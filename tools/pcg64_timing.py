"""Timing of the actual run (actuator noise, the actual run's event script) with numpy's Generator(PCG64) streams on the
device, next to the same run with legacy RandomState (MT19937) streams, both seeded on the device, at N = 1,024 and
16,384 robots.  Three rows per generator kind:
  solver call   Solver.held_closed_loop(seeds=) / (pcg_seeds=): host clock around the synchronising call (seed words
                up, seeding kernel, loop, results and final states down), after a warm-up call; the two kinds alternate,
                three calls each, median and spread printed;
  loop alone    the device-pointer loop (mpcb_held_closed_loop_actual_device / _pcg64_device) on torch tensors, CUDA
                events around the launch, generators restored from a seeded copy before each of five launches, mean;
  seeding       the seeding kernel alone (mpcb_rng_seed_device / mpcb_pcg64_seed_device), CUDA events, mean of 20.
Each kind's loop outputs are checked against its own solver call, and the PCG64 solver call against the rngs=[default_rng]
path of math_mpc_batch.  numpy's SeedSequence.spawn(N), with which the PCG64 solver call advances its SeedSequence on
the host, is timed alone too.
usage: python tools/pcg64_timing.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import importlib, statistics, subprocess, time
import numpy as np, torch
mt = importlib.import_module("diplomjourney_b200.math_model_tree")
from diplomjourney_b200 import _native as nat, config

TICKS = 400
params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, TICKS)
OUT = ("ticks", "status", "log", "final")
kw = dict(first_threshold=1e10, events=mt.ACTUAL_EVENTS, radius_u_turn=mt.radius_u_turn)


def equal(a, b, keys=OUT):
    return all(np.array_equal(a[k], b[k], equal_nan=k in ("log", "final")) for k in keys)


def events_ms(ext, fn, reps, before=None):
    """mean device time of fn() over reps launches on the solver's stream, CUDA events around each launch"""
    total = 0.0
    for _ in range(reps):
        if before:
            before()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(ext):
            e0.record(ext)
            fn()
            e1.record(ext)
        e1.synchronize()
        total += e0.elapsed_time(e1)
    return total / reps


try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()[0]
except (OSError, IndexError):
    card = torch.cuda.get_device_name(0)
print(f"device: {card}", flush=True)
s = mt._solver()
ext = torch.cuda.ExternalStream(s.stream)
rng = np.random.default_rng(5)
for n in (1024, 16384):
    init = np.zeros((n, 5)); init[:, :2] = rng.uniform(-1, 1, (n, 2)); init[:, 2] = rng.uniform(-0.5, 7, n)
    init[:, 3] = rng.choice([0.0, 0.3, 0.6], n)
    tgt = np.tile([2.0, 3.0], (n, 1)) + rng.uniform(-1, 1, (n, 2))
    org = np.zeros((n, 2))
    mt_seeds = rng.integers(0, 2 ** 32, n)
    root_entropy = int(rng.integers(0, 2 ** 63))
    calls = {"MT19937": lambda: s.held_closed_loop(params, init, tgt, org, seeds=mt_seeds, **kw),
             "PCG64": lambda: s.held_closed_loop(params, init, tgt, org, pcg_seeds=np.random.SeedSequence(root_entropy), **kw)}
    times = {k: [] for k in calls}
    res = {k: c() for k, c in calls.items()}            # warm-up
    for _ in range(3):
        for k, c in calls.items():
            t0 = time.perf_counter(); res[k] = c(); times[k].append(time.perf_counter() - t0)
    for k in calls:
        r = res[k]
        print(f"solver call, {k:7s} N={n}: median {statistics.median(times[k]) * 1e3:.2f} ms "
              f"(calls {', '.join(f'{t * 1e3:.2f}' for t in times[k])} ms), {r['ticks'].sum()} ticks, "
              f"{r['ticks'].sum() / statistics.median(times[k]):.3e} ticks/s", flush=True)
    t0 = time.perf_counter(); kids = np.random.SeedSequence(root_entropy).spawn(n); dt = time.perf_counter() - t0
    print(f"host, SeedSequence.spawn({n}) alone (the PCG64 solver call advances its SeedSequence with it): "
          f"{dt * 1e3:.2f} ms", flush=True)
    via_rngs = mt.math_mpc_batch(init, tgt, max_ticks=TICKS, origin=org, isActual=True, events=True, device_noise=True,
                                 rngs=[np.random.default_rng(c) for c in kids])
    print(f"PCG64 solver call equal to math_mpc_batch(rngs=[default_rng(child)]): {equal(res['PCG64'], via_rngs)}",
          flush=True)

    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    d_init, d_tgt, d_org, d_thr = dev(init), dev(tgt), dev(org), dev(np.full(n, 1e10))
    d_log = torch.empty((n, TICKS, 5), dtype=torch.float64, device="cuda")
    d_tk, d_st = (torch.empty(n, dtype=torch.int32, device="cuda") for _ in range(2))
    d_fin = torch.empty((n, 6), dtype=torch.float64, device="cuda")
    d_keys = dev(mt_seeds.astype(np.uint32).view(np.int32))
    ent, stride, spawn = nat.pcg64_seed_words(np.random.SeedSequence(root_entropy), n)
    d_ent, d_spawn = dev(ent.view(np.int32)), dev(spawn.view(np.int32))
    gens = {"MT19937": torch.empty((n, 625), dtype=torch.int32, device="cuda"),
            "PCG64": torch.empty((n, 6), dtype=torch.int64, device="cuda")}
    seed = {"MT19937": lambda: s.seed_generators_device(n, d_keys.data_ptr(), 0, gens["MT19937"].data_ptr()),
            "PCG64": lambda: s.seed_pcg64_device(n, d_ent.data_ptr(), ent.size, stride, d_spawn.data_ptr(),
                                                 spawn.shape[1], gens["PCG64"].data_ptr())}
    loop = {"MT19937": lambda: s.held_closed_loop_device_actual(
                params, n, d_init.data_ptr(), d_tgt.data_ptr(), d_org.data_ptr(), d_thr.data_ptr(), 0,
                gens["MT19937"].data_ptr(), d_log.data_ptr(), d_tk.data_ptr(), d_st.data_ptr(), d_fin.data_ptr(),
                events=mt.ACTUAL_EVENTS, radius_u_turn=mt.radius_u_turn),
            "PCG64": lambda: s.held_closed_loop_device_pcg64(
                params, n, d_init.data_ptr(), d_tgt.data_ptr(), d_org.data_ptr(), d_thr.data_ptr(), 0,
                gens["PCG64"].data_ptr(), d_log.data_ptr(), d_tk.data_ptr(), d_st.data_ptr(), d_fin.data_ptr(),
                events=mt.ACTUAL_EVENTS, radius_u_turn=mt.radius_u_turn)}
    for k in ("MT19937", "PCG64"):
        with torch.cuda.stream(ext):
            seed[k]()
        s.sync()
        seeded = gens[k].clone()

        def restore():
            with torch.cuda.stream(ext):
                gens[k].copy_(seeded)
                d_log.fill_(float("nan"))
            s.sync()

        restore(); loop[k](); s.sync()                  # warm-up
        ms = events_ms(ext, loop[k], 5, restore)
        out = dict(log=d_log.cpu().numpy(), ticks=d_tk.cpu().numpy(), status=d_st.cpu().numpy(), final=d_fin.cpu().numpy())
        print(f"loop alone,  {k:7s} N={n}: {ms:.2f} ms per launch (CUDA events, mean of 5), "
              f"equal to its solver call: {equal(out, res[k])}", flush=True)
        seed[k](); s.sync()
        sm = events_ms(ext, seed[k], 20)
        rec_bytes = n * (625 * 4 if k == "MT19937" else 48)
        print(f"seeding,     {k:7s} N={n}: {sm * 1e3:.1f} us per launch (CUDA events, mean of 20), "
              f"{rec_bytes / (sm * 1e-3) / 1e9:.1f} GB/s of records written", flush=True)
