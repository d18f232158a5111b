"""Timing of the online controller's "actual" run (actuator noise, the actual run's event script) as ONE launch of the
device-resident loop (math_mpc_batch(..., isActual=True, device_noise=True)), next to the per-tick path that draws the
noise on the host (one batched launch per tick) and to the noise-free device loop on the same robots.  Host clock
around the synchronising call, after one warm-up call of the same shape.  The math_mpc_batch rows with rngs= include
handing the generators' states over (RandomState.get_state / set_state, ~0.1 ms per robot in numpy); the "solver call"
rows time Solver.held_closed_loop alone on states packed beforehand, with and without them, so the loop's own cost
shows.  The seeded rows build the same generators on the device from the integer seeds instead (seeds=): through
math_mpc_batch, through the host entry (final states copied back), and as seeding kernel + device-pointer loop on torch
tensors; the seeding kernel alone is timed with CUDA events.  Each seeded row says whether its outputs equal the rngs
path's (math_mpc_batch rows) or the packed-state solver call's.
usage: python tools/actual_loop_timing.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import time, numpy as np, importlib, torch
mt = importlib.import_module("diplomjourney_b200.math_model_tree")
from diplomjourney_b200 import _native as nat, config
params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, 400)
rng = np.random.default_rng(1)
OUT = ("ticks", "status", "log", "final")


def timed(**kw):
    t0 = time.perf_counter()
    r = mt.math_mpc_batch(init, tgt, max_ticks=400, origin=org, events=True, **kw)
    return time.perf_counter() - t0, r


def line(name, dt, r):
    return (f"{name} N={n}: {dt * 1e3:.2f} ms, {r['ticks'].sum()} ticks, {r['ticks'].sum() / dt:.3e} ticks/s, "
            f"status {np.bincount(r['status'], minlength=4)}")


def equal(a, b, keys=OUT):
    return all(np.array_equal(a[k], b[k], equal_nan=k in ("log", "final")) for k in keys)


def seed_kernel_ms(s, ext, n, keys, key_len, out, reps=20):
    """mean time of one seeding launch, CUDA events around `reps` launches on the solver's stream"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(ext):
        s.seed_generators_device(n, keys.data_ptr(), key_len, out.data_ptr())          # warm-up
        e0.record(ext)
        for _ in range(reps):
            s.seed_generators_device(n, keys.data_ptr(), key_len, out.data_ptr())
        e1.record(ext)
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


s = mt._solver()
ext = torch.cuda.ExternalStream(s.stream)
for n in (1, 1024, 16384):
    init = np.zeros((n, 5)); init[:, :2] = rng.uniform(-1, 1, (n, 2)); init[:, 2] = rng.uniform(-0.5, 7, n)
    tgt = np.tile([2.0, 3.0], (n, 1)) + rng.uniform(-1, 1, (n, 2))
    org = np.zeros((n, 2))
    seeds = rng.integers(0, 2 ** 32, n)
    gens = lambda: [np.random.RandomState(x) for x in seeds]
    timed(isActual=True, device_noise=True, rngs=gens())                    # warm-up
    dt, r = timed(isActual=True, device_noise=True, rngs=gens())
    print(line("device loop, actuator noise", dt, r), flush=True)
    timed(isActual=True, device_noise=True, seeds=seeds)
    dt, rs = timed(isActual=True, device_noise=True, seeds=seeds)
    print(line("device loop, actuator noise, seeded on the device", dt, rs) + f", equal to the rngs path: {equal(rs, r)}",
          flush=True)
    timed()
    dt, r0 = timed()
    print(line("device loop, noise-free", dt, r0), flush=True)
    packed = mt._pack_generators(gens())
    kw = dict(first_threshold=1e10, events=mt.ACTUAL_EVENTS, radius_u_turn=mt.radius_u_turn)
    for name, extra in (("solver call, actuator noise", dict(rng_state=packed)), ("solver call, noise-free", {})):
        call = lambda: s.held_closed_loop(params, init, tgt, org, **kw, **extra)
        call()
        t0 = time.perf_counter(); rc = call(); dt = time.perf_counter() - t0
        print(line(name, dt, rc), flush=True)
        if extra:
            ref = rc
    call = lambda: s.held_closed_loop(params, init, tgt, org, seeds=seeds, **kw)
    call()
    t0 = time.perf_counter(); rh = call(); dt = time.perf_counter() - t0
    print(line("seeded host entry, actuator noise", dt, rh) +
          f", equal to the packed-state solver call (generators too): {equal(rh, ref, OUT + ('rng_state',))}", flush=True)

    # the same run on torch tensors: seeding kernel + mpcb_held_closed_loop_actual_device, no host copy
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    d_init, d_tgt, d_org, d_thr = dev(init), dev(tgt), dev(org), dev(np.full(n, 1e10))
    d_keys = dev(seeds.astype(np.uint32).view(np.int32))
    d_rng = torch.empty((n, 625), dtype=torch.int32, device="cuda")
    d_log = torch.empty((n, 400, 5), dtype=torch.float64, device="cuda")
    d_tk, d_st = (torch.empty(n, dtype=torch.int32, device="cuda") for _ in range(2))
    d_fin = torch.empty((n, 6), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()

    def device_run():
        with torch.cuda.stream(ext):
            d_log.fill_(float("nan"))
            s.seed_generators_device(n, d_keys.data_ptr(), 0, d_rng.data_ptr())
            s.held_closed_loop_device_actual(params, n, d_init.data_ptr(), d_tgt.data_ptr(), d_org.data_ptr(),
                                             d_thr.data_ptr(), 0, d_rng.data_ptr(), d_log.data_ptr(), d_tk.data_ptr(),
                                             d_st.data_ptr(), d_fin.data_ptr(), events=mt.ACTUAL_EVENTS,
                                             radius_u_turn=mt.radius_u_turn)
        s.sync()

    device_run()
    t0 = time.perf_counter(); device_run(); dt_dev = time.perf_counter() - t0
    rd = dict(log=d_log.cpu().numpy(), ticks=d_tk.cpu().numpy(), status=d_st.cpu().numpy(), final=d_fin.cpu().numpy(),
              rng_state=d_rng.cpu().numpy().view(np.uint32))
    print(line("seeding + device loop on torch tensors, actuator noise", dt_dev, rd) +
          f", equal to the packed-state solver call (generators too): {equal(rd, ref, OUT + ('rng_state',))}", flush=True)
    ms = seed_kernel_ms(s, ext, n, d_keys, 0, d_rng)
    print(f"seeding kernel alone N={n}: {ms * 1e3:.1f} us per launch (CUDA events, mean of 20), "
          f"{ms / (dt_dev * 1e3) * 100:.2f} % of the torch-tensor row", flush=True)
    if n == 1024:
        dt, h = timed(isActual=True, rngs=gens())
        same = np.array_equal(h["ticks"], r["ticks"]) and np.allclose(h["log"], r["log"], rtol=0, atol=1e-9, equal_nan=True)
        print(line("per-tick path, actuator noise", dt, h) + f", equal to the device loop: {same}", flush=True)

n = 65536
big = rng.integers(0, 2 ** 32, (n, 3)).astype(np.uint32)
d_rng = torch.empty((n, 625), dtype=torch.int32, device="cuda")
for key_len, keys in ((0, big[:, 0]), (3, big)):
    d_keys = torch.from_numpy(np.ascontiguousarray(keys).view(np.int32)).cuda()
    torch.cuda.synchronize()
    ms = seed_kernel_ms(s, ext, n, d_keys, key_len, d_rng)
    print(f"seeding kernel alone N={n}, key_len={key_len}: {ms * 1e3:.1f} us per launch (CUDA events, mean of 20), "
          f"{n * 625 * 4 / (ms * 1e-3) / 1e9:.0f} GB/s of records written", flush=True)
