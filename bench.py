#!/usr/bin/env python
"""bench.py -- MPC inner-loop benchmark (BASELINE.json metric: candidate rollouts/s and MPC solves/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg2|cfg4] [--dump-outputs DIR]

Headline workload at every N (weak scaling: fixed work per GPU, robots are independent -- no collective):
  cfg2 = BASELINE.json configs[1]: 1,024 independent robots per GPU, horizon 3, FULL tree
  (math_model.py:159-200) with the MM tracking cost (math_model.py:82-86) on the default
  acceleration-window control grid 11 x 41 (math_model_tree.py:239-256 at v=0.5, beta=0; S=451):
  91,733,851 leaf rollouts per robot, 9.39e10 per step.  Scenarios: numpy default_rng(0) over the
  distribution of run_math_model.py:235-239.  A "step" is one batched solve of all robots.

One JSON line on stdout (rank 0).  `value` = rollouts/s with inputs resident in HBM (device
API, CUDA events on the library's stream, max over ranks); `e2e` = the same through the
host-buffer C-ABI call (pinned host inputs copied H2D and results copied D2H inside the timed
region).  Further legs of the same line:
  cfg4_strong  BASELINE configs[3]: all 65,536 scenarios (H=4, 16x16 grid) sharded by contiguous ranges over the N
               GPUs -- strong scaling, no collective -- with 32 of them re-solved exhaustively
  split_tree   (N > 1) BASELINE configs[4]: ONE tree (H=6, 16x16 grid, 2.8e14 leaves) split over the N GPUs by first
               control and reconciled by the library's own NCCL all-gather of 16-byte (cost, index) records
  bigtree      (N = 1) configs[2] / configs[4] whole trees on one GPU over 64 seeded scenarios each
  leafwalk     (N = 1) the one-thread-per-leaf kernel north_star prescribes, on the same workload
`--impl reference` times the CPU port of the reference path (oracle/ref_port.py: per-node scipy.integrate.quad,
Python loops) on all host cores, on a bounded slice of the same workload.
"""
from __future__ import annotations

import argparse
import glob
import json
import math
import os
import re
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the bench leaves the tree as it found it (it may be read-only)

import numpy as np  # noqa: E402

H = 3
N_ROBOTS = 1024
SM_COUNT = 148
MUFU_PER_CLK_SM = 16       # XU lanes per SM per clock (SURVEY 8d)
FP32_PER_CLK_SM = 128

# What the pass-1 kernels execute per rollout: FP32-pipe lane slots (an FFMA2 / FADD2 is two) and XU operations counted
# in the SASS of their inner loops (profiles/r2_sass_loops.txt; tools/sass_loops.py prints them from the built library),
# instr = warp instructions x 32 / rollouts of the whole kernel as ncu counts them (smsp__inst_executed.sum,
# profiles/r2j_cfg2_full.txt, r2j_leafwalk_full.txt, r1l_cfg2_full.txt).
EXECUTED = {
    # row screen loop of prefixn_kernel<.,2,true>: per node and leaf PAIR 7 FFMA2 + 1 FADD2 + 1 FMNMX3 + 1/2 (LDS.128 + LDS.64),
    # no MUFU; one more FFMA per node and speed ROW (fma(kWd^2, r, D2s), 1/42 per rollout on the 11 x 41 grid)
    "prefix_screen": dict(kernel="prefixn_kernel<true,2,true> (pass 1, row screen loop)", fp32=8.05, mufu=0.0, instr=6.1),
    # full loop of prefixn_kernel<.,2,false>: per node and leaf pair 7 FFMA2 + 1 FADD2 + 2 MUFU.SQRT + 1 FMNMX3 + 1 LDS.128
    "prefix_full": dict(kernel="prefixn_kernel<true,2,false> (pass 1)", fp32=8.0, mufu=1.0, instr=6.95),
    # leafwalk_kernel<1,true,1>, H=3: 7 MUFU (sin + cos per step, one sqrt), 15 scalar FP32 ops, 56.6 instructions in all
    "leafwalk": dict(kernel="leafwalk_kernel<1,true,1> (pass 1)", fp32=15.0, mufu=7.0, instr=56.6),
}


def workload(name):
    from oracle import closed_form as C
    if name == "cfg4":   # configs[3] shape, trimmed batch: 16x16 grid, H=4 (4.29e9 leaves per scenario)
        V = np.linspace(0.0, 1.0, 16)
        B = np.linspace(-math.radians(60), math.radians(60), 16)
        return dict(name="cfg4: FULL tree, H=4, 16x16 linspace grid (S=256), MM cost", V=V, B=B, H=4, n=32, seed=1)
    V, B = C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0)
    return dict(name="cfg2: 1024 robots/GPU, FULL tree, H=3, acceleration-window grid 11x41 (S=451), MM cost",
                V=np.array(V), B=np.array(B), H=3, n=N_ROBOTS, seed=0)


def config_of(wl):
    """The `config` object of the JSON line -- the same keys from both arms."""
    S = len(wl["V"]) * len(wl["B"])
    return dict(workload=wl["name"], robots_per_gpu=wl["n"], H=wl["H"], S=S, leaves_per_solve=S ** wl["H"],
                l2="flushed between timed steps (256 MiB fill)", selection="float64 first-minimum argmin")


def peaks():
    p = dict(sm_max_mhz=1965.0, hbm_gbs=6650.0, src="fallback")
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            m = json.load(f)
        p.update(sm_max_mhz=float(m["sm_max_mhz"]), hbm_gbs=float(m["hbm_gbs"]), src="measured")
    except Exception:
        pass
    return p


def ncu_record(kernel_key):
    """Figures of the committed ncu --set full capture of the dominant kernel (profiles/*_full.txt, newest round first):
    DRAM traffic per launch and the pipe utilisations.  None when no capture of that kernel is committed."""
    want = {"prefix_screen": r"prefixn_kernel<1, 2, 1>", "prefix_full": r"prefixn_kernel<1, 2(, 0)?>\(",
            "leafwalk": r"leafwalk_kernel<1, 1, 1>"}[kernel_key]
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_full.txt")), reverse=True):
        try:
            txt = open(path).read()
        except OSError:
            continue
        for block in txt.split("\n== ")[1:]:
            if not re.search(want, block.splitlines()[0]):
                continue
            def val(name):
                m = re.search(r"^" + re.escape(name) + r" = ([0-9.eE+-]+) ?(\S*)", block, re.M)
                if not m:
                    return None
                scale = {"Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "byte": 1.0}.get(m.group(2), 1.0)
                return float(m.group(1)) * scale
            rd, wr = val("dram__bytes_read.sum"), val("dram__bytes_write.sum")
            return dict(file=os.path.relpath(path, ROOT), traffic=None if rd is None else int(rd + (wr or 0.0)),
                        fma_pipe_pct=val("sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active"),
                        xu_pipe_pct=val("sm__inst_executed_pipe_xu.avg.pct_of_peak_sustained_active"),
                        issue_pct=val("smsp__issue_active.avg.pct_of_peak_sustained_active"),
                        kernel_ms=val("gpu__time_duration.sum"))
    return None


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
                getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
            }
            while not self._stop_evt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.02)
        except Exception as e:  # NVML missing: report it rather than fail the bench
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        busy = s[len(s) // 4:] if s else []
        return dict(sm_mhz=(statistics.median(busy) if busy else None), sm_max_mhz=self.max_mhz,
                    reasons=sorted(self.reasons), samples=len(s))


def cpu_sample(wl, seconds_target=12.0, procs=None):
    """Bounded sample of the same workload on the host cores with the reference-style port."""
    from oracle import closed_form as C
    from oracle import ref_port as P
    procs = procs or os.cpu_count() or 1
    scen = C.random_scenarios(max(procs, 8), wl["seed"])
    S = len(wl["V"]) * len(wl["B"])
    if wl["H"] != 3:
        raise SystemExit("the reference CPU path is hard-coded to H=3 (math_model.py:160-186)")
    # ~33 us per leaf per core (measured on the B200 box's hosts) -> second-level subtrees per process for ~12 s
    n_i1 = max(1, min(S, int(seconds_target / (33e-6 * S))))
    leaves, wall, per = P.timed_sample_full(list(wl["V"]), list(wl["B"]), scen, "mm", n_i1, procs)
    return dict(value=leaves / wall, unit="rollouts/s", cores=procs, kind="port",
                sample=f"{procs} processes x {n_i1} second-level subtrees ({n_i1 * S} leaves each) of the FULL H=3 "
                       f"S={S} tree, per-node scipy.integrate.quad as in math_model.py:90-114; {wall:.1f}s wall",
                rollouts_per_s_per_core=leaves / sum(per))


def closed_form_cpu(wl):
    """The same solve with the float64 closed-form C port on all cores (context, not the baseline)."""
    from oracle import c_oracle as K
    from oracle import closed_form as C
    s = C.random_scenarios(2, wl["seed"])
    K.solve_full(s[0][:3], s[0][3:5], s[0][:2], wl["V"], wl["B"], wl["H"])   # warm (builds the .so)
    t = time.perf_counter()
    K.solve_full(s[1][:3], s[1][3:5], s[1][:2], wl["V"], wl["B"], wl["H"])
    dt = time.perf_counter() - t
    S = len(wl["V"]) * len(wl["B"])
    return dict(value=S ** wl["H"] / dt, unit="rollouts/s", cores=os.cpu_count(),
                note="oracle/mpc_oracle.c: float64 closed form with prefix sharing, pthreads, 1 solve")


def held_metrics(solver, nat, C, device_index):
    """MPC solves/s of the online (HELD, CoordinateTree-pruned) controller -- the other half of the
    BASELINE metric: (a) whole closed loops resident on the device for a batch of robots,
    (b) one tick through the reference-API call on host buffers, (c) a 1,024-robot batch on the
    FULL scripts' 201x121 grid (S=24,321 candidates per solve)."""
    from diplomjourney_b200 import config
    out = {}
    rng = np.random.default_rng(0)
    n = 4096
    params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, 256)
    init = np.zeros((n, 5)); init[:, 2] = rng.uniform(-1, 1, n)
    ang = init[:, 2] + rng.uniform(-0.5, 0.5, n); d = rng.uniform(1.0, 4.0, n)
    tgt = np.stack([d * np.cos(ang), d * np.sin(ang)], 1)
    for _ in range(3):
        t = time.perf_counter()
        r = solver.held_closed_loop(params, init, tgt, [[0.0, 0.0]], first_threshold=1e10)
        dt = time.perf_counter() - t
    out["closed_loop_batch"] = dict(robots=n, ticks=int(r["ticks"].sum()), seconds=dt,
                                    solves_per_s=float(r["ticks"].sum() / dt), S_max=451,
                                    note="mpcb_held_closed_loop_host: whole math_mpc loops on the device, host wall incl. copies")
    V, B = C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0)
    x = C.random_scenarios(1, 3)[0]
    reps = 300
    cfgv = (C.CONFIG["L"], C.CONFIG["delta_t"], C.CONFIG["v_min"])

    def per_call(fn):
        fn()
        t = time.perf_counter()
        for _ in range(reps):
            fn()
        return (time.perf_counter() - t) / reps

    def generic():
        solver.set_grid(V, B, *cfgv)
        solver.solve(nat.MODE_HELD, nat.COST_TREE, 3, x[:3], x[3:5], x[:2])

    def tick():
        solver.held_tick(V, B, *cfgv, nat.COST_TREE, 3, x[:3], x[3:5], x[:2])

    dt = per_call(generic)
    out["single_tick_host_api"] = dict(us_per_solve=dt * 1e6, solves_per_s=1.0 / dt, S=len(V) * len(B),
                                       note="Solver.set_grid + Solver.solve per tick (two C calls, numpy marshalling): host "
                                            "buffers, one launch, one synchronisation")
    dt = per_call(tick)
    solver.set_option("zero_copy", 0)
    dt_staged = per_call(tick)
    solver.set_option("zero_copy", 1)
    out["single_tick_c_abi"] = dict(us_per_solve=dt * 1e6, solves_per_s=1.0 / dt, us_per_solve_staged_copies=dt_staged * 1e6,
                                    note="mpcb_held_tick_host through ctypes (what math_model_tree.predictive_control calls): "
                                         "window lists + one HELD solve in one C call; inputs and results in mapped pinned "
                                         "host memory (one launch, one synchronisation, no copy); staged = one copy each way")
    if hasattr(solver, "solve_held_windows"):
        # 1,024 robots with DIFFERENT (v, beta): per-robot acceleration windows built on the device, one launch
        m = 1024
        sc = C.random_scenarios(m, 5)
        vb = np.stack([rng.uniform(0.0, 0.99, m), rng.uniform(-1.0, 1.0, m)], 1)
        for _ in range(3):
            t = time.perf_counter()
            solver.solve_held_windows(params, sc[:, :3], vb, sc[:, 3:5], sc[:, :2])
            dt = time.perf_counter() - t
        out["batch_per_robot_windows"] = dict(robots=m, seconds=dt, solves_per_s=m / dt,
                                              note="mpcb_solve_held_windows_host: one tick of 1,024 robots, each with its own "
                                                   "acceleration window (math_model_tree.py:239-256) built on the device")
    Vf, Bf = C.grid_full_default()
    solver.set_grid(Vf, Bf, C.CONFIG["L"], C.CONFIG["delta_t"], C.CONFIG["v_min"])
    sc = C.random_scenarios(1024, 1)
    for _ in range(3):
        t = time.perf_counter()
        solver.solve(nat.MODE_HELD, nat.COST_TREE, 3, sc[:, :3], sc[:, 3:5], sc[:, :2])
        dt = time.perf_counter() - t
    out["batch_201x121"] = dict(robots=1024, S=int(Vf.size * Bf.size), seconds=dt, solves_per_s=1024 / dt,
                                rollouts_per_s=1024 * Vf.size * Bf.size / dt)
    return out


BIGTREES = (("configs[2] H=5 32x32", 5, 32), ("configs[4] H=6 16x16", 6, 16))


def bigtree_scenarios(C, n=64):
    """Scenario set of the big-tree legs: the config.py scenario, the tie-heavy one (its optimum stands still, 6.3e6
    leaves tie exactly at H=6), a target behind the robot, a target one step away, and seeded random ones over the
    distribution of run_math_model.py:235-239."""
    from diplomjourney_b200 import config as cfg
    named = [("config.py", [cfg.x_0, cfg.y_0, cfg.phi_0, cfg.x_t, cfg.y_t]),
             ("tie-heavy", list(C.random_scenarios(3, 77)[0])),
             ("target behind", [0.0, 0.0, 0.0, -3.0, 0.5]),
             ("target one step away", [0.0, 0.0, 0.3, 0.04, 0.02])]
    rnd = C.random_scenarios(n - len(named), 2)
    return named + [(f"rng(2)[{i}]", list(x)) for i, x in enumerate(rnd)]


def pinned_bigtree():
    """Exhaustive (prune=0) records of the config.py scenario on the big trees, run once on eight GPUs and committed
    (profiles/r2_bigtree_exhaustive.json): the independent pin of the pruned answers."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_bigtree_exhaustive.json")) as f:
            return json.load(f)
    except OSError:
        return {}


def bigtree_metrics(solver, nat, C):
    """BASELINE configs[2] and configs[4]: ONE oversized FULL tree per solve on this GPU through the host API with the
    exact branch-and-bound -- the only way such a tree is solved in finite time.  Pruning is by bounds, so the time
    depends on the scenario: 64 seeded scenarios per tree, median / p90 / worst reported, the config.py scenario
    checked against the committed exhaustive record."""
    from diplomjourney_b200 import config as cfg
    out = {}
    pins = pinned_bigtree()
    scen = bigtree_scenarios(C)
    solver.set_option("prune", 1)
    for name, Hh, n in BIGTREES:
        V = np.linspace(0.0, cfg.v_max, n)
        B = np.linspace(-cfg.beta_max, cfg.beta_max, n)
        solver.set_grid(V, B, cfg.L, cfg.delta_t, cfg.v_min)
        solver.solve(nat.MODE_FULL, nat.COST_MM, Hh, scen[0][1][:3], scen[0][1][3:5], scen[0][1][:2])     # tables, scratch
        times, rec = [], {}
        for label, x in scen:
            t = time.perf_counter()
            r = solver.solve(nat.MODE_FULL, nat.COST_MM, Hh, x[:3], x[3:5], x[:2])
            times.append(time.perf_counter() - t)
            rec[label] = (int(r["index"][0]), float(r["cost"][0]))
        stt = solver.stats()
        order = np.argsort(times)
        pin = pins.get(name)
        entry = dict(leaves=int(stt["leaves_per_solve"]), scenarios=len(scen),
                     seconds_median=float(np.median(times)), seconds_p90=float(np.percentile(times, 90)),
                     seconds_worst=float(max(times)), worst_scenario=scen[int(order[-1])][0],
                     seconds_config_py=times[0], seconds_tie_heavy=times[1],
                     solves_per_s_median=1.0 / float(np.median(times)),
                     config_py=dict(leaf=rec["config.py"][0], cost=rec["config.py"][1]))
        if pin:
            same = pin["leaf"] == rec["config.py"][0] and pin["cost"] == rec["config.py"][1]
            entry["config_py"]["exhaustive_pin"] = dict(file="profiles/r2_bigtree_exhaustive.json", same=bool(same),
                                                        exhaustive_seconds=pin.get("seconds"), gpus=pin.get("gpus"))
            if not same:
                raise SystemExit(f"PARITY FAILURE in bench: pruned {name} answer {rec['config.py']} differs from the exhaustive pin {pin}")
        out[name] = entry
    solver.set_option("prune", 0)
    return out


def run_reference(args):
    wl = workload(args.workload)
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    for i in range(args.warmup + args.steps):
        r = cpu_sample(wl, seconds_target=float(os.environ.get("MPCB_CPU_SAMPLE_SECONDS", "6.0")))
        if i >= args.warmup:
            vals.append(r)
    v = statistics.mean(x["value"] for x in vals)
    last = vals[-1]
    S = len(wl["V"]) * len(wl["B"])
    line = dict(metric="candidate rollouts/s (MPC inner loop)", value=v, unit="rollouts/s", impl="reference",
                n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * (S ** wl["H"] * wl["n"]) / v, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f64", data="synthetic", config=config_of(wl),
                solves_per_s=v / S ** wl["H"],
                cpu_baseline=dict(value=v, unit="rollouts/s", cores=last["cores"], kind="port", sample=last["sample"]),
                e2e=dict(value=v, unit="rollouts/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                note="ms_per_step is extrapolated from the timed slice: the reference cannot finish one step")
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ multi-GPU legs
def leg_cfg4_strong(solver, nat, C, torch, dist, dev, ext, world, rank, n_total):
    """BASELINE configs[3]: `n_total` scenarios (default_rng(1)), H=4, 16x16 grid, FULL tree (4.29e9 leaves each),
    sharded by contiguous ranges over the ranks -- STRONG scaling, no data-path collective.  Exact branch-and-bound
    (the library default); 32 scenarios are re-solved with prune=0 (every leaf evaluated) and compared bit for bit.
    Device API on resident inputs, CUDA events on the library's stream, max over ranks."""
    from diplomjourney_b200.distributed import shard_range
    Hh = 4
    V = np.linspace(0.0, 1.0, 16)
    B = np.linspace(-math.radians(60), math.radians(60), 16)
    solver.set_grid(V, B, C.CONFIG["L"], C.CONFIG["delta_t"], C.CONFIG["v_min"])
    solver.set_option("prune", 1)
    sc_all = C.random_scenarios(n_total, 1)
    lo, hi = shard_range(n_total, world, rank)
    sc = sc_all[lo:hi]
    n = hi - lo
    st = torch.from_numpy(np.ascontiguousarray(sc[:, :3])).to(dev)
    tg = torch.from_numpy(np.ascontiguousarray(sc[:, 3:5])).to(dev)
    og = torch.from_numpy(np.ascontiguousarray(sc[:, :2])).to(dev)
    oc = torch.empty(n, dtype=torch.float64, device=dev)
    oi = torch.empty(n, dtype=torch.int64, device=dev)
    ou = torch.empty(n, 2, dtype=torch.float64, device=dev)
    chunk = 4096

    def run(i0, i1, c, i, u):
        for b in range(i0, i1, chunk):
            e = min(b + chunk, i1)
            solver.solve_device(nat.MODE_FULL, nat.COST_MM, Hh, e - b, st[b:e].data_ptr(), tg[b:e].data_ptr(),
                                og[b:e].data_ptr(), 0, 0, c[b - i0:].data_ptr(), i[b - i0:].data_ptr(), 0,
                                u[b - i0:].data_ptr())

    with torch.cuda.stream(ext):
        run(0, min(n, 256), oc, oi, ou)                       # warm-up: tables, scratch
    solver.sync()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(ext):
        e0.record()
        run(0, n, oc, oi, ou)
        e1.record()
    solver.sync()
    torch.cuda.synchronize()
    sec = torch.tensor([e0.elapsed_time(e1) * 1e-3], dtype=torch.float64, device=dev)
    # checksums over ALL scenarios (identical at every N, or the sharding changed an answer)
    chk = torch.stack([oi.sum().to(torch.float64), oc.sum(), (oi < 0).sum().to(torch.float64)])
    # exhaustive re-solve of this rank's first 32/world scenarios
    k = min(n, max(1, 32 // world))
    solver.set_option("prune", 0)
    xc = torch.empty(k, dtype=torch.float64, device=dev)
    xi = torch.empty(k, dtype=torch.int64, device=dev)
    xu = torch.empty(k, 2, dtype=torch.float64, device=dev)
    x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(ext):
        x0.record()
        run(0, k, xc, xi, xu)
        x1.record()
    solver.sync()
    torch.cuda.synchronize()
    same = bool(torch.equal(xi, oi[:k]) and torch.equal(xc, oc[:k]) and torch.equal(xu, ou[:k]))
    ex_sec = torch.tensor([x0.elapsed_time(x1) * 1e-3], dtype=torch.float64, device=dev)
    bad = torch.tensor([0.0 if same else 1.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(sec, op=dist.ReduceOp.MAX)
        dist.all_reduce(ex_sec, op=dist.ReduceOp.MAX)
        dist.all_reduce(chk, op=dist.ReduceOp.SUM)
        dist.all_reduce(bad, op=dist.ReduceOp.SUM)
    if float(bad[0]) != 0.0:
        raise SystemExit("PARITY FAILURE in bench: cfg4_strong pruned and exhaustive solves disagree")
    leaves = (len(V) * len(B)) ** Hh
    oracle = None
    if rank == 0:
        from oracle import c_oracle as K
        o = K.solve_full(sc[0, :3], sc[0, 3:5], sc[0, :2], V, B, Hh, C.COST_MM)
        ok = int(oi[0]) == o["index"] and abs(float(oc[0]) - o["cost"]) <= 1e-12 * abs(o["cost"])
        oracle = f"scenario 0 vs the float64 C oracle: {'identical' if ok else 'MISMATCH'}"
        if not ok:
            raise SystemExit("PARITY FAILURE in bench: cfg4_strong " + oracle)
    solver.set_option("prune", 1)
    return dict(workload=f"configs[3]: {n_total} scenarios, FULL tree, H=4, 16x16 grid (S=256), MM cost, sharded by "
                         f"contiguous ranges over {world} GPU(s)", scaling="strong", scenarios=n_total,
                leaves_per_scenario=leaves, seconds=float(sec[0]), solves_per_s=n_total / float(sec[0]),
                effective_rollouts_per_s=n_total * leaves / float(sec[0]), mode="exact branch-and-bound (prune=1)",
                checksum=dict(index_sum=int(chk[0]), cost_sum=float(chk[1]), no_leaf=int(chk[2])),
                exhaustive_check=dict(scenarios=k * world, identical=True, seconds=float(ex_sec[0]),
                                      rollouts_per_s=k * world * leaves / float(ex_sec[0])),
                oracle=oracle, collective="none (independent scenarios)")


def leg_split_tree(solver, nat, C, torch, dist, dev, ext, world, rank):
    """BASELINE configs[4]: ONE robot, H=6, 16x16 grid = 2.815e14 leaves, split over the ranks by contiguous ranges
    of the first control (mpcb_solve_tree_split_device): every rank solves its share, ONE ncclAllGather of the
    16-byte (cost, index) records on the library's own communicator, local lexicographic minimum, local re-roll of
    the winner.  CUDA events on the library's stream, max over ranks; the records of all ranks must agree, and equal
    a whole-tree solve on one GPU.  Scenarios: config.py and the tie-heavy one."""
    from diplomjourney_b200 import config as cfg
    ids = [nat.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    comm = nat.NcclComm(solver, world, rank, ids[0])
    V = np.linspace(0.0, cfg.v_max, 16)
    B = np.linspace(-cfg.beta_max, cfg.beta_max, 16)
    solver.set_grid(V, B, cfg.L, cfg.delta_t, cfg.v_min)
    S = 256
    out = dict(communicator="library-owned NCCL communicator (mpcb_nccl_comm_create), one 16-byte all-gather per solve",
               runs=[])
    scen = [("config.py", np.array([cfg.x_0, cfg.y_0, cfg.phi_0, cfg.x_t, cfg.y_t], dtype=np.float64)),
            ("tie-heavy", np.array(C.random_scenarios(3, 77)[0], dtype=np.float64))]
    oc = torch.empty(1, dtype=torch.float64, device=dev)
    oi = torch.empty(1, dtype=torch.int64, device=dev)
    ot = torch.empty(8 * 3, dtype=torch.float64, device=dev)
    ou = torch.empty(2, dtype=torch.float64, device=dev)
    # (H, prune, repetitions): the config tree with the exact branch-and-bound; a 1.1e12-leaf tree with every leaf
    # evaluated (the split path at rollouts/s scale)
    for Hh, prune, reps in ((6, 1, 3), (5, 0, 1)):
        for label, x in scen:
            solver.set_option("prune", prune)
            st = torch.from_numpy(x[:3].copy()).to(dev)
            tg = torch.from_numpy(x[3:5].copy()).to(dev)
            og = torch.from_numpy(x[:2].copy()).to(dev)

            def once():
                solver.solve_tree_split_device(comm, nat.COST_MM, Hh, 1, st.data_ptr(), tg.data_ptr(), og.data_ptr(), 0,
                                               oc.data_ptr(), oi.data_ptr(), ot.data_ptr(), ou.data_ptr())
            with torch.cuda.stream(ext):
                once()                                            # warm-up (NCCL connection set-up on the first call)
            solver.sync()
            best = None
            for _ in range(reps):
                dist.barrier()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                with torch.cuda.stream(ext):
                    e0.record()
                    once()
                    e1.record()
                solver.sync()
                torch.cuda.synchronize()
                tt = torch.tensor([e0.elapsed_time(e1) * 1e-3], dtype=torch.float64, device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                best = float(tt[0]) if best is None else min(best, float(tt[0]))
            recs = [None] * world
            dist.all_gather_object(recs, (float(oc[0]), int(oi[0]), ot[:3 * Hh].cpu().numpy().tobytes()))
            agree = all(r == recs[0] for r in recs)
            whole_same = None
            if rank == 0 and prune == 1:                          # the same tree on ONE GPU (no split, no collective)
                w = solver.solve(nat.MODE_FULL, nat.COST_MM, Hh, x[:3], x[3:5], x[:2])
                whole_same = bool(int(w["index"][0]) == recs[0][1] and float(w["cost"][0]) == recs[0][0]
                                  and w["traj"][0].tobytes() == recs[0][2])
            flag = torch.tensor([0.0 if agree and whole_same is not False else 1.0], dtype=torch.float64, device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.SUM)
            if float(flag[0]) != 0.0:
                raise SystemExit(f"PARITY FAILURE in bench: split tree H={Hh} {label}: ranks agree={agree}, equals whole tree={whole_same}")
            leaves = S ** Hh
            out["runs"].append(dict(scenario=label, H=Hh, leaves=leaves, mode="exact branch-and-bound" if prune else "every leaf evaluated",
                                    seconds=best, solves_per_s=1.0 / best, effective_rollouts_per_s=leaves / best,
                                    leaf=recs[0][1], cost=recs[0][0], ranks_agree=True, equals_one_gpu_whole_tree=whole_same))
    # the exhaustive H=5 answers must equal the pruned ones of the same tree
    solver.set_option("prune", 1)
    for label, x in scen:
        w = solver.solve(nat.MODE_FULL, nat.COST_MM, 5, x[:3], x[3:5], x[:2])
        ex = [r for r in out["runs"] if r["H"] == 5 and r["scenario"] == label][0]
        if int(w["index"][0]) != ex["leaf"] or float(w["cost"][0]) != ex["cost"]:
            raise SystemExit(f"PARITY FAILURE in bench: split tree H=5 {label}: exhaustive split and pruned whole tree disagree")
        ex["equals_pruned_whole_tree"] = True
    out["limiter"] = ("pruned: launch latency of the solve chain plus the all-gather (tens of microseconds) against a "
                      "sub-millisecond solve; exhaustive: the pass-1 kernel, the collective is invisible")
    comm.close()
    return out


def leg_leafwalk(solver, nat, C, torch, dev, ext, wl, scen, pk):
    """The one-thread-per-leaf kernel north_star prescribes (accounting A: 2H+1 MUFU per rollout), same workload (all
    robots: the persistent grid needs a few hundred ms of work per launch to hide its tail)."""
    n = len(scen)
    Hh = wl["H"]
    S = len(wl["V"]) * len(wl["B"])
    solver.set_grid(wl["V"], wl["B"], C.CONFIG["L"], C.CONFIG["delta_t"], C.CONFIG["v_min"])
    solver.set_option("algo", nat.ALGO_LEAFWALK)
    solver.set_option("prune", 0)
    st = torch.from_numpy(np.ascontiguousarray(scen[:n, :3])).to(dev)
    tg = torch.from_numpy(np.ascontiguousarray(scen[:n, 3:5])).to(dev)
    og = torch.from_numpy(np.ascontiguousarray(scen[:n, :2])).to(dev)
    oc = torch.empty(n, dtype=torch.float64, device=dev)
    oi = torch.empty(n, dtype=torch.int64, device=dev)

    def step():
        solver.solve_device(nat.MODE_FULL, nat.COST_MM, Hh, n, st.data_ptr(), tg.data_ptr(), og.data_ptr(), 0, 0,
                            oc.data_ptr(), oi.data_ptr(), 0, 0)
    with torch.cuda.stream(ext):
        step()
    solver.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3
    with torch.cuda.stream(ext):
        e0.record()
        for _ in range(reps):
            step()
        e1.record()
    solver.sync()
    torch.cuda.synchronize()
    rate = reps * n * S ** Hh / (e0.elapsed_time(e1) * 1e-3)
    solver.set_option("algo", nat.ALGO_AUTO)
    ex = EXECUTED["leafwalk"]
    clk = pk["sm_max_mhz"] * 1e6
    return dict(kernel=ex["kernel"], robots=n, rollouts_per_s=rate, index_checksum=int(oi.sum()),
                xu_frac=rate * ex["mufu"] / (SM_COUNT * MUFU_PER_CLK_SM * clk),
                issue_frac=rate * ex["instr"] / (SM_COUNT * FP32_PER_CLK_SM * clk),
                accounting_A_frac=rate * (2 * Hh + 1) / (SM_COUNT * MUFU_PER_CLK_SM * clk),
                executed=dict(mufu_per_rollout=ex["mufu"], instructions_per_rollout=ex["instr"]))


def dump_outputs(directory, tensors, dist, world, rank):
    """Writes the arrays a caller of the timed step receives as DIR/<name>.npy in float64 (the int64 leaf index is
    exact there), every robot of every rank in the global robot order: ~106 KB a GPU for cfg2, so nothing is sampled."""
    arrays = {k: t.cpu().numpy().astype(np.float64) for k, t in tensors.items()}
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, arrays)
        arrays = {k: np.concatenate([p[k] for p in parts]) for k in arrays}
    if rank == 0:
        os.makedirs(directory, exist_ok=True)
        for k, a in arrays.items():
            np.save(os.path.join(directory, k + ".npy"), a)


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from diplomjourney_b200 import _native as nat
    from oracle import closed_form as C   # scenario generator + parity gate only

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)

    wl = workload(args.workload)
    Hh, n = wl["H"], wl["n"]
    S = len(wl["V"]) * len(wl["B"])
    leaves_per_solve = S ** Hh
    solver = nat.Solver(local)
    solver.set_grid(wl["V"], wl["B"], C.CONFIG["L"], C.CONFIG["delta_t"], C.CONFIG["v_min"])
    solver.set_option("algo", {"auto": nat.ALGO_AUTO, "prefix": nat.ALGO_PREFIX, "leafwalk": nat.ALGO_LEAFWALK}[args.algo])
    # the headline evaluates EVERY leaf (as the reference does); the exact branch-and-bound is reported separately
    solver.set_option("prune", 0)
    if args.nodes_per_thread:
        solver.set_option("nodes_per_thread", args.nodes_per_thread)
    if args.screen is not None:
        solver.set_option("screen", args.screen)
    screen = 1 if args.screen is None else args.screen

    # each rank owns its own robots (contiguous ranges of the global batch): no data-path collective
    scen = C.random_scenarios(n * world, wl["seed"])[rank * n:(rank + 1) * n]
    st_h = torch.from_numpy(np.ascontiguousarray(scen[:, :3])).pin_memory()
    tg_h = torch.from_numpy(np.ascontiguousarray(scen[:, 3:5])).pin_memory()
    og_h = torch.from_numpy(np.ascontiguousarray(scen[:, :2])).pin_memory()
    st, tg, og = st_h.to(dev), tg_h.to(dev), og_h.to(dev)
    oc = torch.empty(n, dtype=torch.float64, device=dev)
    oi = torch.empty(n, dtype=torch.int64, device=dev)
    ot = torch.empty(n, Hh, 3, dtype=torch.float64, device=dev)
    ou = torch.empty(n, 2, dtype=torch.float64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2
    ext = torch.cuda.ExternalStream(solver.stream, device=dev)

    def step_device():
        solver.solve_device(nat.MODE_FULL, nat.COST_MM, Hh, n, st.data_ptr(), tg.data_ptr(), og.data_ptr(), 0, 0,
                            oc.data_ptr(), oi.data_ptr(), ot.data_ptr(), ou.data_ptr())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing (value + roofline)
    with torch.cuda.stream(ext):
        for _ in range(args.warmup):
            flush.fill_(1)
            step_device()
    stats = solver.stats()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(ext):
        t0.record()
        for k in range(args.steps):
            flush.fill_(k & 0xFF)                 # L2 flush between timed iterations (inside the region)
            evs[k][0].record()
            step_device()
            evs[k][1].record()
        t1.record()
    barrier()
    clocks = sampler.stop()
    total_ms = t0.elapsed_time(t1)
    step_ms = [a.elapsed_time(b) for a, b in evs]
    tt = torch.tensor([total_ms, statistics.mean(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms, kern_ms = float(tt[0]), float(tt[1])
    rollouts_per_step = leaves_per_solve * n * world
    value = rollouts_per_step * args.steps / (total_ms * 1e-3)
    dev_index = oi.cpu().numpy().copy()
    dev_cost = oc.cpu().numpy().copy()
    if args.dump_outputs:
        # the last timed step's outputs, before the later legs reuse the buffers
        dump_outputs(args.dump_outputs, dict(cost=oc, index=oi, traj=ot, first_control=ou), dist, world, rank)

    # ---------------- end-to-end through the host-buffer C-ABI call (pinned inputs, H2D + D2H inside)
    out_np = None
    for _ in range(max(1, args.warmup)):
        out_np = solver.solve(nat.MODE_FULL, nat.COST_MM, Hh, st_h.numpy(), tg_h.numpy(), og_h.numpy())
    barrier()
    e0 = time.perf_counter()
    for _ in range(args.steps):
        out_np = solver.solve(nat.MODE_FULL, nat.COST_MM, Hh, st_h.numpy(), tg_h.numpy(), og_h.numpy())
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - e0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = rollouts_per_step * args.steps / float(te[0])
    h2d = n * (3 + 2 + 2) * 8
    d2h = n * (8 + 8 + 3 * Hh * 8 + 16)

    # ---------------- parity gate on the benchmark's own output: every robot of the device-timed step equals the
    # host-API step bit for bit, and an evenly spaced sub-sample of >= 64 robots equals the float64 C oracle
    if not (np.array_equal(dev_index, out_np["index"]) and np.array_equal(dev_cost, out_np["cost"])):
        raise SystemExit("PARITY FAILURE in bench: device-API and host-API steps disagree")
    parity = None
    if rank == 0:
        from oracle import c_oracle as K
        chk = list(range(0, n, max(1, n // 64)))[:64] if Hh == 3 else list(range(min(2, n)))
        ok = 0
        for i in chk:
            o = K.solve_full(scen[i, :3], scen[i, 3:5], scen[i, :2], wl["V"], wl["B"], Hh, C.COST_MM)
            ok += int(out_np["index"][i] == o["index"] and abs(out_np["cost"][i] - o["cost"]) <= 1e-12 * o["cost"]
                      and np.allclose(out_np["traj"][i], o["traj"], rtol=0, atol=1e-12))
        parity = (f"{ok}/{len(chk)} robots (every {max(1, n // 64)}th) identical to the float64 C oracle (index, cost rtol 1e-12, "
                  f"trajectory atol 1e-12); all {n} robots identical between the device-API and host-API steps")
        if ok != len(chk):
            raise SystemExit("PARITY FAILURE in bench: " + parity)

    # ---------------- same step with the exact branch-and-bound on (identical results, fewer leaves evaluated)
    pruned = None
    if args.algo != "leafwalk":
        solver.set_option("prune", 1)
        with torch.cuda.stream(ext):
            step_device()
        barrier()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(ext):
            p0.record()
            for _ in range(args.steps):
                step_device()
            p1.record()
        barrier()
        pst = solver.stats()
        same = bool(np.array_equal(oi.cpu().numpy(), out_np["index"]) and np.array_equal(oc.cpu().numpy(), out_np["cost"]))
        tp = torch.tensor([p0.elapsed_time(p1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tp, op=dist.ReduceOp.MAX)
        parents = pst["units"] * n
        pruned = dict(ms_per_step=float(tp[0]) / args.steps, solves_per_s=n * world * args.steps / (float(tp[0]) * 1e-3),
                      evaluated_fraction=1.0 - pst["pruned_units"] / max(parents, 1), same_records_as_unpruned=same,
                      kernel_launches_per_step=pst["kernel_launches"],
                      note="option prune=1 (the library default): exact branch-and-bound -- nodes and subtrees whose leaves "
                           "provably cannot reach the refinement window are skipped, identical records; `value` above "
                           "is measured with prune=0 (every leaf evaluated)")
        if not same:
            raise SystemExit("PARITY FAILURE in bench: pruned and unpruned solves disagree")
        solver.set_option("prune", 0)
    solver.set_option("algo", nat.ALGO_AUTO)

    full = args.algo == "auto" and args.workload == "cfg2" and not args.no_legs
    pk = peaks()
    held = held_metrics(solver, nat, C, local) if rank == 0 and world == 1 and full else None
    bigtree = bigtree_metrics(solver, nat, C) if rank == 0 and world == 1 and full else None
    leafwalk = leg_leafwalk(solver, nat, C, torch, dev, ext, wl, scen, pk) if rank == 0 and world == 1 and full else None
    cfg4 = leg_cfg4_strong(solver, nat, C, torch, dist, dev, ext, world, rank, args.cfg4_scenarios) if full else None
    split = leg_split_tree(solver, nat, C, torch, dist, dev, ext, world, rank) if full and world > 1 else None

    if rank == 0:
        clk_hz = pk["sm_max_mhz"] * 1e6
        mufu_peak = SM_COUNT * MUFU_PER_CLK_SM * clk_hz
        fp32_peak = SM_COUNT * FP32_PER_CLK_SM * clk_hz
        per_gpu_rate = leaves_per_solve * n / (kern_ms * 1e-3)           # rollouts/s of one GPU, per step
        key = "leafwalk" if stats["algo"] == nat.ALGO_LEAFWALK else ("prefix_screen" if screen == 1 else "prefix_full")
        ex = EXECUTED[key]
        fp32_frac = per_gpu_rate * ex["fp32"] / fp32_peak
        xu_frac = per_gpu_rate * ex["mufu"] / mufu_peak
        bound_is_xu = xu_frac > fp32_frac
        ncu = ncu_record(key)
        roofline = dict(
            bound="xu" if bound_is_xu else "fp32",
            unit="Tlane-op/s",
            achieved=(per_gpu_rate * ex["mufu"] if bound_is_xu else per_gpu_rate * ex["fp32"]) / 1e12,
            peak=(mufu_peak if bound_is_xu else fp32_peak) / 1e12,
            frac=max(fp32_frac, xu_frac),
            traffic=ncu["traffic"] if ncu else None,
            note="the path is neither HBM- nor tensor-bound (SURVEY 8d): frac = work the dominant kernel EXECUTES per rollout "
                 "on its binding pipe (FP32 lanes or XU/MUFU, counted in its SASS) x measured rollouts/s / that pipe's peak",
            kernel=ex["kernel"], kernel_ms_per_step=kern_ms,
            executed=dict(fp32_lane_ops_per_rollout=ex["fp32"], mufu_per_rollout=ex["mufu"],
                          instructions_per_rollout=ex["instr"], fp32_frac=fp32_frac, xu_frac=xu_frac,
                          issue_frac=per_gpu_rate * ex["instr"] / fp32_peak, source="profiles/r2_sass_loops.txt"),
            ncu=ncu,
            accounting_A=dict(mufu_per_rollout=2 * Hh + 1, frac=per_gpu_rate * (2 * Hh + 1) / mufu_peak,
                              note="SURVEY 8d: one thread per leaf walks H steps; the prefix kernel shares prefixes and does not "
                                   "execute this work, so > 1 is expected for it"),
            accounting_B=dict(mufu_per_rollout=3, frac=per_gpu_rate * 3 / mufu_peak),
            hbm=dict(algorithmic_bytes_per_step=h2d + d2h, gbs=(h2d + d2h) / (kern_ms * 1e-3) / 1e9,
                     peak_gbs=pk["hbm_gbs"]),
            peak_src=f"{pk['src']} sm_max_mhz={pk['sm_max_mhz']:.0f} x {SM_COUNT} SMs x {FP32_PER_CLK_SM} FP32 lanes "
                     f"(x {MUFU_PER_CLK_SM} MUFU) per clock per SM")
        line = dict(
            metric="candidate rollouts/s (MPC inner loop)", value=value, unit="rollouts/s", n_gpus=world,
            steps=args.steps, warmup=args.warmup, ms_per_step=total_ms / args.steps, higher_is_better=True,
            scaling="weak", vs_baseline=None, dtype="f32", data="synthetic", config=config_of(wl),
            solves_per_s=n * world * args.steps / (total_ms * 1e-3),
            roofline=roofline,
            e2e=dict(value=e2e_value, unit="rollouts/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                     solves_per_s=n * world * args.steps / float(te[0])),
            gpu_launches=stats["kernel_launches"] * args.steps,
            clocks=clocks, parity=parity, pruned=pruned,
            refine=dict(segments=stats["refine_segments"], candidates=stats["refine_candidates"]),
            cfg4_strong=cfg4, split_tree=split, held=held, bigtree=bigtree, leafwalk=leafwalk,
        )
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_sample(wl)
            line["cpu_closed_form"] = closed_form_cpu(wl)
        print(json.dumps(line), flush=True)
    solver.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg4"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-legs", action="store_true", help="headline only (kernel experiments)")
    ap.add_argument("--cfg4-scenarios", type=int, default=65536, help="scenarios of the cfg4_strong leg")
    ap.add_argument("--nodes-per-thread", type=int, default=0, choices=[0, 1, 2, 4],
                    help="prefix pass 1: depth-(H-1) nodes per thread (0 = library default)")
    ap.add_argument("--screen", type=int, default=None, choices=[0, 1],
                    help="exhaustive prefix pass 1: 0 = MUFU.SQRT per leaf, 1 = screened (library default)")
    ap.add_argument("--algo", default="auto", choices=["auto", "prefix", "leafwalk"],
                    help="expansion kernel: prefix (default for this workload) or the one-thread-per-leaf design")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs (cost, index, traj, first_control) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU step's outputs; the reference arm only counts leaves")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
