"""Cost of the closed loops' per-tick trace (mpcb_set_loop_trace): kernel time of the device entries on torch tensors
with the trace off and on, next to the parent commit's library (no trace), and the wall clock of the reference run
math_mpc([0,0,0,0,0], [2,3], False) per tick against the module switch device_loop = True.

  * mpcb_held_closed_loop_device: the programmed run (noise-free; no device entry takes an event script without noise,
    so no events), first threshold 1e10, max_ticks 512
  * mpcb_held_closed_loop_actual_device: the actual run with the actual run's event script, generators seeded on the
    device from integer seeds (mpcb_rng_seed_device) before every launch, outside the timed window
at 1,024 and 16,384 robots, H = 3.  Per configuration the three variants (parent, trace off, trace on) run in turn,
five rounds, one launch each: CUDA events around the one launch on the handle's stream; mean, min and max of the five.
Outputs of the parent and of trace-off are compared bit for bit, and trace-on's log with trace-off's.

usage: python tools/loop_trace_timing.py [--parent build/variants/lib_parent.so]
(build the parent's library from a git worktree of the parent commit with diplomjourney_b200.build.build_library(
force=True, out=...))"""
import argparse
import ctypes as C
import importlib
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from diplomjourney_b200 import _native as nat, config  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--parent", default=os.path.join(ROOT, "build", "variants", "lib_parent.so"))
ap.add_argument("--rounds", type=int, default=5)
args = ap.parse_args()

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True)
print(f"GPU: {q.stdout.strip().splitlines()[0] if q.returncode == 0 else 'nvidia-smi failed: ' + q.stderr.strip()}")
print(f"torch {torch.__version__}, device {torch.cuda.get_device_name(0)}")


class Lib:
    """A handle of one build of the library (ctypes, so that two builds live in one process)."""

    def __init__(self, path):
        self.lib = lib = C.CDLL(path)
        vp = C.c_void_p
        lib.mpcb_create.argtypes = [C.c_int, C.POINTER(vp)]
        lib.mpcb_stream.argtypes = [vp]
        lib.mpcb_stream.restype = vp
        lib.mpcb_destroy.argtypes = [vp]
        loop = [vp, C.POINTER(nat.LoopParams), C.c_int64, vp, vp, vp, vp, vp, vp, vp, vp]
        lib.mpcb_held_closed_loop_device.argtypes = loop
        lib.mpcb_held_closed_loop_actual_device.argtypes = loop[:8] + [vp, C.c_int32, C.c_double, vp] + loop[8:] + [vp]
        lib.mpcb_rng_seed_device.argtypes = [vp, C.c_int64, vp, C.c_int32, vp]
        self.traced = hasattr(lib, "mpcb_set_loop_trace")
        if self.traced:
            lib.mpcb_set_loop_trace.argtypes = [vp, C.POINTER(nat.LoopTrace)]
        self.h = vp()
        assert lib.mpcb_create(0, C.byref(self.h)) == 0
        self.stream = torch.cuda.ExternalStream(lib.mpcb_stream(self.h))

    def ck(self, rc):
        assert rc == 0, rc


mt = importlib.import_module("diplomjourney_b200.math_model_tree")
ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
T = 512
params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, T)
ev, n_ev = nat._event_script(mt.ACTUAL_EVENTS)
libs = {"parent": Lib(args.parent), "new": Lib(nat.load()._name)}
assert not libs["parent"].traced and libs["new"].traced
variants = (("parent", "parent", False), ("trace off", "new", False), ("trace on", "new", True))

for n in (1024, 16384):
    rng = np.random.default_rng(n)
    init = np.zeros((n, 5))
    init[:, :2] = rng.uniform(-1, 1, (n, 2))
    init[:, 2] = rng.uniform(-0.5, 7.0, n)
    init[:, 3] = rng.choice([0.0, 0.0, 0.3, 0.6], n)
    tgt = np.tile([2.0, 3.0], (n, 1)) + rng.uniform(-1, 1, (n, 2))
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    d_init, d_tgt, d_org, d_thr = cuda(init), cuda(tgt), cuda(np.zeros((n, 2))), cuda(np.full(n, 1e10))
    d_keys = cuda(rng.integers(0, 2 ** 32, n).astype(np.uint32).view(np.int32))
    f64 = dict(dtype=torch.float64, device="cuda")
    out = {name: dict(log=torch.empty((n, T, 5), **f64), ticks=torch.empty(n, dtype=torch.int32, device="cuda"),
                      status=torch.empty(n, dtype=torch.int32, device="cuda"), final=torch.empty((n, 6), **f64),
                      rng=torch.empty((n, 625), dtype=torch.int32, device="cuda")) for name, _, _ in variants}
    trace = dict(pred=torch.empty((n, T, 3, 3), **f64), control=torch.empty((n, T, 2), **f64), cost=torch.empty((n, T), **f64))
    mem = sum(t.numel() * 8 for t in trace.values())
    print(f"\nN={n}: trace memory {mem / 2 ** 20:.1f} MiB = N * max_ticks * (3H + 3) * 8 bytes "
          f"(max_ticks {T}, H 3)", flush=True)
    for run in ("programmed", "actual"):
        times = {name: [] for name, _, _ in variants}
        for r in range(args.rounds + 1):                    # round 0 warms every variant up and is not counted
            for name, which, traced in variants:
                L, o = libs[which], out[name]
                o["log"].fill_(float("nan"))
                for t in trace.values():
                    t.fill_(float("nan"))
                if run == "actual":
                    L.ck(L.lib.mpcb_rng_seed_device(L.h, n, ptr(d_keys), 0, ptr(o["rng"])))
                torch.cuda.synchronize()
                if traced:
                    L.ck(L.lib.mpcb_set_loop_trace(L.h, C.byref(nat.LoopTrace(*(trace[k].data_ptr() for k in
                                                                                 ("pred", "control", "cost"))))))
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(L.stream)
                if run == "programmed":
                    L.ck(L.lib.mpcb_held_closed_loop_device(L.h, C.byref(params), n, ptr(d_init), ptr(d_tgt), ptr(d_org),
                                                            ptr(d_thr), None, ptr(o["log"]), ptr(o["ticks"]),
                                                            ptr(o["status"])))
                else:
                    L.ck(L.lib.mpcb_held_closed_loop_actual_device(
                        L.h, C.byref(params), n, ptr(d_init), ptr(d_tgt), ptr(d_org), ptr(d_thr), None, ev, n_ev,
                        mt.radius_u_turn, ptr(o["rng"]), ptr(o["log"]), ptr(o["ticks"]), ptr(o["status"]),
                        ptr(o["final"])))
                e1.record(L.stream)
                e1.synchronize()
                if r:
                    times[name].append(e0.elapsed_time(e1))
        a, b, c = (out[name] for name, _, _ in variants)
        keys = ("log", "ticks", "status") + (("final", "rng") if run == "actual" else ())
        same_parent = all(torch.equal(a[k].nan_to_num(-7.0), b[k].nan_to_num(-7.0)) for k in keys)
        same_traced = all(torch.equal(b[k].nan_to_num(-7.0), c[k].nan_to_num(-7.0)) for k in keys)
        tk = b["ticks"].cpu().numpy()
        print(f"  {run} run (mean ticks {tk.mean():.1f}, max {tk.max()}): outputs parent == trace off: {same_parent}, "
              f"trace off == trace on: {same_traced}", flush=True)
        base = np.mean(times["parent"])
        for name, _, _ in variants:
            ms = np.array(times[name])
            print(f"    {name:9s}: {ms.mean():8.3f} ms (min {ms.min():.3f}, max {ms.max():.3f}, "
                  f"spread {100 * (ms.max() - ms.min()) / ms.mean():.1f} %)  {100 * (ms.mean() / base - 1):+.2f} % vs parent",
                  flush=True)
    del out, trace
    torch.cuda.empty_cache()

# the reference's programmed run: the per-tick math_mpc against one launch
print("\nmath_mpc([0,0,0,0,0], [2,3], False), wall clock (perf_counter around the call, which ends in a sync):")
walls = {False: [], True: []}
for r in range(4):                                          # round 0 warms both up
    for dev in (False, True):
        mt = importlib.reload(mt)
        mt.reset_state()
        mt.device_loop = dev
        t0 = time.perf_counter()
        mt.math_mpc([0, 0, 0, 0, 0], [2, 3], False)
        dt = time.perf_counter() - t0
        if r:
            walls[dev].append(dt)
        ticks = mt.p - 1
for dev, name in ((False, "per tick"), (True, "device_loop")):
    w = np.array(walls[dev]) * 1e3
    print(f"  {name:16s}: {w.mean():8.2f} ms per run (min {w.min():.2f}, max {w.max():.2f}), "
          f"{w.mean() / ticks * 1e3:.1f} us per tick over {ticks} ticks")
