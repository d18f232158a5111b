"""Cost of the FULL-tree closed loop (mpcb_full_closed_loop_*, run_batch), next to the parent commit's library, which
returned to the host every tick (enqueue the solve, apply, read the running count back, synchronise).

  * host entry, parent vs new: wall clock (perf_counter around the call, which ends in a synchronisation); the parent
    also on a second handle of its own: with few robots the run is mostly the refinement scan of a handful of solves,
    whose time depends on where the handle's buffers lie, so two handles of one build differ by themselves
  * device entry (new): CUDA events around the call on the handle's stream -- the whole run
  * the device entry's call alone on the host clock: the first call of a workload captures and instantiates the loop
    graph and launches it; the timed rounds find it in the handle's cache and only launch it
Workloads: the acceleration-window grid 11 x 41 (S = 451, math_model_tree.py:239-256 at v = 0.5, beta = 0), H = 3, MM
cost, scenarios of oracle.closed_form.random_scenarios (start and target up to 10 m apart), max_ticks 256, default
pruning, at N = 1, 64 and 1,024 robots; and N = 1,024 exhaustive (prune = 0) with max_ticks 4.  Per workload the three
variants run in turn, --rounds rounds after one warm-up round; every output (log rows incl. the NaN rows, ticks,
status) of the new host entry and of the device entry is compared bit for bit with the parent's.

usage: python tools/full_loop_timing.py [--parent build/variants/lib_parent.so] [--rounds 5]
(build the parent's library from a git worktree of the parent commit with diplomjourney_b200.build.build_library(
force=True, out=...))"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from diplomjourney_b200 import _native as nat, config  # noqa: E402
from oracle import closed_form as CF  # noqa: E402

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
        lib.mpcb_last_error.argtypes = [vp]
        lib.mpcb_last_error.restype = C.c_char_p
        lib.mpcb_set_grid.argtypes = [vp, vp, C.c_int, vp, C.c_int, C.c_double, C.c_double, C.c_double]
        lib.mpcb_set_option.argtypes = [vp, C.c_char_p, C.c_double]
        full = [vp, C.c_int, C.c_int, C.c_int64, vp, vp, vp, vp, C.c_double, C.c_int, vp, vp, vp]
        lib.mpcb_full_closed_loop_host.argtypes = full
        self.device_entry = hasattr(lib, "mpcb_full_closed_loop_device")
        if self.device_entry:
            lib.mpcb_full_closed_loop_device.argtypes = full
        self.h = vp()
        assert lib.mpcb_create(0, C.byref(self.h)) == 0
        self.stream = torch.cuda.ExternalStream(lib.mpcb_stream(self.h))

    def ck(self, rc):
        assert rc == 0, (rc, self.lib.mpcb_last_error(self.h))


V = np.array(CF.vector_of_velocities(0.5))
B = np.array(CF.vector_of_beta_angles(0.0))
H = 3
libs = {"parent": Lib(args.parent), "parent2": Lib(args.parent), "new": Lib(nat.load()._name),
        "new_dev": Lib(nat.load()._name)}      # the device entry on a handle of its own: each handle keeps one graph
assert not libs["parent"].device_entry and libs["new"].device_entry
for L in libs.values():
    L.ck(L.lib.mpcb_set_grid(L.h, V.ctypes.data, V.size, B.ctypes.data, B.size, config.L, config.delta_t, 0.0))
print(f"grid {V.size} x {B.size} (S = {V.size * B.size}), H = {H}, MM cost, eps {config.eps}")

hp = lambda a: C.c_void_p(a.ctypes.data)
dp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
workloads = [(1, 256, 1), (64, 256, 1), (1024, 256, 1), (1024, 4, 0)]
for n, T, prune in workloads:
    sc = CF.random_scenarios(n, 2024 + n)
    ini, tgt, org = (np.ascontiguousarray(x) for x in (sc[:, :3], sc[:, 3:5], sc[:, :2]))
    ang = np.arctan(sc[:, 3] / sc[:, 4]) - sc[:, 2]
    thr = 10000 * np.sqrt((sc[:, 3] - sc[:, 0]) ** 2 + (sc[:, 4] - sc[:, 1]) ** 2) + 10 * ang ** 2 + 100 * 1000 ** 2
    for L in libs.values():
        L.ck(L.lib.mpcb_set_option(L.h, b"prune", float(prune)))
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    d_in = [cuda(ini), cuda(tgt), cuda(org), cuda(thr)]
    out = {k: dict(log=np.empty((n, T, 5)), ticks=np.empty(n, np.int32), status=np.empty(n, np.int32))
           for k in ("parent host", "parent2 host", "new host")}
    d_out = dict(log=torch.empty((n, T, 5), dtype=torch.float64, device="cuda"),
                 ticks=torch.empty(n, dtype=torch.int32, device="cuda"),
                 status=torch.empty(n, dtype=torch.int32, device="cuda"))
    times = {k: [] for k in ("parent host", "parent2 host", "new host", "device entry", "device call (host clock)")}
    for r in range(args.rounds + 1):                        # round 0 warms every variant up and is not counted
        for name in ("parent host", "parent2 host", "new host"):
            L, o = libs[name.split()[0]], out[name]
            t0 = time.perf_counter()
            L.ck(L.lib.mpcb_full_closed_loop_host(L.h, nat.COST_MM, H, n, hp(ini), hp(tgt), hp(org), hp(thr), config.eps,
                                                  T, hp(o["log"]), hp(o["ticks"]), hp(o["status"])))
            if r:
                times[name].append((time.perf_counter() - t0) * 1e3)
        L = libs["new_dev"]
        d_out["log"].fill_(float("nan"))
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(L.stream)
        t0 = time.perf_counter()
        L.ck(L.lib.mpcb_full_closed_loop_device(L.h, nat.COST_MM, H, n, *(dp(x) for x in d_in), config.eps, T,
                                                dp(d_out["log"]), dp(d_out["ticks"]), dp(d_out["status"])))
        t1 = time.perf_counter()
        e1.record(L.stream)
        e1.synchronize()
        if r:
            times["device entry"].append(e0.elapsed_time(e1))
            times["device call (host clock)"].append((t1 - t0) * 1e3)
        else:
            first_call = (t1 - t0) * 1e3
    dev = {k: v.cpu().numpy() for k, v in d_out.items()}
    same = lambda a, b: all(np.array_equal(a[k], b[k], equal_nan=True) for k in ("log", "ticks", "status"))
    par = out["parent host"]
    tk = par["ticks"]
    print(f"\nN={n}, max_ticks {T}, prune {prune}: ticks mean {tk.mean():.1f}, max {tk.max()}, status counts "
          f"{np.bincount(par['status'], minlength=4).tolist()}; bit-identical to the parent: its 2nd handle "
          f"{same(out['parent2 host'], par)}, new host {same(out['new host'], par)}, device entry {same(dev, par)}",
          flush=True)
    print(f"    first device call (capture + instantiate + launch, host clock): {first_call:.3f} ms")
    base = np.mean(times["parent host"])
    for name, ms in times.items():
        ms = np.array(ms)
        rel = f"  {100 * (ms.mean() / base - 1):+.2f} % vs parent host" if name != "device call (host clock)" else ""
        print(f"    {name:25s}: {ms.mean():9.3f} ms (min {ms.min():.3f}, max {ms.max():.3f}, "
              f"spread {100 * (ms.max() - ms.min()) / ms.mean():.1f} %){rel}", flush=True)
for L in libs.values():
    L.lib.mpcb_destroy(L.h)
