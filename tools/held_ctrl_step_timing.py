"""What stepping the online controller one tick at a time costs (mpcb_held_ctrl_step_device), against the whole closed
loop in one launch and against the per-tick host path, for 1,024 and 16,384 robots, H = 3:

  (a) identity plant: the step loop (one step launch and one read of the running count per tick) vs
      mpcb_held_closed_loop_device on the same robots; plus the steps alone, enqueued back to back without the read
      (CUDA events), i.e. what one step kernel costs against one tick of the loop kernel;
  (b) math_mpc_batch(isActual=True, actuator=fn) with a torch-vectorised actuator vs the per-tick path
      _math_mpc_batch_ticks (one batched windows solve per tick, noise drawn on the host).

    python tools/held_ctrl_step_timing.py [--reps 5]

Prints the card's name and power limit first; every time is the median of --reps runs with min and max.
"""
import argparse
import ctypes
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from diplomjourney_b200 import _native as nat, config  # noqa: E402
from diplomjourney_b200 import math_model_tree as mt  # noqa: E402


def spread(xs):
    xs = sorted(xs)
    return f"{statistics.median(xs) * 1e3:9.2f} ms [{xs[0] * 1e3:.2f} .. {xs[-1] * 1e3:.2f}]"


def robots(n, seed):
    rng = np.random.default_rng(seed)
    init = np.zeros((n, 5))
    init[:, :2] = rng.uniform(-1, 1, (n, 2))
    init[:, 2] = rng.uniform(-0.5, 7.0, n)
    init[:, 3] = rng.choice([0.0, 0.0, 0.3, 0.6], n)
    tgt = np.tile([2.0, 3.0], (n, 1)) + rng.uniform(-1, 1, (n, 2))
    return init, tgt, np.zeros((n, 2)), np.full(n, 1e10)


def identity(s, n, reps):
    params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, 256)
    init, tgt, org, thr = robots(n, n)
    dev = torch.device("cuda", 0)
    st = torch.cuda.ExternalStream(s.stream, device=dev)
    with torch.cuda.stream(st):
        t_init, t_tgt, t_org, t_thr = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (init, tgt, org, thr))
        log = torch.full((n, params.max_ticks, 5), float("nan"), dtype=torch.float64, device=dev)
        ticks = torch.empty(n, dtype=torch.int32, device=dev)
        status = torch.empty(n, dtype=torch.int32, device=dev)
        ctrl = torch.empty((n, ctypes.sizeof(nat.HeldCtrl)), dtype=torch.uint8, device=dev)
        prop = torch.empty((n, 5), dtype=torch.float64, device=dev)
        running = torch.zeros(1, dtype=torch.int32, device=dev)
    vp = lambda t: ctypes.c_void_p(t.data_ptr())

    def loop():
        rc = s.lib.mpcb_held_closed_loop_device(s.h, ctypes.byref(params), n, vp(t_init), vp(t_tgt), vp(t_org), vp(t_thr),
                                                None, vp(log), vp(ticks), vp(status))
        assert rc == 0

    def init_ctrl():
        s.held_ctrl_init_device(params, n, t_init.data_ptr(), t_tgt.data_ptr(), t_org.data_ptr(), t_thr.data_ptr(), 0,
                                ctrl.data_ptr())

    def step():
        with torch.cuda.stream(st):
            running.zero_()
        s.held_ctrl_step_device(params, n, ctrl.data_ptr(), proposal=prop.data_ptr(), running=running.data_ptr())

    def step_loop():
        init_ctrl()
        k = 0
        while True:
            step()
            k += 1
            with torch.cuda.stream(st):                 # the read follows the step on the solver's stream
                if not int(running.item()):
                    return k

    t_loop, t_steps, t_free = [], [], []
    loop(); step_loop(); s.sync()                               # warm-up
    for _ in range(reps):
        t0 = time.perf_counter(); loop(); s.sync(); t_loop.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); k = step_loop(); s.sync(); t_steps.append(time.perf_counter() - t0)
        # the same k steps enqueued back to back, no read of the running count: device time of the steps alone
        init_ctrl()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(k):
            step()
        e1.record(st)
        e1.synchronize()
        t_free.append(e0.elapsed_time(e1) * 1e-3)
    with torch.cuda.stream(st):
        tk = ticks.cpu().numpy()
    assert k == tk.max() + 1, (k, tk.max())           # the last step only commits
    steps_per_tick = k / max(1, tk.max())
    print(f"(a) robots {n:6d}: ticks max {tk.max()} sum {tk.sum()}, {k} steps")
    print(f"    closed loop, one launch      {spread(t_loop)}   {statistics.median(t_loop) / tk.max() * 1e6:8.1f} us per tick of the longest robot")
    print(f"    step loop (read per step)    {spread(t_steps)}   {statistics.median(t_steps) / k * 1e6:8.1f} us per step")
    print(f"    steps back to back (events)  {spread(t_free)}   {statistics.median(t_free) / k * 1e6:8.1f} us per step  ({steps_per_tick:.3f} steps per tick)")


def actual(s, n, reps, per_tick_reps):
    init, tgt, org, _ = robots(n, 7 * n)
    gen = torch.Generator(device="cuda:0")

    def fn(commanded, running):                     # a vectorised actuator: jitter of up to 5 mm/s and 1 degree
        j = torch.rand(commanded.shape, generator=gen, device=commanded.device, dtype=torch.float64) - 0.5
        return commanded + j * torch.tensor([0.01, 0.035], dtype=torch.float64, device=commanded.device)

    run = dict(max_ticks=256, origin=org, isActual=True, events=True)
    t_act, t_tick = [], []
    gen.manual_seed(0)
    mt.math_mpc_batch(init, tgt, actuator=fn, **run)     # warm-up
    for _ in range(reps):
        gen.manual_seed(0)
        t0 = time.perf_counter(); a = mt.math_mpc_batch(init, tgt, actuator=fn, **run); t_act.append(time.perf_counter() - t0)
    first = np.empty(n)                             # the first thresholds math_mpc_batch computes
    saved = (mt.x_t, mt.y_t, mt.x_0, mt.y_0)
    for i in range(n):
        mt.x_t, mt.y_t, mt.x_0, mt.y_0 = tgt[i, 0], tgt[i, 1], org[i, 0], org[i, 1]
        first[i] = mt.control_criterion([org[i, 0], org[i, 1], mt.phi_0])
    mt.x_t, mt.y_t, mt.x_0, mt.y_0 = saved
    for _ in range(per_tick_reps):
        gens = [np.random.RandomState(i) for i in range(n)]
        t0 = time.perf_counter()
        h = mt._math_mpc_batch_ticks(init, tgt, org, first, 256, None, True, gens, True)
        t_tick.append(time.perf_counter() - t0)
    print(f"(b) robots {n:6d}: actuator= ticks max {a['ticks'].max()} sum {a['ticks'].sum()}; per-tick path ticks max "
          f"{h['ticks'].max()} sum {h['ticks'].sum()}")
    print(f"    math_mpc_batch(actuator=)    {spread(t_act)}   {statistics.median(t_act) / a['ticks'].max() * 1e6:8.1f} us per step")
    print(f"    per-tick path                {spread(t_tick)}   {statistics.median(t_tick) / h['ticks'].max() * 1e6:8.1f} us per tick")
    print(f"    speed-up {statistics.median(t_tick) / statistics.median(t_act):.1f}x")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--per-tick-reps", type=int, default=3, help="runs of the per-tick path at 1,024 robots (one at 16,384)")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    print("GPU:", q.stdout.strip().splitlines()[0] if q.returncode == 0 else "nvidia-smi unavailable")
    print("torch", torch.__version__, "| CUDA", torch.version.cuda)
    s = mt._solver()
    for n in (1024, 16384):
        identity(s, n, args.reps)
    for n in (1024, 16384):
        actual(s, n, args.reps, args.per_tick_reps if n <= 1024 else 1)


if __name__ == "__main__":
    main()
