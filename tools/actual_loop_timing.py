"""Timing of the online controller's "actual" run (actuator noise, the actual run's event script) as ONE launch of the
device-resident loop (math_mpc_batch(..., isActual=True, device_noise=True)), next to the per-tick path that draws the
noise on the host (one batched launch per tick) and to the noise-free device loop on the same robots.  Host clock
around the synchronising call, after one warm-up call of the same shape.  The math_mpc_batch rows include handing the
generators' states over (RandomState.get_state / set_state, ~0.1 ms per robot in numpy); the "solver call" rows time
Solver.held_closed_loop alone on states packed beforehand, with and without them, so the loop's own cost shows.
usage: python tools/actual_loop_timing.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import time, numpy as np, importlib
mt = importlib.import_module("diplomjourney_b200.math_model_tree")
from diplomjourney_b200 import _native as nat, config
params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, 400)
rng = np.random.default_rng(1)


def timed(**kw):
    t0 = time.perf_counter()
    r = mt.math_mpc_batch(init, tgt, max_ticks=400, origin=org, events=True, **kw)
    return time.perf_counter() - t0, r


def line(name, dt, r):
    return (f"{name} N={n}: {dt * 1e3:.2f} ms, {r['ticks'].sum()} ticks, {r['ticks'].sum() / dt:.3e} ticks/s, "
            f"status {np.bincount(r['status'], minlength=4)}")


for n in (1, 1024, 16384):
    init = np.zeros((n, 5)); init[:, :2] = rng.uniform(-1, 1, (n, 2)); init[:, 2] = rng.uniform(-0.5, 7, n)
    tgt = np.tile([2.0, 3.0], (n, 1)) + rng.uniform(-1, 1, (n, 2))
    org = np.zeros((n, 2))
    seeds = rng.integers(0, 2 ** 32, n)
    gens = lambda: [np.random.RandomState(s) for s in seeds]
    timed(isActual=True, device_noise=True, rngs=gens())                    # warm-up
    dt, r = timed(isActual=True, device_noise=True, rngs=gens())
    print(line("device loop, actuator noise", dt, r), flush=True)
    timed()
    dt, r0 = timed()
    print(line("device loop, noise-free", dt, r0), flush=True)
    packed = mt._pack_generators(gens())
    for name, kw in (("solver call, actuator noise", dict(rng_state=packed)), ("solver call, noise-free", {})):
        call = lambda: mt._solver().held_closed_loop(params, init, tgt, org, first_threshold=1e10, events=mt.ACTUAL_EVENTS,
                                                     radius_u_turn=mt.radius_u_turn, **kw)
        call()
        t0 = time.perf_counter(); rs = call(); dt = time.perf_counter() - t0
        print(line(name, dt, rs), flush=True)
    if n == 1024:
        dt, h = timed(isActual=True, rngs=gens())
        same = np.array_equal(h["ticks"], r["ticks"]) and np.allclose(h["log"], r["log"], rtol=0, atol=1e-9, equal_nan=True)
        print(line("per-tick path, actuator noise", dt, h) + f", equal to the device loop: {same}", flush=True)
