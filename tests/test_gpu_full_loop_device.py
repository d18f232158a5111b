"""GPU: the FULL-tree closed loop as one graph launch -- mpcb_full_closed_loop_device on torch tensors against
mpcb_full_closed_loop_host, bit for bit (log rows, ticks, status and the per-tick trace), over the golden grids, both
costs, horizons 1-4, the pruning and screening options, robots on target at entry, first-tick NO_LEAF and short runs;
handle reuse after a grid / option / size change, chained launches, trace consumption and two devices at once."""
import math

import numpy as np
import pytest
import torch

from diplomjourney_b200 import _native as nat, config

pytestmark = pytest.mark.gpu

GRIDS = ("g4x5", "g5x7", "g3x9")


@pytest.fixture(scope="module")
def grids(golden):
    g = golden("full_h3")
    out = {}
    for name in GRIDS:
        cases = [c for c in g["cases"] if c["grid"] == name]
        sc = np.array([[c["scenario"][k] for k in ("x_0", "y_0", "phi_0", "x_t", "y_t")] for c in cases], float)
        out[name] = (np.array(cases[0]["vector_v"]), np.array(cases[0]["vector_beta"]), sc)
    return out


def _solver(grid, device=0, **options):
    s = nat.Solver(device)
    s.set_grid(grid[0], grid[1], config.L, config.delta_t, 0.0)
    for k, v in options.items():
        s.set_option(k, v)
    return s


def _first_threshold(sc):
    """control_criterion of each start pose with the line starting there (run_batch's first threshold)."""
    ang = np.arctan(sc[:, 3] / sc[:, 4]) - sc[:, 2]
    return 10000 * np.sqrt((sc[:, 3] - sc[:, 0]) ** 2 + (sc[:, 4] - sc[:, 1]) ** 2) + 10 * ang ** 2 + 100 * 1000 ** 2


def _random_scenarios(n, seed):
    rng = np.random.default_rng(seed)
    sc = np.zeros((n, 5))
    sc[:, :2] = rng.uniform(-1, 1, (n, 2))
    sc[:, 2] = rng.uniform(-0.5, 7.0, n)
    sc[:, 3:5] = sc[:, :2] + rng.uniform(0.3, 1.5, (n, 2)) * rng.choice([-1, 1], (n, 2))
    return sc


def _boundary_target(x, y, eps):
    """A target whose distance from (x, y) the on-target test must round as is_on_target does: dx * dx + dy * dy,
    each product rounded, is <= eps, but either fused form fma(dx, dx, dy * dy) / fma(dy, dy, dx * dx) is > eps."""
    from fractions import Fraction as F
    fma = lambda a, b, c: float(F(a) * F(b) + F(c))          # one rounding, as an FMA rounds
    for i in range(20000):
        ddx = 0.011 + 1e-6 * i
        base = math.sqrt(eps - ddx * ddx)
        for k in range(-4, 5):
            tx, ty = x + ddx, y + base + k * 2.0 ** -60
            dx, dy = tx - x, ty - y
            if dx * dx + dy * dy <= eps and fma(dx, dx, dy * dy) > eps and fma(dy, dy, dx * dx) > eps:
                return tx, ty
    raise AssertionError("no boundary target found")


def _host(s, cost, H, sc, thr, T):
    return s.full_closed_loop(cost, H, sc[:, :3], sc[:, 3:5], sc[:, :2], first_threshold=thr, eps=config.eps,
                              max_ticks=T, trace=True)


class _DeviceRun:
    """Inputs and NaN-filled outputs of one device-entry run, as torch tensors on the solver's device."""

    def __init__(self, s, cost, H, sc, thr, T, trace=True):
        dev = torch.device("cuda", s.device)
        f64 = dict(dtype=torch.float64, device=dev)
        t = lambda a: torch.tensor(np.ascontiguousarray(a), **f64)
        N = sc.shape[0]
        self.inp = [t(sc[:, :3]), t(sc[:, 3:5]), t(sc[:, :2]), None if thr is None else t(thr)]
        self.out = dict(log=torch.full((N, T, 5), math.nan, **f64),
                        ticks=torch.full((N,), -9, dtype=torch.int32, device=dev),
                        status=torch.full((N,), -9, dtype=torch.int32, device=dev))
        if trace:
            self.out.update(pred=torch.full((N, T, H, 3), math.nan, **f64), control=torch.full((N, T, 2), math.nan, **f64),
                            cost=torch.full((N, T), math.nan, **f64))
        self.args = (s, dev, cost, H, N, T, trace)
        self.launch()

    def launch(self):
        s, dev, cost, H, N, T, trace = self.args
        torch.cuda.synchronize(dev)                   # the library's stream does not wait for torch's
        ptr = lambda x: 0 if x is None else x.data_ptr()
        o = self.out
        s.full_closed_loop_device(cost, H, N, *(ptr(x) for x in self.inp), config.eps, T, ptr(o["log"]),
                                  ptr(o["ticks"]), ptr(o["status"]),
                                  trace=(ptr(o["pred"]), ptr(o["control"]), ptr(o["cost"])) if trace else None)

    def result(self):
        return {k: v.cpu().numpy() for k, v in self.out.items()}


def _device(s, cost, H, sc, thr, T, trace=True):
    run = _DeviceRun(s, cost, H, sc, thr, T, trace)
    s.sync()
    return run.result()


def _assert_same(dev, host, what=""):
    for k in dev:
        np.testing.assert_array_equal(dev[k], host[k], err_msg=f"{what} {k}")


@pytest.mark.parametrize("H", [1, 2, 3, 4])
@pytest.mark.parametrize("cost", [nat.COST_MM, nat.COST_TREE])
@pytest.mark.parametrize("grid", GRIDS)
def test_device_entry_equals_host_entry_on_golden_scenarios(grids, grid, cost, H):
    sc = grids[grid][2]
    T = 80
    s = _solver(grids[grid])
    thr = _first_threshold(sc)
    host = _host(s, cost, H, sc, thr, T)
    launches = s.stats()["kernel_launches"]
    dev = _device(s, cost, H, sc, thr, T)
    _assert_same(dev, host, f"{grid} cost {cost} H {H}")
    # the host entry counts the kernels of every tick run, the device entry those of one tick; a robot that found no
    # leaf stopped on the tick after its last logged one
    ticks_run = (host["ticks"] + (host["status"] == nat.LOOP_NO_LEAF)).max()
    assert ticks_run > 0 and launches == ticks_run * s.stats()["kernel_launches"]
    s.close()


@pytest.mark.parametrize("prune,screen", [(1, 2), (0, 0), (0, 1), (0, 2)])
def test_device_entry_equals_host_entry_with_pruning_and_screening(grids, prune, screen):
    sc = _random_scenarios(64, 3)
    s = _solver(grids["g5x7"], prune=prune, screen=screen)
    thr = _first_threshold(sc)
    host = _host(s, nat.COST_MM, 3, sc, thr, 60)
    assert s.stats()["algo"] == nat.ALGO_PREFIX                 # the exhaustive prefix pass 1 is what screen selects
    _assert_same(_device(s, nat.COST_MM, 3, sc, thr, 60), host, f"prune {prune} screen {screen}")
    s.close()


@pytest.mark.parametrize("T", [1, 4, 200])
def test_on_target_at_entry_no_leaf_and_short_runs(grids, T):
    """Robots on target at entry never run (one on the eps boundary, where an FMA would round it off target), robots whose first threshold is 0 stop at
    their first tick with NO_LEAF, and max_ticks cuts the others short."""
    sc = _random_scenarios(48, 7)
    sc[:6, 3:5] = sc[:6, :2] + [[0.0, 0.0], [0.01, -0.02], [0.02, 0.0], [-0.02, 0.01], [0.0, 0.0316], [0.05, 0.0]]
    sc[4, 3:5] = _boundary_target(sc[4, 0], sc[4, 1], config.eps)   # on target only if the test is not contracted
    thr = _first_threshold(sc)
    thr[10:16] = 0.0
    s = _solver(grids["g4x5"])
    host = _host(s, nat.COST_MM, 3, sc, None if T == 200 else thr, T)
    dev = _device(s, nat.COST_MM, 3, sc, None if T == 200 else thr, T)
    _assert_same(dev, host, f"T {T}")
    st = host["status"]
    assert (st[:5] == nat.LOOP_ON_TARGET).all() and (host["ticks"][:5] == 0).all()
    if T != 200:
        assert (st[10:16] == nat.LOOP_NO_LEAF).all()
    if T < 200:
        assert (st == nat.LOOP_MAX_TICKS).any()
    s.close()


def test_no_robots_launches_nothing(grids):
    s = _solver(grids["g4x5"])
    s.full_closed_loop_device(nat.COST_MM, 3, 0, 0, 0, 0, 0, config.eps, 10, 0, 0, 0)
    r = s.full_closed_loop(nat.COST_MM, 3, np.zeros((0, 3)), np.zeros((0, 2)), np.zeros((0, 2)), max_ticks=10)
    assert r["log"].shape == (0, 10, 5)
    s.sync()
    s.close()


def test_handle_reuse_after_grid_option_and_size_changes(grids):
    """One handle across a new grid, a toggled option and a larger batch equals a fresh handle each time."""
    small, large = _random_scenarios(8, 1), _random_scenarios(96, 2)
    T = 40
    s = _solver(grids["g4x5"])
    runs = [("g4x5", {}, small), ("g5x7", {}, small), ("g5x7", {"prune": 0}, small), ("g5x7", {"prune": 1}, small),
            ("g5x7", {"prune": 1}, large), ("g3x9", {"prune": 1}, large)]
    prev_grid = "g4x5"
    for grid, opts, sc in runs:
        if grid != prev_grid:
            s.set_grid(grids[grid][0], grids[grid][1], config.L, config.delta_t, 0.0)
            prev_grid = grid
        for k, v in opts.items():
            s.set_option(k, v)
        thr = _first_threshold(sc)
        got = _device(s, nat.COST_MM, 3, sc, thr, T)
        fresh = _solver(grids[grid], **opts)
        _assert_same(got, _device(fresh, nat.COST_MM, 3, sc, thr, T), f"{grid} {opts} N {len(sc)}")
        fresh.close()
    s.close()


def test_same_addresses_new_contents(grids):
    """A second call through the same tensors (the handle launches the graph it kept) runs on their new contents."""
    a, b = _random_scenarios(32, 31), _random_scenarios(32, 32)
    s, ref = _solver(grids["g5x7"]), _solver(grids["g5x7"])   # host runs on another handle: s keeps its graph
    run = _DeviceRun(s, nat.COST_MM, 3, a, _first_threshold(a), 50)
    s.sync()
    _assert_same(run.result(), _host(ref, nat.COST_MM, 3, a, _first_threshold(a), 50), "first")
    per_tick = s.stats()["kernel_launches"]
    for t, v in zip(run.inp, (b[:, :3], b[:, 3:5], b[:, :2], _first_threshold(b))):
        t.copy_(torch.from_numpy(np.ascontiguousarray(v)))
    for k, t in run.out.items():
        t.fill_(-9 if k in ("ticks", "status") else math.nan)
    run.launch()
    s.sync()
    assert s.stats()["kernel_launches"] == per_tick
    _assert_same(run.result(), _host(ref, nat.COST_MM, 3, b, _first_threshold(b), 50), "second")
    s.close()
    ref.close()


def test_chained_device_calls_each_equal_their_host_run(grids):
    a, b = _random_scenarios(64, 11), _random_scenarios(64, 12)
    s = _solver(grids["g5x7"])
    ra = _DeviceRun(s, nat.COST_TREE, 3, a, _first_threshold(a), 50)
    rb = _DeviceRun(s, nat.COST_TREE, 3, b, None, 50)         # enqueued behind the first, no sync in between
    s.sync()
    _assert_same(ra.result(), _host(s, nat.COST_TREE, 3, a, _first_threshold(a), 50), "first")
    _assert_same(rb.result(), _host(s, nat.COST_TREE, 3, b, None, 50), "second")
    s.close()


def test_rejected_device_call_consumes_the_trace(grids):
    sc = _random_scenarios(4, 5)
    s = _solver(grids["g4x5"])
    sentinel = torch.full((4 * 10 * 3 * 3,), -7.0, dtype=torch.float64, device="cuda")
    s.set_loop_trace(sentinel.data_ptr(), 0, 0)
    with pytest.raises(nat.MpcbError):                       # max_ticks < 1
        s.full_closed_loop_device(nat.COST_MM, 3, 4, 1, 1, 1, 0, config.eps, 0, 1, 1, 1)
    r = _device(s, nat.COST_MM, 3, sc, None, 10, trace=False)
    assert (r["ticks"] > 0).all()
    assert (sentinel == -7.0).all()
    for bad in (dict(N=-1), dict(N=1 << 31)):
        with pytest.raises(nat.MpcbError):
            s.full_closed_loop_device(nat.COST_MM, 3, bad["N"], 1, 1, 1, 0, config.eps, 10, 1, 1, 1)
    with pytest.raises(nat.MpcbError):                       # null pointer
        s.full_closed_loop_device(nat.COST_MM, 3, 4, 0, 1, 1, 0, config.eps, 10, 1, 1, 1)
    s.close()
    s = nat.Solver(0)
    with pytest.raises(nat.MpcbError) as e:                  # no grid
        s.full_closed_loop_device(nat.COST_MM, 3, 4, 1, 1, 1, 0, config.eps, 10, 1, 1, 1)
    assert e.value.code == -3
    s.close()


def _ngpus():
    try:
        return nat.load().mpcb_device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_ngpus() < 2, reason="needs 2 GPUs")
def test_two_devices_from_one_host_thread(grids):
    """One loop enqueued per device before either is waited for; each equals its run alone."""
    scs = [_random_scenarios(128, 21), _random_scenarios(128, 22)]
    solvers = [_solver(grids["g5x7"], device=d) for d in (0, 1)]
    runs = [_DeviceRun(s, nat.COST_MM, 3, sc, _first_threshold(sc), 60) for s, sc in zip(solvers, scs)]
    for s in solvers:
        s.sync()
    for d, (s, sc, run) in enumerate(zip(solvers, scs, runs)):
        alone = _solver(grids["g5x7"], device=d)
        _assert_same(run.result(), _device(alone, nat.COST_MM, 3, sc, _first_threshold(sc), 60), f"device {d}")
        alone.close()
        s.close()
