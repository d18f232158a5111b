"""GPU: the device returns the float64 oracle's choice far from the world origin, and on the on-target boundary.

Robot logs in UTM coordinates put robots at easting ~5e5 m, northing ~5e6 m.  There every rounding of the reference's
line distance is worth tens of cost units, so the device must form it in the reference's own order, and the fp32
windows must cover the rounding noise the float64 costs then carry.  Regions: the world point (shift, 0.9 shift) for
shifts 0 .. 5e6 m, line origins 0-300 m off the start, targets 5-3,000 m away, headings accumulated to +-10..60 rad.

Bars: identical index; cost rtol 1e-12; trajectories within 4 ulp of the coordinate (atol 1e-12 is below one ulp at
5e6 m).  The closed loops are compared with the per-tick loop driven by the float64 oracle (tests/oracle_backend.py):
identical ticks and status, log rows within 4 ulp.  The knife edges put a robot exactly where is_on_target's separately
rounded dx*dx + dy*dy and either FMA-contracted form disagree."""
import importlib
import math
from fractions import Fraction

import numpy as np
import pytest

from diplomjourney_b200 import config
from oracle import c_oracle as K
from oracle import closed_form as C
from oracle_backend import OracleBackend

pytestmark = pytest.mark.gpu

nat = pytest.importorskip("diplomjourney_b200._native")

COSTS = {C.COST_MM: nat.COST_MM, C.COST_TREE: nat.COST_TREE}
L, DT, VMIN = C.CONFIG["L"], C.CONFIG["delta_t"], C.CONFIG["v_min"]
SHIFTS = [0.0, 1e3, 1e5, 5e5, 5e6]
V, B = np.array([0.0, 0.3, 0.6, 1.0]), np.linspace(-1.0, 1.0, 7)        # S = 28, H = 3: 21,952 leaves


@pytest.fixture(scope="module")
def solver():
    s = nat.Solver(0)
    yield s
    s.close()


def world_scenarios(shift, seed, n=6):
    """(state, target, origin) around the world point (shift, 0.9 shift): the line origin on the start or 0.5-300 m
    off it, targets 5-3,000 m away, headings also accumulated outside [-pi, pi]."""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n):
        st = np.array([shift + rng.uniform(-10, 10), 0.9 * shift + rng.uniform(-10, 10), rng.uniform(-math.pi, math.pi)])
        if k % 3 == 2:
            st[2] += rng.choice([-1.0, 1.0]) * rng.uniform(10, 60)
        dist = [5.0, 12.0, 40.0, 300.0, 3000.0, 8.0][k % 6] * rng.uniform(0.6, 1.0)
        ang = rng.uniform(-math.pi, math.pi)
        tg = st[:2] + dist * np.array([math.cos(ang), math.sin(ang)])
        off = [0.0, 0.5, 5.0, 60.0, 300.0, 20.0][k % 6] * rng.uniform(0.5, 1.0)
        oa = rng.uniform(-math.pi, math.pi)
        out.append((st, tg, st[:2] + off * np.array([math.cos(oa), math.sin(oa)])))
    return out


def _batch(shift, seed):
    sc = world_scenarios(shift, seed)
    return (np.array([s for s, _, _ in sc]), np.array([t for _, t, _ in sc]), np.array([o for _, _, o in sc]))


def _ulps(a, ref):
    """|a - ref| in units of the last place of the coordinate (at least that of 1.0)"""
    a, ref = np.asarray(a, float), np.asarray(ref, float)
    u = np.abs(a - ref) / np.spacing(np.maximum(np.abs(ref), 1.0))
    return np.where(np.isnan(a) & np.isnan(ref), 0.0, u)          # NaN against a number stays NaN and fails


def _check(res, i, ref, what):
    assert res["index"][i] == ref["index"], (what, i, res["index"][i], ref["index"], res["cost"][i], ref["cost"])
    assert res["cost"][i] == pytest.approx(ref["cost"], rel=1e-12), what
    assert _ulps(res["traj"][i], ref["traj"]).max() <= 4, what
    np.testing.assert_array_equal(res["first_control"][i], ref["first_control"], err_msg=what)


FULL_PATHS = [("leafwalk", dict(algo=nat.ALGO_LEAFWALK))] + \
    [(f"prefix screen {sc} npt {npt}", dict(algo=nat.ALGO_PREFIX, prune=0, screen=sc, nodes_per_thread=npt))
     for sc in (0, 1, 2) for npt in (2, 4)] + \
    [(f"prefix prune {pr} cut {cut}", dict(algo=nat.ALGO_PREFIX, prune=pr, subtree_cut=cut))
     for pr in (0, 1) for cut in (1, 3)]
_DEFAULTS = dict(algo=nat.ALGO_AUTO, prune=1, screen=2, nodes_per_thread=4, subtree_cut=2)


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
@pytest.mark.parametrize("shift", SHIFTS)
def test_full_paths_pick_the_oracles_leaf(solver, shift, cost):
    """Every FULL pass-1 flavour (leafwalk; prefix with each screen and nodes per thread; pruned and unpruned with the
    tile and the frontier cut) against the C oracle, in every region."""
    st, tg, og = _batch(shift, int(shift) % 1000 + 31)
    refs = [K.solve_full(st[i], tg[i], og[i], V, B, 3, cost) for i in range(len(st))]
    solver.set_grid(V, B, L, DT, VMIN)
    try:
        for name, opts in FULL_PATHS:
            for k, v in opts.items():
                solver.set_option(k, v)
            res = solver.solve(nat.MODE_FULL, COSTS[cost], 3, st, tg, og)
            for i, ref in enumerate(refs):
                _check(res, i, ref, f"{name} shift {shift:g}")
    finally:
        for k, v in _DEFAULTS.items():
            solver.set_option(k, v)


@pytest.mark.parametrize("small_path", [1, 0])
@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_held_paths_pick_the_oracles_leaf(solver, cost, small_path):
    """HELD solves, the one-launch float64 kernel and the fp32 + refinement pipeline, with and without the slow-down
    override, in every region."""
    solver.set_grid(V, B, L, DT, VMIN)
    solver.set_option("small_path", small_path)
    try:
        for shift in SHIFTS:
            st, tg, og = _batch(shift, int(shift) % 1000 + 43)
            for slow in (0, nat.FLAG_SLOW):
                res = solver.solve(nat.MODE_HELD, COSTS[cost], 3, st, tg, og, flags=np.full(len(st), slow, np.uint8))
                for i in range(len(st)):
                    ref = K.solve_held(st[i], tg[i], og[i], V, B, 3, cost, slow=bool(slow), v_min=VMIN)
                    _check(res, i, ref, f"small_path {small_path} slow {slow} shift {shift:g}")
                    if cost == C.COST_TREE and shift >= 1e5:
                        # no heading term, and the device's sincos moves no position rounded at this size: every
                        # operation is the oracle's, correctly rounded -- so the very bits (A^2 + B^2 not contracted)
                        assert res["cost"][i] == ref["cost"], (shift, i, res["cost"][i], ref["cost"])
    finally:
        solver.set_option("small_path", 1)


def test_held_windows_pick_the_oracles_leaf(solver):
    """One online tick per robot with its own acceleration window (mpcb_solve_held_windows), both costs, in every
    region, against the oracle answering the same tick."""
    be = OracleBackend()
    for cost in (nat.COST_TREE, nat.COST_MM):
        params = nat.LoopParams.from_config(config, cost, 3, 1)
        for shift in SHIFTS:
            st, tg, og = _batch(shift, int(shift) % 1000 + 59)
            rng = np.random.default_rng(int(shift) % 1000)
            vb = np.stack([rng.uniform(0.0, 1.0, len(st)), rng.uniform(-0.5, 0.5, len(st))], axis=1)
            fl = np.array([0, nat.FLAG_SLOW] * (len(st) // 2), np.uint8)
            res = solver.solve_held_windows(params, st, vb, tg, og, flags=fl)
            ref = be.solve_held_windows(params, st, vb, tg, og, flags=fl)
            np.testing.assert_array_equal(res["shape"], ref["shape"])
            np.testing.assert_array_equal(res["index"], ref["index"], err_msg=f"shift {shift:g}")
            np.testing.assert_allclose(res["cost"], ref["cost"], rtol=1e-12, atol=0)
            assert _ulps(res["traj"], ref["traj"]).max() <= 4
            np.testing.assert_array_equal(res["first_control"], ref["first_control"])


# ---------------------------------------------------------------- the fp32 stage against the windows
def _eps_model(s, origin, H, cost, prefix, smax, dphimax, direct=False, world=True):
    """Python mirror of the error bounds prep_kernel computes: tol/2 (the value pass 2 filters with), or with
    ``direct`` tol1/2 (the form pass 1 ranks with).  ``world=False`` leaves out the term for the float64 rounding at
    the solve's coordinates (DESIGN.md section 3.3), to show what it covers."""
    xs, ys, p0, xt, yt = s
    wl, wh = (10.0, math.sqrt(10.0)) if cost == C.COST_MM else (100.0, 0.0)
    A, Bc = yt - origin[1], xt - origin[0]
    norm = math.sqrt(A * A + Bc * Bc)
    e0 = wl * ((A * xs - Bc * ys) + (xt * origin[1] - yt * origin[0])) / norm
    hp0 = wh * (C.heading_reference(xt, yt) - p0)
    Rtot = H * smax
    Rl = smax if prefix else Rtot
    Gl = wh * (dphimax if prefix else H * dphimax)
    E, Hh, Q = abs(e0) + wl * Rtot, abs(hp0) + wh * H * dphimax, wl * Rl
    Phi, X, Y = abs(p0) + H * dphimax, abs(xs) + Rtot, abs(ys) + Rtot
    dphi = H * 2.0 ** -53 * Phi
    dp = H * 2.0 ** -52 * (X + Y) + H * smax * dphi
    de = wl * (2.0 ** -51 * (abs(A) * X + abs(Bc) * Y + abs(xt * origin[1]) + abs(yt * origin[0])) / norm + dp)
    dh = wh * dphi
    Mw = (1e4 * dp + 2 * de * (2 * E + de) + 2 * dh * (2 * Hh + dh)) * 2.0 ** 23 if world else 0.0
    M = 1e4 * Rl * 16 + 4 * Q * (2 * E + Q) + 4 * Gl * (Gl + 2 * Hh) + Mw
    if not prefix:
        M += 1e4 * Rtot * 8 * max(1.0, H * dphimax / math.pi)
    if direct:
        d0 = math.hypot(xt - xs, yt - ys)
        Vmax = 1e4 * (d0 + Rtot) + (E + Q) ** 2 + (Hh + Gl) ** 2
        if prefix:
            M = max(M, 3 * 1e4 * (d0 + Rtot) + 2 * 1e4 * smax + 4 * (E + Q) ** 2 + 3 * (Hh + Gl) ** 2 + Vmax + Mw)
        else:
            M = M + 4 * 1e4 * (d0 + Rtot) + 4 * (E + Q) ** 2 + 3 * (Hh + Gl) ** 2 + Vmax
    return M * 2.0 ** -23


@pytest.mark.parametrize("direct", [0, 1])
@pytest.mark.parametrize("algo", [nat.ALGO_LEAFWALK, nat.ALGO_PREFIX])
@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_fp32_values_stay_inside_the_windows_far_from_the_world_origin(solver, cost, algo, direct):
    """Every leaf's fp32 value (dump_leaves; dump_direct = the form pass 1 ranks with) lies within tol/2 (tol1/2) of
    the oracle's float64 cost, in every region.  Without the world-coordinate term the 5e6 m region is far outside."""
    solver.set_grid(V, B, L, DT, VMIN)
    solver.set_option("dump_direct", direct)
    vv, _, dphi = C.control_tables(V, B, L, DT)
    smax, dphimax = float(np.max(vv) * DT), float(np.max(np.abs(dphi)))
    try:
        for shift in SHIFTS:
            worst = worst_without = 0.0
            for st, tg, og in world_scenarios(shift, int(shift) % 1000 + 71):
                s = np.r_[st, tg]
                _, J = solver.dump_leaves(nat.MODE_FULL, COSTS[cost], 3, st, tg, og, algo=algo)
                Jo = K.full_leaf_costs(st, tg, og, V, B, 3, cost)
                _, x, y, _ = C.full_leaf_costs(st, tg, og, V, B, 3, cost, return_xy=True)
                special = (x == og[0]) & (y == og[1])          # leaves on the line origin carry 1e8 / 1e10
                assert np.all(np.abs(J - Jo)[special] <= 1e-6 * Jo[special])
                err = np.abs(J - Jo)[~special].max()
                args = (s, og, 3, cost, algo == nat.ALGO_PREFIX, smax, dphimax, bool(direct))
                worst = max(worst, err / _eps_model(*args))
                worst_without = max(worst_without, err / _eps_model(*args, world=False))
            print(f"{cost} algo {algo} direct {direct} shift {shift:g}: worst |J32 - J64| = {worst:.3g} of the window "
                  f"half-width ({worst_without:.3g} without the world-coordinate term)")
            assert worst < 1.0, (shift, worst)
            if shift == 5e6:
                assert worst_without > 1.0
    finally:
        solver.set_option("dump_direct", 0)


# ---------------------------------------------------------------- closed loops
def _on_target(x, y, tx, ty):
    return (tx - x) ** 2 + (ty - y) ** 2 <= config.eps          # is_on_target: each square rounded, then the sum


def _full_loop_on_oracle(cost, H, sc, T, grid=(V, B)):
    """math_model.py's closed loop (one FULL solve per tick with the carried threshold, stall repeats the previous
    return, stop on target / after two repeated positions / at T ticks), every solve answered by the oracle."""
    be = OracleBackend()
    be.set_grid(*grid, L, DT)
    N = len(sc)
    log, ticks, status = np.full((N, T, 5), np.nan), np.zeros(N, np.int32), np.zeros(N, np.int32)
    for n, s in enumerate(sc):
        x, tg, og, thr, ret, k = s[:3].copy(), s[3:5], s[:2], math.inf, None, 0
        if _on_target(x[0], x[1], *tg):
            status[n] = nat.LOOP_ON_TARGET
            continue
        for t in range(T):
            r = be.solve(nat.MODE_FULL, cost, H, x, tg, og, threshold=thr)
            if r["index"][0] >= 0:
                ret, thr = list(r["traj"][0, 0]) + list(r["first_control"][0]), float(r["cost"][0])
            elif ret is None:
                status[n] = nat.LOOP_NO_LEAF
                break
            log[n, t] = ret
            ticks[n] = t + 1
            if ret[0] == x[0] and ret[1] == x[1]:
                k += 1
            x = np.array(ret[:3])
            if k == 2:
                status[n] = nat.LOOP_STALLED
                break
            if _on_target(x[0], x[1], *tg):
                status[n] = nat.LOOP_ON_TARGET
                break
            if t + 1 >= T:
                status[n] = nat.LOOP_MAX_TICKS
    return dict(log=log, ticks=ticks, status=status)


def _held_loop_runs(ini, tgt, org, T):
    """math_mpc_batch: the per-tick loop answered by the oracle, and the device-resident loop."""
    mt = importlib.reload(importlib.import_module("diplomjourney_b200.math_model_tree"))
    try:
        mt._backend = OracleBackend()
        ref = mt.math_mpc_batch(ini, tgt, max_ticks=T, origin=org, host_loop=True)
        mt._backend = None
        dev = mt.math_mpc_batch(ini, tgt, max_ticks=T, origin=org)
    finally:
        mt._backend = None
    return ref, dev


def _same_loops(dev, ref, what):
    np.testing.assert_array_equal(dev["ticks"], ref["ticks"], err_msg=what)
    np.testing.assert_array_equal(dev["status"], ref["status"], err_msg=what)
    for n, t in enumerate(ref["ticks"]):
        assert _ulps(dev["log"][n, :t], ref["log"][n, :t]).max(initial=0) <= 4, (what, n)


def test_held_closed_loop_far_from_the_world_origin():
    """The online controller's closed loop of shifted robots, the line origin off the start, on the device and per
    tick on the oracle."""
    rng = np.random.default_rng(3)
    ini, tgt, org = [], [], []
    for shift in SHIFTS:
        for k in range(2):
            x = np.array([shift + rng.uniform(-5, 5), 0.9 * shift + rng.uniform(-5, 5)])
            ini.append([x[0], x[1], rng.uniform(-math.pi, math.pi) + 20.0 * k, 0.5, 0.0])
            tgt.append(x + rng.uniform(0.8, 2.0, 2) * rng.choice([-1, 1], 2))
            org.append(x + rng.uniform(-3, 3, 2) * k)
    ref, dev = _held_loop_runs(np.array(ini), np.array(tgt), np.array(org), 200)
    _same_loops(dev, ref, "held")
    assert (ref["ticks"] > 1).all()


def test_full_closed_loop_far_from_the_world_origin():
    """The FULL-tree closed loop (one graph launch) of shifted robots against the oracle-driven per-tick loop."""
    rng = np.random.default_rng(5)
    sc = []
    for shift in SHIFTS:
        for _ in range(2):
            x = np.array([shift + rng.uniform(-5, 5), 0.9 * shift + rng.uniform(-5, 5)])
            sc.append([x[0], x[1], rng.uniform(-math.pi, math.pi), *(x + rng.uniform(0.3, 1.2, 2) * rng.choice([-1, 1], 2))])
    sc = np.array(sc)
    s = nat.Solver(0)
    try:
        s.set_grid(V, B, L, DT, VMIN)
        for cost in (nat.COST_MM, nat.COST_TREE):
            dev = s.full_closed_loop(cost, 3, sc[:, :3], sc[:, 3:5], sc[:, :2], eps=config.eps, max_ticks=60)
            _same_loops(dev, _full_loop_on_oracle(cost, 3, sc, 60), f"full cost {cost}")
    finally:
        s.close()


# ---------------------------------------------------------------- knife edges of the on-target test
def _fma(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))          # one rounding, as an FMA rounds


def _boundary_target(x, y, eps):
    """A target whose squared distance from (x, y) is <= eps when each product is rounded (is_on_target), but > eps in
    either FMA-contracted form."""
    for i in range(20000):
        ddx = 0.011 + 1e-6 * i
        base = math.sqrt(eps - ddx * ddx)
        for k in range(-4, 5):
            tx, ty = x + ddx, y + base + k * 2.0 ** -60
            dx, dy = tx - x, ty - y
            if dx * dx + dy * dy <= eps and _fma(dx, dx, dy * dy) > eps and _fma(dy, dy, dx * dx) > eps:
                return tx, ty
    raise AssertionError("no boundary target found")


def _fixed_point(pose_of, x, y):
    """The target on the boundary around the pose that the solve towards that very target produces."""
    tg = _boundary_target(x, y, config.eps)
    for _ in range(20):
        px, py = pose_of(tg)
        nt = _boundary_target(px, py, config.eps)
        if nt == tg:
            return tg
        tg = nt
    raise AssertionError("the pose did not settle")


def test_held_loop_robot_on_the_boundary_at_entry():
    ini = np.array([[0.3, -0.2, 0.4, 0.5, 0.0], [1.1, 0.7, 2.0, 0.3, 0.1]])
    tgt = np.array([_boundary_target(0.3, -0.2, config.eps), [2.0, 2.5]])
    org = np.array([[0.0, 0.0], [0.0, 0.0]])
    ref, dev = _held_loop_runs(ini, tgt, org, 100)
    assert ref["status"][0] == nat.LOOP_ON_TARGET and ref["ticks"][0] == 0
    _same_loops(dev, ref, "held on target at entry")


def test_full_loop_robot_whose_first_pose_lands_on_the_boundary():
    """The first accepted pose of a FULL robot lies on the boundary of its target: the loop must stop after one tick,
    as the reference's does.  (A grid without a standstill speed, heading away from the side the boundary target is
    placed on: else the pose that settles is the start itself, on target at entry.)"""
    grid = (np.array([0.3, 0.6, 1.0]), B)
    st = np.array([0.2, 0.1, 0.5 * math.pi])
    be = OracleBackend()
    be.set_grid(*grid, L, DT)

    def first_pose(tg):
        r = be.solve(nat.MODE_FULL, nat.COST_MM, 3, st, tg, st[:2])
        return tuple(r["traj"][0, 0, :2])
    p = first_pose((st[0] + 0.02, st[1] + 0.08))
    tg = _fixed_point(first_pose, *p)
    sc = np.array([[*st, *tg]])
    ref = _full_loop_on_oracle(nat.COST_MM, 3, sc, 30, grid)
    assert ref["status"][0] == nat.LOOP_ON_TARGET and ref["ticks"][0] == 1
    s = nat.Solver(0)
    try:
        s.set_grid(*grid, L, DT, VMIN)
        dev = s.full_closed_loop(nat.COST_MM, 3, sc[:, :3], sc[:, 3:5], sc[:, :2], eps=config.eps, max_ticks=30)
    finally:
        s.close()
    _same_loops(dev, ref, "full boundary pose")


def test_held_loop_predicted_terminal_pose_on_the_boundary():
    """The terminal pose of a held robot's first predicted trajectory lies on the boundary of its target: the
    finishing heuristic counts m there (math_model_tree.py:392-414) exactly when the reference does."""
    params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, 1)
    be = OracleBackend()
    ini = np.array([0.2, 0.1, 0.5, 0.9, 0.0])
    org = np.array([0.0, 0.0])

    def terminal(tg):
        r = be.solve_held_windows(params, ini[:3], ini[3:5], tg, org)
        return tuple(r["traj"][0, -1, :2])
    p = terminal((0.5, 0.3))
    tg = _fixed_point(terminal, *p)
    ref, dev = _held_loop_runs(ini[None], np.array([tg]), org[None], 100)
    assert ref["robots"][0]["m"] >= 1
    _same_loops(dev, ref, "held boundary terminal pose")
    assert int(dev["final"][0, 5]) == ref["robots"][0]["m"]
