"""GPU parity: the CUDA path (through the C ABI, libmpcb200.so) against the float64 oracle and
the golden fixtures produced by the reference's own functions.

Bars (SURVEY 8d): the winning leaf index is IDENTICAL to the float64 oracle's (the refinement
pass re-evaluates near-minimal leaves in float64 with the reference's formula), cost rtol 1e-12,
trajectory atol 1e-12.  The fp32 stage is checked separately against its own error model."""
import math

import numpy as np
import pytest

from oracle import c_oracle as K
from oracle import closed_form as C

pytestmark = pytest.mark.gpu

nat = pytest.importorskip("diplomjourney_b200._native")

COSTS = {C.COST_MM: nat.COST_MM, C.COST_TREE: nat.COST_TREE}
L, DT, VMIN = C.CONFIG["L"], C.CONFIG["delta_t"], C.CONFIG["v_min"]


@pytest.fixture(scope="module")
def solver():
    s = nat.Solver(0)
    yield s
    s.close()


def _check(res, i, ref, H):
    assert res["index"][i] == ref["index"], (res["index"][i], ref["index"], res["cost"][i], ref["cost"])
    assert res["cost"][i] == pytest.approx(ref["cost"], rel=1e-12)
    np.testing.assert_allclose(res["traj"][i], ref["traj"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(res["first_control"][i], ref["first_control"], rtol=0, atol=0)


@pytest.mark.parametrize("algo", [nat.ALGO_LEAFWALK, nat.ALGO_PREFIX])
def test_full_golden_reference_outputs(solver, golden, algo):
    g = golden("full_h3")
    solver.set_option("algo", algo)
    try:
        for case in g["cases"]:
            sc = case["scenario"]
            solver.set_grid(case["vector_v"], case["vector_beta"], L, DT, VMIN)
            prev = None
            for tick in case["ticks"]:
                r = solver.solve(nat.MODE_FULL, nat.COST_MM, 3, tick["state"], (sc["x_t"], sc["y_t"]),
                                 (sc["x_0"], sc["y_0"]), threshold=tick["threshold"])
                if r["index"][0] >= 0:
                    ret = list(r["traj"][0, 0]) + list(r["first_control"][0])
                    np.testing.assert_allclose(ret, tick["ret"], rtol=0, atol=1e-12)
                    np.testing.assert_allclose(r["traj"][0], np.array(tick["traj"]), rtol=0, atol=1e-12)
                    assert r["cost"][0] == pytest.approx(tick["criterion_after"], rel=1e-12)
                else:  # stall: nothing beats the carried threshold, the reference repeats itself
                    assert tick["ret"] == prev and tick["criterion_after"] == tick["threshold"]
                prev = tick["ret"]
    finally:
        solver.set_option("algo", nat.ALGO_AUTO)


@pytest.mark.parametrize("small_path", [1, 0])
def test_held_golden_reference_outputs(solver, golden, small_path):
    """small_path=1: one-launch float64 kernel; 0: the general fp32 leafwalk + float64 refinement pipeline."""
    g = golden("held_single")
    solver.set_option("small_path", small_path)
    for c in g["cases"]:
        solver.set_grid(c["vector_v"], c["vector_beta"], L, DT, VMIN)
        r = solver.solve(nat.MODE_HELD, nat.COST_TREE, 3, c["state"], c["target"], c["origin"],
                         flags=nat.FLAG_SLOW if c["slow"] else 0)
        ret = list(r["traj"][0, 0]) + list(r["first_control"][0])
        np.testing.assert_allclose(ret, c["ret"], rtol=0, atol=1e-12)
        np.testing.assert_allclose(r["traj"][0], np.array(c["traj"]), rtol=0, atol=1e-12)
        assert solver.stats()["kernel_launches"] == (1 if small_path else 8)   # prep, pass 1, reduce, pass 2, 3 x candidates, finalize
    solver.set_option("small_path", 1)


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
@pytest.mark.parametrize("H", [1, 2, 3, 4])
@pytest.mark.parametrize("algo", [nat.ALGO_LEAFWALK, nat.ALGO_PREFIX])
def test_full_small_trees_vs_oracle(solver, cost, H, algo):
    V, B = [0.0, 0.3, 0.6, 1.0], np.linspace(-1, 1, 7)
    solver.set_grid(V, B, L, DT, VMIN)
    solver.set_option("algo", algo)
    try:
        sc = C.random_scenarios(24, 100 + H)
        res = solver.solve(nat.MODE_FULL, COSTS[cost], H, sc[:, :3], sc[:, 3:5], sc[:, :2])
        for i, s in enumerate(sc):
            _check(res, i, K.solve_full(s[:3], s[3:], s[:2], V, B, H, cost), H)
    finally:
        solver.set_option("algo", nat.ALGO_AUTO)


@pytest.mark.parametrize("algo", [nat.ALGO_LEAFWALK, nat.ALGO_PREFIX])
@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_fp32_stage_within_error_model(solver, algo, cost):
    """All-leaf dump of the fp32 stage vs float64 oracle: the per-leaf error stays inside the
    window the refinement pass assumes (P.tol/2), with margin."""
    V, B = [0.0, 0.3, 0.6, 1.0], np.linspace(-1, 1, 9)
    solver.set_grid(V, B, L, DT, VMIN)
    H = 3
    sc = C.random_scenarios(12, 5)
    # plus near-target starts (NEAR regime) and off-line origins
    near = sc[:4].copy()
    near[:, 3] = near[:, 0] + 0.07
    near[:, 4] = near[:, 1] - 0.05
    worst = 0.0
    for s, origin in [(s, s[:2]) for s in sc] + [(s, s[:2] + [0.4, -0.2]) for s in near]:
        xy, J = solver.dump_leaves(nat.MODE_FULL, COSTS[cost], H, s[:3], s[3:5], origin, algo=algo)
        Jo, xo, yo, _ = C.full_leaf_costs(s[:3], s[3:5], origin, V, B, H, cost, return_xy=True)
        ok = Jo < 1e7     # the "on the origin" leaves carry 1e8/1e10 and are compared relatively
        err = np.abs(J - Jo)
        worst = max(worst, err[ok].max())
        assert np.all(err[~ok] <= 1e-6 * Jo[~ok])
        np.testing.assert_allclose(xy[:, 0], xo, atol=2e-5)
        np.testing.assert_allclose(xy[:, 1], yo, atol=2e-5)
    # error model (prep_kernel): eps = tol/2; measured error must stay below it
    reach = (1 if algo == nat.ALGO_PREFIX else H) * 1.0 * DT
    eps_model = (1e4 * reach * 16 + (0 if algo == nat.ALGO_PREFIX else 1e4 * H * DT * 8)) * 2.0 ** -23
    assert worst < eps_model, (worst, eps_model)


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_full_default_window_grid_vs_oracle(solver, cost):
    """S=451 (11x41 acceleration window), H=3: 9.2e7 leaves per solve, prefix kernel."""
    V, B = C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0)
    solver.set_grid(V, B, L, DT, VMIN)
    sc = C.random_scenarios(6, 42)
    res = solver.solve(nat.MODE_FULL, COSTS[cost], 3, sc[:, :3], sc[:, 3:5], sc[:, :2])
    assert solver.stats()["algo"] == nat.ALGO_PREFIX
    for i, s in enumerate(sc):
        _check(res, i, K.solve_full(s[:3], s[3:], s[:2], V, B, 3, cost), 3)


def test_held_full_resolution_grid_batch(solver):
    """HELD on the FULL scripts' 201x121 grid (S=24,321) for a batch of robots, both costs."""
    V, B = C.grid_full_default()
    solver.set_grid(V, B, L, DT, VMIN)
    sc = C.random_scenarios(16, 9)
    for cost in (C.COST_MM, C.COST_TREE):
        res = solver.solve(nat.MODE_HELD, COSTS[cost], 3, sc[:, :3], sc[:, 3:5], sc[:, :2])
        for i, s in enumerate(sc):
            _check(res, i, K.solve_held(s[:3], s[3:], s[:2], V, B, 3, cost), 3)


def test_zero_velocity_exact_ties_pick_first_leaf(solver):
    V, B = [0.0], np.linspace(-1, 1, 5)
    solver.set_grid(V, B, L, DT, VMIN)
    for mode in (nat.MODE_FULL, nat.MODE_HELD):
        for origin in ((0.0, 0.0), (1.0, 2.0)):      # second: start IS the origin -> special case on every leaf
            r = solver.solve(mode, nat.COST_MM, 3, [1.0, 2.0, 0.3], (3.0, 4.0), origin)
            assert r["index"][0] == 0
    # v=0 at the last step only: 5-way exact tie below one parent -> lowest beta index
    V2 = [0.0, 1.0]
    solver.set_grid(V2, B, L, DT, VMIN)
    s = [0.0, 0.0, 0.0]
    tgt = (0.1, 0.0)   # two steps at v=1 land on it; third step must stop
    r = solver.solve(nat.MODE_FULL, nat.COST_TREE, 3, s, tgt, (-1.0, 0.0))
    ref = K.solve_full(s, tgt, (-1.0, 0.0), V2, B, 3, C.COST_TREE)
    assert r["index"][0] == ref["index"]


def test_threshold_and_split_ranges(solver):
    V, B = [0.0, 0.5, 1.0], np.linspace(-1, 1, 5)
    solver.set_grid(V, B, L, DT, VMIN)
    s = C.random_scenarios(1, 5)[0]
    whole = solver.solve(nat.MODE_FULL, nat.COST_MM, 3, s[:3], s[3:5], s[:2])
    ref = K.solve_full(s[:3], s[3:], s[:2], V, B, 3)
    assert whole["index"][0] == ref["index"]
    # threshold exactly at the minimum -> strict '<' rejects (math_model.py:195)
    r = solver.solve(nat.MODE_FULL, nat.COST_MM, 3, s[:3], s[3:5], s[:2], threshold=whole["cost"][0])
    assert r["index"][0] == -1 and r["cost"][0] == whole["cost"][0]
    r = solver.solve(nat.MODE_FULL, nat.COST_MM, 3, s[:3], s[3:5], s[:2], threshold=np.nextafter(whole["cost"][0], np.inf))
    assert r["index"][0] == whole["index"][0]
    # contiguous first-control shares recombine to the whole-tree answer
    parts = [solver.solve(nat.MODE_FULL, nat.COST_MM, 3, s[:3], s[3:5], s[:2], i0_range=rg)
             for rg in ((0, 4), (4, 9), (9, 15))]
    for p, rg in zip(parts, ((0, 4), (4, 9), (9, 15))):
        pr = K.solve_full(s[:3], s[3:], s[:2], V, B, 3, i0_range=rg)
        assert p["index"][0] == pr["index"]
    best = min(parts, key=lambda r: (r["cost"][0], r["index"][0]))
    assert best["index"][0] == whole["index"][0]


def test_degenerate_inputs_do_not_select_a_leaf(solver):
    V, B = [0.0, 0.5, 1.0], np.linspace(-1, 1, 5)
    solver.set_grid(V, B, L, DT, VMIN)
    # target == line origin: 0/0 in the line distance -> every cost NaN -> no leaf (reference: ZeroDivisionError)
    r = solver.solve(nat.MODE_FULL, nat.COST_MM, 3, [0.0, 0.0, 0.0], (1.0, 1.0), (1.0, 1.0))
    assert r["index"][0] == -1 and math.isnan(r["cost"][0])
    with pytest.raises(nat.MpcbError):
        solver.set_grid([], B, L, DT, VMIN)
    with pytest.raises(nat.MpcbError):
        solver.solve(nat.MODE_FULL, nat.COST_MM, 3, [0.0, 0.0, 0.0], (1.0, 1.0), (0.0, 0.0))  # grid was dropped


def test_prefix_multi_chunk_table_and_reference_default_grid(solver):
    """S > 1024 makes the prefix kernel stream the leaf table through shared memory in chunks.
    (a) 30x50 grid, H=2 and 3 restricted to a few first controls; (b) the reference's own default
    201x121 grid (S=24,321, math_model.py:23-30) at H=2: 5.9e8 leaves, the tree the reference cannot allocate."""
    V, B = np.linspace(0.0, 1.0, 30), np.linspace(-1.0, 1.0, 50)
    solver.set_grid(V, B, L, DT, VMIN)
    solver.set_option("algo", nat.ALGO_PREFIX)
    try:
        sc = C.random_scenarios(3, 21)
        res = solver.solve(nat.MODE_FULL, nat.COST_MM, 2, sc[:, :3], sc[:, 3:5], sc[:, :2])
        for i, s in enumerate(sc):
            _check(res, i, K.solve_full(s[:3], s[3:], s[:2], V, B, 2, C.COST_MM), 2)
        s = sc[0]
        r = solver.solve(nat.MODE_FULL, nat.COST_TREE, 3, s[:3], s[3:5], s[:2], i0_range=(1490, 1500))
        o = K.solve_full(s[:3], s[3:], s[:2], V, B, 3, C.COST_TREE, i0_range=(1490, 1500))
        assert r["index"][0] == o["index"] and r["cost"][0] == pytest.approx(o["cost"], rel=1e-12)
        Vd, Bd = C.grid_full_default()
        solver.set_grid(Vd, Bd, L, DT, VMIN)
        s = np.array([0.0, 0.0, 0.0, 1.0, 5.0])          # config.py start and target; the start IS the line origin
        r = solver.solve(nat.MODE_FULL, nat.COST_MM, 2, s[:3], s[3:5], s[:2])
        assert solver.stats()["leaves_per_solve"] == 24321 ** 2
        _check(r, 0, K.solve_full(s[:3], s[3:], s[:2], Vd, Bd, 2, C.COST_MM), 2)
    finally:
        solver.set_option("algo", nat.ALGO_AUTO)


@pytest.mark.parametrize("algo", [nat.ALGO_LEAFWALK, nat.ALGO_PREFIX])
def test_long_horizons(solver, algo):
    """H = 6 and 8 (the reference hard-codes 3): index decoding over many digits, 64-bit paths."""
    solver.set_option("algo", algo)
    try:
        for H, V, B in ((6, [0.2, 1.0], np.linspace(-0.9, 0.9, 4)), (8, [0.5, 1.0], [-0.8, 0.0, 0.8])):
            solver.set_grid(V, B, L, DT, VMIN)
            sc = C.random_scenarios(4, 30 + H)
            res = solver.solve(nat.MODE_FULL, nat.COST_TREE, H, sc[:, :3], sc[:, 3:5], sc[:, :2])
            for i, s in enumerate(sc):
                _check(res, i, K.solve_full(s[:3], s[3:], s[:2], V, B, H, C.COST_TREE), H)
    finally:
        solver.set_option("algo", nat.ALGO_AUTO)


def test_config0_default_full_tree_subtrees(solver):
    """BASELINE configs[0]: run_math_model.py's default scenario -- start (0,0,0), target (1,5), H=3 on the
    201x121 grid: 1.44e13 leaves (the reference's np.empty([S**3, 3]) is a 345 TB allocation).  Here: three
    first-control subtrees (5.9e8 leaves each) against the C oracle; the whole tree is timed in profiles/."""
    Vd, Bd = C.grid_full_default()
    solver.set_grid(Vd, Bd, L, DT, VMIN)
    s = np.array([0.0, 0.0, 0.0, 1.0, 5.0])
    for i0 in (0, 12160, 24320):
        r = solver.solve(nat.MODE_FULL, nat.COST_MM, 3, s[:3], s[3:5], s[:2], i0_range=(i0, i0 + 1))
        o = K.solve_full(s[:3], s[3:], s[:2], Vd, Bd, 3, C.COST_MM, i0_range=(i0, i0 + 1))
        assert r["index"][0] == o["index"], (i0, r["index"][0], o["index"])
        assert r["cost"][0] == pytest.approx(o["cost"], rel=1e-12)
        np.testing.assert_allclose(r["traj"][0], o["traj"], rtol=0, atol=1e-12)


def _eps_model(s, origin, H, cost, prefix, smax, dphimax, direct=False):
    """Python mirror of the error bounds prep_kernel computes: tol/2 (the value pass 2 filters with), or with
    ``direct`` tol1/2 (the cheaper direct form the prefix pass 1 ranks with)."""
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
    # float64 rounding at the solve's coordinates (heading, position, line-distance sum; DESIGN.md section 3.3)
    Phi, X, Y = abs(p0) + H * dphimax, abs(xs) + Rtot, abs(ys) + Rtot
    dphi = H * 2.0 ** -53 * Phi
    dp = H * 2.0 ** -52 * (X + Y) + H * smax * dphi
    de = wl * (2.0 ** -51 * (abs(A) * X + abs(Bc) * Y + abs(xt * origin[1]) + abs(yt * origin[0])) / norm + dp)
    dh = wh * dphi
    Mw = (1e4 * dp + 2 * de * (2 * E + de) + 2 * dh * (2 * Hh + dh)) * 2.0 ** 23
    M = 1e4 * Rl * 16 + 4 * Q * (2 * E + Q) + 4 * Gl * (Gl + 2 * Hh) + Mw
    if not prefix:
        M += 1e4 * Rtot * 8 * max(1.0, H * dphimax / math.pi)
    if direct:
        d0 = math.hypot(xt - xs, yt - ys)
        Vmax = 1e4 * (d0 + Rtot) + (E + Q) ** 2 + (Hh + Gl) ** 2      # the accumulating FFMAs round at this size
        if prefix:
            M1 = 3 * 1e4 * (d0 + Rtot) + 2 * 1e4 * smax + 4 * (E + Q) ** 2 + 3 * (Hh + Gl) ** 2 + Vmax + Mw
            M = max(M, M1)
        else:
            M = M + 4 * 1e4 * (d0 + Rtot) + 4 * (E + Q) ** 2 + 3 * (Hh + Gl) ** 2 + Vmax
    return M * 2.0 ** -23


@pytest.mark.parametrize("algo", [nat.ALGO_LEAFWALK, nat.ALGO_PREFIX, "prefix_direct", "leafwalk_direct"])
@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_fp32_stage_error_stays_inside_the_refinement_window(solver, algo, cost):
    """Every leaf of many small trees (far / near the target / far off the tracked line): the fp32 value the
    kernels compare lies within the per-solve window half-width eps that the refinement pass assumes.
    "prefix_direct" / "leafwalk_direct" dump the values the two pass-1 kernels RANK with (leaf_val_direct,
    leaf_walk_direct) against their own bound tol1/2."""
    direct = algo in ("prefix_direct", "leafwalk_direct")
    if direct:
        algo = nat.ALGO_PREFIX if algo == "prefix_direct" else nat.ALGO_LEAFWALK
    solver.set_option("dump_direct", 1 if direct else 0)
    V, B = [0.0, 0.3, 0.6, 1.0], np.linspace(-1, 1, 9)
    solver.set_grid(V, B, L, DT, VMIN)
    vv, bb, dphi = C.control_tables(V, B, L, DT)
    smax, dphimax = float(np.max(vv) * DT), float(np.max(np.abs(dphi)))
    H = 3
    sc = C.random_scenarios(10, 77)
    cases = [(s, s[:2]) for s in sc]
    for s in sc[:5]:
        n = s.copy(); n[3], n[4] = n[0] + 0.06, n[1] + 0.04           # NEAR regime
        cases.append((n, n[:2]))
        cases.append((s, s[:2] + np.array([3.0, -2.0])))              # robot metres away from the tracked line
    worst_ratio = 0.0
    for s, origin in cases:
        _, J = solver.dump_leaves(nat.MODE_FULL, COSTS[cost], H, s[:3], s[3:5], origin, algo=algo)
        Jo = C.full_leaf_costs(s[:3], s[3:5], origin, V, B, H, cost)
        ok = Jo < 1e7
        eps = _eps_model(s, origin, H, cost, algo == nat.ALGO_PREFIX, smax, dphimax, direct)
        worst_ratio = max(worst_ratio, float(np.abs(J - Jo)[ok].max() / eps))
    solver.set_option("dump_direct", 0)
    assert worst_ratio < 1.0, worst_ratio


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_branch_and_bound_is_exact(solver, cost):
    """option prune=1 (default) skips depth-(H-1) nodes that provably cannot hold the argmin and, with subtree_cut
    (H >= 3; 1 = per 256-node tile, 3 = frontier descent from the root incl. its overflow fallback, 2 = auto),
    whole subtrees that cannot: the answers must be bit-identical to
    prune=0 (every leaf evaluated) and to the oracle -- on wide-speed grids where most nodes are cut, on the narrow
    acceleration window where few are, on a deep tree with a tiny grid (a tile straddles many depth-(H-2) nodes) and
    on a grid with S > 1024 restricted to a few first controls (warp-queue kernel walking the survivor list)."""
    grids = [(np.linspace(0.0, 1.0, 16), np.linspace(-np.radians(60), np.radians(60), 16), 3, 8, None),
             (C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0), 3, 4, None),
             (np.linspace(0.0, 1.0, 6), np.linspace(-1.0, 1.0, 7), 4, 8, None),
             (np.linspace(0.0, 1.0, 3), np.linspace(-1.0, 1.0, 4), 5, 6, None),
             (np.linspace(0.0, 1.0, 30), np.linspace(-1.0, 1.0, 50), 3, 2, (1480, 1500))]
    solver.set_option("algo", nat.ALGO_PREFIX)
    try:
        for V, B, H, n, i0 in grids:
            solver.set_grid(V, B, L, DT, VMIN)
            sc = C.random_scenarios(n, 500 + H)
            sc[0, 3:5] = sc[0, :2] + [0.05, 0.02]                      # one robot already next to its target
            args = (nat.MODE_FULL, COSTS[cost], H, sc[:, :3], sc[:, 3:5], sc[:, :2])
            solver.set_option("prune", 0)
            full = solver.solve(*args, i0_range=i0)
            assert solver.stats()["pruned_units"] == 0
            solver.set_option("prune", 1)
            pruned = {}
            for subtree, cap in ((0, None), (1, None), (2, None), (3, None), (3, 48)):   # cap 48: a frontier overflows -> tile path
                solver.set_option("subtree_cut", subtree)
                solver.set_option("frontier_cap", cap or 2 ** 22)
                cut = solver.solve(*args, i0_range=i0)
                st = solver.stats()
                pruned[(subtree, cap)] = st["pruned_units"]
                assert 0 <= st["pruned_units"] <= st["units"] * n, (subtree, cap, st)
                np.testing.assert_array_equal(cut["index"], full["index"])
                np.testing.assert_array_equal(cut["cost"], full["cost"])
                np.testing.assert_array_equal(cut["traj"], full["traj"])
                for i, s in enumerate(sc):
                    _check(cut, i, K.solve_full(s[:3], s[3:], s[:2], V, B, H, cost, i0_range=i0), H)
                if len(V) == 16:
                    assert st["pruned_units"] > 0.2 * st["units"] * n      # v in [0,1]: many nodes cannot win
    finally:
        solver.set_option("subtree_cut", 2)
        solver.set_option("frontier_cap", 2 ** 22)
        solver.set_option("prune", 1)
        solver.set_option("algo", nat.ALGO_AUTO)


def test_branch_and_bound_random_sweep(solver):
    """A few hundred random scenarios per grid -- robots facing away from, next to and far from their targets, robots off
    the tracked line, a grid that cannot stop, one that starts from rest, one with reverse speeds -- solved exhaustively
    and with both subtree-cut modes: bit-identical records (tools/prune_sweep.py is the long version)."""
    n = 128
    cases = [(C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0), 3),
             (np.linspace(0, 1, 16), np.linspace(-np.radians(60), np.radians(60), 16), 3),
             (np.linspace(0.1, 1, 7), np.linspace(-1.4, 1.4, 9), 4),
             (np.linspace(-0.5, 1, 5), np.linspace(-1, 1, 5), 5)]
    solver.set_option("algo", nat.ALGO_PREFIX)
    try:
        for ci, (V, B, H) in enumerate(cases):
            solver.set_grid(V, B, L, DT, VMIN)
            sc = C.random_scenarios(n, 2000 + ci)
            k = n // 8
            sc[:k, 3:5] = sc[:k, :2] + np.random.default_rng(ci).uniform(-0.1, 0.1, (k, 2))
            sc[k:2 * k, 3:5] = sc[k:2 * k, :2] + np.random.default_rng(ci + 50).uniform(-300, 300, (k, 2))
            origin = sc[:, :2].copy()
            origin[2 * k:3 * k] += np.random.default_rng(ci + 99).uniform(-5, 5, (k, 2))
            for cost in (nat.COST_MM, nat.COST_TREE):
                args = (nat.MODE_FULL, cost, H, sc[:, :3], sc[:, 3:5], origin)
                solver.set_option("prune", 0)
                ref = solver.solve(*args)
                solver.set_option("prune", 1)
                for mode in (1, 3):
                    solver.set_option("subtree_cut", mode)
                    cut = solver.solve(*args)
                    for key in ("index", "cost", "traj", "first_control"):
                        np.testing.assert_array_equal(cut[key], ref[key], err_msg=f"case {ci} cost {cost} mode {mode} {key}")
    finally:
        solver.set_option("subtree_cut", 2)
        solver.set_option("prune", 1)
        solver.set_option("algo", nat.ALGO_AUTO)


def test_many_segments_per_solve(solver):
    """One solve with 65,536 segments (H=4 on the 16x16 grid, 4.3e9 leaves): from 32,768 segments per solve on, the
    per-solve reduction of the segment minima and the compaction of the work list run grid-wide instead of on one
    CTA per solve.  Exhaustive and pruned against the C oracle."""
    V, B = np.linspace(0.0, 1.0, 16), np.linspace(-np.radians(60), np.radians(60), 16)
    solver.set_grid(V, B, L, DT, VMIN)
    s = C.random_scenarios(1, 4242)[0]
    o = K.solve_full(s[:3], s[3:], s[:2], V, B, 4, C.COST_MM)
    try:
        for prune in (0, 1):
            solver.set_option("prune", prune)
            r = solver.solve(nat.MODE_FULL, nat.COST_MM, 4, s[:3], s[3:5], s[:2])
            assert solver.stats()["segments"] == 65536
            _check(r, 0, o, 4)
    finally:
        solver.set_option("prune", 1)


def test_slow_flag_is_held_only(solver):
    """MPCB_FLAG_SLOW is the online controller's override; a FULL solve must ignore it (both algorithms)."""
    V, B = [0.2, 0.6, 1.0], np.linspace(-1, 1, 5)
    solver.set_grid(V, B, L, DT, VMIN)
    s = C.random_scenarios(1, 3)[0]
    ref = K.solve_full(s[:3], s[3:], s[:2], V, B, 3, C.COST_MM)
    for algo in (nat.ALGO_LEAFWALK, nat.ALGO_PREFIX):
        solver.set_option("algo", algo)
        r = solver.solve(nat.MODE_FULL, nat.COST_MM, 3, s[:3], s[3:5], s[:2], flags=nat.FLAG_SLOW)
        assert r["index"][0] == ref["index"] and r["cost"][0] == pytest.approx(ref["cost"], rel=1e-12)
    solver.set_option("algo", nat.ALGO_AUTO)
    held = solver.solve(nat.MODE_HELD, nat.COST_TREE, 3, s[:3], s[3:5], s[:2], flags=nat.FLAG_SLOW)
    o = K.solve_held(s[:3], s[3:], s[:2], V, B, 3, C.COST_TREE, slow=True)
    assert held["index"][0] == o["index"] and held["first_control"][0, 0] == 0.4     # max(min V, v_min)


def test_large_heading_changes_stay_exact(solver):
    """Short wheelbase => up to ~1.7 rad of heading change per step: sin.approx/cos.approx leave their accurate
    range in the leafwalk kernel; the window model widens with it and the result stays the float64 argmin."""
    V, B = [0.3, 1.0], np.linspace(-1.0, 1.0, 7)
    Lshort = 0.05
    for algo in (nat.ALGO_LEAFWALK, nat.ALGO_PREFIX):
        solver.set_option("algo", algo)
        solver.set_grid(V, B, Lshort, DT, VMIN)
        sc = C.random_scenarios(12, 909)
        res = solver.solve(nat.MODE_FULL, nat.COST_MM, 4, sc[:, :3], sc[:, 3:5], sc[:, :2])
        for i, s in enumerate(sc):
            _check(res, i, K.solve_full(s[:3], s[3:], s[:2], V, B, 4, C.COST_MM, L=Lshort), 4)
    solver.set_option("algo", nat.ALGO_AUTO)


@pytest.mark.parametrize("small_path", [1, 0])
def test_skip_flag(solver, small_path):
    """MPCB_FLAG_SKIP: entries of a batch that are not to be solved come back as (NaN, -1) on every path."""
    V, B = C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0)
    solver.set_grid(V, B, L, DT, VMIN)
    solver.set_option("small_path", small_path)
    sc = C.random_scenarios(4, 8)
    flags = np.array([0, nat.FLAG_SKIP, nat.FLAG_SLOW, nat.FLAG_SKIP | nat.FLAG_SLOW], np.uint8)
    r = solver.solve(nat.MODE_HELD, nat.COST_TREE, 3, sc[:, :3], sc[:, 3:5], sc[:, :2], flags=flags)
    solver.set_option("small_path", 1)
    assert list(r["index"][[1, 3]]) == [-1, -1] and np.all(np.isnan(r["cost"][[1, 3]]))
    for i, slow in ((0, False), (2, True)):
        o = K.solve_held(sc[i, :3], sc[i, 3:5], sc[i, :2], V, B, 3, C.COST_TREE, slow=slow)
        assert r["index"][i] == o["index"] and r["cost"][i] == pytest.approx(o["cost"], rel=1e-12)
    full = solver.solve(nat.MODE_FULL, nat.COST_MM, 2, sc[:, :3], sc[:, 3:5], sc[:, :2], flags=flags)
    assert list(full["index"][[1, 3]]) == [-1, -1] and full["index"][0] >= 0 and full["index"][2] >= 0


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_several_nodes_per_thread_is_bit_identical(solver, cost):
    """option nodes_per_thread=2 / 4 (exhaustive prefix pass 1 with several depth-(H-1) nodes per thread) does the same
    arithmetic per node: identical results to nodes_per_thread=1 and to the oracle, including ragged last tiles,
    a robot on the line origin, a robot next to its target (NEAR regime) and a chunked table (S > 1024)."""
    grids = [(np.linspace(0.0, 1.0, 11), np.linspace(-1.0, 1.0, 13), 3, 6),        # 143^2 nodes: ragged tiles
             (C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0), 3, 4),
             (np.linspace(0.1, 1.0, 30), np.linspace(-1.0, 1.0, 41), 2, 5)]        # S = 1230: two table chunks
    solver.set_option("algo", nat.ALGO_PREFIX)
    solver.set_option("prune", 0)
    try:
        for V, B, H, n in grids:
            solver.set_grid(V, B, L, DT, VMIN)
            sc = C.random_scenarios(n, 900 + H)
            sc[0, 3:5] = sc[0, :2] + [0.05, 0.02]
            solver.set_option("nodes_per_thread", 1)
            one = solver.solve(nat.MODE_FULL, COSTS[cost], H, sc[:, :3], sc[:, 3:5], sc[:, :2])
            for npt in (2, 4):
                solver.set_option("nodes_per_thread", npt)
                two = solver.solve(nat.MODE_FULL, COSTS[cost], H, sc[:, :3], sc[:, 3:5], sc[:, :2])
                for k in ("index", "cost", "traj", "first_control"):
                    np.testing.assert_array_equal(two[k], one[k])
            for i, s in enumerate(sc):
                _check(two, i, K.solve_full(s[:3], s[3:], s[:2], V, B, H, cost), H)
    finally:
        solver.set_option("nodes_per_thread", 2)                       # library default
        solver.set_option("prune", 1)
        solver.set_option("algo", nat.ALGO_AUTO)


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_screened_pass1_is_exact(solver, cost):
    """option screen=1 (default of the exhaustive prefix pass 1: the MUFU.SQRT of a leaf is only spent in nodes that
    hold a leaf which can still matter, against the probe's upper bound) returns the records of screen=0 and of the
    oracle: ragged tiles, a robot on its line origin, one next to its target (NEAR), zero-velocity exact ties, a
    chunked table (S > 1024), first-control ranges (a range whose held sequences give no bound at all included) and
    carried thresholds."""
    grids = [(np.linspace(0.0, 1.0, 11), np.linspace(-1.0, 1.0, 13), 3, 8),
             (C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0), 3, 6),
             (C.vector_of_velocities(0.01), C.vector_of_beta_angles(0.9), 3, 4),       # clipped window with v = 0 rows
             (np.linspace(0.1, 1.0, 30), np.linspace(-1.0, 1.0, 41), 2, 5),           # S = 1230: two table chunks
             (np.linspace(0.0, 1.0, 6), np.linspace(-1.0, 1.0, 7), 4, 4)]
    solver.set_option("algo", nat.ALGO_PREFIX)
    solver.set_option("prune", 0)
    try:
        for V, B, H, n in grids:
            solver.set_grid(V, B, L, DT, VMIN)
            S = len(V) * len(B)
            sc = C.random_scenarios(n, 1200 + H + S)
            sc[0, 3:5] = sc[0, :2] + [0.05, 0.02]                   # next to its target
            sc[1, 3:5] = sc[1, :2] + [0.0, 1e-3]                    # the optimum stands still: exact ties
            thr = np.full(n, np.inf); thr[2] = 1.0                  # nothing beats this one
            for rng_ in (None, (0, max(1, S // 3)), (S // 2, S // 2 + 1)):
                res = []
                for scr in (0, 1):
                    solver.set_option("screen", scr)
                    res.append(solver.solve(nat.MODE_FULL, COSTS[cost], H, sc[:, :3], sc[:, 3:5], sc[:, :2], threshold=thr,
                                            i0_range=rng_))
                for k in ("index", "cost", "traj", "first_control"):
                    np.testing.assert_array_equal(res[1][k], res[0][k], err_msg=f"{k} S={S} H={H} range={rng_}")
                if rng_ is None and S ** H <= 3e7:
                    for i, s_ in enumerate(sc):
                        o = K.solve_full(s_[:3], s_[3:], s_[:2], V, B, H, cost, threshold=thr[i])
                        assert res[1]["index"][i] == o["index"], (S, H, i)
    finally:
        solver.set_option("screen", 1)
        solver.set_option("prune", 1)
        solver.set_option("algo", nat.ALGO_AUTO)


@pytest.mark.parametrize("algo", [nat.ALGO_LEAFWALK, nat.ALGO_PREFIX])
def test_candidate_list_sizes_give_identical_records(solver, algo):
    """option candidate_list: the in-window leaves of the refinement pass are listed and evaluated in float64 one thread
    each; with a list that is too small (5 entries) the excess -- and with 0 every one -- is evaluated by the thread that
    found it.  Same records in every case, also with many exact ties (zero-velocity leaves) and under pruning."""
    V, B = np.linspace(0.0, 1.0, 9), np.linspace(-1.0, 1.0, 11)
    solver.set_grid(V, B, L, DT, VMIN)
    sc = C.random_scenarios(12, 77)
    sc[1, 3:5] = sc[1, :2] + [0.0, 1e-3]                        # the optimum stands still: thousands of tied candidates
    solver.set_option("algo", algo)
    try:
        for prune in (0, 1):
            solver.set_option("prune", prune)
            res = []
            for cap in (1 << 20, 5, 0):
                solver.set_option("candidate_list", cap)
                res.append(solver.solve(nat.MODE_FULL, nat.COST_MM, 3, sc[:, :3], sc[:, 3:5], sc[:, :2]))
                assert solver.stats()["refine_candidates"] >= len(sc)
            for r in res[1:]:
                for k in ("index", "cost", "traj", "first_control"):
                    np.testing.assert_array_equal(r[k], res[0][k])
            for i, s_ in enumerate(sc):
                _check(res[0], i, K.solve_full(s_[:3], s_[3:], s_[:2], V, B, 3, C.COST_MM), 3)
    finally:
        solver.set_option("candidate_list", -1)
        solver.set_option("prune", 1)
        solver.set_option("algo", nat.ALGO_AUTO)


def test_node_list_sizes_give_identical_records(solver):
    """option node_list (prefix algorithm): the refinement pass lists the nodes whose bound reaches into the window and a
    second kernel scans each with one warp; with a list that is too small (3 entries: a warp whose nodes do not fit scans
    them itself and leaves its reserved slots empty) and with 0 (every node scanned where it is found) the records, the
    number of refined segments and the number of candidates are the same -- exhaustive and pruned, many exact ties."""
    V, B = np.linspace(0.0, 1.0, 9), np.linspace(-1.0, 1.0, 11)
    solver.set_grid(V, B, L, DT, VMIN)
    sc = C.random_scenarios(12, 78)
    sc[1, 3:5] = sc[1, :2] + [0.0, 1e-3]                        # the optimum stands still: thousands of tied candidates
    solver.set_option("algo", nat.ALGO_PREFIX)
    try:
        for prune in (0, 1):
            solver.set_option("prune", prune)
            res, stats = [], []
            for cap in (1 << 15, 3, 0):
                solver.set_option("node_list", cap)
                res.append(solver.solve(nat.MODE_FULL, nat.COST_MM, 3, sc[:, :3], sc[:, 3:5], sc[:, :2]))
                st = solver.stats()
                stats.append((st["refine_segments"], st["refine_candidates"]))
            assert stats[0] == stats[1] == stats[2] and stats[0][1] >= len(sc), stats
            for r in res[1:]:
                for k in ("index", "cost", "traj", "first_control"):
                    np.testing.assert_array_equal(r[k], res[0][k])
            for i, s_ in enumerate(sc):
                _check(res[0], i, K.solve_full(s_[:3], s_[3:], s_[:2], V, B, 3, C.COST_MM), 3)
    finally:
        solver.set_option("node_list", 1 << 15)
        solver.set_option("prune", 1)
        solver.set_option("algo", nat.ALGO_AUTO)


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_fp32_prefilter_changes_nothing(solver, cost):
    """option prefilter (pruned pass 1: the node bound is first evaluated in fp32 with a margin of 8 error bounds): it may
    only drop nodes the float64 test drops as well, so the records AND the number of pruned nodes are those of
    prefilter=0 -- on the benchmark grid, a 16x16 grid at H=4 (tile path and frontier descent) and a chunked table."""
    cases = [(C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0), 3, 24, 2),
             (np.linspace(0.0, 1.0, 16), np.linspace(-math.radians(60), math.radians(60), 16), 4, 6, 1),
             (np.linspace(0.0, 1.0, 16), np.linspace(-math.radians(60), math.radians(60), 16), 4, 6, 3),
             (np.linspace(0.1, 1.0, 30), np.linspace(-1.0, 1.0, 41), 2, 8, 2)]
    solver.set_option("algo", nat.ALGO_PREFIX)
    solver.set_option("prune", 1)
    try:
        for V, B, H, n, cutmode in cases:
            solver.set_grid(V, B, L, DT, VMIN)
            solver.set_option("subtree_cut", cutmode)
            sc = C.random_scenarios(n, 4100 + H)
            sc[0, 3:5] = sc[0, :2] + [0.05, 0.02]
            res, pruned = [], []
            for pf in (0, 1):
                solver.set_option("prefilter", pf)
                res.append(solver.solve(nat.MODE_FULL, COSTS[cost], H, sc[:, :3], sc[:, 3:5], sc[:, :2]))
                pruned.append(solver.stats()["pruned_units"])
            for k in ("index", "cost", "traj", "first_control"):
                np.testing.assert_array_equal(res[1][k], res[0][k])
            # the upper bound tightens in a timing-dependent order, so the counts may differ by the few nodes that sit
            # between two values of it -- not by the thousands a wrong margin would produce
            assert abs(pruned[1] - pruned[0]) <= 1e-3 * max(pruned[0], 1), (pruned, len(V) * len(B), H)
    finally:
        solver.set_option("prefilter", 1)
        solver.set_option("subtree_cut", 2)
        solver.set_option("algo", nat.ALGO_AUTO)
