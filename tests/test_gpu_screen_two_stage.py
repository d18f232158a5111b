"""The two-stage screen of the exhaustive prefix pass 1 (option screen=2, the default; DESIGN.md section 3.5).

Stage 1 forms only every leaf's distance and bounds the line and heading terms per node (csrc/mpcb_screen.cuh); only
the nodes it passes go through the one-stage screen (screen=1).  Its bound is sound, so the records must be
bit-identical to screen=1 and to screen=0 (a MUFU.SQRT per leaf, no bound at all): index, cost, trajectory and first
control, for both costs and 1, 2 and 4 nodes per thread, on the scenario sets of the screened and branch-and-bound parity
tests, on the pair-table layouts around S = 1024 and on exact ties."""
import numpy as np
import pytest

from oracle import c_oracle as K
from oracle import closed_form as C

pytestmark = pytest.mark.gpu

nat = pytest.importorskip("diplomjourney_b200._native")

COSTS = {C.COST_MM: nat.COST_MM, C.COST_TREE: nat.COST_TREE}
L, DT, VMIN = C.CONFIG["L"], C.CONFIG["delta_t"], C.CONFIG["v_min"]
KEYS = ("index", "cost", "traj", "first_control")

# (V, B, H, robots, first-control range)
SCREENED_SET = [(np.linspace(0.0, 1.0, 11), np.linspace(-1.0, 1.0, 13), 3, 8, None),
                (C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0), 3, 6, None),
                (C.vector_of_velocities(0.01), C.vector_of_beta_angles(0.9), 3, 4, None),      # clipped window, v = 0 rows
                (np.linspace(0.1, 1.0, 30), np.linspace(-1.0, 1.0, 41), 2, 5, None),          # S = 1230: two chunks, flat loop
                (np.linspace(0.0, 1.0, 6), np.linspace(-1.0, 1.0, 7), 4, 4, None)]
BNB_SET = [(np.linspace(0.0, 1.0, 16), np.linspace(-np.radians(60), np.radians(60), 16), 3, 8, None),
           (np.linspace(0.0, 1.0, 3), np.linspace(-1.0, 1.0, 4), 5, 6, None),
           (np.linspace(0.0, 1.0, 30), np.linspace(-1.0, 1.0, 50), 3, 2, (1480, 1500))]
# around S = 1024: 31 x 33 (no row table, one chunk), 32 x 32 (the row table fills the chunk exactly), 16 x 63 (row
# table, odd rows padded), 25 x 41 (two chunks)
EDGE_SET = [(np.linspace(0.0, 1.0, nv), np.linspace(-1.0, 1.0, nb), 3, 7, None)
            for nv, nb in ((31, 33), (32, 32), (16, 63), (25, 41))]


@pytest.fixture(scope="module")
def solver():
    s = nat.Solver(0)
    s.set_option("algo", nat.ALGO_PREFIX)
    s.set_option("prune", 0)
    yield s
    s.close()


def _scenarios(n, seed, S):
    sc = C.random_scenarios(n, seed)
    sc[0, 3:5] = sc[0, :2] + [0.05, 0.02]                       # next to its target (NEAR)
    if n > 1:
        sc[1, 3:5] = sc[1, :2] + [0.0, 1e-3]                    # the optimum stands still: exact ties
    thr = np.full(n, np.inf)
    if n > 2:
        thr[2] = 1.0                                            # nothing beats this one
    return sc, thr


def _rows_fit(V, B):
    return 2 * len(V) * ((len(B) + 1) // 2) <= 1024


def _three_screens(solver, V, B, H, sc, thr, cost, i0):
    res, st = {}, {}
    for scr in (0, 1, 2):
        solver.set_option("screen", scr)
        res[scr] = solver.solve(nat.MODE_FULL, COSTS[cost], H, sc[:, :3], sc[:, 3:5], sc[:, :2], threshold=thr, i0_range=i0)
        st[scr] = solver.stats()
    return res, st


@pytest.mark.parametrize("npt", [1, 2, 4])
@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
@pytest.mark.parametrize("which", ["screened", "bnb", "edges"])
def test_two_stage_screen_is_bit_identical(solver, which, cost, npt):
    grids = {"screened": SCREENED_SET, "bnb": BNB_SET, "edges": EDGE_SET}[which]
    solver.set_option("nodes_per_thread", npt)
    try:
        for gi, (V, B, H, n, i0) in enumerate(grids):
            solver.set_grid(V, B, L, DT, VMIN)
            S = len(V) * len(B)
            sc, thr = _scenarios(n, 1300 + 17 * gi + H + S, S)
            ranges = [i0] if i0 is not None else [None, (0, max(1, S // 3)), (S // 2, S // 2 + 1)]
            for rg in ranges:
                res, st = _three_screens(solver, V, B, H, sc, thr, cost, rg)
                for k in KEYS:
                    np.testing.assert_array_equal(res[2][k], res[1][k], err_msg=f"{k} S={S} H={H} range={rg} npt={npt}")
                    np.testing.assert_array_equal(res[2][k], res[0][k], err_msg=f"{k} S={S} H={H} range={rg} npt={npt}")
                assert st[0]["stage2_units"] == 0 and st[1]["stage2_units"] == 0
                assert 0 <= st[2]["stage2_units"] <= st[2]["units"] * n
                if npt == 1 or not _rows_fit(V, B):
                    assert st[2]["stage2_units"] == 0                  # stage 1 only runs on the row table, NPT >= 2
                if which == "screened" and rg is None and S ** H <= 3e7:
                    for i, s_ in enumerate(sc):
                        o = K.solve_full(s_[:3], s_[3:], s_[:2], V, B, H, cost, threshold=thr[i])
                        assert res[2]["index"][i] == o["index"], (S, H, i)
    finally:
        solver.set_option("nodes_per_thread", 2)
        solver.set_option("screen", 2)


def test_two_stage_screen_on_exact_ties(solver):
    """Designed exact ties: a zero-speed grid row, a robot whose start is its line origin, and v = 0 at the last step
    only (a 5-way tie below one parent): the first minimum must come back under every screen."""
    B = np.linspace(-1, 1, 5)
    cases = [([0.0, 0.5, 1.0], B, [1.0, 2.0, 0.3], (3.0, 4.0), (0.0, 0.0)),
             ([0.0, 0.5, 1.0], B, [1.0, 2.0, 0.3], (3.0, 4.0), (1.0, 2.0)),
             ([0.0, 1.0], B, [0.0, 0.0, 0.0], (0.1, 0.0), (-1.0, 0.0))]
    try:
        for V, B_, s, tgt, org in cases:
            solver.set_grid(V, B_, L, DT, VMIN)
            for cost in (C.COST_MM, C.COST_TREE):
                ref = K.solve_full(s, tgt, org, V, B_, 3, cost)
                st = np.tile(np.asarray(s, float), (64, 1))                 # 64 copies: whole warps of tied nodes
                res = {}
                for scr in (0, 1, 2):
                    solver.set_option("screen", scr)
                    res[scr] = solver.solve(nat.MODE_FULL, COSTS[cost], 3, st, np.tile(tgt, (64, 1)), np.tile(org, (64, 1)))
                for k in KEYS:
                    np.testing.assert_array_equal(res[2][k], res[0][k])
                    np.testing.assert_array_equal(res[2][k], res[1][k])
                assert np.all(res[2]["index"] == ref["index"])
    finally:
        solver.set_option("screen", 2)


def test_two_stage_screen_on_the_bench_workload(solver):
    """The cfg2 bench workload (11 x 41 acceleration window, H = 3, MM cost), 256 robots of its default_rng(0) batch:
    identical records under the three screens, and stage 1 passes only a small share of the nodes."""
    V, B = C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0)
    solver.set_grid(V, B, L, DT, VMIN)
    sc = C.random_scenarios(1024, 0)[::4]
    n = len(sc)
    thr = np.full(n, np.inf)
    try:
        res, st = _three_screens(solver, V, B, 3, sc, thr, C.COST_MM, None)
        for k in KEYS:
            np.testing.assert_array_equal(res[2][k], res[0][k])
            np.testing.assert_array_equal(res[2][k], res[1][k])
        frac = st[2]["stage2_units"] / (st[2]["units"] * n)
        print(f"stage 1 passed {st[2]['stage2_units']} of {st[2]['units'] * n} nodes ({100 * frac:.4f} %)")
        assert 0 < st[2]["stage2_units"] and frac < 0.05
    finally:
        solver.set_option("screen", 2)
