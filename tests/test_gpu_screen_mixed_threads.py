"""The two-stage screen (screen=2) where the nodes one thread holds take different paths.

With nodes_per_thread = 2 or 4 a thread holds nodes 1024/NPT apart.  Stage 1 screens every node in the FAR regime,
whatever the thread's other nodes are: in the NEAR regime, unmoved on the line origin (both scored by the scalar
loop), or past the tree's last node.  The records must stay bit-identical to screen=1 and screen=0, and the nodes
stage 1 passes in such threads are counted in stage2_units."""
import math

import numpy as np
import pytest

from oracle import c_oracle as K
from oracle import closed_form as C

pytestmark = pytest.mark.gpu

nat = pytest.importorskip("diplomjourney_b200._native")

COSTS = {C.COST_MM: nat.COST_MM, C.COST_TREE: nat.COST_TREE}
L, DT, VMIN = C.CONFIG["L"], C.CONFIG["delta_t"], C.CONFIG["v_min"]
KEYS = ("index", "cost", "traj", "first_control")


@pytest.fixture(scope="module")
def solver():
    s = nat.Solver(0)
    s.set_option("algo", nat.ALGO_PREFIX)
    s.set_option("prune", 0)
    yield s
    s.close()


def _three_screens(solver, H, sc, cost, npt):
    solver.set_option("nodes_per_thread", npt)
    res, st = {}, {}
    for scr in (0, 1, 2):
        solver.set_option("screen", scr)
        res[scr] = solver.solve(nat.MODE_FULL, COSTS[cost], H, sc[:, :3], sc[:, 3:5], sc[:, :2])
        st[scr] = solver.stats()
    return res, st


def _near_far_scenarios(n, seed):
    """Targets 0.12 to 0.3 from the start.  A step is at most v dt = 0.05 long, so the depth-2 nodes lie within 0.1
    of the start, and a node is NEAR when its target is closer than 4 steps = 0.2: these targets split the nodes of
    every solve into NEAR and FAR ones, and nodes 1024/NPT apart (other speed rows) fall on both sides.  The line
    origin is the start, so the nodes that stand still on the v = 0 row are the unmoved special case."""
    rng = np.random.default_rng(seed)
    x0, y0, p0 = rng.uniform(-5, 5, n), rng.uniform(-5, 5, n), rng.uniform(-math.pi, math.pi, n)
    d = np.linspace(0.12, 0.3, n)
    ang = p0 + rng.uniform(-math.pi, math.pi, n)
    return np.stack([x0, y0, p0, x0 + d * np.cos(ang), y0 + d * np.sin(ang)], axis=1)


@pytest.mark.parametrize("npt", [2, 4])
@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_near_far_and_unmoved_nodes_in_one_thread(solver, cost, npt):
    V, B = np.linspace(0.0, 1.0, 11), np.linspace(-1.0, 1.0, 13)         # S = 143, 20,449 depth-2 nodes
    solver.set_grid(V, B, L, DT, VMIN)
    sc = _near_far_scenarios(8, 4100 + npt)
    try:
        res, st = _three_screens(solver, 3, sc, cost, npt)
        for k in KEYS:
            np.testing.assert_array_equal(res[2][k], res[1][k], err_msg=f"{k} npt={npt}")
            np.testing.assert_array_equal(res[2][k], res[0][k], err_msg=f"{k} npt={npt}")
        for i, s_ in enumerate(sc):
            o = K.solve_full(s_[:3], s_[3:], s_[:2], V, B, 3, cost)
            assert res[2]["index"][i] == o["index"], i
    finally:
        solver.set_option("nodes_per_thread", 4)
        solver.set_option("screen", 2)


@pytest.mark.parametrize("npt", [2, 4])
@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_nodes_next_to_empty_slots_are_screened(solver, cost, npt):
    """A tree of 225 depth-2 nodes (S = 15, H = 3) is smaller than a CTA's thread count (512 with two nodes per thread,
    256 with four), so every thread holds one node and empty slots.  Stage 1 still screens that node.  The optimum of
    each of these solves lies in a FAR node, and that node passes stage 1 (its leaf lies below the upper bound), so
    stage2_units >= robots; a kernel that skipped stage 1 in threads with empty slots would count 0."""
    V, B = np.linspace(0.0, 1.0, 3), np.linspace(-1.0, 1.0, 5)
    solver.set_grid(V, B, L, DT, VMIN)
    sc = C.random_scenarios(16, 4200 + npt)
    try:
        res, st = _three_screens(solver, 3, sc, cost, npt)
        for k in KEYS:
            np.testing.assert_array_equal(res[2][k], res[1][k], err_msg=f"{k} npt={npt}")
            np.testing.assert_array_equal(res[2][k], res[0][k], err_msg=f"{k} npt={npt}")
        assert st[0]["stage2_units"] == 0 and st[1]["stage2_units"] == 0
        assert len(sc) <= st[2]["stage2_units"] <= st[2]["units"] * len(sc)
        for i, s_ in enumerate(sc):
            o = K.solve_full(s_[:3], s_[3:], s_[:2], V, B, 3, cost)
            assert res[2]["index"][i] == o["index"], i
    finally:
        solver.set_option("nodes_per_thread", 4)
        solver.set_option("screen", 2)
