"""The pair table of stage 1 of the two-stage screen travels with each launch of the exhaustive pass 1 as a kernel
parameter (RowPairs, csrc/mpcb_types.cuh; DESIGN.md section 3.5).  Its capacity is that of the row table, 512 pairs:
a grid whose row table fits runs stage 1, one that does not runs the flat one-stage screen; both must return the
records of screen=0.  Because the table is passed by value, two handles holding different grids on one device may
solve at the same time."""
import numpy as np
import pytest

from oracle import closed_form as C

pytestmark = pytest.mark.gpu

nat = pytest.importorskip("diplomjourney_b200._native")

L, DT, VMIN = C.CONFIG["L"], C.CONFIG["delta_t"], C.CONFIG["v_min"]
KEYS = ("index", "cost", "traj", "first_control")
K_ROW_PAIR_CAP = 512                                    # kRowPairCap = kLeafChunk / 2


def _solver(grid):
    s = nat.Solver(0)
    s.set_option("algo", nat.ALGO_PREFIX)
    s.set_option("prune", 0)
    s.set_grid(*grid, L, DT, VMIN)
    return s


def _grid(nv, nb):
    return np.linspace(0.0, 1.0, nv), np.linspace(-1.0, 1.0, nb)


@pytest.mark.parametrize("nv,nb,stage1", [(32, 32, True), (16, 63, True), (31, 33, False), (33, 31, False)])
def test_table_capacity_edges(nv, nb, stage1):
    """32 x 32 and 16 x 63 fill the 512 pairs exactly (stage 1 runs: the node of each optimum passes it, so some
    node does); 31 x 33 and 33 x 31 need 527 and 528 pairs (no row table, the flat screen: stage 1 never runs)."""
    assert (nv * ((nb + 1) // 2) <= K_ROW_PAIR_CAP) == stage1
    s = _solver(_grid(nv, nb))
    try:
        sc = C.random_scenarios(6, 4100 + nv * nb)
        S = nv * nb
        res = {}
        for scr in (0, 2):
            s.set_option("screen", scr)
            res[scr] = s.solve(nat.MODE_FULL, nat.COST_MM, 3, sc[:, :3], sc[:, 3:5], sc[:, :2], i0_range=(S // 2, S // 2 + 4))
            st = s.stats()
        for k in KEYS:
            np.testing.assert_array_equal(res[2][k], res[0][k], err_msg=k)
        assert (st["stage2_units"] > 0) == stage1, st["stage2_units"]
    finally:
        s.close()


def test_two_handles_with_different_grids_interleaved():
    """Two handles on one device, each with its own grid (the bench's 11 x 41 window and a 16 x 31 grid), solving on
    their own streams in alternation without synchronising in between: every record equals that of a solve on a
    fresh handle that holds only its grid."""
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available()
    grids = [(C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0)), _grid(16, 31)]
    H, n, rounds = 3, 64, 3
    scen = [C.random_scenarios(n, 5200 + 31 * r) for r in range(rounds)]
    ref = []
    for g in grids:
        s = _solver(g)
        try:
            ref.append([s.solve(nat.MODE_FULL, nat.COST_MM, H, sc[:, :3], sc[:, 3:5], sc[:, :2]) for sc in scen])
        finally:
            s.close()
    solvers = [_solver(g) for g in grids]
    try:
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.float64)).cuda()
        ins = [(dev(sc[:, :3]), dev(sc[:, 3:5]), dev(sc[:, :2])) for sc in scen]
        torch.cuda.synchronize()
        outs = {}
        for r in range(rounds):
            for h, s in enumerate(solvers):
                o = dict(cost=torch.empty(n, dtype=torch.float64, device="cuda"),
                         index=torch.empty(n, dtype=torch.int64, device="cuda"),
                         traj=torch.empty((n, H, 3), dtype=torch.float64, device="cuda"),
                         first_control=torch.empty((n, 2), dtype=torch.float64, device="cuda"))
                st, tg, og = ins[r]
                s.solve_device(nat.MODE_FULL, nat.COST_MM, H, n, st.data_ptr(), tg.data_ptr(), og.data_ptr(), 0, 0,
                               o["cost"].data_ptr(), o["index"].data_ptr(), o["traj"].data_ptr(),
                               o["first_control"].data_ptr())
                outs[h, r] = o
        for s in solvers:
            s.sync()
        for (h, r), o in outs.items():
            for k in KEYS:
                np.testing.assert_array_equal(o[k].cpu().numpy(), ref[h][r][k], err_msg=f"handle {h} round {r} {k}")
    finally:
        for s in solvers:
            s.close()
