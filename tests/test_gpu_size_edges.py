"""GPU parity at the sizes where the launch plan switches sides.

Every solve goes through make_plan / fill_args / solve_core (csrc/mpcb_api.cu): they pick the algorithm, the width of
the leaf and node indices, the table layouts and how tiles are grouped into segments and batches from the tree's size.
The parity suite (test_gpu_parity.py) mostly runs small grids and small batches, i.e. one side of each switch; this
module runs the other side and compares it with the float64 C oracle and with the GPU's own other configurations.

``_plan`` restates the plan's arithmetic, so that each test first asserts which side of a switch it is on (and that
``solver.stats()`` agrees where the library reports the value); a change of a threshold cannot silently turn a case
into a copy of a small-tree test.

Bars (as in test_gpu_parity.py): leaf index identical to the oracle's, cost rtol 1e-12, trajectory atol 1e-12, first
control exactly equal; two GPU configurations that must agree are compared bit for bit."""
import contextlib
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
TWO32 = 1 << 32

# library constants the plan is made of
K_THREADS = 256            # mpcb_types.cuh:17 (MPCB_THREADS): units per prefix tile, leafwalk's index step
K_LEAF_PER_THREAD = 8      # mpcb_types.cuh:117: a leafwalk tile is 256 * 8 leaves
K_LEAF_CHUNK = 1024        # mpcb_types.cuh:24: pair-table entries staged in shared memory at a time
K_SEG_CAP = 1 << 22        # mpcb_handle.cuh:27: tiles per batch before a segment holds several tiles
K_TILE_BATCH = 1 << 23     # mpcb_handle.cuh:28: tiles per subtree-cut batch
K_WIDE_REDUCE = 1 << 15    # mpcb_handle.cuh:29: segments per solve from which the reduction runs grid-wide

# library defaults of every option this module sets (mpcb_handle.cuh:45-63)
DEFAULTS = dict(algo=nat.ALGO_AUTO, prune=1, screen=1, nodes_per_thread=2, subtree_cut=2, frontier_cap=1 << 22,
                small_path=1)


def _plan(S, H, N, i0_range=None, algo=nat.ALGO_AUTO, mode=nat.MODE_FULL, nb=None, small_path=1):
    """The launch plan of one mpcb_solve_batch_host call, as csrc/mpcb_api.cu computes it.  ``algo`` is the option's
    value; ``nb`` (beta count) is needed for the row table only, ``small_path`` for HELD solves only."""
    p = {}
    if mode == nat.MODE_HELD:                                              # make_plan, mpcb_api.cu:91-95
        prefix, u_begin, u_end, leaves = False, 0, S, S
    else:
        sub = S ** (H - 1)                                                 # :96-98
        lo, hi = (0, S) if i0_range is None else i0_range                  # :99
        if algo == nat.ALGO_AUTO:                                          # :104-106
            algo = nat.ALGO_PREFIX if H >= 2 and sub * N >= 32768 else nat.ALGO_LEAFWALK
        if H < 2:                                                          # :107
            algo = nat.ALGO_LEAFWALK
        prefix = algo == nat.ALGO_PREFIX
        per_i0 = sub // S if prefix else sub                               # :109-116: depth-(H-1) nodes or leaves
        u_begin, u_end = lo * per_i0, hi * per_i0
        leaves = (hi - lo) * sub                                           # :117
    full = mode == nat.MODE_FULL
    p.update(algo=nat.ALGO_PREFIX if prefix else nat.ALGO_LEAFWALK, u_begin=u_begin, u_end=u_end,
             units=u_end - u_begin, leaves_per_solve=leaves)
    # fill_args
    p["idx32"] = not prefix and u_end < TWO32                              # :129
    p["node32"] = prefix and u_end < TWO32 and S ** max(H - 2, 0) < TWO32  # :131-135 (fd32[1].d = S^(H-2))
    p["lw_smem"] = not prefix and full and S <= 4096                       # :146
    digits, r = [], K_THREADS                                              # :140-143: kThreads in base S
    for _ in range(H):
        digits.append(r % S if full else 0)
        r = r // S if full else 0
    digits.reverse()
    p["low_step"] = all(d == 0 for d in digits[:-1])                       # mpcb_kernels.cu:1506-1513 (LOW walk)
    p["kind"] = 2 if not full else (1 if p["idx32"] else 0)                # mpcb_kernels.cu:2017
    p["ht"] = H if H in (2, 3, 4) else 0                                   # mpcb_kernels.cu:1587-1590 (pass 1)
    p["digit_walk"] = not prefix and p["kind"] == 1 and p["ht"] > 0        # mpcb_kernels.cu:1499
    tile_units = K_THREADS if prefix else K_THREADS * K_LEAF_PER_THREAD    # :145
    # solve_core
    tiles = -(-p["units"] // tile_units)                                   # :395
    tps = max(1, -(-(tiles * N) // K_SEG_CAP))                             # :398-400
    segs = -(-tiles // tps) if tiles else 0                                # :403
    p.update(tiles_per_solve=tiles, tps=tps, segs_per_solve=segs, total_segs=segs * N,   # :404
             wide_reduce=segs >= K_WIDE_REDUCE,                            # :525
             tile_batches=-(-(tiles * N) // K_TILE_BATCH))                 # :481,515 (subtree_cut=1, pruned prefix)
    if nb is not None:                                                     # ensure_tables, :205-206
        nv = S // nb
        p["rows_fit"] = 2 * nv * ((nb + 1) // 2) <= K_LEAF_CHUNK
        p["chunks"] = -(-S // K_LEAF_CHUNK)                                # mpcb_kernels.cu:1023 (flat table)
    # host entry: HELD solves of few candidates take the one-launch float64 kernel (:717), small batches zero-copy (:614)
    p["held_small"] = (mode == nat.MODE_HELD and bool(small_path) and S <= 4096 and (nb or 0) <= 4096 and N <= 8192)
    p["zero_copy"] = p["held_small"] and N <= 64
    p["segments"] = 0 if p["held_small"] else p["total_segs"]              # solve_held_small resets the stats (:650)
    return p


def _assert_stats(solver, p):
    st = solver.stats()
    for k in ("algo", "units", "leaves_per_solve", "segments"):
        assert st[k] == p[k], (k, st[k], p[k])
    return st


@pytest.fixture(scope="module")
def solver():
    s = nat.Solver(0)
    yield s
    s.close()


@contextlib.contextmanager
def _options(solver, **opts):
    """Sets ``opts`` for the block; afterwards every option this module touches is back at the library default."""
    try:
        for k, v in opts.items():
            solver.set_option(k, v)
        yield
    finally:
        for k, v in DEFAULTS.items():
            solver.set_option(k, v)


def _check(res, i, ref):
    assert res["index"][i] == ref["index"], (i, res["index"][i], ref["index"], res["cost"][i], ref["cost"])
    assert res["cost"][i] == pytest.approx(ref["cost"], rel=1e-12)
    np.testing.assert_allclose(res["traj"][i], ref["traj"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(res["first_control"][i], ref["first_control"], rtol=0, atol=0)


def _same(a, b, msg=""):
    for k in KEYS:
        np.testing.assert_array_equal(a[k], b[k], err_msg=f"{msg} {k}")


def _mixed(n, seed):
    """A batch that takes every per-solve branch: robots on their line origin (rows 0, 2, 4, 6..) and off it (1, 3),
    next to the target (2), an optimum that stands still (3: the start lies on the line, 1 mm from the target), a
    threshold nothing beats (4) and an entry not to be solved (5).  With a v = 0 grid row, leaves that end in a
    v = 0 step tie exactly with their siblings of that row."""
    sc = C.random_scenarios(n, seed)
    origin = sc[:, :2].copy()
    origin[1] += (3.0, -2.0)                      # the tracked line passes metres from the robot
    sc[2, 3:5] = sc[2, :2] + (0.05, 0.02)         # NEAR regime
    sc[3, 3:5] = sc[3, :2] + (0.0, 1e-3)
    origin[3] = sc[3, :2] - (0.0, 1.0)
    thr = np.full(n, np.inf)
    thr[4] = 1.0
    flags = np.zeros(n, np.uint8)
    flags[5] = nat.FLAG_SKIP
    return dict(sc=sc, origin=origin, thr=thr, flags=flags)


def _solve(solver, mode, cost, H, b, rows=slice(None), i0_range=None):
    return solver.solve(mode, COSTS[cost], H, b["sc"][rows, :3], b["sc"][rows, 3:5], b["origin"][rows],
                        threshold=b["thr"][rows], flags=b["flags"][rows], i0_range=i0_range)


def _check_full(res, b, V, B, H, cost, i0_range=None, rows=None):
    """Every robot of the batch (or ``rows``) against the oracle; skipped entries come back as (NaN, -1)."""
    for i in range(len(b["sc"])) if rows is None else rows:
        if b["flags"][i] & nat.FLAG_SKIP:
            assert res["index"][i] == -1 and math.isnan(res["cost"][i])
            continue
        s = b["sc"][i]
        _check(res, i, K.solve_full(s[:3], s[3:5], b["origin"][i], V, B, H, cost, threshold=b["thr"][i],
                                    i0_range=i0_range))


# ---------------------------------------------------------------------------------------------------------------
# 1. leafwalk FULL trees on wide grids: the digit walk of pass 1 and where its control table lives

B41 = np.array(C.vector_of_beta_angles(0.0))           # the acceleration window's 41 steering angles
LEAFWALK_GRIDS = {
    # name: V, B, H, i0_range, (low_step, lw_smem, kind, ht)
    "S255_H3": (np.linspace(0.0, 1.0, 15), np.linspace(-1.0, 1.0, 17), 3, None, (False, True, 1, 3)),
    "S256_H3": (np.linspace(0.0, 1.0, 16), np.linspace(-1.0, 1.0, 16), 3, None, (False, True, 1, 3)),
    "S451_H3": (np.linspace(0.0, 0.5, 11), B41, 3, None, (True, True, 1, 3)),
    "S4096_H2": (np.linspace(0.0, 1.0, 64), np.linspace(-1.0, 1.0, 64), 2, None, (True, True, 1, 2)),
    "S4160_H2": (np.linspace(0.0, 1.0, 64), np.linspace(-1.0, 1.0, 65), 2, None, (True, False, 1, 2)),
    "S451_H4": (np.linspace(0.0, 0.5, 11), B41, 4, (44, 46), (True, True, 1, 4)),
    "S90_H5": (np.linspace(0.0, 1.0, 9), np.linspace(-1.0, 1.0, 10), 5, (89, 90), (False, True, 0, 0)),
}


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
@pytest.mark.parametrize("name", list(LEAFWALK_GRIDS))
def test_leafwalk_wide_grids_vs_oracle(solver, name, cost):
    """Pass 1 of the leafwalk kernel keeps a leaf's control digits in registers and adds kThreads = 256 per leaf: with
    S < 256 the step has two digits (general carry), S = 256 is "10" in base S, S > 256 steps the last digit only (LOW).
    Its {dphi, s} table sits in shared memory up to S = 4096 and is read from global memory above.  H = 4 runs the
    HT = 4 walk up to leaf 4.2e9; H = 5 the generic HT = 0 loop with 64-bit leaf indices above 5.8e9."""
    V, B, H, rg, (low, smem, kind, ht) = LEAFWALK_GRIDS[name]
    S, n = len(V) * len(B), 7
    p = _plan(S, H, n, rg, nat.ALGO_LEAFWALK)
    assert (p["low_step"], p["lw_smem"], p["kind"], p["ht"]) == (low, smem, kind, ht)
    assert p["digit_walk"] == (kind == 1)
    if name == "S451_H4":
        assert (p["u_begin"], p["u_end"]) == (4_036_289_444, 4_219_757_146) and p["u_end"] < TWO32
    if name == "S90_H5":
        assert p["u_begin"] == 5_839_290_000 and p["leaves_per_solve"] == 65_610_000
    solver.set_grid(V, B, L, DT, VMIN)
    b = _mixed(n, 100 + S + H)
    with _options(solver, algo=nat.ALGO_LEAFWALK):
        res = _solve(solver, nat.MODE_FULL, cost, H, b, i0_range=rg)
        _assert_stats(solver, p)
    _check_full(res, b, V, B, H, cost, rg)


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_default_plan_one_robot_reference_grid_is_leafwalk(solver, cost):
    """ALGO_AUTO sends one robot at H = 2 on the reference's own 201x121 grid (24,321 parents < 32,768) to the leafwalk
    kernel, with its control table in global memory (S > 4096) and the LOW digit walk."""
    Vd, Bd = C.grid_full_default()
    S = len(Vd) * len(Bd)
    p = _plan(S, 2, 1)
    assert p["algo"] == nat.ALGO_LEAFWALK and not p["lw_smem"] and p["digit_walk"] and p["low_step"]
    solver.set_grid(Vd, Bd, L, DT, VMIN)
    if cost == C.COST_MM:
        s, origin = np.array([0.0, 0.0, 0.0, 1.0, 5.0]), np.array([0.0, 0.0])   # config.py: start on the line origin
    else:
        s = C.random_scenarios(1, 61)[0]
        origin = s[:2] + (-2.0, 4.0)
    r = solver.solve(nat.MODE_FULL, COSTS[cost], 2, s[:3], s[3:5], origin)
    st = _assert_stats(solver, p)
    assert st["algo"] == nat.ALGO_LEAFWALK
    _check(r, 0, K.solve_full(s[:3], s[3:5], origin, Vd, Bd, 2, cost))        # 5.9e8 leaves


def test_bench_leafwalk_workload_vs_oracle(solver):
    """The bench's leafwalk leg (11x41 acceleration window, H = 3, MM cost, its first 64 robots), which reports only
    a rate and an index checksum, against the oracle."""
    V, B = C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0)
    S, n = len(V) * len(B), 64
    p = _plan(S, 3, n, None, nat.ALGO_LEAFWALK)
    assert S == 451 and p["digit_walk"] and p["low_step"] and p["lw_smem"]
    sc = C.random_scenarios(1024, 0)[:n]                                       # bench.py: workload "cfg2", seed 0
    solver.set_grid(V, B, L, DT, VMIN)
    with _options(solver, algo=nat.ALGO_LEAFWALK, prune=0):
        res = solver.solve(nat.MODE_FULL, nat.COST_MM, 3, sc[:, :3], sc[:, 3:5], sc[:, :2])
        _assert_stats(solver, p)
    for i, s in enumerate(sc):                                                 # 64 x 9.2e7 = 5.9e9 leaves
        _check(res, i, K.solve_full(s[:3], s[3:5], s[:2], V, B, 3, C.COST_MM))


# ---------------------------------------------------------------------------------------------------------------
# 2-4. 64-bit leaf and node indices, with an exact tie across 2^32

V260 = np.linspace(1.0, 0.0, 13)          # descending: v = 0 is row iv = 12, i.e. controls 240 .. 259
B260 = np.linspace(-1.0, 1.0, 20)
S260 = 260
TIE_NODE = TWO32 // S260                  # 16,519,104: controls (244, 95, 4)


def _tie_batch(n, seed, D):
    """_mixed batch whose row 0 is the designed tie: start (0, 0) on its line origin, target = the float64 pose of
    node TIE_NODE at depth D (the oracle's own tables and steps).  COST_TREE is >= 0 and 0 on the target (on the line
    too), and a v = 0 step neither moves nor turns: every v = 0 descendant of that node costs exactly what the node
    does, and the first minimum is its lowest one."""
    vv, _, dphi = C.control_tables(V260, B260, L, DT)
    start = np.array([0.0, 0.0, 0.3])
    assert C.leaf_controls(TIE_NODE, S260, D)[-3:] == [244, 95, 4]
    pose = C.rollout(start, C.leaf_controls(TIE_NODE, S260, D), vv, dphi, DT)[-1]
    b = _mixed(n, seed)
    b["sc"][0] = (*start, pose[0], pose[1])
    b["origin"][0] = start[:2]
    return b


@pytest.mark.parametrize("i0_range", [(244, 245), (259, 260)])
def test_leafwalk_64bit_leaf_indices_across_2_32(solver, i0_range):
    """S = 260, H = 4: first control 244 holds leaves 4,288,544,000 .. 4,306,119,999, across 2^32; 259 lies wholly
    above.  The leafwalk kernel takes its 64-bit index path (KIND 0), the prefix kernel's node indices still fit
    32 bits; both against the oracle and against each other."""
    H, n = 4, 7
    pl = _plan(S260, H, n, i0_range, nat.ALGO_LEAFWALK)
    pp = _plan(S260, H, n, i0_range, nat.ALGO_PREFIX)
    assert pl["kind"] == 0 and not pl["idx32"] and pl["leaves_per_solve"] == 17_576_000
    if i0_range == (244, 245):
        assert (pl["u_begin"], pl["u_end"]) == (4_288_544_000, 4_306_120_000) and pl["u_begin"] < TWO32 < pl["u_end"]
    else:
        assert pl["u_begin"] == 4_552_184_000 > TWO32
    assert pp["node32"] and pp["u_end"] < TWO32
    b = _tie_batch(n, 4000 + i0_range[0], 3)
    refs = {i: K.solve_full(b["sc"][i, :3], b["sc"][i, 3:5], b["origin"][i], V260, B260, H, C.COST_TREE,
                            threshold=b["thr"][i], i0_range=i0_range) for i in range(n) if i != 5}
    if i0_range == (244, 245):             # precondition: the tie is the lowest of the v = 0 leaves 4,294,967,280 .. 299
        assert refs[0]["index"] == TIE_NODE * S260 + 240 == 4_294_967_280 and refs[0]["cost"] < 1e-9
    solver.set_grid(V260, B260, L, DT, VMIN)
    out = {}
    for algo, p in ((nat.ALGO_LEAFWALK, pl), (nat.ALGO_PREFIX, pp)):
        with _options(solver, algo=algo):
            out[algo] = _solve(solver, nat.MODE_FULL, C.COST_TREE, H, b, i0_range=i0_range)
            _assert_stats(solver, p)
        for i, ref in refs.items():
            _check(out[algo], i, ref)
        assert out[algo]["index"][5] == -1 and math.isnan(out[algo]["cost"][5])
    _same(out[nat.ALGO_LEAFWALK], out[nat.ALGO_PREFIX], "leafwalk vs prefix")


def test_prefix_64bit_node_decode_across_2_32(solver):
    """S = 260, H = 5, first control 244: depth-4 node indices 4,288,544,000 .. 4,306,119,999 straddle 2^32, so the
    prefix kernels decode nodes with 64-bit dividers (node32 = 0).  Exhaustive (screened or not, 1/2/4 nodes per
    thread), pruned (no subtree cut, tile cut, frontier descent, frontier overflow into the tile walk) and the
    leafwalk kernel (64-bit leaves) must agree bit for bit; the designed tie's v = 0 leaves hang below depth-4 nodes
    4,294,967,280 .. 299 on both sides of 2^32."""
    H, n, rg = 5, 6, (244, 245)
    p = _plan(S260, H, n, rg, nat.ALGO_PREFIX)
    assert not p["node32"] and (p["u_begin"], p["u_end"]) == (4_288_544_000, 4_306_120_000)
    assert p["u_begin"] < TIE_NODE * S260 + 240 < TWO32 < TIE_NODE * S260 + 259 < p["u_end"]
    assert p["leaves_per_solve"] == 4_569_760_000
    pl = _plan(S260, H, n, rg, nat.ALGO_LEAFWALK)
    assert pl["kind"] == 0 and pl["ht"] == 0
    b = _tie_batch(n, 4500, 3)
    solver.set_grid(V260, B260, L, DT, VMIN)
    runs = {}
    with _options(solver, algo=nat.ALGO_PREFIX, prune=0):
        for screen in (0, 1):
            for npt in (1, 2, 4):
                solver.set_option("screen", screen)
                solver.set_option("nodes_per_thread", npt)
                runs[("exhaustive", screen, npt)] = _solve(solver, nat.MODE_FULL, C.COST_TREE, H, b, i0_range=rg)
                _assert_stats(solver, p)
        solver.set_option("prune", 1)
        for cut, cap in ((0, 1 << 22), (1, 1 << 22), (3, 1 << 22), (3, 48)):    # cap 48: the frontier overflows
            solver.set_option("subtree_cut", cut)
            solver.set_option("frontier_cap", cap)
            runs[("pruned", cut, cap)] = _solve(solver, nat.MODE_FULL, C.COST_TREE, H, b, i0_range=rg)
            _assert_stats(solver, p)
    with _options(solver, algo=nat.ALGO_LEAFWALK):
        runs["leafwalk"] = _solve(solver, nat.MODE_FULL, C.COST_TREE, H, b, i0_range=rg)
        _assert_stats(solver, pl)
    ref_run = runs[("exhaustive", 0, 1)]
    for key, r in runs.items():
        _same(r, ref_run, str(key))
    # 4,569,760,000 leaves (the designed tie only)
    o = K.solve_full(b["sc"][0, :3], b["sc"][0, 3:5], b["origin"][0], V260, B260, H, C.COST_TREE, i0_range=rg)
    assert o["index"] == (TIE_NODE * S260 + 240) * S260 + 240 == 1_116_691_493_040 and o["cost"] < 1e-9
    _check(ref_run, 0, o)


# ---------------------------------------------------------------------------------------------------------------
# 5-6. segments of several tiles, several tile-cut batches

def test_segments_of_several_tiles(solver):
    """Prefix, S = 255, H = 4, 65 robots: 64,771 tiles per solve (odd) and 4.2e6 tiles in the batch, so a segment is two
    tiles (the last one of every solve one) and the per-solve reduction runs one CTA per solve; solved one at a time,
    a solve is 64,771 one-tile segments reduced grid-wide.  Leafwalk on the same grid with 3 robots: 6.2e6 tiles, two
    per segment.  All bit-identical, pruned too, and equal to the oracle."""
    V, B, H, n = np.linspace(0.0, 1.0, 15), np.linspace(-1.0, 1.0, 17), 4, 65
    S = 255
    p = _plan(S, H, n, None, nat.ALGO_PREFIX)
    assert (p["tiles_per_solve"], p["tps"], p["segs_per_solve"]) == (64_771, 2, 32_386) and not p["wide_reduce"]
    p1 = _plan(S, H, 1, None, nat.ALGO_PREFIX)
    assert (p1["tps"], p1["segs_per_solve"]) == (1, 64_771) and p1["wide_reduce"]
    pl = _plan(S, H, 3, None, nat.ALGO_LEAFWALK)
    assert (pl["tiles_per_solve"], pl["tps"]) == (2_064_576, 2) and pl["digit_walk"]
    b = _mixed(n, 5000)
    solver.set_grid(V, B, L, DT, VMIN)
    with _options(solver, algo=nat.ALGO_PREFIX, prune=0):
        batch = _solve(solver, nat.MODE_FULL, C.COST_MM, H, b)
        _assert_stats(solver, p)
        singles = [_solve(solver, nat.MODE_FULL, C.COST_MM, H, b, rows=slice(i, i + 1)) for i in range(n)]
        _assert_stats(solver, p1)
        solver.set_option("prune", 1)
        pruned = _solve(solver, nat.MODE_FULL, C.COST_MM, H, b)
    for k in KEYS:
        np.testing.assert_array_equal(np.concatenate([r[k] for r in singles]), batch[k], err_msg=k)
    _same(pruned, batch, "pruned")
    with _options(solver, algo=nat.ALGO_LEAFWALK):
        lw = _solve(solver, nat.MODE_FULL, C.COST_MM, H, b, rows=slice(0, 3))
        _assert_stats(solver, pl)
    for k in KEYS:
        np.testing.assert_array_equal(lw[k], batch[k][:3], err_msg=f"leafwalk {k}")
    _check_full(batch, b, V, B, H, C.COST_MM, rows=(0, 1))                       # 2 x 4.2e9 = 8.5e9 leaves


def test_several_tile_cut_batches(solver):
    """Pruned prefix with the per-tile subtree cut, 16x16 grid (+-60 deg), H = 4, 160 robots: 10,485,760 tiles, i.e. two
    batches of the tile test (the second one partial) and three tiles per segment; bit-identical to the exhaustive
    solve of all 6.9e11 leaves."""
    V, B, H, n = np.linspace(0.0, 1.0, 16), np.linspace(-math.radians(60), math.radians(60), 16), 4, 160
    p = _plan(256, H, n, None, nat.ALGO_PREFIX)
    assert p["tiles_per_solve"] * n == 10_485_760 and p["tile_batches"] == 2 and p["tps"] == 3
    assert K_TILE_BATCH < p["tiles_per_solve"] * n < 2 * K_TILE_BATCH
    b = _mixed(n, 6000)
    solver.set_grid(V, B, L, DT, VMIN)
    with _options(solver, algo=nat.ALGO_PREFIX, prune=1, subtree_cut=1):
        cut = _solve(solver, nat.MODE_FULL, C.COST_MM, H, b)
        st = _assert_stats(solver, p)
        assert st["pruned_units"] > 0
        solver.set_option("prune", 0)
        full = _solve(solver, nat.MODE_FULL, C.COST_MM, H, b)
        _assert_stats(solver, p)
    _same(cut, full, "subtree_cut=1 vs exhaustive")


# ---------------------------------------------------------------------------------------------------------------
# 7. pair-table layouts around S = 1024

@pytest.mark.parametrize("nv,nb,rows_fit,chunks", [(31, 33, False, 1), (32, 32, True, 1), (25, 41, False, 2)])
def test_pair_table_layouts_near_1024(solver, nv, nb, rows_fit, chunks):
    """The prefix pass 1 reads the per-control pair table by speed row when it fits one shared-memory chunk, else
    flat, in chunks of 1024 controls.  31x33 (S = 1023): no rows, one chunk; 32x32: rows fit exactly; 25x41
    (S = 1025): two chunks, the second of one control.  Exhaustive (screened or not) and pruned, H = 3 on three
    first controls."""
    V, B, H, n = np.linspace(0.0, 1.0, nv), np.linspace(-1.0, 1.0, nb), 3, 7
    S = nv * nb
    rg = (S // 2, S // 2 + 3)
    p = _plan(S, H, n, rg, nat.ALGO_PREFIX, nb=nb)
    assert (p["rows_fit"], p["chunks"]) == (rows_fit, chunks)
    b = _mixed(n, 7000 + S)
    solver.set_grid(V, B, L, DT, VMIN)
    runs = []
    with _options(solver, algo=nat.ALGO_PREFIX, prune=0):
        for screen in (0, 1):
            solver.set_option("screen", screen)
            runs.append(_solve(solver, nat.MODE_FULL, C.COST_MM, H, b, i0_range=rg))
            _assert_stats(solver, p)
        solver.set_option("prune", 1)
        runs.append(_solve(solver, nat.MODE_FULL, C.COST_MM, H, b, i0_range=rg))
        _assert_stats(solver, p)
    for r in runs[1:]:
        _same(r, runs[0], f"S={S}")
    _check_full(runs[0], b, V, B, H, C.COST_MM, rg)


# ---------------------------------------------------------------------------------------------------------------
# 8. HELD solves beyond H = 3 and across the limits of the one-launch path

def _held_batch(n, seed):
    b = _mixed(n, seed)
    b["flags"][6::3] |= nat.FLAG_SLOW                                          # the online controller's slow-down
    return b


def _check_held(res, b, V, B, H, cost, rows, cache=None):
    for i in rows:
        if b["flags"][i] & nat.FLAG_SKIP:
            assert res["index"][i] == -1 and math.isnan(res["cost"][i])
            continue
        s = b["sc"][i]
        key = (i, len(B), H, cost)
        ref = cache.get(key) if cache is not None else None
        if ref is None:
            ref = K.solve_held(s[:3], s[3:5], b["origin"][i], V, B, H, cost, threshold=b["thr"][i],
                               slow=bool(b["flags"][i] & nat.FLAG_SLOW))
            if cache is not None:
                cache[key] = ref
        _check(res, i, ref)


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
@pytest.mark.parametrize("H", [1, 2, 5, 8])
def test_held_horizons_and_path_limits(solver, H, cost):
    """HELD at H = 1, 2, 5, 8 with and without the slow-down flag, on the one-launch float64 path and on the general
    pipeline: 64x64 (S = 4096, the one-launch path may take it) and 64x65 (S = 4160, the general pipeline even with
    small_path = 1), 64 robots (zero-copy) and 65 (staged copies)."""
    cache = {}
    for nb in (64, 65):
        V, B = np.linspace(0.0, 1.0, 64), np.linspace(-1.0, 1.0, nb)
        S = 64 * nb
        solver.set_grid(V, B, L, DT, VMIN)
        b = _held_batch(65, 8000 + H)
        for small_path in (1, 0):
            per_n = {}
            for n in (64, 65):
                p = _plan(S, H, n, mode=nat.MODE_HELD, nb=nb, small_path=small_path)
                assert p["held_small"] == (small_path == 1 and S == 4096)
                assert p["zero_copy"] == (p["held_small"] and n == 64)
                with _options(solver, small_path=small_path):
                    per_n[n] = _solve(solver, nat.MODE_HELD, cost, H, b, rows=slice(0, n))
                    st = _assert_stats(solver, p)
                assert (st["kernel_launches"] == 1) == p["held_small"]
                _check_held(per_n[n], b, V, B, H, cost, range(n), cache)
            for k in KEYS:
                np.testing.assert_array_equal(per_n[64][k], per_n[65][k][:64], err_msg=f"S={S} small={small_path} {k}")


def test_held_batch_past_the_one_launch_limit(solver):
    """8,193 HELD solves in one call exceed the one-launch path's 8,192 and run the general pipeline: bit-identical to
    the same robots in batches of 4,096 on that pipeline, equal to the one-launch path's batches of 4,096 (whose
    tan(beta) is the device's), and to the oracle on every 256th robot."""
    V, B, H, n = [0.0, 0.3, 0.6, 1.0], np.linspace(-1.0, 1.0, 7), 3, 8193
    S = 28
    p = _plan(S, H, n, mode=nat.MODE_HELD, nb=len(B))
    assert not p["held_small"] and p["segments"] == n
    assert _plan(S, H, 4096, mode=nat.MODE_HELD, nb=len(B))["held_small"]
    b = _held_batch(n, 9000)
    solver.set_grid(V, B, L, DT, VMIN)
    for cost in (C.COST_MM, C.COST_TREE):
        whole = _solve(solver, nat.MODE_HELD, cost, H, b)
        _assert_stats(solver, p)
        parts = {}
        for small_path in (0, 1):
            with _options(solver, small_path=small_path):
                rs = [_solve(solver, nat.MODE_HELD, cost, H, b, rows=slice(k, min(k + 4096, n))) for k in range(0, n, 4096)]
                assert (solver.stats()["kernel_launches"] == 1) == bool(small_path)   # the last part is one robot
            parts[small_path] = {k: np.concatenate([r[k] for r in rs]) for k in KEYS}
        _same(parts[0], whole, f"{cost} batches of 4096, general pipeline")
        np.testing.assert_array_equal(parts[1]["index"], whole["index"])
        np.testing.assert_array_equal(parts[1]["first_control"], whole["first_control"])
        np.testing.assert_allclose(parts[1]["cost"], whole["cost"], rtol=1e-12, atol=0)
        np.testing.assert_allclose(parts[1]["traj"], whole["traj"], rtol=0, atol=1e-12)
        _check_held(whole, b, V, B, H, cost, range(0, n, 256))
