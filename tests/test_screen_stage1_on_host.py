"""Stage 1 of the two-stage screen (option screen=2, DESIGN.md section 3.5), checked on the CPU.

csrc/mpcb_screen.cuh -- the header the kernel includes -- is compiled for the host with g++ next to a replay of the
fp32 arithmetic of the screen loop.  For every depth-(H-1) node of small trees (several grids, both costs, so the heading
term on and off, robots on and off their line origin) and a range of screen bounds cn, including for each node the
smallest cn at which the screen flags it:
  * the bound's q, gg and t ranges hold the q, gg and t of every leaf of the node;
  * no node whose stage-2 maximum of fma(t, t, -dd) is positive -- a real hit or a false one -- is rejected by stage 1.
The bound has no slack to spare, and the test shows it: with T one ulp lower, or the heading interval one ulp
narrower, it fails."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import closed_form as C

L, DT = C.CONFIG["L"], C.CONFIG["delta_t"]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32

GRIDS = [(np.linspace(0.0, 1.0, 6), np.linspace(-1.0, 1.0, 7), 3),
         (np.linspace(0.1, 1.0, 4), np.linspace(-1.0, 1.0, 9), 3),
         (C.vector_of_velocities(0.5), C.vector_of_beta_angles(0.0), 2),                  # the bench's 11 x 41 window
         (np.linspace(-0.5, 1.0, 5), np.linspace(-np.radians(60), np.radians(60), 8), 3)]  # reversing speeds


@pytest.fixture(scope="module")
def lib():
    src = os.path.join(ROOT, "tests", "native", "screen_host.cpp")
    out_dir = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "screen_host.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-std=c++17", "-I", os.path.join(ROOT, "diplomjourney_b200", "csrc"),
                           src, "-o", so])
    lib = ctypes.CDLL(so)
    fp = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
    lib.mpcb_test_screen.argtypes = [ctypes.c_int, fp, fp, ctypes.c_int, ctypes.c_longlong, fp, fp, ctypes.c_int, fp]
    lib.mpcb_test_knife_edge_cn.argtypes = [ctypes.c_int, fp, ctypes.c_int, ctypes.c_longlong, fp, fp]
    return lib


def _table(V, B):
    """GridTables::leaf32 as the library builds it: {a, b, r, g} per control, rounded to fp32."""
    vv, _, dphi = C.control_tables(V, B, L, DT)
    s = vv * DT
    return np.ascontiguousarray(np.stack([s * np.cos(dphi), s * np.sin(dphi), s * s, 3.16227766016837952 * dphi], 1).astype(F32))


def _box(tab):
    return np.ascontiguousarray([tab[:, 0].min(), tab[:, 0].max(), tab[:, 1].min(), tab[:, 1].max(),
                                 tab[:, 3].min(), tab[:, 3].max()], F32)


def _node_regs(V, B, H, x, cost):
    """fp32 direct-form registers (u2s, w2s, D2s, nu, nw, eh, nhh) of every depth-(H-1) node, as node_regs forms them from
    the float64 node frame.  The line origin is x[5:7]."""
    vv, _, dphi = C.control_tables(V, B, L, DT)
    S, s = len(vv), vv * DT
    xs, ys, p0, xt, yt, ox, oy = x
    wl, wh = (10.0, math.sqrt(10.0)) if cost == C.COST_MM else (100.0, 0.0)
    X, Y, P = np.array([xs]), np.array([ys]), np.array([p0])
    for _ in range(H - 1):
        P = (P[:, None] + dphi[None, :]).ravel()
        X = np.repeat(X, S) + np.tile(s, len(X)) * np.cos(P)
        Y = np.repeat(Y, S) + np.tile(s, len(Y)) * np.sin(P)
    cp, sp = np.cos(P), np.sin(P)
    relx, rely = xt - X, yt - Y
    u, w = cp * relx + sp * rely, cp * rely - sp * relx
    A, Bc, Cc = yt - oy, xt - ox, xt * oy - yt * ox
    norm = math.hypot(A, Bc)
    ep = wl * (A * X - Bc * Y + Cc) / norm
    gx, gy = wl * A / norm, -wl * Bc / norm
    hp = wh * (C.heading_reference(xt, yt) - P)
    kWd = 1e4
    regs = np.stack([(-2.0 * kWd * kWd * u).astype(F32), (-2.0 * kWd * kWd * w).astype(F32),
                     (kWd * kWd * (u * u + w * w)).astype(F32), (cp * gx + sp * gy).astype(F32), (cp * gy - sp * gx).astype(F32),
                     ep.astype(F32), -(hp.astype(F32))], 1)
    return np.ascontiguousarray(regs, F32)


def _scenarios(n, seed):
    """start (x, y, phi), target, line origin: the first half start on their line origin, the rest elsewhere"""
    sc = C.random_scenarios(n, seed)
    rng = np.random.default_rng(seed)
    origin = sc[:, :2].copy()
    origin[n // 2:] += rng.uniform(-2.0, 2.0, (n - n // 2, 2))
    return np.concatenate([sc, origin], 1)


def _run(lib, tab, box, head, regs, cn, tshrink=0):
    out = np.zeros((len(regs), 16), F32)
    lib.mpcb_test_screen(len(tab), tab, box, int(head), len(regs), regs, np.ascontiguousarray(cn, F32), tshrink, out)
    return out


def _knife(lib, tab, head, regs):
    out = np.zeros(len(regs), F32)
    lib.mpcb_test_knife_edge_cn(len(tab), tab, int(head), len(regs), regs, out)
    return out


def _cases(lib, V, B, H, cost, n, seed):
    """(table, head, regs, cn) over every node of n trees: each node's knife-edge cn, values around it, and negative ones
    (false hits: t < 0 with t^2 > dd)"""
    tab, head = _table(V, B), cost == C.COST_MM
    regs = np.concatenate([_node_regs(V, B, H, x, cost) for x in _scenarios(n, seed)])
    knife = _knife(lib, tab, head, regs)
    ok = np.isfinite(knife)
    regs, knife = regs[ok], knife[ok]
    scales = [1.0, 1.0 + 2.0 ** -20, 1.0 - 2.0 ** -20, 1.001, 0.999, 1.1, 0.9, 0.5, -0.5, -1.0, -3.0]
    cn = np.concatenate([(knife * F32(k)).astype(F32) for k in scales])
    return tab, head, np.ascontiguousarray(np.tile(regs, (len(scales), 1))), cn, len(regs)


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
@pytest.mark.parametrize("gi", range(len(GRIDS)))
def test_stage1_bound_holds_every_leaf_and_rejects_no_flagged_node(lib, gi, cost):
    V, B, H = GRIDS[gi]
    tab, head, regs, cn, nodes = _cases(lib, V, B, H, cost, 6, 40 + gi)
    assert nodes > 100
    o = _run(lib, tab, _box(tab), head, regs, cn)
    assert np.all(o[:, 10] <= o[:, 8]) and np.all(o[:, 9] <= o[:, 11]), "a leaf's q outside the bound's q range"
    if head:
        assert np.all(o[:, 14] <= o[:, 12]) and np.all(o[:, 13] <= o[:, 15]), "a leaf's gg outside the gg range"
    assert np.all(o[:, 6] <= o[:, 4]) and np.all(o[:, 5] <= o[:, 7]), "a leaf's t outside [tlo, thi]"
    flagged = o[:, 0] > 0
    assert flagged.sum() > nodes                                     # knife edges and above: many flagged nodes
    rejected = flagged & (o[:, 3] == 0)
    assert not rejected.any(), f"{rejected.sum()} flagged nodes rejected by stage 1"
    assert (o[:, 3] == 0).any()                                     # and stage 1 does reject (below the knife edge)


def test_stage1_fails_with_a_tighter_bound(lib):
    """A grid of one control makes stage 1 exactly stage 2 (the box is that control): at each node's knife-edge cn,
    a T one ulp lower rejects flagged nodes.  On a real grid a heading interval one ulp narrower misses leaves."""
    V, B = [0.7], [0.3]
    tab = _table(V, B)
    regs = np.concatenate([_node_regs(V, B, 3, x, C.COST_MM) for x in _scenarios(400, 7)])
    knife = _knife(lib, tab, True, regs)
    ok = np.isfinite(knife)
    regs, knife = np.ascontiguousarray(regs[ok]), knife[ok]
    exact = _run(lib, tab, _box(tab), True, regs, knife)
    assert np.all(exact[:, 0] > 0) and np.all(exact[:, 3] == 1)
    tight = _run(lib, tab, _box(tab), True, regs, knife, tshrink=1)
    assert np.sum(tight[:, 3] == 0) > len(regs) // 10, "T one ulp lower should reject flagged nodes"

    V, B, H = GRIDS[0]
    tab, head, regs, cn, _ = _cases(lib, V, B, H, C.COST_MM, 6, 40)
    box = _box(tab)
    narrow = box.copy()
    narrow[4], narrow[5] = np.nextafter(box[4], F32(np.inf)), np.nextafter(box[5], F32(-np.inf))
    o = _run(lib, tab, narrow, head, regs, cn)
    assert np.any(o[:, 12] < o[:, 14]) or np.any(o[:, 13] > o[:, 15]), "a narrower heading interval should miss leaves"
