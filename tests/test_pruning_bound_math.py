"""The inequality behind the exact branch-and-bound (DESIGN.md section 3.5), checked numerically on the CPU.

The CUDA code (`projection_range`, `lower_bound_from`, `subtree_lower_bound` in csrc/mpcb_bounds.cuh) cuts a node when a lower bound on
the cost of every leaf `k` control steps below it exceeds the best cost known.  This file restates that bound in numpy
and checks, for EVERY node of small trees, that it never exceeds the true minimum over the node's leaves (float64
oracle) -- i.e. that cutting by it cannot lose the argmin -- and that it is much tighter than the isotropic bound
(`d >= D - k s_max`, `|q| <= wl k s_max`) it replaced.  The second half compiles the SHIPPED source, csrc/mpcb_bounds.cuh
(the header the kernels include), for the host with g++ and runs the same check on it, so the proof is about the code
that runs, not about a copy.  The GPU-side proof is tests/test_gpu_parity.py::test_branch_and_bound_is_exact."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import closed_form as C

L, DT = 0.5, 0.05
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _quad_min(e, Q):
    """min over |q| <= Q of q^2 + e q"""
    ae = np.abs(e)
    return np.where(ae <= 2 * Q, -0.25 * e * e, Q * (Q - ae))


def _bounds(V, B, H, x, k, cost, want_poses=False, og=None):
    """(isotropic bound, heading-aware bound, true minimum over the leaves below) for every depth-(H-k) node; the
    line origin `og` is the start unless given."""
    vv, bb, dphi = C.control_tables(V, B, L, DT)
    S = len(vv)
    s = vv * DT
    smax, smin, dmax = np.abs(s).max(), s.min(), np.abs(dphi).max()
    st, tg = x[:3], x[3:5]
    og = x[:2] if og is None else og
    wl, wh = (10.0, math.sqrt(10.0)) if cost == C.COST_MM else (100.0, 0.0)
    J = C.full_leaf_costs(st, tg, og, V, B, H, cost)
    X, Y, P = np.array([st[0]]), np.array([st[1]]), np.array([st[2]])
    for _ in range(H - k):                                            # poses of the depth-(H-k) nodes, leaf order
        P = (P[:, None] + dphi[None, :]).ravel()
        X = np.repeat(X, S) + np.tile(s, len(X)) * np.cos(P)
        Y = np.repeat(Y, S) + np.tile(s, len(Y)) * np.sin(P)
    relx, rely = tg[0] - X, tg[1] - Y
    D = np.hypot(relx, rely)
    A, Bc = tg[1] - og[1], tg[0] - og[0]
    e = wl * ((A * X - Bc * Y) + tg[0] * og[1] - tg[1] * og[0]) / math.hypot(A, Bc)
    hp = wh * (C.heading_reference(tg[0], tg[1]) - P)
    reach_iso = k * smax
    Q = wl * k * smax
    if smin < 0:
        reach = np.full_like(D, reach_iso)
        q_lo, q_hi = np.full_like(D, -Q), np.full_like(D, Q)
    else:
        def proj_range(cg, sg):
            """[lo, hi] of sum_i s_i cos(angle_i) for a direction at (cos, |sin|) = (cg, sg) from the present heading"""
            lo, hi = np.zeros_like(D), np.zeros_like(D)
            for i in range(1, k + 1):
                a = i * dmax
                if a >= math.pi:
                    cmax, cmin = np.ones_like(D), -np.ones_like(D)
                else:
                    ci, si = math.cos(a), math.sin(a)
                    cmax = np.where(cg >= ci, 1.0, cg * ci + sg * si)
                    cmin = np.where(-cg >= ci, -1.0, cg * ci - sg * si)
                hi += np.where(cmax >= 0, smax * cmax, smin * cmax)
                lo += np.where(cmin <= 0, smax * cmin, smin * cmin)
            return lo, hi
        _, reach = proj_range((relx * np.cos(P) + rely * np.sin(P)) / D, np.abs(relx * np.sin(P) - rely * np.cos(P)) / D)
        # scaled line offset q = wl * sum_i s_i (n . h_i), n = gradient direction of the signed line distance
        nx, ny = A / math.hypot(A, Bc), -Bc / math.hypot(A, Bc)
        lo, hi = proj_range(nx * np.cos(P) + ny * np.sin(P), np.abs(nx * np.sin(P) - ny * np.cos(P)))
        q_lo, q_hi = wl * lo, wl * hi
    base = 1e4 * D + e * e + hp * hp
    heading = _quad_min(-2 * hp, wh * k * dmax)
    qv = np.minimum(np.maximum(-e, q_lo), q_hi)                      # vertex of q^2 + 2 e q clamped into [q_lo, q_hi]
    rest = qv * (qv + 2 * e) + heading
    rest_iso = _quad_min(2 * e, Q) + heading
    true_min = J.reshape(len(D), -1).min(axis=1)
    poses = (X, Y, P)
    near = np.minimum(reach, D)                                      # a distance cannot become negative
    if want_poses:
        return base - 1e4 * near + rest, true_min, poses, (smax, smin, dmax, wl, wh)
    return base - 1e4 * reach_iso + rest_iso, base - 1e4 * near + rest, true_min, J.min()


GRIDS = {
    "window": (np.array(C.vector_of_velocities(0.5))[::2], np.array(C.vector_of_beta_angles(0.0))[::4]),   # cannot stop
    "from-rest": (np.linspace(0.0, 1.0, 6), np.linspace(-math.radians(60), math.radians(60), 7)),
    "wide-steer": (np.linspace(0.2, 1.0, 4), np.linspace(-1.4, 1.4, 9)),                                   # dphi_max 0.58 rad
    "reverse": (np.linspace(-0.5, 1.0, 5), np.linspace(-1.0, 1.0, 5)),                                     # isotropic fallback
}


@pytest.mark.parametrize("grid", sorted(GRIDS))
@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_subtree_bound_never_exceeds_the_true_minimum(grid, cost):
    V, B = GRIDS[grid]
    sc = C.random_scenarios(10, 11)
    sc[0, 3:5] = sc[0, :2] + [0.05, 0.02]                 # target next to the robot
    sc[1, 2] = math.atan2(sc[1, 4] - sc[1, 1], sc[1, 3] - sc[1, 0]) + math.pi      # facing exactly away
    sc[2, 2] = math.atan2(sc[2, 4] - sc[2, 1], sc[2, 3] - sc[2, 0])                # facing exactly at the target
    for x in sc:
        for k in (1, 2, 3):
            iso, new, true_min, _ = _bounds(V, B, 3, x, k, cost)
            ok = true_min < 1e7                           # the "on the line origin" special case only raises costs
            slack = true_min[ok] - new[ok]
            assert slack.min() >= -1e-7 * max(1.0, np.abs(true_min[ok]).max() * 1e-6), (grid, k, slack.min())
            assert np.all(iso[ok] <= new[ok] + 1e-9)      # never looser than the bound it replaced


def test_heading_aware_bound_is_what_makes_the_cut_bite():
    """Fraction of depth-(H-1) nodes that survive `bound <= optimum + tol` over random scenarios: close to all of them
    with the isotropic bound on the acceleration-window grid (the robot cannot stop or turn round in one step, yet the
    bound pretends it can), a few per cent with the heading-aware bound."""
    V, B = GRIDS["window"]
    surv_iso, surv_new = [], []
    for x in C.random_scenarios(12, 3):
        iso, new, _, jstar = _bounds(V, B, 3, x, 1, C.COST_MM)
        surv_iso.append(np.mean(iso <= jstar + 0.02))
        surv_new.append(np.mean(new <= jstar + 0.02))
    assert np.mean(surv_iso) > 0.8
    assert np.mean(surv_new) < 0.05


def test_line_offset_interval_matters_for_the_tree_cost():
    """With the tree script's cost (line weight 1e4) the line term dominates the differences between leaves; bounding
    the line offset by the interval the heading range allows, instead of +-wl k s_max, is what cuts there."""
    V, B = GRIDS["window"]
    surv_iso, surv_new = [], []
    for x in C.random_scenarios(12, 3):
        iso, new, _, jstar = _bounds(V, B, 3, x, 1, C.COST_TREE)
        surv_iso.append(np.mean(iso <= jstar + 0.02))
        surv_new.append(np.mean(new <= jstar + 0.02))
    assert np.mean(surv_new) < 0.25 * np.mean(surv_iso), (np.mean(surv_iso), np.mean(surv_new))


def tol_model(x, og, H, cost, smax, dphimax):
    """Python mirror of the window widths prep_kernel gives a prefix-algorithm solve (csrc/mpcb_kernels.cu, DESIGN.md
    section 3.3): (tol, tol1), each twice an error bound, incl. the float64 rounding at the solve's coordinates."""
    xs, ys, p0, xt, yt = x
    ox, oy = og
    wl, wh = (10.0, math.sqrt(10.0)) if cost == C.COST_MM else (100.0, 0.0)
    A, Bc = yt - oy, xt - ox
    norm = math.sqrt(A * A + Bc * Bc)
    e0 = wl * ((A * xs - Bc * ys) + (xt * oy - yt * ox)) / norm
    hp0 = wh * (C.heading_reference(xt, yt) - p0)
    d0 = math.hypot(xt - xs, yt - ys)
    Rtot, Rl, Gl = H * smax, smax, wh * dphimax
    E, Hh, Q = abs(e0) + wl * Rtot, abs(hp0) + wh * H * dphimax, wl * Rl
    Phi, X, Y = abs(p0) + H * dphimax, abs(xs) + Rtot, abs(ys) + Rtot
    dphi = H * 2.0 ** -53 * Phi
    dp = H * 2.0 ** -52 * (X + Y) + H * smax * dphi
    de = wl * (2.0 ** -51 * (abs(A) * X + abs(Bc) * Y + abs(xt * oy) + abs(yt * ox)) / norm + dp)
    dh = wh * dphi
    Mw = (1e4 * dp + 2 * de * (2 * E + de) + 2 * dh * (2 * Hh + dh)) * 2.0 ** 23
    M = 1e4 * Rl * 16 + 4 * Q * (2 * E + Q) + 4 * Gl * (Gl + 2 * Hh) + Mw
    Dmax, E1, H1 = d0 + Rtot, E + Q, Hh + Gl
    Vmax = 1e4 * Dmax + E1 * E1 + H1 * H1
    M1 = 3e4 * Dmax + 2e4 * smax + 4 * E1 * E1 + 3 * H1 * H1 + Vmax + Mw
    tol = 2 * M * 2.0 ** -23
    return tol, max(tol, 2 * M1 * 2.0 ** -23)


# ---------------------------------------------------------------- the shipped CUDA source, compiled for the host
@pytest.fixture(scope="module")
def shipped_bound():
    """diplomjourney_b200/csrc/mpcb_bounds.cuh (the file the kernels include) built with g++ behind a C entry point."""
    src = os.path.join(ROOT, "tests", "native", "bounds_host.cpp")
    out_dir = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "bounds_host.so")
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-std=c++17", "-I", os.path.join(ROOT, "diplomjourney_b200", "csrc"),
                           "-I", cuda_inc, src, "-o", so])
    lib = ctypes.CDLL(so)
    dp = ctypes.POINTER(ctypes.c_double)
    lib.mpcb_test_subtree_lower_bounds.argtypes = [ctypes.c_double] * 3 + [dp, ctypes.c_longlong, dp, dp, dp, ctypes.c_int, dp]

    def bound(x, cost, poses, consts, k, og=None):
        """J lower bound (absolute cost) of every node in `poses` with k steps to go, by the library's own code (line
        origin `og`, default the start)."""
        X, Y, P = poses
        smax, smin, dmax, wl, wh = consts
        xs, ys, p0, xt, yt = x
        ox, oy = (xs, ys) if og is None else og
        c0, s0 = math.cos(p0), math.sin(p0)
        # SolveParams exactly as prep_kernel builds them (csrc/mpcb_kernels.cu); e0 in the reference's order
        A, Bc = yt - oy, xt - ox
        norm = math.sqrt(A * A + Bc * Bc)
        rx, ry = xt - xs, yt - ys
        u0, w0, d0 = c0 * rx + s0 * ry, c0 * ry - s0 * rx, math.hypot(rx, ry)
        e0 = wl * ((A * xs - Bc * ys) + (xt * oy - yt * ox)) / norm
        nx0, ny0 = wl * (A * c0 - Bc * s0) / norm, wl * (-A * s0 - Bc * c0) / norm
        hp0 = wh * (C.heading_reference(xt, yt) - p0)
        kbase = 1e4 * d0 + e0 * e0 + hp0 * hp0
        solve = np.array([u0, w0, d0, e0, nx0, ny0, hp0, wl, wh])
        xi = np.ascontiguousarray(c0 * (X - xs) + s0 * (Y - ys))      # node poses in the start frame
        eta = np.ascontiguousarray(-s0 * (X - xs) + c0 * (Y - ys))
        psi = np.ascontiguousarray(P - p0)
        out = np.empty_like(xi)
        p = lambda a: a.ctypes.data_as(dp)
        lib.mpcb_test_subtree_lower_bounds(smax, smin, dmax, p(solve), len(xi), p(xi), p(eta), p(psi), k, p(out))
        if k in (1, 2):     # ... and the fp32 pre-filter (nodes: one step, tiles: two) on the same nodes, with the model's error bound
            out32 = np.empty(len(xi), np.float32)
            lib.mpcb_test_prefilter32(smax, smin, dmax, p(solve), len(xi), p(xi), p(eta), p(psi),
                                      out32.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), k)
            _, tol1 = tol_model(x, (ox, oy), 3, cost, smax, dmax)
            bound.prefilter = (out32.astype(np.float64), out, tol1)
        return kbase + out
    lib.mpcb_test_prefilter32.argtypes = [ctypes.c_double] * 3 + [dp, ctypes.c_longlong, dp, dp, dp, ctypes.POINTER(ctypes.c_float),
                                          ctypes.c_int]
    return bound


@pytest.mark.parametrize("grid", sorted(GRIDS))
@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_shipped_bound_code_never_exceeds_the_true_minimum(shipped_bound, grid, cost):
    """The same check on the code the kernels run: mpcb_bounds.cuh compiled for the host must (a) stay below the
    float64 oracle's minimum over the leaves of every node, and (b) agree with the numpy restatement above."""
    V, B = GRIDS[grid]
    sc = C.random_scenarios(8, 23)
    sc[0, 3:5] = sc[0, :2] + [0.05, 0.02]
    sc[1, 2] = math.atan2(sc[1, 4] - sc[1, 1], sc[1, 3] - sc[1, 0]) + math.pi
    for x in sc:
        for k in (1, 2, 3):
            new, true_min, poses, consts = _bounds(V, B, 3, x, k, cost, want_poses=True)
            lb = shipped_bound(x, cost, poses, consts, k)
            ok = true_min < 1e7
            scale = max(1.0, np.abs(true_min[ok]).max())
            assert (true_min[ok] - lb[ok]).min() >= -1e-10 * scale, (grid, k, (true_min[ok] - lb[ok]).min())
            np.testing.assert_allclose(lb[ok], new[ok], rtol=0, atol=1e-8 * scale)


@pytest.mark.parametrize("grid", sorted(GRIDS))
@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_fp32_prefilter_stays_within_its_margin_of_the_float64_bound(shipped_bound, grid, cost):
    """The pruned pass 1 drops a node early when the bound evaluated in FLOAT exceeds the upper bound by 8 tol1.  That is
    only sound if |lb32 - lb64| stays (well) below 8 tol1: measured here on every depth-2 node of small trees with the
    shipped code, including a robot next to its target and robots far from their line (large anchors)."""
    V, B = GRIDS[grid]
    sc = C.random_scenarios(10, 29)
    sc[0, 3:5] = sc[0, :2] + [0.05, 0.02]
    sc[1, 3:5] = sc[1, :2] + [60.0, -45.0]                            # a far target: large kWd d
    for steps in (1, 2):                                              # node test (children) and tile test (two levels)
        worst = 0.0
        for x in sc:
            new, true_min, poses, consts = _bounds(V, B, 3, x, steps, cost, want_poses=True)
            shipped_bound(x, cost, poses, consts, steps)
            lb32, lb64, tol1 = shipped_bound.prefilter
            ok = np.isfinite(lb64)
            err = np.abs(lb32[ok] - lb64[ok]).max()
            worst = max(worst, err / tol1)
            assert err <= tol1, (grid, cost, steps, err, tol1)        # the analysis in mpcb_bounds.cuh; the kernel allows 8x
        assert worst > 0.0
        print(f"fp32 pre-filter, {steps} step(s): worst |lb32 - lb64| = {worst:.3f} tol1 ({grid}, {cost})")


WORLD_SHIFTS = [0.0, 1e3, 1e5, 5e5, 5e6]


def world_bound_scenarios(shift, seed):
    """(x, origin) around the world point (shift, 0.9 shift): the line origin 0-300 m off the start, headings accumulated
    to +-10..60 rad as closed loops leave them, targets 30-3,000 m away, and one robot next to its target."""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(8):
        x = C.random_scenarios(1, seed * 10 + k)[0]
        x[[0, 3]] += shift
        x[[1, 4]] += 0.9 * shift
        og = x[:2] + rng.uniform(-300, 300, 2) * [0.0, 0.02, 0.1, 1.0][k % 4]
        if k % 3 == 1:
            x[2] += rng.choice([-1.0, 1.0]) * rng.uniform(10, 60)
        if k % 4 == 2:
            ang, dist = rng.uniform(-math.pi, math.pi), rng.uniform(30, 3000)
            x[3:5] = x[:2] + dist * np.array([math.cos(ang), math.sin(ang)])
        if k == 7:
            x[3:5] = x[:2] + [0.05, 0.02]
        out.append((x, og))
    return out


@pytest.mark.parametrize("grid", sorted(GRIDS))
@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_shipped_bound_cuts_only_what_the_window_allows_far_from_the_world_origin(shipped_bound, grid, cost):
    """Off the line origin and far from the world origin the oracle's float64 costs carry rounding noise that grows with
    the coordinates (tens of cost units at 5e6 m), which the bound, formed from anchors in the start frame, does not.
    The kernel cuts a node when LB > UB + tol1 + tol, so what must hold is LB <= true_min + tol1 + tol with the windows
    prep_kernel computes (tol_model) -- for every node of small trees, with the shipped code, in every region -- and the
    fp32 pre-filter must stay within tol1 of the float64 bound."""
    V, B = GRIDS[grid]
    for shift in WORLD_SHIFTS:
        worst, worst32 = -np.inf, 0.0
        for x, og in world_bound_scenarios(shift, int(shift) % 997 + 3):
            for k in (1, 2, 3):
                _, true_min, poses, consts = _bounds(V, B, 3, x, k, cost, want_poses=True, og=og)
                lb = shipped_bound(x, cost, poses, consts, k, og=og)
                tol, tol1 = tol_model(x, og, 3, cost, consts[0], consts[2])
                ok = np.isfinite(true_min)
                excess = (lb[ok] - true_min[ok]).max()
                assert excess <= tol1 + tol, (shift, k, excess, tol1 + tol)
                worst = max(worst, excess / (tol1 + tol))
                if k in (1, 2):
                    lb32, lb64, ptol1 = shipped_bound.prefilter
                    fin = np.isfinite(lb64)
                    err = np.abs(lb32[fin] - lb64[fin]).max()
                    assert err <= ptol1, (shift, k, err, ptol1)
                    worst32 = max(worst32, err / ptol1)
        print(f"{grid} {cost} shift {shift:g}: worst (LB - true min) = {worst:.3g} (tol1 + tol), "
              f"|lb32 - lb64| = {worst32:.3g} tol1")
