"""The shipped float64 leaf evaluation far from the world origin, on the CPU.

Robot logs often carry UTM coordinates (easting ~5e5 m, northing ~5e6 m).  There the products in the reference's line
distance, |(y_t-y_0) x - (x_t-x_0) y + x_t y_0 - y_t x_0|, are ~1e13, and every rounding of that sum is worth tens of
cost units: the library only returns the reference's own float64 choice if it rounds exactly as the reference does, in
the reference's order -- ((A x - B y) + x_t y_0) - y_t x_0, no FMA contraction.  These tests compile
csrc/mpcb_exact.cuh (what the refinement and the final re-roll evaluate) for the host with g++ -ffp-contract=off and
compare it BIT FOR BIT with the C oracle (oracle/mpc_oracle.c, the same libm) on every leaf of small trees, at world
shifts up to 5e6 m, with the line origin up to 300 m off the start, for both costs, FULL and HELD trees and the slow-down
override; and the argmin of whole trees.  The fp32 side of the same regions (the error model, the bounds) is
tests/test_pruning_bound_math.py; the device paths are tests/test_gpu_world_coordinates.py."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import c_oracle as K
from oracle import closed_form as C

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
L, DT, VMIN = C.CONFIG["L"], C.CONFIG["delta_t"], C.CONFIG["v_min"]
SHIFTS = [0.0, 1e3, 1e5, 5e5, 5e6]
V, B = np.linspace(0.0, 1.0, 6), np.linspace(-1.0, 1.0, 7)      # S = 42, H = 3: 74,088 leaves


@pytest.fixture(scope="module")
def host():
    out_dir = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "exact_host_world.so")
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-std=c++17",
                           "-I", os.path.join(ROOT, "diplomjourney_b200", "csrc"), "-I", cuda_inc,
                           os.path.join(ROOT, "tests", "native", "exact_host.cpp"), "-o", so])
    lib = ctypes.CDLL(so)
    dp = ctypes.POINTER(ctypes.c_double)
    lib.mpcb_test_exact_costs.argtypes = [dp, ctypes.c_int, dp, ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                          ctypes.c_int, ctypes.c_int, ctypes.c_int, dp, dp, dp, ctypes.c_int,
                                          ctypes.c_double, ctypes.c_longlong, dp]
    return lib


def _shipped_costs(lib, mode, cost, H, state, target, origin, slow=False):
    """every leaf's cost by mpcb::exact_cost (mode 0 FULL, 1 HELD)"""
    v, b = np.ascontiguousarray(V), np.ascontiguousarray(B)
    st, tg, og = (np.ascontiguousarray(np.asarray(a, np.float64)) for a in (state[:3], target, origin))
    n = (v.size * b.size) ** (H if mode == 0 else 1)
    out = np.empty(n)
    p = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    lib.mpcb_test_exact_costs(p(v), v.size, p(b), b.size, L, DT, mode, 0 if cost == C.COST_MM else 1, H,
                              p(st), p(tg), p(og), 1 if slow else 0, VMIN, n, p(out))
    return out


def world_scenarios(shift, seed, n=4):
    """(state, target, origin) around the world point (shift, 0.9 shift): the line origin 0-300 m off the start (the
    first one ON the start: the reference's d_l = 1000 special case), targets 5-3,000 m away, headings also accumulated
    outside [-pi, pi] as closed loops produce them."""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n):
        st = np.array([shift + rng.uniform(-10, 10), 0.9 * shift + rng.uniform(-10, 10), rng.uniform(-math.pi, math.pi)])
        if k == 3:
            st[2] += rng.choice([-1.0, 1.0]) * rng.uniform(10, 60)
        dist = [8.0, 40.0, 3000.0, 300.0][k % 4] * rng.uniform(0.6, 1.0)
        ang = rng.uniform(-math.pi, math.pi)
        tg = st[:2] + dist * np.array([math.cos(ang), math.sin(ang)])
        off = [0.0, 5.0, 300.0, 60.0][k % 4] * rng.uniform(0.5, 1.0)
        oa = rng.uniform(-math.pi, math.pi)
        og = st[:2] + off * np.array([math.cos(oa), math.sin(oa)])
        out.append((st, tg, og))
    return out


def _bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
@pytest.mark.parametrize("shift", SHIFTS)
def test_full_tree_costs_are_the_oracles_bit_for_bit(host, shift, cost):
    """Every leaf of FULL trees (H = 3) around the world point: the shipped evaluation returns the oracle's bits."""
    for st, tg, og in world_scenarios(shift, int(shift) % 1000 + 7):
        J = _shipped_costs(host, 0, cost, 3, st, tg, og)
        Jo = K.full_leaf_costs(st, tg, og, V, B, 3, cost)
        bad = np.flatnonzero(_bits(J) != _bits(Jo))
        assert bad.size == 0, (shift, cost, bad.size, float(np.abs(J - Jo)[bad].max()))


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
@pytest.mark.parametrize("shift", SHIFTS)
def test_held_tree_costs_are_the_oracles_bit_for_bit(host, shift, cost):
    """Every candidate of HELD trees, with and without the slow-down override (every velocity := max(min V, v_min))."""
    for slow in (False, True):
        for st, tg, og in world_scenarios(shift, int(shift) % 1000 + 11):
            J = _shipped_costs(host, 1, cost, 3, st, tg, og, slow=slow)
            Jo = K.solve_held(st, tg, og, V, B, 3, cost, slow=slow, v_min=VMIN)["leaf_costs"]
            assert np.array_equal(_bits(J), _bits(Jo)), (shift, cost, slow, float(np.abs(J - Jo).max()))


def test_start_on_the_line_origin_far_from_the_world_origin(host):
    """The robot starts ON the line origin (d_l = 1000 for a leaf that has not moved) at 5e6 m: v = 0 leaves take the
    special case, all others the reference's line distance -- both bit for bit."""
    Vz = np.array([0.0, 0.4, 1.0])
    for shift in (5e5, 5e6):
        st = np.array([shift + 0.3, 0.9 * shift - 0.7, 0.4])
        tg, og = st[:2] + [6.0, -2.5], st[:2].copy()
        for cost in (C.COST_MM, C.COST_TREE):
            for mode in (0, 1):
                v, b = np.ascontiguousarray(Vz), np.ascontiguousarray(B)
                n = (v.size * b.size) ** (3 if mode == 0 else 1)
                out = np.empty(n)
                p = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
                host.mpcb_test_exact_costs(p(v), v.size, p(b), b.size, L, DT, mode, 0 if cost == C.COST_MM else 1, 3,
                                           p(st), p(tg), p(og), 0, VMIN, n, p(out))
                Jo = (K.full_leaf_costs(st, tg, og, Vz, B, 3, cost) if mode == 0
                      else K.solve_held(st, tg, og, Vz, B, 3, cost)["leaf_costs"])
                assert np.array_equal(_bits(out), _bits(Jo)), (shift, cost, mode)
                assert np.sum(out >= 1e8) >= B.size          # the special case did occur


@pytest.mark.parametrize("cost", [C.COST_MM, C.COST_TREE])
def test_argmin_of_whole_trees_is_the_oracles(host, cost):
    """The decision itself: the first minimum over whole FULL trees, shipped evaluation against the C oracle's solve,
    at every shift (both report the lowest index of the smallest cost)."""
    for shift in SHIFTS:
        for st, tg, og in world_scenarios(shift, int(shift) % 1000 + 19, n=2):
            J = _shipped_costs(host, 0, cost, 3, st, tg, og)
            o = K.solve_full(st, tg, og, V, B, 3, cost)
            assert int(np.argmin(J)) == o["index"], (shift, cost)
            assert J.min() == o["cost"]


def test_a_precomputed_line_constant_picks_another_leaf_at_utm_northings(host):
    """Why the order matters: with x_t y_0 - y_t x_0 added as one precomputed constant (what the library did before)
    the float64 costs of this 5e6 m TREE tree move by tens of units and the first minimum is another leaf.  The shipped
    evaluation picks the oracle's."""
    st, tg, og = _UTM_CASE
    J = _shipped_costs(host, 0, C.COST_TREE, 3, st, tg, og)
    Jo, x, y, _ = C.full_leaf_costs(st, tg, og, V, B, 3, C.COST_TREE, return_xy=True)
    assert np.array_equal(_bits(J), _bits(K.full_leaf_costs(st, tg, og, V, B, 3, C.COST_TREE)))
    A, Bc = tg[1] - og[1], tg[0] - og[0]
    lineC = tg[0] * og[1] - tg[1] * og[0]
    dl = np.abs((A * x - Bc * y) + lineC) / math.sqrt(A * A + Bc * Bc)
    J_const = 10000 * np.sqrt((tg[0] - x) ** 2 + (tg[1] - y) ** 2) + 10000 * dl ** 2
    assert np.abs(J_const - Jo).max() > 1.0
    assert int(np.argmin(J_const)) != int(np.argmin(Jo))
    assert int(np.argmin(J)) == K.solve_full(st, tg, og, V, B, 3, C.COST_TREE)["index"]


# a robot 5 m from its target and its line origin at easting 5.0e6 m, northing 4.5e6 m (start, target, line origin)
_UTM_CASE = (np.array([4999993.571, 4499997.925, -3.105]), np.array([4999988.821, 4499996.349]),
             np.array([4999989.631, 4499999.257]))
