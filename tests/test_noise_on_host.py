"""The actuator noise of the device-resident "actual" run, compiled for the HOST with g++ and checked on the CPU.

csrc/mpcb_noise.cuh (numpy's legacy MT19937 stream over the (key, pos) record RandomState.get_state() hands out, its
random() and masked-rejection randint(), and the two actuator functions of math_model_tree.py:259-275) is plain
host/device code.  tests/native/noise_host.cpp builds it into a small shared object; every value and every final
(key, pos) must equal np.random.RandomState's, bit for bit.  Also here: the argument checks of
math_mpc_batch(..., device_noise=True), which run before any solver is touched."""
import ctypes
import importlib
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEEDS = (0, 1, 2 ** 32 - 1)
POSITIONS = (0, 1, 623, 624)


@pytest.fixture(scope="module")
def host():
    out_dir = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "noise_host.so")
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-std=c++17",
                           "-I", os.path.join(ROOT, "diplomjourney_b200", "csrc"), "-I", cuda_inc,
                           os.path.join(ROOT, "tests", "native", "noise_host.cpp"), "-o", so])
    lib = ctypes.CDLL(so)
    vp, ll = ctypes.c_void_p, ctypes.c_longlong
    lib.mpcb_test_mt_words.argtypes = [vp, ll, vp]
    lib.mpcb_test_random_sample.argtypes = [vp, ll, vp]
    lib.mpcb_test_randint.argtypes = [vp, ctypes.c_int, ctypes.c_int, ll, vp]
    lib.mpcb_test_actuators.argtypes = [vp, ll, vp, vp, vp, vp]
    return lib


def _generator(seed, pos):
    """A RandomState with the key of ``seed`` and the stream position ``pos`` (pos = 624: as seeded, the first draw
    twists; pos = 0: a twist has just happened)."""
    rs = np.random.RandomState(seed)
    key = rs.get_state()[1]
    rs.set_state(("MT19937", key, pos))
    return rs


def _record(rs):
    st = rs.get_state()
    return np.concatenate([st[1].astype(np.uint32), np.array([st[2]], np.uint32)])


def _assert_same_state(rec, rs):
    np.testing.assert_array_equal(rec, _record(rs))


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@pytest.mark.parametrize("pos", POSITIONS)
@pytest.mark.parametrize("seed", SEEDS)
def test_raw_words_random_and_randint_equal_numpy(host, seed, pos):
    """Raw tempered words, random() and the three randint ranges of the actuator functions, each over several twists,
    and the final (key, pos) after each."""
    n = 2000
    rs = _generator(seed, pos)
    rec = _record(rs)
    words = np.empty(n, np.uint32)
    host.mpcb_test_mt_words(_p(rec), n, _p(words))
    np.testing.assert_array_equal(words, rs.randint(0, 2 ** 32, size=n, dtype=np.uint32))   # one word per value
    _assert_same_state(rec, rs)

    rs = _generator(seed, pos)
    rec = _record(rs)
    u = np.empty(n)
    host.mpcb_test_random_sample(_p(rec), n, _p(u))
    want = np.array([rs.random() for _ in range(n)])
    np.testing.assert_array_equal(u.view(np.uint64), want.view(np.uint64))
    _assert_same_state(rec, rs)

    for lo, hi in ((0, 5), (-100, 10), (-5, 5), (3, 4)):
        rs = _generator(seed, pos)
        rec = _record(rs)
        k = np.empty(n, np.int64)
        host.mpcb_test_randint(_p(rec), lo, hi, n, _p(k))
        np.testing.assert_array_equal(k, [rs.randint(lo, hi) for _ in range(n)], err_msg=f"randint({lo}, {hi})")
        _assert_same_state(rec, rs)


@pytest.mark.parametrize("pos", POSITIONS)
@pytest.mark.parametrize("seed", SEEDS)
def test_actuator_functions_equal_the_module(host, seed, pos):
    """actual_velocity then actual_beta, tick after tick, == the module's get_actual_velocity / get_actual_beta_angle on
    the same RandomState (the reference's functions with the generator passed in): v_ref below, at and above the 0.4
    switch, results bit for bit and the final (key, pos)."""
    mt = importlib.import_module("diplomjourney_b200.math_model_tree")
    n = 3000
    rng = np.random.default_rng(seed % 1000 + pos)
    v_ref = rng.choice([0.0, 0.05, 0.39999999999999997, 0.4, 0.4000000000000001, 0.7, 0.995], n)
    b_ref = rng.uniform(-1.05, 1.05, n)
    b_ref[:7] = (0.0, -1.0471975511965976, 1.0471975511965976, 0.5, -0.5, 1e-17, -0.0)
    rs = _generator(seed, pos)
    rec = _record(rs)
    v_out, b_out = np.empty(n), np.empty(n)
    host.mpcb_test_actuators(_p(rec), n, _p(v_ref), _p(b_ref), _p(v_out), _p(b_out))
    want_v, want_b = np.empty(n), np.empty(n)
    for i in range(n):
        want_v[i] = mt.get_actual_velocity(float(v_ref[i]), rs)
        want_b[i] = mt.get_actual_beta_angle(float(b_ref[i]), rs)
    np.testing.assert_array_equal(v_out.view(np.uint64), want_v.view(np.uint64))
    np.testing.assert_array_equal(b_out.view(np.uint64), want_b.view(np.uint64))
    _assert_same_state(rec, rs)
    assert (v_out != v_ref).sum() > n // 3 and (b_out != b_ref).sum() > n // 3     # the noise did fire


def test_device_noise_argument_errors():
    """math_mpc_batch(..., device_noise=True) rejects what one CTA per robot cannot reproduce, before it touches a
    solver (the module's solver is replaced by an object without methods: reaching it would raise AttributeError)."""
    mt = importlib.reload(importlib.import_module("diplomjourney_b200.math_model_tree"))
    mt._backend = object()
    one, two = [[0, 0, 0, 0, 0]], [[0, 0, 0, 0, 0]] * 2
    with pytest.raises(ValueError):                 # noise needs the actual run
        mt.math_mpc_batch(one, [[2, 3]], device_noise=True, rngs=[np.random.RandomState(1)])
    with pytest.raises(ValueError):                 # the device path is not the per-tick path
        mt.math_mpc_batch(one, [[2, 3]], isActual=True, device_noise=True, host_loop=True, rngs=[np.random.RandomState(1)])
    with pytest.raises(ValueError):                 # one shared generator interleaves its draws over the robots
        mt.math_mpc_batch(two, [[2, 3]], isActual=True, device_noise=True)
    with pytest.raises(ValueError):                 # one generator per robot
        mt.math_mpc_batch(two, [[2, 3]], isActual=True, device_noise=True, rngs=[np.random.RandomState(1)])
    with pytest.raises(TypeError):                  # numpy's Generator (PCG64) is another stream
        mt.math_mpc_batch(two, [[2, 3]], isActual=True, device_noise=True,
                          rngs=[np.random.RandomState(1), np.random.default_rng(2)])
    with pytest.raises(TypeError):
        mt.math_mpc_batch(one, [[2, 3]], isActual=True, device_noise=True, rngs=[7])
    before = np.random.get_state()
    with pytest.raises(ValueError):
        mt.math_mpc_batch(two, [[2, 3]], isActual=True, device_noise=True)
    after = np.random.get_state()
    assert after[2] == before[2] and np.array_equal(after[1], before[1])           # nothing was drawn
    mt._backend = None
