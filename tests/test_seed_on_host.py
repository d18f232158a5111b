"""The seeding of the actual run's generators, compiled for the HOST with g++ and checked on the CPU.

csrc/mpcb_noise.cuh's mt_seed (numpy's mt19937_seed, RandomState(int)) and mt_seed_by_array (mt19937_init_by_array,
RandomState(array)) are plain host/device code.  tests/native/seed_host.cpp builds them, next to the draws of
tests/native/noise_host.cpp, into a small shared object; every record (key[624] + pos) must equal
RandomState(seed).get_state(), and the stream drawn from it numpy's, bit for bit.  Also here: the argument checks of
math_mpc_batch(..., seeds=), which run before any solver is created."""
import ctypes
import importlib
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INT_SEEDS = (0, 1, 5, 5489, 19650218, 2 ** 31, 2 ** 32 - 1)
KEY_LENGTHS = (1, 2, 623, 624, 625, 1000)


@pytest.fixture(scope="module")
def host():
    out_dir = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "seed_host.so")
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-std=c++17",
                           "-I", os.path.join(ROOT, "diplomjourney_b200", "csrc"), "-I", cuda_inc,
                           os.path.join(ROOT, "tests", "native", "seed_host.cpp"),
                           os.path.join(ROOT, "tests", "native", "noise_host.cpp"), "-o", so])
    lib = ctypes.CDLL(so)
    vp, ll = ctypes.c_void_p, ctypes.c_longlong
    lib.mpcb_test_mt_seed.argtypes = [vp, ctypes.c_uint32]
    lib.mpcb_test_mt_seed_by_array.argtypes = [vp, vp, ctypes.c_int]
    lib.mpcb_test_mt_words.argtypes = [vp, ll, vp]
    lib.mpcb_test_actuators.argtypes = [vp, ll, vp, vp, vp, vp]
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _record(rs):
    st = rs.get_state()
    return np.concatenate([st[1].astype(np.uint32), np.array([st[2]], np.uint32)])


def _seeded(host, seed):
    """The record the shipped code builds for RandomState(seed): an int, or a list (a key)."""
    rec = np.full(625, 0xDEADBEEF, np.uint32)          # every word must be written
    if isinstance(seed, list):
        key = np.array(seed, np.uint32)
        host.mpcb_test_mt_seed_by_array(_p(rec), _p(key), key.size)
    else:
        host.mpcb_test_mt_seed(_p(rec), seed)
    return rec


def _key(k):
    """A key of k words that includes 0 and 2^32 - 1."""
    key = np.random.default_rng(k).integers(0, 2 ** 32, k, dtype=np.uint64)
    key[0] = 2 ** 32 - 1
    key[k // 2] = 0
    if k > 2:
        key[-1] = 2 ** 32 - 1
    return [int(x) for x in key]


SEEDS = [s for s in INT_SEEDS] + [_key(k) for k in KEY_LENGTHS] + [[5], [0], [2 ** 32 - 1, 0]]
IDS = [f"int{s}" for s in INT_SEEDS] + [f"key{k}" for k in KEY_LENGTHS] + ["key[5]", "key[0]", "key[max,0]"]


@pytest.mark.parametrize("seed", SEEDS, ids=IDS)
def test_seeded_record_equals_numpy(host, seed):
    """key[624] and pos == RandomState(seed).get_state(), word for word."""
    np.testing.assert_array_equal(_seeded(host, seed), _record(np.random.RandomState(seed)))


def test_integer_seed_and_one_word_key_are_different_streams(host):
    assert not np.array_equal(_seeded(host, 5), _seeded(host, [5]))
    np.testing.assert_array_equal(_seeded(host, [5]), _record(np.random.RandomState([5])))


@pytest.mark.parametrize("seed", [0, 2 ** 32 - 1, _key(2), _key(700)], ids=["int0", "intmax", "key2", "key700"])
def test_stream_after_seeding_equals_numpy(host, seed):
    """The first 2,000 raw words after seeding, then the actuator draws (velocity, then beta, tick after tick), and the
    final (key, pos) -- all from the shipped seeding, against the same RandomState."""
    mt = importlib.import_module("diplomjourney_b200.math_model_tree")
    rec = _seeded(host, seed)
    rs = np.random.RandomState(seed)
    n = 2000
    words = np.empty(n, np.uint32)
    host.mpcb_test_mt_words(_p(rec), n, _p(words))
    np.testing.assert_array_equal(words, rs.randint(0, 2 ** 32, size=n, dtype=np.uint32))
    rng = np.random.default_rng(1)
    v_ref = rng.choice([0.0, 0.3, 0.4, 0.7], n)
    b_ref = rng.uniform(-1.05, 1.05, n)
    v_out, b_out = np.empty(n), np.empty(n)
    host.mpcb_test_actuators(_p(rec), n, _p(v_ref), _p(b_ref), _p(v_out), _p(b_out))
    want_v = np.empty(n)
    want_b = np.empty(n)
    for i in range(n):
        want_v[i] = mt.get_actual_velocity(float(v_ref[i]), rs)
        want_b[i] = mt.get_actual_beta_angle(float(b_ref[i]), rs)
    np.testing.assert_array_equal(v_out.view(np.uint64), want_v.view(np.uint64))
    np.testing.assert_array_equal(b_out.view(np.uint64), want_b.view(np.uint64))
    np.testing.assert_array_equal(rec, _record(rs))


def test_seed_keys_forms():
    """_native.seed_keys: [N] integer seeds -> key_len 0, [N][K] keys -> key_len K (also K == 1), uint32, values kept."""
    from diplomjourney_b200 import _native as nat
    k, n = nat.seed_keys([0, 5, 2 ** 32 - 1], 3)
    assert n == 0 and k.dtype == np.uint32 and k.tolist() == [0, 5, 2 ** 32 - 1]
    k, n = nat.seed_keys(np.array([[5], [7]]), 2)
    assert n == 1 and k.shape == (2, 1) and k.dtype == np.uint32
    k, n = nat.seed_keys([[1, 2 ** 32 - 1], [3, 4]], 2)
    assert n == 2 and k.tolist() == [[1, 2 ** 32 - 1], [3, 4]]
    k, n = nat.seed_keys(np.array([2 ** 32 - 1], np.uint64), 1)
    assert k.tolist() == [2 ** 32 - 1]


def test_seeds_argument_errors():
    """math_mpc_batch(..., seeds=) rejects bad seeds before it creates a solver (the module's solver is replaced by an
    object without methods: reaching it would raise AttributeError), with numpy's wording for out-of-range values; and
    np.random is not touched."""
    mt = importlib.reload(importlib.import_module("diplomjourney_b200.math_model_tree"))
    mt._backend = object()
    two = [[0, 0, 0, 0, 0]] * 2
    run = lambda seeds, **kw: mt.math_mpc_batch(two, [[2, 3]], **{"isActual": True, "device_noise": True,
                                                                  "seeds": seeds, **kw})
    before = np.random.get_state()
    with pytest.raises(ValueError, match="rngs"):                # seeds and rngs
        run([1, 2], rngs=[np.random.RandomState(1), np.random.RandomState(2)])
    with pytest.raises(ValueError, match="device_noise"):        # seeds need the device loop
        run([1, 2], device_noise=False)
    with pytest.raises(ValueError, match="device_noise"):
        mt.math_mpc_batch(two, [[2, 3]], seeds=[1, 2])
    with pytest.raises(ValueError, match="isActual"):
        run([1, 2], isActual=False)
    for bad in ([1, 2, 3], [1], [[1, 2]] * 3, []):            # one row per robot
        with pytest.raises(ValueError, match="rows"):
            run(bad)
    with pytest.raises(ValueError, match="non-empty"):           # an empty key
        run([[], []])
    for bad in ([[[1, 2]], [[3, 4]]], 7, [[1, 2], [3]]):      # a key that is not 1-d, a scalar, ragged keys
        with pytest.raises(ValueError):
            run(bad)
    for bad in ([-1, 2], [1, 2 ** 32], [[1, 2 ** 32]] * 2, [[0, -1], [0, 0]], [2 ** 70, 1], np.array([1, -5])):
        with pytest.raises(ValueError, match=r"Seed must be between 0 and 2\*\*32 - 1"):
            run(bad)
    with pytest.raises(TypeError):                               # not integers
        run([1.5, 2.0])
    with pytest.raises(TypeError):
        run(["a", "b"])
    after = np.random.get_state()
    assert after[2] == before[2] and np.array_equal(after[1], before[1])
    mt._backend = None
