"""numpy's Generator(PCG64) stream of the device-resident "actual" run, compiled for the HOST with g++ and checked on the CPU.

csrc/mpcb_pcg64.cuh (the 128-bit LCG step and XSL-RR output, the buffered 32-bit draws, random(), Lemire's integers(),
SeedSequence -> PCG64 seeding, and the PCG64 actuator functions) is plain host/device code.  tests/native/pcg64_host.cpp
builds it into a small shared object; every value and every final bit_generator.state must equal numpy's, bit for bit.
Also here: the packing of seeds into SeedSequence words and the argument checks of math_mpc_batch / Solver, which run
before any solver is touched."""
import ctypes
import importlib
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MULT = (2549297995355413924 << 64) + 4865540595714422341
M128 = (1 << 128) - 1
RANGES = ((0, 5), (-100, 10), (-5, 5), (3, 4))


@pytest.fixture(scope="module")
def host():
    out_dir = os.path.join(ROOT, "tests", "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "pcg64_host.so")
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-std=c++17",
                           "-I", os.path.join(ROOT, "diplomjourney_b200", "csrc"), "-I", cuda_inc,
                           os.path.join(ROOT, "tests", "native", "pcg64_host.cpp"), "-o", so])
    lib = ctypes.CDLL(so)
    vp, ll, i = ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int
    lib.mpcb_test_pcg64_seed.argtypes = [vp, i, vp, i, vp]
    lib.mpcb_test_pcg64_draws.argtypes = [vp, ll, vp, vp, vp, vp]
    lib.mpcb_test_pcg64_actuators.argtypes = [vp, ll, vp, vp, vp, vp]
    return lib


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _words(x):
    """SeedSequence's little-endian 32-bit words of an integer or a sequence of integers (written here from numpy's
    documentation, independently of the package's packer)."""
    if isinstance(x, (list, tuple)):
        return [w for v in x for w in _words(v)]
    w = [x & 0xFFFFFFFF]
    x >>= 32
    while x:
        w.append(x & 0xFFFFFFFF)
        x >>= 32
    return w


def _record(g):
    st = g.bit_generator.state
    s, inc = st["state"]["state"], st["state"]["inc"]
    return np.array([s >> 64, s & (2 ** 64 - 1), inc >> 64, inc & (2 ** 64 - 1), st["has_uint32"], st["uinteger"]],
                    np.uint64)


def _generator(rec):
    g = np.random.Generator(np.random.PCG64())
    r = [int(x) for x in rec]
    g.bit_generator.state = {"bit_generator": "PCG64", "state": {"state": (r[0] << 64) | r[1], "inc": (r[2] << 64) | r[3]},
                             "has_uint32": r[4], "uinteger": r[5]}
    return g


def _seeded(host, entropy_words, spawn_words):
    ent = np.array(entropy_words, np.uint32)
    sp = np.array(spawn_words, np.uint32) if len(spawn_words) else None
    rec = np.empty(6, np.uint64)
    host.mpcb_test_pcg64_seed(_p(ent), ent.size, _p(sp), 0 if sp is None else sp.size, _p(rec))
    return rec


ENTROPIES = (0, 1, 2 ** 32 - 1, 2 ** 32, 2 ** 64 + 5, 2 ** 100 + 3, 2 ** 160 + 2 ** 130 + 9, [1, 2, 3, 4, 5, 6],
             [2 ** 40, 7], [0])
SPAWN_KEYS = ((), (0,), (5,), (2 ** 32 + 1,), (3, 2 ** 33), (7, 0))


@pytest.mark.parametrize("spawn_key", SPAWN_KEYS)
@pytest.mark.parametrize("entropy", ENTROPIES, ids=str)
def test_seeding_equals_seedsequence(host, entropy, spawn_key):
    """Entropies of 1, 2, 4 and more than 4 words (integers and sequences), with no spawn key and with spawn keys of one
    or two elements (elements >= 2^32 included): the record equals Generator(PCG64(SeedSequence(...))).bit_generator.state."""
    want = _record(np.random.Generator(np.random.PCG64(np.random.SeedSequence(entropy, spawn_key=spawn_key))))
    np.testing.assert_array_equal(_seeded(host, _words(entropy), _words(list(spawn_key))), want)


def test_default_rng_and_spawn_equal_the_packer(host):
    """The package's packer (_native.pcg64_seed_words): integer seeds as default_rng(s), and SeedSequence(root).spawn(N)
    children, through the shipped seeding; the packer does not advance the SeedSequence."""
    from diplomjourney_b200 import _native as nat
    seeds = [0, 1, 2 ** 32 - 1, 2 ** 32, 2 ** 100 + 3, 123456789]
    ent, stride, spawn = nat.pcg64_seed_words(seeds, len(seeds))
    assert stride == ent.shape[1] and spawn is None
    for i, s in enumerate(seeds):
        np.testing.assert_array_equal(_seeded(host, ent[i], []), _record(np.random.default_rng(s)), err_msg=str(s))
        np.testing.assert_array_equal(nat.pcg64_record(np.random.default_rng(s).bit_generator),
                                      _record(np.random.default_rng(s)))
    for root in (np.random.SeedSequence(2024), np.random.SeedSequence(2 ** 90 + 1, spawn_key=(4,)),
                 np.random.SeedSequence([5, 6, 7, 8, 9])):
        root.spawn(3)                               # the children continue the counter
        ent, stride, spawn = nat.pcg64_seed_words(root, 5)
        assert stride == 0 and root.n_children_spawned == 3
        kids = root.spawn(5)
        for i, k in enumerate(kids):
            np.testing.assert_array_equal(_seeded(host, ent, spawn[i]), _record(np.random.default_rng(k)))


def _ops(seed, n):
    """an interleaved random() / integers() script over the actuator ranges and a one-value range"""
    r = np.random.default_rng(seed)
    ops = r.integers(0, 2, n).astype(np.int32)
    pick = r.integers(0, len(RANGES), n)
    lo = np.array([RANGES[k][0] for k in pick], np.int64)
    hi = np.array([RANGES[k][1] for k in pick], np.int64)
    return ops, lo, hi


def _run(host, rec, ops, lo, hi):
    rec = rec.copy()
    val = np.empty(ops.size)
    host.mpcb_test_pcg64_draws(_p(rec), ops.size, _p(ops), _p(lo), _p(hi), _p(val))
    return val, rec


def _numpy_run(g, ops, lo, hi):
    return np.array([g.random() if o == 0 else float(g.integers(a, b)) for o, a, b in zip(ops, lo, hi)])


@pytest.mark.parametrize("start", ["fresh", "mid_even", "mid_odd"])
@pytest.mark.parametrize("seed", [0, 7, 2 ** 63 + 11])
def test_streams_equal_numpy(host, seed, start):
    """random() and integers(lo, hi) interleaved, from a fresh state and from mid-stream states with has_uint32 = 0
    and 1: values and the final state bit for bit."""
    g = np.random.default_rng(seed)
    if start != "fresh":
        g.random(17)
        g.integers(0, 5, 4 if start == "mid_even" else 3)
    rec = _record(g)
    assert rec[4] == (1 if start == "mid_odd" else 0)
    ops, lo, hi = _ops(seed % 1000, 4000)
    val, out = _run(host, rec, ops, lo, hi)
    want = _numpy_run(g, ops, lo, hi)
    np.testing.assert_array_equal(val.view(np.uint64), want.view(np.uint64))
    np.testing.assert_array_equal(out, _record(g))


def _state_before(target, inc):
    """the state whose next step lands on ``target``: s = (target - inc) * M^-1 mod 2^128"""
    return ((target - inc) * pow(MULT, -1, 1 << 128)) & M128


@pytest.mark.parametrize("lo,hi", [(0, 5), (-100, 10), (-5, 5)])
@pytest.mark.parametrize("case", ["low_rejected", "buffer_rejected", "both_rejected"])
def test_lemire_rejection_branch(host, lo, hi, case):
    """States built to hit Lemire's rejection (probability ~range / 2^32 in a random stream): a 64-bit output whose low
    word is 0 (rejected, then the buffered high half is taken), a buffered upper half of 0 (rejected, then a new
    output), and an output of 0 (both halves rejected)."""
    rng_excl = hi - lo
    assert (2 ** 32 - rng_excl) % rng_excl > 0         # a zero word is below the threshold
    inc = (987654321 << 1) | 1
    if case == "low_rejected":
        target, has, u = 0x12345678_00000000, 0, 0     # hi = 0: output = lo, its low 32 bits 0
    elif case == "buffer_rejected":
        target, has, u = (3 << 64) | 0x1111_2222_3333_4444, 1, 0
    else:
        target, has, u = 0, 0, 0
    g = _generator([0, 0, inc >> 64, inc & (2 ** 64 - 1), has, u])
    s = _state_before(target, inc)
    st = g.bit_generator.state
    st["state"]["state"] = s
    g.bit_generator.state = st
    rec = _record(g)
    ops = np.array([1, 1, 0, 1], np.int32)
    lo_a, hi_a = np.full(4, lo, np.int64), np.full(4, hi, np.int64)
    val, out = _run(host, rec, ops, lo_a, hi_a)
    g2 = _generator(rec)
    first = g2.integers(lo, hi)
    after = g2.bit_generator.state
    if case == "low_rejected":          # the low word rejected, the buffered high half taken: one output, two words
        assert after["state"]["state"] == target and after["has_uint32"] == 0
    elif case == "buffer_rejected":     # the buffered 0 rejected, then the low half of a new output
        assert after["state"]["state"] == target and after["has_uint32"] == 1
    else:                               # both halves of the output 0 rejected: numpy stepped again
        assert after["state"]["state"] != target
    want = np.array([float(first)] + list(_numpy_run(g2, ops[1:], lo_a[1:], hi_a[1:])))
    np.testing.assert_array_equal(val.view(np.uint64), want.view(np.uint64))
    np.testing.assert_array_equal(out, _record(g2))


@pytest.mark.parametrize("seed", [0, 1, 2 ** 40 + 9])
def test_actuator_functions_equal_the_module(host, seed):
    """actual_velocity then actual_beta with PCG64, tick after tick, == the module's get_actual_velocity /
    get_actual_beta_angle driven by a numpy Generator: v_ref on both sides of the 0.4 switch, results and final state."""
    mt = importlib.import_module("diplomjourney_b200.math_model_tree")
    n = 3000
    rng = np.random.default_rng(seed % 1000 + 5)
    v_ref = rng.choice([0.0, 0.05, 0.39999999999999997, 0.4, 0.4000000000000001, 0.7, 0.995], n)
    b_ref = rng.uniform(-1.05, 1.05, n)
    g = np.random.default_rng(seed)
    g.integers(0, 5)                                    # start with a buffered half
    rec = _record(g)
    v_out, b_out = np.empty(n), np.empty(n)
    host.mpcb_test_pcg64_actuators(_p(rec), n, _p(v_ref), _p(b_ref), _p(v_out), _p(b_out))
    want_v = np.empty(n)
    want_b = np.empty(n)
    for i in range(n):
        want_v[i] = mt.get_actual_velocity(float(v_ref[i]), g)
        want_b[i] = mt.get_actual_beta_angle(float(b_ref[i]), g)
    np.testing.assert_array_equal(v_out.view(np.uint64), want_v.view(np.uint64))
    np.testing.assert_array_equal(b_out.view(np.uint64), want_b.view(np.uint64))
    np.testing.assert_array_equal(rec, _record(g))
    assert (v_out != v_ref).sum() > n // 3 and (b_out != b_ref).sum() > n // 3


def test_mirror_keeps_randomstate_behaviour():
    """With a RandomState the mirror functions draw randint as before: the same values as the reference's expressions."""
    mt = importlib.import_module("diplomjourney_b200.math_model_tree")
    a, b = np.random.RandomState(5), np.random.RandomState(5)
    for v in (0.1, 0.6) * 200:
        want = v + (b.randint(0, 5) / 1000 if v < 0.4 else b.randint(-100, 10) / 1000) if b.random() < 0.7 else v
        assert mt.get_actual_velocity(v, a) == want
    assert a.get_state()[2] == b.get_state()[2]


def test_argument_errors():
    """math_mpc_batch / Solver refuse what the PCG64 device loop cannot reproduce, before any solver is touched (the
    module's solver is replaced by an object without methods: reaching it would raise AttributeError)."""
    from diplomjourney_b200 import _native as nat
    mt = importlib.reload(importlib.import_module("diplomjourney_b200.math_model_tree"))
    mt._backend = object()
    two = [[0, 0, 0, 0, 0]] * 2
    kw = dict(isActual=True, device_noise=True)
    with pytest.raises(TypeError, match="mixes"):
        mt.math_mpc_batch(two, [[2, 3]], rngs=[np.random.default_rng(1), np.random.RandomState(2)], **kw)
    for bg in (np.random.PCG64DXSM(1), np.random.Philox(1), np.random.SFC64(1), np.random.MT19937(1)):
        with pytest.raises(TypeError, match=type(bg).__name__):
            mt.math_mpc_batch(two, [[2, 3]], rngs=[np.random.Generator(bg), np.random.default_rng(2)], **kw)
    with pytest.raises(ValueError):
        mt.math_mpc_batch(two, [[2, 3]], rngs=[np.random.default_rng(1)] * 2, seeds=np.random.SeedSequence(1), **kw)
    with pytest.raises(ValueError, match="pool_size"):
        mt.math_mpc_batch(two, [[2, 3]], seeds=np.random.SeedSequence(1, pool_size=8), **kw)
    with pytest.raises(ValueError, match="non-negative"):
        mt.math_mpc_batch(two, [[2, 3]], seeds=[1, -1], generator="pcg64", **kw)
    with pytest.raises(ValueError):                     # a SeedSequence seeds Generator(PCG64) only
        mt.math_mpc_batch(two, [[2, 3]], seeds=np.random.SeedSequence(1), generator="mt19937", **kw)
    with pytest.raises(ValueError):
        mt.math_mpc_batch(two, [[2, 3]], seeds=[1, 2], generator="philox", **kw)
    with pytest.raises(ValueError):                     # the selector is for seeds
        mt.math_mpc_batch(two, [[2, 3]], rngs=[np.random.default_rng(1)] * 2, generator="pcg64", **kw)
    with pytest.raises(ValueError):                     # one row per robot
        mt.math_mpc_batch(two, [[2, 3]], seeds=[1], generator="pcg64", **kw)
    with pytest.raises(ValueError):                     # a SeedSequence, too, runs on the device only
        mt.math_mpc_batch(two, [[2, 3]], isActual=True, seeds=np.random.SeedSequence(1))
    mt._backend = None
    with pytest.raises(ValueError, match="non-negative"):
        nat.pcg64_seed_words([5, -3], 2)
    with pytest.raises(ValueError):                     # words of different lengths above the pool size
        nat.pcg64_seed_words([1, 2 ** 200], 2)
    with pytest.raises(TypeError):
        nat.pcg64_seed_words([1.5, 2], 2)
    with pytest.raises(ValueError):
        nat.Solver.held_closed_loop(object(), None, [[0] * 5], [[2, 3]], [[0, 0]], seeds=[1],
                                    pcg_seeds=np.random.SeedSequence(1))
    with pytest.raises(ValueError):
        nat.Solver.held_closed_loop(object(), None, [[0] * 5], [[2, 3]], [[0, 0]], rng_state=np.zeros((1, 625)),
                                    pcg_state=np.zeros((1, 6), np.uint64))
    with pytest.raises(TypeError):
        nat.pcg64_record(np.random.PCG64DXSM(1))
