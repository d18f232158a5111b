"""GPU: the actual run (math_mpc(..., True), actuator noise) with its generators SEEDED ON THE DEVICE from numpy seeds --
math_mpc_batch(..., device_noise=True, seeds=), Solver.held_closed_loop(seeds=) / mpcb_held_closed_loop_seeded_host,
mpcb_rng_seed_device -- and the device-pointer entry mpcb_held_closed_loop_actual_device on torch tensors.  Robot i must
draw exactly the stream of np.random.RandomState(seeds[i]): every result equals the rngs= path (generators built by
numpy, handed over with get_state / set_state) bit for bit, and the generators end in the same states."""
import ctypes
import importlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KEYS = ("actual_result_trajectory_x", "actual_result_trajectory_y", "actual_result_trajectory_phi",
        "actual_result_trajectory_v", "actual_result_trajectory_beta")
OUT = ("ticks", "status", "log", "final")


def _module():
    mt = importlib.reload(importlib.import_module("diplomjourney_b200.math_model_tree"))
    mt._backend = None
    return mt


def _record(rs):
    st = rs.get_state()
    return np.concatenate([st[1].astype(np.uint32), np.array([st[2]], np.uint32)])


def _random_robots(n, seed):
    rng = np.random.default_rng(seed)
    init = np.zeros((n, 5))
    init[:, :2] = rng.uniform(-1, 1, (n, 2))
    init[:, 2] = rng.uniform(-0.5, 7.0, n)
    init[:, 3] = rng.choice([0.0, 0.0, 0.3, 0.6], n)
    tgt = np.tile([2.0, 3.0], (n, 1)) + rng.uniform(-1, 1, (n, 2))
    seeds = rng.integers(0, 2 ** 32, n)
    seeds[:2] = (0, 2 ** 32 - 1)
    return init, tgt, seeds


def _assert_same(a, b, keys=OUT):
    for k in keys:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)     # NaN rows included


def test_reference_seeds_in_one_launch(golden):
    """The seeds of held_actual.json (and a few more) as ONE batch with seeds=: the reference's logs at 1e-9, and
    bit for bit what rngs=[RandomState(s)] gives."""
    mt = _module()
    nat = mt._native
    cases = golden("held_actual")["cases"]
    seeds = [c["seed"] for c in cases] + [3, 23, 77, 0, 2 ** 32 - 1]
    n = len(seeds)
    init, tgt, org = np.zeros((n, 5)), np.tile([2.0, 3.0], (n, 1)), np.zeros((n, 2))
    before = np.random.get_state()
    d = mt.math_mpc_batch(init, tgt, max_ticks=400, origin=org, isActual=True, events=True, device_noise=True,
                          seeds=seeds)
    after = np.random.get_state()
    assert after[2] == before[2] and np.array_equal(after[1], before[1])          # np.random untouched
    assert sorted(d) == sorted(OUT)
    r = mt.math_mpc_batch(init, tgt, max_ticks=400, origin=org, isActual=True, events=True, device_noise=True,
                          rngs=[np.random.RandomState(s) for s in seeds])
    _assert_same(d, r)
    for i, c in enumerate(cases):
        ref = np.array([c["log"][k][1:] for k in KEYS], dtype=float).T
        assert d["ticks"][i] == c["p"] - 1 == ref.shape[0]
        np.testing.assert_allclose(d["log"][i, :ref.shape[0]], ref, rtol=0, atol=1e-9)
        assert np.isnan(d["log"][i, ref.shape[0]:]).all()
        assert d["final"][i, 5] == c["m"]
        assert d["status"][i] == (nat.LOOP_STALLED if c["recursive"] else nat.LOOP_ON_TARGET)


@pytest.mark.parametrize("events", [True, False, "custom"])
def test_random_batch_seeds_equal_rngs(events, monkeypatch):
    """256 random robots (seeds 0 and 2^32 - 1 among them) with the actual script, without events and with a custom
    script: seeds= equals rngs= (log, ticks, status, final), and the states Solver.held_closed_loop(seeds=) returns equal
    the RandomState objects after the rngs= run."""
    mt = _module()
    nat = mt._native
    init, tgt, seeds = _random_robots(256, {True: 21, False: 22, "custom": 23}[events])
    org = np.zeros((256, 2))
    if events == "custom":
        events = [(3, nat.EVENT_TURN_LEFT, 1.5, 0.0), (25, nat.EVENT_NEW_TARGET, 1.0, -2.0),
                  (25, nat.EVENT_TURN_RIGHT, 1.0, 0.0), (40, nat.EVENT_NEW_TARGET, -1.5, 2.5)]
    gens = [np.random.RandomState(s) for s in seeds]
    r = mt.math_mpc_batch(init, tgt, max_ticks=300, origin=org, isActual=True, events=events, device_noise=True,
                          rngs=gens)
    seen = {}
    plain = nat.Solver.held_closed_loop

    def keep_states(self, *a, **kw):               # the call math_mpc_batch makes, with the final states kept
        kw["return_rng_state"] = True
        seen.update(plain(self, *a, **kw))
        return seen

    monkeypatch.setattr(nat.Solver, "held_closed_loop", keep_states)
    d = mt.math_mpc_batch(init, tgt, max_ticks=300, origin=org, isActual=True, events=events, device_noise=True,
                          seeds=seeds)
    _assert_same(d, r)
    np.testing.assert_array_equal(seen["rng_state"], np.stack([_record(g) for g in gens]))
    st = np.bincount(d["status"], minlength=4)
    assert st[nat.LOOP_ON_TARGET] >= 32 and len(set(d["ticks"].tolist())) > 20, st


@pytest.mark.parametrize("K", [1, 2, 624, 700])
def test_keys_equal_randomstate_of_the_row(K):
    """[N][K] keys: robot i draws RandomState(list(keys[i])) -- also for K == 1, where RandomState(int) is another
    stream; log, ticks, status, final and the final generator states equal the rng_state= path's."""
    from diplomjourney_b200 import _native as nat, config
    mt = _module()
    params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, 200)
    n = 64
    init, tgt, _ = _random_robots(n, 30 + K)
    keys = np.random.default_rng(K).integers(0, 2 ** 32, (n, K), dtype=np.uint64)
    keys[0, 0], keys[1, -1] = 0, 2 ** 32 - 1
    s = nat.Solver(0)
    kw = dict(first_threshold=1e10, events=mt.ACTUAL_EVENTS, radius_u_turn=mt.radius_u_turn)
    d = s.held_closed_loop(params, init, tgt, [[0.0, 0.0]], seeds=keys, **kw)
    packed = mt._pack_generators([np.random.RandomState(row.tolist()) for row in keys])
    r = s.held_closed_loop(params, init, tgt, [[0.0, 0.0]], rng_state=packed, **kw)
    _assert_same(d, r, OUT + ("rng_state",))
    if K == 1:
        w = s.held_closed_loop(params, init, tgt, [[0.0, 0.0]], seeds=keys[:, 0], **kw)
        assert not np.array_equal(w["rng_state"], d["rng_state"])
    s.close()


def _torch():
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available()
    return torch


def _u32(torch, a):
    """a uint32 numpy array as an int32 CUDA tensor of the same bits"""
    return torch.from_numpy(np.ascontiguousarray(a, np.uint32).view(np.int32)).cuda()


def _host_u32(t):
    return t.cpu().numpy().view(np.uint32)


@pytest.mark.parametrize("key_len", [0, 3])
def test_seeding_kernel_65536_generators(key_len):
    """mpcb_rng_seed_device at N = 65,536 (164 MB of records): a spread sample of 512 records, the last included, equals
    RandomState(seed).get_state()."""
    from diplomjourney_b200 import _native as nat
    torch = _torch()
    n = 65536
    rng = np.random.default_rng(40 + key_len)
    keys = rng.integers(0, 2 ** 32, (n, key_len) if key_len else n, dtype=np.uint64).astype(np.uint32)
    keys.flat[0], keys.flat[-1] = 2 ** 32 - 1, 0
    s = nat.Solver(0)
    d_keys = _u32(torch, keys)
    out = torch.full((n, 625), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    s.seed_generators_device(n, d_keys.data_ptr(), key_len, out.data_ptr())
    s.sync()
    got = _host_u32(out)
    for i in np.unique(np.r_[np.linspace(0, n - 1, 512).astype(np.int64), n - 1]):
        seed = keys[i].tolist() if key_len else int(keys[i])
        np.testing.assert_array_equal(got[i], _record(np.random.RandomState(seed)), err_msg=f"generator {i}")
    s.close()


def test_device_entries_on_torch_tensors():
    """Seeding + mpcb_held_closed_loop_actual_device on torch tensors: bit for bit the seeded host entry; a second run
    from new starts on the same device state buffer equals the rng_state= path run twice with the same RandomState
    objects; a record with pos = 1000 behaves as pos = 624."""
    from diplomjourney_b200 import _native as nat, config
    torch = _torch()
    mt = _module()
    n, ticks = 512, 300
    params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, ticks)
    init, tgt, seeds = _random_robots(n, 50)
    init2 = _random_robots(n, 51)[0]
    org = np.zeros((n, 2))
    thr = np.full(n, 1e10)
    ev = dict(events=mt.ACTUAL_EVENTS, radius_u_turn=mt.radius_u_turn)
    s = nat.Solver(0)
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    d_tgt, d_org, d_thr = cuda(tgt), cuda(org), cuda(thr)
    d_rng = torch.empty((n, 625), dtype=torch.int32, device="cuda")
    d_keys = _u32(torch, seeds.astype(np.uint32))

    def run(start, rng_state):
        log = torch.full((n, ticks, 5), float("nan"), dtype=torch.float64, device="cuda")
        tk = torch.empty(n, dtype=torch.int32, device="cuda")
        stt = torch.empty(n, dtype=torch.int32, device="cuda")
        fin = torch.empty((n, 6), dtype=torch.float64, device="cuda")
        d_init = cuda(start)
        torch.cuda.synchronize()
        s.held_closed_loop_device_actual(params, n, d_init.data_ptr(), d_tgt.data_ptr(), d_org.data_ptr(),
                                         d_thr.data_ptr(), 0, rng_state.data_ptr(), log.data_ptr(), tk.data_ptr(),
                                         stt.data_ptr(), fin.data_ptr(), **ev)
        s.sync()
        return dict(log=log.cpu().numpy(), ticks=tk.cpu().numpy(), status=stt.cpu().numpy(), final=fin.cpu().numpy(),
                    rng_state=_host_u32(rng_state).copy())

    torch.cuda.synchronize()
    s.seed_generators_device(n, d_keys.data_ptr(), 0, d_rng.data_ptr())
    first = run(init, d_rng)
    host = s.held_closed_loop(params, init, tgt, org, first_threshold=thr, seeds=seeds, **ev)
    _assert_same(first, host, OUT + ("rng_state",))
    second = run(init2, d_rng)                       # chained: the generators continue on the device

    gens = [np.random.RandomState(x) for x in seeds]
    for start, want in ((init, first), (init2, second)):
        r = s.held_closed_loop(params, start, tgt, org, first_threshold=thr, rng_state=mt._pack_generators(gens), **ev)
        for g, st in zip(gens, r["rng_state"]):
            g.set_state(("MT19937", st[:624].copy(), int(st[624])))
        _assert_same(want, r, OUT + ("rng_state",))
    assert (second["ticks"] > 0).all() and not np.array_equal(first["rng_state"], second["rng_state"])

    # pos = 1000 twists before its first draw, as pos = 624 does (every robot here draws at least once)
    fresh = mt._pack_generators([np.random.RandomState(x) for x in seeds])
    odd = fresh.copy()
    odd[::2, 624] = 1000
    a, b = run(init, _u32(torch, fresh)), run(init, _u32(torch, odd))
    assert (a["ticks"] > 0).all()
    _assert_same(a, b, OUT + ("rng_state",))
    s.close()


def test_seeding_abi_rejections():
    """The entries' argument errors are MPCB_ERR_INVALID; N == 0 is OK and launches nothing."""
    from diplomjourney_b200 import _native as nat, config
    torch = _torch()
    s = nat.Solver(0)
    lib = s.lib
    keys = torch.zeros(8, dtype=torch.int32, device="cuda")
    out = torch.zeros((8, 625), dtype=torch.int32, device="cuda")
    k, o = ctypes.c_void_p(keys.data_ptr()), ctypes.c_void_p(out.data_ptr())
    for N, kp, kl, op in ((4, k, -1, o), (4, k, 4097, o), (4, None, 0, o), (4, k, 0, None), (-1, k, 0, o)):
        assert lib.mpcb_rng_seed_device(s.h, N, kp, kl, op) == -1, (N, kl)
    assert lib.mpcb_rng_seed_device(s.h, 0, None, 0, None) == 0
    assert lib.mpcb_rng_seed_device(s.h, 2, k, 4, o) == 0
    s.sync()

    params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, 16)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    ini, tg, og = dev(np.zeros((1, 5))), dev(np.array([[2.0, 3.0]])), dev(np.zeros((1, 2)))
    log = torch.empty((1, 16, 5), dtype=torch.float64, device="cuda")
    tk, st = torch.empty(1, dtype=torch.int32, device="cuda"), torch.empty(1, dtype=torch.int32, device="cuda")
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    bad_kind = (nat.LoopEvent * 1)(nat.LoopEvent(1, 9, 0.0, 0.0))
    torch.cuda.synchronize()
    for N, events, n_ev, rng in ((1, None, 0, None), (1, bad_kind, 1, o), (1, None, -1, o), (-1, None, 0, o)):
        rc = lib.mpcb_held_closed_loop_actual_device(s.h, ctypes.byref(params), N, p(ini), p(tg), p(og), None, None,
                                                     events, n_ev, 0.0, rng, p(log), p(tk), p(st), None)
        assert rc == -1, (N, n_ev)
    h_ini, h_tg, h_og = np.zeros((1, 5)), np.array([[2.0, 3.0]]), np.zeros((1, 2))
    h_log, h_tk, h_st = np.empty((1, 16, 5)), np.empty(1, np.int32), np.empty(1, np.int32)
    hp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    h_keys = np.zeros(1, np.uint32)
    for kp, kl in ((None, 0), (hp(h_keys), 4097), (hp(h_keys), -2)):
        rc = lib.mpcb_held_closed_loop_seeded_host(s.h, ctypes.byref(params), 1, hp(h_ini), hp(h_tg), hp(h_og), None,
                                                   None, None, 0, 0.0, kp, kl, None, hp(h_log), hp(h_tk), hp(h_st), None)
        assert rc == -1, kl
    with pytest.raises(ValueError):                  # one source of generators
        s.held_closed_loop(params, h_ini, h_tg, h_og, seeds=[1], rng_state=np.zeros((1, 625), np.uint32))
    s.close()
