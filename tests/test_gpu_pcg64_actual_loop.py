"""GPU: the actual run (math_mpc(..., True), actuator noise) with numpy's Generator(PCG64) streams on the device --
math_mpc_batch(..., device_noise=True) with rngs=[default_rng(...)], seeds=SeedSequence(...), integer seeds with
generator="pcg64", Solver.held_closed_loop(pcg_state= / pcg_seeds=), and the device-pointer entries
mpcb_pcg64_seed_device / mpcb_held_closed_loop_pcg64_device on torch tensors.  Robot i must draw exactly the stream its
Generator draws on the per-tick path: ticks, status and every Generator's final bit_generator.state are equal, logs and
final rows at the per-tick comparison's 1e-9 bar (as for the RandomState run); device paths among themselves are equal bit
for bit, NaN rows included."""
import copy
import importlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

OUT = ("ticks", "status", "log", "final")


def _module():
    mt = importlib.reload(importlib.import_module("diplomjourney_b200.math_model_tree"))
    mt._backend = None
    return mt


def _random_robots(n, seed):
    rng = np.random.default_rng(seed)
    init = np.zeros((n, 5))
    init[:, :2] = rng.uniform(-1, 1, (n, 2))
    init[:, 2] = rng.uniform(-0.5, 7.0, n)
    init[:, 3] = rng.choice([0.0, 0.0, 0.3, 0.6], n)          # speeds on both sides of 0.4 m/s
    tgt = np.tile([2.0, 3.0], (n, 1)) + rng.uniform(-1, 1, (n, 2))
    seeds = [int(s) for s in rng.integers(0, 2 ** 63, n)]
    seeds[:3] = (0, 2 ** 32 - 1, 2 ** 100 + 3)
    return init, tgt, seeds


def _states(gens):
    return [g.bit_generator.state for g in gens]


def _assert_same(a, b, keys=OUT):
    for k in keys:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)     # NaN rows included


CUSTOM = [(3, 3, 1.5, 0.0), (25, 1, 1.0, -2.0), (25, 3, 1.0, 0.0), (40, 1, -1.5, 2.5)]


@pytest.mark.parametrize("events", [True, "custom"])
def test_generators_equal_the_per_tick_path(events, monkeypatch):
    """256 robots, default_rng(seed) each: device_noise=True against the per-tick path with copies of the same
    Generators (the custom script applied on the per-tick path by the module's own turn / new_target functions)."""
    mt = _module()
    nat = mt._native
    init, tgt, seeds = _random_robots(256, {True: 61, "custom": 62}[events])
    org = np.zeros((256, 2))
    dev_g = [np.random.default_rng(s) for s in seeds]
    for g in dev_g[::3]:
        g.integers(0, 5)                                  # some start with a buffered half
    host_g = copy.deepcopy(dev_g)
    script, host_events = (events, events) if events is True else (CUSTOM, True)
    if events == "custom":
        fns = {nat.EVENT_NEW_TARGET: lambda px, py, pphi, a, b, pv: mt.new_target(px, py, pphi, a, b, pv),
               nat.EVENT_TURN_LEFT: lambda px, py, pphi, a, b, pv: mt.turn_left(px, py, pphi, a, pv),
               nat.EVENT_TURN_RIGHT: lambda px, py, pphi, a, b, pv: mt.turn_right(px, py, pphi, a, pv)}

        def robot_events(ctx, tick, px, py, pphi, pv, isActual):      # _robot_events with the custom script
            todo = [e for e in CUSTOM if e[0] == tick]
            if not todo:
                return
            g = vars(mt)
            saved = {k: g[k] for k in mt._EVENT_KEYS}
            g.update({k: ctx[k] for k in mt._EVENT_KEYS})
            try:
                for _, kind, a, b in todo:
                    fns[kind](px, py, pphi, a, b, pv)
                ctx.update({k: g[k] for k in mt._EVENT_KEYS})
            finally:
                g.update(saved)

        monkeypatch.setattr(mt, "_robot_events", robot_events)
    d = mt.math_mpc_batch(init, tgt, max_ticks=300, origin=org, isActual=True, rngs=dev_g, events=script,
                          device_noise=True)
    h = mt.math_mpc_batch(init, tgt, max_ticks=300, origin=org, isActual=True, rngs=host_g, events=host_events)
    np.testing.assert_array_equal(d["ticks"], h["ticks"])
    np.testing.assert_array_equal(d["status"], h["status"])
    np.testing.assert_allclose(d["log"], h["log"], rtol=0, atol=1e-9, equal_nan=True)
    assert (np.isnan(d["log"]) == np.isnan(h["log"])).all()
    for i, c in enumerate(h["robots"]):
        want = [c["x_t"], c["y_t"], c["x_0"], c["y_0"], c["steps_for_slowing"], c["m"]]
        cols = [0, 1, 2, 3, 5] if h["status"][i] == nat.LOOP_NO_LEAF else list(range(6))
        np.testing.assert_allclose(d["final"][i, cols], np.array(want, float)[cols], rtol=0, atol=1e-9, err_msg=str(i))
    assert _states(dev_g) == _states(host_g)
    assert len({s["has_uint32"] for s in _states(dev_g)}) == 2           # both buffer states handed back
    st = np.bincount(d["status"], minlength=4)
    assert st[nat.LOOP_ON_TARGET] >= 32 and len(set(d["ticks"].tolist())) > 20, st


def test_seedsequence_and_integer_seeds_equal_rngs():
    """seeds=SeedSequence(root) equals rngs=[default_rng(c) for c in SeedSequence(root).spawn(N)] and advances root's
    n_children_spawned by N (a second call continues with the next children); integer seeds with generator="pcg64"
    equal rngs=[default_rng(s)]."""
    mt = _module()
    n = 256
    init, tgt, seeds = _random_robots(n, 63)
    kw = dict(max_ticks=300, origin=np.zeros((n, 2)), isActual=True, events=True, device_noise=True)
    root = np.random.SeedSequence(20241021, spawn_key=(7,))
    for call in range(2):
        before = root.n_children_spawned
        d = mt.math_mpc_batch(init, tgt, seeds=root, **kw)
        assert root.n_children_spawned == before + n
        kids = np.random.SeedSequence(20241021, spawn_key=(7,)).spawn(before + n)[before:]
        r = mt.math_mpc_batch(init, tgt, rngs=[np.random.default_rng(k) for k in kids], **kw)
        _assert_same(d, r)
    d = mt.math_mpc_batch(init, tgt, seeds=seeds, generator="pcg64", **kw)
    gens = [np.random.default_rng(s) for s in seeds]
    r = mt.math_mpc_batch(init, tgt, rngs=gens, **kw)
    _assert_same(d, r)
    legacy = mt.math_mpc_batch(init, tgt, seeds=[s % 2 ** 32 for s in seeds], **kw)      # integer seeds stay legacy
    assert not np.array_equal(legacy["log"], d["log"], equal_nan=True)


def test_solver_states_and_device_entries_on_torch_tensors():
    """Solver.held_closed_loop(pcg_seeds=) returns the states the rngs= path leaves; mpcb_pcg64_seed_device +
    mpcb_held_closed_loop_pcg64_device on torch tensors, chained twice on the same state buffer, equal the host entry run
    twice with the state it hands back -- results and states bit for bit."""
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available()
    from diplomjourney_b200 import _native as nat, config
    mt = _module()
    n, ticks = 512, 300
    params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, ticks)
    init, tgt, seeds = _random_robots(n, 64)
    init2 = _random_robots(n, 65)[0]
    org, thr = np.zeros((n, 2)), np.full(n, 1e10)
    ev = dict(events=mt.ACTUAL_EVENTS, radius_u_turn=mt.radius_u_turn)
    s = nat.Solver(0)
    root = np.random.SeedSequence(99)
    ent, stride, spawn = nat.pcg64_seed_words(root, n)
    host = s.held_closed_loop(params, init, tgt, org, first_threshold=thr, pcg_seeds=root, **ev)
    gens = [np.random.default_rng(c) for c in np.random.SeedSequence(99).spawn(n)]
    r = s.held_closed_loop(params, init, tgt, org, first_threshold=thr,
                           pcg_state=np.stack([nat.pcg64_record(g.bit_generator) for g in gens]), **ev)
    _assert_same(host, r, OUT + ("pcg_state",))
    host2 = s.held_closed_loop(params, init2, tgt, org, first_threshold=thr, pcg_state=host["pcg_state"], **ev)

    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    d_tgt, d_org, d_thr = cuda(tgt), cuda(org), cuda(thr)
    d_ent = cuda(ent.view(np.int32))
    d_spawn = cuda(spawn.view(np.int32))
    d_pcg = torch.full((n, 6), -1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    s.seed_pcg64_device(n, d_ent.data_ptr(), ent.size, stride, d_spawn.data_ptr(), spawn.shape[1], d_pcg.data_ptr())
    s.sync()
    seeded = d_pcg.cpu().numpy().view(np.uint64)
    np.testing.assert_array_equal(seeded, np.stack([nat.pcg64_record(np.random.default_rng(c).bit_generator)
                                                    for c in np.random.SeedSequence(99).spawn(n)]))

    def run(start):
        log = torch.full((n, ticks, 5), float("nan"), dtype=torch.float64, device="cuda")
        tk = torch.empty(n, dtype=torch.int32, device="cuda")
        stt = torch.empty(n, dtype=torch.int32, device="cuda")
        fin = torch.empty((n, 6), dtype=torch.float64, device="cuda")
        d_init = cuda(start)
        torch.cuda.synchronize()
        s.held_closed_loop_device_pcg64(params, n, d_init.data_ptr(), d_tgt.data_ptr(), d_org.data_ptr(),
                                        d_thr.data_ptr(), 0, d_pcg.data_ptr(), log.data_ptr(), tk.data_ptr(),
                                        stt.data_ptr(), fin.data_ptr(), **ev)
        s.sync()
        return dict(log=log.cpu().numpy(), ticks=tk.cpu().numpy(), status=stt.cpu().numpy(), final=fin.cpu().numpy(),
                    pcg_state=d_pcg.cpu().numpy().view(np.uint64).copy())

    first = run(init)
    _assert_same(first, host, OUT + ("pcg_state",))
    second = run(init2)                                   # chained: the generators continue on the device
    _assert_same(second, host2, OUT + ("pcg_state",))
    assert (second["ticks"] > 0).all() and not np.array_equal(first["pcg_state"], second["pcg_state"])
    s.close()


def test_pcg64_abi_rejections():
    """The PCG64 entries' argument errors are MPCB_ERR_INVALID, checked before anything is copied; N == 0 is OK."""
    import ctypes
    torch = pytest.importorskip("torch")
    from diplomjourney_b200 import _native as nat, config
    s = nat.Solver(0)
    lib = s.lib
    ent = torch.zeros(8, dtype=torch.int32, device="cuda")
    out = torch.zeros((8, 6), dtype=torch.int64, device="cuda")
    e, o = ctypes.c_void_p(ent.data_ptr()), ctypes.c_void_p(out.data_ptr())
    for N, ep, el, es, sp, sl, op in ((4, e, 0, 0, None, 0, o), (4, e, 4097, 0, None, 0, o), (4, e, 2, 3, None, 0, o),
                                      (4, e, 2, 0, None, 1, o), (4, e, 2, 0, e, -1, o), (4, None, 2, 0, None, 0, o),
                                      (4, e, 2, 0, None, 0, None), (-1, e, 2, 0, None, 0, o)):
        assert lib.mpcb_pcg64_seed_device(s.h, N, ep, el, es, sp, sl, op) == -1, (N, el, es, sl)
    assert lib.mpcb_pcg64_seed_device(s.h, 0, None, 1, 0, None, 0, None) == 0
    assert lib.mpcb_pcg64_seed_device(s.h, 2, e, 2, 2, e, 2, o) == 0
    s.sync()
    params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, 16)
    good = nat.pcg64_record(np.random.default_rng(1).bit_generator)
    for i, bad in ((4, 2), (5, 2 ** 32), (3, int(good[3]) ^ 1)):
        st = good.copy()
        st[i] = bad
        with pytest.raises(nat.MpcbError):
            s.held_closed_loop(params, np.zeros((1, 5)), [[2.0, 3.0]], [[0.0, 0.0]], pcg_state=st[None])
    r = s.held_closed_loop(params, np.zeros((1, 5)), [[2.0, 3.0]], [[0.0, 0.0]], pcg_state=good[None])
    assert r["ticks"][0] > 0
    s.close()
