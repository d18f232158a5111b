"""GPU: the "actual" run of the online controller (math_mpc(..., True), actuator noise from numpy.random) as ONE launch
of the device-resident closed loop, math_mpc_batch(..., isActual=True, device_noise=True) /
mpcb_held_closed_loop_actual_host.  Every robot draws from its own RandomState on the device; the results must equal
the reference's seeded runs and the per-tick path (one batched solve per tick, noise drawn on the host by the module's
own get_actual_velocity / get_actual_beta_angle), and every generator must end in the very state the per-tick path
leaves it in -- which pins the number of words each robot consumed."""
import ctypes
import importlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KEYS = ("actual_result_trajectory_x", "actual_result_trajectory_y", "actual_result_trajectory_phi",
        "actual_result_trajectory_v", "actual_result_trajectory_beta")


def _module():
    mt = importlib.reload(importlib.import_module("diplomjourney_b200.math_model_tree"))
    mt._backend = None
    return mt


def _generators(seeds, pos=None):
    gens = [np.random.RandomState(s) for s in seeds]
    if pos is not None:                                  # same keys, another stream position
        for g, p in zip(gens, pos):
            g.set_state(("MT19937", g.get_state()[1], int(p)))
    return gens


def _assert_same_generators(a, b):
    for i, (ga, gb) in enumerate(zip(a, b)):
        sa, sb = ga.get_state(), gb.get_state()
        assert sa[2] == sb[2], (i, sa[2], sb[2])
        np.testing.assert_array_equal(sa[1], sb[1], err_msg=f"robot {i}")


def _random_robots(n, seed):
    rng = np.random.default_rng(seed)
    init = np.zeros((n, 5))
    init[:, :2] = rng.uniform(-1, 1, (n, 2))
    init[:, 2] = rng.uniform(-0.5, 7.0, n)
    init[:, 3] = rng.choice([0.0, 0.0, 0.3, 0.6], n)
    tgt = np.tile([2.0, 3.0], (n, 1)) + rng.uniform(-1, 1, (n, 2))
    return init, tgt, rng.integers(0, 2 ** 32, n)


def _device_equals_per_tick(mt, init, tgt, seeds, events, max_ticks=300, pos=None, host_events=None):
    """The device path and the per-tick path on the same robots and seeds: identical ticks, status and final
    generator states; logs and final line/target/slow-down/m at the existing 1e-9 bar."""
    n = init.shape[0]
    org = np.zeros((n, 2))
    dev_g, host_g = _generators(seeds, pos), _generators(seeds, pos)
    d = mt.math_mpc_batch(init, tgt, max_ticks=max_ticks, origin=org, isActual=True, rngs=dev_g, events=events,
                          device_noise=True)
    h = mt.math_mpc_batch(init, tgt, max_ticks=max_ticks, origin=org, isActual=True, rngs=host_g,
                          events=events if host_events is None else host_events)
    np.testing.assert_array_equal(d["ticks"], h["ticks"])
    np.testing.assert_array_equal(d["status"], h["status"])
    np.testing.assert_allclose(d["log"], h["log"], rtol=0, atol=1e-9, equal_nan=True)
    for i, c in enumerate(h["robots"]):
        want = [c["x_t"], c["y_t"], c["x_0"], c["y_0"], c["steps_for_slowing"], c["m"]]
        cols = [0, 1, 2, 3, 5] if h["status"][i] == mt._native.LOOP_NO_LEAF else list(range(6))
        # (the per-tick path stops a no-leaf robot before its slow-down counter is decremented; the loop after it)
        np.testing.assert_allclose(d["final"][i, cols], np.array(want, float)[cols], rtol=0, atol=1e-9, err_msg=str(i))
    _assert_same_generators(dev_g, host_g)
    assert "robots" not in d
    return d


def test_reference_seeded_runs_in_one_launch(golden):
    """Both reference runs (held_actual.json: 195 and 198 ticks, all four operator events, well over 624 words each, so
    the generators twist on the device) plus extra seeds, as ONE batch; the extra seeds also against the per-tick path."""
    mt = _module()
    nat = mt._native
    cases = golden("held_actual")["cases"]
    seeds = [c["seed"] for c in cases] + [3, 23, 77, 2 ** 32 - 1]
    n = len(seeds)
    init, tgt = np.zeros((n, 5)), np.tile([2.0, 3.0], (n, 1))
    d = _device_equals_per_tick(mt, init, tgt, seeds, True, max_ticks=400)
    for i, c in enumerate(cases):
        ref = np.array([c["log"][k][1:] for k in KEYS], dtype=float).T
        assert d["ticks"][i] == c["p"] - 1 == ref.shape[0]
        np.testing.assert_allclose(d["log"][i, :ref.shape[0]], ref, rtol=0, atol=1e-9)
        assert np.isnan(d["log"][i, ref.shape[0]:]).all()
        assert d["final"][i, 5] == c["m"]
        assert d["status"][i] == (nat.LOOP_STALLED if c["recursive"] else nat.LOOP_ON_TARGET)


@pytest.mark.parametrize("events", [True, False, "custom"])
def test_random_batch_equals_the_per_tick_path(events, monkeypatch):
    """256 robots with random starts, targets, speeds and seeds, with the actual run's event script, without events,
    and with a custom script (on the per-tick path applied by the module's own turn_left / new_target / turn_right)."""
    mt = _module()
    nat = mt._native
    init, tgt, seeds = _random_robots(256, {True: 1, False: 2, "custom": 3}[events])
    if events == "custom":
        script = [(3, nat.EVENT_TURN_LEFT, 1.5, 0.0), (25, nat.EVENT_NEW_TARGET, 1.0, -2.0), (25, nat.EVENT_TURN_RIGHT, 1.0, 0.0),
                  (40, nat.EVENT_NEW_TARGET, -1.5, 2.5)]
        fns = {nat.EVENT_NEW_TARGET: lambda px, py, pphi, a, b, pv: mt.new_target(px, py, pphi, a, b, pv),
               nat.EVENT_TURN_LEFT: lambda px, py, pphi, a, b, pv: mt.turn_left(px, py, pphi, a, pv),
               nat.EVENT_TURN_RIGHT: lambda px, py, pphi, a, b, pv: mt.turn_right(px, py, pphi, a, pv)}

        def robot_events(ctx, tick, px, py, pphi, pv, isActual):      # _robot_events with the custom script
            todo = [e for e in script if e[0] == tick]
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
        d = _device_equals_per_tick(mt, init, tgt, seeds, script, host_events=True)
        assert (d["ticks"] > 40).sum() >= 8
    else:
        d = _device_equals_per_tick(mt, init, tgt, seeds, events)
        if events:
            assert (d["ticks"] > 110).sum() >= 4
    st = np.bincount(d["status"], minlength=4)
    assert st[nat.LOOP_ON_TARGET] >= 32 and len(set(d["ticks"].tolist())) > 20, st


def test_one_robot_on_the_module_generator(golden):
    """N = 1 with rngs=None after np.random.seed(seed): the reference's run, and np.random ends in the state a
    sequential math_mpc([0,0,0,0,0], [2,3], True) leaves it in.  Two robots on the one module generator are refused."""
    mt = _module()
    c = golden("held_actual")["cases"][0]
    np.random.seed(c["seed"])
    d = mt.math_mpc_batch([[0, 0, 0, 0, 0]], [[2, 3]], max_ticks=400, origin=[[0, 0]], isActual=True, events=True,
                          device_noise=True)
    after_device = np.random.get_state()
    ref = np.array([c["log"][k][1:] for k in KEYS], dtype=float).T
    assert d["ticks"][0] == c["p"] - 1 == ref.shape[0]
    np.testing.assert_allclose(d["log"][0, :ref.shape[0]], ref, rtol=0, atol=1e-9)
    mt.x_0, mt.y_0, mt.phi_0 = 0, 0, 0
    mt.reset_state()
    np.random.seed(c["seed"])
    mt.math_mpc([0, 0, 0, 0, 0], [2, 3], True)
    after_sequential = np.random.get_state()
    assert after_device[2] == after_sequential[2] and after_device[3:] == after_sequential[3:]
    np.testing.assert_array_equal(after_device[1], after_sequential[1])
    np.testing.assert_allclose(d["log"][0, :ref.shape[0], 0], np.array(mt.actual_result_trajectory_x[1:], float),
                               rtol=0, atol=1e-9)
    with pytest.raises(ValueError):
        mt.math_mpc_batch([[0, 0, 0, 0, 0]] * 2, [[2, 3]], isActual=True, device_noise=True)


def test_generators_about_to_twist_and_stalling_robots():
    """Generators that start at pos 620..624 (a twist within the first tick or two, on the device) and robots that
    stall: the tick that ends in the repeated-position stop still draws, as the per-tick path does."""
    mt = _module()
    nat = mt._native
    init, tgt, seeds = _random_robots(96, 7)
    pos = 620 + np.arange(96) % 5
    d = _device_equals_per_tick(mt, init, tgt, seeds, False, pos=pos)
    assert (d["status"] == nat.LOOP_STALLED).sum() >= 8 and (d["status"] == nat.LOOP_ON_TARGET).sum() >= 8


def test_many_robots_per_cta_with_generators():
    """4,096 robots (several per CTA, each CTA reloads its shared generator per robot) == the same robots in slices of
    64, generators included; the caller's rng_state array is not modified."""
    from diplomjourney_b200 import _native as nat, config
    mt = _module()
    params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, 256)
    init, tgt, seeds = _random_robots(4096, 11)
    st = mt._pack_generators(_generators(seeds))
    st[::7, 624] = np.arange(0, 4096, 7) % 625
    st0 = st.copy()
    s = nat.Solver(0)
    big = s.held_closed_loop(params, init, tgt, [[0.0, 0.0]], first_threshold=1e10, rng_state=st)
    np.testing.assert_array_equal(st, st0)
    assert (big["rng_state"][:, 624] != st0[:, 624]).mean() > 0.9
    for lo in range(0, 4096, 512):
        part = s.held_closed_loop(params, init[lo:lo + 64], tgt[lo:lo + 64], [[0.0, 0.0]], first_threshold=1e10,
                                  rng_state=st[lo:lo + 64])
        for k in ("ticks", "status", "log", "final", "rng_state"):
            np.testing.assert_array_equal(big[k][lo:lo + 64], part[k], err_msg=k)
    assert nat.LOOP_ON_TARGET in set(big["status"].tolist())
    s.close()


def test_actual_entry_rejects_bad_generator_states():
    """mpcb_held_closed_loop_actual_host: a null rng_state or a pos outside [0, 624] is MPCB_ERR_INVALID."""
    from diplomjourney_b200 import _native as nat, config
    mt = _module()
    params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, 16)
    s = nat.Solver(0)
    st = mt._pack_generators(_generators([1, 2]))
    st[1, 624] = 625
    with pytest.raises(nat.MpcbError) as e:
        s.held_closed_loop(params, np.zeros((2, 5)), [[2.0, 3.0]], [[0.0, 0.0]], rng_state=st)
    assert e.value.code == -1 and "robot 1" in str(e.value)
    ini, tg, og = np.zeros((1, 5)), np.array([[2.0, 3.0]]), np.zeros((1, 2))
    log, ticks, status = np.empty((1, 16, 5)), np.empty(1, np.int32), np.empty(1, np.int32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    rc = s.lib.mpcb_held_closed_loop_actual_host(s.h, ctypes.byref(params), 1, p(ini), p(tg), p(og), None, None, None, 0,
                                                 0.0, None, p(log), p(ticks), p(status), None)
    assert rc == -1
    s.close()
