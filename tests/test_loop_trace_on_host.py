"""CPU: the host side of the closed loops' per-tick trace.  ``math_model_tree._replay_trace`` rebuilds the module state
``math_mpc`` leaves (every log list, p, m, recursive, steps_for_slowing, the line, optimal_trajectory ...) from what the
device loop returns -- log, trace (pred, control), final and the event script.  Fed with the reference's own lists, or
with a sequential math_mpc on the oracle backend whose commands are captured per tick, it must give that very state back."""
import importlib

import numpy as np
import pytest

from oracle_backend import OracleBackend

FIVE = ("result_trajectory_x", "result_trajectory_y", "result_trajectory_phi", "result_trajectory_v",
        "result_trajectory_beta")


def _module():
    mt = importlib.reload(importlib.import_module("diplomjourney_b200.math_model_tree"))
    mt._backend = OracleBackend()
    return mt


def _fresh(mt):
    ctx = {}
    mt.reset_state(ctx)
    ctx.update(phi_0=mt.phi_0, optimal_criterion=mt.optimal_criterion)
    return ctx


def test_programmed_run_from_the_reference_lists(golden):
    """held_closed_loop.json (151 ticks, turn_right / turn_left / new_target): log, pred, control and final built from
    the reference's lists give back all 20 of its lists and its final globals."""
    mt = _module()
    nat = mt._native
    log = golden("held_closed_loop")["log"]
    fin = log["final"]
    rows = np.array([log[k][1:] for k in FIVE], float).T
    T = rows.shape[0]
    pred = np.array([[[log[f"predicted_trajectory_{c}_anim{j}"][k] for c in ("x", "y", "phi")] for j in range(3)]
                     for k in range(T)])
    final = [fin["x_t"], fin["y_t"], fin["x_0"], fin["y_0"], fin["steps_for_slowing"], fin["m"]]
    g = _fresh(mt)
    mt._replay_trace(g, [0, 0, 0, 0, 0], rows, pred, rows[:, 3:5], T, nat.LOOP_ON_TARGET, final, mt.DEMO_EVENTS, False)
    lists = [k for k in log if k != "final"]
    assert len(lists) == 20
    for key in lists:
        got = np.array(g[key], float)
        assert got.shape == (len(log[key]),), key
        np.testing.assert_allclose(got, log[key], rtol=0, atol=1e-9, err_msg=key)
    assert (g["p"], g["m"], g["steps_for_slowing"], g["recursive"]) == \
        (fin["p"], fin["m"], fin["steps_for_slowing"], fin["recursive"])
    assert (g["x_0"], g["y_0"], g["phi_0"]) == pytest.approx((fin["x_0"], fin["y_0"], fin["phi_0"]), abs=1e-9)
    assert g["t"] == 0 and g["optimal_criterion"] == mt.sys.maxsize
    np.testing.assert_array_equal(np.array(g["optimal_trajectory"][0])[:, :3], pred[-1])
    assert (g["result_v"], g["result_beta"]) == (rows[-1, 3], rows[-1, 4])


def _sequential_with_trace(mt, monkeypatch, init, target, isActual):
    """math_mpc(init, target, isActual) on the oracle backend with predictive_control wrapped: per tick the commanded
    (v, beta) it returns and the poses of optimal_trajectory it leaves -- what the device loop's trace holds."""
    pred, control = [], []
    inner = mt.predictive_control

    def traced(*a):
        r = inner(*a)
        control.append((r[3], r[4]))
        pred.append([[q[0], q[1], q[2]] for q in mt.optimal_trajectory[0]])
        return r

    monkeypatch.setattr(mt, "predictive_control", traced)
    mt.math_mpc(init, target, isActual)
    return np.array(pred, float), np.array(control, float)


def _assert_state_equal(mt, g):
    """Every entry of the rebuilt state equals the module global of the same name, lists element for element."""
    for key, val in g.items():
        want = getattr(mt, key)
        if key == "optimal_trajectory":
            np.testing.assert_array_equal(np.array(val[0], float), np.array(want[0], float), err_msg=key)
        elif isinstance(val, list):
            assert len(val) == len(want), key
            np.testing.assert_array_equal(np.array(val, float), np.array(want, float), err_msg=key)
        else:
            assert val == want, (key, val, want)


@pytest.mark.parametrize("case", ["actual", "stall", "short"])
def test_sequential_run_is_rebuilt_exactly(case, golden, monkeypatch):
    """The actual run of held_actual.json (actuator noise, all four events, seed 5), the 'Recursive error' stall of
    held_short_loops.json (the stop tick still logs, p does not advance) and an event-free short run: the state rebuilt
    from log, trace and final equals the module state of the sequential run, every list and global."""
    mt = _module()
    nat = mt._native
    isActual = case == "actual"
    if isActual:
        c = golden("held_actual")["cases"][0]
        np.random.seed(c["seed"])
        init, target = [0, 0, 0, 0, 0], [2, 3]
    else:
        c = golden("held_short_loops")["cases"][3 if case == "stall" else 0]
        assert c["recursive"] == (case == "stall")
        init, target = list(c["init"]), list(c["target"])
    g = _fresh(mt)
    pred, control = _sequential_with_trace(mt, monkeypatch, init, target, isActual)
    pre = "actual_" if isActual else ""
    rows = np.array([getattr(mt, pre + k)[1:] for k in FIVE], float).T
    T = rows.shape[0]
    assert pred.shape == (T, 3, 3) and control.shape == (T, 2)
    if not isActual:
        np.testing.assert_array_equal(control, rows[:, 3:5])
    status = nat.LOOP_STALLED if mt.recursive else nat.LOOP_ON_TARGET
    final = [mt.x_t, mt.y_t, mt.x_0, mt.y_0, mt.steps_for_slowing, mt.m]
    mt._replay_trace(g, init, rows, pred, control, T, status, final, mt.ACTUAL_EVENTS if isActual else mt.DEMO_EVENTS,
                     isActual)
    _assert_state_equal(mt, g)
    if isActual:
        assert (g["p"], g["m"], g["recursive"]) == (c["p"], c["m"], c["recursive"])
    else:
        assert (g["p"] - 1, g["m"], g["recursive"], g["steps_for_slowing"]) == \
            (c["ticks"], c["m"], c["recursive"], c["steps_for_slowing"])


def test_device_loop_refuses_states_it_cannot_start_from():
    """math_mpc with device_loop = True refuses a carried m and a carried optimal_trajectory with an empty first window before
    any solver is touched."""
    mt = _module()
    mt._backend = None                       # nothing may reach a solver
    mt.device_loop = True
    mt.m = 1
    with pytest.raises(ValueError, match="m == 0"):
        mt.math_mpc([0, 0, 0, 0, 0], [2, 3], False)
    mt.m = 0
    mt.optimal_trajectory = [[[0.1, 0.2, 0.3, 0.5, 0.0]] * 3]
    with pytest.raises(ValueError, match="empty"):
        mt.math_mpc([0, 0, 0, 5.0, 0], [2, 3], False)
    assert mt._backend is None
