"""Drop-in for the reference's ``math_model_tree.py``: the online ("CoordinateTree-pruned")
controller.  Same module-level names, function signatures and log lists
(math_model_tree.py:19-717); every MPC tick is one HELD solve on the GPU.

HELD semantics (math_model_tree.py:308-361 + CoordinateTree.py:20-30): node k of layer d is
the child of node k of layer d-1, so candidate k applies control k = (v, beta) for all three
steps; S = |V|*|B| candidates, 3S node expansions.  The reference allocates a
``CoordinateTree(S)`` of S+S^2+S^3 slots per tick to hold them; here nothing is allocated.

Deliberate differences: importing does not run ``math_mpc`` twice nor open figures
(math_model_tree.py:719-941 is plotting, out of scope); ``run_default_experiment()`` performs
the two calls of math_model_tree.py:736-738.
"""
import math
import sys

import numpy as np

from . import _native
from .config import (L, beta_acc_max, beta_max, delta_beta, delta_t, delta_v,
                     eps, phi_0, v_acc_max, v_max, v_min, x_0, x_t, y_0, y_t, eps_beta)
from .CoordinateTree import CoordinateTree  # noqa: F401  (part of the module surface)

# the reference's ``from scipy import *`` (math_model_tree.py:11) shadows ``import random`` with
# numpy.random on the author's SciPy, so randint's upper bound is exclusive (SURVEY 8f)
random = np.random

# vehicle state (math_model_tree.py:19-24)
beta = 0
v = 0
phi = phi_0
x = x_0
y = y_0

prediction_horizon = 3

vector_v_no_constraint = np.round(np.arange(v, v_max + 0.1, 0.1), 3)
vector_beta_no_constraint = np.round(np.arange(-beta_max, beta_max + math.pi / 96, math.pi / 96), 3)

result_vector_x = [x]
result_vector_y = [y]
result_vector_phi = [phi]

radius_u_turn = L / np.sin(beta_max)

_backend = None     # tests may inject a CPU checker here; the product default is the CUDA library
_device = 0


def is_on_target(actual_x, actual_y, target_x, target_y):
    """[reached?, squared distance] (math_model_tree.py:48-52)."""
    d2 = (target_x - actual_x) ** 2 + (target_y - actual_y) ** 2
    return [bool(d2 <= eps), d2]


def get_distance_from_line(x_a, y_a):
    """SQUARED distance to the start->target line, 1000**2 on the line origin itself
    (math_model_tree.py:56-62)."""
    if x_a == x_0 and y_a == y_0:
        distance = 1000
    else:
        distance = abs((y_t - y_0) * x_a - (x_t - x_0) * y_a + x_t * y_0 - y_t * x_0) / \
            math.sqrt((y_t - y_0) ** 2 + (x_t - x_0) ** 2)
    return distance ** 2


def get_distance_from_target(x_a, y_a):
    return math.sqrt((x_t - x_a) ** 2 + (y_t - y_a) ** 2)


def v_x(time, _velocity, _phi):
    return _velocity * np.cos(_phi)


def v_y(time, _velocity, _phi):
    return _velocity * np.sin(_phi)


def v_phi(time, _velocity, angle_beta):
    return (_velocity / L) * math.tan(angle_beta)


def control_criterion(predicted_coordinates):
    """math_model_tree.py:82-87."""
    return 10000 * get_distance_from_target(predicted_coordinates[0], predicted_coordinates[1]) + \
        10000 * get_distance_from_line(predicted_coordinates[0], predicted_coordinates[1])


# scipy.integrate.quad over time-constant integrands (math_model_tree.py:91-108) in closed form
def integrate_velocity(velocity_function, velocity_value, _phi, t_start, t_stop):
    return velocity_function(t_start, velocity_value, _phi) * (t_stop - t_start)


def integrate_angle(angle_function, velocity_value, angle_value, t_start, t_stop):
    return angle_function(t_start, velocity_value, angle_value) * (t_stop - t_start)


def coordinate_x(_v, _phi):
    return v_x(0, _v, _phi) * delta_t


def coordinate_y(_v, _phi):
    return v_y(0, _v, _phi) * delta_t


def angle_phi(_v, _beta):
    return v_phi(0, _v, _beta) * delta_t


def iteration_of_predict(_global_coordinates, _v, _angle):
    """One bicycle-model step; returns [x, y, phi, v, beta] (math_model_tree.py:111-115)."""
    heading = _global_coordinates[2] + angle_phi(_v, _angle)
    return [_global_coordinates[0] + coordinate_x(_v, heading),
            _global_coordinates[1] + coordinate_y(_v, heading), heading, _v, _angle]


def new_target(actual_x, actual_y, actual_phi, target_x, target_y, actual_velocity):
    """The tracked line restarts at the current pose (math_model_tree.py:118-129)."""
    global x_t, y_t, x_0, y_0, phi_0
    x_t, y_t = target_x, target_y
    x_0, y_0, phi_0 = actual_x, actual_y, actual_phi
    plot_from_actual_to_target(actual_x, actual_y, actual_phi, target_x, target_y)
    slow_down(math.radians(30))


def plot_from_actual_to_target(initial_x, initial_y, initial_phi, target_x, target_y):
    """Plotting is out of scope (math_model_tree.py:132-139)."""


# Quadrant tables of turn_left / turn_right (math_model_tree.py:142-215): the synthetic target is
#   x + sx1*distance*fx1(tau) + sx2*radius_u_turn*fx2(tau),  y likewise,
# with tau = phi - offset.  Same arithmetic and evaluation order as the reference's four branches.
_LEFT = (
    (math.pi / 2, (-1, np.cos, -1, np.sin), (-1, np.sin, +1, np.cos)),
    (math.pi, (+1, np.sin, -1, np.cos), (-1, np.cos, -1, np.sin)),
    (3 * math.pi / 2, (+1, np.cos, +1, np.sin), (+1, np.sin, -1, np.cos)),
    (0.0, (-1, np.sin, +1, np.cos), (+1, np.cos, +1, np.sin)),
)
_RIGHT = (
    (math.pi / 2, (+1, np.cos, -1, np.sin), (+1, np.sin, +1, np.cos)),
    (math.pi, (-1, np.sin, -1, np.cos), (+1, np.cos, -1, np.sin)),
    (3 * math.pi / 2, (-1, np.cos, +1, np.sin), (-1, np.sin, -1, np.cos)),
    (0.0, (+1, np.sin, +1, np.cos), (-1, np.cos, +1, np.sin)),
)


def _quadrant(actual_phi):
    if math.pi / 2 <= actual_phi <= 3 * math.pi / 2:
        return 0 if actual_phi <= math.pi else 1
    return 2 if actual_phi <= 2 * math.pi else 3


def _turn(table, actual_x, actual_y, actual_phi, distance, actual_velocity):
    offset, (sx1, fx1, sx2, fx2), (sy1, fy1, sy2, fy2) = table[_quadrant(actual_phi)]
    tau = actual_phi - offset if offset else actual_phi
    target_x = actual_x + sx1 * (distance * fx1(tau)) + sx2 * (radius_u_turn * fx2(tau))
    target_y = actual_y + sy1 * (distance * fy1(tau)) + sy2 * (radius_u_turn * fy2(tau))
    new_target(actual_x, actual_y, actual_phi, target_x, target_y, actual_velocity)
    slow_down(math.radians(90))


def turn_left(actual_x, actual_y, actual_phi, distance, actual_velocity):
    _turn(_LEFT, actual_x, actual_y, actual_phi, distance, actual_velocity)


def turn_right(actual_x, actual_y, actual_phi, distance, actual_velocity):
    _turn(_RIGHT, actual_x, actual_y, actual_phi, distance, actual_velocity)


def slow_down(delta_teta):
    """0 / 10 / 20 slowed ticks by turn angle; > 90 deg leaves the counter alone
    (math_model_tree.py:219-226)."""
    global steps_for_slowing
    a = abs(delta_teta)
    if a < math.radians(10):
        steps_for_slowing = 0
    elif a <= math.radians(45):
        steps_for_slowing = 10
    elif a <= math.radians(90):
        steps_for_slowing = 20


def find_closest_value(target_value, vector_of_values):
    """Unused by the reference; kept with its (quirky) semantics (math_model_tree.py:229-236)."""
    result_value, temp = 0, sys.maxsize
    for value in vector_of_values:
        if abs(target_value - value) < temp:
            result_value, temp = value, target_value - value
    return result_value


def vector_of_velocities(actual_velocity):
    """Velocities reachable within one tick, 0 <= v < v_max (math_model_tree.py:239-246)."""
    half = (v_acc_max * delta_t) / delta_v
    window = (actual_velocity + delta_v * (i - half) for i in range(1 + 2 * int(half)))
    return [pv for pv in window if (not pv < 0) and pv < v_max]


def vector_of_beta_angles(actual_beta):
    """Steering angles reachable within one tick (math_model_tree.py:249-256)."""
    half = (math.degrees(beta_acc_max) * delta_t) / math.degrees(delta_beta)
    window = (actual_beta + delta_beta * (i - half) for i in range(1 + 2 * int(half)))
    return [pa for pa in window if abs(pa) <= (beta_max + math.radians(eps_beta))]


def _randint(rng, lo, hi):
    """randint(lo, hi) of a RandomState; a numpy Generator draws the same range with integers(lo, hi)."""
    if isinstance(rng, np.random.Generator):
        return int(rng.integers(lo, hi))
    return rng.randint(lo, hi)


def get_actual_velocity(velocity_ref, rng=None):
    """Actuator disturbance (math_model_tree.py:259-267).  ``rng``: a numpy RandomState or Generator standing in for the
    module-level generator (one per robot in ``math_mpc_batch``)."""
    rng = random if rng is None else rng
    if rng.random() < 0.7:
        if velocity_ref < 0.4:
            return velocity_ref + (_randint(rng, 0, 5) / 1000)
        return velocity_ref + (_randint(rng, -100, 10) / 1000)
    return velocity_ref


def get_actual_beta_angle(beta_ref, rng=None):
    rng = random if rng is None else rng
    if rng.random() < 0.7:
        return beta_ref + math.radians(_randint(rng, -5, 5))
    return beta_ref


def _solver():
    global _backend
    if _backend is None:
        _backend = _native.default_solver(_device)
    return _backend


def _log_names(isActual):
    pre = "actual_" if isActual else ""
    return [[pre + "predicted_trajectory_%s_anim%d" % (c, k) for k in range(3)] for c in ("x", "y", "phi")]


def predictive_control(_initial_x, _initial_y, _initial_phi, _target_x, _target_y, _vector_v,
                       _vector_beta, isActual):
    """One online MPC tick (math_model_tree.py:278-496).  As in the reference, the cost reads the
    module globals x_t, y_t, x_0, y_0 -- the target arguments are not used."""
    g = globals()
    found = None
    # an empty window has no candidate: the reference's loops do not execute, no leaf improves and the previous
    # trajectory is handed back (the np.min at math_model_tree.py:313 sits INSIDE the velocity loop)
    if np.size(_vector_beta) * np.size(_vector_v) > 0:
        slowing = g["steps_for_slowing"] > 0
        solver = _solver()
        flags = _native.FLAG_SLOW if slowing else 0
        if hasattr(solver, "held_tick"):         # the CUDA library: window lists and solve in one C call
            cost, k, traj, (v_used, beta_used) = solver.held_tick(
                _vector_v, _vector_beta, L, delta_t, v_min, _native.COST_TREE, prediction_horizon,
                (_initial_x, _initial_y, _initial_phi), (x_t, y_t), (x_0, y_0), optimal_criterion, flags)
            traj = traj.copy()
        else:                                    # a test double with the two-call interface
            solver.set_grid(_vector_v, _vector_beta, L, delta_t, v_min)
            r = solver.solve(_native.MODE_HELD, _native.COST_TREE, prediction_horizon,
                             [_initial_x, _initial_y, _initial_phi], [x_t, y_t], [x_0, y_0],
                             threshold=optimal_criterion, flags=flags)
            cost, k, traj, (v_used, beta_used) = r["cost"][0], int(r["index"][0]), r["traj"][0], r["first_control"][0]
        if k >= 0:
            if not slowing:                      # hand back the caller's own objects where possible
                v_used, beta_used = _vector_v[k // np.size(_vector_beta)], _vector_beta[k % np.size(_vector_beta)]
            found = (traj, v_used, beta_used, cost)
    return _finish_tick(g, found, isActual)


def _finish_tick(g, found, isActual):
    """Everything predictive_control does around the tree solve (math_model_tree.py:301-305,361-429), on the state
    dict ``g``: the module globals for the reference API, one dict per robot for ``math_mpc_batch``.
    ``found`` = (poses[H][3], v, beta, cost) of a leaf that beat the threshold, or None."""
    g["t"] += delta_t
    g["actual_time_arr_for_plotting" if isActual else "time_arr_for_plotting"].append(g["t"])
    if found is not None:
        traj, v_used, beta_used, cost = found
        g["optimal_trajectory"] = [[[p[0], p[1], p[2], v_used, beta_used] for p in traj]]
        g["result_v"], g["result_beta"] = v_used, beta_used
        g["optimal_criterion"] = cost
    g["steps_for_slowing"] -= 1

    best = g["optimal_trajectory"][0]
    poses = [[best[k][c] for k in range(3)] for c in range(3)]          # [x|y|phi][step]
    for names, vals in zip(_log_names(isActual), poses):
        for name, val in zip(names, vals):
            g[name].append(val)

    # finishing heuristic (math_model_tree.py:388-414): once the third predicted pose is on target,
    # the next two ticks hand out the second and then the third pose of that tick's prediction
    pick = 0
    if g["m"] == 2:
        pick = 2
    elif g["m"] == 1:
        pick = 1
        g["m"] += 1
    elif is_on_target(poses[0][2], poses[1][2], g["x_t"], g["y_t"])[0]:
        g["m"] += 1
    result_x, result_y, result_phi = poses[0][pick], poses[1][pick], poses[2][pick]
    result_v, result_beta = g["result_v"], g["result_beta"]

    if not isActual:
        g["result_trajectory_x"].append(result_x)
        g["result_trajectory_y"].append(result_y)
        g["result_trajectory_phi"].append(result_phi)
        g["result_trajectory_v"].append(result_v)
        g["result_trajectory_beta"].append(result_beta)
        g["result_trajectory_angle_speed"].append((result_v / L) * np.tan(result_beta))
    else:
        g["actual_result_trajectory_x"].append(result_x)
        g["actual_result_trajectory_y"].append(result_y)
        g["actual_result_trajectory_phi"].append(result_phi)
    g["optimal_criterion"] = sys.maxsize       # the online controller re-arms the threshold every tick
    return [result_x, result_y, result_phi, result_v, result_beta]


def add_plot_polygon(coordinates_of_vertexes):
    """Plotting is out of scope (math_model_tree.py:499-502)."""


need_scatter = False
scripted_events = True      # the demo run's operator events at ticks 1/60/90/110; set False for a plain run
# EXTENSION: math_mpc runs the whole loop in one launch of the device-resident loop (a module switch like the two above:
# a keyword would change math_mpc's signature, which is the reference's)
device_loop = False


# the programmed run's script (math_model_tree.py:564-569) in the form mpcb_held_closed_loop_events takes
DEMO_EVENTS = ((60, _native.EVENT_TURN_RIGHT, 2.0, 0.0), (90, _native.EVENT_TURN_LEFT, 2.0, 0.0),
               (110, _native.EVENT_NEW_TARGET, 2.0, 3.0))
# the actual run's script (:617-624): new_target(2, 3) after the first tick, then the programmed run's
ACTUAL_EVENTS = ((1, _native.EVENT_NEW_TARGET, 2.0, 3.0),) + DEMO_EVENTS


def _scripted_events(tick, px, py, pphi, pv, isActual):
    """Operator events of the demo run (math_model_tree.py:564-569,617-624)."""
    if not scripted_events:
        return
    if isActual and tick == 1:
        new_target(px, py, pphi, 2, 3, pv)
    if tick == 60:
        turn_right(px, py, pphi, 2, pv)
    if tick == 90:
        turn_left(px, py, pphi, 2, pv)
    if tick == 110:
        new_target(px, py, pphi, 2, 3, pv)


def math_mpc(initial_coordinates, target_coordinates, isActual):
    """Closed loop (math_model_tree.py:515-635): initial [x, y, phi, v, beta], target [x_t, y_t].
    EXTENSION: with the module switch ``device_loop = True`` the whole loop runs as ONE launch of the device-resident
    closed loop and leaves every module list and global as the per-tick run would (see ``_math_mpc_device``)."""
    global x, y, phi, x_t, y_t, v, beta, recursive, need_scatter, p, t
    if device_loop:
        return _math_mpc_device(initial_coordinates, target_coordinates, isActual)
    p, t = 1, 0
    x_t, y_t = target_coordinates[0], target_coordinates[1]
    recursive = False
    plot_from_actual_to_target(x_0, y_0, phi_0, x_t, y_t)

    px, py, pphi, pv, pbeta = (initial_coordinates[k] for k in range(5))
    x_previous, y_previous = px, py
    if not isActual:
        x, y, phi, v, beta = px, py, pphi, pv, pbeta
    while not is_on_target(px, py, x_t, y_t)[0]:
        previous_v = pv
        coordinates = predictive_control(px, py, pphi, x_t, y_t, vector_of_velocities(pv),
                                         vector_of_beta_angles(pbeta), isActual)
        px, py, pphi = coordinates[0], coordinates[1], coordinates[2]
        if isActual:
            pv = get_actual_velocity(coordinates[3])
            pbeta = get_actual_beta_angle(coordinates[4])
            actual_result_trajectory_v.append(pv)
            actual_result_trajectory_beta.append(pbeta)
            actual_result_trajectory_angle_speed.append((pv / L) * np.tan(pbeta))
        else:
            pv, pbeta = coordinates[3], coordinates[4]
            x, y, phi, v, beta = px, py, pphi, pv, pbeta
        if recursive:                            # second identical position in a row ("Recursive error.")
            break
        elif px == x_previous and py == y_previous:
            recursive = True
        _scripted_events(p, px, py, pphi, pv, isActual)
        x_previous, y_previous = px, py
        p += 1
        if not isActual:
            result_x_velocity.append(pv * np.cos(pphi))
            result_x_acceleration.append(((pv - previous_v) / delta_t) * np.cos(pphi))
            result_y_velocity.append(pv * np.sin(pphi))
            result_y_acceleration.append(((pv - previous_v) / delta_t) * np.sin(pphi))
    t = 0


# ticks math_mpc's device loop may run; the reference's loop has no bound
DEVICE_LOOP_MAX_TICKS = 4096


def _math_mpc_device(initial_coordinates, target_coordinates, isActual):
    """``math_mpc`` as one ``held_closed_loop`` launch with the trace: the loop starts from the module state
    (optimal_criterion as the first threshold, steps_for_slowing, the line x_0, y_0, the demo or actual event script
    when ``scripted_events`` is set; the actual run draws from ``np.random``), and ``_replay_trace`` rebuilds the
    module's lists and globals from the log and the trace."""
    global x, y, phi, x_t, y_t, v, beta, recursive, p, t
    from . import config as _cfg
    ini = np.array([[float(initial_coordinates[k]) for k in range(5)]])
    if m != 0:
        raise ValueError(f"math_mpc with device_loop starts with the finishing heuristic's m == 0, not {m}: the device "
                         "loop has no way to take a carried m (reset m, or set device_loop = False)")
    carried = optimal_trajectory != [[[0]]]
    if carried and not (vector_of_velocities(ini[0, 3]) and vector_of_beta_angles(ini[0, 4])):
        raise ValueError("math_mpc with device_loop: the first acceleration window is empty, so the reference would hand "
                         "back the carried optimal_trajectory, which the device loop does not hold "
                         "(set device_loop = False)")
    params = _native.LoopParams.from_config(_cfg, _native.COST_TREE, prediction_horizon, DEVICE_LOOP_MAX_TICKS)
    script = (ACTUAL_EVENTS if isActual else DEMO_EVENTS) if scripted_events else None
    kw = dict(first_threshold=[float(optimal_criterion)], slow_steps=[int(steps_for_slowing)], events=script,
              radius_u_turn=radius_u_turn, trace=True)
    tgt = [[float(target_coordinates[0]), float(target_coordinates[1])]]
    org = [[float(x_0), float(y_0)]]
    if isActual:
        r = _solver().held_closed_loop(params, ini, tgt, org, rng_state=_pack_generators([random]), **kw)
    else:
        r = _solver().held_closed_loop(params, ini, tgt, org, **kw)
    status = int(r["status"][0])
    if status == _native.LOOP_MAX_TICKS:
        raise RuntimeError(f"math_mpc with device_loop: no stop within {DEVICE_LOOP_MAX_TICKS} ticks")
    p, t = 1, 0
    x_t, y_t = target_coordinates[0], target_coordinates[1]
    recursive = False
    if not isActual:
        x, y, phi, v, beta = (initial_coordinates[k] for k in range(5))
    if status == _native.LOOP_NO_LEAF:
        if carried:
            raise ValueError("math_mpc with device_loop: no leaf beat optimal_criterion on the first tick, so the "
                             "reference would hand back the carried optimal_trajectory (set device_loop = False)")
        raise IndexError("no leaf beat optimal_criterion on the first tick: optimal_trajectory is still the placeholder")
    if isActual:                            # the draws the robot made on the device
        old = random.get_state()
        st = r["rng_state"][0]
        random.set_state((old[0], st[:624].copy(), int(st[624]), old[3], old[4]))
    k = int(r["ticks"][0])
    _replay_trace(globals(), ini[0], r["log"][0], r["pred"][0], r["control"][0], k, status, r["final"][0], script,
                  isActual)
    if not isActual and k:
        x, y, phi, v, beta = r["log"][0, k - 1]


def _replay_trace(g, init, log, pred, control, ticks, status, final, script, isActual):
    """The state ``math_mpc`` leaves in ``g`` (the module globals, or one robot's dict from ``reset_state``) when it runs
    one robot alone, rebuilt from that robot's device loop: init[5], log[ticks][5], the trace pred[ticks][H][3] and
    control[ticks][2], status, final[6] = x_t, y_t, x_0, y_0, steps_for_slowing, m, and the event script it ran with.
    Appends to g's log lists as the per-tick run appends to them (math_model_tree.py:542-635, _finish_tick)."""
    pre = "actual_" if isActual else ""
    names = _log_names(isActual)
    tt = 0
    xprev, yprev, pv_prev = init[0], init[1], init[3]
    rec, pp = False, 1
    for k in range(ticks):
        tt += delta_t
        g[pre + "time_arr_for_plotting"].append(tt)
        for c in range(3):
            for j, name in enumerate(names[c]):
                g[name].append(pred[k][j][c])
        px, py, pphi, pv, pbeta = log[k]
        cv, cb = control[k]
        g[pre + "result_trajectory_x"].append(px)
        g[pre + "result_trajectory_y"].append(py)
        g[pre + "result_trajectory_phi"].append(pphi)
        if isActual:                         # the applied (noisy) values, logged by math_mpc after the tick
            g["actual_result_trajectory_v"].append(pv)
            g["actual_result_trajectory_beta"].append(pbeta)
            g["actual_result_trajectory_angle_speed"].append((pv / L) * np.tan(pbeta))
        else:
            g["result_trajectory_v"].append(cv)
            g["result_trajectory_beta"].append(cb)
            g["result_trajectory_angle_speed"].append((cv / L) * np.tan(cb))
        if rec:                              # the "Recursive error." tick
            break
        if px == xprev and py == yprev:
            rec = True
        xprev, yprev = px, py
        pp += 1
        if not isActual:
            g["result_x_velocity"].append(pv * np.cos(pphi))
            g["result_x_acceleration"].append(((pv - pv_prev) / delta_t) * np.cos(pphi))
            g["result_y_velocity"].append(pv * np.sin(pphi))
            g["result_y_acceleration"].append(((pv - pv_prev) / delta_t) * np.sin(pphi))
        pv_prev = pv
    # every event goes through new_target, which restarts the line at the robot's pose of that tick
    fired = [e[0] for e in (script or ()) if e[0] < ticks or (e[0] == ticks and status != _native.LOOP_STALLED)]
    if fired:
        g["phi_0"] = log[max(fired) - 1][2]
    g.update(x_t=final[0], y_t=final[1], x_0=final[2], y_0=final[3], steps_for_slowing=int(final[4]), m=int(final[5]),
             p=pp, recursive=rec, t=0)
    if ticks:
        cv, cb = control[ticks - 1]
        g["optimal_trajectory"] = [[[q[0], q[1], q[2], cv, cb] for q in pred[ticks - 1]]]
        g["result_v"], g["result_beta"] = cv, cb
        g["optimal_criterion"] = sys.maxsize


def _replayed_robots(r, ini, first, script, isActual):
    """``robots`` of a device-loop result with the trace: per robot the state ``math_mpc`` leaves when it runs that robot
    alone (``_replay_trace`` on a fresh ``reset_state`` dict)."""
    robots = []
    for i in range(ini.shape[0]):
        ctx = {}
        reset_state(ctx)
        ctx.update(phi_0=phi_0, optimal_criterion=first[i])
        _replay_trace(ctx, ini[i], r["log"][i], r["pred"][i], r["control"][i], int(r["ticks"][i]), int(r["status"][i]),
                      r["final"][i], script, isActual)
        robots.append(ctx)
    return robots


_EVENT_KEYS = ("x_t", "y_t", "x_0", "y_0", "phi_0", "steps_for_slowing")


def _robot_events(ctx, tick, px, py, pphi, pv, isActual):
    """The scripted operator events for ONE robot of a batch: new_target / turn_left / turn_right / slow_down work on
    the module globals, so the robot's line, target and slow-down counter are swapped in, the event applied, and
    swapped out again (events are rare: four ticks of a run)."""
    if tick not in (1, 60, 90, 110):
        return
    g = globals()
    saved = {k: g[k] for k in _EVENT_KEYS}
    g.update({k: ctx[k] for k in _EVENT_KEYS})
    try:
        _scripted_events(tick, px, py, pphi, pv, isActual)
        ctx.update({k: g[k] for k in _EVENT_KEYS})
    finally:
        g.update(saved)


def _math_mpc_batch_ticks(ini, tgt, org, first, max_ticks, cost_kind, isActual, rngs, events):
    """The tick loop of ``math_mpc`` (math_model_tree.py:542-635) for N robots at once: per tick ONE batched device
    solve in which every robot has its own acceleration window (``mpcb_solve_held_windows``), then the reference's
    per-robot host bookkeeping -- finishing heuristic, logs, actuator noise drawn from the robot's own generator,
    stall detection, scripted events."""
    from . import config as _cfg
    n = ini.shape[0]
    params = _native.LoopParams.from_config(_cfg, _native.COST_TREE if cost_kind is None else cost_kind,
                                            prediction_horizon, max_ticks)
    robots = []
    for i in range(n):
        ctx = {}
        reset_state(ctx)
        ctx.update(x_t=tgt[i, 0], y_t=tgt[i, 1], x_0=org[i, 0], y_0=org[i, 1], phi_0=phi_0, optimal_criterion=first[i],
                   pose=[ini[i, k] for k in range(5)], previous=(ini[i, 0], ini[i, 1]), status=None, ticks=0,
                   rng=None if rngs is None else rngs[i], out=[])
        robots.append(ctx)
    solver = _solver()
    for _ in range(max_ticks):
        live = [c for c in robots if c["status"] is None]
        for c in live:
            if is_on_target(c["pose"][0], c["pose"][1], c["x_t"], c["y_t"])[0]:
                c["status"] = _native.LOOP_ON_TARGET
        live = [c for c in live if c["status"] is None]
        if not live:
            break
        r = solver.solve_held_windows(
            params, [c["pose"][:3] for c in live], [c["pose"][3:5] for c in live],
            [[c["x_t"], c["y_t"]] for c in live], [[c["x_0"], c["y_0"]] for c in live],
            threshold=[float(c["optimal_criterion"]) for c in live],
            flags=[_native.FLAG_SLOW if c["steps_for_slowing"] > 0 else 0 for c in live])
        for k, c in enumerate(live):
            found = None
            if r["index"][k] >= 0:
                found = (r["traj"][k], r["first_control"][k, 0], r["first_control"][k, 1], r["cost"][k])
            elif c["optimal_trajectory"] == [[[0]]]:
                c["status"] = _native.LOOP_NO_LEAF          # the reference raises IndexError on the placeholder
                continue
            px, py, pphi, cv, cb = _finish_tick(c, found, isActual)
            if isActual:
                pv, pbeta = get_actual_velocity(cv, c["rng"]), get_actual_beta_angle(cb, c["rng"])
                c["actual_result_trajectory_v"].append(pv)
                c["actual_result_trajectory_beta"].append(pbeta)
                c["actual_result_trajectory_angle_speed"].append((pv / L) * np.tan(pbeta))
            else:
                pv, pbeta = cv, cb
            c["pose"] = [px, py, pphi, pv, pbeta]
            c["out"].append([px, py, pphi, pv, pbeta])
            c["ticks"] += 1
            if c["recursive"]:
                c["status"] = _native.LOOP_STALLED
                continue
            if (px, py) == c["previous"]:
                c["recursive"] = True
            if events:
                _robot_events(c, c["p"], px, py, pphi, pv, isActual)
            c["previous"] = (px, py)
            c["p"] += 1
    log = np.full((n, max_ticks, 5), np.nan)
    for i, c in enumerate(robots):
        if c["status"] is None:
            c["status"] = _native.LOOP_ON_TARGET if is_on_target(c["pose"][0], c["pose"][1], c["x_t"], c["y_t"])[0] \
                else _native.LOOP_MAX_TICKS
        if c["out"]:
            log[i, :len(c["out"])] = c["out"]
    return dict(log=log, ticks=np.array([c["ticks"] for c in robots], np.int32),
                status=np.array([c["status"] for c in robots], np.int32), robots=robots)


def _pack_generators(gens):
    """[N][625] uint32: key[624] + pos of each generator's legacy MT19937 state (RandomState.get_state())."""
    out = np.empty((len(gens), 625), np.uint32)
    for i, g in enumerate(gens):
        st = g.get_state()
        out[i, :624], out[i, 624] = st[1], st[2]
    return out


def _generator_kind(rngs):
    """"mt19937" when every entry is a RandomState, "pcg64" when every entry is a Generator over PCG64; anything else
    is a TypeError that names the offending type."""
    kinds = set()
    for g in rngs:
        if isinstance(g, np.random.RandomState):
            kinds.add("mt19937")
        elif isinstance(g, np.random.Generator):
            if type(g.bit_generator) is not np.random.PCG64:
                raise TypeError("rngs entries that are numpy Generators must draw from PCG64 (np.random.default_rng), "
                                f"not {type(g.bit_generator).__name__}")
            kinds.add("pcg64")
        else:
            raise TypeError(f"rngs entries must be numpy RandomState or Generator(PCG64), not {type(g)!r}")
    if len(kinds) > 1:
        raise TypeError("rngs mixes numpy RandomState and Generator(PCG64) entries: the device loop runs one kind")
    return kinds.pop() if kinds else "mt19937"


def _math_mpc_batch_device_noise(params, ini, tgt, org, first, rngs, events, seeds=None, kind="mt19937", logs=False):
    """The actual run on the device (mpcb_held_closed_loop_actual): each robot draws from its own generator, whose state
    goes to the device as get_state() and comes back through set_state (has_gauss / cached_gaussian kept).  With
    ``seeds`` (already checked by ``_native.seed_keys``) the generators are seeded on the device and stay there.
    ``kind="pcg64"``: numpy Generator(PCG64) streams (mpcb_held_closed_loop_pcg64): the bit generators' state, inc,
    has_uint32 and uinteger go to the device and come back; ``seeds`` then is a SeedSequence or integer seeds.
    ``logs=True``: the loop also writes its trace, and the result carries ``robots`` (``_replayed_robots``)."""
    script = ACTUAL_EVENTS if events is True else list(events or ())
    kw = dict(first_threshold=first, events=script or None, radius_u_turn=radius_u_turn, trace=logs)
    if kind == "pcg64":
        if seeds is not None:
            r = _solver().held_closed_loop(params, ini, tgt, org, pcg_seeds=seeds, return_rng_state=False, **kw)
        else:
            r = _solver().held_closed_loop(params, ini, tgt, org,
                                           pcg_state=np.stack([_native.pcg64_record(g.bit_generator) for g in rngs]), **kw)
            for g, st in zip(rngs, r.pop("pcg_state")):
                g.bit_generator.state = _native.pcg64_state(st)
    elif seeds is not None:
        r = _solver().held_closed_loop(params, ini, tgt, org, seeds=seeds, return_rng_state=False, **kw)
    else:
        gens = [random] if rngs is None else rngs
        r = _solver().held_closed_loop(params, ini, tgt, org, rng_state=_pack_generators(gens), **kw)
        for g, st in zip(gens, r.pop("rng_state")):
            old = g.get_state()
            g.set_state((old[0], st[:624].copy(), int(st[624]), old[3], old[4]))
    if logs:
        r["robots"] = _replayed_robots(r, ini, first, script, True)
    return r


def _math_mpc_batch_actuator(params, ini, tgt, org, first, events, actuator):
    """The actual run with the caller's actuator model in place of get_actual_velocity / get_actual_beta_angle: the
    online controller stepped one tick at a time on the device (``mpcb_held_ctrl_step_device``), ``actuator`` run
    between two steps on the solver's stream, so that nothing waits for the device but the one read of the running
    count per step.  The committed rows (the proposal's pose with the applied v, beta) are appended to the log on the
    device."""
    import ctypes

    import torch
    solver = _solver()
    n, T = ini.shape[0], params.max_ticks
    script = ACTUAL_EVENTS if events is True else list(events or ())
    if any(int(e[1]) not in (_native.EVENT_NEW_TARGET, _native.EVENT_TURN_LEFT, _native.EVENT_TURN_RIGHT) for e in script):
        raise ValueError("event kinds are _native.EVENT_NEW_TARGET, EVENT_TURN_LEFT or EVENT_TURN_RIGHT")
    dev = torch.device("cuda", solver.device)
    f64 = dict(dtype=torch.float64, device=dev)
    with torch.cuda.device(dev), torch.cuda.stream(torch.cuda.ExternalStream(solver.stream, device=dev)):
        ini_d, tgt_d = torch.tensor(ini, **f64), torch.tensor(np.ascontiguousarray(tgt), **f64)
        org_d, first_d = torch.tensor(np.ascontiguousarray(org), **f64), torch.tensor(first, **f64)
        ctrl = torch.empty((n, ctypes.sizeof(_native.HeldCtrl)), dtype=torch.uint8, device=dev)
        log = torch.full((n, T, 5), math.nan, **f64)
        proposal, measured = torch.empty((n, 5), **f64), torch.empty((n, 5), **f64)
        running = torch.zeros(1, dtype=torch.int32, device=dev)
        count = torch.zeros(n, dtype=torch.int64, device=dev)      # rows each robot has committed
        rows = torch.arange(n, device=dev) * T
        # the script's tick s goes to the step that commits tick s, the same events for every robot
        step_events = {}
        for s in sorted({int(e[0]) for e in script}):
            todo = [e for e in script if int(e[0]) == s]
            ev = (_native.LoopEvent * len(todo))(*(_native.LoopEvent(s, int(k), float(a), float(b)) for _, k, a, b in todo))
            row = np.frombuffer(bytes(ev), np.uint8)
            step_events[s] = (torch.tensor(np.tile(row, (n, 1)), device=dev), len(todo))
        solver.held_ctrl_init_device(params, n, ini_d.data_ptr(), tgt_d.data_ptr(), org_d.data_ptr(), first_d.data_ptr(),
                                     0, ctrl.data_ptr())
        solver.held_ctrl_step_device(params, n, ctrl.data_ptr(), proposal=proposal.data_ptr(), running=running.data_ptr())
        step = 0
        while int(running.item()):
            step += 1
            mask = ~torch.isnan(proposal[:, 0])
            applied = torch.as_tensor(actuator(proposal[:, 3:5].clone(), mask), **f64).reshape(n, 2)
            measured[:, :3] = proposal[:, :3]
            measured[:, 3:] = applied
            flat, lf = rows + count.clamp(max=T - 1), log.view(-1, 5)
            lf[flat] = torch.where(mask[:, None], measured, lf[flat])
            count += mask
            running.zero_()
            ev, n_ev = step_events.get(step, (None, 0))
            solver.held_ctrl_step_device(params, n, ctrl.data_ptr(), measured.data_ptr(),
                                         0 if ev is None else ev.data_ptr(), n_ev, radius_u_turn, proposal.data_ptr(),
                                         running.data_ptr())
        rec = ctrl.cpu().numpy()
        log = log.cpu().numpy()
    d, w = rec.view(np.float64), rec.view(np.int32)
    R = _native.HeldCtrl
    line = d[:, R.line.offset // 8:R.line.offset // 8 + 4]
    final = np.concatenate([line, w[:, [R.slow_steps.offset // 4, R.m.offset // 4]].astype(np.float64)], axis=1)
    return dict(log=log, ticks=w[:, R.ticks.offset // 4].copy(), status=w[:, R.status.offset // 4].copy(), final=final)


def math_mpc_batch(initial_coordinates, target_coordinates, max_ticks=512, origin=None, cost_kind=None,
                   isActual=False, rngs=None, events=False, host_loop=False, device_noise=False, seeds=None,
                   generator=None, logs=False, actuator=None):
    """EXTENSION (not in the reference): the closed loop of ``math_mpc`` for a whole batch of robots.
    ``initial_coordinates`` [N][5] = x, y, phi, v, beta; ``target_coordinates`` [N][2].  The tracked line starts at
    the module's x_0, y_0 unless ``origin`` [N][2] is given.

    * ``isActual=False``: executed on the GPU without returning to the host between ticks (one CTA per robot,
      ``mpcb_held_closed_loop``).  ``events=True`` adds the demo run's scripted operator events (:564-569: turn_right
      at tick 60, turn_left at 90, new_target(2, 3) at 110), ``events=[(tick, kind, a, b), ...]`` any other script
      (``_native.EVENT_*``); they too are applied on the device, to each robot's own pose.  The dict then also carries
      ``final[N][6]`` = x_t, y_t, x_0, y_0, steps_for_slowing, m.
    * ``isActual=True`` (actuator noise, math_model_tree.py:259-275,590-597; ``rngs`` = one numpy RandomState per
      robot, default the module generator; ``events=True`` = the demo script, :617-624): the host draws the noise and
      applies the events between ticks, and every tick is ONE batched device solve with per-robot acceleration windows
      (``mpcb_solve_held_windows``).  The returned dict then also carries ``robots``: per robot the state and log
      lists of the reference module (``actual_result_trajectory_x`` ...).  ``host_loop=True`` takes this per-tick
      path for a noise-free run as well (events then = the demo script, applied by the module's own functions).
    * ``isActual=True, device_noise=True``: the whole noisy run in ONE launch (``mpcb_held_closed_loop_actual``): every
      robot draws from its own generator on the device, draw for draw as the per-tick path draws from it, and
      ``rngs[i]`` is left in exactly the state the per-tick path leaves it in.  ``rngs=None`` uses (and advances) the
      module generator ``np.random``, for N == 1 only: one generator shared by several robots interleaves their draws,
      which one CTA per robot cannot reproduce.  ``events=True`` is the actual run's script (new_target(2, 3) after tick
      1, then the demo script), or any ``[(tick, kind, a, b), ...]``.  Returns log, ticks, status and final as the
      noise-free device loop does (``robots`` with ``logs=True``).
    * ``isActual=True, device_noise=True, seeds=...`` in place of ``rngs``: robot i draws the stream of
      ``np.random.RandomState(seeds[i])``, seeded on the device from ``seeds`` [N] (integer seeds) or [N][K] (keys; a
      row is a key even when K == 1, see ``_native.seed_keys``).  No generator object is built and ``np.random`` is
      not touched; the generators' final states are not returned (``_native.Solver.held_closed_loop(..., seeds=)``
      returns them).  Same result keys as with ``rngs``.
    * numpy's Generator (PCG64, ``np.random.default_rng``) in place of RandomState: ``rngs`` may be all RandomState or
      all Generator(PCG64) -- on the per-tick path and with ``device_noise=True``, where the Generators are advanced
      exactly as the per-tick path advances them.  With ``device_noise=True``, ``seeds=np.random.SeedSequence(...)``
      gives robot i the stream of ``default_rng(seeds.spawn(N)[i])`` and advances ``seeds`` as ``spawn(N)`` does;
      integer ``seeds`` with ``generator="pcg64"`` give robot i ``default_rng(seeds[i])`` (without the selector
      integer seeds keep their RandomState meaning).
    * ``logs=True`` on the device paths (``isActual=False``, or ``device_noise=True``): the loop also writes what every
      tick logs besides the 5-list, and the dict carries ``pred[N][max_ticks][H][3]`` (optimal_trajectory's poses),
      ``control[N][max_ticks][2]`` (the commanded v, beta, before actuator noise), ``cost[N][max_ticks]`` and ``robots``:
      per robot the module state ``math_mpc`` leaves when it runs that robot alone -- every log list of
      ``reset_state``, p, m, recursive, steps_for_slowing, x_t, y_t, x_0, y_0, phi_0, t, optimal_trajectory, result_v,
      result_beta.  (Unlike the per-tick path's ``robots``, result_{x,y}_{velocity,acceleration} are filled, as
      ``math_mpc`` fills them.)

    * ``isActual=True, actuator=fn``: the actual run with the caller's actuator model in place of
      get_actual_velocity / get_actual_beta_angle, the controller stepped on the device one tick at a time
      (``mpcb_held_ctrl_step_device``).  ``fn(commanded, running)`` gets a float64 CUDA tensor [N][2] of this tick's
      commanded (v, beta) (NaN rows for robots without a proposal) and a bool mask of the robots with one, on the
      solver's stream, and returns the applied [N][2]; the tick commits the proposed pose with those.  Events as with
      ``device_noise``.  Returns log, ticks, status and final as the device loops do.  Not together with ``rngs``,
      ``seeds``, ``device_noise``, ``host_loop`` or ``logs``.

    Returns dict(log[N][max_ticks][5], ticks[N], status[N])."""
    if actuator is not None:
        if not isActual:
            raise ValueError("actuator= replaces the actual run's actuator noise: it needs isActual=True")
        clash = [k for k, on in (("rngs", rngs is not None), ("seeds", seeds is not None), ("device_noise", device_noise),
                                 ("host_loop", host_loop), ("logs", logs)) if on]
        if clash:
            raise ValueError(f"actuator= is the actuator model of the stepped run; it does not go with {', '.join(clash)}")
        if not callable(actuator):
            raise TypeError("actuator must be callable: fn(commanded[N][2], running[N]) -> applied[N][2]")
    from . import config as _cfg
    ini = np.asarray(initial_coordinates, dtype=np.float64).reshape(-1, 5)
    org = np.array([[x_0, y_0]], dtype=np.float64) if origin is None else np.asarray(origin, np.float64).reshape(-1, 2)
    tgt = np.asarray(target_coordinates, dtype=np.float64).reshape(-1, 2)
    n = ini.shape[0]
    kind = "mt19937"
    if generator not in (None, "mt19937", "pcg64"):
        raise ValueError(f"generator must be 'mt19937' or 'pcg64', not {generator!r}")
    if generator is not None and seeds is None:
        raise ValueError("generator= says which stream integer seeds= start; rngs= carry their own kind")
    if seeds is not None:
        if rngs is not None:
            raise ValueError("seeds and rngs both give the robots' generators: pass one of them")
        if not device_noise:
            raise ValueError("seeds seed the generators on the device: they need isActual=True, device_noise=True")
        if isinstance(seeds, np.random.SeedSequence) or generator == "pcg64":
            if generator == "mt19937":
                raise ValueError("a SeedSequence seeds numpy's Generator(PCG64), not the legacy RandomState")
            _native.pcg64_seed_words(seeds, n)          # numpy's refusals, before any solver is touched
            kind = "pcg64"
        else:
            seeds = _native.seed_keys(seeds, n)[0]
    if device_noise:
        if not isActual:
            raise ValueError("device_noise=True is the actual run's actuator noise: it needs isActual=True")
        if host_loop:
            raise ValueError("device_noise=True runs the whole loop on the device; host_loop=True is the per-tick path")
        if rngs is None and seeds is None:
            if n != 1:
                raise ValueError("rngs=None shares the module generator among the robots, which interleaves their draws; "
                                 "pass one numpy RandomState per robot (or run one robot)")
        elif rngs is not None:
            rngs = list(rngs)
            if len(rngs) != n:
                raise ValueError(f"rngs holds {len(rngs)} generators for {n} robots")
            kind = _generator_kind(rngs)
    org = np.broadcast_to(org, (n, 2))
    tgt = np.broadcast_to(tgt, (n, 2))
    # optimal_criterion before the first tick = control_criterion of the line origin (math_model_tree.py:676)
    saved = (x_t, y_t, x_0, y_0)
    g = globals()
    first = np.empty(n)
    try:
        for i in range(n):
            g.update(x_t=tgt[i, 0], y_t=tgt[i, 1], x_0=org[i, 0], y_0=org[i, 1])
            first[i] = control_criterion([org[i, 0], org[i, 1], phi_0])
    finally:
        g.update(x_t=saved[0], y_t=saved[1], x_0=saved[2], y_0=saved[3])
    params = _native.LoopParams.from_config(_cfg, _native.COST_TREE if cost_kind is None else cost_kind,
                                            prediction_horizon, max_ticks)
    if actuator is not None:
        return _math_mpc_batch_actuator(params, ini, tgt, org, first, events, actuator)
    if device_noise:
        return _math_mpc_batch_device_noise(params, ini, tgt, org, first, rngs, events, seeds, kind, logs)
    if isActual or host_loop:
        if not isinstance(events, bool) and events is not None:
            raise ValueError("a custom event script runs on the device loop only (isActual=False, host_loop=False); "
                             "the per-tick path applies the demo script (events=True) with the module's own functions")
        return _math_mpc_batch_ticks(ini, tgt, org, first, max_ticks, cost_kind, isActual, rngs, bool(events))
    script = DEMO_EVENTS if events is True else list(events or ())
    r = _solver().held_closed_loop(params, ini, tgt, org, first_threshold=first, events=script or None,
                                   radius_u_turn=radius_u_turn, trace=logs)
    if logs:
        r["robots"] = _replayed_robots(r, ini, first, script, False)
    return r


def reset_state(g=None):
    """(Re)creates the state the reference sets up at math_model_tree.py:638-717 -- in the module globals, or in the
    dict ``g`` (one robot of ``math_mpc_batch``)."""
    own = g is not None
    g = globals() if g is None else g
    g.update(t=0, dt=delta_t, time_arr_for_plotting=[0], actual_time_arr_for_plotting=[0],
             optimal_trajectory=[[[0]]], result_v=0, result_beta=0, m=0, steps_for_slowing=0,
             recursive=False, p=1)
    for pre in ("", "actual_"):
        g[pre + "result_trajectory_phi"] = [phi_0]
        g[pre + "result_trajectory_x"] = [x_0]
        g[pre + "result_trajectory_y"] = [y_0]
        for name in ("result_x_velocity", "result_x_acceleration", "result_y_velocity", "result_y_acceleration",
                     "result_trajectory_v", "result_trajectory_beta", "result_trajectory_angle_speed"):
            g[pre + name] = [0]
        for c in ("x", "y", "phi"):
            for k in range(3):
                g[pre + "predicted_trajectory_%s_anim%d" % (c, k)] = []
    for name in ("v_max_vector", "v_max_vector_minus", "v_acc_max_vector", "v_acc_max_vector_minus",
                 "beta_max_vector", "beta_max_vector_minus", "angle_speed_max_vector",
                 "angle_speed_max_vector_minus"):
        g[name] = []
    if not own:
        g["optimal_criterion"] = control_criterion([x_0, y_0, phi_0])


reset_state()


def run_default_experiment():
    """math_model_tree.py:736-738: the programmed run, then the run with actuator noise."""
    global m
    math_mpc([0, 0, 0, 0, 0], [2, 3], False)
    m = 0
    math_mpc([0, 0, 0, 0, 0], [2, 3], True)
