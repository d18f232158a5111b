"""Shared body of ``math_model`` and ``run_math_model`` (the reference keeps two copies of the
same functions: math_model.py:40-231 and run_math_model.py:42-228).

``install(g)`` defines the reference's function surface inside the module namespace ``g``.
All state stays where the reference keeps it -- module globals of the installing module
(``optimal_criterion``, ``optimal_trajectory``, ``t``, ``x_t`` ...) -- so user code that
rebinds ``math_model.x_t`` or reads ``math_model.optimal_criterion`` keeps working.

The scalar helpers are closed forms of the reference's expressions; ``predictive_control``
hands the whole tree to the CUDA library (no CPU fallback).
"""
from __future__ import annotations

import math

import numpy as np

from . import _native


def default_grids(g):
    """math_model.py:23-30: absolute grids, rounded to 3 decimals."""
    vector_v = np.round(np.arange(g["v"], g["v_max"] + g["delta_v"], g["delta_v"]), 3)
    vector_beta = np.round(np.arange(-g["beta_max"], g["beta_max"] + g["delta_beta"], g["delta_beta"]), 3)
    return vector_v, vector_beta


def install(g, placeholder_trajectory):
    def is_on_target(actual_x, actual_y, target_x, target_y):
        # math_model.py:40-44
        return bool((target_x - actual_x) ** 2 + (target_y - actual_y) ** 2 <= g["eps"])

    def get_distance_from_line(x_a, y_a):
        # math_model.py:48-54 (1000 when the point IS the line origin)
        if x_a == g["x_0"] and y_a == g["y_0"]:
            return 1000
        x_t, y_t, x_0, y_0 = g["x_t"], g["y_t"], g["x_0"], g["y_0"]
        return abs((y_t - y_0) * x_a - (x_t - x_0) * y_a + x_t * y_0 - y_t * x_0) / \
            math.sqrt((y_t - y_0) ** 2 + (x_t - x_0) ** 2)

    def get_distance_from_target(x_a, y_a):
        return math.sqrt((g["x_t"] - x_a) ** 2 + (g["y_t"] - y_a) ** 2)

    def saturation(value, value_mplt):
        return max(-value_mplt, min(value_mplt, value))

    def v_x(time, _velocity, _phi):
        return _velocity * np.cos(_phi)

    def v_y(time, _velocity, _phi):
        return _velocity * np.sin(_phi)

    def v_phi(time, _velocity, angle_beta):
        return (_velocity / g["L"]) * math.tan(angle_beta)

    def control_criterion(predicted_coordinates):
        # math_model.py:82-86
        angle_from_line = np.arctan(g["x_t"] / g["y_t"]) - predicted_coordinates[2]
        d = get_distance_from_target(predicted_coordinates[0], predicted_coordinates[1])
        dl = get_distance_from_line(predicted_coordinates[0], predicted_coordinates[1])
        return 10000 * d + 10 * angle_from_line ** 2 + 100 * dl ** 2

    # The reference integrates time-constant integrands with scipy.integrate.quad
    # (math_model.py:90-107); the integral is integrand * (t_stop - t_start).
    def integrate_velocity(velocity_function, velocity_value, _phi, t_start, t_stop):
        return velocity_function(t_start, velocity_value, _phi) * (t_stop - t_start)

    def integrate_angle(angle_function, velocity_value, angle_value, t_start, t_stop):
        return angle_function(t_start, velocity_value, angle_value) * (t_stop - t_start)

    def coordinate_x(_v, _phi):
        return v_x(0, _v, _phi) * g["delta_t"]

    def coordinate_y(_v, _phi):
        return v_y(0, _v, _phi) * g["delta_t"]

    def angle_phi(_v, _beta):
        return v_phi(0, _v, _beta) * g["delta_t"]

    def iteration_of_predict(_global_coordinates, _v, _angle):
        # math_model.py:110-114
        _phi = angle_phi(_v, _angle)
        heading = _global_coordinates[2] + _phi
        return [_global_coordinates[0] + coordinate_x(_v, heading),
                _global_coordinates[1] + coordinate_y(_v, heading), heading]

    def _solver():
        s = g.get("_backend")
        if s is None:
            s = g["_backend"] = _native.default_solver(g.get("_device", 0))
        key = (tuple(np.asarray(g["vector_v"], float)), tuple(np.asarray(g["vector_beta"], float)),
               g["L"], g["delta_t"])
        if g.get("_grid_key") != key or getattr(s, "_owner", None) is not g:
            s.set_grid(g["vector_v"], g["vector_beta"], g["L"], g["delta_t"], 0.0)
            g["_grid_key"] = key
            s._owner = g
        return s

    def predictive_control(_initial_x, _initial_y, _initial_phi, _initial_velocity, _target_x, _target_y):
        """One MPC tick on the FULL tree (math_model.py:136-231).  As in the reference the
        target arguments are ignored: the cost reads the module globals x_t, y_t, x_0, y_0."""
        g["t"] += g["delta_t"]
        x_t, y_t, x_0, y_0 = g["x_t"], g["y_t"], g["x_0"], g["y_0"]
        x_t / y_t                                                   # ZeroDivisionError like math_model.py:83
        1 / math.sqrt((y_t - y_0) ** 2 + (x_t - x_0) ** 2)          # ... and math_model.py:52-53
        H = g["prediction_horizon"]
        r = _solver().solve(_native.MODE_FULL, _native.COST_MM, H, [_initial_x, _initial_y, _initial_phi],
                            [x_t, y_t], [x_0, y_0], threshold=g["optimal_criterion"])
        if r["index"][0] >= 0:                                      # strict '<' against the carried optimum
            traj = r["traj"][0]
            v0, b0 = r["first_control"][0]
            first = np.array([traj[0, 0], traj[0, 1], traj[0, 2], v0, b0])
            g["optimal_trajectory"] = [np.array([first] + [traj[k].copy() for k in range(1, H)], dtype=object)]
            g["optimal_criterion"] = r["cost"][0]
            g["last_leaf_index"] = int(r["index"][0])
        # otherwise the previously accepted path is returned again (stall; math_model.py:217-221)
        best = g["optimal_trajectory"][0][0]
        return [best[0], best[1], best[2], best[3], best[4]]

    def leaf_cloud(_initial_x, _initial_y, _initial_phi, leaf_begin=0, count=None):
        """Terminal (x, y) and cost of every leaf in enumeration order -- the data behind the
        reference's green scatter of ``third_field_x/y`` (math_model.py:192-193,204).  Small trees
        only (16 bytes per leaf come back to the host)."""
        xy, cost = _solver().dump_leaves(_native.MODE_FULL, _native.COST_MM, g["prediction_horizon"],
                                         [_initial_x, _initial_y, _initial_phi], [g["x_t"], g["y_t"]],
                                         [g["x_0"], g["y_0"]], leaf_begin=leaf_begin, count=count)
        return xy[:, 0], xy[:, 1], cost

    def run_scenario(max_ticks=None, verbose=False):
        """The closed loop of math_model.py:234-254: tick until on target, stop after the
        position repeated twice ("Recursive error")."""
        x, y, phi, v, beta = g["x"], g["y"], g["phi"], g["v"], g["beta"]
        x_previous, y_previous = x, y
        k, p, path = 0, 1, [(x, y, phi)]
        while not is_on_target(x, y, g["x_t"], g["y_t"]):
            x, y, phi, v, beta = predictive_control(x, y, phi, v, g["x_t"], g["y_t"])
            path.append((x, y, phi))
            if x == x_previous and y == y_previous:
                k += 1
            if k == 2:
                if verbose:
                    print("Recursive error")
                break
            x_previous, y_previous = x, y
            if verbose:
                print("Iteration number = " + str(p))
            p += 1
            if max_ticks is not None and p > max_ticks:
                break
        g.update(x=x, y=y, phi=phi, v=v, beta=beta)
        return path

    def run_batch(scenarios, max_ticks=256, trace=False):
        """EXTENSION (not in the reference): the closed loop of run_math_model.py:233-276 for a whole batch of
        scenarios at once -- rows of [x_0, y_0, phi_0, x_t, y_t]; the tracked line starts at each robot's start
        pose and ``optimal_criterion`` is seeded from it, as run_math_model.py:251-252 does.  Every tick is ONE
        batched FULL solve on the GPU with the carried thresholds; per-robot bookkeeping (repeat counter,
        is_on_target) stays on the device.  Returns dict(log[N][max_ticks][5], ticks[N], status[N]); ``trace=True``
        adds per tick pred[N][max_ticks][H][3] (the poses of optimal_trajectory, the previous path again on a stall),
        control[N][max_ticks][2] and cost[N][max_ticks] (NaN on a stall)."""
        sc = np.asarray(scenarios, dtype=np.float64).reshape(-1, 5)
        first = np.empty(sc.shape[0])
        for i, (sx, sy, sphi, tx, ty) in enumerate(sc):
            ang = np.arctan(tx / ty) - sphi
            first[i] = 10000 * math.sqrt((tx - sx) ** 2 + (ty - sy) ** 2) + 10 * ang ** 2 + 100 * 1000 ** 2
        return _solver().full_closed_loop(_native.COST_MM, g["prediction_horizon"], sc[:, :3], sc[:, 3:5], sc[:, :2],
                                          first_threshold=first, eps=g["eps"], max_ticks=max_ticks, trace=trace)

    def reset_scenario(x_0, y_0, phi_0, x_t, y_t):
        """run_math_model.py:233-252: new start/target, optimum re-seeded from the start pose."""
        g.update(x_0=x_0, y_0=y_0, phi_0=phi_0, x_t=x_t, y_t=y_t, x=x_0, y=y_0, phi=phi_0, v=0, beta=0, t=0)
        g["optimal_trajectory"] = list(placeholder_trajectory)
        g["optimal_criterion"] = control_criterion([x_0, y_0, phi_0])

    for name, fn in list(locals().items()):
        if callable(fn) and not name.startswith("_") and name not in ("g",):
            fn.__module__ = g.get("__name__", fn.__module__)
            g[name] = fn
    g["optimal_trajectory"] = list(placeholder_trajectory)
    g["optimal_criterion"] = control_criterion([g["x_0"], g["y_0"], g["phi_0"]])
