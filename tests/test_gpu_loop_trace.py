"""GPU: the per-tick trace of the device closed loops (mpcb_set_loop_trace) -- the predicted trajectory, the commanded
(v, beta) and the accepted cost of every tick, written by the loop kernels on out_log's row -- and what is built on it:
math_mpc with device_loop = True (the whole reference run in one launch, module lists and globals as the per-tick run
leaves them), math_mpc_batch(..., logs=True) (``robots`` from the device paths) and run_batch(..., trace=True)."""
import ctypes
import importlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# lists the per-tick batch path leaves at their reset_state value (math_mpc fills them, the device rebuild too)
NOT_ON_THE_PER_TICK_PATH = ("result_x_velocity", "result_x_acceleration", "result_y_velocity", "result_y_acceleration")


def _module():
    mt = importlib.reload(importlib.import_module("diplomjourney_b200.math_model_tree"))
    mt._backend = None
    return mt


def _random_robots(n, seed):
    rng = np.random.default_rng(seed)
    init = np.zeros((n, 5))
    init[:, :2] = rng.uniform(-1, 1, (n, 2))
    init[:, 2] = rng.uniform(-0.5, 7.0, n)
    init[:, 3] = rng.choice([0.0, 0.0, 0.3, 0.6], n)
    tgt = np.tile([2.0, 3.0], (n, 1)) + rng.uniform(-1, 1, (n, 2))
    return init, tgt, rng.integers(0, 2 ** 32, n)


def _module_state(mt):
    """Every list reset_state creates and the globals math_mpc sets, as they stand in the module."""
    g = {}
    mt.reset_state(g)
    keys = list(g) + ["p", "m", "recursive", "steps_for_slowing", "x_t", "y_t", "x_0", "y_0", "phi_0", "t",
                      "optimal_criterion", "x", "y", "phi", "v", "beta"]
    return {k: getattr(mt, k) for k in keys}


def _assert_states_close(a, b, what):
    assert a.keys() == b.keys()
    for k in a:
        if k == "optimal_trajectory":
            np.testing.assert_allclose(np.array(a[k][0], float), np.array(b[k][0], float), rtol=0, atol=1e-9,
                                       err_msg=f"{what}: {k}")
        elif isinstance(a[k], list):
            assert len(a[k]) == len(b[k]), (what, k, len(a[k]), len(b[k]))
            np.testing.assert_allclose(np.array(a[k], float), np.array(b[k], float), rtol=0, atol=1e-9,
                                       err_msg=f"{what}: {k}")
        elif k == "optimal_criterion":
            assert a[k] == pytest.approx(b[k], rel=1e-12), (what, k)
        else:
            assert a[k] == pytest.approx(b[k], abs=1e-9), (what, k, a[k], b[k])


def test_demo_run_in_one_launch(golden):
    """math_mpc([0,0,0,0,0], [2,3], False) with device_loop = True after reset_state(): held_closed_loop.json's 20 lists and
    final globals, from ONE kernel launch."""
    mt = _module()
    mt.reset_state()
    mt.device_loop = True
    mt.math_mpc([0, 0, 0, 0, 0], [2, 3], False)
    assert mt._solver().stats()["kernel_launches"] == 1
    log = golden("held_closed_loop")["log"]
    for key in [k for k in log if k != "final"]:
        got = np.array(getattr(mt, key), float)
        assert got.shape == (len(log[key]),), key
        np.testing.assert_allclose(got, log[key], rtol=0, atol=1e-9, err_msg=key)
    fin = log["final"]
    assert (mt.p, mt.m, mt.steps_for_slowing, mt.recursive) == (fin["p"], fin["m"], fin["steps_for_slowing"],
                                                                fin["recursive"])
    assert (mt.x_t, mt.y_t, mt.x_0, mt.y_0, mt.phi_0) == pytest.approx(
        (fin["x_t"], fin["y_t"], fin["x_0"], fin["y_0"], fin["phi_0"]), abs=1e-9)
    assert mt.t == 0 and mt.optimal_criterion == mt.sys.maxsize


def test_actual_run_in_one_launch(golden):
    """After np.random.seed(seed), math_mpc(..., True) with device_loop = True equals held_actual.json, leaves the module
    lists and globals the per-tick math_mpc(..., True) leaves on the GPU, and np.random in the same state."""
    for c in golden("held_actual")["cases"]:
        mt = _module()
        np.random.seed(c["seed"])
        mt.device_loop = True
        mt.math_mpc([0, 0, 0, 0, 0], [2, 3], True)
        dev, dev_rng = _module_state(mt), np.random.get_state()
        for key, ref in c["log"].items():
            np.testing.assert_allclose(np.array(getattr(mt, key), float), ref, rtol=0, atol=1e-9, err_msg=key)
        assert (mt.p, mt.m, mt.recursive) == (c["p"], c["m"], c["recursive"])
        mt = _module()
        np.random.seed(c["seed"])
        mt.math_mpc([0, 0, 0, 0, 0], [2, 3], True)
        seq, seq_rng = _module_state(mt), np.random.get_state()
        _assert_states_close(dev, seq, f"seed {c['seed']}")
        assert dev_rng[2:] == seq_rng[2:]
        np.testing.assert_array_equal(dev_rng[1], seq_rng[1])


def _recording(mt, monkeypatch):
    """_finish_tick of the per-tick path, recording per robot and tick what the trace holds."""
    inner = mt._finish_tick

    def rec(g, found, isActual):
        out = inner(g, found, isActual)
        g.setdefault("_pred", []).append([[q[0], q[1], q[2]] for q in g["optimal_trajectory"][0]])
        g.setdefault("_ctl", []).append((g["result_v"], g["result_beta"]))
        g.setdefault("_cost", []).append(np.nan if found is None else found[3])
        return out

    monkeypatch.setattr(mt, "_finish_tick", rec)


@pytest.mark.parametrize("kind", ["mt19937", "pcg64", "noise_free"])
def test_batch_logs_equal_the_per_tick_path(kind, monkeypatch):
    """256 random robots: math_mpc_batch(..., logs=True) on the device (actual run with RandomState or Generator(PCG64)
    per robot and the actual run's script; the noise-free run with the demo script) against the per-tick path on the
    same robots -- pred / control / cost equal its per-tick trajectory, command and accepted cost, and ``robots`` equal
    its ``robots`` on every list both fill."""
    mt = _module()
    nat = mt._native
    init, tgt, seeds = _random_robots(256, {"mt19937": 81, "pcg64": 82, "noise_free": 83}[kind])
    kw = dict(max_ticks=300, origin=np.zeros((256, 2)), events=True)
    if kind == "noise_free":
        d = mt.math_mpc_batch(init, tgt, logs=True, **kw)
        _recording(mt, monkeypatch)
        h = mt.math_mpc_batch(init, tgt, host_loop=True, **kw)
    else:
        make = (lambda s: np.random.RandomState(s)) if kind == "mt19937" else (lambda s: np.random.default_rng(s))
        d = mt.math_mpc_batch(init, tgt, isActual=True, rngs=[make(s) for s in seeds], device_noise=True, logs=True, **kw)
        _recording(mt, monkeypatch)
        h = mt.math_mpc_batch(init, tgt, isActual=True, rngs=[make(s) for s in seeds], **kw)
    np.testing.assert_array_equal(d["ticks"], h["ticks"])
    np.testing.assert_array_equal(d["status"], h["status"])
    np.testing.assert_allclose(d["log"], h["log"], rtol=0, atol=1e-9, equal_nan=True)
    for i, (c, r) in enumerate(zip(h["robots"], d["robots"])):
        k = int(d["ticks"][i])
        assert np.isnan(d["pred"][i, k:]).all() and np.isnan(d["control"][i, k:]).all() and np.isnan(d["cost"][i, k:]).all()
        if k:
            np.testing.assert_allclose(d["pred"][i, :k], c["_pred"], rtol=0, atol=1e-9, err_msg=str(i))
            np.testing.assert_allclose(d["control"][i, :k], c["_ctl"], rtol=0, atol=1e-9, err_msg=str(i))
            np.testing.assert_allclose(d["cost"][i, :k], c["_cost"], rtol=1e-12, atol=0, equal_nan=True, err_msg=str(i))
        if kind == "noise_free":
            np.testing.assert_array_equal(d["control"][i, :k], d["log"][i, :k, 3:5])
        for key, val in r.items():
            if isinstance(val, list) and key not in NOT_ON_THE_PER_TICK_PATH and key != "optimal_trajectory":
                assert len(val) == len(c[key]), (i, key)
                np.testing.assert_allclose(np.array(val, float), np.array(c[key], float), rtol=0, atol=1e-9,
                                           err_msg=f"robot {i}: {key}")
        same = ["p", "m", "recursive", "x_t", "y_t", "x_0", "y_0", "phi_0", "result_v", "result_beta"]
        if d["status"][i] != nat.LOOP_NO_LEAF:      # the per-tick path stops that robot before its counter moves
            same.append("steps_for_slowing")
        for key in same:
            assert r[key] == pytest.approx(c[key], abs=1e-9), (i, key, r[key], c[key])
        if k:
            np.testing.assert_allclose(np.array(r["optimal_trajectory"][0], float),
                                       np.array(c["optimal_trajectory"][0], float), rtol=0, atol=1e-9)
            if kind == "noise_free":
                assert len(r["result_x_velocity"]) == (k if d["status"][i] != nat.LOOP_STALLED else k - 1) + 1
    st = np.bincount(d["status"], minlength=4)
    assert st[nat.LOOP_ON_TARGET] >= 32 and len(set(d["ticks"].tolist())) > 20, st


def _pcg_records(seeds):
    from diplomjourney_b200 import _native as nat
    return np.stack([nat.pcg64_record(np.random.default_rng(s).bit_generator) for s in seeds])


def test_outputs_are_the_same_with_and_without_a_trace():
    """Every host entry: log, ticks, status, final and generator states bit for bit with and without a trace.  A trace
    set before a call that fails its argument checks is consumed by it: the next call writes none."""
    from diplomjourney_b200 import _native as nat, config
    mt = _module()
    n = 512
    params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, 256)
    init, tgt, seeds = _random_robots(n, 91)
    org, thr = np.zeros((n, 2)), np.full(n, 1e10)
    s = nat.Solver(0)
    ev = dict(events=mt.ACTUAL_EVENTS, radius_u_turn=mt.radius_u_turn, first_threshold=thr)
    gens = mt._pack_generators([np.random.RandomState(int(x)) for x in seeds])
    variants = {"events": dict(events=mt.DEMO_EVENTS, radius_u_turn=mt.radius_u_turn, first_threshold=thr),
                "rng_state": dict(rng_state=gens, **ev), "seeds": dict(seeds=seeds, **ev),
                "pcg_state": dict(pcg_state=_pcg_records(seeds), **ev),
                "pcg_seeds": dict(pcg_seeds=[int(x) for x in seeds], **ev)}
    for name, kw in variants.items():
        a = s.held_closed_loop(params, init, tgt, org, **kw)
        b = s.held_closed_loop(params, init, tgt, org, trace=True, **kw)
        assert set(b) - set(a) == {"pred", "control", "cost"}
        for k in a:
            np.testing.assert_array_equal(a[k], b[k], err_msg=f"{name}: {k}")
        done = np.arange(params.max_ticks)[None, :] < b["ticks"][:, None]
        assert np.isfinite(b["pred"][done]).all() and np.isnan(b["pred"][~done]).all(), name
        assert np.isfinite(b["control"][done]).all() and np.isnan(b["control"][~done]).all(), name
        if name == "events":
            np.testing.assert_array_equal(b["control"][done], b["log"][done][:, 3:5])
    # consumed by a failing call
    sentinel = [np.full((n, params.max_ticks, 3, 3), 7.0), np.full((n, params.max_ticks, 2), 7.0),
                np.full((n, params.max_ticks), 7.0)]
    bad = gens.copy()
    bad[3, 624] = 625
    s.set_loop_trace(*(x.ctypes.data for x in sentinel))
    with pytest.raises(nat.MpcbError):
        s.held_closed_loop(params, init, tgt, org, rng_state=bad, **ev)
    s.held_closed_loop(params, init, tgt, org, rng_state=gens, **ev)
    assert all((x == 7.0).all() for x in sentinel)
    s.set_loop_trace(*(x.ctypes.data for x in sentinel))
    s.set_loop_trace()                                      # cleared
    s.held_closed_loop(params, init, tgt, org, **variants["events"])
    assert all((x == 7.0).all() for x in sentinel)
    s.close()


def test_device_entries_fill_torch_tensors():
    """mpcb_held_closed_loop_device, _actual_device and _pcg64_device with a trace on torch tensors: the host entry's
    trace on every row a robot ticked, rows after its last tick left as they were."""
    torch = pytest.importorskip("torch")
    from diplomjourney_b200 import _native as nat, config
    mt = _module()
    n, T = 1024, 300
    params = nat.LoopParams.from_config(config, nat.COST_TREE, 3, T)
    init, tgt, seeds = _random_robots(n, 92)
    org, thr = np.zeros((n, 2)), np.full(n, 1e10)
    s = nat.Solver(0)
    ev = dict(events=mt.ACTUAL_EVENTS, radius_u_turn=mt.radius_u_turn)
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    d_init, d_tgt, d_org, d_thr = cuda(init), cuda(tgt), cuda(org), cuda(thr)
    gens = mt._pack_generators([np.random.RandomState(int(x)) for x in seeds])
    for name in ("noise_free", "mt19937", "pcg64"):
        out = dict(log=torch.full((n, T, 5), 7.0, dtype=torch.float64, device="cuda"),
                   pred=torch.full((n, T, 3, 3), 7.0, dtype=torch.float64, device="cuda"),
                   control=torch.full((n, T, 2), 7.0, dtype=torch.float64, device="cuda"),
                   cost=torch.full((n, T), 7.0, dtype=torch.float64, device="cuda"))
        tk, stt = (torch.empty(n, dtype=torch.int32, device="cuda") for _ in range(2))
        trace = tuple(out[k].data_ptr() for k in ("pred", "control", "cost"))
        ptr = lambda t: ctypes.c_void_p(t.data_ptr())
        torch.cuda.synchronize()
        if name == "noise_free":
            s.set_loop_trace(*trace)
            s._ck(s.lib.mpcb_held_closed_loop_device(s.h, ctypes.byref(params), n, ptr(d_init), ptr(d_tgt), ptr(d_org),
                                                     ptr(d_thr), None, ptr(out["log"]), ptr(tk), ptr(stt)))
            host = s.held_closed_loop(params, init, tgt, org, first_threshold=thr, trace=True)
        elif name == "mt19937":
            d_rng = cuda(gens.view(np.int32))
            s.held_closed_loop_device_actual(params, n, d_init.data_ptr(), d_tgt.data_ptr(), d_org.data_ptr(),
                                             d_thr.data_ptr(), 0, d_rng.data_ptr(), out["log"].data_ptr(), tk.data_ptr(),
                                             stt.data_ptr(), trace=trace, **ev)
            host = s.held_closed_loop(params, init, tgt, org, first_threshold=thr, rng_state=gens, trace=True, **ev)
        else:
            d_pcg = cuda(_pcg_records(seeds).view(np.int64))
            s.held_closed_loop_device_pcg64(params, n, d_init.data_ptr(), d_tgt.data_ptr(), d_org.data_ptr(),
                                            d_thr.data_ptr(), 0, d_pcg.data_ptr(), out["log"].data_ptr(), tk.data_ptr(),
                                            stt.data_ptr(), trace=trace, **ev)
            host = s.held_closed_loop(params, init, tgt, org, first_threshold=thr, pcg_state=_pcg_records(seeds),
                                      trace=True, **ev)
        s.sync()
        ticks = tk.cpu().numpy()
        np.testing.assert_array_equal(ticks, host["ticks"])
        done = np.arange(T)[None, :] < ticks[:, None]
        for k in ("log", "pred", "control", "cost"):
            got = out[k].cpu().numpy()
            np.testing.assert_array_equal(got[done], host[k][done], err_msg=f"{name}: {k}")
            assert (got[~done] == 7.0).all(), (name, k)
    s.close()


def test_full_batch_trace_equals_the_per_tick_solves(golden):
    """run_batch(..., trace=True) on 64 seeded scenarios of the 5 x 7 grid: pred is the per-tick predictive_control's
    optimal_trajectory on every tick, stall ticks (the previous path again) included; control is the log's v, beta, and
    cost the accepted leaf's cost (NaN on a stall)."""
    rm = importlib.import_module("diplomjourney_b200.run_math_model")
    case = [c for c in golden("full_h3")["cases"] if c["grid"] == "g5x7"][0]
    rm._backend = None
    rm._grid_key = None
    rm.vector_v, rm.vector_beta = np.array(case["vector_v"]), np.array(case["vector_beta"])
    rng = np.random.default_rng(5)
    n, T = 64, 120
    sc = np.zeros((n, 5))
    sc[:, :2] = rng.uniform(-1, 1, (n, 2))
    sc[:, 2] = rng.uniform(-0.5, 7.0, n)
    sc[:, 3:5] = sc[:, :2] + rng.uniform(0.3, 1.5, (n, 2)) * rng.choice([-1, 1], (n, 2))
    r = rm.run_batch(sc, max_ticks=T, trace=True)
    H = rm.prediction_horizon
    assert r["pred"].shape == (n, T, H, 3) and r["control"].shape == (n, T, 2) and r["cost"].shape == (n, T)
    stalls = compared = 0
    for i in range(n):
        k = int(r["ticks"][i])
        assert np.isnan(r["pred"][i, k:]).all() and np.isnan(r["cost"][i, k:]).all()
        np.testing.assert_array_equal(r["control"][i, :k], r["log"][i, :k, 3:5])
        rm.reset_scenario(*sc[i])
        x, y, phi = sc[i, :3]
        for t in range(k):
            before = rm.optimal_criterion
            ret = rm.predictive_control(x, y, phi, 0, rm.x_t, rm.y_t)
            if not np.allclose(ret[:3], r["log"][i, t, :3], rtol=0, atol=1e-9):
                break                            # a knife-edge tie decided the other way: stop comparing this robot
            want = np.array([[q[0], q[1], q[2]] for q in rm.optimal_trajectory[0]], float)
            np.testing.assert_allclose(r["pred"][i, t], want, rtol=0, atol=1e-9, err_msg=f"scenario {i} tick {t}")
            accepted = rm.optimal_criterion != before
            assert np.isnan(r["cost"][i, t]) == (not accepted), (i, t)
            if accepted:
                assert r["cost"][i, t] == pytest.approx(rm.optimal_criterion, rel=1e-12)
            stalls += not accepted
            compared += 1
            x, y, phi = ret[:3]
    assert compared >= 0.9 * r["ticks"].sum() and stalls > 0, (compared, stalls)
    rm._backend = None
