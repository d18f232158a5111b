"""GPU: the online controller stepped one tick at a time on per-robot records in device memory
(mpcb_held_ctrl_init_device / mpcb_held_ctrl_step_device), so that a caller's plant closes the loop.  With the identity
plant the steps are the device closed loop bit for bit; with numpy's noise drawn on the host they are the actual run;
with per-robot events each robot is its own one-robot loop; with a plant that moves the robot the steps equal a host loop
built from the per-tick solve and the module's own bookkeeping."""
import ctypes
import importlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _module():
    mt = importlib.reload(importlib.import_module("diplomjourney_b200.math_model_tree"))
    mt._backend = None
    return mt


def _nat():
    from diplomjourney_b200 import _native
    return _native


def _params(H=3, cost=None, max_ticks=256):
    from diplomjourney_b200 import config
    nat = _nat()
    return nat.LoopParams.from_config(config, nat.COST_TREE if cost is None else cost, H, max_ticks)


def _robots(n, seed):
    """Random robots, plus: two on target at entry, two that find no leaf on their first tick (first threshold -1), and
    two that face away from their target on the tracked line with v = 0, so that standing still is their best move and
    they stall.  Returns init, target, origin, first threshold."""
    rng = np.random.default_rng(seed)
    init = np.zeros((n + 6, 5))
    init[:n, :2] = rng.uniform(-1, 1, (n, 2))
    init[:n, 2] = rng.uniform(-0.5, 7.0, n)
    init[:n, 3] = rng.choice([0.0, 0.0, 0.3, 0.6], n)
    init[:n, 4] = rng.choice([0.0, 0.2, -0.2], n)
    tgt = np.tile([2.0, 3.0], (n + 6, 1))
    tgt[:n] += rng.uniform(-1, 1, (n, 2))
    org = np.zeros((n + 6, 2))
    thr = np.full(n + 6, 1e10)
    init[n:n + 2, :2] = tgt[n:n + 2]                                     # on target at entry
    thr[n + 2:n + 4] = -1.0                                               # no leaf on the first tick
    init[n + 4:n + 6] = [[1.0, 1.5, np.arctan2(-1.5, -1.0) + 2 * np.pi, 0.0, 0.0]] * 2    # stall
    return init, tgt, org, thr


def _per_step_events(script, n):
    """{step: [n][k] LoopEvent bytes} of a script shared by all robots: its tick s goes to the step that commits tick s."""
    nat = _nat()
    out = {}
    for s in sorted({e[0] for e in script}):
        todo = [e for e in script if e[0] == s]
        ev = (nat.LoopEvent * len(todo))(*(nat.LoopEvent(0, k, a, b) for _, k, a, b in todo))
        out[s] = np.tile(np.frombuffer(bytes(ev), np.uint8), (n, 1))
    return out


class StepRun:
    """Records of N robots on a solver, stepped until no robot runs.  ``plant(step, proposal, mask) -> measured``
    (device tensors) or None for measured = NULL; ``events`` {step: [N][k * 24] uint8 LoopEvent rows}."""

    def __init__(self, s, params, init, tgt, org, thr=None, slow=None):
        self.s, self.p, self.N = s, params, len(init)
        dev = torch.device("cuda", s.device)
        self.dev = dev
        self.stream = torch.cuda.ExternalStream(s.stream, device=dev)
        f64 = dict(dtype=torch.float64, device=dev)
        with torch.cuda.stream(self.stream):
            self.inp = [torch.tensor(np.ascontiguousarray(a, np.float64), **f64) for a in (init, tgt, org)]
            self.thr = None if thr is None else torch.tensor(np.asarray(thr, np.float64), **f64)
            self.slow = None if slow is None else torch.tensor(np.asarray(slow, np.int32), device=dev)
            self.ctrl = torch.empty((self.N, ctypes.sizeof(_nat().HeldCtrl)), dtype=torch.uint8, device=dev)
            self.proposal = torch.empty((self.N, 5), **f64)
            self.measured = torch.empty((self.N, 5), **f64)
            self.running = torch.zeros(1, dtype=torch.int32, device=dev)
        self.init()

    def init(self):
        with torch.cuda.stream(self.stream):
            self.s.held_ctrl_init_device(self.p, self.N, *(t.data_ptr() for t in self.inp),
                                         0 if self.thr is None else self.thr.data_ptr(),
                                         0 if self.slow is None else self.slow.data_ptr(), self.ctrl.data_ptr())
        self.k = 0
        self.props = []

    def step(self, plant=None, events=None, radius=0.0, sync=False):
        """One step; returns the running count (the one read of the step)."""
        with torch.cuda.stream(self.stream):
            meas = 0
            if plant is not None and self.k > 0:
                mask = ~torch.isnan(self.proposal[:, 0])
                self.measured.copy_(plant(self.k, self.proposal, mask))
                if sync:
                    torch.cuda.synchronize(self.dev)
                meas = self.measured.data_ptr()
            ev = (events or {}).get(self.k)
            evt = None if ev is None else torch.tensor(ev, device=self.dev)
            self.running.zero_()
            self.s.held_ctrl_step_device(self.p, self.N, self.ctrl.data_ptr(), meas, 0 if evt is None else evt.data_ptr(),
                                         0 if ev is None else ev.shape[1] // 24, radius, self.proposal.data_ptr(),
                                         self.running.data_ptr())
            self.props.append(self.proposal.clone())
            self.k += 1
            return int(self.running.item())

    def run(self, **kw):
        while self.step(**kw):
            assert self.k <= self.p.max_ticks + 1
        return self

    def records(self):
        with torch.cuda.stream(self.stream):
            raw = self.ctrl.cpu().numpy()
        return (_nat().HeldCtrl * self.N).from_buffer_copy(raw.tobytes()), raw

    def log(self):
        """The proposals as a closed loop's log [N][max_ticks][5] (proposal of step k = row k, NaN after)."""
        with torch.cuda.stream(self.stream):
            P = torch.stack(self.props).cpu().numpy()                 # [steps][N][5]
        out = np.full((self.N, self.p.max_ticks, 5), np.nan)
        k = min(P.shape[0], self.p.max_ticks)
        out[:, :k] = P[:k].transpose(1, 0, 2)
        assert np.isnan(P[self.p.max_ticks:]).all()
        return out

    def result(self):
        recs, _ = self.records()
        return dict(log=self.log(), ticks=np.array([r.ticks for r in recs], np.int32),
                    status=np.array([r.status for r in recs], np.int32),
                    final=np.array([list(r.line) + [r.slow_steps, r.m] for r in recs], np.float64))


def _assert_same_run(step, loop, what=""):
    for k in ("log", "ticks", "status", "final"):
        np.testing.assert_array_equal(step[k], loop[k], err_msg=f"{what}: {k}")


@pytest.mark.parametrize("H, cost, max_ticks, script", [
    (1, 1, 256, False), (2, 0, 256, True), (3, 1, 256, True), (3, 0, 40, False), (4, 1, 256, False), (4, 0, 120, True)])
def test_identity_plant_is_the_closed_loop(H, cost, max_ticks, script):
    """measured = NULL and measured = the proposal handed back: the stacked proposals, ticks, status and the records'
    line, slow_steps and m equal held_closed_loop with final, bit for bit -- with and without the demo script as
    per-step events, robots on target at entry, first-tick no-leaf robots, stalls and max_ticks."""
    mt = _module()
    nat = mt._native
    s = nat.Solver(0)
    params = _params(H, cost, max_ticks)
    init, tgt, org, thr = _robots(250, 100 + H + 10 * cost)
    n = len(init)
    kw = dict(events=list(mt.DEMO_EVENTS), radius_u_turn=mt.radius_u_turn) if script else {}
    loop = s.held_closed_loop(params, init, tgt, org, first_threshold=thr, **kw)
    ev = _per_step_events(mt.DEMO_EVENTS, n) if script else None
    a = StepRun(s, params, init, tgt, org, thr).run(events=ev, radius=mt.radius_u_turn).result()
    _assert_same_run(a, loop, "measured NULL")
    b = StepRun(s, params, init, tgt, org, thr).run(plant=lambda k, prop, mask: prop, events=ev,
                                                    radius=mt.radius_u_turn).result()
    _assert_same_run(b, loop, "measured = proposal")
    st = loop["status"]
    assert (st[n - 6:n - 4] == nat.LOOP_ON_TARGET).all() and (loop["ticks"][n - 6:n - 4] == 0).all()
    assert (st[n - 4:n - 2] == nat.LOOP_NO_LEAF).all()
    assert (st[n - 2:] == nat.LOOP_STALLED).all()
    if max_ticks < 200:
        assert (st == nat.LOOP_MAX_TICKS).sum() >= 8
    if script:
        assert (loop["ticks"] > 110).sum() >= 4


def _host_draws(gens, mt):
    def fn(commanded, running):
        c, m = commanded.cpu().numpy(), running.cpu().numpy()
        out = np.full_like(c, np.nan)
        for i in np.flatnonzero(m):
            out[i, 0] = mt.get_actual_velocity(c[i, 0], gens[i])
            out[i, 1] = mt.get_actual_beta_angle(c[i, 1], gens[i])
        return torch.from_numpy(out).to(commanded.device)
    return fn


def _assert_same_generators(a, b):
    for i, (ga, gb) in enumerate(zip(a, b)):
        if isinstance(ga, np.random.Generator):
            assert ga.bit_generator.state == gb.bit_generator.state, i
        else:
            sa, sb = ga.get_state(), gb.get_state()
            assert sa[2] == sb[2], i
            np.testing.assert_array_equal(sa[1], sb[1], err_msg=str(i))


@pytest.mark.parametrize("kind", ["mt19937", "pcg64"])
def test_actuator_from_host_generators_is_the_actual_run(kind, golden):
    """math_mpc_batch(actuator=fn), fn drawing get_actual_* from each robot's own generator on the host, equals
    device_noise=True on the same seeds bit for bit, generators included; the reference's seeded runs at 1e-9."""
    mt = _module()
    nat = mt._native
    cases = golden("held_actual")["cases"]
    rng = np.random.default_rng(5)
    seeds = [c["seed"] for c in cases] + [int(x) for x in rng.integers(0, 2 ** 32, 62)]
    n = len(seeds)
    init = np.zeros((n, 5))
    tgt = np.tile([2.0, 3.0], (n, 1))
    init[len(cases):, :2] = rng.uniform(-1, 1, (n - len(cases), 2))
    init[len(cases):, 2] = rng.uniform(-0.5, 7.0, n - len(cases))
    tgt[len(cases):] += rng.uniform(-1, 1, (n - len(cases), 2))
    make = (lambda: [np.random.RandomState(x) for x in seeds]) if kind == "mt19937" else \
        (lambda: [np.random.default_rng(x) for x in seeds])
    run = dict(max_ticks=400, origin=np.zeros((n, 2)), isActual=True, events=True)
    g_dev, g_host = make(), make()
    d = mt.math_mpc_batch(init, tgt, rngs=g_dev, device_noise=True, **run)
    a = mt.math_mpc_batch(init, tgt, actuator=_host_draws(g_host, mt), **run)
    _assert_same_run(a, d, kind)
    _assert_same_generators(g_dev, g_host)
    if kind == "mt19937":
        keys = ("actual_result_trajectory_x", "actual_result_trajectory_y", "actual_result_trajectory_phi",
                "actual_result_trajectory_v", "actual_result_trajectory_beta")
        for i, c in enumerate(cases):
            ref = np.array([c["log"][k][1:] for k in keys], dtype=float).T
            assert a["ticks"][i] == c["p"] - 1 == ref.shape[0]
            np.testing.assert_allclose(a["log"][i, :ref.shape[0]], ref, rtol=0, atol=1e-9)
            assert a["final"][i, 5] == c["m"]
            assert a["status"][i] == (nat.LOOP_STALLED if c["recursive"] else nat.LOOP_ON_TARGET)
    assert (a["status"] == nat.LOOP_ON_TARGET).sum() >= 8 and (a["ticks"] > 110).sum() >= 4


def test_per_robot_events():
    """Robots of one batch get different new_target / turn events at different ticks through the step's events (empty
    slots kind 0); each robot equals a one-robot held_closed_loop with its own script, bit for bit."""
    mt = _module()
    nat = mt._native
    s = nat.Solver(0)
    params = _params(3, nat.COST_TREE, 300)
    init, tgt, org, thr = _robots(40, 7)
    n = len(init)
    rng = np.random.default_rng(8)
    scripts = []
    for i in range(n):
        t1, t2 = sorted(rng.choice(np.arange(2, 60), 2, replace=False))
        kind2 = int(rng.choice([nat.EVENT_TURN_LEFT, nat.EVENT_TURN_RIGHT, nat.EVENT_NEW_TARGET]))
        sc = [(int(t1), nat.EVENT_NEW_TARGET, float(rng.uniform(-2, 3)), float(rng.uniform(-2, 3))),
              (int(t2), kind2, float(rng.uniform(0.5, 2.5)), float(rng.uniform(-2, 3)))]
        if i % 3 == 0:                                  # two events after one tick, in script order
            sc.append((int(t2), nat.EVENT_TURN_RIGHT, 1.0, 0.0))
        scripts.append(sc if i % 5 else [])             # some robots without any event
    ev = {}
    for t in sorted({e[0] for sc in scripts for e in sc}):
        rows = np.zeros((n, 3 * 24), np.uint8)          # three slots per robot, kind 0 = empty
        for i, sc in enumerate(scripts):
            todo = [e for e in sc if e[0] == t]
            if todo:
                arr = (nat.LoopEvent * len(todo))(*(nat.LoopEvent(12345, k, a, b) for _, k, a, b in todo))
                rows[i, :24 * len(todo)] = np.frombuffer(bytes(arr), np.uint8)
        ev[t] = rows
    r = StepRun(s, params, init, tgt, org, thr).run(events=ev, radius=mt.radius_u_turn).result()
    for i, sc in enumerate(scripts):
        one = s.held_closed_loop(params, init[i:i + 1], tgt[i:i + 1], org[i:i + 1], first_threshold=thr[i:i + 1],
                                 events=sc or None, radius_u_turn=mt.radius_u_turn)
        for k in ("log", "ticks", "status", "final"):
            np.testing.assert_array_equal(r[k][i:i + 1], one[k], err_msg=f"robot {i}: {k}")
    assert (r["ticks"] > 40).sum() >= 10


def _perturb(k, prop, n0=0):
    """The test plant: the proposed pose moved by a deterministic few millimetres / milliradians per robot and tick; robots
    n % 7 == 3 are held at their previous committed position on tick 9 (a repeated position taken from the plant)."""
    n = np.arange(n0, n0 + prop.shape[0])
    out = prop.copy()
    out[:, 0] += 2e-3 * np.cos(0.7 * n + 1.3 * k)
    out[:, 1] += 2e-3 * np.sin(0.9 * n + 0.4 * k)
    out[:, 2] += 1e-3 * np.cos(0.3 * n + 2.1 * k)
    return out


def test_plant_that_moves_the_robot_equals_a_host_loop():
    """measured != proposal: windows, the stop test and the repeated-position test are taken from the measured state.
    The steps equal a host loop written from Solver.solve_held_windows and the module's _finish_tick on the same
    measured states, at 1e-9."""
    mt = _module()
    nat = mt._native
    s = nat.Solver(0)
    params = _params(3, nat.COST_TREE, 200)
    init, tgt, org, thr = _robots(120, 21)
    n = len(init)
    held = np.arange(n) % 7 == 3
    prev = {"xy": init[:, :2].copy()}

    def plant_np(k, prop, mask):
        out = _perturb(k, prop)
        if k == 9:
            out[held, :2] = prev["xy"][held]
        prev["xy"] = np.where(mask[:, None], out[:, :2], prev["xy"])
        return out

    def plant(k, prop, mask):
        return torch.from_numpy(plant_np(k, prop.cpu().numpy(), mask.cpu().numpy())).to(prop.device)

    r = StepRun(s, params, init, tgt, org, thr).run(plant=plant).result()

    # the host loop
    prev["xy"] = init[:, :2].copy()
    robots = []
    for i in range(n):
        c = {}
        mt.reset_state(c)
        c.update(x_t=tgt[i, 0], y_t=tgt[i, 1], x_0=org[i, 0], y_0=org[i, 1], optimal_criterion=thr[i],
                 pose=list(init[i]), previous=(init[i, 0], init[i, 1]), status=None, ticks=0, recursive=False)
        robots.append(c)
    log = np.full((n, params.max_ticks, 5), np.nan)
    k = 0
    while True:
        live = []                                       # robot numbers (identical robots are distinct robots)
        for i, c in enumerate(robots):
            if c["status"] is not None:
                continue
            if mt.is_on_target(c["pose"][0], c["pose"][1], c["x_t"], c["y_t"])[0]:
                c["status"] = nat.LOOP_ON_TARGET
            elif c["ticks"] >= params.max_ticks:
                c["status"] = nat.LOOP_MAX_TICKS
            else:
                live.append(i)
        if not live:
            break
        lc = [robots[i] for i in live]
        w = s.solve_held_windows(params, [c["pose"][:3] for c in lc], [c["pose"][3:5] for c in lc],
                                 [[c["x_t"], c["y_t"]] for c in lc], [[c["x_0"], c["y_0"]] for c in lc],
                                 threshold=[float(c["optimal_criterion"]) for c in lc],
                                 flags=[nat.FLAG_SLOW if c["steps_for_slowing"] > 0 else 0 for c in lc])
        prop = np.full((n, 5), np.nan)
        for j, i in enumerate(live):
            c = robots[i]
            found = None
            if w["index"][j] >= 0:
                found = (w["traj"][j], w["first_control"][j, 0], w["first_control"][j, 1], w["cost"][j])
            elif c["optimal_trajectory"] == [[[0]]]:
                c["status"] = nat.LOOP_NO_LEAF
                c["steps_for_slowing"] -= 1
                continue
            prop[i] = mt._finish_tick(c, found, False)
        k += 1
        mask = ~np.isnan(prop[:, 0])
        meas = plant_np(k, prop, mask)
        for i in np.flatnonzero(mask):
            c = robots[i]
            log[i, c["ticks"]] = prop[i]
            c["pose"] = list(meas[i])
            c["ticks"] += 1
            if c["recursive"]:
                c["status"] = nat.LOOP_STALLED
            elif (meas[i, 0], meas[i, 1]) == c["previous"]:
                c["recursive"] = True
            c["previous"] = (meas[i, 0], meas[i, 1])
    np.testing.assert_array_equal(r["ticks"], [c["ticks"] for c in robots])
    np.testing.assert_array_equal(r["status"], [c["status"] for c in robots])
    np.testing.assert_allclose(r["log"], log, rtol=0, atol=1e-9, equal_nan=True)
    want = np.array([[c["x_t"], c["y_t"], c["x_0"], c["y_0"], c["steps_for_slowing"], c["m"]] for c in robots], float)
    np.testing.assert_array_equal(r["final"], want)
    assert (r["status"][held] == nat.LOOP_STALLED).sum() >= 8
    assert (r["status"] == nat.LOOP_ON_TARGET).sum() >= 30


def test_edge_cases():
    """N = 0; a step after every robot stopped (NaN rows, running 0, records unchanged); re-initialised records; two
    handles stepping in alternation; the plant on the solver's stream without per-step synchronisation; refusals."""
    mt = _module()
    nat = mt._native
    s, s2 = nat.Solver(0), nat.Solver(0)
    params = _params(3, nat.COST_TREE, 150)
    init, tgt, org, thr = _robots(60, 31)
    ref = s.held_closed_loop(params, init, tgt, org, first_threshold=thr)

    # N = 0: nothing to do, nothing read
    s.held_ctrl_init_device(params, 0, 0, 0, 0, 0, 0, 0)
    s.held_ctrl_step_device(params, 0, 0)
    s.sync()

    # after the last step
    a = StepRun(s, params, init, tgt, org, thr).run()
    _assert_same_run(a.result(), ref)
    _, before = a.records()
    assert a.step() == 0 and torch.isnan(a.props[-1]).all()
    _, after = a.records()
    np.testing.assert_array_equal(before, after)

    # re-initialised records, part-way through a run
    a.init()
    for _ in range(17):
        a.step()
    a.init()
    _assert_same_run(a.run().result(), ref, "re-initialised")

    # two handles in alternation, each on its own stream
    half = len(init) // 2
    b1 = StepRun(s, params, init[:half], tgt[:half], org[:half], thr[:half])
    b2 = StepRun(s2, params, init[half:], tgt[half:], org[half:], thr[half:])
    run1 = run2 = True
    while run1 or run2:
        if run1:
            run1 = b1.step()
        if run2:
            run2 = b2.step()
    r1, r2 = b1.result(), b2.result()
    for k in ("log", "ticks", "status", "final"):
        np.testing.assert_array_equal(np.concatenate([r1[k], r2[k]]), ref[k], err_msg=k)

    # a torch plant on the solver's stream, no per-step synchronisation == the same with one after every plant call
    def plant(k, prop, mask):
        d = torch.arange(prop.shape[0], device=prop.device, dtype=torch.float64)
        out = prop.clone()
        out[:, 0] += 1e-3 * torch.cos(0.7 * d + 1.3 * k)
        out[:, 3] = torch.clamp(out[:, 3] * 0.98, min=0.0)
        return out
    x = StepRun(s, params, init, tgt, org, thr).run(plant=plant).result()
    y = StepRun(s, params, init, tgt, org, thr).run(plant=plant, sync=True).result()
    for k in ("log", "ticks", "status", "final"):
        np.testing.assert_array_equal(x[k], y[k], err_msg=k)
    assert not np.array_equal(x["log"], ref["log"])

    # refusals
    c = a.ctrl.data_ptr()
    ev = torch.zeros(len(init) * 65 * 24, dtype=torch.uint8, device=a.dev)

    def refused(fn):
        with pytest.raises(nat.MpcbError) as e:
            fn()
        assert e.value.code == -1
    for n_ev, evp in ((-1, ev.data_ptr()), (65, ev.data_ptr()), (1, 0)):
        refused(lambda: s.held_ctrl_step_device(params, len(init), c, 0, evp, n_ev))
    refused(lambda: s.held_ctrl_step_device(params, len(init), 0))
    refused(lambda: s.held_ctrl_step_device(params, -1, c))
    refused(lambda: s.held_ctrl_init_device(params, len(init), 0, *(t.data_ptr() for t in a.inp[1:]), 0, 0, c))
    refused(lambda: s.held_ctrl_init_device(params, len(init), *(t.data_ptr() for t in a.inp), 0, 0, 0))
    for field, bad in (("H", 0), ("H", 9), ("max_ticks", 0), ("n_v", 0), ("n_beta", 129)):
        p = _params(3, nat.COST_TREE, 150)
        setattr(p, field, bad)
        refused(lambda: s.held_ctrl_step_device(p, len(init), c))
        refused(lambda: s.held_ctrl_init_device(p, len(init), *(t.data_ptr() for t in a.inp), 0, 0, c))
    s.held_ctrl_step_device(params, len(init), c, 0, ev.data_ptr(), 64)     # 64 slots of kind 0: accepted
    s.sync()
