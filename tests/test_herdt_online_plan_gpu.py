"""Plans of the on-line Herdt2010 generator: wg_herdt_online_tick_plan (HerdtOnline.tick_plan, tick_plan_device).

A plan is the QP a robot solved at the tick it fired, expanded over its horizon.  It is checked without trusting the plan
kernel: a RefRobot of test_herdt_online_gpu (the C++ mirror's per-tick logic over the period API) records the QP input of
each period it runs, the dense QP entry (Context.herdt_qp_solve) solves it again, and numpy expands the solution with the
dynamics matrices of RigidBodySystem::compute_dyn_cjerk (rigid-body-system.cpp:377-452).  The oracle's own closed loop
(herdt_oracle.Sim) checks the same plans against the reference's code path.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import herdt_oracle as ho
from test_herdt_online_gpu import RefRobot, _back_row, _init15

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "walkgen_b200.h")
N = 16
TS = 0.005
PRW = ("prw_com_x", "prw_com_y", "prw_cop_x", "prw_cop_y")
SENTINEL = 0x5A


def _wg():
    import jrl_walkgen_b200 as wg
    return wg


@pytest.fixture(scope="module")
def mctx(ctx):
    ctx.herdt_set_params()
    ctx.herdt_mpc_set_params()
    return ctx


@pytest.fixture()
def era_ctx(ctx):
    """The datref-era settings of test_herdt_online_gpu.era_ctx; restored afterwards."""
    wg = _wg()
    ctx.herdt_set_params()
    p = wg.herdt_mpc_default_params()
    p.foot_vel_limit = 0.0
    p.return_to_centre = 0
    ctx.herdt_mpc_set_params(p)
    yield ctx
    ctx.herdt_mpc_set_params()


def expand_axis(c, u, T, h):
    """(CoM [N][3], CoP [N]) of one axis from its initial state c (3) and jerks u (N)."""
    k = np.arange(1, N + 1, dtype=np.float64)
    d = (np.arange(N)[:, None] - np.arange(N)[None, :]).astype(np.float64)
    low = d >= 0
    Sp = np.column_stack([np.ones(N), k * T, k * k * T * T / 2])
    Up = np.where(low, (1 + 3 * d + 3 * d * d) * T ** 3 / 6, 0.0)
    Sv = np.column_stack([np.zeros(N), np.ones(N), k * T])
    Uv = np.where(low, (2 * d + 1) * T * T / 2, 0.0)
    Ua = np.where(low, T, 0.0)
    Sz = np.column_stack([np.ones(N), k * T, k * k * T * T / 2 - h / 9.81])
    Uz = np.where(low, (1 + 3 * d + 3 * d * d) * T ** 3 / 6 - T * h / 9.81, 0.0)
    com = np.column_stack([Sp @ c + Up @ u, Sv @ c + Uv @ u, c[2] + Ua @ u])
    return com, Sz @ c + Uz @ u


def expected_plans(ctx, qins, times, qp_counts):
    """The plans of the recorded QP inputs: solved by the dense QP entry, expanded by numpy."""
    wg = _wg()
    out = ctx.herdt_qp_solve(qins)
    T, h = ctx.herdt_params.T, ctx.herdt_params.com_height
    p = np.zeros(len(qins), dtype=wg.HERDT_PLAN_DTYPE)
    for i, (q, o) in enumerate(zip(qins, out)):
        ns = (int(o["n_vars"]) - 2 * N) // 2
        r = p[i]
        r["time"] = times[i]; r["qp_count"] = qp_counts[i]
        r["com_x"] = q["com_x"]; r["com_y"] = q["com_y"]
        r["jerk_x"] = o["x"][:N]; r["jerk_y"] = o["x"][N:2 * N]
        for f in ("sup_x", "sup_y", "sup_yaw", "sup_foot", "sup_phase", "sup_step", "sup_changed"):
            r[f] = q[f]
        r["n_steps"] = ns; r["fail"] = o["fail"]; r["iterations"] = o["iterations"]
        for s in range(ns):
            k = int(np.argmax(q["sup_step"][1:] == s + 1)) + 1
            r["step_x"][s] = o["x"][2 * N + s]; r["step_y"][s] = o["x"][2 * N + ns + s]
            r["step_yaw"][s] = q["sup_yaw"][k]; r["step_sample"][s] = k; r["step_foot"][s] = q["sup_foot"][k]
        r["prw_com_x"], r["prw_cop_x"] = expand_axis(q["com_x"], o["x"][:N], T, h)
        r["prw_com_y"], r["prw_cop_y"] = expand_axis(q["com_y"], o["x"][N:2 * N], T, h)
    return p


def assert_plan_equal(got, want):
    """Bitwise outside the expanded horizon, within 1e-12 on it."""
    g, w = got.copy(), want.copy()
    for f in PRW:
        assert np.abs(g[f] - w[f]).max() < 1e-12, (f, np.abs(g[f] - w[f]).max())
        g[f] = 0.0; w[f] = 0.0
    if g.tobytes() != w.tobytes():
        bad = [f for f in g.dtype.names if g[f].tobytes() != w[f].tobytes()]
        raise AssertionError(f"plan fields differ: {bad}")


class PlanRobot(RefRobot):
    """RefRobot that keeps (QP input, clock, qp_count) of the period it runs at a tick in `fired` (None otherwise)."""

    def tick(self, cmd=None):
        wg = _wg()
        self.fired = None
        if not self.running:
            return None, 0
        st = self.st
        if cmd is not None:
            if cmd["flags"] & wg.CMD_VEL:
                st["new_ref"][0] = cmd["vel"]
            if cmd["flags"] & wg.CMD_STOP:
                st["ending_phase"] = 1
        clock = st["clock"][0] + TS
        if st["online_mode"][0] and clock + 0.00001 > st["upper_time_limit"][0]:
            t, s, q = self.ctx.herdt_mpc_run(st, 1, ticks=True, steps=True, qp_in=True)
            self.fired = (q[0].copy(), float(s[0, 0]["time"]), int(st["qp_count"][0]))
            rows = t[0]
            self.q[-1]["left"] = rows[0]["left"]; self.q[-1]["right"] = rows[0]["right"]
            for k in range(1, 20):
                self.q.append(np.array(rows[k], dtype=wg.TICK_DTYPE))
            self.q.append(_back_row(st).copy())
        else:
            st["clock"] = clock
            if st["online_mode"][0] and st["ending_phase"][0] and clock >= st["time_to_stop"][0]:
                st["online_mode"] = 0
        if not self.q:
            self.running = False
            return None, 0
        return self.q.popleft(), 1


def _fleet_script():
    """The 48-robot script of test_online_ticks_bitwise_equal_per_robot_mirror: starts over ticks 0..39, two restarts of
    running robots, velocity and yaw commands (bursts inside one QP period), :stoppg at random ticks; 1500 ticks."""
    wg = _wg()
    rng = np.random.default_rng(2026)
    B, NT = 48, 1500
    starts = rng.permutation(np.arange(B) % 40)
    events = {}
    for b in range(B):
        init = _init15(x=0.0316055 + rng.uniform(-0.5, 0.5), y=rng.uniform(-0.5, 0.5), dx=0.02 if b % 5 == 0 else 0.0)
        init[9] = init[12] = init[0] - 0.0316055
        events.setdefault(int(starts[b]), []).append((b, init))
    for b, t in ((3, 300), (17, 777)):
        events.setdefault(t, []).append((b, _init15(y=0.2 * (b % 2))))
    cmds = np.zeros((NT, B), dtype=wg.HERDT_COMMAND_DTYPE)
    for b in range(B):
        for t in rng.choice(np.arange(40, NT - 100), size=6, replace=False):
            cmds["flags"][t, b] = wg.CMD_VEL
            cmds["vel"][t, b] = (rng.uniform(-0.2, 0.3), rng.uniform(-0.15, 0.15), rng.uniform(-0.3, 0.3))
    for b in (5, 6):
        t0 = 401 + 3 * b
        for k, dt in enumerate((0, 4, 9, 15)):
            cmds["flags"][t0 + dt, b] = wg.CMD_VEL
            cmds["vel"][t0 + dt, b] = (0.05 * k, -0.03 * k, 0.1 * (k - 1))
    for b in rng.choice([b for b in range(B) if b not in (3, 17)], size=16, replace=False):
        cmds["flags"][int(rng.integers(100, 1100)), b] |= wg.CMD_STOP
    return B, NT, events, cmds


@pytest.fixture(scope="module")
def fleet_reference(mctx):
    """Rows, running flags, final states and the plan of every (tick, robot) firing of the per-robot mirror."""
    wg = _wg()
    B, NT, events, cmds = _fleet_script()
    robots = [PlanRobot(mctx) for _ in range(B)]
    rows = np.zeros((NT, B), dtype=wg.TICK_DTYPE)
    run = np.zeros((NT, B), dtype=np.int8)
    keys, qins, times, counts = [], [], [], []
    for t in range(NT):
        for b, init in events.get(t, []):
            robots[b].start(init)
        for b, r in enumerate(robots):
            row, ok = r.tick(cmds[t, b])
            run[t, b] = ok
            if ok:
                rows[t, b] = row
            if r.fired is not None:
                keys.append((t, b)); qins.append(r.fired[0]); times.append(r.fired[1]); counts.append(r.fired[2])
    plans = expected_plans(mctx, np.array(qins), times, counts)
    st = np.concatenate([r.st for r in robots])
    return {"rows": rows, "run": run, "states": st, "plans": dict(zip(keys, plans))}


def _bounds(NT, events, per_call):
    cuts = set(range(0, NT, per_call)) | set(events) | {NT}
    return sorted(cuts)


@pytest.mark.gpu
@pytest.mark.parametrize("per_call", [1, 7, 20])
def test_plans_bitwise_equal_per_robot_mirror(mctx, fleet_reference, per_call):
    wg = _wg()
    B, NT, events, cmds = _fleet_script()
    ref = fleet_reference
    h = mctx.herdt_online(B)
    plans = np.zeros(B, dtype=wg.HERDT_PLAN_DTYPE)
    plans.view(np.uint8)[:] = SENTINEL
    rows = np.zeros((NT, B), dtype=wg.TICK_DTYPE)
    run = np.zeros((NT, B), dtype=np.int8)
    checked = 0
    try:
        cuts = _bounds(NT, events, per_call)
        for a, b in zip(cuts[:-1], cuts[1:]):
            if a in events:
                h.start([i for i, _ in events[a]], np.array([init for _, init in events[a]]))
            before = plans.copy()
            r, q, pt = h.tick_plan(b - a, plans, cmds[a:b])
            rows[a:b] = r; run[a:b] = q
            for i in range(B):
                fired = [t for t in range(a, b) if (t, i) in ref["plans"]]
                if not fired:
                    assert pt[i] == -1 and plans[i].tobytes() == before[i].tobytes(), (a, i)
                    continue
                assert pt[i] == fired[-1] - a, (a, i, pt[i], fired)
                assert_plan_equal(plans[i], ref["plans"][(fired[-1], i)])
                checked += 1
        st = h.states()
    finally:
        h.destroy()
    assert np.array_equal(run, ref["run"])
    assert rows.tobytes() == ref["rows"].tobytes()
    assert st.tobytes() == ref["states"].tobytes()
    assert checked >= (len(ref["plans"]) if per_call == 1 else len(ref["plans"]) // 2)
    # the script exercised previewed steps and both feet
    allp = np.array(list(ref["plans"].values()))
    assert (allp["n_steps"] == 2).any() and (allp["n_steps"] == 1).any() and (allp["fail"] == 0).all()


def _era_plans(era_ctx, script, name):
    """One robot of the TestHerdt2010 script through the handle, 10 ticks per call (at most one QP per call) -> (plans in
    firing order, firing ticks, states after each firing call, rows [ticks])."""
    wg = _wg()
    gold = ho.load_golden(name)
    NT = len(gold) + 40

    def edit(st):
        st["sup_steps_left"] = 2; st["nb_steps_ssds"] = 2
        st["sup_x"], st["sup_y"], st["sup_yaw"] = 0.0, 0.1, 0.0

    cmds = np.zeros((NT, 1), dtype=wg.HERDT_COMMAND_DTYPE)
    for t, v, stop in script:
        cmds["vel"][t, 0] = v
        cmds["flags"][t, 0] = wg.CMD_VEL | (wg.CMD_STOP if stop else 0)
    h = era_ctx.herdt_online(1)
    out, ticks, states = [], [], []
    rows = np.zeros(NT, dtype=wg.TICK_DTYPE)
    run = np.zeros(NT, dtype=np.int8)
    try:
        h.start([0], _init15())
        st = h.states(); edit(st); h.set_states(st)
        plans = np.zeros(1, dtype=wg.HERDT_PLAN_DTYPE)
        for a in range(0, NT, 10):
            r, q, pt = h.tick_plan(min(10, NT - a), plans, cmds[a:a + 10])
            rows[a:a + len(r)] = r[:, 0]; run[a:a + len(q)] = q[:, 0]
            if pt[0] >= 0:
                out.append(plans[0].copy()); ticks.append(a + int(pt[0])); states.append(h.states()[0])
    finally:
        h.destroy()
    assert run[:len(gold)].all() and not run[len(gold):].any()
    return np.array(out), ticks, np.array(states), rows, len(gold)


@pytest.mark.gpu
@pytest.mark.parametrize("name,script,events", [("online", ho.ONLINE_SCRIPT, ho.ONLINE_EVENTS),
                                                ("emergency", ho.EMERGENCY_SCRIPT, ho.EMERGENCY_EVENTS)])
def test_plans_follow_the_reference_code_path(era_ctx, name, script, events):
    plans, ticks, states, rows, n = _era_plans(era_ctx, script, name)
    sim, _ = ho.run_online_script(n, events, datref_era=True, logging=True)
    ins, X, _, _ = sim.log()
    sim.close()
    assert len(plans) == len(ins), (len(plans), len(ins))
    for f in ("sup_phase", "sup_foot", "sup_step", "sup_changed"):
        assert np.array_equal(plans[f], ins[f]), f
    # Footsteps and the first previewed sample, which the period executes, meet the closed-loop tests' 1e-6 m.  Farther out
    # the horizon magnifies the jerks' own differences between the two solvers (U of sample k = 1 weighs a jerk by T^3/6 =
    # 1.7e-4, sample 16 by 0.12 and the 16 jerks together by 0.68), so the whole horizon is held to 1e-4 m.
    T, h = era_ctx.herdt_params.T, era_ctx.herdt_params.com_height
    steps = first = horizon = 0.0
    for p, q, x in zip(plans, ins, X):
        ns = int(q["sup_step"][N])
        assert p["n_steps"] == ns
        for s in range(ns):
            steps = max(steps, abs(p["step_x"][s] - x[2 * N + s]), abs(p["step_y"][s] - x[2 * N + ns + s]))
        for axis, (c, u) in enumerate(((q["com_x"], x[:N]), (q["com_y"], x[N:2 * N]))):
            com, cop = expand_axis(c, u, T, h)
            err = np.maximum(np.abs(p[("prw_com_x", "prw_com_y")[axis]][:, 0] - com[:, 0]),
                             np.abs(p[("prw_cop_x", "prw_cop_y")[axis]] - cop))
            first, horizon = max(first, err[0]), max(horizon, err.max())
    print(f"{name}: {len(plans)} plans, max |plan - oracle|: footsteps {steps:.2e}, sample 1 {first:.2e}, "
          f"horizon {horizon:.2e}")
    assert steps < 1e-6 and first < 1e-6 and horizon < 1e-4, (steps, first, horizon)
    # return_to_centre = 0: the period applies jerk_x[0] / jerk_y[0], so previewed sample 1 is the state's CoM after the tick
    assert np.abs(plans["prw_com_x"][:, 0] - states["com_x"]).max() < 1e-12
    assert np.abs(plans["prw_com_y"][:, 0] - states["com_y"]).max() < 1e-12
    # and sample j of the period is the row popped 8 + j ticks after the firing tick (7 + j after the first QP)
    for i, (p, t) in enumerate(zip(plans, ticks)):
        lag = 7 if i == 0 else 8
        for j in range(1, 20):
            tj = j * TS
            for axis, f in ((0, "com_x"), (1, "com_y")):
                c, u = p[f], p[("jerk_x", "jerk_y")[axis]][0]
                want = c[0] + tj * c[1] + 0.5 * tj * tj * c[2] + tj ** 3 * u / 6.0
                assert abs(rows[t + lag + j][f][0] - want) < 1e-12, (i, j, f)


@pytest.mark.gpu
def test_entries_of_robots_that_do_not_fire_are_untouched(mctx):
    """Robots never started, stopped, past time_to_stop and draining their deques, or without a QP instant in a short call:
    plan_tick -1 and their entries keep the caller's bytes; host and device modes give the same bytes."""
    wg = _wg()
    B, NT = 8, 760
    cmds = np.zeros((NT, B), dtype=wg.HERDT_COMMAND_DTYPE)
    cmds["flags"][:, :] = wg.CMD_VEL
    cmds["vel"][:, :] = (0.15, 0.02, 0.05)
    for b, t in ((2, 5), (3, 120), (4, 181), (5, 243), (6, 300)):
        cmds["flags"][t, b] |= wg.CMD_STOP
    lengths = [5, 20, 3, 13, 1, 40, 9, 2, 17]
    hh, hd = mctx.herdt_online(B), mctx.herdt_online(B)
    d_plans = mctx.alloc(B * wg.HERDT_PLAN_DTYPE.itemsize)
    d_pt = mctx.alloc(B * 4)
    seen = {"never": 0, "stopped": 0, "draining": 0, "between_instants": 0}
    try:
        for h in (hh, hd):
            h.start(np.arange(1, B))
        a, n = 0, 0
        while a < NT:
            m = min(lengths[n % len(lengths)], NT - a)
            plans = np.zeros(B, dtype=wg.HERDT_PLAN_DTYPE)
            plans.view(np.uint8)[:] = SENTINEL
            _, q, pt = hh.tick_plan(m, plans, cmds[a:a + m])
            mctx._check(mctx.lib.wg_memset_device(mctx.h, d_plans.ptr, SENTINEL, d_plans.nbytes))
            mctx._check(mctx.lib.wg_memset_device(mctx.h, d_pt.ptr, 0x7F, d_pt.nbytes))
            d_cmd = mctx.to_device(cmds[a:a + m])
            hd.tick_plan_device(m, d_plans, d_cmd, None, None, d_pt)
            mctx.sync(); d_cmd.free()
            assert d_plans.download(wg.HERDT_PLAN_DTYPE, (B,)).tobytes() == plans.tobytes()
            assert d_pt.download(np.int32, (B,)).tobytes() == pt.tobytes()
            st = hh.states()
            for b in range(B):
                untouched = plans[b].tobytes() == bytes([SENTINEL]) * wg.HERDT_PLAN_DTYPE.itemsize
                assert untouched == (pt[b] == -1), (a, b, pt[b])
                if pt[b] != -1:
                    assert plans[b]["qp_count"] == st[b]["qp_count"] and plans[b]["time"] > 0
                    continue
                if b == 0:
                    seen["never"] += 1
                elif not q[:, b].any():
                    seen["stopped"] += 1
                elif not st[b]["online_mode"]:
                    seen["draining"] += 1
                else:
                    seen["between_instants"] += 1
            a += m; n += 1
        assert hh.states().tobytes() == hd.states().tobytes()
    finally:
        hh.destroy(); hd.destroy(); d_plans.free(); d_pt.free()
    assert all(v > 0 for v in seen.values()), seen


@pytest.mark.gpu
def test_launches_per_tick_and_no_allocation_in_steady_state(mctx):
    """Five launches per tick with plans (either pointer), four with both NULL, whether no robot, some or all fire; with
    WG_MEM_DEVICE no call allocates once the buffers exist."""
    from test_kajita_online_gpu import _free_device_memory
    wg = _wg()
    B = 64
    h = mctx.herdt_online(B)
    d_plans = mctx.alloc(B * wg.HERDT_PLAN_DTYPE.itemsize)
    d_pt = mctx.alloc(B * 4)
    try:
        def launches(n, plans=True, pt=True):
            out = []
            for _ in range(n):
                l0 = mctx.launches
                h.tick_plan_device(1, d_plans if plans else None, d_plan_tick=d_pt if pt else None)
                out.append(mctx.launches - l0)
            mctx.sync()
            return out

        assert set(launches(3)) == {5}                     # nothing started
        h.start(np.arange(B))
        assert set(launches(1)) == {5}                     # every robot fires
        assert set(launches(3, pt=False) + launches(3, plans=False)) == {5}
        assert set(launches(10, plans=False, pt=False)) == {4}
        h.start(np.arange(0, B, 2))
        assert set(launches(1)) == {5}                     # half the robots fire
        assert set(launches(40)) == {5}
    finally:
        h.destroy(); d_plans.free(); d_pt.free()
    # steady state at 4096 robots, 20 ticks per call
    B = 4096
    h = mctx.herdt_online(B)
    d_plans = mctx.alloc(B * wg.HERDT_PLAN_DTYPE.itemsize)
    d_pt = mctx.alloc(B * 4)
    d_rows, d_run = mctx.alloc(20 * B * wg.TICK_DTYPE.itemsize), mctx.alloc(20 * B)
    try:
        for t in range(20):
            h.start(np.arange(t, B, 20))
            h.tick_plan_device(1, d_plans, None, d_rows, d_run, d_pt)
        free0 = None
        for call in range(30):
            if call == 10:
                mctx.sync()
                free0 = _free_device_memory()
            h.tick_plan_device(20, d_plans, None, d_rows, d_run, d_pt)
        mctx.sync()
        assert _free_device_memory() == free0
        assert (d_pt.download(np.int32, (B,)) >= 0).all()
    finally:
        h.destroy(); d_plans.free(); d_pt.free(); d_rows.free(); d_run.free()


@pytest.mark.gpu
def test_refusals_change_nothing(mctx, ctx):
    """The tick's refusals and device plans that are not 16-byte aligned return WG_ERR_INVALID and leave states, deques and
    the caller's plans as they were (a twin handle that never saw the refused calls ticks on bitwise equal)."""
    wg = _wg()
    from jrl_walkgen_b200 import _capi
    INVALID = _capi.WG_ERR_INVALID
    B = 6
    cmds = np.zeros((120, B), dtype=wg.HERDT_COMMAND_DTYPE)
    cmds["flags"][:, :] = wg.CMD_VEL
    cmds["vel"][:, :] = (0.2, 0.0, 0.1)
    h, twin = mctx.herdt_online(B), mctx.herdt_online(B)
    d_plans = mctx.alloc(B * wg.HERDT_PLAN_DTYPE.itemsize + 16)
    try:
        for x in (h, twin):
            x.start([0, 2, 3, 5])
            x.tick(37, cmds[:37])
        saved = h.save()
        plans = np.zeros(B, dtype=wg.HERDT_PLAN_DTYPE)
        plans.view(np.uint8)[:] = SENTINEL
        pt = np.full(B, 77, dtype=np.int32)
        mctx._check(mctx.lib.wg_memset_device(mctx.h, d_plans.ptr, SENTINEL, d_plans.nbytes))
        lib = mctx.lib
        cmd1 = np.ascontiguousarray(cmds[37:38])
        refused = [lib.wg_herdt_online_tick_plan(h.h, wg.WG_MEM_HOST, -1, None, None, None, plans.ctypes.data, pt.ctypes.data),
                   lib.wg_herdt_online_tick_plan(h.h, 7, 1, None, None, None, plans.ctypes.data, pt.ctypes.data),
                   lib.wg_herdt_online_tick_plan(h.h, wg.WG_MEM_DEVICE, 1, None, None, None, C.c_void_p(d_plans.ptr + 8), None),
                   lib.wg_herdt_online_tick_plan(h.h, wg.WG_MEM_DEVICE, 1, None, None, None, C.c_void_p(d_plans.ptr + 4), None),
                   lib.wg_herdt_online_tick_plan(h.h, wg.WG_MEM_HOST, -3, cmd1.ctypes.data, None, None, None, None)]
        assert refused == [INVALID] * len(refused), refused
        mctx.sync()
        assert h.save().tobytes() == saved.tobytes()
        assert (plans.view(np.uint8) == SENTINEL).all() and (pt == 77).all()
        assert (d_plans.download(np.uint8, (d_plans.nbytes,)) == SENTINEL).all()
        pa = np.zeros(B, dtype=wg.HERDT_PLAN_DTYPE)
        ra, qa, ta = h.tick_plan(83, pa, cmds[37:])
        rb, qb = twin.tick(83, cmds[37:])
        assert qa.tobytes() == qb.tobytes() and ra.tobytes() == rb.tobytes() and qa[:, [0, 2, 3, 5]].all()
        assert h.save().tobytes() == twin.save().tobytes()
        assert (ta[[0, 2, 3, 5]] >= 0).all() and (ta[[1, 4]] == -1).all()
    finally:
        h.destroy(); twin.destroy(); d_plans.free()
    bare = wg.Context(0)
    try:
        hb = bare.herdt_online(2)
        want = bare.lib.wg_herdt_online_tick(hb.h, wg.WG_MEM_HOST, 1, None, None, None)
        assert want == _capi.WG_ERR_NOT_READY
        p2 = np.zeros(2, dtype=wg.HERDT_PLAN_DTYPE)
        assert bare.lib.wg_herdt_online_tick_plan(hb.h, wg.WG_MEM_HOST, 1, None, None, None, p2.ctypes.data, None) == want
        assert not p2.view(np.uint8).any()
        hb.destroy()
    finally:
        bare.close()


@pytest.mark.gpu
def test_forked_branches_plan_like_fresh_copies(mctx):
    """Live robots copied into K branches each, every branch under its own velocity, ticked until each fires: the branch
    plans differ from each other, and each equals the plan of the same robot copied into another handle at another index
    and ticked the same way, byte for byte."""
    wg = _wg()
    L, K = 8, 4
    live = mctx.herdt_online(L)
    rng = np.random.default_rng(11)
    lc = np.zeros((57, L), dtype=wg.HERDT_COMMAND_DTYPE)
    lc["flags"][::9] = wg.CMD_VEL
    lc["vel"][::9] = rng.uniform(-0.1, 0.2, size=(len(lc[::9]), L, 3))
    cand = np.column_stack([np.linspace(0.0, 0.3, K), np.linspace(-0.1, 0.1, K), np.linspace(-0.2, 0.2, K)])
    nb = L * K
    bc = np.zeros((20, nb), dtype=wg.HERDT_COMMAND_DTYPE)
    bc["flags"][0] = wg.CMD_VEL
    bc["vel"][0] = np.tile(cand, (L, 1))
    perm = rng.permutation(nb).astype(np.int32)
    br, fresh = mctx.herdt_online(nb), mctx.herdt_online(nb)
    try:
        for t in range(8):
            live.start([t])
            live.tick(1, lc[t:t + 1])
        live.tick(49, lc[8:])
        br.copy_from(live, src_idx=np.repeat(np.arange(L), K))
        pb = np.zeros(nb, dtype=wg.HERDT_PLAN_DTYPE)
        _, _, tb = br.tick_plan(20, pb, bc)
        fresh.copy_from(live, src_idx=np.repeat(np.arange(L), K), dst_idx=perm)
        fc = np.zeros_like(bc)
        fc[:, perm] = bc
        pf = np.zeros(nb, dtype=wg.HERDT_PLAN_DTYPE)
        _, _, tf = fresh.tick_plan(20, pf, fc)
    finally:
        live.destroy(); br.destroy(); fresh.destroy()
    assert (tb >= 0).all()
    assert pf[perm].tobytes() == pb.tobytes() and tf[perm].tobytes() == tb.tobytes()
    for r in range(L):
        branch = pb[r * K:(r + 1) * K]
        assert len({p.tobytes() for p in branch}) == K
        assert len({p["time"] for p in branch}) == 1 and len({p["qp_count"] for p in branch}) == 1


def test_plan_layout_matches_the_header(tmp_path):
    """sizeof and field offsets of wg_herdt_plan, compiled against the header, equal HERDT_PLAN_DTYPE's."""
    wg = _wg()
    d = wg.HERDT_PLAN_DTYPE
    prog = tmp_path / "plan.c"
    body = "\n".join(f'  printf("{f} %zu\\n", offsetof(wg_herdt_plan, {f}));' for f in d.names)
    prog.write_text(f'#include <stddef.h>\n#include <stdio.h>\n#include "{HEADER}"\nint main(void) {{\n'
                    f'  printf("sizeof %zu\\n", sizeof(wg_herdt_plan));\n{body}\n  return 0;\n}}\n')
    exe = tmp_path / "plan"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(prog)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out["sizeof"]) == d.itemsize == 1888 and d.itemsize % 16 == 0
    for f in d.names:
        assert int(out[f]) == d.fields[f][1], f
