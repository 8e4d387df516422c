"""The on-line Herdt2010 generator (wg_herdt_online_*, Context.herdt_online): B robots advanced one 5 ms control tick at a
time, each with its own start tick, commands and deques.

The reference here is the C++ mirror's per-tick logic, restated per robot in Python over the period API with one robot and
one period (Context.herdt_mpc_run(B = 1, nsteps = 1)): PatternGeneratorInterface::RunOneStepOfTheControlLoop
(walkgen_host_pgi.cpp:503-542), ZMPVelocityReferencedQP::OnLine (walkgen_host.cpp:550-597) and the buffered start rows of
InitOnLine (walkgen_host.cpp:485-502).  Both run the same device code per robot, so rows, running flags and states must be
bitwise equal.
"""
import ctypes as C
from collections import deque

import numpy as np
import pytest

import herdt_oracle as ho
from test_herdt_mpc_gpu import ACC, rows_from_ticks

TS = 0.005


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
    """The datref-era settings of test_herdt_mpc_gpu.era_ctx; restored afterwards."""
    wg = _wg()
    ctx.herdt_set_params()
    p = wg.herdt_mpc_default_params()
    p.foot_vel_limit = 0.0
    p.return_to_centre = 0
    ctx.herdt_mpc_set_params(p)
    yield ctx
    ctx.herdt_mpc_set_params()


def _back_row(st):
    """The row a state holds as the deques' not-yet-emitted back element (com_back, feet at index 2)."""
    wg = _wg()
    r = np.zeros((), dtype=wg.TICK_DTYPE)
    cb = st["com_back"][0]
    r["com_x"] = cb[0:3]; r["com_y"] = cb[3:6]; r["com_z"] = cb[6]; r["yaw"] = cb[7]; r["dyaw"] = cb[8]
    r["zmp_x"] = cb[9]; r["zmp_y"] = cb[10]
    r["left"] = st["foot"][0, 0, 2]; r["right"] = st["foot"][0, 1, 2]
    return r


class RefRobot:
    """One robot of the C++ mirror: PGI tick, OnLine, deques, over the period API with B = 1."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.running = False
        self.st = None
        self.q = deque()

    def start(self, init15, edit=None):
        wg = _wg()
        st = np.zeros(1, dtype=wg.MPC_STATE_DTYPE)
        init = np.ascontiguousarray(init15, dtype=np.float64)
        self.ctx._check(self.ctx.lib.wg_herdt_mpc_init15(self.ctx.h, wg.WG_MEM_HOST, 1, init.ctypes.data, 0, st.ctypes.data))
        if edit:
            edit(st)
        self.st = st
        self.q = deque(_back_row(st).copy() for _ in range(8))   # TimeBuffer_ / Ts buffered samples
        self.running = True

    def tick(self, cmd=None):
        """-> (row or None, running flag) of one RunOneStepOfTheControlLoop."""
        wg = _wg()
        if not self.running:
            return None, 0
        st = self.st
        if cmd is not None:
            if cmd["flags"] & wg.CMD_VEL:
                st["new_ref"][0] = cmd["vel"]
            if cmd["flags"] & wg.CMD_STOP:
                st["ending_phase"] = 1
        clock = st["clock"][0] + TS
        if st["online_mode"][0]:
            if clock + 0.00001 > st["upper_time_limit"][0]:
                assert len(self.q) + 20 <= wg.HERDT_ONLINE_QUEUE
                t, _, _ = self.ctx.herdt_mpc_run(st, 1, ticks=True)     # advances the clock by Ts and runs the end test
                rows = t[0]
                self.q[-1]["left"] = rows[0]["left"]; self.q[-1]["right"] = rows[0]["right"]
                for k in range(1, 20):
                    self.q.append(np.array(rows[k], dtype=wg.TICK_DTYPE))
                self.q.append(_back_row(st).copy())
            else:
                st["clock"] = clock
                if st["ending_phase"][0] and clock >= st["time_to_stop"][0]:
                    st["online_mode"] = 0
        else:
            st["clock"] = clock
        if not self.q:
            self.running = False
            return None, 0
        return self.q.popleft(), 1


def _init15(x=0.0316055, y=0.0, dx=0.0, dy=0.0, yaw=0.0, feet_dx=0.0):
    return np.array([x, dx, 0.0, y, dy, 0.0, 0.7116911, yaw, 0.0,
                     feet_dx, y + 0.09, 0.0, feet_dx, y - 0.09, 0.0])


def _run_batch(h, nticks, events, commands):
    """Tick the handle over [0, nticks), calling start(idx, init) before the ticks listed in `events` {tick: [(idx, init15,
    edit)]}; returns rows and running [nticks][B]."""
    wg = _wg()
    rows = np.zeros((nticks, h.B), dtype=wg.TICK_DTYPE)
    run = np.zeros((nticks, h.B), dtype=np.int8)
    bounds = sorted(set([0, nticks] + list(events)))
    for a, b in zip(bounds[:-1], bounds[1:]):
        if a in events:
            idx = [i for i, _, _ in events[a]]
            h.start(idx, np.array([init for _, init, _ in events[a]]))
            edits = [(i, e) for i, _, e in events[a] if e]
            if edits:
                st = h.states()
                for i, e in edits:
                    one = st[i:i + 1].copy(); e(one); st[i] = one[0]
                h.set_states(st)
        r, q = h.tick(b - a, commands[a:b])
        rows[a:b] = r; run[a:b] = q
    return rows, run


def _run_reference(ctx, B, nticks, events, commands):
    wg = _wg()
    robots = [RefRobot(ctx) for _ in range(B)]
    rows = np.zeros((nticks, B), dtype=wg.TICK_DTYPE)
    run = np.zeros((nticks, B), dtype=np.int8)
    for t in range(nticks):
        for i, init, e in events.get(t, []):
            robots[i].start(init, e)
        for b, r in enumerate(robots):
            row, ok = r.tick(commands[t, b])
            run[t, b] = ok
            if ok:
                rows[t, b] = row
    return rows, run, robots


@pytest.mark.gpu
def test_online_ticks_bitwise_equal_per_robot_mirror(mctx):
    """48 robots started over ticks 0..39 (every QP phase), two restarts of running robots, velocity commands with yaw
    rates (several inside one QP period: only the last before the instant counts), :stoppg at random ticks; 1500 ticks."""
    wg = _wg()
    rng = np.random.default_rng(2026)
    B, NT = 48, 1500
    starts = rng.permutation(np.arange(B) % 40)
    events = {}
    for b in range(B):
        init = _init15(x=0.0316055 + rng.uniform(-0.5, 0.5), y=rng.uniform(-0.5, 0.5),
                       dx=0.02 if b % 5 == 0 else 0.0, feet_dx=0.0)
        init[9] = init[12] = init[0] - 0.0316055
        events.setdefault(int(starts[b]), []).append((b, init, None))
    for b, t in ((3, 300), (17, 777)):
        events.setdefault(t, []).append((b, _init15(y=0.2 * (b % 2)), None))
    cmds = np.zeros((NT, B), dtype=wg.HERDT_COMMAND_DTYPE)
    for b in range(B):
        for t in rng.choice(np.arange(40, NT - 100), size=6, replace=False):
            cmds["flags"][t, b] = wg.CMD_VEL
            cmds["vel"][t, b] = (rng.uniform(-0.2, 0.3), rng.uniform(-0.15, 0.15), rng.uniform(-0.3, 0.3))
    for b in (5, 6):                                # bursts of commands inside one QP period
        t0 = 401 + 3 * b
        for k, dt in enumerate((0, 4, 9, 15)):
            cmds["flags"][t0 + dt, b] = wg.CMD_VEL
            cmds["vel"][t0 + dt, b] = (0.05 * k, -0.03 * k, 0.1 * (k - 1))
    stoppers = rng.choice([b for b in range(B) if b not in (3, 17)], size=16, replace=False)   # 3 and 17 restart running
    for b in stoppers:
        t = int(rng.integers(100, 1100))
        cmds["flags"][t, b] |= wg.CMD_STOP

    h = mctx.herdt_online(B)
    try:
        rows, run = _run_batch(h, NT, events, cmds)
        st = h.states()
    finally:
        h.destroy()
    ref_rows, ref_run, robots = _run_reference(mctx, B, NT, events, cmds)
    ref_st = np.concatenate([r.st for r in robots])
    assert np.array_equal(run, ref_run)
    assert rows.tobytes() == ref_rows.tobytes()
    assert st.tobytes() == ref_st.tobytes()
    # the inputs did what they are meant to: robots stopped, others still running, yaw commands turned the trunk
    stopped = (run[-1] == 0)
    assert stopped.sum() >= 8 and (~stopped).sum() >= 16
    assert np.abs(st["trunk_yaw"][:, 0]).max() > 0.1 and (st["fail_count"] == 0).all()
    assert (st["qp_count"] > 0).all()


def _check_datref(rows36, gold):
    """_gpu_full_datref's tolerances (test_herdt_mpc_gpu.py) on rows compared from datref row 0."""
    n = len(rows36)
    g = gold[:n, 1:37]
    err = np.abs(rows36 - g)
    VEL = np.zeros(36, bool); VEL[[4, 5]] = True
    tail = gold[:n, 0] > 111.0
    strict = err.copy(); strict[np.ix_(tail, VEL)] = 0.0
    assert strict[:, ~ACC].max() < 1e-6, (strict[:, ~ACC].max(), np.unravel_index((strict * ~ACC).argmax(), err.shape))
    assert err[:, [0, 1, 7, 8]].max() < 5e-7
    if tail.any():
        assert err[np.ix_(tail, VEL)].max() < 2e-6
    assert err[:, ACC].max() < 1e-4
    return err


def _datref_copies(era_ctx, name, script):
    """8 copies of a TestHerdt2010 script in one batch, started at 8 different ticks, events delivered as per-tick commands
    (an event sent after tick t is applied before the copy's tick t + 1)."""
    wg = _wg()
    gold = ho.load_golden(name)
    starts = [0, 1, 5, 8, 13, 19, 26, 37]
    B = len(starts)
    NT = max(starts) + len(gold) + 40

    def edit(st):
        st["sup_steps_left"] = 2; st["nb_steps_ssds"] = 2
        st["sup_x"], st["sup_y"], st["sup_yaw"] = 0.0, 0.1, 0.0

    events = {s: [(c, _init15(), edit)] for c, s in enumerate(starts)}
    cmds = np.zeros((NT, B), dtype=wg.HERDT_COMMAND_DTYPE)
    one = np.zeros(NT, dtype=wg.HERDT_COMMAND_DTYPE)
    for t, v, stop in script:
        one["vel"][t] = v
        one["flags"][t] = wg.CMD_VEL | (wg.CMD_STOP if stop else 0)
    for c, s in enumerate(starts):
        cmds[s:, c] = one[:NT - s]
    h = era_ctx.herdt_online(B)
    try:
        rows, run = _run_batch(h, NT, events, cmds)
    finally:
        h.destroy()
    # the per-robot reference of one copy (the copies are the same robot shifted in time)
    ref_rows, ref_run, _ = _run_reference(era_ctx, 1, NT, {0: [(0, _init15(), edit)]}, one[:, None])
    ref_stop = int(np.argmin(ref_run[:, 0]))
    assert ref_run[:ref_stop, 0].all() and not ref_run[ref_stop:, 0].any()
    assert ref_stop == len(gold), (ref_stop, len(gold))
    worst = 0.0
    for c, s in enumerate(starts):
        r = run[s:, c]
        stop = int(np.argmin(r))
        assert r[:stop].all() and not r[stop:].any() and not run[:s, c].any()
        assert stop == ref_stop, (c, stop, ref_stop)
        mine = rows[s:s + stop, c]
        assert mine.tobytes() == ref_rows[:stop, 0].tobytes()
        err = _check_datref(rows_from_ticks(mine), gold)
        worst = max(worst, err[:, ~ACC].max())
    return worst, len(gold)


@pytest.mark.gpu
def test_online_reproduces_whole_online_datref_from_row_zero(era_ctx):
    worst, n = _datref_copies(era_ctx, "online", ho.ONLINE_SCRIPT)
    print(f"online datref, 8 copies: {n} rows each, max |tick rows - datref| {worst:.2e}")


@pytest.mark.gpu
def test_online_reproduces_whole_emergency_stop_datref_from_row_zero(era_ctx):
    worst, n = _datref_copies(era_ctx, "emergency", ho.EMERGENCY_SCRIPT)
    print(f"emergency datref, 8 copies: {n} rows each, max |tick rows - datref| {worst:.2e}")


def _boundary_setup(rng, B, NT):
    wg = _wg()
    cmds = np.zeros((NT, B), dtype=wg.HERDT_COMMAND_DTYPE)
    for b in range(B):
        for t in rng.choice(NT, size=5, replace=False):
            cmds["flags"][t, b] = wg.CMD_VEL
            cmds["vel"][t, b] = (rng.uniform(-0.2, 0.3), rng.uniform(-0.15, 0.15), rng.uniform(-0.2, 0.2))
    cmds["flags"][60, 2] |= wg.CMD_STOP
    return cmds


@pytest.mark.gpu
def test_online_call_boundaries_and_memory_modes(mctx):
    """tick(N) = N x tick(1) = the device-resident form; robots never started stay untouched (device rows keep their bytes,
    host rows are zero, running 0, state records zero)."""
    wg = _wg()
    rng = np.random.default_rng(7)
    B, NT, T1 = 12, 700, 13
    never = [4, 9]
    first = [0, 1, 2, 3, 5]
    second = [6, 7, 8, 10, 11]
    cmds = _boundary_setup(rng, B, NT)

    def starts(h, k):
        h.start(first if k == 0 else second)

    # (a) two calls
    ha = mctx.herdt_online(B)
    starts(ha, 0)
    ra1, qa1 = ha.tick(T1, cmds[:T1])
    starts(ha, 1)
    ra2, qa2 = ha.tick(NT - T1, cmds[T1:])
    ra, qa, sa = np.concatenate([ra1, ra2]), np.concatenate([qa1, qa2]), ha.states()
    ha.destroy()
    # (b) one tick per call
    hb = mctx.herdt_online(B)
    rb, qb = [], []
    for t in range(NT):
        if t in (0, T1):
            starts(hb, 0 if t == 0 else 1)
        r, q = hb.tick(1, cmds[t:t + 1])
        rb.append(r); qb.append(q)
    rb, qb, sb = np.concatenate(rb), np.concatenate(qb), hb.states()
    hb.destroy()
    # (c) device-resident buffers, rows pre-filled with a byte pattern
    hc = mctx.herdt_online(B)
    d_cmd = mctx.to_device(cmds)
    d_rows = mctx.alloc(NT * B * wg.TICK_DTYPE.itemsize)
    d_run = mctx.alloc(NT * B)
    mctx._check(mctx.lib.wg_memset_device(mctx.h, d_rows.ptr, 0xA5, d_rows.nbytes))
    mctx._check(mctx.lib.wg_memset_device(mctx.h, d_run.ptr, 0x7F, d_run.nbytes))
    starts(hc, 0)
    hc.tick_device(T1, d_cmd, d_rows, d_run)
    starts(hc, 1)
    off = T1 * B
    mctx._check(mctx.lib.wg_herdt_online_tick(hc.h, wg.WG_MEM_DEVICE, NT - T1,
                                              C.c_void_p(d_cmd.ptr + off * wg.HERDT_COMMAND_DTYPE.itemsize),
                                              C.c_void_p(d_rows.ptr + off * wg.TICK_DTYPE.itemsize), C.c_void_p(d_run.ptr + off)))
    mctx.sync()
    rc_ = d_rows.download(wg.TICK_DTYPE, (NT, B)); qc = d_run.download(np.int8, (NT, B)); sc = hc.states()
    hc.destroy(); d_cmd.free(); d_rows.free(); d_run.free()

    assert qa.tobytes() == qb.tobytes() == qc.tobytes()
    assert ra.tobytes() == rb.tobytes()
    assert sa.tobytes() == sb.tobytes() == sc.tobytes()
    live = qa.astype(bool)
    assert ra[live].tobytes() == rc_[live].tobytes()
    assert (rc_[~live].view(np.uint8) == 0xA5).all()             # device rows of idle robots: untouched
    assert (ra[~live].view(np.uint8) == 0).all()                 # host rows of idle robots: zero
    assert not qa[:, never].any() and (sa[never].view(np.uint8) == 0).all()
    assert not qa[:T1, second].any() and qa[T1:, second].all() and qa[:, [0, 1, 3, 5]].all()
    assert not qa[-1, 2] and qa[:100, 2].all()                   # :stoppg at tick 60: robot 2 ran dry and stopped
    assert (sa["qp_count"][[0, 1, 3, 5]] > 30).all() and 0 < sa["qp_count"][2] < 30


@pytest.mark.gpu
def test_online_launches_per_tick_do_not_depend_on_firing(mctx):
    """Four launches per tick whether no robot, some robots or all robots fire, on every call."""
    wg = _wg()
    B = 64
    h = mctx.herdt_online(B)
    try:
        def launches(n):
            out = []
            for _ in range(n):
                l0 = mctx.launches
                h.tick_device(1)
                out.append(mctx.launches - l0)
            mctx.sync()
            return out

        none = launches(5)                               # nothing started
        h.start(np.arange(B))                             # every robot fires on its first tick and every 20 ticks
        q0 = h.states()["qp_count"].copy()
        allf = launches(1)
        assert (h.states()["qp_count"] == q0 + 1).all()
        launches(10)
        h.start(np.arange(0, B, 2))                       # half the robots restarted: they fire now, the others (tick 12) do not
        q0 = h.states()["qp_count"].copy()
        some = launches(1)
        fired = h.states()["qp_count"] - q0
        assert (fired[::2] == 1).all() and (fired[1::2] == 0).all()
        rest = launches(40)
    finally:
        h.destroy()
    counts = none + allf + some + rest
    assert set(counts) == {4}, counts


@pytest.mark.gpu
def test_online_refusals_change_nothing(mctx, ctx):
    """Every refusal returns WG_ERR_INVALID and leaves states and deques as they were (checked bitwise against a twin
    handle that never saw the refused calls); without parameters tick returns what wg_herdt_mpc_run_batch returns."""
    wg = _wg()
    from jrl_walkgen_b200 import _capi
    INVALID = _capi.WG_ERR_INVALID
    B = 6
    rng = np.random.default_rng(3)
    cmds = _boundary_setup(rng, B, 120)
    h, twin = mctx.herdt_online(B), mctx.herdt_online(B)
    try:
        for x in (h, twin):
            x.start([0, 2, 3, 5])
            x.tick(37, cmds[:37])
        st0 = h.states()
        lib = mctx.lib
        i15 = np.ascontiguousarray(np.tile(_init15(), (3, 1)))
        def start(idx, init=i15, n=None, stride=15):
            a = None if idx is None else np.ascontiguousarray(idx, dtype=np.int32)
            nn = len(idx) if n is None else n
            return lib.wg_herdt_online_start(h.h, nn, None if a is None else a.ctypes.data,
                                             None if init is None else init.ctypes.data, stride)
        refused = [start([0, 1], n=-1), start([0, 6, 1]), start([-1, 1, 2]), start([1, 4, 1]), start(None, n=2),
                   start([0, 1], init=None), start([0, 1], stride=-1),
                   lib.wg_herdt_online_tick(h.h, wg.WG_MEM_HOST, -1, None, None, None),
                   lib.wg_herdt_online_tick(h.h, 7, 1, None, None, None)]
        assert refused == [INVALID] * len(refused), refused
        assert lib.wg_herdt_online_create(mctx.h, -1, C.byref(C.c_void_p())) == INVALID
        assert h.states().tobytes() == st0.tobytes()
        ra, qa = h.tick(83, cmds[37:])
        rb, qb = twin.tick(83, cmds[37:])
        assert qa.tobytes() == qb.tobytes() and ra.tobytes() == rb.tobytes() and qa[:, [0, 2, 3, 5]].all()
        assert h.states().tobytes() == twin.states().tobytes()
    finally:
        h.destroy(); twin.destroy()
    # a context without Herdt parameters: the status of wg_herdt_mpc_run_batch
    bare = wg.Context(0)
    try:
        hb = bare.herdt_online(2)
        st = np.zeros(2, dtype=wg.MPC_STATE_DTYPE)
        want = bare.lib.wg_herdt_mpc_run_batch(bare.h, wg.WG_MEM_HOST, 2, 1, st.ctypes.data, None, None, None, None)
        assert want == _capi.WG_ERR_NOT_READY
        assert bare.lib.wg_herdt_online_tick(hb.h, wg.WG_MEM_HOST, 1, None, None, None) == want
        i1 = np.ascontiguousarray(_init15())
        assert bare.lib.wg_herdt_online_start(hb.h, 1, np.zeros(1, np.int32).ctypes.data, i1.ctypes.data, 0) == want
        hb.destroy()
    finally:
        bare.close()
