"""The on-line Kajita2003 generator (wg_kajita_online_*, Context.kajita_online): B walks advanced one 5 ms control tick at a
time, each refilling its queues from its own step stack.

The reference here is the C++ mirror's per-tick logic, restated per walk in Python over the on-line stream with one walk
(Context.kajita_stream(B = 1)): PatternGeneratorInterface::RunOneStepOfTheControlLoop, Kajita branch
(walkgen_host_pgi.cpp:503-542), and the step stack's AddStandardOnLineStep / RemoveFirstStepInTheStack / StopOnLineStep
(:105-130).  Both run the same front-end kernel per walk, so the ZMP reference, feet, step types, clock and running flags
must be bitwise equal; the CoM comes from preview runs that hold other walks, so it agrees within the stream's chunked
tolerances (test_kajita_stream.py::_check_chunked).
"""
import ctypes as C
import os
import subprocess
from collections import deque

import numpy as np
import pytest

import zmpdisc_oracle as zo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "walkgen_b200.h")
GAINS = (0.005, 1.6, 0.814)
COM_H = 0.814
T = 0.005
EXACT = ("zmp_px", "zmp_py", "zmp_theta", "zmp_time", "left", "right", "step_type", "com_z", "com_yaw")


def _wg():
    import jrl_walkgen_b200 as wg
    return wg


def _step(sx, sy, theta=0.0, ss=0.78, ds=0.02):
    wg = _wg()
    s = np.zeros((), dtype=wg.REL_STEP_DTYPE)
    s["sx"], s["sy"], s["theta"], s["ss_time"], s["ds_time"], s["step_type"] = sx, sy, theta, ss, ds, 1
    return s


# ------------------------------------------------------------------------------------------------
# layout (no GPU)
# ------------------------------------------------------------------------------------------------
def test_tick_and_command_layouts_match_the_header(tmp_path):
    wg = _wg()
    fields = {"wg_kajita_tick": wg.KAJITA_TICK_DTYPE, "wg_kajita_command": wg.KAJITA_COMMAND_DTYPE}
    lines = []
    for s, dt in fields.items():
        lines.append(f'  printf("{s} sizeof %zu\\n", sizeof({s}));')
        for f in dt.names:
            lines.append(f'  printf("{s} {f} %zu\\n", offsetof({s}, {f}));')
    lines.append('  printf("chunk %d %d %d %d\\n", WG_KAJITA_ONLINE_CHUNK, WG_KAJITA_PUSH, WG_KAJITA_STANDARD, WG_KAJITA_STOP);')
    prog = tmp_path / "layout.c"
    prog.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "' + HEADER + '"\nint main(void) {\n' + "\n".join(lines)
                    + "\n  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(prog)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines()
    got = {tuple(l.split()[:2]): l.split()[2:] for l in out}
    for s, dt in fields.items():
        assert int(got[(s, "sizeof")][0]) == dt.itemsize
        for f in dt.names:
            assert int(got[(s, f)][0]) == dt.fields[f][1], (s, f)
    assert [int(v) for v in got[("chunk", out[-1].split()[1])]] == [wg.KAJITA_PUSH, wg.KAJITA_STANDARD, wg.KAJITA_STOP]
    assert int(out[-1].split()[1]) == wg.KAJITA_ONLINE_CHUNK
    assert wg.KAJITA_TICK_DTYPE.itemsize % 16 == 0


# ------------------------------------------------------------------------------------------------
# the reference: one walk of the mirror's tick over a one-walk stream
# ------------------------------------------------------------------------------------------------
class RefWalk:
    """One walk of the mirror: step stack, keep parity, on-line flags, queues as a deque of rows."""

    def __init__(self, ctx, params, com_height=COM_H):
        wg = _wg()
        self.ctx, self.p, self.ch = ctx, params, com_height
        self.NL = ctx.gains.NL
        self.s = ctx.kajita_stream(1, params)
        self.running = self.online = self.transition = False
        self.lives = []            # realised step lists of finished walks (start steps and every refill step)

    def _run(self, steps, flags, feet=None):
        wg = _wg()
        self.s.append(np.array([0, len(steps)], dtype=np.int64), np.array(steps, dtype=wg.REL_STEP_DTYPE).reshape(-1),
                      np.array([flags], dtype=np.int32), feet)
        out = self.s.host_outputs()
        self.s.run(**out)
        n, k = int(self.s.sample_offsets[1]), int(self.s.com_counts[0])
        rows = np.zeros(n, dtype=wg.KAJITA_TICK_DTYPE)
        rows["zmp_px"], rows["zmp_py"] = out["zmpref_xy"][:, 0], out["zmpref_xy"][:, 1]
        rows["zmp_theta"] = rows["com_yaw"] = out["zmp_theta"]
        rows["com_z"] = self.ch
        rows["left"], rows["right"], rows["step_type"] = out["left"], out["right"], out["step_type"]
        for i in range(n):                        # the mirror's clock: T accumulated sample by sample
            rows["zmp_time"][i] = self.clock
            self.clock += T
        self.q.extend(rows[i] for i in range(n))
        for j in range(k):                        # CoM of walk samples previewed .. previewed + k - 1
            r = self.q[self.previewed - self.popped + j]
            r["com_x"], r["com_y"] = out["com_out"][j, :3], out["com_out"][j, 3:]
            r["zmp_out"] = out["zmp_out"][j]
        self.previewed += k
        self.realised.extend(np.array(steps, dtype=wg.REL_STEP_DTYPE).reshape(-1))

    def start(self, steps, feet, keep=1):
        wg = _wg()
        self.q, self.stack, self.realised = deque(), deque(), []
        self.clock, self.previewed, self.popped = 0.0, 0, 0
        self.keep = keep
        self._run(steps, wg.STREAM_START, np.asarray(feet, dtype=np.float64).reshape(1, 6))
        self.running = self.online = True
        self.transition = False

    def _standard(self, sx, sy, theta):
        return _step(sx, sy + self.keep * 0.19, theta, self.p.t_single, self.p.t_double)

    def tick(self, cmd=None):
        """-> (row or None, running flag) of one RunOneStepOfTheControlLoop."""
        wg = _wg()
        if not self.running:
            return None, 0
        if cmd is not None and self.online:
            f = int(cmd["flags"])
            if f & wg.KAJITA_PUSH:
                self.stack.append(cmd["step"].copy())
            if f & wg.KAJITA_STANDARD:
                self.stack.append(self._standard(cmd["step"]["sx"], cmd["step"]["sy"], cmd["step"]["theta"]))
                self.keep = -self.keep
            if f & wg.KAJITA_STOP:
                if len(self.stack) % 2 == 0:
                    self.keep = -self.keep
                self.stack.clear()
                self.transition = True
        NL = self.NL
        if self.online and len(self.q) <= 2 * NL + 1:
            if not self.stack:
                self.stack.append(self._standard(0.0, 0.0, 0.0))
                self.keep = -self.keep
            f = self.stack.popleft()
            last = not self.stack and self.transition
            self._run([f], wg.STREAM_FINISH if last else 0)
            if last:
                self.online = self.transition = False
                self.lives.append(np.array(self.realised, dtype=wg.REL_STEP_DTYPE))
        if len(self.q) <= 2 * NL:
            self.running = False
            return None, 0
        self.popped += 1
        return self.q.popleft(), 1

    def destroy(self):
        self.s.destroy()


# ------------------------------------------------------------------------------------------------
# the script: staggered starts, random commands, stops, restarts, very short pushed steps
# ------------------------------------------------------------------------------------------------
def make_script(B, nticks, seed, params):
    wg = _wg()
    rng = np.random.default_rng(seed)
    cmds = np.zeros((nticks, B), dtype=wg.KAJITA_COMMAND_DTYPE)
    u = rng.random((nticks, B))
    std, push = u < 0.006, (u >= 0.006) & (u < 0.014)
    st = cmds["step"]
    st["sx"][std] = rng.uniform(-0.1, 0.2, std.sum()); st["sy"][std] = rng.uniform(-0.02, 0.02, std.sum())
    st["theta"][std] = rng.uniform(-8, 8, std.sum())
    cmds["flags"][std] = wg.KAJITA_STANDARD
    npush = int(push.sum())
    side = rng.choice([-0.19, 0.19], npush)
    st["sx"][push] = rng.uniform(-0.05, 0.15, npush); st["sy"][push] = side + rng.uniform(-0.02, 0.02, npush)
    st["theta"][push] = rng.uniform(-5, 5, npush)
    # as short as the stream accepts: 0.005 s of double support and no single support is a one-sample segment
    st["ss_time"][push] = rng.choice([0.0, 0.0, 0.05, 0.3, 0.7], npush)
    st["ds_time"][push] = rng.choice([0.005, 0.02, 0.1], npush)
    st["step_type"][push] = 1
    cmds["flags"][push] = wg.KAJITA_PUSH
    starts = {}
    stop_at = {}
    for b in range(B):
        starts.setdefault(7 * b, []).append(b)
        if b % 4 != 3:
            # STOP, then no command until the walk has ended (pushes would keep the stack from emptying), except a
            # STANDARD step after the STOP for every eighth walk: it becomes the last step; restart for half of them
            s = int(rng.integers(7 * b + 150, 900))
            cmds[s:2500, b] = np.zeros((), dtype=wg.KAJITA_COMMAND_DTYPE)
            cmds["flags"][s, b] = wg.KAJITA_STOP
            if b % 8 == 0:
                cmds["flags"][s + 3, b] = wg.KAJITA_STANDARD
                cmds["step"]["sx"][s + 3, b] = 0.1
            stop_at[b] = s
            if b % 2 == 0:
                starts.setdefault(int(rng.integers(2500, 2800)), []).append(b)
    lists, feet, keep = {}, {}, {}
    for t, walks in starts.items():
        for b in walks:
            n = int(rng.integers(1, 4))
            side = 1.0 if rng.random() < 0.5 else -1.0
            l = [_step(0.0, side * 0.095)]
            for i in range(n):
                side = -side
                l.append(_step(rng.uniform(0.0, 0.2), side * 0.19, rng.uniform(-5, 5)))
            lists[(t, b)] = np.array(l, dtype=wg.REL_STEP_DTYPE)
            feet[(t, b)] = zo.INIT_FEET + rng.uniform(-0.01, 0.01, 6) * [1, 1, 0, 1, 1, 0]
            keep[(t, b)] = int(rng.choice([-1, 1]))
    return dict(B=B, nticks=nticks, cmds=cmds, starts=starts, lists=lists, feet=feet, keep=keep, stop_at=stop_at)


def drive_handle(ctx, sc, N, mem=None, params=None):
    wg = _wg()
    B, nt = sc["B"], sc["nticks"]
    h = ctx.kajita_online(B, params, com_height=COM_H)
    rows = np.zeros((nt, B), dtype=wg.KAJITA_TICK_DTYPE)
    run = np.zeros((nt, B), dtype=np.int8)
    dev = mem == wg.WG_MEM_DEVICE
    if dev:
        d_rows, d_run = ctx.alloc(rows.nbytes), ctx.alloc(run.nbytes)
        ctx._check(ctx.lib.wg_memset_device(ctx.h, d_rows.ptr, 0xA5, d_rows.nbytes))
        ctx._check(ctx.lib.wg_memset_device(ctx.h, d_run.ptr, 0x7F, d_run.nbytes))
    bounds = sorted(set([0, nt] + [t for t in sc["starts"] if t < nt]))
    try:
        for a, b in zip(bounds[:-1], bounds[1:]):
            if a in sc["starts"]:
                w = sc["starts"][a]
                h.start(w, [sc["lists"][(a, i)] for i in w], [sc["feet"][(a, i)] for i in w], [sc["keep"][(a, i)] for i in w])
            for c0 in range(a, b, N):
                c1 = min(b, c0 + N)
                if dev:
                    r = C.c_void_p(d_rows.ptr + c0 * B * wg.KAJITA_TICK_DTYPE.itemsize)
                    q = C.c_void_p(d_run.ptr + c0 * B)
                    ctx._check(ctx.lib.wg_kajita_online_tick(h.h, wg.WG_MEM_DEVICE, c1 - c0,
                                                             np.ascontiguousarray(sc["cmds"][c0:c1]).ctypes.data, r, q))
                else:
                    rows[c0:c1], run[c0:c1] = h.tick(c1 - c0, sc["cmds"][c0:c1])
        if dev:
            ctx.sync()
            rows = d_rows.download(wg.KAJITA_TICK_DTYPE, (nt, B))
            run = d_run.download(np.int8, (nt, B))
        state = h.state()
    finally:
        h.destroy()
        if dev:
            d_rows.free(); d_run.free()
    return rows, run, state


def drive_reference(ctx, sc, params):
    wg = _wg()
    B, nt = sc["B"], sc["nticks"]
    refs = [RefWalk(ctx, params) for _ in range(B)]
    rows = np.zeros((nt, B), dtype=wg.KAJITA_TICK_DTYPE)
    run = np.zeros((nt, B), dtype=np.int8)
    try:
        for t in range(nt):
            for b in sc["starts"].get(t, []):
                refs[b].start(sc["lists"][(t, b)], sc["feet"][(t, b)], sc["keep"][(t, b)])
            for b in range(B):
                r, q = refs[b].tick(sc["cmds"][t, b])
                if q:
                    rows[t, b] = r
                    run[t, b] = 1
        lives = [r.lives for r in refs]
        state = (np.array([len(r.q) if r.running else 0 for r in refs]), np.array([len(r.stack) for r in refs]),
                 np.array([int(r.running) for r in refs]), np.array([int(r.online) for r in refs]))
    finally:
        for r in refs:
            r.destroy()
    return rows, run, lives, state


def assert_rows(got, want, run):
    assert got.shape == want.shape
    for f in EXACT:
        assert np.array_equal(got[f], want[f]), f
    sel = run == 1
    dx = np.abs(got["com_x"][sel] - want["com_x"][sel]); dy = np.abs(got["com_y"][sel] - want["com_y"][sel])
    assert max(dx[:, 0].max(), dy[:, 0].max()) < 1e-11
    assert max(dx.max(), dy.max()) < 1e-8
    assert np.abs(got["zmp_out"][sel] - want["zmp_out"][sel]).max() < 1e-9


@pytest.fixture(scope="module")
def kctx(ctx):
    wg = _wg()
    ctx.preview_set_gains(wg.preview_gains(*GAINS, wg.MODE_WITHOUT_INITIALPOS))
    return ctx


@pytest.fixture(scope="module")
def script(kctx):
    wg = _wg()
    p = wg.zmpdisc_default_params()
    sc = make_script(64, 3000, 5, p)
    ref = drive_reference(kctx, sc, p)
    return sc, ref, p


# ------------------------------------------------------------------------------------------------
# 1. the reference, bitwise, whatever the number of ticks per call
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 7, 20, 160, 400])
def test_matches_reference_walks_any_ticks_per_call(kctx, script, N):
    sc, (rrows, rrun, _, rstate), p = script
    rows, run, state = drive_handle(kctx, sc, N, params=p)
    assert np.array_equal(run, rrun)
    assert_rows(rows, rrows, run)
    assert not rows[run == 0].view(np.uint8).any()             # host rows of walks not running are zero
    q, s, r, o = state
    assert np.array_equal(s, rstate[1]) and np.array_equal(r, rstate[2]) and np.array_equal(o, rstate[3])
    # the script covers what it is meant to: refills several times within one call, stops and restarts
    assert run[:, ::2].sum(axis=0).min() > 0 and (np.diff(run.astype(int), axis=0) == -1).sum() >= 40
    assert (np.diff(run.astype(int), axis=0) == 1).sum() >= 63 + 20


# ------------------------------------------------------------------------------------------------
# 2. off-line cross-check of whole walks
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_finished_walks_are_the_offline_plan_of_their_steps(kctx, script):
    wg = _wg()
    sc, (rrows, rrun, lives, _), p = script
    rows, run, _ = drive_handle(kctx, sc, 20, params=p)
    NL = kctx.gains.NL
    checked = 0
    for b in range(sc["B"]):
        if not lives[b]:
            continue
        steps = lives[b][0]
        t0 = 7 * b
        n = int(np.argmin(run[t0:, b])) if (run[t0:, b] == 0).any() else len(run) - t0
        got = rows[t0:t0 + n, b]
        plan = kctx.kajita_plan(np.array([0, len(steps)], dtype=np.int64), steps, sc["feet"][(t0, b)].reshape(1, 6), p)
        ns = plan.total_samples
        z = np.zeros((ns, 2)); th = np.zeros(ns); ty = np.zeros((ns, 3), dtype=np.int32)
        left = np.zeros(ns, dtype=wg.KAJITA_FOOT_DTYPE); right = np.zeros(ns, dtype=wg.KAJITA_FOOT_DTYPE)
        plan.discretize(z, th, left, right, ty)
        st = np.zeros((1, 8)); com = np.zeros((ns, 6)); zmp = np.zeros((ns, 2))
        plan.run(st, com, zmp)
        plan.destroy()
        assert n == ns - 2 * NL, (b, n, ns)
        assert np.array_equal(got["zmp_px"], z[:n, 0]) and np.array_equal(got["zmp_py"], z[:n, 1])
        assert np.array_equal(got["zmp_theta"], th[:n]) and np.array_equal(got["step_type"], ty[:n])
        assert np.array_equal(got["left"], left[:n]) and np.array_equal(got["right"], right[:n])
        c = np.hstack([got["com_x"], got["com_y"]])
        dc = np.abs(c - com[:n])
        assert dc[:, [0, 3]].max() < 1e-11 and dc.max() < 1e-8
        assert np.abs(got["zmp_out"] - zmp[:n]).max() < 1e-9
        checked += 1
    assert checked >= 20


# ------------------------------------------------------------------------------------------------
# 3. the mirror's own on-line script (tests/cpp host_api_test kajita2003 OnLine)
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def exe():
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "cpp")], check=True)
    return os.path.join(ROOT, "tests", "cpp", "host_api_test")


@pytest.mark.gpu
def test_mirror_online_script(exe, tmp_path, ctx):
    """:StartOnLineStepSequencing with four steps, default steps while the queues run low, :StopOnLineStepSequencing before
    tick 1000.  The mirror's start leaves its four steps on the stack (its first refill takes the support-foot step again):
    the handle gets them pushed raw, one per tick on ticks 0..3, all before its first refill (the queue starts with 1120
    samples)."""
    wg = _wg()
    out = tmp_path / "online.dat"
    r = subprocess.run([exe, "kajita2003", "OnLine", str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    mirror = np.loadtxt(out)
    ctx.preview_set_gains(wg.preview_gains(0.005, 1.6, 0.8078, wg.MODE_WITHOUT_INITIALPOS))
    h = ctx.kajita_online(1, com_height=0.8078)
    try:
        steps = zo.steps_from_seq("0.0 -0.105 0.0 0.2 0.21 0.0 0.2 -0.21 0.0 0.2 0.21 0.0")
        h.start([0], [steps], [zo.INIT_FEET], [1])
        nt = 40000
        cmds = np.zeros((nt, 1), dtype=wg.KAJITA_COMMAND_DTYPE)
        cmds["step"][:4, 0] = steps
        cmds["flags"][:4, 0] = wg.KAJITA_PUSH
        cmds["flags"][1000, 0] = wg.KAJITA_STOP
        r_, q_ = h.tick(nt, cmds)
    finally:
        h.destroy()
        ctx.preview_set_gains(wg.preview_gains(*GAINS, wg.MODE_WITHOUT_INITIALPOS))
    n = int(q_[:, 0].sum())
    assert n == mirror.shape[0] and q_[:n, 0].all() and not q_[n:, 0].any()
    g = r_[:n, 0]
    got = np.column_stack([(np.arange(n) + 1) * 0.005, g["com_x"][:, 0], g["com_y"][:, 0], g["com_z"], g["com_yaw"],
                           g["com_x"][:, 1], g["com_y"][:, 1], g["zmp_px"], g["zmp_py"],
                           np.ascontiguousarray(g["left"]).view(np.float64).reshape(n, 6),
                           np.ascontiguousarray(g["right"]).view(np.float64).reshape(n, 6)])
    # the file holds 11 significant digits (scientific, 10 after the point)
    tol = 1e-9 * np.abs(mirror) + 1e-15
    tol[:, [1, 2]] += 1e-10
    tol[:, [5, 6]] += 1e-8
    bad = np.abs(got - mirror) > tol
    assert not bad.any(), (np.argwhere(bad)[:5], np.abs(got - mirror).max(axis=0))


# ------------------------------------------------------------------------------------------------
# 4. edges
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_host_and_device_modes_bitwise(kctx, script):
    """Device rows of walks that do not pop are untouched (the byte pattern stays), host rows are zero; popped rows and
    running flags are bitwise equal."""
    wg = _wg()
    sc, _, p = script
    small = dict(sc, nticks=1200)
    hr, hq, hs = drive_handle(kctx, small, 20, params=p)
    dr, dq, ds = drive_handle(kctx, small, 20, mem=wg.WG_MEM_DEVICE, params=p)
    assert np.array_equal(hq, dq)
    assert hr[hq == 1].tobytes() == dr[dq == 1].tobytes()
    assert (dr[dq == 0].view(np.uint8) == 0xA5).all() and not hr[hq == 0].view(np.uint8).any()
    assert all(np.array_equal(a, b) for a, b in zip(hs, ds))


@pytest.mark.gpu
def test_null_rows_and_running_and_ignored_commands(kctx):
    """NULL rows / running advance the walks as the full call does; commands to walks not started, stopped or off line
    change nothing."""
    wg = _wg()
    B = 6
    steps = zo.steps_from_seq("0.0 -0.095 0.0 0.1 0.19 0.0")
    a, b = kctx.kajita_online(B), kctx.kajita_online(B)
    try:
        for h in (a, b):
            h.start([0, 2, 4], [steps] * 3, [zo.INIT_FEET] * 3)
        noise = np.zeros((300, B), dtype=wg.KAJITA_COMMAND_DTYPE)
        noise["flags"][:, [1, 3, 5]] = wg.KAJITA_STANDARD           # walks never started
        noise["step"]["sx"][:, [1, 3, 5]] = 0.1
        ra, qa = a.tick(300, noise)
        for c0 in range(0, 300, 50):
            b.tick(50, None, rows=False, running=(c0 % 100 == 0))
        rb, qb = b.tick(0)
        assert rb.shape == (0, B)
        assert all(np.array_equal(x, y) for x, y in zip(a.state(), b.state()))
        assert not qa[:, [1, 3, 5]].any() and not any(ra[:, [1, 3, 5]].tobytes())
        r1, _ = a.tick(200)
        r2, _ = b.tick(200)
        assert r1.tobytes() == r2.tobytes()
    finally:
        a.destroy(); b.destroy()


@pytest.mark.gpu
def test_refusals_change_nothing(kctx):
    wg = _wg()
    B = 8
    steps = zo.steps_from_seq("0.0 -0.095 0.0 0.1 0.19 0.0 0.1 -0.19 0.0")
    # no gains: WG_ERR_NOT_READY; a default step longer than max_step_time: WG_ERR_INVALID
    bare = wg.Context(0)
    try:
        with pytest.raises(wg.WalkgenError) as ei:
            bare.kajita_online(4)
        assert ei.value.code == -5
    finally:
        bare.close()
    with pytest.raises(wg.WalkgenError) as ei:
        kctx.kajita_online(4, max_step_time=0.5)
    assert ei.value.code == -3
    A, R = kctx.kajita_online(B), kctx.kajita_online(B)
    lib = kctx.lib

    def refused(fn):
        with pytest.raises(wg.WalkgenError) as ei:
            fn()
        assert ei.value.code == -3

    try:
        for h in (A, R):
            h.start(np.arange(0, B, 2), [steps] * 4, [zo.INIT_FEET] * 4, [1, -1, 1, -1])
            h.tick(250)
        long = steps.copy(); long["ss_time"][2] = 0.9
        refused(lambda: A.start([B], [steps], [zo.INIT_FEET]))
        refused(lambda: A.start([1, 1], [steps, steps], [zo.INIT_FEET] * 2))
        refused(lambda: A.start([1, 3], [steps, long], [zo.INIT_FEET] * 2))
        refused(lambda: A.start([1], [steps], [zo.INIT_FEET], [0]))
        refused(lambda: A.start([1], [steps[:0]], [zo.INIT_FEET]))
        refused(lambda: kctx._check(lib.wg_kajita_online_tick(A.h, wg.WG_MEM_HOST, -1, None, None, None)))
        refused(lambda: kctx._check(lib.wg_kajita_online_tick(A.h, 2, 1, None, None, None)))
        for flags, step in ((wg.KAJITA_STOP | wg.KAJITA_PUSH, steps[1]), (wg.KAJITA_STOP | wg.KAJITA_STANDARD, steps[1]),
                            (wg.KAJITA_PUSH | wg.KAJITA_STANDARD, steps[1]), (8, steps[1]), (wg.KAJITA_PUSH, long[2])):
            cmds = np.zeros((30, B), dtype=wg.KAJITA_COMMAND_DTYPE)
            cmds["flags"][29, 6] = flags
            cmds["step"][29, 6] = step
            refused(lambda: A.tick(30, cmds))
        assert all(np.array_equal(x, y) for x, y in zip(A.state(), R.state()))
        cmds = np.zeros((1500, B), dtype=wg.KAJITA_COMMAND_DTYPE)
        cmds["flags"][10, :] = wg.KAJITA_STOP
        ra, qa = A.tick(1500, cmds)
        rr, qr = R.tick(1500, cmds)
        assert ra.tobytes() == rr.tobytes() and qa.tobytes() == qr.tobytes()
        assert qa[0, ::2].all() and not qa[-1].any()
    finally:
        A.destroy(); R.destroy()


def _free_device_memory():
    cudart = C.CDLL("libcudart.so.12")
    free, total = C.c_size_t(), C.c_size_t()
    assert cudart.cudaMemGetInfo(C.byref(free), C.byref(total)) == 0
    return free.value


@pytest.mark.gpu
def test_launches_per_call_and_no_allocation_in_steady_state(kctx):
    """B = 4096 walks started together: every call of 20 ticks is four launches when a walk refills in it (the stream's
    front end and preview, the scatter, the gather) and one when none does; after warm-up no call allocates."""
    wg = _wg()
    B, N = 4096, 20
    steps = zo.steps_from_seq("0.0 -0.095 0.0")
    h = kctx.kajita_online(B)
    d_rows, d_run = kctx.alloc(N * B * wg.KAJITA_TICK_DTYPE.itemsize), kctx.alloc(N * B)
    try:
        h.start(np.arange(B), [steps] * B, np.tile(zo.INIT_FEET, (B, 1)))
        counts, refills = [], []
        free0 = None
        for call in range(48):
            if call == 24:
                kctx.sync()
                free0 = _free_device_memory()
            q0 = h.state()[0]
            l0 = kctx.launches
            h.tick_device(N, None, d_rows, d_run)
            counts.append(kctx.launches - l0)
            refills.append(bool((h.state()[0] > q0 - N).any()))
        kctx.sync()
        free1 = _free_device_memory()
        assert h.state()[2].all()
    finally:
        h.destroy()
        d_rows.free(); d_run.free()
    assert sum(refills) >= 6 and not all(refills)
    assert all(c == (4 if r else 1) for c, r in zip(counts, refills)), list(zip(counts, refills))
    assert free1 == free0
