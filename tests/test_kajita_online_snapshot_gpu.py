"""Whole walks of the on-line Kajita2003 generator (wg_kajita_online_save / restore / copy): checkpoints, rewinds, forks for
footstep lookahead and migration.

A walk is its record (the owned stream's walk, popped, clock, keep and the tick flags), its preview carry, its queue (front
first) and its step stack.  A walk brought back by restore or copy must go on as the original does: the ZMP reference,
feet, step types, clock and running flags bitwise, and the CoM bitwise where the preview sees the same batch, within the
stream's chunked tolerances otherwise (test_kajita_online_gpu.assert_rows).
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import zmpdisc_oracle as zo
from test_kajita_online_gpu import COM_H, GAINS, RefWalk, assert_rows, make_script

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "walkgen_b200.h")
N = 20            # ticks per call


def _wg():
    import jrl_walkgen_b200 as wg
    return wg


@pytest.fixture(scope="module")
def kctx(ctx):
    wg = _wg()
    ctx.preview_set_gains(wg.preview_gains(*GAINS, wg.MODE_WITHOUT_INITIALPOS))
    return ctx


class Fleet:
    """A handle driven by a make_script script, tick by tick in calls of at most N ticks, starts at their ticks."""

    def __init__(self, ctx, sc, B=None, idx=None, params=None):
        self.sc = sc
        self.B = sc["B"] if B is None else B
        self.idx = np.arange(sc["B"]) if idx is None else np.asarray(idx)     # script walk i lives at walk idx[i]
        self.h = ctx.kajita_online(self.B, params, com_height=COM_H)
        self.t = 0
        self.started = -1

    def cmds(self, t0, t1):
        wg = _wg()
        c = np.zeros((t1 - t0, self.B), dtype=wg.KAJITA_COMMAND_DTYPE)
        c[:, self.idx] = self.sc["cmds"][t0:t1]
        return c

    def start_due(self):
        if self.t in self.sc["starts"] and self.started != self.t:
            self.started = self.t
            w = self.sc["starts"][self.t]
            t = self.t
            self.h.start(self.idx[w], [self.sc["lists"][(t, i)] for i in w], [self.sc["feet"][(t, i)] for i in w],
                         [self.sc["keep"][(t, i)] for i in w])

    def run(self, t1, starts=True):
        """-> rows, running of ticks [t, t1), script columns."""
        out_r, out_q = [], []
        while self.t < t1:
            if starts:
                self.start_due()
            nxt = min([t1, self.t + N] + [s for s in self.sc["starts"] if self.t < s < t1])
            r, q = self.h.tick(nxt - self.t, self.cmds(self.t, nxt))
            out_r.append(r[:, self.idx]); out_q.append(q[:, self.idx])
            self.t = nxt
        if not out_r:
            return None, None
        return np.concatenate(out_r), np.concatenate(out_q)

    def destroy(self):
        self.h.destroy()


def _same(a, b):
    wa, ca, qa, sa = a
    wb, cb, qb, sb = b
    return (wa.tobytes() == wb.tobytes() and ca.tobytes() == cb.tobytes() and qa.tobytes() == qb.tobytes()
            and len(sa) == len(sb) and all(x.tobytes() == y.tobytes() for x, y in zip(sa, sb)))


@pytest.fixture(scope="module")
def script():
    wg = _wg()
    p = wg.zmpdisc_default_params()
    return make_script(48, 3000, 17, p), p


# ------------------------------------------------------------------------------------------------
# layout (no GPU)
# ------------------------------------------------------------------------------------------------
def test_online_walk_layout_matches_the_header(tmp_path):
    wg = _wg()
    d = wg.KAJITA_ONLINE_WALK_DTYPE
    lines = ['  printf("sizeof %zu\\n", sizeof(wg_kajita_online_walk));']
    lines += [f'  printf("{f} %zu\\n", offsetof(wg_kajita_online_walk, {f}));' for f in d.names]
    prog = tmp_path / "walk.c"
    prog.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "' + HEADER + '"\nint main(void) {\n' + "\n".join(lines)
                    + "\n  return 0;\n}\n")
    exe = tmp_path / "walk"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(prog)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out["sizeof"]) == d.itemsize == 624
    for f in d.names:
        assert int(out[f]) == d.fields[f][1], f
    assert int(out["stream"]) == 0 and int(out["popped"]) == 576
    assert list(d.names) == ["stream", "popped", "clock", "keep", "running", "online", "transition", "stacked", "pad_"]


# ------------------------------------------------------------------------------------------------
# phases, canonical records, device saves
# ------------------------------------------------------------------------------------------------
SAVE_AT = [0, 14, 300, 600, 900, 1200, 1500, 1800, 2100, 2400, 2600, 2700, 2850, 3000]


def _phases(w):
    e = w["stream"]["samples_emitted"]
    return dict(never=(e == 0) & (w["running"] == 0), fresh=(w["running"] == 1) & (w["popped"] == 0),
                stacked=(w["online"] == 1) & (w["stacked"] > 0), stop_pending=w["transition"] == 1,
                end_phase=(w["online"] == 0) & (w["running"] == 1), stopped=(e > 0) & (w["running"] == 0))


def _check_canonical(h, rec):
    w, c, q, s = rec
    NL1 = h.carry_rows
    for i in range(len(w)):
        e, p = int(w["stream"]["samples_emitted"][i]), int(w["stream"]["steps_previewed"][i])
        nq = e - int(w["popped"][i])
        assert not q[i, nq:].view(np.uint8).any()
        stale = q[i, nq - (e - p):nq] if e > p else q[i, :0]
        assert not stale["com_x"].any() and not stale["com_y"].any() and not stale["zmp_out"].any()
        assert not w["pad_"][i].any() and not w["stream"]["pad_"][i]
        assert not c[i, min(e, NL1):].any()
        assert len(s[i]) == w["stacked"][i]
        if e == 0:
            z = w[i:i + 1].copy()
            assert z["keep"][0] == 1
            z["keep"] = 0
            assert not z.view(np.uint8).any() and not q[i].view(np.uint8).any() and not c[i].any()


@pytest.mark.gpu
def test_saves_cover_every_phase_are_canonical_and_device_saves_equal_host_saves(kctx, script):
    wg = _wg()
    sc, p = script
    F = Fleet(kctx, sc, params=p)
    n = sc["B"]
    R = F.h.ring_rows
    d_w, d_c, d_q = kctx.alloc(n * 624), kctx.alloc(n * F.h.carry_rows * 16), kctx.alloc(n * R * 224)
    seen = {k: False for k in ("never", "fresh", "stacked", "stop_pending", "end_phase", "stopped", "restarted")}
    restarted = set(b for t, ws in sc["starts"].items() if t >= 2500 for b in ws)
    try:
        for t in SAVE_AT:
            F.run(t)
            F.start_due()
            rec = F.h.save()
            _check_canonical(F.h, rec)
            for k, m in _phases(rec[0]).items():
                seen[k] |= bool(m.any())
            w = rec[0]
            for b in restarted:
                if t >= 2500 and w["running"][b] and w["stream"]["samples_emitted"][b] < 2000:
                    seen["restarted"] = True
            # device save: same bytes
            idx = np.arange(n)[::-1].copy()
            stacks = F.h.save_device(n, d_w, d_c, d_q, idx)
            kctx.sync()
            got = (d_w.download(wg.KAJITA_ONLINE_WALK_DTYPE, (n,)), d_c.download(np.float64, (n, F.h.carry_rows, 2)),
                   d_q.download(wg.KAJITA_TICK_DTYPE, (n, R)), stacks)
            want = (rec[0][idx], rec[1][idx], rec[2][idx], [rec[3][i] for i in idx])
            assert _same(got, want), t
            # state() agrees with the records
            qd, st, rn, on = F.h.state()
            assert np.array_equal(st, w["stacked"]) and np.array_equal(rn, w["running"]) and np.array_equal(on, w["online"])
            assert np.array_equal(qd, w["stream"]["samples_emitted"] - w["popped"])
        assert all(seen.values()), seen
    finally:
        F.destroy(); d_w.free(); d_c.free(); d_q.free()


@pytest.mark.gpu
def test_a_restarted_walk_saves_as_a_fresh_one(kctx):
    """Walk 0 walks, stops and restarts over its stale ring; walk 1 starts fresh at the same tick with the same steps and
    commands: the two save to the same bytes."""
    wg = _wg()
    steps = zo.steps_from_seq("0.0 -0.095 0.0 0.1 0.19 0.0 0.1 -0.19 0.0")
    h = kctx.kajita_online(2)
    try:
        h.start([0], [steps], [zo.INIT_FEET], [-1])
        c = np.zeros((1800, 2), dtype=wg.KAJITA_COMMAND_DTYPE)
        c["flags"][5, 0] = wg.KAJITA_PUSH
        c["step"][5, 0] = steps[1]
        c["flags"][400, 0] = wg.KAJITA_STOP
        h.tick(1800, c)
        assert h.state()[2][0] == 0
        h.start([0, 1], [steps, steps], [zo.INIT_FEET] * 2, [1, 1])
        c = np.zeros((250, 2), dtype=wg.KAJITA_COMMAND_DTYPE)
        for col in (0, 1):
            c["flags"][[3, 100], col] = [wg.KAJITA_STANDARD, wg.KAJITA_PUSH]
            c["step"]["sx"][3, col] = 0.1
            c["step"][100, col] = steps[2]
        for k in range(0, 250, 50):
            h.tick(50, c[k:k + 50])
            a, b = h.save([0]), h.save([1])
            assert _same(a, b), k
        assert a[0]["stacked"][0] > 0 or a[0]["popped"][0] > 0
    finally:
        h.destroy()


# ------------------------------------------------------------------------------------------------
# round trips
# ------------------------------------------------------------------------------------------------
def _continue(A, F, t1):
    ra, qa = A.run(t1, starts=False)
    rf, qf = F.run(t1, starts=False)
    return (ra, qa), (rf, qf)


@pytest.mark.gpu
@pytest.mark.parametrize("t0", [14, 900, 1800])
def test_round_trip_into_a_fresh_handle_continues_bitwise(kctx, script, t0):
    """Host save -> restore into a fresh handle at the same indices, and device save -> device restore: both go on bitwise
    for 2 NL + 400 ticks and more (every restored row, the carry and a stop consumed)."""
    wg = _wg()
    sc, p = script
    n = sc["B"]
    NL = kctx.gains.NL
    t1 = min(sc["nticks"], t0 + 2 * NL + 1200)
    sc2 = dict(sc, starts={t: w for t, w in sc["starts"].items() if t <= t0})
    A = Fleet(kctx, sc2, params=p)
    Fh, Fd = Fleet(kctx, sc2, params=p), Fleet(kctx, sc2, params=p)
    try:
        A.run(t0)
        A.start_due()
        rec = A.h.save()
        Fh.h.restore(*rec)
        R = A.h.ring_rows
        d_w, d_c, d_q = kctx.alloc(n * 624), kctx.alloc(n * A.h.carry_rows * 16), kctx.alloc(n * R * 224)
        try:
            stacks = A.h.save_device(n, d_w, d_c, d_q)
            Fd.h.restore_device(n, d_w, d_c, d_q, stacks)
        finally:
            kctx.sync()
            d_w.free(); d_c.free(); d_q.free()
        for F in (Fh, Fd):
            F.t = t0
            assert _same(F.h.save(), rec)
        ra, qa = A.run(t1, starts=False)
        for F in (Fh, Fd):
            rf, qf = F.run(t1, starts=False)
            assert np.array_equal(qa, qf)
            assert ra.tobytes() == rf.tobytes()
            assert _same(F.h.save(), A.h.save())
        assert t1 - t0 >= 2 * NL + 400 and (np.diff(qa.astype(int), axis=0) == -1).any()
    finally:
        A.destroy(); Fh.destroy(); Fd.destroy()


@pytest.mark.gpu
def test_restore_into_other_indices_and_another_B(kctx, script):
    """Restore into permuted indices of a handle of another B: ZMP, feet, step types, clock and running flags bitwise, the
    CoM within the chunked tolerances."""
    sc, p = script
    n = sc["B"]
    NL = kctx.gains.NL
    t0 = 900
    sc2 = dict(sc, starts={t: w for t, w in sc["starts"].items() if t <= t0})
    perm = np.random.default_rng(3).permutation(70)[:n]
    A = Fleet(kctx, sc2, params=p)
    G = Fleet(kctx, sc2, B=70, idx=perm, params=p)
    try:
        A.run(t0)
        A.start_due()
        G.h.restore(*A.h.save(), idx=perm)
        G.t = t0
        ra, qa = A.run(t0 + 2 * NL + 500, starts=False)
        rg, qg = G.run(t0 + 2 * NL + 500, starts=False)
        assert np.array_equal(qa, qg)
        assert_rows(rg, ra, qa)
    finally:
        A.destroy(); G.destroy()


# ------------------------------------------------------------------------------------------------
# forks: footstep lookahead
# ------------------------------------------------------------------------------------------------
def _candidates():
    wg = _wg()
    c = np.zeros(4, dtype=wg.KAJITA_COMMAND_DTYPE)
    c["flags"] = [wg.KAJITA_PUSH, wg.KAJITA_PUSH, wg.KAJITA_STANDARD, wg.KAJITA_STOP]
    c["step"]["sx"] = [0.15, 0.0, 0.1, 0.0]
    c["step"]["sy"] = [0.19, -0.19, 0.0, 0.0]
    c["step"]["theta"] = [5.0, -3.0, 2.0, 0.0]
    c["step"]["ss_time"] = [0.7, 0.3, 0.0, 0.0]
    c["step"]["ds_time"] = [0.1, 0.02, 0.0, 0.0]
    c["step"]["step_type"] = [1, 1, 0, 0]
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("into", ["same_handle", "second_handle"])
def test_fork_into_branches(kctx, into):
    """32 walks fork into 4 branches each, within one handle or into a second; each branch takes another candidate (two
    pushed steps, a standard step, a STOP) and must be the mirror's walk with that command history.  The sources save to the
    same bytes before and after the fork."""
    wg = _wg()
    p = wg.zmpdisc_default_params()
    NL = kctx.gains.NL
    S, K, T0 = 32, 4, 520
    sc = make_script(S, 3000, 29, p)
    sc["starts"] = {t: w for t, w in sc["starts"].items() if t < T0}
    sc["cmds"]["flags"][sc["cmds"]["flags"] == wg.KAJITA_STOP] = 0
    A = Fleet(kctx, sc, B=S + (S * K if into == "same_handle" else 0), params=p)
    D = A if into == "same_handle" else Fleet(kctx, sc, B=S * K, params=p)
    base = S if into == "same_handle" else 0
    src = np.repeat(np.arange(S), K).astype(np.int32)
    dst = (base + np.arange(S * K)).astype(np.int32)
    cand = _candidates()
    T1 = 2 * NL + 1000
    refs = []
    try:
        A.run(T0)
        before = A.h.save(np.arange(S))
        D.h.copy_from(A.h, src_idx=src, dst_idx=dst)
        assert _same(A.h.save(np.arange(S)), before)
        cmds = np.zeros((T1, D.B), dtype=wg.KAJITA_COMMAND_DTYPE)
        cmds[0, dst] = np.tile(cand, S)
        rows, run = [], []
        for k in range(0, T1, N):
            r, q = D.h.tick(min(N, T1 - k), cmds[k:k + N])
            rows.append(r[:, dst]); run.append(q[:, dst])
        rows, run = np.concatenate(rows), np.concatenate(run)
        # the mirror of every branch: the source's script, then the branch's candidate
        want_r = np.zeros_like(rows); want_q = np.zeros_like(run)
        for s in range(S):
            for k in range(K):
                ref = RefWalk(kctx, p)
                refs.append(ref)
                for t in range(T0):
                    for b in sc["starts"].get(t, []):
                        if b == s:
                            ref.start(sc["lists"][(t, b)], sc["feet"][(t, b)], sc["keep"][(t, b)])
                    ref.tick(sc["cmds"][t, s])
                j = s * K + k
                for t in range(T1):
                    r, q = ref.tick(cand[k] if t == 0 else None)
                    if q:
                        want_r[t, j], want_q[t, j] = r, 1
                ref.destroy()
        assert np.array_equal(run, want_q)
        assert_rows(rows, want_r, run)
        assert run.any(axis=0).all() and not run[-1, 3::K].any()       # the STOP branches have ended
    finally:
        A.destroy()
        if D is not A:
            D.destroy()


# ------------------------------------------------------------------------------------------------
# refusals
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusals_change_nothing(kctx):
    wg = _wg()
    B = 6
    steps = zo.steps_from_seq("0.0 -0.095 0.0 0.1 0.19 0.0 0.1 -0.19 0.0")
    A, X = kctx.kajita_online(B), kctx.kajita_online(B)
    lib = kctx.lib

    def refused(fn):
        with pytest.raises(wg.WalkgenError) as ei:
            fn()
        assert ei.value.code == -3

    others = []
    try:
        for h in (A, X):
            h.start([0, 1, 2, 3], [steps] * 4, [zo.INIT_FEET] * 4, [1, -1, 1, -1])
            c = np.zeros((700, B), dtype=wg.KAJITA_COMMAND_DTYPE)
            for k in range(3):          # pushed in the last ticks: at most one is taken by a refill before the save
                c["flags"][695 + k, 1] = wg.KAJITA_PUSH; c["step"][695 + k, 1] = steps[1 + k % 2]
            c["flags"][10, 2] = wg.KAJITA_STOP
            h.tick(700, c)
        ref = A.save()
        st0 = A.state()
        good = X.save()
        w, cy, q, s = good

        def unchanged():
            assert _same(A.save(), ref)
            assert all(np.array_equal(a, b) for a, b in zip(A.state(), st0))

        def bad_record(i, **kw):
            ww = w.copy()
            for k, v in kw.items():
                if k.startswith("stream_"):
                    ww["stream"][k[7:]][i] = v
                else:
                    ww[k][i] = v
            ss = list(s)
            return ww, cy, q, ss

        assert w["stacked"][1] > 0 and w["online"][1] == 1 and w["running"][4] == 0
        cases = [bad_record(1, stream_open=0), bad_record(1, stream_steps_previewed=3), bad_record(1, running=2),
                 bad_record(1, online=-1), bad_record(1, transition=2), bad_record(0, running=0),
                 bad_record(4, transition=1), bad_record(4, online=1), bad_record(1, keep=0), bad_record(1, popped=-1),
                 bad_record(1, popped=int(w["stream"]["samples_emitted"][1]) + 1),
                 bad_record(0, popped=int(w["stream"]["samples_emitted"][0]) - A.ring_rows - 1),
                 bad_record(0, popped=int(w["stream"]["samples_emitted"][0]) - 2 * kctx.gains.NL + 1),
                 bad_record(1, stacked=-1), bad_record(1, stacked=int(w["stacked"][1]) + 1)]
        # a walk off line with a stack: walk 2 has stopped (online 0)
        c2 = bad_record(2, stacked=1)
        c2[3][2] = steps[1:2]
        cases.append(c2)
        badstep = [x.copy() for x in s]
        badstep[1][0]["ss_time"] = 0.95           # longer than max_step_time
        cases.append((w, cy, q, badstep))
        for rec in cases:
            refused(lambda: A.restore(*rec))
            unchanged()
        # device records: the same checks after the read-back
        n = B
        R = A.ring_rows
        d_w, d_c, d_q = kctx.alloc(n * 624), kctx.alloc(n * A.carry_rows * 16), kctx.alloc(n * R * 224)
        others += [d_w, d_c, d_q]
        d_c.upload(cy); d_q.upload(q)
        for rec in cases[:3]:
            d_w.upload(rec[0])
            refused(lambda: A.restore_device(n, d_w, d_c, d_q, rec[3]))
            unchanged()
        # arguments
        refused(lambda: A.restore(w, cy, q, s, idx=[0, 0, 1, 2, 3, 4]))
        refused(lambda: A.restore(w, cy, q, s, idx=[0, 1, 2, 3, 4, B]))
        refused(lambda: kctx._check(lib.wg_kajita_online_restore(A.h, wg.WG_MEM_HOST, B + 1, None, w.ctypes.data, cy.ctypes.data,
                                                                 q.ctypes.data, None, 0)))
        refused(lambda: kctx._check(lib.wg_kajita_online_restore(A.h, 2, B, None, w.ctypes.data, cy.ctypes.data, q.ctypes.data,
                                                                 None, 0)))
        refused(lambda: kctx._check(lib.wg_kajita_online_restore(A.h, wg.WG_MEM_HOST, -1, None, None, None, None, None, 0)))
        refused(lambda: kctx._check(lib.wg_kajita_online_restore(A.h, wg.WG_MEM_HOST, B, None, w.ctypes.data, None,
                                                                 q.ctypes.data, None, 0)))
        refused(lambda: kctx._check(lib.wg_kajita_online_restore(A.h, wg.WG_MEM_DEVICE, B, None, C.c_void_p(d_w.ptr + 8),
                                                                 C.c_void_p(d_c.ptr), C.c_void_p(d_q.ptr), None, 0)))
        buf = np.zeros(8, dtype=wg.REL_STEP_DTYPE)
        total = int(st0[1].sum())
        assert total > 0
        refused(lambda: kctx._check(lib.wg_kajita_online_save(A.h, wg.WG_MEM_HOST, B, None, w.copy().ctypes.data, cy.copy().ctypes.data,
                                                              q.copy().ctypes.data, buf.ctypes.data, total - 1, None)))
        refused(lambda: kctx._check(lib.wg_kajita_online_save(A.h, wg.WG_MEM_HOST, 1, np.array([B], dtype=np.int32).ctypes.data,
                                                              w.copy().ctypes.data, cy.copy().ctypes.data, q.copy().ctypes.data,
                                                              buf.ctypes.data, 8, None)))
        refused(lambda: kctx._check(lib.wg_kajita_online_save(A.h, 2, 1, None, w.copy().ctypes.data, cy.copy().ctypes.data,
                                                              q.copy().ctypes.data, buf.ctypes.data, 8, None)))
        refused(lambda: kctx._check(lib.wg_kajita_online_save(A.h, wg.WG_MEM_DEVICE, 1, None, C.c_void_p(d_w.ptr + 8),
                                                              C.c_void_p(d_c.ptr), C.c_void_p(d_q.ptr), buf.ctypes.data, 8, None)))
        unchanged()
        # copies
        refused(lambda: A.copy_from(A, src_idx=[0, 1], dst_idx=[1, 2]))
        refused(lambda: A.copy_from(X, src_idx=[0, 1], dst_idx=[2, 2]))
        refused(lambda: A.copy_from(X, src_idx=[0], dst_idx=[B]))
        refused(lambda: kctx._check(lib.wg_kajita_online_copy(A.h, -1, None, X.h, None)))
        refused(lambda: kctx._check(lib.wg_kajita_online_copy(A.h, B + 1, None, X.h, None)))
        longer = kctx.kajita_online(B, max_step_time=1.0)
        others.append(longer)
        assert longer.ring_rows != A.ring_rows
        refused(lambda: A.copy_from(longer, src_idx=[0], dst_idx=[5]))
        kctx.preview_set_gains(wg.preview_gains(0.005, 1.2, 0.814, wg.MODE_WITHOUT_INITIALPOS))
        try:
            shortnl = kctx.kajita_online(B)
            others.append(shortnl)
        finally:
            kctx.preview_set_gains(wg.preview_gains(*GAINS, wg.MODE_WITHOUT_INITIALPOS))
        refused(lambda: A.copy_from(shortnl, src_idx=[0], dst_idx=[5]))
        c1 = wg.Context(0)
        try:
            c1.preview_set_gains(wg.preview_gains(*GAINS, wg.MODE_WITHOUT_INITIALPOS))
            Y = c1.kajita_online(B)
            refused(lambda: A.copy_from(Y, src_idx=[0], dst_idx=[5]))
            Y.destroy()
        finally:
            c1.close()
        unchanged()
    finally:
        A.destroy(); X.destroy()
        for o in others:
            (o.free if hasattr(o, "free") else o.destroy)()


# ------------------------------------------------------------------------------------------------
# launches, allocation, migration
# ------------------------------------------------------------------------------------------------
def _free_device_memory():
    cudart = C.CDLL("libcudart.so.12")
    free, total = C.c_size_t(), C.c_size_t()
    assert cudart.cudaMemGetInfo(C.byref(free), C.byref(total)) == 0
    return free.value


@pytest.mark.gpu
def test_launches_per_call_and_no_allocation_in_steady_state(kctx):
    """save, restore and copy are two launches each, host or device records; a device save or copy allocates nothing once
    its buffers exist."""
    wg = _wg()
    n = 64
    steps = zo.steps_from_seq("0.0 -0.095 0.0 0.1 0.19 0.0")
    A, Bh = kctx.kajita_online(n), kctx.kajita_online(n)
    R = A.ring_rows
    d_w, d_c, d_q = kctx.alloc(n * 624), kctx.alloc(n * A.carry_rows * 16), kctx.alloc(n * R * 224)
    try:
        A.start(np.arange(n), [steps] * n, np.tile(zo.INIT_FEET, (n, 1)))
        A.tick(300)
        rec = A.save()
        idx = np.arange(n)[::-1].copy()

        def count(f):
            l0 = kctx.launches
            f()
            return kctx.launches - l0

        got = {k: [] for k in ("save_host", "save_device", "copy", "restore_host", "restore_device")}
        for it in range(4):
            if it == 2:
                kctx.sync()
                free0 = _free_device_memory()
            got["save_host"].append(count(lambda: A.save(idx)))
            got["save_device"].append(count(lambda: A.save_device(n, d_w, d_c, d_q)))
            got["copy"].append(count(lambda: Bh.copy_from(A, src_idx=idx)))
            got["restore_host"].append(count(lambda: Bh.restore(*rec, idx=idx)))
            got["restore_device"].append(count(lambda: Bh.restore_device(n, d_w, d_c, d_q, rec[3])))
        kctx.sync()
        free1 = _free_device_memory()
    finally:
        A.destroy(); Bh.destroy(); d_w.free(); d_c.free(); d_q.free()
    assert got == {k: [2] * 4 for k in got}, got
    assert free1 == free0


@pytest.mark.gpu
def test_migration_between_devices(kctx, script):
    """Save on device 0, restore on device 1, go on: bitwise what staying on device 0 gives."""
    wg = _wg()
    if wg.device_count() < 2:
        pytest.skip("one visible device")
    sc, p = script
    NL = kctx.gains.NL
    t0 = 900
    sc2 = dict(sc, starts={t: w for t, w in sc["starts"].items() if t <= t0})
    A = Fleet(kctx, sc2, params=p)
    c1 = wg.Context(1)
    try:
        c1.preview_set_gains(wg.preview_gains(*GAINS, wg.MODE_WITHOUT_INITIALPOS))
        M = Fleet(c1, sc2, params=p)
        A.run(t0)
        A.start_due()
        M.h.restore(*A.h.save())
        M.t = t0
        ra, qa = A.run(t0 + 2 * NL + 400, starts=False)
        rm, qm = M.run(t0 + 2 * NL + 400, starts=False)
        assert np.array_equal(qa, qm)
        assert_rows(rm, ra, qa)
        M.destroy()
    finally:
        A.destroy()
        c1.close()
