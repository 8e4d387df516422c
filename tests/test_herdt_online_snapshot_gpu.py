"""Whole robots of the on-line Herdt2010 generator: wg_herdt_online_save / restore / copy (HerdtOnline.save, restore,
save_device, restore_device, copy_from).

A record is the robot's state, its deques front first and its {count, running} slot.  What a record means is checked without
trusting save and restore to agree with each other: a RefRobot (the C++ mirror's per-tick logic over the period API, from
test_herdt_online_gpu) seeded with the record's state, its first `count` rows and its running flag must tick bitwise equal to
a robot restored from it.
"""
import ctypes as C
import os
import subprocess
from collections import deque

import numpy as np
import pytest

from test_herdt_online_gpu import RefRobot, _init15

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "walkgen_b200.h")
B = 48
NEVER = (44, 45, 46, 47)          # robots of the scenario that are never started
SAVE_TICKS = (311, 457, 602)      # the scenario's live handle is saved before these ticks
T2 = 420                          # ticks run after a save


def _wg():
    import jrl_walkgen_b200 as wg
    return wg


@pytest.fixture(scope="module")
def mctx(ctx):
    ctx.herdt_set_params()
    ctx.herdt_mpc_set_params()
    return ctx


def _scenario(seed, nticks, n=B):
    """The staggered fleet of test_herdt_online_gpu: starts over ticks 0..39, two restarts of running robots, velocity
    commands with yaw rates (a burst of four inside one QP period), :stoppg at random ticks; NEVER are never started.
    -> (starts {tick: [robot]}, commands [nticks][n])."""
    wg = _wg()
    rng = np.random.default_rng(seed)
    live = [b for b in range(n) if b not in NEVER]
    starts = {}
    for b, t in zip(live, rng.permutation(np.arange(len(live)) % 40)):
        starts.setdefault(int(t), []).append(b)
    for b, t in ((3, 150), (17, 260)):
        starts.setdefault(t, []).append(b)
    cmds = np.zeros((nticks, n), dtype=wg.HERDT_COMMAND_DTYPE)
    for b in range(n):
        for t in rng.choice(np.arange(40, nticks), size=int(nticks / 150), replace=False):
            cmds["flags"][t, b] = wg.CMD_VEL
            cmds["vel"][t, b] = (rng.uniform(-0.2, 0.3), rng.uniform(-0.15, 0.15), rng.uniform(-0.3, 0.3))
    for k, dt in enumerate((0, 4, 9, 15)):
        cmds["flags"][401 + dt, 5] = wg.CMD_VEL
        cmds["vel"][401 + dt, 5] = (0.05 * k, -0.03 * k, 0.1 * (k - 1))
    for b in rng.choice([b for b in live if b not in (3, 17)], size=16, replace=False):
        cmds["flags"][int(rng.integers(60, 560)), b] |= wg.CMD_STOP
    return starts, cmds


def _init_of(b):
    i = _init15(x=0.0316055 + 0.01 * b, y=0.02 * (b % 7))
    i[9] = i[12] = 0.01 * b
    return i


def _tick_to(h, t0, t1, starts, cmds):
    """Ticks [t0, t1) of the scenario on h (starts before their tick) -> rows, running [t1 - t0][B]."""
    rows, run = [], []
    bounds = sorted(set([t0, t1] + [t for t in starts if t0 < t < t1]))
    for a, b in zip(bounds[:-1], bounds[1:]):
        if a in starts:
            h.start(starts[a], np.array([_init_of(r) for r in starts[a]]))
        r, q = h.tick(b - a, cmds[a:b])
        rows.append(r); run.append(q)
    return np.concatenate(rows), np.concatenate(run)


def _ref_from(ctx, rec1):
    """A RefRobot seeded from a record (an array of one): st = record.state, q = deque(record.rows[:count]),
    running = record.running."""
    wg = _wg()
    r = RefRobot(ctx)
    r.st = rec1["state"].copy()
    r.q = deque(np.array(rec1["rows"][0][k], dtype=wg.TICK_DTYPE) for k in range(int(rec1["count"][0])))
    r.running = bool(rec1["running"][0])
    return r


def _ref_ticks(robots, cmds):
    wg = _wg()
    n = len(cmds)
    rows = np.zeros((n, len(robots)), dtype=wg.TICK_DTYPE)
    run = np.zeros((n, len(robots)), dtype=np.int8)
    for t in range(n):
        for b, r in enumerate(robots):
            row, ok = r.tick(cmds[t, b])
            run[t, b] = ok
            if ok:
                rows[t, b] = row
    return rows, run


def _rows_past_count_zero(recs):
    q = _wg().HERDT_ONLINE_QUEUE
    past = np.arange(q)[None, :] >= recs["count"][:, None]
    return (recs["rows"][past].view(np.uint8) == 0).all()


@pytest.fixture(scope="module")
def live(mctx):
    """The scenario's live handle, saved (host and device form) before each of SAVE_TICKS and ticked to the last save + T2."""
    wg = _wg()
    nt = SAVE_TICKS[-1] + T2
    starts, cmds = _scenario(11, nt)
    h = mctx.herdt_online(B)
    saves, dev, t = {}, {}, 0
    rows, run = [], []
    try:
        for ts in SAVE_TICKS + (nt,):
            r, q = _tick_to(h, t, ts, starts, cmds)
            rows.append(r); run.append(q)
            t = ts
            if ts == nt:
                break
            saves[ts] = h.save()
            d = mctx.alloc(B * wg.ONLINE_ROBOT_DTYPE.itemsize)
            h.save_device(B, d)
            dev[ts] = d.download(wg.ONLINE_ROBOT_DTYPE, (B,))
            d.free()
        final = h.save()
        states = h.states()
    finally:
        h.destroy()
    return dict(starts=starts, cmds=cmds, rows=np.concatenate(rows), run=np.concatenate(run), saves=saves, dev=dev,
                final=final, states=states, nt=nt)


@pytest.mark.gpu
def test_saves_hit_every_phase_and_device_saves_equal_host_saves(live):
    """The save ticks catch robots just before a firing tick (9 rows held), on one (28 rows), mid-period, in the ending phase,
    stopped after :stoppg and never started; the device form of a save is bitwise the host form."""
    seen = set()
    for ts, rec in live["saves"].items():
        assert rec.tobytes() == live["dev"][ts].tobytes()
        assert _rows_past_count_zero(rec)
        run, cnt, st = rec["running"] == 1, rec["count"], rec["state"]
        online = run & (st["online_mode"] == 1)
        seen |= {k for k, m in (("before_fire", online & (cnt == 9)), ("on_fire", online & (cnt == 28)),
                                ("mid", online & (cnt > 9) & (cnt < 28)), ("ending", run & (st["ending_phase"] == 1)),
                                ("stopped", ~run & (st["qp_count"] > 0)), ("never", ~run & (st["qp_count"] == 0))) if m.any()}
        idle = ~run
        assert (cnt[idle] == 0).all()
        assert (rec[list(NEVER)].view(np.uint8) == 0).all()
    assert seen == {"before_fire", "on_fire", "mid", "ending", "stopped", "never"}, seen


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["host", "device"])
def test_round_trip_into_a_fresh_handle_continues_bitwise(mctx, live, form):
    """Records saved at a tick, restored into a fresh handle and run under the same commands: rows, running flags, final
    states and final saves equal the live handle's, bitwise."""
    wg = _wg()
    cmds, nt = live["cmds"], live["nt"]
    for ts in SAVE_TICKS:
        rec = live["saves"][ts]
        h = mctx.herdt_online(B)
        try:
            if form == "host":
                h.restore(rec)
            else:
                d = mctx.to_device(rec)
                h.restore_device(B, d)
                d.free()
            assert h.save().tobytes() == rec.tobytes()
            rows, run = _tick_to(h, ts, nt, {t: v for t, v in live["starts"].items() if t >= ts}, cmds)
            final, states = h.save(), h.states()
        finally:
            h.destroy()
        assert nt - ts >= 400
        assert run.tobytes() == live["run"][ts:].tobytes()
        assert rows.tobytes() == live["rows"][ts:].tobytes()
        assert states.tobytes() == live["states"].tobytes()
        assert final.tobytes() == live["final"].tobytes()
    assert live["run"][-1].sum() >= 12 and (live["states"]["fail_count"] == 0).all()
    assert wg.ONLINE_ROBOT_DTYPE.itemsize == 8448


@pytest.mark.gpu
def test_restored_robots_tick_like_the_mirror_seeded_from_the_record(mctx, live):
    """A robot restored from a record and a RefRobot seeded from the same record tick bitwise equal for T2 ticks."""
    wg = _wg()
    ts = SAVE_TICKS[1]
    rec = live["saves"][ts]
    cmds = live["cmds"][ts:ts + T2]
    assert not any(ts <= t < ts + T2 for t in live["starts"])
    h = mctx.herdt_online(B)
    try:
        h.restore(rec)
        rows, run = h.tick(T2, cmds)
        st = h.states()
    finally:
        h.destroy()
    robots = [_ref_from(mctx, rec[b:b + 1]) for b in range(B)]
    ref_rows, ref_run = _ref_ticks(robots, cmds)
    assert np.array_equal(run, ref_run)
    assert rows.tobytes() == ref_rows.tobytes()
    assert st.tobytes() == np.concatenate([r.st for r in robots]).tobytes()
    assert wg.HERDT_ONLINE_QUEUE == 29


@pytest.mark.gpu
def test_records_are_canonical_whatever_the_ring_head(mctx, live):
    """One record restored into robots whose rings sit at different heads, then ticked the same way, saves to equal records
    on every tick: robot k of the handle is saved and restored into itself after k_off[k] ticks, which puts its ring head
    back at row 0, so after M ticks the heads are (M - k_off[k]) mod 29, all different.  The records also equal the live
    robot's at the next save tick.  Rows past count are zero; stopped and never-started robots save as running = 0,
    count = 0 and ignore commands after a restore."""
    wg = _wg()
    ts, t_next = SAVE_TICKS[0], SAVE_TICKS[1]
    rec = live["saves"][ts]
    live_run = rec["running"] == 1
    j = int(np.flatnonzero(live_run & (rec["state"]["online_mode"] == 1) & (rec["state"]["ending_phase"] == 0))[0])
    k_off = (0, 3, 7, 11, 16, 22, 27)
    K = len(k_off)
    g = mctx.herdt_online(K)
    try:
        for k in range(K):                 # robot k starts k ticks late: the rings sit at K different heads
            g.start([k])
            g.tick(1)
        g.tick(33)
        g.restore(np.repeat(rec[j:j + 1], K))
        cj = np.ascontiguousarray(np.repeat(live["cmds"][ts:t_next, j:j + 1], K, axis=1))
        for m in range(t_next - ts):
            for k in range(K):
                if m == k_off[k]:
                    g.restore(g.save([k]), [k])
            r, q = g.tick(1, cj[m:m + 1])
            assert q[0].all() and (r[0].tobytes()[:r.itemsize] * K) == r[0].tobytes(), m
            s = g.save()
            assert (s.tobytes()[:s.itemsize] * K) == s.tobytes(), m
            assert _rows_past_count_zero(s), m
        assert s[0].tobytes() == live["saves"][t_next][j].tobytes()
    finally:
        g.destroy()
    # idle robots (stopped and never started): running = 0, count = 0, and after a restore they ignore commands
    rec = live["saves"][SAVE_TICKS[-1]]
    idle = np.flatnonzero(rec["running"] == 0)
    assert len(idle) >= len(NEVER) + 2
    assert (rec["count"][idle] == 0).all()
    h = mctx.herdt_online(len(idle))
    try:
        h.restore(rec[idle])
        cmds = np.zeros((30, len(idle)), dtype=wg.HERDT_COMMAND_DTYPE)
        cmds["flags"] = wg.CMD_VEL | wg.CMD_STOP
        cmds["vel"] = (0.2, 0.1, 0.1)
        _, run = h.tick(30, cmds)
        assert not run.any()
        assert h.save().tobytes() == rec[idle].tobytes()
    finally:
        h.destroy()


@pytest.mark.gpu
def test_fork_into_branches(mctx, live):
    """32 robots copied four times each into a 128-robot handle, each branch under its own commands: every branch equals a
    RefRobot seeded from its source's record; the branch given the source's own commands equals the source's own
    continuation; the sources are unchanged by the copy and by the branch ticks.  Also a same-handle copy between disjoint
    sets and the NULL-index forms."""
    wg = _wg()
    ts, NB, K, TB = SAVE_TICKS[1], 32, 4, 200
    rec = live["saves"][ts]
    sel = np.concatenate([np.flatnonzero(rec["running"] == 1)[:NB - 2], np.flatnonzero(rec["running"] == 0)[:2]])
    assert len(sel) == NB
    rng = np.random.default_rng(5)
    cmds_src = live["cmds"][ts:ts + TB]
    src = mctx.herdt_online(B)
    dst = mctx.herdt_online(NB * K)
    try:
        src.restore(rec)
        before = src.save()
        dst.copy_from(src, src_idx=np.repeat(sel, K), dst_idx=np.arange(NB * K))
        assert src.save().tobytes() == before.tobytes()
        branch_recs = dst.save()
        assert branch_recs.tobytes() == np.repeat(before[sel], K).tobytes()
        # branch k of source i: 0 its source's commands, 1 other velocities, 2 a stop, 3 no command
        bc = np.zeros((TB, NB * K), dtype=wg.HERDT_COMMAND_DTYPE)
        for i in range(NB):
            bc[:, K * i] = cmds_src[:, sel[i]]
            for t in rng.choice(TB, size=4, replace=False):
                bc["flags"][t, K * i + 1] = wg.CMD_VEL
                bc["vel"][t, K * i + 1] = (rng.uniform(-0.2, 0.3), rng.uniform(-0.15, 0.15), rng.uniform(-0.3, 0.3))
            bc["flags"][int(rng.integers(0, 60)), K * i + 2] = wg.CMD_STOP
        brows, brun = dst.tick(TB, bc)
        bst = dst.states()
        assert src.save().tobytes() == before.tobytes()
        srows, srun = src.tick(TB, cmds_src)
        s_after = src.save()
        d_after = dst.save()
    finally:
        src.destroy(); dst.destroy()
    robots = [_ref_from(mctx, before[sel[i // K]:sel[i // K] + 1]) for i in range(NB * K)]
    ref_rows, ref_run = _ref_ticks(robots, bc)
    assert np.array_equal(brun, ref_run)
    assert brows.tobytes() == ref_rows.tobytes()
    assert bst.tobytes() == np.concatenate([r.st for r in robots]).tobytes()
    own = np.arange(0, NB * K, K)
    assert brun[:, own].tobytes() == srun[:, sel].tobytes()
    assert brows[:, own].tobytes() == srows[:, sel].tobytes()
    assert d_after[own].tobytes() == s_after[sel].tobytes()
    assert not np.array_equal(brows[:, own + 1], brows[:, own])      # the branches did diverge
    assert (bst["ending_phase"][own[:NB - 2] + 2] == 1).all()

    # same handle, disjoint sets; then the NULL-index forms (all robots, and dst 0..n-1 from named sources)
    h = mctx.herdt_online(B)
    g = mctx.herdt_online(B)
    try:
        h.restore(rec)
        a, b = np.arange(0, 10), np.arange(20, 30)
        h.copy_from(h, src_idx=a, dst_idx=b)
        s = h.save()
        assert s[b].tobytes() == rec[a].tobytes()
        keep = np.setdiff1d(np.arange(B), b)
        assert s[keep].tobytes() == rec[keep].tobytes()
        c = live["cmds"][ts:ts + 60].copy()
        c[:, b] = c[:, a]
        r, q = h.tick(60, c)
        assert r[:, a].tobytes() == r[:, b].tobytes() and q[:, a].tobytes() == q[:, b].tobytes()
        g.copy_from(h)
        assert g.save().tobytes() == h.save().tobytes()
        g.restore(rec)
        g.copy_from(h, src_idx=[7, 7, 3])
        s = g.save(); hs = h.save()
        assert s[:3].tobytes() == hs[[7, 7, 3]].tobytes() and s[3:].tobytes() == rec[3:].tobytes()
        g.restore(rec)
        g.copy_from(h, dst_idx=[40, 41])
        s = g.save()
        assert s[[40, 41]].tobytes() == hs[[0, 1]].tobytes() and s[:40].tobytes() == rec[:40].tobytes()
    finally:
        h.destroy(); g.destroy()


def _saves(*hs):
    return [h.save().tobytes() for h in hs]


@pytest.mark.gpu
def test_refusals_change_no_robot(mctx):
    """Every refused call returns WG_ERR_INVALID and leaves every robot of every handle bitwise unchanged."""
    wg = _wg()
    from jrl_walkgen_b200 import _capi
    INVALID = _capi.WG_ERR_INVALID
    H, D = wg.WG_MEM_HOST, wg.WG_MEM_DEVICE
    lib = mctx.lib
    n8 = 8
    a, b, c = mctx.herdt_online(n8), mctx.herdt_online(n8), mctx.herdt_online(n8 + 2)
    other = wg.Context(0)               # a second context on the same device
    x = other.herdt_online(n8)
    d_rec = mctx.alloc(n8 * wg.ONLINE_ROBOT_DTYPE.itemsize + 16)
    try:
        a.start(np.arange(n8)); b.start([1, 3, 5])
        a.tick(31); b.tick(17)
        good = a.save()
        assert (good["running"] == 1).all() and (good["count"] > 0).all()
        base = _saves(a, b, c)
        out = np.zeros(n8 + 1, dtype=wg.ONLINE_ROBOT_DTYPE)

        def ids(v):
            return None if v is None else np.ascontiguousarray(v, dtype=np.int32)

        def P(arr):
            return None if arr is None else arr.ctypes.data

        def save(n, idx, mem=H, where="ok"):
            p = {"ok": out.ctypes.data if mem != D else d_rec.ptr, "null": None, "odd": d_rec.ptr + 8}[where]
            ii = ids(idx)                   # kept alive across the call
            return lib.wg_herdt_online_save(a.h, mem, n, P(ii), p)

        def restore(recs, idx, mem=H, n=None, where="ok"):
            r = np.ascontiguousarray(recs, dtype=wg.ONLINE_ROBOT_DTYPE)
            if mem == D:
                d_rec.upload(r)
            p = {"ok": d_rec.ptr if mem == D else r.ctypes.data, "null": None, "odd": d_rec.ptr + 8}[where]
            ii = ids(idx)
            return lib.wg_herdt_online_restore(a.h, mem, len(r) if n is None else n, P(ii), p)

        def copy(dst, n, didx, src, sidx):
            di, si = ids(didx), ids(sidx)
            return lib.wg_herdt_online_copy(dst.h, n, P(di), src.h, P(si))

        def bad(**kw):
            r = good[:4].copy()
            for f, v in kw.items():
                r[f][2] = v
            return r

        cases = {
            "save: index out of range": lambda: save(2, [0, 8]),
            "save: negative index": lambda: save(2, [-1, 0]),
            "save: n < 0": lambda: save(-1, None),
            "save: n > B, NULL indices": lambda: save(n8 + 1, None),
            "save: NULL records": lambda: save(2, None, where="null"),
            "save: NULL device records": lambda: save(2, None, mem=D, where="null"),
            "save: unknown mem": lambda: save(2, None, mem=7),
            "save: misaligned device records": lambda: save(2, None, mem=D, where="odd"),
            "restore: index out of range": lambda: restore(good[:2], [3, 8]),
            "restore: repeated index": lambda: restore(good[:3], [1, 2, 1]),
            "restore: n < 0": lambda: restore(good[:2], None, n=-1),
            "restore: n > B, NULL indices": lambda: restore(np.concatenate([good, good[:1]]), None),
            "restore: NULL records": lambda: restore(good[:2], None, where="null"),
            "restore: NULL device records": lambda: restore(good[:2], None, mem=D, where="null"),
            "restore: unknown mem": lambda: restore(good[:2], None, mem=7),
            "restore: misaligned device records": lambda: restore(good[:2], None, mem=D, where="odd"),
            "copy: destination out of range": lambda: copy(b, 2, [0, 8], a, [0, 1]),
            "copy: source out of range": lambda: copy(b, 2, [0, 1], a, [0, -3]),
            "copy: repeated destination": lambda: copy(b, 3, [0, 1, 0], a, [0, 1, 2]),
            "copy: a robot both source and destination": lambda: copy(a, 2, [0, 5], a, [5, 6]),
            "copy: NULL source indices meet the destination": lambda: copy(a, 2, [1, 7], a, None),
            "copy: handles of two contexts": lambda: copy(b, 2, None, x, None),
            "copy: handles of two contexts, reversed": lambda: copy(x, 2, None, a, None),
            "copy: n < 0": lambda: copy(b, -1, None, a, None),
            "copy: n > B, NULL indices": lambda: copy(b, n8 + 1, None, c, None),
            "copy: n > source B, NULL source indices": lambda: copy(c, n8 + 1, None, a, None),
        }
        for mem, tag in ((H, "host"), (D, "device")):
            for rule, kw in (("count < 0", dict(count=-1)), ("count > 29", dict(count=30)), ("running = 2", dict(running=2)),
                             ("running = -1", dict(running=-1)), ("running = 0 with rows held", dict(running=0))):
                cases[f"restore {tag}: {rule}"] = (lambda m=mem, k=kw: restore(bad(**k), [4, 5, 6, 7], mem=m))
        for name, call in cases.items():
            rc = call()
            assert rc == INVALID, (name, rc)
            assert _saves(a, b, c) == base, name
            assert x.save().tobytes() == np.zeros(n8, dtype=wg.ONLINE_ROBOT_DTYPE).tobytes(), name
        # the same calls with valid arguments go through
        assert restore(good[:4], [4, 5, 6, 7], mem=D) == 0 and restore(good[:4], [4, 5, 6, 7]) == 0
        assert copy(a, 2, [0, 5], a, [6, 7]) == 0 and copy(c, n8, None, a, None) == 0
        mctx.sync()
    finally:
        d_rec.free()
        a.destroy(); b.destroy(); c.destroy(); x.destroy()
        other.close()


@pytest.mark.gpu
def test_launches_per_call(mctx):
    """save = 1 launch, copy = 1, restore = 1 from host records and 2 from device records, on every call."""
    wg = _wg()
    n = 16
    a, b = mctx.herdt_online(n), mctx.herdt_online(n)
    d = mctx.alloc(n * wg.ONLINE_ROBOT_DTYPE.itemsize)
    try:
        a.start(np.arange(n)); a.tick(25)
        idx = np.arange(n)[::-1].copy()
        rec = a.save()

        def count(f):
            l0 = mctx.launches
            f()
            return mctx.launches - l0

        got = {k: [] for k in ("save_host", "save_device", "copy", "restore_host", "restore_device")}
        for _ in range(3):
            got["save_host"].append(count(lambda: a.save(idx)))
            got["save_device"].append(count(lambda: a.save_device(n, d)))
            got["copy"].append(count(lambda: b.copy_from(a, src_idx=idx)))
            got["restore_host"].append(count(lambda: b.restore(rec, idx)))
            got["restore_device"].append(count(lambda: b.restore_device(n, d, idx)))
        mctx.sync()
    finally:
        d.free(); a.destroy(); b.destroy()
    want = {"save_host": 1, "save_device": 1, "copy": 1, "restore_host": 1, "restore_device": 2}
    assert got == {k: [v] * 3 for k, v in want.items()}, got


@pytest.mark.gpu
def test_migration_between_devices(mctx, live):
    """Save on device 0, restore on device 1, continue: bitwise what staying on device 0 gives."""
    wg = _wg()
    if wg.device_count() < 2:
        pytest.skip("one visible device")
    ts = SAVE_TICKS[1]
    rec, cmds = live["saves"][ts], live["cmds"][ts:ts + T2]
    c1 = wg.Context(1)
    try:
        c1.herdt_set_params(); c1.herdt_mpc_set_params()
        h1 = c1.herdt_online(B)
        h1.restore(rec)
        rows, run = h1.tick(T2, cmds)
        final = h1.save()
        h1.destroy()
    finally:
        c1.close()
    h0 = mctx.herdt_online(B)
    try:
        h0.restore(rec)
        rows0, run0 = h0.tick(T2, cmds)
        final0 = h0.save()
    finally:
        h0.destroy()
    assert run.tobytes() == run0.tobytes() and rows.tobytes() == rows0.tobytes() and final.tobytes() == final0.tobytes()


def test_record_layout_matches_the_header(tmp_path):
    """sizeof and field offsets of wg_herdt_online_robot, compiled against the header, equal ONLINE_ROBOT_DTYPE's."""
    wg = _wg()
    d = wg.ONLINE_ROBOT_DTYPE
    prog = tmp_path / "robot.c"
    fields = ["rows", "state", "count", "running", "pad_"]
    body = "\n".join(f'  printf("{f} %zu\\n", offsetof(wg_herdt_online_robot, {f}));' for f in fields)
    prog.write_text(f'#include <stddef.h>\n#include <stdio.h>\n#include "{HEADER}"\nint main(void) {{\n'
                    f'  printf("sizeof %zu\\n", sizeof(wg_herdt_online_robot));\n{body}\n  return 0;\n}}\n')
    exe = tmp_path / "robot"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(prog)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out["sizeof"]) == d.itemsize == 8448
    assert int(out["rows"]) == 0
    for f in fields:
        assert int(out[f]) == d.fields[f][1], f
    assert d.fields["rows"][0].shape == (wg.HERDT_ONLINE_QUEUE,)
