"""Whole walks of the on-line Kajita2003 generator: wg_kajita_stream_save / restore / copy (KajitaStream.save, restore,
save_device, restore_device, copy_from).

A record is the walk's state between runs (support frame, feet, last step, filter history), its preview state and its
counters; its carry is the last NL-1 ZMP samples the preview has not consumed yet.  Restored and copied walks are checked
against walks that ran the same history.  The preview's CoM bits depend on the run boundaries and, under the per-launch CTA
shape, on the number of walks in a launch; every stream of this module runs under CTA shape 1 (as
test_kajita_stream::test_restart_matches_fresh_stream does) and every bitwise comparison keeps the run boundaries.
"""
import os
import subprocess

import numpy as np
import pytest

from test_kajita_stream import Drive, batch_lists, reference_com, sched_ragged

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "walkgen_b200.h")
GAINS = (0.005, 1.6, 0.8078)
NL1 = 319                         # carry rows at NL = 320
N_LEAD = 640                      # lead-in samples at the default preview_time of 1.6 s
B = 48
NEVER = (44, 45, 46, 47)          # walks of the fleet that are never started
LATE = (40, 41, 42)               # walk LATE[k] starts with the support-foot step alone in run SAVES[k]
RESTART = (0, 36, 37, 38, 39)     # restarted with new lists in run RS (walk 0 after finishing in run 0, the others while open)
SAVES = (3, 8, 13)                # the fleet is saved after these runs
RS = 6


def _wg():
    import jrl_walkgen_b200 as wg
    return wg


@pytest.fixture(scope="module")
def gctx():
    wg = _wg()
    c = wg.Context(0)
    c.preview_set_gains(wg.preview_gains(*GAINS, wg.MODE_WITHOUT_INITIALPOS))
    c.preview_set_cta_shape(1)
    yield c
    c.preview_set_cta_shape(-1)
    c.close()


def _scenario():
    """The 48-walk ragged fleet -> (lists, feet, runs); runs[r] = (steps each walk appends in run r, {walk: (new list, new
    feet)} for the walks that restart in run r).  Walk 0 runs its whole list in run 0; LATE[k] appends its first step alone in
    run SAVES[k]; RESTART walks append one step per run from RS to the last save; NEVER walks have no steps."""
    lists, feet = batch_lists(B, seed=61)
    new, new_feet = batch_lists(len(RESTART), seed=62)
    for b in NEVER:
        lists[b] = lists[b][:0]
    rng = np.random.default_rng(63)
    cur, pos, runs, r = list(lists), np.zeros(B, dtype=int), [], 0
    while r <= SAVES[-1] or any(pos[b] < len(cur[b]) for b in range(B)):
        restarts = {}
        if r == RS:
            for k, b in enumerate(RESTART):
                restarts[b] = (new[k], new_feet[k])
                cur[b], pos[b] = new[k], 0
        take = np.zeros(B, dtype=int)
        for b in range(B):
            left = len(cur[b]) - pos[b]
            if b == 0 and r == 0:
                t = left
            elif b in LATE:
                k = LATE.index(b)
                t = 0 if r < SAVES[k] else 1 if r == SAVES[k] else int(rng.integers(0, 4))
            elif b in RESTART and RS <= r <= SAVES[-1]:
                t = 1
            else:
                t = int(rng.integers(0, 4))
            take[b] = min(t, left)
        pos += take
        runs.append((take, restarts))
        r += 1
    runs.append((np.zeros(B, dtype=int), {}))            # one empty run at the end
    return lists, feet, runs


def _run(d, runs, first):
    """Runs first.. of a scenario on a Drive (restarts applied before their run)."""
    for take, restarts in runs[first:]:
        for b, (lst, f) in restarts.items():
            d.lists[b], d.pos[b], d.done[b] = lst, 0, False
            d.feet[b] = f
        d.step(take)


def _device_save(ctx, s, n):
    wg = _wg()
    dw, dc = ctx.alloc(n * wg.KAJITA_STREAM_WALK_DTYPE.itemsize), ctx.alloc(max(n * s.carry_rows * 16, 16))
    try:
        s.save_device(n, dw, dc if s.with_preview else None)
        ctx.sync()
        return dw.download(wg.KAJITA_STREAM_WALK_DTYPE, (n,)), (dc.download(np.float64, (n, s.carry_rows, 2))
                                                                  if s.with_preview else None)
    finally:
        dw.free(); dc.free()


def _tails_zero(walks, carry):
    count = walks["samples_emitted"] - walks["steps_previewed"]
    past = np.arange(carry.shape[1])[None, :] >= count[:, None]
    return not carry[past].any()


def _same(a, b):
    """Two saves (walks, carry) bitwise equal."""
    return a[0].tobytes() == b[0].tobytes() and (a[1] is None and b[1] is None or a[1].tobytes() == b[1].tobytes())


def _assert_runs_equal(runs_a, runs_b):
    assert len(runs_a) == len(runs_b)
    for r, ((so, co, cnt, oa), (so2, co2, cnt2, ob)) in enumerate(zip(runs_a, runs_b)):
        assert np.array_equal(so, so2) and np.array_equal(co, co2) and np.array_equal(cnt, cnt2), r
        assert oa.keys() == ob.keys()
        for k in oa:
            assert oa[k].tobytes() == ob[k].tobytes(), (r, k)


@pytest.fixture(scope="module")
def live(gctx):
    """The fleet run along its schedule, saved (host and device form) after each of SAVES, with what a continuation from
    each save needs (lists, feet, positions)."""
    lists, feet, runs = _scenario()
    d = Drive(gctx, list(lists), feet.copy())
    saves = {}
    for r in range(len(runs)):
        _run(d, runs[:r + 1], r)
        if r in SAVES:
            saves[r] = dict(rec=d.s.save(), dev=_device_save(gctx, d.s, B), state=d.s.state(), lists=list(d.lists),
                            feet=d.feet.copy(), pos=d.pos.copy(), done=d.done.copy())
    res = dict(runs=runs, d=d, saves=saves, final=d.s.save(), state=d.s.state())
    yield res
    d.s.destroy()


@pytest.mark.gpu
def test_saves_hit_every_phase_and_device_saves_equal_host_saves(live):
    """The saves catch walks never started (all-zero record and carry), just started (the lead-in alone), mid-walk,
    finished and restarted; every record's counters are wg_kajita_stream_state's; carry rows past the count are zero; the
    device form of a save is bitwise the host form."""
    seen = set()
    for r in SAVES:
        sv = live["saves"][r]
        w, c = sv["rec"]
        _, emitted, previewed, is_open = sv["state"]
        assert np.array_equal(w["samples_emitted"], emitted) and np.array_equal(w["steps_previewed"], previewed)
        assert np.array_equal(w["open"], is_open) and not w["pad_"].any()
        assert _same(sv["rec"], sv["dev"])
        assert c.shape == (B, NL1, 2) and _tails_zero(w, c)
        assert np.array_equal(w["steps_previewed"], np.maximum(0, w["samples_emitted"] - NL1))
        for b in range(B):
            e, o = int(w["samples_emitted"][b]), int(w["open"][b])
            if e == 0:
                seen.add("never")
                assert w[b].tobytes() == bytes(w.itemsize) and not c[b].any()
            elif o == 1 and e == N_LEAD:
                seen.add("just started")
            elif o == 1:
                seen.add("mid-walk")
            else:
                seen.add("finished")
            if b in RESTART and r >= RS and e > 0:
                seen.add("restarted")
        for b in NEVER:
            assert w[b].tobytes() == bytes(w.itemsize)
        k = SAVES.index(r)
        assert w["open"][LATE[k]] == 1 and w["samples_emitted"][LATE[k]] == N_LEAD
    assert seen == {"never", "just started", "mid-walk", "finished", "restarted"}, seen
    assert live["saves"][SAVES[0]]["rec"][0]["open"][0] == 0 and live["saves"][SAVES[0]]["rec"][0]["samples_emitted"][0] > 0
    _, _, _, is_open = live["state"]
    assert not is_open.any()


def _com_since_start(runs_out, starts):
    """Per walk b of `starts` (walk -> run of its last START): its CoM and ZMP rows of every run from then on, concatenated."""
    com, zmp = {b: [] for b in starts}, {b: [] for b in starts}
    for r, (so, co, cnt, out) in enumerate(runs_out):
        for b, r0 in starts.items():
            if r >= r0 and cnt[b]:
                com[b].append(out["com_out"][co[b]:co[b] + cnt[b]])
                zmp[b].append(out["zmp_out"][co[b]:co[b] + cnt[b]])
    return ({b: np.concatenate(v) if v else np.zeros((0, 6)) for b, v in com.items()},
            {b: np.concatenate(v) if v else np.zeros((0, 2)) for b, v in zmp.items()})


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["host", "device"])
def test_round_trip_into_a_fresh_stream_continues_bitwise(gctx, live, form):
    """Records saved after a run, restored into a fresh stream and continued along the same remaining schedule: every
    front-end row, every CoM / ZMP row, wg_kajita_stream_state and the final saves equal the live stream's, bitwise.  Each
    walk's CoM over all runs (the live stream's before the save, the restored one's after it) agrees with
    wg_kajita_run_batch on its whole list."""
    runs, d = live["runs"], live["d"]
    for r in SAVES:
        sv = live["saves"][r]
        f = Drive(gctx, list(sv["lists"]), sv["feet"].copy())
        try:
            f.pos[:] = sv["pos"]; f.done[:] = sv["done"]
            walks, carry = sv["rec"]
            if form == "host":
                f.s.restore(walks, carry)
            else:
                dw, dc = gctx.to_device(walks), gctx.to_device(carry)
                f.s.restore_device(B, dw, dc)
                dw.free(); dc.free()
            assert _same(f.s.save(), sv["rec"])
            for a, b in zip(f.s.state()[1:], sv["state"][1:]):
                assert np.array_equal(a, b)
            _run(f, runs, r + 1)
            _assert_runs_equal(f.runs, d.runs[r + 1:])
            for a, b in zip(f.s.state(), live["state"]):
                assert a.tobytes() == b.tobytes()
            assert _same(f.s.save(), live["final"])
            runs_out = d.runs[:r + 1] + f.runs
            final_lists, final_feet = list(f.lists), f.feet.copy()
        finally:
            f.s.destroy()
    # the CoM of every walk since its last START, against the off-line pipeline on the list it ran
    walks_ = [b for b in range(B) if b not in NEVER]
    starts = {b: (RS if b in RESTART else 0) for b in walks_}
    com, zmp = _com_since_start(runs_out, starts)
    ref = reference_com(gctx, [final_lists[b] for b in walks_], final_feet[walks_])
    off = ref["offsets"]
    for j, b in enumerate(walks_):
        k = max(0, int(off[j + 1] - off[j]) - NL1)
        assert len(com[b]) == k, (b, len(com[b]), k)
        dc = np.abs(com[b] - ref["com"][off[j]:off[j] + k])
        assert dc[:, [0, 3]].max(initial=0) < 1e-11 and dc.max(initial=0) < 1e-8, (b, dc.max(axis=0))
        assert np.abs(zmp[b] - ref["zmp"][off[j]:off[j] + k]).max(initial=0) < 1e-9, b
    assert np.abs(live["state"][0][walks_] - ref["state"]).max() < 1e-9


@pytest.mark.gpu
def test_records_are_canonical(gctx):
    """One walk saved from two streams, at index 2 of one that held a longer walk there before and at index 0 of a fresh
    one, gives equal bytes after every run.  A 0.5 s preview_time makes the lead-in 200 samples, so right after the START
    the carry holds 200 of its 319 rows and the longer walk's rows past them are stale on the device: the saves zero them.
    A save after a restore returns the records, in any index order."""
    wg = _wg()
    p = wg.zmpdisc_default_params()
    p.preview_time = 0.5
    lists, feet = batch_lists(6, seed=111)
    order = sorted(range(6), key=lambda b: -len(lists[b]))
    long_, W = lists[order[0]], lists[order[1]]
    assert len(long_) >= 8 and len(W) >= 4
    e0 = long_[:0]
    P = Drive(gctx, [e0, e0, long_, e0], np.tile(feet[0], (4, 1)), params=p)
    Q = Drive(gctx, [W.copy(), e0, e0], np.tile(feet[0], (3, 1)), params=p)
    R = gctx.kajita_stream(4, params=p)
    try:
        for _ in range(3):
            P.step([0, 0, 2, 0])
        P.lists[2], P.pos[2], P.done[2] = W, 0, False
        takes = [1, 2] + [1] * (len(W) - 3)
        for i, t in enumerate(takes):
            P.step([0, 0, t, 0])
            Q.step([t, 0, 0])
            pw, pc = P.s.save()
            qw, qc = Q.s.save()
            assert pw[2].tobytes() == qw[0].tobytes() and pc[2].tobytes() == qc[0].tobytes(), i
            assert _tails_zero(pw, pc) and _tails_zero(qw, qc)
            if i == 0:
                assert pw["samples_emitted"][2] == 200 and pw["steps_previewed"][2] == 0
            R.restore(pw, pc)
            assert _same(R.save(), (pw, pc))
            perm = np.array([3, 1, 0, 2])
            R.restore(pw[perm], pc[perm], idx=perm[::-1].copy())
            assert _same(R.save(perm[::-1].copy()), (pw[perm], pc[perm]))
        assert pw["open"][2] == 0 and qw["open"][0] == 0
    finally:
        P.s.destroy(); Q.s.destroy(); R.destroy()


@pytest.mark.gpu
def test_fork_into_branches(gctx):
    """16 walks copied four times each into a 64-walk stream; branch k of each appends candidate step k and FINISH.  Every
    branch's rows, CoM and final save are bitwise those of a stream that ran the same history and the same candidate with
    the same run boundaries.  The sources save to the same bytes before the copy, after it and after the branches ran.  Also
    a same-stream copy between disjoint sets and the NULL-index forms."""
    wg = _wg()
    NB, K = 16, 4
    lists, feet = batch_lists(NB, seed=71)
    hist = [np.ones(NB, dtype=int)] * 3                  # every walk still open after three runs
    cand = np.zeros(K, dtype=wg.REL_STEP_DTYPE)
    cand["sx"] = (0.05, 0.15, 0.25, 0.1)
    cand["theta"] = (0.0, 5.0, -5.0, 10.0)
    cand["ss_time"], cand["ds_time"], cand["step_type"] = 0.78, 0.02, 1
    S = Drive(gctx, [l.copy() for l in lists], feet.copy())
    Br = gctx.kajita_stream(NB * K)
    T, U = gctx.kajita_stream(NB), gctx.kajita_stream(NB)
    fin = wg.STREAM_FINISH
    try:
        for t in hist:
            S.step(t)
        assert all(len(l) > 3 for l in lists)
        last_sy = np.array([S.lists[i][S.pos[i] - 1]["sy"] for i in range(NB)])

        def cand_steps(k):
            st = np.repeat(cand[k:k + 1], NB)
            st["sy"] = -np.sign(last_sy) * 0.2
            return st

        before = S.s.save()
        Br.copy_from(S.s, src_idx=np.repeat(np.arange(NB), K))
        assert _same(S.s.save(), before)
        bw, bc = Br.save()
        assert bw.tobytes() == np.repeat(before[0], K).tobytes() and bc.tobytes() == np.repeat(before[1], K, axis=0).tobytes()
        steps = np.concatenate([cand_steps(k)[i:i + 1] for i in range(NB) for k in range(K)])
        Br.append(np.arange(NB * K + 1, dtype=np.int64), steps, np.full(NB * K, fin, dtype=np.int32))
        so, co, cnt = Br.sample_offsets.copy(), Br.com_offsets.copy(), Br.com_counts.copy()
        out = Br.host_outputs()
        Br.run(**out)
        assert _same(S.s.save(), before)
        bsave = Br.save()
        for k in range(K):
            R = Drive(gctx, [l.copy() for l in lists], feet.copy())
            try:
                for t in hist:
                    R.step(t)
                R.s.append(np.arange(NB + 1, dtype=np.int64), cand_steps(k), np.full(NB, fin, dtype=np.int32))
                rso, rco, rcnt = R.s.sample_offsets.copy(), R.s.com_offsets.copy(), R.s.com_counts.copy()
                ro = R.s.host_outputs()
                R.s.run(**ro)
                rw, rc = R.s.save()
            finally:
                R.s.destroy()
            for i in range(NB):
                j = K * i + k
                for key in ("zmpref_xy", "zmp_theta", "left", "right", "step_type"):
                    assert out[key][so[j]:so[j + 1]].tobytes() == ro[key][rso[i]:rso[i + 1]].tobytes(), (i, k, key)
                assert cnt[j] == rcnt[i] > 0
                for key in ("com_out", "zmp_out"):
                    assert out[key][co[j]:co[j] + cnt[j]].tobytes() == ro[key][rco[i]:rco[i] + rcnt[i]].tobytes(), (i, k, key)
                assert bsave[0][j].tobytes() == rw[i].tobytes() and bsave[1][j].tobytes() == rc[i].tobytes(), (i, k)
        assert not bsave[0]["open"].any()
        zr = out["zmpref_xy"]
        assert zr[so[0]:so[1]].tobytes() != zr[so[1]:so[2]].tobytes()          # the branches did diverge

        # same stream, disjoint sets; then the NULL-index forms
        T.restore(*before)
        a, b = np.arange(0, 4), np.arange(8, 12)
        T.copy_from(T, src_idx=a, dst_idx=b)
        tw, tc = T.save()
        keep = np.setdiff1d(np.arange(NB), b)
        assert tw[b].tobytes() == before[0][a].tobytes() and tc[b].tobytes() == before[1][a].tobytes()
        assert tw[keep].tobytes() == before[0][keep].tobytes() and tc[keep].tobytes() == before[1][keep].tobytes()
        U.copy_from(T)
        assert _same(U.save(), (tw, tc))
        U.restore(*before)
        U.copy_from(T, src_idx=[7, 7, 3])
        uw, uc = U.save()
        assert uw[:3].tobytes() == tw[[7, 7, 3]].tobytes() and uc[:3].tobytes() == tc[[7, 7, 3]].tobytes()
        assert uw[3:].tobytes() == before[0][3:].tobytes()
        U.restore(*before)
        U.copy_from(T, dst_idx=[14, 15])
        uw, _ = U.save()
        assert uw[[14, 15]].tobytes() == tw[[0, 1]].tobytes() and uw[:14].tobytes() == before[0][:14].tobytes()
    finally:
        S.s.destroy(); Br.destroy(); T.destroy(); U.destroy()


def _saves(*ss):
    return [s.save() for s in ss]


@pytest.mark.gpu
def test_refusals_change_no_walk(gctx):
    """Every refused call returns WG_ERR_INVALID and leaves every walk of every stream, and its counters, bitwise unchanged."""
    wg = _wg()
    from jrl_walkgen_b200 import _capi
    INVALID = _capi.WG_ERR_INVALID
    H, D = wg.WG_MEM_HOST, wg.WG_MEM_DEVICE
    WALK = wg.KAJITA_STREAM_WALK_DTYPE
    lib = gctx.lib
    n8 = 8
    lists, feet = batch_lists(10, seed=81)
    A = Drive(gctx, [l.copy() for l in lists[:n8]], feet[:n8].copy())
    A2 = Drive(gctx, [l.copy() for l in lists[:n8]], feet[:n8].copy())          # A's twin
    C = Drive(gctx, [l.copy() for l in lists], feet.copy())
    NP = Drive(gctx, [l.copy() for l in lists[:n8]], feet[:n8].copy(), with_preview=False)
    gctx.preview_set_gains(wg.preview_gains(0.005, 1.2, 0.8078, wg.MODE_WITHOUT_INITIALPOS))
    try:
        nl = gctx.kajita_stream(n8)                   # NL = 240
    finally:
        gctx.preview_set_gains(wg.preview_gains(*GAINS, wg.MODE_WITHOUT_INITIALPOS))
    other = wg.Context(0)                             # a second context on the same device
    other.preview_set_gains(wg.preview_gains(*GAINS, wg.MODE_WITHOUT_INITIALPOS))
    x = other.kajita_stream(n8)
    d_w, d_c = gctx.alloc((n8 + 1) * WALK.itemsize + 16), gctx.alloc((n8 + 1) * NL1 * 16 + 16)
    a, c, np_ = A.s, C.s, NP.s
    try:
        for t in (np.ones(n8, dtype=int), np.full(n8, 2)):
            A.step(t); A2.step(t); NP.step(t)
        C.step(np.r_[np.ones(4, dtype=int), np.zeros(6, dtype=int)])
        good = a.save()
        npgood = np_.save()
        assert nl.carry_rows == 239 and (good[0]["open"] == 1).all() and npgood[1] is None
        streams = (a, c, np_, nl)
        base = _saves(*streams)
        zero_x = (np.zeros(n8, dtype=WALK), np.zeros((n8, NL1, 2)))
        out_w, out_c = np.zeros(n8 + 1, dtype=WALK), np.zeros((n8 + 1, NL1, 2))

        def ids(v):
            return None if v is None else np.ascontiguousarray(v, dtype=np.int32)

        def P(arr):
            return None if arr is None else arr.ctypes.data

        def save(s, n, idx, mem=H, w="ok", cr="ok"):
            pw = {"ok": d_w.ptr if mem == D else out_w.ctypes.data, "null": None, "odd": d_w.ptr + 8}[w]
            pc = {"ok": d_c.ptr if mem == D else out_c.ctypes.data, "null": None, "odd": d_c.ptr + 8}[cr]
            ii = ids(idx)
            return lib.wg_kajita_stream_save(s.h, mem, n, P(ii), pw, pc)

        def restore(s, rec, idx, mem=H, n=None, w="ok", cr="ok"):
            r = np.ascontiguousarray(rec[0], dtype=WALK)
            cc = np.ascontiguousarray(rec[1] if rec[1] is not None else np.zeros((len(r), 1, 2)))
            if mem == D:
                d_w.upload(r); d_c.upload(cc)
            pw = {"ok": d_w.ptr if mem == D else r.ctypes.data, "null": None, "odd": d_w.ptr + 8}[w]
            pc = {"ok": d_c.ptr if mem == D else cc.ctypes.data, "null": None, "odd": d_c.ptr + 8}[cr]
            ii = ids(idx)
            return lib.wg_kajita_stream_restore(s.h, mem, len(r) if n is None else n, P(ii), pw, pc)

        def copy(dst, n, didx, src, sidx):
            di, si = ids(didx), ids(sidx)
            return lib.wg_kajita_stream_copy(dst.h, n, P(di), src.h, P(si))

        def bad(**kw):
            r = good[0][:4].copy()
            for f, v in kw.items():
                r[f][2] = v
            return r, good[1][:4].copy()

        g4 = (good[0][:4], good[1][:4])
        cases = {
            "save: index out of range": lambda: save(a, 2, [0, 8]),
            "save: negative index": lambda: save(a, 2, [-1, 0]),
            "save: n < 0": lambda: save(a, -1, None),
            "save: n > B, NULL indices": lambda: save(a, n8 + 1, None),
            "save: NULL walks": lambda: save(a, 2, None, w="null"),
            "save: NULL carry with preview": lambda: save(a, 2, None, cr="null"),
            "save: NULL device carry with preview": lambda: save(a, 2, None, mem=D, cr="null"),
            "save: carry without preview": lambda: save(np_, 2, None),
            "save: device carry without preview": lambda: save(np_, 2, None, mem=D),
            "save: unknown mem": lambda: save(a, 2, None, mem=7),
            "save: misaligned device walks": lambda: save(a, 2, None, mem=D, w="odd"),
            "save: misaligned device carry": lambda: save(a, 2, None, mem=D, cr="odd"),
            "restore: index out of range": lambda: restore(a, (good[0][:2], good[1][:2]), [3, 8]),
            "restore: repeated index": lambda: restore(a, (good[0][:3], good[1][:3]), [1, 2, 1]),
            "restore: device records, repeated index": lambda: restore(a, (good[0][:3], good[1][:3]), [1, 2, 1], mem=D),
            "restore: n < 0": lambda: restore(a, g4, None, n=-1),
            "restore: n > B, NULL indices": lambda: restore(a, (np.concatenate([good[0], good[0][:1]]),
                                                                 np.concatenate([good[1], good[1][:1]])), None),
            "restore: NULL walks": lambda: restore(a, g4, None, w="null"),
            "restore: NULL carry with preview": lambda: restore(a, g4, None, cr="null"),
            "restore: NULL device carry with preview": lambda: restore(a, g4, None, mem=D, cr="null"),
            "restore: carry without preview": lambda: restore(np_, (npgood[0][:4], None), None),
            "restore: device carry without preview": lambda: restore(np_, (npgood[0][:4], None), None, mem=D),
            "restore: unknown mem": lambda: restore(a, g4, None, mem=7),
            "restore: misaligned device walks": lambda: restore(a, g4, None, mem=D, w="odd"),
            "restore: misaligned device carry": lambda: restore(a, g4, None, mem=D, cr="odd"),
            "copy: destination out of range": lambda: copy(c, 2, [0, 10], a, [0, 1]),
            "copy: source out of range": lambda: copy(c, 2, [0, 1], a, [0, -3]),
            "copy: repeated destination": lambda: copy(c, 3, [0, 1, 0], a, [0, 1, 2]),
            "copy: a walk both source and destination": lambda: copy(a, 2, [0, 5], a, [5, 6]),
            "copy: NULL source indices meet the destination": lambda: copy(a, 2, [1, 7], a, None),
            "copy: streams of two contexts": lambda: copy(a, 2, None, x, None),
            "copy: streams of two contexts, reversed": lambda: copy(x, 2, None, a, None),
            "copy: NL differs": lambda: copy(a, 2, None, nl, None),
            "copy: NL differs, reversed": lambda: copy(nl, 2, None, a, None),
            "copy: with_preview differs": lambda: copy(a, 2, None, np_, None),
            "copy: with_preview differs, reversed": lambda: copy(np_, 2, None, a, None),
            "copy: n < 0": lambda: copy(c, -1, None, a, None),
            "copy: n > B, NULL indices": lambda: copy(a, n8 + 1, None, c, None),
            "copy: n > source B, NULL source indices": lambda: copy(c, n8 + 1, None, a, None),
        }
        for mem, tag in ((H, "host"), (D, "device")):
            for rule, kw in (("open = 2", dict(open=2)), ("open = -1", dict(open=-1)),
                             ("negative samples_emitted", dict(samples_emitted=-1, steps_previewed=0)),
                             ("steps_previewed off by one", dict(steps_previewed=int(good[0]["steps_previewed"][2]) + 1)),
                             ("open with zero samples", dict(samples_emitted=0, steps_previewed=0, open=1))):
                cases[f"restore {tag}: {rule}"] = (lambda m=mem, k=kw: restore(a, bad(**k), [4, 5, 6, 7], mem=m))
        for name, call in cases.items():
            rc = call()
            assert rc == INVALID, (name, rc)
            got = _saves(*streams)
            assert all(_same(g, h) for g, h in zip(got, base)), name
            assert _same(x.save(), zero_x), name

        # a pending append: every call on the stream, as source or as destination, is refused; the run then gives what the
        # twin gives
        take = np.ones(n8, dtype=int)
        off, steps, flags = A.plan(take)
        a.append(off, steps, flags, A.feet)
        pending = {
            "save": lambda: save(a, 2, None),
            "save, device": lambda: save(a, 2, None, mem=D),
            "restore": lambda: restore(a, g4, [4, 5, 6, 7]),
            "restore, device": lambda: restore(a, g4, [4, 5, 6, 7], mem=D),
            "copy into it": lambda: copy(a, 2, [0, 1], c, [0, 1]),
            "copy from it": lambda: copy(c, 2, [0, 1], a, [0, 1]),
            "copy within it": lambda: copy(a, 2, [0, 1], a, [2, 3]),
        }
        for name, call in pending.items():
            rc = call()
            assert rc == INVALID, (name, rc)
            got = _saves(c, np_, nl)
            assert all(_same(g, h) for g, h in zip(got, base[1:])), name
        A.execute()
        A2.step(take)
        _assert_runs_equal(A.runs, A2.runs)
        assert _same(a.save(), A2.s.save())
        # the same calls with valid arguments go through
        g4 = a.save([0, 1, 2, 3])
        assert restore(a, g4, [4, 5, 6, 7], mem=D) == 0 and restore(a, g4, [4, 5, 6, 7]) == 0
        assert copy(a, 2, [0, 5], a, [6, 7]) == 0 and copy(c, n8, None, a, None) == 0
        gctx.sync()
    finally:
        d_w.free(); d_c.free()
        for s in (a, A2.s, c, np_, nl):
            s.destroy()
        x.destroy()
        other.close()


@pytest.mark.gpu
def test_without_preview_round_trip(gctx):
    """A front-end-only stream saves records with no carry (None), a zero preview state and zero steps previewed; restored
    (host and device form) into fresh streams, the walks continue bitwise."""
    n = 12
    lists, feet = batch_lists(n, seed=91)
    sched = sched_ragged(lists, 92)
    cut = 3
    A = Drive(gctx, [l.copy() for l in lists], feet.copy(), with_preview=False)
    F = Drive(gctx, [l.copy() for l in lists], feet.copy(), with_preview=False)
    G = Drive(gctx, [l.copy() for l in lists], feet.copy(), with_preview=False)
    try:
        assert A.s.carry_rows == 0
        for t in sched[:cut]:
            A.step(t)
        rec = A.s.save()
        w, c = rec
        assert c is None and not w["preview_state"].any() and not w["steps_previewed"].any() and (w["samples_emitted"] > 0).any()
        assert _same(rec, _device_save(gctx, A.s, n))
        F.s.restore(w, None)
        dw = gctx.to_device(w)
        G.s.restore_device(n, dw, None)
        dw.free()
        for d in (F, G):
            d.pos[:] = A.pos; d.done[:] = A.done
            assert _same(d.s.save(), rec)
        k0 = len(A.runs)
        for t in sched[cut:]:
            A.step(t); F.step(t); G.step(t)
        _assert_runs_equal(F.runs, A.runs[k0:])
        _assert_runs_equal(G.runs, A.runs[k0:])
        fin = A.s.save()
        assert _same(F.s.save(), fin) and _same(G.s.save(), fin) and not fin[0]["open"].any()
    finally:
        A.s.destroy(); F.s.destroy(); G.s.destroy()


@pytest.mark.gpu
def test_launches_per_call(gctx):
    """save = 1 launch (host or device records), copy = 1, restore = 1 from host records and 2 from device records."""
    n = 16
    lists, feet = batch_lists(n, seed=101)
    A = Drive(gctx, lists, feet.copy())
    b = gctx.kajita_stream(n)
    d_w, d_c = gctx.alloc(n * 576), gctx.alloc(n * NL1 * 16)
    try:
        for _ in range(2):
            A.step(np.ones(n, dtype=int))
        idx = np.arange(n)[::-1].copy()
        w, c = A.s.save()

        def count(f):
            l0 = gctx.launches
            f()
            return gctx.launches - l0

        got = {k: [] for k in ("save_host", "save_device", "copy", "restore_host", "restore_device")}
        for _ in range(3):
            got["save_host"].append(count(lambda: A.s.save(idx)))
            got["save_device"].append(count(lambda: A.s.save_device(n, d_w, d_c)))
            got["copy"].append(count(lambda: b.copy_from(A.s, src_idx=idx)))
            got["restore_host"].append(count(lambda: b.restore(w, c, idx)))
            got["restore_device"].append(count(lambda: b.restore_device(n, d_w, d_c, idx)))
        gctx.sync()
    finally:
        d_w.free(); d_c.free(); A.s.destroy(); b.destroy()
    want = {"save_host": 1, "save_device": 1, "copy": 1, "restore_host": 1, "restore_device": 2}
    assert got == {k: [v] * 3 for k, v in want.items()}, got


@pytest.mark.gpu
def test_migration_between_devices(gctx):
    """Save on device 0, restore on device 1, continue: bitwise what staying on device 0 gives."""
    wg = _wg()
    if wg.device_count() < 2:
        pytest.skip("one visible device")
    n = 16
    lists, feet = batch_lists(n, seed=121)
    sched = sched_ragged(lists, 122)
    A = Drive(gctx, [l.copy() for l in lists], feet.copy())
    c1 = wg.Context(1)
    try:
        c1.preview_set_gains(wg.preview_gains(*GAINS, wg.MODE_WITHOUT_INITIALPOS))
        c1.preview_set_cta_shape(1)
        for t in sched[:3]:
            A.step(t)
        rec = A.s.save()
        M = Drive(c1, [l.copy() for l in lists], feet.copy())
        M.pos[:] = A.pos; M.done[:] = A.done
        M.s.restore(*rec)
        k0 = len(A.runs)
        for t in sched[3:]:
            A.step(t); M.step(t)
        _assert_runs_equal(M.runs, A.runs[k0:])
        assert _same(M.s.save(), A.s.save())
        M.s.destroy()
    finally:
        A.s.destroy()
        c1.close()


def test_record_layout_matches_the_header(tmp_path):
    """sizeof and field offsets of wg_kajita_stream_walk, compiled against the header, equal KAJITA_STREAM_WALK_DTYPE's."""
    wg = _wg()
    d = wg.KAJITA_STREAM_WALK_DTYPE
    prog = tmp_path / "walk.c"
    fields = list(d.names)
    body = "\n".join(f'  printf("{f} %zu\\n", offsetof(wg_kajita_stream_walk, {f}));' for f in fields)
    prog.write_text(f'#include <stddef.h>\n#include <stdio.h>\n#include "{HEADER}"\nint main(void) {{\n'
                    f'  printf("sizeof %zu\\n", sizeof(wg_kajita_stream_walk));\n{body}\n  return 0;\n}}\n')
    exe = tmp_path / "walk"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-o", str(exe), str(prog)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out["sizeof"]) == d.itemsize == 576
    for f in fields:
        assert int(out[f]) == d.fields[f][1], f
    assert int(out["hist"]) == 240 and int(out["preview_state"]) == 496
    assert fields == ["support", "prev_support", "left", "right", "zmp_theta", "samples_emitted", "final0", "last", "hist",
                      "preview_state", "steps_previewed", "open", "pad_"]
