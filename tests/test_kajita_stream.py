"""On-line Kajita2003 generator (wg_kajita_stream): footsteps appended to running walks, ZMP reference, feet and CoM streamed.

The front end is bitwise the off-line one (wg_zmpdisc_run_batch on each walk's whole list) under any schedule of appends.
The CoM is bitwise wg_kajita_run_batch when whole walks go in one run, and within the tolerances test_preview.py uses
between kernel shapes when the preview runs in chunks (the scan tiles then fall on other ticks).
"""
import numpy as np
import pytest

import zmpdisc_oracle as zo

PROFILES = ("StraightWalking", "Circle", "PbFlorentSeq1", "PbFlorentSeq2")
DATREF_TOL = 1.2e-7
GAINS = (0.005, 1.6, 0.8078)


@pytest.fixture(scope="module")
def sctx():
    import jrl_walkgen_b200 as wg
    c = wg.Context(0)
    c.preview_set_gains(wg.preview_gains(*GAINS, wg.MODE_WITHOUT_INITIALPOS))
    yield c
    c.close()


def _cat(lists):
    import jrl_walkgen_b200 as wg
    off = np.concatenate([[0], np.cumsum([len(s) for s in lists])]).astype(np.int64)
    return off, np.concatenate(lists).astype(wg.REL_STEP_DTYPE)


def batch_lists(B, seed):
    from jrl_walkgen_b200 import workloads as W
    off, steps, feet = W.kajita_steps_batch(B, seed=seed)
    return [steps[off[b]:off[b + 1]].copy() for b in range(B)], feet


def edge_lists():
    """The walks of test_zmpdisc.py::test_cuda_edge_cases_match_oracle."""
    rng = np.random.default_rng(11)
    base = zo.profile_steps("PbFlorentSeq1")
    timed = base.copy()
    timed["ss_time"] = rng.uniform(0.4, 1.2, len(base)).round(2)
    timed["ds_time"] = rng.uniform(0.02, 0.3, len(base)).round(2)
    over = zo.profile_steps("StraightWalking").copy()
    over["step_type"][4:9] = [3, 4, 5, 3, 4]
    short = zo.profile_steps("StraightWalking").copy()
    short["ss_time"][5], short["ds_time"][5] = 0.03, 0.01
    lists = [base[:1].copy(), timed, over, short, zo.profile_steps("Circle")]
    feet = np.tile(zo.INIT_FEET, (len(lists), 1))
    feet[1] = [0.01, 0.1, 5.0, -0.01, -0.09, -3.0]
    return lists, feet


def edge_params():
    import jrl_walkgen_b200 as wg
    p = wg.zmpdisc_default_params()
    p.omega = 4.0
    p.zmp_neutral[0], p.zmp_neutral[1] = 0.01, -0.005
    p.zmp_shift[0], p.zmp_shift[1], p.zmp_shift[2], p.zmp_shift[3] = 0.015, 0.02, 0.01, 0.005
    p.step_height = 0.05
    p.t_single, p.t_double = 0.7, 0.1
    return p


# ---- schedules: per run, the number of steps each walk appends ------------------------------------------------------
def sched_one(lists):
    return [np.ones(len(lists), dtype=int)] * (max(len(s) for s in lists))


def sched_whole(lists):
    return [np.array([len(s) for s in lists])]


def sched_ragged(lists, seed):
    rng = np.random.default_rng(seed)
    left = np.array([len(s) for s in lists])
    runs = []
    while left.sum() > 0:
        take = np.minimum(rng.integers(0, 4, len(lists)), left)
        runs.append(take)
        left = left - take
    runs.append(np.zeros(len(lists), dtype=int))     # one empty run at the end
    return runs


class Drive:
    """Pushes walks through a stream along a schedule; a walk starts with its first append and finishes with its last.
    Collects, per walk, the concatenated front-end samples and, in the layout of wg_kajita_run_batch, the CoM / ZMP."""

    def __init__(self, ctx, lists, feet, params=None, with_preview=True, mem=None, ref_offsets=None):
        import jrl_walkgen_b200 as wg
        self.wg, self.ctx, self.lists, self.feet = wg, ctx, lists, np.ascontiguousarray(feet, dtype=np.float64)
        self.B = len(lists)
        self.s = ctx.kajita_stream(self.B, params, with_preview)
        self.mem = wg.WG_MEM_HOST if mem is None else mem
        self.pos = np.zeros(self.B, dtype=int)
        self.done = np.zeros(self.B, dtype=bool)
        self.samples = [[] for _ in range(self.B)]
        self.ref_offsets = ref_offsets
        if ref_offsets is not None:
            n = int(ref_offsets[-1])
            self.com, self.zmp = np.zeros((n, 6)), np.zeros((n, 2))
        self.previewed = np.zeros(self.B, dtype=np.int64)
        self.com_count = 0
        self.runs = []

    def plan(self, take):
        wg = self.wg
        flags = np.zeros(self.B, dtype=np.int32)
        chunks = []
        for b in range(self.B):
            t = int(take[b]) if not self.done[b] else 0
            p = self.pos[b]
            if t > 0 and p == 0:
                flags[b] |= wg.STREAM_START
            if t > 0 and p + t == len(self.lists[b]):
                flags[b] |= wg.STREAM_FINISH
                self.done[b] = True
            chunks.append(self.lists[b][p:p + t])
            self.pos[b] = p + t
        off, steps = _cat(chunks)
        return off, steps, flags

    def step(self, take):
        off, steps, flags = self.plan(take)
        self.s.append(off, steps, flags, self.feet)
        return self.execute()

    def execute(self):
        wg, s = self.wg, self.s
        so, co, cnt = s.sample_offsets.copy(), s.com_offsets.copy(), s.com_counts.copy()
        out = s.host_outputs(com=s.with_preview)
        if self.mem == wg.WG_MEM_HOST:
            s.run(**out)
        else:
            dev = {}
            for k, a in out.items():
                dev[k] = self.ctx.alloc(max(a.nbytes, 16))
                self.ctx.lib.wg_memset_device(self.ctx.h, dev[k].ptr, 0, max(a.nbytes, 16))
            s.run(**dev, mem=wg.WG_MEM_DEVICE)
            self.ctx.sync()
            for k, a in out.items():
                out[k] = dev[k].download(a.dtype, a.shape)
                dev[k].free()
        z, th = out["zmpref_xy"], out["zmp_theta"]
        left = out["left"].view(np.float64).reshape(-1, 6)
        right = out["right"].view(np.float64).reshape(-1, 6)
        for b in range(self.B):
            a, e = int(so[b]), int(so[b + 1])
            if e > a:
                self.samples[b].append((z[a:e], th[a:e], left[a:e], right[a:e], out["step_type"][a:e]))
        if s.with_preview:
            self.com_count += int(cnt.sum())
            if self.ref_offsets is not None:
                for b in np.nonzero(cnt)[0]:
                    k, r = int(cnt[b]), int(self.ref_offsets[b] + self.previewed[b])
                    self.com[r:r + k] = out["com_out"][co[b]:co[b] + k]
                    self.zmp[r:r + k] = out["zmp_out"][co[b]:co[b] + k]
            self.previewed += cnt
        self.runs.append((so, co, cnt, out))
        return out

    def walk(self, b):
        parts = self.samples[b]
        return tuple(np.concatenate([p[i] for p in parts]) for i in range(5))


def reference_front(ctx, lists, feet, params=None):
    import jrl_walkgen_b200 as wg
    off, steps = _cat(lists)
    plan = ctx.kajita_plan(off, steps, feet, params)
    n = plan.total_samples
    z = np.zeros((n, 2)); th = np.zeros(n); types = np.zeros((n, 3), dtype=np.int32)
    left = np.zeros(n, dtype=wg.KAJITA_FOOT_DTYPE); right = np.zeros(n, dtype=wg.KAJITA_FOOT_DTYPE)
    plan.discretize(z, th, left, right, types)
    so = plan.sample_offsets
    left, right = left.view(np.float64).reshape(n, 6), right.view(np.float64).reshape(n, 6)
    plan.destroy()
    return [(z[so[b]:so[b + 1]], th[so[b]:so[b + 1]], left[so[b]:so[b + 1]], right[so[b]:so[b + 1]], types[so[b]:so[b + 1]])
            for b in range(len(lists))]


def reference_com(ctx, lists, feet):
    off, steps = _cat(lists)
    plan = ctx.kajita_plan(off, steps, feet)
    n, B = plan.total_samples, len(lists)
    st = np.zeros((B, 8)); com = np.zeros((n, 6)); zmp = np.zeros((n, 2)); zref = np.zeros((n, 2))
    plan.run(st, com, zmp, zref)
    res = dict(offsets=plan.sample_offsets.copy(), total_steps=plan.total_steps, state=st, com=com, zmp=zmp, zref=zref)
    plan.destroy()
    return res


def assert_front_equal(d, ref):
    for b, want in enumerate(ref):
        got = d.walk(b)
        for name, g, w in zip(("zmpref", "theta", "left", "right", "types"), got, want):
            assert g.shape == w.shape and np.array_equal(g, w), (b, name)


# ------------------------------------------------------------------------------------------------
# 1. front end, bitwise, any schedule
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("schedule", ["one", "ragged", "whole"])
def test_front_end_bitwise_any_schedule(sctx, schedule):
    lists, feet = batch_lists(96, seed=3)
    lists += [zo.profile_steps(n) for n in PROFILES]
    feet = np.vstack([feet, np.tile(zo.INIT_FEET, (len(PROFILES), 1))])
    ref = reference_front(sctx, lists, feet)
    runs = {"one": sched_one, "whole": sched_whole, "ragged": lambda l: sched_ragged(l, 7)}[schedule](lists)
    d = Drive(sctx, lists, feet, with_preview=False)
    for take in runs:
        d.step(take)
    assert_front_equal(d, ref)
    _, emitted, _, is_open = d.s.state()
    assert np.array_equal(emitted, [len(r[0]) for r in ref]) and not is_open.any()
    for i, name in enumerate(PROFILES):   # the datrefs of TestKajita2003
        b = 96 + i
        z, _, left, right, _ = d.walk(b)
        g = zo.golden(name)
        err = np.abs(np.hstack([left[:len(g)], right[:len(g)], z[:len(g)]]) - g).max()
        assert err < DATREF_TOL, (name, err)
    d.s.destroy()


# ------------------------------------------------------------------------------------------------
# 2. edge cases, one step per run, both parameter sets
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("which", ["default", "edge"])
def test_edge_cases_bitwise(sctx, which):
    import jrl_walkgen_b200 as wg
    lists, feet = edge_lists()
    params = wg.zmpdisc_default_params() if which == "default" else edge_params()
    ref = reference_front(sctx, lists, feet, params)
    d = Drive(sctx, lists, feet, params=params, with_preview=False)
    for take in sched_one(lists):
        d.step(take)
    assert_front_equal(d, ref)
    assert d.runs[0][2].sum() == 0
    # the one-step walk was START|FINISH in the first run: lead-in + end phase at once
    so = d.runs[0][0]
    assert so[1] - so[0] == len(ref[0][0])
    d.s.destroy()


# ------------------------------------------------------------------------------------------------
# 3. CoM
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [0, 1, 2])
def test_whole_walks_com_bitwise(sctx, shape):
    lists, feet = batch_lists(40, seed=9)
    sctx.preview_set_cta_shape(shape)
    try:
        ref = reference_com(sctx, lists, feet)
        d = Drive(sctx, lists, feet, ref_offsets=ref["offsets"])
        d.step(sched_whole(lists)[0])
        st, emitted, previewed, _ = d.s.state()
    finally:
        sctx.preview_set_cta_shape(-1)
    assert np.array_equal(d.com, ref["com"]) and np.array_equal(d.zmp, ref["zmp"])
    assert np.array_equal(st, ref["state"])
    assert np.array_equal(d.runs[0][0], ref["offsets"]) and np.array_equal(d.runs[0][1], ref["offsets"])
    assert d.com_count == previewed.sum() == ref["total_steps"]
    d.s.destroy()


def _check_chunked(ref, d):
    st, _, previewed, _ = d.s.state()
    assert d.com_count == previewed.sum() == ref["total_steps"]
    dc = np.abs(d.com - ref["com"])
    assert dc[:, [0, 3]].max() < 1e-11 and dc.max() < 1e-8, dc.max(axis=0)
    assert np.abs(d.zmp - ref["zmp"]).max() < 1e-9
    assert np.abs(st - ref["state"]).max() < 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["direct", "recursive"])
def test_chunked_com_b40_and_oracle(sctx, mode):
    import jrl_walkgen_b200 as wg
    import oracle_lib as ol
    B = 40
    lists, feet = batch_lists(B, seed=9)
    sctx.preview_set_sum_mode(wg.PREVIEW_SUM_DIRECT if mode == "direct" else wg.PREVIEW_SUM_RECURSIVE)
    try:
        ref = reference_com(sctx, lists, feet)
        for sched in (sched_one(lists), sched_ragged(lists, 3)):
            d = Drive(sctx, lists, feet, ref_offsets=ref["offsets"])
            for take in sched:
                d.step(take)
            _check_chunked(ref, d)
            d.s.destroy()
    finally:
        sctx.preview_set_sum_mode(wg.PREVIEW_SUM_AUTO)
    # the oracle chain: zmpdisc_oracle -> OneIterationOfPreview
    po = zo.default_params()
    z_o = np.concatenate([zo.run(po, lists[b], feet[b])["zmp"][:, :2] for b in range(B)])
    og = ol.OracleGains(*GAINS, 1)
    st_o = np.zeros((B, 8))
    com_o, zmp_o, nsteps = ol.oracle_preview_batch(og, ref["offsets"], np.ascontiguousarray(z_o), st_o)
    assert nsteps == ref["total_steps"]
    assert np.abs(d.com - com_o).max() < 1e-9 and np.abs(d.zmp - zmp_o).max() < 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["direct", "recursive"])
def test_chunked_com_b4096(sctx, mode):
    import jrl_walkgen_b200 as wg
    B = 4096
    lists, feet = batch_lists(B, seed=0)
    sctx.preview_set_sum_mode(wg.PREVIEW_SUM_DIRECT if mode == "direct" else wg.PREVIEW_SUM_RECURSIVE)
    try:
        ref = reference_com(sctx, lists, feet)
        d = Drive(sctx, lists, feet, ref_offsets=ref["offsets"])
        for take in sched_ragged(lists, 5):
            d.step(take)
        _check_chunked(ref, d)
        d.s.destroy()
    finally:
        sctx.preview_set_sum_mode(wg.PREVIEW_SUM_AUTO)


# ------------------------------------------------------------------------------------------------
# 4. host and device modes
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_host_and_device_modes_bitwise(sctx):
    import jrl_walkgen_b200 as wg
    lists, feet = batch_lists(40, seed=4)
    sched = sched_ragged(lists, 11)
    dh = Drive(sctx, lists, feet)
    dd = Drive(sctx, lists, feet, mem=wg.WG_MEM_DEVICE)
    for take in sched:
        dh.step(take)
        dd.step(take)
    for (so, co, cnt, oh), (so2, co2, cnt2, od) in zip(dh.runs, dd.runs):
        assert np.array_equal(so, so2) and np.array_equal(co, co2) and np.array_equal(cnt, cnt2)
        for k in oh:
            assert np.array_equal(oh[k], od[k]), k
    sh = dh.s.state()[0]
    d_st = sctx.alloc(len(lists) * 64)
    dd.s.state(d_st, mem=wg.WG_MEM_DEVICE)
    sctx.sync()
    assert np.array_equal(d_st.download(np.float64, (len(lists), 8)), sh)
    d_st.free()
    dh.s.destroy(); dd.s.destroy()


# ------------------------------------------------------------------------------------------------
# 5. restart
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_restart_matches_fresh_stream(sctx):
    """Walks 0..3 restart with START at run 3 while walks 4..7 go on: every run from then on is the run of a stream in
    which walks 0..3 start at run 3."""
    lists, feet = batch_lists(8, seed=21)
    new, feet2 = batch_lists(4, seed=22)
    sctx.preview_set_cta_shape(1)
    try:
        A = Drive(sctx, lists, feet)
        F = Drive(sctx, [l[:0] for l in lists[:4]] + lists[4:], feet)
        for r in range(3):
            A.step(np.ones(8, dtype=int))
            F.step(np.r_[np.zeros(4, dtype=int), np.ones(4, dtype=int)])
        # restart walks 0..3 of A with new lists (their old walks are still open)
        for b in range(4):
            A.lists[b], A.pos[b], A.done[b] = new[b], 0, False
            F.lists[b] = new[b]
        A.feet[:4] = feet2; F.feet[:4] = feet2
        while not (A.done.all() and F.done.all()):
            A.step(np.ones(8, dtype=int))
            F.step(np.ones(8, dtype=int))
        assert len(A.runs) == len(F.runs) < 100
        for r in range(3, len(A.runs)):
            (so, co, cnt, oa), (so2, co2, cnt2, of) = A.runs[r], F.runs[r]
            assert np.array_equal(so, so2) and np.array_equal(co, co2) and np.array_equal(cnt, cnt2), r
            for k in oa:
                assert np.array_equal(oa[k], of[k]), (r, k)
        assert np.array_equal(A.s.state()[0], F.s.state()[0])
    finally:
        sctx.preview_set_cta_shape(-1)
    # the restarted walks' front end is the off-line one on their new lists
    ref = reference_front(sctx, new, feet2)
    for b in range(4):
        got = [np.concatenate([p[i] for p in A.samples[b][3:]]) for i in range(5)]
        for g, w in zip(got, ref[b]):
            assert np.array_equal(g, w), b
    A.s.destroy(); F.s.destroy()


# ------------------------------------------------------------------------------------------------
# 6. refusals
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refused_appends_change_nothing(sctx):
    import jrl_walkgen_b200 as wg
    lists, feet = batch_lists(6, seed=31)
    S = Drive(sctx, lists, feet)
    R = Drive(sctx, lists, feet)
    B = 6

    def refused(off, steps, flags, init_feet=feet, code=-3):
        with pytest.raises(wg.WalkgenError) as ei:
            S.s.append(off, steps, flags, init_feet)
        assert ei.value.code == code

    one = lists[0][:2].copy()
    z = np.zeros(B, dtype=np.int32)
    # before anything: steps for walks that are not open, FINISH on a closed walk, START without steps or feet
    refused(np.r_[0, np.full(B, 2)], one, z)
    refused(np.zeros(B + 1, dtype=np.int64), one[:0], np.r_[wg.STREAM_FINISH, np.zeros(B - 1, dtype=np.int32)])
    refused(np.zeros(B + 1, dtype=np.int64), one[:0], np.r_[wg.STREAM_START, np.zeros(B - 1, dtype=np.int32)])
    refused(np.r_[0, np.full(B, 2)], one, np.r_[wg.STREAM_START, np.zeros(B - 1, dtype=np.int32)], init_feet=None)
    sched = sched_ragged(lists, 2)
    for i, take in enumerate(sched):
        if i == 2:
            bad = lists[1][:3].copy()
            bad["ds_time"][1], bad["ss_time"][1] = 0.001, 0.5        # rounds to zero double-support samples
            refused(np.r_[0, np.full(B, 3)], bad, np.r_[wg.STREAM_START, np.zeros(B - 1, dtype=np.int32)])
            off, steps, flags = S.plan(take)                          # a valid append before an un-run one: refused
            S.s.append(off, steps, flags, feet)
            refused(off, steps, flags)
            S.execute()
            R.step(take)
            continue
        S.step(take)
        R.step(take)
        if i == len(sched) - 1:                                       # every walk closed: FINISH / steps refused
            refused(np.zeros(B + 1, dtype=np.int64), one[:0], np.full(B, wg.STREAM_FINISH, dtype=np.int32))
            refused(np.r_[0, np.full(B, 2)], one, z)
    for (so, co, cnt, os_), (so2, co2, cnt2, or_) in zip(S.runs, R.runs):
        assert np.array_equal(so, so2) and np.array_equal(co, co2) and np.array_equal(cnt, cnt2)
        for k in os_:
            assert np.array_equal(os_[k], or_[k]), k
    assert np.array_equal(S.s.state()[0], R.s.state()[0])
    S.s.destroy(); R.s.destroy()


@pytest.mark.gpu
def test_gains_of_another_nl_are_refused(sctx):
    import jrl_walkgen_b200 as wg
    lists, feet = batch_lists(4, seed=41)
    s = sctx.kajita_stream(4)
    off, steps = _cat([l[:2] for l in lists])
    s.append(off, steps, np.full(4, wg.STREAM_START, dtype=np.int32), feet)
    try:
        sctx.preview_set_gains(wg.preview_gains(0.005, 1.2, 0.8078, wg.MODE_WITHOUT_INITIALPOS))
        with pytest.raises(wg.WalkgenError) as ei:
            s.run(**s.host_outputs())
        assert ei.value.code == -5
    finally:
        sctx.preview_set_gains(wg.preview_gains(*GAINS, wg.MODE_WITHOUT_INITIALPOS))
    s.run(**s.host_outputs())          # the same NL again: the pending run goes through
    assert s.state()[1].sum() == s.sample_offsets[-1]
    s.destroy()
    with pytest.raises(wg.WalkgenError) as ei:    # front end only: no CoM outputs
        f = sctx.kajita_stream(4, with_preview=False)
        try:
            f.append(off, steps, np.full(4, wg.STREAM_START, dtype=np.int32), feet)
            f.run(com_out=np.zeros((10, 6)))
        finally:
            f.destroy()
    assert ei.value.code == -3


# ------------------------------------------------------------------------------------------------
# 7. steady state
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_steady_state_launches(sctx):
    """After warm-up every run of one step per walk is two kernel launches: the front end and the preview."""
    import jrl_walkgen_b200 as wg
    lists, feet = batch_lists(64, seed=51)
    long = [np.concatenate([l[:1]] + [l[1:-1]] * 60 + [l[-1:]]) for l in lists]     # 60+ steps per walk
    s = sctx.kajita_stream(64)
    d_out = {k: sctx.alloc(1 << 22) for k in ("zmpref_xy", "com_out", "zmp_out")}
    one = np.arange(65, dtype=np.int64)
    for r in range(60):
        steps = np.concatenate([l[r:r + 1] for l in long])
        flags = np.full(64, wg.STREAM_START if r == 0 else 0, dtype=np.int32)
        s.append(one, steps, flags, feet)
        before = sctx.launches
        s.run(**d_out, mem=wg.WG_MEM_DEVICE)
        if r >= 10:
            assert sctx.launches - before == 2, (r, sctx.launches - before)
    sctx.sync()
    for b in d_out.values():
        b.free()
    s.destroy()
