"""Two-stage preview control (SURVEY 8a row a4: ZMPPreviewControlWithMultiBodyZMP::FirstStageOfControl /
EvaluateMultiBodyZMP / SecondStageOfControl, src/PreviewControl/ZMPPreviewControlWithMultiBodyZMP.cpp:317-479) pinned to
the reference's OWN object code.

oracle/_ref/libwalkgen_ref.so holds ZMPPreviewControlWithMultiBodyZMP.cpp compiled where it lies; the robot model and the
whole-body realisation it calls are test doubles without a model (oracle/ref_glue_twostage.cc): the multibody ZMP is a
stream the test supplies.  Everything else - FIFOs, both preview stages, the delta ZMP, the NL-delayed sum, the gains
(ComputeOptimalWeights through dgges_ inside Setup) - is the reference's code.
  * CPU: the restatement oracle_two_stage_run against that object: bitwise.
  * GPU: wg_preview_run_batch -> wg_preview_delta_zmp -> wg_preview_stage2_run_batch on the stream the reference's FIFOs
    hold, against the same object at 1e-9 m.  Where oracle/_ref is not built, the GPU tests compare with OracleTwoStage
    instead: the bitwise restatement run on the oracle's Riccati gains, which agree with the reference's dgges_ gains to
    2e-9 relative; the tests of the reference object itself need oracle/_ref.
"""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol
import preview_ref as pr
from test_preview_ref import straight_walking_zmpref, synth_walk

D = ol.D
HAVE_REF = pr.lib() is not None and hasattr(pr.lib(), "ref_twostage_new")
needs_ref = pytest.mark.skipif(not HAVE_REF, reason="oracle/_ref/libwalkgen_ref.so (reference object code) not built")
T, TP, ZC, NL = 0.005, 1.6, 0.807709, 320


class RefTwoStage:
    def __init__(self):
        if not pr.lapack_available():
            pytest.skip("no LAPACK with dgges_ in this image")
        self.r = pr.lib()
        self.r.ref_twostage_new.restype = C.c_void_p
        self.r.ref_twostage_new.argtypes = [C.c_double] * 3
        self.r.ref_twostage_delete.argtypes = [C.c_void_p]
        self.r.ref_twostage_get_gains.restype = C.c_int
        self.r.ref_twostage_get_gains.argtypes = [C.c_void_p, D, D, D, D, D, D, C.c_int]
        self.r.ref_twostage_run.restype = C.c_long
        self.r.ref_twostage_run.argtypes = [C.c_void_p, D, C.c_long, D, C.c_long, D, C.c_int, D, D, D, C.POINTER(C.c_long)]
        self.h = self.r.ref_twostage_new(T, TP, ZC)

    def close(self):
        self.r.ref_twostage_delete(self.h)

    def run(self, zref, zmb, start, strategy=1):
        L = len(zref)
        s1 = np.zeros((L, 6)); dl = np.zeros((L, 2)); fin = np.zeros((L, 6))
        ticks = C.c_long(0)
        zref = np.ascontiguousarray(zref); zmb = np.ascontiguousarray(zmb)
        start = np.ascontiguousarray(start, dtype=np.float64)
        n = self.r.ref_twostage_run(self.h, ol.dptr(zref), L, ol.dptr(zmb), len(zmb), ol.dptr(start), strategy, ol.dptr(s1),
                                    ol.dptr(dl), ol.dptr(fin), C.byref(ticks))
        assert n >= 0
        return s1[:ticks.value], dl[:ticks.value], fin[:n]

    def gains(self):
        """The gains the reference computed for itself inside Setup (only valid after a run)."""
        g = ol.OracleGains.__new__(ol.OracleGains)
        g.A = np.zeros(9); g.B = np.zeros(3); g.C = np.zeros(3); g.Kx = np.zeros(3)
        F = np.zeros(4096); ks = C.c_double()
        g.NL = self.r.ref_twostage_get_gains(self.h, ol.dptr(g.A), ol.dptr(g.B), ol.dptr(g.C), ol.dptr(g.Kx), C.byref(ks),
                                             ol.dptr(F), 4096)
        g.F = F[:g.NL].copy(); g.Ks = ks.value
        return g


def oracle_two_stage(g, zref, zmb, start):
    o = ol.oracle()
    o.oracle_two_stage_run.restype = C.c_long
    o.oracle_two_stage_run.argtypes = [D, D, D, D, C.c_double, D, C.c_int, D, C.c_long, D, C.c_long, D, D, D, D,
                                       C.POINTER(C.c_long)]
    L = len(zref)
    s1 = np.zeros((L, 6)); dl = np.zeros((L, 2)); fin = np.zeros((L, 6))
    ticks = C.c_long(0)
    zref = np.ascontiguousarray(zref); zmb = np.ascontiguousarray(zmb); start = np.ascontiguousarray(start[:2], dtype=np.float64)
    n = o.oracle_two_stage_run(ol.dptr(g.A), ol.dptr(g.B), ol.dptr(g.C), ol.dptr(g.Kx), g.Ks, ol.dptr(g.F), g.NL, ol.dptr(zref),
                               L, ol.dptr(zmb), len(zmb), ol.dptr(start), ol.dptr(s1), ol.dptr(dl), ol.dptr(fin), C.byref(ticks))
    assert n >= 0
    return s1[:ticks.value], dl[:ticks.value], fin[:n]


class OracleTwoStage:
    """Stand-in for RefTwoStage (ZMPCOM_TRAJECTORY_FULL only) where oracle/_ref is not built: oracle_two_stage_run, which
    test_restatement_matches_reference_object holds bitwise equal to the reference object for the same gains, on the
    oracle's own gains (Riccati fixed point) in place of the reference's dgges_ solve."""

    def __init__(self):
        self.g = ol.OracleGains(T, TP, ZC, 1)

    def close(self):
        pass

    def run(self, zref, zmb, start):
        return oracle_two_stage(self.g, zref, zmb, start)

    def gains(self):
        return self.g


def synthetic_multibody_zmp(com1, k0=0):
    """A stand-in for the multibody model: the cart-table ZMP at 0.9 zc plus a slow disturbance, a function of the
    first-stage CoM of the same tick (what the reference evaluates through IK + inverse dynamics)."""
    k = np.arange(k0, k0 + len(com1))
    h = 0.9 * ZC / 9.81
    return np.column_stack([com1[:, 0] - h * com1[:, 2] + 0.003 * np.sin(0.02 * k),
                            com1[:, 3] - h * com1[:, 5] + 0.002 * np.cos(0.015 * k)])


def stage1_only(g, zeff, start):
    st = np.zeros((1, 8)); st[0, 0] = start[0]; st[0, 3] = start[1]
    com, _, steps = ol.oracle_preview_batch(g, np.array([0, len(zeff)], dtype=np.int64), zeff, st)
    return com[:steps]


def effective_stream(zref):
    """What the reference's FIFO holds: Setup pushes ZMPRefPositions[i + 1 + NL] after having loaded [0, NL), so sample NL
    never enters (ZMPPreviewControlWithMultiBodyZMP.cpp:550-557, :660)."""
    return np.ascontiguousarray(np.concatenate([zref[:NL], zref[NL + 1:]]))


@pytest.fixture(scope="module")
def ref_obj():
    r = RefTwoStage() if HAVE_REF else OracleTwoStage()
    z = straight_walking_zmpref()
    r.run(z[:2 * NL + 8], np.zeros((2 * NL + 8, 2)), (0.0, 0.0, ZC))   # makes the object compute its gains
    yield r
    r.close()


@needs_ref
def test_restatement_matches_reference_object(ref_obj):
    """oracle_two_stage_run == the reference object: first-stage CoM, delta ZMP stream and final CoM, bitwise, on the
    StraightWalking reference and on random walks; and the count of ticks / global steps."""
    g = ref_obj.gains()
    assert g.NL == NL
    rng = np.random.default_rng(5)
    walks = [straight_walking_zmpref()] + [synth_walk(rng, int(L)) for L in (700, 1500, 2 * NL + 1, 2 * NL + 2)]
    for w in walks:
        start = (w[0, 0] + 0.001, w[0, 1] - 0.002, ZC)
        com1 = stage1_only(g, effective_stream(w), start)
        zmb = synthetic_multibody_zmp(com1)
        s1r, dlr, finr = ref_obj.run(w, zmb, start)
        s1o, dlo, fino = oracle_two_stage(g, w, zmb, start)
        assert len(finr) == len(fino) == len(w) - 2 * NL and len(s1r) == len(s1o) == len(w) - NL
        assert np.array_equal(s1r, s1o)
        assert np.array_equal(dlr, dlo)
        assert np.array_equal(finr, fino)
        assert np.array_equal(s1o, com1[:len(s1o)])                # the first stage is the plain preview loop on the FIFO's stream
        # the second stage really moves the CoM (millimetres), i.e. the test would see a wrong delay or sign
        if len(finr) > 200:
            assert np.abs(finr[:, 0] - s1r[:len(finr), 0]).max() > 1e-4


@needs_ref
def test_first_stage_only_strategy(ref_obj):
    """ZMPCOM_TRAJECTORY_FIRST_STAGE_ONLY: the final CoM is the first stage's, delayed by NL ticks."""
    g = ref_obj.gains()
    w = straight_walking_zmpref()[:1500]
    start = (0.0, 0.0, ZC)
    s1, _, fin = ref_obj.run(w, np.zeros((len(w), 2)), start, strategy=3)
    assert len(fin) > 0 and np.array_equal(fin, s1[:len(fin)])
    assert np.array_equal(s1, stage1_only(g, effective_stream(w), start)[:len(s1)])


@pytest.mark.gpu
def test_gpu_two_stage_vs_reference_object(ctx, ref_obj):
    """The batched product path (first stage, delta ZMP, second stage with the NL-delayed sum fused into the store) on a ragged
    batch, host and device memory, against the reference object walk by walk."""
    import jrl_walkgen_b200 as wg
    g = ref_obj.gains()
    gains = wg.preview_gains(T, TP, ZC, 1)
    assert gains.NL == NL
    # the product's own gains (structure-preserving doubling) agree with the reference's (dgges_) to 2e-9 relative; use the
    # reference's here so that the comparison is on the recursion alone
    gains.Ks = g.Ks
    for i in range(3):
        gains.Kx[i] = g.Kx[i]
    for i in range(NL):
        gains.F[i] = g.F[i]
    ctx.preview_set_gains(gains)
    rng = np.random.default_rng(9)
    walks = [straight_walking_zmpref()] + [synth_walk(rng, int(L)) for L in rng.integers(2 * NL + 40, 3000, size=6)]
    effs = [effective_stream(w) for w in walks]
    offsets = np.concatenate([[0], np.cumsum([len(e) for e in effs])]).astype(np.int64)
    zeff = np.concatenate(effs)
    n = len(zeff)
    starts = [(w[0, 0] + 0.001, w[0, 1] - 0.002, ZC) for w in walks]
    plan = ctx.preview_plan(offsets)
    st1 = np.zeros((len(walks), 8))
    for b, s in enumerate(starts):
        st1[b, 0] = s[0]; st1[b, 3] = s[1]
    com1 = np.zeros((n, 6))
    plan.run(zeff, st1, com1, None, True)
    zmb = np.zeros((n, 2))
    for b in range(len(walks)):
        o, e = int(offsets[b]), int(offsets[b + 1])
        zmb[o:e] = synthetic_multibody_zmp(com1[o:e])
    delta = np.zeros((n, 2))
    plan.delta_zmp(zeff, zmb, delta)
    st2 = np.zeros((len(walks), 8))
    fin = np.zeros((n, 6)); dz = np.zeros((n, 2))
    plan.run_stage2(delta, com1, st2, fin, dz)
    worst = 0.0
    for b, w in enumerate(walks):
        o = int(offsets[b])
        ticks = len(effs[b]) - NL + 1
        s1r, dlr, finr = ref_obj.run(w, zmb[o:o + ticks], starts[b])
        assert len(finr) == len(effs[b]) - 2 * NL + 1
        assert np.abs(com1[o:o + len(s1r)] - s1r).max() < 1e-9
        assert np.abs(delta[o:o + len(dlr)] - dlr).max() < 1e-9
        e = np.abs(fin[o:o + len(finr)] - finr).max()
        worst = max(worst, e)
        assert e < 1e-9, (b, e)
    # device-resident: same bits as the host path
    d = {k: ctx.to_device(v) for k, v in dict(z=zeff, mb=zmb, com1=com1).items()}
    d_delta = ctx.alloc(delta.nbytes); d_fin = ctx.alloc(fin.nbytes); d_st = ctx.to_device(np.zeros((len(walks), 8)))
    plan.delta_zmp(d["z"], d["mb"], d_delta, mem=wg.WG_MEM_DEVICE)
    plan.run_stage2(d_delta, d["com1"], d_st, d_fin, None, mem=wg.WG_MEM_DEVICE)
    ctx.sync()
    fin_d = d_fin.download(np.float64, (n, 6))
    assert np.array_equal(d_delta.download(np.float64, (n, 2)), delta)
    for b in range(len(walks)):
        o = int(offsets[b]); steps = len(effs[b]) - NL + 1
        assert np.array_equal(fin_d[o:o + steps], fin[o:o + steps])
    for v in list(d.values()) + [d_delta, d_fin, d_st]:
        v.free()
    plan.destroy()
    print(f"two-stage: max |final CoM - reference object| = {worst:.2e} over {len(walks)} walks")


@pytest.mark.gpu
def test_cpp_class_mirror_two_stage_vs_reference_object(ref_obj, tmp_path):
    """The ZMPPreviewControlWithMultiBodyZMP class mirror (jrl_walkgen_b200/host) driven tick by tick - EvaluateStartingCoM,
    Setup, then OneGlobalStepOfControl + UpdateTheZMPRefQueue - with a model robot whose zeroMomentumPoint() is a function
    of the CoM the realisation was handed, and its batched RunWholeTrajectory, against the reference object fed the same
    multibody ZMP stream: every final CoM within 1e-9 (the product's gains agree with the reference's dgges_ gains to 2e-9
    relative; both sides use their own here)."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run(["make", "-s", "-C", os.path.join(root, "tests", "cpp")], check=True)
    w = straight_walking_zmpref()[:2200]
    fin_path, out_path = tmp_path / "zref.bin", tmp_path / "twostage.bin"
    np.ascontiguousarray(w).tofile(fin_path)
    r = subprocess.run([os.path.join(root, "tests", "cpp", "host_api_test"), "twostage", str(fin_path), str(out_path), "100000"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = np.fromfile(out_path)
    steps, nb = int(raw[0]), int(raw[1])
    serial = raw[2:2 + 6 * steps].reshape(steps, 6)
    batched = raw[2 + 6 * steps:].reshape(nb, 6)
    assert steps == nb == len(w) - 2 * NL
    g = ref_obj.gains()
    start = (w[0, 0] + 0.001, w[0, 1] - 0.002, ZC)
    com1 = stage1_only(g, effective_stream(w), start)
    zmb = synthetic_multibody_zmp(com1)
    s1r, dlr, finr = ref_obj.run(w, zmb, start)
    assert len(finr) == steps
    e1, e2 = np.abs(serial - finr).max(), np.abs(batched - finr).max()
    print(r.stdout.strip(), f"; vs reference object: tick by tick {e1:.2e}, batched {e2:.2e}")
    assert e1 < 1e-8 and e2 < 1e-8
