"""Kajita2003 preview control pinned to the reference's OWN object code.

oracle/_ref/libwalkgen_ref.so holds /root/reference/src/PreviewControl/PreviewControl.cpp and
OptimalControllerSolver.cpp compiled where they lie (oracle/Makefile, over the stand-in MAL header of
oracle/ref_shim; LAPACK dgges_/dgetrf_/dgetri_ resolved from the OpenBLAS inside the image's SciPy wheel).
  * CPU (-m "not gpu"): the restatement oracle/oracle_preview.cpp against that object code - BITWISE for the recursion
    (PreviewControl.cpp:324-484, all three entry points), 2e-9 relative for the gains (ComputeOptimalWeights through
    dgges_, :198-322, against the oracle's Riccati fixed point and the product's host SDA solve).
  * GPU: preview_fused_kernel, wg_preview_one_iteration and the host class mirror's 1-D variants against the same
    object code, on the ZMP reference of TestKajita2003's StraightWalking profile and on random walks, at 1e-9 m.
"""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as ol
import preview_ref as pr
import zmpdisc_oracle as zo

needs_ref = pytest.mark.skipif(pr.lib() is None, reason="oracle/_ref/libwalkgen_ref.so (reference object code) not built")
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "preview_ref.npz")

TOL_COM = 1e-9     # m; north_star asks 1e-6 m for CoM/ZMP trajectories
CONFIGS = [(0.005, 1.6, 0.814, 1), (0.005, 1.6, 0.807709, 1), (0.01, 1.6, 0.814, 0), (0.005, 0.8, 0.75, 1)]


def synth_walk(rng, L):
    z = np.zeros((L, 2))
    k = 0; x = 0.0; side = 1.0
    while k < L:
        n = int(rng.integers(120, 200))
        z[k:k + n, 0] = x; z[k:k + n, 1] = side * 0.095
        x += rng.uniform(0.05, 0.25); side = -side; k += n
    return z


def straight_walking_zmpref():
    """ZMP reference of TestKajita2003 StraightWalking (4002 samples; its first 3362 rows are datref columns 35-36,
    asserted here at the datref's 1e-7 truncation)."""
    o = zo.run(zo.default_params(), zo.profile_steps("StraightWalking"))
    z = np.ascontiguousarray(o["zmp"][:, :2])
    g = zo.golden("StraightWalking")
    assert np.abs(z[:len(g)] - g[:, -2:]).max() < 1.2e-7
    return z


def gpu_preview_inputs():
    """The StraightWalking ZMP reference and 64 seeded random walks, with their seeded initial states."""
    rng = np.random.default_rng(21)
    walks = [straight_walking_zmpref()] + [synth_walk(rng, int(L)) for L in rng.integers(900, 5200, size=64)]
    st0 = rng.normal(scale=0.01, size=(len(walks), 8)); st0[0] = 0.0
    return walks, st0


def sample_rows(steps, b, count):
    """Fixed, seeded sample of `count` preview steps of walk b (its first and last step included), sorted."""
    r = 1 + np.random.default_rng([21, b]).choice(steps - 2, size=count - 2, replace=False)
    return np.sort(np.concatenate([[0, steps - 1], r]).astype(np.int64))


def ref_with_gains(g, T, Tp, zc):
    rp = pr.RefPreview(1, False)
    rp.set_gains(T, Tp, zc, g.Kx, g.Ks, g.F)
    return rp


# ------------------------------------------------------------------------------------------------
# CPU: restatement vs reference object code
# ------------------------------------------------------------------------------------------------
@needs_ref
@pytest.mark.parametrize("T,Tp,zc,mode", CONFIGS)
def test_reference_gains_vs_oracle_and_product(T, Tp, zc, mode):
    """ComputeOptimalWeights of the reference (generalized Schur form through dgges_) against the oracle's Riccati
    fixed point and the product's structure-preserving doubling: three different algorithms for the same
    stabilising solution.  Measured agreement 9e-10 relative for R = 1e-6 (mode 1), 1e-14 for mode 0."""
    if not pr.lapack_available():
        pytest.skip("no LAPACK with dgges_ in this image")
    import jrl_walkgen_b200 as wg
    rp = pr.RefPreview(mode, False)
    rp.compute_weights(T, Tp, zc, mode)
    g = rp.gains(); rp.close()
    o = ol.OracleGains(T, Tp, zc, mode)
    p = wg.preview_gains(T, Tp, zc, mode)
    assert g["NL"] == o.NL == p.NL
    for cand_F, cand_Ks, cand_Kx in ((o.F, o.Ks, o.Kx), (np.array(p.F[:p.NL]), p.Ks, np.array(p.Kx[:]))):
        assert np.abs(g["F"] - cand_F).max() <= 2e-9 * np.abs(g["F"]).max()
        assert abs(g["Ks"] - cand_Ks) <= 2e-9 * abs(g["Ks"])
        assert np.allclose(g["Kx"], cand_Kx, rtol=2e-9)
    assert np.array_equal(g["A"], o.A) and np.array_equal(g["B"], o.B) and np.array_equal(g["C"], o.C)
    assert np.array_equal(g["A"], np.array(p.A[:])) and np.array_equal(g["B"], np.array(p.B[:]))


@needs_ref
def test_reference_gains_through_plugin_commands():
    """:samplingperiod / :previewcontroltime / :comheight with automatic weights (PreviewControl.cpp:512-548)."""
    if not pr.lapack_available():
        pytest.skip("no LAPACK with dgges_ in this image")
    rp = pr.RefPreview(1, True)
    rp.call_method(":samplingperiod", "0.005")
    rp.call_method(":previewcontroltime", "1.6")
    rp.call_method(":comheight", "0.814")
    g = rp.gains(); rp.close()
    o = ol.OracleGains(0.005, 1.6, 0.814, 1)
    assert g["NL"] == 320 and abs(g["Ks"] - o.Ks) <= 2e-9 * o.Ks


@needs_ref
@pytest.mark.parametrize("simulation", [True, False])
@pytest.mark.parametrize("use_lindex", [False, True])
def test_oracle_recursion_is_bitwise_the_reference(simulation, use_lindex):
    """OneIterationOfPreview (:324-374) of the reference object over whole trajectories (FIFO popped per tick as
    ZMPPreviewControlWithMultiBodyZMP.cpp:393-438 does, or lindex = k) == oracle_preview_run, bit for bit."""
    o = ol.OracleGains(0.005, 1.6, 0.807709, 1)
    rp = ref_with_gains(o, 0.005, 1.6, 0.807709)
    rng = np.random.default_rng(11)
    walks = [straight_walking_zmpref()] + [synth_walk(rng, int(L)) for L in (320, 321, 2000, 4500)]
    for z in walks:
        st = rng.normal(scale=0.01, size=8); st_o = st.copy()
        com, zmp, steps = rp.run(z, st, simulation, use_lindex)
        com_o, zmp_o, steps_o = ol.oracle_preview_batch(o, [0, len(z)], z, st_o, simulation)
        assert steps == steps_o == len(z) - 320 + 1
        assert np.array_equal(com[:steps], com_o[:steps]) and np.array_equal(zmp[:steps], zmp_o[:steps])
        assert np.array_equal(st, st_o)
    # window longer than the FIFO: the reference LTHROWs (:341-344), the oracle returns an error
    st = np.zeros(8)
    assert rp.run(walks[1][:319], st)[2] == -1
    rp.close()


@needs_ref
def test_oracle_1d_variants_are_bitwise_the_reference():
    """OneIterationOfPreview1D: deque overload (:376-421) and vector overload with its wrap-around branch (:423-484)."""
    o = ol.OracleGains(0.005, 1.6, 0.814, 1)
    rp = ref_with_gains(o, 0.005, 1.6, 0.814)
    rng = np.random.default_rng(12)
    z = synth_walk(rng, 1500)
    # deque overload over a trajectory == the x axis of the 2-D recursion
    st4 = rng.normal(scale=0.01, size=4)
    st8 = np.array([st4[0], st4[1], st4[2], 0, 0, 0, st4[3], 0.0])
    com1, zmp1, steps = rp.run_1d_deque(z[:, 0], st4)
    zz = z.copy(); zz[:, 1] = 0
    com_o, zmp_o, steps_o = ol.oracle_preview_batch(o, [0, 1500], zz, st8)
    assert steps == steps_o
    assert np.array_equal(com1[:steps], com_o[:steps, :3]) and np.array_equal(zmp1[:steps], zmp_o[:steps, 0])
    # vector overload: plain branch (TestSize >= 0) and wrap-around branch.  The wrap-around loop indexes F with the
    # absolute buffer index (:459), so it is only memory-safe for a circular buffer of exactly NL samples.
    D = ol.D
    for (L, lindex) in ((1500, 0), (1500, 700), (1500, 1180), (320, 0), (320, 1), (320, 137), (320, 319)):
        buf = z[:L, 1].copy()
        x0 = rng.normal(scale=0.01, size=3); s0 = float(rng.normal(scale=0.01))
        for sim in (True, False):
            rc, x, s, zo_ = rp.step_1d_vector(buf, lindex, x0, s0, sim)
            xo = x0.copy(); so = C.c_double(s0); zout = C.c_double()
            rc_o = ol.oracle().oracle_preview_step_1d_wrap(ol.dptr(o.A), ol.dptr(o.B), ol.dptr(o.C), ol.dptr(o.Kx), o.Ks,
                                                           ol.dptr(o.F), o.NL, ol.dptr(xo), C.byref(so), ol.dptr(buf), L,
                                                           lindex, C.byref(zout), int(sim))
            assert rc == rc_o == 0
            assert np.array_equal(x, xo) and s == so.value and zo_ == zout.value
    rp.close()


@needs_ref
def test_read_precomputed_file_goes_through_float(tmp_path):
    """ReadPrecomputedFile parses every gain into a `float` (PreviewControl.cpp:157-176): a 17-digit file comes back
    rounded to single precision.  The product's PreviewControl::ReadPrecomputedFile mirror does the same
    (tests/cpp/host_api_test.cpp)."""
    o = ol.OracleGains(0.005, 1.6, 0.814, 1)
    path = os.path.join(tmp_path, "gains.ini")
    pr.write_precomputed_file(path, 0.814, 0.005, 1.6, o.Kx, o.Ks, o.F)
    rp = pr.RefPreview(1, False)
    rp.read_file(path)
    g = rp.gains(); rp.close()
    assert g["NL"] == 320 and g["T"] == 0.005 and g["zc"] == 0.814
    assert np.array_equal(g["F"], o.F.astype(np.float32).astype(np.float64))
    assert np.array_equal(g["Kx"], o.Kx.astype(np.float32).astype(np.float64))
    assert g["Ks"] == float(np.float32(o.Ks))
    assert np.array_equal(g["A"], o.A) and np.array_equal(g["C"], o.C)


# ------------------------------------------------------------------------------------------------
# GPU: the CUDA path against the reference object code
# ------------------------------------------------------------------------------------------------
def _gpu_run(ctx, gains, offsets, z, st0, simulation=True):
    ctx.preview_set_gains(gains)
    plan = ctx.preview_plan(offsets)
    n = int(offsets[-1])
    st = st0.copy()
    com = np.zeros((n, 6)); zmp = np.zeros((n, 2))
    plan.run(z, st, com, zmp, simulation)
    plan.destroy()
    return com, zmp, st


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [-1, 0, 2, 3])
@pytest.mark.parametrize("own_gains", [False, True])
def test_gpu_preview_vs_reference_object(ctx, own_gains, shape):
    """The batch preview kernels (shape -1: the default choice for this batch size; 0: preview_rec_kernel at 64 x 8; 2:
    preview_rec_warp_kernel, the one a batch of thousands of walks runs through; 3: 256 x 2, small batches) against PreviewControl::OneIterationOfPreview of the reference object on the StraightWalking
    ZMP reference and 64 random walks.  own_gains=False: both sides use the product's gains (pins the recursion; the
    reference's output is stored, at 96 seeded steps of every walk, in tests/golden/preview_ref.npz); own_gains=True: the
    reference object computes its own gains through dgges_ (pins gains + recursion end to end); where oracle/_ref is not
    built, the oracle's recursion on the oracle's own gains (Riccati fixed point, independent of the product's doubling solve,
    2e-9 relative from dgges_) stands in for it."""
    import jrl_walkgen_b200 as wg
    T, Tp, zc = 0.005, 1.6, 0.807709
    gains = wg.preview_gains(T, Tp, zc, 1)
    rp = og = None
    if own_gains and pr.lib() is not None:
        if not pr.lapack_available():
            pytest.skip("no LAPACK with dgges_ in this image")
        rp = pr.RefPreview(1, False)
        rp.compute_weights(T, Tp, zc, 1)
    elif own_gains:
        og = ol.OracleGains(T, Tp, zc, 1)
    else:
        gold = np.load(GOLDEN)
    walks, st0 = gpu_preview_inputs()
    offsets = np.concatenate([[0], np.cumsum([len(w) for w in walks])]).astype(np.int64)
    z = np.concatenate(walks)
    ctx.preview_set_cta_shape(shape)
    for simulation in (True, False):
        try:
            com, zmp, st = _gpu_run(ctx, gains, offsets, z, st0, simulation)
        except Exception:
            ctx.preview_set_cta_shape(-1)
            raise
        worst = 0.0
        tag = "sim" if simulation else "nosim"
        for b, w in enumerate(walks):
            steps = len(w) - 320 + 1
            o = int(offsets[b])
            if rp is not None or og is not None:
                sr = st0[b].copy()
                com_r, zmp_r, steps_r = rp.run(w, sr, simulation) if rp is not None else \
                    ol.oracle_preview_batch(og, [0, len(w)], w, sr, simulation)
                assert steps_r == steps
                rows = np.arange(steps)
                com_r, zmp_r = com_r[:steps, [0, 3]], zmp_r[:steps]
            else:
                rows = sample_rows(steps, b, 96)
                assert np.array_equal(rows, gold[tag + "_rows"][b])
                com_r, zmp_r, sr = gold[tag + "_com_x_y"][b], gold[tag + "_zmp"][b], gold[tag + "_state"][b]
            e = max(np.abs(com[o + rows][:, [0, 3]] - com_r).max(), np.abs(zmp[o + rows] - zmp_r).max())
            worst = max(worst, e)
            assert np.allclose(st[b, :6], sr[:6], atol=1e-8, rtol=0)
        assert worst < (TOL_COM if simulation else 1e-7), worst
    ctx.preview_set_cta_shape(-1)
    if rp is not None:
        rp.close()


@pytest.mark.gpu
def test_gpu_one_iteration_vs_reference_object(ctx):
    """wg_preview_one_iteration (the per-tick call of the class mirror) over 200 consecutive ticks of the
    StraightWalking reference == the reference object (its output stored in tests/golden/preview_ref.npz), tick by tick."""
    import jrl_walkgen_b200 as wg
    gains = wg.preview_gains(0.005, 1.6, 0.807709, 1)
    ctx.preview_set_gains(gains)
    z = straight_walking_zmpref()[600:600 + 320 + 200]
    gold = np.load(GOLDEN)
    com_r, zmp_r = gold["one_iteration_com"], gold["one_iteration_zmp"]
    x = np.zeros(3); y = np.zeros(3); sx = sy = 0.0
    for k in range(200):
        x, y, sx, sy, zx, zy = ctx.preview_one_iteration(x, y, sx, sy, z[k:k + 320])
        assert np.abs(x - com_r[k, :3]).max() < 1e-9 and np.abs(y - com_r[k, 3:]).max() < 1e-9
        assert abs(zx - zmp_r[k, 0]) < 1e-9 and abs(zy - zmp_r[k, 1]) < 1e-9


@needs_ref
@pytest.mark.gpu
def test_cpp_mirror_1d_variants_and_precomputed_file_vs_reference_object(tmp_path):
    """The host class mirror (PreviewControl::ReadPrecomputedFile, OneIterationOfPreview1D deque and vector overloads
    including the wrap-around branch of PreviewControl.cpp:448-466) driven by tests/cpp/host_api_test.cpp, against the
    reference object that read the SAME gains file (both parse the gains through `float`)."""
    import struct
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run(["make", "-s", "-C", os.path.join(root, "tests", "cpp")], check=True)
    exe = os.path.join(root, "tests", "cpp", "host_api_test")
    o = ol.OracleGains(0.005, 1.6, 0.814, 1)
    ini = os.path.join(tmp_path, "gains.ini")
    pr.write_precomputed_file(ini, 0.814, 0.005, 1.6, o.Kx, o.Ks, o.F)
    rp = pr.RefPreview(1, False)
    rp.read_file(ini)
    rng = np.random.default_rng(31)
    z = synth_walk(rng, 1200)[:, 0].copy()
    cases = []
    for (L, lindex) in ((1500, 0), (1500, 700), (1500, 1180), (320, 0), (320, 1), (320, 137), (320, 319)):
        for sim in (1, 0):
            cases.append((L, lindex, sim, rng.normal(scale=0.01, size=3), float(rng.normal(scale=0.01)),
                          synth_walk(rng, L)[:, 1].copy()))
    fin = os.path.join(tmp_path, "in.bin"); fout = os.path.join(tmp_path, "out.bin")
    with open(fin, "wb") as f:
        f.write(struct.pack("2i", len(z), len(cases)) + z.tobytes())
        for (L, lindex, sim, x0, s0, buf) in cases:
            f.write(struct.pack("4i", L, lindex, sim, 0) + x0.tobytes() + struct.pack("d", s0) + buf.tobytes())
    r = subprocess.run([exe, "preview1d", ini, fin, fout], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    got = np.fromfile(fout)
    steps = len(z) - 320 + 1
    traj = got[:4 * steps].reshape(steps, 4)
    st4 = np.zeros(4)
    com_r, zmp_r, steps_r = rp.run_1d_deque(z, st4)
    assert steps_r == steps
    assert np.abs(traj[:, :3] - com_r[:steps]).max() < 1e-9 and np.abs(traj[:, 3] - zmp_r[:steps]).max() < 1e-9
    rows = got[4 * steps:4 * steps + 5 * len(cases)].reshape(len(cases), 5)
    for row, (L, lindex, sim, x0, s0, buf) in zip(rows, cases):
        rc, x, s, zz = rp.step_1d_vector(buf, lindex, x0, s0, bool(sim))
        assert rc == 0
        assert np.abs(row[:3] - x).max() < 1e-9 and abs(row[3] - s) < 1e-9 and abs(row[4] - zz) < 1e-9, (L, lindex, sim)
    rp.close()
    print("class-mirror OneIterationOfPreview latency per tick: %.1f us" % got[-1])
