"""Wieber2006 generator (SURVEY 8f rank 3: ZMPQPWithConstraint, n = 150 jerks, m <= 600 CoP rows, QLD) pinned to the
reference's OWN object code: src/ZMPRefTrajectoryGeneration/ZMPQPWithConstraint.cpp compiled where it lies into oracle/_ref
(its ZMPDiscretization member, which only produces the input buffers, replaced by a do-nothing class; ql0001_ is the
reference's).  The reference holds no golden data for this generator.
  * CPU: the restatement oracle/oracle_wieber.cpp (with the reference's ql0001_) against that object: polygons and the
    whole CoM / ZMP output, bitwise.
  * GPU: wg_wieber_run_batch against the same object at north_star's tolerance (1e-6 m on CoM / ZMP).  Where oracle/_ref is
    not built, the GPU tests compare with wieber_oracle.OracleWieber instead, which reproduces that object's trajectory to
    1e-7 m; the tests of the reference object itself need oracle/_ref.
"""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol
import dimitrov_oracle as do
import wieber_oracle as wo
import zmpdisc_oracle as zo

HAVE_REF = ol.ref() is not None and hasattr(ol.ref(), "ref_wieber_new")
needs_ref = pytest.mark.skipif(not HAVE_REF, reason="oracle/_ref/libwalkgen_ref.so (reference object code) not built")


def short_walk(nsteps=4, sx=0.2):
    seq = "0.0 -0.095 0.0 " + " ".join(f"{sx} {0.19 if k % 2 == 0 else -0.19} 0.0" for k in range(nsteps)) + \
        f" 0.0 {0.19 if nsteps % 2 == 0 else -0.19} 0.0"
    return zo.run(zo.default_params(), zo.steps_from_seq(seq))


@pytest.fixture(scope="module")
def ref_gen():
    r = wo.RefWieber() if HAVE_REF else wo.OracleWieber()
    yield r
    r.close()


@needs_ref
def test_polygons_are_those_of_the_reference_generator(ref_gen):
    """BuildLinearConstraintInequalities of ZMPQPWithConstraint == oracle_fcals_build (rows A, B and the time windows), bitwise,
    on the four TestKajita2003 profiles."""
    for name in ("StraightWalking", "Circle", "PbFlorentSeq1", "PbFlorentSeq2"):
        w = zo.run(zo.default_params(), zo.profile_steps(name))
        rows, times, nr = ref_gen.polygons(w)
        lci = do.fcals(w["left"], w["right"], w["types"][:, 1])
        assert len(lci) == len(rows) and np.array_equal(lci["rows"], nr), name
        for p in range(len(lci)):
            k = int(nr[p])
            assert np.array_equal(lci["A"][p, :k], rows[p, :k, :2]) and np.array_equal(lci["B"][p, :k], rows[p, :k, 2]), (name, p)
        assert np.array_equal(lci["t_start"], times[:, 0]) and np.array_equal(lci["t_end"], times[:, 1]), name


@needs_ref
def test_restatement_matches_reference_object_bitwise(ref_gen):
    """BuildZMPTrajectoryFromFootTrajectory on a four-step walk: every CoM / ZMP sample the loop writes."""
    w = short_walk(4)
    rc, com_r, zmp_r = ref_gen.run(w)
    k, com_o, zmp_o, info = wo.run(w)
    assert rc == 0 and k > 100, (rc, k)
    assert np.array_equal(com_r, com_o)
    assert np.array_equal(zmp_r, zmp_o)
    assert (info[:, 1] == 0).all() and info[:, 2].max() > 0            # constraints do become active
    n_rows = k * 4
    assert np.abs(com_o[:n_rows, 0]).max() > 0.1                       # the CoM really moved forward
    print(f"wieber: {k} QP periods, m in [{info[:, 0].min()}, {info[:, 0].max()}], active rows up to {info[:, 2].max()}")


def walk_steps(nsteps=4, sx=0.2):
    seq = "0.0 -0.095 0.0 " + " ".join(f"{sx} {0.19 if k % 2 == 0 else -0.19} 0.0" for k in range(nsteps)) + \
        f" 0.0 {0.19 if nsteps % 2 == 0 else -0.19} 0.0"
    return zo.steps_from_seq(seq)


@pytest.mark.gpu
@pytest.mark.parametrize("materialize_pu", [0, 1])
def test_gpu_wieber_generator_matches_reference_object(ctx, ref_gen, materialize_pu):
    """wg_wieber_run_batch (ZMPDiscretization -> polygons -> 150-variable QP per 20 ms -> LIPM, all on the device) on a ragged
    batch of walks against the reference's ZMPQPWithConstraint object code fed the feet / ZMP buffers of the restated
    ZMPDiscretization: every CoM / ZMP sample the loop writes within 1e-6 m (north_star), the same number of periods."""
    import jrl_walkgen_b200 as wg
    walks = [walk_steps(4, 0.2), walk_steps(3, 0.1), walk_steps(6, 0.25), zo.profile_steps("StraightWalking")]
    feet = np.array([zo.INIT_FEET] * len(walks), dtype=np.float64).reshape(len(walks), -1)
    from jrl_walkgen_b200 import _capi
    par = _capi.WieberParams()
    ctx.lib.wg_wieber_default_params(C.byref(par))
    par.materialize_pu = materialize_pu        # 0: rank-structured rows (default); 1: the dense Pu of the reference
    ctx.wieber_set_params(par)
    out = ctx.wieber_run(walks, feet)
    assert (out["status"] == 0).all(), out["status"]
    so = out["sample_offsets"]
    worst = 0.0
    for b, steps in enumerate(walks):
        w = zo.run(zo.default_params(), steps)
        rc, com_r, zmp_r = ref_gen.run(w)
        assert rc == 0
        o, e = int(so[b]), int(so[b + 1])
        assert e - o == len(com_r)
        k = int(out["periods_done"][b])
        assert k == int(out["period_counts"][b])
        rows = 4 * k
        ec = np.abs(out["com"][o:o + rows] - com_r[:rows, :6]).max()
        ez = np.abs(out["zmp"][o:e] - zmp_r[:, :2]).max()
        worst = max(worst, ec, ez)
        assert ec < 1e-6 and ez < 1e-6, (b, ec, ez)
        assert (com_r[rows:, :6] == 0).all() and (out["com"][o + rows:e] == 0).all()
    print(f"wieber GPU ({'dense Pu' if materialize_pu else 'ranked rows'}) vs reference object: max |CoM, ZMP| deviation {worst:.2e} m; periods {out['periods_done']}, "
          f"active-set changes per QP {out['qp_iterations'].sum() / out['periods_done'].sum():.1f}")


@needs_ref
def test_reference_qld_regularises_the_hessian_and_the_rule_is_restated():
    """Finding of this pin: the Wieber2006 Hessian (beta PPu'PPu + alpha VPu'VPu, 75 samples of 20 ms) has eigenvalues down to
    3e-10 (cond 5e11).  ql0001_ does not factorise it as given: ql0002_ adds a multiple of I until every Cholesky pivot exceeds
    vsmall = eps = 1e-8 (qld.cpp:809-918).  wg_qld_diagonal_boost restates that rule (host arithmetic): with the diag it returns
    (1.9e-8) the reference's closed-loop trajectory is reproduced by an independent extended-precision solver to 1e-9 m, while
    the exact minimiser of the QP as stated lies 5.7e-2 m (ZMP) away from what the reference outputs."""
    import ctypes as C
    from jrl_walkgen_b200 import _capi
    lib = _capi.load()
    Cm, _, _ = wo.constants()
    ev = np.linalg.eigvalsh(Cm)
    assert ev.min() < 1e-8 and ev.max() / ev.min() > 1e11
    Cf = np.asfortranarray(Cm)
    boost = lib.wg_qld_diagonal_boost(150, 150, Cf.ctypes.data, 1e-8)
    assert 1e-8 < boost < 1e-7
    assert lib.wg_qld_diagonal_boost(150, 150, Cf.ctypes.data, 0.0) == 0.0
    well = np.asfortranarray(np.eye(5) * 3.0 + 0.1)
    assert lib.wg_qld_diagonal_boost(5, 5, well.ctypes.data, 1e-8) == 0.0          # well conditioned: QLD adds nothing
    w = short_walk(4)
    o = wo._ora()
    o.oracle_wieber_set_boost.argtypes = [C.c_double]
    try:
        o.oracle_wieber_set_solver(0)
        k0, com_q, zmp_q, _ = wo.run(w)
        o.oracle_wieber_set_solver(2); o.oracle_wieber_set_boost(boost)
        k1, com_b, zmp_b, _ = wo.run(w)
        o.oracle_wieber_set_boost(0.0)
        k2, com_e, zmp_e, _ = wo.run(w)
    finally:
        o.oracle_wieber_set_solver(0); o.oracle_wieber_set_boost(0.0)
    assert k0 == k1 == k2 > 0
    n = 4 * k0
    assert np.abs(com_q[:n, :6] - com_b[:n, :6]).max() < 1e-7 and np.abs(zmp_q[:n, :2] - zmp_b[:n, :2]).max() < 1e-8
    gap = np.abs(zmp_q[:n, :2] - zmp_e[:n, :2]).max()
    assert gap > 1e-3
    print(f"QLD adds {boost:.3e} I; reference vs exact solve of the regularised QP: ZMP {np.abs(zmp_q[:n, :2] - zmp_b[:n, :2]).max():.1e} m; "
          f"vs the QP as stated: {gap:.1e} m")


@pytest.mark.gpu
def test_cpp_class_mirror_zmpqpwithconstraint_and_ql0001(ref_gen, tmp_path):
    """ZMPQPWithConstraint::GetZMPDiscretization (":setpbwconstraint", the ZMPRefTrajectoryGeneration commands) and ql0001_ with
    the reference's signature, through the C++ class mirror (tests/cpp/host_api_test.cpp): CoM / ZMP of the whole walk against
    the reference object within 1e-6 m."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run(["make", "-s", "-C", os.path.join(root, "tests", "cpp")], check=True)
    out = tmp_path / "wieber.bin"
    r = subprocess.run([os.path.join(root, "tests", "cpp", "host_api_test"), "wieber", str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = np.fromfile(out)
    n, k = int(raw[0]), int(raw[1])
    rows = raw[2:].reshape(n, 8)
    w = short_walk(4)
    rc, com_r, zmp_r = ref_gen.run(w)
    assert rc == 0 and len(com_r) == n
    e = max(np.abs(rows[:4 * k, :6] - com_r[:4 * k, :6]).max(), np.abs(rows[:, 6:] - zmp_r[:, :2]).max())
    print(r.stdout.strip(), f"; vs reference object {e:.2e} m")
    assert e < 1e-6
