"""Dimitrov2008 path (support polygons -> constraint matrices -> PLDP -> LIPM): oracle pins (CPU) and CUDA parity (GPU).

Pins (SURVEY 8c: the reference ships no test or datref for this generator - parity unpinned by golden vectors):
  * the convex hull and BuildLinearConstraintInequalities restatements against what the reference's OWN object code
    (ConvexHull.cpp, FootConstraintsAsLinearSystem.cpp) returns on the same inputs - bitwise, stored in
    tests/golden/dimitrov_ref.npz (tests/golden/make_dimitrov_ref.py);
  * the receding-horizon loop against the same loop driven through the reference's own PLDPSolver object - bitwise (stored
    solutions for the straight walk; the whole-generator cases run that object from oracle/_ref);
  * size-independent properties: every previewed CoP lies in its support polygon, the solution is the constrained
    optimum of the reference's cost.
"""
import ctypes as C
import os

import numpy as np
import pytest

import dimitrov_oracle as do
import oracle_lib as ol
import pldp_oracle as po
import zmpdisc_oracle as zo

PROFILES = ("StraightWalking", "Circle", "PbFlorentSeq1", "PbFlorentSeq2")
needs_ref = pytest.mark.skipif(ol.ref() is None or not hasattr(ol.ref(), "ref_fcals_build"),
                               reason="oracle/_ref (reference object code) not built")
REF = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dimitrov_ref.npz"))


def feet_of(name):
    o = zo.run(zo.default_params(), zo.profile_steps(name))
    return o["left"], o["right"], o["types"][:, 1].copy(), o


def assert_same_lci(a, b):
    assert len(a) == len(b)
    for k in ("rows", "similar"):
        assert (a[k] == b[k]).all(), k
    for k in ("A", "B", "center", "t_start", "t_end"):
        assert a[k].tobytes() == b[k].tobytes(), (k, np.abs(a[k] - b[k]).max())


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_oracle_convex_hull_equals_reference_object_code():
    """400 seeded point sets (tests/golden/make_dimitrov_ref.py): two feet with the same or different headings (collinear
    corners, up to 8 vertices), random points, and points with exact ties and collinear triples."""
    for trial in range(len(REF["hull"])):
        pts = REF["hull_points"][trial, :REF["hull_npts"][trial]]
        a, b = do.hull(pts), REF["hull"][trial, :REF["hull_count"][trial]]
        assert a.tobytes() == b.tobytes(), (trial, pts, a, b)


@pytest.mark.parametrize("name", PROFILES)
def test_oracle_fcals_equals_reference_object_code_on_the_kajita_profiles(name):
    left, right, lt, _ = feet_of(name)
    a = do.fcals(left, right, lt)
    b = np.zeros(len(REF["fcals_%s_rows" % name]), dtype=do.LCI)   # the reference reports no first_sample / state / rc
    for k in ("rows", "similar", "A", "B", "center", "t_start", "t_end"):
        b[k] = REF["fcals_%s_%s" % (name, k)]
    assert_same_lci(a, b)
    assert (a["rc"] == 0).all()
    # structure: the walk opens and closes in double support, polygons tile the clock without gaps
    assert a["state"][0] == 3 and a["state"][-1] == 3
    assert (a["t_start"][1:] == a["t_end"][:-1]).all()
    assert a["t_end"][-1] == do.clock(len(left))[-1]
    assert set(a["rows"][a["state"] != 3]) == {4}


def test_oracle_fcals_polygons_contain_their_centre_and_the_support_foot():
    left, right, lt, _ = feet_of("Circle")
    P = do.fcals(left, right, lt)
    for p in P:
        r = p["rows"]
        w = p["A"][:r] @ p["center"] + p["B"][:r]
        assert (w > 0).all()
        i = p["first_sample"]
        for f, z in ((left[i], left[i][2]), (right[i], right[i][2])):
            if z < 1e-5:     # a foot on the ground: its ankle lies inside the polygon
                assert (p["A"][:r] @ f[:2] + p["B"][:r] > 0).all()


def test_oracle_constants_match_independent_numpy_construction():
    from jrl_walkgen_b200 import workloads as W
    K = do.Constants()
    Kn = W.DimitrovConstants()
    for k in ("iLQ", "OptB", "OptC", "Pu", "Px"):
        np.testing.assert_allclose(getattr(K, k), getattr(Kn, k), rtol=1e-9, atol=1e-12, err_msg=k)
    np.testing.assert_allclose(K.iPu @ K.Pu, np.eye(16), atol=1e-7)
    np.testing.assert_allclose(K.iPu, Kn.iPu, rtol=1e-6, atol=1e-6)


def test_oracle_loop_equals_the_loop_driven_through_the_reference_pldp_object():
    """BuildZMPTrajectoryFromFootTrajectory, PLDP branch: the oracle's loop against the same loop with the solve done by
    the reference's PLDPSolver object (hot-start memory inside the object, as in the reference; its solutions stored):
    X bitwise, period by period, up to the period at which the reference's solver would print "PB ON constraint" and call
    exit(0)."""
    left, right, lt, _ = feet_of("StraightWalking")
    par = do.default_params()
    out = do.run(left, right, lt, par)
    per = out["periods"]
    # FINDING: with the reference's own tolerance handling (a constraint within m_tol of its bound is pushed m_tol
    # further, PLDPSolver.cpp:617-618) the hot-started start point of period 17 violates a kept constraint by
    # 1.0000000036e-8 > m_tol, which the reference answers with exit(0) (:822-828).
    assert out["failed_at"] == 17 and per["status"][17] == 2
    assert (per["rc"][:17] == 0).all() and (per["status"][:17] == 0).all()
    K = do.Constants(par)
    P = do.fcals(left, right, lt, par)
    st = 0.0
    for li in range(17):
        xk = per["xk"][li].copy()
        pb = do.build_constraints(K, P, st, xk)
        assert pb["m"] == per["m"][li] and pb["n_first"] == per["n_first"][li]
        assert st == per["t_start"][li]
        X = REF["loop_X"][li]
        jx = 0.0
        jy = 0.0
        for j in range(16):          # the reference's sequential sum (:1382-1400)
            jx += K.iLQ[j, 0] * X[j]
            jy += K.iLQ[j, 0] * X[j + 16]
        assert jx == per["jerk_x"][li] and jy == per["jerk_y"][li], li
        st += par.T


REF_OBJECT_CASES = ("StraightWalking", "StraightWalking@500", "StraightWalking@900", "Circle@200", "Circle@300", "Circle@640",
                    "Circle@1000", "PbFlorentSeq1@700", "PbFlorentSeq1@1500", "PbFlorentSeq2@1200")


@needs_ref
@pytest.mark.parametrize("case", REF_OBJECT_CASES)
def test_oracle_equals_the_reference_generator_object(case):
    """The reference's OWN ZMPConstrainedQPFastFormulation object (its .cpp compiled into oracle/_ref together with
    LinearizedInvertedPendulum2D.cpp and privatepgtypes.cpp; constructor -> InitConstants, then
    BuildZMPTrajectoryFromFootTrajectory in PLDP mode) against the oracle:
      * InitConstants(): Px, Pu = iLQ Pu', iLQ, OptB, OptC BITWISE (both axes' blocks; off-diagonal blocks zero); iPu is LAPACK's
        LU inverse in the reference (MAL_INVERSE) and agrees to 1e-15 relative;
      * the whole loop - polygon look-up by accumulated clocks, DPx / DPu / D, the PLDP solve with the real SimilarConstraints
        flags and hot starts, jerk recovery through iLQ, LIPM interpolation - BITWISE on CoM (x, dx, ddx, y, dy, ddy) and ZMP for
        every period up to the one at which the reference stops, once both sides hold the same iPu; and the stop falls on the
        same period for the same reason: exit(0) after "PB ON constraint" (trapped by the glue) <-> status 2, IFAIL / return -1
        <-> a NaN solution (status 0 with rc -1, or 3 when more than 2N rows were activated).
    "<profile>@<k>" hands the generator the feet buffers from sample k on: every unshifted walk stops at its 18th period (the
    m_tol drift of the hot start during the initial double support), so later phases - single support, rotated feet, the
    duplicated half-planes of arcs - are reached this way; 10 cases, 17 + 148 + 82 + 40 + 34 + 2 + 2 + 77 + 47 + 75 periods.
    With LAPACK's own inverse (1 ulp away) the solver's m_tol pushes (PLDPSolver.cpp:617-618) land differently: 3e-8 m over
    the 17 periods of the unshifted walk - the reason the comparison pins the inverse.  Subprocess: see the glue's exit trap."""
    import json
    import os
    import subprocess
    import sys
    import preview_ref as pr
    if not pr.lapack_available():
        pytest.skip("no LAPACK with dgetrf_/dgetri_ in this image (the reference's MAL_INVERSE)")
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, os.path.join(here, "dimitrov_ref_object.py"), case], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["constants_bitwise"] and d["iPu_rel"] < 1e-14 and d["iPu_Pu_identity"] < 1e-12
    assert d["oracle_stop"] is not None and d["periods_compared"] == d["oracle_stop"]
    if d["ref_rc"] == -100:
        assert d["oracle_stop_status"] == 2, d            # exit(0): negative step length after an infeasible hot start
    else:
        assert d["ref_rc"] == -1 and d["oracle_stop_status"] in (0, 3), d
    if d["periods_compared"]:
        assert d["com_bitwise"] and d["com_err"] == 0.0 and d["zmp_err"] == 0.0, d
    if case == "StraightWalking":
        assert d["periods_compared"] == 17 and d["ref_rc_lapack_inverse"] == -100
        assert d["com_err_lapack_inverse"] < 1e-7 and d["zmp_err_lapack_inverse"] < 1e-7


@needs_ref
@pytest.mark.parametrize("name", PROFILES)
def test_oracle_loop_equals_reference_pldp_object_with_real_similar_flags_whole_walks(name):
    """Every period of all four TestKajita2003 profiles (843 periods) through the reference's PLDPSolver object fed with
    the REAL m_SimilarConstraints of the reference's FootConstraintsAsLinearSystem object code, cold_restart on both
    sides (a fresh solver object where the oracle re-solves from the cold start point): jerks bitwise equal, and where
    the oracle stops on NaN (duplicated half-plane) the reference's SolveProblem returns -1 as well.  Runs in a
    subprocess: a reference exit(0) must not end pytest."""
    import json
    import os
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, os.path.join(here, "dimitrov_ref_loop.py"), name], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["done"] and res["flagged_rows"] > 1000
    expect = {"StraightWalking": (185, None), "Circle": (55, 55), "PbFlorentSeq1": (147, 147), "PbFlorentSeq2": (456, 456)}[name]
    assert (res["compared"], res["failed_at"]) == expect
    assert res["restarts"] >= 2
    if res["failed_at"] is not None:
        assert res["ref_rc_at_stop"] == -1


def test_oracle_loop_stops_like_the_reference_on_duplicated_hull_rows():
    """FINDING: for rotated parallel feet the reference's hull keeps collinear corners (the cross product is not exactly
    0), the final double-support polygon then carries the same half-plane twice, and as soon as both copies are active
    E E^T is singular: Cholesky yields NaN, SolveProblem returns -1 (PLDPSolver.cpp:955-964) and the generator stops
    (IFAIL, ZMPConstrainedQPFastFormulation.cpp:1373-1377).  The polygons are bitwise those of the reference's object
    code (test above), so this is the reference's behaviour on its own Circle profile."""
    left, right, lt, _ = feet_of("Circle")
    par = do.default_params()
    par.cold_restart = 1
    P = do.fcals(left, right, lt, par)
    last = P[-1]
    assert last["rows"] == 6 and (last["A"][1] == last["A"][2]).all() and last["B"][1] == last["B"][2]
    out = do.run(left, right, lt, par)
    assert out["failed_at"] is not None and out["periods"]["rc"][-1] == -1
    assert np.isnan(out["periods"]["jerk_x"][-1])


def test_oracle_robust_mode_completes_every_profile():
    """cold_restart + merge_duplicate_rows (both NOT in the reference, both off by default): every TestKajita2003 profile
    runs to its last period; the polygons only lose rows that repeat their predecessor."""
    par = do.default_params()
    par.cold_restart = 1
    par.merge_duplicate_rows = 1
    for name in PROFILES:
        left, right, lt, _ = feet_of(name)
        out = do.run(left, right, lt, par)
        assert out["failed_at"] is None and len(out["periods"]) == do.period_count(len(left), par), name
        assert set(out["periods"]["status"]) <= {0, 5}
        P0, P1 = do.fcals(left, right, lt), do.fcals(left, right, lt, par)
        assert len(P0) == len(P1) and (P1["rows"] <= P0["rows"]).all() and (P1["rows"] >= 4).all()
        assert (P1["rows"][P0["state"] != 3] == 4).all()
    left, right, lt, _ = feet_of("Circle")
    assert do.fcals(left, right, lt)[-1]["rows"] == 6 and do.fcals(left, right, lt, par)[-1]["rows"] == 4


@pytest.mark.parametrize("name", PROFILES)
def test_oracle_loop_properties(name):
    """Size-independent properties of the generated walk (cold_restart = 1 so that the walk continues where the
    reference would exit): the CoP after every period lies inside the support polygon of its instant (tolerance: the
    solver's m_tol hack lets a bound be crossed by ~1e-8 per period), the CoM follows the feet, accelerations bounded."""
    left, right, lt, o = feet_of(name)
    par = do.default_params()
    par.cold_restart = 1
    out = do.run(left, right, lt, par)
    per = out["periods"]
    good = len(per) if out["failed_at"] is None else out["failed_at"]
    assert good > 50
    assert set(per["status"][:good]) <= {0, 5}
    P = do.fcals(left, right, lt, par)
    for k in range(good):
        # the reference constrains the CoP predicted for t + (i+1) T with the polygon of t + i T (:849-862 vs Px row i)
        t = per["t_start"][k]
        p = P[np.searchsorted(P["t_end"], t, side="left")]
        z = out["zmp"][20 * k + 19]
        r = p["rows"]
        assert (p["A"][:r] @ z + p["B"][:r] > -1e-6).all(), (k, p["A"][:r] @ z + p["B"][:r])
    n = 20 * good
    mid = 0.5 * (left[:n, :2] + right[:n, :2])
    assert np.abs(out["com"][:n, [0, 3]] - mid).max() < 0.15
    assert np.abs(out["com"][:n, [2, 5]]).max() < 5.0
    assert per["iterations"][:good].max() < 40


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_constants_match_oracle(ctx):
    K = do.Constants()
    G = ctx.dimitrov_set_params()
    for k in ("iLQ", "OptB", "OptC", "Pu", "Px"):
        np.testing.assert_allclose(G[k], getattr(K, k), rtol=1e-12, atol=1e-14, err_msg=k)
    np.testing.assert_allclose(G["iPu"], K.iPu, rtol=1e-9, atol=1e-9)


@pytest.mark.gpu
def test_gpu_convex_hull_matches_oracle_bitwise(ctx):
    rng = np.random.default_rng(11)
    B = 2048
    pts = rng.uniform(-1, 1, (B, 8, 2))
    pts[::2] = np.round(pts[::2] * 4) / 4
    for b in range(0, B, 5):       # parallel feet
        x0, x1 = rng.uniform(-0.2, 0.2, 2)
        k = 0
        for (x, y) in ((x0, 0.095), (x1, -0.095)):
            for lx, ly in ((1, -1), (1, 1), (-1, 1), (-1, -1)):
                pts[b, k] = (x + lx * 0.085, y + ly * 0.03); k += 1
    hull, cnt = ctx.convex_hull_batch(pts)
    checked = 0
    for b in range(B):
        if len(np.unique(pts[b], axis=0)) < 3:
            continue
        h = do.hull(pts[b])
        assert cnt[b] == len(h), (b, pts[b], h, hull[b])
        assert hull[b, :cnt[b]].tobytes() == h.tobytes(), b
        checked += 1
    assert checked > B * 0.9


@pytest.mark.gpu
@pytest.mark.parametrize("name", PROFILES)
def test_gpu_fcals_matches_oracle(ctx, name):
    """The polygons of the four TestKajita2003 profiles from the SAME feet buffers (the oracle's): rows, similar flags,
    clock stamps and first samples identical; A, B, centre to 1e-12 (device sin/cos differ from glibc's in the last
    bit when the feet are rotated; bitwise when they are not)."""
    left, right, lt, o = feet_of(name)
    ref = do.fcals(left, right, lt)
    ctx.dimitrov_set_params()
    got = ctx.fcals_build(left, right, o["types"])
    assert len(got) == len(ref)
    for k in ("rows", "first_sample", "state", "rc"):
        assert (got[k] == ref[k]).all(), k
    for k in ("t_start", "t_end"):
        assert got[k].tobytes() == ref[k].tobytes(), k
    for k in ("A", "B", "center"):
        np.testing.assert_allclose(got[k], ref[k], rtol=0, atol=1e-12, err_msg=k)
    # SimilarConstraints are exact-equality tests on slopes (A_i == -A_j): a last-bit difference of sin/cos flips
    # them for rotated feet; they only select a bit-neutral shortcut inside the solver
    assert (got["similar"] == ref["similar"]).mean() > 0.9
    if name == "StraightWalking":
        for k in ("A", "B", "center", "similar"):
            assert got[k].tobytes() == ref[k].tobytes(), k


def _gpu_params(cold):
    import jrl_walkgen_b200 as wg
    p = wg.dimitrov_default_params()
    p.cold_restart = cold
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("cold", (0, 1))
@pytest.mark.parametrize("name", PROFILES)
def test_gpu_dimitrov_closed_loop_matches_oracle(ctx, name, cold):
    """footsteps -> ZMPDiscretization -> polygons -> PLDP loop -> CoM/ZMP, all on the device, against the oracle chain:
    cold = 0 the reference-faithful mode (the walk stops where the reference would exit), cold = 1 with cold restarts."""
    steps = zo.profile_steps(name)
    o = zo.run(zo.default_params(), steps)
    par = do.default_params()
    par.cold_restart = cold
    ref = do.run(o["left"], o["right"], o["types"][:, 1].copy(), par)
    ctx.dimitrov_set_params(_gpu_params(cold))
    out = ctx.dimitrov_run([steps], [zo.INIT_FEET])
    per, rper = out["periods"][0], ref["periods"]
    assert out["status"][0] == (0 if ref["failed_at"] is None else 1)
    good = len(rper) if ref["failed_at"] is None else ref["failed_at"]
    if ref["failed_at"] is not None and rper["rc"][-1] == -1:
        # a NaN stop (both copies of a duplicated half-plane active, see the CPU test): WHEN the second copy enters the
        # active set hangs on last-bit ties between the two copies, i.e. on sin/cos of the rotated feet
        assert per["rc"][-1] == -1 and abs(len(per) - len(rper)) <= 3, (len(per), len(rper))
        good = min(good, len(per) - 1)
        per, rper = per[:good], rper[:good]
    else:
        assert len(per) == len(rper), (len(per), len(rper))
    assert (per["m"] == rper["m"]).all() and (per["n_first"] == rper["n_first"]).all()
    assert (per["status"] == rper["status"]).all() and (per["rc"] == rper["rc"]).all()
    assert per["t_start"].tobytes() == rper["t_start"].tobytes()
    same_sets = np.mean([set(a[a >= 0]) == set(b[b >= 0]) for a, b in zip(per["active"][:good], rper["active"][:good])])
    assert same_sets > 0.98, same_sets
    n = 20 * good      # (sample 20*good is written twice: extrapolated by period good-1, then by period good if it runs)
    np.testing.assert_allclose(out["com"][:n, [0, 3]], ref["com"][:n, [0, 3]], rtol=0, atol=1e-6)     # north_star: 1e-6 m
    np.testing.assert_allclose(out["zmp"][:n], ref["zmp"][:n], rtol=0, atol=1e-6)
    np.testing.assert_allclose(out["com"][:n], ref["com"][:n], rtol=0, atol=1e-5)
    if name == "StraightWalking":      # no rotated foot: every operation is the same IEEE operation on both sides
        assert out["com"][:n].tobytes() == ref["com"][:n].tobytes()
        assert out["zmp"][:n].tobytes() == ref["zmp"][:n].tobytes()
        assert (per["active"] == rper["active"]).all() and (per["iterations"] == rper["iterations"]).all()
    nw = 20 * (out["periods_done"][0] - (1 if out["status"][0] else 0)) + 1    # rows the GPU loop wrote
    assert np.abs(out["com"][nw:]).max() == 0.0
    # rows the loop does not reach keep the discretised ZMP reference
    np.testing.assert_array_equal(out["zmp"][nw:], o["zmp"][nw:, :2])


@pytest.mark.gpu
@needs_ref
def test_gpu_dimitrov_equals_the_reference_generator_object(ctx, tmp_path):
    """wg_dimitrov_run_batch (defaults = the reference's semantics) against the reference's OWN ZMPConstrainedQPFastFormulation
    object on TestKajita2003's straight walk: the reference ends the process at its 18th period (exit(0), trapped by the glue);
    the GPU walk stops there with status 1, and the 340 rows of CoM (x, dx, ddx, y, dy, ddy) and ZMP before it are BITWISE the
    object's when it holds the product's iPu, and within 1e-7 m when it keeps LAPACK's own inverse."""
    import json
    import os
    import subprocess
    import sys
    import preview_ref as pr
    if not pr.lapack_available():
        pytest.skip("no LAPACK with dgetrf_/dgetri_ in this image (the reference's MAL_INVERSE)")
    G = ctx.dimitrov_set_params(_gpu_params(0))
    np.save(tmp_path / "ipu.npy", np.ascontiguousarray(G["iPu"]))
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, os.path.join(here, "dimitrov_ref_object.py"), "StraightWalking",
                        str(tmp_path / "rows.npz"), str(tmp_path / "ipu.npy")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["ref_rc"] == -100 and d["periods_compared"] == 17
    rows = np.load(tmp_path / "rows.npz")
    out = ctx.dimitrov_run([zo.profile_steps("StraightWalking")], [zo.INIT_FEET])
    assert out["status"][0] == 1 and out["periods_done"][0] in (17, 18)
    n = 340
    assert out["com"][:n].tobytes() == rows["com"].tobytes()
    assert out["zmp"][:n].tobytes() == rows["zmp"].tobytes()
    assert np.abs(out["com"][:n] - rows["com_lapack"]).max() < 1e-7 and np.abs(out["zmp"][:n] - rows["zmp_lapack"]).max() < 1e-7


@pytest.mark.gpu
@pytest.mark.parametrize("name", PROFILES)
def test_gpu_dimitrov_robust_mode_matches_oracle(ctx, name):
    """cold_restart + merge_duplicate_rows: every profile completes on the device as in the oracle."""
    import jrl_walkgen_b200 as wg
    steps = zo.profile_steps(name)
    o = zo.run(zo.default_params(), steps)
    par = do.default_params()
    par.cold_restart = 1; par.merge_duplicate_rows = 1
    ref = do.run(o["left"], o["right"], o["types"][:, 1].copy(), par)
    gp = wg.dimitrov_default_params()
    gp.cold_restart = 1; gp.merge_duplicate_rows = 1
    ctx.dimitrov_set_params(gp)
    out = ctx.dimitrov_run([steps], [zo.INIT_FEET])
    per, rper = out["periods"][0], ref["periods"]
    assert out["status"][0] == 0 and ref["failed_at"] is None and len(per) == len(rper) == out["period_counts"][0]
    assert (per["m"] == rper["m"]).all() and set(per["status"]) <= {0, 5}
    # The cold-restart decision is the reference's `violation > m_tol` test on a violation that the solver's own
    # tolerance handling parks AT m_tol (1.0000000x e-8): with rotated feet (device sin/cos differ from glibc's in the
    # last bit) the two sides can decide differently, and since PLDP never drops a constraint inside a solve the
    # restarted period ends on a different vertex.  Parity is therefore asserted up to the first differing decision
    # (456 of 497 periods on PbFlorentSeq2, all periods on the other profiles); the rest is checked by property.
    differ = np.nonzero(per["status"] != rper["status"])[0]
    good = len(per) if len(differ) == 0 else int(differ[0])
    assert good >= 0.9 * len(per), (good, len(per))
    if name != "PbFlorentSeq2":
        assert good == len(per)
    n = 20 * good
    np.testing.assert_allclose(out["com"][:n, [0, 3]], ref["com"][:n, [0, 3]], rtol=0, atol=1e-6)
    np.testing.assert_allclose(out["zmp"][:n], ref["zmp"][:n], rtol=0, atol=1e-6)
    P = ctx.fcals_build(o["left"], o["right"], o["types"])
    Pr = do.fcals(o["left"], o["right"], o["types"][:, 1].copy(), par)
    assert (P["rows"] == Pr["rows"]).all()
    for k in range(len(per)):         # every period, including those after a differing decision: CoP inside its polygon
        pk = P[np.searchsorted(P["t_end"], per["t_start"][k], side="left")]
        r = pk["rows"]
        assert (pk["A"][:r] @ out["zmp"][20 * k + 19] + pk["B"][:r] > -1e-6).all(), k
    ctx.dimitrov_set_params()


@pytest.mark.gpu
def test_gpu_dimitrov_batch_properties(ctx):
    """A ragged batch of random walks: the CoP after every period inside the polygon of its instant, walks independent
    of their batch neighbours (same walk alone = same bits), straight walks complete."""
    from jrl_walkgen_b200 import workloads as W
    off, steps, feet = W.kajita_steps_batch(48, seed=5)
    walks = [steps[off[b]:off[b + 1]] for b in range(48)]
    ctx.dimitrov_set_params(_gpu_params(1))
    out = ctx.dimitrov_run(walks, feet)
    assert set(out["status"]) <= {0, 1}
    # straight walks (no rotated foot) run the same IEEE operations as the oracle: same stops (some end with the NaN
    # exit of the reference when the closing double-support hull carries two nearly identical vertical edges), same bits
    straight = [b for b in range(48) if (walks[b]["theta"] == 0).all()]
    assert len(straight) > 5
    par = do.default_params()
    par.cold_restart = 1
    completed = 0
    for b in straight:
        s0, s1 = out["sample_offsets"][b], out["sample_offsets"][b + 1]
        o = zo.run(zo.default_params(), walks[b].astype(zo.REL_STEP_DTYPE), feet[b])
        ref = do.run(o["left"], o["right"], o["types"][:, 1].copy(), par)
        assert out["status"][b] == (0 if ref["failed_at"] is None else 1), b
        assert out["periods_done"][b] == len(ref["periods"]), b
        good = len(ref["periods"]) - (0 if ref["failed_at"] is None else 1)
        assert out["com"][s0:s0 + 20 * good].tobytes() == ref["com"][:20 * good].tobytes(), b
        completed += ref["failed_at"] is None
        if ref["failed_at"] is None:
            assert out["periods_done"][b] == out["period_counts"][b]
    assert completed >= len(straight) // 2
    solo = ctx.dimitrov_run([walks[7]], [feet[7]])
    s0, s1 = out["sample_offsets"][7], out["sample_offsets"][8]
    assert out["com"][s0:s1].tobytes() == solo["com"].tobytes()
    for b in (0, 7, 31):
        s0, s1 = out["sample_offsets"][b], out["sample_offsets"][b + 1]
        per = out["periods"][b]
        good = len(per) - (1 if out["status"][b] else 0)
        assert set(per["status"][:good]) <= {0, 5}
        P = ctx.fcals_build(out["left"][s0:s1], out["right"][s0:s1], out["types"][s0:s1])
        for k in range(good):
            t = per["t_start"][k]
            p = P[np.searchsorted(P["t_end"], t, side="left")]
            z = out["zmp"][s0 + 20 * k + 19]
            r = p["rows"]
            assert (p["A"][:r] @ z + p["B"][:r] > -1e-6).all(), (b, k)


@pytest.mark.gpu
def test_gpu_dimitrov_edge_cases(ctx):
    """Error conventions and degenerate inputs of the Dimitrov entry points: too few period records and too small a
    polygon capacity are refused (WG_ERR_INVALID), a context without constants answers WG_ERR_NOT_READY, a walk that is
    a single (initial) step - double support from the first to the last sample - runs and matches the oracle."""
    import jrl_walkgen_b200 as wg
    from jrl_walkgen_b200 import _capi
    steps = zo.profile_steps("StraightWalking")
    # (1) not ready: a fresh context has no Dimitrov constants
    c2 = wg.Context(0)
    try:
        plan = wg.KajitaPlan(c2, np.array([0, len(steps)], dtype=np.int64), steps, zo.INIT_FEET)
        rc = c2.lib.wg_dimitrov_run_batch(c2.h, plan.h, wg.WG_MEM_HOST, None, None, None, None, None, None, None, None)
        assert rc == _capi.WG_ERR_NOT_READY
        plan.destroy()
    finally:
        c2.close()
    # (2) period records: one fewer than the loop needs
    ctx.dimitrov_set_params()
    plan = wg.KajitaPlan(ctx, np.array([0, len(steps)], dtype=np.int64), steps, zo.INIT_FEET)
    need = int(ctx.lib.wg_dimitrov_period_count(C.byref(ctx.dimitrov_params), int(plan.total_samples)))
    assert need == 185
    per = np.zeros(need, dtype=wg.DIMITROV_PERIOD_DTYPE)
    po = np.array([0, need - 1], dtype=np.int64)
    rc = ctx.lib.wg_dimitrov_run_batch(ctx.h, plan.h, wg.WG_MEM_HOST, None, None, None, None,
                                       po.ctypes.data_as(_capi.c_i64_p), per.ctypes.data, None, None)
    assert rc == _capi.WG_ERR_INVALID
    plan.destroy()
    # (3) polygon capacity
    o = zo.run(zo.default_params(), steps)
    with pytest.raises(wg.WalkgenError):
        ctx.fcals_build(o["left"], o["right"], o["types"], cap=5)
    # (4) a walk of one step: the whole buffer is one double-support polygon
    one = steps[:1].copy()
    o1 = zo.run(zo.default_params(), one)
    ref = do.run(o1["left"], o1["right"], o1["types"][:, 1].copy())
    out = ctx.dimitrov_run([one], [zo.INIT_FEET])
    P = ctx.fcals_build(o1["left"], o1["right"], o1["types"])
    assert len(P) == 1 and P["state"][0] == 3 and P["rows"][0] == 4
    assert out["status"][0] == (0 if ref["failed_at"] is None else 1) and out["periods_done"][0] == len(ref["periods"])
    good = len(ref["periods"]) - (0 if ref["failed_at"] is None else 1)
    assert out["com"][:20 * good].tobytes() == ref["com"][:20 * good].tobytes()
