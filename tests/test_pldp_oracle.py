"""Pins for the PLDP / OptCholesky oracle (oracle/oracle_pldp.cpp) - all CPU.

The reference ships no test or golden data for PLDPSolver (SURVEY 8c: parity unpinned by golden vectors); the pin is
what the reference's OWN object code (PLDPSolver.cpp / OptCholesky.cpp) returns on identical seeded inputs, stored in
tests/golden/pldp_ref.npz (tests/golden/make_pldp_ref.py) and compared bitwise.  OptCholesky additionally reproduces the reference's only test, tests/TestOptCholesky.cpp
(||A A^T - L L^T||_F <= 1e-6 on a 12 x 15 uniform matrix, rows added one by one; then full Cholesky + inverse).
"""
import os

import numpy as np

import pldp_oracle as po
from jrl_walkgen_b200 import workloads as W

REF = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pldp_ref.npz"))


def test_oracle_optcholesky_reproduces_testoptcholesky():
    rng = np.random.default_rng(0)
    A = rng.uniform(0.0, 1.0, size=(12, 15))                       # tests/TestOptCholesky.cpp:94-103
    L = np.zeros((12, 12))
    rows = np.arange(12, dtype=np.int32)
    for k in range(12):                                             # AddActiveConstraint one by one, :128-140
        po.lib().oracle_optcholesky_add_rows(0, 12, 15, 12, A.ctypes.data, rows.ctypes.data, k, k + 1, L.ctypes.data)
    assert np.linalg.norm(A @ A.T - L @ L.T) <= 1e-6                # :143-150
    M = A @ A.T
    L2 = np.zeros((12, 12)); iL = np.zeros((12, 12))
    po.lib().oracle_optcholesky_full(12, M.ctypes.data, L2.ctypes.data)          # :155-165
    po.lib().oracle_optcholesky_inverse(12, 12, L2.ctypes.data, iL.ctypes.data)  # :166-177
    assert np.linalg.norm(M - L2 @ L2.T) <= 1e-6
    assert np.abs(iL @ L2 - np.eye(12)).max() < 1e-9
    assert np.allclose(L2, np.linalg.cholesky(M), atol=1e-12)


def test_oracle_optcholesky_equals_reference_object_code():
    rng = np.random.default_rng(1)
    for mode, nb, cu in ((0, 12, 15), (1, 20, 32)):
        if mode == 0:
            A = rng.uniform(0.0, 1.0, size=(nb, cu))
        else:
            A = rng.uniform(-1.0, 1.0, size=(cu, nb + 1))           # column-major, leading dimension nb + 1
        A = np.ascontiguousarray(A)
        rows = rng.permutation(nb)[:10].astype(np.int32)
        L = np.zeros((nb, nb))
        po.lib().oracle_optcholesky_add_rows(mode, nb, cu, nb, A.ctypes.data, rows.ctypes.data, 0, 10, L.ctypes.data)
        assert np.array_equal(L, REF["optchol_L%d" % mode])         # bitwise


def test_oracle_pldp_equals_reference_object_code_cold_and_hot():
    """Cold start and a hot-started sequence: X bitwise equal to the reference's PLDPSolver (the 1.3 ms wall-clock cap
    of the reference does not bind on these ~50 us problems)."""
    K, pb = W.pldp_batch(40, seed=3)
    n_act = []
    for b in range(20):
        Xr = REF["cold_X"][b]                                       # fresh solver: no hot-start memory
        X, info, act = po.oracle_solve(K, pb, b, hot=None, starting=True)
        assert info[0] == 0 and info[1] == 0
        assert np.array_equal(X, Xr), (b, np.abs(X - Xr).max())
        n_act.append(info[3])
    assert max(n_act) >= 3                                          # constraints do get activated
    # hot-started receding-horizon sequences on one solver object each: the previous active set and ZMP solution
    # are reused (PLDPSolver.cpp:296-317, :763-778), NumberOfRemovedConstraints = rows of the sample that left
    kept = compared = overshoot = 0
    for seq in range(4):
        rng = np.random.default_rng([9, seq])
        polys = W._support_polygons(rng, K.N, K.T, count=K.N + 25)
        xk_r = np.zeros(6); xk_r[0], xk_r[3] = polys[0][0]
        xk_o = xk_r.copy()
        hot = np.zeros(1, dtype=po.STATE)
        n_removed = 0
        for t in range(25):
            p_o = W.pldp_problem_from(K, polys[t:t + K.N], xk_o)
            X, info, act = po.oracle_solve(K, W.pldp_pack(K, [p_o]), 0, hot=hot, starting=(t == 0), n_removed=n_removed)
            if info[1] == 2:
                # The `tmp2 = -m_tol` clamp (PLDPSolver.cpp:617-618) lets the iterate overshoot an active row by up to
                # m_tol per solve; once the hot-started point violates a row by more than m_tol the step length turns
                # negative and the reference calls exit(0) (:822-828).  The oracle reports status 2 instead; the
                # reference must not be driven there inside the test process.
                overshoot += 1
                assert np.isnan(REF["hot_X"][seq, t]).all()
                break
            Xr = REF["hot_X"][seq, t]
            assert info[0] == 0 and info[1] == 0
            assert np.array_equal(X, Xr), (seq, t, np.abs(X - Xr).max())
            compared += 1
            kept += int(hot["n_prev"][0])
            n_removed = p_o["n_first"]
            xk_r = W.pldp_advance(K, xk_r, Xr); xk_o = W.pldp_advance(K, xk_o, X)
    assert compared >= 40
    assert kept > 0                                                 # the hot start did carry constraints over


def test_oracle_pldp_similar_constraints_semantics_equal_reference_object_code():
    """ComputeAlpha's `A_j = -A_i` reuse (PLDPSolver.cpp:570-590) driven by SimilarConstraints.
    (a) flags consistent with the matrix (row li is the exact negation of row li + similar[li], as FindSimilarConstraints
        guarantees): reference object == oracle with the flags == oracle without them, bitwise - the reuse is bit-neutral;
    (b) backward flags that do NOT match the matrix: the reference reuses -tmp1 of the other row anyway; the oracle
        restates that exactly (bitwise equal X and activation order), and the result differs from the flag-less solve."""
    K, pb = W.pldp_batch(24, seed=11)
    differ = 0
    for b in range(24):
        m = int(pb["m"][b])
        sim_ok = np.ascontiguousarray(pb["similar"][b])
        assert (sim_ok[:m] != 0).sum() == m // 2
        X0, i0, a0 = po.oracle_solve(K, pb, b, starting=True)
        X1, i1, a1 = po.oracle_solve(K, pb, b, starting=True, similar=sim_ok)
        Xr = REF["similar_X"][b]
        assert np.array_equal(X1, Xr) and np.array_equal(X0, X1) and np.array_equal(a0, a1)
        rng = np.random.default_rng([11, b])
        sim_bad = np.zeros(128, dtype=np.int32)
        for li in range(1, m):
            if rng.random() < 0.3:
                sim_bad[li] = -int(rng.integers(1, min(li, 5) + 1))
        X2, i2, a2 = po.oracle_solve(K, pb, b, starting=True, similar=sim_bad)
        if i2[1] != 0:
            assert REF["similar_bad_rc"][b] == -1
            continue          # a wrong reuse can drive the step length negative: the reference would exit(0) there, so
                              # it has a stored solve only where the oracle predicts a clean one
        Xr2, rc = REF["similar_bad_X"][b], REF["similar_bad_rc"][b]
        assert np.array_equal(X2, Xr2, equal_nan=True) and rc == i2[0], (b, np.abs(X2 - Xr2).max())
        differ += int(not np.array_equal(X2, X0))
    assert differ >= 2
    # forward / out-of-range flags: the reference reads stale or uninitialised memory; the oracle refuses (status 6)
    sim_fwd = np.zeros(128, dtype=np.int32); sim_fwd[0] = 2
    assert po.oracle_solve(K, pb, 0, starting=True, similar=sim_fwd)[1][1] == 6


def test_oracle_pldp_solution_is_the_constrained_optimum():
    """Property: X minimises 1/2 |v|^2 + D.v over {A v + b >= 0}: feasibility and KKT with multipliers -v2 >= 0."""
    K, pb = W.pldp_batch(30, seed=5)
    for b in range(30):
        X, info, act = po.oracle_solve(K, pb, b, starting=True)
        m = int(pb["m"][b])
        A = pb["DPu"][b, :(m + 1) * 32].reshape(32, m + 1).T[:m]
        s = A @ X + pb["DPx"][b, :m]
        assert s.min() > -1e-7
        k = info[3]
        E = A[act[:k]]
        g = X + pb["D"][b]                                          # gradient
        if k:
            lam, *_ = np.linalg.lstsq(E.T, g, rcond=None)
            assert np.abs(E.T @ lam - g).max() < 1e-6
            assert np.abs(s[act[:k]]).max() < 1e-6                  # active rows are tight
        else:
            assert np.abs(g).max() < 1e-9
