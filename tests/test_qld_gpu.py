"""General dense QP (wg_qld_solve_batch, the ql0001_ calling convention) against the reference's OWN ql0001_ object code
(oracle/_ref: src/Mathematics/qld.cpp compiled where it lies) on identical inputs.  Where that object code is not built,
the inequality-only families are checked against the oracle's exact Goldfarb-Idnani solver (oracle/oracle_qp.cpp)
instead: the QPs are strictly convex, so the minimiser and the set of positive multipliers are unique.  Equalities and
bounds are reduced to that case exactly (exact_qp_eq_bounds); the failure-code test checks the exact solver's own
"inconsistent" code; the Wieber test solves the QP with QLD's diagonal boost added, in extended precision, which reproduces
ql0001_ there.

Criteria (north_star): identical optimal active sets, solution within 1e-6 (relative to its scale), KKT residuals <= 1e-9.
Problem families: random strictly convex QPs of the sizes the reference's callers use (Herdt n = 36 / m = 75, Wieber
n = 150 / m = 300 ... 450), with equalities, with finite bounds, per-QP and shared Hessians, infeasible rows, ragged m."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol

D = ol.D
IP = C.POINTER(C.c_int)


def ref_qld(Cm, d, A, b, me=0, xl=None, xu=None):
    """One call of the reference's ql0001_ (dummy row / mmax = m + 1 as QPProblem::solve and ZMPQPWithConstraint pass it)."""
    r = ol.ref()
    n = len(d); m = len(b)
    mmax = m + 1
    a = np.zeros((n, mmax)); a[:, :m] = A.T                      # column-major, leading dimension mmax
    bb = np.zeros(mmax); bb[:m] = b
    c = np.asfortranarray(Cm).copy(order="F")
    xl = np.full(n, -1e8) if xl is None else np.array(xl, dtype=np.float64)
    xu = np.full(n, 1e8) if xu is None else np.array(xu, dtype=np.float64)
    mnn = m + 2 * n
    x = np.zeros(n); u = np.zeros(mnn)
    lwar = 3 * n * n // 2 + 10 * n + 2 * mmax + 20000
    war = np.zeros(lwar); iwar = np.zeros(n + 10, dtype=np.int32); iwar[0] = 1
    ci = lambda v: C.byref(C.c_int(v))
    ifail = C.c_int(0)
    eps = C.c_double(1e-8)
    dd = np.array(d, dtype=np.float64)
    r.ref_ql0001(ci(m), ci(me), ci(mmax), ci(n), ci(n), ci(mnn), ol.dptr(c), ol.dptr(dd), ol.dptr(a), ol.dptr(bb), ol.dptr(xl),
                 ol.dptr(xu), ol.dptr(x), ol.dptr(u), ci(0), C.byref(ifail), ci(0), ol.dptr(war), ci(lwar),
                 iwar.ctypes.data_as(IP), ci(len(iwar)), C.byref(eps))
    return x, u, ifail.value


def exact_qp(Cm, d, A, b, extended=False):
    """min 1/2 x'Cx + d'x s.t. A x + b >= 0 by the oracle's textbook solver (in x87 extended precision with extended=True)
    -> (x, u [m], rc): rc 0 on success, 3 for inconsistent constraints."""
    n, m = len(d), len(b)
    Cc = np.ascontiguousarray(Cm, dtype=np.float64); dd = np.ascontiguousarray(d, dtype=np.float64)
    Ac = np.ascontiguousarray(A, dtype=np.float64).reshape(m, n) if m else np.zeros((1, n))
    bc = np.ascontiguousarray(b, dtype=np.float64) if m else np.zeros(1)
    x = np.zeros(n); u = np.zeros(max(m, 1))
    o = ol.oracle()
    f = o.oracle_qp_solve_ld if extended else o.oracle_qp_solve
    f.restype = C.c_int
    f.argtypes = [C.c_int, C.c_int, D, D, D, D, D, D, C.c_void_p]
    rc = f(n, m, ol.dptr(Cc), ol.dptr(dd), ol.dptr(Ac), ol.dptr(bc), ol.dptr(x), ol.dptr(u), None)
    return x, u[:m], rc


def exact_qp_eq_bounds(Cm, d, A, b, me, xl, xu):
    """exact_qp with QLD's equalities (rows < me: A x + b = 0) and bounds xl <= x <= xu: the equalities are eliminated
    through a null-space basis, the bounds become rows, and the equality multipliers follow from stationarity.
    -> (x, u [m + 2n] in QLD's layout [rows | lower bounds | upper bounds], rc)."""
    n, m = len(d), len(b)
    Ai = np.vstack([A[me:], np.eye(n), -np.eye(n)]); bi = np.concatenate([b[me:], -np.asarray(xl), np.asarray(xu)])
    Ae = A[:me]
    if me:
        Q, R = np.linalg.qr(Ae.T, mode="complete")
        Z = Q[:, me:]
        x0 = Q[:, :me] @ np.linalg.solve(R[:me].T, -b[:me])
    else:
        Z, x0 = np.eye(n), np.zeros(n)
    y, ui, rc = exact_qp(Z.T @ Cm @ Z, Z.T @ (Cm @ x0 + d), Ai @ Z, Ai @ x0 + bi)
    x = x0 + Z @ y
    ue = np.linalg.lstsq(Ae.T, Cm @ x + d - Ai.T @ ui, rcond=None)[0] if me else np.zeros(0)
    return x, np.concatenate([ue, ui]), rc


def inequality_qp(Cm, d, A, b):
    """The pin of the inequality-only families: the reference's ql0001_ where oracle/_ref is built, else exact_qp."""
    return ref_qld(Cm, d, A, b) if ol.ref() is not None else exact_qp(Cm, d, A, b)


def random_qp(rng, n, m, cond=1e3, active_frac=0.3):
    """Strictly convex QP with a known interior-ish structure: rows are random half-spaces, a fraction of them cutting off
    the unconstrained minimiser."""
    Q, _ = np.linalg.qr(rng.normal(size=(n, n)))
    ev = np.exp(rng.uniform(0, np.log(cond), n))
    Cm = (Q * ev) @ Q.T
    Cm = 0.5 * (Cm + Cm.T)
    d = rng.normal(size=n) * np.sqrt(ev.mean())
    x0 = -np.linalg.solve(Cm, d)
    A = rng.normal(size=(m, n))
    # A x + b >= 0 feasible at the point xf, violated at x0 for some rows
    xf = x0 + rng.normal(size=n) * 0.5
    slack = rng.uniform(0.05, 1.0, m)
    b = -A @ xf + slack
    cut = rng.random(m) < active_frac
    b[cut] = -A[cut] @ (0.5 * (x0 + xf)) - 0 * slack[cut] + (A[cut] @ (xf - x0)).clip(min=0) * 0.0
    # make sure xf stays feasible for the cutting rows
    viol = A @ xf + b
    b[viol < 0.01] += (0.01 - viol[viol < 0.01])
    return Cm, d, A, b


def kkt(Cm, d, A, b, x, u_rows, xl=None, xu=None, u_lo=None, u_up=None, me=0):
    grad = Cm @ x + d - A.T @ u_rows
    if u_lo is not None:
        grad = grad - u_lo + u_up
    s = A @ x + b
    scale = max(1.0, np.abs(d).max())
    stat = np.abs(grad).max() / scale
    rown = np.maximum(np.linalg.norm(A, axis=1), 1e-30)
    feas = min((s[me:] / rown[me:]).min() if len(s) > me else 0.0, 0.0)
    if xl is not None:
        feas = min(feas, (x - xl).min(), (xu - x).min())
        comp_b = max(np.abs(u_lo * (x - xl)).max(), np.abs(u_up * (xu - x)).max()) / scale
    else:
        comp_b = 0.0
    eq = np.abs(s[:me] / rown[:me]).max() if me else 0.0
    comp = max(np.abs(u_rows[me:] * s[me:]).max() / scale if len(s) > me else 0.0, comp_b)
    return stat, feas, eq, comp


def compare(ctx_out, k, Cm, d, A, b, me=0, xl=None, xu=None, xtol=1e-6):
    x, u, ifail, it = ctx_out
    m, n = A.shape
    xr, ur, fr = ref_qld(Cm, d, A, b, me, xl, xu) if (me or xl is not None) else inequality_qp(Cm, d, A, b)
    assert fr == 0 and ifail[k] == 0, (k, fr, ifail[k])
    sc = max(1.0, np.abs(xr).max())
    ex = np.abs(x[k] - xr).max() / sc
    assert ex < xtol, (k, ex)
    big = max(np.abs(ur[:m]).max(initial=0.0), 1e-12)
    act_g = set(np.nonzero(np.abs(u[k, :m]) > 1e-7 * big)[0]); act_r = set(np.nonzero(np.abs(ur[:m]) > 1e-7 * big)[0])
    assert act_g == act_r, (k, sorted(act_g ^ act_r))
    assert (u[k, me:m] >= -1e-12 * big).all()
    has_b = xl is not None
    stat, feas, eq, comp = kkt(Cm, d, A, b, x[k], u[k, :m], xl, xu, u[k, m:m + n] if has_b else None,
                               u[k, m + n:m + 2 * n] if has_b else None, me)
    assert stat < 1e-9 and feas > -1e-9 and eq < 1e-9 and comp < 1e-9, (k, stat, feas, eq, comp)
    return ex, max(stat, -feas, eq, comp)




@pytest.mark.gpu
@pytest.mark.parametrize("n,m,count", [(36, 75, 24), (150, 300, 6), (150, 450, 4), (8, 5, 16), (64, 0, 3)])
def test_gpu_dense_qp_matches_reference_ql0001(ctx, n, m, count):
    rng = np.random.default_rng(100 + n + m)
    probs = [random_qp(rng, n, m) for _ in range(count)] if m else \
        [(lambda Cm, d, A, b: (Cm, d, np.zeros((0, n)), np.zeros(0)))(*random_qp(rng, n, 3)) for _ in range(count)]
    mmax = m + 1
    Cs = np.stack([p[0] for p in probs]); ds = np.stack([p[1] for p in probs])
    As = np.zeros((count, mmax, n)); bs = np.zeros((count, mmax))
    for k, p in enumerate(probs):
        As[k, :m] = p[2]; bs[k, :m] = p[3]
    out = ctx.qld_solve(ds, As, bs, np.full(count, m), C_=Cs)
    worst = (0.0, 0.0)
    for k, p in enumerate(probs):
        e = compare(out, k, *p)
        worst = (max(worst[0], e[0]), max(worst[1], e[1]))
    print(f"n={n} m={m}: max rel |x - x_ql0001| {worst[0]:.2e}, KKT {worst[1]:.2e}, iterations mean {out[3].mean():.1f} max {out[3].max()}")


@pytest.mark.gpu
def test_gpu_dense_qp_equalities_bounds_shared_hessian_and_ragged_m(ctx):
    rng = np.random.default_rng(7)
    n, mmax = 40, 61
    Cm, _, _, _ = random_qp(rng, n, 4)
    ctx.qld_set_shared_hessian(Cm)
    probs = []
    for k in range(20):
        m = int(rng.integers(10, 61))
        me = int(rng.integers(0, 4))
        _, d, A, b = random_qp(rng, n, m)
        x0 = -np.linalg.solve(Cm, d)
        xf = x0 + rng.normal(size=n) * 0.3
        b = -A @ xf + rng.uniform(0.05, 0.5, m)
        b[:me] = -A[:me] @ xf                                       # equalities hold at xf
        tight = rng.random(m) < 0.3
        tight[:me] = False
        b[tight] = -A[tight] @ (0.6 * xf + 0.4 * x0) + np.maximum(A[tight] @ (0.6 * xf + 0.4 * x0) - A[tight] @ xf, 0) * 0 
        viol = A[me:] @ xf + b[me:]
        b[me:][viol < 0.01] += 0.01 - viol[viol < 0.01]
        xl = xf - rng.uniform(0.2, 2.0, n); xu = xf + rng.uniform(0.2, 2.0, n)
        probs.append((d, A, b, me, xl, xu))
    B = len(probs)
    ds = np.stack([p[0] for p in probs])
    As = np.zeros((B, mmax, n)); bs = np.zeros((B, mmax))
    for k, p in enumerate(probs):
        As[k, :len(p[2])] = p[1]; bs[k, :len(p[2])] = p[2]
    ms = np.array([len(p[2]) for p in probs]); mes = np.array([p[3] for p in probs])
    xl = np.stack([p[4] for p in probs]); xu = np.stack([p[5] for p in probs])
    out = ctx.qld_solve(ds, As, bs, ms, me=mes, xl=xl, xu=xu)
    x, u, ifail, it = out
    worst = 0.0
    nb_active = 0
    for k, (d, A, b, me, l, h) in enumerate(probs):
        m = len(b)
        xr, ur, fr = ref_qld(Cm, d, A, b, me, l, h) if ol.ref() is not None else exact_qp_eq_bounds(Cm, d, A, b, me, l, h)
        assert fr == 0 and ifail[k] == 0, (k, fr, ifail[k])
        assert np.abs(x[k] - xr).max() < 1e-6 * max(1.0, np.abs(xr).max()), k
        worst = max(worst, np.abs(x[k] - xr).max())
        big = max(np.abs(ur).max(), 1e-12)
        # rows, lower bounds, upper bounds: same active sets; QLD's layout u = [m rows | n lower | n upper]
        ug = u[k, :m + 2 * n]
        assert set(np.nonzero(np.abs(ug) > 1e-7 * big)[0]) == set(np.nonzero(np.abs(ur) > 1e-7 * big)[0]), k
        nb_active += int((np.abs(u[k, m:m + 2 * n]) > 1e-7 * big).sum())
        stat, feas, eq, comp = kkt(Cm, d, A, b, x[k], u[k, :m], l, h, u[k, m:m + n], u[k, m + n:m + 2 * n], me)
        assert stat < 1e-9 and feas > -1e-9 and eq < 1e-9 and comp < 1e-9, (k, stat, feas, eq, comp)
        assert (x[k] >= l - 1e-9).all() and (x[k] <= h + 1e-9).all()
    assert nb_active > 0                                              # bounds were exercised
    print(f"equalities + bounds + shared Hessian: max |x - x_ql0001| {worst:.2e}, active bounds {nb_active}")


@pytest.mark.gpu
def test_gpu_dense_qp_failure_codes(ctx):
    """Inconsistent constraints report ifail > 10 like QLD; an indefinite Hessian is refused with 2; a bad m with 5."""
    rng = np.random.default_rng(3)
    n = 6
    Cm = np.eye(n)
    A = np.zeros((3, 4, n)); b = np.zeros((3, 4))
    A[:, 0, 0] = 1.0; b[:, 0] = -1.0          # x0 >= 1
    A[:, 1, 0] = -1.0; b[:, 1] = -1.0         # x0 <= -1: inconsistent with row 0
    d = rng.normal(size=(3, n))
    Cs = np.stack([Cm, Cm, Cm])
    Cs[1, 2, 2] = -1.0
    x, u, ifail, it = ctx.qld_solve(d, A, b, np.array([2, 2, 9]), C_=Cs)
    assert ifail[0] > 10 and ifail[1] == 2 and ifail[2] == 5
    if ol.ref() is not None:
        assert ref_qld(Cm, d[0], A[0, :2], b[0, :2])[2] > 10
    else:
        assert exact_qp(Cm, d[0], A[0, :2], b[0, :2])[2] == 3


@pytest.mark.gpu
def test_gpu_dense_qp_on_wieber_qps_reproduces_ql0001_regularisation(ctx):
    """QPs of the Wieber2006 generator (cond(C) = 5e11): with eps = 1e-8 - QLD's diagonal boost, on the host for a shared
    Hessian and inside qld_factor_kernel for per-QP Hessians - the solver reproduces the reference's ql0001_; with eps = 0 it
    returns the minimiser of the QP as stated, whose objective is lower than that of ql0001_'s answer."""
    import ctypes as C
    import dimitrov_oracle as do
    import wieber_oracle as wo
    from test_wieber import short_walk
    N, T = 75, 0.02
    Cm, OptB, OptC = wo.constants()
    w = short_walk(4)
    L, R, st, t, z = wo.inputs(w)
    lci = do.fcals(w["left"], w["right"], w["types"][:, 1])
    o = ol.oracle()
    o.oracle_wieber_build.argtypes = [C.c_int, C.c_double, C.c_double, C.c_int, C.c_void_p, C.c_double, D, D, D, C.POINTER(C.c_int)]
    probs = []
    rng = np.random.default_rng(1)
    for li in (100, 120, 150, 200, 260, 330):
        xk = rng.normal(scale=[0.02, 0.05, 0.2, 0.02, 0.05, 0.2])
        Px = np.zeros(8 * N + 1); Pu = np.zeros((8 * N + 1) * 2 * N); nb = C.c_int(0)
        assert o.oracle_wieber_build(N, T, li * T, len(lci), lci.ctypes.data, 0.80, ol.dptr(xk), ol.dptr(Px), ol.dptr(Pu), C.byref(nb)) == 0
        m = nb.value
        A = Pu[:(m + 1) * 2 * N].reshape(2 * N, m + 1).T[:m].copy(); b = Px[:m].copy()
        zr = np.concatenate([z[li * 4 + 4 * np.arange(N), 0], z[li * 4 + 4 * np.arange(N), 1]])
        probs.append((OptB @ xk - OptC @ zr, A, b))
    mmax = max(len(p[2]) for p in probs) + 1
    B = len(probs)
    ds = np.stack([p[0] for p in probs]); As = np.zeros((B, mmax, 2 * N)); bs = np.zeros((B, mmax))
    for k, p in enumerate(probs):
        As[k, :len(p[2])] = p[1]; bs[k, :len(p[2])] = p[2]
    ms = np.array([len(p[2]) for p in probs])
    boost = ctx.qld_set_shared_hessian(Cm, eps=1e-8)
    assert 1e-8 < boost < 1e-7
    # ql0001_, or without oracle/_ref the QP with QLD's boost added solved in extended precision (the chain that reproduces
    # the reference's Wieber trajectory: test_reference_qld_regularises_the_hessian_and_the_rule_is_restated)
    Cb = Cm + boost * np.eye(len(Cm))
    ql = (lambda d, A, b: ref_qld(Cm, d, A, b)) if ol.ref() is not None else (lambda d, A, b: exact_qp(Cb, d, A, b, True))
    shared = ctx.qld_solve(ds, As, bs, ms)
    per_qp = ctx.qld_solve(ds, As, bs, ms, C_=np.stack([Cm] * B), eps=1e-8)
    ctx.qld_set_shared_hessian(Cm, eps=0.0)
    exact = ctx.qld_solve(ds, As, bs, ms)
    f = lambda x, d: 0.5 * x @ (Cm @ x) + d @ x
    for k, (d, A, b) in enumerate(probs):
        xr, ur, fr = ql(d, A, b)
        assert fr == 0 and shared[2][k] == 0 and per_qp[2][k] == 0 and exact[2][k] == 0
        sc = max(1.0, np.abs(xr).max())
        assert np.abs(shared[0][k] - xr).max() < 1e-6 * sc, (k, np.abs(shared[0][k] - xr).max())
        assert np.abs(per_qp[0][k] - xr).max() < 1e-5 * sc, (k, np.abs(per_qp[0][k] - xr).max())
        act = lambda u: set(np.nonzero(u[:len(b)] > 1e-7 * max(ur.max(), 1e-12))[0])
        assert act(shared[1][k]) == act(ur) == act(per_qp[1][k]), k
        assert (A @ exact[0][k] + b).min() > -1e-8          # the bound the reference itself checks (:1085)
        assert f(exact[0][k], d) <= f(xr, d) + 1e-9 * abs(f(xr, d))
    print(f"Wieber QPs: |x - x_ql0001| shared {max(np.abs(shared[0][k] - ql(*probs[k])[0]).max() for k in range(B)):.2e}, "
          f"per-QP factor {max(np.abs(per_qp[0][k] - ql(*probs[k])[0]).max() for k in range(B)):.2e}; iterations {shared[3]}")


@pytest.mark.gpu
def test_gpu_dense_qp_covers_the_qldandlq_call_of_the_dimitrov_generator(ctx):
    """ZMPConstrainedQPFastFormulation.cpp:1297-1305: in QLDANDLQ mode the generator hands ql0001_ the SAME per-period problem the
    PLDP branch solves (Hessian = identity in the variables L_Q' u, D, the dense (m + 1) x 32 matrix DPu, DPx).  The mode is
    fixed to PLDP in the constructor (:55) and has no setter, so the branch is unreachable in the reference; the call itself is
    covered here: the period QPs of TestKajita2003's straight walk through wg_qld_solve_batch against ql0001_, and against the
    PLDP solution of the same problem (PLDP never drops a row: its objective can only be higher or equal)."""
    import dimitrov_oracle as do
    import pldp_oracle as po
    import zmpdisc_oracle as zo
    w = zo.run(zo.default_params(), zo.profile_steps("StraightWalking"))
    lci = do.fcals(w["left"], w["right"], w["types"][:, 1])
    K = do.Constants()
    N = 16
    rng = np.random.default_rng(2)
    probs = []
    for k in range(24):
        t0 = 0.1 * int(rng.integers(5, 150))
        xk = rng.normal(scale=[0.03, 0.1, 0.3, 0.03, 0.1, 0.3])
        xk[0] += 0.2 * t0 / 3.0
        pr = do.build_constraints(K, lci, t0, xk)
        m = pr["m"]
        A = pr["DPu"].reshape(2 * N, m + 1).T[:m].copy()
        probs.append((pr["D"].copy(), A, pr["DPx"].copy()))
    mmax = max(len(p[2]) for p in probs) + 1
    B = len(probs)
    ds = np.stack([p[0] for p in probs]); As = np.zeros((B, mmax, 2 * N)); bs = np.zeros((B, mmax))
    for k, p in enumerate(probs):
        As[k, :len(p[2])] = p[1]; bs[k, :len(p[2])] = p[2]
    ctx.qld_set_shared_hessian(np.eye(2 * N), eps=1e-8)
    x, u, ifail, it = ctx.qld_solve(ds, As, bs, np.array([len(p[2]) for p in probs]))
    feasible = 0
    for k, (d, A, b) in enumerate(probs):
        xr, ur, fr = inequality_qp(np.eye(2 * N), d, A, b)
        if fr != 0:
            assert ifail[k] != 0, k                  # random states can make a period infeasible: both must say so
            continue
        feasible += 1
        compare((x, u, ifail, it), k, np.eye(2 * N), d, A, b)
    assert feasible >= B // 2
    print(f"Dimitrov QLDANDLQ call: {feasible} feasible period QPs identical to ql0001_ (active sets, x, KKT), iterations mean {it.mean():.1f}")
