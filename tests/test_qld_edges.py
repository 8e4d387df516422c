"""The dense QP solver (wg_qld_solve_batch, wg_qld_solve_batch_ranked) at the edges of the contract its header states: the
ranked entry, dependent and degenerate rows, zero rows, the n / m limits, padded layouts, device memory, a batch large
enough that every CTA of the persistent grid solves several QPs, and a caller's shared Hessian next to the Wieber
generator's.  Calls the Context wrapper cannot express (nmax > n, padded strides, u / iterations / me = NULL, device
memory, the ranked entry) go straight to the C ABI through ctypes.

The reference is independent of the kernel: the problem is materialised in numpy (ranked rows expanded into the dense
m x 2N matrix, bounds as rows), its equalities are eliminated through an SVD null space (so rank-deficient equality blocks
work), and the rest is solved by the oracle's Goldfarb-Idnani method in x87 extended precision (oracle_qp_solve_ld).
Every GPU answer is also certified by a KKT check in long double: stationarity, primal feasibility, inequality multipliers
>= 0 and complementarity, each <= 1e-9 relative.  Where oracle/_ref is built, the reference's own ql0001_ is compared too.
Tolerances for cond(C) <= 1e4: x within 1e-10 of the reference relative to its scale, identical active sets (multipliers
above 1e-7 of the largest).  Where rows are dependent their multipliers are not unique: there only x, the inequality
multipliers that are unique and the KKT certificate are compared."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol
from jrl_walkgen_b200 import _capi

LD = np.longdouble
D = ol.D
WG_MEM_HOST, WG_MEM_DEVICE, WG_ERR_INVALID = _capi.WG_MEM_HOST, _capi.WG_MEM_DEVICE, _capi.WG_ERR_INVALID
QLD_MAX_N, QLD_MAX_M = 160, 1024
XTOL = 1e-10


# ---------------------------------------------------------------------------------------------------------------------
# reference helpers (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def eliminate(Ae, be, rtol=1e-12):
    """The solutions of Ae x + be = 0 through the SVD of Ae: -> (x0, Z, consistent), every solution x0 + Z y, Z an
    orthonormal basis of the null space of Ae (n - rank columns).  Works on rank-deficient blocks."""
    Ae = np.asarray(Ae, dtype=np.float64).reshape(-1, np.shape(Ae)[-1])
    n = Ae.shape[1]
    if len(Ae) == 0:
        return np.zeros(n), np.eye(n), True
    U, s, Vt = np.linalg.svd(Ae)
    r = int((s > rtol * s.max()).sum()) if s.max() > 0 else 0
    x0 = Vt[:r].T @ ((U[:, :r].T @ -np.asarray(be, dtype=np.float64)) / s[:r])
    res = Ae @ x0 + be
    scale = np.abs(be).max() + np.linalg.norm(Ae, axis=1).max() * np.abs(x0).max()
    return x0, Vt[r:].T, bool(np.abs(res).max() <= 1e-9 * scale)


def first_inconsistent(Ae, be):
    """0-based index of the first equality row that cannot hold together with the rows before it, or -1."""
    for j in range(len(be)):
        if not eliminate(Ae[:j + 1], be[:j + 1])[2]:
            return j
    return -1


def ranked_dense(A0, A1, samp, uz, N):
    """The m x 2N matrix of rank-structured rows: element (r, k + N ax) = A_ax[r] uz[s - k] for k <= s = min(samp[r], N - 1)."""
    m = len(A0)
    A = np.zeros((m, 2 * N))
    for r in range(m):
        s = min(int(samp[r]), N - 1)
        col = uz[s - np.arange(s + 1)]
        A[r, :s + 1] = A0[r] * col
        A[r, N:N + s + 1] = A1[r] * col
    return A


def _oracle_ld(Cm, d, A, b):
    n, m = len(d), len(b)
    Cc = np.ascontiguousarray(0.5 * (Cm + Cm.T)); dd = np.ascontiguousarray(d, dtype=np.float64)
    Ac = np.ascontiguousarray(A, dtype=np.float64).reshape(m, n) if m else np.zeros((1, n))
    bc = np.ascontiguousarray(b, dtype=np.float64) if m else np.zeros(1)
    x = np.zeros(n); u = np.zeros(max(m, 1))
    f = ol.oracle().oracle_qp_solve_ld
    f.restype = C.c_int
    f.argtypes = [C.c_int, C.c_int, D, D, D, D, D, D, C.c_void_p]
    rc = f(n, m, ol.dptr(Cc), ol.dptr(dd), ol.dptr(Ac), ol.dptr(bc), ol.dptr(x), ol.dptr(u), None)
    return x, u[:m], rc


def reference(p):
    """min 1/2 x'Cx + d'x  s.t.  A[:me] x + b = 0, A[me:] x + b >= 0, xl <= x <= xu, solved without the kernel.
    -> (x, u in QLD's layout [m rows | n lower | n upper], status): status 0, 10 + j (1-based j) for an equality row that
    contradicts the ones before it, 3 when the inequalities cannot be met.  Kept in p["_ref"]."""
    if "_ref" not in p:
        p["_ref"] = _reference(p)
    return p["_ref"]


def _reference(p):
    Cm, d, A, b, me = p["C"], p["d"], p["A"], p["b"], p.get("me", 0)
    xl, xu = p.get("xl"), p.get("xu")
    n, m = len(d), len(b)
    j = first_inconsistent(A[:me], b[:me])
    if j >= 0:
        return None, None, 10 + j + 1
    x0, Z, _ = eliminate(A[:me], b[:me])
    assert Z.shape[1] > 0, "the equalities fix x: not a case of this suite"
    Ai, bi = A[me:], b[me:]
    if xl is not None:
        Ai = np.vstack([Ai, np.eye(n), -np.eye(n)]); bi = np.concatenate([bi, -xl, xu])
    y, ui, rc = _oracle_ld(Z.T @ Cm @ Z, Z.T @ (Cm @ x0 + d), Ai @ Z, Ai @ x0 + bi)
    if rc != 0:
        return None, None, rc
    x = x0 + Z @ y
    ue = np.linalg.lstsq(A[:me].T, Cm @ x + d - Ai.T @ ui, rcond=None)[0] if me else np.zeros(0)
    return x, np.concatenate([ue, ui]), 0


def kkt_ld(p, x, u):
    """KKT residuals of (x, u) in long double, each relative: stationarity, equality and inequality feasibility, dual
    feasibility of the inequality and bound multipliers, complementarity."""
    Cm, d, A, b = (np.asarray(p[k], dtype=LD) for k in ("C", "d", "A", "b"))
    me = p.get("me", 0)
    n, m = len(d), len(b)
    x_, u_ = np.asarray(x, dtype=LD), np.asarray(u, dtype=LD)
    A = A.reshape(m, n)
    g = Cm @ x_ + d - A.T @ u_[:m]
    bounds = p.get("xl") is not None
    if bounds:
        xl, xu = np.asarray(p["xl"], dtype=LD), np.asarray(p["xu"], dtype=LD)
        g = g - u_[m:m + n] + u_[m + n:m + 2 * n]
    scale = max(1.0, float(np.abs(d).max()), float(np.abs(Cm @ x_).max()))
    xs = max(1.0, float(np.abs(x_).max()))
    big = max(1.0, float(np.abs(u_).max(initial=0.0)))
    rown = np.sqrt((A * A).sum(axis=1)); rown[rown == 0] = 1
    s = (A @ x_ + b) / rown
    r = {"stat": float(np.abs(g).max()) / scale,
         "eq": float(np.abs(s[:me]).max(initial=0)) / xs,
         "feas": float(max(0, -s[me:].min(initial=0))) / xs,
         "dual": float(max(0, -u_[me:m].min(initial=0))) / big,
         "comp": float(np.abs(u_[me:m] * s[me:]).max(initial=0)) / scale}
    if bounds:
        r["feas"] = max(r["feas"], float(max(0, -(x_ - xl).min(), -(xu - x_).min())) / xs)
        r["dual"] = max(r["dual"], float(max(0, -u_[m:m + 2 * n].min())) / big)
        r["comp"] = max(r["comp"], float(max(np.abs(u_[m:m + n] * (x_ - xl)).max(),
                                             np.abs(u_[m + n:m + 2 * n] * (xu - x_)).max())) / scale)
    return r


def certify(p, x, u, tol=1e-9, what=""):
    r = kkt_ld(p, x, u)
    assert max(r.values()) <= tol, (what, r)
    return max(r.values())


def active(u, big=None):
    big = max(np.abs(u).max(initial=0.0), 1e-12) if big is None else big
    return set(np.nonzero(np.abs(u) > 1e-7 * big)[0])


def check_against_reference(p, x, u, what, sets=True, ineq_u=False):
    """x within XTOL of the reference, the KKT certificate, and identical active sets (sets) or, where the equality rows
    are dependent, identical inequality multipliers (ineq_u); u in QLD's layout.  -> (|dx| relative, KKT)."""
    xr, ur, st = reference(p)
    assert st == 0, (what, st)
    m = len(p["b"])
    ex = np.abs(x - xr).max() / max(1.0, np.abs(xr).max())
    assert ex < XTOL, (what, ex)
    if sets:
        lay = len(ur)
        assert active(u[:lay], max(np.abs(ur).max(initial=0), 1e-12)) == active(ur), (what, sorted(active(u[:lay]) ^ active(ur)))
    if ineq_u:
        me = p.get("me", 0)
        assert np.abs(u[me:] - ur[me:]).max(initial=0) <= 1e-7 * max(1.0, np.abs(ur[me:]).max(initial=0)), what
    k = certify(p, x, u, what=what)
    if ol.ref() is not None:
        from test_qld_gpu import ref_qld
        xq, _, fq = ref_qld(p["C"], p["d"], p["A"], p["b"], p.get("me", 0), p.get("xl"), p.get("xu"))
        assert fq == 0 and np.abs(xq - xr).max() < 1e-6 * max(1.0, np.abs(xr).max()), what
    return ex, k


def spd(rng, n, cond=1e2):
    Q, _ = np.linalg.qr(rng.normal(size=(n, n)))
    ev = np.exp(rng.uniform(0, np.log(cond), n))
    Cm = (Q * ev) @ Q.T
    return 0.5 * (Cm + Cm.T)


def make_qp(rng, n, m, me=0, bounds=False, cond=1e2, Cm=None, spread=3.0):
    """A feasible strictly convex QP: the rows hold at xf (equalities exactly, inequalities with a random slack), the
    unconstrained minimiser lies `spread` away, so that a good share of the rows and bounds is active."""
    Cm = spd(rng, n, cond) if Cm is None else Cm
    xf = rng.normal(size=n)
    x0 = xf + spread * rng.normal(size=n)
    A = rng.normal(size=(m, n))
    b = -A @ xf + rng.uniform(0.0, 1.0, m)
    b[:me] = -A[:me] @ xf
    p = {"C": Cm, "d": -Cm @ x0, "A": A, "b": b, "me": me}
    if bounds:
        p["xl"] = xf - rng.uniform(0.2, 2.0, n); p["xu"] = xf + rng.uniform(0.2, 2.0, n)
    return p


# ---------------------------------------------------------------------------------------------------------------------
# the C ABI through ctypes
# ---------------------------------------------------------------------------------------------------------------------
def pack(probs, n, nmax=None, mmax=None, a_pad=0, b_pad=0, u_pad=0, fill=0.0):
    """ql0001_'s layout for a batch: C column-major with leading dimension nmax, A column-major with leading dimension
    mmax at stride a_stride = mmax n + a_pad, b at stride mmax + b_pad.  Padding holds `fill`."""
    B = len(probs)
    nmax = n if nmax is None else nmax
    mmax = max(len(p["b"]) for p in probs) if mmax is None else mmax
    bounds = probs[0].get("xl") is not None
    a_stride, b_stride = mmax * n + a_pad, mmax + b_pad
    A = np.full((B, max(a_stride, 1)), fill); b = np.full((B, max(b_stride, 1)), fill); Cc = np.full((B, nmax * n), fill)
    for k, p in enumerate(probs):
        m = len(p["b"])
        A[k, :mmax * n].reshape(n, mmax)[:, :m] = np.asarray(p["A"]).reshape(m, n).T
        b[k, :m] = p["b"]
        Cc[k].reshape(n, nmax)[:, :n] = p["C"].T
    out = {"probs": probs, "n": n, "nmax": nmax, "mmax": mmax, "a_stride": a_stride, "b_stride": b_stride,
           "u_stride": mmax + (2 * n if bounds else 0) + u_pad, "A": A, "b": b, "C": Cc,
           "d": np.stack([p["d"] for p in probs]).astype(np.float64),
           "m": np.array([p.get("m", len(p["b"])) for p in probs], dtype=np.int32),
           "me": np.array([p.get("me", 0) for p in probs], dtype=np.int32)}
    if bounds:
        out["xl"] = np.stack([p["xl"] for p in probs]); out["xu"] = np.stack([p["xu"] for p in probs])
    return out


def solve_raw(ctx, pk, shared=False, mem=WG_MEM_HOST, eps=0.0, no_u=False, no_it=False, no_me=False, ranked=None):
    """One wg_qld_solve_batch (or, with ranked = (A0, A1, samp, row_stride, uz, N), wg_qld_solve_batch_ranked) call.
    -> (rc, x, u, ifail, iterations)."""
    B, n = pk["d"].shape
    q = _capi.QldBatch()
    q.n, q.nmax, q.mmax, q.shared_hessian, q.eps = pk.get("n_call", n), pk["nmax"], pk["mmax"], int(shared), float(eps)
    q.a_stride, q.b_stride, q.u_stride = pk["a_stride"], pk["b_stride"], pk["u_stride"]
    x = np.zeros((B, n)); u = np.full((B, pk["u_stride"]), 7.0)
    ifail = np.full(B, -99, dtype=np.int32); it = np.full(B, -99, dtype=np.int32)
    ins = {"m": pk["m"], "me": None if no_me else pk["me"], "C": None if shared else pk["C"], "d": pk["d"], "A": pk["A"],
           "b": pk["b"], "xl": pk.get("xl"), "xu": pk.get("xu")}
    outs = {"x": x, "u": None if no_u else u, "ifail": ifail, "iterations": None if no_it else it}
    bufs = []
    if ranked is not None or mem == WG_MEM_DEVICE:
        def dev(a):
            if a is None:
                return None
            buf = ctx.to_device(np.ascontiguousarray(a)); bufs.append(buf)
            return buf.ptr
        for k, a in ins.items():
            setattr(q, k, dev(a))
        dout = {k: dev(a) for k, a in outs.items()}
        for k, p in dout.items():
            setattr(q, k, p)
    else:
        for k, a in list(ins.items()) + list(outs.items()):
            setattr(q, k, None if a is None else a.ctypes.data)
    try:
        if ranked is None:
            rc = ctx.lib.wg_qld_solve_batch(ctx.h, mem, B, C.byref(q))
        else:
            A0, A1, samp, row_stride, uz, N = ranked
            rp = [dev(np.ascontiguousarray(A0, dtype=np.float64)), dev(np.ascontiguousarray(A1, dtype=np.float64)),
                  dev(np.ascontiguousarray(samp, dtype=np.uint8)), dev(np.ascontiguousarray(uz, dtype=np.float64))]
            rc = ctx.lib.wg_qld_solve_batch_ranked(ctx.h, mem, B, C.byref(q), C.c_void_p(rp[0]), C.c_void_p(rp[1]),
                                                   C.c_void_p(rp[2]), C.c_longlong(row_stride), C.c_void_p(rp[3]), N)
        if rc == 0 and bufs:
            ctx.sync()
            for k, a in outs.items():
                if a is not None:
                    a[...] = bufs[[b.ptr for b in bufs].index(dout[k])].download(a.dtype, a.shape)
    finally:
        for buf in bufs:
            buf.free()
    return rc, x, u, ifail, it


def solve_ok(ctx, pk, **kw):
    rc, x, u, ifail, it = solve_raw(ctx, pk, **kw)
    assert rc == 0, (rc, ctx.lib.wg_last_error(ctx.h).decode())
    return x, u, ifail, it


def sm_count():
    cudart = C.CDLL("libcudart.so.12")       # the runtime the library is linked against, already loaded
    v = C.c_int(0)
    assert cudart.cudaDeviceGetAttribute(C.byref(v), 16, 0) == 0        # cudaDevAttrMultiProcessorCount
    return v.value


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference helpers themselves
# ---------------------------------------------------------------------------------------------------------------------
def test_svd_elimination_on_rank_deficient_equality_blocks():
    rng = np.random.default_rng(11)
    for n in (3, 6, 10):
        e = rng.normal(size=(3, n))
        xf = rng.normal(size=n)
        blocks = [np.vstack([e[0], e[0]]),                                  # duplicated
                  np.vstack([e[0], -2.5 * e[0], e[1]]),                     # scaled
                  np.vstack([e[0], e[1], e[0] - 3 * e[1], e[2]]),           # linear combination
                  np.zeros((2, n)),                                         # zero rows (b = 0: no constraint)
                  e[:1]]
        for Ae in blocks:
            be = -Ae @ xf
            x0, Z, ok = eliminate(Ae, be)
            rank = np.linalg.matrix_rank(Ae) if Ae.any() else 0
            assert ok and Z.shape == (n, n - rank)
            assert np.abs(Z.T @ Z - np.eye(n - rank)).max(initial=0) < 1e-13
            assert np.abs(Ae @ Z).max(initial=0) < 1e-12 and np.abs(Ae @ x0 + be).max() < 1e-12
            # every solution of the block is x0 + Z y: xf is one
            y = Z.T @ (xf - x0)
            assert np.abs(x0 + Z @ y - xf).max() < 1e-12
            assert first_inconsistent(Ae, be) == -1
        # an inconsistent dependent row: 2 e0 x + b != 2 (e0 x + b0)
        Ae = np.vstack([e[0], e[1], 2.0 * e[0]])
        be = -Ae @ xf; be[2] += 0.3
        assert not eliminate(Ae, be)[2] and first_inconsistent(Ae, be) == 2
        Ae = np.vstack([e[0], np.zeros(n)]); be = np.array([0.1, -1e-3])        # a zero row with b != 0
        assert first_inconsistent(Ae, be) == 1


def test_ranked_rows_expand_to_the_toeplitz_product():
    """Row r of the expansion is (A0[r], A1[r]) times row samp[r] of the lower-triangular Toeplitz matrix of uz, on both
    axes: checked against scipy's Toeplitz matrix and against the points P_ax = Uz x_ax the ranked kernel scans."""
    from scipy.linalg import toeplitz
    rng = np.random.default_rng(12)
    for N in (1, 3, 16, 75, 80):
        uz = rng.uniform(0.2, 1.0, N) * 0.7 ** np.arange(N)
        Uz = toeplitz(uz, np.zeros(N))
        m = 40
        A0, A1 = rng.normal(size=m), rng.normal(size=m)
        samp = rng.integers(0, N, m); samp[0] = 0; samp[-1] = N - 1
        A = ranked_dense(A0, A1, samp, uz, N)
        assert np.array_equal(A, np.hstack([A0[:, None] * Uz[samp], A1[:, None] * Uz[samp]]))
        x = rng.normal(size=2 * N)
        pts = np.stack([Uz @ x[:N], Uz @ x[N:]])
        assert np.abs(A @ x - (A0 * pts[0, samp] + A1 * pts[1, samp])).max() < 1e-13


def test_reference_solutions_pass_the_long_double_certificate():
    """reference() on QPs with dependent equalities and bounds satisfies KKT in long double; a solution moved by 1e-7 or a
    multiplier of the wrong sign does not; an equality-only QP agrees with the direct solve of its KKT system."""
    rng = np.random.default_rng(13)
    for k in range(30):
        n = int(rng.integers(4, 12)); m = int(rng.integers(3, 15))
        p = make_qp(rng, n, m, me=2, bounds=k % 2 == 0)
        p["A"] = np.vstack([p["A"][:2], 2.0 * p["A"][:1], p["A"][2:]]); p["b"] = np.concatenate([p["b"][:2], 2.0 * p["b"][:1], p["b"][2:]])
        p["me"] = 3
        x, u, st = reference(p)
        assert st == 0
        assert certify(p, x, u) < 1e-12
        r = kkt_ld(p, x + 1e-7, u)
        assert max(r.values()) > 1e-9
        ui = np.nonzero(u[3:] > 1e-6)[0]
        if len(ui):
            bad = u.copy(); bad[3 + ui[0]] = -bad[3 + ui[0]]
            assert max(kkt_ld(p, x, bad).values()) > 1e-9
        if ol.ref() is not None:
            from test_qld_gpu import ref_qld
            xq, _, fq = ref_qld(p["C"], p["d"], p["A"], p["b"], 3, p.get("xl"), p.get("xu"))
            assert fq == 0 and np.abs(xq - x).max() < 1e-8 * max(1, np.abs(x).max())
    # equalities only (full row rank): [C -A'; A 0] [x; u] = [-d; -b]
    n, me = 8, 3
    p = make_qp(rng, n, me, me=me)
    Kk = np.block([[p["C"], -p["A"].T], [p["A"], np.zeros((me, me))]])
    sol = np.linalg.solve(Kk, np.concatenate([-p["d"], -p["b"]]))
    x, u, st = reference(p)
    assert st == 0 and np.abs(x - sol[:n]).max() < 1e-12 and np.abs(u - sol[n:]).max() < 1e-10
    # inconsistent inequalities: 3, inconsistent equalities: 10 + j
    p = {"C": np.eye(2), "d": np.zeros(2), "A": np.array([[1.0, 0.0], [-1.0, 0.0]]), "b": np.array([-1.0, -1.0]), "me": 0}
    assert reference(p)[2] == 3
    assert reference({k: v for k, v in p.items() if k != "_ref"} | {"me": 2})[2] == 12


# ---------------------------------------------------------------------------------------------------------------------
# GPU 1: the ranked entry against the dense entry and the reference
# ---------------------------------------------------------------------------------------------------------------------
RANKED_CASES = [(1, 0, False, 0), (1, 1, True, 0), (1, 6, True, 1), (3, 0, True, 0), (3, 1, False, 0), (3, 12, True, 2),
                (16, 3, True, 0), (16, 7, False, 2), (16, 7, True, 2), (16, 40, True, 2), (75, 1, True, 0), (75, 20, True, 2),
                (75, 37, False, 2), (75, 600, True, 2), (80, 0, True, 0), (80, 39, True, 2), (80, 200, False, 2)]


def ranked_batch(rng, N, mmax, bounds, me, count=5, cond=1e2):
    uz = rng.uniform(0.5, 1.0, N) * 0.6 ** np.arange(N)
    n = 2 * N
    probs, rows = [], []
    for k in range(count):
        m = mmax if k == 0 else int(rng.integers(0, mmax + 1))                # ragged m, one QP at mmax
        mek = min(me, m)
        A0, A1 = rng.normal(size=m), rng.normal(size=m)
        samp = rng.integers(0, N, m).astype(np.uint8)
        if m:
            samp[0] = 0; samp[-1] = N - 1
        A = ranked_dense(A0, A1, samp, uz, N)
        Cm = spd(rng, n, cond)
        xf = rng.normal(size=n) * 0.3
        x0 = xf + rng.normal(size=n)
        b = -A @ xf + rng.uniform(0.0, 0.2, m)
        b[:mek] = -A[:mek] @ xf
        p = {"C": Cm, "d": -Cm @ x0, "A": A, "b": b, "me": mek}
        if bounds:
            p["xl"] = xf - rng.uniform(0.1, 0.8, n); p["xu"] = xf + rng.uniform(0.1, 0.8, n)
        probs.append(p); rows.append((A0, A1, samp))
    rs = max(mmax, 1)
    A0s = np.zeros((count, rs)); A1s = np.zeros((count, rs)); ss = np.zeros((count, rs), dtype=np.uint8)
    for k, (a0, a1, s) in enumerate(rows):
        A0s[k, :len(a0)] = a0; A1s[k, :len(a1)] = a1; ss[k, :len(s)] = s
    return probs, (A0s, A1s, ss, rs, uz, N)


@pytest.mark.gpu
@pytest.mark.parametrize("N,mmax,bounds,me", RANKED_CASES)
def test_gpu_ranked_entry_matches_dense_entry_and_reference(ctx, N, mmax, bounds, me):
    """wg_qld_solve_batch_ranked on rank-structured rows == wg_qld_solve_batch on the materialised matrix (identical
    active sets, x to 1e-10) == the reference; mmax < N / 2 included (the scan's 4N doubles of scratch must not overlap
    the multipliers), samples 0 and N - 1 in every QP, ragged m."""
    rng = np.random.default_rng(1000 * N + mmax + 7 * bounds + me)
    probs, rk = ranked_batch(rng, N, mmax, bounds, me)
    pk = pack(probs, 2 * N, mmax=mmax)
    xr_, ur_, fr_, itr = solve_ok(ctx, pk, ranked=rk, mem=WG_MEM_DEVICE)
    xd_, ud_, fd_, itd = solve_ok(ctx, pk)
    worst = 0.0
    for k, p in enumerate(probs):
        assert fr_[k] == 0 and fd_[k] == 0, (k, fr_[k], fd_[k])
        lay = len(p["b"]) + (4 * N if bounds else 0)
        big = max(np.abs(ud_[k, :lay]).max(initial=0), 1e-12)
        assert active(ur_[k, :lay], big) == active(ud_[k, :lay], big), k
        assert np.abs(xr_[k] - xd_[k]).max() < XTOL * max(1.0, np.abs(xd_[k]).max()), k
        for x, u, what in ((xr_[k], ur_[k], "ranked"), (xd_[k], ud_[k], "dense")):
            worst = max(worst, check_against_reference(p, x, u[:lay], (what, k))[0])
    print(f"N={N} mmax={mmax}: ranked / dense vs reference |dx| <= {worst:.1e}, iterations {itr.tolist()}")


@pytest.mark.gpu
def test_gpu_ranked_entry_refusals(ctx):
    """n != 2N and host memory are refused with WG_ERR_INVALID; nothing is solved."""
    rng = np.random.default_rng(5)
    probs, rk = ranked_batch(rng, 16, 10, False, 0, count=2)
    pk = pack(probs, 32, mmax=10)
    assert solve_raw(ctx, dict(pk, n_call=30, nmax=32), ranked=rk, mem=WG_MEM_DEVICE)[0] == WG_ERR_INVALID
    assert solve_raw(ctx, pk, ranked=rk, mem=WG_MEM_HOST)[0] == WG_ERR_INVALID
    assert solve_raw(ctx, pk, ranked=rk, mem=WG_MEM_DEVICE)[0] == 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU 2: dependent equalities
# ---------------------------------------------------------------------------------------------------------------------
def dependent_eq_qp(rng, kind):
    """Equality rows of which some depend on the earlier ones, then inequalities that cut the unconstrained minimiser."""
    n = int(rng.integers(4, 13))
    e = rng.normal(size=(2, n))
    Ae = {"dup": np.vstack([e[0], e[0]]), "scaled": np.vstack([e[0], -2.0 * e[0]]),
          "comb": np.vstack([e[0], e[1], 0.5 * e[0] - 1.5 * e[1]]), "mixed": np.vstack([e[0], 2.0 * e[0], e[1], e[0] + e[1]])}[kind]
    me = len(Ae)
    mi = int(rng.integers(4, 12))
    xf = rng.normal(size=n)
    Ai = rng.normal(size=(mi, n))
    Cm = np.eye(n) if rng.random() < 0.5 else spd(rng, n, 1e2)
    p = {"C": Cm, "d": rng.normal(size=n) * 3 - Cm @ xf, "A": np.vstack([Ae, Ai]),
         "b": np.concatenate([-Ae @ xf, -Ai @ xf + rng.uniform(0.0, 0.5, mi)]), "me": me}
    return p, me - np.linalg.matrix_rank(Ae)


@pytest.mark.gpu
def test_gpu_dependent_equalities_keep_inequality_rows_droppable(ctx):
    """Consistent equality rows that depend on earlier ones (duplicated, scaled, linear combinations) are skipped; the
    inequality rows added after them must stay droppable, or their multipliers go negative with ifail = 0.  400 QPs; the
    dual steps that drop rows must actually occur in a good share of them."""
    rng = np.random.default_rng(21)
    kinds = ["dup", "scaled", "comb", "mixed"]
    by_n = {}
    for k in range(400):
        p, skipped = dependent_eq_qp(rng, kinds[k % 4])
        by_n.setdefault(len(p["d"]), []).append((p, skipped))
    total = dropped = 0
    worst = 0.0
    for n, group in sorted(by_n.items()):
        probs = [g[0] for g in group]
        x, u, ifail, it = solve_ok(ctx, pack(probs, n))
        for k, (p, skipped) in enumerate(group):
            m, me = len(p["b"]), p["me"]
            assert ifail[k] == 0, (n, k, ifail[k])
            assert (u[k, me:m] >= -1e-9 * max(1.0, np.abs(u[k, :m]).max())).all(), (n, k, u[k, me:m].min())
            worst = max(worst, check_against_reference(p, x[k], u[k, :m], (n, k), sets=False, ineq_u=True)[0])
            total += 1
            dropped += int(it[k] > np.count_nonzero(u[k, :m]) + skipped)
    assert total == 400 and dropped >= 40, (total, dropped)
    print(f"dependent equalities: {total} QPs, {dropped} with dropped rows, |dx| <= {worst:.1e}")


@pytest.mark.gpu
def test_gpu_inconsistent_dependent_equalities_report_the_row(ctx):
    """An equality row that contradicts the earlier rows it depends on: ifail = 10 + j (1-based), like the reference."""
    rng = np.random.default_rng(22)
    probs, want = [], []
    n = 7
    for k in range(24):
        e = rng.normal(size=(2, n)); xf = rng.normal(size=n)
        Ae = [np.vstack([e[0], e[0]]), np.vstack([e[0], e[1], 3.0 * e[0]]), np.vstack([e[0], e[1], e[0] - e[1]])][k % 3]
        be = -Ae @ xf; be[-1] += rng.choice([-1, 1]) * rng.uniform(0.01, 1.0)
        Ai = rng.normal(size=(5, n))
        p = {"C": spd(rng, n), "d": rng.normal(size=n), "A": np.vstack([Ae, Ai]),
             "b": np.concatenate([be, -Ai @ xf + 0.1]), "me": len(Ae)}
        assert reference(p)[2] == 10 + len(Ae)
        probs.append(p); want.append(10 + len(Ae))
    x, u, ifail, it = solve_ok(ctx, pack(probs, n))
    assert ifail.tolist() == want
    for k, p in enumerate(probs):           # on failure x is the unconstrained minimiser
        assert np.abs(x[k] + np.linalg.solve(p["C"], p["d"])).max() < 1e-10 * max(1, np.abs(x[k]).max())


# ---------------------------------------------------------------------------------------------------------------------
# GPU 3: degenerate inequalities and zero rows
# ---------------------------------------------------------------------------------------------------------------------
def degenerate_qp(rng, n, kind):
    Cm = spd(rng, n, 1e2)
    xf = rng.normal(size=n)
    x0 = xf + 3 * rng.normal(size=n)
    A = rng.normal(size=(6, n))
    b = -A @ xf + rng.uniform(0.0, 0.5, 6)
    if kind == "dup":                        # exact duplicates of every row
        A = np.vstack([A, A]); b = np.concatenate([b, b])
    elif kind == "parallel":                 # the same normals with other offsets (some tighter, some looser), interleaved
        A = np.vstack([A, 2.0 * A, A]); b = np.concatenate([b, 2.0 * b + rng.uniform(-0.4, 0.4, 6), b - rng.uniform(0, 0.3, 6)])
    elif kind == "dependent":                # sums of pairs of rows, tightened: met only after the pair is given up
        S = A[:3] + A[3:]
        A = np.vstack([A, S]); b = np.concatenate([b, b[:3] + b[3:] - rng.uniform(0.05, 0.5, 3)])
    return {"C": Cm, "d": -Cm @ x0, "A": A, "b": b, "me": 0}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["dup", "parallel", "dependent"])
def test_gpu_degenerate_inequalities(ctx, kind):
    """Duplicated rows, parallel rows with other offsets, and rows that depend on the active set (the pure dual step):
    x equals the reference's, the KKT certificate holds (the multipliers of dependent rows are not unique)."""
    rng = np.random.default_rng({"dup": 31, "parallel": 32, "dependent": 33}[kind])
    n = 9
    probs = [degenerate_qp(rng, n, kind) for _ in range(60)]
    x, u, ifail, it = solve_ok(ctx, pack(probs, n))
    worst = 0.0
    for k, p in enumerate(probs):
        assert ifail[k] == 0, (k, ifail[k])
        worst = max(worst, check_against_reference(p, x[k], u[k, :len(p["b"])], k, sets=False)[0])
    print(f"{kind}: |dx| <= {worst:.1e}, iterations mean {it.mean():.1f} max {it.max()}")


@pytest.mark.gpu
def test_gpu_zero_rows(ctx):
    """A row of zeros with b >= 0 is no constraint (u = 0, x as without it); with b < 0 it cannot be met: ifail = 10 + j,
    as the header states.  An equality row of zeros is redundant with b = 0 and inconsistent (10 + j) with b != 0."""
    rng = np.random.default_rng(41)
    n = 8
    base = [make_qp(rng, n, 10, me=1) for _ in range(6)]
    probs, want = [], []
    for k, p in enumerate(base):
        for j, bz, me_z in ((4, 0.0, False), (4, 0.5, False), (7, -0.25, False), (0, 0.0, True), (0, 0.4, True), (9, -1e-3, False)):
            q = dict(p)
            A = p["A"].copy(); b = p["b"].copy()
            A = np.insert(A, j, 0.0, axis=0); b = np.insert(b, j, bz)
            q["A"], q["b"] = A, b
            q["me"] = p["me"] + (1 if me_z else 0)
            if me_z:
                assert j < q["me"]
            bad = (bz < 0) or (me_z and bz != 0)
            assert (reference(q)[2] != 0) == bad
            probs.append(q); want.append(10 + j + 1 if bad else 0)
    x, u, ifail, it = solve_ok(ctx, pack(probs, n))
    assert ifail.tolist() == want, [(k, int(ifail[k]), w) for k, w in enumerate(want) if ifail[k] != w]
    for k, q in enumerate(probs):
        if want[k] == 0:
            m = len(q["b"])
            check_against_reference(q, x[k], u[k, :m], k, sets=False)
            zr = np.nonzero(~q["A"].any(axis=1))[0]
            assert (u[k, zr] == 0).all()
    if ol.ref() is not None:                 # the reference's ql0001_ on the same zero rows
        from test_qld_gpu import ref_qld
        for k, q in enumerate(probs[:6]):
            fq = ref_qld(q["C"], q["d"], q["A"], q["b"], q["me"])[2]
            assert (fq > 10) == (want[k] > 10), (k, fq, want[k])


# ---------------------------------------------------------------------------------------------------------------------
# GPU 4: dimension limits
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_one_variable(ctx):
    rng = np.random.default_rng(51)
    probs = []
    for k in range(8):
        p = make_qp(rng, 1, int(rng.integers(0, 5)), bounds=k % 2 == 1)
        probs.append(p)
    mmax = max(len(p["b"]) for p in probs)
    for bounds in (False, True):
        grp = [p for p in probs if (p.get("xl") is not None) == bounds]
        x, u, ifail, it = solve_ok(ctx, pack(grp, 1, mmax=mmax))
        for k, p in enumerate(grp):
            m = len(p["b"])
            lay = u[k, :m + 2] if bounds else u[k, :m]
            assert ifail[k] == 0
            check_against_reference(p, x[k], lay, k)


@pytest.mark.gpu
def test_gpu_largest_problem_n160_m1024(ctx):
    """n = WG_QLD_MAX_N, m = WG_QLD_MAX_M, with bounds and equalities, per-QP and shared Hessians."""
    rng = np.random.default_rng(52)
    n, m = QLD_MAX_N, QLD_MAX_M
    Cm = spd(rng, n, 1e2)
    probs = [make_qp(rng, n, m, me=3, bounds=True, Cm=Cm, spread=1.0) for _ in range(2)]
    per_qp = solve_ok(ctx, pack(probs, n))
    ctx.qld_set_shared_hessian(Cm)
    shared = solve_ok(ctx, pack(probs, n), shared=True)
    for k, p in enumerate(probs):
        for x, u, ifail, it in (per_qp, shared):
            assert ifail[k] == 0
            ex, kk = check_against_reference(p, x[k], u[k], k)
        print(f"n=160 m=1024: active rows {len(active(per_qp[1][k]))}, iterations {per_qp[3][k]}, |dx| {ex:.1e}")


@pytest.mark.gpu
def test_gpu_vertex_solutions_fill_every_slot(ctx):
    """Optima with exactly n active rows (a vertex: the active set reaches its capacity n), with n active bounds and m = 0,
    and with n + 1 rows through the same point (degenerate: any n of them carry the optimum)."""
    rng = np.random.default_rng(53)
    n = 10
    vertex, box, over = [], [], []
    for k in range(8):
        Cm = spd(rng, n)
        xs = rng.normal(size=n)
        A = rng.normal(size=(n, n)); lam = rng.uniform(0.5, 2.0, n)
        vertex.append({"C": Cm, "d": -Cm @ xs + A.T @ lam, "A": A, "b": -A @ xs, "me": 0})
        lo = rng.random(n) < 0.5
        xl = xs - np.where(lo, 0.0, 1.0); xu = xs + np.where(lo, 1.0, 0.0)        # x* on a corner of the box
        mu = rng.uniform(0.5, 2.0, n)
        box.append({"C": Cm, "d": -Cm @ xs + np.where(lo, mu, -mu), "A": np.zeros((0, n)), "b": np.zeros(0), "me": 0, "xl": xl, "xu": xu})
        A1 = rng.normal(size=(n + 1, n)); lam1 = rng.uniform(0.5, 2.0, n + 1)
        over.append({"C": Cm, "d": -Cm @ xs + A1.T @ lam1, "A": A1, "b": -A1 @ xs, "me": 0, "xs": xs})
    x, u, ifail, it = solve_ok(ctx, pack(vertex, n))
    for k, p in enumerate(vertex):
        assert ifail[k] == 0 and len(active(u[k])) == n
        check_against_reference(p, x[k], u[k], ("vertex", k))
    x, u, ifail, it = solve_ok(ctx, pack(box, n, mmax=0))
    for k, p in enumerate(box):
        assert ifail[k] == 0 and len(active(u[k])) == n
        check_against_reference(p, x[k], u[k], ("box", k))
    x, u, ifail, it = solve_ok(ctx, pack(over, n))
    for k, p in enumerate(over):
        assert ifail[k] == 0, ("n + 1 rows", k, ifail[k])
        assert np.abs(x[k] - p["xs"]).max() < XTOL * max(1, np.abs(p["xs"]).max())
        assert len(active(u[k])) <= n
        certify(p, x[k], u[k], what=("n + 1 rows", k))


@pytest.mark.gpu
def test_gpu_n_plus_one_inconsistent_rows(ctx):
    """n + 1 rows with an empty intersection (x_i >= 0 for all i and sum x <= -1): ifail > 10, x the unconstrained minimiser."""
    rng = np.random.default_rng(54)
    n = 6
    probs = []
    for k in range(6):
        A = np.vstack([np.eye(n), -np.ones((1, n))])
        perm = rng.permutation(n + 1)
        p = {"C": spd(rng, n), "d": rng.normal(size=n), "A": A[perm], "b": np.concatenate([np.zeros(n), [-1.0]])[perm], "me": 0}
        assert reference(p)[2] == 3
        probs.append(p)
    x, u, ifail, it = solve_ok(ctx, pack(probs, n))
    assert (ifail > 10).all() and (ifail <= 10 + n + 1).all(), ifail
    for k, p in enumerate(probs):
        assert np.abs(x[k] + np.linalg.solve(p["C"], p["d"])).max() < 1e-10 * max(1, np.abs(x[k]).max())


# ---------------------------------------------------------------------------------------------------------------------
# GPU 5: layouts and memory, bitwise against the plain host call
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_layouts_and_memory_are_bitwise_the_plain_call(ctx):
    """nmax = n + 3, padded a_stride / b_stride / u_stride (padding NaN: it must not be read), u = NULL, iterations = NULL,
    me = NULL against all-zero me, and WG_MEM_DEVICE: every x, u, ifail and iteration count bitwise equal to the plain host
    call with exact strides."""
    rng = np.random.default_rng(61)
    n = 14
    probs = [make_qp(rng, n, int(rng.integers(5, 30)), me=int(rng.integers(0, 3)), bounds=True) for _ in range(12)]
    mmax = 32
    plain = solve_ok(ctx, pack(probs, n, mmax=mmax))
    for k, p in enumerate(probs):
        assert plain[2][k] == 0
        m = len(p["b"])
        check_against_reference(p, plain[0][k], plain[1][k, :m + 2 * n], k)
    lay = lambda out, us: (out[0], out[1][:, :us], out[2], out[3])
    us = mmax + 2 * n

    def same(a, b, what):
        for i, name in enumerate(("x", "u", "ifail", "iterations")):
            assert np.array_equal(a[i], b[i]), (what, name)

    padded = pack(probs, n, nmax=n + 3, mmax=mmax, a_pad=5, b_pad=3, u_pad=4, fill=np.nan)
    same(lay(solve_ok(ctx, padded), us), plain, "padded")
    same(solve_ok(ctx, pack(probs, n, mmax=mmax), mem=WG_MEM_DEVICE), plain, "device")
    same(lay(solve_ok(ctx, padded, mem=WG_MEM_DEVICE), us), plain, "padded device")
    x, u, ifail, it = solve_ok(ctx, pack(probs, n, mmax=mmax), no_u=True, no_it=True)
    assert np.array_equal(x, plain[0]) and np.array_equal(ifail, plain[2])
    assert (u == 7.0).all() and (it == -99).all()                              # nothing written where NULL was passed
    noeq = [dict(p, me=0) for p in probs]
    z = solve_ok(ctx, pack(noeq, n, mmax=mmax))
    same(solve_ok(ctx, pack(noeq, n, mmax=mmax), no_me=True), z, "me = NULL")
    same(solve_ok(ctx, pack(noeq, n, mmax=mmax), no_me=True, mem=WG_MEM_DEVICE), z, "me = NULL, device")


# ---------------------------------------------------------------------------------------------------------------------
# GPU 6: the persistent grid
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_persistent_grid_every_qp_as_if_alone(ctx):
    """B = 2 SMs 3 + 5 QPs (each CTA of the persistent grid solves several), good ones mixed with every failure code: 2
    (indefinite per-QP C, eps = 0), 5 (m > mmax, me > m), > 10 (inconsistent rows).  Each result is bitwise that of the same
    QP solved alone with B = 1: a failure does not disturb its neighbours, nor does the scratch a CTA reuses."""
    rng = np.random.default_rng(71)
    n, mmax = 12, 24
    B = 2 * sm_count() * 3 + 5
    probs, want = [], []
    for k in range(B):
        p = make_qp(rng, n, int(rng.integers(0, mmax + 1)), me=int(rng.integers(0, 3)), bounds=True)
        p["me"] = min(p["me"], len(p["b"]))
        kind = k % 7
        if kind == 1:                                         # indefinite Hessian
            p["C"] = p["C"].copy(); p["C"][3, 3] = -1.0
            want.append(2)
        elif kind == 3:                                       # m > mmax
            p["m"] = mmax + 1; want.append(5)
        elif kind == 5 and len(p["b"]) >= 2:                  # me > m
            p["m"] = len(p["b"]); p["me"] = len(p["b"]) + 1; want.append(5)
        elif kind == 6 and len(p["b"]) >= 2:                  # a row that contradicts the last: x_0 <= xl_0 - 1
            p["A"] = p["A"].copy(); p["b"] = p["b"].copy()
            p["A"][-1] = 0; p["A"][-1, 0] = -1.0; p["b"][-1] = p["xl"][0] - 1.0
            want.append(-1)
        else:
            want.append(0)
        probs.append(p)
    pk = pack(probs, n, mmax=mmax)
    x, u, ifail, it = solve_ok(ctx, pk)
    for k, p in enumerate(probs):
        one = solve_ok(ctx, pack([p], n, mmax=mmax))
        assert np.array_equal(one[0][0], x[k]) and np.array_equal(one[1][0], u[k]), k
        assert one[2][0] == ifail[k] and one[3][0] == it[k], k
        if want[k] == -1:
            assert ifail[k] > 10, (k, ifail[k])
        else:
            assert ifail[k] == want[k], (k, ifail[k], want[k])
        if want[k] == 0 and k % 23 == 0:
            m = len(p["b"])
            check_against_reference(p, x[k], u[k, :m + 2 * n], k)
    print(f"persistent grid: B={B}, ifail counts {np.unique(ifail, return_counts=True)}")


# ---------------------------------------------------------------------------------------------------------------------
# GPU 7: a caller's shared Hessian next to the Wieber generator's
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [150, 40])
def test_gpu_wieber_run_keeps_the_callers_shared_hessian(ctx, n):
    """A caller installs its shared Hessian, runs a short Wieber batch, and solves with shared_hessian = 1: the answer is
    the one for the caller's Hessian (n = 150 is the generator's own size, n = 40 another), and the generator's output
    does not depend on the caller's Hessian."""
    import zmpdisc_oracle as zo
    from test_wieber import walk_steps
    rng = np.random.default_rng(80 + n)
    Cm = spd(rng, n, 1e2)
    probs = [make_qp(rng, n, 30, Cm=Cm) for _ in range(4)]
    walks = [walk_steps(2, 0.1)]
    feet = np.array([zo.INIT_FEET], dtype=np.float64).reshape(1, -1)
    ctx.wieber_set_params()
    w0 = ctx.wieber_run(walks, feet)
    ctx.qld_set_shared_hessian(Cm)
    before = solve_ok(ctx, pack(probs, n), shared=True)
    w1 = ctx.wieber_run(walks, feet)
    after = solve_ok(ctx, pack(probs, n), shared=True)
    for i in range(4):
        assert np.array_equal(before[i], after[i])
    for k, p in enumerate(probs):
        assert after[2][k] == 0
        check_against_reference(p, after[0][k], after[1][k], k)
    assert (w0["status"] == 0).all() and int(w0["periods_done"][0]) > 0
    assert np.array_equal(w0["com"], w1["com"]) and np.array_equal(w0["zmp"], w1["zmp"])
