"""ctypes access to the Wieber2006 restatement (oracle/oracle_wieber.cpp) and to the reference's OWN ZMPQPWithConstraint
object code (oracle/_ref, glue oracle/ref_glue_wieber.cc).  TEST INFRASTRUCTURE ONLY."""
import ctypes as C

import numpy as np

import dimitrov_oracle as do
import oracle_lib as ol

D = ol.D
IP = C.POINTER(C.c_int)
N_DEFAULT, T_DEFAULT = 75, 0.02          # m_QP_N, m_QP_T (ZMPQPWithConstraint.cpp:71-72)
_bound = False


def _ora():
    global _bound
    o = ol.oracle()
    if not _bound:
        o.oracle_wieber_run.restype = C.c_long
        o.oracle_wieber_run.argtypes = [C.c_long, D, D, IP, D, D, D, C.c_double, C.c_double, C.c_double, C.c_double,
                                        C.c_double, C.c_int, C.c_double, C.c_long, IP]
        o.oracle_wieber_constants.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double, D, D, D]
        o.oracle_wieber_set_qld.argtypes = [C.c_void_p]
        r = ol.ref()
        if r is not None:
            o.oracle_wieber_set_qld(C.cast(r.ref_ql0001, C.c_void_p))   # the reference's own ql0001_
        _bound = True
    return o


def inputs(walk):
    """walk: output of zmpdisc_oracle.run -> (left4, right4, left step types, clock, zmp3)."""
    L = do._feet4(walk["left"]); R = do._feet4(walk["right"])
    st = np.ascontiguousarray(walk["types"][:, 1], dtype=np.int32)
    t = do.clock(len(L))
    z = np.ascontiguousarray(walk["zmp"][:, :3], dtype=np.float64)
    return L, R, st, t, z


def constants(N=N_DEFAULT, T=T_DEFAULT, alpha=200.0, beta=1000.0):
    n = 2 * N
    Cm = np.zeros((n, n)); OptB = np.zeros((n, 6)); OptC = np.zeros((n, n))
    _ora().oracle_wieber_constants(N, T, alpha, beta, ol.dptr(Cm), ol.dptr(OptB), ol.dptr(OptC))
    return Cm, OptB, OptC


def run(walk, cx=0.04, cy=0.04, T=T_DEFAULT, N=N_DEFAULT, sole=(0.25, 0.14), max_periods=0):
    """-> (periods or -(1 + failing period), com [n][7], zmp [n][3], info [periods][3] = m, ifail, active rows)."""
    L, R, st, t, z = inputs(walk)
    n = len(L)
    com = np.zeros((n, 7)); zz = z.copy()
    info = np.zeros((n, 3), dtype=np.int32)
    k = _ora().oracle_wieber_run(n, ol.dptr(L), ol.dptr(R), st.ctypes.data_as(IP), ol.dptr(t), ol.dptr(zz), ol.dptr(com),
                                 sole[0], sole[1], cx, cy, T, N, 0.005, max_periods, info.ctypes.data_as(IP))
    return k, com, zz, info[:max(k, 0)]


class RefWieber:
    def __init__(self, sole=(0.25, 0.14)):
        self.r = ol.ref()
        self.r.ref_wieber_new.restype = C.c_void_p
        self.r.ref_wieber_new.argtypes = [C.c_double, C.c_double]
        self.r.ref_wieber_delete.argtypes = [C.c_void_p]
        self.r.ref_wieber_run.restype = C.c_int
        self.r.ref_wieber_run.argtypes = [C.c_void_p, C.c_long, D, D, IP, D, D, D, C.c_double, C.c_double, C.c_double, C.c_uint]
        self.r.ref_wieber_polygons.restype = C.c_int
        self.r.ref_wieber_polygons.argtypes = [C.c_void_p, C.c_long, D, D, IP, D, C.c_double, C.c_double, C.c_int, C.c_int, D, D, IP]
        self.h = self.r.ref_wieber_new(*sole)

    def close(self):
        self.r.ref_wieber_delete(self.h)

    def run(self, walk, cx=0.04, cy=0.04, T=T_DEFAULT, N=N_DEFAULT):
        L, R, st, t, z = inputs(walk)
        n = len(L)
        com = np.zeros((n, 7)); zz = z.copy()
        rc = self.r.ref_wieber_run(self.h, n, ol.dptr(L), ol.dptr(R), st.ctypes.data_as(IP), ol.dptr(t), ol.dptr(zz), ol.dptr(com),
                                   cx, cy, T, N)
        return rc, com, zz

    def polygons(self, walk, cx=0.04, cy=0.04, cap=512):
        L, R, st, t, z = inputs(walk)
        rows = np.zeros((cap, 8, 3)); times = np.zeros((cap, 2)); nr = np.zeros(cap, dtype=np.int32)
        n = self.r.ref_wieber_polygons(self.h, len(L), ol.dptr(L), ol.dptr(R), st.ctypes.data_as(IP), ol.dptr(t), cx, cy, cap, 8,
                                       ol.dptr(rows), ol.dptr(times), nr.ctypes.data_as(IP))
        return rows[:n], times[:n], nr[:n]


class OracleWieber:
    """Stand-in for RefWieber.run where oracle/_ref is not built: the restatement oracle/oracle_wieber.cpp (bitwise the
    reference object when both use the reference's ql0001_) with its QP solved in extended precision on the Hessian plus
    QLD's diagonal boost (wg_qld_diagonal_boost, QLD's rule restated).  That chain reproduces the reference object's
    trajectory to 1e-7 m (CoM) / 1e-8 m (ZMP): test_reference_qld_regularises_the_hessian_and_the_rule_is_restated."""

    def __init__(self):
        from jrl_walkgen_b200 import _capi
        Cf = np.asfortranarray(constants()[0])
        self.boost = _capi.load().wg_qld_diagonal_boost(2 * N_DEFAULT, 2 * N_DEFAULT, Cf.ctypes.data, 1e-8)

    def close(self):
        pass

    def run(self, walk):
        o = _ora()
        o.oracle_wieber_set_boost.argtypes = [C.c_double]
        o.oracle_wieber_set_solver(2); o.oracle_wieber_set_boost(self.boost)
        try:
            k, com, zz, _ = run(walk)
        finally:
            o.oracle_wieber_set_solver(0); o.oracle_wieber_set_boost(0.0)
        return (0 if k > 0 else -1), com, zz

