"""jrl_walkgen_b200 - B200-native batched backend for jrl-walkgen's ZMP pattern-generation hot path.

The product is ``libwalkgen_b200.so`` (hand-written CUDA for sm_100a behind the C ABI in
``include/walkgen_b200.h``) plus the C++ class mirror in ``jrl_walkgen_b200/host/``.  This Python
package is a thin numpy-facing driver over the C ABI used by ``tests/`` and ``bench.py``; it holds
no algorithmic code and has no CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi
from ._capi import (MODE_WITH_INITIALPOS, MODE_WITHOUT_INITIALPOS, WG_MEM_DEVICE, WG_MEM_HOST,
                    HerdtMpcParams, HerdtParams, PreviewGains, WalkgenError)

QP_INPUT_DTYPE, QP_OUTPUT_DTYPE = _capi.herdt_dtypes()
FOOT_DTYPE, TICK_DTYPE, MPC_STATE_DTYPE, MPC_STEP_DTYPE = _capi.herdt_mpc_dtypes()
TICKS_PER_STEP = _capi.HERDT_TICKS_PER_STEP
ACTIVE_SET_DTYPE = _capi.herdt_active_set_dtype()
PLDP_STATE_DTYPE, PLDP_INFO_DTYPE = _capi.pldp_dtypes()
REL_STEP_DTYPE, KAJITA_FOOT_DTYPE = _capi.kajita_dtypes()
KAJITA_STREAM_WALK_DTYPE = _capi.kajita_stream_walk_dtype()
KAJITA_TICK_DTYPE, KAJITA_COMMAND_DTYPE = _capi.kajita_online_dtypes()
KAJITA_ONLINE_WALK_DTYPE = _capi.kajita_online_walk_dtype()
KAJITA_PUSH, KAJITA_STANDARD, KAJITA_STOP = _capi.WG_KAJITA_PUSH, _capi.WG_KAJITA_STANDARD, _capi.WG_KAJITA_STOP
KAJITA_ONLINE_CHUNK = _capi.KAJITA_ONLINE_CHUNK
LCI_DTYPE, DIMITROV_PERIOD_DTYPE = _capi.dimitrov_dtypes()
HERDT_COMMAND_DTYPE = _capi.herdt_command_dtype()
CMD_VEL, CMD_STOP = _capi.WG_CMD_VEL, _capi.WG_CMD_STOP
HERDT_ONLINE_QUEUE = _capi.HERDT_ONLINE_QUEUE
ONLINE_ROBOT_DTYPE = _capi.herdt_online_robot_dtype()
HERDT_PLAN_DTYPE = _capi.herdt_plan_dtype()
# init15 of the TestHerdt2010 start at rest: CoM (x, dx, ddx, y, dy, ddy, z), trunk yaw and rate, left and right foot (x, y, theta)
HERDT_INIT15 = (0.0316055, 0.0, 0.0, 0.0, 0.0, 0.0, 0.7116911, 0.0, 0.0, 0.0, 0.09, 0.0, 0.0, -0.09, 0.0)
DimitrovParams = _capi.DimitrovParams

__all__ = ["MultiContext", "LCI_DTYPE", "DIMITROV_PERIOD_DTYPE", "DimitrovParams", "dimitrov_default_params", "Context", "PreviewPlan", "KajitaPlan", "KajitaStream", "HerdtOnline",
           "KajitaOnline", "KAJITA_ONLINE_WALK_DTYPE", "KAJITA_TICK_DTYPE", "KAJITA_COMMAND_DTYPE", "KAJITA_PUSH", "KAJITA_STANDARD", "KAJITA_STOP",
           "KAJITA_ONLINE_CHUNK",
           "HERDT_COMMAND_DTYPE", "CMD_VEL", "CMD_STOP", "HERDT_ONLINE_QUEUE", "ONLINE_ROBOT_DTYPE", "HERDT_PLAN_DTYPE", "HERDT_INIT15",
           "STREAM_START", "STREAM_FINISH", "zmpdisc_default_params", "REL_STEP_DTYPE", "KAJITA_FOOT_DTYPE", "KAJITA_STREAM_WALK_DTYPE", "preview_gains", "herdt_default_params", "herdt_mpc_default_params", "HerdtParams", "HerdtMpcParams",
           "PLDP_STATE_DTYPE", "PLDP_INFO_DTYPE", "FOOT_DTYPE", "TICK_DTYPE", "MPC_STATE_DTYPE", "MPC_STEP_DTYPE", "TICKS_PER_STEP", "QP_INPUT_DTYPE",
           "QP_OUTPUT_DTYPE", "ACTIVE_SET_DTYPE", "WalkgenError", "device_count",
           "MODE_WITH_INITIALPOS", "MODE_WITHOUT_INITIALPOS", "WG_MEM_HOST", "WG_MEM_DEVICE"]


def device_count() -> int:
    return _capi.load().wg_device_count()


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, DeviceBuffer):
        return C.c_void_p(a.ptr)
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def _indices(idx):
    return None if idx is None else np.ascontiguousarray(idx, dtype=np.int32).reshape(-1)


def _copy_indices(src_idx, dst_idx, B):
    """(n, src, dst) of a whole-record copy: n is the length of the index arrays given, B when neither is."""
    si, di = _indices(src_idx), _indices(dst_idx)
    n = len(di) if di is not None else (len(si) if si is not None else B)
    assert si is None or len(si) == n
    return n, si, di


def herdt_default_params(sole_length=0.25, sole_width=0.14) -> HerdtParams:
    """Constants of ZMPVelocityReferencedQP's ctor (ZMPVelocityReferencedQP.cpp:61-118) for a given sole size
    (the reference reads it from the robot model; 0.25 x 0.14 m is the sample robot's, fitted from the datref)."""
    p = HerdtParams()
    _capi.load().wg_herdt_default_params(sole_length, sole_width, C.byref(p))
    return p


def herdt_mpc_default_params() -> HerdtMpcParams:
    """Constants of ZMPVelocityReferencedQP's ctor and the TestHerdt2010 script (step timing 0.7/0.1 s)."""
    p = HerdtMpcParams()
    _capi.load().wg_herdt_mpc_default_params(C.byref(p))
    return p


def dimitrov_default_params() -> "_capi.DimitrovParams":
    """The constants of ZMPConstrainedQPFastFormulation's ctor (ZMPConstrainedQPFastFormulation.cpp:79-96)."""
    p = _capi.DimitrovParams()
    _capi.load().wg_dimitrov_default_params(C.byref(p))
    return p


def zmpdisc_default_params() -> "_capi.ZmpDiscParams":
    """The ZMPDiscretization / FootTrajectoryGenerationStandard parameters tests/CommonTools.cpp:56-69 sets."""
    p = _capi.ZmpDiscParams()
    _capi.load().wg_zmpdisc_default_params(C.byref(p))
    return p


PREVIEW_SUM_AUTO, PREVIEW_SUM_DIRECT, PREVIEW_SUM_RECURSIVE = 0, 1, 2   # wg_preview_set_sum_mode


def preview_gains(T=0.005, preview_time=1.6, zc=0.814, mode=MODE_WITHOUT_INITIALPOS) -> PreviewGains:
    """Host Riccati solve: PreviewControl::ComputeOptimalWeights (PreviewControl.cpp:198-322)."""
    g = PreviewGains()
    rc = _capi.load().wg_preview_gains(T, preview_time, zc, mode, C.byref(g))
    if rc != 0:
        raise WalkgenError(rc, "wg_preview_gains")
    return g


class DeviceBuffer:
    """A device allocation owned by a Context (plain pointer + size)."""

    def __init__(self, ctx, nbytes):
        self.ctx = ctx
        self.nbytes = int(nbytes)
        p = C.c_void_p()
        ctx._check(ctx.lib.wg_malloc_device(ctx.h, self.nbytes, C.byref(p)))
        self.ptr = p.value

    def upload(self, arr):
        arr = np.ascontiguousarray(arr)
        assert arr.nbytes <= self.nbytes
        self.ctx._check(self.ctx.lib.wg_memcpy_h2d(self.ctx.h, self.ptr, arr.ctypes.data, arr.nbytes))
        self.ctx.sync()
        return self

    def download(self, dtype, shape):
        out = np.empty(shape, dtype=dtype)
        assert out.nbytes <= self.nbytes
        self.ctx._check(self.ctx.lib.wg_memcpy_d2h(self.ctx.h, out.ctypes.data, self.ptr, out.nbytes))
        self.ctx.sync()
        return out

    def free(self):
        if self.ptr:
            self.ctx.lib.wg_free_device(self.ctx.h, self.ptr)
            self.ptr = None


class Context:
    """One per GPU (wg_ctx).  Raises WalkgenError(WG_ERR_NO_DEVICE) when there is no GPU."""

    def __init__(self, device=0):
        self.lib = _capi.load()
        h = C.c_void_p()
        rc = self.lib.wg_ctx_create(device, C.byref(h))
        if rc != 0:
            raise WalkgenError(rc, "wg_ctx_create: no usable CUDA device (there is no CPU fallback)")
        self.h = h
        self.device = device

    def _check(self, rc):
        if rc != 0:
            raise WalkgenError(rc, self.lib.wg_last_error(self.h).decode())

    def close(self):
        if self.h:
            self.lib.wg_ctx_destroy(self.h)
            self.h = None

    def sync(self):
        self._check(self.lib.wg_sync(self.h))

    def alloc(self, nbytes) -> DeviceBuffer:
        return DeviceBuffer(self, nbytes)

    def to_device(self, arr) -> DeviceBuffer:
        arr = np.ascontiguousarray(arr)
        return DeviceBuffer(self, max(arr.nbytes, 8)).upload(arr)

    def pinned(self, shape, dtype=np.float64):
        """numpy view on pinned host memory (kept alive by the returned array's base)."""
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        self._check(self.lib.wg_malloc_pinned(self.h, max(n, 8), C.byref(p)))
        buf = (C.c_char * max(n, 8)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
        return arr

    def timer_start(self):
        self._check(self.lib.wg_timer_start(self.h))

    def timer_stop_ms(self) -> float:
        ms = C.c_float()
        self._check(self.lib.wg_timer_stop_ms(self.h, C.byref(ms)))
        return ms.value

    @property
    def launches(self) -> int:
        return self.lib.wg_launch_count(self.h)

    def reset_launches(self):
        self.lib.wg_launch_count_reset(self.h)

    def prof_begin(self, capacity):
        self._check(self.lib.wg_prof_begin(self.h, int(capacity)))

    def prof_end(self):
        """-> {kernel_id: (launches, total_ms)} for the kernels that ran since prof_begin."""
        self._check(self.lib.wg_prof_end(self.h))
        out = {}
        for kid in range(12):
            n = C.c_longlong(); ms = C.c_double()
            self._check(self.lib.wg_prof_get(self.h, kid, C.byref(n), C.byref(ms)))
            if n.value:
                out[kid] = (n.value, ms.value)
        return out

    def fp64_peak_tflops(self) -> float:
        v = C.c_double()
        self._check(self.lib.wg_measure_fp64_peak(self.h, C.byref(v)))
        return v.value

    # ---- Kajita preview control ---------------------------------------------------------
    def preview_set_gains(self, gains: PreviewGains):
        self._check(self.lib.wg_preview_set_gains(self.h, C.byref(gains)))
        self.gains = gains

    def preview_set_sum_mode(self, mode: int):
        """wg_preview_set_sum_mode: PREVIEW_SUM_AUTO / _DIRECT / _RECURSIVE."""
        self._check(self.lib.wg_preview_set_sum_mode(self.h, int(mode)))

    def preview_set_cta_shape(self, shape: int):
        """wg_preview_set_cta_shape: -1 per launch (default), 0 = 64 x 8, 1 = 128 x 4, 2 = one warp per trajectory, 3 = 256 x 2."""
        self._check(self.lib.wg_preview_set_cta_shape(self.h, int(shape)))

    def preview_sum_info(self):
        """(mode in use, relative residual of the fit F[i] = w' L^i v) - wg_preview_sum_info."""
        m, r = C.c_int(0), C.c_double(0.0)
        self._check(self.lib.wg_preview_sum_info(self.h, C.byref(m), C.byref(r)))
        return m.value, r.value

    def preview_plan(self, offsets) -> "PreviewPlan":
        return PreviewPlan(self, offsets)

    def kajita_plan(self, step_offsets, steps, init_feet, params=None) -> "KajitaPlan":
        """The step stacks of B walks, resident on the GPU (wg_kajita_plan_create)."""
        return KajitaPlan(self, step_offsets, steps, init_feet, params)

    def kajita_stream(self, B, params=None, with_preview=True) -> "KajitaStream":
        """B walks whose footsteps arrive while they run (wg_kajita_stream_create)."""
        return KajitaStream(self, B, params, with_preview)

    def kajita_online(self, B, params=None, com_height=0.814, max_step_time=0.8) -> "KajitaOnline":
        """B walks driven one 5 ms control tick at a time, each refilling its queues from its own step stack
        (wg_kajita_online_create); needs preview gains on the context."""
        return KajitaOnline(self, B, params, com_height, max_step_time)

    def preview_one_iteration(self, x, y, sx, sy, window_xy, simulation=True):
        """PreviewControl::OneIterationOfPreview for one instance (host buffers)."""
        x = np.array(x, dtype=np.float64)
        y = np.array(y, dtype=np.float64)
        w = np.ascontiguousarray(window_xy, dtype=np.float64)
        csx, csy, zx, zy = C.c_double(sx), C.c_double(sy), C.c_double(), C.c_double()
        D = _capi.c_double_p
        rc = self.lib.wg_preview_one_iteration(self.h, x.ctypes.data_as(D), y.ctypes.data_as(D), C.byref(csx),
                                               C.byref(csy), w.ctypes.data_as(D), w.shape[0], C.byref(zx),
                                               C.byref(zy), int(simulation))
        self._check(rc)
        return x, y, csx.value, csy.value, zx.value, zy.value


    # ---- Herdt2010 velocity-referenced QP ----------------------------------------------------
    def herdt_set_params(self, params: HerdtParams = None):
        self.herdt_params = params or herdt_default_params()
        self._check(self.lib.wg_herdt_set_params(self.h, C.byref(self.herdt_params)))

    def herdt_qp_solve(self, inputs, outputs=None, mem=WG_MEM_HOST, count=None):
        """wg_herdt_qp_solve_batch.  Host mode: numpy arrays of QP_INPUT_DTYPE -> QP_OUTPUT_DTYPE."""
        if mem == WG_MEM_HOST:
            inputs = np.ascontiguousarray(inputs, dtype=QP_INPUT_DTYPE)
            B = len(inputs)
            if outputs is None:
                outputs = np.zeros(B, dtype=QP_OUTPUT_DTYPE)
            self._check(self.lib.wg_herdt_qp_solve_batch(self.h, mem, B, inputs.ctypes.data, outputs.ctypes.data))
            return outputs
        self._check(self.lib.wg_herdt_qp_solve_batch(self.h, mem, int(count), _ptr(inputs), _ptr(outputs)))
        return outputs

    def preview_gains_batch(self, params, mode=MODE_WITHOUT_INITIALPOS, f_stride=None):
        """wg_preview_gains_batch on host arrays: params [B][3] = (T, preview_time, zc) -> (heads, F [B][f_stride])."""
        params = np.ascontiguousarray(params, dtype=np.float64)
        B = len(params)
        if f_stride is None:
            f_stride = int(np.max(np.floor(params[:, 1] / params[:, 0]))) + 1 if B else 1
        heads = np.zeros(B, dtype=_capi.preview_gains_head_dtype())
        F = np.zeros((B, f_stride))
        self._check(self.lib.wg_preview_gains_batch(self.h, WG_MEM_HOST, B, params.ctypes.data, int(mode), heads.ctypes.data,
                                                    F.ctypes.data, int(f_stride)))
        return heads, F

    # ---- general dense QP (ql0001_ convention) ---------------------------------------------------
    def qld_set_shared_hessian(self, Cmat, eps=0.0):
        """eps > 0: QLD's diagonal boost rule with vsmall = eps first (returns the multiple of I that was added)."""
        Cmat = np.asfortranarray(Cmat, dtype=np.float64)
        n = Cmat.shape[0]
        self._check(self.lib.wg_qld_set_shared_hessian(self.h, n, n, Cmat.ctypes.data, float(eps)))
        return self.lib.wg_qld_shared_boost(self.h)

    def qld_solve(self, d, A, b, m, C_=None, me=None, xl=None, xu=None, want_u=True, eps=0.0):
        """wg_qld_solve_batch on host arrays.  d [B][n]; A [B][mmax][n] (row r of QP k = A[k, r]; converted here to the
        column-major layout of ql0001_); b [B][mmax]; m [B]; C_ [B][n][n] symmetric, or None for the shared Hessian.
        Returns x [B][n], u [B][mmax (+ 2n)], ifail [B], iterations [B]."""
        d = np.ascontiguousarray(d, dtype=np.float64)
        B, n = d.shape
        A = np.asarray(A, dtype=np.float64)
        mmax = A.shape[1]
        Acm = np.ascontiguousarray(np.transpose(A, (0, 2, 1)))          # [B][n][mmax]: element (r, i) at r + i * mmax
        b = np.ascontiguousarray(b, dtype=np.float64)
        m = np.ascontiguousarray(m, dtype=np.int32)
        q = _capi.QldBatch()
        q.n = n; q.nmax = n; q.mmax = mmax
        q.shared_hessian = 1 if C_ is None else 0
        q.eps = float(eps)
        keep = [d, Acm, b, m]
        q.m = m.ctypes.data; q.d = d.ctypes.data; q.A = Acm.ctypes.data; q.a_stride = mmax * n
        q.b = b.ctypes.data; q.b_stride = mmax
        if C_ is not None:
            C_ = np.ascontiguousarray(C_, dtype=np.float64); keep.append(C_)
            q.C = C_.ctypes.data
        if me is not None:
            me = np.ascontiguousarray(me, dtype=np.int32); keep.append(me)
            q.me = me.ctypes.data
        nb = 0
        if xl is not None:
            xl = np.ascontiguousarray(xl, dtype=np.float64); xu = np.ascontiguousarray(xu, dtype=np.float64)
            keep += [xl, xu]
            q.xl = xl.ctypes.data; q.xu = xu.ctypes.data
            nb = 2 * n
        x = np.zeros((B, n)); u = np.zeros((B, mmax + nb)); ifail = np.zeros(B, dtype=np.int32); it = np.zeros(B, dtype=np.int32)
        q.x = x.ctypes.data; q.u = u.ctypes.data if want_u else None; q.u_stride = mmax + nb
        q.ifail = ifail.ctypes.data; q.iterations = it.ctypes.data
        self._check(self.lib.wg_qld_solve_batch(self.h, WG_MEM_HOST, B, C.byref(q)))
        return x, u, ifail, it

    def herdt_qp_solve_warm(self, inputs, guess=None, age=1, outputs=None, active=None):
        """wg_herdt_qp_solve_batch_warm on host arrays -> (outputs, optimal active sets)."""
        inputs = np.ascontiguousarray(inputs, dtype=QP_INPUT_DTYPE)
        B = len(inputs)
        if outputs is None:
            outputs = np.zeros(B, dtype=QP_OUTPUT_DTYPE)
        if active is None:
            active = np.zeros(B, dtype=ACTIVE_SET_DTYPE)
        if guess is not None:
            guess = np.ascontiguousarray(guess, dtype=ACTIVE_SET_DTYPE)
            assert len(guess) == B
        self._check(self.lib.wg_herdt_qp_solve_batch_warm(self.h, WG_MEM_HOST, B, inputs.ctypes.data, outputs.ctypes.data,
                                                          guess.ctypes.data if guess is not None else None, int(age),
                                                          active.ctypes.data))
        return outputs, active


    # ---- Herdt2010 closed loop -----------------------------------------------------------------
    def herdt_mpc_set_params(self, params: HerdtMpcParams = None):
        if not hasattr(self, "herdt_params"):
            self.herdt_set_params()
        self.herdt_mpc_params = params or herdt_mpc_default_params()
        self._check(self.lib.wg_herdt_mpc_set_params(self.h, C.byref(self.herdt_mpc_params)))

    def herdt_mpc_init(self, B, init9=(0.0316055, 0.0, 0.7116911, 0.0, 0.09, 0.0, 0.0, -0.09, 0.0), device=False):
        """InitOnLine for B instances -> host array of MPC_STATE_DTYPE, or a DeviceBuffer when device=True.
        init9: one start configuration (broadcast) or an array [B][9]."""
        init = np.ascontiguousarray(init9, dtype=np.float64)
        stride = 0 if init.ndim == 1 else 9
        assert init.size == 9 or init.shape == (B, 9)
        if device:
            buf = self.alloc(B * MPC_STATE_DTYPE.itemsize)
            self._check(self.lib.wg_herdt_mpc_init(self.h, WG_MEM_DEVICE, B, init.ctypes.data, stride, buf.ptr))
            return buf
        states = np.zeros(B, dtype=MPC_STATE_DTYPE)
        self._check(self.lib.wg_herdt_mpc_init(self.h, WG_MEM_HOST, B, init.ctypes.data, stride, states.ctypes.data))
        return states

    def herdt_mpc_run(self, states, nsteps, vel_ref=None, ticks=False, steps=False, qp_in=False):
        """wg_herdt_mpc_run_batch on host arrays: advances `states` in place; returns (ticks, steps, qp_in)
        arrays for the outputs requested (else None)."""
        assert states.dtype == MPC_STATE_DTYPE and states.flags["C_CONTIGUOUS"]
        B = len(states)
        ref = None if vel_ref is None else np.ascontiguousarray(np.broadcast_to(vel_ref, (B, 3)), dtype=np.float64)
        t = np.zeros((B, nsteps * TICKS_PER_STEP), dtype=TICK_DTYPE) if ticks else None
        s = np.zeros((B, nsteps), dtype=MPC_STEP_DTYPE) if steps else None
        q = np.zeros(B, dtype=QP_INPUT_DTYPE) if qp_in else None
        self._check(self.lib.wg_herdt_mpc_run_batch(self.h, WG_MEM_HOST, B, int(nsteps), states.ctypes.data, _ptr(ref),
                                                    _ptr(t), _ptr(s), _ptr(q)))
        return t, s, q

    def herdt_mpc_run_device(self, d_states, B, nsteps, d_vel_ref=None, d_ticks=None, d_steps=None, d_qp_in=None):
        """Device-resident form (asynchronous on the context stream)."""
        self._check(self.lib.wg_herdt_mpc_run_batch(self.h, WG_MEM_DEVICE, int(B), int(nsteps), _ptr(d_states),
                                                    _ptr(d_vel_ref), _ptr(d_ticks), _ptr(d_steps), _ptr(d_qp_in)))

    def herdt_online(self, B) -> "HerdtOnline":
        """B robots driven one 5 ms control tick at a time (wg_herdt_online_create)."""
        return HerdtOnline(self, B)


    # ---- Dimitrov PLDP / OptCholesky ------------------------------------------------------------
    def pldp_set_constants(self, iPu, Px, Pu):
        """The arrays the PLDPSolver ctor borrows (PLDPSolver.hh:48-52), CardU = 16."""
        iPu, Px, Pu = (np.ascontiguousarray(a, dtype=np.float64) for a in (iPu, Px, Pu))
        D = _capi.c_double_p
        self._check(self.lib.wg_pldp_set_constants(self.h, iPu.shape[0], iPu.ctypes.data_as(D), Px.ctypes.data_as(D),
                                                   Pu.ctypes.data_as(D)))

    def pldp_solve(self, pb, hot=None, hot_start=True, starting=None, n_removed=None, similar=None, max_iterations=0,
                   mem=WG_MEM_HOST, B=None, X=None, info=None, ranked=False, similar_stride=None):
        """wg_pldp_solve_batch.  pb: dict with D [B][32], m [B] int32, DPu [B][dpu_stride], DPx [B][dpx_stride],
        ZMPRef [B][32], XkYk [B][6], dpu_stride, dpx_stride (numpy arrays, or DeviceBuffers with mem=WG_MEM_DEVICE).
        ranked=True: wg_pldp_solve_batch_ranked on pb["a0"], pb["a1"] [B][row_stride] float64 and pb["ri"] [B][row_stride]
        uint8 (pb["row_stride"]) instead of DPu.  Returns (X, info)."""
        if mem == WG_MEM_HOST:
            B = len(pb["m"])
            X = np.zeros((B, 32)) if X is None else X
            info = np.zeros(B, dtype=PLDP_INFO_DTYPE) if info is None else info
        names = ("D", "m", "DPu", "DPx", "ZMPRef", "XkYk")
        keep = [None if (ranked and k == "DPu") else (np.ascontiguousarray(pb[k]) if mem == WG_MEM_HOST else pb[k]) for k in names]
        rk = None
        if ranked:
            rk = [np.ascontiguousarray(pb[k]) if mem == WG_MEM_HOST else pb[k] for k in ("a0", "a1", "ri")]
        opt = [None if a is None else (np.ascontiguousarray(a, dtype=np.int32) if mem == WG_MEM_HOST else a)
               for a in (similar, n_removed, starting)]
        def vp(a):
            p = _ptr(a)
            return None if p is None else p.value
        if similar_stride is None:
            similar_stride = 0 if opt[0] is None or mem != WG_MEM_HOST else opt[0].shape[1]
        b = _capi.PldpBatch(D=vp(keep[0]), m=vp(keep[1]), DPu=vp(keep[2]), dpu_stride=int(pb.get("dpu_stride", 0)),
                            DPx=vp(keep[3]), dpx_stride=int(pb["dpx_stride"]), ZMPRef=vp(keep[4]), XkYk=vp(keep[5]),
                            X=vp(X), similar=vp(opt[0]), similar_stride=int(similar_stride),
                            n_removed=vp(opt[1]), starting=vp(opt[2]), hot=vp(hot), hot_start=int(bool(hot_start)),
                            max_iterations=int(max_iterations), info=vp(info))
        if ranked:
            self._check(self.lib.wg_pldp_solve_batch_ranked(self.h, mem, int(B), C.byref(b), vp(rk[0]), vp(rk[1]), vp(rk[2]),
                                                            int(pb["row_stride"])))
        else:
            self._check(self.lib.wg_pldp_solve_batch(self.h, mem, int(B), C.byref(b)))
        return X, info

    def optcholesky_add_rows(self, A, rows, L, mode, nb_max, card_u, nb_constraints, k0, k1):
        """OptCholesky::AddActiveConstraint for rows[:, k0:k1] of every instance (host arrays; L updated in place)."""
        A = np.ascontiguousarray(A, dtype=np.float64); rows = np.ascontiguousarray(rows, dtype=np.int32)
        assert L.flags["C_CONTIGUOUS"] and L.dtype == np.float64
        B = A.shape[0]
        self._check(self.lib.wg_optcholesky_add_rows_batch(self.h, WG_MEM_HOST, B, mode, nb_max, card_u, nb_constraints,
                                                           A.ctypes.data, A[0].size, rows.ctypes.data, rows.shape[1],
                                                           k0, k1, L.ctypes.data, L[0].size))
        return L

    def optcholesky_full(self, A, inverse=True):
        """ComputeNormalCholeskyOnANormal (+ ComputeInverseCholeskyNormal(1)) for A [B][n][n] -> (L, iL)."""
        A = np.ascontiguousarray(A, dtype=np.float64)
        B, n, _ = A.shape
        L = np.zeros_like(A); iL = np.zeros_like(A) if inverse else None
        self._check(self.lib.wg_optcholesky_full_batch(self.h, WG_MEM_HOST, B, n, A.ctypes.data, L.ctypes.data,
                                                       None if iL is None else iL.ctypes.data, n))
        return L, iL


    # ---- Dimitrov2008 front to back ------------------------------------------------------------------------------
    def dimitrov_set_params(self, params=None):
        """InitConstants(): -> dict of the constant matrices (one axis block, row-major)."""
        self.dimitrov_params = params if params is not None else dimitrov_default_params()
        out = {k: np.zeros(shape) for k, shape in (("iPu", (16, 16)), ("Px", (16, 3)), ("Pu", (16, 16)),
                                                   ("iLQ", (16, 16)), ("OptB", (16, 3)), ("OptC", (16, 16)))}
        self._check(self.lib.wg_dimitrov_set_params(self.h, C.byref(self.dimitrov_params),
                                                    *[out[k].ctypes.data for k in ("iPu", "Px", "Pu", "iLQ", "OptB", "OptC")]))
        return out

    def convex_hull_batch(self, points):
        """DoComputeConvexHull for [B][n][2] point sets -> (hull [B][8][2], counts [B])."""
        pts = np.ascontiguousarray(points, dtype=np.float64)
        B, n = pts.shape[0], pts.shape[1]
        hull = np.zeros((B, 8, 2)); cnt = np.zeros(B, dtype=np.int32)
        self._check(self.lib.wg_convex_hull_batch(self.h, WG_MEM_HOST, B, n, pts.ctypes.data, hull.ctypes.data, cnt.ctypes.data))
        return hull, cnt

    def fcals_build(self, left, right, types, cap=None):
        """BuildLinearConstraintInequalities for ONE feet buffer (left/right: [n][6] floats or KAJITA_FOOT_DTYPE,
        types [n][3]) -> LCI_DTYPE records."""
        L = np.ascontiguousarray(left).view(np.float64).reshape(-1, 6)
        R = np.ascontiguousarray(right).view(np.float64).reshape(-1, 6)
        ty = np.ascontiguousarray(types, dtype=np.int32).reshape(-1, 3)
        n = len(L)
        cap = cap or 1024
        so = np.array([0, n], dtype=np.int64); lo = np.array([0, cap], dtype=np.int64)
        out = np.zeros(cap, dtype=LCI_DTYPE); cnt = np.zeros(1, dtype=np.int32)
        if not hasattr(self, "dimitrov_params"):
            self.dimitrov_set_params()
        self._check(self.lib.wg_fcals_build_batch(self.h, WG_MEM_HOST, 1, so.ctypes.data_as(_capi.c_i64_p), L.ctypes.data,
                                                  R.ctypes.data, ty.ctypes.data, lo.ctypes.data_as(_capi.c_i64_p),
                                                  out.ctypes.data, cnt.ctypes.data))
        return out[:cnt[0]]

    def dimitrov_run(self, walks, init_feet, zmpdisc_params=None, want_feet=True):
        """footsteps -> ZMPDiscretization -> support polygons -> PLDP receding-horizon loop -> CoM / ZMP at 5 ms for a
        list of step arrays.  -> dict(com, zmp, left, right, types, periods (list per walk), status, periods_done,
        sample_offsets)."""
        if not hasattr(self, "dimitrov_params"):
            self.dimitrov_set_params()
        B = len(walks)
        off = np.concatenate([[0], np.cumsum([len(w) for w in walks])]).astype(np.int64)
        steps = np.ascontiguousarray(np.concatenate([np.asarray(w, dtype=REL_STEP_DTYPE) for w in walks]))
        plan = KajitaPlan(self, off, steps, np.ascontiguousarray(init_feet, dtype=np.float64), zmpdisc_params)
        try:
            so = plan.sample_offsets
            ns = int(so[-1])
            pc = [int(self.lib.wg_dimitrov_period_count(C.byref(self.dimitrov_params), int(so[b + 1] - so[b]))) for b in range(B)]
            po = np.concatenate([[0], np.cumsum(pc)]).astype(np.int64)
            com = np.zeros((ns, 6)); zmp = np.zeros((ns, 2))
            left = np.zeros(ns, dtype=KAJITA_FOOT_DTYPE) if want_feet else None
            right = np.zeros(ns, dtype=KAJITA_FOOT_DTYPE) if want_feet else None
            per = np.zeros(max(1, int(po[-1])), dtype=DIMITROV_PERIOD_DTYPE)
            status = np.zeros(B, dtype=np.int32); done = np.zeros(B, dtype=np.int32)
            self._check(self.lib.wg_dimitrov_run_batch(self.h, plan.h, WG_MEM_HOST, com.ctypes.data, zmp.ctypes.data,
                                                       _ptr(left), _ptr(right), po.ctypes.data_as(_capi.c_i64_p),
                                                       per.ctypes.data, status.ctypes.data, done.ctypes.data))
            types = None
            if want_feet:
                types = np.zeros((ns, 3), dtype=np.int32)
                plan.discretize(step_type=types)
        finally:
            plan.destroy()
        return {"com": com, "zmp": zmp, "left": left, "right": right, "types": types, "status": status,
                "periods_done": done, "periods": [per[po[b]:po[b] + done[b]] for b in range(B)],
                "period_counts": np.array(pc), "sample_offsets": so}

    # ---- Wieber2006 generator ------------------------------------------------------------------
    def wieber_set_params(self, params=None):
        if params is None:
            params = _capi.WieberParams()
            self.lib.wg_wieber_default_params(C.byref(params))
        self.wieber_params = params
        self._check(self.lib.wg_wieber_set_params(self.h, C.byref(params)))

    def wieber_run(self, walks, init_feet, zmpdisc_params=None, want_feet=False):
        """footsteps -> ZMPDiscretization -> support polygons -> per-period dense QP -> CoM / ZMP at 5 ms for a list of step
        arrays.  -> dict(com, zmp, left, right, status, periods_done, period_counts, qp_iterations, sample_offsets)."""
        if not hasattr(self, "wieber_params"):
            self.wieber_set_params()
        B = len(walks)
        off = np.concatenate([[0], np.cumsum([len(w) for w in walks])]).astype(np.int64)
        steps = np.ascontiguousarray(np.concatenate([np.asarray(w, dtype=REL_STEP_DTYPE) for w in walks]))
        plan = KajitaPlan(self, off, steps, np.ascontiguousarray(init_feet, dtype=np.float64), zmpdisc_params)
        try:
            so = plan.sample_offsets
            ns = int(so[-1])
            pc = [int(self.lib.wg_wieber_period_count(C.byref(self.wieber_params), int(so[b + 1] - so[b]))) for b in range(B)]
            com = np.zeros((ns, 6)); zmp = np.zeros((ns, 2))
            left = np.zeros(ns, dtype=KAJITA_FOOT_DTYPE) if want_feet else None
            right = np.zeros(ns, dtype=KAJITA_FOOT_DTYPE) if want_feet else None
            status = np.zeros(B, dtype=np.int32); done = np.zeros(B, dtype=np.int32); its = np.zeros(B, dtype=np.int64)
            self._check(self.lib.wg_wieber_run_batch(self.h, plan.h, WG_MEM_HOST, com.ctypes.data, zmp.ctypes.data, _ptr(left),
                                                     _ptr(right), status.ctypes.data, done.ctypes.data, its.ctypes.data))
        finally:
            plan.destroy()
        return {"com": com, "zmp": zmp, "left": left, "right": right, "status": status, "periods_done": done,
                "period_counts": np.array(pc), "qp_iterations": its, "sample_offsets": so}


class MultiContext:
    """wg_multi: several GPUs from one process (instance i -> device i mod G, statistics all-reduced over NCCL)."""

    def __init__(self, device_mask=0):
        self.lib = _capi.load()
        h = C.c_void_p()
        rc = self.lib.wg_multi_create(int(device_mask), C.byref(h))
        if rc != 0:
            raise WalkgenError(rc, "wg_multi_create failed (no CUDA device?)")
        self.h = h
        self.size = self.lib.wg_multi_size(h)
        self.nccl_version = self.lib.wg_multi_nccl_version(h)

    def herdt_set_params(self, hp=None, mp=None):
        self.hp = hp or herdt_default_params()
        self.mp = mp or herdt_mpc_default_params()
        rc = self.lib.wg_multi_herdt_set_params(self.h, C.byref(self.hp), C.byref(self.mp))
        if rc != 0:
            raise WalkgenError(rc, self.lib.wg_multi_last_error(self.h).decode())

    def herdt_mpc_sweep(self, vel_ref, periods, chunk=10,
                        init9=(0.0316055, 0.0, 0.7116911, 0.0, 0.09, 0.0, 0.0, -0.09, 0.0)):
        v = np.ascontiguousarray(vel_ref, dtype=np.float64)
        i9 = np.ascontiguousarray(init9, dtype=np.float64)
        st = _capi.MultiStats()
        rc = self.lib.wg_multi_herdt_mpc_sweep(self.h, len(v), int(periods), int(chunk), v.ctypes.data, i9.ctypes.data, C.byref(st))
        if rc != 0:
            raise WalkgenError(rc, self.lib.wg_multi_last_error(self.h).decode())
        G = st.devices
        return {"instances": st.instances, "periods": st.periods, "seconds": st.seconds, "qp_solves": st.qp_solves,
                "failures": st.failures, "iterations": st.iterations, "still_online": st.still_online, "devices": G,
                "reduced_by_nccl": bool(st.reduced_by_nccl), "nccl_version": st.nccl_version,
                "device_ms": [float(st.device_ms[k]) for k in range(G)],
                "device_instances": [int(st.device_instances[k]) for k in range(G)],
                "device_launches": [int(st.device_launches[k]) for k in range(G)]}

    def close(self):
        if self.h:
            self.lib.wg_multi_destroy(self.h)
            self.h = None


class KajitaPlan:
    """Footsteps -> ZMP reference + feet (ZMPDiscretization) -> CoM (preview control) for a ragged batch of walks."""

    def __init__(self, ctx: Context, step_offsets, steps, init_feet, params=None):
        self.ctx = ctx
        self.params = params if params is not None else zmpdisc_default_params()
        self.step_offsets = np.ascontiguousarray(step_offsets, dtype=np.int64)
        self.B = len(self.step_offsets) - 1
        steps = np.ascontiguousarray(steps, dtype=REL_STEP_DTYPE)
        feet = np.ascontiguousarray(init_feet, dtype=np.float64).reshape(self.B, 6)
        h = C.c_void_p()
        ctx._check(ctx.lib.wg_kajita_plan_create(ctx.h, C.byref(self.params), self.B,
                                                 self.step_offsets.ctypes.data_as(_capi.c_i64_p), steps.ctypes.data,
                                                 feet.ctypes.data, C.byref(h)))
        self.h = h
        so = ctx.lib.wg_kajita_plan_sample_offsets(h)
        self.sample_offsets = np.ctypeslib.as_array(so, shape=(self.B + 1,)).copy()
        self.total_samples = int(ctx.lib.wg_kajita_plan_total_samples(h))
        self.total_steps = int(ctx.lib.wg_kajita_plan_total_steps(h))

    def set_steps(self, steps, init_feet=None):
        self.ctx._check(self.ctx.lib.wg_kajita_plan_set_steps(self.h, _ptr(steps), _ptr(init_feet)))

    def discretize(self, zmpref_xy=None, zmp_theta=None, left=None, right=None, step_type=None, mem=WG_MEM_HOST):
        """ZMPDiscretization::GetZMPDiscretization for every walk."""
        self.ctx._check(self.ctx.lib.wg_zmpdisc_run_batch(self.ctx.h, self.h, mem, _ptr(zmpref_xy), _ptr(zmp_theta),
                                                          _ptr(left), _ptr(right), _ptr(step_type)))

    def run(self, state, com_out=None, zmp_out=None, zmpref_xy=None, left=None, right=None, simulation=True,
            mem=WG_MEM_HOST):
        """Footsteps -> CoM on the GPU."""
        self.ctx._check(self.ctx.lib.wg_kajita_run_batch(self.ctx.h, self.h, mem, _ptr(state), _ptr(com_out),
                                                         _ptr(zmp_out), _ptr(zmpref_xy), _ptr(left), _ptr(right),
                                                         int(simulation)))

    def destroy(self):
        if self.h:
            self.ctx.lib.wg_kajita_plan_destroy(self.h)
            self.h = None


STREAM_START, STREAM_FINISH = 1, 2


class KajitaStream:
    """On-line Kajita2003 generator for B walks: InitOnLine / OnLineAddFoot / EndPhaseOfTheWalking, batched, with the
    preview loop consuming each walk's new ZMP reference (wg_kajita_stream_*).  One append plans one run."""

    def __init__(self, ctx: Context, B, params=None, with_preview=True):
        self.ctx = ctx
        self.B = int(B)
        self.params = params if params is not None else zmpdisc_default_params()
        self.with_preview = bool(with_preview)
        h = C.c_void_p()
        ctx._check(ctx.lib.wg_kajita_stream_create(ctx.h, C.byref(self.params), self.B, int(self.with_preview), C.byref(h)))
        self.h = h
        self.carry_rows = int(ctx.lib.wg_kajita_stream_carry_rows(h))   # NL-1 with preview, 0 without
        self.sample_offsets = np.zeros(self.B + 1, dtype=np.int64)
        self.com_offsets = np.zeros(self.B + 1, dtype=np.int64)
        self.com_counts = np.zeros(self.B, dtype=np.int64)

    def append(self, step_offsets, steps, flags=None, init_feet=None):
        """Plan the next run: walk b appends steps[step_offsets[b]:step_offsets[b+1]] with flags[b] (STREAM_START /
        STREAM_FINISH).  Refreshes sample_offsets, com_offsets and com_counts (the row layout of the run)."""
        off = np.ascontiguousarray(step_offsets, dtype=np.int64)
        assert len(off) == self.B + 1
        steps = np.ascontiguousarray(steps, dtype=REL_STEP_DTYPE)
        fl = None if flags is None else np.ascontiguousarray(flags, dtype=np.int32)
        feet = None if init_feet is None else np.ascontiguousarray(init_feet, dtype=np.float64).reshape(self.B, 6)
        lib = self.ctx.lib
        self.ctx._check(lib.wg_kajita_stream_append(self.h, off.ctypes.data_as(_capi.c_i64_p), steps.ctypes.data if len(steps) else None,
                                                    _ptr(fl), _ptr(feet)))
        self.sample_offsets = np.ctypeslib.as_array(lib.wg_kajita_stream_sample_offsets(self.h), shape=(self.B + 1,)).copy()
        self.com_offsets = np.ctypeslib.as_array(lib.wg_kajita_stream_com_offsets(self.h), shape=(self.B + 1,)).copy()
        self.com_counts = np.ctypeslib.as_array(lib.wg_kajita_stream_com_counts(self.h), shape=(self.B,)).copy()
        return self.sample_offsets, self.com_offsets, self.com_counts

    def host_outputs(self, com=True):
        """Zeroed host arrays sized for the planned run: zmpref, zmp_theta, left, right, step_type (and com_out, zmp_out)."""
        n, m = int(self.sample_offsets[-1]), int(self.com_offsets[-1])
        out = dict(zmpref_xy=np.zeros((n, 2)), zmp_theta=np.zeros(n), left=np.zeros(n, dtype=KAJITA_FOOT_DTYPE),
                   right=np.zeros(n, dtype=KAJITA_FOOT_DTYPE), step_type=np.zeros((n, 3), dtype=np.int32))
        if com and self.with_preview:
            out.update(com_out=np.zeros((m, 6)), zmp_out=np.zeros((m, 2)))
        return out

    def run(self, zmpref_xy=None, zmp_theta=None, left=None, right=None, step_type=None, com_out=None, zmp_out=None,
            simulation=True, mem=WG_MEM_HOST):
        """Run the planned append (wg_kajita_stream_run); any output may be None."""
        self.ctx._check(self.ctx.lib.wg_kajita_stream_run(self.h, mem, _ptr(zmpref_xy), _ptr(zmp_theta), _ptr(left), _ptr(right),
                                                          _ptr(step_type), _ptr(com_out), _ptr(zmp_out), int(simulation)))

    def state(self, preview_state=None, mem=WG_MEM_HOST):
        """-> (preview_state [B][8] or None, samples_emitted [B], steps_previewed [B], open [B])."""
        if preview_state is None and self.with_preview and mem == WG_MEM_HOST:
            preview_state = np.zeros((self.B, 8))
        emitted = np.zeros(self.B, dtype=np.int64); previewed = np.zeros(self.B, dtype=np.int64)
        is_open = np.zeros(self.B, dtype=np.int32)
        self.ctx._check(self.ctx.lib.wg_kajita_stream_state(self.h, mem, _ptr(preview_state), _ptr(emitted), _ptr(previewed),
                                                            _ptr(is_open)))
        return preview_state, emitted, previewed, is_open

    def save(self, idx=None):
        """-> (walks [n] of KAJITA_STREAM_WALK_DTYPE, carry [n][carry_rows][2] or None without preview) of the walks idx
        (all B when None): wg_kajita_stream_save."""
        ia = _indices(idx)
        n = self.B if ia is None else len(ia)
        walks = np.zeros(n, dtype=KAJITA_STREAM_WALK_DTYPE)
        carry = np.zeros((n, self.carry_rows, 2)) if self.with_preview else None
        self.ctx._check(self.ctx.lib.wg_kajita_stream_save(self.h, WG_MEM_HOST, n, _ptr(ia), walks.ctypes.data, _ptr(carry)))
        return walks, carry

    def restore(self, walks, carry, idx=None):
        """Write host records and carry rows into the walks idx (0..len(walks)-1 when None); all or nothing."""
        rec = np.ascontiguousarray(walks, dtype=KAJITA_STREAM_WALK_DTYPE).reshape(-1)
        c = None if carry is None else np.ascontiguousarray(carry, dtype=np.float64)
        assert c is None or c.shape == (len(rec), self.carry_rows, 2)
        ia = _indices(idx)
        assert ia is None or len(ia) == len(rec)
        self.ctx._check(self.ctx.lib.wg_kajita_stream_restore(self.h, WG_MEM_HOST, len(rec), _ptr(ia), rec.ctypes.data, _ptr(c)))

    def save_device(self, n, d_walks, d_carry, idx=None):
        """Device-resident save of n walks into d_walks, d_carry (None without preview); asynchronous on the context stream."""
        self.ctx._check(self.ctx.lib.wg_kajita_stream_save(self.h, WG_MEM_DEVICE, int(n), _ptr(_indices(idx)), _ptr(d_walks),
                                                           _ptr(d_carry)))

    def restore_device(self, n, d_walks, d_carry, idx=None):
        """Device-resident restore of n walks from d_walks, d_carry (waits for the check of the records)."""
        self.ctx._check(self.ctx.lib.wg_kajita_stream_restore(self.h, WG_MEM_DEVICE, int(n), _ptr(_indices(idx)), _ptr(d_walks),
                                                              _ptr(d_carry)))

    def copy_from(self, src: "KajitaStream", src_idx=None, dst_idx=None):
        """Walk src_idx[i] of src -> walk dst_idx[i] of this stream, on the device (wg_kajita_stream_copy); n is the length of
        the index arrays given, B of this stream when neither is."""
        n, si, di = _copy_indices(src_idx, dst_idx, self.B)
        self.ctx._check(self.ctx.lib.wg_kajita_stream_copy(self.h, n, _ptr(di), src.h, _ptr(si)))

    def destroy(self):
        if self.h:
            self.ctx.lib.wg_kajita_stream_destroy(self.h)
            self.h = None


class KajitaOnline:
    """On-line Kajita2003 generator for B walks: RunOneStepOfTheControlLoop's Kajita branch batched, each walk with its own
    start tick, step stack, commands (PUSH, :addstandardonlinestep, :StopOnLineStepSequencing) and queues
    (wg_kajita_online_*)."""

    def __init__(self, ctx: Context, B, params=None, com_height=0.814, max_step_time=0.8):
        self.ctx = ctx
        self.B = int(B)
        self.params = params if params is not None else zmpdisc_default_params()
        h = C.c_void_p()
        ctx._check(ctx.lib.wg_kajita_online_create(ctx.h, C.byref(self.params), self.B, float(com_height), float(max_step_time),
                                                   C.byref(h)))
        self.h = h
        self.ring_rows = int(ctx.lib.wg_kajita_online_ring_rows(h))
        self.carry_rows = int(ctx.lib.wg_kajita_online_carry_rows(h))   # NL-1

    def start(self, idx, steps, init_feet, keep_last=None):
        """:StartOnLineStepSequencing for the walks idx: steps is one REL_STEP_DTYPE list per walk (its first step the
        support-foot step), init_feet [len(idx)][6], keep_last [len(idx)] of +-1 or None (+1)."""
        idx = np.ascontiguousarray(idx, dtype=np.int32).reshape(-1)
        lists = [np.asarray(s, dtype=REL_STEP_DTYPE).reshape(-1) for s in steps]
        assert len(lists) == len(idx)
        off = np.concatenate([[0], np.cumsum([len(s) for s in lists])]).astype(np.int64)
        st = np.ascontiguousarray(np.concatenate(lists) if lists else np.zeros(0, dtype=REL_STEP_DTYPE))
        feet = np.ascontiguousarray(init_feet, dtype=np.float64).reshape(len(idx), 6)
        keep = None if keep_last is None else np.ascontiguousarray(keep_last, dtype=np.int32).reshape(len(idx))
        self.ctx._check(self.ctx.lib.wg_kajita_online_start(self.h, len(idx), idx.ctypes.data, off.ctypes.data_as(_capi.c_i64_p),
                                                            st.ctypes.data, feet.ctypes.data, _ptr(keep)))

    def tick(self, nticks, commands=None, rows=True, running=True):
        """nticks ticks on host arrays: commands [nticks][B] of KAJITA_COMMAND_DTYPE or None -> (rows [nticks][B] of
        KAJITA_TICK_DTYPE, running [nticks][B] int8), each None when not asked for."""
        n = int(nticks)
        cmd = None if commands is None else np.ascontiguousarray(commands, dtype=KAJITA_COMMAND_DTYPE)
        assert cmd is None or cmd.shape == (n, self.B)
        r = np.zeros((n, self.B), dtype=KAJITA_TICK_DTYPE) if rows else None
        run = np.zeros((n, self.B), dtype=np.int8) if running else None
        self.ctx._check(self.ctx.lib.wg_kajita_online_tick(self.h, WG_MEM_HOST, n, _ptr(cmd), _ptr(r), _ptr(run)))
        return r, run

    def tick_device(self, nticks, commands=None, d_rows=None, d_running=None):
        """Device-resident rows and running flags (asynchronous on the context stream); commands stay a host array."""
        cmd = None if commands is None else np.ascontiguousarray(commands, dtype=KAJITA_COMMAND_DTYPE)
        assert cmd is None or cmd.shape == (int(nticks), self.B)
        self.ctx._check(self.ctx.lib.wg_kajita_online_tick(self.h, WG_MEM_DEVICE, int(nticks), _ptr(cmd), _ptr(d_rows),
                                                           _ptr(d_running)))

    def state(self):
        """-> (queued int64 [B], stacked int32 [B], running int32 [B], online int32 [B])."""
        q = np.zeros(self.B, dtype=np.int64)
        s, r, o = (np.zeros(self.B, dtype=np.int32) for _ in range(3))
        self.ctx._check(self.ctx.lib.wg_kajita_online_state(self.h, q.ctypes.data, s.ctypes.data, r.ctypes.data, o.ctypes.data))
        return q, s, r, o

    def _stack_buffer(self, idx):
        """A host array for the stacks of the walks idx (all B when None), sized from state()."""
        stacked = self.state()[1]
        cap = int(stacked.sum() if idx is None else stacked[np.asarray(idx, dtype=np.int64)].sum())
        return np.zeros(max(cap, 1), dtype=REL_STEP_DTYPE), cap

    @staticmethod
    def _split_stacks(walks, buf):
        ends = np.cumsum(walks["stacked"].astype(np.int64))
        return [buf[e - k:e].copy() for e, k in zip(ends, walks["stacked"].astype(np.int64))]

    def save(self, idx=None):
        """-> (walks [n] of KAJITA_ONLINE_WALK_DTYPE, carry [n][carry_rows][2], queue [n][ring_rows] of KAJITA_TICK_DTYPE,
        stacks: one REL_STEP_DTYPE array per walk, front first) of the walks idx (all B when None)."""
        ia = _indices(idx)
        n = self.B if ia is None else len(ia)
        walks = np.zeros(n, dtype=KAJITA_ONLINE_WALK_DTYPE)
        carry = np.zeros((n, self.carry_rows, 2))
        queue = np.zeros((n, self.ring_rows), dtype=KAJITA_TICK_DTYPE)
        buf, cap = self._stack_buffer(ia)
        ln = C.c_int64()
        self.ctx._check(self.ctx.lib.wg_kajita_online_save(self.h, WG_MEM_HOST, n, _ptr(ia), walks.ctypes.data, carry.ctypes.data,
                                                           queue.ctypes.data, buf.ctypes.data, cap, C.byref(ln)))
        return walks, carry, queue, self._split_stacks(walks, buf)

    @staticmethod
    def _join_stacks(stacks):
        lists = [np.asarray(s, dtype=REL_STEP_DTYPE).reshape(-1) for s in stacks]
        buf = np.ascontiguousarray(np.concatenate(lists) if lists else np.zeros(0, dtype=REL_STEP_DTYPE))
        return buf, len(buf)

    def restore(self, walks, carry, queue, stacks, idx=None):
        """Write host records, carry rows, queues and stacks into the walks idx (0..len(walks)-1 when None); all or nothing."""
        rec = np.ascontiguousarray(walks, dtype=KAJITA_ONLINE_WALK_DTYPE).reshape(-1)
        n = len(rec)
        c = np.ascontiguousarray(carry, dtype=np.float64)
        q = np.ascontiguousarray(queue, dtype=KAJITA_TICK_DTYPE)
        assert c.shape == (n, self.carry_rows, 2) and q.shape == (n, self.ring_rows)
        ia = _indices(idx)
        assert ia is None or len(ia) == n
        buf, ln = self._join_stacks(stacks)
        self.ctx._check(self.ctx.lib.wg_kajita_online_restore(self.h, WG_MEM_HOST, n, _ptr(ia), rec.ctypes.data, c.ctypes.data,
                                                              q.ctypes.data, buf.ctypes.data if ln else None, ln))

    def save_device(self, n, d_walks, d_carry, d_queue, idx=None):
        """Device-resident save of n walks into d_walks, d_carry, d_queue (asynchronous on the context stream) -> the stacks,
        one REL_STEP_DTYPE array per walk."""
        ia = _indices(idx)
        buf, cap = self._stack_buffer(ia)
        k = self.state()[1][np.arange(int(n)) if ia is None else ia].astype(np.int64)
        ln = C.c_int64()
        self.ctx._check(self.ctx.lib.wg_kajita_online_save(self.h, WG_MEM_DEVICE, int(n), _ptr(ia), _ptr(d_walks), _ptr(d_carry),
                                                           _ptr(d_queue), buf.ctypes.data, cap, C.byref(ln)))
        ends = np.cumsum(k)
        return [buf[e - m:e].copy() for e, m in zip(ends, k)]

    def restore_device(self, n, d_walks, d_carry, d_queue, stacks, idx=None):
        """Device-resident restore of n walks from d_walks, d_carry, d_queue and the host stacks (reads the records back)."""
        buf, ln = self._join_stacks(stacks)
        self.ctx._check(self.ctx.lib.wg_kajita_online_restore(self.h, WG_MEM_DEVICE, int(n), _ptr(_indices(idx)), _ptr(d_walks),
                                                              _ptr(d_carry), _ptr(d_queue), buf.ctypes.data if ln else None, ln))

    def copy_from(self, src: "KajitaOnline", src_idx=None, dst_idx=None):
        """Walk src_idx[i] of src -> walk dst_idx[i] of this handle, on the device (wg_kajita_online_copy); n is the length of
        the index arrays given, B of this handle when neither is."""
        n, si, di = _copy_indices(src_idx, dst_idx, self.B)
        self.ctx._check(self.ctx.lib.wg_kajita_online_copy(self.h, n, _ptr(di), src.h, _ptr(si)))

    def destroy(self):
        if self.h:
            self.ctx.lib.wg_kajita_online_destroy(self.h)
            self.h = None


class HerdtOnline:
    """On-line Herdt2010 generator for B robots: RunOneStepOfTheControlLoop batched, each robot with its own start tick,
    commands (:setVelReference, :stoppg) and deques (wg_herdt_online_*)."""

    def __init__(self, ctx: Context, B):
        self.ctx = ctx
        self.B = int(B)
        h = C.c_void_p()
        ctx._check(ctx.lib.wg_herdt_online_create(ctx.h, self.B, C.byref(h)))
        self.h = h

    def start(self, idx, init15=HERDT_INIT15):
        """:HerdtOnline for the robots idx; init15: one start configuration (broadcast) or an array [len(idx)][15]."""
        idx = np.ascontiguousarray(idx, dtype=np.int32).reshape(-1)
        init = np.ascontiguousarray(init15, dtype=np.float64)
        stride = 0 if init.ndim == 1 else 15
        assert init.size == 15 or init.shape == (len(idx), 15)
        self.ctx._check(self.ctx.lib.wg_herdt_online_start(self.h, len(idx), idx.ctypes.data, init.ctypes.data, stride))

    def tick(self, nticks, commands=None, rows=True, running=True):
        """nticks ticks on host arrays: commands [nticks][B] of HERDT_COMMAND_DTYPE or None -> (rows [nticks][B] of
        TICK_DTYPE, running [nticks][B] int8), each None when not asked for."""
        n = int(nticks)
        cmd = None if commands is None else np.ascontiguousarray(commands, dtype=HERDT_COMMAND_DTYPE)
        assert cmd is None or cmd.shape == (n, self.B)
        r = np.zeros((n, self.B), dtype=TICK_DTYPE) if rows else None
        run = np.zeros((n, self.B), dtype=np.int8) if running else None
        self.ctx._check(self.ctx.lib.wg_herdt_online_tick(self.h, WG_MEM_HOST, n, _ptr(cmd), _ptr(r), _ptr(run)))
        return r, run

    def tick_device(self, nticks, d_commands=None, d_rows=None, d_running=None):
        """Device-resident form (asynchronous on the context stream)."""
        self.ctx._check(self.ctx.lib.wg_herdt_online_tick(self.h, WG_MEM_DEVICE, int(nticks), _ptr(d_commands), _ptr(d_rows),
                                                          _ptr(d_running)))

    def tick_plan(self, nticks, plans, commands=None, rows=True, running=True):
        """tick(), and the plan of every robot that fires (wg_herdt_online_tick_plan): plans, a host array [B] of
        HERDT_PLAN_DTYPE, is updated in place for the robots that fire (the last firing of the call wins), the other
        entries keep their bytes -> (rows, running, plan_tick [B] int32: index of the last firing in the call, or -1)."""
        n = int(nticks)
        cmd = None if commands is None else np.ascontiguousarray(commands, dtype=HERDT_COMMAND_DTYPE)
        assert cmd is None or cmd.shape == (n, self.B)
        assert plans is None or (plans.dtype == HERDT_PLAN_DTYPE and plans.shape == (self.B,) and plans.flags["C_CONTIGUOUS"])
        r = np.zeros((n, self.B), dtype=TICK_DTYPE) if rows else None
        run = np.zeros((n, self.B), dtype=np.int8) if running else None
        pt = np.full(self.B, -1, dtype=np.int32)
        self.ctx._check(self.ctx.lib.wg_herdt_online_tick_plan(self.h, WG_MEM_HOST, n, _ptr(cmd), _ptr(r), _ptr(run),
                                                               _ptr(plans), _ptr(pt)))
        return r, run, pt

    def tick_plan_device(self, nticks, d_plans, d_commands=None, d_rows=None, d_running=None, d_plan_tick=None):
        """Device-resident form of tick_plan (asynchronous on the context stream)."""
        self.ctx._check(self.ctx.lib.wg_herdt_online_tick_plan(self.h, WG_MEM_DEVICE, int(nticks), _ptr(d_commands),
                                                               _ptr(d_rows), _ptr(d_running), _ptr(d_plans),
                                                               _ptr(d_plan_tick)))

    @property
    def d_states(self) -> int:
        """Device address of the B MPC_STATE_DTYPE records."""
        return self.ctx.lib.wg_herdt_online_states(self.h)

    def states(self):
        """Host copy of the B state records."""
        out = np.zeros(self.B, dtype=MPC_STATE_DTYPE)
        self.ctx._check(self.ctx.lib.wg_memcpy_d2h(self.ctx.h, out.ctypes.data, self.d_states, out.nbytes))
        self.ctx.sync()
        return out

    def set_states(self, states):
        """Write B state records (e.g. a copy from states(), edited) back to the device."""
        st = np.ascontiguousarray(states, dtype=MPC_STATE_DTYPE)
        assert st.shape == (self.B,)
        self.ctx._check(self.ctx.lib.wg_memcpy_h2d(self.ctx.h, self.d_states, st.ctypes.data, st.nbytes))
        self.ctx.sync()

    def save(self, idx=None):
        """-> host records [n] of ONLINE_ROBOT_DTYPE of the robots idx (all B when None): wg_herdt_online_save."""
        ia = _indices(idx)
        out = np.zeros(self.B if ia is None else len(ia), dtype=ONLINE_ROBOT_DTYPE)
        self.ctx._check(self.ctx.lib.wg_herdt_online_save(self.h, WG_MEM_HOST, len(out), _ptr(ia), out.ctypes.data))
        return out

    def restore(self, records, idx=None):
        """Write host records (ONLINE_ROBOT_DTYPE) into the robots idx (0..len(records)-1 when None); all or nothing."""
        rec = np.ascontiguousarray(records, dtype=ONLINE_ROBOT_DTYPE).reshape(-1)
        ia = _indices(idx)
        assert ia is None or len(ia) == len(rec)
        self.ctx._check(self.ctx.lib.wg_herdt_online_restore(self.h, WG_MEM_HOST, len(rec), _ptr(ia), rec.ctypes.data))

    def save_device(self, n, d_out, idx=None):
        """Device-resident save of n robots into d_out (asynchronous on the context stream)."""
        self.ctx._check(self.ctx.lib.wg_herdt_online_save(self.h, WG_MEM_DEVICE, int(n), _ptr(_indices(idx)), _ptr(d_out)))

    def restore_device(self, n, d_in, idx=None):
        """Device-resident restore of n records from d_in (waits for the check of the records)."""
        self.ctx._check(self.ctx.lib.wg_herdt_online_restore(self.h, WG_MEM_DEVICE, int(n), _ptr(_indices(idx)), _ptr(d_in)))

    def copy_from(self, src: "HerdtOnline", src_idx=None, dst_idx=None):
        """Robot src_idx[i] of src -> robot dst_idx[i] of this handle, on the device (wg_herdt_online_copy); n is the
        length of the index arrays given, B of this handle when neither is."""
        n, si, di = _copy_indices(src_idx, dst_idx, self.B)
        self.ctx._check(self.ctx.lib.wg_herdt_online_copy(self.h, n, _ptr(di), src.h, _ptr(si)))

    def destroy(self):
        if self.h:
            self.ctx.lib.wg_herdt_online_destroy(self.h)
            self.h = None


class PreviewPlan:
    def __init__(self, ctx: Context, offsets):
        self.ctx = ctx
        self.offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self.B = len(self.offsets) - 1
        h = C.c_void_p()
        ctx._check(ctx.lib.wg_preview_plan_create(ctx.h, self.B, self.offsets.ctypes.data_as(_capi.c_i64_p),
                                                  C.byref(h)))
        self.h = h
        self.total_steps = ctx.lib.wg_preview_plan_total_steps(h)
        self.total_samples = ctx.lib.wg_preview_plan_total_samples(h)

    def run(self, zmpref_xy, state, com_out=None, zmp_out=None, simulation=True, mem=WG_MEM_HOST):
        self.ctx._check(self.ctx.lib.wg_preview_run_batch(self.ctx.h, self.h, mem, _ptr(zmpref_xy), _ptr(state),
                                                          _ptr(com_out), _ptr(zmp_out), int(simulation)))

    def run_pos(self, zmpref_xy, state, com_pos_out, simulation=True, mem=WG_MEM_HOST):
        """wg_preview_run_batch_pos: only the CoM position (x, y) of every step."""
        self.ctx._check(self.ctx.lib.wg_preview_run_batch_pos(self.ctx.h, self.h, mem, _ptr(zmpref_xy), _ptr(state),
                                                              _ptr(com_pos_out), int(simulation)))

    def delta_zmp(self, zmpref_xy, zmp_multibody_xy, delta_out, mem=WG_MEM_HOST):
        """wg_preview_delta_zmp: delta[k] = zmpref[k + 1] - zmp_multibody[k] (EvaluateMultiBodyZMP)."""
        self.ctx._check(self.ctx.lib.wg_preview_delta_zmp(self.ctx.h, self.h, mem, _ptr(zmpref_xy), _ptr(zmp_multibody_xy),
                                                          _ptr(delta_out)))

    def run_stage2(self, delta_zmp_xy, com_stage1, state2, com_final_out, dzmp_out=None, mem=WG_MEM_HOST):
        """wg_preview_stage2_run_batch: SecondStageOfControl over the whole delta-ZMP stream."""
        self.ctx._check(self.ctx.lib.wg_preview_stage2_run_batch(self.ctx.h, self.h, mem, _ptr(delta_zmp_xy), _ptr(com_stage1),
                                                                 _ptr(state2), _ptr(com_final_out), _ptr(dzmp_out)))

    def destroy(self):
        if self.h:
            self.ctx.lib.wg_preview_plan_destroy(self.h)
            self.h = None
