"""ctypes binding of the C ABI declared in include/walkgen_b200.h.

This module is *plumbing*: it loads ``libwalkgen_b200.so`` (built in-tree by
``jrl_walkgen_b200/csrc/Makefile``) and declares argument types.  It never falls back to a
CPU implementation: if the library is missing, or no CUDA device is present when a context
is requested, it raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libwalkgen_b200.so")

WG_OK = 0
WG_ERR_NO_DEVICE = -1
WG_ERR_CUDA = -2
WG_ERR_INVALID = -3
WG_ERR_ALLOC = -4
WG_ERR_NOT_READY = -5
WG_ERR_WINDOW = -6
WG_MEM_HOST = 0
WG_MEM_DEVICE = 1
WG_PREVIEW_MAX_NL = 2048
MODE_WITH_INITIALPOS = 0
MODE_WITHOUT_INITIALPOS = 1

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)
c_i64_p = C.POINTER(C.c_int64)


class WalkgenError(RuntimeError):
    def __init__(self, code, msg=""):
        super().__init__(f"walkgen_b200 error {code}: {msg}")
        self.code = code


class PreviewGains(C.Structure):
    """Mirror of wg_preview_gains_t."""
    _fields_ = [
        ("A", C.c_double * 9),
        ("B", C.c_double * 3),
        ("C", C.c_double * 3),
        ("Kx", C.c_double * 3),
        ("Ks", C.c_double),
        ("T", C.c_double),
        ("preview_time", C.c_double),
        ("zc", C.c_double),
        ("mode", C.c_int),
        ("NL", C.c_int),
        ("F", C.c_double * WG_PREVIEW_MAX_NL),
    ]


class HerdtParams(C.Structure):
    """Mirror of wg_herdt_params."""
    _fields_ = [("T", C.c_double), ("com_height", C.c_double), ("w_jerk", C.c_double), ("w_vel", C.c_double),
                ("w_cop", C.c_double), ("cop_half_x", C.c_double), ("cop_half_y", C.c_double),
                ("ds_feet_distance", C.c_double), ("foot_hull_x", C.c_double * 5), ("foot_hull_y", C.c_double * 5),
                ("lipm_T", C.c_double)]


class HerdtMpcParams(C.Structure):
    """Mirror of wg_herdt_mpc_params."""
    _fields_ = [("Ts", C.c_double), ("time_buffer", C.c_double), ("step_period", C.c_double),
                ("ds_period", C.c_double), ("dsss_period", C.c_double), ("t_single", C.c_double),
                ("t_double", C.c_double), ("step_height", C.c_double), ("hip_lower", C.c_double * 2),
                ("hip_upper", C.c_double * 2), ("foot_vel_limit", C.c_double), ("hip_acc_limit", C.c_double),
                ("feet_cross_limit", C.c_double), ("nb_steps_ssds", C.c_int32), ("return_to_centre", C.c_int32),
                ("warm_start", C.c_int32), ("reserved", C.c_int32)]


class PldpBatch(C.Structure):
    """Mirror of wg_pldp_batch."""
    _fields_ = [("D", C.c_void_p), ("m", C.c_void_p), ("DPu", C.c_void_p), ("dpu_stride", C.c_longlong),
                ("DPx", C.c_void_p), ("dpx_stride", C.c_longlong), ("ZMPRef", C.c_void_p), ("XkYk", C.c_void_p),
                ("X", C.c_void_p), ("similar", C.c_void_p), ("similar_stride", C.c_longlong),
                ("n_removed", C.c_void_p), ("starting", C.c_void_p), ("hot", C.c_void_p), ("hot_start", C.c_int32),
                ("max_iterations", C.c_int32), ("info", C.c_void_p)]


class MultiStats(C.Structure):
    """Mirror of wg_multi_stats."""
    _fields_ = [("instances", C.c_longlong), ("periods", C.c_longlong), ("seconds", C.c_double), ("qp_solves", C.c_double),
                ("failures", C.c_double), ("iterations", C.c_double), ("still_online", C.c_double), ("devices", C.c_int32),
                ("reduced_by_nccl", C.c_int32), ("nccl_version", C.c_int32), ("reserved", C.c_int32),
                ("device_ms", C.c_float * 16), ("device_instances", C.c_longlong * 16), ("device_launches", C.c_longlong * 16)]


class QldBatch(C.Structure):
    """Mirror of wg_qld_batch."""
    _fields_ = [("n", C.c_int32), ("nmax", C.c_int32), ("mmax", C.c_int32), ("shared_hessian", C.c_int32),
                ("m", C.c_void_p), ("me", C.c_void_p), ("C", C.c_void_p), ("d", C.c_void_p), ("A", C.c_void_p),
                ("a_stride", C.c_longlong), ("b", C.c_void_p), ("b_stride", C.c_longlong), ("xl", C.c_void_p),
                ("xu", C.c_void_p), ("x", C.c_void_p), ("u", C.c_void_p), ("u_stride", C.c_longlong),
                ("ifail", C.c_void_p), ("iterations", C.c_void_p), ("eps", C.c_double)]


class WieberParams(C.Structure):
    """Mirror of wg_wieber_params."""
    _fields_ = [("T", C.c_double), ("sampling_period", C.c_double), ("com_height", C.c_double), ("alpha", C.c_double),
                ("beta", C.c_double), ("constraint_x", C.c_double), ("constraint_y", C.c_double),
                ("sole_length", C.c_double), ("sole_width", C.c_double), ("qld_eps", C.c_double), ("N", C.c_int32),
                ("materialize_pu", C.c_int32)]


class ZmpDiscParams(C.Structure):
    """Mirror of wg_zmpdisc_params."""
    _fields_ = [("sampling_period", C.c_double), ("preview_time", C.c_double), ("t_single", C.c_double),
                ("t_double", C.c_double), ("step_height", C.c_double), ("omega", C.c_double),
                ("modulation", C.c_double), ("zmp_neutral", C.c_double * 2), ("zmp_shift", C.c_double * 4),
                ("foot_b", C.c_double), ("foot_h", C.c_double), ("foot_f", C.c_double), ("filter_time", C.c_double)]


class DimitrovParams(C.Structure):
    """Mirror of wg_dimitrov_params."""
    _fields_ = [("T", C.c_double), ("sampling_period", C.c_double), ("com_height", C.c_double), ("alpha", C.c_double),
                ("beta", C.c_double), ("constraint_x", C.c_double), ("constraint_y", C.c_double),
                ("sole_length", C.c_double), ("sole_width", C.c_double), ("max_iterations", C.c_int32),
                ("cold_restart", C.c_int32), ("merge_duplicate_rows", C.c_int32), ("reserved", C.c_int32)]


def dimitrov_dtypes():
    """numpy mirrors of wg_lci (272 B) and wg_dimitrov_period (224 B)."""
    np = _np()
    lci = np.dtype([("A", "f8", (8, 2)), ("B", "f8", 8), ("center", "f8", 2), ("t_start", "f8"), ("t_end", "f8"),
                    ("rows", "i4"), ("first_sample", "i4"), ("state", "i4"), ("rc", "i4"), ("similar", "i4", 8)])
    period = np.dtype([("t_start", "f8"), ("xk", "f8", 6), ("jerk_x", "f8"), ("jerk_y", "f8"), ("m", "i4"),
                       ("n_first", "i4"), ("rc", "i4"), ("status", "i4"), ("iterations", "i4"), ("n_active", "i4"),
                       ("active", "i4", 32)])
    assert lci.itemsize == 272 and period.itemsize == 224
    return lci, period


def kajita_dtypes():
    """numpy mirrors of wg_rel_step (48 B) and wg_foot_sample (48 B)."""
    np = _np()
    step = np.dtype([("sx", "f8"), ("sy", "f8"), ("theta", "f8"), ("ss_time", "f8"), ("ds_time", "f8"),
                     ("step_type", "i4"), ("reserved", "i4")])
    foot = np.dtype([("x", "f8"), ("y", "f8"), ("z", "f8"), ("theta", "f8"), ("omega", "f8"), ("omega2", "f8")])
    assert step.itemsize == 48 and foot.itemsize == 48
    return step, foot


def kajita_stream_walk_dtype():
    """numpy mirror of wg_kajita_stream_walk (576 B): one whole walk of wg_kajita_stream, its carry rows apart."""
    np = _np()
    step, foot = kajita_dtypes()
    d = np.dtype([("support", "f8", 6), ("prev_support", "f8", 2), ("left", foot), ("right", foot), ("zmp_theta", "f8"),
                  ("samples_emitted", "i8"), ("final0", "f8", 2), ("last", step), ("hist", "f8", (16, 2)),
                  ("preview_state", "f8", 8), ("steps_previewed", "i8"), ("open", "i4"), ("pad_", "i4")])
    assert d.itemsize == 576 and d.fields["hist"][1] == 240 and d.fields["preview_state"][1] == 496
    return d


def pldp_dtypes():
    """numpy mirrors of wg_pldp_state (392 B) and wg_pldp_info (144 B)."""
    np = _np()
    state = np.dtype([("prev_zmp", "f8", 32), ("prev_active", "i4", 32), ("n_prev", "i4"), ("pad_", "i4")])
    info = np.dtype([("rc", "i4"), ("status", "i4"), ("iterations", "i4"), ("n_active", "i4"), ("active", "i4", 32)])
    assert state.itemsize == 392 and info.itemsize == 144
    return state, info


KAJITA_ONLINE_CHUNK = 160
WG_KAJITA_PUSH = 1
WG_KAJITA_STANDARD = 2
WG_KAJITA_STOP = 4


def kajita_online_dtypes():
    """numpy mirrors of wg_kajita_tick (224 B) and wg_kajita_command (64 B)."""
    np = _np()
    step, foot = kajita_dtypes()
    tick = np.dtype([("com_x", "f8", 3), ("com_y", "f8", 3), ("com_z", "f8"), ("com_yaw", "f8"), ("zmp_px", "f8"),
                     ("zmp_py", "f8"), ("zmp_theta", "f8"), ("zmp_time", "f8"), ("zmp_out", "f8", 2), ("left", foot),
                     ("right", foot), ("step_type", "i4", 3), ("pad_", "i4")])
    cmd = np.dtype([("step", step), ("flags", "i4"), ("pad_", "i4", 3)])
    assert tick.itemsize == 224 and cmd.itemsize == 64
    return tick, cmd


def kajita_online_walk_dtype():
    """numpy mirror of wg_kajita_online_walk (624 B): one whole walk of wg_kajita_online, its carry, queue and stack apart."""
    np = _np()
    d = np.dtype([("stream", kajita_stream_walk_dtype()), ("popped", "i8"), ("clock", "f8"), ("keep", "i4"), ("running", "i4"),
                  ("online", "i4"), ("transition", "i4"), ("stacked", "i4"), ("pad_", "i4", 3)])
    assert d.itemsize == 624 and d.fields["popped"][1] == 576
    return d


HERDT_N = 16
HERDT_TICKS_PER_STEP = 20
HERDT_MAX_VARS = 36
HERDT_MAX_ROWS = 75


def _np():
    import numpy as np
    return np


def herdt_dtypes():
    """numpy mirrors of wg_herdt_qp_input (784 B) and wg_herdt_qp_output (960 B)."""
    np = _np()
    N = HERDT_N
    qin = np.dtype([
        ("com_x", "f8", 3), ("com_y", "f8", 3), ("ref_x", "f8", N), ("ref_y", "f8", N),
        ("sup_x", "f8", N + 1), ("sup_y", "f8", N + 1), ("sup_yaw", "f8", N + 1),
        ("sup_foot", "i1", N + 1), ("sup_phase", "i1", N + 1), ("sup_step", "i1", N + 1),
        ("sup_changed", "i1", N + 1), ("pad_", "i1", 4)])
    qout = np.dtype([
        ("x", "f8", HERDT_MAX_VARS), ("lagr", "f8", HERDT_MAX_ROWS + 1), ("com_next_x", "f8", 3),
        ("com_next_y", "f8", 3), ("n_vars", "i4"), ("n_rows", "i4"), ("fail", "i4"), ("iterations", "i4")])
    assert qin.itemsize == 784 and qout.itemsize == 960
    return qin, qout


def preview_gains_head_dtype():
    """numpy mirror of wg_preview_gains_head (184 B)."""
    np = _np()
    d = np.dtype([("A", "f8", 9), ("B", "f8", 3), ("C", "f8", 3), ("Kx", "f8", 3), ("Ks", "f8"), ("T", "f8"),
                  ("preview_time", "f8"), ("zc", "f8"), ("mode", "i4"), ("NL", "i4")])
    assert d.itemsize == 184
    return d


def herdt_active_set_dtype():
    """numpy mirror of wg_herdt_active_set (48 B)."""
    np = _np()
    d = np.dtype([("rows", "i1", 40), ("n", "i1"), ("step_pi", "i1", 2), ("pad_", "i1", 5)])
    assert d.itemsize == 48
    return d


def herdt_mpc_dtypes():
    """numpy mirrors of wg_herdt_foot_sample, wg_herdt_tick (256 B), wg_herdt_mpc_state, wg_herdt_mpc_step (144 B)."""
    np = _np()
    foot = np.dtype([("x", "f8"), ("y", "f8"), ("z", "f8"), ("theta", "f8"), ("dx", "f8"), ("dy", "f8"),
                     ("dz", "f8"), ("dtheta", "f8"), ("ddx", "f8"), ("ddy", "f8")])
    tick = np.dtype([("com_x", "f8", 3), ("com_y", "f8", 3), ("com_z", "f8"), ("yaw", "f8"), ("dyaw", "f8"),
                     ("zmp_x", "f8"), ("zmp_y", "f8"), ("pad_", "f8"), ("left", foot), ("right", foot)])
    state = np.dtype([
        ("clock", "f8"), ("upper_time_limit", "f8"), ("time_to_stop", "f8"), ("new_ref", "f8", 3), ("ref", "f8", 3),
        ("com_x", "f8", 3), ("com_y", "f8", 3), ("com_height", "f8"), ("trunk_yaw", "f8", 3),
        ("trunk_t_yaw", "f8", 2), ("support_time_passed", "f8"), ("sup_time_limit", "f8"),
        ("sup_start_time", "f8"), ("sup_x", "f8"), ("sup_y", "f8"), ("sup_yaw", "f8"), ("poly_z", "f8", 5),
        ("com_front", "f8", 6), ("com_back", "f8", 11), ("foot", foot, (2, 3)),
        ("sup_phase", "i4"), ("sup_foot", "i4"), ("sup_steps_left", "i4"), ("sup_step_number", "i4"),
        ("sup_nb_instants", "i4"), ("sup_changed", "i4"), ("in_translation", "i4"), ("in_rotation", "i4"),
        ("post_rotation", "i4"), ("steps_after_rotation", "i4"), ("fsm_support_foot", "i4"),
        ("online_mode", "i4"), ("ending_phase", "i4"), ("running", "i4"), ("nb_steps_ssds", "i4"),
        ("qp_count", "i4"), ("fail_count", "i4"), ("last_fail", "i4"), ("iterations_total", "i8"),
        ("warm", herdt_active_set_dtype())])
    step = np.dtype([("time", "f8"), ("com_x", "f8", 3), ("com_y", "f8", 3), ("jerk_x", "f8"), ("jerk_y", "f8"),
                     ("next_foot_x", "f8"), ("next_foot_y", "f8"), ("sup_x", "f8"), ("sup_y", "f8"),
                     ("sup_yaw", "f8"), ("sup_foot", "i4"), ("sup_phase", "i4"), ("n_prw_steps", "i4"),
                     ("fail", "i4"), ("iterations", "i4"), ("n_active", "i4"), ("pad_", "i4", 2)])
    assert foot.itemsize == 80 and tick.itemsize == 256 and step.itemsize == 144 and state.itemsize == 1000
    return foot, tick, state, step


HERDT_ONLINE_QUEUE = 29
WG_CMD_VEL = 1
WG_CMD_STOP = 2


def herdt_command_dtype():
    """numpy mirror of wg_herdt_command (32 B)."""
    np = _np()
    d = np.dtype([("vel", "f8", 3), ("flags", "i4"), ("pad_", "i4")])
    assert d.itemsize == 32
    return d


def herdt_online_robot_dtype():
    """numpy mirror of wg_herdt_online_robot (8448 B): one whole robot of wg_herdt_online, deques front first."""
    np = _np()
    _, tick, state, _ = herdt_mpc_dtypes()
    d = np.dtype([("rows", tick, (HERDT_ONLINE_QUEUE,)), ("state", state), ("count", "i4"), ("running", "i4"),
                  ("pad_", "i4", 4)])
    assert d.itemsize == 8448 and d.fields["rows"][1] == 0
    return d


def herdt_plan_dtype():
    """numpy mirror of wg_herdt_plan (1888 B): the QP of one firing robot of wg_herdt_online, expanded over its horizon."""
    np = _np()
    N = HERDT_N
    d = np.dtype([("time", "f8"), ("com_x", "f8", 3), ("com_y", "f8", 3), ("jerk_x", "f8", N), ("jerk_y", "f8", N),
                  ("prw_com_x", "f8", (N, 3)), ("prw_com_y", "f8", (N, 3)), ("prw_cop_x", "f8", N), ("prw_cop_y", "f8", N),
                  ("sup_x", "f8", N + 1), ("sup_y", "f8", N + 1), ("sup_yaw", "f8", N + 1),
                  ("step_x", "f8", 2), ("step_y", "f8", 2), ("step_yaw", "f8", 2),
                  ("sup_foot", "i1", N + 1), ("sup_phase", "i1", N + 1), ("sup_step", "i1", N + 1),
                  ("sup_changed", "i1", N + 1), ("step_sample", "i1", 2), ("step_foot", "i1", 2),
                  ("n_steps", "i4"), ("fail", "i4"), ("iterations", "i4"), ("qp_count", "i4"), ("pad_", "i4", 2)])
    assert d.itemsize == 1888
    return d


# name -> (restype, argtypes); also the list checked against include/walkgen_b200.h by the tests
SIGNATURES = {
    "wg_version": (C.c_int, []),
    "wg_device_count": (C.c_int, []),
    "wg_ctx_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "wg_ctx_destroy": (C.c_int, [C.c_void_p]),
    "wg_sync": (C.c_int, [C.c_void_p]),
    "wg_last_error": (C.c_char_p, [C.c_void_p]),
    "wg_ctx_stream": (C.c_void_p, [C.c_void_p]),
    "wg_malloc_device": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "wg_free_device": (C.c_int, [C.c_void_p, C.c_void_p]),
    "wg_malloc_pinned": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "wg_free_pinned": (C.c_int, [C.c_void_p, C.c_void_p]),
    "wg_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "wg_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "wg_memset_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t]),
    "wg_timer_start": (C.c_int, [C.c_void_p]),
    "wg_timer_stop_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "wg_launch_count": (C.c_longlong, [C.c_void_p]),
    "wg_launch_count_reset": (None, [C.c_void_p]),
    "wg_prof_begin": (C.c_int, [C.c_void_p, C.c_int]),
    "wg_prof_end": (C.c_int, [C.c_void_p]),
    "wg_prof_get": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_longlong), c_double_p]),
    "wg_measure_fp64_peak": (C.c_int, [C.c_void_p, c_double_p]),
    "wg_multi_create": (C.c_int, [C.c_ulonglong, C.POINTER(C.c_void_p)]),
    "wg_multi_destroy": (C.c_int, [C.c_void_p]),
    "wg_multi_size": (C.c_int, [C.c_void_p]),
    "wg_multi_ctx": (C.c_void_p, [C.c_void_p, C.c_int]),
    "wg_multi_nccl_version": (C.c_int, [C.c_void_p]),
    "wg_multi_last_error": (C.c_char_p, [C.c_void_p]),
    "wg_multi_herdt_set_params": (C.c_int, [C.c_void_p, C.POINTER(HerdtParams), C.POINTER(HerdtMpcParams)]),
    "wg_multi_herdt_mpc_sweep": (C.c_int, [C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                           C.POINTER(MultiStats)]),
    "wg_preview_gains": (C.c_int, [C.c_double, C.c_double, C.c_double, C.c_int, C.POINTER(PreviewGains)]),
    "wg_preview_gains_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                         C.c_longlong]),
    "wg_preview_set_gains": (C.c_int, [C.c_void_p, C.POINTER(PreviewGains)]),
    "wg_preview_sum_fit": (C.c_double, [C.POINTER(PreviewGains)]),
    "wg_preview_set_sum_mode": (C.c_int, [C.c_void_p, C.c_int]),
    "wg_preview_set_cta_shape": (C.c_int, [C.c_void_p, C.c_int]),
    "wg_preview_sum_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_double)]),
    "wg_preview_plan_create": (C.c_int, [C.c_void_p, C.c_int, c_i64_p, C.POINTER(C.c_void_p)]),
    "wg_preview_plan_destroy": (C.c_int, [C.c_void_p]),
    "wg_preview_plan_total_steps": (C.c_int64, [C.c_void_p]),
    "wg_preview_plan_total_samples": (C.c_int64, [C.c_void_p]),
    "wg_preview_run_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_int]),
    "wg_preview_run_batch_pos": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "wg_preview_delta_zmp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_preview_stage2_run_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p]),
    "wg_preview_one_iteration": (C.c_int, [C.c_void_p, c_double_p, c_double_p, c_double_p, c_double_p,
                                           c_double_p, C.c_int, c_double_p, c_double_p, C.c_int]),
    "wg_herdt_default_params": (None, [C.c_double, C.c_double, C.POINTER(HerdtParams)]),
    "wg_herdt_set_params": (C.c_int, [C.c_void_p, C.POINTER(HerdtParams)]),
    "wg_herdt_qp_solve_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "wg_herdt_qp_solve_batch_warm": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                               C.c_void_p]),
    "wg_pldp_set_constants": (C.c_int, [C.c_void_p, C.c_int, c_double_p, c_double_p, c_double_p]),
    "wg_pldp_solve_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(PldpBatch)]),
    "wg_pldp_solve_batch_ranked": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(PldpBatch), C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_longlong]),
    "wg_optcholesky_add_rows_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                                C.c_void_p, C.c_longlong, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                C.c_void_p, C.c_longlong]),
    "wg_optcholesky_full_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_int]),
    "wg_qld_set_shared_hessian": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_double]),
    "wg_qld_shared_boost": (C.c_double, [C.c_void_p]),
    "wg_qld_diagonal_boost": (C.c_double, [C.c_int, C.c_int, C.c_void_p, C.c_double]),
    "wg_qld_solve_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(QldBatch)]),
    "wg_qld_solve_batch_ranked": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(QldBatch), C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_longlong, C.c_void_p, C.c_int]),
    "wg_wieber_default_params": (None, [C.POINTER(WieberParams)]),
    "wg_wieber_set_params": (C.c_int, [C.c_void_p, C.POINTER(WieberParams)]),
    "wg_wieber_period_count": (C.c_int64, [C.POINTER(WieberParams), C.c_int64]),
    "wg_wieber_run_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_zmpdisc_default_params": (None, [C.POINTER(ZmpDiscParams)]),
    "wg_steps_support_foot": (C.c_int, [C.c_void_p, C.c_int, c_int_p, C.c_int, C.c_double, C.c_double]),
    "wg_steps_arc": (C.c_int, [C.c_void_p, C.c_int, c_int_p, C.c_double, C.c_double, C.c_double, C.c_int, C.c_double,
                               C.c_double, c_int_p]),
    "wg_steps_last_support": (C.c_int, [C.c_void_p, C.c_int, c_int_p, C.c_int, C.c_double, C.c_double]),
    "wg_zmpdisc_sample_count": (C.c_int64, [C.POINTER(ZmpDiscParams), C.c_int, C.c_void_p]),
    "wg_kajita_plan_create": (C.c_int, [C.c_void_p, C.POINTER(ZmpDiscParams), C.c_int, c_i64_p, C.c_void_p, C.c_void_p,
                                        C.POINTER(C.c_void_p)]),
    "wg_kajita_plan_destroy": (C.c_int, [C.c_void_p]),
    "wg_kajita_plan_sample_offsets": (c_i64_p, [C.c_void_p]),
    "wg_kajita_plan_total_samples": (C.c_int64, [C.c_void_p]),
    "wg_kajita_plan_total_steps": (C.c_int64, [C.c_void_p]),
    "wg_kajita_plan_set_steps": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_zmpdisc_run_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p]),
    "wg_kajita_run_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_int]),
    "wg_kajita_stream_create": (C.c_int, [C.c_void_p, C.POINTER(ZmpDiscParams), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "wg_kajita_stream_destroy": (C.c_int, [C.c_void_p]),
    "wg_kajita_stream_append": (C.c_int, [C.c_void_p, c_i64_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_kajita_stream_sample_offsets": (c_i64_p, [C.c_void_p]),
    "wg_kajita_stream_com_offsets": (c_i64_p, [C.c_void_p]),
    "wg_kajita_stream_com_counts": (c_i64_p, [C.c_void_p]),
    "wg_kajita_stream_run": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_int]),
    "wg_kajita_stream_state": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_kajita_stream_carry_rows": (C.c_int, [C.c_void_p]),
    "wg_kajita_stream_save": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_kajita_stream_restore": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_kajita_stream_copy": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_kajita_online_create": (C.c_int, [C.c_void_p, C.POINTER(ZmpDiscParams), C.c_int, C.c_double, C.c_double,
                                          C.POINTER(C.c_void_p)]),
    "wg_kajita_online_destroy": (C.c_int, [C.c_void_p]),
    "wg_kajita_online_ring_rows": (C.c_int, [C.c_void_p]),
    "wg_kajita_online_start": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, c_i64_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_kajita_online_tick": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_kajita_online_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_kajita_online_carry_rows": (C.c_int, [C.c_void_p]),
    "wg_kajita_online_save": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "wg_kajita_online_restore": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_int64]),
    "wg_kajita_online_copy": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_dimitrov_default_params": (None, [C.POINTER(DimitrovParams)]),
    "wg_dimitrov_set_params": (C.c_int, [C.c_void_p, C.POINTER(DimitrovParams)] + [C.c_void_p] * 6),
    "wg_dimitrov_period_count": (C.c_int64, [C.POINTER(DimitrovParams), C.c_int64]),
    "wg_convex_hull_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_fcals_build_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_i64_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       c_i64_p, C.c_void_p, C.c_void_p]),
    "wg_dimitrov_run_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, c_i64_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_herdt_mpc_default_params": (None, [C.POINTER(HerdtMpcParams)]),
    "wg_herdt_mpc_set_params": (C.c_int, [C.c_void_p, C.POINTER(HerdtMpcParams)]),
    "wg_herdt_mpc_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "wg_herdt_mpc_init15": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "wg_herdt_mpc_stats": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "wg_herdt_mpc_run_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "wg_herdt_online_create": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "wg_herdt_online_destroy": (C.c_int, [C.c_void_p]),
    "wg_herdt_online_start": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "wg_herdt_online_tick": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "wg_herdt_online_states": (C.c_void_p, [C.c_void_p]),
    "wg_herdt_online_tick_plan": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p]),
    "wg_herdt_online_save": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "wg_herdt_online_restore": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "wg_herdt_online_copy": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
}

_lib = None


def load():
    """Load the product library; raise (never fall back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise WalkgenError(
            WG_ERR_NO_DEVICE,
            f"{LIB_PATH} not built - run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means the ABI header and library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
