/* walkgen_b200.h - C ABI of the B200-native batched ZMP pattern-generation backend.
 *
 * This is the drop-in boundary for the jrl-walkgen hot path (SURVEY.md section 8b).  The reference
 * has no C ABI of its own apart from ql0001_ (src/Mathematics/qld.hh:27-31); every entry point below
 * names the reference interface it replaces.  Conventions:
 *   - plain pointers and sizes only; no C++/torch types cross this boundary;
 *   - every function returns 0 (WG_OK) or a negative wg_status; none throws or calls exit()
 *     (the reference LTHROWs / exit(0)s on these paths: PreviewControl.cpp:341-344, :394-399,
 *     PLDPSolver.cpp:822-828);
 *   - `mem` says where the *bulk* buffers of a call live: WG_MEM_HOST (the library stages them
 *     through the context's stream: H2D, kernels, D2H) or WG_MEM_DEVICE (used in place, no copies; device arrays must be
 *     16-byte aligned - anything cudaMalloc / wg_malloc returns is -, the preview entries refuse others with WG_ERR_INVALID).
 *     Small metadata arrays documented as "host" are always host pointers;
 *   - calls are asynchronous on the context's CUDA stream when mem == WG_MEM_DEVICE; call wg_sync()
 *     before reading results.  With WG_MEM_HOST the call returns after the D2H copy completed;
 *   - all arithmetic is FP64 (the reference is double throughout);
 *   - there is NO CPU fallback: without a CUDA device wg_ctx_create fails with WG_ERR_NO_DEVICE.
 */
#ifndef WALKGEN_B200_H
#define WALKGEN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum wg_status {
  WG_OK = 0,
  WG_ERR_NO_DEVICE = -1,   /* no CUDA device / driver: the product never falls back to the CPU */
  WG_ERR_CUDA = -2,        /* a CUDA runtime call failed; see wg_last_error()                     */
  WG_ERR_INVALID = -3,     /* bad argument                                                        */
  WG_ERR_ALLOC = -4,
  WG_ERR_NOT_READY = -5,   /* e.g. preview gains not set                                          */
  WG_ERR_WINDOW = -6       /* fewer ZMP samples than the preview window (PreviewControl.cpp:341)  */
} wg_status;

enum { WG_MEM_HOST = 0, WG_MEM_DEVICE = 1 };

typedef struct wg_ctx wg_ctx;

/* ------------------------------------------------------------------------------------------------
 * Context, memory, synchronisation
 * ---------------------------------------------------------------------------------------------- */
int wg_version(void);                               /* (major<<16)|(minor<<8)|patch                */
int wg_device_count(void);                          /* 0 when no usable CUDA device                */
int wg_ctx_create(int device, wg_ctx **out);        /* one context per GPU / per process rank      */
int wg_ctx_destroy(wg_ctx *ctx);
int wg_sync(wg_ctx *ctx);                           /* cudaStreamSynchronize on the context stream */
const char *wg_last_error(wg_ctx *ctx);             /* message of the last failure (never NULL)    */
void *wg_ctx_stream(wg_ctx *ctx);                   /* the cudaStream_t, for callers that time it  */
int wg_malloc_device(wg_ctx *ctx, size_t bytes, void **out);
int wg_free_device(wg_ctx *ctx, void *p);
int wg_malloc_pinned(wg_ctx *ctx, size_t bytes, void **out);
int wg_free_pinned(wg_ctx *ctx, void *p);
int wg_memcpy_h2d(wg_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);  /* async */
int wg_memcpy_d2h(wg_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);  /* async */
int wg_memset_device(wg_ctx *ctx, void *dst_dev, int value, size_t bytes);          /* async */
/* CUDA-event stopwatch on the context stream (for bench.py; torch events cannot see this stream). */
int wg_timer_start(wg_ctx *ctx);
int wg_timer_stop_ms(wg_ctx *ctx, float *ms);       /* records, synchronises, returns elapsed ms   */
/* Number of kernels this library launched on this context since creation / last reset. */
long long wg_launch_count(wg_ctx *ctx);
void wg_launch_count_reset(wg_ctx *ctx);
/* Per-kernel CUDA-event profiler on the context stream.  Between wg_prof_begin(capacity = max number of
 * kernel launches to record) and wg_prof_end every kernel this library launches is bracketed by an event
 * pair; wg_prof_get returns the launch count and the summed duration of one kernel id:
 *   2 Herdt QP solve, 3 Herdt closed-loop periods, 4 PLDP solve, 5 OptCholesky, 6 preview (fused FIR + scan),
 *   7 ZMPDiscretization, 8 support polygons (FCALS / convex hull), 9 Dimitrov receding-horizon loop, 10 dense QP (qld),
 *   11 Wieber2006 generator (assembly + interpolation kernels). */
int wg_prof_begin(wg_ctx *ctx, int capacity);
int wg_prof_end(wg_ctx *ctx);                        /* synchronises the stream and accumulates      */
int wg_prof_get(wg_ctx *ctx, int kernel_id, long long *launches, double *total_ms);
/* FP64 FMA peak micro-benchmark (register-resident DFMA chains on every SM): TFLOP/s. */
int wg_measure_fp64_peak(wg_ctx *ctx, double *tflops);

/* ------------------------------------------------------------------------------------------------
 * Several GPUs from one process (SURVEY 8e).  The instances of this path are independent: a sharded run deals instance i to
 * device i mod G, every device runs the same kernel sequence on its share from its own host thread, no collective on the data
 * path; the per-device statistics are all-reduced ONCE over NCCL at the end (ncclCommInitAll communicators, libnccl.so.2 bound
 * at run time with dlopen; WG_NCCL_LIB overrides the name).  Without NCCL the statistics are summed on the host and
 * wg_multi_stats::reduced_by_nccl is 0.  (One process per GPU over torch.distributed, as bench.py --gpus N runs it, needs none
 * of this: every rank simply creates its own wg_ctx.)
 * ---------------------------------------------------------------------------------------------- */
typedef struct wg_multi wg_multi;
int wg_multi_create(unsigned long long device_mask, wg_multi **out);   /* bit d selects device d; 0 = every visible device */
int wg_multi_destroy(wg_multi *m);
int wg_multi_size(const wg_multi *m);                                   /* G                                             */
wg_ctx *wg_multi_ctx(wg_multi *m, int k);                               /* the context of the k-th selected device       */
int wg_multi_nccl_version(const wg_multi *m);                           /* e.g. 22703, 0 when NCCL is not in use          */
const char *wg_multi_last_error(const wg_multi *m);

typedef struct wg_multi_stats {
  long long instances, periods;
  double seconds;                 /* CUDA-event time of the slowest device (MAX all-reduce)                               */
  double qp_solves, failures, iterations, still_online;   /* SUM all-reduce over the devices                              */
  int32_t devices, reduced_by_nccl, nccl_version, reserved;
  float device_ms[16];            /* per device: time, share and kernel launches                                          */
  long long device_instances[16], device_launches[16];
} wg_multi_stats;

/* struct wg_herdt_params / wg_herdt_mpc_params are declared further down */
struct wg_herdt_params;
struct wg_herdt_mpc_params;
int wg_multi_herdt_set_params(wg_multi *m, const struct wg_herdt_params *hp, const struct wg_herdt_mpc_params *mp);
/* BASELINE configs[4] inside the library: `instances` Herdt2010 closed loops (InitOnLine from init9, constant velocity
 * reference vel_ref [instances][3], HOST array) advanced by `periods` QP periods in launches of `chunk` periods (<= 0: 10),
 * sharded i -> device i mod G, states device resident from start to end. */
int wg_multi_herdt_mpc_sweep(wg_multi *m, long long instances, int periods, int chunk, const double *vel_ref,
                             const double *init9, wg_multi_stats *out);

/* ------------------------------------------------------------------------------------------------
 * Kajita2003 preview control
 *   replaces PreviewControl::ComputeOptimalWeights        (src/PreviewControl/PreviewControl.cpp:198-322)
 *            OptimalControllerSolver::ComputeWeights       (src/PreviewControl/OptimalControllerSolver.cpp:200-352)
 *            PreviewControl::OneIterationOfPreview         (src/PreviewControl/PreviewControl.cpp:324-374)
 *            PreviewControl::OneIterationOfPreview1D (x2)  (src/PreviewControl/PreviewControl.cpp:376-484)
 * ---------------------------------------------------------------------------------------------- */
#define WG_PREVIEW_MAX_NL 2048

enum { WG_PREVIEW_MODE_WITH_INITIALPOS = 0,      /* OptimalControllerSolver.hh:144 */
       WG_PREVIEW_MODE_WITHOUT_INITIALPOS = 1 }; /* OptimalControllerSolver.hh:143 */

typedef struct wg_preview_gains_t {
  double A[9];   /* cart-table state matrix, row-major   (PreviewControl.cpp:204-206) */
  double B[3];   /*                                      (PreviewControl.cpp:208-210) */
  double C[3];   /* zmp = C x, C = [1, 0, -zc/9.81]      (PreviewControl.cpp:212-214) */
  double Kx[3];  /* state feedback                       (PreviewControl.cpp:279-280) */
  double Ks;     /* integral gain                        (PreviewControl.cpp:278)     */
  double T, preview_time, zc;
  int mode;
  int NL;        /* preview window = (int)(preview_time/T) (PreviewControl.cpp:317-319) */
  double F[WG_PREVIEW_MAX_NL];
} wg_preview_gains_t;

/* Host-side Riccati solve (runs once per parameter change, as in the reference).  The reference
 * calls LAPACK dgges_ on the symplectic pencil (Laub); here the same stabilising solution is
 * obtained with the structure-preserving doubling algorithm. */
int wg_preview_gains(double T, double preview_time, double zc, int mode, wg_preview_gains_t *out);

/* The same solve for B parameter sets at once on the device (one thread per set; the reference has a single-instance
 * OptimalControllerSolver only): params [B][3] = (T, preview_time, zc); heads [B]; F [B][f_stride] with f_stride >= the
 * largest NL (entries past NL are left untouched in device memory, zero in host memory).  A set the solve refuses
 * (T <= 0, NL > f_stride, singular pencil) gets NL = 0 and Ks = NaN. */
typedef struct wg_preview_gains_head {
  double A[9], B[3], C[3], Kx[3], Ks;
  double T, preview_time, zc;
  int32_t mode, NL;
} wg_preview_gains_head;              /* 184 bytes */
int wg_preview_gains_batch(wg_ctx *ctx, int mem, int B, const double *params, int mode, wg_preview_gains_head *heads,
                           double *F, long long f_stride);

/* Upload gains to the context (constant memory image used by the kernels). */
int wg_preview_set_gains(wg_ctx *ctx, const wg_preview_gains_t *gains);

/* How the batched kernels evaluate the preview sum  sum_{i<NL} F[i] p[k+i]  of OneIterationOfPreview (PreviewControl.cpp:346-352).
 * The weights OptimalControllerSolver::ComputeWeights produces are F[i] = (1/(R+b'Pb)) b' ((A-bK)')^i P c'Q
 * (OptimalControllerSolver.cpp:323-345), a matrix-geometric sequence, so the sum obeys a stable BACKWARD linear recurrence in k
 * and costs ~70 flop per tick instead of 1280: the batch run becomes HBM bound instead of FP64 bound.  wg_preview_set_gains fits
 * that structure to the table it is given (extended precision); when sum_i |F[i] - fit| <= WG_PREVIEW_REC_TOL * sum_i |F[i]| the
 * recursive kernel is used (AUTO), otherwise - e.g. a table read from a file with few digits - the direct 320-tap sum.  The two
 * differ by the summation order of the same products: ~1e-14 relative on the sum, < 1e-12 m on CoM / ZMP (tests/test_preview*.py).
 *   DIRECT    always the direct sum
 *   RECURSIVE refuse (WG_ERR_INVALID) instead of falling back when the weights do not have the structure
 * wg_preview_sum_info: which of the two the next run uses, and the fit residual (relative; -1: no fit possible). */
enum { WG_PREVIEW_SUM_AUTO = 0, WG_PREVIEW_SUM_DIRECT = 1, WG_PREVIEW_SUM_RECURSIVE = 2 };
#define WG_PREVIEW_REC_TOL 1e-12
double wg_preview_sum_fit(const wg_preview_gains_t *gains);   /* host only: the relative fit residual of a gain set, -1: none */
int wg_preview_set_sum_mode(wg_ctx *ctx, int mode);
int wg_preview_sum_info(wg_ctx *ctx, int *mode_in_use, double *fit_residual);
/* Tuning knob: the CTA shape of the batch kernels.  -1 (default) = chosen per launch from the number of trajectories (the
 * recursive sum runs one warp per trajectory from 1792 trajectories up, four warps per trajectory below that, eight below 768);
 * 0 = 64 threads x 8 CTAs/SM, 1 = 128 x 4, 2 = 32 x 16 (one warp per trajectory), 3 = 256 x 2 (falls back to 1 when the window does not fit).  Results do not depend on it beyond the summation order (1e-14).  The
 * environment variable WG_PREVIEW_SHAPE, read once per process, overrides both. */
int wg_preview_set_cta_shape(wg_ctx *ctx, int shape);

/* A plan describes a ragged batch of B trajectories: trajectory b owns ZMP-reference samples
 * [offsets[b], offsets[b+1]) of a packed array of interleaved (px,py) pairs.  A trajectory of L
 * samples yields L-NL+1 preview steps (step k consumes the window [k, k+NL), exactly what
 * OneIterationOfPreview reads from the FIFO at lindex=k).  offsets is a HOST array of B+1 entries. */
typedef struct wg_preview_plan wg_preview_plan;
int wg_preview_plan_create(wg_ctx *ctx, int B, const int64_t *offsets_host, wg_preview_plan **out);
int wg_preview_plan_destroy(wg_preview_plan *plan);
int64_t wg_preview_plan_total_steps(const wg_preview_plan *plan);   /* sum of (L_b-NL+1)^+ */
int64_t wg_preview_plan_total_samples(const wg_preview_plan *plan); /* offsets[B]           */

/* Run every preview step of every trajectory of the plan.
 *   zmpref_xy : [total_samples][2]  in      ZMP reference (px,py)
 *   state     : [B][8]              in/out  {x, dx, ddx, y, dy, ddy, sxzmp, syzmp}: the arguments
 *                                           x, y, sxzmp, syzmp of OneIterationOfPreview
 *   com_out   : [total_samples][6]  out     row offsets[b]+k = (x,dx,ddx,y,dy,ddy) after step k
 *   zmp_out   : [total_samples][2]  out     row offsets[b]+k = (zmpx2, zmpy2) of step k
 *                                           (rows past a trajectory's last step: left untouched with
 *                                           WG_MEM_DEVICE, zero with WG_MEM_HOST)
 *   simulation: the `Simulation` flag (accumulate sxzmp += zmpref - zmp, PreviewControl.cpp:363-367)
 * com_out / zmp_out may be NULL. */
int wg_preview_run_batch(wg_ctx *ctx, wg_preview_plan *plan, int mem, const double *zmpref_xy,
                         double *state, double *com_out, double *zmp_out, int simulation);

/* Output selection: the same run, writing only the CoM POSITION of every step, com_pos_out [total_samples][2] = (x, y) after
 * step k (rows past a trajectory's last step as in wg_preview_run_batch's zmp_out).  16 bytes per step leave the GPU instead of
 * 64 - the host-buffer path is bound by that traffic.  `state` still receives the full final state. */
int wg_preview_run_batch_pos(wg_ctx *ctx, wg_preview_plan *plan, int mem, const double *zmpref_xy, double *state,
                             double *com_pos_out, int simulation);

/* Second stage of the two-stage scheme (ZMPPreviewControlWithMultiBodyZMP::EvaluateMultiBodyZMP / SecondStageOfControl,
 * src/PreviewControl/ZMPPreviewControlWithMultiBodyZMP.cpp:447-479, :317-376), for callers that own the multibody model:
 *   1. wg_preview_run_batch(simulation = 1) is the first stage: com_out row k = m_PC1x / m_PC1y after tick k;
 *   2. the caller evaluates its robot's multibody ZMP for every first-stage tick (zmp_multibody_xy, same row indexing);
 *   3. wg_preview_delta_zmp forms the stream the reference pushes into m_FIFODeltaZMPPositions:
 *        delta[k] = zmpref[k + 1] - zmp_multibody[k]   (m_FIFOZMPRefPositions[0] AFTER the first stage popped it; the last
 *        sample of a trajectory, which has no successor, gets 0);
 *   4. wg_preview_stage2_run_batch runs the same preview controller on the delta stream (Simulation = true, state2 =
 *      {m_Deltax, m_Deltay, m_sxDeltazmp, m_syDeltazmp}, zero after SetupFirstPhase) and writes
 *        com_final_out row n = com_stage1 row n + (m_Deltax, m_Deltay) after step n   (all three derivatives, :352-356),
 *      the CoM the reference hands back NL ticks after the first stage computed it (step n consumes delta[n, n + NL)).
 *      dzmp_out (or NULL) receives Deltazmpx2 / Deltazmpy2.  Rows n > L - 2 NL + 1 of a trajectory of L samples are computed
 *      from delta rows the first stage never produces (the caller's padding) and have no counterpart in the reference.
 * The reference's own FIFO bookkeeping (Setup skips ZMPRefPositions[NL], :660) lives in the class mirror
 * (jrl_walkgen_b200/host), which feeds these entry points the stream the FIFOs actually hold. */
int wg_preview_delta_zmp(wg_ctx *ctx, wg_preview_plan *plan, int mem, const double *zmpref_xy,
                         const double *zmp_multibody_xy, double *delta_out);
int wg_preview_stage2_run_batch(wg_ctx *ctx, wg_preview_plan *plan, int mem, const double *delta_zmp_xy,
                                const double *com_stage1, double *state2, double *com_final_out, double *dzmp_out);

/* Single-call form of OneIterationOfPreview for the class wrappers (batch of one, one step):
 * host pointers; x[3], y[3], sxzmp, syzmp in/out; window = NL pairs starting at ZMPPositions[lindex]. */
int wg_preview_one_iteration(wg_ctx *ctx, double *x, double *y, double *sxzmp, double *syzmp,
                             const double *window_xy, int n_available, double *zmpx2, double *zmpy2,
                             int simulation);

/* ------------------------------------------------------------------------------------------------
 * Herdt2010 velocity-referenced QP (N = 16 previewed samples of T = 0.1 s)
 *   replaces GeneratorVelRef::build_invariant_part / update_problem / build_constraints
 *                (src/ZMPRefTrajectoryGeneration/generator-vel-ref.cpp:588-674, :285-474, :555-584)
 *            RelativeFeetInequalities::set_vertices / compute_linear_system
 *                (src/Mathematics/relative-feet-inequalities.cpp:186-234, :265-319)
 *            QPProblem::add_term_to / solve          (src/ZMPRefTrajectoryGeneration/qp-problem.cpp:411-547, :246-407)
 *            ql0001_ / ql0002_                       (src/Mathematics/qld.cpp:378-2090)
 *            LinearizedInvertedPendulum2D::Interpolation / OneIteration
 *                (src/PreviewControl/LinearizedInvertedPendulum2D.cpp:157-264)
 * ---------------------------------------------------------------------------------------------- */
#define WG_HERDT_N 16            /* QP_N_, ZMPVelocityReferencedQP.cpp:65                        */
#define WG_HERDT_MAX_STEPS 2     /* previewed steps ns in {0,1,2} for StepPeriod = 8 samples     */
#define WG_HERDT_MAX_VARS (2 * WG_HERDT_N + 2 * WG_HERDT_MAX_STEPS)            /* 36 */
#define WG_HERDT_MAX_ROWS (1 + 4 * WG_HERDT_N + 5 * WG_HERDT_MAX_STEPS)        /* 75: dummy row + CoP + feet */

enum { WG_LEFT = 0, WG_RIGHT = 1 };  /* foot_type_e, privatepgtypes.hh:47-50 */
enum { WG_SS = 0, WG_DS = 1 };       /* PhaseType,   privatepgtypes.hh:65-68 */

/* Generator + robot constants (one set per context). */
typedef struct wg_herdt_params {
  double T;                 /* QP sampling period, 0.1          (ZMPVelocityReferencedQP.cpp:63)   */
  double com_height;        /* QP model height, 0.814           (ZMPVelocityReferencedQP.cpp:103)  */
  double w_jerk;            /* JERK_MIN weight 1e-5             (ZMPVelocityReferencedQP.cpp:118)  */
  double w_vel;             /* INSTANT_VELOCITY weight 1.0      (ZMPVelocityReferencedQP.cpp:116)  */
  double w_cop;             /* COP_CENTERING weight 1e-6        (ZMPVelocityReferencedQP.cpp:117)  */
  double cop_half_x;        /* 0.5*sole_length - SecurityMarginX (FootHalfSize.cpp:62-68)          */
  double cop_half_y;        /* 0.5*sole_width  - SecurityMarginY                                   */
  double ds_feet_distance;  /* DSFeetDistance_ 0.2              (relative-feet-inequalities.cpp:45) */
  double foot_hull_x[5];    /* LeftFPosEdgesX_                  (relative-feet-inequalities.cpp:51) */
  double foot_hull_y[5];    /* LeftFPosEdgesY_ (right = -left)  (relative-feet-inequalities.cpp:52) */
  double lipm_T;            /* control period for the 5 ms interpolation, 0.005                    */
} wg_herdt_params;

/* Defaults of the reference for a sole of (length, width) metres and margins 0.04 m. */
void wg_herdt_default_params(double sole_length, double sole_width, wg_herdt_params *out);

/* Everything GeneratorVelRef reads when it assembles one QP (one instance):
 * IntermedData_->State().CoM, Ref.Global.{X,Y}_vec and Solution_.SupportStates_deq[0..N]. */
typedef struct wg_herdt_qp_input {
  double com_x[3], com_y[3];                       /* (c, dc, ddc) per axis                          */
  double ref_x[WG_HERDT_N], ref_y[WG_HERDT_N];     /* velocity reference in the global frame         */
  double sup_x[WG_HERDT_N + 1];                    /* support_state_t::X   [0] = current, [i] = previewed */
  double sup_y[WG_HERDT_N + 1];                    /* support_state_t::Y                             */
  double sup_yaw[WG_HERDT_N + 1];                  /* support_state_t::Yaw                           */
  int8_t sup_foot[WG_HERDT_N + 1];                 /* WG_LEFT / WG_RIGHT                             */
  int8_t sup_phase[WG_HERDT_N + 1];                /* WG_SS / WG_DS                                  */
  int8_t sup_step[WG_HERDT_N + 1];                 /* support_state_t::StepNumber                    */
  int8_t sup_changed[WG_HERDT_N + 1];              /* support_state_t::StateChanged                  */
  int8_t pad_[4];
} wg_herdt_qp_input;                               /* 784 bytes */

/* solution_t as filled by QPProblem::solve (qp-problem.cpp:281-293) plus the first 0.1 s of CoM/ZMP. */
typedef struct wg_herdt_qp_output {
  double x[WG_HERDT_MAX_VARS];      /* Solution_vec: jerk_x[16], jerk_y[16], foot_x[ns], foot_y[ns]       */
  double lagr[WG_HERDT_MAX_ROWS + 1]; /* ConstrLagr_vec; row 0 is the reference's all-zero dummy row      */
  double com_next_x[3], com_next_y[3]; /* CoM_ after OneIteration(x[0], x[N]) (LIPM2D.cpp:230-264)        */
  int32_t n_vars;                   /* 2N + 2ns                                                           */
  int32_t n_rows;                   /* m_ = 1 + 4N + 5ns (incl. dummy row)                                */
  int32_t fail;                     /* 0 ok (QLD ifail convention: >0 failure)                            */
  int32_t iterations;               /* active-set changes (adds + drops)                                  */
} wg_herdt_qp_output;

/* Optimal active set of one solve, as a warm start for the next solve of the same instance: the 0-based rows (without the
 * dummy row: CoP row 4 i + e of previewed sample i, foot row 4N + 5 s + e of previewed step s) in activation order, and where
 * the previewed steps start, so that a later solve can shift the rows by the samples that left the horizon. */
typedef struct wg_herdt_active_set {
  int8_t rows[40];                  /* -1 padded                                                            */
  int8_t n;                         /* 0: no guess (cold start)                                             */
  int8_t step_pi[2];                /* previewed sample (1..N) at which previewed step 1 / 2 starts, 0 = none */
  int8_t pad_[5];
} wg_herdt_active_set;              /* 48 bytes */

int wg_herdt_set_params(wg_ctx *ctx, const wg_herdt_params *params);

/* Build and solve B independent QPs.  in/out are arrays of B structs (host or device per `mem`). */
int wg_herdt_qp_solve_batch(wg_ctx *ctx, int mem, int B, const wg_herdt_qp_input *in,
                            wg_herdt_qp_output *out);

/* The same solve, warm started.  guess[b] (or NULL) is the active set a solve of the same instance `age` QP periods earlier
 * ended on (age 0: the same QP): its rows are shifted by the samples / steps that left the horizon, taken as equalities all
 * at once, guesses whose multiplier comes out negative are dropped, and the dual active-set iteration continues from that
 * pair.  The QP is strictly convex, so the optimum - x, multipliers, active set - is the one of the cold start; only the
 * path (and `iterations`) changes.  active_out[b] (or NULL; may alias guess) receives the optimal active set. */
int wg_herdt_qp_solve_batch_warm(wg_ctx *ctx, int mem, int B, const wg_herdt_qp_input *in, wg_herdt_qp_output *out,
                                 const wg_herdt_active_set *guess, int age, wg_herdt_active_set *active_out);

/* ------------------------------------------------------------------------------------------------
 * Herdt2010 closed loop: the whole ZMPVelocityReferencedQP::OnLine cycle on the device, batched
 *   replaces ZMPVelocityReferencedQP::InitOnLine / OnLine      (ZMPVelocityReferencedQP.cpp:213-319, :324-458)
 *            SupportFSM::update_vel_reference / set_support_state (src/PreviewControl/SupportFSM.cpp:58-153)
 *            GeneratorVelRef::preview_support_states / compute_global_reference (generator-vel-ref.cpp:71-134, :212-229)
 *            OrientationsPreview::preview_orientations / interpolate_trunk_orientation (OrientationsPreview.cpp:80-418)
 *            LinearizedInvertedPendulum2D::Interpolation / OneIteration (LinearizedInvertedPendulum2D.cpp:157-264)
 *            OnLineFootTrajectoryGeneration::interpolate_feet_positions (OnLineFootTrajectoryGeneration.cpp:51-346)
 *            the 5 ms deques popped by CoMAndFootOnlyStrategy::OneGlobalStepOfControl (CoMAndFootOnlyStrategy.cpp:56-124)
 * One "step" is one QP period (QP_T_ = 0.1 s = 20 control ticks): FSM + orientation preview + QP build and
 * solve + 20 interpolated CoM / ZMP / feet samples.  Every instance carries its own state, so B instances
 * advance independently (different velocity references, phases, stop commands).
 * ---------------------------------------------------------------------------------------------- */
typedef struct wg_herdt_mpc_params {
  double Ts;                /* m_SamplingPeriod 0.005            (ZMPVelocityReferencedQP.cpp:64)  */
  double time_buffer;       /* TimeBuffer_ 0.04                  (:62)                             */
  double step_period;       /* SupportFSM StepPeriod 0.8         (:77)                             */
  double ds_period;         /* DSPeriod 1e9                      (:78)                             */
  double dsss_period;       /* DSSSPeriod 0.8                    (:79)                             */
  double t_single;          /* :singlesupporttime (TestHerdt2010: 0.7)                             */
  double t_double;          /* :doublesupporttime (TestHerdt2010: 0.1)                             */
  double step_height;       /* 0.05                              (rigid-body-system.cpp:66)        */
  double hip_lower[2];      /* hip-yaw joint limits [left, right] (OrientationsPreview.cpp:48-66)  */
  double hip_upper[2];
  double foot_vel_limit;    /* |upperVelocityBound| of the hip yaw joint (:67-68)                  */
  double hip_acc_limit;     /* uaLimitHipYaw_ 0.1                (:71)                             */
  double feet_cross_limit;  /* uLimitFeet_ 5 deg                 (:73)                             */
  int32_t nb_steps_ssds;    /* SupportFSM NbStepsSSDS 2 (:80); :numberstepsbeforestop overrides    */
  int32_t return_to_centre; /* 1: end-of-walk jerk towards the feet centre (:410-421, since 3.1.8);
                               0: always apply the QP jerk (the code the committed datrefs were made with) */
  int32_t warm_start;       /* 1: every QP starts from the previous period's optimal active set, shifted by one sample
                               (same optimum, another path: +8 % closed-loop rate measured); 0 (default): cold start as
                               QLD does                                                                               */
  int32_t reserved;
} wg_herdt_mpc_params;

void wg_herdt_mpc_default_params(wg_herdt_mpc_params *out);

/* One 5 ms foot sample: the fields of FootAbsolutePosition this path writes (pgtypes.hh:141-170).
 * theta in degrees as in the reference; omega/omega2 are identically 0 on this path (:omega 0.0). */
typedef struct wg_herdt_foot_sample {
  double x, y, z, theta;
  double dx, dy, dz, dtheta;
  double ddx, ddy;
} wg_herdt_foot_sample;                /* 80 bytes */

/* One 5 ms output row: what one tick pops from the four deques. */
typedef struct wg_herdt_tick {
  double com_x[3], com_y[3];           /* COMState x[0..2], y[0..2]                                   */
  double com_z, yaw, dyaw;             /* COMState z[0], yaw[0], yaw[1]                               */
  double zmp_x, zmp_y;                 /* ZMPPosition px, py (world frame)                            */
  double pad_;
  wg_herdt_foot_sample left, right;
} wg_herdt_tick;                       /* 256 bytes */

#define WG_HERDT_TICKS_PER_STEP 20     /* QP_T_ / m_SamplingPeriod */

/* Per-instance persistent state of ZMPVelocityReferencedQP and its helpers (plain data; the host may
 * read and edit it between calls, e.g. new_ref for Reference(), ending_phase for :stoppg). */
typedef struct wg_herdt_mpc_state {
  double clock;                        /* PGI m_InternalClock                                         */
  double upper_time_limit;             /* UpperTimeLimitToUpdate_                                     */
  double time_to_stop;                 /* m_TimeToStopOnLineMode                                      */
  double new_ref[3];                   /* NewVelRef_ (dx, dy, dyaw): set by Reference()               */
  double ref[3];                       /* VelRef_.Local after SupportFSM::update_vel_reference        */
  double com_x[3], com_y[3];           /* CoM_ (LIPM state at the QP instants)                        */
  double com_height;                   /* m_ComHeight of the LIPM (start height, NOT the QP's 0.814)  */
  double trunk_yaw[3];                 /* OrientPrw_ TrunkState_.yaw                                  */
  double trunk_t_yaw[2];               /* TrunkStateT_.yaw[0..1]                                      */
  double support_time_passed;          /* OrientationsPreview::SupportTimePassed_                     */
  double sup_time_limit, sup_start_time, sup_x, sup_y, sup_yaw;   /* IntermedData_->SupportState()    */
  double poly_z[5];                    /* swing-height quartic, reset on support change               */
  double com_front[6];                 /* FinalCOMTraj_deq[0]: x[0..2], y[0..2]                       */
  double com_back[11];                 /* the not-yet-emitted last CoM/ZMP sample (wg_herdt_tick[0..10]) */
  wg_herdt_foot_sample foot[2][3];     /* [left,right][deque index 0, size-2, size-1]                 */
  int32_t sup_phase, sup_foot, sup_steps_left, sup_step_number, sup_nb_instants, sup_changed;
  int32_t in_translation, in_rotation, post_rotation, steps_after_rotation, fsm_support_foot;
  int32_t online_mode, ending_phase, running, nb_steps_ssds;
  int32_t qp_count, fail_count, last_fail;
  int64_t iterations_total;            /* active-set changes summed over all QPs of this instance     */
  wg_herdt_active_set warm;            /* optimal active set of the last QP (warm start of the next one, see
                                          wg_herdt_mpc_params::warm_start); n = 0 after InitOnLine        */
} wg_herdt_mpc_state;

/* Summary of one QP period (optional output). */
typedef struct wg_herdt_mpc_step {
  double time;                         /* clock at which the QP was solved                            */
  double com_x[3], com_y[3];           /* CoM_ after the period                                       */
  double jerk_x, jerk_y;               /* applied jerk (Solution_vec[0], [N])                         */
  double next_foot_x, next_foot_y;     /* first previewed foot placement (0 when none)                */
  double sup_x, sup_y, sup_yaw;        /* current support frame                                       */
  int32_t sup_foot, sup_phase, n_prw_steps, fail;
  int32_t iterations, n_active, pad_[2];
} wg_herdt_mpc_step;                   /* 144 bytes */

int wg_herdt_mpc_set_params(wg_ctx *ctx, const wg_herdt_mpc_params *params);

/* InitOnLine for B instances.  init9 = {com x, y, z, left foot x, y, theta(deg), right foot x, y, theta(deg)};
 * instance b reads init9 + b*init_stride (init_stride = 0 broadcasts one start configuration; the array is a
 * HOST pointer).  `states` is host or device memory per `mem`.  The 8 buffered start samples
 * (TimeBuffer_/m_SamplingPeriod) of the deques are implied by the state. */
int wg_herdt_mpc_init(wg_ctx *ctx, int mem, int B, const double *init9, int init_stride,
                      wg_herdt_mpc_state *states);

/* The same for a start that is not at rest: init15 = {com x, dx, ddx, y, dy, ddy, z, trunk yaw (rad), trunk yaw rate,
 * left foot x, y, theta(deg), right foot x, y, theta(deg)} - InitOnLine copies the whole lStartingCOMState into CoM_ and hands it
 * to OrientationsPreview::CurrentTrunkState (ZMPVelocityReferencedQP.cpp:292-301). */
int wg_herdt_mpc_init15(wg_ctx *ctx, int mem, int B, const double *init15, int init_stride, wg_herdt_mpc_state *states);

/* qp_count, fail_count, iterations_total summed over B DEVICE-resident states and the number of instances still on line, into
 * four DEVICE doubles (asynchronous on the context stream): the statistics a sharded run reduces across GPUs. */
int wg_herdt_mpc_stats(wg_ctx *ctx, int B, const wg_herdt_mpc_state *d_states, double *d_out4);

/* Advance every instance by `nsteps` QP periods.
 *   vel_ref : [B][3] or NULL   new (dx, dy, dyaw) written to new_ref before the first period
 *   ticks   : [B][nsteps*20] or NULL  the rows popped at ticks 7+20k .. 26+20k of each period k (the sample a
 *             period inherits at the back of the deques, final only now, then its first 19 new samples)
 *   steps   : [B][nsteps] or NULL     per-period summaries
 *   qp_in   : [B] or NULL             the QP input of each instance's LAST period (workload capture)
 * Instances whose on-line mode ended (:stoppg + preview horizon elapsed) are left untouched.
 * A period is three kernel launches (FSM + QP record, the solver of wg_herdt_qp_solve_batch, interpolation + state update). */
int wg_herdt_mpc_run_batch(wg_ctx *ctx, int mem, int B, int nsteps, wg_herdt_mpc_state *states,
                           const double *vel_ref, wg_herdt_tick *ticks, wg_herdt_mpc_step *steps,
                           wg_herdt_qp_input *qp_in);

/* ------------------------------------------------------------------------------------------------
 * Herdt2010 on-line generator, one 5 ms control tick at a time, for B robots
 *   replaces PatternGeneratorInterface::RunOneStepOfTheControlLoop, Herdt branch (PatternGeneratorInterfacePrivate.cpp:1246-1336):
 *            ZMPVelocityReferencedQP::OnLine (ZMPVelocityReferencedQP.cpp:324-458) and the pop of the four deques by
 *            CoMAndFootOnlyStrategy::OneGlobalStepOfControl (CoMAndFootOnlyStrategy.cpp:56-124);
 *            :HerdtOnline (InitOnLine), :setVelReference (Reference()) and :stoppg between ticks.
 * Every robot keeps its own clock, deques and commands, so robots started at different ticks and commanded at different
 * ticks advance together.  One tick of robot b is what one RunOneStepOfTheControlLoop does for that robot alone:
 *   - its command of this tick is applied (WG_CMD_VEL writes new_ref, WG_CMD_STOP sets ending_phase);
 *   - its clock advances by Ts;
 *   - while on line, the end-of-on-line test runs, and when clock + 1e-5 > upper_time_limit one QP period fires (the
 *     same device code as wg_herdt_mpc_run_batch): the back element of the deques takes the new feet, then the period's
 *     samples 1..19 and the state's com_back / foot[.][2] sample are appended;
 *   - one element is popped into rows[t][b] and running[t][b] = 1; when the deques are empty the robot stops for good
 *     (running[t][b] = 0 from then on, until it is started again).
 * A robot that is not started, or has stopped, is not advanced and ignores its commands: its running entry is 0 and its row
 * is untouched with WG_MEM_DEVICE, zero with WG_MEM_HOST.
 *
 * Memory: the deques of a robot are a ring of WG_HERDT_ONLINE_QUEUE wg_herdt_tick rows in device memory.  A robot holds at
 * most 29 rows before a pop (8 buffered at the start plus 20 at the first tick; 9 + 20 at each later QP instant); a QP
 * instant that would overflow the ring (possible only after the states were edited) stops the robot's on-line mode with
 * last_fail = -1 instead.  Per robot: 7424 B of queue, 1000 B of state, 5120 B of staged period rows, 1760 B of QP records:
 * about 15.3 GB for 10^6 robots.
 * Parameters come from wg_herdt_set_params / wg_herdt_mpc_set_params and are read at tick time; without them start and tick
 * return WG_ERR_NOT_READY.  A tick is four kernel launches whatever number of robots fire; with WG_MEM_DEVICE it does not
 * synchronise, and once its buffers exist it allocates nothing.
 * ---------------------------------------------------------------------------------------------- */
#define WG_HERDT_ONLINE_QUEUE 29
enum { WG_CMD_VEL = 1, WG_CMD_STOP = 2 };

typedef struct wg_herdt_command {      /* one robot, one tick; applied before that tick                          */
  double vel[3];                       /* WG_CMD_VEL: :setVelReference dx dy dyaw (new_ref)                      */
  int32_t flags;                       /* WG_CMD_VEL | WG_CMD_STOP (:stoppg); 0 = no command                     */
  int32_t pad_;
} wg_herdt_command;                    /* 32 bytes */

typedef struct wg_herdt_online wg_herdt_online;
int wg_herdt_online_create(wg_ctx *ctx, int B, wg_herdt_online **out);
int wg_herdt_online_destroy(wg_herdt_online *h);
/* :HerdtOnline for the n robots idx_host[0..n): state as wg_herdt_mpc_init15 (robot idx[i] reads init15_host +
 * i*init_stride; stride 0 broadcasts), deques = the 8 buffered start samples (TimeBuffer_/Ts, the state's com_back and
 * feet), clock restarted at 0.  Robots not listed keep running.  Refused with WG_ERR_INVALID, nothing changed: n < 0,
 * init_stride < 0, an index out of [0, B) or repeated, NULL arrays with n > 0.  Waits for the context stream. */
int wg_herdt_online_start(wg_herdt_online *h, int n, const int32_t *idx_host, const double *init15_host, int init_stride);
/* nticks control ticks for every started robot.  In `mem`, each may be NULL:
 *   commands [nticks][B]   command of robot b before tick t
 *   rows     [nticks][B]   the popped COMState / ZMPPosition / feet
 *   running  [nticks][B]   1 = RunOneStepOfTheControlLoop returned true
 * Refused with WG_ERR_INVALID, nothing changed: nticks < 0 or an unknown mem. */
int wg_herdt_online_tick(wg_herdt_online *h, int mem, int nticks, const wg_herdt_command *commands, wg_herdt_tick *rows,
                         int8_t *running);
/* The B state records in DEVICE memory (plain data, editable between calls as wg_herdt_mpc_run_batch's are). */
wg_herdt_mpc_state *wg_herdt_online_states(wg_herdt_online *h);

/* ------------------------------------------------------------------------------------------------
 * Dimitrov PLDP solver and OptCholesky, batched (QP_N = 16: control vector of 2N = 32 entries)
 *   replaces PLDPSolver::PLDPSolver / SolveProblem / ComputeInitialSolution / ComputeProjectedDescentDirection /
 *            ComputeAlpha / StoreCurrentZMPSolution   (src/Mathematics/PLDPSolver.cpp:56-135, :287-1032)
 *            OptCholesky::AddActiveConstraint(s) / UpdateCholeskyMatrixNormal / UpdateCholeskyMatrixFortran /
 *            ComputeNormalCholeskyOnANormal / ComputeInverseCholeskyNormal (src/Mathematics/OptCholesky.cpp:78-302)
 * ---------------------------------------------------------------------------------------------- */
#define WG_PLDP_CARDU 16                 /* m_CardV = QP_N                                          */
#define WG_PLDP_NVAR (2 * WG_PLDP_CARDU)  /* 32                                                      */
#define WG_PLDP_MAX_ROWS 128             /* NbOfConstraints <= 8 rows x QP_N samples ("bounded to 8 constraints per support
                                            foot", ZMPConstrainedQPFastFormulation.cpp:775-777); larger m is refused  */

/* Constants the PLDPSolver ctor borrows (PLDPSolver.hh:48-52): iPu, Px, Pu are CardU x CardU, CardU x 3, CardU x CardU
 * row-major host arrays.  (iLQ is only read by the reference's debug dumps and is not needed.) */
int wg_pldp_set_constants(wg_ctx *ctx, int card_u, const double *iPu, const double *Px, const double *Pu);

/* Hot-start memory of one solver instance: m_PreviouslyActivatedConstraints and m_PreviousZMPSolution. */
typedef struct wg_pldp_state {
  double prev_zmp[WG_PLDP_NVAR];
  int32_t prev_active[WG_PLDP_NVAR];
  int32_t n_prev;
  int32_t pad_;
} wg_pldp_state;

typedef struct wg_pldp_info {
  int32_t rc;          /* return value of SolveProblem: 0, or -1 when X[0] / X[CardU] is NaN or Inf (PLDPSolver.cpp:955-964) */
  int32_t status;      /* 0 ok; 1 start point violated a constraint by more than m_tol ("PB ON constraint", :611-616);
                          2 negative step length (the reference calls exit(0), :822-828); 3 active-set capacity;
                          4 iteration cap reached (stands in for the 1.3 ms wall-clock cap, :890-900);
                          6 a SimilarConstraints entry points forward or outside the problem (device-side batches; host-side
                            ones are refused with WG_ERR_INVALID); 7 m outside [0, WG_PLDP_MAX_ROWS] (X = NaN, rc = -1)   */
  int32_t iterations;  /* m_ItNb                                                                                       */
  int32_t n_active;
  int32_t active[WG_PLDP_NVAR];   /* m_ActivatedConstraints in activation order, -1 padded                             */
} wg_pldp_info;

/* Arguments of B calls of PLDPSolver::SolveProblem (PLDPSolver.hh:60-68), one per instance b.  All pointers live in
 * the memory space given by `mem`. */
typedef struct wg_pldp_batch {
  const double *D;        /* [B][32]  CstPartOfTheCostFunction                                                    */
  const int32_t *m;       /* [B]      NbOfConstraints                                                             */
  const double *DPu;      /* instance b at DPu + b*dpu_stride: LinearPartOfConstraints, column-major with leading
                             dimension m[b]+1 (element (r,c) at r + c*(m[b]+1)), 32 columns                       */
  long long dpu_stride;
  const double *DPx;      /* instance b at DPx + b*dpx_stride: CstPartOfConstraints [m[b]]                        */
  long long dpx_stride;
  const double *ZMPRef;   /* [B][32]                                                                              */
  const double *XkYk;     /* [B][6]   (x, dx, ddx, y, dy, ddy)                                                    */
  double *X;              /* [B][32]  out                                                                         */
  const int32_t *similar; /* [B][similar_stride] SimilarConstraints, or NULL.  similar[li] = s != 0 makes ComputeAlpha take
                             the product of row li as minus that of row li + s when that row is not active
                             (PLDPSolver.cpp:570-590), exactly as the reference does; s must be <= 0 with li + s >= 0 (the
                             reference only ever builds -2 / -3, FootConstraintsAsLinearSystem.cpp:53-92).  For flags that
                             match the matrix the reuse is bit-neutral, so NULL gives the same result                    */
  long long similar_stride;
  const int32_t *n_removed; /* [B] NumberOfRemovedConstraints, or NULL (0)                                        */
  const int32_t *starting;  /* [B] StartingSequence, or NULL (true)                                               */
  wg_pldp_state *hot;     /* [B] in/out hot-start memory, or NULL                                                 */
  int32_t hot_start;      /* m_HotStart (the reference hard-codes true, PLDPSolver.cpp:65)                        */
  int32_t max_iterations; /* <= 0: 128                                                                            */
  wg_pldp_info *info;     /* [B] out, or NULL                                                                     */
} wg_pldp_batch;

int wg_pldp_solve_batch(wg_ctx *ctx, int mem, int B, const wg_pldp_batch *batch);

/* The same solve with the constraint matrix in the rank-structured form every call of the reference has: row r of the
 * matrix BuildConstraintMatrices writes (ZMPConstrainedQPFastFormulation.cpp:885-905) is
 *     element (r, k + 16 ax) = A_r(ax) * Pu[k][i_r]
 * with A_r = the half-plane normal of the row, i_r = the previewed sample it belongs to and Pu the matrix given to
 * wg_pldp_set_constants.  The caller passes A0 = A_r(0), A1 = A_r(1) and sample = i_r ([B][row_stride] each, row_stride >=
 * max m) instead of batch->DPu (ignored, may be NULL): 17 bytes per row instead of 256 cross PCIe / HBM, the products are
 * formed where they are used by the same single IEEE multiplication the reference stores, and X / the activation sequence
 * are bitwise those of wg_pldp_solve_batch on the materialised matrix. */
int wg_pldp_solve_batch_ranked(wg_ctx *ctx, int mem, int B, const wg_pldp_batch *batch, const double *A0, const double *A1,
                               const uint8_t *sample, long long row_stride);

/* OptCholesky, B instances: compute rows k0..k1-1 of L for the active rows rows[b][0..k1) of A_b (rows 0..k0-1 of L
 * must already be there: this is AddActiveConstraint called k1-k0 times).  mode 1 = MODE_FORTRAN (A column-major,
 * leading dimension nb_constraints+1), mode 0 = MODE_NORMAL (A row-major, card_u columns).  L is row-major with leading
 * dimension nb_max, as the storage SetL() hands to the reference. */
int wg_optcholesky_add_rows_batch(wg_ctx *ctx, int mem, int B, int mode, int nb_max, int card_u, int nb_constraints,
                                  const double *A, long long a_stride, const int32_t *rows, int rows_stride, int k0,
                                  int k1, double *L, long long l_stride);
/* ComputeNormalCholeskyOnANormal (A: [B][n][n] row-major, may be NULL to keep L) and, when iL != NULL,
 * ComputeInverseCholeskyNormal on the leading inv_size x inv_size block. */
int wg_optcholesky_full_batch(wg_ctx *ctx, int mem, int B, int n, const double *A, double *L, double *iL, int inv_size);

/* ------------------------------------------------------------------------------------------------
 * General dense strictly convex QP, batched, in the ql0001_ calling convention
 *   replaces ql0001_ / ql0002_ (src/Mathematics/qld.hh:27-31, qld.cpp:378-2090) for callers that hand it a dense problem:
 *            ZMPQPWithConstraint (Wieber2006, n = 150, m <= 600: ZMPQPWithConstraint.cpp:1040-1046) and the QLD / QLDANDLQ
 *            branches of ZMPConstrainedQPFastFormulation (:1297-1320)
 *     min 1/2 x'Cx + d'x   s.t.  a_j'x + b_j = 0 (j < me),  a_j'x + b_j >= 0 (me <= j < m),  xl <= x <= xu
 * Arrays are laid out as ql0001_ wants them: C column-major with leading dimension nmax, A column-major with leading
 * dimension mmax (row j of QP k at A + k a_stride + j, its element i at + i mmax), multipliers u = m rows, then n lower
 * bounds, then n upper bounds (qld.cpp:520-536).  One CTA per QP; dual active-set method in range-space form (qld.cu).
 * ifail: 0 ok; 1 iteration limit 40 (m + n) (QLD :459); 2 C not positive definite and eps = 0 (with eps > 0 the diagonal is
 * boosted as QLD does, :809-918); 3 more than n active rows; 5 bad dimensions; 10 + j: constraint j (1-based) cannot be satisfied
 * together with the active ones (QLD's ifail > 10).  On failure x is the unconstrained minimiser.  A row of zeros is
 * inconsistent (10 + j) when b_j < 0 (inequality) or b_j != 0 (equality), and ignored with u_j = 0 otherwise.  Equality rows
 * that depend on earlier ones are skipped when consistent (their multipliers are then not unique: the solver returns one
 * choice) and reported as 10 + j when not.
 * ---------------------------------------------------------------------------------------------- */
#define WG_QLD_MAX_N 160
#define WG_QLD_MAX_M 1024

typedef struct wg_qld_batch {
  int32_t n, nmax;            /* variables; leading dimension of C (>= n)                                        */
  int32_t mmax;               /* leading dimension of A = rows allocated per QP (>= every m; the reference passes m + 1) */
  int32_t shared_hessian;     /* 1: every QP has the Hessian given to wg_qld_set_shared_hessian (C ignored)      */
  const int32_t *m;           /* [B] constraints of each QP                                                      */
  const int32_t *me;          /* [B] equalities among them (the first me rows), or NULL (0)                      */
  const double *C;            /* [B][nmax * n]                                                                   */
  const double *d;            /* [B][n]                                                                          */
  const double *A;            /* QP k at A + k * a_stride                                                        */
  long long a_stride;         /* >= mmax * n                                                                     */
  const double *b;            /* QP k at b + k * b_stride: [m]                                                   */
  long long b_stride;
  const double *xl, *xu;      /* [B][n] each, or both NULL (no bounds; the reference passes -1e8 / +1e8)          */
  double *x;                  /* [B][n]        out                                                               */
  double *u;                  /* [B][u_stride] out, or NULL; entries past m (+ 2n) of each row are set to 0        */
  long long u_stride;         /* >= mmax (+ 2 n when bounds are given)                                           */
  int32_t *ifail;             /* [B]           out                                                               */
  int32_t *iterations;        /* [B]           out (active-set changes), or NULL                                 */
  double eps;                 /* per-QP Hessians: > 0 applies QLD's diagonal boost rule with vsmall = eps (the accuracy
                                 argument of ql0001_; see wg_qld_set_shared_hessian) instead of refusing a Hessian whose
                                 pivots fall below it; 0: factorise C as given, ifail 2 when it is not positive definite */
} wg_qld_batch;

/* The Hessian shared by every QP of later wg_qld_solve_batch(shared_hessian = 1) calls (both reference generators have a
 * constant C): its Cholesky factor is inverted once, on the host in extended precision.  C: column-major, leading dimension
 * nmax.  eps > 0 applies QLD's own treatment of the Hessian first (ql0002_, qld.cpp:809-918): QLD factorises C + diag I, diag
 * found by its 2 x 2 minor test and by doubling steps until every Cholesky pivot exceeds vsmall = eps (the accuracy argument
 * of ql0001_, 1e-8 in every call of the reference).  For a well conditioned C diag is 0; for the reference's generators
 * (eigenvalues down to 2e-9) it is not, and ql0001_'s results are those of the regularised problem - pass the reference's eps
 * to reproduce them, 0 to solve the problem as stated.  wg_qld_shared_boost returns the diag that was added.  The Wieber2006
 * generator keeps its Hessian apart: running it does not replace the one installed here. */
int wg_qld_set_shared_hessian(wg_ctx *ctx, int n, int nmax, const double *C, double eps);
double wg_qld_shared_boost(wg_ctx *ctx);
/* The rule alone (host arithmetic, no device): the multiple of I that ql0001_(eps) adds to C before factorising it. */
double wg_qld_diagonal_boost(int n, int nmax, const double *C, double eps);
int wg_qld_solve_batch(wg_ctx *ctx, int mem, int B, const wg_qld_batch *batch);

/* The same solve for constraint matrices of the rank structure both QP generators of the reference build
 * (ZMPQPWithConstraint.cpp:613-626, ZMPConstrainedQPFastFormulation.cpp:885-905): n = 2N and row r of QP k is
 *     element (r, j + N ax) = A_ax[r] * uz[sample[r] - j]   for j <= sample[r], 0 beyond     (ax = 0, 1)
 * i.e. a half-plane normal (A0, A1) applied to previewed sample `sample[r]` of the lower-triangular Toeplitz map uz from the
 * jerks to the CoP.  A0, A1, sample: [B][row_stride] (row_stride >= mmax), uz_dev: N DEVICE doubles; batch->A is ignored.  The
 * m x n matrix (360 KB per Wieber QP) is neither materialised nor streamed: the violation scan works on the N points Uz x.
 * Device memory only (mem = WG_MEM_DEVICE).  Same results as the dense entry on the materialised matrix up to rounding.
 * sample[r] is not validated: a value >= N is read as N - 1. */
int wg_qld_solve_batch_ranked(wg_ctx *ctx, int mem, int B, const wg_qld_batch *batch, const double *A0, const double *A1,
                              const unsigned char *sample, long long row_stride, const double *uz_dev, int N);

/* ------------------------------------------------------------------------------------------------
 * Kajita2003 front end: footsteps -> 5 ms ZMP reference and feet trajectories, batched
 *   replaces StepStackHandler::ReadStepSequenceAccordingToWalkMode / PrepareForSupportFoot /
 *                CreateArcInStepStack / FinishOnTheLastCorrectSupportFoot
 *                (src/StepStackHandler.cpp:128-175, :754-764, :299-457, :872-883)            [host]
 *            ZMPDiscretization::GetZMPDiscretization = InitOnLine + OnLineAddFoot per step +
 *                EndPhaseOfTheWalking + FilterOutValues + UpdateCurrentSupportFootPosition
 *                (src/ZMPRefTrajectoryGeneration/ZMPDiscretization.cpp:145-175, :319-513, :573-1020,
 *                 :1129-1300, :1046-1107, :515-561)                                          [device]
 *            FootTrajectoryGenerationStandard::UpdateFootPosition (first overload) and the
 *                Polynome3/4/5 boundary-value polynomials
 *                (src/FootTrajectoryGeneration/FootTrajectoryGenerationStandard.cpp:409-563,
 *                 src/Mathematics/PolynomeFoot.cpp:38-56, :103-126, :177-200)                 [device]
 * The output ZMP reference has exactly the layout wg_preview_run_batch consumes, so footsteps -> CoM runs
 * without leaving the GPU (wg_kajita_run_batch).
 * ---------------------------------------------------------------------------------------------- */
typedef struct wg_rel_step {      /* RelativeFootPosition (include/jrl/walkgen/pgtypes.hh)                  */
  double sx, sy;                  /* next support foot in the frame of the current one (m)                   */
  double theta;                   /* relative yaw in DEGREES, as in :stepseq                                 */
  double ss_time, ds_time;        /* SStime / DStime; ds_time == 0 selects the generator's defaults          */
  int32_t step_type;              /* 1 normal; 3/4/5 = step-over ZMP shifts (ZMPDiscretization.cpp:700-728)   */
  int32_t reserved;
} wg_rel_step;                    /* 48 bytes */

typedef struct wg_zmpdisc_params {
  double sampling_period;         /* :samplingperiod       0.005                                             */
  double preview_time;            /* :previewcontroltime   1.6                                               */
  double t_single, t_double;      /* :singlesupporttime / :doublesupporttime (0.78 / 0.02 in the tests)      */
  double step_height;             /* :stepheight           0.07                                              */
  double omega;                   /* :omega (degrees)      0.0                                               */
  double modulation;              /* m_ModulationSupportCoefficient = 0.9 (ZMPDiscretization.cpp:99)         */
  double zmp_neutral[2];          /* m_ZMPNeutralPosition (0, 0)                                             */
  double zmp_shift[4];            /* :ZMPShiftParameters (only used by step types 3/4/5)                     */
  double foot_b, foot_h, foot_f;  /* m_FootB/H/F: heel, ankle height, toe lengths for the omega correction   */
  double filter_time;             /* 0.05: window of the sin^2 smoothing filter (ZMPDiscretization.cpp:237)  */
} wg_zmpdisc_params;

void wg_zmpdisc_default_params(wg_zmpdisc_params *p);   /* the values of tests/CommonTools.cpp:56-69 */

typedef struct wg_foot_sample {   /* the fields of FootAbsolutePosition this path writes */
  double x, y, z, theta, omega, omega2;    /* theta, omega in degrees */
} wg_foot_sample;                 /* 48 bytes */

/* StepStackHandler on the host (tiny, sequential, string/command driven in the reference).  Each appends to
 * steps[*n] (capacity cap) and returns WG_OK or WG_ERR_INVALID when full.  keep_last is m_KeepLastCorrectSupportFoot. */
int wg_steps_support_foot(wg_rel_step *steps, int cap, int *n, int support_foot, double ss, double ds);
int wg_steps_arc(wg_rel_step *steps, int cap, int *n, double x, double y, double arc_deg, int support_foot,
                 double ss, double ds, int *keep_last);
int wg_steps_last_support(wg_rel_step *steps, int cap, int *n, int keep_last, double ss, double ds);

/* Number of 5 ms samples GetZMPDiscretization emits for a step list (host arithmetic only):
 * 2*NL lead-in + sum over steps 1.. of round((DS+SS)/T) + round(Tdble/(2T)) + 3*NL. */
int64_t wg_zmpdisc_sample_count(const wg_zmpdisc_params *p, int n_steps, const wg_rel_step *steps);

/* A Kajita plan = the step stacks of B walks (what StepStackHandler holds when :finish / :stepseq arrives), resident
 * on the GPU.  Walk b owns steps [step_offsets[b], step_offsets[b+1]) (HOST arrays; uploaded once, a few KB per
 * walk); init_feet[b] = {left x, y, theta, right x, y, theta} (InitLeft/RightFootAbsolutePosition, theta in degrees).
 * The plan computes the sample offsets of the ragged batch (walk b owns samples [so[b], so[b+1])) and, when preview
 * gains are set on the context, an internal wg_preview_plan over them. */
typedef struct wg_kajita_plan wg_kajita_plan;
int wg_kajita_plan_create(wg_ctx *ctx, const wg_zmpdisc_params *p, int B, const int64_t *step_offsets_host,
                          const wg_rel_step *steps_host, const double *init_feet_host, wg_kajita_plan **out);
int wg_kajita_plan_destroy(wg_kajita_plan *plan);
const int64_t *wg_kajita_plan_sample_offsets(const wg_kajita_plan *plan);   /* host array of B+1 entries */
int64_t wg_kajita_plan_total_samples(const wg_kajita_plan *plan);
int64_t wg_kajita_plan_total_steps(const wg_kajita_plan *plan);             /* preview steps, sum of L_b-NL+1 */
/* Replace the step values of every walk (same step counts and timings, hence the same sample offsets): the H2D copy
 * a caller streaming new footstep plans pays per batch.  Asynchronous on the context stream. */
int wg_kajita_plan_set_steps(wg_kajita_plan *plan, const wg_rel_step *steps_host, const double *init_feet_host);

/* ZMPDiscretization::GetZMPDiscretization for every walk of the plan.  Outputs (any may be NULL), `mem` says where
 * they live: zmpref_xy [total][2] (px, py) filtered = FinalZMPPositions; zmp_theta [total] (degrees);
 * left/right [total] feet; step_type [total][3] = stepType of the ZMP, left-foot and right-foot samples. */
int wg_zmpdisc_run_batch(wg_ctx *ctx, wg_kajita_plan *plan, int mem, double *zmpref_xy, double *zmp_theta,
                         wg_foot_sample *left, wg_foot_sample *right, int32_t *step_type);

/* Footsteps -> CoM: GetZMPDiscretization followed by the preview loop of wg_preview_run_batch on the same device
 * buffers; the ZMP reference only leaves the GPU if zmpref_xy != NULL.  state/com_out/zmp_out as in
 * wg_preview_run_batch.  With WG_MEM_HOST the walks are processed in chunks and the D2H copy of a chunk's outputs
 * overlaps the kernels of the next one. */
int wg_kajita_run_batch(wg_ctx *ctx, wg_kajita_plan *plan, int mem, double *state, double *com_out, double *zmp_out,
                        double *zmpref_xy, wg_foot_sample *left, wg_foot_sample *right, int simulation);

/* On-line form: B walks whose footsteps arrive while they run, each walk's state kept on the device between runs.
 *   replaces ZMPDiscretization::InitOnLine (src/ZMPRefTrajectoryGeneration/ZMPDiscretization.cpp:319-513),
 *            ZMPDiscretization::OnLineAddFoot (:573-1020) and ZMPDiscretization::EndPhaseOfTheWalking (:1129-1300),
 *            each driving the preview loop over the new part of the ZMP FIFO                               [device]
 * Each run emits what one append scheduled.  For walk b, flags[b] selects:
 *   WG_STREAM_START   (re)start the walk (InitOnLine); its state is dropped.  The append's first step is the support-foot
 *                     step (step 0 of a plan's list): the run emits the 2*NL lead-in, then one segment per further step.
 *                     The preview state of the walk is zeroed.  init_feet_host[b] as in wg_kajita_plan_create.
 *   (no flag)         each appended step is one OnLineAddFoot and emits its segment.
 *   WG_STREAM_FINISH  after this append's steps, EndPhaseOfTheWalking (n_end + 3*NL samples); the walk closes.
 * A walk with no steps and no flags is untouched.  START|FINISH on a whole step list is exactly one walk of a plan: the
 * samples a walk emits over all its runs, concatenated, are bitwise what wg_zmpdisc_run_batch gives for its whole list.
 *
 * wg_kajita_stream_append plans the next run on the host (the step timings size it) and starts an asynchronous H2D copy
 * of its steps; steps, offsets and flags are host arrays (step_offsets [B+1], walk b appends steps [off[b], off[b+1]) of
 * steps_host; flags_host [B] may be NULL for no flags).  Refused with WG_ERR_INVALID, every walk left unchanged: steps for a
 * walk that is not open and has no START; START with zero steps or with init_feet_host == NULL; FINISH on a closed walk;
 * a step timing that wg_kajita_plan_create refuses; an append while the previous one has not been run.
 *
 * wg_kajita_stream_run executes the pending append (a run with none pending does nothing).  Outputs live in `mem` and
 * each may be NULL; their rows:
 *   zmpref_xy [][2], zmp_theta [], left [], right [], step_type [][3]: walk b's new samples are rows [so[b], so[b+1]),
 *       compact and in order (so = wg_kajita_stream_sample_offsets).
 *   com_out [][6], zmp_out [][2]: walk b's com_counts[b] new preview steps are the first rows of [co[b], co[b+1])
 *       (co = wg_kajita_stream_com_offsets).  Row j is the walk's preview step steps_previewed_before + j, the row
 *       wg_kajita_run_batch writes at offsets[b] + steps_previewed_before + j.  Rows past the count: untouched with
 *       WG_MEM_DEVICE, zero with WG_MEM_HOST.  A walk's preview consumes its samples as they arrive: after a run it has
 *       previewed max(0, samples_emitted - NL + 1) steps, so FINISH completes the walk's preview.
 * with_preview = 1 needs preview gains on the context (WG_ERR_NOT_READY otherwise) and keeps their NL: a run after gains of
 * another NL were set is refused with WG_ERR_NOT_READY.  Gains of the same NL and the sum mode are read at run time, as
 * wg_kajita_run_batch does.  With with_preview = 0 the stream is the front end only and com_out / zmp_out must be NULL.
 * The offsets returned below describe the pending append (or the last one run); they stay valid until the next append.
 * In steady state a run allocates nothing and creates no stream or event; buffers grow when a run needs more. */
typedef struct wg_kajita_stream wg_kajita_stream;
enum { WG_STREAM_START = 1, WG_STREAM_FINISH = 2 };
int wg_kajita_stream_create(wg_ctx *ctx, const wg_zmpdisc_params *p, int B, int with_preview, wg_kajita_stream **out);
int wg_kajita_stream_destroy(wg_kajita_stream *s);
int wg_kajita_stream_append(wg_kajita_stream *s, const int64_t *step_offsets_host, const wg_rel_step *steps_host,
                            const int32_t *flags_host, const double *init_feet_host);
const int64_t *wg_kajita_stream_sample_offsets(const wg_kajita_stream *s);  /* B+1: rows of the samples the run emits */
const int64_t *wg_kajita_stream_com_offsets(const wg_kajita_stream *s);     /* B+1: rows reserved for its preview steps */
const int64_t *wg_kajita_stream_com_counts(const wg_kajita_stream *s);      /* B: preview steps each walk gets          */
int wg_kajita_stream_run(wg_kajita_stream *s, int mem, double *zmpref_xy, double *zmp_theta, wg_foot_sample *left,
                         wg_foot_sample *right, int32_t *step_type, double *com_out, double *zmp_out, int simulation);
/* After the last run: preview_state [B][8] (in `mem`; as wg_preview_run_batch's state) and, in host arrays of B entries,
 * the samples each walk emitted and the preview steps it ran since its START, and whether it is open.  Any may be NULL.
 * With WG_MEM_HOST the call waits for the stream. */
int wg_kajita_stream_state(wg_kajita_stream *s, int mem, double *preview_state, int64_t *samples_emitted,
                           int64_t *steps_previewed, int32_t *open);

/* ------------------------------------------------------------------------------------------------
 * Dimitrov2008 front to back: feet trajectories -> support polygons -> per-period constraint matrices ->
 * PLDP solve -> LIPM, closed loop on the device (one warp owns one walk for its whole duration)
 *   replaces ComputeConvexHull::DoComputeConvexHull                     (src/Mathematics/ConvexHull.cpp:87-203)
 *            FootConstraintsAsLinearSystem::BuildLinearConstraintInequalities / ComputeLinearSystem /
 *                FindSimilarConstraints          (src/Mathematics/FootConstraintsAsLinearSystem.cpp:258-539, :94-256, :53-92)
 *            ZMPConstrainedQPFastFormulation::InitConstants = InitializeMatrixPbConstants +
 *                BuildingConstantPartOfTheObjectiveFunction(+QLDANDLQ) + BuildingConstantPartOfConstraintMatrices
 *                (src/ZMPRefTrajectoryGeneration/ZMPConstrainedQPFastFormulation.cpp:158-246, :390-614, :616-720)  [host]
 *            ZMPConstrainedQPFastFormulation::BuildConstraintMatrices (:759-1022) and the PLDP branch of
 *                BuildZMPTrajectoryFromFootTrajectory (:1095-1480), GetZMPDiscretization (:1483-1520)            [device]
 *            LinearizedInvertedPendulum2D::Interpolation / OneIteration (src/PreviewControl/LinearizedInvertedPendulum2D.cpp:157-264)
 * ---------------------------------------------------------------------------------------------- */
#define WG_LCI_MAX_ROWS 8              /* "bounded to 8 constraints per support foot (double support case)", :775-777 */

typedef struct wg_lci {               /* LinearConstraintInequality_t (include/jrl/walkgen/pgtypes.hh:168-177): A z + B >= 0 */
  double A[WG_LCI_MAX_ROWS][2];
  double B[WG_LCI_MAX_ROWS];
  double center[2];
  double t_start, t_end;              /* StartingTime, EndingTime (the accumulated 5 ms clock of the feet samples)       */
  int32_t rows;
  int32_t first_sample;               /* index of the 5 ms sample that opened the polygon                                */
  int32_t state;                      /* 1 right foot is support (left flying), 2 left foot is support, 3 double support */
  int32_t rc;                         /* 0, or -1 when ComputeLinearSystem reports "Linear system ill-computed" (:244-249) */
  int32_t similar[WG_LCI_MAX_ROWS];   /* SimilarConstraints                                                              */
} wg_lci;                             /* 272 bytes */

typedef struct wg_dimitrov_params {
  double T;                           /* m_QP_T 0.1                                                                      */
  double sampling_period;             /* m_SamplingPeriod 0.005                                                          */
  double com_height;                  /* m_ComHeight 0.80                                                                */
  double alpha, beta;                 /* m_Alpha 200, m_Beta 1000                                                        */
  double constraint_x, constraint_y;  /* :setdimitrovconstraint  0.04 0.04                                               */
  double sole_length, sole_width;     /* CjrlFoot::getSoleSize of both feet (robot data; HRP-2 test robot: 0.25 x 0.14)  */
  int32_t max_iterations;             /* PLDP iteration cap standing in for the 1.3 ms wall-clock cap; <= 0: 128         */
  int32_t cold_restart;               /* what to do when a hot-started solve finds its start point infeasible by more
                                         than m_tol ("PB ON constraint" then a negative step: the reference prints and
                                         calls exit(0), PLDPSolver.cpp:611-616, :822-828).  0 (default, the reference's
                                         observable behaviour short of killing the process): the walk stops there with
                                         status 1.  1: the period is solved again from the cold start point
                                         (StartingSequence semantics, no kept constraints) and flagged status 5.        */
  int32_t merge_duplicate_rows;       /* 0 (default): the polygons of the reference, bit for bit.  1: a half-plane that
                                         repeats its predecessor (all three coefficients within 1e-9: the reference's hull
                                         keeps corners that are collinear only up to rounding) is dropped, which removes
                                         the singular active sets behind the reference's NaN / IFAIL stops.               */
  int32_t reserved;
} wg_dimitrov_params;

void wg_dimitrov_default_params(wg_dimitrov_params *p);

/* The constants of InitConstants() for QP_N = 16 (host arithmetic, uploaded to the context; also installs them as the
 * PLDP constants of wg_pldp_solve_batch).  Any out pointer may be NULL.  Row-major: iPu, Pu, iLQ, OptC [16][16] (one
 * axis block); Px, OptB [16][3]. */
int wg_dimitrov_set_params(wg_ctx *ctx, const wg_dimitrov_params *p, double *iPu, double *Px, double *Pu, double *iLQ,
                           double *OptB, double *OptC);

/* DoComputeConvexHull for B point sets of n points each (xy [B][n][2], n <= 8): hull_xy [B][8][2], counts [B]. */
int wg_convex_hull_batch(wg_ctx *ctx, int mem, int B, int n, const double *xy, double *hull_xy, int32_t *counts);

/* BuildLinearConstraintInequalities for a ragged batch of feet buffers: walk b owns samples
 * [sample_offsets[b], sample_offsets[b+1]) of left/right/step_type (step_type [total][3] as written by
 * wg_zmpdisc_run_batch: ZMP, left foot, right foot; only the left foot's is read) and writes at most
 * lci_offsets[b+1]-lci_offsets[b] polygons at lci + lci_offsets[b]; n_lci[b] = number found (a walk that needs more
 * fails with WG_ERR_INVALID in host mode and n_lci[b] = -needed in device mode).  sample_offsets / lci_offsets are
 * HOST arrays; the others live in `mem`.  Sample i of a walk carries time = the 5 ms clock accumulated i times. */
int wg_fcals_build_batch(wg_ctx *ctx, int mem, int B, const int64_t *sample_offsets, const wg_foot_sample *left,
                         const wg_foot_sample *right, const int32_t *step_type, const int64_t *lci_offsets,
                         wg_lci *lci, int32_t *n_lci);

typedef struct wg_dimitrov_period {   /* one iteration of the loop of BuildZMPTrajectoryFromFootTrajectory */
  double t_start;                     /* StartingTime                                                       */
  double xk[6];                       /* LIPM state the QP was built for (x, dx, ddx, y, dy, ddy)            */
  double jerk_x, jerk_y;              /* ptX[0], ptX[N]                                                      */
  int32_t m;                          /* NbOfConstraints                                                     */
  int32_t n_first;                    /* NextNumberOfRemovedConstraints                                      */
  int32_t rc, status;                 /* as wg_pldp_info; status 5 = solved again from the cold start (cold_restart) */
  int32_t iterations, n_active;
  int32_t active[WG_PLDP_NVAR];
} wg_dimitrov_period;                 /* 224 bytes */

/* Number of QP periods the loop runs for a feet buffer of n samples (host arithmetic, the loop bound of :1190-1194). */
int64_t wg_dimitrov_period_count(const wg_dimitrov_params *p, int64_t n_samples);

/* GetZMPDiscretization of ZMPConstrainedQPFastFormulation for every walk of a Kajita plan: ZMPDiscretization, then
 * FootConstraintsAsLinearSystem, then the receding-horizon PLDP loop.  Outputs (any may be NULL) live in `mem`:
 *   com_out [total][6]   COMStates x[0..2], y[0..2]; rows the loop does not reach are zero
 *   zmp_out [total][2]   ZMPRefPositions px, py after the loop (rows it does not reach keep the discretised reference)
 *   left/right [total]   feet
 *   periods              walk b's periods at periods + period_offsets[b] (period_offsets: HOST array of B+1 entries,
 *                        period_offsets[b+1]-period_offsets[b] >= wg_dimitrov_period_count of the walk), or NULL
 *   status [B]           0, 1 = a PLDP solve failed: NaN (the reference prints IFAIL and returns -1, :1373-1377) or
 *                        an infeasible hot start (the reference calls exit(0)); the walk stops at that period,
 *                        2 = no polygon covers a sample time ("HERE 3", :800-804), 3 = polygon capacity,
 *                        4 = ZMPDiscretization refused the walk
 *   periods_done [B]     periods attempted (the failing one included) */
int wg_dimitrov_run_batch(wg_ctx *ctx, wg_kajita_plan *plan, int mem, double *com_out, double *zmp_out,
                          wg_foot_sample *left, wg_foot_sample *right, const int64_t *period_offsets,
                          wg_dimitrov_period *periods, int32_t *status, int32_t *periods_done);

/* ------------------------------------------------------------------------------------------------
 * Wieber2006 front to back: feet trajectories -> support polygons -> per-period dense QP (n = 2N = 150 jerks, m <= 8N CoP
 * rows) -> LIPM, batched over walks
 *   replaces ZMPQPWithConstraint::BuildLinearConstraintInequalities / ComputeLinearSystem
 *                (src/ZMPRefTrajectoryGeneration/ZMPQPWithConstraint.cpp:229-502, :94-228)
 *            ZMPQPWithConstraint::BuildMatricesPxPu (:504-663) and BuildZMPTrajectoryFromFootTrajectory (:665-1338: constant
 *                matrices, the receding-horizon loop, ql0001_, the feasibility check of the solution, the 5 ms interpolation)
 *            ZMPQPWithConstraint::GetZMPDiscretization (:1340-1387)
 * ---------------------------------------------------------------------------------------------- */
#define WG_WIEBER_MAX_N 80

typedef struct wg_wieber_params {
  double T;                           /* m_QP_T 0.02            (:71)                                                   */
  double sampling_period;             /* m_SamplingPeriod 0.005 (:78)                                                   */
  double com_height;                  /* ComHeight 0.80         (:674)                                                  */
  double alpha, beta;                 /* 200, 1000              (:691)                                                  */
  double constraint_x, constraint_y;  /* :setpbwconstraint XY, 0.04 0.04 (:68-69)                                        */
  double sole_length, sole_width;     /* CjrlFoot::getSoleSize (robot data)                                             */
  double qld_eps;                     /* Eps handed to ql0001_, 1e-8 (:734): QLD regularises the Hessian with it (see
                                         wg_qld_set_shared_hessian); 0 solves the QP as stated                          */
  int32_t N;                          /* m_QP_N 75              (:72); 2N <= WG_QLD_MAX_N                               */
  int32_t materialize_pu;             /* 0 (default): the rows go to the solver as (A_r(0), A_r(1), i_r)
                                         (wg_qld_solve_batch_ranked); 1: the dense (m + 1) x 2N matrix Pu is written out in
                                         ql0001_'s layout and solved through wg_qld_solve_batch, as the reference does       */
} wg_wieber_params;

void wg_wieber_default_params(wg_wieber_params *p);
/* Constant matrices (host, the reference's summation order) and the Hessian of the dense solver (wg_qld_set_shared_hessian). */
int wg_wieber_set_params(wg_ctx *ctx, const wg_wieber_params *p);
/* Number of QP periods the loop runs for a feet buffer of n samples (the loop bound of :993-995). */
int64_t wg_wieber_period_count(const wg_wieber_params *p, int64_t n_samples);
/* GetZMPDiscretization of ZMPQPWithConstraint for every walk of a Kajita plan.  Outputs (any may be NULL) live in `mem`:
 *   com_out [total][6]   COMStates x[0..2], y[0..2]; rows the loop does not reach are zero
 *   zmp_out [total][2]   ZMPRefPositions px, py after the loop (rows it does not reach keep the discretised reference)
 *   left / right [total] feet
 *   status [B]           0; 1 = the QP failed or its solution violates a row by more than 1e-8 (the reference prints and
 *                        returns -1, :1048-1052, :1085-1104); 2 = no polygon covers a sample time ("HERE 3", :545-549);
 *                        3 = polygon capacity; 4 = ZMPDiscretization refused the walk.  A failed walk stops at that period
 *   periods_done [B]     QP periods attempted
 *   qp_iterations [B]    active-set changes summed over the walk's QPs */
int wg_wieber_run_batch(wg_ctx *ctx, wg_kajita_plan *plan, int mem, double *com_out, double *zmp_out, wg_foot_sample *left,
                        wg_foot_sample *right, int32_t *status, int32_t *periods_done, long long *qp_iterations);

#ifdef __cplusplus
}
#endif
#endif /* WALKGEN_B200_H */
