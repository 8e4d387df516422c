// wg_common.h - internal definitions shared by the CUDA translation units of libwalkgen_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include "../../include/walkgen_b200.h"

#define WG_VERSION ((0 << 16) | (1 << 8) | 0)

// Kernel ids of the per-kernel CUDA-event profiler (wg_prof_*): bench.py reads the average launch
// duration of each kernel over the timed region from these.
enum { WG_K_PREVIEW_FIR = 0, WG_K_PREVIEW_RECUR = 1, WG_K_HERDT_QP = 2, WG_K_HERDT_MPC = 3, WG_K_PLDP = 4,
       WG_K_OPTCHOL = 5, WG_K_PREVIEW_FUSED = 6, WG_K_ZMPDISC = 7, WG_K_FCALS = 8, WG_K_DIMITROV = 9, WG_K_QLD = 10, WG_K_WIEBER = 11,
       WG_K_COUNT = 12 };

struct wg_prof_state {
  bool on = false;
  std::vector<cudaEvent_t> ev;   // pairs (start, stop)
  std::vector<int> kid;          // kernel id of pair i
  size_t used = 0;               // pairs recorded since wg_prof_begin
  long long launches[WG_K_COUNT] = {0};
  double total_ms[WG_K_COUNT] = {0};
};

struct wg_ctx {
  wg_prof_state prof;
  int device = -1;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  long long launches = 0;
  char err[512] = {0};
  // preview control
  bool preview_ready = false;
  wg_preview_gains_t preview_gains;
  std::vector<unsigned char> preview_image;   // host image of the kernels' __constant__ block (PreviewConsts + taps)
  unsigned long long preview_gen = 0;         // bumped by wg_preview_set_gains
  void *preview_tick = nullptr;               // buffers of wg_preview_one_iteration (preview.cu)
  int preview_sum_mode = WG_PREVIEW_SUM_AUTO;  // wg_preview_set_sum_mode
  int preview_cta_shape = -1;                 // wg_preview_set_cta_shape (-1: per launch)
  bool preview_rec_ok = false;                // the window weights fit w' L^i v within WG_PREVIEW_REC_TOL (rec_setup, preview.cu)
  double preview_rec_residual = -1.0;
  void *preview_rec_dev = nullptr;            // device tables of preview_rec_kernel
  // Herdt constants (herdt_qp.cu)
  void *herdt = nullptr;
  // Herdt closed loop (herdt_mpc.cu)
  void *herdt_mpc = nullptr;
  // PLDP constants (pldp.cu)
  void *pldp = nullptr;
  // Dimitrov front-to-back pipeline (dimitrov.cu)
  void *dimitrov = nullptr;
  // dense QP solver (qld.cu) and the Wieber2006 generator on top of it (wieber.cu)
  void *qld = nullptr;
  void *wieber = nullptr;
};

inline int wg_fail(wg_ctx *ctx, int code, const char *what, cudaError_t e = cudaSuccess)
{
  if (ctx) {
    if (e != cudaSuccess)
      snprintf(ctx->err, sizeof ctx->err, "%s: %s", what, cudaGetErrorString(e));
    else
      snprintf(ctx->err, sizeof ctx->err, "%s", what);
  }
  return code;
}

#define WG_CUDA(ctx, call)                                                   \
  do {                                                                       \
    cudaError_t e__ = (call);                                                \
    if (e__ != cudaSuccess) return wg_fail((ctx), WG_ERR_CUDA, #call, e__);  \
  } while (0)

#define WG_LAUNCHED(ctx)                                                     \
  do {                                                                       \
    (ctx)->launches++;                                                       \
    cudaError_t e__ = cudaGetLastError();                                    \
    if (e__ != cudaSuccess) return wg_fail((ctx), WG_ERR_CUDA, "kernel launch", e__); \
  } while (0)

// Bracket a kernel launch with profiler events (no-ops unless wg_prof_begin was called).
inline void wg_prof_start(wg_ctx *ctx, int kid)
{
  wg_prof_state &p = ctx->prof;
  if (!p.on || 2 * (p.used + 1) > p.ev.size()) return;
  p.kid[p.used] = kid;
  cudaEventRecord(p.ev[2 * p.used], ctx->stream);
}
inline void wg_prof_stop(wg_ctx *ctx)
{
  wg_prof_state &p = ctx->prof;
  if (!p.on || 2 * (p.used + 1) > p.ev.size()) return;
  cudaEventRecord(p.ev[2 * p.used + 1], ctx->stream);
  p.used++;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE, per-function attribute: keep the largest value set so far
// per (device, kernel) instead of in function-local statics (a second context on another GPU must set it again, a second
// context on the same GPU must not lower it).  Kernels that need at most 48 KB are left alone.
extern "C" int wgi_smem_attr(wg_ctx *ctx, const void *func, size_t bytes);
#define WG_SMEM_ATTR(ctx, func, bytes)                                              \
  do {                                                                              \
    int rc__ = wgi_smem_attr((ctx), reinterpret_cast<const void *>(func), (bytes)); \
    if (rc__ != WG_OK) return rc__;                                                 \
  } while (0)

// Grow-only device scratch: make *buf hold at least `bytes` (8 for a zero-byte request), *cap being its size in bytes.  A
// buffer that must grow is freed after the context stream drains (earlier launches may still read it); on return *buf is
// never null.
extern "C" int wgi_grow_scratch(wg_ctx *ctx, void **buf, size_t *cap, size_t bytes);

// preview.cu internals used by zmpdisc.cu (the footsteps -> CoM pipeline): launch the fused preview kernel over `count`
// trajectories listed in the device array d_order.
extern "C" int wgi_preview_launch_range(wg_ctx *ctx, wg_preview_plan *pl, const int *d_order, int count,
                                        const double *d_zmp, double *d_state, double *d_com, double *d_zmpout,
                                        int simulation, const double *d_com_add = nullptr, int pos_only = 0);
// Replace the offsets of a plan's B trajectories (same B, no allocation); the copy is asynchronous on the context stream.
extern "C" int wgi_preview_plan_set_offsets(wg_preview_plan *pl, const int64_t *offsets_host);

// zmpdisc.cu / pldp.cu internals used by dimitrov.cu
struct wgi_kajita_view {
  int B;
  const int64_t *samp_off, *step_off;   // host, B+1 entries
  const int64_t *d_samp_off;            // device
  const int *d_zd_status;               // device, per walk
  double sampling_period;
};
extern "C" int wgi_kajita_discretize_device(wg_ctx *ctx, wg_kajita_plan *pl, double **zmpref, wg_foot_sample **left,
                                            wg_foot_sample **right, int32_t **types, wgi_kajita_view *view);
extern "C" const void *wgi_pldp_device_consts(wg_ctx *ctx);   // PldpConsts on the device, or nullptr
// The dense QP solver with the Wieber2006 generator's own shared Hessian, kept apart from the one a caller installs with
// wg_qld_set_shared_hessian.  wgi_qld_solve_generator: device memory; A0 = nullptr selects the dense rows of batch->A, else
// the rank-structured rows of wg_qld_solve_batch_ranked.
extern "C" int wgi_qld_set_generator_hessian(wg_ctx *ctx, int n, int nmax, const double *C, double eps);
extern "C" int wgi_qld_solve_generator(wg_ctx *ctx, int B, const wg_qld_batch *q, const double *A0, const double *A1,
                                       const unsigned char *sample, long long row_stride, const double *uz_dev, int N);

struct wg_device_guard {
  int prev = -1;
  explicit wg_device_guard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~wg_device_guard() { if (prev >= 0) cudaSetDevice(prev); }
};
