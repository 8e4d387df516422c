// herdt_qp.cu - batched Herdt2010 velocity-referenced QP for sm_100a: host constants, kernels, C ABI.
// Device algorithm: herdt_qp.cuh.
#include "herdt_qp.cuh"
#include <algorithm>
#include <vector>
#include <cmath>

namespace {

using herdt::Consts;
using herdt::N;

struct HerdtState {
  Consts h_consts;
  Consts *d_consts = nullptr;
  bool ready = false;
  // staging for WG_MEM_HOST calls
  wg_herdt_qp_input *d_in = nullptr; size_t cap_in = 0;
  wg_herdt_qp_output *d_out = nullptr; size_t cap_out = 0;
  int *d_next = nullptr;          // work counter of herdt_qp_kernel
  double *d_T = nullptr; size_t cap_T = 0;   // per-warp T slices
  wg_herdt_active_set *d_act = nullptr; size_t cap_act = 0;   // staging of the warm-start sets (WG_MEM_HOST)
  // WG_MEM_HOST pipeline: upload / download streams and per-chunk events
  cudaStream_t up = nullptr, down = nullptr;
  cudaEvent_t ev_up[2] = {nullptr}, ev_k[2] = {nullptr}, ev0 = nullptr;
};

HerdtState *state_of(wg_ctx *ctx)
{
  if (!ctx->herdt) ctx->herdt = new HerdtState();
  return static_cast<HerdtState *>(ctx->herdt);
}

// Constant matrices in extended precision (the only place an inverse is formed):
//   Uv, Uz, Sv, Sz: RigidBodySystem::compute_dyn_cjerk (src/PreviewControl/rigid-body-system.cpp:377-452)
//   Qc = w_jerk I + w_vel Uv'Uv + w_cop Uz'Uz: GeneratorVelRef::build_invariant_part (generator-vel-ref.cpp:588-614)
void compute_consts(const wg_herdt_params &P, Consts &C)
{
  typedef long double L;
  const L T = P.T, h = P.com_height, g = 9.81L;
  L Uv[N][N], Uz[N][N], Sv[N][3], Qc[N][N], Gi[N][2 * N];
  for (int i = 0; i < N; ++i) {
    Sv[i][0] = 0; Sv[i][1] = 1; Sv[i][2] = (i + 1) * T;
    C.Sz[i][0] = 1.0; C.Sz[i][1] = (double)((i + 1) * T);
    C.Sz[i][2] = (double)((L)(i + 1) * (i + 1) * T * T * 0.5L - h / g);
    for (int j = 0; j < N; ++j) {
      const int d = i - j;
      Uv[i][j] = (j <= i) ? (2 * d + 1) * T * T * 0.5L : 0.0L;
      Uz[i][j] = (j <= i) ? (1 + 3 * d + 3 * d * d) * T * T * T / 6.0L - T * h / g : 0.0L;
    }
  }
  for (int d = 0; d < N; ++d) {
    // the device uses exactly the doubles the reference computes (rigid-body-system.cpp:438-441)
    C.uz[d] = (1 + 3 * d + 3 * d * d) * P.T * P.T * P.T / 6.0 - P.T * P.com_height / 9.81;
  }
  for (int i = 0; i < N; ++i) {
    double s2 = 0.0;
    for (int j = 0; j <= i; ++j) { Uz[i][j] = C.uz[i - j]; s2 += C.uz[i - j] * C.uz[i - j]; }
    C.uz2[i] = s2;
  }
  for (int i = 0; i < N; ++i)
    for (int j = 0; j < N; ++j) {
      L s = (i == j) ? (L)P.w_jerk : 0.0L;
      for (int k = 0; k < N; ++k) s += (L)P.w_vel * Uv[k][i] * Uv[k][j] + (L)P.w_cop * Uz[k][i] * Uz[k][j];
      Qc[i][j] = s;
      C.Qc[i][j] = (double)s;
    }
  // Gauss-Jordan inverse with partial pivoting
  for (int i = 0; i < N; ++i)
    for (int j = 0; j < N; ++j) { Gi[i][j] = Qc[i][j]; Gi[i][N + j] = (i == j) ? 1.0L : 0.0L; }
  for (int c = 0; c < N; ++c) {
    int piv = c;
    for (int r = c + 1; r < N; ++r)
      if (fabsl(Gi[r][c]) > fabsl(Gi[piv][c])) piv = r;
    if (piv != c)
      for (int j = 0; j < 2 * N; ++j) std::swap(Gi[piv][j], Gi[c][j]);
    const L d = Gi[c][c];
    for (int j = 0; j < 2 * N; ++j) Gi[c][j] /= d;
    for (int r = 0; r < N; ++r)
      if (r != c) {
        const L f = Gi[r][c];
        if (f != 0.0L)
          for (int j = 0; j < 2 * N; ++j) Gi[r][j] -= f * Gi[c][j];
      }
  }
  L G0[N][N], K1[N][N], K3[N][N];
  for (int i = 0; i < N; ++i)
    for (int j = 0; j < N; ++j) G0[i][j] = 0.5L * (Gi[i][N + j] + Gi[j][N + i]);
  for (int i = 0; i < N; ++i)
    for (int j = 0; j < N; ++j) {
      L a = 0, b = 0;
      for (int k = 0; k < N; ++k) { a += G0[i][k] * Uz[j][k]; b += G0[i][k] * Uv[j][k]; }
      K1[i][j] = a; K3[i][j] = b;
      C.K1[i][j] = (double)a; C.K3[i][j] = (double)b;
    }
  for (int i = 0; i < N; ++i) {
    for (int j = 0; j < N; ++j) {
      L a = 0;
      for (int k = 0; k < N; ++k) a += Uz[i][k] * K1[k][j];
      C.G[i][j] = (double)a;
    }
    for (int c = 0; c < 3; ++c) {
      L a = 0;
      for (int k = 0; k < N; ++k) a += K3[i][k] * Sv[k][c];
      C.K4[i][c] = (double)a;
    }
  }
  for (int i = 0; i < N; ++i)   // symmetrise G in double
    for (int j = 0; j < i; ++j) { double v = 0.5 * (C.G[i][j] + C.G[j][i]); C.G[i][j] = C.G[j][i] = v; }
  C.P = P;
}

constexpr int QP_WARPS = 4;  // warps (instances) per block

__global__ void __launch_bounds__(QP_WARPS * 32, 4)
herdt_qp_kernel(int B, const Consts *__restrict__ Cp, const wg_herdt_qp_input *__restrict__ in,
                wg_herdt_qp_output *__restrict__ out, int *__restrict__ next_instance, double *__restrict__ scratchT,
                herdt::LaunchOpts opt)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  herdt::Work *works = reinterpret_cast<herdt::Work *>(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const Consts &C = *Cp;
  herdt::Work &s = works[warp];
  double *Tw = scratchT + ((size_t)blockIdx.x * QP_WARPS + warp) * herdt::TRI;
  // solve times differ (10-42 active-set iterations): every warp takes its next instance from a work counter
  for (;;) {
    int b = 0;
    if (lane == 0) b = atomicAdd(next_instance, 1);
    b = __shfl_sync(0xffffffffu, b, 0);
    if (b >= B) break;
    if (opt.fire && !*reinterpret_cast<const int *>(opt.fire + (size_t)b * opt.fire_stride)) continue;   // closed loop: no QP this period
    // stage the 784-byte input record
    {
      const double *src = reinterpret_cast<const double *>(in + b);
      double *dst = reinterpret_cast<double *>(&s.in);
      for (int e = lane; e < (int)(sizeof(wg_herdt_qp_input) / 8); e += 32) dst[e] = __ldg(src + e);
    }
    __syncwarp();
    int q = 0;
    const wg_herdt_active_set *guess =
        opt.guess ? reinterpret_cast<const wg_herdt_active_set *>(opt.guess + (size_t)b * opt.guess_stride) : nullptr;
    const herdt::Result r = herdt::solve_warp(s, C, lane, q, Tw, guess, opt.age);
    if (opt.active_out) {   // may alias the guess: the solve is done with it
      wg_herdt_active_set *ao = reinterpret_cast<wg_herdt_active_set *>(opt.active_out + (size_t)b * opt.active_stride);
      const int nq = r.fail ? 0 : q;
      for (int e = lane; e < (int)sizeof(ao->rows); e += 32) ao->rows[e] = (e < nq) ? (int8_t)s.W[e] : (int8_t)-1;
      if (lane == 0) {
        int p1 = 0, p2 = 0;
        for (int k = N; k >= 1; --k) { const int sn = s.in.sup_step[k]; if (sn == 1) p1 = k; else if (sn == 2) p2 = k; }
        ao->n = (int8_t)nq; ao->step_pi[0] = (int8_t)p1; ao->step_pi[1] = (int8_t)p2;
        for (int e = 0; e < 5; ++e) ao->pad_[e] = 0;
      }
    }
    // ---- write wg_herdt_qp_output (960 B)
    wg_herdt_qp_output &o = out[b];
    const int ns = (r.n_vars - 2 * N) / 2;
    for (int e = lane; e < WG_HERDT_MAX_VARS; e += 32) {
      double v = 0.0;
      if (e < 2 * N) v = s.jr[e >> 4][e & 15];
      else if (e < 2 * N + ns) v = s.ff[0][e - 2 * N];
      else if (e < 2 * N + 2 * ns) v = s.ff[1][e - 2 * N - ns];
      o.x[e] = v;
    }
    for (int e = lane; e < WG_HERDT_MAX_ROWS + 1; e += 32) o.lagr[e] = 0.0;
    __syncwarp();
    for (int j = lane; j < q && !r.fail; j += 32) o.lagr[1 + s.W[j]] = s.u[j];
    if (lane < 6) {
      // LinearizedInvertedPendulum2D::OneIteration with T = QP period (LinearizedInvertedPendulum2D.cpp:230-264)
      const int ax = lane / 3, c = lane % 3;
      const double T = C.P.T;
      const double *cm = ax ? s.in.com_y : s.in.com_x;
      const double jk = s.jr[ax][0];
      double v;
      if (c == 0) v = cm[0] + T * cm[1] + T * T / 2.0 * cm[2] + jk * (T * T * T / 6.0);
      else if (c == 1) v = cm[1] + T * cm[2] + jk * (T * T / 2.0);
      else v = cm[2] + jk * T;
      (ax ? o.com_next_y : o.com_next_x)[c] = v;
    }
    if (lane == 0) { o.n_vars = r.n_vars; o.n_rows = r.n_rows; o.fail = r.fail; o.iterations = r.iterations; }
    __syncwarp();
  }
}

}  // namespace

void wg_herdt_release(wg_ctx *ctx)
{
  if (!ctx->herdt) return;
  HerdtState *st = static_cast<HerdtState *>(ctx->herdt);
  cudaFree(st->d_consts); cudaFree(st->d_in); cudaFree(st->d_out); cudaFree(st->d_next); cudaFree(st->d_T); cudaFree(st->d_act);
  if (st->up) cudaStreamDestroy(st->up);
  if (st->down) cudaStreamDestroy(st->down);
  for (int c = 0; c < 2; ++c) { if (st->ev_up[c]) cudaEventDestroy(st->ev_up[c]); if (st->ev_k[c]) cudaEventDestroy(st->ev_k[c]); }
  if (st->ev0) cudaEventDestroy(st->ev0);
  delete st;
  ctx->herdt = nullptr;
}

// used by herdt_mpc.cu
const herdt::Consts *wg_herdt_device_consts(wg_ctx *ctx)
{
  HerdtState *st = static_cast<HerdtState *>(ctx->herdt);
  return (st && st->ready) ? st->d_consts : nullptr;
}
const herdt::Consts *wg_herdt_host_consts(wg_ctx *ctx)
{
  HerdtState *st = static_cast<HerdtState *>(ctx->herdt);
  return (st && st->ready) ? &st->h_consts : nullptr;
}

extern "C" {

void wg_herdt_default_params(double sole_length, double sole_width, wg_herdt_params *p)
{
  if (!p) return;
  std::memset(p, 0, sizeof *p);
  p->T = 0.1;                 // QP_T_,  ZMPVelocityReferencedQP.cpp:63
  p->com_height = 0.814;      // CoMHeight_ of the QP model, ZMPVelocityReferencedQP.cpp:103
  p->w_jerk = 0.00001;        // ZMPVelocityReferencedQP.cpp:118
  p->w_vel = 1.0;             // :116
  p->w_cop = 0.000001;        // :117
  p->cop_half_x = 0.5 * sole_length - 0.04;   // FootHalfSize.cpp:62-68, margins relative-feet-inequalities.cpp:47-49
  p->cop_half_y = 0.5 * sole_width - 0.04;
  p->ds_feet_distance = 0.2;  // relative-feet-inequalities.cpp:45
  const double X[5] = {-0.28, -0.2, 0.0, 0.2, 0.28}, Y[5] = {-0.2, -0.3, -0.4, -0.3, -0.2};  // :51-52
  for (int i = 0; i < 5; ++i) { p->foot_hull_x[i] = X[i]; p->foot_hull_y[i] = Y[i]; }
  p->lipm_T = 0.005;
}

int wg_herdt_set_params(wg_ctx *ctx, const wg_herdt_params *params)
{
  if (!ctx || !params || !(params->T > 0.0) || !(params->w_jerk > 0.0) || !(params->w_cop > 0.0))
    return WG_ERR_INVALID;
  wg_device_guard guard(ctx->device);
  HerdtState *st = state_of(ctx);
  compute_consts(*params, st->h_consts);
  if (!st->d_consts) WG_CUDA(ctx, cudaMalloc(&st->d_consts, sizeof(Consts)));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  WG_CUDA(ctx, cudaMemcpy(st->d_consts, &st->h_consts, sizeof(Consts), cudaMemcpyHostToDevice));
  st->ready = true;
  return WG_OK;
}

static int herdt_launch(wg_ctx *ctx, HerdtState *st, int B, const wg_herdt_qp_input *d_in, wg_herdt_qp_output *d_out,
                        const herdt::LaunchOpts &opt = herdt::LaunchOpts())
{
  const size_t smem = sizeof(herdt::Work) * QP_WARPS;
  WG_SMEM_ATTR(ctx, herdt_qp_kernel, smem);
  int per_sm = (int)((227 * 1024) / (smem + 1024));
  if (per_sm < 1) per_sm = 1;
  int blocks = (B + QP_WARPS - 1) / QP_WARPS;
  const int cap = ctx->sm_count * per_sm;
  if (blocks > cap) blocks = cap;   // persistent: a multiple of the SM count, grid-stride over instances
  if (!st->d_next) WG_CUDA(ctx, cudaMalloc(&st->d_next, sizeof(int)));
  int rc = wgi_grow_scratch(ctx, reinterpret_cast<void **>(&st->d_T), &st->cap_T, sizeof(double) * blocks * QP_WARPS * herdt::TRI);
  if (rc != WG_OK) return rc;
  WG_CUDA(ctx, cudaMemsetAsync(st->d_next, 0, sizeof(int), ctx->stream));
  wg_prof_start(ctx, WG_K_HERDT_QP);
  herdt_qp_kernel<<<blocks, QP_WARPS * 32, smem, ctx->stream>>>(B, st->d_consts, d_in, d_out, st->d_next, st->d_T, opt);
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  return WG_OK;
}

int wg_herdt_qp_solve_batch(wg_ctx *ctx, int mem, int B, const wg_herdt_qp_input *in, wg_herdt_qp_output *out)
{
  if (!ctx || B < 0 || (B > 0 && (!in || !out))) return WG_ERR_INVALID;
  HerdtState *st = state_of(ctx);
  if (!st->ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_herdt_set_params not called");
  if (B == 0) return WG_OK;
  wg_device_guard guard(ctx->device);
  if (mem == WG_MEM_DEVICE) return herdt_launch(ctx, st, B, in, out);
  if (mem != WG_MEM_HOST) return WG_ERR_INVALID;
  int rc;
  if ((rc = wgi_grow_scratch(ctx, reinterpret_cast<void **>(&st->d_in), &st->cap_in, sizeof(wg_herdt_qp_input) * (size_t)B)) != WG_OK ||
      (rc = wgi_grow_scratch(ctx, reinterpret_cast<void **>(&st->d_out), &st->cap_out, sizeof(wg_herdt_qp_output) * (size_t)B)) != WG_OK)
    return rc;
  // at most two large chunks (small launches waste the tail of the persistent grid: 8 chunks of 2048 measured 18 % SLOWER than
  // the unpipelined call): the upload of chunk c+1 and the download of chunk c-1 overlap the kernel of chunk c
  if (!st->up) {
    WG_CUDA(ctx, cudaStreamCreateWithFlags(&st->up, cudaStreamNonBlocking));
    WG_CUDA(ctx, cudaStreamCreateWithFlags(&st->down, cudaStreamNonBlocking));
    for (int c = 0; c < 2; ++c) {
      WG_CUDA(ctx, cudaEventCreateWithFlags(&st->ev_up[c], cudaEventDisableTiming));
      WG_CUDA(ctx, cudaEventCreateWithFlags(&st->ev_k[c], cudaEventDisableTiming));
    }
    WG_CUDA(ctx, cudaEventCreateWithFlags(&st->ev0, cudaEventDisableTiming));
  }
  const int nch = std::max(1, std::min(2, B / 4096));
  WG_CUDA(ctx, cudaEventRecord(st->ev0, ctx->stream));
  WG_CUDA(ctx, cudaStreamWaitEvent(st->up, st->ev0, 0));
  for (int c = 0; c < nch; ++c) {
    const size_t b0 = (size_t)B * c / nch, b1 = (size_t)B * (c + 1) / nch;
    WG_CUDA(ctx, cudaMemcpyAsync(st->d_in + b0, in + b0, sizeof(wg_herdt_qp_input) * (b1 - b0), cudaMemcpyHostToDevice, st->up));
    WG_CUDA(ctx, cudaEventRecord(st->ev_up[c], st->up));
    WG_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, st->ev_up[c], 0));
    if ((rc = herdt_launch(ctx, st, (int)(b1 - b0), st->d_in + b0, st->d_out + b0)) != WG_OK) return rc;
    WG_CUDA(ctx, cudaEventRecord(st->ev_k[c], ctx->stream));
    WG_CUDA(ctx, cudaStreamWaitEvent(st->down, st->ev_k[c], 0));
    WG_CUDA(ctx, cudaMemcpyAsync(out + b0, st->d_out + b0, sizeof(wg_herdt_qp_output) * (b1 - b0), cudaMemcpyDeviceToHost, st->down));
  }
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  WG_CUDA(ctx, cudaStreamSynchronize(st->down));
  return WG_OK;
}

int wg_herdt_qp_solve_batch_warm(wg_ctx *ctx, int mem, int B, const wg_herdt_qp_input *in, wg_herdt_qp_output *out,
                                 const wg_herdt_active_set *guess, int age, wg_herdt_active_set *active_out)
{
  if (!ctx || B < 0 || age < 0 || (B > 0 && (!in || !out))) return WG_ERR_INVALID;
  HerdtState *st = state_of(ctx);
  if (!st->ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_herdt_set_params not called");
  if (B == 0) return WG_OK;
  wg_device_guard guard(ctx->device);
  herdt::LaunchOpts opt;
  opt.age = age;
  opt.guess_stride = opt.active_stride = sizeof(wg_herdt_active_set);
  if (mem == WG_MEM_DEVICE) {
    opt.guess = reinterpret_cast<const unsigned char *>(guess);
    opt.active_out = reinterpret_cast<unsigned char *>(active_out);
    return herdt_launch(ctx, st, B, in, out, opt);
  }
  if (mem != WG_MEM_HOST) return WG_ERR_INVALID;
  int rc;
  if ((rc = wgi_grow_scratch(ctx, reinterpret_cast<void **>(&st->d_in), &st->cap_in, sizeof(wg_herdt_qp_input) * (size_t)B)) != WG_OK ||
      (rc = wgi_grow_scratch(ctx, reinterpret_cast<void **>(&st->d_out), &st->cap_out, sizeof(wg_herdt_qp_output) * (size_t)B)) != WG_OK)
    return rc;
  if ((rc = wgi_grow_scratch(ctx, reinterpret_cast<void **>(&st->d_act), &st->cap_act, sizeof(wg_herdt_active_set) * (size_t)B)) != WG_OK)
    return rc;
  WG_CUDA(ctx, cudaMemcpyAsync(st->d_in, in, sizeof(wg_herdt_qp_input) * (size_t)B, cudaMemcpyHostToDevice, ctx->stream));
  if (guess) {
    WG_CUDA(ctx, cudaMemcpyAsync(st->d_act, guess, sizeof(wg_herdt_active_set) * (size_t)B, cudaMemcpyHostToDevice, ctx->stream));
    opt.guess = reinterpret_cast<const unsigned char *>(st->d_act);
  }
  opt.active_out = reinterpret_cast<unsigned char *>(st->d_act);
  rc = herdt_launch(ctx, st, B, st->d_in, st->d_out, opt);
  if (rc != WG_OK) return rc;
  WG_CUDA(ctx, cudaMemcpyAsync(out, st->d_out, sizeof(wg_herdt_qp_output) * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream));
  if (active_out)
    WG_CUDA(ctx, cudaMemcpyAsync(active_out, st->d_act, sizeof(wg_herdt_active_set) * (size_t)B, cudaMemcpyDeviceToHost, ctx->stream));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return WG_OK;
}

}  // extern "C"

// used by herdt_mpc.cu: the solve of one closed-loop period on device-resident records, skipping the instances that do not
// fire, warm started from / writing back the active set kept in each instance's state
int wg_herdt_qp_solve_device(wg_ctx *ctx, int B, const wg_herdt_qp_input *in, wg_herdt_qp_output *out,
                             const herdt::LaunchOpts &opt)
{
  HerdtState *st = state_of(ctx);
  if (!st->ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_herdt_set_params not called");
  return herdt_launch(ctx, st, B, in, out, opt);
}
