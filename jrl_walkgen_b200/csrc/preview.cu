// preview.cu - batched Kajita2003 cart-table preview control for sm_100a.
//
// Replaces PreviewControl::OneIterationOfPreview (src/PreviewControl/PreviewControl.cpp:324-374) and
// its 1-D variants (:376-484) for whole ragged batches of trajectories, and the host-side gain
// computation PreviewControl::ComputeOptimalWeights (:198-322) / OptimalControllerSolver::ComputeWeights
// (src/PreviewControl/OptimalControllerSolver.cpp:200-352).
//
// B200-first restructuring.  The reference evaluates, per 5 ms tick and per axis,
//     u = -Kx.x + Ks.s + sum_{i<NL} F[i] * p[k+i]          (640 MACs through a deque of 48-byte structs)
// and then the 3-state update.  One kernel, preview_fused_kernel, does all of it; one CTA owns one
// trajectory and walks it in tiles of 8 x (threads per CTA) ticks (512 by default):
//   (1) FIR.  The preview sum does not depend on the state, so it is a FIR filter of the ZMP reference
//       (>94% of the flops: 1280 of 1360 per step).  Each thread produces R=8 consecutive outputs for
//       both axes from a register-resident sliding window: per tap it issues ONE 128-bit shared-memory
//       load and 16 DFMAs, so the FP64 pipe (64 DFMA/clk/SM), not the LSU, is the limiter.  The ZMP tile
//       is staged once per tile in shared memory (coalesced 128-bit global loads) with a 9/8 padding so
//       that the stride-8 per-thread windows are bank-conflict free.
//   (2) Recursion as a scan.  Per axis the controller is the linear recurrence X' = M X + g_k on the
//       4-state X = (x, dx, ddx, s) with a CONSTANT closed-loop matrix M (spectral radius 0.983), so the
//       serial chain of the reference is replaced by: every thread runs its 8 ticks from a zero state
//       (thread 0: from the carried state) in the reference's statement order; a Kogge-Stone scan over the
//       CTA's threads combines them with the constant matrices M^(8 d), d = 1..32 (warp shuffles inside a warp,
//       one shared-memory exchange of the four warp totals across warps); every thread then re-runs its 8 ticks from its true start state and
//       emits CoM and ZMP.  The last tick's state is carried to the next tile in shared memory.
//   (3) Stores.  A lane owns 8 consecutive ticks (the sliding window wants that), which is the worst layout for
//       stores (32 lines per instruction); CoM/ZMP rows are therefore staged two ticks at a time in the dead tile
//       buffer and written with consecutive lanes on consecutive 16 bytes.
// The FIR result never goes to HBM: traffic is the streaming minimum (16 B in per tick + the NL-sample
// halo once per tile, 64 B out).
//
#include "wg_common.h"
#include <atomic>
#include <mutex>
#include <cstdlib>
#include <vector>
#include <cmath>
#include <algorithm>
#include <type_traits>

// ---------------------------------------------------------------------------------------------
// Host: gains by structure-preserving doubling (SDA) for the DARE
//     P = A'PA - A'Pb (R + b'Pb)^-1 b'PA + c'Qc
// ---------------------------------------------------------------------------------------------
#define WG_HD __host__ __device__

namespace {

struct Mat {  // tiny dense n x n (n <= 4), row-major
  int n;
  double a[16];
  WG_HD double &operator()(int i, int j) { return a[i * n + j]; }
  WG_HD double operator()(int i, int j) const { return a[i * n + j]; }
};

WG_HD Mat mat_zero(int n)
{
  Mat C;
  C.n = n;
  for (int i = 0; i < 16; ++i) C.a[i] = 0.0;
  return C;
}
WG_HD Mat mm(const Mat &A, const Mat &B)
{
  Mat C = mat_zero(A.n);
  for (int i = 0; i < A.n; ++i)
    for (int j = 0; j < A.n; ++j) {
      double s = 0;
      for (int k = 0; k < A.n; ++k) s += A(i, k) * B(k, j);
      C(i, j) = s;
    }
  return C;
}
WG_HD Mat tr(const Mat &A)
{
  Mat C = mat_zero(A.n);
  for (int i = 0; i < A.n; ++i)
    for (int j = 0; j < A.n; ++j) C(i, j) = A(j, i);
  return C;
}
WG_HD Mat add(const Mat &A, const Mat &B)
{
  Mat C = mat_zero(A.n);
  for (int i = 0; i < A.n * A.n; ++i) C.a[i] = A.a[i] + B.a[i];
  return C;
}
// X = W^-1 B by Gaussian elimination with partial pivoting.
WG_HD bool solve(Mat W, Mat B, Mat &X)
{
  int n = W.n;
  for (int c = 0; c < n; ++c) {
    int piv = c;
    for (int r = c + 1; r < n; ++r)
      if (fabs(W(r, c)) > fabs(W(piv, c))) piv = r;
    if (W(piv, c) == 0.0) return false;
    if (piv != c)
      for (int j = 0; j < n; ++j) {
        double t = W(piv, j); W(piv, j) = W(c, j); W(c, j) = t;
        t = B(piv, j); B(piv, j) = B(c, j); B(c, j) = t;
      }
    for (int r = c + 1; r < n; ++r) {
      double f = W(r, c) / W(c, c);
      for (int j = c; j < n; ++j) W(r, j) -= f * W(c, j);
      for (int j = 0; j < n; ++j) B(r, j) -= f * B(c, j);
    }
  }
  X.n = n;
  for (int j = 0; j < n; ++j)
    for (int r = n - 1; r >= 0; --r) {
      double s = B(r, j);
      for (int k = r + 1; k < n; ++k) s -= W(r, k) * X(k, j);
      X(r, j) = s / W(r, r);
    }
  return true;
}

WG_HD bool dare_sda(const Mat &A0, const double *b, const double *c, double Q, double R, Mat &P)
{
  int n = A0.n;
  Mat A = A0, G = mat_zero(n), H = mat_zero(n), I = mat_zero(n);
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) {
      G(i, j) = b[i] * b[j] / R;
      H(i, j) = c[i] * Q * c[j];
      I(i, j) = (i == j);
    }
  for (int it = 0; it < 200; ++it) {
    Mat W = add(I, mm(G, H));
    Mat WiA = mat_zero(n), WiG = mat_zero(n);
    if (!solve(W, A, WiA)) return false;   // W^-1 A
    if (!solve(W, G, WiG)) return false;   // W^-1 G
    Mat At = tr(A);
    Mat A1 = mm(A, WiA);
    Mat G1 = add(G, mm(mm(A, WiG), At));
    Mat H1 = add(H, mm(mm(At, H), WiA));
    double diff = 0, norm = 0;
    for (int i = 0; i < n * n; ++i) {
      diff = fmax(diff, fabs(H1.a[i] - H.a[i]));
      norm = fmax(norm, fabs(H1.a[i]));
    }
    A = A1; G = G1; H = H1;
    if (diff <= 1e-16 * norm) break;
  }
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) P(i, j) = 0.5 * (H(i, j) + H(j, i));
  P.n = n;
  return true;
}

// PreviewControl::ComputeOptimalWeights + OptimalControllerSolver::ComputeWeights for one (T, preview time, zc, mode):
// the head (A, B, C, Kx, Ks) and the NL window weights.  Host (wg_preview_gains) and device (preview_gains_kernel, one
// thread per parameter set) run this same code.
WG_HD int gains_core(double T, double preview_time, double zc, int mode, wg_preview_gains_head *out, double *F, int f_cap)
{
  if (!(T > 0.0) || !(preview_time > 0.0)) return WG_ERR_INVALID;
  const int NL = (int)(preview_time / T);
  if (NL <= 0 || NL > WG_PREVIEW_MAX_NL || NL > f_cap) return WG_ERR_INVALID;
  out->T = T; out->preview_time = preview_time; out->zc = zc; out->mode = mode; out->NL = NL;
  const double A[9] = {1.0, T, T * T / 2.0, 0.0, 1.0, T, 0.0, 0.0, 1.0};
  const double B[3] = {T * T * T / 6.0, T * T / 2.0, T};
  const double C[3] = {1.0, 0.0, -zc / 9.81};
  for (int i = 0; i < 9; ++i) out->A[i] = A[i];
  for (int i = 0; i < 3; ++i) { out->B[i] = B[i]; out->C[i] = C[i]; out->Kx[i] = 0.0; }
  out->Ks = 0.0;

  Mat Ax = mat_zero(0);
  double bx[4] = {0, 0, 0, 0}, cx[4] = {0, 0, 0, 0}, Q = 1.0, R;
  if (mode == WG_PREVIEW_MODE_WITHOUT_INITIALPOS) {
    // augmented (integrated error, state increment) system, PreviewControl.cpp:237-262
    R = 1e-6;
    Ax.n = 4;
    Ax(0, 0) = 1.0;
    for (int j = 0; j < 3; ++j) {
      double s = 0;
      for (int l = 0; l < 3; ++l) s += C[l] * A[l * 3 + j];
      Ax(0, j + 1) = s;
      for (int i = 0; i < 3; ++i) Ax(i + 1, j + 1) = A[i * 3 + j];
    }
    for (int l = 0; l < 3; ++l) { bx[0] += C[l] * B[l]; bx[l + 1] = B[l]; }
    cx[0] = 1.0;
  } else if (mode == WG_PREVIEW_MODE_WITH_INITIALPOS) {
    R = 1e-5;
    Ax.n = 3;
    for (int i = 0; i < 9; ++i) Ax.a[i] = A[i];
    for (int i = 0; i < 3; ++i) { bx[i] = B[i]; cx[i] = C[i]; }
  } else {
    return WG_ERR_INVALID;
  }
  int n = Ax.n;
  Mat P = mat_zero(n);
  if (!dare_sda(Ax, bx, cx, Q, R, P)) return WG_ERR_INVALID;

  double Pb[4] = {0, 0, 0, 0}, bPb = 0;
  for (int i = 0; i < n; ++i) {
    for (int j = 0; j < n; ++j) Pb[i] += P(i, j) * bx[j];
  }
  for (int i = 0; i < n; ++i) bPb += bx[i] * Pb[i];
  const double la = 1.0 / (R + bPb);
  Mat PA = mm(P, Ax);
  double K[4] = {0, 0, 0, 0};
  for (int j = 0; j < n; ++j) {
    double s = 0;
    for (int l = 0; l < n; ++l) s += bx[l] * PA(l, j);
    K[j] = s * la;
  }
  // F[k] = la b' ((A - bK)')^k (P c'Q | c'Q)
  double rec[4] = {0, 0, 0, 0}, nxt[4];
  for (int i = 0; i < n; ++i) rec[i] = cx[i] * Q;
  if (mode == WG_PREVIEW_MODE_WITHOUT_INITIALPOS) {
    for (int i = 0; i < n; ++i) { nxt[i] = 0; for (int j = 0; j < n; ++j) nxt[i] += P(i, j) * rec[j]; }
    for (int i = 0; i < n; ++i) rec[i] = nxt[i];
  }
  for (int k = 0; k < NL; ++k) {
    double s = 0;
    for (int l = 0; l < n; ++l) s += la * bx[l] * rec[l];
    F[k] = s;
    for (int i = 0; i < n; ++i) {
      nxt[i] = 0;
      for (int j = 0; j < n; ++j) nxt[i] += (Ax(j, i) - bx[j] * K[i]) * rec[j];
    }
    for (int i = 0; i < n; ++i) rec[i] = nxt[i];
  }
  out->Ks = K[0];
  if (mode == WG_PREVIEW_MODE_WITHOUT_INITIALPOS)
    for (int i = 0; i < 3; ++i) out->Kx[i] = K[i + 1];
  else
    for (int i = 0; i < 3; ++i) out->Kx[i] = K[i];
  return WG_OK;
}

}  // namespace

extern "C" int wg_preview_gains(double T, double preview_time, double zc, int mode, wg_preview_gains_t *out)
{
  if (!out) return WG_ERR_INVALID;
  std::memset(out, 0, sizeof *out);
  wg_preview_gains_head h;
  const int rc = gains_core(T, preview_time, zc, mode, &h, out->F, WG_PREVIEW_MAX_NL);
  if (rc != WG_OK) return rc;
  std::memcpy(out->A, h.A, sizeof h.A); std::memcpy(out->B, h.B, sizeof h.B); std::memcpy(out->C, h.C, sizeof h.C);
  std::memcpy(out->Kx, h.Kx, sizeof h.Kx);
  out->Ks = h.Ks; out->T = T; out->preview_time = preview_time; out->zc = zc; out->mode = mode; out->NL = h.NL;
  return WG_OK;
}

// Batched gains (SURVEY 8f rank 4): one thread per (T, preview time, zc).  ~20 doubling steps on 4 x 4 matrices and an
// NL-step 4-vector recursion per instance: a few 10^4 flops, register / local-memory resident.
__global__ void __launch_bounds__(64)
preview_gains_kernel(int B, const double *__restrict__ params, int mode, wg_preview_gains_head *__restrict__ heads,
                     double *__restrict__ F, long long f_stride)
{
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  wg_preview_gains_head h;
  const int rc = gains_core(params[3 * (size_t)b], params[3 * (size_t)b + 1], params[3 * (size_t)b + 2], mode, &h,
                            F + (size_t)b * f_stride, (int)(f_stride > WG_PREVIEW_MAX_NL ? WG_PREVIEW_MAX_NL : f_stride));
  if (rc != WG_OK) {
    h.NL = 0; h.mode = mode; h.Ks = 0.0 / 0.0;
    h.T = params[3 * (size_t)b]; h.preview_time = params[3 * (size_t)b + 1]; h.zc = params[3 * (size_t)b + 2];
  }
  heads[b] = h;
}

extern "C" int wg_preview_gains_batch(wg_ctx *ctx, int mem, int B, const double *params, int mode,
                                      wg_preview_gains_head *heads, double *F, long long f_stride)
{
  if (!ctx || B < 0 || f_stride <= 0 || (B > 0 && (!params || !heads || !F))) return WG_ERR_INVALID;
  if (mode != WG_PREVIEW_MODE_WITHOUT_INITIALPOS && mode != WG_PREVIEW_MODE_WITH_INITIALPOS) return WG_ERR_INVALID;
  if (B == 0) return WG_OK;
  wg_device_guard guard(ctx->device);
  const double *d_par = params; wg_preview_gains_head *d_heads = heads; double *d_F = F;
  void *tmp = nullptr;
  const size_t nb = (size_t)B, bytes_par = sizeof(double) * 3 * nb, bytes_h = sizeof(wg_preview_gains_head) * nb,
               bytes_F = sizeof(double) * nb * (size_t)f_stride;
  if (mem == WG_MEM_HOST) {
    WG_CUDA(ctx, cudaMalloc(&tmp, bytes_par + bytes_h + bytes_F));
    d_par = static_cast<double *>(tmp);
    d_heads = reinterpret_cast<wg_preview_gains_head *>(static_cast<char *>(tmp) + bytes_par);
    d_F = reinterpret_cast<double *>(static_cast<char *>(tmp) + bytes_par + bytes_h);
    cudaError_t e = cudaMemcpyAsync(tmp, params, bytes_par, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_F, 0, bytes_F, ctx->stream);
    if (e != cudaSuccess) { cudaFree(tmp); return wg_fail(ctx, WG_ERR_CUDA, "wg_preview_gains_batch", e); }
  } else if (mem != WG_MEM_DEVICE) return WG_ERR_INVALID;
  preview_gains_kernel<<<(B + 63) / 64, 64, 0, ctx->stream>>>(B, d_par, mode, d_heads, d_F, f_stride);
  ctx->launches++;
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess && mem == WG_MEM_HOST) {
    e = cudaMemcpyAsync(heads, d_heads, bytes_h, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(F, d_F, bytes_F, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  }
  if (tmp) cudaFree(tmp);
  if (e != cudaSuccess) return wg_fail(ctx, WG_ERR_CUDA, "wg_preview_gains_batch", e);
  return WG_OK;
}

// ---------------------------------------------------------------------------------------------
// Device side
// ---------------------------------------------------------------------------------------------
constexpr int FIR_R = 8;                      // ticks per thread
constexpr int SCAN_LEVELS = 6;                // M^(8 d), d = 1, 2, 4, ..., 32 threads

struct PreviewConsts {
  double A[9], B[3], C[3], Kx[3], Ks;
  int NL, NLpad;
  // P[sim][l] = M_sim^(FIR_R * 2^l), row-major 4x4; M_sim is the closed-loop one-tick matrix of the
  // 4-state (x, dx, ddx, s) with (sim = 1) or without (sim = 0) the integrated-error update.
  double P[2][SCAN_LEVELS][16];
  // One tick is X' = M X + g f + h p (f = preview sum, p = ZMP reference of the tick).  State after the FIR_R ticks
  // of a thread started from zero: sum_r G[sim][r] f_r + H[sim][r] p_r with G[r] = M^(FIR_R-1-r) g, same for H.
  double G[2][FIR_R][4], H[2][FIR_R][4];
  // ---- recursive evaluation of the preview sum (preview_rec_kernel; see rec_setup): the window weights of
  // OptimalControllerSolver::ComputeWeights are F[i] = w' L^i v with L = (A - b K)' (OptimalControllerSolver.cpp:323-345), so
  // W_k = sum_{i<NL} L^i v p[k+i] obeys the BACKWARD recurrence W_k = L W_{k+1} + v p[k] - (L^NL v) p[k+NL], f_k = w' W_k.
  double RF0[FIR_R], RFN[FIR_R];       // w' L^i v and w' L^(NL+i) v, i < FIR_R: the local triangular sums of a thread
  double RV[FIR_R][4], RVN[FIR_R][4];  // L^r v and L^(NL+r) v: a thread's local total sum_r RV[r] p[r] - RVN[r] p[r+NL]
  double RW[FIR_R + 1][4];             // rows w' L^j, j = 0..FIR_R: tick r of a thread adds RW[FIR_R - r] . W_in
  double RP[SCAN_LEVELS][16];          // L^(FIR_R 2^l), row-major
};
__constant__ PreviewConsts c_pc;
__constant__ double c_F[WG_PREVIEW_MAX_NL + 8];

// The FIR taps are DFMA operands straight from the constant bank (no load instruction in the inner loop), so the gains
// live in ONE __constant__ block per device, while gains belong to a context.  Every context keeps a host image of the
// block; preview_bind() (called under g_pv_mutex right before each launch) re-uploads it when the block currently holds
// another context's gains (or older gains of this one), after draining the device so that no running kernel sees the
// switch.  Two contexts on one GPU with different gains therefore stay correct; they just do not overlap.
namespace {
struct PreviewImage {
  PreviewConsts pc;
  double F[WG_PREVIEW_MAX_NL + 8];
};
std::mutex g_pv_mutex;
std::atomic<unsigned long long> g_pv_gen_counter{0};
unsigned long long g_pv_bound[64];   // generation of the gains held by each device's __constant__ block (0 = none)

int preview_bind(wg_ctx *ctx)
{
  if (ctx->device < 0 || ctx->device >= 64) return WG_ERR_INVALID;
  if (g_pv_bound[ctx->device] == ctx->preview_gen) return WG_OK;
  const PreviewImage *im = reinterpret_cast<const PreviewImage *>(ctx->preview_image.data());
  WG_CUDA(ctx, cudaDeviceSynchronize());
  WG_CUDA(ctx, cudaMemcpyToSymbol(c_pc, &im->pc, sizeof im->pc));
  WG_CUDA(ctx, cudaMemcpyToSymbol(c_F, im->F, sizeof im->F));
  g_pv_bound[ctx->device] = ctx->preview_gen;
  return WG_OK;
}
}  // namespace

constexpr int PV_MAX_CHUNKS = 16;

struct wg_preview_plan {
  wg_ctx *ctx;
  int B;
  int NL;
  int64_t total_samples, total_steps;
  int64_t *d_offsets;
  int *d_order;        // trajectories sorted by decreasing length (longest CTAs are scheduled first)
  // staging buffers for WG_MEM_HOST calls
  double *d_zmp, *d_state, *d_com, *d_zmpout, *d_add;
  // WG_MEM_HOST pipeline: chunk c = trajectories [chunk_first[c], chunk_first[c+1]) (contiguous sample ranges); its
  // upload, kernel and downloads run on three streams so that H2D, compute and D2H of different chunks overlap
  int n_chunks;
  int chunk_first[PV_MAX_CHUNKS + 1];
  int64_t chunk_samp[PV_MAX_CHUNKS + 1];   // offsets[chunk_first[c]]
  int *d_order_chunked;                    // trajectories sorted by decreasing length inside each chunk
  cudaStream_t up_stream, down_stream;
  cudaEvent_t ev_up[PV_MAX_CHUNKS], ev_k[PV_MAX_CHUNKS], ev_done;
};

__device__ __forceinline__ int pad9(int e) { return e + (e >> 3); }
__device__ __forceinline__ int swz8(int e) { return e ^ ((e >> 3) & 7); }   // XOR swizzle of 16-byte slots in groups of 8

// One tick of OneIterationOfPreview for one axis, in the reference's statement order
// (PreviewControl.cpp:346-367): u, x <- A x + B u, zmp = C x, s += p - zmp.
struct Axis {
  double x0, x1, x2, s;
};
template <bool SIM>
__device__ __forceinline__ double preview_tick(Axis &a, double f, double pk)
{
  double r = c_pc.Kx[0] * a.x0;
  r = fma(c_pc.Kx[1], a.x1, r);
  r = fma(c_pc.Kx[2], a.x2, r);
  const double u = fma(c_pc.Ks, a.s, -r) + f;
  // A = [[1,T,T^2/2],[0,1,T],[0,0,1]]
  const double n0 = fma(c_pc.A[2], a.x2, fma(c_pc.A[1], a.x1, a.x0));
  const double n1 = fma(c_pc.A[5], a.x2, a.x1);
  a.x0 = fma(u, c_pc.B[0], n0);
  a.x1 = fma(u, c_pc.B[1], n1);
  a.x2 = fma(u, c_pc.B[2], a.x2);
  const double z = fma(c_pc.C[2], a.x2, fma(c_pc.C[1], a.x1, c_pc.C[0] * a.x0));
  if (SIM) a.s += (pk - z);
  return z;
}

__device__ __forceinline__ Axis axis_zero()
{
  Axis a;
  a.x0 = a.x1 = a.x2 = a.s = 0.0;
  return a;
}
__device__ __forceinline__ void operator+=(Axis &a, const Axis &b)
{
  a.x0 += b.x0; a.x1 += b.x1; a.x2 += b.x2; a.s += b.s;
}
// c += g a, component by component
__device__ __forceinline__ void axpy(Axis &c, const double *g, double a)
{
  c.x0 = fma(g[0], a, c.x0); c.x1 = fma(g[1], a, c.x1);
  c.x2 = fma(g[2], a, c.x2); c.s = fma(g[3], a, c.s);
}
__device__ __forceinline__ Axis shfl_up(const Axis &a, int d)
{
  Axis r;
  r.x0 = __shfl_up_sync(0xffffffffu, a.x0, d); r.x1 = __shfl_up_sync(0xffffffffu, a.x1, d);
  r.x2 = __shfl_up_sync(0xffffffffu, a.x2, d); r.s = __shfl_up_sync(0xffffffffu, a.s, d);
  return r;
}
__device__ __forceinline__ Axis shfl_down(const Axis &a, int d)
{
  Axis r;
  r.x0 = __shfl_down_sync(0xffffffffu, a.x0, d); r.x1 = __shfl_down_sync(0xffffffffu, a.x1, d);
  r.x2 = __shfl_down_sync(0xffffffffu, a.x2, d); r.s = __shfl_down_sync(0xffffffffu, a.s, d);
  return r;
}
// The two records of 8 doubles: a walk's state {x,dx,ddx,y,dy,ddy,sx,sy} (state arrays, s_carry) and a scan total
// {x axis, y axis} (s_tot, s_totb, s_halo).
__device__ __forceinline__ void load_state(const double *q, Axis &x, Axis &y)
{
  x.x0 = q[0]; x.x1 = q[1]; x.x2 = q[2]; x.s = q[6];
  y.x0 = q[3]; y.x1 = q[4]; y.x2 = q[5]; y.s = q[7];
}
__device__ __forceinline__ void store_state(double *q, const Axis &x, const Axis &y)
{
  q[0] = x.x0; q[1] = x.x1; q[2] = x.x2; q[6] = x.s;
  q[3] = y.x0; q[4] = y.x1; q[5] = y.x2; q[7] = y.s;
}
__device__ __forceinline__ void load_pair(const double *q, Axis &x, Axis &y)
{
  x.x0 = q[0]; x.x1 = q[1]; x.x2 = q[2]; x.s = q[3];
  y.x0 = q[4]; y.x1 = q[5]; y.x2 = q[6]; y.s = q[7];
}
__device__ __forceinline__ void store_pair(double *q, const Axis &x, const Axis &y)
{
  q[0] = x.x0; q[1] = x.x1; q[2] = x.x2; q[3] = x.s;
  q[4] = y.x0; q[5] = y.x1; q[6] = y.x2; q[7] = y.s;
}

// c += P n, P a row-major 4 x 4 matrix
__device__ __forceinline__ void scan_combine(Axis &c, const double *__restrict__ P, const Axis &n)
{
  c.x0 = fma(P[0], n.x0, fma(P[1], n.x1, fma(P[2], n.x2, fma(P[3], n.s, c.x0))));
  c.x1 = fma(P[4], n.x0, fma(P[5], n.x1, fma(P[6], n.x2, fma(P[7], n.s, c.x1))));
  c.x2 = fma(P[8], n.x0, fma(P[9], n.x1, fma(P[10], n.x2, fma(P[11], n.s, c.x2))));
  c.s = fma(P[12], n.x0, fma(P[13], n.x1, fma(P[14], n.x2, fma(P[15], n.s, c.s))));
}

// ---- Phases shared by the kernels below (the phase numbers are those of their comments).
// (2a) local aggregate: the cart-table state after a thread's FIR_R ticks started from zero, as the linear map of its inputs
// (preview sums ax / ay, ZMP reference pk); the thread that owns the tile's first tick (carry_in) adds M^8 x the carried state,
// which it also returns in (inx, iny).
template <bool SIM>
__device__ __forceinline__ void local_aggregate(const double *ax, const double *ay, const double2 *pk, bool carry_in,
                                                const double *s_carry, const double (*Pm)[16], Axis &cx, Axis &cy,
                                                Axis &inx, Axis &iny)
{
  cx = axis_zero(); cy = axis_zero();
  inx = cx; iny = cy;
  const double(*Gm)[4] = c_pc.G[SIM ? 1 : 0];
  const double(*Hm)[4] = c_pc.H[SIM ? 1 : 0];
#pragma unroll
  for (int r = 0; r < FIR_R; ++r) {
    axpy(cx, Gm[r], ax[r]);
    axpy(cy, Gm[r], ay[r]);
    if (SIM) {
      axpy(cx, Hm[r], pk[r].x);
      axpy(cy, Hm[r], pk[r].y);
    }
  }
  if (carry_in) {
    load_state(s_carry, inx, iny);
    scan_combine(cx, Pm[0], inx);
    scan_combine(cy, Pm[0], iny);
  }
}

// (2b) Kogge-Stone scan UP the lanes of a warp: c_t += M^(8d) c_{t-d}
__device__ __forceinline__ void scan_up(Axis &cx, Axis &cy, int lane, const double (*Pm)[16])
{
#pragma unroll
  for (int l = 0; l < 5; ++l) {
    const int d = 1 << l;
    const Axis a = shfl_up(cx, d), b = shfl_up(cy, d);
    if (lane >= d) {
      scan_combine(cx, Pm[l], a);
      scan_combine(cy, Pm[l], b);
    }
  }
}

// (1b) local pass: ax[r], ay[r] = the part of f of tick 8t + r that comes from this thread's own 8 samples and their partners NL
// further on; (bx, by) = the thread's total, W at tick 8t for a zero state at tick 8t + 8; pk = the thread's own ZMP reference
// (the `ZMPPositions[lindex]` of the integrator).  The ring of samples has CAP slots; the kernel's slot mapping comes in as
// own(j) = sample j of the thread (slot own0 + j) and ring(i) = the sample in slot i.
template <bool SIM, class Own, class Ring>
__device__ __forceinline__ void local_pass(Own own, Ring ring, int own0, int NL, int CAP, double *ax, double *ay, double2 *pk,
                                           Axis &bx, Axis &by)
{
  bx = axis_zero();
  by = bx;
#pragma unroll
  for (int r = 0; r < FIR_R; ++r) { ax[r] = 0.0; ay[r] = 0.0; }
#pragma unroll
  for (int j = 0; j < FIR_R; ++j) {
    const double2 a = own(j);
    int fi = own0 + j + NL;
    if (fi >= CAP) fi -= CAP;
    const double2 f = ring(fi);
    pk[j] = SIM ? a : make_double2(0.0, 0.0);
#pragma unroll
    for (int r = 0; r <= j; ++r) {
      ax[r] = fma(c_pc.RF0[j - r], a.x, ax[r]); ax[r] = fma(c_pc.RFN[j - r], f.x, ax[r]);
      ay[r] = fma(c_pc.RF0[j - r], a.y, ay[r]); ay[r] = fma(c_pc.RFN[j - r], f.y, ay[r]);
    }
    bx.x0 = fma(c_pc.RV[j][0], a.x, bx.x0); bx.x0 = fma(c_pc.RVN[j][0], f.x, bx.x0);
    bx.x1 = fma(c_pc.RV[j][1], a.x, bx.x1); bx.x1 = fma(c_pc.RVN[j][1], f.x, bx.x1);
    bx.x2 = fma(c_pc.RV[j][2], a.x, bx.x2); bx.x2 = fma(c_pc.RVN[j][2], f.x, bx.x2);
    bx.s = fma(c_pc.RV[j][3], a.x, bx.s); bx.s = fma(c_pc.RVN[j][3], f.x, bx.s);
    by.x0 = fma(c_pc.RV[j][0], a.y, by.x0); by.x0 = fma(c_pc.RVN[j][0], f.y, by.x0);
    by.x1 = fma(c_pc.RV[j][1], a.y, by.x1); by.x1 = fma(c_pc.RVN[j][1], f.y, by.x1);
    by.x2 = fma(c_pc.RV[j][2], a.y, by.x2); by.x2 = fma(c_pc.RVN[j][2], f.y, by.x2);
    by.s = fma(c_pc.RV[j][3], a.y, by.s); by.s = fma(c_pc.RVN[j][3], f.y, by.s);
  }
}

// (1c) Kogge-Stone scan DOWN the lanes of a warp: c_t += L^(8d) c_{t+d}
__device__ __forceinline__ void scan_down(Axis &bx, Axis &by, int lane)
{
#pragma unroll
  for (int l = 0; l < 5; ++l) {
    const int d = 1 << l;
    const Axis a = shfl_down(bx, d), b = shfl_down(by, d);
    if (lane + d < 32) {
      scan_combine(bx, c_pc.RP[l], a);
      scan_combine(by, c_pc.RP[l], b);
    }
  }
}

// (1d) f of tick r += (w' L^(8 - r)) . W_in, W_in = (ix, iy) the true W at the thread's end
__device__ __forceinline__ void add_window(double *ax, double *ay, const Axis &ix, const Axis &iy)
{
#pragma unroll
  for (int r = 0; r < FIR_R; ++r) {
    const double *g = c_pc.RW[FIR_R - r];
    ax[r] = fma(g[0], ix.x0, fma(g[1], ix.x1, fma(g[2], ix.x2, fma(g[3], ix.s, ax[r]))));
    ay[r] = fma(g[0], iy.x0, fma(g[1], iy.x1, fma(g[2], iy.x2, fma(g[3], iy.s, ay[r]))));
  }
}

// ADD: second stage of ZMPPreviewControlWithMultiBodyZMP (SecondStageOfControl, ZMPPreviewControlWithMultiBodyZMP.cpp:317-376):
// the stream is the delta ZMP, and the CoM rows written are com_add (the first stage's CoM of the same tick) + the state.
// POS: output selection for callers that only consume the CoM position (wg_preview_run_batch_pos): the (x, y) pair of a tick
// goes out through the 16-byte path of the ZMP (zmp = the position array, com = nullptr): 16 B per step leave the GPU, not 64.
template <bool SIM, int FIR_THREADS, int MIN_CTAS, bool ADD = false, bool POS = false>
__global__ void __launch_bounds__(FIR_THREADS, MIN_CTAS)
preview_fused_kernel(const int *__restrict__ order, const int64_t *__restrict__ offsets,
                     const double2 *__restrict__ p, double *__restrict__ state, double *__restrict__ com,
                     double *__restrict__ zmp, const double *__restrict__ com_add = nullptr)
{
  constexpr int FIR_TILE = FIR_R * FIR_THREADS;   // ticks per tile
  extern __shared__ double2 sp[];             // padded tile of (px,py), then the scan exchange area
  __shared__ double s_tot[FIR_THREADS / 32 + 1][8];   // warp totals of the scan (x axis 0..3, y axis 4..7)
  __shared__ double s_carry[8];
  const int b = order[blockIdx.x];
  const int64_t o = offsets[b];
  const int L = (int)(offsets[b + 1] - o);
  const int NL = c_pc.NL, NLpad = c_pc.NLpad;
  const int nsteps = L - NL + 1;
  if (nsteps <= 0) return;
  const int t = threadIdx.x, lane = t & 31;
  const int span = FIR_TILE + NLpad;           // samples one tile needs
  if (t < 8) s_carry[t] = state[8 * (size_t)b + t];   // {x,dx,ddx,y,dy,ddy,sx,sy}
  const double(*Pm)[16] = c_pc.P[SIM ? 1 : 0];

  for (int start = 0; start < nsteps; start += FIR_TILE) {
    __syncthreads();
    const double2 *src = p + o + start;
    const int avail = L - start;               // samples that exist from `start` on
    for (int e = t; e < span; e += FIR_THREADS) {
      double2 v = make_double2(0.0, 0.0);
      if (e < avail) v = __ldg(src + e);
      sp[pad9(e)] = v;
    }
    __syncthreads();

    // ---- (1) FIR: ax[r], ay[r] = sum_i F[i] p[start + 8t + r + i]
    double ax[FIR_R], ay[FIR_R], wx[FIR_R], wy[FIR_R];
#pragma unroll
    for (int r = 0; r < FIR_R; ++r) {
      ax[r] = 0.0; ay[r] = 0.0;
      double2 v = sp[pad9(FIR_R * t + r)];
      wx[r] = v.x; wy[r] = v.y;
    }
    // window invariant at tap j: w[(j+r) % 8] holds p[8t + r + j]
    const double2 *wp = sp + pad9(FIR_R * t + FIR_R);   // next sample to enter the window
    // threads whose 8 ticks all lie past the trajectory's last step (ragged last tile) skip the FIR: their
    // ax/ay stay 0 and nothing downstream of the scan reads them (the scan only propagates upwards)
    const int ntaps = (start + FIR_R * t < nsteps) ? NLpad : 0;
    for (int jj = 0; jj < ntaps; jj += FIR_R) {
#pragma unroll
      for (int u = 0; u < FIR_R; ++u) {
        const double f = c_F[jj + u];
#pragma unroll
        for (int r = 0; r < FIR_R; ++r) {
          ax[r] = fma(f, wx[(u + r) % FIR_R], ax[r]);
          ay[r] = fma(f, wy[(u + r) % FIR_R], ay[r]);
        }
        double2 v = wp[u];                        // p[8t + 8 + jj + u]; 8-aligned group => no pad inside
        wx[u] = v.x; wy[u] = v.y;
      }
      wp += FIR_R + 1;                            // 8 samples + 1 padding slot
    }
    // the ZMP reference of the thread's own ticks (the `ZMPPositions[lindex]` of the error integrator) is
    // re-read from the tile in both passes below rather than kept in registers across the scan
    const double2 *own = sp + pad9(FIR_R * t);
    double2 pk[FIR_R];                          // kept in registers: the tile buffer becomes the store staging area
#pragma unroll
    for (int r = 0; r < FIR_R; ++r) pk[r] = SIM ? own[r] : make_double2(0.0, 0.0);

    // ---- (2a) local aggregate: state after this thread's 8 ticks started from zero, as the linear map of its
    //      inputs (thread 0 adds M^8 x the carried state)
    Axis cx, cy, inx, iny;
    local_aggregate<SIM>(ax, ay, pk, t == 0, s_carry, Pm, cx, cy, inx, iny);
    // ---- (2b) Kogge-Stone scan over threads: c_t += M^(8d) c_{t-d}
    scan_up(cx, cy, lane, Pm);
    if (lane == 31) store_pair(s_tot[t >> 5], cx, cy);
    __syncthreads();
    // ---- (2c) true start state of this thread = inclusive result of thread t-1
    Axis sx, sy;
    {
      const int w = t >> 5;
      Axis vx, vy;                         // W_w, the state entering this warp
      vx.x0 = vx.x1 = vx.x2 = vx.s = 0.0;
      vy.x0 = vy.x1 = vy.x2 = vy.s = 0.0;
      for (int v = 0; v < w; ++v) {        // W_{v+1} = M^256 W_v + T_v
        const double *n = s_tot[v];
        Axis nx, ny;
        nx.x0 = n[0]; nx.x1 = n[1]; nx.x2 = n[2]; nx.s = n[3];
        ny.x0 = n[4]; ny.x1 = n[5]; ny.x2 = n[6]; ny.s = n[7];
        scan_combine(nx, Pm[5], vx);
        scan_combine(ny, Pm[5], vy);
        vx = nx; vy = ny;
      }
      const Axis wx_in = vx, wy_in = vy;
      if (w > 0) {
#pragma unroll
        for (int l = 0; l < 6; ++l) {
          if (((lane + 1) >> l) & 1) {
            Axis zx, zy;
            zx.x0 = zx.x1 = zx.x2 = zx.s = 0.0;
            zy.x0 = zy.x1 = zy.x2 = zy.s = 0.0;
            scan_combine(zx, Pm[l], vx);
            scan_combine(zy, Pm[l], vy);
            vx = zx; vy = zy;
          }
        }
        cx.x0 += vx.x0; cx.x1 += vx.x1; cx.x2 += vx.x2; cx.s += vx.s;
        cy.x0 += vy.x0; cy.x1 += vy.x1; cy.x2 += vy.x2; cy.s += vy.s;
      }
      sx.x0 = __shfl_up_sync(0xffffffffu, cx.x0, 1); sx.x1 = __shfl_up_sync(0xffffffffu, cx.x1, 1);
      sx.x2 = __shfl_up_sync(0xffffffffu, cx.x2, 1); sx.s = __shfl_up_sync(0xffffffffu, cx.s, 1);
      sy.x0 = __shfl_up_sync(0xffffffffu, cy.x0, 1); sy.x1 = __shfl_up_sync(0xffffffffu, cy.x1, 1);
      sy.x2 = __shfl_up_sync(0xffffffffu, cy.x2, 1); sy.s = __shfl_up_sync(0xffffffffu, cy.s, 1);
      if (lane == 0) {
        if (w == 0) { sx = inx; sy = iny; }
        else { sx = wx_in; sy = wy_in; }
      }
    }
    // ---- (2d) final pass: emit CoM / ZMP of the valid ticks.  A lane owns 8 consecutive ticks, so direct stores would
    //      put 32 different 128-byte lines behind every store instruction (measured: 0.34 ms of the 0.83 ms pass).  The
    //      warp stages two ticks per lane in its slice of the (now dead) tile buffer - every FIR read of the tile
    //      happened before the barrier above - and copies the slice out with consecutive lanes on consecutive 16 bytes.
    const int k0 = start + FIR_R * t;
    const int last = min(start + FIR_TILE, nsteps) - 1;   // last valid tick of this tile
    {
      constexpr int CHUNK_C = 7, CHUNK_Z = 3;     // double2 per lane and round: 6 (+1 pad) of CoM, 2 (+1 pad) of ZMP
      double2 *stg_c = sp + (t >> 5) * (32 * (CHUNK_C + CHUNK_Z));
      double2 *stg_z = stg_c + 32 * CHUNK_C;
      const int kw = start + FIR_R * (t & ~31);   // first tick of this warp
      double2 *gc = reinterpret_cast<double2 *>(com) + 3 * (o + kw);
      double2 *gz = reinterpret_cast<double2 *>(zmp) + (o + kw);
#pragma unroll
      for (int j = 0; j < FIR_R / 2; ++j) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int r = 2 * j + h;
          if (k0 + r <= last) {
            const double zx = preview_tick<SIM>(sx, ax[r], pk[r].x);
            const double zy = preview_tick<SIM>(sy, ay[r], pk[r].y);
            double2 *q = stg_c + CHUNK_C * lane + 3 * h;
            q[0] = make_double2(sx.x0, sx.x1);
            q[1] = make_double2(sx.x2, sy.x0);
            q[2] = make_double2(sy.x1, sy.x2);
            stg_z[CHUNK_Z * lane + h] = POS ? make_double2(sx.x0, sy.x0) : make_double2(zx, zy);
          }
        }
        __syncwarp();
        if (com) {
#pragma unroll
          for (int it = 0; it < 6; ++it) {
            const int idx = 32 * it + lane, c = idx / 6, part = idx - 6 * c;
            const int row = kw + FIR_R * c + 2 * j;             // first of the two ticks of lane c in this round
            if (row + (part >= 3) <= last) {
              double2 v = stg_c[CHUNK_C * c + part];
              if (ADD) {
                const double2 a = __ldg(reinterpret_cast<const double2 *>(com_add) + 3 * (o + kw) + 3 * (FIR_R * c + 2 * j) + part);
                v.x += a.x; v.y += a.y;
              }
              gc[3 * (FIR_R * c + 2 * j) + part] = v;
            }
          }
        }
        if (zmp) {
#pragma unroll
          for (int it = 0; it < 2; ++it) {
            const int idx = 32 * it + lane, c = idx >> 1, part = idx & 1;
            const int row = kw + FIR_R * c + 2 * j + part;
            if (row <= last) gz[FIR_R * c + 2 * j + part] = stg_z[CHUNK_Z * c + part];
          }
        }
        __syncwarp();
      }
    }
    if (k0 <= last && last < k0 + FIR_R) store_state(s_carry, sx, sy);   // the thread that ran the tile's last valid tick carries the state
  }
  __syncthreads();
  if (t < 8) state[8 * (size_t)b + t] = s_carry[t];
}

// ---------------------------------------------------------------------------------------------
// preview_rec_kernel: the same batch run with the preview sum evaluated RECURSIVELY (HBM bound instead of FP64 bound).
//
// The window weights of the reference are F[i] = w' L^i v (see rec_setup), so with W_k = sum_{i<NL} L^i v p[k+i]
//     f_k = w' W_k,      W_k = L W_{k+1} + v p[k] - (L^NL v) p[k+NL]        (spectral radius of L: 0.983)
// a stable BACKWARD linear recurrence: 1280 flop of window sum per tick become ~70.  Per tile of 8 x THREADS ticks:
//   (1a) W at the tile's end directly from the halo samples already staged in shared memory (sum_{i<NL} E[i] p[end+i],
//        one table row per sample, reduced over the CTA): tiles stay independent of each other and of the processing order;
//   (1b) every thread: its 8 ticks from a zero end state - the 8-tap triangular sums with F[0..7] and -F[NL..NL+7] - and
//        its local total sum_r L^r (v p[r] - L^NL v p[r+NL]);
//   (1c) Kogge-Stone scan over threads, running DOWN the tile (shuffle-down, constant matrices L^(8 d)), warp totals through
//        shared memory, the per-lane power (L^8)^(31-lane) of the state entering the warp from a 4 KB table;
//   (1d) f of tick r += (w' L^(8-r)) . (true W at the thread's end).
// Then phases (2a)-(2d) of preview_fused_kernel unchanged (forward scan of the cart-table state, staged stores).
// Deviation of f from the direct sum: 1e-14 relative (it is a different summation order of the same 320 products);
// measured on CoM / ZMP against the reference's object code: see tests/test_preview_ref.py.
// ---------------------------------------------------------------------------------------------
// 256-bit global accesses (LDG.256 / STG.256, sm_100): one whole 32-byte sector per thread; `al32` = the address is 32-byte
// aligned (uniform over the CTA), otherwise two 128-bit accesses
__device__ __forceinline__ void st32g(double *p, double a, double b, double c, double d, bool al32)
{
  if (al32) asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};\n" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
  else {
    reinterpret_cast<double2 *>(p)[0] = make_double2(a, b);
    reinterpret_cast<double2 *>(p)[1] = make_double2(c, d);
  }
}
__device__ __forceinline__ void ld32g(const double *p, double &a, double &b, double &c, double &d, bool al32)
{
  if (al32) asm volatile("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];\n" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
  else {
    const double2 u = __ldg(reinterpret_cast<const double2 *>(p)), v = __ldg(reinterpret_cast<const double2 *>(p) + 1);
    a = u.x; b = u.y; c = v.x; d = v.y;
  }
}
// cp.async (LDGSTS): 16 bytes global -> shared without a register round trip; src_size 0 writes zeros
__device__ __forceinline__ void cp_async16(double2 *dst_smem, const double2 *src_gmem, unsigned src_size)
{
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst_smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(src_gmem), "r"(src_size) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

template <bool SIM, int FIR_THREADS, int MIN_CTAS, bool ADD = false, bool POS = false>
__global__ void __launch_bounds__(FIR_THREADS, MIN_CTAS)
preview_rec_kernel(const int *__restrict__ order, const int64_t *__restrict__ offsets,
                   const double2 *__restrict__ p, double *__restrict__ state, double *__restrict__ com,
                   double *__restrict__ zmp, const double *__restrict__ com_add, const double2 *__restrict__ Etab,
                   const double2 *__restrict__ lanepow)
{
  constexpr int FIR_TILE = FIR_R * FIR_THREADS;   // ticks per tile
  constexpr int NW = FIR_THREADS / 32;
  constexpr unsigned FULL = 0xffffffffu;
  // Ring of 2 tiles + the window, 9/8 padded: sample e of the trajectory lives in slot pad9(e mod CAP).  While tile i is
  // computed, the FIR_TILE new samples tile i + 1 needs arrive through cp.async in the slots tile i - 1 used for its own
  // samples; the slots of tile i's own samples are dead after phase (1) and stage its stores.  Nothing is loaded twice.
  extern __shared__ double2 sp[];
  __shared__ double s_tot[NW + 1][8];         // warp totals of the forward scan (x axis 0..3, y axis 4..7)
  __shared__ double s_totb[NW + 1][8];        // warp totals of the backward scan
  __shared__ double s_halo[NW][8];            // per-warp partial sums of W at the tile's end
  __shared__ double s_carry[8];
  const int b = order[blockIdx.x];
  const int64_t o = offsets[b];
  const int L = (int)(offsets[b + 1] - o);
  const int NL = c_pc.NL, NLpad = c_pc.NLpad;
  const int nsteps = L - NL + 1;
  if (nsteps <= 0) return;
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const int CAP = 2 * FIR_TILE + NLpad;        // ring capacity in samples (a multiple of 8)
  if (t < 8) s_carry[t] = state[8 * (size_t)b + t];   // {x,dx,ddx,y,dy,ddy,sx,sy}
  const double(*Pm)[16] = c_pc.P[SIM ? 1 : 0];
  const double2 *src = p + o;
  // first tile: samples [0, FIR_TILE + NLpad); samples past the trajectory read as zero (src-size 0 zero-fills)
  for (int e = t; e < FIR_TILE + NLpad; e += FIR_THREADS) cp_async16(sp + pad9(e), src + (e < L ? e : 0), e < L ? 16u : 0u);
  cp_async_commit();
  int base = 0;                                // slot index (before padding) of sample `start`

  for (int start = 0; start < nsteps; start += FIR_TILE) {
    cp_async_wait_all();
    __syncthreads();                           // this tile's samples have landed; the previous tile's staged stores are out
    if (start + FIR_TILE < nsteps) {           // prefetch what the next tile adds: samples [start + span, start + span + FIR_TILE)
      const int first = start + FIR_TILE + NLpad;
#pragma unroll
      for (int u = 0; u < FIR_R; ++u) {
        const int e = t + u * FIR_THREADS;
        int ri = base + FIR_TILE + NLpad + e;
        if (ri >= CAP) ri -= CAP;
        const bool in = first + e < L;
        cp_async16(sp + pad9(ri), src + (in ? first + e : 0), in ? 16u : 0u);
      }
      cp_async_commit();
    }
    const int own0 = (base + FIR_R * t >= CAP) ? base + FIR_R * t - CAP : base + FIR_R * t;   // slot of this thread's first sample

    // ---- (1a) W at the tile's end (x: h[0..3], y: h[4..7]), partial sums of this thread's halo samples
    {
      double h[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) h[j] = 0.0;
      for (int i = t; i < NL; i += FIR_THREADS) {
        const double2 e01 = __ldg(Etab + 2 * i), e23 = __ldg(Etab + 2 * i + 1);
        int hi = base + FIR_TILE + i;
        if (hi >= CAP) hi -= CAP;
        const double2 q = sp[pad9(hi)];
        h[0] = fma(e01.x, q.x, h[0]); h[1] = fma(e01.y, q.x, h[1]); h[2] = fma(e23.x, q.x, h[2]); h[3] = fma(e23.y, q.x, h[3]);
        h[4] = fma(e01.x, q.y, h[4]); h[5] = fma(e01.y, q.y, h[5]); h[6] = fma(e23.x, q.y, h[6]); h[7] = fma(e23.y, q.y, h[7]);
      }
      // warp sum of 8 values with 9 shuffles: halve the set of values a lane carries at each of the first three levels
      double k4[4], k2[2], k1;
      {
        const bool up = (lane & 16) != 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const double send = up ? h[j] : h[4 + j];
          k4[j] = (up ? h[4 + j] : h[j]) + __shfl_xor_sync(FULL, send, 16);
        }
      }
      {
        const bool up = (lane & 8) != 0;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const double send = up ? k4[j] : k4[2 + j];
          k2[j] = (up ? k4[2 + j] : k4[j]) + __shfl_xor_sync(FULL, send, 8);
        }
      }
      {
        const bool up = (lane & 4) != 0;
        const double send = up ? k2[0] : k2[1];
        k1 = (up ? k2[1] : k2[0]) + __shfl_xor_sync(FULL, send, 4);
      }
      k1 += __shfl_xor_sync(FULL, k1, 2);
      k1 += __shfl_xor_sync(FULL, k1, 1);
      if ((lane & 3) == 0) s_halo[w][((lane & 16) ? 4 : 0) + ((lane & 8) ? 2 : 0) + ((lane & 4) ? 1 : 0)] = k1;
    }

    // ---- (1b) local pass
    double ax[FIR_R], ay[FIR_R];
    double2 pk[FIR_R];
    Axis bx, by;
    const double2 *own = sp + pad9(own0);
    local_pass<SIM>([&](int j) { return own[j]; }, [&](int i) { return sp[pad9(i)]; }, own0, NL, CAP, ax, ay, pk, bx, by);
    // ---- (1c) Kogge-Stone scan DOWN the tile (segmented per warp)
    scan_down(bx, by, lane);
    if (lane == 0) store_pair(s_totb[w], bx, by);
    __syncthreads();      // every read of the tile buffer is done: it becomes the store staging area below
    {
      // state entering this warp from above: V_(NW-1) = W at the tile's end, V_(u-1) = T_u + L^256 V_u
      Axis vx, vy;
      vx.x0 = vx.x1 = vx.x2 = vx.s = 0.0;
      vy = vx;
#pragma unroll
      for (int u = 0; u < NW; ++u) {
        vx.x0 += s_halo[u][0]; vx.x1 += s_halo[u][1]; vx.x2 += s_halo[u][2]; vx.s += s_halo[u][3];
        vy.x0 += s_halo[u][4]; vy.x1 += s_halo[u][5]; vy.x2 += s_halo[u][6]; vy.s += s_halo[u][7];
      }
      for (int u = NW - 1; u > w; --u) {
        const double *n = s_totb[u];
        Axis nx, ny;
        nx.x0 = n[0]; nx.x1 = n[1]; nx.x2 = n[2]; nx.s = n[3];
        ny.x0 = n[4]; ny.x1 = n[5]; ny.x2 = n[6]; ny.s = n[7];
        scan_combine(nx, c_pc.RP[5], vx);
        scan_combine(ny, c_pc.RP[5], vy);
        vx = nx; vy = ny;
      }
      // true W at this thread's end (tick 8t + 8) = inclusive result of lane + 1 (nothing for lane 31) + (L^8)^(31-lane) V
      Axis ix, iy;
      ix.x0 = __shfl_down_sync(FULL, bx.x0, 1); ix.x1 = __shfl_down_sync(FULL, bx.x1, 1);
      ix.x2 = __shfl_down_sync(FULL, bx.x2, 1); ix.s = __shfl_down_sync(FULL, bx.s, 1);
      iy.x0 = __shfl_down_sync(FULL, by.x0, 1); iy.x1 = __shfl_down_sync(FULL, by.x1, 1);
      iy.x2 = __shfl_down_sync(FULL, by.x2, 1); iy.s = __shfl_down_sync(FULL, by.s, 1);
      if (lane == 31) { ix.x0 = ix.x1 = ix.x2 = ix.s = 0.0; iy = ix; }
      {
        const double2 *lp = lanepow + 8 * (31 - lane);
        double Pl[16];
#pragma unroll
        for (int e = 0; e < 8; ++e) { const double2 q = __ldg(lp + e); Pl[2 * e] = q.x; Pl[2 * e + 1] = q.y; }
        scan_combine(ix, Pl, vx);
        scan_combine(iy, Pl, vy);
      }
      // ---- (1d)
      add_window(ax, ay, ix, iy);
    }

    // ---- (2a) local aggregate of the cart-table recursion (as preview_fused_kernel)
    Axis cx, cy, inx, iny;
    local_aggregate<SIM>(ax, ay, pk, t == 0, s_carry, Pm, cx, cy, inx, iny);
    // ---- (2b) Kogge-Stone scan UP the tile
    scan_up(cx, cy, lane, Pm);
    if (lane == 31) store_pair(s_tot[w], cx, cy);
    __syncthreads();
    // ---- (2c) true start state of this thread = inclusive result of thread t-1
    Axis sx, sy;
    {
      Axis vx, vy;                         // W_w, the state entering this warp
      vx.x0 = vx.x1 = vx.x2 = vx.s = 0.0;
      vy.x0 = vy.x1 = vy.x2 = vy.s = 0.0;
      for (int v = 0; v < w; ++v) {        // W_{v+1} = M^256 W_v + T_v
        const double *n = s_tot[v];
        Axis nx, ny;
        nx.x0 = n[0]; nx.x1 = n[1]; nx.x2 = n[2]; nx.s = n[3];
        ny.x0 = n[4]; ny.x1 = n[5]; ny.x2 = n[6]; ny.s = n[7];
        scan_combine(nx, Pm[5], vx);
        scan_combine(ny, Pm[5], vy);
        vx = nx; vy = ny;
      }
      const Axis wx_in = vx, wy_in = vy;
      if (w > 0) {
#pragma unroll
        for (int l = 0; l < 6; ++l) {
          if (((lane + 1) >> l) & 1) {
            Axis zx, zy;
            zx.x0 = zx.x1 = zx.x2 = zx.s = 0.0;
            zy.x0 = zy.x1 = zy.x2 = zy.s = 0.0;
            scan_combine(zx, Pm[l], vx);
            scan_combine(zy, Pm[l], vy);
            vx = zx; vy = zy;
          }
        }
        cx.x0 += vx.x0; cx.x1 += vx.x1; cx.x2 += vx.x2; cx.s += vx.s;
        cy.x0 += vy.x0; cy.x1 += vy.x1; cy.x2 += vy.x2; cy.s += vy.s;
      }
      sx.x0 = __shfl_up_sync(0xffffffffu, cx.x0, 1); sx.x1 = __shfl_up_sync(0xffffffffu, cx.x1, 1);
      sx.x2 = __shfl_up_sync(0xffffffffu, cx.x2, 1); sx.s = __shfl_up_sync(0xffffffffu, cx.s, 1);
      sy.x0 = __shfl_up_sync(0xffffffffu, cy.x0, 1); sy.x1 = __shfl_up_sync(0xffffffffu, cy.x1, 1);
      sy.x2 = __shfl_up_sync(0xffffffffu, cy.x2, 1); sy.s = __shfl_up_sync(0xffffffffu, cy.s, 1);
      if (lane == 0) {
        if (w == 0) { sx = inx; sy = iny; }
        else { sx = wx_in; sy = wy_in; }
      }
    }
    // ---- (2d) final pass, rows stored straight from registers
    const int k0 = start + FIR_R * t;
    const int last = min(start + FIR_TILE, nsteps) - 1;   // last valid tick of this tile
    {
      double *gc = com ? com + 6 * (size_t)(o + k0) : nullptr;
      double *gz = zmp ? zmp + 2 * (size_t)(o + k0) : nullptr;
      const double *ga = ADD ? com_add + 6 * (size_t)(o + k0) : nullptr;
      const bool c32 = ((reinterpret_cast<uintptr_t>(gc) | (ADD ? reinterpret_cast<uintptr_t>(ga) : 0)) & 31) == 0;
      const bool z32 = (reinterpret_cast<uintptr_t>(gz) & 31) == 0;
#pragma unroll
      for (int j = 0; j < FIR_R / 2; ++j) {
        const int r0 = 2 * j, r1 = 2 * j + 1;
        if (k0 + r1 <= last) {                 // both ticks of the pair are valid
          const double zx0 = preview_tick<SIM>(sx, ax[r0], pk[r0].x);
          const double zy0 = preview_tick<SIM>(sy, ay[r0], pk[r0].y);
          double a0 = sx.x0, a1 = sx.x1, a2 = sx.x2, a3 = sy.x0, a4 = sy.x1, a5 = sy.x2;
          const double u0 = POS ? sx.x0 : zx0, u1 = POS ? sy.x0 : zy0;
          const double zx1 = preview_tick<SIM>(sx, ax[r1], pk[r1].x);
          const double zy1 = preview_tick<SIM>(sy, ay[r1], pk[r1].y);
          if (com) {
            double b0 = sx.x0, b1 = sx.x1, b2 = sx.x2, b3 = sy.x0, b4 = sy.x1, b5 = sy.x2;
            if (ADD) {
              double q[12];
              ld32g(ga + 6 * r0, q[0], q[1], q[2], q[3], c32);
              ld32g(ga + 6 * r0 + 4, q[4], q[5], q[6], q[7], c32);
              ld32g(ga + 6 * r0 + 8, q[8], q[9], q[10], q[11], c32);
              a0 += q[0]; a1 += q[1]; a2 += q[2]; a3 += q[3]; a4 += q[4]; a5 += q[5];
              b0 += q[6]; b1 += q[7]; b2 += q[8]; b3 += q[9]; b4 += q[10]; b5 += q[11];
            }
            st32g(gc + 6 * r0, a0, a1, a2, a3, c32);
            st32g(gc + 6 * r0 + 4, a4, a5, b0, b1, c32);
            st32g(gc + 6 * r0 + 8, b2, b3, b4, b5, c32);
          }
          if (zmp) st32g(gz + 2 * r0, u0, u1, POS ? sx.x0 : zx1, POS ? sy.x0 : zy1, z32);
        } else if (k0 + r0 <= last) {          // the trajectory ends on the first tick of the pair
          const double zx0 = preview_tick<SIM>(sx, ax[r0], pk[r0].x);
          const double zy0 = preview_tick<SIM>(sy, ay[r0], pk[r0].y);
          if (com) {
            double a0 = sx.x0, a1 = sx.x1, a2 = sx.x2, a3 = sy.x0, a4 = sy.x1, a5 = sy.x2;
            if (ADD) {
              const double2 q0 = __ldg(reinterpret_cast<const double2 *>(ga + 6 * r0));
              const double2 q1 = __ldg(reinterpret_cast<const double2 *>(ga + 6 * r0) + 1);
              const double2 q2 = __ldg(reinterpret_cast<const double2 *>(ga + 6 * r0) + 2);
              a0 += q0.x; a1 += q0.y; a2 += q1.x; a3 += q1.y; a4 += q2.x; a5 += q2.y;
            }
            double2 *g2 = reinterpret_cast<double2 *>(gc + 6 * r0);
            g2[0] = make_double2(a0, a1); g2[1] = make_double2(a2, a3); g2[2] = make_double2(a4, a5);
          }
          if (zmp) *reinterpret_cast<double2 *>(gz + 2 * r0) = POS ? make_double2(sx.x0, sy.x0) : make_double2(zx0, zy0);
        }
      }
    }
    if (k0 <= last && last < k0 + FIR_R) store_state(s_carry, sx, sy);   // the thread that ran the tile's last valid tick carries the state
    base += FIR_TILE;
    if (base >= CAP) base -= CAP;
  }
  __syncthreads();
  if (t < 8) state[8 * (size_t)b + t] = s_carry[t];
}

// ---------------------------------------------------------------------------------------------
// preview_rec_warp_kernel: the recursive evaluation with ONE WARP per trajectory (CTA = 32 threads, tile = 256 ticks).
// Same arithmetic as preview_rec_kernel; what a single warp changes:
//   * no cross-warp phase, no __syncthreads: W at the tile's end (the halo sum) is folded into lane 31's local total BEFORE the
//     downward scan (c_31 += L^8 W_end), so the scan delivers the true W of every lane and the per-lane power table is not read;
//     the carried cart-table state enters lane 0 of the upward scan the same way;
//   * the samples live in a ring of TILE + NLpad slots: once phase (1b) has read a lane's own 8 samples their slots are dead and
//     receive (cp.async) the 256 samples the next tile adds while phases (1c)-(2d) run; the ring is XOR-swizzled, not padded
//     (slot s lives at s ^ ((s >> 3) & 7): the stride-8 reads of the local pass and the lane-contiguous accesses are both
//     conflict free): 9.2 KB at NL = 320;
//   * the E table rows of a lane's halo samples are fetched five at a time, one 256-bit load per row, before they are used (one
//     exposed L1/L2 latency per five samples instead of one per sample);
//   * the CoM rows leave through the bulk-copy engine: a lane stages the 384 bytes of its 8 ticks in its own slot behind the ring
//     (400-byte stride: conflict-free 128-bit stores) and hands them over with ONE cp.async.bulk request per tile.  A warp-wide
//     256-bit store of this row layout touches 32 different 128-byte lines, and the LSU tag stage - not HBM - was what the stores
//     cost; measured on configs[1]: 39.2 G steps/s with direct stores, 42.4 with one request per tick pair (16 warps/SM), 43.8 per
//     four ticks (13 warps/SM), 47.2 per tile (22 KB of shared memory per warp: 10 warps/SM, 140 registers, no spills).
//     UBLKCP takes its operands in uniform registers, so a request issued by every lane for its own slot becomes a
//     ~10-instruction loop per lane (11 % of the kernel's instructions).  Instead, after the warp has staged the tile, ONE
//     elected lane issues all 32 requests: lane i's request depends only on i and the tile, its operands are warp-uniform, and
//     a whole tile's 32 requests unroll to ~5 instructions each (0.310 -> 0.298 ms per launch on configs[1]).  The ZMP pair (one
//     sector per lane) stays a 256-bit store: a second request per lane costs more than it saves (38.7 G steps/s at 8 warps/SM).
// ---------------------------------------------------------------------------------------------
constexpr int RW_TILE = FIR_R * 32;
constexpr int RW_U = 5;                        // halo samples per lane fetched together

// shared -> global through the bulk-copy engine (cp.async.bulk, UBLKCP): 16-byte aligned addresses and size
__device__ __forceinline__ void bulk_store(double *dst, unsigned src_smem, unsigned bytes)
{
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(dst), "r"(src_smem), "r"(bytes) : "memory");
}
// true in exactly one lane of the (converged) warp: what the compiler needs to issue a request once, not once per lane
__device__ __forceinline__ bool elect_one()
{
  unsigned r;
  asm volatile("{\n .reg .pred p;\n elect.sync _|p, 0xffffffff;\n selp.u32 %0, 1, 0, p;\n}\n" : "=r"(r));
  return r != 0;
}

template <bool SIM, bool ADD = false, bool POS = false>
__global__ void __launch_bounds__(32, 10)
preview_rec_warp_kernel(const int *__restrict__ order, const int64_t *__restrict__ offsets,
                        const double2 *__restrict__ p, double *__restrict__ state, double *__restrict__ com,
                        double *__restrict__ zmp, const double *__restrict__ com_add, const double2 *__restrict__ Etab)
{
  constexpr unsigned FULL = 0xffffffffu;
  extern __shared__ double2 sp[];             // the ring (XOR-swizzled), then 32 staging slots of 7 double2
  __shared__ double s_halo[8];                // W at the tile's end (x: 0..3, y: 4..7)
  __shared__ double s_carry[8];
  const int b = order[blockIdx.x];
  const int64_t o = offsets[b];
  const int L = (int)(offsets[b + 1] - o);
  const int NL = c_pc.NL, NLpad = c_pc.NLpad;
  const int nsteps = L - NL + 1;
  if (nsteps <= 0) return;
  const int lane = threadIdx.x;
  const int CAP = RW_TILE + NLpad;             // ring capacity in samples (a multiple of 8)
  // per-lane staging of the CoM rows of one tick pair (96 B, lane stride 112 B: conflict-free 128-bit stores) behind the ring
  double2 *stage = sp + CAP + 25 * lane;
  if (lane < 8) s_carry[lane] = state[8 * (size_t)b + lane];   // {x,dx,ddx,y,dy,ddy,sx,sy}
  const double(*Pm)[16] = c_pc.P[SIM ? 1 : 0];
  const double2 *src = p + o;
  // first tile: samples [0, TILE + NLpad) fill the whole ring; samples past the trajectory read as zero
  for (int e = lane; e < CAP; e += 32) cp_async16(sp + swz8(e), src + (e < L ? e : 0), e < L ? 16u : 0u);
  cp_async_commit();
  int base = 0;                                // ring slot of sample `start`

  for (int start = 0; start < nsteps; start += RW_TILE) {
    cp_async_wait_all();
    __syncwarp();                              // this tile's samples have landed
    int own0 = base + FIR_R * lane;            // slot of this lane's first sample
    if (own0 >= CAP) own0 -= CAP;

    // ---- (1a) W at the tile's end, partial sums over this lane's halo samples
    {
      double h[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) h[j] = 0.0;
      int hb = base + RW_TILE;
      if (hb >= CAP) hb -= CAP;
      for (int i0 = lane; i0 < NL; i0 += 32 * RW_U) {
        double2 e01[RW_U], e23[RW_U], q[RW_U];
#pragma unroll
        for (int u = 0; u < RW_U; ++u) {
          const int i = i0 + 32 * u;
          const bool in = i < NL;
          const int ii = in ? i : 0;
          ld32g(reinterpret_cast<const double *>(Etab + 2 * ii), e01[u].x, e01[u].y, e23[u].x, e23[u].y, true);   // one 32-byte row
          int hi = hb + ii;
          if (hi >= CAP) hi -= CAP;
          q[u] = in ? sp[swz8(hi)] : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int u = 0; u < RW_U; ++u) {
          h[0] = fma(e01[u].x, q[u].x, h[0]); h[1] = fma(e01[u].y, q[u].x, h[1]);
          h[2] = fma(e23[u].x, q[u].x, h[2]); h[3] = fma(e23[u].y, q[u].x, h[3]);
          h[4] = fma(e01[u].x, q[u].y, h[4]); h[5] = fma(e01[u].y, q[u].y, h[5]);
          h[6] = fma(e23[u].x, q[u].y, h[6]); h[7] = fma(e23[u].y, q[u].y, h[7]);
        }
      }
      // warp sum of 8 values with 9 shuffles: halve the set of values a lane carries at each of the first three levels
      double k4[4], k2[2], k1;
      {
        const bool up = (lane & 16) != 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const double send = up ? h[j] : h[4 + j];
          k4[j] = (up ? h[4 + j] : h[j]) + __shfl_xor_sync(FULL, send, 16);
        }
      }
      {
        const bool up = (lane & 8) != 0;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const double send = up ? k4[j] : k4[2 + j];
          k2[j] = (up ? k4[2 + j] : k4[j]) + __shfl_xor_sync(FULL, send, 8);
        }
      }
      {
        const bool up = (lane & 4) != 0;
        const double send = up ? k2[0] : k2[1];
        k1 = (up ? k2[1] : k2[0]) + __shfl_xor_sync(FULL, send, 4);
      }
      k1 += __shfl_xor_sync(FULL, k1, 2);
      k1 += __shfl_xor_sync(FULL, k1, 1);
      if ((lane & 3) == 0) s_halo[((lane & 16) ? 4 : 0) + ((lane & 8) ? 2 : 0) + ((lane & 4) ? 1 : 0)] = k1;
    }

    // ---- (1b) local pass (as preview_rec_kernel)
    double ax[FIR_R], ay[FIR_R];
    double2 pk[FIR_R];
    Axis bx, by;
    {
      const double2 *own = sp + own0;          // own0 is a multiple of 8: sample j of the block sits at j ^ ((own0 >> 3) & 7)
      const int osw = (own0 >> 3) & 7;
      local_pass<SIM>([&](int j) { return own[j ^ osw]; }, [&](int i) { return sp[swz8(i)]; }, own0, NL, CAP, ax, ay, pk, bx, by);
    }
    __syncwarp();          // every read of this tile's samples is done; s_halo is written
    // the slots of the tile's own samples are dead: they receive what the next tile adds, samples [start + CAP, start + CAP + TILE)
    if (start + RW_TILE < nsteps) {
      const int first = start + CAP;
#pragma unroll
      for (int u = 0; u < FIR_R; ++u) {
        const int e = lane + 32 * u;
        int ri = base + e;
        if (ri >= CAP) ri -= CAP;
        const bool in = first + e < L;
        cp_async16(sp + swz8(ri), src + (in ? first + e : 0), in ? 16u : 0u);
      }
      cp_async_commit();
    }
    // ---- (1c) lane 31 takes W at the tile's end, then Kogge-Stone DOWN the tile: c_t += L^(8d) c_{t+d}
    Axis ix, iy;                               // W at tick 8 lane + 8 (the end of this lane's ticks)
    load_pair(s_halo, ix, iy);
    if (lane == 31) {
      scan_combine(bx, c_pc.RP[0], ix);
      scan_combine(by, c_pc.RP[0], iy);
    }
    scan_down(bx, by, lane);
    {
      const Axis a = shfl_down(bx, 1), b = shfl_down(by, 1);
      if (lane != 31) { ix = a; iy = b; }
    }
    // ---- (1d)
    add_window(ax, ay, ix, iy);

    // ---- (2a) local aggregate of the cart-table recursion; lane 0 takes the carried state
    Axis cx, cy, inx, iny;
    local_aggregate<SIM>(ax, ay, pk, lane == 0, s_carry, Pm, cx, cy, inx, iny);
    // ---- (2b) Kogge-Stone scan UP the tile
    scan_up(cx, cy, lane, Pm);
    // ---- (2c) true start state of this lane = inclusive result of lane - 1
    Axis sx = shfl_up(cx, 1), sy = shfl_up(cy, 1);
    if (lane == 0) { sx = inx; sy = iny; }
    __syncwarp();                              // s_carry and s_halo have been read
    // ---- (2d) final pass, rows stored straight from registers, CoM pairs through the bulk-copy engine (16-byte alignment is
    //      all it asks)
    const int k0 = start + FIR_R * lane;
    const int last = min(start + RW_TILE, nsteps) - 1;   // last valid tick of this tile
    {
      double *gc = com ? com + 6 * (size_t)(o + k0) : nullptr;
      double *gz = zmp ? zmp + 2 * (size_t)(o + k0) : nullptr;
      const double *ga = ADD ? com_add + 6 * (size_t)(o + k0) : nullptr;
      const bool c32 = ((reinterpret_cast<uintptr_t>(gc) | (ADD ? reinterpret_cast<uintptr_t>(ga) : 0)) & 31) == 0;
      const bool z32 = (reinterpret_cast<uintptr_t>(gz) & 31) == 0;
      const bool bulk = com != nullptr;        // CoM pairs through the bulk-copy engine (16-byte alignment is all it asks)
      if (bulk) {                              // the previous tile's requests have read the staging slots
        asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
        __syncwarp();
      }
#pragma unroll
      for (int j = 0; j < FIR_R / 2; ++j) {
        const int r0 = 2 * j, r1 = 2 * j + 1;
        if (k0 + r1 <= last) {                 // both ticks of the pair are valid
          const double zx0 = preview_tick<SIM>(sx, ax[r0], pk[r0].x);
          const double zy0 = preview_tick<SIM>(sy, ay[r0], pk[r0].y);
          double a0 = sx.x0, a1 = sx.x1, a2 = sx.x2, a3 = sy.x0, a4 = sy.x1, a5 = sy.x2;
          const double u0 = POS ? sx.x0 : zx0, u1 = POS ? sy.x0 : zy0;
          const double zx1 = preview_tick<SIM>(sx, ax[r1], pk[r1].x);
          const double zy1 = preview_tick<SIM>(sy, ay[r1], pk[r1].y);
          if (com) {
            double b0 = sx.x0, b1 = sx.x1, b2 = sx.x2, b3 = sy.x0, b4 = sy.x1, b5 = sy.x2;
            if (ADD) {
              double q[12];
              ld32g(ga + 6 * r0, q[0], q[1], q[2], q[3], c32);
              ld32g(ga + 6 * r0 + 4, q[4], q[5], q[6], q[7], c32);
              ld32g(ga + 6 * r0 + 8, q[8], q[9], q[10], q[11], c32);
              a0 += q[0]; a1 += q[1]; a2 += q[2]; a3 += q[3]; a4 += q[4]; a5 += q[5];
              b0 += q[6]; b1 += q[7]; b2 += q[8]; b3 += q[9]; b4 += q[10]; b5 += q[11];
            }
            if (bulk) {
              double2 *sg = stage + 6 * j;
              sg[0] = make_double2(a0, a1); sg[1] = make_double2(a2, a3); sg[2] = make_double2(a4, a5);
              sg[3] = make_double2(b0, b1); sg[4] = make_double2(b2, b3); sg[5] = make_double2(b4, b5);
            } else {
              st32g(gc + 6 * r0, a0, a1, a2, a3, c32);
              st32g(gc + 6 * r0 + 4, a4, a5, b0, b1, c32);
              st32g(gc + 6 * r0 + 8, b2, b3, b4, b5, c32);
            }
          }
          if (zmp) st32g(gz + 2 * r0, u0, u1, POS ? sx.x0 : zx1, POS ? sy.x0 : zy1, z32);
        } else if (k0 + r0 <= last) {          // the trajectory ends on the first tick of the pair
          const double zx0 = preview_tick<SIM>(sx, ax[r0], pk[r0].x);
          const double zy0 = preview_tick<SIM>(sy, ay[r0], pk[r0].y);
          if (com) {
            double a0 = sx.x0, a1 = sx.x1, a2 = sx.x2, a3 = sy.x0, a4 = sy.x1, a5 = sy.x2;
            if (ADD) {
              const double2 q0 = __ldg(reinterpret_cast<const double2 *>(ga + 6 * r0));
              const double2 q1 = __ldg(reinterpret_cast<const double2 *>(ga + 6 * r0) + 1);
              const double2 q2 = __ldg(reinterpret_cast<const double2 *>(ga + 6 * r0) + 2);
              a0 += q0.x; a1 += q0.y; a2 += q1.x; a3 += q1.y; a4 += q2.x; a5 += q2.y;
            }
            double2 *g2 = reinterpret_cast<double2 *>(gc + 6 * r0);
            g2[0] = make_double2(a0, a1); g2[1] = make_double2(a2, a3); g2[2] = make_double2(a4, a5);
          }
          if (zmp) *reinterpret_cast<double2 *>(gz + 2 * r0) = POS ? make_double2(sx.x0, sy.x0) : make_double2(zx0, zy0);
        }
      }
      // one lane hands every lane's whole tick pairs to the bulk-copy engine: lane i's request depends on i and on the tile only,
      // so its operands are warp-uniform and each request is one UBLKCP (issued from every lane, each request costs a
      // ~10-instruction loop over the lanes, 11 % of the kernel's instructions)
      if (bulk) {
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        __syncwarp();
        if (elect_one()) {
          const int nt = last - start + 1;     // valid ticks of this tile
          double *g = com + 6 * (size_t)(o + start);
          const unsigned sa = (unsigned)__cvta_generic_to_shared(sp + CAP);
          if (nt >= RW_TILE) {                 // a whole tile: 32 requests of 384 B, constant offsets
#pragma unroll
            for (int i = 0; i < 32; ++i) bulk_store(g + 6 * FIR_R * i, sa + 400u * i, 96u * (FIR_R / 2));
          } else {
            for (int i = 0; i < 32 && FIR_R * i + 1 < nt; ++i)   // lane i's whole tick pairs
              bulk_store(g + 6 * FIR_R * i, sa + 400u * i, 96u * (unsigned)min(FIR_R / 2, (nt - FIR_R * i) / 2));
          }
          asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
        }
      }
    }
    if (k0 <= last && last < k0 + FIR_R) store_state(s_carry, sx, sy);   // the lane that ran the tile's last valid tick carries the state
    base += RW_TILE;
    if (base >= CAP) base -= CAP;
  }
  __syncwarp();
  asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");     // every row handed to the bulk-copy engine has been written
  if (lane < 8) state[8 * (size_t)b + lane] = s_carry[lane];
}

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
namespace {

// Closed-loop one-tick matrix of the 4-state (x, dx, ddx, s) and its powers M^(8 2^l), in extended precision.
void scan_matrices(const wg_preview_gains_t &g, bool sim, double (*P)[16], double (*G)[4], double (*H)[4])
{
  typedef long double LD;
  LD M[4][4];
  for (int j = 0; j < 4; ++j) {
    LD x[3] = {0, 0, 0}, s = 0;
    if (j < 3) x[j] = 1; else s = 1;
    const LD u = (LD)g.Ks * s - ((LD)g.Kx[0] * x[0] + (LD)g.Kx[1] * x[1] + (LD)g.Kx[2] * x[2]);
    LD n[3];
    for (int i = 0; i < 3; ++i)
      n[i] = (LD)g.A[3 * i] * x[0] + (LD)g.A[3 * i + 1] * x[1] + (LD)g.A[3 * i + 2] * x[2] + (LD)g.B[i] * u;
    const LD z = (LD)g.C[0] * n[0] + (LD)g.C[1] * n[1] + (LD)g.C[2] * n[2];
    for (int i = 0; i < 3; ++i) M[i][j] = n[i];
    M[3][j] = sim ? s - z : s;
  }
  auto square = [](LD X[4][4]) {
    LD Y[4][4];
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 4; ++j) {
        LD a = 0;
        for (int k = 0; k < 4; ++k) a += X[i][k] * X[k][j];
        Y[i][j] = a;
      }
    std::memcpy(X, Y, sizeof Y);
  };
  if (G && H) {
    // g = column of f, h = column of p of one tick; G[r] = M^(FIR_R-1-r) g, H[r] = M^(FIR_R-1-r) h
    LD g4[4], h4[4] = {0, 0, 0, 0};
    LD zb = 0;
    for (int i = 0; i < 3; ++i) { g4[i] = (LD)g.B[i]; zb += (LD)g.C[i] * (LD)g.B[i]; }
    g4[3] = sim ? -zb : (LD)0;
    h4[3] = sim ? (LD)1 : (LD)0;
    for (int r = FIR_R - 1; r >= 0; --r) {
      for (int i = 0; i < 4; ++i) { G[r][i] = (double)g4[i]; H[r][i] = (double)h4[i]; }
      LD gn[4], hn[4];
      for (int i = 0; i < 4; ++i) {
        gn[i] = 0; hn[i] = 0;
        for (int k = 0; k < 4; ++k) { gn[i] += M[i][k] * g4[k]; hn[i] += M[i][k] * h4[k]; }
      }
      std::memcpy(g4, gn, sizeof gn); std::memcpy(h4, hn, sizeof hn);
    }
  }
  for (int r = 1; r < FIR_R; r <<= 1) square(M);   // M^FIR_R (FIR_R is a power of two)
  for (int l = 0; l < SCAN_LEVELS; ++l) {
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 4; ++j) P[l][4 * i + j] = (double)M[i][j];
    square(M);
  }
}


// Constants of preview_rec_kernel.  The window weights are fitted as F[i] = w' L^i v in extended precision: L = (A - b K)' is
// formed from the head of the gain set (for MODE_WITHOUT_INITIALPOS the augmented error system of PreviewControl.cpp:237-262
// with K = (Ks, Kx)), w = b, and v is the least-squares solution of the NL x n system (column-scaled, Gram-Schmidt twice).
// Weights that OptimalControllerSolver::ComputeWeights produced have this structure up to their own rounding (measured
// residual 4e-15 of sum |F|); a table that does not (e.g. read from a file with few digits) keeps the direct sum.
// Returns sum |F[i] - w' L^i v| / sum |F[i]|, or -1 when the structure cannot be formed.  tables = E [NLpad][4] (L^i v, zero
// past NL) followed by lane powers [32][16] ((L^FIR_R)^m, row-major).
double rec_setup(const wg_preview_gains_t &g, PreviewConsts &pc, std::vector<double> &tables)
{
  typedef long double LD;
  const int NL = g.NL;
  int n = 0;
  LD Ax[4][4], bx[4] = {0, 0, 0, 0}, K[4] = {0, 0, 0, 0};
  for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) Ax[i][j] = 0;
  if (g.mode == WG_PREVIEW_MODE_WITHOUT_INITIALPOS) {
    n = 4;
    Ax[0][0] = 1;
    for (int j = 0; j < 3; ++j) {
      LD a = 0;
      for (int l = 0; l < 3; ++l) a += (LD)g.C[l] * (LD)g.A[3 * l + j];
      Ax[0][j + 1] = a;
      for (int i = 0; i < 3; ++i) Ax[i + 1][j + 1] = g.A[3 * i + j];
    }
    for (int l = 0; l < 3; ++l) { bx[0] += (LD)g.C[l] * (LD)g.B[l]; bx[l + 1] = g.B[l]; }
    K[0] = g.Ks;
    for (int j = 0; j < 3; ++j) K[j + 1] = g.Kx[j];
  } else if (g.mode == WG_PREVIEW_MODE_WITH_INITIALPOS) {
    n = 3;
    for (int i = 0; i < 3; ++i) { for (int j = 0; j < 3; ++j) Ax[i][j] = g.A[3 * i + j]; bx[i] = g.B[i]; K[i] = g.Kx[i]; }
  } else {
    return -1.0;
  }
  if (NL < 2 * n) return -1.0;
  LD L[4][4];
  for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) L[i][j] = (i < n && j < n) ? Ax[j][i] - bx[j] * K[i] : (LD)0;
  // rows r_i = (L')^i w: r_i . v = w' L^i v
  std::vector<LD> M((size_t)NL * 4, 0), Q((size_t)NL * 4, 0);
  {
    LD r[4] = {bx[0], bx[1], bx[2], bx[3]};
    for (int i = 0; i < NL; ++i) {
      for (int a = 0; a < 4; ++a) M[4 * (size_t)i + a] = r[a];
      LD nx[4] = {0, 0, 0, 0};
      for (int a = 0; a < 4; ++a) for (int b = 0; b < 4; ++b) nx[a] += L[b][a] * r[b];
      for (int a = 0; a < 4; ++a) r[a] = nx[a];
    }
  }
  LD sc[4] = {1, 1, 1, 1}, R[4][4], y[4] = {0, 0, 0, 0}, v[4] = {0, 0, 0, 0};
  for (int a = 0; a < 4; ++a) for (int b = 0; b < 4; ++b) R[a][b] = 0;
  for (int a = 0; a < n; ++a) {
    LD m = 0;
    for (int i = 0; i < NL; ++i) m = std::max(m, fabsl(M[4 * (size_t)i + a]));
    if (!(m > 0)) return -1.0;
    sc[a] = m;
  }
  for (int j = 0; j < n; ++j) {
    for (int i = 0; i < NL; ++i) Q[4 * (size_t)i + j] = M[4 * (size_t)i + j] / sc[j];
    for (int rep = 0; rep < 2; ++rep)
      for (int a = 0; a < j; ++a) {
        LD c = 0;
        for (int i = 0; i < NL; ++i) c += Q[4 * (size_t)i + a] * Q[4 * (size_t)i + j];
        R[a][j] += c;
        for (int i = 0; i < NL; ++i) Q[4 * (size_t)i + j] -= c * Q[4 * (size_t)i + a];
      }
    LD nn = 0;
    for (int i = 0; i < NL; ++i) nn += Q[4 * (size_t)i + j] * Q[4 * (size_t)i + j];
    nn = sqrtl(nn);
    if (!(nn > 1e-12L)) return -1.0;     // the Krylov rows do not span n directions: no unique fit
    R[j][j] = nn;
    for (int i = 0; i < NL; ++i) Q[4 * (size_t)i + j] /= nn;
  }
  for (int j = 0; j < n; ++j) for (int i = 0; i < NL; ++i) y[j] += Q[4 * (size_t)i + j] * (LD)g.F[i];
  for (int j = n - 1; j >= 0; --j) {
    LD a = y[j];
    for (int b = j + 1; b < n; ++b) a -= R[j][b] * v[b];
    v[j] = a / R[j][j];
  }
  for (int j = 0; j < n; ++j) v[j] /= sc[j];
  LD res = 0, tot = 0;
  for (int i = 0; i < NL; ++i) {
    LD fh = 0;
    for (int a = 0; a < n; ++a) fh += M[4 * (size_t)i + a] * v[a];
    res += fabsl((LD)g.F[i] - fh);
    tot += fabsl((LD)g.F[i]);
  }
  if (!(tot > 0) || !(res == res)) return -1.0;
  // x_i = L^i v, i <= NL + FIR_R
  const int NLpad = (NL + FIR_R - 1) / FIR_R * FIR_R;
  tables.assign((size_t)NLpad * 4 + 32 * 16, 0.0);
  {
    LD x[4] = {v[0], v[1], v[2], v[3]};
    for (int i = 0; i < NL + FIR_R; ++i) {
      LD f = 0;
      for (int a = 0; a < 4; ++a) f += bx[a] * x[a];
      if (i < NL) for (int a = 0; a < 4; ++a) tables[4 * (size_t)i + a] = (double)x[a];
      if (i < FIR_R) { pc.RF0[i] = (double)f; for (int a = 0; a < 4; ++a) pc.RV[i][a] = (double)x[a]; }
      if (i >= NL) { pc.RFN[i - NL] = (double)-f; for (int a = 0; a < 4; ++a) pc.RVN[i - NL][a] = (double)-x[a]; }   // negated: pure FMAs
      LD nx[4] = {0, 0, 0, 0};
      for (int a = 0; a < 4; ++a) for (int b = 0; b < 4; ++b) nx[a] += L[a][b] * x[b];
      for (int a = 0; a < 4; ++a) x[a] = nx[a];
    }
  }
  {
    LD r[4] = {bx[0], bx[1], bx[2], bx[3]};          // w' L^j
    for (int j = 0; j <= FIR_R; ++j) {
      for (int a = 0; a < 4; ++a) pc.RW[j][a] = (double)r[a];
      LD nx[4] = {0, 0, 0, 0};
      for (int a = 0; a < 4; ++a) for (int b = 0; b < 4; ++b) nx[a] += r[b] * L[b][a];
      for (int a = 0; a < 4; ++a) r[a] = nx[a];
    }
  }
  auto mul = [](LD X[4][4], LD Y[4][4], LD Z[4][4]) {
    LD T[4][4];
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 4; ++j) {
        LD a = 0;
        for (int k = 0; k < 4; ++k) a += X[i][k] * Y[k][j];
        T[i][j] = a;
      }
    std::memcpy(Z, T, sizeof T);
  };
  LD P8[4][4];
  std::memcpy(P8, L, sizeof P8);
  for (int r = 1; r < FIR_R; r <<= 1) mul(P8, P8, P8);            // L^FIR_R
  {
    LD Pl[4][4];
    std::memcpy(Pl, P8, sizeof Pl);
    for (int l = 0; l < SCAN_LEVELS; ++l) {
      for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) pc.RP[l][4 * i + j] = (double)Pl[i][j];
      mul(Pl, Pl, Pl);
    }
    LD Pm[4][4];
    for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) Pm[i][j] = (i == j) ? 1 : 0;
    double *lp = tables.data() + (size_t)NLpad * 4;
    for (int m = 0; m < 32; ++m) {
      for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) lp[16 * m + 4 * i + j] = (double)Pm[i][j];
      mul(P8, Pm, Pm);
    }
  }
  return (double)(res / tot);
}

}  // namespace

// One launch of a preview kernel: the 96 KB check, the gains of this context in the device's __constant__ block, the
// shared-memory opt-in and the profiler bracket.
template <class... P, class... A>
static int preview_launch(wg_ctx *ctx, void (*kern)(P...), int count, int threads, size_t smem, const char *too_large,
                          A... args)
{
  if (smem > 96 * 1024) return wg_fail(ctx, WG_ERR_INVALID, too_large);
  std::lock_guard<std::mutex> lock(g_pv_mutex);
  { const int rc = preview_bind(ctx); if (rc != WG_OK) return rc; }
  WG_SMEM_ATTR(ctx, kern, smem);
  wg_prof_start(ctx, WG_K_PREVIEW_FUSED);
  kern<<<count, threads, smem, ctx->stream>>>(args...);
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  return WG_OK;
}

// The kernel of variant <SIM, ADD, POS> in the family (direct sum, recursive, recursive one-warp) and CTA shape that
// wgi_preview_launch_range chose, with the dynamic shared memory that shape needs.
template <bool SIM, bool ADD, bool POS>
static int preview_launch_variant(wg_ctx *ctx, wg_preview_plan *pl, bool recursive, int shape, const int *d_order, int count,
                                  const double2 *pz, double *d_state, double *d_com, double *d_zmpout, const double *d_com_add)
{
  const int NLpad = (pl->NL + FIR_R - 1) / FIR_R * FIR_R;
  const int64_t *off = pl->d_offsets;
  if (!recursive) {
    // tile = 8 x threads ticks; the tile buffer doubles as the store staging area (320 double2 per warp)
    auto smem = [&](int threads) {
      const int span = FIR_R * threads + NLpad;
      return sizeof(double2) * std::max<size_t>((size_t)(span + (span >> 3) + 2), (size_t)(threads / 32) * 320);
    };
    const char *msg = "preview window too large for the FIR tile";
    switch (shape) {
    case 1: return preview_launch(ctx, preview_fused_kernel<SIM, 128, 4, ADD, POS>, count, 128, smem(128), msg, d_order, off, pz, d_state, d_com, d_zmpout, d_com_add);
    case 2: return preview_launch(ctx, preview_fused_kernel<SIM, 32, 16, ADD, POS>, count, 32, smem(32), msg, d_order, off, pz, d_state, d_com, d_zmpout, d_com_add);
    default: return preview_launch(ctx, preview_fused_kernel<SIM, 64, 8, ADD, POS>, count, 64, smem(64), msg, d_order, off, pz, d_state, d_com, d_zmpout, d_com_add);
    }
  }
  const double2 *E = reinterpret_cast<const double2 *>(ctx->preview_rec_dev);
  const char *msg = "preview window too large for the tile";
  if (shape == 2)   // swizzled ring + 32 staging slots of 400 B
    return preview_launch(ctx, preview_rec_warp_kernel<SIM, ADD, POS>, count, 32, sizeof(double2) * (size_t)(RW_TILE + NLpad + 25 * 32),
                          msg, d_order, off, pz, d_state, d_com, d_zmpout, d_com_add, E);
  auto smem = [&](int threads) {   // ring of two tiles + the window
    const int cap = 2 * FIR_R * threads + NLpad;
    return sizeof(double2) * (size_t)(cap + (cap >> 3) + 2);
  };
  const double2 *lp = E + 2 * (size_t)NLpad;
  switch (shape) {
  case 1: return preview_launch(ctx, preview_rec_kernel<SIM, 128, 4, ADD, POS>, count, 128, smem(128), msg, d_order, off, pz, d_state, d_com, d_zmpout, d_com_add, E, lp);
  case 3: return preview_launch(ctx, preview_rec_kernel<SIM, 256, 2, ADD, POS>, count, 256, smem(256), msg, d_order, off, pz, d_state, d_com, d_zmpout, d_com_add, E, lp);
  default: return preview_launch(ctx, preview_rec_kernel<SIM, 64, 8, ADD, POS>, count, 64, smem(64), msg, d_order, off, pz, d_state, d_com, d_zmpout, d_com_add, E, lp);
  }
}

extern "C" {

int wg_preview_set_gains(wg_ctx *ctx, const wg_preview_gains_t *g)
{
  if (!ctx || !g || g->NL <= 0 || g->NL > WG_PREVIEW_MAX_NL) return WG_ERR_INVALID;
  wg_device_guard guard(ctx->device);
  static_assert((FIR_R & (FIR_R - 1)) == 0, "FIR_R must be a power of two");
  ctx->preview_image.assign(sizeof(PreviewImage), 0);
  PreviewImage *im = reinterpret_cast<PreviewImage *>(ctx->preview_image.data());
  PreviewConsts &pc = im->pc;
  std::memcpy(pc.A, g->A, sizeof pc.A);
  std::memcpy(pc.B, g->B, sizeof pc.B);
  std::memcpy(pc.C, g->C, sizeof pc.C);
  std::memcpy(pc.Kx, g->Kx, sizeof pc.Kx);
  pc.Ks = g->Ks;
  pc.NL = g->NL;
  pc.NLpad = (g->NL + FIR_R - 1) / FIR_R * FIR_R;
  scan_matrices(*g, false, pc.P[0], pc.G[0], pc.H[0]);
  scan_matrices(*g, true, pc.P[1], pc.G[1], pc.H[1]);
  std::copy(g->F, g->F + g->NL, im->F);          // the rest of F stays zero: the FIR runs over NLpad taps
  // recursive evaluation of the preview sum: usable when the weights have the structure ComputeWeights gives them
  {
    std::vector<double> tables;
    ctx->preview_rec_residual = rec_setup(*g, pc, tables);
    ctx->preview_rec_ok = ctx->preview_rec_residual >= 0.0 && ctx->preview_rec_residual <= WG_PREVIEW_REC_TOL;
    if (ctx->preview_rec_dev) { WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); cudaFree(ctx->preview_rec_dev); ctx->preview_rec_dev = nullptr; }
    if (ctx->preview_rec_ok) {
      WG_CUDA(ctx, cudaMalloc(&ctx->preview_rec_dev, sizeof(double) * tables.size()));
      WG_CUDA(ctx, cudaMemcpy(ctx->preview_rec_dev, tables.data(), sizeof(double) * tables.size(), cudaMemcpyHostToDevice));
    }
  }
  ctx->preview_gains = *g;
  ctx->preview_gen = ++g_pv_gen_counter;           // the device block is refreshed lazily by preview_bind()
  ctx->preview_ready = true;
  return WG_OK;
}

double wg_preview_sum_fit(const wg_preview_gains_t *g)
{
  if (!g || g->NL <= 0 || g->NL > WG_PREVIEW_MAX_NL) return -1.0;
  PreviewConsts pc;
  std::vector<double> tables;
  return rec_setup(*g, pc, tables);
}

// internal (tests): the constants of preview_rec_kernel for a gain set, flat: RF0[8] RFN[8] RV[8][4] RVN[8][4] RW[9][4] RP[6][16],
// then E[NLpad][4] and the lane powers [32][16].  Returns the number of doubles (or -1), writes at most cap of them.
long long wgi_preview_rec_dump(const wg_preview_gains_t *g, double *out, long long cap)
{
  if (!g || g->NL <= 0 || g->NL > WG_PREVIEW_MAX_NL) return -1;
  PreviewConsts pc;
  std::vector<double> tables;
  if (rec_setup(*g, pc, tables) < 0.0) return -1;
  std::vector<double> flat;
  flat.insert(flat.end(), pc.RF0, pc.RF0 + FIR_R);
  flat.insert(flat.end(), pc.RFN, pc.RFN + FIR_R);
  flat.insert(flat.end(), &pc.RV[0][0], &pc.RV[0][0] + FIR_R * 4);
  flat.insert(flat.end(), &pc.RVN[0][0], &pc.RVN[0][0] + FIR_R * 4);
  flat.insert(flat.end(), &pc.RW[0][0], &pc.RW[0][0] + (FIR_R + 1) * 4);
  flat.insert(flat.end(), &pc.RP[0][0], &pc.RP[0][0] + SCAN_LEVELS * 16);
  flat.insert(flat.end(), tables.begin(), tables.end());
  for (long long i = 0; i < (long long)flat.size() && i < cap; ++i) out[i] = flat[(size_t)i];
  return (long long)flat.size();
}

int wg_preview_set_sum_mode(wg_ctx *ctx, int mode)
{
  if (!ctx || mode < WG_PREVIEW_SUM_AUTO || mode > WG_PREVIEW_SUM_RECURSIVE) return WG_ERR_INVALID;
  if (mode == WG_PREVIEW_SUM_RECURSIVE && ctx->preview_ready && !ctx->preview_rec_ok)
    return wg_fail(ctx, WG_ERR_INVALID, "the window weights of this context are not of the form w' L^i v");
  ctx->preview_sum_mode = mode;
  return WG_OK;
}

int wg_preview_set_cta_shape(wg_ctx *ctx, int shape)
{
  if (!ctx || shape < -1 || shape > 3) return WG_ERR_INVALID;
  ctx->preview_cta_shape = shape;
  return WG_OK;
}

int wg_preview_sum_info(wg_ctx *ctx, int *mode_in_use, double *fit_residual)
{
  if (!ctx) return WG_ERR_INVALID;
  if (!ctx->preview_ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_preview_set_gains not called");
  if (mode_in_use)
    *mode_in_use = (ctx->preview_sum_mode != WG_PREVIEW_SUM_DIRECT && ctx->preview_rec_ok) ? WG_PREVIEW_SUM_RECURSIVE : WG_PREVIEW_SUM_DIRECT;
  if (fit_residual) *fit_residual = ctx->preview_rec_residual;
  return WG_OK;
}

int wg_preview_plan_create(wg_ctx *ctx, int B, const int64_t *offsets, wg_preview_plan **out)
{
  if (!ctx || !out || B < 0 || (B > 0 && !offsets)) return WG_ERR_INVALID;
  if (!ctx->preview_ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_preview_set_gains not called");
  wg_device_guard guard(ctx->device);
  *out = nullptr;
  const int NL = ctx->preview_gains.NL;
  if (B > 0 && offsets[0] != 0) return wg_fail(ctx, WG_ERR_INVALID, "offsets[0] must be 0");
  int64_t total_steps = 0;
  std::vector<int> order(B);
  for (int b = 0; b < B; ++b) {
    const int64_t L = offsets[b + 1] - offsets[b];
    if (L < 0 || L > 0x3fffffff) return wg_fail(ctx, WG_ERR_INVALID, "offsets must be non-decreasing");
    if (L >= NL) total_steps += L - NL + 1;
    order[b] = b;
  }
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
    return offsets[a + 1] - offsets[a] > offsets[b + 1] - offsets[b];
  });
  wg_preview_plan *pl = new (std::nothrow) wg_preview_plan();
  if (!pl) return WG_ERR_ALLOC;
  std::memset(pl, 0, sizeof *pl);
  pl->ctx = ctx; pl->B = B; pl->NL = NL;
  pl->total_samples = B > 0 ? offsets[B] : 0;
  pl->total_steps = total_steps;
  // chunks of about equal sample counts, at least 8 trajectories each
  pl->n_chunks = std::max(1, std::min(PV_MAX_CHUNKS, B / 8));
  {
    const int64_t total = B > 0 ? offsets[B] : 0;
    int b = 0;
    pl->chunk_first[0] = 0;
    for (int c = 1; c < pl->n_chunks; ++c) {
      const int64_t target = total * c / pl->n_chunks;
      while (b < B && offsets[b] < target) ++b;
      pl->chunk_first[c] = std::max(b, pl->chunk_first[c - 1]);
    }
    pl->chunk_first[pl->n_chunks] = B;
    for (int c = 0; c <= pl->n_chunks; ++c) pl->chunk_samp[c] = B > 0 ? offsets[pl->chunk_first[c]] : 0;
  }
  std::vector<int> order_chunked(B);
  for (int b = 0; b < B; ++b) order_chunked[b] = b;
  for (int c = 0; c < pl->n_chunks; ++c)
    std::stable_sort(order_chunked.begin() + pl->chunk_first[c], order_chunked.begin() + pl->chunk_first[c + 1], [&](int a, int b) {
      return offsets[a + 1] - offsets[a] > offsets[b + 1] - offsets[b];
    });
  cudaError_t e = cudaMalloc(&pl->d_offsets, sizeof(int64_t) * (B + 1));
  if (e == cudaSuccess) e = cudaMalloc(&pl->d_order, sizeof(int) * std::max(1, B));
  if (e == cudaSuccess) e = cudaMalloc(&pl->d_order_chunked, sizeof(int) * std::max(1, B));
  if (e == cudaSuccess && B > 0)
    e = cudaMemcpyAsync(pl->d_order_chunked, order_chunked.data(), sizeof(int) * B, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&pl->up_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&pl->down_stream, cudaStreamNonBlocking);
  for (int c = 0; c < PV_MAX_CHUNKS && e == cudaSuccess; ++c) {
    e = cudaEventCreateWithFlags(&pl->ev_up[c], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&pl->ev_k[c], cudaEventDisableTiming);
  }
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&pl->ev_done, cudaEventDisableTiming);
  if (e == cudaSuccess && B > 0)
    e = cudaMemcpyAsync(pl->d_offsets, offsets, sizeof(int64_t) * (B + 1), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess && B > 0)
    e = cudaMemcpyAsync(pl->d_order, order.data(), sizeof(int) * B, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) {
    wg_fail(ctx, WG_ERR_CUDA, "wg_preview_plan_create", e);
    wg_preview_plan_destroy(pl);
    return WG_ERR_CUDA;
  }
  *out = pl;
  return WG_OK;
}

int wg_preview_plan_destroy(wg_preview_plan *pl)
{
  if (!pl) return WG_OK;
  wg_device_guard guard(pl->ctx->device);
  cudaStreamSynchronize(pl->ctx->stream);
  if (pl->up_stream) { cudaStreamSynchronize(pl->up_stream); cudaStreamDestroy(pl->up_stream); }
  if (pl->down_stream) { cudaStreamSynchronize(pl->down_stream); cudaStreamDestroy(pl->down_stream); }
  for (int c = 0; c < PV_MAX_CHUNKS; ++c) { if (pl->ev_up[c]) cudaEventDestroy(pl->ev_up[c]); if (pl->ev_k[c]) cudaEventDestroy(pl->ev_k[c]); }
  if (pl->ev_done) cudaEventDestroy(pl->ev_done);
  cudaFree(pl->d_offsets); cudaFree(pl->d_order); cudaFree(pl->d_order_chunked);
  cudaFree(pl->d_zmp); cudaFree(pl->d_state); cudaFree(pl->d_com); cudaFree(pl->d_zmpout); cudaFree(pl->d_add);
  delete pl;
  return WG_OK;
}

// Internal (zmpdisc.cu, wg_kajita_stream): give the plan's B trajectories new offsets, in its own device array.  The copy is
// asynchronous on the context stream: offsets_host must stay unchanged until the stream has passed it.
int wgi_preview_plan_set_offsets(wg_preview_plan *pl, const int64_t *offsets_host)
{
  wg_ctx *ctx = pl->ctx;
  int64_t total_steps = 0;
  for (int b = 0; b < pl->B; ++b) {
    const int64_t L = offsets_host[b + 1] - offsets_host[b];
    if (L >= pl->NL) total_steps += L - pl->NL + 1;
  }
  pl->total_samples = pl->B > 0 ? offsets_host[pl->B] : 0;
  pl->total_steps = total_steps;
  if (pl->B > 0)
    WG_CUDA(ctx, cudaMemcpyAsync(pl->d_offsets, offsets_host, sizeof(int64_t) * (pl->B + 1), cudaMemcpyHostToDevice, ctx->stream));
  return WG_OK;
}

int64_t wg_preview_plan_total_steps(const wg_preview_plan *pl) { return pl ? pl->total_steps : 0; }
int64_t wg_preview_plan_total_samples(const wg_preview_plan *pl) { return pl ? pl->total_samples : 0; }

// Launch over `count` trajectories listed in d_order (device array of trajectory indices of this plan).
int wgi_preview_launch_range(wg_ctx *ctx, wg_preview_plan *pl, const int *d_order, int count, const double *d_zmp,
                            double *d_state, double *d_com, double *d_zmpout, int simulation, const double *d_com_add,
                            int pos_only)
{
  if (pl->total_steps == 0 || count <= 0) return WG_OK;
  // CTA shape: 0 = 64 threads x 8 CTAs/SM, 1 = 128 x 4, 2 = one warp per trajectory (preview_rec_warp_kernel), 3 = 256 x 2 (2 and 3:
  // the recursive sum only).  WG_PREVIEW_SHAPE / wg_preview_set_cta_shape force one; otherwise the recursive path takes the shape
  // that is fastest for the number of trajectories of THIS launch, measured on walks of configs[1] (G steps/s):
  //   walks     32    64    128    256    512   1024   1536   2048   3072   4096
  //   64 x 8     -     -      -    8.8   14.8   23.9   27.5   31.2   34.2   34.7
  //   128 x 4   2.2   4.2    8.0  14.1   21.3   27.4   31.7   32.2   34.8   35.4
  //   256 x 2   2.7   5.1    9.7  16.4   23.8     -      -      -      -      -
  //   one warp   -     -      -    5.7   11.2   22.0   29.8   36.9   43.6   48.7
  // (ten one-warp CTAs per SM need 1480 trajectories to fill 148 SMs; below that more warps per trajectory finish sooner).
  // The direct sum stays at 64 x 8 (measured 0.752 ms vs 0.778 (128 x 4) and 0.766 (32 x 16) on config 2).
  static int forced = -2;
  if (forced == -2) {
    const char *e = getenv("WG_PREVIEW_SHAPE");
    forced = e ? atoi(e) : -1;
  }
  const bool recursive = ctx->preview_sum_mode != WG_PREVIEW_SUM_DIRECT && ctx->preview_rec_ok;
  int shape = forced >= 0 ? forced : ctx->preview_cta_shape >= 0 ? ctx->preview_cta_shape : !recursive ? 0 : count >= 1792 ? 2 : count >= 768 ? 1 : 3;
  if (shape == 3) {      // eight warps per trajectory (tiles of 2048 ticks): the ring of two tiles + the window must fit 96 KB
    const int NLpad = (pl->NL + FIR_R - 1) / FIR_R * FIR_R, cap = 2 * FIR_R * 256 + NLpad;
    if (!recursive || sizeof(double2) * (size_t)(cap + (cap >> 3) + 2) > 96 * 1024) shape = 1;
  }
  if (ctx->preview_sum_mode == WG_PREVIEW_SUM_RECURSIVE && !ctx->preview_rec_ok)
    return wg_fail(ctx, WG_ERR_INVALID, "WG_PREVIEW_SUM_RECURSIVE: the window weights of this context are not of the form w' L^i v");
  // variant: position only (the CoM (x, y) pair leaves through the ZMP path), the second stage (always with the integrated
  // error, ZMPPreviewControlWithMultiBodyZMP.cpp:343-347), or the plain run
  const double2 *pz = reinterpret_cast<const double2 *>(d_zmp);
  auto launch = [&](auto sim, auto add, auto pos) {
    return preview_launch_variant<sim, add, pos>(ctx, pl, recursive, shape, d_order, count, pz, d_state, pos ? nullptr : d_com,
                                                 d_zmpout, add ? d_com_add : nullptr);
  };
  const std::true_type T{};
  const std::false_type F{};
  if (pos_only) return simulation ? launch(T, F, T) : launch(F, F, T);
  if (d_com_add && d_com) return launch(T, T, F);
  return simulation ? launch(T, F, F) : launch(F, F, F);
}

static int preview_run(wg_ctx *ctx, wg_preview_plan *pl, int mem, const double *zmpref_xy, double *state,
                       double *com_out, double *zmp_out, int simulation, const double *com_add, int pos_only = 0)
{
  if (!ctx || !pl || pl->ctx != ctx || !state || (!zmpref_xy && pl->total_samples > 0)) return WG_ERR_INVALID;
  if (!ctx->preview_ready || ctx->preview_gains.NL != pl->NL)
    return wg_fail(ctx, WG_ERR_NOT_READY, "gains changed since the plan was created");
  wg_device_guard guard(ctx->device);
  if (pl->B == 0) return WG_OK;
  if (mem == WG_MEM_DEVICE) {
    // the kernels move rows with 128-bit (and wider) accesses and hand CoM rows to the bulk-copy engine: 16-byte aligned arrays
    if ((reinterpret_cast<uintptr_t>(zmpref_xy) | reinterpret_cast<uintptr_t>(com_out) | reinterpret_cast<uintptr_t>(zmp_out) |
         reinterpret_cast<uintptr_t>(com_add)) & 15)
      return wg_fail(ctx, WG_ERR_INVALID, "preview: device arrays must be 16-byte aligned");
    return wgi_preview_launch_range(ctx, pl, pl->d_order, pl->B, zmpref_xy, state, com_out, zmp_out, simulation, com_add, pos_only);
  }
  if (mem != WG_MEM_HOST) return WG_ERR_INVALID;
  const size_t ns = (size_t)pl->total_samples;
  if (com_add && !pl->d_add) WG_CUDA(ctx, cudaMalloc(&pl->d_add, sizeof(double) * 6 * std::max<size_t>(1, ns)));
  if (!pl->d_zmp) WG_CUDA(ctx, cudaMalloc(&pl->d_zmp, sizeof(double) * 2 * std::max<size_t>(1, ns)));
  if (!pl->d_state) WG_CUDA(ctx, cudaMalloc(&pl->d_state, sizeof(double) * 8 * pl->B));
  if (com_out && !pl->d_com) {  // zero once: rows past a trajectory's last step read back as 0 in host mode
    WG_CUDA(ctx, cudaMalloc(&pl->d_com, sizeof(double) * 6 * std::max<size_t>(1, ns)));
    WG_CUDA(ctx, cudaMemsetAsync(pl->d_com, 0, sizeof(double) * 6 * std::max<size_t>(1, ns), ctx->stream));
  }
  if (zmp_out && !pl->d_zmpout) {
    WG_CUDA(ctx, cudaMalloc(&pl->d_zmpout, sizeof(double) * 2 * std::max<size_t>(1, ns)));
    WG_CUDA(ctx, cudaMemsetAsync(pl->d_zmpout, 0, sizeof(double) * 2 * std::max<size_t>(1, ns), ctx->stream));
  }
  // ---- pipelined over chunks: upload (up_stream) -> kernel (ctx->stream) -> downloads (down_stream)
  WG_CUDA(ctx, cudaMemcpyAsync(pl->d_state, state, sizeof(double) * 8 * pl->B, cudaMemcpyHostToDevice, ctx->stream));
  WG_CUDA(ctx, cudaEventRecord(pl->ev_done, ctx->stream));          // allocations / memsets / previous call are done
  WG_CUDA(ctx, cudaStreamWaitEvent(pl->up_stream, pl->ev_done, 0));
  for (int c = 0; c < pl->n_chunks; ++c) {
    const int b0 = pl->chunk_first[c], b1 = pl->chunk_first[c + 1];
    const size_t s0 = (size_t)pl->chunk_samp[c], cnt = (size_t)(pl->chunk_samp[c + 1] - pl->chunk_samp[c]);
    if (b1 <= b0) continue;
    if (cnt) WG_CUDA(ctx, cudaMemcpyAsync(pl->d_zmp + 2 * s0, zmpref_xy + 2 * s0, sizeof(double) * 2 * cnt, cudaMemcpyHostToDevice, pl->up_stream));
    if (cnt && com_add)
      WG_CUDA(ctx, cudaMemcpyAsync(pl->d_add + 6 * s0, com_add + 6 * s0, sizeof(double) * 6 * cnt, cudaMemcpyHostToDevice, pl->up_stream));
    WG_CUDA(ctx, cudaEventRecord(pl->ev_up[c], pl->up_stream));
    WG_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, pl->ev_up[c], 0));
    int rc = wgi_preview_launch_range(ctx, pl, pl->d_order_chunked + b0, b1 - b0, pl->d_zmp, pl->d_state,
                                      com_out ? pl->d_com : nullptr, zmp_out ? pl->d_zmpout : nullptr, simulation,
                                      com_add ? pl->d_add : nullptr, pos_only);
    if (rc != WG_OK) return rc;
    WG_CUDA(ctx, cudaEventRecord(pl->ev_k[c], ctx->stream));
    WG_CUDA(ctx, cudaStreamWaitEvent(pl->down_stream, pl->ev_k[c], 0));
    if (com_out && cnt)
      WG_CUDA(ctx, cudaMemcpyAsync(com_out + 6 * s0, pl->d_com + 6 * s0, sizeof(double) * 6 * cnt, cudaMemcpyDeviceToHost, pl->down_stream));
    if (zmp_out && cnt)
      WG_CUDA(ctx, cudaMemcpyAsync(zmp_out + 2 * s0, pl->d_zmpout + 2 * s0, sizeof(double) * 2 * cnt, cudaMemcpyDeviceToHost, pl->down_stream));
  }
  WG_CUDA(ctx, cudaMemcpyAsync(state, pl->d_state, sizeof(double) * 8 * pl->B, cudaMemcpyDeviceToHost, ctx->stream));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  WG_CUDA(ctx, cudaStreamSynchronize(pl->down_stream));
  return WG_OK;
}

int wg_preview_run_batch(wg_ctx *ctx, wg_preview_plan *pl, int mem, const double *zmpref_xy, double *state,
                         double *com_out, double *zmp_out, int simulation)
{
  return preview_run(ctx, pl, mem, zmpref_xy, state, com_out, zmp_out, simulation, nullptr);
}

int wg_preview_run_batch_pos(wg_ctx *ctx, wg_preview_plan *pl, int mem, const double *zmpref_xy, double *state,
                             double *com_pos_out, int simulation)
{
  if (!com_pos_out) return WG_ERR_INVALID;
  return preview_run(ctx, pl, mem, zmpref_xy, state, nullptr, com_pos_out, simulation, nullptr, 1);
}

int wg_preview_stage2_run_batch(wg_ctx *ctx, wg_preview_plan *pl, int mem, const double *delta_zmp_xy,
                                const double *com_stage1, double *state2, double *com_final_out, double *dzmp_out)
{
  if (!com_stage1 || !com_final_out) return WG_ERR_INVALID;
  return preview_run(ctx, pl, mem, delta_zmp_xy, state2, com_final_out, dzmp_out, 1, com_stage1);
}

}  // extern "C"

// EvaluateMultiBodyZMP (ZMPPreviewControlWithMultiBodyZMP.cpp:464-469): after the first stage popped its FIFO,
// delta[k] = ZMPRef[k + 1] - ZMPmultibody[k].
__global__ void __launch_bounds__(256)
delta_zmp_kernel(int B, const int64_t *__restrict__ offsets, const double2 *__restrict__ ref, const double2 *__restrict__ mb,
                 double2 *__restrict__ delta)
{
  for (int b = blockIdx.y; b < B; b += gridDim.y) {
    const int64_t o = offsets[b], L = offsets[b + 1] - o;
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < L; k += (int64_t)gridDim.x * blockDim.x) {
      double2 d = make_double2(0.0, 0.0);
      if (k + 1 < L) { const double2 r = ref[o + k + 1], m = mb[o + k]; d = make_double2(r.x - m.x, r.y - m.y); }
      delta[o + k] = d;
    }
  }
}

extern "C" int wg_preview_delta_zmp(wg_ctx *ctx, wg_preview_plan *pl, int mem, const double *zmpref_xy,
                                    const double *zmp_multibody_xy, double *delta_out)
{
  if (!ctx || !pl || pl->ctx != ctx || !zmpref_xy || !zmp_multibody_xy || !delta_out) return WG_ERR_INVALID;
  wg_device_guard guard(ctx->device);
  if (pl->B == 0 || pl->total_samples == 0) return WG_OK;
  const size_t ns = (size_t)pl->total_samples;
  const double *d_ref = zmpref_xy, *d_mb = zmp_multibody_xy;
  double *d_out = delta_out;
  if (mem == WG_MEM_HOST) {
    if (!pl->d_zmp) WG_CUDA(ctx, cudaMalloc(&pl->d_zmp, sizeof(double) * 2 * ns));
    if (!pl->d_add) WG_CUDA(ctx, cudaMalloc(&pl->d_add, sizeof(double) * 6 * ns));   // scratch here; d_zmpout must stay zero past the last step
    WG_CUDA(ctx, cudaMemcpyAsync(pl->d_zmp, zmpref_xy, sizeof(double) * 2 * ns, cudaMemcpyHostToDevice, ctx->stream));
    WG_CUDA(ctx, cudaMemcpyAsync(pl->d_add, zmp_multibody_xy, sizeof(double) * 2 * ns, cudaMemcpyHostToDevice, ctx->stream));
    d_ref = pl->d_zmp; d_mb = pl->d_add; d_out = pl->d_add;   // in place: element k only reads mb[k]
  } else if (mem != WG_MEM_DEVICE) return WG_ERR_INVALID;
  const int64_t avg = (pl->total_samples + pl->B - 1) / pl->B;
  dim3 grid((unsigned)std::max<int64_t>(1, std::min<int64_t>(64, (avg + 255) / 256)), (unsigned)std::min(pl->B, 65535));
  delta_zmp_kernel<<<grid, 256, 0, ctx->stream>>>(pl->B, pl->d_offsets, reinterpret_cast<const double2 *>(d_ref),
                                                 reinterpret_cast<const double2 *>(d_mb), reinterpret_cast<double2 *>(d_out));
  WG_LAUNCHED(ctx);
  if (mem == WG_MEM_HOST) {
    WG_CUDA(ctx, cudaMemcpyAsync(delta_out, d_out, sizeof(double) * 2 * ns, cudaMemcpyDeviceToHost, ctx->stream));
    WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return WG_OK;
}

// ---- single tick for the class wrappers (PreviewControl::OneIterationOfPreview called once per 5 ms tick) ----
// One CTA: the 2 x NL window products are reduced over 128 threads, thread 0 then runs the tick in the reference's
// statement order.  Window, state and results live in ONE mapped pinned host buffer owned by the context (zero copy:
// the kernel reads 16 NL bytes over PCIe and writes 10 doubles back), so a tick is one launch + one stream
// synchronisation: no allocation, no plan, no memcpy calls.
struct PreviewTickBuf {
  double *h = nullptr;      // pinned, mapped: [2 NLmax window | 8 state | 2 zmp]
  double *d = nullptr;      // device alias of h
  int cap_nl = 0;
};

template <bool SIM>
__global__ void __launch_bounds__(128)
preview_tick_kernel(const double2 *__restrict__ win, double *__restrict__ io)
{
  __shared__ double2 part[4];
  const int NL = c_pc.NL, t = threadIdx.x;
  double fx = 0.0, fy = 0.0;
  for (int i = t; i < NL; i += 128) {
    const double2 v = win[i];
    fx = fma(c_F[i], v.x, fx);
    fy = fma(c_F[i], v.y, fy);
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    fx += __shfl_down_sync(0xffffffffu, fx, d);
    fy += __shfl_down_sync(0xffffffffu, fy, d);
  }
  if ((t & 31) == 0) part[t >> 5] = make_double2(fx, fy);
  __syncthreads();
  if (t == 0) {
    fx = (part[0].x + part[1].x) + (part[2].x + part[3].x);
    fy = (part[0].y + part[1].y) + (part[2].y + part[3].y);
    Axis ax, ay;
    ax.x0 = io[0]; ax.x1 = io[1]; ax.x2 = io[2]; ax.s = io[6];
    ay.x0 = io[3]; ay.x1 = io[4]; ay.x2 = io[5]; ay.s = io[7];
    const double2 p0 = win[0];
    const double zx = preview_tick<SIM>(ax, fx, p0.x);
    const double zy = preview_tick<SIM>(ay, fy, p0.y);
    io[0] = ax.x0; io[1] = ax.x1; io[2] = ax.x2; io[6] = ax.s;
    io[3] = ay.x0; io[4] = ay.x1; io[5] = ay.x2; io[7] = ay.s;
    io[8] = zx; io[9] = zy;
  }
}

extern "C" {

void wg_preview_release(wg_ctx *ctx)
{
  if (ctx && ctx->preview_rec_dev) { cudaFree(ctx->preview_rec_dev); ctx->preview_rec_dev = nullptr; }
  PreviewTickBuf *tb = static_cast<PreviewTickBuf *>(ctx->preview_tick);
  if (!tb) return;
  if (tb->h) cudaFreeHost(tb->h);
  delete tb;
  ctx->preview_tick = nullptr;
}

int wg_preview_one_iteration(wg_ctx *ctx, double *x, double *y, double *sxzmp, double *syzmp,
                             const double *window_xy, int n_available, double *zmpx2, double *zmpy2,
                             int simulation)
{
  if (!ctx || !x || !y || !sxzmp || !syzmp || !window_xy || !zmpx2 || !zmpy2) return WG_ERR_INVALID;
  if (!ctx->preview_ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_preview_set_gains not called");
  const int NL = ctx->preview_gains.NL;
  if (n_available < NL) return wg_fail(ctx, WG_ERR_WINDOW, "ZMPPositions.size()<m_SizeOfPreviewWindow");
  wg_device_guard guard(ctx->device);
  PreviewTickBuf *tb = static_cast<PreviewTickBuf *>(ctx->preview_tick);
  if (!tb) { tb = new (std::nothrow) PreviewTickBuf(); if (!tb) return WG_ERR_ALLOC; ctx->preview_tick = tb; }
  if (tb->cap_nl < NL) {
    if (tb->h) { cudaFreeHost(tb->h); tb->h = nullptr; tb->cap_nl = 0; }
    WG_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(&tb->h), sizeof(double) * (2 * (size_t)NL + 10), cudaHostAllocMapped));
    WG_CUDA(ctx, cudaHostGetDevicePointer(reinterpret_cast<void **>(&tb->d), tb->h, 0));
    tb->cap_nl = NL;
  }
  std::memcpy(tb->h, window_xy, sizeof(double) * 2 * (size_t)NL);
  double *io = tb->h + 2 * (size_t)tb->cap_nl;
  for (int i = 0; i < 3; ++i) { io[i] = x[i]; io[3 + i] = y[i]; }
  io[6] = *sxzmp; io[7] = *syzmp;
  {
    std::lock_guard<std::mutex> lock(g_pv_mutex);
    const int rc = preview_bind(ctx);
    if (rc != WG_OK) return rc;
    const double2 *dw = reinterpret_cast<const double2 *>(tb->d);
    double *dio = tb->d + 2 * (size_t)tb->cap_nl;
    if (simulation) preview_tick_kernel<true><<<1, 128, 0, ctx->stream>>>(dw, dio);
    else preview_tick_kernel<false><<<1, 128, 0, ctx->stream>>>(dw, dio);
    WG_LAUNCHED(ctx);
  }
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < 3; ++i) { x[i] = io[i]; y[i] = io[3 + i]; }
  *sxzmp = io[6]; *syzmp = io[7];
  *zmpx2 = io[8]; *zmpy2 = io[9];
  return WG_OK;
}

}  // extern "C"
