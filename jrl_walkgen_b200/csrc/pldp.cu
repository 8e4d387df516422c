// pldp.cu - batched Dimitrov PLDP solver and OptCholesky for sm_100a.
//
// Replaces PLDPSolver::SolveProblem and its helpers (src/Mathematics/PLDPSolver.cpp:287-1007) and
// OptCholesky (src/Mathematics/OptCholesky.cpp:92-302) for whole batches of independent problems.
//
// One warp owns one problem.  The control vector has 2N = 32 entries = one per lane, so the iterate V_k, the
// descent direction c, the projected direction d live in registers (one double per lane) and move with shuffles;
// the Cholesky factor of E E^T (at most 32 x 32: PLDP never drops a constraint and E has 32 columns) is packed in
// shared memory.  The constraint matrix (m+1) x 32, column-major exactly as the reference receives it, is read
// from global memory / L2 by "row per lane" loops (consecutive lanes read consecutive rows: coalesced).
//
// Arithmetic follows the reference statement by statement with NON-fused multiplies and adds (__dmul_rn/__dadd_rn)
// in the reference's summation order throughout, so that on identical inputs the iterates, the step lengths and therefore the
// sequence of activated constraints are the same as the reference's x86-64 object code (which has no FMA
// contraction at -O3 without -march).  Differences by design: the wall-clock cap of 1.3 ms (PLDPSolver.cpp:69,
// :890-900) becomes an iteration cap, and the paths on which the reference calls exit(0) (:822-828) or prints
// return a status instead.
#include "wg_common.h"
#include <algorithm>
#include <vector>
#include <cmath>

#include "pldp.cuh"

namespace {

struct PldpHost {
  PldpConsts h;
  PldpConsts *d = nullptr;
  bool ready = false;
  // staging for WG_MEM_HOST calls
  void *buf[13] = {nullptr};
  size_t cap[13] = {0};
  int *d_next = nullptr;   // work counter of pldp_kernel
  // WG_MEM_HOST pipeline
  cudaStream_t up = nullptr, down = nullptr;
  cudaEvent_t ev_up[4] = {nullptr}, ev_k[4] = {nullptr}, ev0 = nullptr;
};

// The rank-structured form of the constraint matrix (wg_pldp_solve_batch_ranked): per instance three arrays of m entries.
struct PldpRanked {
  const double *a0, *a1;      // [B][row_stride]
  const unsigned char *ri;    // [B][row_stride]
  long long row_stride;
};

// One instance per warp.  RANKED = false: the dense (m+1) x 32 column-major matrix the reference hands to SolveProblem, read
// from L2 (8 CTAs/SM at 64 registers).  RANKED = true: the matrix is formed on the fly from (A_r(0), A_r(1), i_r) and the
// context's Pu (RankMat): 17 bytes per row instead of 256, nothing re-read from L2 (4 CTAs/SM at 128 registers).
template <bool RANKED>
__global__ void __launch_bounds__(PLDP_WARPS * 32, RANKED ? 4 : 8)
pldp_kernel(int B, const PldpConsts *__restrict__ Cp, const double *__restrict__ D, const int *__restrict__ mvec,
            const double *__restrict__ DPu, long long dpu_stride, const double *__restrict__ DPx, long long dpx_stride,
            const double *__restrict__ ZMPRef, const double *__restrict__ XkYk, double *__restrict__ X,
            const int *__restrict__ similar, long long similar_stride, const int *__restrict__ nremoved,
            const int *__restrict__ starting, wg_pldp_state *__restrict__ hot, int hot_start, int max_iter,
            double tol, wg_pldp_info *__restrict__ info, int a_cap, int *__restrict__ next_problem, PldpRanked rk)
{
  __shared__ PldpWarp ws[PLDP_WARPS];
  __shared__ double s_t1[PLDP_WARPS][WG_PLDP_MAX_ROWS];     // SimilarConstraints scratch (see pldp_solve_warp)
  __shared__ unsigned s_amask[PLDP_WARPS][4];
  __shared__ double sPu[RANKED ? 2 * PLDP_N * PLDP_N : 1];   // Pu and its transpose
  __shared__ double s_rowa[RANKED ? PLDP_WARPS : 1][2][RANKED ? WG_PLDP_MAX_ROWS : 1];   // the instance's (A_r(0), A_r(1)) ...
  __shared__ unsigned char s_rowi[RANKED ? PLDP_WARPS : 1][RANKED ? WG_PLDP_MAX_ROWS : 4];   // ... and i_r, staged once
  extern __shared__ __align__(16) double sA[];   // a_cap doubles per warp: the instance's constraint matrix (0: read it from L2)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const PldpConsts &C = *Cp;
  PldpWarp &w = ws[warp];
  constexpr int N = PLDP_N;
  if (RANKED) {
    for (int e = threadIdx.x; e < N * N; e += blockDim.x) { sPu[e] = C.Pu[e]; sPu[N * N + e] = C.PuT[e]; }
    __syncthreads();
  }
  // iteration counts differ (5-33 on the bench workload): every warp takes its next problem from a work counter
  for (;;) {
    int b = 0;
    if (lane == 0) b = atomicAdd(next_problem, 1);
    b = __shfl_sync(0xffffffffu, b, 0);
    if (b >= B) break;
    const int m = mvec[b];
    if (m < 0 || m > WG_PLDP_MAX_ROWS) {
      // device-side batches are not validated on the host: refuse the instance instead of ignoring rows past 128
      X[(size_t)b * PLDP_U + lane] = nan("");
      if (info) {
        if (lane == 0) { info[b].rc = -1; info[b].status = 7; info[b].iterations = 0; info[b].n_active = 0; }
        info[b].active[lane] = -1;
      }
      continue;
    }
    const int ld = m + 1;
    const double *A = RANKED ? nullptr : DPu + (size_t)b * dpu_stride;
    if (!RANKED && a_cap > 0 && ld * PLDP_U <= a_cap) {
      // stage the (m+1) x 32 column-major matrix once: every iteration re-reads all of it
      double *dst = sA + (size_t)warp * a_cap;
      const int n = ld * PLDP_U;
      __syncwarp();
      if ((((size_t)A) & 15) == 0) {
        const double2 *src2 = reinterpret_cast<const double2 *>(A);
        double2 *dst2 = reinterpret_cast<double2 *>(dst);
        for (int e = lane; e < (n >> 1); e += 32) dst2[e] = __ldg(src2 + e);
        if ((n & 1) && lane == 0) dst[n - 1] = A[n - 1];
      } else {
        for (int e = lane; e < n; e += 32) dst[e] = A[e];
      }
      __syncwarp();
      A = dst;
    }
    const double *bv = DPx + (size_t)b * dpx_stride;
    const bool start = starting ? starting[b] != 0 : true;
    const double Dl = D[(size_t)b * PLDP_U + lane];
    const double *zr = ZMPRef + (size_t)b * PLDP_U;
    const double *xk = XkYk + (size_t)b * 6;
    const bool hs = hot && hot_start;
    PldpRes r;
    const PldpSim simv{similar ? similar + (size_t)b * similar_stride : nullptr, s_t1[warp], s_amask[warp]};
    const PldpSim *simp = similar ? &simv : nullptr;
    double Vk;
    if (RANKED) {
      const size_t ro = (size_t)b * rk.row_stride;
      __syncwarp();
      for (int e = lane; e < m; e += 32) {
        s_rowa[warp][0][e] = rk.a0[ro + e];
        s_rowa[warp][1][e] = rk.a1[ro + e];
        const unsigned char i_r = rk.ri[ro + e];
        s_rowi[warp][e] = i_r < N ? i_r : 0;      // host-side batches are validated; a bad device-side index must not read outside Pu
      }
      __syncwarp();
      const RankMat M{s_rowa[warp][0], s_rowa[warp][1], s_rowi[warp], sPu, sPu + N * N};
      Vk = pldp_solve_warp(C, w, M, m, bv, Dl, zr, xk, hs && !start, hs ? hot[b].prev_zmp : nullptr,
                           hs ? hot[b].n_prev : 0, hs ? hot[b].prev_active : nullptr,
                           nremoved ? nremoved[b] : 0, max_iter, tol, lane, r, simp);
    } else {
      const DenseMat M{A, ld};
      Vk = pldp_solve_warp(C, w, M, m, bv, Dl, zr, xk, hs && !start, hs ? hot[b].prev_zmp : nullptr,
                           hs ? hot[b].n_prev : 0, hs ? hot[b].prev_active : nullptr,
                           nremoved ? nremoved[b] : 0, max_iter, tol, lane, r, simp);
    }
    const int status = r.status, it = r.it, k = r.k, kproj = r.kproj;
    const double v2 = r.v2;
    const int ii = lane & (N - 1), ax = lane >> 4;
    // ---- results
    X[(size_t)b * PLDP_U + lane] = Vk;
    const double x0 = bcast(Vk, 0), xn = bcast(Vk, N);
    int rc = 0;
    if (isnan(x0) || isnan(xn) || isinf(x0) || isinf(xn)) rc = -1;   // PLDPSolver.cpp:955-964
    if (hot && hot_start) {
      // keep the rows whose multiplier is negative (:909-920) and store the ZMP solution (:1009-1032)
      const unsigned keep = __ballot_sync(0xffffffffu, lane < kproj && v2 < 0.0);
      if (lane < kproj && v2 < 0.0) hot[b].prev_active[__popc(keep & ((1u << lane) - 1u))] = w.active[lane];
      if (lane == 0) hot[b].n_prev = __popc(keep);
      double z = 0.0;
#pragma unroll 2
      for (int j = 0; j < N; ++j) z = add(z, mul(C.Pu[j * N + ii], bcast(Vk, j + N * ax)));
#pragma unroll
      for (int j = 0; j < 3; ++j) z = add(z, mul(C.Px[ii * 3 + j], xk[3 * ax + j]));
      hot[b].prev_zmp[lane] = z;
    }
    if (info) {
      if (lane == 0) { info[b].rc = rc; info[b].status = status; info[b].iterations = it; info[b].n_active = k; }
      info[b].active[lane] = (lane < k) ? w.active[lane] : -1;
    }
    __syncwarp();
  }
}

// OptCholesky batched: rows k0..k-1 of L for the active rows `rows` of each instance's A.
//   mode 1 (MODE_FORTRAN): A column-major, element (r, c) at A[r + c (nb_constraints + 1)]  (OptCholesky.cpp:171-223)
//   mode 0 (MODE_NORMAL):  A row-major,    element (r, c) at A[r card_u + c]                 (OptCholesky.cpp:123-169)
// L is row-major with leading dimension nb_max (the caller-owned storage the reference writes into).
__global__ void __launch_bounds__(128)
optchol_kernel(int B, int mode, int nb_max, int card_u, int nb_constraints, const double *__restrict__ A,
               long long a_stride, const int *__restrict__ rows, int rows_stride, int k0, int k1,
               double *__restrict__ Lout, long long l_stride)
{
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int b = blockIdx.x * 4 + warp; b < B; b += gridDim.x * 4) {
    const double *Ab = A + (size_t)b * a_stride;
    const int *act = rows + (size_t)b * rows_stride;
    double *L = Lout + (size_t)b * l_stride;
    const long long rs = mode ? 1 : card_u, cs = mode ? (nb_constraints + 1) : 1;
    for (int i = k0; i < k1; ++i) {
      const double *ri = Ab + (size_t)act[i] * rs;
      // columns j = 0..i, 32 at a time; the recurrence over j is sequential, lane (j % 32) finalises L(i,j)
      for (int j = 0; j <= i; ++j) {
        const double *rj = Ab + (size_t)act[j] * rs;
        // M(i,j) in the reference's order, then r -= L(i,k) L(j,k) for k < j: one lane does the serial sum
        // (bit-faithful); different (i,j) pairs cannot run ahead because of the recurrence on L(i,k<j).
        if (lane == 0) {
          double r = 0.0;
          for (int c = 0; c < card_u; ++c) r = add(r, mul(ri[c * cs], rj[c * cs]));
          const double *Li = L + (size_t)i * nb_max, *Lj = L + (size_t)j * nb_max;
          for (int kk = 0; kk < j; ++kk) r = add(r, -mul(Li[kk], Lj[kk]));
          L[(size_t)i * nb_max + j] = (j != i) ? r / Lj[j] : sqrt(r);
        }
        __syncwarp();
      }
    }
  }
}

// ComputeNormalCholeskyOnANormal (OptCholesky.cpp:225-259) + ComputeInverseCholeskyNormal (:261-302), one warp each.
__global__ void __launch_bounds__(128)
optchol_full_kernel(int B, int n, const double *__restrict__ A, double *__restrict__ Lout, double *__restrict__ iLout,
                    int inv_size)
{
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int b = blockIdx.x * 4 + warp; b < B; b += gridDim.x * 4) {
    const double *Ab = A ? A + (size_t)b * n * n : nullptr;
    double *L = Lout + (size_t)b * n * n;
    double *iL = iLout ? iLout + (size_t)b * n * n : nullptr;
    if (Ab) {
      for (int i = 0; i < n; ++i) {
        for (int j = 0; j <= i; ++j) {
          if (lane == 0) {
            double r = Ab[(size_t)i * n + j];
            for (int kk = 0; kk < j; ++kk) r = add(r, -mul(L[(size_t)i * n + kk], L[(size_t)j * n + kk]));
            L[(size_t)i * n + j] = (j != i) ? r / L[(size_t)j * n + j] : sqrt(r);
          }
          __syncwarp();
        }
      }
    }
    if (iL) {
      // columns lj are independent of each other: lane-strided over lj, serial down the column as the reference
      for (int lj = inv_size - 1 - lane; lj >= 0; lj -= 32) {
        const double inv = 1 / L[(size_t)lj * n + lj];
        iL[(size_t)lj * n + lj] = inv;
      }
      __syncwarp();
      // iL(li,lj) = -iL(lj,lj) * sum_{lk=lj+1..} iL(li,lk) L(lk,lj): needs iL(li, lk>lj) -> process lj descending
      for (int lj = inv_size - 1; lj >= 0; --lj) {
        const double inv = iL[(size_t)lj * n + lj];
        for (int li = lj + 1 + lane; li < inv_size; li += 32) {
          double r = 0.0;
          for (int lk = lj + 1; lk < inv_size; ++lk) r = add(r, mul(iL[(size_t)li * n + lk], L[(size_t)lk * n + lj]));
          iL[(size_t)li * n + lj] = mul(-inv, r);
        }
        __syncwarp();
      }
    }
  }
}

PldpHost *pldp_of(wg_ctx *ctx)
{
  if (!ctx->pldp) ctx->pldp = new PldpHost();
  return static_cast<PldpHost *>(ctx->pldp);
}

int grid_for(wg_ctx *ctx, int B, int warps) { int g = (B + warps - 1) / warps; int cap = ctx->sm_count * 8; return g < cap ? (g > 0 ? g : 1) : cap; }

}  // namespace

extern "C" const void *wgi_pldp_device_consts(wg_ctx *ctx)
{
  PldpHost *p = static_cast<PldpHost *>(ctx->pldp);
  return (p && p->ready) ? p->d : nullptr;
}

void wg_pldp_release(wg_ctx *ctx)
{
  if (!ctx->pldp) return;
  PldpHost *p = static_cast<PldpHost *>(ctx->pldp);
  cudaFree(p->d); cudaFree(p->d_next);
  if (p->up) cudaStreamDestroy(p->up);
  if (p->down) cudaStreamDestroy(p->down);
  for (int c = 0; c < 4; ++c) { if (p->ev_up[c]) cudaEventDestroy(p->ev_up[c]); if (p->ev_k[c]) cudaEventDestroy(p->ev_k[c]); }
  if (p->ev0) cudaEventDestroy(p->ev0);
  for (void *b : p->buf) cudaFree(b);
  delete p;
  ctx->pldp = nullptr;
}

extern "C" {

int wg_pldp_set_constants(wg_ctx *ctx, int card_u, const double *iPu, const double *Px, const double *Pu)
{
  if (!ctx || !iPu || !Px || !Pu) return WG_ERR_INVALID;
  if (card_u != PLDP_N) return wg_fail(ctx, WG_ERR_INVALID, "PLDP kernels are built for CardU = 16 (QP_N of the reference)");
  wg_device_guard guard(ctx->device);
  PldpHost *p = pldp_of(ctx);
  const int N = PLDP_N;
  std::memcpy(p->h.iPu, iPu, sizeof p->h.iPu);
  std::memcpy(p->h.Px, Px, sizeof p->h.Px);
  std::memcpy(p->h.Pu, Pu, sizeof p->h.Pu);
  for (int k = 0; k < PLDP_N; ++k)
    for (int i = 0; i < PLDP_N; ++i) p->h.PuT[i * PLDP_N + k] = Pu[k * PLDP_N + i];
  // PLDPSolver::PrecomputeiPuPx, PLDPSolver.cpp:264-285 (same summation order)
  std::memset(p->h.iPuPx, 0, sizeof p->h.iPuPx);
  for (int i = 0; i < N; ++i)
    for (int j = 0; j < 3; ++j)
      for (int k = 0; k < N; ++k) {
        const double tmp = iPu[k * N + i] * Px[k * 3 + j];
        p->h.iPuPx[i * 6 + j] += tmp;
        p->h.iPuPx[(i + N) * 6 + j + 3] += tmp;
      }
  if (!p->d) WG_CUDA(ctx, cudaMalloc(&p->d, sizeof(PldpConsts)));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  WG_CUDA(ctx, cudaMemcpy(p->d, &p->h, sizeof(PldpConsts), cudaMemcpyHostToDevice));
  p->ready = true;
  return WG_OK;
}

}  // extern "C"

// Common body of wg_pldp_solve_batch (ranked == nullptr) and wg_pldp_solve_batch_ranked.
static int pldp_solve_impl(wg_ctx *ctx, int mem, int B, const wg_pldp_batch *pb, const PldpRanked *ranked)
{
  if (!ctx || !pb || B < 0) return WG_ERR_INVALID;
  PldpHost *p = pldp_of(ctx);
  if (!p->ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_pldp_set_constants not called");
  if (B == 0) return WG_OK;
  if (!pb->D || !pb->m || !pb->DPx || !pb->ZMPRef || !pb->XkYk || !pb->X) return WG_ERR_INVALID;
  if (!ranked && (!pb->DPu || pb->dpu_stride <= 0)) return WG_ERR_INVALID;
  if (ranked && (!ranked->a0 || !ranked->a1 || !ranked->ri || ranked->row_stride <= 0)) return WG_ERR_INVALID;
  if (pb->dpx_stride <= 0) return WG_ERR_INVALID;
  if (pb->similar && pb->similar_stride <= 0) return WG_ERR_INVALID;
  if (mem == WG_MEM_HOST) {
    // host-side batches are validated here (device-side ones by the kernel: status 7 / 6)
    for (int b = 0; b < B; ++b) {
      const long long m = pb->m[b];
      if (m < 0 || m > WG_PLDP_MAX_ROWS) return wg_fail(ctx, WG_ERR_INVALID, "m[b] outside [0, WG_PLDP_MAX_ROWS]");
      if (!ranked && pb->dpu_stride < (m + 1) * PLDP_U) return wg_fail(ctx, WG_ERR_INVALID, "dpu_stride < (m[b]+1)*32");
      if (ranked && ranked->row_stride < m) return wg_fail(ctx, WG_ERR_INVALID, "row_stride < m[b]");
      if (pb->dpx_stride < m) return wg_fail(ctx, WG_ERR_INVALID, "dpx_stride < m[b]");
      if (pb->similar) {
        if (pb->similar_stride < m) return wg_fail(ctx, WG_ERR_INVALID, "similar_stride < m[b]");
        const int32_t *sm = pb->similar + (size_t)b * pb->similar_stride;
        for (long long r = 0; r < m; ++r)
          if (sm[r] > 0 || r + sm[r] < 0)
            return wg_fail(ctx, WG_ERR_INVALID, "SimilarConstraints must be 0 or point backward inside the problem");
      }
      if (ranked) {
        const unsigned char *ri = ranked->ri + (size_t)b * ranked->row_stride;
        for (long long r = 0; r < m; ++r)
          if (ri[r] >= PLDP_N) return wg_fail(ctx, WG_ERR_INVALID, "previewed sample index of a row >= 16");
      }
    }
  }
  wg_device_guard guard(ctx->device);
  const int max_iter = pb->max_iterations > 0 ? pb->max_iterations : 4 * PLDP_KMAX;
  const double tol = 1e-8;   // m_tol, PLDPSolver.cpp:66
  wg_pldp_batch d = *pb;
  PldpRanked dr = ranked ? *ranked : PldpRanked{nullptr, nullptr, nullptr, 0};
  // launch over instances [b0, b0 + n) of the device-side batch `d`
  auto launch = [&](int b0, int n) -> int {
    int grid = (n + PLDP_WARPS - 1) / PLDP_WARPS;
    // Measured (16 384 cold-started problems, m ~ 68): constraint matrix staged in shared memory, 8 warps/SM: 4.57 ms; read
    // from L2 (the batch's matrices, 290 MB, stream through once per iteration of their own warp), 32 warps/SM at 64
    // registers: 3.53 ms, 2.85 ms with the work counter (24 warps/SM at 80 registers: 3.10 ms).  The solver is a chain of dependent FP64 operations: resident warps
    // hide more than shared memory saves.  WG_PLDP_STAGE=1 restores the staged variant.
    static const int stage = getenv("WG_PLDP_STAGE") ? atoi(getenv("WG_PLDP_STAGE")) : 0;
    int a_cap = (stage && !ranked) ? (int)((pb->dpu_stride + 1) & ~1LL) : 0;
    size_t smem = sizeof(double) * (size_t)a_cap * PLDP_WARPS;
    if (smem > 190 * 1024) { a_cap = 0; smem = 0; }
    WG_SMEM_ATTR(ctx, pldp_kernel<false>, smem);
    const int per_sm = smem ? (int)((227 * 1024) / (smem + (sizeof(PldpWarp) + 1100) * PLDP_WARPS + 1024)) : (ranked ? 4 : 8);
    if (grid > ctx->sm_count * (per_sm > 0 ? per_sm : 1)) grid = ctx->sm_count * (per_sm > 0 ? per_sm : 1);
    if (!p->d_next) WG_CUDA(ctx, cudaMalloc(&p->d_next, sizeof(int)));
    WG_CUDA(ctx, cudaMemsetAsync(p->d_next, 0, sizeof(int), ctx->stream));
    const size_t o = (size_t)b0;
    wg_prof_start(ctx, WG_K_PLDP);
    if (ranked) {
      const PldpRanked rk{dr.a0 + o * dr.row_stride, dr.a1 + o * dr.row_stride, dr.ri + o * dr.row_stride, dr.row_stride};
      pldp_kernel<true><<<grid, PLDP_WARPS * 32, 0, ctx->stream>>>(
          n, p->d, d.D + o * PLDP_U, d.m + o, nullptr, 0, d.DPx + o * d.dpx_stride, d.dpx_stride,
          d.ZMPRef + o * PLDP_U, d.XkYk + o * 6, d.X + o * PLDP_U, d.similar ? d.similar + o * d.similar_stride : nullptr,
          d.similar_stride, d.n_removed ? d.n_removed + o : nullptr, d.starting ? d.starting + o : nullptr,
          d.hot ? d.hot + o : nullptr, pb->hot_start, max_iter, tol, d.info ? d.info + o : nullptr, 0, p->d_next, rk);
    } else {
      pldp_kernel<false><<<grid, PLDP_WARPS * 32, smem, ctx->stream>>>(
          n, p->d, d.D + o * PLDP_U, d.m + o, d.DPu + o * d.dpu_stride, d.dpu_stride, d.DPx + o * d.dpx_stride, d.dpx_stride,
          d.ZMPRef + o * PLDP_U, d.XkYk + o * 6, d.X + o * PLDP_U, d.similar ? d.similar + o * d.similar_stride : nullptr,
          d.similar_stride, d.n_removed ? d.n_removed + o : nullptr, d.starting ? d.starting + o : nullptr,
          d.hot ? d.hot + o : nullptr, pb->hot_start, max_iter, tol, d.info ? d.info + o : nullptr, a_cap, p->d_next,
          PldpRanked{nullptr, nullptr, nullptr, 0});
    }
    wg_prof_stop(ctx);
    WG_LAUNCHED(ctx);
    return WG_OK;
  };
  if (mem == WG_MEM_DEVICE) return launch(0, B);
  if (mem != WG_MEM_HOST) return WG_ERR_INVALID;
  // ---- host buffers: stage, then up to 4 chunks pipelined over upload / kernel / download streams (the upload of the
  // constraint matrices, 17 KB per problem, is twice the kernel time)
  const size_t nb = (size_t)B;
  struct Item { int slot; const void *src; size_t per; const void **dst; };
  const Item in[] = {
      {0, pb->D, sizeof(double) * PLDP_U, (const void **)&d.D},
      {1, pb->m, sizeof(int), (const void **)&d.m},
      {2, ranked ? nullptr : pb->DPu, ranked ? 0 : sizeof(double) * (size_t)pb->dpu_stride, (const void **)&d.DPu},
      {10, ranked ? ranked->a0 : nullptr, ranked ? sizeof(double) * (size_t)ranked->row_stride : 0, (const void **)&dr.a0},
      {11, ranked ? ranked->a1 : nullptr, ranked ? sizeof(double) * (size_t)ranked->row_stride : 0, (const void **)&dr.a1},
      {12, ranked ? ranked->ri : nullptr, ranked ? sizeof(unsigned char) * (size_t)ranked->row_stride : 0, (const void **)&dr.ri},
      {3, pb->DPx, sizeof(double) * (size_t)pb->dpx_stride, (const void **)&d.DPx},
      {4, pb->ZMPRef, sizeof(double) * PLDP_U, (const void **)&d.ZMPRef},
      {5, pb->XkYk, sizeof(double) * 6, (const void **)&d.XkYk},
      {6, pb->similar, pb->similar ? sizeof(int) * (size_t)pb->similar_stride : 0, (const void **)&d.similar},
      {7, pb->n_removed, pb->n_removed ? sizeof(int) : 0, (const void **)&d.n_removed},
      {8, pb->starting, pb->starting ? sizeof(int) : 0, (const void **)&d.starting}};
  for (const Item &it : in) {
    if (!it.src) continue;
    int rc = wgi_grow_scratch(ctx, &p->buf[it.slot], &p->cap[it.slot], it.per * nb);
    if (rc != WG_OK) return rc;
    *it.dst = p->buf[it.slot];
  }
  // outputs + hot-start state share one allocation: X | info | hot
  const size_t ox = 0, oi = ox + sizeof(double) * PLDP_U * nb, oh = oi + sizeof(wg_pldp_info) * nb;
  int rc = wgi_grow_scratch(ctx, &p->buf[9], &p->cap[9], oh + sizeof(wg_pldp_state) * nb);
  if (rc != WG_OK) return rc;
  char *base = static_cast<char *>(p->buf[9]);
  d.X = reinterpret_cast<double *>(base + ox);
  d.info = pb->info ? reinterpret_cast<wg_pldp_info *>(base + oi) : nullptr;
  d.hot = pb->hot ? reinterpret_cast<wg_pldp_state *>(base + oh) : nullptr;
  if (!p->up) {
    WG_CUDA(ctx, cudaStreamCreateWithFlags(&p->up, cudaStreamNonBlocking));
    WG_CUDA(ctx, cudaStreamCreateWithFlags(&p->down, cudaStreamNonBlocking));
    for (int c = 0; c < 4; ++c) {
      WG_CUDA(ctx, cudaEventCreateWithFlags(&p->ev_up[c], cudaEventDisableTiming));
      WG_CUDA(ctx, cudaEventCreateWithFlags(&p->ev_k[c], cudaEventDisableTiming));
    }
    WG_CUDA(ctx, cudaEventCreateWithFlags(&p->ev0, cudaEventDisableTiming));
  }
  const int nch = std::max(1, std::min(4, B / 2048));
  WG_CUDA(ctx, cudaEventRecord(p->ev0, ctx->stream));
  WG_CUDA(ctx, cudaStreamWaitEvent(p->up, p->ev0, 0));
  for (int c = 0; c < nch; ++c) {
    const size_t b0 = nb * c / nch, b1 = nb * (c + 1) / nch, n = b1 - b0;
    for (const Item &it : in)
      if (it.src)
        WG_CUDA(ctx, cudaMemcpyAsync(static_cast<char *>(p->buf[it.slot]) + b0 * it.per, static_cast<const char *>(it.src) + b0 * it.per,
                                     it.per * n, cudaMemcpyHostToDevice, p->up));
    if (pb->hot) WG_CUDA(ctx, cudaMemcpyAsync(d.hot + b0, pb->hot + b0, sizeof(wg_pldp_state) * n, cudaMemcpyHostToDevice, p->up));
    WG_CUDA(ctx, cudaEventRecord(p->ev_up[c], p->up));
    WG_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, p->ev_up[c], 0));
    if ((rc = launch((int)b0, (int)n)) != WG_OK) return rc;
    WG_CUDA(ctx, cudaEventRecord(p->ev_k[c], ctx->stream));
    WG_CUDA(ctx, cudaStreamWaitEvent(p->down, p->ev_k[c], 0));
    WG_CUDA(ctx, cudaMemcpyAsync(pb->X + b0 * PLDP_U, d.X + b0 * PLDP_U, sizeof(double) * PLDP_U * n, cudaMemcpyDeviceToHost, p->down));
    if (pb->info) WG_CUDA(ctx, cudaMemcpyAsync(pb->info + b0, d.info + b0, sizeof(wg_pldp_info) * n, cudaMemcpyDeviceToHost, p->down));
    if (pb->hot) WG_CUDA(ctx, cudaMemcpyAsync(pb->hot + b0, d.hot + b0, sizeof(wg_pldp_state) * n, cudaMemcpyDeviceToHost, p->down));
  }
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  WG_CUDA(ctx, cudaStreamSynchronize(p->down));
  return WG_OK;
}

extern "C" {

int wg_pldp_solve_batch(wg_ctx *ctx, int mem, int B, const wg_pldp_batch *pb)
{
  return pldp_solve_impl(ctx, mem, B, pb, nullptr);
}

int wg_pldp_solve_batch_ranked(wg_ctx *ctx, int mem, int B, const wg_pldp_batch *pb, const double *A0, const double *A1,
                               const uint8_t *sample, long long row_stride)
{
  const PldpRanked rk{A0, A1, sample, row_stride};
  return pldp_solve_impl(ctx, mem, B, pb, &rk);
}

int wg_optcholesky_add_rows_batch(wg_ctx *ctx, int mem, int B, int mode, int nb_max, int card_u, int nb_constraints,
                                  const double *A, long long a_stride, const int *rows, int rows_stride, int k0, int k1,
                                  double *L, long long l_stride)
{
  if (!ctx || B < 0 || nb_max <= 0 || card_u <= 0 || k0 < 0 || k1 < k0 || k1 > nb_max || (mode != 0 && mode != 1))
    return WG_ERR_INVALID;
  if (B == 0 || k1 == k0) return WG_OK;
  if (!A || !rows || !L || rows_stride < k1) return WG_ERR_INVALID;   // UpdateCholeskyMatrix* returns -1 on null A / L
  wg_device_guard guard(ctx->device);
  PldpHost *p = pldp_of(ctx);
  const double *dA = A; const int *drows = rows; double *dL = L;
  const size_t nb = (size_t)B;
  if (mem == WG_MEM_HOST) {
    int rc;
    if ((rc = wgi_grow_scratch(ctx, &p->buf[2], &p->cap[2], sizeof(double) * (size_t)a_stride * nb)) != WG_OK) return rc;
    if ((rc = wgi_grow_scratch(ctx, &p->buf[6], &p->cap[6], sizeof(int) * (size_t)rows_stride * nb)) != WG_OK) return rc;
    if ((rc = wgi_grow_scratch(ctx, &p->buf[9], &p->cap[9], sizeof(double) * (size_t)l_stride * nb)) != WG_OK) return rc;
    WG_CUDA(ctx, cudaMemcpyAsync(p->buf[2], A, sizeof(double) * (size_t)a_stride * nb, cudaMemcpyHostToDevice, ctx->stream));
    WG_CUDA(ctx, cudaMemcpyAsync(p->buf[6], rows, sizeof(int) * (size_t)rows_stride * nb, cudaMemcpyHostToDevice, ctx->stream));
    WG_CUDA(ctx, cudaMemcpyAsync(p->buf[9], L, sizeof(double) * (size_t)l_stride * nb, cudaMemcpyHostToDevice, ctx->stream));
    dA = static_cast<const double *>(p->buf[2]); drows = static_cast<const int *>(p->buf[6]); dL = static_cast<double *>(p->buf[9]);
  } else if (mem != WG_MEM_DEVICE) {
    return WG_ERR_INVALID;
  }
  wg_prof_start(ctx, WG_K_OPTCHOL);
  optchol_kernel<<<grid_for(ctx, B, 4), 128, 0, ctx->stream>>>(B, mode, nb_max, card_u, nb_constraints, dA, a_stride, drows,
                                                               rows_stride, k0, k1, dL, l_stride);
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  if (mem == WG_MEM_HOST) {
    WG_CUDA(ctx, cudaMemcpyAsync(L, dL, sizeof(double) * (size_t)l_stride * nb, cudaMemcpyDeviceToHost, ctx->stream));
    WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return WG_OK;
}

int wg_optcholesky_full_batch(wg_ctx *ctx, int mem, int B, int n, const double *A, double *L, double *iL, int inv_size)
{
  if (!ctx || B < 0 || n <= 0 || !L || inv_size < 0 || inv_size > n) return WG_ERR_INVALID;
  if (B == 0) return WG_OK;
  wg_device_guard guard(ctx->device);
  PldpHost *p = pldp_of(ctx);
  const size_t bytes = sizeof(double) * (size_t)n * n * B;
  const double *dA = A; double *dL = L, *diL = iL;
  if (mem == WG_MEM_HOST) {
    int rc;
    if ((rc = wgi_grow_scratch(ctx, &p->buf[2], &p->cap[2], bytes)) != WG_OK) return rc;
    if ((rc = wgi_grow_scratch(ctx, &p->buf[9], &p->cap[9], 2 * bytes)) != WG_OK) return rc;
    if (A) WG_CUDA(ctx, cudaMemcpyAsync(p->buf[2], A, bytes, cudaMemcpyHostToDevice, ctx->stream));
    dL = static_cast<double *>(p->buf[9]); diL = iL ? dL + (size_t)n * n * B : nullptr;
    WG_CUDA(ctx, cudaMemcpyAsync(dL, L, bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (iL) WG_CUDA(ctx, cudaMemcpyAsync(diL, iL, bytes, cudaMemcpyHostToDevice, ctx->stream));
    dA = A ? static_cast<const double *>(p->buf[2]) : nullptr;
  } else if (mem != WG_MEM_DEVICE) {
    return WG_ERR_INVALID;
  }
  wg_prof_start(ctx, WG_K_OPTCHOL);
  optchol_full_kernel<<<grid_for(ctx, B, 4), 128, 0, ctx->stream>>>(B, n, dA, dL, diL, inv_size);
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  if (mem == WG_MEM_HOST) {
    WG_CUDA(ctx, cudaMemcpyAsync(L, dL, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (iL) WG_CUDA(ctx, cudaMemcpyAsync(iL, diL, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return WG_OK;
}

}  // extern "C"
