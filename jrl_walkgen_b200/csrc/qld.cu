// qld.cu - batched dense strictly convex QP in the ql0001_ calling convention, for sm_100a.
//
// Replaces ql0001_ / ql0002_ (src/Mathematics/qld.cpp:378-2090; Powell's ZQPCVX dual method) for the callers that hand it a
// general dense problem: ZMPQPWithConstraint (Wieber2006: n = 150, m <= 600, ZMPQPWithConstraint.cpp:1040-1046) and the QLD
// branches of ZMPConstrainedQPFastFormulation (:1297-1320):
//      min 1/2 x'Cx + d'x   s.t.  a_j'x + b_j  = 0 (j < me),  a_j'x + b_j >= 0 (me <= j < m),  xl <= x <= xu.
//
// B200-first formulation.  One CTA owns one QP (QPs are taken from a work counter).  The method is the dual active-set method
// of Goldfarb and Idnani in its RANGE-SPACE form, the same iteration herdt_qp.cuh runs in point space, written in the
// variables v = L'x of the Cholesky factor C = L L' (Hessian = identity there): with X = L^-1 at hand, a row a_p becomes
// y_p = X a_p, the Gram matrix of the active rows is Y'Y, and the only factorisation that changes during the solve is the
// inverse Cholesky factor T of Y'Y (grown by a row per added constraint, shrunk by Givens rotations per dropped one), next
// to the columns Y of the active rows.  A null-space / orthogonal-factor implementation (QLD, QuadProg) rotates an n x n
// matrix on every active-set change - a chain of n - q dependent Givens rotations; here an active-set change costs two
// triangular n x n products with X (coalesced, n independent dot products each) and O(q^2 + q n) work on T and Y, which is
// what a CTA does well, and it is cheapest exactly where the reference's problems live: few active rows (q << n).
// Working through the FACTOR matters: the Hessians of the reference's generators have condition numbers around 5e11
// (ZMPQPWithConstraint), and products with an explicit H^-1 lose cond(H) eps = 5e-5 of relative accuracy - measured: jerks off
// by 40 % on Wieber's QPs -, products with X lose sqrt(cond) eps = 7e-11.  X is formed once per Hessian (qld_factor_kernel;
// once per BATCH, in extended precision on the host, when the Hessian is shared, as in both reference generators whose C is
// constant) and lives in L2; per-iteration HBM traffic is the m x n constraint matrix.
// Pivoting follows QLD: the row with the largest violation normalised by its Euclidean norm (qld.cpp:1255-1331).
#include "wg_common.h"
#include <algorithm>
#include <vector>
#include <cmath>

namespace {

constexpr int QT = 256;              // threads per CTA
constexpr int QW = QT / 32;

// A Hessian shared by every QP of a batch, factorised once on the host.
struct SharedHessian {
  double *d_hinv = nullptr;          // [n*n] X = L^-1 in symmetric storage
  double *d_c = nullptr;             // [n*n] the Hessian itself, symmetric dense
  int n = 0;
  double boost = 0.0;                // the multiple of I QLD's rule added to it
};

struct QldState {
  SharedHessian caller;              // wg_qld_set_shared_hessian
  SharedHessian generator;           // the Wieber2006 generator's own (wgi_qld_set_generator_hessian): a caller's stays put
  // per-call scratch
  double *d_hinv = nullptr; size_t cap_hinv = 0;     // [B][n*n] per-QP inverses
  double *d_work = nullptr; size_t cap_work = 0;     // per-CTA Z (n x qcap) and T (packed)
  int *d_next = nullptr;
  int *d_fail = nullptr; size_t cap_fail = 0;
  // staging for WG_MEM_HOST
  void *d_stage = nullptr; size_t cap_stage = 0;
};

QldState *state_of(wg_ctx *ctx)
{
  if (!ctx->qld) ctx->qld = new QldState();
  return static_cast<QldState *>(ctx->qld);
}

__device__ __forceinline__ int tri(int i) { return (i * (i + 1)) >> 1; }

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// block-wide sum / argmin through a small shared scratch area (QW doubles + QW ints); every thread gets the result
__device__ double block_sum(double v, double *red)
{
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int w = 0; w < QW; ++w) t += red[w];
  return t;
}
__device__ void block_argmin(double &v, int &idx, double *red, int *redi)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (ov < v || (ov == v && oi < idx)) { v = ov; idx = oi; }
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = v; redi[threadIdx.x >> 5] = idx; }
  __syncthreads();
  v = red[0]; idx = redi[0];
#pragma unroll
  for (int w = 1; w < QW; ++w)
    if (red[w] < v || (red[w] == v && redi[w] < idx)) { v = red[w]; idx = redi[w]; }
}

// ---------------------------------------------------------------------------------------------------------------
// X = L^-1 (C = L L') of `count` symmetric positive definite matrices, one CTA each, in place in the n x n output block,
// stored SYMMETRICALLY: S[a][b] = X[max(a,b)][min(a,b)], so that both products the solver needs read it coalesced:
//   y = X a   : y_i = sum_{j <= i} S[j n + i] a_j          z = X'v : z_j = sum_{i >= j} S[i n + j] v_i.
// fail[b] = 1 when a pivot is not positive (QLD boosts the diagonal there, qld.cpp:809-854; this solver refuses).
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(QT)
qld_factor_kernel(int count, int n, int nmax, const double *__restrict__ C, long long c_stride, double *__restrict__ Sout,
                  int *__restrict__ fail, double vsmall)
{
  extern __shared__ double sm[];
  double *dinv = sm, *wv = sm + n;
  __shared__ double red[QW];
  __shared__ int redi[QW];
  __shared__ int bad, jfail;
  __shared__ double s_diag;
  const int t = threadIdx.x;
  for (int b = blockIdx.x; b < count; b += gridDim.x) {
    const double *Cb = C + (size_t)b * c_stride;
    double *W = Sout + (size_t)b * n * n;
    // QLD's first estimate of the multiple of I to add (qld.cpp:814-843; see qld_diagonal_boost)
    double dg = 0.0;
    if (vsmall > 0.0) {
      for (int e = t; e < n * n; e += QT) {
        const int i = e / n, j = e - i * n;
        const double gii = Cb[(size_t)i * nmax + i];
        if (j == i) dg = fmax(dg, vsmall - gii);
        else if (j > i) {
          const double gjj = Cb[(size_t)j * nmax + j], gij = Cb[(size_t)j * nmax + i];
          double ga = -fmin(gii, gjj);
          const double gb = fabs(gii - gjj) + fabs(gij);
          if (gb > 0.0) ga += gij * gij / gb;
          dg = fmax(dg, ga);
        }
      }
      int dummy = 0;
      double neg = -dg;
      block_argmin(neg, dummy, red, redi);
      dg = -neg;
    }
    bool boosted = dg > 0.0;
    if (t == 0) { bad = 0; s_diag = dg; }
    __syncthreads();
    for (int pass = 0; pass < 200; ++pass) {
      if (t == 0) { if (boosted) s_diag = 2.0 * s_diag; jfail = -1; }
      __syncthreads();
      const double diag = s_diag;
      for (int e = t; e < n * n; e += QT) {
        const int i = e / n, j = e - i * n;
        W[e] = (j <= i) ? Cb[(size_t)j * nmax + i] + (j == i ? diag : 0.0) : 0.0;      // lower triangle of the column-major C
      }
      __syncthreads();
      for (int j = 0; j < n; ++j) {
        if (t == 0) {
          const double p = W[j * n + j];
          if (vsmall > 0.0 ? (p < vsmall) : !(p > 0.0)) { jfail = j; }
          else { const double l = sqrt(p); W[j * n + j] = l; dinv[j] = 1.0 / l; }
        }
        __syncthreads();
        if (jfail >= 0) break;
        const double il = dinv[j];
        for (int i = j + 1 + t; i < n; i += QT) W[i * n + j] *= il;
        __syncthreads();
        // trailing update of the lower triangle: W[i][k] -= W[i][j] W[k][j], j < k <= i
        const int r = n - 1 - j;
        for (int e = t; e < r * r; e += QT) {
          const int ii = e / r, kk = e - ii * r;
          if (kk <= ii) {
            const int i = j + 1 + ii, k = j + 1 + kk;
            W[i * n + k] -= W[i * n + j] * W[k * n + j];
          }
        }
        __syncthreads();
      }
      if (jfail < 0) break;
      if (!(vsmall > 0.0)) {           // no QLD treatment asked for: refuse the Hessian
        if (t == 0) { bad = 1; }
        // finish with a harmless factor so that the kernel below reads defined memory
        for (int e = t; e < n * n; e += QT) { const int i = e / n, j = e - i * n; W[e] = (i == j) ? 1.0 : 0.0; }
        for (int i = t; i < n; i += QT) dinv[i] = 1.0;
        __syncthreads();
        break;
      }
      // qld.cpp:893-918: w solves R w = e_j-like with the part of the factor found so far; diag += vsmall - pivot / |w|^2
      if (t == 0) {
        const int j = jfail;
        const double temp = W[j * n + j];
        wv[j] = 1.0;
        double sumx = 1.0;
        for (int k = j - 1; k >= 0; --k) {
          double sum = 0.0;
          for (int i = k + 1; i <= j; ++i) sum -= W[i * n + k] * wv[i];     // R(k, i) = L(i, k)
          wv[k] = sum / W[k * n + k];
          sumx += wv[k] * wv[k];
        }
        s_diag = s_diag + vsmall - temp / sumx;
      }
      boosted = true;
      __syncthreads();
    }
    // X = L^-1, column c by forward substitution, written transposed into the strict upper triangle: X[i][c] at W[c][i]
    for (int c = t; c < n; c += QT) {
      for (int i = c + 1; i < n; ++i) {
        double s = W[i * n + c] * dinv[c];
        for (int k = c + 1; k < i; ++k) s = fma(W[i * n + k], W[c * n + k], s);
        W[c * n + i] = -s * dinv[i];
      }
    }
    __syncthreads();
    for (int e = t; e < n * n; e += QT) {
      const int i = e / n, j = e - i * n;
      if (j < i) W[e] = W[j * n + i]; else if (j == i) W[e] = dinv[i];
    }
    if (t == 0 && fail) fail[b] = bad;
    __syncthreads();
  }
}

// y = X a through the symmetric storage of X: y_i = sum_{j <= i} S[j n + i] a_j.  One thread per row, consecutive threads on
// consecutive addresses, 8 independent accumulators: the dependent FMA chain is n / 8 long and the n loads of a thread are
// independent of it.  (A warp per row with a shuffle reduction was measured slower: 19 dependent load + 5-round reductions per
// warp and product, 34 % of the kernel's samples.)
__device__ __forceinline__ void tri_lower_mv(const double *__restrict__ S, int n, const double *a, double *y, int t)
{
  for (int i = t; i < n; i += QT) {
    double s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const double *col = S + i;
    int j = 0;
    for (; j + 7 <= i; j += 8) {
#pragma unroll
      for (int k = 0; k < 8; ++k) s[k] = fma(col[(size_t)(j + k) * n], a[j + k], s[k]);
    }
    for (; j <= i; ++j) s[0] = fma(col[(size_t)j * n], a[j], s[0]);
    y[i] = ((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7]));
  }
}
// x = X'v: x_j = sum_{i >= j} X[i][j] v_i = sum_{i >= j} S[i n + j] v_i (same access pattern)
__device__ __forceinline__ void tri_upper_mv(const double *__restrict__ S, int n, const double *v, double *x, int t)
{
  for (int j = t; j < n; j += QT) {
    double s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const double *col = S + j;
    int i = j;
    for (; i + 7 < n; i += 8) {
#pragma unroll
      for (int k = 0; k < 8; ++k) s[k] = fma(col[(size_t)(i + k) * n], v[i + k], s[k]);
    }
    for (; i < n; ++i) s[0] = fma(col[(size_t)i * n], v[i], s[0]);
    x[j] = ((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7]));
  }
}
// dots[k] = Q_k . y for the q active rows: a warp takes four rows at a time (four independent load / reduce chains)
__device__ __forceinline__ void basis_dots(const double *__restrict__ Y, const int *slot, int q, int n, const double *y, double *dots,
                                           int warp, int lane)
{
  for (int k0 = 4 * warp; k0 < q; k0 += 4 * QW) {
    double s[4] = {0, 0, 0, 0};
    const double *qk[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) qk[c] = Y + (size_t)slot[min(k0 + c, q - 1)] * n;
    for (int j = lane; j < n; j += 32) {
      const double yj = y[j];
#pragma unroll
      for (int c = 0; c < 4; ++c) s[c] = fma(qk[c][j], yj, s[c]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int c = 0; c < 4; ++c) s[c] += __shfl_xor_sync(0xffffffffu, s[c], o);
    }
    if (lane == 0) {
#pragma unroll
      for (int c = 0; c < 4; ++c) if (k0 + c < q) dots[k0 + c] = s[c];
    }
  }
}
// part[w][r] = sum over the columns j of chunk w of A(r, j) * (x ? x[j] : A(r, j)): the m x n column-major constraint matrix is
// read once, consecutive lanes on consecutive rows (coalesced), 4 rows per lane in flight; the caller sums the QW partials.
__device__ __forceinline__ void rows_partial(const double *__restrict__ A, int mmax, int m, int n, const double *x, double *part,
                                             int pstride, int warp, int lane)
{
  constexpr int RPL = 8;                      // rows per lane in flight
  const int chunk = (n + QW - 1) / QW, j0 = warp * chunk, j1 = min(n, j0 + chunk);
  double *pw = part + (size_t)warp * pstride;
  for (int base = 0; base < m; base += 32 * RPL) {
    double s[RPL];
#pragma unroll
    for (int k = 0; k < RPL; ++k) s[k] = 0.0;
    for (int j = j0; j < j1; ++j) {
      const double *col = A + (size_t)j * mmax + base + lane;
      const double xj = x ? x[j] : 0.0;
#pragma unroll
      for (int k = 0; k < RPL; ++k) {
        const double a = (base + lane + 32 * k < m) ? col[32 * k] : 0.0;
        s[k] = fma(a, x ? xj : a, s[k]);
      }
    }
#pragma unroll
    for (int k = 0; k < RPL; ++k)
      if (base + lane + 32 * k < m) pw[base + lane + 32 * k] = s[k];
  }
}

struct QldArgs {
  int B, n, nmax, mmax, qcap;
  int pstride;                              // stride of the QW partial row sums in shared memory: >= mmax, and QW pstride >= 4N (RANKED)
  const int *m, *me;
  const double *C; long long c_stride;      // per-QP Hessians (refinement), or the shared one with stride 0
  const double *S; long long h_stride;      // X = L^-1 in symmetric storage; stride 0: shared
  const int *hfail;                         // per Hessian (index b, or 0 when shared), may be null
  const double *d;
  const double *A; long long a_stride;
  const double *b; long long b_stride;
  const double *xl, *xu;
  double *x;
  double *u; long long u_stride;
  int *ifail, *iterations;
  double *work; long long work_stride;      // per CTA
  int *next;
  // rank-structured rows (RANKED kernel): row r of QP b = (A0, A1) x row `samp` of the lower-triangular Toeplitz matrix uz
  const double *A0, *A1; const unsigned char *samp; long long row_stride;
  const double *uz; int N;
};

// ---------------------------------------------------------------------------------------------------------------
// The solver.  Shared memory: x, v, v0, ap, yp, yd [n each]; inrm [m + 2n]; u, g, w, r [qcap each]; W, slot [qcap ints];
// active flags [m + 2n bytes]; free-slot stack [qcap ints].  v = L'x is the iterate, x = X'v is refreshed after every step.
// ---------------------------------------------------------------------------------------------------------------
// RANKED: the m x n matrix is never read (nor materialised by the caller): element (r, k + N ax) = A_ax[r] uz[samp[r] - k],
// k <= samp[r].  The violation scan then works on the N "points" P_ax = Uz x_ax (two Toeplitz products out of shared memory) and
// costs two multiplications per row; the row handed to the factor is rebuilt from (A0, A1, samp).  Everything else is the
// dense kernel.  (Wieber2006: 360 KB of matrix per QP and active-set change no longer cross HBM.)
template <bool RANKED>
__global__ void __launch_bounds__(QT, 2)
qld_kernel(QldArgs P)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double red[QW];
  __shared__ int redi[QW];
  __shared__ int s_b;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int n = P.n, qcap = P.qcap, mmax = P.mmax, pstride = P.pstride;
  const bool bounds = (P.xl != nullptr) && (P.xu != nullptr);
  const int mtot_max = mmax + (bounds ? 2 * n : 0);
  double *x = reinterpret_cast<double *>(smem_raw);
  double *v = x + n, *v0 = v + n, *ap = v0 + n, *yp = ap + n, *yd = yp + n;
  double *inrm = yd + n;
  double *part = inrm + mtot_max;                                         // QW x pstride partial row sums
  double *u = part + (size_t)QW * pstride, *g = u + qcap, *w = g + qcap, *r = w + qcap;
  int *Wc = reinterpret_cast<int *>(r + qcap);
  int *slot = Wc + qcap, *freeslot = slot + qcap;
  signed char *sgn = reinterpret_cast<signed char *>(freeslot + qcap);   // sign of an active (equality) row
  unsigned char *act = reinterpret_cast<unsigned char *>(sgn + qcap);
  const int N = RANKED ? P.N : 0;
  double *pts = part, *uzs = part + 2 * N, *rn2 = part + 3 * N;          // RANKED: P_x, P_y [N each], uz [N], |uz row|^2 [N]
  double *Y = P.work + (size_t)blockIdx.x * P.work_stride;                // n x qcap, column `slot` at Y + slot * n
  double *T = Y + (size_t)n * qcap;                                       // packed lower triangle, row j at T + tri(j)
  const double INF = __longlong_as_double(0x7ff0000000000000LL);

  for (;;) {
    if (t == 0) s_b = atomicAdd(P.next, 1);
    __syncthreads();
    const int b = s_b;
    __syncthreads();
    if (b >= P.B) break;
    const int m = P.m[b], me = P.me ? P.me[b] : 0;
    const double *A = RANKED ? nullptr : P.A + (size_t)b * P.a_stride, *bv = P.b + (size_t)b * P.b_stride;
    const double *A0 = RANKED ? P.A0 + (size_t)b * P.row_stride : nullptr, *A1 = RANKED ? P.A1 + (size_t)b * P.row_stride : nullptr;
    const unsigned char *samp = RANKED ? P.samp + (size_t)b * P.row_stride : nullptr;
    const double *dv = P.d + (size_t)b * n;
    const double *S = P.S + (size_t)b * P.h_stride;
    const double *Cm = P.C ? P.C + (size_t)b * P.c_stride : nullptr;
    const double *xl = bounds ? P.xl + (size_t)b * n : nullptr, *xu = bounds ? P.xu + (size_t)b * n : nullptr;
    // neq: equality rows processed (added, or skipped as redundant); qeq: equality rows in the active set, positions 0..qeq-1
    int fail = 0, iters = 0, q = 0, neq = 0, qeq = 0;
    if (m < 0 || m > mmax || me < 0 || me > m) fail = 5;                  // QLD ifail 5: wrong dimensions
    if (!fail && P.hfail && P.hfail[P.h_stride ? b : 0]) fail = 2;
    const int mtot = fail ? 0 : m + (bounds ? 2 * n : 0);

    // ---- unconstrained optimum v0 = -X d, x = X'v0; row norms, flags
    for (int i = t; i < n; i += QT) ap[i] = dv[i];
    __syncthreads();
    tri_lower_mv(S, n, ap, v0, t);
    if (RANKED) {
      for (int i = t; i < N; i += QT) uzs[i] = P.uz[i];
      __syncthreads();
      for (int i = t; i < N; i += QT) { double a = 0.0; for (int k = 0; k <= i; ++k) a = fma(uzs[k], uzs[k], a); rn2[i] = a; }
    } else if (!fail) rows_partial(A, mmax, m, n, nullptr, part, pstride, warp, lane);
    __syncthreads();
    for (int i = t; i < n; i += QT) { v0[i] = -v0[i]; v[i] = v0[i]; }
    for (int rr = t; rr < mtot; rr += QT) {
      double s = 1.0;
      if (rr < m) {
        if (RANKED) s = (A0[rr] * A0[rr] + A1[rr] * A1[rr]) * rn2[min((int)samp[rr], N - 1)];
        else {
          s = 0.0;
#pragma unroll
          for (int wq = 0; wq < QW; ++wq) s += part[(size_t)wq * pstride + rr];
        }
      }
      // a zero row is scaled by 1, so that its violation is b itself: with b < 0 it is picked, found dependent on any active
      // set and reported as inconsistent (ifail 10 + j); with b >= 0 it is never violated
      inrm[rr] = s > 0.0 ? rsqrt(s) : 1.0;
      act[rr] = 0;
    }
    __syncthreads();
    tri_upper_mv(S, n, v, x, t);
    for (int k = t; k < qcap; k += QT) freeslot[k] = qcap - 1 - k;
    __syncthreads();
    int nfree = qcap;
    const int maxit = 40 * (mtot + n);
    bool done = fail != 0;

    while (!done) {
      // ---- the row to add: equalities first, in order; then the most violated inequality (normalised)
      int p; double sp; int sign = 1;
      double xn2 = 0.0;
      for (int i = t; i < n; i += QT) xn2 = fma(x[i], x[i], xn2);
      const double xnorm = sqrt(block_sum(xn2, red));
      if (neq < me) {
        p = neq;
        double s = 0.0;
        if (RANKED) {
          const int ip = min((int)samp[p], N - 1);
          for (int j = t; j <= ip; j += QT) s = fma(uzs[ip - j], A0[p] * x[j] + A1[p] * x[j + N], s);
        } else {
          for (int j = t; j < n; j += QT) s = fma(A[p + (size_t)j * mmax], x[j], s);
        }
        sp = block_sum(s, red) + bv[p];
        if (sp > 0.0) { sign = -1; sp = -sp; }
      } else {
        double best = INF; int bi = 0x7fffffff;
        if (RANKED) {
          // points P_ax[i] = sum_{k <= i} uz[i - k] x[ax N + k]: warp per (axis, sample)
          for (int e = t; e < 2 * N; e += QT) {
            const int ax = e >= N, i = ax ? e - N : e;
            const double *xa = x + ax * N;
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
            int k = 0;
            for (; k + 3 <= i; k += 4) {
              a0 = fma(uzs[i - k], xa[k], a0); a1 = fma(uzs[i - k - 1], xa[k + 1], a1);
              a2 = fma(uzs[i - k - 2], xa[k + 2], a2); a3 = fma(uzs[i - k - 3], xa[k + 3], a3);
            }
            for (; k <= i; ++k) a0 = fma(uzs[i - k], xa[k], a0);
            pts[e] = (a0 + a1) + (a2 + a3);
          }
        } else rows_partial(A, mmax, m, n, x, part, pstride, warp, lane);
        __syncthreads();
        for (int rr = t; rr < mtot; rr += QT) {
          if (act[rr] || rr < me) continue;          // equalities are all taken above
          double s, scale;
          if (rr < m) {
            if (RANKED) {
              const int ip = min((int)samp[rr], N - 1);
              s = A0[rr] * pts[ip] + A1[rr] * pts[N + ip];
            } else {
              s = 0.0;
#pragma unroll
              for (int wq = 0; wq < QW; ++wq) s += part[(size_t)wq * pstride + rr];
            }
            const double bb = bv[rr];
            s += bb;
            scale = fabs(bb) * inrm[rr] + xnorm;
          } else if (rr < m + n) {
            const int i = rr - m;
            s = x[i] - xl[i]; scale = fabs(xl[i]) + xnorm;
          } else {
            const int i = rr - m - n;
            s = xu[i] - x[i]; scale = fabs(xu[i]) + xnorm;
          }
          const double sv = s * inrm[rr];
          // converged rows: violation below 1e-11 of the row's own scale (distance units)
          if (sv < -1e-11 * (scale + 1e-300) && sv < best) { best = sv; bi = rr; }
        }
        block_argmin(best, bi, red, redi);
        if (bi == 0x7fffffff) break;             // no violated row left: optimal
        p = bi;
        sp = best / inrm[p];
      }
      // a_p into shared memory (bounds: +- unit vector)
      for (int j = t; j < n; j += QT) {
        double a;
        if (p < m) {
          if (RANKED) {
            const int ip = min((int)samp[p], N - 1), ax = j >= N, k = ax ? j - N : j;
            a = (k <= ip) ? sign * (ax ? A1[p] : A0[p]) * uzs[ip - k] : 0.0;
          } else a = sign * A[p + (size_t)j * mmax];
        }
        else if (p < m + n) a = (j == p - m) ? 1.0 : 0.0;
        else a = (j == p - m - n) ? -1.0 : 0.0;
        ap[j] = a;
      }
      __syncthreads();
      // y_p = X a_p, M_pp = |y_p|^2
      tri_lower_mv(S, n, ap, yp, t);
      __syncthreads();
      double mpp = 0.0;
      for (int i = t; i < n; i += QT) mpp = fma(yp[i], yp[i], mpp);
      const double Mpp = block_sum(mpp, red);
      double up = 0.0;
      bool added = false;
      while (!added && !done) {
        if (++iters > maxit) { fail = 1; done = true; break; }
        // w = Q'y_p (warp per active row): the coordinates of y_p in the orthonormal basis Q of the active rows (Y = Q R)
        basis_dots(Y, slot, q, n, yp, w, warp, lane);
        __syncthreads();
        // yd = y_p - Q w: the part of y_p orthogonal to the active rows, with one re-orthogonalisation pass (Gram-Schmidt
        // twice: |yd| stays accurate when y_p lies almost inside the span, which is the rule for adjacent CoP rows)
        for (int i = t; i < n; i += QT) {
          double s0 = yp[i], s1 = 0.0, s2 = 0.0, s3 = 0.0;
          int k = 0;
          for (; k + 3 < q; k += 4) {
            s0 = fma(-w[k], Y[(size_t)slot[k] * n + i], s0); s1 = fma(-w[k + 1], Y[(size_t)slot[k + 1] * n + i], s1);
            s2 = fma(-w[k + 2], Y[(size_t)slot[k + 2] * n + i], s2); s3 = fma(-w[k + 3], Y[(size_t)slot[k + 3] * n + i], s3);
          }
          for (; k < q; ++k) s0 = fma(-w[k], Y[(size_t)slot[k] * n + i], s0);
          yd[i] = (s0 + s1) + (s2 + s3);
        }
        __syncthreads();
        basis_dots(Y, slot, q, n, yd, g, warp, lane);
        __syncthreads();
        double dsq = 0.0;
        for (int i = t; i < n; i += QT) {
          double s0 = yd[i], s1 = 0.0, s2 = 0.0, s3 = 0.0;
          int k = 0;
          for (; k + 3 < q; k += 4) {
            s0 = fma(-g[k], Y[(size_t)slot[k] * n + i], s0); s1 = fma(-g[k + 1], Y[(size_t)slot[k + 1] * n + i], s1);
            s2 = fma(-g[k + 2], Y[(size_t)slot[k + 2] * n + i], s2); s3 = fma(-g[k + 3], Y[(size_t)slot[k + 3] * n + i], s3);
          }
          for (; k < q; ++k) s0 = fma(-g[k], Y[(size_t)slot[k] * n + i], s0);
          const double s = (s0 + s1) + (s2 + s3);
          yd[i] = s;
          dsq = fma(s, s, dsq);
        }
        for (int k = t; k < q; k += QT) w[k] += g[k];
        const double delta = block_sum(dsq, red);             // = a_p' (H^-1 - H^-1 N (N'H^-1 N)^-1 N'H^-1) a_p
        // r = R^-1 w = T'w: the dual step direction
        double t1 = INF; int l = 0x7fffffff;
        for (int j = t; j < q; j += QT) {
          double s = 0.0;
          for (int rr = j; rr < q; ++rr) s = fma(T[tri(rr) + j], w[rr], s);
          r[j] = s;
          if (s > 0.0 && j >= qeq) {                        // equality rows are never dropped
            const double tj = u[j] / s;
            if (tj < t1) { t1 = tj; l = j; }
          }
        }
        block_argmin(t1, l, red, redi);
        const bool dependent = !(delta > 1e-22 * Mpp);
        const double t2 = dependent ? INF : -sp / delta;
        const double tt = fmin(t1, t2);
        if (!(tt < INF)) {
          // the row is a combination of the active rows and cannot be satisfied
          if (neq < me && fabs(sp) * inrm[p] <= 1e-9 * (fabs(bv[p]) * inrm[p] + xnorm + 1e-300)) { act[p] = 0; ++neq; added = true; break; }   // redundant equality
          fail = 10 + p + 1; done = true; break;            // QLD: ifail > 10, constraint ifail - 10 inconsistent
        }
        if (!dependent) {
          // step along yd in the factor's variables, x = X'v
          for (int i = t; i < n; i += QT) v[i] = fma(tt, yd[i], v[i]);
          __syncthreads();
          tri_upper_mv(S, n, v, x, t);
          sp += tt * delta;
        }
        for (int j = t; j < q; j += QT) u[j] = fma(-tt, r[j], u[j]);
        up += tt;
        __syncthreads();
        if (t2 <= t1) {
          // full step: row p becomes active; new basis vector yd / |yd|, new row of T = R^-T
          if (q >= qcap || nfree <= 0) { fail = 3; done = true; break; }
          const double idd = rsqrt(delta);
          for (int j = t; j < q; j += QT) T[tri(q) + j] = -r[j] * idd;
          const int sl = freeslot[nfree - 1];
          for (int i = t; i < n; i += QT) Y[(size_t)sl * n + i] = yd[i] * idd;
          if (t == 0) { T[tri(q) + q] = idd; Wc[q] = p; slot[q] = sl; u[q] = up; sgn[q] = (signed char)sign; act[p] = 1; }
          --nfree; ++q;
          if (neq < me) { ++neq; ++qeq; }
          added = true;
          __syncthreads();
          break;
        }
        // partial step: multiplier l reached zero -> drop row l.  Warp 0 rotates rows (l, rr), rr > l, of T so that column l
        // vanishes below row l and deletes row / column l (herdt_qp.cuh drop_row); the same rotations, kept in g (cosines)
        // and w (sines), are then applied to the basis vectors Q_l, Q_rr by all threads (Q -> Q G').
        if (warp == 0) {
          for (int j = lane; j < q; j += 32) yd[j] = (j <= l) ? T[tri(l) + j] : 0.0;     // yd: rotating copy of row l (q <= n)
          __syncwarp();
          for (int rr = l + 1; rr < q; ++rr) {
            const double *Tr = T + tri(rr);
            const double p1 = yd[l], p2 = Tr[l];
            const double ih = rsqrt(p1 * p1 + p2 * p2);
            const double c_ = p1 * ih, s_ = p2 * ih;
            __syncwarp();
            double *Tn = T + tri(rr - 1);
            for (int j = lane; j <= rr; j += 32) {
              const double x1 = yd[j], x2 = Tr[j];
              yd[j] = c_ * x1 + s_ * x2;
              const double nr = c_ * x2 - s_ * x1;
              if (j < l) Tn[j] = nr;
              else if (j > l) Tn[j - 1] = nr;
            }
            if (lane == 0) { g[rr] = c_; w[rr] = s_; }
            __syncwarp();
          }
        }
        __syncthreads();
        {
          const int sl_l = slot[l];
          for (int i = t; i < n; i += QT) {
            double ql = Y[(size_t)sl_l * n + i];
            for (int rr = l + 1; rr < q; ++rr) {
              double *qr = Y + (size_t)slot[rr] * n + i;
              const double c_ = g[rr], s_ = w[rr], b2 = *qr;
              *qr = c_ * b2 - s_ * ql;
              ql = c_ * ql + s_ * b2;
            }
          }
        }
        __syncthreads();
        if (warp == 0) {
          if (lane == 0) { act[Wc[l]] = 0; freeslot[nfree] = slot[l]; }
          __syncwarp();
          for (int base = l; base < q - 1; base += 32) {
            const int j = base + lane;
            const bool mv = j < q - 1;
            const int Wn = mv ? Wc[j + 1] : 0, sn = mv ? slot[j + 1] : 0;
            const double un = mv ? u[j + 1] : 0.0;
            const signed char gn = mv ? sgn[j + 1] : (signed char)1;
            __syncwarp();
            if (mv) { Wc[j] = Wn; slot[j] = sn; u[j] = un; sgn[j] = gn; }
            __syncwarp();
          }
        }
        ++nfree; --q;
        __syncthreads();
        if (dependent) continue;   // sp unchanged by a pure dual step
        // recompute the violation of p on the moved point
        double s = 0.0;
        for (int j = t; j < n; j += QT) s = fma(ap[j], x[j], s);
        s = block_sum(s, red);
        if (p < m) sp = s + sign * bv[p];
        else if (p < m + n) sp = s - xl[p - m];
        else sp = s + xu[p - m - n];
      }
    }

    // (No Newton step on the stationarity residual here: H^-1 res leaves the active rows, and with cond(H) = 5e11 its rounding
    // noise moved vertex solutions of Wieber's QPs 2e-7 outside their active rows - measured.  v is kept by projected steps,
    // each orthogonal to every active row, so the active rows hold to rounding and x = X'v needs no repair.)
    // ---- results: x, multipliers in QLD's layout (m rows, n lower bounds, n upper bounds; qld.cpp:520-536)
    if (fail) {
      __syncthreads();
      tri_upper_mv(S, n, v0, x, t);
      __syncthreads();
    }
    for (int i = t; i < n; i += QT) P.x[(size_t)b * n + i] = x[i];
    if (P.u) {
      double *uo = P.u + (size_t)b * P.u_stride;
      for (int k = t; k < P.u_stride; k += QT) uo[k] = 0.0;             // the whole row: no stale values past m + 2n
      __syncthreads();
      if (!fail)
        for (int k = t; k < q; k += QT) {
          const int pk = Wc[k];
          const int dst = pk < m ? pk : (bounds ? pk : -1);
          if (dst >= 0 && dst < P.u_stride) uo[dst] = sgn[k] * u[k];
        }
    }
    if (t == 0) {
      P.ifail[b] = fail;
      if (P.iterations) P.iterations[b] = iters;
    }
    __syncthreads();
  }
}

size_t qld_smem_bytes(int n, int mmax, int pstride, int qcap, bool bounds)
{
  const size_t mtot = (size_t)mmax + (bounds ? 2 * (size_t)n : 0);
  size_t s = sizeof(double) * (6 * (size_t)n + mtot + (size_t)QW * pstride + 4 * (size_t)qcap) + sizeof(int) * 3 * (size_t)qcap + qcap + mtot;
  return (s + 15) & ~(size_t)15;
}

int hinv_launch(wg_ctx *ctx, int count, int n, int nmax, const double *d_C, long long c_stride, double *d_hinv, int *d_fail,
                double vsmall)
{
  const int blocks = std::max(1, std::min(count, ctx->sm_count * 2));
  qld_factor_kernel<<<blocks, QT, sizeof(double) * 2 * n, ctx->stream>>>(count, n, nmax, d_C, c_stride, d_hinv, d_fail, vsmall);
  WG_LAUNCHED(ctx);
  return WG_OK;
}

}  // namespace

void wg_qld_release(wg_ctx *ctx)
{
  if (!ctx->qld) return;
  QldState *st = static_cast<QldState *>(ctx->qld);
  for (SharedHessian *h : {&st->caller, &st->generator}) { cudaFree(h->d_hinv); cudaFree(h->d_c); }
  cudaFree(st->d_hinv); cudaFree(st->d_work); cudaFree(st->d_next);
  cudaFree(st->d_fail); cudaFree(st->d_stage);
  delete st;
  ctx->qld = nullptr;
}

// QLD does not factorise the Hessian it is given but G + diag I (ql0002_, qld.cpp:809-918, lql = true): diag starts as
// twice the largest of (vsmall - g_ii) and of the 2 x 2 minor bounds -min(g_ii, g_jj) + g_ij^2 / (|g_ii - g_jj| + |g_ij|);
// whenever a Cholesky pivot then falls below vsmall, diag grows by vsmall - pivot / |w|^2 (w: the direction of smallest
// curvature found so far), is DOUBLED, and the factorisation restarts.  vsmall is the `eps` the caller hands to ql0001_
// (1e-8 in every call of the reference).  For the reference's generators this matters: their Hessians have eigenvalues down
// to 2e-9, QLD regularises them, and its solutions differ from the exact minimiser by 40 % in the flat directions.  This
// function restates that rule in QLD's operation order and returns the multiple of I that QLD adds (0: none).
static double qld_diagonal_boost(int n, int nmax, const double *C, double vsmall)
{
  if (!(vsmall > 0.0)) return 0.0;
  auto g = [&](int i, int j) { return C[(size_t)j * nmax + i]; };   // symmetric
  std::vector<double> gd(n);
  double diag = 0.0;
  for (int i = 0; i < n; ++i) {
    gd[i] = g(i, i);
    diag = std::max(diag, vsmall - gd[i]);
    for (int j = i + 1; j < n; ++j) {
      double ga = -std::min(gd[i], g(j, j));
      const double gb = std::fabs(gd[i] - g(j, j)) + std::fabs(g(i, j));
      if (gb > 0.0) ga += g(i, j) * g(i, j) / gb;
      diag = std::max(diag, ga);
    }
  }
  if (!(diag > 0.0)) diag = 0.0;
  std::vector<double> R((size_t)n * n, 0.0), w(n);     // R upper triangular, R(i, j) at i * n + j
  bool boosted = diag > 0.0;
  for (int pass = 0; pass < 200; ++pass) {
    if (boosted) diag = 2.0 * diag;                    // L70: diag = diagr * diag
    boosted = false;
    int jfail = -1; double temp = 0.0;
    for (int j = 0; j < n && jfail < 0; ++j) {
      for (int i = 0; i <= j; ++i) {
        temp = (i == j) ? gd[i] + diag : g(i, j);
        for (int k = 0; k < i; ++k) temp -= R[(size_t)k * n + i] * R[(size_t)k * n + j];
        if (i < j) R[(size_t)i * n + j] = temp / R[(size_t)i * n + i];
      }
      if (temp < vsmall) { jfail = j; break; }
      R[(size_t)j * n + j] = std::sqrt(temp);
    }
    if (jfail < 0) return diag;
    // L140-L160: w solves R(0..j-1, 0..j-1) w = -R(0..j-1, j), w_j = 1
    const int j = jfail;
    w[j] = 1.0;
    double sumx = 1.0;
    for (int k = j - 1; k >= 0; --k) {
      double sum = 0.0;
      for (int i = k + 1; i <= j; ++i) sum -= R[(size_t)k * n + i] * w[i];
      w[k] = sum / R[(size_t)k * n + k];
      sumx += w[k] * w[k];
    }
    diag = diag + vsmall - temp / sumx;
    boosted = true;
  }
  return diag;
}

// Factorise C (+ QLD's boost) into slot h.  The slot keeps its previous Hessian when C is refused.
static int install_shared_hessian(wg_ctx *ctx, SharedHessian &h, int n, int nmax, const double *C_in, double eps)
{
  if (!ctx || n <= 0 || n > WG_QLD_MAX_N || nmax < n || !C_in) return WG_ERR_INVALID;
  wg_device_guard guard(ctx->device);
  const double boost = qld_diagonal_boost(n, nmax, C_in, eps);
  std::vector<double> Cb(C_in, C_in + (size_t)nmax * n);
  for (int i = 0; i < n; ++i) Cb[(size_t)i * nmax + i] += boost;
  const double *C = Cb.data();
  // the inverse in extended precision on the host: once per Hessian, and the generators' Hessians (sums of products of
  // integrator matrices over 75 samples) are badly conditioned
  typedef long double LD;
  std::vector<LD> L((size_t)n * n, 0), X((size_t)n * n, 0);
  for (int j = 0; j < n; ++j) {
    LD p = C[(size_t)j * nmax + j];
    for (int k = 0; k < j; ++k) p -= L[(size_t)j * n + k] * L[(size_t)j * n + k];
    if (!(p > 0)) return wg_fail(ctx, WG_ERR_INVALID, "shared Hessian: C is not positive definite");
    const LD l = sqrtl(p);
    L[(size_t)j * n + j] = l;
    for (int i = j + 1; i < n; ++i) {
      LD v = C[(size_t)j * nmax + i];
      for (int k = 0; k < j; ++k) v -= L[(size_t)i * n + k] * L[(size_t)j * n + k];
      L[(size_t)i * n + j] = v / l;
    }
  }
  for (int c = 0; c < n; ++c) {          // X = L^-1
    X[(size_t)c * n + c] = 1 / L[(size_t)c * n + c];
    for (int i = c + 1; i < n; ++i) {
      LD s = 0;
      for (int k = c; k < i; ++k) s += L[(size_t)i * n + k] * X[(size_t)k * n + c];
      X[(size_t)i * n + c] = -s / L[(size_t)i * n + i];
    }
  }
  std::vector<double> H((size_t)n * n), Cs((size_t)n * n);     // H: X in symmetric storage (see qld_factor_kernel)
  for (int a = 0; a < n; ++a)
    for (int b = 0; b <= a; ++b) {
      H[(size_t)a * n + b] = H[(size_t)b * n + a] = (double)X[(size_t)a * n + b];
      Cs[(size_t)a * n + b] = Cs[(size_t)b * n + a] = C[(size_t)b * nmax + a];
    }
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (h.n != n) {
    cudaFree(h.d_hinv); cudaFree(h.d_c);
    h.d_hinv = h.d_c = nullptr; h.n = 0;
    WG_CUDA(ctx, cudaMalloc(&h.d_hinv, sizeof(double) * n * n));
    WG_CUDA(ctx, cudaMalloc(&h.d_c, sizeof(double) * n * n));
    h.n = n;
  }
  WG_CUDA(ctx, cudaMemcpy(h.d_hinv, H.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice));
  WG_CUDA(ctx, cudaMemcpy(h.d_c, Cs.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice));
  h.boost = boost;
  return WG_OK;
}

extern "C" {

int wg_qld_set_shared_hessian(wg_ctx *ctx, int n, int nmax, const double *C, double eps)
{
  return ctx ? install_shared_hessian(ctx, state_of(ctx)->caller, n, nmax, C, eps) : WG_ERR_INVALID;
}

int wgi_qld_set_generator_hessian(wg_ctx *ctx, int n, int nmax, const double *C, double eps)
{
  return ctx ? install_shared_hessian(ctx, state_of(ctx)->generator, n, nmax, C, eps) : WG_ERR_INVALID;
}

double wg_qld_diagonal_boost(int n, int nmax, const double *C, double eps)
{
  if (n <= 0 || nmax < n || !C) return 0.0;
  return qld_diagonal_boost(n, nmax, C, eps);
}

double wg_qld_shared_boost(wg_ctx *ctx) { return ctx && ctx->qld ? static_cast<QldState *>(ctx->qld)->caller.boost : 0.0; }

struct RankedRows { const double *A0, *A1; const unsigned char *samp; long long row_stride; const double *uz; int N; };

// generator: shared_hessian = 1 means the generator's Hessian (wgi_qld_set_generator_hessian), not the caller's
static int qld_solve_impl(wg_ctx *ctx, int mem, int B, const wg_qld_batch *q, const RankedRows *rk, bool generator)
{
  if (!ctx || !q || B < 0) return WG_ERR_INVALID;
  if (B == 0) return WG_OK;
  const int n = q->n, nmax = q->nmax, mmax = q->mmax;
  if (n <= 0 || n > WG_QLD_MAX_N || mmax < 0 || mmax > WG_QLD_MAX_M || !q->m || !q->d || !q->x || !q->ifail ||
      (mmax > 0 && ((!rk && !q->A) || !q->b)) || (!q->shared_hessian && (!q->C || nmax < n)) || ((q->xl == nullptr) != (q->xu == nullptr)))
    return WG_ERR_INVALID;
  if ((!rk && q->a_stride < (long long)mmax * n) || q->b_stride < mmax || (q->u && q->u_stride < mmax)) return WG_ERR_INVALID;
  if (rk && (mem != WG_MEM_DEVICE || rk->N * 2 != n || !rk->A0 || !rk->A1 || !rk->samp || !rk->uz || rk->row_stride < mmax || rk->N > 255))
    return WG_ERR_INVALID;
  wg_device_guard guard(ctx->device);
  QldState *st = state_of(ctx);
  const SharedHessian &sh = generator ? st->generator : st->caller;
  if (q->shared_hessian && (sh.n != n || !sh.d_hinv))
    return wg_fail(ctx, WG_ERR_NOT_READY, "wg_qld_set_shared_hessian not called for this n");
  const bool bounds = q->xl != nullptr;
  const size_t nb = (size_t)B;
  int rc;
  wg_qld_batch d = *q;       // device view of the batch
  std::vector<std::pair<void *, std::pair<const void *, size_t>>> downloads;
  if (mem == WG_MEM_HOST) {
    // one staging block: every array of the batch, uploaded; results downloaded after the launch
    const size_t szC = q->shared_hessian ? 0 : sizeof(double) * nb * nmax * n;
    const size_t sz_m = sizeof(int) * nb, sz_d = sizeof(double) * nb * n, szA = sizeof(double) * nb * q->a_stride,
                 szb = sizeof(double) * nb * q->b_stride, szu = q->u ? sizeof(double) * nb * q->u_stride : 0;
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    size_t off = 0;
    const size_t o_m = off; off += al(sz_m);
    const size_t o_me = off; off += q->me ? al(sz_m) : 0;
    const size_t o_C = off; off += al(szC);
    const size_t o_d = off; off += al(sz_d);
    const size_t o_A = off; off += al(szA);
    const size_t o_b = off; off += al(szb);
    const size_t o_xl = off; off += bounds ? al(sz_d) : 0;
    const size_t o_xu = off; off += bounds ? al(sz_d) : 0;
    const size_t o_x = off; off += al(sz_d);
    const size_t o_u = off; off += al(szu);
    const size_t o_f = off; off += al(sz_m);
    const size_t o_it = off; off += al(sz_m);
    if ((rc = wgi_grow_scratch(ctx, &st->d_stage, &st->cap_stage, off)) != WG_OK) return rc;
    char *base = static_cast<char *>(st->d_stage);
    auto up = [&](size_t o, const void *src, size_t bytes) -> cudaError_t {
      return bytes ? cudaMemcpyAsync(base + o, src, bytes, cudaMemcpyHostToDevice, ctx->stream) : cudaSuccess;
    };
    WG_CUDA(ctx, up(o_m, q->m, sz_m));
    if (q->me) WG_CUDA(ctx, up(o_me, q->me, sz_m));
    WG_CUDA(ctx, up(o_C, q->C, szC));
    WG_CUDA(ctx, up(o_d, q->d, sz_d));
    WG_CUDA(ctx, up(o_A, q->A, szA));
    WG_CUDA(ctx, up(o_b, q->b, szb));
    if (bounds) { WG_CUDA(ctx, up(o_xl, q->xl, sz_d)); WG_CUDA(ctx, up(o_xu, q->xu, sz_d)); }
    d.m = reinterpret_cast<const int *>(base + o_m);
    d.me = q->me ? reinterpret_cast<const int *>(base + o_me) : nullptr;
    d.C = szC ? reinterpret_cast<const double *>(base + o_C) : nullptr;
    d.d = reinterpret_cast<const double *>(base + o_d);
    d.A = reinterpret_cast<const double *>(base + o_A);
    d.b = reinterpret_cast<const double *>(base + o_b);
    d.xl = bounds ? reinterpret_cast<const double *>(base + o_xl) : nullptr;
    d.xu = bounds ? reinterpret_cast<const double *>(base + o_xu) : nullptr;
    d.x = reinterpret_cast<double *>(base + o_x);
    d.u = q->u ? reinterpret_cast<double *>(base + o_u) : nullptr;
    d.ifail = reinterpret_cast<int *>(base + o_f);
    d.iterations = q->iterations ? reinterpret_cast<int *>(base + o_it) : nullptr;
    downloads.push_back({q->x, {d.x, sz_d}});
    if (q->u) downloads.push_back({q->u, {d.u, szu}});
    downloads.push_back({q->ifail, {d.ifail, sz_m}});
    if (q->iterations) downloads.push_back({q->iterations, {d.iterations, sz_m}});
  } else if (mem != WG_MEM_DEVICE) return WG_ERR_INVALID;

  QldArgs a;
  a.B = B; a.n = n; a.nmax = q->shared_hessian ? n : nmax; a.mmax = mmax;
  a.qcap = std::min(n + (bounds ? 0 : 0), WG_QLD_MAX_N);
  a.m = d.m; a.me = d.me;
  a.d = d.d; a.A = d.A; a.a_stride = q->a_stride; a.b = d.b; a.b_stride = q->b_stride;
  a.xl = d.xl; a.xu = d.xu; a.x = d.x; a.u = d.u; a.u_stride = q->u_stride; a.ifail = d.ifail; a.iterations = d.iterations;
  if (q->shared_hessian) {
    a.S = sh.d_hinv; a.h_stride = 0; a.hfail = nullptr;
    a.C = sh.d_c; a.c_stride = 0;
  } else {
    if ((rc = wgi_grow_scratch(ctx, reinterpret_cast<void **>(&st->d_hinv), &st->cap_hinv, sizeof(double) * nb * n * n)) != WG_OK) return rc;
    if ((rc = wgi_grow_scratch(ctx, reinterpret_cast<void **>(&st->d_fail), &st->cap_fail, sizeof(int) * nb)) != WG_OK) return rc;
    if ((rc = hinv_launch(ctx, B, n, nmax, d.C, (long long)nmax * n, st->d_hinv, st->d_fail, q->eps)) != WG_OK) return rc;
    a.S = st->d_hinv; a.h_stride = (long long)n * n; a.hfail = st->d_fail;
    a.C = d.C; a.c_stride = (long long)nmax * n;
  }
  a.A0 = a.A1 = nullptr; a.samp = nullptr; a.row_stride = 0; a.uz = nullptr; a.N = 0;
  if (rk) { a.A0 = rk->A0; a.A1 = rk->A1; a.samp = rk->samp; a.row_stride = rk->row_stride; a.uz = rk->uz; a.N = rk->N; }
  // the partial row sums are also the ranked kernel's 4N doubles of points, uz and row norms: the multipliers start after both
  a.pstride = std::max(mmax, rk ? (4 * rk->N + QW - 1) / QW : 0);
  const size_t smem = qld_smem_bytes(n, mmax, a.pstride, a.qcap, bounds);
  if (smem > 200 * 1024) return wg_fail(ctx, WG_ERR_INVALID, "wg_qld_solve_batch: problem too large for shared memory");
  if (rk) WG_SMEM_ATTR(ctx, qld_kernel<true>, smem);
  else WG_SMEM_ATTR(ctx, qld_kernel<false>, smem);
  int per_sm = (int)std::min<size_t>(2, (220 * 1024) / (smem + 1024));
  if (per_sm < 1) per_sm = 1;
  const int blocks = std::max(1, std::min(B, ctx->sm_count * per_sm));
  a.work_stride = (long long)n * a.qcap + (long long)a.qcap * (a.qcap + 1) / 2;
  if ((rc = wgi_grow_scratch(ctx, reinterpret_cast<void **>(&st->d_work), &st->cap_work,
                             sizeof(double) * (size_t)blocks * a.work_stride)) != WG_OK)
    return rc;
  a.work = st->d_work;
  if (!st->d_next) WG_CUDA(ctx, cudaMalloc(&st->d_next, sizeof(int)));
  a.next = st->d_next;
  WG_CUDA(ctx, cudaMemsetAsync(st->d_next, 0, sizeof(int), ctx->stream));
  wg_prof_start(ctx, WG_K_QLD);
  if (rk) qld_kernel<true><<<blocks, QT, smem, ctx->stream>>>(a);
  else qld_kernel<false><<<blocks, QT, smem, ctx->stream>>>(a);
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  for (auto &dl : downloads)
    WG_CUDA(ctx, cudaMemcpyAsync(dl.first, dl.second.first, dl.second.second, cudaMemcpyDeviceToHost, ctx->stream));
  if (mem == WG_MEM_HOST) WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return WG_OK;
}

int wg_qld_solve_batch(wg_ctx *ctx, int mem, int B, const wg_qld_batch *q) { return qld_solve_impl(ctx, mem, B, q, nullptr, false); }

int wg_qld_solve_batch_ranked(wg_ctx *ctx, int mem, int B, const wg_qld_batch *q, const double *A0, const double *A1,
                              const unsigned char *sample, long long row_stride, const double *uz_dev, int N)
{
  RankedRows rk = {A0, A1, sample, row_stride, uz_dev, N};
  return qld_solve_impl(ctx, mem, B, q, &rk, false);
}

int wgi_qld_solve_generator(wg_ctx *ctx, int B, const wg_qld_batch *q, const double *A0, const double *A1,
                            const unsigned char *sample, long long row_stride, const double *uz_dev, int N)
{
  RankedRows rk = {A0, A1, sample, row_stride, uz_dev, N};
  return qld_solve_impl(ctx, WG_MEM_DEVICE, B, q, A0 ? &rk : nullptr, true);
}

}  // extern "C"
