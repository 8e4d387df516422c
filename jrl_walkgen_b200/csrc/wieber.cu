// wieber.cu - the Wieber2006 generator (ZMPQPWithConstraint) front to back, batched over walks, for sm_100a.
//
// Replaces ZMPQPWithConstraint::BuildLinearConstraintInequalities / BuildMatricesPxPu / BuildZMPTrajectoryFromFootTrajectory /
// GetZMPDiscretization (src/ZMPRefTrajectoryGeneration/ZMPQPWithConstraint.cpp:229-502, :504-663, :665-1338, :1340-1387).
//
// A walk is a serial chain of QP periods (the LIPM state a QP is built for comes out of the previous one), so the batch axis is
// the walk: per period three launches over all walks that are still running -
//   wieber_pre_kernel   (one CTA per walk)  the N previewed polygons by the reference's clock rules, Px, the dense (m + 1) x 2N
//                                           matrix Pu in ql0001_'s column-major layout, and D = OptB x_k - OptC ZMPRef;
//   qld_kernel          (qld.cu)            the n = 2N = 150, m <= 8N = 600 QP, Hessian shared by the whole batch;
//   wieber_post_kernel  (one CTA per walk)  the reference's feasibility check of the solution (:1070-1105), the 5 ms CoM / ZMP
//                                           samples of the period and x_{k+1} = A x_k + B u.
// The constant matrices (:700-770, :905-990) are formed once on the host in the reference's summation order.
#include "wg_common.h"
#include <algorithm>
#include <cmath>
#include <cstddef>
#include <vector>

extern "C" int wgi_fcals_launch(wg_ctx *ctx, int B, const int64_t *d_samp_off, const wg_foot_sample *left,
                                const wg_foot_sample *right, const int32_t *types, const int64_t *d_lci_off, wg_lci *lci,
                                int32_t *n_lci, double hw, double hh, double sampling_period, size_t max_n,
                                const double **d_clock_out);

namespace {

constexpr int WB_T = 256;
constexpr int WB_MAXN = WG_WIEBER_MAX_N;            // 80 previewed samples
constexpr int WB_MAXROWS = WG_LCI_MAX_ROWS * WB_MAXN;

struct WbConsts {
  int N, interval, ld;              // previewed samples, 5 ms samples per QP period, leading dimension of Pu (8N + 1)
  double T, Ts, zc;
  double pz[WB_MAXN];               // (1 + 3d + 3d^2) T^3 / 6 - T zc / g      (:616-625)
  double sz[WB_MAXN][3];            // 1, (i+1) T, (i+1)^2 T^2 / 2 - zc / g    (:600-612)
  double optc[WB_MAXN];             // beta (1 + 3d + 3d^2) T^3 / 6: OptC = beta PPu' is Toeplitz
  double OptB[2 * WB_MAXN][6];
};

struct WbWalk {                     // per-walk loop state
  double xk[6];
  int li, status, done, hint;       // period index, 0 / failure code, finished, polygon index of the last StartingTime
  long long iterations;
};

struct WbHost {
  wg_wieber_params par;
  WbConsts h;
  WbConsts *d = nullptr;
  bool ready = false;
  std::vector<double> Ccm;          // the Hessian (column-major), kept to re-install it in the dense solver
  std::vector<double> start_h;      // StartingTime of period li: T added li times (:993-997)
  double *d_start = nullptr; size_t cap_start = 0;
  void *buf[16] = {nullptr};
  size_t cap[16] = {0};
};

WbHost *wb_of(wg_ctx *ctx)
{
  if (!ctx->wieber) ctx->wieber = new WbHost();
  return static_cast<WbHost *>(ctx->wieber);
}

// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(WB_T)
wieber_pre_kernel(int B, const WbConsts *__restrict__ Kp, const int64_t *__restrict__ samp_off,
                  const double *__restrict__ start_time, const int64_t *__restrict__ lci_off, const wg_lci *__restrict__ lci,
                  const int32_t *__restrict__ n_lci, const int *__restrict__ zd_status, const double *__restrict__ zmp,
                  WbWalk *__restrict__ walks, int32_t *__restrict__ m_out, double *__restrict__ Px, double *__restrict__ Pu,
                  double *__restrict__ Dv, double *__restrict__ A0g, double *__restrict__ A1g, unsigned char *__restrict__ sampg)
{
  __shared__ int s_poly[WB_MAXN], s_row0[WB_MAXN + 1];
  __shared__ int s_m, s_go;
  __shared__ double s_a0[WB_MAXROWS], s_a1[WB_MAXROWS];
  __shared__ unsigned char s_ri[WB_MAXROWS];
  __shared__ double s_xk[6], s_ref[2 * WB_MAXN];
  const WbConsts &K = *Kp;
  const int N = K.N, ld = K.ld, t = threadIdx.x;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    WbWalk &w = walks[b];
    const int64_t s0 = samp_off[b];
    const int n = (int)(samp_off[b + 1] - s0);
    const int np = n_lci[b];
    const wg_lci *L = lci + lci_off[b];
    __syncthreads();
    if (t == 0) {
      int go = !w.done;
      int m = 0;
      if (go && w.li == 0) {
        if (zd_status && zd_status[b]) { w.status = 4; go = 0; }
        else if (np <= 0 || np > (int)(lci_off[b + 1] - lci_off[b])) { w.status = 3; go = 0; }
      }
      if (go) {
        const double ST = start_time[w.li];
        // the loop bound of :993-995
        if (!(ST < L[np - 1].t_end - (unsigned)N * K.T)) go = 0;
        else {
          // the polygon that contains StartingTime (:531-549); StartingTime only grows, so the search resumes at the last hit
          int it = w.hint;
          while (it < np && !(ST >= L[it].t_start && ST <= L[it].t_end)) ++it;
          if (it >= np) { it = 0; while (it < np && !(ST >= L[it].t_start && ST <= L[it].t_end)) ++it; }
          if (it >= np) { w.status = 2; go = 0; }                       // "HERE 3"
          else {
            w.hint = it;
            // one polygon step at most per previewed sample (:567-577, :583-592)
            for (int i = 0; i < N; ++i) {
              const double ltime = ST + i * K.T;
              if (ltime > L[it].t_end) ++it;
              if (it >= np) { m = -1; break; }
              s_poly[i] = it; s_row0[i] = m;
              m += L[it].rows;
            }
            if (m < 0 || m > ld - 1) { w.status = 2; go = 0; }
            else s_row0[N] = m;
          }
        }
        if (!go) w.done = 1;
      }
      s_go = go; s_m = go ? m : 0;
      if (go) for (int c = 0; c < 6; ++c) s_xk[c] = w.xk[c];
    }
    __syncthreads();
    const int m = s_m;
    if (t == 0) m_out[b] = m;
    double *Db = Dv + (size_t)b * 2 * N;
    if (!s_go) {                                  // finished walk: an empty QP with a zero gradient
      for (int i = t; i < 2 * N; i += WB_T) Db[i] = 0.0;
      continue;
    }
    const int li = w.li;
    for (int i = t; i < N; i += WB_T) {
      const wg_lci &P = L[s_poly[i]];
      const int r0 = s_row0[i];
      for (int j = 0; j < P.rows; ++j) { s_a0[r0 + j] = P.A[j][0]; s_a1[r0 + j] = P.A[j][1]; s_ri[r0 + j] = (unsigned char)i; }
      const int64_t row = s0 + (int64_t)li * K.interval + (int64_t)i * K.interval;
      const bool in = row < s0 + n;
      s_ref[i] = in ? zmp[2 * row] : 0.0; s_ref[i + N] = in ? zmp[2 * row + 1] : 0.0;
    }
    __syncthreads();
    // Px (:594-612)
    double *Pxb = Px + (size_t)b * ld, *Pub = Pu ? Pu + (size_t)b * ld * 2 * N : nullptr;
    for (int r = t; r < m; r += WB_T) {
      const int i = s_ri[r];
      const wg_lci &P = L[s_poly[i]];
      const int j = r - s_row0[i];
      Pxb[r] = (s_xk[0] * K.sz[i][0] + s_xk[1] * K.sz[i][1] + s_xk[2] * K.sz[i][2]) * s_a0[r] +
               (s_xk[3] * K.sz[i][0] + s_xk[4] * K.sz[i][1] + s_xk[5] * K.sz[i][2]) * s_a1[r] + P.B[j];
    }
    // rank-structured rows for wg_qld_solve_batch_ranked: (A_r(0), A_r(1), i_r) - 17 bytes per row instead of 2N doubles
    if (A0g)
      for (int r = t; r < m; r += WB_T) { A0g[(size_t)b * ld + r] = s_a0[r]; A1g[(size_t)b * ld + r] = s_a1[r]; sampg[(size_t)b * ld + r] = s_ri[r]; }
    // Pu (:613-626): element (r, k) = A_r(0) pz(i_r - k), (r, k + N) = A_r(1) pz(i_r - k), k <= i_r; zero elsewhere
    for (int k = 0; Pu && k < N; ++k) {
      double *cx = Pub + (size_t)k * ld, *cy = Pub + (size_t)(k + N) * ld;
      for (int r = t; r < m; r += WB_T) {
        const int i = s_ri[r];
        const double v = (k <= i) ? K.pz[i - k] : 0.0;
        cx[r] = s_a0[r] * v; cy[r] = s_a1[r] * v;
      }
    }
    // D = OptB x_k - OptC ZMPRef (:1000-1030); OptC(i, k) = beta pu(k - i), k >= i, per axis
    for (int i = t; i < 2 * N; i += WB_T) {
      const int ax = i >= N, ii = ax ? i - N : i;
      double t1 = 0.0, t2 = 0.0;
      for (int k = ii; k < N; ++k) t1 += K.optc[k - ii] * s_ref[k + ax * N];
      for (int k = 0; k < 6; ++k) t2 += K.OptB[i][k] * s_xk[k];
      Db[i] = t2 - t1;
    }
  }
}

__global__ void __launch_bounds__(WB_T)
wieber_post_kernel(int B, const WbConsts *__restrict__ Kp, const int64_t *__restrict__ samp_off,
                   const int32_t *__restrict__ m_in, const double *__restrict__ Px, const double *__restrict__ Pu,
                   const double *__restrict__ X, const int32_t *__restrict__ ifail, const int32_t *__restrict__ iters,
                   WbWalk *__restrict__ walks, double *__restrict__ com, double *__restrict__ zmp,
                   const double *__restrict__ A0g, const double *__restrict__ A1g, const unsigned char *__restrict__ sampg)
{
  __shared__ int s_bad;
  __shared__ double s_x[2 * WB_MAXN], s_pt[2 * WB_MAXN];
  const WbConsts &K = *Kp;
  const int N = K.N, ld = K.ld, t = threadIdx.x;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    WbWalk &w = walks[b];
    __syncthreads();
    if (w.done) continue;
    const int m = m_in[b];
    if (t == 0) s_bad = (ifail[b] != 0);
    for (int i = t; i < 2 * N; i += WB_T) s_x[i] = X[(size_t)b * 2 * N + i];
    __syncthreads();
    // vnlValConstraint = Pu X + Px >= -1e-8 (:1056-1105; a violated row makes the reference return -1)
    const double *Pub = Pu ? Pu + (size_t)b * ld * 2 * N : nullptr, *Pxb = Px + (size_t)b * ld;
    if (A0g) {
      // rank-structured rows: Pu X = A_r(0) (Uz X_x)_i + A_r(1) (Uz X_y)_i
      for (int e = t; e < 2 * N; e += WB_T) {
        const int ax = e >= N, i = ax ? e - N : e;
        double a = 0.0;
        for (int k = 0; k <= i; ++k) a += K.pz[i - k] * s_x[ax * N + k];
        s_pt[e] = a;
      }
      __syncthreads();
      if (!s_bad)
        for (int r = t; r < m; r += WB_T) {
          const int i = sampg[(size_t)b * ld + r];
          if (A0g[(size_t)b * ld + r] * s_pt[i] + A1g[(size_t)b * ld + r] * s_pt[N + i] + Pxb[r] < -1e-8) s_bad = 1;
        }
    } else if (!s_bad)
      for (int r = t; r < m; r += WB_T) {
        double s = 0.0;
        for (int j = 0; j < 2 * N; ++j) s += Pub[r + (size_t)j * ld] * s_x[j];
        if (s + Pxb[r] < -1e-8) s_bad = 1;
      }
    __syncthreads();
    if (s_bad) {
      if (t == 0) { w.status = 1; w.done = 1; }
      continue;
    }
    const int64_t s0 = samp_off[b];
    const int n = (int)(samp_off[b + 1] - s0);
    const double jx = s_x[0], jy = s_x[N];
    const double *xk = w.xk;
    if (t < K.interval) {
      const int64_t row = (int64_t)w.li * K.interval + t;
      if (row < n) {
        const double s = (t + 1) * K.Ts;
        const double c0 = xk[0] + s * xk[1] + 0.5 * s * s * xk[2] + s * s * s * jx / 6.0;
        const double c1 = xk[1] + s * xk[2] + 0.5 * s * s * jx;
        const double c2 = xk[2] + s * jx;
        const double c3 = xk[3] + s * xk[4] + 0.5 * s * s * xk[5] + s * s * s * jy / 6.0;
        const double c4 = xk[4] + s * xk[5] + 0.5 * s * s * jy;
        const double c5 = xk[5] + s * jy;
        if (com) { double *c = com + 6 * (s0 + row); c[0] = c0; c[1] = c1; c[2] = c2; c[3] = c3; c[4] = c4; c[5] = c5; }
        const double cz = -K.zc / 9.81;
        zmp[2 * (s0 + row)] = 1.0 * c0 + 0.0 * c1 + cz * c2;
        zmp[2 * (s0 + row) + 1] = 1.0 * c3 + 0.0 * c4 + cz * c5;
      }
    }
    __syncthreads();
    if (t == 0) {
      const double T = K.T;
      const double B0 = T * T * T / 6.0, B1 = T * T / 2.0;
      const double nx0 = xk[0] + T * xk[1] + T * T / 2.0 * xk[2] + jx * B0;
      const double nx1 = xk[1] + T * xk[2] + jx * B1;
      const double nx2 = xk[2] + jx * T;
      const double ny0 = xk[3] + T * xk[4] + T * T / 2.0 * xk[5] + jy * B0;
      const double ny1 = xk[4] + T * xk[5] + jy * B1;
      const double ny2 = xk[5] + jy * T;
      w.xk[0] = nx0; w.xk[1] = nx1; w.xk[2] = nx2; w.xk[3] = ny0; w.xk[4] = ny1; w.xk[5] = ny2;
      w.li += 1;
      w.iterations += iters ? iters[b] : 0;
    }
  }
}

__global__ void wieber_finish_kernel(int B, const WbWalk *__restrict__ walks, int32_t *__restrict__ status,
                                     int32_t *__restrict__ periods_done, long long *__restrict__ iterations)
{
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  if (status) status[b] = walks[b].status;
  if (periods_done) periods_done[b] = walks[b].li + (walks[b].status == 1 ? 1 : 0);   // the failing period counts as attempted
  if (iterations) iterations[b] = walks[b].iterations;
}

// Host constants in the reference's summation order (uBLAS prod: k ascending from 0).
int make_constants(const wg_wieber_params &p, WbHost *H, std::vector<double> &Ccm)
{
  const int N = p.N, n = 2 * N;
  const double T = p.T, alpha = p.alpha, beta = p.beta;
  WbConsts &K = H->h;
  std::memset(&K, 0, sizeof K);
  K.N = N; K.ld = 8 * N + 1; K.T = T; K.Ts = p.sampling_period; K.zc = p.com_height;
  K.interval = (int)(T / p.sampling_period);
  if (K.interval < 1 || K.interval > WB_T) return WG_ERR_INVALID;
  for (int d = 0; d < N; ++d) {
    K.pz[d] = (1 + 3 * d + 3 * d * d) * T * T * T / 6.0 - T * p.com_height / 9.81;
    K.optc[d] = beta * ((1 + 3 * d + 3 * d * d) * T * T * T / 6.0);
    K.sz[d][0] = 1.0; K.sz[d][1] = T * (d + 1); K.sz[d][2] = (d + 1) * (d + 1) * T * T / 2 - p.com_height / 9.81;
  }
  std::vector<double> PPu((size_t)n * n, 0.0), VPu((size_t)n * n, 0.0), PPx((size_t)n * 6, 0.0), VPx((size_t)n * 6, 0.0);
  for (int i = 0; i < N; ++i) {
    VPx[(size_t)i * 6 + 1] = 1.0; VPx[(size_t)i * 6 + 2] = (i + 1) * T;
    VPx[(size_t)(i + N) * 6 + 4] = 1.0; VPx[(size_t)(i + N) * 6 + 5] = (i + 1) * T;
    PPx[(size_t)i * 6 + 0] = 1.0; PPx[(size_t)i * 6 + 1] = (i + 1) * T; PPx[(size_t)i * 6 + 2] = (i + 1) * (i + 1) * T * T * 0.5;
    PPx[(size_t)(i + N) * 6 + 3] = 1.0; PPx[(size_t)(i + N) * 6 + 4] = (i + 1) * T;
    PPx[(size_t)(i + N) * 6 + 5] = (i + 1) * (i + 1) * T * T * 0.5;
    for (int j = 0; j <= i; ++j) {
      const double v = (2 * (i - j) + 1) * T * T * 0.5, q = (1 + 3 * (i - j) + 3 * (i - j) * (i - j)) * T * T * T / 6.0;
      VPu[(size_t)i * n + j] = VPu[(size_t)(i + N) * n + j + N] = v;
      PPu[(size_t)i * n + j] = PPu[(size_t)(i + N) * n + j + N] = q;
    }
  }
  // C = beta PPu'PPu + alpha VPu'VPu (:905-925), column-major for ql0001_ (symmetric)
  Ccm.assign((size_t)n * n, 0.0);
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) {
      double l1 = 0.0, l2 = 0.0;
      for (int k = 0; k < n; ++k) { l1 += PPu[(size_t)k * n + i] * PPu[(size_t)k * n + j]; l2 += VPu[(size_t)k * n + i] * VPu[(size_t)k * n + j]; }
      Ccm[(size_t)j * n + i] = beta * l1 + alpha * l2;
    }
  // OptB = alpha VPu'VPx + beta PPu'PPx (:960-969)
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < 6; ++j) {
      double b1 = 0.0, b2 = 0.0;
      for (int k = 0; k < n; ++k) { b1 += PPu[(size_t)k * n + i] * PPx[(size_t)k * 6 + j]; b2 += VPu[(size_t)k * n + i] * VPx[(size_t)k * 6 + j]; }
      double v = alpha * b2;
      v += beta * b1;
      K.OptB[i][j] = v;
    }
  return WG_OK;
}

}  // namespace

void wg_wieber_release(wg_ctx *ctx)
{
  if (!ctx->wieber) return;
  WbHost *p = static_cast<WbHost *>(ctx->wieber);
  cudaFree(p->d); cudaFree(p->d_start);
  for (void *b : p->buf) cudaFree(b);
  delete p;
  ctx->wieber = nullptr;
}

extern "C" {

void wg_wieber_default_params(wg_wieber_params *p)
{
  if (!p) return;
  std::memset(p, 0, sizeof *p);
  p->T = 0.02; p->N = 75;                          // m_QP_T, m_QP_N (ZMPQPWithConstraint.cpp:71-72)
  p->sampling_period = 0.005;                      // :78
  p->com_height = 0.80;                            // ComHeight of BuildZMPTrajectoryFromFootTrajectory, :674
  p->alpha = 200.0; p->beta = 1000.0;              // :691
  p->constraint_x = 0.04; p->constraint_y = 0.04;  // :68-69
  p->sole_length = 0.25; p->sole_width = 0.14;     // robot data (HRP-2 test robot, SURVEY 8c)
  p->qld_eps = 1e-8;                               // Eps handed to ql0001_, :734
}

int wg_wieber_set_params(wg_ctx *ctx, const wg_wieber_params *p)
{
  if (!ctx || !p || !(p->T > 0.0) || !(p->sampling_period > 0.0) || p->N < 1 || p->N > WB_MAXN || 2 * p->N > WG_QLD_MAX_N)
    return WG_ERR_INVALID;
  wg_device_guard guard(ctx->device);
  WbHost *H = wb_of(ctx);
  int rc = make_constants(*p, H, H->Ccm);
  if (rc != WG_OK) return rc;
  if ((rc = wgi_qld_set_generator_hessian(ctx, 2 * p->N, 2 * p->N, H->Ccm.data(), p->qld_eps)) != WG_OK) return rc;
  H->par = *p;
  if (!H->d) WG_CUDA(ctx, cudaMalloc(&H->d, sizeof(WbConsts)));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  WG_CUDA(ctx, cudaMemcpy(H->d, &H->h, sizeof(WbConsts), cudaMemcpyHostToDevice));
  H->start_h.clear();
  H->ready = true;
  return WG_OK;
}

int64_t wg_wieber_period_count(const wg_wieber_params *p, int64_t n_samples)
{
  if (!p || n_samples < 1) return 0;
  double t = 0.0;
  for (int64_t i = 1; i < n_samples; ++i) t += p->sampling_period;
  const double horizon = (unsigned)p->N * p->T;
  int64_t c = 0;
  for (double st = 0.0; st < t - horizon; st += p->T) ++c;
  return c;
}

int wg_wieber_run_batch(wg_ctx *ctx, wg_kajita_plan *plan, int mem, double *com_out, double *zmp_out, wg_foot_sample *left,
                        wg_foot_sample *right, int32_t *status, int32_t *periods_done, long long *qp_iterations)
{
  if (!ctx || !plan) return WG_ERR_INVALID;
  if (mem != WG_MEM_HOST && mem != WG_MEM_DEVICE) return WG_ERR_INVALID;
  WbHost *H = wb_of(ctx);
  if (!H->ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_wieber_set_params not called");
  wg_device_guard guard(ctx->device);
  const bool host = mem == WG_MEM_HOST;
  const wg_wieber_params &par = H->par;
  const int N = par.N, nv = 2 * N, ld = 8 * N + 1;
  // ---- GetZMPDiscretization (:1355-1364)
  double *d_zmp = host ? nullptr : zmp_out;
  wg_foot_sample *d_left = host ? nullptr : left, *d_right = host ? nullptr : right;
  int32_t *d_types = nullptr;
  wgi_kajita_view V;
  int rc = wgi_kajita_discretize_device(ctx, plan, &d_zmp, &d_left, &d_right, &d_types, &V);
  if (rc != WG_OK) return rc;
  if (std::fabs(V.sampling_period - par.sampling_period) > 1e-15)
    return wg_fail(ctx, WG_ERR_INVALID, "sampling period of the plan differs from wg_wieber_params");
  const int B = V.B;
  const size_t nb = (size_t)B, ns = (size_t)V.samp_off[B];
  int64_t max_n = 0;
  std::vector<int64_t> lci_off(B + 1);
  lci_off[0] = 0;
  for (int b = 0; b < B; ++b) {
    max_n = std::max(max_n, V.samp_off[b + 1] - V.samp_off[b]);
    lci_off[b + 1] = lci_off[b] + 2 * (V.step_off[b + 1] - V.step_off[b]) + 6;
  }
  const int64_t max_periods = wg_wieber_period_count(&par, max_n);
  if ((int64_t)H->start_h.size() < max_periods + 2) {
    H->start_h.resize((size_t)max_periods + 2);
    double st = 0.0;
    for (size_t i = 0; i < H->start_h.size(); ++i) { H->start_h[i] = st; st += par.T; }
    if (H->cap_start < H->start_h.size()) {
      WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
      cudaFree(H->d_start); H->d_start = nullptr;
      WG_CUDA(ctx, cudaMalloc(&H->d_start, sizeof(double) * H->start_h.size()));
      H->cap_start = H->start_h.size();
    }
    WG_CUDA(ctx, cudaMemcpy(H->d_start, H->start_h.data(), sizeof(double) * H->start_h.size(), cudaMemcpyHostToDevice));
  }
  const size_t nl = (size_t)lci_off[B];
  if ((rc = wgi_grow_scratch(ctx, &H->buf[0], &H->cap[0], sizeof(int64_t) * (nb + 1))) != WG_OK) return rc;
  if ((rc = wgi_grow_scratch(ctx, &H->buf[1], &H->cap[1], sizeof(wg_lci) * nl)) != WG_OK) return rc;
  if ((rc = wgi_grow_scratch(ctx, &H->buf[2], &H->cap[2], sizeof(int32_t) * 4 * nb)) != WG_OK) return rc;
  if ((rc = wgi_grow_scratch(ctx, &H->buf[3], &H->cap[3], sizeof(WbWalk) * nb)) != WG_OK) return rc;
  if ((rc = wgi_grow_scratch(ctx, &H->buf[4], &H->cap[4], sizeof(double) * nb * ld)) != WG_OK) return rc;
  const bool dense = par.materialize_pu != 0;
  if (dense) { if ((rc = wgi_grow_scratch(ctx, &H->buf[5], &H->cap[5], sizeof(double) * nb * ld * nv)) != WG_OK) return rc; }
  else { if ((rc = wgi_grow_scratch(ctx, &H->buf[9], &H->cap[9], (sizeof(double) * 2 + 1) * nb * ld + 64)) != WG_OK) return rc; }
  if ((rc = wgi_grow_scratch(ctx, &H->buf[6], &H->cap[6], sizeof(double) * nb * nv * 2)) != WG_OK) return rc;
  int64_t *d_lo = static_cast<int64_t *>(H->buf[0]);
  wg_lci *d_lci = static_cast<wg_lci *>(H->buf[1]);
  int32_t *d_nlci = static_cast<int32_t *>(H->buf[2]), *d_m = d_nlci + nb, *d_ifail = d_m + nb, *d_it = d_ifail + nb;
  WbWalk *d_walks = static_cast<WbWalk *>(H->buf[3]);
  double *d_Px = static_cast<double *>(H->buf[4]), *d_Pu = dense ? static_cast<double *>(H->buf[5]) : nullptr;
  double *d_A0 = dense ? nullptr : static_cast<double *>(H->buf[9]), *d_A1 = dense ? nullptr : d_A0 + nb * ld;
  unsigned char *d_samp = dense ? nullptr : reinterpret_cast<unsigned char *>(d_A1 + nb * ld);
  const double *d_uz = reinterpret_cast<const double *>(reinterpret_cast<const char *>(H->d) + offsetof(WbConsts, pz));
  double *d_D = static_cast<double *>(H->buf[6]), *d_X = d_D + nb * nv;
  WG_CUDA(ctx, cudaMemcpyAsync(d_lo, lci_off.data(), sizeof(int64_t) * (nb + 1), cudaMemcpyHostToDevice, ctx->stream));
  WG_CUDA(ctx, cudaMemsetAsync(d_walks, 0, sizeof(WbWalk) * nb, ctx->stream));
  double *d_com = com_out;
  if (host && com_out) {
    if ((rc = wgi_grow_scratch(ctx, &H->buf[7], &H->cap[7], sizeof(double) * 6 * ns)) != WG_OK) return rc;
    d_com = static_cast<double *>(H->buf[7]);
  }
  if (d_com) WG_CUDA(ctx, cudaMemsetAsync(d_com, 0, sizeof(double) * 6 * ns, ctx->stream));
  // ---- BuildLinearConstraintInequalities (:229-502)
  const double *d_clock = nullptr;
  rc = wgi_fcals_launch(ctx, B, V.d_samp_off, d_left, d_right, d_types, d_lo, d_lci, d_nlci, 0.5 * par.sole_length - par.constraint_x,
                        0.5 * par.sole_width - par.constraint_y, par.sampling_period, (size_t)max_n, &d_clock);
  if (rc != WG_OK) return rc;
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // lci_off is a pageable temporary
  // ---- the loop (:993-1330)
  wg_qld_batch q;
  std::memset(&q, 0, sizeof q);
  q.n = nv; q.nmax = nv; q.mmax = ld; q.shared_hessian = 1;
  q.m = d_m; q.d = d_D; q.A = d_Pu; q.a_stride = (long long)ld * nv; q.b = d_Px; q.b_stride = ld;   // A: dense mode only
  q.x = d_X; q.ifail = d_ifail; q.iterations = d_it;
  const int grid = std::max(1, std::min(B, ctx->sm_count * 4));
  for (int64_t li = 0; li < max_periods; ++li) {
    wg_prof_start(ctx, WG_K_WIEBER);
    wieber_pre_kernel<<<grid, WB_T, 0, ctx->stream>>>(B, H->d, V.d_samp_off, H->d_start, d_lo, d_lci, d_nlci, V.d_zd_status,
                                                     d_zmp, d_walks, d_m, d_Px, d_Pu, d_D, d_A0, d_A1, d_samp);
    wg_prof_stop(ctx);
    WG_LAUNCHED(ctx);
    rc = wgi_qld_solve_generator(ctx, B, &q, d_A0, d_A1, d_samp, ld, d_uz, N);     // d_A0 = nullptr in dense mode
    if (rc != WG_OK) return rc;
    wg_prof_start(ctx, WG_K_WIEBER);
    wieber_post_kernel<<<grid, WB_T, 0, ctx->stream>>>(B, H->d, V.d_samp_off, d_m, d_Px, d_Pu, d_X, d_ifail, d_it, d_walks,
                                                      d_com, d_zmp, d_A0, d_A1, d_samp);
    wg_prof_stop(ctx);
    WG_LAUNCHED(ctx);
  }
  // one more pre pass so that walks whose loop bound is reached exactly at max_periods are marked done (no effect otherwise)
  int32_t *d_status = status, *d_done = periods_done;
  long long *d_iter = qp_iterations;
  if (host) {
    if ((rc = wgi_grow_scratch(ctx, &H->buf[8], &H->cap[8], (sizeof(int32_t) * 2 + sizeof(long long)) * nb)) != WG_OK) return rc;
    d_iter = static_cast<long long *>(H->buf[8]);
    d_status = reinterpret_cast<int32_t *>(d_iter + nb); d_done = d_status + nb;
  }
  wieber_finish_kernel<<<(B + 127) / 128, 128, 0, ctx->stream>>>(B, d_walks, d_status, d_done, d_iter);
  WG_LAUNCHED(ctx);
  if (host) {
    if (com_out) WG_CUDA(ctx, cudaMemcpyAsync(com_out, d_com, sizeof(double) * 6 * ns, cudaMemcpyDeviceToHost, ctx->stream));
    if (zmp_out) WG_CUDA(ctx, cudaMemcpyAsync(zmp_out, d_zmp, sizeof(double) * 2 * ns, cudaMemcpyDeviceToHost, ctx->stream));
    if (left) WG_CUDA(ctx, cudaMemcpyAsync(left, d_left, sizeof(wg_foot_sample) * ns, cudaMemcpyDeviceToHost, ctx->stream));
    if (right) WG_CUDA(ctx, cudaMemcpyAsync(right, d_right, sizeof(wg_foot_sample) * ns, cudaMemcpyDeviceToHost, ctx->stream));
    if (status) WG_CUDA(ctx, cudaMemcpyAsync(status, d_status, sizeof(int32_t) * nb, cudaMemcpyDeviceToHost, ctx->stream));
    if (periods_done) WG_CUDA(ctx, cudaMemcpyAsync(periods_done, d_done, sizeof(int32_t) * nb, cudaMemcpyDeviceToHost, ctx->stream));
    if (qp_iterations) WG_CUDA(ctx, cudaMemcpyAsync(qp_iterations, d_iter, sizeof(long long) * nb, cudaMemcpyDeviceToHost, ctx->stream));
    WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return WG_OK;
}

}  // extern "C"
