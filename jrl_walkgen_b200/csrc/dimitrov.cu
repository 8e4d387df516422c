// dimitrov.cu - the Dimitrov2008 generator front to back on the device, for sm_100a.
//
// Replaces (see include/walkgen_b200.h for the file:line list)
//   ComputeConvexHull::DoComputeConvexHull, FootConstraintsAsLinearSystem::{BuildLinearConstraintInequalities,
//   ComputeLinearSystem, FindSimilarConstraints}, ZMPConstrainedQPFastFormulation::{InitConstants,
//   BuildConstraintMatrices, BuildZMPTrajectoryFromFootTrajectory (PLDP branch)},
//   LinearizedInvertedPendulum2D::{Interpolation, OneIteration}.
//
// Two kernels, both "one warp owns one walk":
//   fcals_kernel      scans the 5 ms feet buffers 32 samples at a time (the support state of a sample is a function
//                     of that sample alone; ballots find the state changes) and the lane sitting on a change builds the
//                     polygon of the new phase: convex hull of the 8 foot corners (double support) or the 4 corners of
//                     the support foot, then the half-plane form.
//   dimitrov_kernel   the receding-horizon loop: per 0.1 s period the warp locates the 16 previewed polygons, builds
//                     the constraint matrix DPu ((m+1) x 32, column-major, exactly the array the reference hands to
//                     PLDPSolver) in SHARED memory - it never exists in HBM -, forms D and DPx, runs the PLDP solve of
//                     pldp.cuh with the hot-start memory kept in shared memory, applies the jerk to the LIPM and writes
//                     the 21 interpolated 5 ms CoM/ZMP samples.  HBM traffic per period: 16 polygon records read
//                     (L2-resident) + 21 x 64 B written.
//
// Arithmetic: compiled with -fmad=false and written in the reference's operation order, so that every discrete decision
// (state changes, hull membership, polygon lookup by the accumulated clocks, PLDP step lengths and activations) falls as
// in the reference's x86-64 object code.  The only non-IEEE-exact operations are sin/cos of the foot yaw (device libm vs
// glibc: last-bit differences when a foot is rotated).
#include "pldp.cuh"
#include <algorithm>
#include <cmath>
#include <map>
#include <new>

namespace {

constexpr int DM_N = PLDP_N;          // 16
constexpr int DM_WARPS = 4;           // loop kernel: 4 warps per CTA, ~9 KB of shared memory per warp
constexpr int FC_WARPS = 4;           // polygon kernel
constexpr int DM_MAXM = WG_LCI_MAX_ROWS * DM_N;   // 128

struct DimConsts {
  double Px[DM_N * 3];
  double Pu[DM_N * DM_N];             // m_Pu = iLQ * Pu'
  double OptB[DM_N * 3];
  double OptC[DM_N * DM_N];
  double iLQc0[DM_N];                 // column 0 of iLQ: NewX[0] = sum_j iLQ(j,0) X[j]
  double T, Ts, zc;
  double hw, hh;                      // half sole sizes minus the security margins
  double horizon;                     // N * T
  int interval;                       // (int)(T / Ts)
  int max_iter;
  int cold_restart;
  int merge_rows;
};

struct DimHost {
  wg_dimitrov_params par;
  DimConsts h;
  DimConsts *d = nullptr;
  bool ready = false;
  double iPu[DM_N * DM_N], iLQ[DM_N * DM_N];
  // clock table and scratch (grow-only)
  double *d_time = nullptr;
  std::vector<double> time_h;
  void *buf[14] = {nullptr};
  size_t cap[14] = {0};
  // the longest-first walk order of the last plan, kept on the device (slot 12)
  const void *order_plan = nullptr; int order_B = 0; int64_t order_total = -1;
  std::map<int64_t, int64_t> period_cache;
};

DimHost *dim_of(wg_ctx *ctx)
{
  if (!ctx->dimitrov) ctx->dimitrov = new DimHost();
  return static_cast<DimHost *>(ctx->dimitrov);
}

// ---------------------------------------------------------------------------------------------------------------
// Convex hull and half-plane form (device; one thread)
// ---------------------------------------------------------------------------------------------------------------
struct P2 { double col, row; };

__device__ __forceinline__ double cross0(const P2 &p0, const P2 &s1, const P2 &s2)
{
  const double x1 = s1.col - p0.col, x2 = s2.col - p0.col, y1 = s1.row - p0.row, y2 = s2.row - p0.row;
  return x1 * y2 - x2 * y1;
}

// DoComputeConvexHull (ConvexHull.cpp:87-203) for n <= 8 points.  The reference's std::set ordered by "cross product about
// p0 > 0" becomes a small array kept in that order; points of equal polar angle are merged as the reference does
// (the farther one stays).  Returns the number of hull vertices (<= 8); hull[0] = the lowest point.
__device__ int dv_convex_hull(const P2 *in, int n, P2 *hull)
{
  P2 p0 = in[0];
  for (int i = 0; i < n; ++i)
    if (in[i].row < p0.row) p0 = in[i];
  P2 lst[8];
  int nl = 0;
  for (int i = 0; i < n; ++i) {
    bool ins = true;
    for (int k = 0; k < nl;) {
      bool del = false;
      if (cross0(p0, lst[k], in[i]) == 0.0) {
        const double x1 = lst[k].col - p0.col, y1 = lst[k].row - p0.row, x2 = in[i].col - p0.col, y2 = in[i].row - p0.row;
        const double d1 = sqrt(x1 * x1 + y1 * y1), d2 = sqrt(x2 * x2 + y2 * y2);
        if (d1 <= d2) del = true; else ins = false;
      }
      if (del) { for (int q = k; q + 1 < nl; ++q) lst[q] = lst[q + 1]; --nl; }
      else ++k;
    }
    if (ins) {
      int pos = 0;
      while (pos < nl && cross0(p0, lst[pos], in[i]) > 0.0) ++pos;
      for (int q = nl; q > pos; --q) lst[q] = lst[q - 1];
      lst[pos] = in[i];
      ++nl;
    }
  }
  int nh = 0;
  hull[nh++] = p0;
  if (nl < 2) { for (int k = 0; k < nl; ++k) hull[nh++] = lst[k]; return nh; }   // the reference reads past end() here
  hull[nh++] = lst[0];
  hull[nh++] = lst[1];
  for (int k = 2; k < nl; ++k) {
    const P2 pi = lst[k];
    bool ok;
    do {
      if (nh >= 2) {
        const P2 s1 = hull[nh - 1], s2 = hull[nh - 2];
        const double x1 = s1.col - s2.col, x2 = pi.col - s2.col, y1 = s1.row - s2.row, y2 = pi.row - s2.row;
        ok = (x1 * y2 - x2 * y1) > 0.0;
      } else ok = true;
      if (!ok) --nh;
    } while (!ok);
    hull[nh++] = pi;
  }
  return nh;
}

// one edge of ComputeLinearSystem (FootConstraintsAsLinearSystem.cpp:151-193 and, for the closing edge, :207-243)
__device__ __forceinline__ void dv_edge(const P2 &from, const P2 &to, const P2 &icpt, double &a, double &b, double &c)
{
  if (fabs(to.col - from.col) > 1e-7) {
    double y1, x1, y2, x2, lmul = -1.0;
    if (to.col < from.col) { lmul = 1.0; y2 = from.row; y1 = to.row; x2 = from.col; x1 = to.col; }
    else { y2 = to.row; y1 = from.row; x2 = to.col; x1 = from.col; }
    a = (y2 - y1) / (x2 - x1);
    b = (icpt.row - a * icpt.col);
    a = lmul * a; b = lmul * b; c = -lmul;
  } else {
    c = 0.0; a = -1.0; b = to.col;
    if (to.row < from.row) { a = -a; b = -b; }
  }
}

// ComputeLinearSystem + FindSimilarConstraints into the record at `o` (every field except t_end, which the lane of the
// NEXT state change owns)
__device__ void dv_write_polygon(wg_lci *o, const P2 *v, int n, double t_start, int first_sample, int state, int merge)
{
  double A0[WG_LCI_MAX_ROWS], A1[WG_LCI_MAX_ROWS], Bv[WG_LCI_MAX_ROWS];
  double C0 = 0.0, C1 = 0.0;
  for (int i = 0; i + 1 < n; ++i) {
    C0 += v[i].col; C1 += v[i].row;
    dv_edge(v[i], v[i + 1], v[i], A0[i], Bv[i], A1[i]);
  }
  C0 += v[n - 1].col; C1 += v[n - 1].row;
  C0 /= (double)n; C1 /= (double)n;
  dv_edge(v[n - 1], v[0], v[0], A0[n - 1], Bv[n - 1], A1[n - 1]);
  if (merge) {
    // NOT in the reference (wg_dimitrov_params.merge_duplicate_rows): drop a half-plane that repeats its predecessor
    int k = 0;
    for (int i = 0; i < n; ++i) {
      if (k > 0 && fabs(A0[i] - A0[k - 1]) <= 1e-9 && fabs(A1[i] - A1[k - 1]) <= 1e-9 && fabs(Bv[i] - Bv[k - 1]) <= 1e-9) continue;
      A0[k] = A0[i]; A1[k] = A1[i]; Bv[k] = Bv[i];
      ++k;
    }
    if (k > 1 && fabs(A0[k - 1] - A0[0]) <= 1e-9 && fabs(A1[k - 1] - A1[0]) <= 1e-9 && fabs(Bv[k - 1] - Bv[0]) <= 1e-9) --k;
    n = k;
  }
  const double W0 = (A0[0] * C0 + A1[0] * C1) + Bv[0], W1 = (A0[1] * C0 + A1[1] * C1) + Bv[1];
  for (int i = 0; i < WG_LCI_MAX_ROWS; ++i) {
    o->A[i][0] = i < n ? A0[i] : 0.0; o->A[i][1] = i < n ? A1[i] : 0.0; o->B[i] = i < n ? Bv[i] : 0.0;
    int sim = 0;
    if (n == 4 && i >= 2 && i < 4 && A0[i - 2] == -A0[i] && A1[i - 2] == -A1[i]) sim = -2;
    if (n == 6 && i >= 3 && i < 6 && A0[i - 3] == -A0[i] && A1[i - 3] == -A1[i]) sim = -3;
    o->similar[i] = sim;
  }
  o->center[0] = C0; o->center[1] = C1;
  o->t_start = t_start;
  o->rows = n;
  o->first_sample = first_sample;
  o->state = state;
  o->rc = (W0 < 0 || W1 < 0) ? -1 : 0;
}

__device__ __forceinline__ void dv_foot_corners(const wg_foot_sample &f, double hw, double hh, P2 *out)
{
  const double lxc[4] = {1.0, 1.0, -1.0, -1.0}, lyc[4] = {-1.0, 1.0, 1.0, -1.0};
  const double s_t = sin(f.theta * M_PI / 180.0), c_t = cos(f.theta * M_PI / 180.0);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    out[j].col = f.x + (lxc[j] * hw * c_t - lyc[j] * hh * s_t);
    out[j].row = f.y + (lxc[j] * hw * s_t + lyc[j] * hh * c_t);
  }
}

__global__ void __launch_bounds__(128)
convex_hull_kernel(int B, int n, const double *__restrict__ xy, double *__restrict__ hull_xy, int32_t *__restrict__ counts)
{
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  P2 in[8], hull[8];
  for (int i = 0; i < n; ++i) { in[i].col = xy[((size_t)b * n + i) * 2]; in[i].row = xy[((size_t)b * n + i) * 2 + 1]; }
  const int nh = dv_convex_hull(in, n, hull);
  for (int i = 0; i < 8; ++i) {
    hull_xy[((size_t)b * 8 + i) * 2] = i < nh ? hull[i].col : 0.0;
    hull_xy[((size_t)b * 8 + i) * 2 + 1] = i < nh ? hull[i].row : 0.0;
  }
  counts[b] = nh;
}

// BuildLinearConstraintInequalities (FootConstraintsAsLinearSystem.cpp:258-539), one warp per walk.
__global__ void __launch_bounds__(FC_WARPS * 32)
fcals_kernel(int B, const DimConsts *__restrict__ Kp, const int64_t *__restrict__ samp_off,
             const wg_foot_sample *__restrict__ left, const wg_foot_sample *__restrict__ right,
             const int32_t *__restrict__ types, const double *__restrict__ clock, const int64_t *__restrict__ lci_off,
             wg_lci *__restrict__ lci, int32_t *__restrict__ n_lci)
{
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const double hw = Kp->hw, hh = Kp->hh;
  for (int b = blockIdx.x * FC_WARPS + warp; b < B; b += gridDim.x * FC_WARPS) {
    const int64_t s0 = samp_off[b];
    const int n = (int)(samp_off[b + 1] - s0);
    const int cap = (int)(lci_off[b + 1] - lci_off[b]);
    wg_lci *out = lci + lci_off[b];
    int carry = 3;      // State before sample 0 (:312-316: i == 0 forces State = 3 before the tests)
    int count = 0, over_i = -1;
    // phase 1, 4 chunks of 32 samples per trip: the 12 strided loads of a trip are issued together (one exposed memory latency per
    // 128 samples; the chunks are still processed in order - state and count carry over)
    constexpr int FC_U = 4;
    for (int cb = 0; cb < n; cb += 32 * FC_U) {
      double lzv[FC_U], rzv[FC_U];
      int tyv[FC_U];
#pragma unroll
      for (int u = 0; u < FC_U; ++u) {
        const int iu = cb + 32 * u + lane;
        lzv[u] = 0.0; rzv[u] = 0.0; tyv[u] = 0;
        if (iu < n) { lzv[u] = left[s0 + iu].z; rzv[u] = right[s0 + iu].z; tyv[u] = types[3 * (s0 + iu) + 1]; }
      }
#pragma unroll
      for (int u = 0; u < FC_U; ++u) {
      const int c0 = cb + 32 * u;
      if (c0 >= n) break;
      const int i = c0 + lane;
      const bool valid = i < n;
      int st = -1;
      double lz = 0.0, rz = 0.0;
      if (valid) {
        lz = lzv[u]; rz = rzv[u];
        const int ty = tyv[u];
        const double thr = 0.00001;
        if (ty >= 10) st = 3;
        else if (lz > thr) st = 2;
        else if (rz > thr) st = 1;
        else if (rz < thr && lz < thr) st = 3;
      }
      // a sample that matches no branch keeps the state of its predecessor
      const unsigned def = __ballot_sync(0xffffffffu, st >= 0);
      const unsigned below = def & ((2u << lane) - 1u);            // definite lanes <= lane
      const int src = below ? 31 - __clz(below) : -1;
      int res = __shfl_sync(0xffffffffu, st, src < 0 ? 0 : src);
      if (src < 0) res = carry;
      int prev = __shfl_up_sync(0xffffffffu, res, 1);
      if (lane == 0) prev = carry;
      const bool boundary = valid && (i == 0 || res != prev);
      const unsigned bm = __ballot_sync(0xffffffffu, boundary);
      const int idx = count + __popc(bm & ((1u << lane) - 1u));
      // phase 1 only records where the support state changes - in the polygon record itself -; the polygons are built
      // afterwards, one per lane
      if (boundary && idx < cap) { out[idx].first_sample = i; out[idx].state = res; }
      const unsigned ov = __ballot_sync(0xffffffffu, boundary && idx == cap);   // the first polygon that does not fit still closes the last
      if (ov) over_i = __shfl_sync(0xffffffffu, i, __ffs(ov) - 1);
      count += __popc(bm);
      const int last = min(31, n - 1 - c0);
      carry = __shfl_sync(0xffffffffu, res, last);
      }
    }
    __syncwarp();
    // ---- phase 2: polygon k of the walk by lane k mod 32 (a walk of configs[1] has ~20 support phases: one round instead of
    //      20 single-lane constructions of ~2.7 k instructions each)
    const int npoly = min(count, cap);
    for (int k0 = 0; k0 < npoly; k0 += 32) {
      const int k = k0 + lane;
      int i = 0, res = 0, inext = -1;
      if (k < npoly) {
        i = out[k].first_sample; res = out[k].state;
        if (k + 1 < npoly) inext = out[k + 1].first_sample;      // read before lane k + 1 rewrites its record
      }
      __syncwarp();
      if (k < npoly) {
        const double t = clock[i];
        const wg_foot_sample L = left[s0 + i], R = right[s0 + i];
        P2 hull[8];
        int nh;
        if (res == 3) {
          P2 pts[8];
          dv_foot_corners(L, hw, hh, pts);
          dv_foot_corners(R, hw, hh, pts + 4);
          nh = dv_convex_hull(pts, 8, hull);
        } else {
          nh = 4;
          if (L.z < R.z) dv_foot_corners(L, hw, hh, hull);
          else dv_foot_corners(R, hw, hh, hull);
        }
        dv_write_polygon(out + k, hull, nh, t, i, res, Kp->merge_rows);
        // EndingTime: the clock of the sample that opens the next polygon (also when that one no longer fits), else the last sample
        out[k].t_end = inext >= 0 ? clock[inext] : (k + 1 < count && over_i >= 0 ? clock[over_i] : clock[n - 1]);
      }
      __syncwarp();
    }
    if (lane == 0) n_lci[b] = count <= cap ? count : -count;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// The receding-horizon loop
// ---------------------------------------------------------------------------------------------------------------
struct DimWarp {
  PldpWarp pw;
  double bv[DM_MAXM + 1];
  double rowa[2][DM_MAXM];
  double zref[PLDP_U];
  double xk[6];
  int prev_active[PLDP_U];
  unsigned char rowi[DM_MAXM];
};

// 4 CTAs/SM (128 registers) measured best at both batch sizes tried: 4096 walks 36.1 ms (3 CTAs/SM at 161 registers: 38 ms, 5
// CTAs/SM at 96 registers: 47.8 ms, 6 at 80 registers with spills: 58 ms); 16 384 walks 111 ms (3: 122 ms, 5: 121 ms).  A walk is
// a serial chain of some hundred periods: per-warp speed (registers, few warps per scheduler) counts as much as residency.
__global__ void __launch_bounds__(DM_WARPS * 32, 3)   // 168 registers, no spills: 32.2 ms per 4096 walks against 33.8 at 4 CTAs / 128 registers
dimitrov_kernel(int B, const DimConsts *__restrict__ Kp, const PldpConsts *__restrict__ Cp,
                const int64_t *__restrict__ samp_off, const double *__restrict__ clock,
                const int64_t *__restrict__ lci_off, const wg_lci *__restrict__ lci, const int32_t *__restrict__ n_lci,
                const int *__restrict__ zd_status, double *__restrict__ com, double *__restrict__ zmp,
                const int64_t *__restrict__ per_off, wg_dimitrov_period *__restrict__ periods,
                int32_t *__restrict__ status_out, int32_t *__restrict__ done_out, int *__restrict__ next_walk,
                const int *__restrict__ order)
{
  __shared__ DimWarp ws[DM_WARPS];
  __shared__ double sPu[DM_N * DM_N], sPuT[DM_N * DM_N];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const DimConsts &K = *Kp;
  const PldpConsts &C = *Cp;
  DimWarp &w = ws[warp];
  constexpr int N = DM_N;
  for (int e = threadIdx.x; e < N * N; e += blockDim.x) { sPu[e] = K.Pu[e]; sPuT[(e % N) * N + e / N] = K.Pu[e]; }
  __syncthreads();
  const double T = K.T, Ts = K.Ts;
  const double tol = 1e-8;   // m_tol, PLDPSolver.cpp:66
  const int ii = lane & (N - 1), ax = lane >> 4;
  // walks differ in length by an order of magnitude: every warp fetches its next walk from a global counter, longest
  // walks first (`order`)
  for (;;) {
    int b = 0;
    if (lane == 0) { b = atomicAdd(next_walk, 1); if (b < B) b = order[b]; }
    b = __shfl_sync(0xffffffffu, b, 0);
    if (b >= B) break;
    const int64_t s0 = samp_off[b];
    const int n = (int)(samp_off[b + 1] - s0);
    const int np = n_lci[b];
    const wg_lci *P = lci + lci_off[b];
    wg_dimitrov_period *per = periods ? periods + per_off[b] : nullptr;
    const int per_cap = periods ? (int)(per_off[b + 1] - per_off[b]) : 0;
    int wstatus = 0;
    if (np <= 0) wstatus = 3;
    if (zd_status && zd_status[b] != 0) wstatus = 4;
    // LIPM state (m_CoM of LinearizedInvertedPendulum2D: zero after InitializeSystem)
    double cx0 = 0.0, cx1 = 0.0, cx2 = 0.0, cy0 = 0.0, cy1 = 0.0, cy2 = 0.0;
    int n_prev = 0, removed = 0;
    bool starting = true;
    int first = 0;         // polygon the previous period started in: the search of :785-795 can resume there
    long li = 0;
    const double t_last = wstatus == 0 ? P[np - 1].t_end : 0.0;
    for (double ST = 0.0; wstatus == 0 && ST < t_last - K.horizon; ST += T, ++li) {
      // ---- BuildConstraintMatrices (:759-1022): locate the polygons of the 16 previewed instants
      while (first < np && !(ST >= P[first].t_start && ST <= P[first].t_end)) ++first;
      if (first >= np) { wstatus = 2; break; }
      int it = first, my_p = first;
      double te = P[it].t_end;
      bool past = false;
#pragma unroll 1
      for (int i = 0; i < N; ++i) {
        const double ltime = ST + i * T;
        if (ltime > te) { ++it; if (it >= np) { past = true; break; } te = P[it].t_end; }
        if (lane == i) my_p = it;
      }
      if (past) { wstatus = 2; break; }
      const int my_rows = lane < N ? P[my_p].rows : 0;
      int incl = my_rows;
#pragma unroll
      for (int o = 1; o < 16; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
      const int m = __shfl_sync(0xffffffffu, incl, N - 1);
      const int roff = incl - my_rows;
      const int n_first = __shfl_sync(0xffffffffu, my_rows, 0);
      if (lane < 6) w.xk[lane] = lane == 0 ? cx0 : lane == 1 ? cx1 : lane == 2 ? cx2 : lane == 3 ? cy0 : lane == 4 ? cy1 : cy2;
      if (lane < N) {
        const wg_lci &q = P[my_p];
        w.zref[lane] = q.center[0];
        w.zref[lane + N] = q.center[1];
        const double zx = cx0 * K.Px[lane * 3 + 0] + cx1 * K.Px[lane * 3 + 1] + cx2 * K.Px[lane * 3 + 2];
        const double zy = cy0 * K.Px[lane * 3 + 0] + cy1 * K.Px[lane * 3 + 1] + cy2 * K.Px[lane * 3 + 2];
#pragma unroll 1
        for (int j = 0; j < my_rows; ++j) {
          const double a0 = q.A[j][0], a1 = q.A[j][1];
          w.rowa[0][roff + j] = a0;
          w.rowa[1][roff + j] = a1;
          w.rowi[roff + j] = lane;
          w.bv[roff + j] = zx * a0 + zy * a1 + q.B[j];
        }
      }
      __syncwarp();
      // DPu (:885-905) is never materialised: element (r, k + N ax) = A_r[ax] * Pu[k N + i_r] is formed where it is used
      // (RankMat, pldp.cuh) by the same single IEEE multiplication the reference stores
      const RankMat M{w.rowa[0], w.rowa[1], w.rowi, sPu, sPuT};
      // D = OptB xk - OptC ZMPRef (:1268-1276), row `lane`
      double Dl;
      {
        double t1 = 0.0, t2 = 0.0;
#pragma unroll 2
        for (int j = 0; j < N; ++j) t1 += K.OptC[ii * N + j] * w.zref[j + N * ax];
        for (int j = 0; j < 3; ++j) t2 += K.OptB[ii * 3 + j] * w.xk[3 * ax + j];
        Dl = t2 - t1;
      }
      __syncwarp();
      // ---- PLDPSolver::SolveProblem, hot-started from the previous period.  A second pass (cold_restart) solves the
      // period again from the cold start point when the reference would print "PB ON constraint" and call exit(0).
      PldpRes r;
      double Vk = 0.0;
      int pstatus = 0;
      for (int attempt = 0; attempt < 2; ++attempt) {
        const bool cold = attempt == 1;
        Vk = pldp_solve_warp(C, w.pw, M, m, w.bv, Dl, w.zref, w.xk, !starting && !cold, w.pw.prev_zmp, cold ? 0 : n_prev,
                             w.prev_active, cold ? 0 : removed, K.max_iter, tol, lane, r);
        pstatus = cold ? (r.status == 0 ? 5 : r.status) : r.status;
        if (cold || !((pstatus == 1 || pstatus == 2) && K.cold_restart)) break;
        __syncwarp();
      }
      starting = false;
      removed = n_first;
      const double x0 = bcast(Vk, 0), xn = bcast(Vk, N);
      int rc = 0;
      if (isnan(x0) || isnan(xn) || isinf(x0) || isinf(xn)) rc = -1;   // PLDPSolver.cpp:955-964
      {
        // keep the rows whose multiplier is negative (:909-920) and store the ZMP solution (:1009-1032)
        const unsigned keep = __ballot_sync(0xffffffffu, lane < r.kproj && r.v2 < 0.0);
        __syncwarp();
        if (lane < r.kproj && r.v2 < 0.0) w.prev_active[__popc(keep & ((1u << lane) - 1u))] = w.pw.active[lane];
        n_prev = __popc(keep);
        double z = 0.0;
#pragma unroll 2
        for (int j = 0; j < N; ++j) z = add(z, mul(C.Pu[j * N + ii], bcast(Vk, j + N * ax)));
#pragma unroll
        for (int j = 0; j < 3; ++j) z = add(z, mul(C.Px[ii * 3 + j], w.xk[3 * ax + j]));
        __syncwarp();
        w.pw.prev_zmp[lane] = z;
      }
      // NewX = iLQ^T X: entries 0 and N (:1382-1400)
      double jx = 0.0, jy = 0.0;
#pragma unroll 2
      for (int j = 0; j < N; ++j) {
        const double vx = bcast(Vk, j), vy = bcast(Vk, j + N);
        jx += K.iLQc0[j] * vx;
        jy += K.iLQc0[j] * vy;
      }
      if (per && li < per_cap) {
        wg_dimitrov_period &o = per[li];
        if (lane == 0) {
          o.t_start = ST;
          o.xk[0] = cx0; o.xk[1] = cx1; o.xk[2] = cx2; o.xk[3] = cy0; o.xk[4] = cy1; o.xk[5] = cy2;
          o.jerk_x = jx; o.jerk_y = jy;
          o.m = m; o.n_first = n_first; o.rc = rc; o.status = pstatus; o.iterations = r.it; o.n_active = r.k;
        }
        o.active[lane] = lane < r.k ? w.pw.active[lane] : -1;
      }
      if (rc != 0 || (pstatus != 0 && pstatus != 5)) { wstatus = 1; ++li; break; }   // IFAIL: the reference returns -1
      // ---- LinearizedInvertedPendulum2D::Interpolation (:157-227): interval + 1 samples
      const long cur = li * K.interval;
      const int loop_end = (int)min((long)K.interval, (long)n - 1 - cur);
      if (lane <= loop_end) {
        const double s = (lane + 1) * Ts;
        const double c0 = cx0 + s * cx1 + 0.5 * s * s * cx2 + s * s * s * jx / 6.0;
        const double c1 = cx1 + s * cx2 + 0.5 * s * s * jx;
        const double c2 = cx2 + s * jx;
        const double d0 = cy0 + s * cy1 + 0.5 * s * s * cy2 + s * s * s * jy / 6.0;
        const double d1 = cy1 + s * cy2 + 0.5 * s * s * jy;
        const double d2 = cy2 + s * jy;
        const double C2 = -K.zc / 9.81;
        const size_t g = (size_t)(s0 + cur + lane);
        if (com) {
          double2 *cp = reinterpret_cast<double2 *>(com + 6 * g);
          cp[0] = make_double2(c0, c1); cp[1] = make_double2(c2, d0); cp[2] = make_double2(d1, d2);
        }
        if (zmp) *reinterpret_cast<double2 *>(zmp + 2 * g) = make_double2(1.0 * c0 + 0.0 * c1 + C2 * c2, 1.0 * d0 + 0.0 * d1 + C2 * d2);
      }
      // ---- OneIteration (:230-264): x = A x + B u
      {
        const double A01 = T, A02 = T * T / 2.0, A12 = T, B0 = T * T * T / 6.0, B1 = T * T / 2.0, B2 = T;
        const double nx0 = ((1.0 * cx0 + A01 * cx1) + A02 * cx2) + jx * B0;
        const double nx1 = ((0.0 * cx0 + 1.0 * cx1) + A12 * cx2) + jx * B1;
        const double nx2 = ((0.0 * cx0 + 0.0 * cx1) + 1.0 * cx2) + jx * B2;
        const double ny0 = ((1.0 * cy0 + A01 * cy1) + A02 * cy2) + jy * B0;
        const double ny1 = ((0.0 * cy0 + 1.0 * cy1) + A12 * cy2) + jy * B1;
        const double ny2 = ((0.0 * cy0 + 0.0 * cy1) + 1.0 * cy2) + jy * B2;
        cx0 = nx0; cx1 = nx1; cx2 = nx2; cy0 = ny0; cy1 = ny1; cy2 = ny2;
      }
      __syncwarp();
    }
    if (lane == 0) {
      if (status_out) status_out[b] = wstatus;
      if (done_out) done_out[b] = (int)li;
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Host: the constants of InitConstants()
// ---------------------------------------------------------------------------------------------------------------
// general inverse by Gauss-Jordan with partial pivoting (the reference calls MAL_INVERSE = LAPACK; 16 x 16, cond ~ 165)
void host_invert(int n, const double *A, double *inv)
{
  std::vector<double> M(A, A + n * n);
  for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) inv[i * n + j] = (i == j) ? 1.0 : 0.0;
  for (int c = 0; c < n; ++c) {
    int p = c;
    for (int r = c + 1; r < n; ++r) if (std::fabs(M[r * n + c]) > std::fabs(M[p * n + c])) p = r;
    if (p != c) for (int j = 0; j < n; ++j) { std::swap(M[p * n + j], M[c * n + j]); std::swap(inv[p * n + j], inv[c * n + j]); }
    const double d = M[c * n + c];
    for (int j = 0; j < n; ++j) { M[c * n + j] /= d; inv[c * n + j] /= d; }
    for (int r = 0; r < n; ++r) {
      if (r == c) continue;
      const double f = M[r * n + c];
      if (f == 0.0) continue;
      for (int j = 0; j < n; ++j) { M[r * n + j] -= f * M[c * n + j]; inv[r * n + j] -= f * inv[c * n + j]; }
    }
  }
}

int make_constants(const wg_dimitrov_params &p, DimHost *H)
{
  constexpr int N = DM_N;
  const double T = p.T, zc = p.com_height, alpha = p.alpha, beta = p.beta;
  if (!(T > 0) || !(p.sampling_period > 0) || !(zc > 0)) return WG_ERR_INVALID;
  std::vector<double> PPu(N * N, 0.0), VPu(N * N, 0.0), PPx(N * 3), VPx(N * 3);
  // InitializeMatrixPbConstants (:158-246)
  for (int i = 0; i < N; ++i) {
    VPx[i * 3 + 0] = 0.0; VPx[i * 3 + 1] = 1.0; VPx[i * 3 + 2] = (i + 1) * T;
    PPx[i * 3 + 0] = 1.0; PPx[i * 3 + 1] = (i + 1) * T; PPx[i * 3 + 2] = (i + 1) * (i + 1) * T * T * 0.5;
    for (int j = 0; j <= i; ++j) {
      VPu[i * N + j] = (2 * (i - j) + 1) * T * T * 0.5;
      PPu[i * N + j] = (1 + 3 * (i - j) + 3 * (i - j) * (i - j)) * T * T * T / 6.0;
    }
    H->h.Px[i * 3 + 0] = 1.0;
    H->h.Px[i * 3 + 1] = (double)(1.0 + i) * T;
    H->h.Px[i * 3 + 2] = (i + 1.0) * (i + 1.0) * T * T * 0.5 - zc / 9.81;
  }
  // BuildingConstantPartOfTheObjectiveFunction (:512-614): OptA = I + beta PPu^T PPu + alpha VPu^T (sic); the Cholesky
  // factorisation of its upper-left block reads the lower triangle only (OptCholesky.cpp:225-259)
  std::vector<double> Q(N * N), L(N * N, 0.0);
  double *iLQ = H->iLQ;
  std::fill(iLQ, iLQ + N * N, 0.0);
  for (int i = 0; i < N; ++i)
    for (int j = 0; j < N; ++j) {
      double t = 0.0;
      for (int k = 0; k < N; ++k) t += PPu[k * N + i] * PPu[k * N + j];
      Q[i * N + j] = ((i == j ? 1.0 : 0.0) + beta * t) + alpha * VPu[j * N + i];
    }
  for (int i = 0; i < N; ++i)
    for (int j = 0; j <= i; ++j) {
      double r = Q[i * N + j];
      for (int k = 0; k < j; ++k) r = r - L[i * N + k] * L[j * N + k];
      if (j != i) L[i * N + j] = r / L[j * N + j];
      else { if (!(r > 0)) return WG_ERR_INVALID; L[i * N + j] = std::sqrt(r); }
    }
  // ComputeInverseCholeskyNormal (OptCholesky.cpp:261-302)
  for (int lj = N - 1; lj >= 0; --lj) {
    const double inv = 1 / L[lj * N + lj];
    iLQ[lj * N + lj] = inv;
    for (int li = lj + 1; li < N; ++li) {
      double r = 0.0;
      for (int lk = lj + 1; lk < N; ++lk) r = r + iLQ[li * N + lk] * L[lk * N + lj];
      iLQ[li * N + lj] = -inv * r;
    }
  }
  std::vector<double> B0(N * 3), C0(N * N), PuT(N * N, 0.0);
  for (int i = 0; i < N; ++i) {
    for (int j = 0; j < 3; ++j) {
      double tv = 0.0, tp = 0.0;
      for (int k = 0; k < N; ++k) { tv += VPu[k * N + i] * VPx[k * 3 + j]; tp += PPu[k * N + i] * PPx[k * 3 + j]; }
      B0[i * 3 + j] = alpha * tv + beta * tp;
    }
    for (int j = 0; j < N; ++j) C0[i * N + j] = beta * PPu[j * N + i];
    // BuildingConstantPartOfConstraintMatrices (:616-680): Pu' then m_Pu = iLQ Pu'
    for (int k = 0; k <= i; ++k)
      PuT[k * N + i] = ((1 + 3 * (i - k) + 3 * (i - k) * (i - k)) * T * T * T / 6.0 - T * zc / 9.81);
  }
  for (int i = 0; i < N; ++i) {
    for (int j = 0; j < 3; ++j) { double t = 0.0; for (int k = 0; k < N; ++k) t += iLQ[i * N + k] * B0[k * 3 + j]; H->h.OptB[i * 3 + j] = t; }
    for (int j = 0; j < N; ++j) {
      double t = 0.0, u = 0.0;
      for (int k = 0; k < N; ++k) { t += iLQ[i * N + k] * C0[k * N + j]; u += iLQ[i * N + k] * PuT[k * N + j]; }
      H->h.OptC[i * N + j] = t;
      H->h.Pu[i * N + j] = u;
    }
    H->h.iLQc0[i] = iLQ[i * N + 0];
  }
  host_invert(N, H->h.Pu, H->iPu);
  H->h.T = T; H->h.Ts = p.sampling_period; H->h.zc = zc;
  // BuildLinearConstraintInequalities (:283-292): half sizes, then the margins
  double hw = p.sole_length, hh = p.sole_width;
  hw *= 0.5; hh *= 0.5;
  hh -= p.constraint_y;
  hw -= p.constraint_x;
  H->h.hw = hw; H->h.hh = hh;
  H->h.horizon = (unsigned)N * T;
  H->h.interval = (int)(T / p.sampling_period);
  H->h.max_iter = p.max_iterations > 0 ? p.max_iterations : 4 * PLDP_KMAX;
  H->h.cold_restart = p.cold_restart;
  H->h.merge_rows = p.merge_duplicate_rows;
  if (H->h.interval < 1 || H->h.interval > 31) return WG_ERR_INVALID;   // interval + 1 samples = one per lane
  return WG_OK;
}

// the accumulated clock of ZMPDiscretization (m_CurrentTime += m_SamplingPeriod per sample) for at least n samples
int ensure_clock(wg_ctx *ctx, DimHost *H, size_t n)
{
  if (H->time_h.size() >= n && H->d_time) return WG_OK;
  size_t cap = std::max<size_t>(n, 2 * H->time_h.size());
  cap = std::max<size_t>(cap, 4096);
  H->time_h.resize(cap);
  double t = 0.0;
  for (size_t i = 0; i < cap; ++i) { H->time_h[i] = t; t += H->par.sampling_period; }
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  cudaFree(H->d_time);
  H->d_time = nullptr;
  WG_CUDA(ctx, cudaMalloc(&H->d_time, sizeof(double) * cap));
  WG_CUDA(ctx, cudaMemcpy(H->d_time, H->time_h.data(), sizeof(double) * cap, cudaMemcpyHostToDevice));
  return WG_OK;
}

int64_t period_count_of(const wg_dimitrov_params &p, int64_t n)
{
  if (n < 1) return 0;
  double t = 0.0;
  for (int64_t i = 1; i < n; ++i) t += p.sampling_period;
  const double horizon = (unsigned)DM_N * p.T;
  int64_t c = 0;
  for (double st = 0.0; st < t - horizon; st += p.T) ++c;
  return c;
}

int launch_fcals(wg_ctx *ctx, DimHost *H, int B, const int64_t *d_samp_off, const wg_foot_sample *left,
                 const wg_foot_sample *right, const int32_t *types, const int64_t *d_lci_off, wg_lci *lci, int32_t *n_lci)
{
  const int grid = std::max(1, std::min((B + FC_WARPS - 1) / FC_WARPS, ctx->sm_count * 8));
  wg_prof_start(ctx, WG_K_FCALS);
  fcals_kernel<<<grid, FC_WARPS * 32, 0, ctx->stream>>>(B, H->d, d_samp_off, left, right, types, H->d_time, d_lci_off, lci, n_lci);
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  return WG_OK;
}

}  // namespace

void wg_dimitrov_release(wg_ctx *ctx)
{
  if (!ctx->dimitrov) return;
  DimHost *p = static_cast<DimHost *>(ctx->dimitrov);
  cudaFree(p->d);
  cudaFree(p->d_time);
  for (void *b : p->buf) cudaFree(b);
  delete p;
  ctx->dimitrov = nullptr;
}

// Used by wieber.cu: BuildLinearConstraintInequalities of ZMPQPWithConstraint (ZMPQPWithConstraint.cpp:229-502) is the same
// scan with the same half-plane arithmetic as FootConstraintsAsLinearSystem's, with its own sole size and security margins.
// d_clock_out: the accumulated 5 ms clock table on the device (>= max_n entries).
extern "C" int wgi_fcals_launch(wg_ctx *ctx, int B, const int64_t *d_samp_off, const wg_foot_sample *left,
                                const wg_foot_sample *right, const int32_t *types, const int64_t *d_lci_off, wg_lci *lci,
                                int32_t *n_lci, double hw, double hh, double sampling_period, size_t max_n,
                                const double **d_clock_out)
{
  DimHost *H = dim_of(ctx);
  if (H->ready && std::fabs(H->par.sampling_period - sampling_period) > 1e-15)
    return wg_fail(ctx, WG_ERR_INVALID, "sampling period differs from the one given to wg_dimitrov_set_params");
  if (!H->ready) H->par.sampling_period = sampling_period;     // clock table only
  int rc = ensure_clock(ctx, H, max_n);
  if (rc != WG_OK) return rc;
  if ((rc = wgi_grow_scratch(ctx, &H->buf[13], &H->cap[13], sizeof(DimConsts))) != WG_OK) return rc;
  DimConsts alt;
  std::memset(&alt, 0, sizeof alt);
  alt.hw = hw; alt.hh = hh; alt.merge_rows = 0;
  WG_CUDA(ctx, cudaMemcpyAsync(H->buf[13], &alt, sizeof alt, cudaMemcpyHostToDevice, ctx->stream));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));            // `alt` is a stack temporary
  const int grid = std::max(1, std::min((B + FC_WARPS - 1) / FC_WARPS, ctx->sm_count * 8));
  wg_prof_start(ctx, WG_K_FCALS);
  fcals_kernel<<<grid, FC_WARPS * 32, 0, ctx->stream>>>(B, static_cast<const DimConsts *>(H->buf[13]), d_samp_off, left, right,
                                                           types, H->d_time, d_lci_off, lci, n_lci);
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  if (d_clock_out) *d_clock_out = H->d_time;
  return WG_OK;
}

extern "C" {

void wg_dimitrov_default_params(wg_dimitrov_params *p)
{
  if (!p) return;
  std::memset(p, 0, sizeof *p);
  p->T = 0.1;                  // m_QP_T, ZMPConstrainedQPFastFormulation.cpp:83
  p->sampling_period = 0.005;  // :86
  p->com_height = 0.80;        // :88
  p->alpha = 200.0;            // :95
  p->beta = 1000.0;            // :96
  p->constraint_x = 0.04;      // :79-80
  p->constraint_y = 0.04;
  p->sole_length = 0.25;       // HRP-2 test robot (SURVEY 8c)
  p->sole_width = 0.14;
  p->max_iterations = 0;
  p->cold_restart = 0;
}

int wg_dimitrov_set_params(wg_ctx *ctx, const wg_dimitrov_params *p, double *iPu, double *Px, double *Pu, double *iLQ,
                           double *OptB, double *OptC)
{
  if (!ctx || !p) return WG_ERR_INVALID;
  wg_device_guard guard(ctx->device);
  DimHost *H = dim_of(ctx);
  DimHost tmp;
  tmp.par = *p;
  int rc = make_constants(*p, &tmp);
  if (rc != WG_OK) return wg_fail(ctx, rc, "wg_dimitrov_params out of range");
  const bool new_clock = !H->ready || H->par.sampling_period != p->sampling_period || H->par.T != p->T;
  H->par = *p;
  H->h = tmp.h;
  std::memcpy(H->iPu, tmp.iPu, sizeof H->iPu);
  std::memcpy(H->iLQ, tmp.iLQ, sizeof H->iLQ);
  if (new_clock) { H->time_h.clear(); H->period_cache.clear(); }
  if ((rc = wg_pldp_set_constants(ctx, DM_N, H->iPu, H->h.Px, H->h.Pu)) != WG_OK) return rc;
  if (!H->d) WG_CUDA(ctx, cudaMalloc(&H->d, sizeof(DimConsts)));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  WG_CUDA(ctx, cudaMemcpy(H->d, &H->h, sizeof(DimConsts), cudaMemcpyHostToDevice));
  H->ready = true;
  constexpr int N = DM_N;
  if (iPu) std::memcpy(iPu, H->iPu, sizeof(double) * N * N);
  if (Px) std::memcpy(Px, H->h.Px, sizeof(double) * N * 3);
  if (Pu) std::memcpy(Pu, H->h.Pu, sizeof(double) * N * N);
  if (iLQ) std::memcpy(iLQ, H->iLQ, sizeof(double) * N * N);
  if (OptB) std::memcpy(OptB, H->h.OptB, sizeof(double) * N * 3);
  if (OptC) std::memcpy(OptC, H->h.OptC, sizeof(double) * N * N);
  return WG_OK;
}

int64_t wg_dimitrov_period_count(const wg_dimitrov_params *p, int64_t n_samples)
{
  if (!p || !(p->T > 0) || !(p->sampling_period > 0)) return -1;
  return period_count_of(*p, n_samples);
}

int wg_convex_hull_batch(wg_ctx *ctx, int mem, int B, int n, const double *xy, double *hull_xy, int32_t *counts)
{
  if (!ctx || B < 0 || n < 1 || n > 8 || !xy || !hull_xy || !counts) return WG_ERR_INVALID;
  if (B == 0) return WG_OK;
  wg_device_guard guard(ctx->device);
  DimHost *H = dim_of(ctx);
  const double *dxy = xy; double *dh = hull_xy; int32_t *dc = counts;
  const size_t nb = (size_t)B;
  if (mem == WG_MEM_HOST) {
    int rc;
    if ((rc = wgi_grow_scratch(ctx, &H->buf[0], &H->cap[0], sizeof(double) * 2 * n * nb)) != WG_OK) return rc;
    if ((rc = wgi_grow_scratch(ctx, &H->buf[1], &H->cap[1], sizeof(double) * 16 * nb)) != WG_OK) return rc;
    if ((rc = wgi_grow_scratch(ctx, &H->buf[2], &H->cap[2], sizeof(int32_t) * nb)) != WG_OK) return rc;
    WG_CUDA(ctx, cudaMemcpyAsync(H->buf[0], xy, sizeof(double) * 2 * n * nb, cudaMemcpyHostToDevice, ctx->stream));
    dxy = static_cast<const double *>(H->buf[0]); dh = static_cast<double *>(H->buf[1]); dc = static_cast<int32_t *>(H->buf[2]);
  } else if (mem != WG_MEM_DEVICE) return WG_ERR_INVALID;
  wg_prof_start(ctx, WG_K_FCALS);
  convex_hull_kernel<<<(B + 127) / 128, 128, 0, ctx->stream>>>(B, n, dxy, dh, dc);
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  if (mem == WG_MEM_HOST) {
    WG_CUDA(ctx, cudaMemcpyAsync(hull_xy, dh, sizeof(double) * 16 * nb, cudaMemcpyDeviceToHost, ctx->stream));
    WG_CUDA(ctx, cudaMemcpyAsync(counts, dc, sizeof(int32_t) * nb, cudaMemcpyDeviceToHost, ctx->stream));
    WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return WG_OK;
}

int wg_fcals_build_batch(wg_ctx *ctx, int mem, int B, const int64_t *sample_offsets, const wg_foot_sample *left,
                         const wg_foot_sample *right, const int32_t *step_type, const int64_t *lci_offsets,
                         wg_lci *lci, int32_t *n_lci)
{
  if (!ctx || B < 0 || !sample_offsets || !left || !right || !step_type || !lci_offsets || !lci || !n_lci) return WG_ERR_INVALID;
  DimHost *H = dim_of(ctx);
  if (!H->ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_dimitrov_set_params not called");
  if (B == 0) return WG_OK;
  wg_device_guard guard(ctx->device);
  int64_t max_n = 0;
  for (int b = 0; b < B; ++b) {
    const int64_t n = sample_offsets[b + 1] - sample_offsets[b];
    if (n < 1 || lci_offsets[b + 1] < lci_offsets[b]) return wg_fail(ctx, WG_ERR_INVALID, "wg_fcals_build_batch: empty walk or negative capacity");
    max_n = std::max(max_n, n);
  }
  int rc;
  if ((rc = ensure_clock(ctx, H, (size_t)max_n)) != WG_OK) return rc;
  const size_t ns = (size_t)sample_offsets[B], nl = (size_t)lci_offsets[B], nb = (size_t)B;
  if ((rc = wgi_grow_scratch(ctx, &H->buf[3], &H->cap[3], sizeof(int64_t) * 2 * (nb + 1))) != WG_OK) return rc;
  int64_t *d_so = static_cast<int64_t *>(H->buf[3]), *d_lo = d_so + (nb + 1);
  WG_CUDA(ctx, cudaMemcpyAsync(d_so, sample_offsets, sizeof(int64_t) * (nb + 1), cudaMemcpyHostToDevice, ctx->stream));
  WG_CUDA(ctx, cudaMemcpyAsync(d_lo, lci_offsets, sizeof(int64_t) * (nb + 1), cudaMemcpyHostToDevice, ctx->stream));
  const wg_foot_sample *dl = left, *dr = right; const int32_t *dt = step_type; wg_lci *dp = lci; int32_t *dn = n_lci;
  if (mem == WG_MEM_HOST) {
    if ((rc = wgi_grow_scratch(ctx, &H->buf[4], &H->cap[4], sizeof(wg_foot_sample) * ns)) != WG_OK) return rc;
    if ((rc = wgi_grow_scratch(ctx, &H->buf[5], &H->cap[5], sizeof(wg_foot_sample) * ns)) != WG_OK) return rc;
    if ((rc = wgi_grow_scratch(ctx, &H->buf[6], &H->cap[6], sizeof(int32_t) * 3 * ns)) != WG_OK) return rc;
    if ((rc = wgi_grow_scratch(ctx, &H->buf[7], &H->cap[7], sizeof(wg_lci) * std::max<size_t>(nl, 1))) != WG_OK) return rc;
    if ((rc = wgi_grow_scratch(ctx, &H->buf[8], &H->cap[8], sizeof(int32_t) * nb)) != WG_OK) return rc;
    WG_CUDA(ctx, cudaMemcpyAsync(H->buf[4], left, sizeof(wg_foot_sample) * ns, cudaMemcpyHostToDevice, ctx->stream));
    WG_CUDA(ctx, cudaMemcpyAsync(H->buf[5], right, sizeof(wg_foot_sample) * ns, cudaMemcpyHostToDevice, ctx->stream));
    WG_CUDA(ctx, cudaMemcpyAsync(H->buf[6], step_type, sizeof(int32_t) * 3 * ns, cudaMemcpyHostToDevice, ctx->stream));
    dl = static_cast<const wg_foot_sample *>(H->buf[4]); dr = static_cast<const wg_foot_sample *>(H->buf[5]);
    dt = static_cast<const int32_t *>(H->buf[6]); dp = static_cast<wg_lci *>(H->buf[7]); dn = static_cast<int32_t *>(H->buf[8]);
    WG_CUDA(ctx, cudaMemsetAsync(dp, 0, sizeof(wg_lci) * nl, ctx->stream));
  } else if (mem != WG_MEM_DEVICE) return WG_ERR_INVALID;
  if ((rc = launch_fcals(ctx, H, B, d_so, dl, dr, dt, d_lo, dp, dn)) != WG_OK) return rc;
  if (mem == WG_MEM_HOST) {
    WG_CUDA(ctx, cudaMemcpyAsync(lci, dp, sizeof(wg_lci) * nl, cudaMemcpyDeviceToHost, ctx->stream));
    WG_CUDA(ctx, cudaMemcpyAsync(n_lci, dn, sizeof(int32_t) * nb, cudaMemcpyDeviceToHost, ctx->stream));
    WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int b = 0; b < B; ++b)
      if (n_lci[b] < 0) return wg_fail(ctx, WG_ERR_INVALID, "wg_fcals_build_batch: a walk has more support polygons than its capacity");
  }
  return WG_OK;
}

int wg_dimitrov_run_batch(wg_ctx *ctx, wg_kajita_plan *plan, int mem, double *com_out, double *zmp_out,
                          wg_foot_sample *left, wg_foot_sample *right, const int64_t *period_offsets,
                          wg_dimitrov_period *periods, int32_t *status, int32_t *periods_done)
{
  if (!ctx || !plan) return WG_ERR_INVALID;
  if (mem != WG_MEM_HOST && mem != WG_MEM_DEVICE) return WG_ERR_INVALID;
  if (periods && !period_offsets) return WG_ERR_INVALID;
  DimHost *H = dim_of(ctx);
  if (!H->ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_dimitrov_set_params not called");
  const PldpConsts *dC = static_cast<const PldpConsts *>(wgi_pldp_device_consts(ctx));
  if (!dC) return wg_fail(ctx, WG_ERR_NOT_READY, "PLDP constants missing");
  wg_device_guard guard(ctx->device);
  const bool host = mem == WG_MEM_HOST;
  // ---- GetZMPDiscretization: feet + discretised ZMP reference on the device
  double *d_zmp = host ? nullptr : zmp_out;
  wg_foot_sample *d_left = host ? nullptr : left, *d_right = host ? nullptr : right;
  int32_t *d_types = nullptr;
  wgi_kajita_view V;
  int rc = wgi_kajita_discretize_device(ctx, plan, &d_zmp, &d_left, &d_right, &d_types, &V);
  if (rc != WG_OK) return rc;
  if (std::fabs(V.sampling_period - H->par.sampling_period) > 1e-15)
    return wg_fail(ctx, WG_ERR_INVALID, "sampling period of the plan differs from wg_dimitrov_params");
  const int B = V.B;
  const size_t nb = (size_t)B, ns = (size_t)V.samp_off[B];
  int64_t max_n = 0;
  std::vector<int64_t> lci_off(B + 1), per_off;
  lci_off[0] = 0;
  for (int b = 0; b < B; ++b) {
    const int64_t n = V.samp_off[b + 1] - V.samp_off[b];
    max_n = std::max(max_n, n);
    // per step: one single-support polygon and one double-support polygon (the swing foot touches down before the
    // single-support phase ends), plus the opening phase and slack
    lci_off[b + 1] = lci_off[b] + 2 * (V.step_off[b + 1] - V.step_off[b]) + 6;
  }
  if (periods) {
    for (int b = 0; b < B; ++b) {
      const int64_t n = V.samp_off[b + 1] - V.samp_off[b];
      auto itc = H->period_cache.find(n);
      const int64_t need = itc != H->period_cache.end() ? itc->second : (H->period_cache[n] = period_count_of(H->par, n));
      if (period_offsets[b + 1] - period_offsets[b] < need)
        return wg_fail(ctx, WG_ERR_INVALID, "wg_dimitrov_run_batch: period_offsets leave too few records for a walk");
    }
  }
  if ((rc = ensure_clock(ctx, H, (size_t)max_n)) != WG_OK) return rc;
  const size_t nl = (size_t)lci_off[B];
  const size_t npr = periods ? (size_t)period_offsets[B] : 0;
  if ((rc = wgi_grow_scratch(ctx, &H->buf[3], &H->cap[3], sizeof(int64_t) * 2 * (nb + 1))) != WG_OK) return rc;
  if ((rc = wgi_grow_scratch(ctx, &H->buf[7], &H->cap[7], sizeof(wg_lci) * nl)) != WG_OK) return rc;
  if ((rc = wgi_grow_scratch(ctx, &H->buf[8], &H->cap[8], sizeof(int32_t) * 3 * nb)) != WG_OK) return rc;
  int64_t *d_lo = static_cast<int64_t *>(H->buf[3]), *d_po = d_lo + (nb + 1);
  wg_lci *d_lci = static_cast<wg_lci *>(H->buf[7]);
  int32_t *d_nlci = static_cast<int32_t *>(H->buf[8]), *d_status = d_nlci + nb, *d_done = d_status + nb;
  WG_CUDA(ctx, cudaMemcpyAsync(d_lo, lci_off.data(), sizeof(int64_t) * (nb + 1), cudaMemcpyHostToDevice, ctx->stream));
  if (periods) WG_CUDA(ctx, cudaMemcpyAsync(d_po, period_offsets, sizeof(int64_t) * (nb + 1), cudaMemcpyHostToDevice, ctx->stream));
  double *d_com = com_out;
  wg_dimitrov_period *d_per = periods;
  int32_t *d_st = status ? status : d_status, *d_dn = periods_done ? periods_done : d_done;
  if (host) {
    d_com = nullptr;
    if (com_out) {
      if ((rc = wgi_grow_scratch(ctx, &H->buf[9], &H->cap[9], sizeof(double) * 6 * ns)) != WG_OK) return rc;
      d_com = static_cast<double *>(H->buf[9]);
    }
    if (periods) {
      if ((rc = wgi_grow_scratch(ctx, &H->buf[10], &H->cap[10], sizeof(wg_dimitrov_period) * std::max<size_t>(npr, 1))) != WG_OK)
        return rc;
      d_per = static_cast<wg_dimitrov_period *>(H->buf[10]);
    }
    d_st = d_status; d_dn = d_done;
  }
  if (d_com) WG_CUDA(ctx, cudaMemsetAsync(d_com, 0, sizeof(double) * 6 * ns, ctx->stream));
  if (d_per) WG_CUDA(ctx, cudaMemsetAsync(d_per, 0, sizeof(wg_dimitrov_period) * npr, ctx->stream));
  // ---- FootConstraintsAsLinearSystem
  if ((rc = launch_fcals(ctx, H, B, V.d_samp_off, d_left, d_right, d_types, d_lo, d_lci, d_nlci)) != WG_OK) return rc;
  // ---- the loop
  const int grid = std::max(1, std::min((B + DM_WARPS - 1) / DM_WARPS, ctx->sm_count * 3));
  if ((rc = wgi_grow_scratch(ctx, &H->buf[11], &H->cap[11], 64)) != WG_OK) return rc;
  int *d_next = static_cast<int *>(H->buf[11]);
  WG_CUDA(ctx, cudaMemsetAsync(d_next, 0, sizeof(int), ctx->stream));
  // longest-processing-time-first order (the sample count is a faithful proxy of the period count); uploaded once per plan
  const size_t order_cap = H->cap[12];
  if ((rc = wgi_grow_scratch(ctx, &H->buf[12], &H->cap[12], sizeof(int) * nb)) != WG_OK) return rc;
  if (H->cap[12] != order_cap) H->order_plan = nullptr;   // a new buffer holds no order yet
  if (H->order_plan != plan || H->order_B != B || H->order_total != (int64_t)ns) {
    std::vector<int> order(B);
    for (int b = 0; b < B; ++b) order[b] = b;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
      return V.samp_off[a + 1] - V.samp_off[a] > V.samp_off[b + 1] - V.samp_off[b];
    });
    WG_CUDA(ctx, cudaMemcpyAsync(H->buf[12], order.data(), sizeof(int) * nb, cudaMemcpyHostToDevice, ctx->stream));
    WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // `order` is a pageable temporary
    H->order_plan = plan; H->order_B = B; H->order_total = (int64_t)ns;
  }
  wg_prof_start(ctx, WG_K_DIMITROV);
  dimitrov_kernel<<<grid, DM_WARPS * 32, 0, ctx->stream>>>(B, H->d, dC, V.d_samp_off, H->d_time, d_lo, d_lci, d_nlci,
                                                              V.d_zd_status, d_com, zmp_out ? d_zmp : nullptr, d_po, d_per,
                                                              d_st, d_dn, d_next, static_cast<const int *>(H->buf[12]));
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  if (host) {
    if (com_out) WG_CUDA(ctx, cudaMemcpyAsync(com_out, d_com, sizeof(double) * 6 * ns, cudaMemcpyDeviceToHost, ctx->stream));
    if (zmp_out) WG_CUDA(ctx, cudaMemcpyAsync(zmp_out, d_zmp, sizeof(double) * 2 * ns, cudaMemcpyDeviceToHost, ctx->stream));
    if (left) WG_CUDA(ctx, cudaMemcpyAsync(left, d_left, sizeof(wg_foot_sample) * ns, cudaMemcpyDeviceToHost, ctx->stream));
    if (right) WG_CUDA(ctx, cudaMemcpyAsync(right, d_right, sizeof(wg_foot_sample) * ns, cudaMemcpyDeviceToHost, ctx->stream));
    if (periods) WG_CUDA(ctx, cudaMemcpyAsync(periods, d_per, sizeof(wg_dimitrov_period) * npr, cudaMemcpyDeviceToHost, ctx->stream));
    if (status) WG_CUDA(ctx, cudaMemcpyAsync(status, d_status, sizeof(int32_t) * nb, cudaMemcpyDeviceToHost, ctx->stream));
    if (periods_done) WG_CUDA(ctx, cudaMemcpyAsync(periods_done, d_done, sizeof(int32_t) * nb, cudaMemcpyDeviceToHost, ctx->stream));
    WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return WG_OK;
}

}  // extern "C"
