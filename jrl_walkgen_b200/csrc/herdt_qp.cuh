// herdt_qp.cuh - warp-per-instance Herdt2010 QP assembly + dual active-set solve (device code).
//
// Replaces, for one instance per warp, GeneratorVelRef::update_problem / build_constraints
// (src/ZMPRefTrajectoryGeneration/generator-vel-ref.cpp:285-674), RelativeFeetInequalities
// (src/Mathematics/relative-feet-inequalities.cpp:89-319), QPProblem::solve (qp-problem.cpp:246-407) and
// ql0001_/ql0002_ (src/Mathematics/qld.cpp:378-2090).
//
// B200-first formulation (DESIGN.md "Herdt QP kernel").  The reference assembles a dense 36x36 Hessian and a
// 75x36 constraint matrix and hands them to QLD, which factorises the Hessian for every solve.  Here nothing
// dense is ever assembled.  The unknowns are x = [jx(16) jy(16) fx(ns) fy(ns)] and
//   * the Hessian is block-diagonal over the two axes with the SAME block  Qx = [[Qc, Cx],[Cx', E]],
//     Qc = a I + b Uv'Uv + c Uz'Uz constant, Cx = -c Uz'V, E = c V'V diagonal (V = step-selection matrix);
//   * every inequality row has the form  a_k * PX[kappa] + b_k * PY[kappa] + d_k >= 0  where the "points"
//     P[kappa] (16 CoP-minus-support offsets + ns relative foot placements) are affine in x with the same
//     coefficient vector theta_kappa for both axes.
// Hence the Gram matrix of the rows in the metric of H^-1 - the only thing a dual active-set method needs - is
//   N_k' H^-1 N_l = (a_k a_l + b_k b_l) * Gamma(kappa_k, kappa_l),   Gamma = theta' Qx^-1 theta   (18 x 18),
// with Gamma = G + t' S^-1 t, G = Uz Qc^-1 Uz' a constant 16x16 matrix and S the ns x ns Schur complement of
// the foot block.  The Goldfarb-Idnani iteration then runs entirely in "point space": the primal iterate is
// the 2 x 18 point coordinates, the dual iterate the multipliers of the <= 32 active rows, and the only
// factorisation is the inverse Cholesky factor T of the active Gram matrix, grown by one row per added
// constraint and shrunk by Givens rotations per dropped one (the batched analogue of OptCholesky's
// row-incremental update, src/Mathematics/OptCholesky.cpp:123-223).  Everything lives in shared memory.
#pragma once
#include "wg_common.h"

namespace herdt {

constexpr int N = WG_HERDT_N;        // 16
constexpr int NPTS = N + 2;          // 18 points
constexpr int MAXM = 4 * N + 10;     // 74 real rows
constexpr int QMAX = 40;             // active-set capacity (> n = 36 independent rows; two slots per lane)
constexpr int TRI = QMAX * (QMAX + 1) / 2;

// Constants of one (T, h, weights) parameter set, computed once on the host in extended precision.
struct Consts {
  double K1[N][N];    // Qc^-1 Uz'
  double G[N][N];     // Uz Qc^-1 Uz'
  double K3[N][N];    // Qc^-1 Uv'
  double K4[N][3];    // K3 Sv
  double Sz[N][3];    // CoP state matrix (rigid-body-system.cpp:425-431)
  double uz[N];       // Uz is Toeplitz: Uz(i,j) = uz[i-j], j <= i
  double uz2[N];      // squared Euclidean norm of row i of Uz
  double Qc[N][N];    // kept for residual checks
  wg_herdt_params P;
};

// Per-warp shared-memory workspace.
struct Work {
  wg_herdt_qp_input in;            // 784 B
  double PX[NPTS + 2], PY[NPTS + 2];
  double Gam[NPTS][NPTS];
  double a[MAXM + 2], b[MAXM + 2], d[MAXM + 2], inrm[MAXM + 2];
  double u[QMAX], gv[QMAX], w[QMAX], r[QMAX], ca[QMAX + 1], cb[QMAX + 1];
  double theta[NPTS][2], sigma[NPTS][2];
  double g[2][N], j0[2][N], Z[2][N], jr[2][N];
  double f0[2][2], ff[2][2];
  double wpt[2][NPTS + 2];
  int W[QMAX], cpt[QMAX + 1];
};

__device__ __forceinline__ int tri(int i) { return (i * (i + 1)) >> 1; }
__device__ __forceinline__ int row_point(int k) { return k < 4 * N ? (k >> 2) : N + (k - 4 * N) / 5; }

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double half_sum(double v)  // sum over the 16 lanes of a half warp
{
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// argmin with deterministic tie-break (lower index wins)
__device__ __forceinline__ void warp_argmin(double &v, int &idx)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    double ov = __shfl_xor_sync(0xffffffffu, v, o);
    int oi = __shfl_xor_sync(0xffffffffu, idx, o);
    if (ov < v || (ov == v && oi < idx)) { v = ov; idx = oi; }
  }
}

// RelativeFeetInequalities::set_vertices + convex_hull_t::rotate + compute_linear_system for one hull
// (relative-feet-inequalities.cpp:186-234, 265-319; privatepgtypes.cpp:152-180).
static __device__ __noinline__ void hull_rows(const wg_herdt_params &P, int foot, int phase, double yaw, bool cop, int sign_foot,
                                 double *A, double *B, double *D)
{
  double X[5], Y[5];
  int nv;
  if (cop) {
    nv = 4;
    const double hw = P.cop_half_x, hh = P.cop_half_y, hhds = P.cop_half_y + P.ds_feet_distance * 0.5;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const double lx = (j < 2) ? 1.0 : -1.0;
      const double lyL = (j == 0 || j == 3) ? 1.0 : -1.0;
      X[j] = lx * hw;
      if (foot == WG_LEFT) Y[j] = (phase == WG_DS) ? lyL * hhds - P.ds_feet_distance * 0.5 : lyL * hh;
      else Y[j] = (phase == WG_DS) ? -lyL * hhds + P.ds_feet_distance * 0.5 : -lyL * hh;
    }
    X[4] = Y[4] = 0.0;
  } else {
    nv = 5;
#pragma unroll
    for (int j = 0; j < 5; ++j) { X[j] = P.foot_hull_x[j]; Y[j] = (foot == WG_LEFT) ? P.foot_hull_y[j] : -P.foot_hull_y[j]; }
  }
  double sn, cs;
  sincos(yaw, &sn, &cs);
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    const double xo = X[j], yo = Y[j];
    X[j] = xo * cs - yo * sn;
    Y[j] = xo * sn + yo * cs;
  }
  const double sg = (sign_foot == WG_LEFT) ? 1.0 : -1.0;
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    if (i < nv) {
      const int k = (i + 1 == nv) ? 0 : i + 1;
      const double dx = Y[i] - Y[k], dy = X[k] - X[i], dc = dx * X[i] + dy * Y[i];
      A[i] = sg * dx; B[i] = sg * dy; D[i] = sg * dc;
    }
  }
}

// Points from a primal iterate (jerks in jr[axis][16], foot placements in ff[axis][2]):
//   P[i]   = -(Uz j)_i + (V f)_i - (Sz c)_i + Vc_i      (generator-vel-ref.cpp:394-447, rows of the CoP constraints)
//   P[N+s] = -(Vf f)_s + Vcf_s                            (generator-vel-ref.cpp:450-474)
static __device__ __noinline__ void points_from_primal(Work &s, const Consts &C, const double (*jr)[N], const double (*ff)[2],
                                          int ns, const double Vf[2][2], const double Vcf[2][2], double *outX,
                                          double *outY, int lane)
{
  const int axis = lane >> 4, i = lane & 15;
  double acc = 0.0;
  for (int k = 0; k <= i; ++k) acc = fma(C.uz[i - k], jr[axis][k], acc);
  const int sn = s.in.sup_step[i + 1];
  const double sel = (sn > 0) ? ff[axis][sn - 1] : (axis ? s.in.sup_y[i + 1] : s.in.sup_x[i + 1]);
  const double p = -acc + sel - s.Z[axis][i];
  (axis ? outY : outX)[i] = p;
  if (i < ns) {
    double v = Vcf[axis][i];
    for (int r = 0; r < ns; ++r) v -= Vf[i][r] * ff[axis][r];
    (axis ? outY : outX)[N + i] = v;
  }
  __syncwarp();
}

struct Result {
  int n_vars, n_rows, fail, iterations;
};

// Optional per-instance side inputs / outputs of herdt_qp_kernel, addressed as base + b * stride bytes so that they can live
// inside larger records (the closed loop keeps the warm-start set inside wg_herdt_mpc_state).
struct LaunchOpts {
  const unsigned char *fire = nullptr;   size_t fire_stride = 0;     // int: 0 = skip instance b
  const unsigned char *guess = nullptr;  size_t guess_stride = 0;    // wg_herdt_active_set of an earlier solve
  unsigned char *active_out = nullptr;   size_t active_stride = 0;   // optimal active set (may alias guess)
  int age = 1;
};

// Drop active row l: rotate rows (l, r), r > l, of the inverse Cholesky factor T so that column l vanishes below row l, then
// delete row and column l (s.w holds the rotating copy of row l); W / cpt / u close the gap.  q is NOT decremented here.
static __device__ __noinline__ void drop_row(Work &s, double *__restrict__ T, int q, int l, int lane, unsigned &actbits)
{
  const int kl = s.W[l];
  if ((kl & 31) == lane) actbits &= ~(1u << (kl >> 5));
#pragma unroll 1
  for (int j = lane; j < q; j += 32) s.w[j] = (j <= l) ? T[tri(l) + j] : 0.0;
  __syncwarp();
#pragma unroll 1
  for (int r = l + 1; r < q; ++r) {
    const double *Tr = T + tri(r);
    const double p1 = s.w[l], p2 = Tr[l];
    const double ih = rsqrt(p1 * p1 + p2 * p2);
    const double c_ = p1 * ih, s_ = p2 * ih;
    __syncwarp();
    double *Tn = T + tri(r - 1);
#pragma unroll 1
    for (int j = lane; j <= r; j += 32) {
      const double x1 = s.w[j], x2 = Tr[j];
      s.w[j] = c_ * x1 + s_ * x2;
      const double nr = c_ * x2 - s_ * x1;
      if (j < l) Tn[j] = nr;
      else if (j > l) Tn[j - 1] = nr;
    }
    __syncwarp();
  }
#pragma unroll 1
  for (int base = 0; base < q; base += 32) {
    const int j = base + lane;
    const bool mv = (j > l && j < q);
    const int Wn = mv ? s.W[j] : 0, cn = mv ? s.cpt[j] : 0;
    const double un = mv ? s.u[j] : 0.0;
    __syncwarp();
    if (mv) { s.W[j - 1] = Wn; s.cpt[j - 1] = cn; s.u[j - 1] = un; }
    __syncwarp();
  }
}

// w = T gv and r = T' w for the current active set (gv in s.gv); returns this lane's share of |w|^2.
static __device__ __noinline__ double tri_products(Work &s, const double *__restrict__ T, int q, int lane)
{
  double wsq = 0.0;
#pragma unroll 1
  for (int j = lane; j < q; j += 32) {
    const double *Tr = T + tri(j);
    double w0 = 0.0, w1 = 0.0;
    int e = 0;
#pragma unroll 2
    for (; e + 1 <= j; e += 2) { w0 = fma(Tr[e], s.gv[e], w0); w1 = fma(Tr[e + 1], s.gv[e + 1], w1); }
    if (e <= j) w0 = fma(Tr[e], s.gv[e], w0);
    const double wv_ = w0 + w1;
    s.w[j] = wv_;
    wsq = fma(wv_, wv_, wsq);
  }
  __syncwarp();
#pragma unroll 1
  for (int j = lane; j < q; j += 32) {
    double r0 = 0.0, r1 = 0.0;
    int r = j;
#pragma unroll 2
    for (; r + 1 < q; r += 2) { r0 = fma(T[tri(r) + j], s.w[r], r0); r1 = fma(T[tri(r + 1) + j], s.w[r + 1], r1); }
    if (r < q) r0 = fma(T[tri(r) + j], s.w[r], r0);
    s.r[j] = r0 + r1;
  }
  __syncwarp();
  return wsq;
}

// Warm start of the dual active-set method from a guessed active set (the optimal set of the previous MPC period, shifted
// by the samples / steps that left the horizon).  A Goldfarb-Idnani iterate is any "S-pair": the minimiser on the active
// rows taken as equalities, with non-negative multipliers.  The guessed rows are taken all at once - T grows by one row per
// independent guess, no violation scan, no step, no ratio test -, the multipliers of the equality-constrained optimum are
// u = -(N' H^-1 N)^-1 s_W(P0) = -T'T s_W(P0), and guesses whose multiplier comes out negative are dropped one at a time
// (most negative first) until the pair is dual feasible.  The main loop then continues from that pair; it reaches the same
// unique optimum as the cold start (strictly convex QP), in a few iterations instead of ~25 when most of the guess is right.
static __device__ __noinline__ void warm_start(Work &s, double *__restrict__ T, int m, int npts, int lane,
                                               const wg_herdt_active_set *__restrict__ hint, int age, int &q,
                                               unsigned &actbits, int &iterations)
{
  const int nh = hint->n;
  if (nh <= 0 || nh > (int)sizeof(hint->rows) || age < 0) return;
  // where the previewed steps of this QP start, to map the foot rows of the guess (a step that starts at previewed sample pi
  // starts at pi - age one QP later; at pi = 1 the foot is down and no longer a variable, generator-vel-ref.cpp:106-128)
  int pi_new[2] = {0, 0};
  for (int k = N; k >= 1; --k) {
    const int sn = s.in.sup_step[k];
    if (sn == 1) pi_new[0] = k; else if (sn == 2) pi_new[1] = k;
  }
  int step_map[2];
#pragma unroll
  for (int o = 0; o < 2; ++o) {
    const int pio = hint->step_pi[o] - age;
    step_map[o] = (hint->step_pi[o] > 0 && pio > 0) ? (pio == pi_new[0] ? 0 : (pio == pi_new[1] ? 1 : -1)) : -1;
  }
#pragma unroll 1
  for (int t = 0; t < nh && q < QMAX - 4; ++t) {
    int p = hint->rows[t];
    if (p < 0) continue;
    if (p < 4 * N) { p -= 4 * age; if (p < 0) continue; }
    else {
      const int so = (p - 4 * N) / 5, e = (p - 4 * N) - 5 * so;
      if (so > 1 || step_map[so] < 0) continue;
      p = 4 * N + 5 * step_map[so] + e;
    }
    if (p >= m) continue;
    const unsigned ab = __shfl_sync(0xffffffffu, actbits, p & 31);
    if ((ab >> (p >> 5)) & 1u) continue;
    if (!(s.inrm[p] > 0.0)) continue;                        // unused (all-zero) row
    const int pp = row_point(p);
    const double ap = s.a[p], bp = s.b[p];
    const double Mpp = (ap * ap + bp * bp) * s.Gam[pp][pp];
#pragma unroll 1
    for (int j = lane; j < q; j += 32) {
      const int k = s.W[j];
      s.gv[j] = (s.a[k] * ap + s.b[k] * bp) * s.Gam[s.cpt[j]][pp];
    }
    __syncwarp();
    const double delta = Mpp - warp_sum(tri_products(s, T, q, lane));
    if (!(delta > 1e-9 * Mpp)) continue;                     // (nearly) dependent on the rows already taken
    const double idd = rsqrt(delta);
#pragma unroll 1
    for (int j = lane; j < q; j += 32) T[tri(q) + j] = -s.r[j] * idd;
    if (lane == 0) { T[tri(q) + q] = idd; s.W[q] = p; s.cpt[q] = pp; s.u[q] = 0.0; }
    if ((p & 31) == lane) actbits |= 1u << (p >> 5);
    ++q; ++iterations;
    __syncwarp();
  }
#pragma unroll 1
  while (q > 0) {
#pragma unroll 1
    for (int j = lane; j < q; j += 32) {
      const int k = s.W[j], kp = s.cpt[j];
      s.gv[j] = s.a[k] * s.PX[kp] + s.b[k] * s.PY[kp] + s.d[k];
    }
    __syncwarp();
    tri_products(s, T, q, lane);
    double umin = 0.0, umax = 0.0; int l = 0x7fffffff;
#pragma unroll 1
    for (int j = lane; j < q; j += 32) {
      const double uj = -s.r[j];
      s.u[j] = uj;
      umax = fmax(umax, uj);
      if (uj < umin) { umin = uj; l = j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) umax = fmax(umax, __shfl_xor_sync(0xffffffffu, umax, o));
    warp_argmin(umin, l);
    __syncwarp();
    if (!(umin < -1e-12 * umax) || l == 0x7fffffff) break;
    drop_row(s, T, q, l, lane, actbits);
    --q; ++iterations;
  }
  if (q == 0) return;
  // move the point onto the S-pair: P = P0 + sum_j Gamma(:, kappa_j) (a_j, b_j) u_j
#pragma unroll 1
  for (int j = lane; j < q; j += 32) {
    const int k = s.W[j];
    const double uj = fmax(s.u[j], 0.0);
    s.u[j] = uj;
    s.ca[j] = uj * s.a[k]; s.cb[j] = uj * s.b[k];
  }
  __syncwarp();
  if (lane < npts) {
    double dx = 0.0, dy = 0.0;
#pragma unroll 2
    for (int j = 0; j < q; ++j) {
      const double gm = s.Gam[lane][s.cpt[j]];
      dx = fma(gm, s.ca[j], dx); dy = fma(gm, s.cb[j], dy);
    }
    s.PX[lane] += dx;
    s.PY[lane] += dy;
  }
  __syncwarp();
}


// Build and solve the QP of the instance in s.in.  On return s.jr / s.ff hold the solution, s.u / s.W / q the
// multipliers of the active rows.  All 32 lanes of the warp must call.
// T: [TRI] doubles of scratch for the inverse Cholesky factor of the active Gram matrix, private to the warp, in global
// memory (herdt_qp_kernel keeps it there to fit 16 warps/SM).
__device__ inline Result solve_warp(Work &s, const Consts &C, int lane, int &q_out, double *__restrict__ T,
                                    const wg_herdt_active_set *__restrict__ hint = nullptr, int hint_age = 1)
{
  const wg_herdt_params &P = C.P;
  const int axis = lane >> 4, i = lane & 15;
  const double wv = P.w_vel, wc = P.w_cop;
  const int ns = s.in.sup_step[N];
  Result res;
  res.n_vars = 2 * N + 2 * ns; res.n_rows = 1 + 4 * N + 5 * ns; res.fail = 0; res.iterations = 0;
  q_out = 0;
  if (ns < 0 || ns > WG_HERDT_MAX_STEPS) { res.fail = 100; return res; }
  const int m = 4 * N + 5 * ns, npts = N + ns;
  const int sn_i = s.in.sup_step[i + 1];
  const double *com = axis ? s.in.com_y : s.in.com_x;
  const double *ref = axis ? s.in.ref_y : s.in.ref_x;

  // ---- selection matrices of the previewed feet (generator-vel-ref.cpp:138-208), redundantly on every lane
  double Vf[2][2] = {{0, 0}, {0, 0}}, Vcf[2][2] = {{0, 0}, {0, 0}};   // Vcf[axis][s]
  for (int ii = 0; ii < N; ++ii) {
    const int k = ii + 1, sn = s.in.sup_step[k];
    if (sn == 1 && s.in.sup_changed[k] && s.in.sup_phase[k] == WG_SS) {
      Vcf[0][0] = s.in.sup_x[k - 1]; Vcf[1][0] = s.in.sup_y[k - 1]; Vf[0][0] = 1.0;
    } else if (sn == 2) {
      Vf[1][0] = -1.0; Vf[1][1] = 1.0;
    }
  }

  // ---- unconstrained optimum: g = Qc^-1 pj,  pj = wv Uv'(Sv c - ref)
  {
    double acc = C.K4[i][0] * com[0] + C.K4[i][1] * com[1] + C.K4[i][2] * com[2];
    for (int k = 0; k < N; ++k) acc = fma(-C.K3[i][k], ref[k], acc);
    s.g[axis][i] = wv * acc;
    s.Z[axis][i] = C.Sz[i][0] * com[0] + C.Sz[i][1] * com[1] + C.Sz[i][2] * com[2];
  }
  __syncwarp();
  double zh;
  {
    double h = 0.0;
    for (int k = 0; k <= i; ++k) h = fma(C.uz[i - k], s.g[axis][k], h);
    zh = s.Z[axis][i] - h;
  }
  // GV[i][s] = sum_{k in step s} G[i][k]
  double GV0 = 0.0, GV1 = 0.0;
  for (int k = 0; k < N; ++k) {
    const int snk = s.in.sup_step[k + 1];
    const double gk = C.G[i][k];
    if (snk == 1) GV0 += gk;
    else if (snk == 2) GV1 += gk;
  }
  const double rhs0 = -wc * half_sum(sn_i == 1 ? zh : 0.0);
  const double rhs1 = -wc * half_sum(sn_i == 2 ? zh : 0.0);
  const double cnt0 = half_sum(sn_i == 1 ? 1.0 : 0.0), cnt1 = half_sum(sn_i == 2 ? 1.0 : 0.0);
  const double V00 = half_sum(sn_i == 1 ? GV0 : 0.0), V01 = half_sum(sn_i == 1 ? GV1 : 0.0);
  const double V11 = half_sum(sn_i == 2 ? GV1 : 0.0);
  double Si00 = 0.0, Si01 = 0.0, Si11 = 0.0;
  if (ns == 1) {
    Si00 = 1.0 / (wc * cnt0 - wc * wc * V00);
  } else if (ns == 2) {
    const double S00 = wc * cnt0 - wc * wc * V00, S01 = -wc * wc * V01, S11 = wc * cnt1 - wc * wc * V11;
    const double det = S00 * S11 - S01 * S01;
    Si00 = S11 / det; Si01 = -S01 / det; Si11 = S00 / det;
  }
  const double tau0 = Si00 * rhs0 + Si01 * rhs1, tau1 = Si01 * rhs0 + Si11 * rhs1;
  if (i < 2) s.f0[axis][i] = (i < ns) ? -(i == 0 ? tau0 : tau1) : 0.0;
  {
    const double vt = (sn_i == 1) ? tau0 : (sn_i == 2 ? tau1 : 0.0);
    double acc = 0.0;
    for (int k = 0; k < N; ++k) acc = fma(C.K1[i][k], __shfl_sync(0xffffffffu, vt, (axis << 4) + k), acc);
    s.j0[axis][i] = -s.g[axis][i] - wc * acc;
  }
  // theta / sigma
  if (axis == 0) {
    const double t0 = (sn_i == 1 ? 1.0 : 0.0) - wc * GV0, t1 = (sn_i == 2 ? 1.0 : 0.0) - wc * GV1;
    s.theta[i][0] = (ns > 0) ? t0 : 0.0; s.theta[i][1] = (ns > 1) ? t1 : 0.0;
  } else if (i < 2) {
    s.theta[N + i][0] = -Vf[i][0]; s.theta[N + i][1] = -Vf[i][1];
  }
  __syncwarp();
  if (lane < NPTS) {
    const double t0 = s.theta[lane][0], t1 = s.theta[lane][1];
    s.sigma[lane][0] = Si00 * t0 + Si01 * t1;
    s.sigma[lane][1] = Si01 * t0 + Si11 * t1;
  }
  __syncwarp();
  for (int e = lane; e < NPTS * NPTS; e += 32) {
    const int k = e / NPTS, l = e - k * NPTS;
    double v = s.sigma[k][0] * s.theta[l][0] + s.sigma[k][1] * s.theta[l][1];
    if (k < N && l < N) v += C.G[k][l];
    s.Gam[k][l] = v;
  }
  points_from_primal(s, C, s.j0, s.f0, ns, Vf, Vcf, s.PX, s.PY, lane);

  // ---- inequality rows (a, b, d) and their inverse Euclidean norms
  if (lane < N) {
    const int k = lane + 1;
    int src = 0;
    for (int kk = 1; kk <= k; ++kk)
      if (s.in.sup_changed[kk]) src = kk;
    double A[5], B[5], D[5];
    hull_rows(P, s.in.sup_foot[src], s.in.sup_phase[src], s.in.sup_yaw[src], true, s.in.sup_foot[k], A, B, D);
    const double th2 = C.uz2[lane] + (sn_i > 0 ? 1.0 : 0.0);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int row = 4 * lane + e;
      s.a[row] = A[e]; s.b[row] = B[e]; s.d[row] = D[e];
      const double n2 = (A[e] * A[e] + B[e] * B[e]) * th2;
      s.inrm[row] = n2 > 0.0 ? rsqrt(n2) : 0.0;
    }
  } else if (lane < N + ns) {
    const int st = lane - N;
    int kf = -1;
    for (int kk = 1; kk <= N; ++kk)
      if (s.in.sup_changed[kk] && s.in.sup_step[kk] == st + 1 && s.in.sup_phase[kk] != WG_DS) kf = kk;
    double A[5] = {0, 0, 0, 0, 0}, B[5] = {0, 0, 0, 0, 0}, D[5] = {0, 0, 0, 0, 0};
    if (kf > 0)
      hull_rows(P, s.in.sup_foot[kf - 1], s.in.sup_phase[kf - 1], s.in.sup_yaw[kf - 1], false, s.in.sup_foot[kf], A, B, D);
    const double th2 = Vf[st][0] * Vf[st][0] + Vf[st][1] * Vf[st][1];
#pragma unroll
    for (int e = 0; e < 5; ++e) {
      const int row = 4 * N + 5 * st + e;
      s.a[row] = A[e]; s.b[row] = B[e]; s.d[row] = D[e];
      const double n2 = (A[e] * A[e] + B[e] * B[e]) * th2;
      s.inrm[row] = n2 > 0.0 ? rsqrt(n2) : 0.0;
    }
  }
  __syncwarp();

  // ---- dual active-set iterations.  Per-row quantities of the active set (<= QMAX = 40 > n = 36 independent rows)
  // live in shared memory and are processed lane-strided (j = lane, lane + 32); the loops are kept rolled on purpose:
  // the iteration body has to stay resident in the instruction cache.
  const double tol = 1e-12;
  const double INF = __longlong_as_double(0x7ff0000000000000LL);
  int q = 0;
  unsigned actbits = 0;    // bit t: row lane + 32 t is active
  int refinements = 0;
  const int maxit = 40 * (m + 2 * N + 4);
  bool done = false;
  if (hint) warm_start(s, T, m, npts, lane, hint, hint_age, q, actbits, res.iterations);
  while (!done) {
    // most violated row, normalised by its Euclidean norm (the pivoting rule of qld.cpp:1255-1331)
    double best = INF;
    int bi = 0x7fffffff;
#pragma unroll 1
    for (int t = 0; t < 3; ++t) {
      const int k = lane + 32 * t;
      if (k < m && !((actbits >> t) & 1u)) {
        const int kp = row_point(k);
        const double sv = (s.a[k] * s.PX[kp] + s.b[k] * s.PY[kp] + s.d[k]) * s.inrm[k];
        if (sv < best) { best = sv; bi = k; }
      }
    }
    warp_argmin(best, bi);
    if (!(best < -tol)) {
      // ---- converged on the incremental points: recover the primal solution from the multipliers, then
      // refine the multipliers so that the active rows hold on points recomputed from that solution
      // (x = x0 + H^-1 N u goes through the precomputed inverse; one or two Newton steps on the dual,
      // du = -(N'H^-1 N)^-1 s_active = -T'T s_active, remove its rounding error)
#pragma unroll 1
      for (int pass = 0;; ++pass) {
        if (lane < NPTS) {
          double wx = 0.0, wy = 0.0;
#pragma unroll 1
          for (int j = 0; j < q; ++j)
            if (s.cpt[j] == lane) { const int k = s.W[j]; wx = fma(s.u[j], s.a[k], wx); wy = fma(s.u[j], s.b[k], wy); }
          s.wpt[0][lane] = wx; s.wpt[1][lane] = wy;
        }
        __syncwarp();
        double sg0 = 0.0, sg1 = 0.0;
#pragma unroll 1
        for (int k = 0; k < npts; ++k) {
          const double wk = s.wpt[axis][k];
          sg0 = fma(s.sigma[k][0], wk, sg0); sg1 = fma(s.sigma[k][1], wk, sg1);
        }
        {
          double acc = 0.0;
#pragma unroll 4
          for (int k = 0; k < N; ++k) {
            const int snk = s.in.sup_step[k + 1];
            const double corr = (snk == 1) ? sg0 : (snk == 2 ? sg1 : 0.0);
            acc = fma(C.K1[i][k], s.wpt[axis][k] - wc * corr, acc);
          }
          s.jr[axis][i] = s.j0[axis][i] - acc;
          if (i < 2) s.ff[axis][i] = (i < ns) ? s.f0[axis][i] + (i == 0 ? sg0 : sg1) : 0.0;
        }
        __syncwarp();
        points_from_primal(s, C, s.jr, s.ff, ns, Vf, Vcf, s.PX, s.PY, lane);
        double vmax = 0.0;
#pragma unroll 1
        for (int j = lane; j < q; j += 32) {
          const int k = s.W[j], kp = s.cpt[j];
          const double sj = s.a[k] * s.PX[kp] + s.b[k] * s.PY[kp] + s.d[k];
          s.gv[j] = sj;
          vmax = fmax(vmax, fabs(sj) * s.inrm[k]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) vmax = fmax(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
        if (!(vmax > 1e-14) || pass >= 3) break;
        __syncwarp();
#pragma unroll 1
        for (int j = lane; j < q; j += 32) {
          const double *Tr = T + tri(j);
          double wv_ = 0.0;
#pragma unroll 4
          for (int e = 0; e <= j; ++e) wv_ = fma(Tr[e], s.gv[e], wv_);
          s.w[j] = wv_;
        }
        __syncwarp();
#pragma unroll 1
        for (int j = lane; j < q; j += 32) {
          double rj = 0.0;
#pragma unroll 4
          for (int r = j; r < q; ++r) rj = fma(T[tri(r) + j], s.w[r], rj);
          s.u[j] -= rj;
        }
        __syncwarp();
      }
      // re-evaluate the inactive rows on those points
      double worst = INF; int wi = 0x7fffffff;
#pragma unroll 1
      for (int t = 0; t < 3; ++t) {
        const int k = lane + 32 * t;
        if (k < m && !((actbits >> t) & 1u)) {
          const int kp = row_point(k);
          const double sv = (s.a[k] * s.PX[kp] + s.b[k] * s.PY[kp] + s.d[k]) * s.inrm[k];
          if (sv < worst) { worst = sv; wi = k; }
        }
      }
      warp_argmin(worst, wi);
      if (!(worst < -tol) || refinements >= 3) { done = true; break; }
      ++refinements;
      best = worst; bi = wi;
    }
    const int p = bi;
    const int pp = row_point(p);
    const double ap = s.a[p], bp = s.b[p];
    const double Mpp = (ap * ap + bp * bp) * s.Gam[pp][pp];
    double up = 0.0;
#pragma unroll 1
    while (true) {
      if (++res.iterations > maxit) { res.fail = 1; done = true; break; }   // QLD ifail 1: too many iterations
      if (q >= QMAX) { res.fail = 3; done = true; break; }                  // active-set capacity exhausted
      // gv_j = N_Wj' H^-1 N_p
#pragma unroll 1
      for (int j = lane; j < q; j += 32) {
        const int k = s.W[j];
        s.gv[j] = (s.a[k] * ap + s.b[k] * bp) * s.Gam[s.cpt[j]][pp];
      }
      __syncwarp();
      double wsq = 0.0;
#pragma unroll 1
      for (int j = lane; j < q; j += 32) {
        const double *Tr = T + tri(j);
        double w0 = 0.0, w1 = 0.0;
        int e = 0;
#pragma unroll 2
        for (; e + 1 <= j; e += 2) { w0 = fma(Tr[e], s.gv[e], w0); w1 = fma(Tr[e + 1], s.gv[e + 1], w1); }
        if (e <= j) w0 = fma(Tr[e], s.gv[e], w0);
        const double wv_ = w0 + w1;
        s.w[j] = wv_;
        wsq = fma(wv_, wv_, wsq);
      }
      __syncwarp();
      double t1 = INF; int l = 0x7fffffff;
#pragma unroll 1
      for (int j = lane; j < q; j += 32) {
        double r0 = 0.0, r1 = 0.0;
        int r = j;
#pragma unroll 2
        for (; r + 1 < q; r += 2) { r0 = fma(T[tri(r) + j], s.w[r], r0); r1 = fma(T[tri(r + 1) + j], s.w[r + 1], r1); }
        if (r < q) r0 = fma(T[tri(r) + j], s.w[r], r0);
        const double rj = r0 + r1;
        s.r[j] = rj;
        if (rj > 0.0) {
          const double tj = s.u[j] / rj;
          if (tj < t1) { t1 = tj; l = j; }
        }
      }
      const double delta = Mpp - warp_sum(wsq);
      warp_argmin(t1, l);
      const double sp = ap * s.PX[pp] + bp * s.PY[pp] + s.d[p];
      const double t2 = (delta > 1e-13 * Mpp) ? -sp / delta : INF;
      const double tt = fmin(t1, t2);
      if (!(tt < INF)) { res.fail = 2; done = true; break; }   // infeasible (QLD ifail 2 family)
      // direction in point space and step
#pragma unroll 1
      for (int j = lane; j < q; j += 32) {
        const int k = s.W[j];
        const double rj = s.r[j];
        s.ca[j] = -rj * s.a[k]; s.cb[j] = -rj * s.b[k];
        s.u[j] = fma(-tt, rj, s.u[j]);
      }
      if (lane == 0) { s.ca[q] = ap; s.cb[q] = bp; s.cpt[q] = pp; }
      __syncwarp();
      if (lane < npts) {
        double dx = 0.0, dy = 0.0;
#pragma unroll 2
        for (int j = 0; j <= q; ++j) {
          const double gm = s.Gam[lane][s.cpt[j]];
          dx = fma(gm, s.ca[j], dx); dy = fma(gm, s.cb[j], dy);
        }
        s.PX[lane] = fma(tt, dx, s.PX[lane]);
        s.PY[lane] = fma(tt, dy, s.PY[lane]);
      }
      up += tt;
      __syncwarp();
      if (t2 <= t1) {
        // full step: row p becomes active; append a row to T (inverse Cholesky factor of the active Gram matrix)
        const double idd = rsqrt(delta);
#pragma unroll 1
        for (int j = lane; j < q; j += 32) T[tri(q) + j] = -s.r[j] * idd;
        if (lane == 0) { T[tri(q) + q] = idd; s.W[q] = p; s.u[q] = up; }
        if ((p & 31) == lane) actbits |= 1u << (p >> 5);
        ++q;
        __syncwarp();
        break;
      }
      // partial step: multiplier l reached zero -> drop row l
      {
        drop_row(s, T, q, l, lane, actbits);
        --q;
      }
    }
  }
  if (res.fail) {  // no solution: report the unconstrained optimum, as a caller-visible placeholder
    s.jr[axis][i] = s.j0[axis][i];
    if (i < 2) s.ff[axis][i] = s.f0[axis][i];
    __syncwarp();
  }
  q_out = q;
  return res;
}

}  // namespace herdt
