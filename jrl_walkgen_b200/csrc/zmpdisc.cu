// zmpdisc.cu - Kajita2003 front end on the GPU: footsteps -> 5 ms ZMP reference + feet trajectories, batched, and the
// footsteps -> CoM pipeline that chains it into the fused preview kernel (preview.cu) without leaving the device.
//
// Replaces (see include/walkgen_b200.h for the line ranges):
//   ZMPDiscretization::GetZMPDiscretization = InitOnLine + OnLineAddFoot per step + EndPhaseOfTheWalking,
//   ZMPDiscretization::FilterOutValues / UpdateCurrentSupportFootPosition,
//   FootTrajectoryGenerationStandard::UpdateFootPosition, Polynome3/4/5,
//   StepStackHandler::PrepareForSupportFoot / CreateArcInStepStack / FinishOnTheLastCorrectSupportFoot (host side).
//
// Kernel design: one WARP owns one walk.  A walk is a chain of segments (lead-in, one per step, end phase); segments
// are sequential (each starts from the last FILTERED sample of the previous one) but the samples of a segment are
// independent given the segment's set-up, so the 32 lanes take samples i = lane, lane+32, ...  The unfiltered ZMP of the
// current segment lives in shared memory (the smoothing window reads samples i-8 .. i+2); every lane carries the same
// copy of the walk state (support frame, feet, polynomial coefficients) in registers, computed redundantly so that no
// broadcast is needed.  The first 8 samples of a segment read already-filtered values of the previous segment AND of
// themselves (a quirk of FilterOutValues' index arithmetic, ZMPDiscretization.cpp:1056-1078): lane 0 runs them serially.
// This translation unit is compiled with -fmad=false: the reference evaluates its polynomials and the filter with
// separate multiplies and adds, and the discrete decisions (lift-off / landing windows) stay on the same side.
#include <algorithm>
#include <cmath>
#include <new>
#include "wg_common.h"

namespace {

constexpr int ZD_WARPS = 4;          // warps (walks in flight) per CTA
constexpr int ZD_THREADS = 32 * ZD_WARPS;
constexpr int ZD_MAXW = 32;          // filter window capacity (n+1 taps; 11 in every reference configuration)
constexpr int ZD_HIST = 16;          // filtered samples of the previous segment kept in shared memory (>= window)
constexpr int ZD_HEAD = 8;           // samples of a segment that depend on filtered history (i - j + 2 < 0 for j <= 10)

struct ZdConsts {
  wg_zmpdisc_params P;
  double window[ZD_MAXW];
  int nw;                            // taps
  int n_lead, n_end, n_tail;         // 2*NL, round(Tdble/(2T)), 3*NL
  int cap;                           // shared-memory capacity (samples) of the per-warp segment buffer
};

struct Poly {
  double c[6];
};
__device__ __forceinline__ double peval(const Poly &p, int n, double t)
{  // Polynome::Compute: running power, separate multiply and add
  double r = 0.0, pt = 1.0;
#pragma unroll
  for (int i = 0; i < 6; ++i)
    if (i < n) {
      r += p.c[i] * pt;
      pt *= t;
    }
  return r;
}
__device__ __forceinline__ Poly poly3(double FT, double FP)
{
  Poly p = {{0, 0, 0, 0, 0, 0}};
  double tmp = FT * FT;
  if (!(FP == 0.0 || FT == 0.0)) {
    p.c[2] = 3.0 * FP / tmp;
    p.c[3] = -2.0 * FP / (tmp * FT);
  }
  return p;
}
__device__ __forceinline__ Poly poly4(double FT, double MP)
{
  Poly p = {{0, 0, 0, 0, 0, 0}};
  double tmp = FT * FT;
  if (!(MP == 0.0 || tmp == 0.0)) {
    p.c[2] = 16.0 * MP / tmp;
    tmp = tmp * FT;
    p.c[3] = -32.0 * MP / tmp;
    tmp = tmp * FT;
    p.c[4] = 16.0 * MP / tmp;
  }
  return p;
}
__device__ __forceinline__ Poly poly5(double FT, double FP)
{
  Poly p = {{0, 0, 0, 0, 0, 0}};
  double tmp = FT * FT * FT;
  if (!(FP == 0.0 || tmp == 0.0)) {
    p.c[3] = 10 * FP / tmp;
    tmp *= FT;
    p.c[4] = -15 * FP / tmp;
    tmp *= FT;
    p.c[5] = 6 * FP / tmp;
  }
  return p;
}

struct Foot {
  double x, y, z, theta, omega, omega2;
};

// Toe / heel rotation of the swing foot for omega != 0 (FootTrajectoryGenerationStandard.cpp:520-563).  Out of line: the
// six sin/cos expansions would otherwise sit in the middle of the sample loop of every step.
__device__ __noinline__ void omega_correction(double lo, double lth, double Bf, double H, double Ff, Foot &f)
{
  double dX, dFZ;
  if (lo < 0) {
    const double X1 = Bf * cos(-lo), X2 = H * sin(-lo), Z1 = H * cos(-lo), Z2 = Bf * sin(-lo);
    dX = -(Bf - X1 + X2);
    dFZ = Z1 + Z2 - H;
  } else {
    const double X1 = Ff * cos(lo), X2 = H * sin(lo), Z1 = H * cos(lo), Z2 = Ff * sin(lo);
    dX = (Ff - X1 + X2);
    dFZ = Z1 + Z2 - H;
  }
  if (dX != 0.0) {
    f.x += cos(lth) * dX;
    f.y += sin(lth) * dX;
  } else {
    f.x += 0.0;
    f.y += 0.0;
  }
  f.z += dFZ;
}

struct Frame {   // m_CurrentSupportFootPosition: rotation (row-major 2x2) + translation
  double r00, r01, r10, r11, tx, ty;
};

__device__ __forceinline__ void update_support(Frame &S, double &ptx, double &pty, const wg_rel_step &s)
{
  ptx = S.tx;
  pty = S.ty;
  const double a = s.theta * M_PI / 180.0;
  const double c = cos(a), sn = sin(a);
  const double n00 = (0.0 + c * S.r00) + -sn * S.r10, n01 = (0.0 + c * S.r01) + -sn * S.r11;
  const double n10 = (0.0 + sn * S.r00) + c * S.r10, n11 = (0.0 + sn * S.r01) + c * S.r11;
  const double v0 = (0.0 + n00 * s.sx) + n01 * s.sy, v1 = (0.0 + n10 * s.sx) + n11 * s.sy;
  S.r00 = n00; S.r01 = n01; S.r10 = n10; S.r11 = n11;
  S.tx += v0;
  S.ty += v1;
}

__device__ __forceinline__ void support_world(const Frame &S, const wg_zmpdisc_params &P, double &wx, double &wy)
{
  wx = ((0.0 + S.r00 * P.zmp_neutral[0]) + S.r01 * P.zmp_neutral[1]) + S.tx * 1.0;
  wy = ((0.0 + S.r10 * P.zmp_neutral[0]) + S.r11 * P.zmp_neutral[1]) + S.ty * 1.0;
}

struct Out {
  double2 *zmpref;
  double *ztheta;
  wg_foot_sample *left, *right;
  int32_t *types;
};

__device__ __forceinline__ void put_foot(wg_foot_sample *dst, int64_t g, const Foot &f)
{
  if (!dst) return;
  double2 *q = reinterpret_cast<double2 *>(dst + g);      // 48-byte records, 16-byte aligned: three 128-bit stores
  q[0] = make_double2(f.x, f.y); q[1] = make_double2(f.z, f.theta); q[2] = make_double2(f.omega, f.omega2);
}

// Filter the head of a segment (samples 0 .. min(len, ZD_HEAD) - 1) serially: they read filtered history.
//   u      unfiltered samples of this segment (shared), ulen = number of distinct entries (clamped reads beyond)
//   hist   the last ZD_HIST filtered samples before this segment (hist[ZD_HIST-1] = FinalZMPPositions.back())
//   F0     number of filtered samples emitted before this segment; final0 = FinalZMPPositions[0]
__device__ void filter_head(const ZdConsts &K, const double2 *u, int len, int ulen, const double2 *hist, int64_t F0,
                            double2 final0, double2 *head)
{
  // A tap that reads filtered history has r = i - j + 2 < 0, i.e. j >= i + 3, and then looks at head[q] with q = 2 i - j - 1
  // <= i - 4: sample i depends on head samples at least four places back.  So the eight head samples are two rounds of four
  // independent ones: lanes 0..3 run samples 4 round + lane, each summing its 11 taps in the reference's order (bitwise the
  // serial loop, a quarter of its instructions).
  const int nh = min(len, ZD_HEAD);
  const int lane = threadIdx.x & 31;
  static_assert(ZD_HEAD == 8, "two rounds of four head samples");
#pragma unroll 1
  for (int round = 0; round < 2; ++round) {
    const int i = 4 * round + lane;
    if (lane < 4 && i < nh) {
      double a0 = 0, a1 = 0;
      const int64_t o = F0 + i - 1 - 2;
#pragma unroll 1
      for (int j = 0; j < K.nw; ++j) {
        int r = i - j + 2;
        double2 v;
        if (r < 0) {
          if (-r < o) {
            const int q = 2 * i - j - 1;          // FinalZMPPositions[o + r] relative to F0
            v = (q >= 0) ? head[q] : hist[ZD_HIST + q];
          } else
            v = final0;
        } else {
          if (r >= len) r = len - 1;
          v = u[min(r, ulen - 1)];
        }
        a0 += K.window[j] * v.x;
        a1 += K.window[j] * v.y;
      }
      head[i] = make_double2(a0, a1);
    }
    __syncwarp();
  }
}

__device__ __forceinline__ double2 filter_body(const ZdConsts &K, const double2 *u, int len, int ulen, int i)
{  // i >= ZD_HEAD: every tap reads this segment's unfiltered samples
  double a0 = 0, a1 = 0;
  for (int j = 0; j < K.nw; ++j) {
    int r = i - j + 2;
    if (r >= len) r = len - 1;
    const double2 v = u[min(r, ulen - 1)];
    a0 += K.window[j] * v.x;
    a1 += K.window[j] * v.y;
  }
  return make_double2(a0, a1);
}

// Filtered ZMP of lead-in sample i (InitOnLine: a ramp from (0, 0) to the neutral position through the 11-tap window).  It depends
// on the parameters only, not on the walk: zmpdisc_lead_kernel tabulates it once per plan with this very code, and the front-end
// kernel reads the table (11 FP64 divisions per sample and walk saved, same bits).
__device__ __forceinline__ double2 lead_sample(const ZdConsts &K, int i)
{
  const wg_zmpdisc_params &P = K.P;
  const int n = K.n_lead;
  const double2 u2 = make_double2(0.0 + (P.zmp_neutral[0] - 0.0) * (2.0 / (double)n),
                                  0.0 + (P.zmp_neutral[1] - 0.0) * (2.0 / (double)n));
  double a0 = 0, a1 = 0;
#pragma unroll 1
  for (int j = 0; j < K.nw; ++j) {
    int r = i - j + 2;
    double2 v;
    if (r < 0)
      v = u2;
    else {
      if (r >= n) r = n - 1;
      const double coef = (double)r / (double)n;
      v = make_double2(0.0 + (P.zmp_neutral[0] - 0.0) * coef, 0.0 + (P.zmp_neutral[1] - 0.0) * coef);
    }
    a0 += K.window[j] * v.x;
    a1 += K.window[j] * v.y;
  }
  return make_double2(a0, a1);
}

__global__ void zmpdisc_lead_kernel(const ZdConsts K, double2 *__restrict__ lead)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < K.n_lead) lead[i] = lead_sample(K, i);
}

// What a walk carries from one segment to the next (besides the last ZD_HIST filtered samples, which live in shared memory):
// m_CurrentSupportFootPosition, the previous support translation, both feet, the theta of FinalZMPPositions.back(), the
// number of samples emitted and FinalZMPPositions[0].
struct ZdWalk {
  Frame S;
  double prev_tx, prev_ty;
  Foot L, R;
  double zmp_theta;
  int64_t F0;
  double2 final0;
};

// Where a segment writes.  Sample F of the walk (counted from its first lead-in sample) goes to row o + F of `out`, and,
// with PACK and pk != nullptr, its filtered ZMP also to row o + F + pk_shift of `pk` (the packed preview input of
// wg_kajita_stream).
struct ZdDst {
  int64_t o;
  double2 *pk;
  int64_t pk_shift;
};
template <bool PACK>
__device__ __forceinline__ void put_zmp(const Out &out, const ZdDst &d, int64_t g, double2 f)
{
  if (out.zmpref) out.zmpref[g] = f;
  if (PACK && d.pk) d.pk[g + d.pk_shift] = f;
}

// InitOnLine: the state of a new walk and its 2*NL lead-in samples ramping from the start ZMP (0,0) to the neutral position
// (init filter).  Fills hist with the last ZD_HIST filtered samples.
template <bool PACK>
__device__ __forceinline__ void zd_lead_in(const ZdConsts &K, ZdWalk &w, const double *feet, const Out &out, const ZdDst &d,
                                           const double2 *lead_tab, double2 *hist, double2 *head, int lane)
{
  w.S = Frame{1.0, 0.0, 0.0, 1.0, 0.0, 0.0};
  w.prev_tx = 0.0; w.prev_ty = 0.0;
  w.L = Foot{feet[0], feet[1], 0.0, feet[2], 0.0, 0.0};
  w.R = Foot{feet[3], feet[4], 0.0, feet[5], 0.0, 0.0};
  w.zmp_theta = 0.0;
  w.F0 = 0;
  const int n = K.n_lead;
#pragma unroll 1
  for (int i = lane; i < n; i += 32) {
    const double2 f = __ldg(lead_tab + i);      // lead_sample(K, i), tabulated once per plan
    const double a0 = f.x, a1 = f.y;
    const int64_t g = d.o + i;
    put_zmp<PACK>(out, d, g, make_double2(a0, a1));
    if (out.ztheta) out.ztheta[g] = 0.0;
    put_foot(out.left, g, w.L);
    put_foot(out.right, g, w.R);
    if (out.types) { out.types[3 * g] = 0; out.types[3 * g + 1] = 10; out.types[3 * g + 2] = 10; }
    if (i >= n - ZD_HIST) hist[i - (n - ZD_HIST)] = make_double2(a0, a1);
    if (i == 0) head[0] = make_double2(a0, a1);
  }
  w.F0 = n;
  __syncwarp();
  w.final0 = head[0];
  __syncwarp();
}

// OnLineAddFoot: the segment of step rel1 (rel0 is the step before it).  Swaps hist / hist2 so that hist holds the new
// history.  Returns 0, or 2 when the step timing or the sample budget (Ltot) does not fit.
template <bool PACK>
__device__ __forceinline__ int zd_add_foot(const ZdConsts &K, ZdWalk &w, const wg_rel_step &rel0, const wg_rel_step &rel1,
                                           const Out &out, const ZdDst &d, int64_t Ltot, double2 *u, double2 *&hist,
                                           double2 *&hist2, double2 *head, Poly *pp, int lane)
{
  const wg_zmpdisc_params &P = K.P;
  const double T = P.sampling_period;
  Frame &S = w.S;
  Foot &L = w.L, &R = w.R;
  double vpre0, vpre1, dTheta, dZmpTheta;
  double lTdble = P.t_double, lTsingle = P.t_single;
  if (rel1.ds_time != 0.0) {
    lTdble = rel1.ds_time;
    lTsingle = rel1.ss_time;
  }
  int who;
  if (rel0.sy < 0) {
    who = -1;
    vpre0 = R.x - L.x; vpre1 = R.y - L.y;
    dTheta = R.theta - L.theta;
    dZmpTheta = R.theta - w.zmp_theta;
  } else {
    who = 1;
    vpre0 = -R.x + L.x; vpre1 = -R.y + L.y;
    dTheta = L.theta - R.theta;
    dZmpTheta = L.theta - w.zmp_theta;
  }
  const int add = (int)(unsigned)round((lTdble + lTsingle) / T);
  update_support(S, w.prev_tx, w.prev_ty, rel0);
  const int n1 = (int)(unsigned)round(lTdble / T);
  const int n2 = (int)(unsigned)round(lTsingle / T);
  if (n1 < 1 || n1 + n2 > add || add > K.cap || w.F0 + add > Ltot) return 2;
  const double2 back = hist[ZD_HIST - 1];
  const double px0 = back.x, py0 = back.y, theta0 = w.zmp_theta;
  double wx, wy;
  support_world(S, P, wx, wy);
  double dx = (wx - px0) / n1, dy = (wy - py0) / n1;
  const int t1 = rel1.step_type;
  if (t1 == 3) { dx = (S.tx + P.zmp_shift[0] - px0) / n1; dy = (S.ty - py0) / n1; }
  if (t1 == 4) { dx = (S.tx + P.zmp_shift[2] - px0) / n1; dy = (S.ty - py0) / n1; }
  if (t1 == 5) {
    dx = (S.tx - (P.zmp_shift[0] + P.zmp_shift[2] + P.zmp_shift[1] + P.zmp_shift[3]) - px0) / n1;
    dy = (S.ty - py0) / n1;
  }
  // unfiltered ZMP of the segment
  for (int k = lane; k < add; k += 32) {
    double2 v;
    if (k < n1)
      v = make_double2(px0 + k * dx, py0 + k * dy);
    else if (k < n1 + n2)
      v = make_double2(wx, wy);
    else
      v = make_double2(0.0, 0.0);
    u[k] = v;
  }
  __syncwarp();
  if ((t1 == 3 || t1 == 4) && lane == 0) {   // step-over profiles: running sums (ZMPDiscretization.cpp:903-931)
    const double sh = (t1 == 3) ? P.zmp_shift[1] : P.zmp_shift[3];
    const double px02 = u[n1 - 1].x, py02 = u[n1 - 1].y;
    const double ex = (S.tx + sh - px02) / n2, ey = (S.ty - py02) / n2;
    for (int k = n1; k < n1 + n2; ++k) u[k] = make_double2(u[k - 1].x + ex, u[k - 1].y + ey);
  }
  __syncwarp();
  filter_head(K, u, add, add, hist, w.F0, w.final0, head);     // whole warp: lanes 0..3 work, two rounds (ends on a __syncwarp)
  // swing-foot set-up (every lane, redundantly)
  const double next_theta = rel1.theta;
  const double rel_theta = next_theta + dTheta, rel_zmp_theta = next_theta + dZmpTheta;
  const double ang = next_theta * M_PI / 180.0;
  const double c = cos(ang), s = sin(ang);
  const double n00 = (0.0 + c * S.r00) + -s * S.r10, n01 = (0.0 + c * S.r01) + -s * S.r11;
  const double n10 = (0.0 + s * S.r00) + c * S.r10, n11 = (0.0 + s * S.r01) + c * S.r11;
  const double vd0 = (0.0 + n00 * rel1.sx) + n01 * rel1.sy, vd1 = (0.0 + n10 * rel1.sx) + n11 * rel1.sy;
  const double vrel0 = vd0 + vpre0, vrel1 = vd1 + vpre1;
  const double mod = lTsingle * P.modulation;
  const double end_lift_param = (lTsingle - mod) * 0.5;
  // the seven boundary-value polynomials of the step live in shared memory (every lane evaluates them at its own
  // time: broadcast reads) instead of 42 registers per lane
  __syncwarp();
  if (lane == 0) {
    pp[0] = poly5(mod, vrel0); pp[1] = poly5(mod, vrel1); pp[2] = poly4(P.t_single, P.step_height);
    pp[3] = poly3(mod, rel_theta); pp[4] = poly3(end_lift_param, P.omega); pp[5] = poly3(mod, 2 * P.omega);
    pp[6] = poly3(lTsingle, rel_zmp_theta);
  }
  __syncwarp();
  const Poly &PX = pp[0], &PY = pp[1], &PZ = pp[2], &PT = pp[3], &PO = pp[4], &PO2 = pp[5], &PZT = pp[6];
  const double end_lift = (P.t_single - mod) * 0.5, start_land = end_lift + mod;
  Foot dsL = L, dsR = R;        // feet during double support: last sample with z = 0
  dsL.z = 0.0;
  dsR.z = 0.0;
  const Foot sup0 = (who == 1) ? dsL : dsR, swg0 = (who == 1) ? dsR : dsL;
  auto swing = [&](int kk) {    // UpdateFootPosition for local index kk = 1 .. n2
    Foot f = {0, 0, 0, 0, 0, 0};
    const double lt = kk * T;
    if (lt < end_lift) {
      f.x = swg0.x; f.y = swg0.y; f.theta = swg0.theta;
    } else if (lt < start_land) {
      f.x = swg0.x + peval(PX, 6, lt - end_lift);
      f.y = swg0.y + peval(PY, 6, lt - end_lift);
      f.theta = swg0.theta + peval(PT, 4, lt - end_lift);
    } else {
      f.x = swg0.x + peval(PX, 6, mod);
      f.y = swg0.y + peval(PY, 6, mod);
      f.theta = swg0.theta + peval(PT, 4, mod);
    }
    f.z = swg0.z + peval(PZ, 5, lt);
    if (lt < end_lift)
      f.omega = peval(PO, 4, lt);
    else if (lt < start_land)
      f.omega = P.omega - peval(PO2, 4, lt - end_lift);
    else
      f.omega = peval(PO, 4, lt - start_land) - P.omega;
    const double lo = f.omega * M_PI / 180.0, lth = f.theta * M_PI / 180.0;
    const double Bf = P.foot_b, H = P.foot_h, Ff = P.foot_f;
    if (lo == 0.0) {            // cos(0) = 1, sin(0) = 0 exactly: the correction vanishes without the trig calls
      const double dX = (Ff - Ff + 0.0), dFZ = H + 0.0 - H;
      f.x += dX;               // x + c*0 = x for finite c
      f.y += dX;
      f.z += dFZ;
    } else {
      omega_correction(lo, lth, Bf, H, Ff, f);   // rarely taken (omega = 0 in every reference profile): out of line
    }
    return f;
  };
  // emit the segment
  for (int i = lane; i < add; i += 32) {
    const double2 f = (i < ZD_HEAD) ? head[i] : filter_body(K, u, add, add, i);
    const int64_t g = d.o + w.F0 + i;
    put_zmp<PACK>(out, d, g, f);
    if (i >= add - ZD_HIST) hist2[i - (add - ZD_HIST)] = f;
    double th;
    int tz, tl, tr;
    Foot fl, fr;
    if (i < n1) {
      th = theta0;
      tz = tl = tr = t1 + 10;
      fl = dsL;
      fr = dsR;
    } else if (i < n1 + n2) {
      const int k = i - n1;
      th = peval(PZT, 4, k * T) + theta0;
      tz = who * rel0.step_type;
      const Foot sw = swing(k + 1);
      if (who == 1) { fl = sup0; fr = sw; tl = -t1; tr = t1; }
      else { fr = sup0; fl = sw; tr = -t1; tl = t1; }
    } else {                    // samples the reference leaves value-initialised
      th = 0.0;
      tz = tl = tr = 0;
      fl = Foot{0, 0, 0, 0, 0, 0};
      fr = fl;
    }
    if (out.ztheta) out.ztheta[g] = th;
    put_foot(out.left, g, fl);
    put_foot(out.right, g, fr);
    if (out.types) { out.types[3 * g] = tz; out.types[3 * g + 1] = tl; out.types[3 * g + 2] = tr; }
  }
  if (add < ZD_HIST)            // very short segment: the older history slides down
    for (int q = lane; q < ZD_HIST - add; q += 32) hist2[q] = hist[q + add];
  __syncwarp();
  // carry: state after the last sample of the segment
  if (add > n1 + n2) {
    L = Foot{0, 0, 0, 0, 0, 0};
    R = L;
    w.zmp_theta = 0.0;
  } else {
    const Foot sw = swing(n2);
    if (who == 1) { L = sup0; R = sw; }
    else { R = sup0; L = sw; }
    w.zmp_theta = (n2 > 0) ? peval(PZT, 4, (n2 - 1) * T) + theta0 : theta0;
  }
  { double2 *t = hist; hist = hist2; hist2 = t; }
  w.F0 += add;
  return 0;
}

// EndPhaseOfTheWalking after the walk's last step `last`: n_end samples to the middle of the feet, then 3*NL at rest.
// Returns 0, or 3 when the phase does not end exactly at Ltot.
template <bool PACK>
__device__ __forceinline__ int zd_end_phase(const ZdConsts &K, ZdWalk &w, const wg_rel_step &last, const Out &out,
                                            const ZdDst &d, int64_t Ltot, double2 *u, const double2 *hist, double2 *head,
                                            int lane)
{
  update_support(w.S, w.prev_tx, w.prev_ty, last);
  const int n = K.n_end, len = K.n_end + K.n_tail;
  if (n < 1 || n > K.cap || w.F0 + len != Ltot) return 3;
  const double2 back = hist[ZD_HIST - 1];
  const double pxf = 0.5 * (w.S.tx + w.prev_tx), pyf = 0.5 * (w.S.ty + w.prev_ty);
  const double dx = (pxf - back.x) / (double)n, dy = (pyf - back.y) / (double)n;
  if (lane == 0) {
    u[0] = make_double2(back.x + dx, back.y + dy);
    for (int k = 1; k < n; ++k) u[k] = make_double2(u[k - 1].x + dx, u[k - 1].y + dy);
  }
  __syncwarp();
  filter_head(K, u, len, n, hist, w.F0, w.final0, head);     // whole warp (ends on a __syncwarp)
  for (int i = lane; i < len; i += 32) {
    const double2 f = (i < ZD_HEAD) ? head[i] : filter_body(K, u, len, n, i);
    const int64_t g = d.o + w.F0 + i;
    put_zmp<PACK>(out, d, g, f);
    if (out.ztheta) out.ztheta[g] = w.zmp_theta;
    put_foot(out.left, g, w.L);
    put_foot(out.right, g, w.R);
    if (out.types) { out.types[3 * g] = 0; out.types[3 * g + 1] = 0; out.types[3 * g + 2] = 0; }
  }
  __syncwarp();
  return 0;
}

// Per-warp slices of the dynamic shared memory: the unfiltered segment (cap), two history buffers, the filtered head.
__device__ __forceinline__ double2 *zd_warp_smem(double2 *smem, const ZdConsts &K, int warp)
{
  return smem + (size_t)warp * (K.cap + 2 * ZD_HIST + ZD_HEAD);
}

// 3 CTAs per SM: 168 registers, no spills (measured 0.72 ms per 4096 walks against 0.77 at 4 CTAs / 128 registers / 56 B of spills, 1.03 at 5)
__global__ void __launch_bounds__(ZD_THREADS, 3)
zmpdisc_kernel(const ZdConsts K, int b0, int b1, const int64_t *__restrict__ step_off,
               const wg_rel_step *__restrict__ steps, const double *__restrict__ init_feet,
               const int64_t *__restrict__ samp_off, Out out, int *__restrict__ status,
               const int *__restrict__ order, int *__restrict__ next_walk, const double2 *__restrict__ lead_tab)
{
  extern __shared__ double2 zd_smem[];
  __shared__ Poly s_poly[ZD_WARPS][7];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double2 *u = zd_warp_smem(zd_smem, K, warp);
  double2 *histA = u + K.cap, *histB = histA + ZD_HIST, *head = histB + ZD_HIST;
  const unsigned FULL = 0xffffffffu;

  // walks differ in length (8-20 steps, arcs): every warp fetches its next walk from a counter, longest walks first
  for (;;) {
    int b = 0;
    if (lane == 0) { b = atomicAdd(next_walk, 1); b = (b0 + b < b1) ? order[b0 + b] : -1; }
    b = __shfl_sync(FULL, b, 0);
    if (b < 0) break;
    const int64_t s0 = step_off[b];
    const int ns = (int)(step_off[b + 1] - s0);
    const ZdDst d = {samp_off[b], nullptr, 0};
    const int64_t Ltot = samp_off[b + 1] - d.o;
    if (ns < 1) {
      if (lane == 0 && status) status[b] = 1;
      continue;
    }
    double2 *hist = histA, *hist2 = histB;
    ZdWalk w;
    zd_lead_in<false>(K, w, init_feet + 6 * b, out, d, lead_tab, hist, head, lane);
    int bad = 0;
    for (int si = 1; si < ns && !bad; ++si) {
      const wg_rel_step rel0 = steps[s0 + si - 1], rel1 = steps[s0 + si];
      bad = zd_add_foot<false>(K, w, rel0, rel1, out, d, Ltot, u, hist, hist2, head, s_poly[warp], lane);
    }
    if (!bad) bad = zd_end_phase<false>(K, w, steps[s0 + ns - 1], out, d, Ltot, u, hist, head, lane);
    if (lane == 0 && status) status[b] = bad;
    __syncwarp();
  }
}

// ---- on-line form (wg_kajita_stream) ----------------------------------------------------------------------------------
// A streamed walk between two runs: exactly what zmpdisc_kernel carries from one segment to the next, plus the last step
// appended (rel0 of the walk's next segment).
struct ZsRec {
  ZdWalk w;
  wg_rel_step last;
  double2 hist[ZD_HIST];
};

// One walk's work in a run (built on the host by wg_kajita_stream_append).
struct ZsWork {
  int32_t b, flags, ns, carry;   // walk, WG_STREAM_* flags, steps appended, preview carry samples placed before the new ones
  int64_t s0;                    // first appended step in the run's step array
  int64_t n;                     // samples this run emits for the walk
  int64_t so, pk;                // output row and packed preview row of the first of them
  double feet[6];                // initial feet (START)
};

// One warp per walk with work, taken from a counter (the list is sorted longest first).  START runs InitOnLine, each
// appended step one OnLineAddFoot, FINISH EndPhaseOfTheWalking; the state record is loaded before and stored after.  With
// a packed preview input (pk != nullptr) the warp also moves the walk's preview carry (its last NL-1 unconsumed ZMP
// samples) in front of the new samples, zeroes the preview state of a START walk, and keeps the new carry.
__global__ void __launch_bounds__(ZD_THREADS, 3)
zmpdisc_stream_kernel(const ZdConsts K, int nwork, const ZsWork *__restrict__ work, const wg_rel_step *__restrict__ steps,
                      ZsRec *__restrict__ rec, Out out, double2 *__restrict__ pk, double2 *__restrict__ carry, int NL1,
                      double *__restrict__ pv_state, int *__restrict__ status, int *__restrict__ next_walk,
                      const double2 *__restrict__ lead_tab)
{
  extern __shared__ double2 zd_smem[];
  __shared__ Poly s_poly[ZD_WARPS][7];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double2 *u = zd_warp_smem(zd_smem, K, warp);
  double2 *histA = u + K.cap, *histB = histA + ZD_HIST, *head = histB + ZD_HIST;
  const unsigned FULL = 0xffffffffu;
  for (;;) {
    int j = 0;
    if (lane == 0) j = atomicAdd(next_walk, 1);
    j = __shfl_sync(FULL, j, 0);
    if (j >= nwork) break;
    const ZsWork &wk = work[j];
    const int b = wk.b;
    ZsRec &r = rec[b];
    const bool start = wk.flags & WG_STREAM_START;
    const int64_t F00 = start ? 0 : r.w.F0;
    const ZdDst d = {wk.so - F00, pk, wk.pk - wk.so};
    const int64_t Ltot = F00 + wk.n;
    if (pk) {
      for (int q = lane; q < wk.carry; q += 32) pk[wk.pk - wk.carry + q] = carry[(int64_t)b * NL1 + q];
      if (start && lane < 8) pv_state[8 * (int64_t)b + lane] = 0.0;
    }
    double2 *hist = histA, *hist2 = histB;
    ZdWalk w;
    wg_rel_step last;
    int si = 0;
    if (start) {
      zd_lead_in<true>(K, w, wk.feet, out, d, lead_tab, hist, head, lane);
      last = steps[wk.s0];
      si = 1;
    } else {
      w = r.w;
      last = r.last;
      if (lane < ZD_HIST) hist[lane] = r.hist[lane];
      __syncwarp();
    }
    int bad = 0;
    for (; si < wk.ns && !bad; ++si) {
      const wg_rel_step rel1 = steps[wk.s0 + si];
      bad = zd_add_foot<true>(K, w, last, rel1, out, d, Ltot, u, hist, hist2, head, s_poly[warp], lane);
      last = rel1;
    }
    if (!bad && (wk.flags & WG_STREAM_FINISH)) bad = zd_end_phase<true>(K, w, last, out, d, Ltot, u, hist, head, lane);
    if (lane == 0) { r.w = w; r.last = last; if (status) status[b] = bad; }
    if (lane < ZD_HIST) r.hist[lane] = hist[lane];
    if (pk) {                 // the new carry: the last min(L, NL-1) samples of carry + new (written by this warp above)
      __syncwarp();
      const int64_t L = wk.carry + wk.n, keep = L < NL1 ? L : NL1;
      for (int q = lane; q < keep; q += 32) carry[(int64_t)b * NL1 + q] = pk[wk.pk - wk.carry + L - keep + q];
    }
    __syncwarp();
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------------------------
struct wg_kajita_plan {
  wg_ctx *ctx;
  int B;
  wg_zmpdisc_params P;
  ZdConsts K;
  std::vector<int64_t> step_off, samp_off;
  int64_t total_steps_in;          // entries of the step array
  int64_t *d_step_off, *d_samp_off;
  wg_rel_step *d_steps;
  double *d_init_feet;
  int *d_status;
  wg_preview_plan *pv;             // nullptr until preview gains are available
  // chunks of consecutive walks for the pipelined host path
  std::vector<int> chunk_first;    // chunk c = walks [chunk_first[c], chunk_first[c+1])
  int *d_order;                    // walks sorted by decreasing length inside each chunk
  int *d_order_all;                // walks sorted by decreasing length over the whole batch (single-launch path)
  int *d_next;                     // work counter of the front-end kernel
  double2 *d_lead;                 // filtered ZMP of the lead-in samples (walk independent), n_lead entries
  // device staging for WG_MEM_HOST calls and scratch for the ZMP reference
  double *d_zmpref, *d_state, *d_com, *d_zmpout, *d_ztheta;
  wg_foot_sample *d_left, *d_right;
  int32_t *d_types;
  cudaStream_t copy_stream;
  std::vector<cudaEvent_t> ev;
};

static int zd_make_consts(const wg_zmpdisc_params *p, ZdConsts *K)
{
  if (!(p->sampling_period > 0) || !(p->preview_time > 0) || !(p->filter_time > 0)) return WG_ERR_INVALID;
  K->P = *p;
  const int n = (int)std::floor(p->filter_time / p->sampling_period);   // InitializeFilter, ZMPDiscretization.cpp:233-257
  if (n < 1 || n + 1 > ZD_MAXW || n + 1 > ZD_HIST || n - 2 > ZD_HEAD) return WG_ERR_INVALID;
  double sum = 0;
  for (int i = 0; i < n + 1; ++i) {
    const double t = std::sin((M_PI * i) / n);
    K->window[i] = t * t;
  }
  for (int i = 0; i < n + 1; ++i) sum += K->window[i];
  for (int i = 0; i < n + 1; ++i) K->window[i] /= sum;
  for (int i = n + 1; i < ZD_MAXW; ++i) K->window[i] = 0.0;
  K->nw = n + 1;
  K->n_lead = (int)(2 * p->preview_time / p->sampling_period);
  K->n_end = (int)(unsigned)std::round(p->t_double / (2 * p->sampling_period));
  K->n_tail = (int)(3.0 * p->preview_time / p->sampling_period);
  K->cap = 0;
  if (K->n_lead < ZD_HIST || K->n_end < 1) return WG_ERR_INVALID;
  return WG_OK;
}

static int zd_step_samples(const wg_zmpdisc_params *p, const wg_rel_step &s)
{
  double ds = p->t_double, ss = p->t_single;
  if (s.ds_time != 0.0) {
    ds = s.ds_time;
    ss = s.ss_time;
  }
  return (int)(unsigned)std::round((ds + ss) / p->sampling_period);
}

static int push_step(wg_rel_step *steps, int cap, int *n, const wg_rel_step &s)
{
  if (!steps || !n || *n < 0 || *n >= cap) return WG_ERR_INVALID;
  steps[(*n)++] = s;
  return WG_OK;
}

extern "C" {

void wg_zmpdisc_default_params(wg_zmpdisc_params *p)
{
  if (!p) return;
  std::memset(p, 0, sizeof *p);
  p->sampling_period = 0.005;
  p->preview_time = 1.6;
  p->t_single = 0.78;
  p->t_double = 0.02;
  p->step_height = 0.07;
  p->omega = 0.0;
  p->modulation = 0.9;
  p->filter_time = 0.05;
  p->foot_b = 0.1;     // only used when omega != 0 (robot specific: CjrlFoot::getAnklePositionInLocalFrame)
  p->foot_h = 0.105;
  p->foot_f = 0.13;
}

int wg_steps_support_foot(wg_rel_step *steps, int cap, int *n, int support_foot, double ss, double ds)
{
  wg_rel_step s;
  std::memset(&s, 0, sizeof s);
  s.sy = support_foot * 0.095;
  s.ss_time = ss;
  s.ds_time = ds;
  s.step_type = 1;
  return push_step(steps, cap, n, s);
}

int wg_steps_arc(wg_rel_step *steps, int cap, int *n, double x, double y, double arc_deg, int support_foot, double ss,
                 double ds, int *keep_last)
{
  // Steps of at most 0.15 m of arc length on a circle of radius |(x, y)| around a centre to the side of the robot; the
  // last one takes the remainder.  Each footprint sits 0.095 m inside / outside the circle.
  const double total = arc_deg * M_PI / 180.0;
  const double radius = std::sqrt(x * x + y * y);
  if (!(radius > 0)) return WG_ERR_INVALID;
  double step_len = 0.15;
  const int whole = (int)std::floor(total * radius / step_len);
  double rest = total * radius - whole * step_len;
  double turn = (step_len / radius) * 180.0 / M_PI;
  double last_turn = (total - (step_len / radius) * whole) * 180.0 / M_PI;
  int dir = -1;
  if (x < 0) { rest = -rest; dir = 1; }
  if (y < 0) { turn = -turn; last_turn = -last_turn; }
  double heading = 0.0;
  int foot = support_foot;
  for (int i = 0; i <= whole; ++i) {
    if (i == whole && rest == 0.0) break;
    const double dth = (i == whole) ? last_turn : turn;
    const double before = heading;
    heading = heading + dth;
    const double c = std::cos(heading * M_PI / 180.0), s = std::sin(heading * M_PI / 180.0);
    const double cp = std::cos(before * M_PI / 180.0), sp = std::sin(before * M_PI / 180.0);
    const double rin = radius + dir * foot * 0.095, rout = radius - dir * foot * 0.095;
    const double wx = rin * s - rout * sp, wy = -(rin * c - rout * cp);
    wg_rel_step st;
    std::memset(&st, 0, sizeof st);
    st.sx = (0.0 + c * wx) + s * wy;      // world displacement expressed in the frame of the new heading
    st.sy = (0.0 + -s * wx) + c * wy;
    st.theta = dth;
    st.ss_time = ss;
    st.ds_time = ds;
    st.step_type = 1;
    int rc = push_step(steps, cap, n, st);
    if (rc != WG_OK) return rc;
    foot = -foot;
  }
  if (keep_last) *keep_last = foot;
  return WG_OK;
}

int wg_steps_last_support(wg_rel_step *steps, int cap, int *n, int keep_last, double ss, double ds)
{
  wg_rel_step s;
  std::memset(&s, 0, sizeof s);
  s.sy = keep_last * 0.19;
  s.ss_time = ss;
  s.ds_time = ds;
  s.step_type = 0;
  return push_step(steps, cap, n, s);
}

int64_t wg_zmpdisc_sample_count(const wg_zmpdisc_params *p, int n_steps, const wg_rel_step *steps)
{
  ZdConsts K;
  if (!p || n_steps < 1 || !steps || zd_make_consts(p, &K) != WG_OK) return -1;
  int64_t n = (int64_t)K.n_lead + K.n_end + K.n_tail;
  for (int i = 1; i < n_steps; ++i) n += zd_step_samples(p, steps[i]);
  return n;
}

int wg_kajita_plan_destroy(wg_kajita_plan *pl)
{
  if (!pl) return WG_OK;
  wg_device_guard guard(pl->ctx->device);
  cudaStreamSynchronize(pl->ctx->stream);
  if (pl->copy_stream) cudaStreamSynchronize(pl->copy_stream);
  if (pl->pv) wg_preview_plan_destroy(pl->pv);
  cudaFree(pl->d_step_off); cudaFree(pl->d_samp_off); cudaFree(pl->d_steps); cudaFree(pl->d_init_feet);
  cudaFree(pl->d_status); cudaFree(pl->d_order); cudaFree(pl->d_order_all); cudaFree(pl->d_next); cudaFree(pl->d_lead);
  cudaFree(pl->d_zmpref); cudaFree(pl->d_state); cudaFree(pl->d_com); cudaFree(pl->d_zmpout); cudaFree(pl->d_ztheta);
  cudaFree(pl->d_left); cudaFree(pl->d_right); cudaFree(pl->d_types);
  for (cudaEvent_t e : pl->ev) cudaEventDestroy(e);
  if (pl->copy_stream) cudaStreamDestroy(pl->copy_stream);
  delete pl;
  return WG_OK;
}

int wg_kajita_plan_create(wg_ctx *ctx, const wg_zmpdisc_params *p, int B, const int64_t *step_off,
                          const wg_rel_step *steps, const double *init_feet, wg_kajita_plan **out)
{
  if (!ctx || !p || !out || B < 1 || !step_off || !steps || !init_feet) return WG_ERR_INVALID;
  *out = nullptr;
  ZdConsts K;
  if (zd_make_consts(p, &K) != WG_OK) return wg_fail(ctx, WG_ERR_INVALID, "wg_zmpdisc_params out of range");
  if (step_off[0] != 0) return wg_fail(ctx, WG_ERR_INVALID, "step_offsets[0] must be 0");
  wg_device_guard guard(ctx->device);
  wg_kajita_plan *pl = new (std::nothrow) wg_kajita_plan();
  if (!pl) return WG_ERR_ALLOC;
  pl->ctx = ctx; pl->B = B; pl->P = *p;
  pl->step_off.assign(step_off, step_off + B + 1);
  pl->samp_off.resize(B + 1);
  pl->samp_off[0] = 0;
  int cap = K.n_end;
  for (int b = 0; b < B; ++b) {
    const int64_t ns = step_off[b + 1] - step_off[b];
    if (ns < 1 || ns > 1000000) { delete pl; return wg_fail(ctx, WG_ERR_INVALID, "every walk needs at least one step"); }
    int64_t n = (int64_t)K.n_lead + K.n_end + K.n_tail;
    for (int64_t i = 1; i < ns; ++i) {
      const wg_rel_step &s = steps[step_off[b] + i];
      const int add = zd_step_samples(p, s);
      double ds = s.ds_time != 0.0 ? s.ds_time : p->t_double, ss = s.ds_time != 0.0 ? s.ss_time : p->t_single;
      const int n1 = (int)(unsigned)std::round(ds / p->sampling_period), n2 = (int)(unsigned)std::round(ss / p->sampling_period);
      if (n1 < 1 || n1 + n2 > add || add > 2800) {
        delete pl;
        return wg_fail(ctx, WG_ERR_INVALID, "step timing out of range (need >= 1 double-support sample, <= 2800 samples per step)");
      }
      cap = std::max(cap, add);
      n += add;
    }
    pl->samp_off[b + 1] = pl->samp_off[b] + n;
  }
  K.cap = (cap + 31) / 32 * 32;
  pl->K = K;
  pl->total_steps_in = step_off[B];
  // chunks: about 16 per batch, at least 8 walks each
  const int nchunks = std::max(1, std::min(16, B / 8));
  for (int c = 0; c <= nchunks; ++c) pl->chunk_first.push_back((int)((int64_t)B * c / nchunks));
  std::vector<int> order(B);
  for (int b = 0; b < B; ++b) order[b] = b;
  for (int c = 0; c < nchunks; ++c)
    std::stable_sort(order.begin() + pl->chunk_first[c], order.begin() + pl->chunk_first[c + 1], [&](int a, int b) {
      return pl->samp_off[a + 1] - pl->samp_off[a] > pl->samp_off[b + 1] - pl->samp_off[b];
    });
  std::vector<int> order_all(B);
  for (int b = 0; b < B; ++b) order_all[b] = b;
  std::stable_sort(order_all.begin(), order_all.end(), [&](int a, int b) {
    return pl->samp_off[a + 1] - pl->samp_off[a] > pl->samp_off[b + 1] - pl->samp_off[b];
  });
  cudaError_t e = cudaMalloc(&pl->d_step_off, sizeof(int64_t) * (B + 1));
  if (e == cudaSuccess) e = cudaMalloc(&pl->d_order_all, sizeof(int) * B);
  if (e == cudaSuccess) e = cudaMalloc(&pl->d_next, sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&pl->d_lead, sizeof(double2) * (size_t)std::max(1, pl->K.n_lead));
  if (e == cudaSuccess) e = cudaMemcpyAsync(pl->d_order_all, order_all.data(), sizeof(int) * B, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMalloc(&pl->d_samp_off, sizeof(int64_t) * (B + 1));
  if (e == cudaSuccess) e = cudaMalloc(&pl->d_steps, sizeof(wg_rel_step) * pl->total_steps_in);
  if (e == cudaSuccess) e = cudaMalloc(&pl->d_init_feet, sizeof(double) * 6 * B);
  if (e == cudaSuccess) e = cudaMalloc(&pl->d_status, sizeof(int) * B);
  if (e == cudaSuccess) e = cudaMalloc(&pl->d_order, sizeof(int) * B);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&pl->copy_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaMemcpyAsync(pl->d_step_off, step_off, sizeof(int64_t) * (B + 1), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(pl->d_samp_off, pl->samp_off.data(), sizeof(int64_t) * (B + 1), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(pl->d_steps, steps, sizeof(wg_rel_step) * pl->total_steps_in, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(pl->d_init_feet, init_feet, sizeof(double) * 6 * B, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(pl->d_order, order.data(), sizeof(int) * B, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(pl->d_status, 0, sizeof(int) * B, ctx->stream);
  if (e == cudaSuccess && pl->K.n_lead > 0) {
    zmpdisc_lead_kernel<<<(pl->K.n_lead + 127) / 128, 128, 0, ctx->stream>>>(pl->K, pl->d_lead);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  for (int i = 0; i < 2 * nchunks + 2 && e == cudaSuccess; ++i) {
    cudaEvent_t ev;
    e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e == cudaSuccess) pl->ev.push_back(ev);
  }
  if (e != cudaSuccess) {
    wg_fail(ctx, WG_ERR_CUDA, "wg_kajita_plan_create", e);
    wg_kajita_plan_destroy(pl);
    return WG_ERR_CUDA;
  }
  if (ctx->preview_ready) {
    int rc = wg_preview_plan_create(ctx, B, pl->samp_off.data(), &pl->pv);
    if (rc != WG_OK) { wg_kajita_plan_destroy(pl); return rc; }
  }
  *out = pl;
  return WG_OK;
}

const int64_t *wg_kajita_plan_sample_offsets(const wg_kajita_plan *pl) { return pl ? pl->samp_off.data() : nullptr; }
int64_t wg_kajita_plan_total_samples(const wg_kajita_plan *pl) { return pl ? pl->samp_off[pl->B] : 0; }
int64_t wg_kajita_plan_total_steps(const wg_kajita_plan *pl) { return (pl && pl->pv) ? wg_preview_plan_total_steps(pl->pv) : 0; }

int wg_kajita_plan_set_steps(wg_kajita_plan *pl, const wg_rel_step *steps, const double *init_feet)
{
  if (!pl || !steps) return WG_ERR_INVALID;
  wg_ctx *ctx = pl->ctx;
  wg_device_guard guard(ctx->device);
  WG_CUDA(ctx, cudaMemcpyAsync(pl->d_steps, steps, sizeof(wg_rel_step) * pl->total_steps_in, cudaMemcpyHostToDevice, ctx->stream));
  if (init_feet)
    WG_CUDA(ctx, cudaMemcpyAsync(pl->d_init_feet, init_feet, sizeof(double) * 6 * pl->B, cudaMemcpyHostToDevice, ctx->stream));
  return WG_OK;
}

}  // extern "C"

static int zd_launch(wg_ctx *ctx, wg_kajita_plan *pl, int b0, int b1, const Out &o)
{
  if (b1 <= b0) return WG_OK;
  const size_t smem = sizeof(double2) * (size_t)ZD_WARPS * (pl->K.cap + 2 * ZD_HIST + ZD_HEAD);
  if (smem > 200 * 1024) return wg_fail(ctx, WG_ERR_INVALID, "step segment too long for the shared-memory buffer");
  WG_SMEM_ATTR(ctx, zmpdisc_kernel, smem);
  const int walks = b1 - b0;
  const int grid = std::max(1, std::min((walks + ZD_WARPS - 1) / ZD_WARPS, ctx->sm_count * 3));
  // the whole batch uses the global longest-first order, a chunk [b0, b1) the per-chunk one (both are permutations of
  // their range stored at positions b0 .. b1-1)
  const int *order = (b0 == 0 && b1 == pl->B) ? pl->d_order_all : pl->d_order;
  WG_CUDA(ctx, cudaMemsetAsync(pl->d_next, 0, sizeof(int), ctx->stream));
  wg_prof_start(ctx, WG_K_ZMPDISC);
  zmpdisc_kernel<<<grid, ZD_THREADS, smem, ctx->stream>>>(pl->K, b0, b1, pl->d_step_off, pl->d_steps, pl->d_init_feet,
                                                         pl->d_samp_off, o, pl->d_status, order, pl->d_next, pl->d_lead);
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  return WG_OK;
}

template <class T>
static int zd_stage(wg_ctx *ctx, T **slot, size_t count)
{
  if (!*slot) WG_CUDA(ctx, cudaMalloc(slot, sizeof(T) * std::max<size_t>(1, count)));
  return WG_OK;
}

static int zd_check_status(wg_ctx *ctx, wg_kajita_plan *pl)
{  // host mode only (the stream is already synchronised): report walks the kernel refused
  std::vector<int> st(pl->B);
  WG_CUDA(ctx, cudaMemcpy(st.data(), pl->d_status, sizeof(int) * pl->B, cudaMemcpyDeviceToHost));
  for (int b = 0; b < pl->B; ++b)
    if (st[b] != 0) return wg_fail(ctx, WG_ERR_INVALID, "zmpdisc: a walk has an invalid step timing");
  return WG_OK;
}

// Internal (dimitrov.cu): run GetZMPDiscretization for every walk of the plan into device buffers.  A NULL *zmpref /
// *left / *right is replaced by the plan's own staging buffer; the step types always go to the plan's buffer.
extern "C" int wgi_kajita_discretize_device(wg_ctx *ctx, wg_kajita_plan *pl, double **zmpref, wg_foot_sample **left,
                                            wg_foot_sample **right, int32_t **types, wgi_kajita_view *view)
{
  if (!ctx || !pl || pl->ctx != ctx) return WG_ERR_INVALID;
  const size_t ns = (size_t)pl->samp_off[pl->B];
  int rc;
  if (!*zmpref) { if ((rc = zd_stage(ctx, &pl->d_zmpref, 2 * ns)) != WG_OK) return rc; *zmpref = pl->d_zmpref; }
  if (!*left) { if ((rc = zd_stage(ctx, &pl->d_left, ns)) != WG_OK) return rc; *left = pl->d_left; }
  if (!*right) { if ((rc = zd_stage(ctx, &pl->d_right, ns)) != WG_OK) return rc; *right = pl->d_right; }
  if ((rc = zd_stage(ctx, &pl->d_types, 3 * ns)) != WG_OK) return rc;
  *types = pl->d_types;
  Out o;
  o.zmpref = reinterpret_cast<double2 *>(*zmpref); o.ztheta = nullptr; o.left = *left; o.right = *right; o.types = *types;
  if ((rc = zd_launch(ctx, pl, 0, pl->B, o)) != WG_OK) return rc;
  view->B = pl->B;
  view->samp_off = pl->samp_off.data();
  view->step_off = pl->step_off.data();
  view->d_samp_off = pl->d_samp_off;
  view->d_zd_status = pl->d_status;
  view->sampling_period = pl->P.sampling_period;
  return WG_OK;
}

extern "C" {

int wg_zmpdisc_run_batch(wg_ctx *ctx, wg_kajita_plan *pl, int mem, double *zmpref_xy, double *zmp_theta,
                         wg_foot_sample *left, wg_foot_sample *right, int32_t *step_type)
{
  if (!ctx || !pl || pl->ctx != ctx) return WG_ERR_INVALID;
  wg_device_guard guard(ctx->device);
  const size_t ns = (size_t)pl->samp_off[pl->B];
  Out o;
  if (mem == WG_MEM_DEVICE) {
    o.zmpref = reinterpret_cast<double2 *>(zmpref_xy); o.ztheta = zmp_theta; o.left = left; o.right = right; o.types = step_type;
    return zd_launch(ctx, pl, 0, pl->B, o);
  }
  if (mem != WG_MEM_HOST) return WG_ERR_INVALID;
  int rc = WG_OK;
  if (zmpref_xy && (rc = zd_stage(ctx, &pl->d_zmpref, 2 * ns)) != WG_OK) return rc;
  if (zmp_theta && (rc = zd_stage(ctx, &pl->d_ztheta, ns)) != WG_OK) return rc;
  if (left && (rc = zd_stage(ctx, &pl->d_left, ns)) != WG_OK) return rc;
  if (right && (rc = zd_stage(ctx, &pl->d_right, ns)) != WG_OK) return rc;
  if (step_type && (rc = zd_stage(ctx, &pl->d_types, 3 * ns)) != WG_OK) return rc;
  o.zmpref = zmpref_xy ? reinterpret_cast<double2 *>(pl->d_zmpref) : nullptr;
  o.ztheta = zmp_theta ? pl->d_ztheta : nullptr;
  o.left = left ? pl->d_left : nullptr;
  o.right = right ? pl->d_right : nullptr;
  o.types = step_type ? pl->d_types : nullptr;
  if ((rc = zd_launch(ctx, pl, 0, pl->B, o)) != WG_OK) return rc;
  if (zmpref_xy) WG_CUDA(ctx, cudaMemcpyAsync(zmpref_xy, pl->d_zmpref, sizeof(double) * 2 * ns, cudaMemcpyDeviceToHost, ctx->stream));
  if (zmp_theta) WG_CUDA(ctx, cudaMemcpyAsync(zmp_theta, pl->d_ztheta, sizeof(double) * ns, cudaMemcpyDeviceToHost, ctx->stream));
  if (left) WG_CUDA(ctx, cudaMemcpyAsync(left, pl->d_left, sizeof(wg_foot_sample) * ns, cudaMemcpyDeviceToHost, ctx->stream));
  if (right) WG_CUDA(ctx, cudaMemcpyAsync(right, pl->d_right, sizeof(wg_foot_sample) * ns, cudaMemcpyDeviceToHost, ctx->stream));
  if (step_type) WG_CUDA(ctx, cudaMemcpyAsync(step_type, pl->d_types, sizeof(int32_t) * 3 * ns, cudaMemcpyDeviceToHost, ctx->stream));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return zd_check_status(ctx, pl);
}

int wg_kajita_run_batch(wg_ctx *ctx, wg_kajita_plan *pl, int mem, double *state, double *com_out, double *zmp_out,
                        double *zmpref_xy, wg_foot_sample *left, wg_foot_sample *right, int simulation)
{
  if (!ctx || !pl || pl->ctx != ctx || !state) return WG_ERR_INVALID;
  if (!ctx->preview_ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_preview_set_gains not called");
  wg_device_guard guard(ctx->device);
  int rc;
  if (!pl->pv && (rc = wg_preview_plan_create(ctx, pl->B, pl->samp_off.data(), &pl->pv)) != WG_OK) return rc;
  const size_t ns = (size_t)pl->samp_off[pl->B];
  Out o;
  o.ztheta = nullptr; o.types = nullptr;
  if (mem == WG_MEM_DEVICE) {
    double *zr = zmpref_xy;
    if (!zr) {
      if ((rc = zd_stage(ctx, &pl->d_zmpref, 2 * ns)) != WG_OK) return rc;
      zr = pl->d_zmpref;
    }
    o.zmpref = reinterpret_cast<double2 *>(zr); o.left = left; o.right = right;
    if ((rc = zd_launch(ctx, pl, 0, pl->B, o)) != WG_OK) return rc;
    return wg_preview_run_batch(ctx, pl->pv, WG_MEM_DEVICE, zr, state, com_out, zmp_out, simulation);
  }
  if (mem != WG_MEM_HOST) return WG_ERR_INVALID;
  // ---- host buffers: chunked, the D2H copies of chunk c run on the copy stream while chunk c+1 computes ------
  if ((rc = zd_stage(ctx, &pl->d_zmpref, 2 * ns)) != WG_OK) return rc;
  if ((rc = zd_stage(ctx, &pl->d_state, 8 * (size_t)pl->B)) != WG_OK) return rc;
  if (com_out && !pl->d_com) {   // zeroed once: rows past a walk's last preview step read back as 0
    WG_CUDA(ctx, cudaMalloc(&pl->d_com, sizeof(double) * 6 * ns));
    WG_CUDA(ctx, cudaMemsetAsync(pl->d_com, 0, sizeof(double) * 6 * ns, ctx->stream));
  }
  if (zmp_out && !pl->d_zmpout) {
    WG_CUDA(ctx, cudaMalloc(&pl->d_zmpout, sizeof(double) * 2 * ns));
    WG_CUDA(ctx, cudaMemsetAsync(pl->d_zmpout, 0, sizeof(double) * 2 * ns, ctx->stream));
  }
  if (left && (rc = zd_stage(ctx, &pl->d_left, ns)) != WG_OK) return rc;
  if (right && (rc = zd_stage(ctx, &pl->d_right, ns)) != WG_OK) return rc;
  WG_CUDA(ctx, cudaMemcpyAsync(pl->d_state, state, sizeof(double) * 8 * pl->B, cudaMemcpyHostToDevice, ctx->stream));
  o.zmpref = reinterpret_cast<double2 *>(pl->d_zmpref);
  o.left = left ? pl->d_left : nullptr;
  o.right = right ? pl->d_right : nullptr;
  const int nchunks = (int)pl->chunk_first.size() - 1;
  for (int c = 0; c < nchunks; ++c) {
    const int b0 = pl->chunk_first[c], b1 = pl->chunk_first[c + 1];
    if ((rc = zd_launch(ctx, pl, b0, b1, o)) != WG_OK) return rc;
    if ((rc = wgi_preview_launch_range(ctx, pl->pv, pl->d_order + b0, b1 - b0, pl->d_zmpref, pl->d_state,
                                       com_out ? pl->d_com : nullptr, zmp_out ? pl->d_zmpout : nullptr, simulation)) != WG_OK)
      return rc;
    WG_CUDA(ctx, cudaEventRecord(pl->ev[c], ctx->stream));
    WG_CUDA(ctx, cudaStreamWaitEvent(pl->copy_stream, pl->ev[c], 0));
    const size_t s0 = (size_t)pl->samp_off[b0], cnt = (size_t)(pl->samp_off[b1] - pl->samp_off[b0]);
    cudaStream_t cs = pl->copy_stream;
    if (com_out) WG_CUDA(ctx, cudaMemcpyAsync(com_out + 6 * s0, pl->d_com + 6 * s0, sizeof(double) * 6 * cnt, cudaMemcpyDeviceToHost, cs));
    if (zmp_out) WG_CUDA(ctx, cudaMemcpyAsync(zmp_out + 2 * s0, pl->d_zmpout + 2 * s0, sizeof(double) * 2 * cnt, cudaMemcpyDeviceToHost, cs));
    if (zmpref_xy) WG_CUDA(ctx, cudaMemcpyAsync(zmpref_xy + 2 * s0, pl->d_zmpref + 2 * s0, sizeof(double) * 2 * cnt, cudaMemcpyDeviceToHost, cs));
    if (left) WG_CUDA(ctx, cudaMemcpyAsync(left + s0, pl->d_left + s0, sizeof(wg_foot_sample) * cnt, cudaMemcpyDeviceToHost, cs));
    if (right) WG_CUDA(ctx, cudaMemcpyAsync(right + s0, pl->d_right + s0, sizeof(wg_foot_sample) * cnt, cudaMemcpyDeviceToHost, cs));
  }
  WG_CUDA(ctx, cudaMemcpyAsync(state, pl->d_state, sizeof(double) * 8 * pl->B, cudaMemcpyDeviceToHost, ctx->stream));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  WG_CUDA(ctx, cudaStreamSynchronize(pl->copy_stream));
  return zd_check_status(ctx, pl);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// On-line form: wg_kajita_stream
// ---------------------------------------------------------------------------------------------------------------
// A run's inputs travel in one blob (pinned on the host, mirrored on the device, one H2D copy per append):
//   ZsWork[nwork] (longest first) | wg_rel_step[steps of the run] | int64 preview offsets[B+1] | int preview order[npv]
struct wg_kajita_stream {
  wg_ctx *ctx;
  int B, with_preview, NL;
  ZdConsts K;                                   // K.cap: the pending run's
  std::vector<int64_t> emitted, previewed;      // per walk since its START, after the last run
  std::vector<int32_t> open;
  std::vector<int64_t> p_emitted, p_previewed;  // the same after the pending run
  std::vector<int32_t> p_open;
  std::vector<int64_t> so, co, cnt;             // row layout of the pending run (or of the last one run)
  bool pending;
  int nwork, npv;
  size_t off_steps, off_po, off_order, bytes;
  unsigned char *h_blob, *d_blob;
  size_t h_cap, d_cap;
  cudaEvent_t ev_staged;                        // the device has consumed h_blob
  ZsRec *d_rec;
  double2 *d_carry, *d_lead, *d_pk;
  double *d_state;
  int *d_status, *d_next;
  size_t pk_cap;
  wg_preview_plan *pv;
  // staging of WG_MEM_HOST runs, grown on demand
  void *d_out[7];
  size_t out_cap[7];
};

// Grow a device buffer to at least `bytes` (half as much again, to amortise).  The old contents are dropped.
static int zs_grow(wg_ctx *ctx, void **p, size_t *cap, size_t bytes)
{
  if (bytes <= *cap && *p) return WG_OK;
  const size_t want = std::max(bytes + bytes / 2, (size_t)256);
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // a kernel of an earlier run may still read the old buffer
  cudaFree(*p);
  *p = nullptr;
  *cap = 0;
  WG_CUDA(ctx, cudaMalloc(p, want));
  *cap = want;
  return WG_OK;
}

static size_t zs_align(size_t x) { return (x + 15) / 16 * 16; }

extern "C" {

int wg_kajita_stream_destroy(wg_kajita_stream *s)
{
  if (!s) return WG_OK;
  wg_device_guard guard(s->ctx->device);
  cudaStreamSynchronize(s->ctx->stream);
  if (s->pv) wg_preview_plan_destroy(s->pv);
  if (s->ev_staged) cudaEventDestroy(s->ev_staged);
  cudaFreeHost(s->h_blob);
  cudaFree(s->d_blob); cudaFree(s->d_rec); cudaFree(s->d_carry); cudaFree(s->d_lead); cudaFree(s->d_pk);
  cudaFree(s->d_state); cudaFree(s->d_status); cudaFree(s->d_next);
  for (void *p : s->d_out) cudaFree(p);
  delete s;
  return WG_OK;
}

int wg_kajita_stream_create(wg_ctx *ctx, const wg_zmpdisc_params *p, int B, int with_preview, wg_kajita_stream **out)
{
  if (!ctx || !p || !out || B < 1) return WG_ERR_INVALID;
  *out = nullptr;
  ZdConsts K;
  if (zd_make_consts(p, &K) != WG_OK) return wg_fail(ctx, WG_ERR_INVALID, "wg_zmpdisc_params out of range");
  if (with_preview && !ctx->preview_ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_preview_set_gains not called");
  wg_device_guard guard(ctx->device);
  wg_kajita_stream *s = new (std::nothrow) wg_kajita_stream();
  if (!s) return WG_ERR_ALLOC;
  s->ctx = ctx; s->B = B; s->with_preview = with_preview ? 1 : 0; s->K = K;
  s->NL = with_preview ? ctx->preview_gains.NL : 0;
  s->emitted.assign(B, 0); s->previewed.assign(B, 0); s->open.assign(B, 0);
  s->so.assign(B + 1, 0); s->co.assign(B + 1, 0); s->cnt.assign(B, 0);
  const int NL1 = std::max(1, s->NL - 1);
  cudaError_t e = cudaMalloc(&s->d_rec, sizeof(ZsRec) * B);
  if (e == cudaSuccess) e = cudaMalloc(&s->d_status, sizeof(int) * B);
  if (e == cudaSuccess) e = cudaMalloc(&s->d_next, sizeof(int));
  if (e == cudaSuccess) e = cudaMalloc(&s->d_lead, sizeof(double2) * (size_t)std::max(1, K.n_lead));
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_staged, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaMemsetAsync(s->d_status, 0, sizeof(int) * B, ctx->stream);
  if (e == cudaSuccess && with_preview) e = cudaMalloc(&s->d_state, sizeof(double) * 8 * B);
  if (e == cudaSuccess && with_preview) e = cudaMemsetAsync(s->d_state, 0, sizeof(double) * 8 * B, ctx->stream);
  if (e == cudaSuccess && with_preview) e = cudaMalloc(&s->d_carry, sizeof(double2) * NL1 * (size_t)B);
  if (e == cudaSuccess) {
    zmpdisc_lead_kernel<<<(K.n_lead + 127) / 128, 128, 0, ctx->stream>>>(K, s->d_lead);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaEventRecord(s->ev_staged, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) {
    wg_fail(ctx, WG_ERR_CUDA, "wg_kajita_stream_create", e);
    wg_kajita_stream_destroy(s);
    return WG_ERR_CUDA;
  }
  if (with_preview) {
    const int rc = wg_preview_plan_create(ctx, B, s->so.data(), &s->pv);
    if (rc != WG_OK) { wg_kajita_stream_destroy(s); return rc; }
  }
  *out = s;
  return WG_OK;
}

const int64_t *wg_kajita_stream_sample_offsets(const wg_kajita_stream *s) { return s ? s->so.data() : nullptr; }
const int64_t *wg_kajita_stream_com_offsets(const wg_kajita_stream *s) { return s ? s->co.data() : nullptr; }
const int64_t *wg_kajita_stream_com_counts(const wg_kajita_stream *s) { return s ? s->cnt.data() : nullptr; }

int wg_kajita_stream_append(wg_kajita_stream *s, const int64_t *step_off, const wg_rel_step *steps, const int32_t *flags,
                            const double *init_feet)
{
  if (!s || !step_off) return WG_ERR_INVALID;
  wg_ctx *ctx = s->ctx;
  const int B = s->B;
  const wg_zmpdisc_params &P = s->K.P;
  if (s->pending) return wg_fail(ctx, WG_ERR_INVALID, "wg_kajita_stream_append: the previous append has not been run");
  if (step_off[0] < 0) return wg_fail(ctx, WG_ERR_INVALID, "step_offsets must be non-negative and non-decreasing");
  for (int b = 0; b < B; ++b)
    if (step_off[b + 1] < step_off[b]) return wg_fail(ctx, WG_ERR_INVALID, "step_offsets must be non-negative and non-decreasing");
  if (step_off[B] > step_off[0] && !steps) return WG_ERR_INVALID;
  // ---- validate and size everything first: a refused append changes nothing ----
  std::vector<int64_t> nsamp(B, 0);
  int cap = 0;
  int64_t nsteps = 0;
  int nwork = 0;
  for (int b = 0; b < B; ++b) {
    const int64_t ns = step_off[b + 1] - step_off[b];
    const int f = flags ? flags[b] : 0;
    if (f & ~(WG_STREAM_START | WG_STREAM_FINISH)) return wg_fail(ctx, WG_ERR_INVALID, "unknown WG_STREAM_* flags");
    const bool start = f & WG_STREAM_START, fin = f & WG_STREAM_FINISH;
    if (start && ns < 1) return wg_fail(ctx, WG_ERR_INVALID, "WG_STREAM_START needs the support-foot step");
    if (start && !init_feet) return wg_fail(ctx, WG_ERR_INVALID, "WG_STREAM_START needs init_feet");
    if (!start && (ns > 0 || fin) && !s->open[b])
      return wg_fail(ctx, WG_ERR_INVALID, "steps or WG_STREAM_FINISH for a walk that is not open");
    if (ns > 1000000) return wg_fail(ctx, WG_ERR_INVALID, "too many steps for one walk");
    int64_t n = start ? s->K.n_lead : 0;
    for (int64_t i = start ? 1 : 0; i < ns; ++i) {   // the test of wg_kajita_plan_create
      const wg_rel_step &st = steps[step_off[b] + i];
      const int add = zd_step_samples(&P, st);
      double ds = st.ds_time != 0.0 ? st.ds_time : P.t_double, ss = st.ds_time != 0.0 ? st.ss_time : P.t_single;
      const int n1 = (int)(unsigned)std::round(ds / P.sampling_period), n2 = (int)(unsigned)std::round(ss / P.sampling_period);
      if (n1 < 1 || n1 + n2 > add || add > 2800)
        return wg_fail(ctx, WG_ERR_INVALID, "step timing out of range (need >= 1 double-support sample, <= 2800 samples per step)");
      cap = std::max(cap, add);
      n += add;
    }
    if (fin) {
      n += s->K.n_end + s->K.n_tail;
      cap = std::max(cap, s->K.n_end);
    }
    nsamp[b] = n;
    if (n > 0) { ++nwork; nsteps += ns; }
  }
  // ---- plan the run ----
  s->p_emitted.resize(B); s->p_previewed.resize(B); s->p_open.resize(B);
  std::vector<int> work_order, pv_order;
  s->so[0] = 0; s->co[0] = 0;
  for (int b = 0; b < B; ++b) {
    const int f = flags ? flags[b] : 0;
    const bool start = f & WG_STREAM_START, fin = f & WG_STREAM_FINISH;
    const int64_t n = nsamp[b];
    const int64_t e0 = start ? 0 : s->emitted[b], p0 = start ? 0 : s->previewed[b];
    int64_t L = 0, k = 0;
    if (n > 0 && s->with_preview) {
      L = (e0 - p0) + n;
      k = std::max<int64_t>(0, L - s->NL + 1);
    }
    s->p_emitted[b] = e0 + n;
    s->p_previewed[b] = p0 + k;
    s->p_open[b] = fin ? 0 : (start ? 1 : s->open[b]);
    s->so[b + 1] = s->so[b] + n;
    s->co[b + 1] = s->co[b] + L;
    s->cnt[b] = k;
    if (n > 0) work_order.push_back(b);
    if (k > 0) pv_order.push_back(b);
  }
  std::stable_sort(work_order.begin(), work_order.end(), [&](int a, int b) { return nsamp[a] > nsamp[b]; });
  std::stable_sort(pv_order.begin(), pv_order.end(), [&](int a, int b) {
    return s->co[a + 1] - s->co[a] > s->co[b + 1] - s->co[b];
  });
  s->nwork = nwork;
  s->npv = (int)pv_order.size();
  s->off_steps = zs_align(sizeof(ZsWork) * nwork);
  s->off_po = s->off_steps + zs_align(sizeof(wg_rel_step) * nsteps);
  s->off_order = s->off_po + zs_align(sizeof(int64_t) * (B + 1));
  s->bytes = s->off_order + zs_align(sizeof(int) * s->npv);
  // ---- stage: wait until the device has read the previous blob, then refill it ----
  wg_device_guard guard(ctx->device);
  WG_CUDA(ctx, cudaEventSynchronize(s->ev_staged));
  if (s->bytes > s->h_cap) {
    cudaFreeHost(s->h_blob);
    s->h_blob = nullptr;
    s->h_cap = 0;
    const size_t want = s->bytes + s->bytes / 2;
    WG_CUDA(ctx, cudaMallocHost(&s->h_blob, want));
    s->h_cap = want;
  }
  ZsWork *wk = reinterpret_cast<ZsWork *>(s->h_blob);
  wg_rel_step *hs = reinterpret_cast<wg_rel_step *>(s->h_blob + s->off_steps);
  int64_t at = 0;
  for (int j = 0; j < nwork; ++j) {
    const int b = work_order[j];
    const int f = flags ? flags[b] : 0;
    const int64_t ns = step_off[b + 1] - step_off[b];
    ZsWork &w = wk[j];
    w.b = b; w.flags = f; w.ns = (int32_t)ns;
    w.carry = (int32_t)((s->co[b + 1] - s->co[b]) - nsamp[b]);
    w.s0 = at; w.n = nsamp[b]; w.so = s->so[b]; w.pk = s->co[b] + w.carry;
    for (int i = 0; i < 6; ++i) w.feet[i] = (f & WG_STREAM_START) ? init_feet[6 * b + i] : 0.0;
    if (ns > 0) std::memcpy(hs + at, steps + step_off[b], sizeof(wg_rel_step) * ns);
    at += ns;
  }
  std::memcpy(s->h_blob + s->off_po, s->co.data(), sizeof(int64_t) * (B + 1));
  if (s->npv) std::memcpy(s->h_blob + s->off_order, pv_order.data(), sizeof(int) * s->npv);
  int rc = zs_grow(ctx, reinterpret_cast<void **>(&s->d_blob), &s->d_cap, s->bytes);
  if (rc != WG_OK) return rc;
  WG_CUDA(ctx, cudaMemcpyAsync(s->d_blob, s->h_blob, s->bytes, cudaMemcpyHostToDevice, ctx->stream));
  if (s->with_preview && (rc = wgi_preview_plan_set_offsets(s->pv, reinterpret_cast<const int64_t *>(s->h_blob + s->off_po))) != WG_OK)
    return rc;
  WG_CUDA(ctx, cudaEventRecord(s->ev_staged, ctx->stream));
  s->K.cap = (cap + 31) / 32 * 32;
  s->pending = true;
  return WG_OK;
}

int wg_kajita_stream_run(wg_kajita_stream *s, int mem, double *zmpref_xy, double *zmp_theta, wg_foot_sample *left,
                         wg_foot_sample *right, int32_t *step_type, double *com_out, double *zmp_out, int simulation)
{
  if (!s) return WG_ERR_INVALID;
  wg_ctx *ctx = s->ctx;
  if (mem != WG_MEM_HOST && mem != WG_MEM_DEVICE) return WG_ERR_INVALID;
  if (!s->with_preview && (com_out || zmp_out))
    return wg_fail(ctx, WG_ERR_INVALID, "wg_kajita_stream_run: com_out / zmp_out need a stream created with_preview");
  if (s->with_preview && (!ctx->preview_ready || ctx->preview_gains.NL != s->NL))
    return wg_fail(ctx, WG_ERR_NOT_READY, "wg_kajita_stream_run: the preview gains' NL changed since the stream was created");
  if (mem == WG_MEM_DEVICE &&
      ((reinterpret_cast<uintptr_t>(zmpref_xy) | reinterpret_cast<uintptr_t>(com_out) | reinterpret_cast<uintptr_t>(zmp_out) |
        reinterpret_cast<uintptr_t>(left) | reinterpret_cast<uintptr_t>(right)) & 15))
    return wg_fail(ctx, WG_ERR_INVALID, "wg_kajita_stream_run: device arrays must be 16-byte aligned");
  if (!s->pending) return WG_OK;
  wg_device_guard guard(ctx->device);
  const int B = s->B;
  const size_t ns = (size_t)s->so[B], nc = (size_t)s->co[B];
  // outputs: the caller's arrays, or (host mode) the stream's staging
  void *dst[7] = {zmpref_xy, zmp_theta, left, right, step_type, com_out, zmp_out};
  const size_t row[7] = {16, 8, sizeof(wg_foot_sample), sizeof(wg_foot_sample), 12, 48, 16};
  const size_t rows[7] = {ns, ns, ns, ns, ns, nc, nc};
  void *dev[7];
  for (int i = 0; i < 7; ++i) {
    dev[i] = dst[i];
    if (mem == WG_MEM_HOST && dst[i]) {
      const int rc = zs_grow(ctx, &s->d_out[i], &s->out_cap[i], row[i] * rows[i]);
      if (rc != WG_OK) return rc;
      dev[i] = s->d_out[i];
    }
  }
  int rc;
  if (s->with_preview && (rc = zs_grow(ctx, reinterpret_cast<void **>(&s->d_pk), &s->pk_cap, sizeof(double2) * nc)) != WG_OK)
    return rc;
  if (s->nwork > 0) {
    Out o;
    o.zmpref = reinterpret_cast<double2 *>(dev[0]); o.ztheta = static_cast<double *>(dev[1]);
    o.left = static_cast<wg_foot_sample *>(dev[2]); o.right = static_cast<wg_foot_sample *>(dev[3]);
    o.types = static_cast<int32_t *>(dev[4]);
    const size_t smem = sizeof(double2) * (size_t)ZD_WARPS * (s->K.cap + 2 * ZD_HIST + ZD_HEAD);
    if (smem > 200 * 1024) return wg_fail(ctx, WG_ERR_INVALID, "step segment too long for the shared-memory buffer");
    WG_SMEM_ATTR(ctx, zmpdisc_stream_kernel, smem);
    const int grid = std::max(1, std::min((s->nwork + ZD_WARPS - 1) / ZD_WARPS, ctx->sm_count * 3));
    const ZsWork *wk = reinterpret_cast<const ZsWork *>(s->d_blob);
    const wg_rel_step *st = reinterpret_cast<const wg_rel_step *>(s->d_blob + s->off_steps);
    WG_CUDA(ctx, cudaMemsetAsync(s->d_next, 0, sizeof(int), ctx->stream));
    wg_prof_start(ctx, WG_K_ZMPDISC);
    zmpdisc_stream_kernel<<<grid, ZD_THREADS, smem, ctx->stream>>>(s->K, s->nwork, wk, st, s->d_rec, o, s->with_preview ? s->d_pk : nullptr,
                                                                  s->d_carry, std::max(0, s->NL - 1), s->d_state, s->d_status,
                                                                  s->d_next, s->d_lead);
    wg_prof_stop(ctx);
    WG_LAUNCHED(ctx);
  }
  if (s->npv > 0) {
    const int *order = reinterpret_cast<const int *>(s->d_blob + s->off_order);
    if ((rc = wgi_preview_launch_range(ctx, s->pv, order, s->npv, reinterpret_cast<const double *>(s->d_pk), s->d_state,
                                       static_cast<double *>(dev[5]), static_cast<double *>(dev[6]), simulation)) != WG_OK)
      return rc;
  }
  if (mem == WG_MEM_HOST) {
    for (int i = 0; i < 7; ++i)
      if (dst[i] && rows[i]) WG_CUDA(ctx, cudaMemcpyAsync(dst[i], dev[i], row[i] * rows[i], cudaMemcpyDeviceToHost, ctx->stream));
    WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int b = 0; b < B; ++b)        // rows past a walk's preview steps read back as zero
      for (int i = 5; i < 7; ++i)
        if (dst[i]) {
          const size_t w = row[i] / sizeof(double);
          double *d = static_cast<double *>(dst[i]);
          std::fill(d + w * (s->co[b] + s->cnt[b]), d + w * s->co[b + 1], 0.0);
        }
    std::vector<int> st(B);
    WG_CUDA(ctx, cudaMemcpy(st.data(), s->d_status, sizeof(int) * B, cudaMemcpyDeviceToHost));
    for (int b = 0; b < B; ++b)
      if (st[b] != 0) return wg_fail(ctx, WG_ERR_INVALID, "zmpdisc: a walk has an invalid step timing");
  }
  s->emitted.swap(s->p_emitted);
  s->previewed.swap(s->p_previewed);
  s->open.swap(s->p_open);
  s->pending = false;
  return WG_OK;
}

int wg_kajita_stream_state(wg_kajita_stream *s, int mem, double *preview_state, int64_t *samples_emitted,
                           int64_t *steps_previewed, int32_t *open)
{
  if (!s || (mem != WG_MEM_HOST && mem != WG_MEM_DEVICE)) return WG_ERR_INVALID;
  wg_ctx *ctx = s->ctx;
  if (preview_state && !s->with_preview) return wg_fail(ctx, WG_ERR_INVALID, "wg_kajita_stream_state: no preview in this stream");
  const int B = s->B;
  if (samples_emitted) std::copy(s->emitted.begin(), s->emitted.end(), samples_emitted);
  if (steps_previewed) std::copy(s->previewed.begin(), s->previewed.end(), steps_previewed);
  if (open) std::copy(s->open.begin(), s->open.end(), open);
  if (preview_state) {
    wg_device_guard guard(ctx->device);
    WG_CUDA(ctx, cudaMemcpyAsync(preview_state, s->d_state, sizeof(double) * 8 * B,
                                 mem == WG_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, ctx->stream));
    if (mem == WG_MEM_HOST) WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return WG_OK;
}

}  // extern "C"
