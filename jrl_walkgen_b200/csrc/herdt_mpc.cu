// herdt_mpc.cu - the Herdt2010 closed loop on the device: one warp owns one walking instance and runs
// ZMPVelocityReferencedQP::OnLine (src/ZMPRefTrajectoryGeneration/ZMPVelocityReferencedQP.cpp:324-458) for it,
// QP period after QP period, without any host round trip:
//   lane 0   SupportFSM (src/PreviewControl/SupportFSM.cpp:58-153), GeneratorVelRef::preview_support_states
//            (generator-vel-ref.cpp:71-134), OrientationsPreview::preview_orientations (OrientationsPreview.cpp:80-251)
//            - branchy integer/compare work, a few hundred instructions;
//   32 lanes the QP (herdt_qp.cuh), compute_global_reference (generator-vel-ref.cpp:212-229);
//   20 lanes the 20 control-rate samples of the period: LinearizedInvertedPendulum2D::Interpolation
//            (LinearizedInvertedPendulum2D.cpp:157-227) and OnLineFootTrajectoryGeneration::interpolate_feet_positions
//            (OnLineFootTrajectoryGeneration.cpp:203-346), one sample per lane.
// The reference's four 5 ms deques are not materialised: the loop only ever reads their elements 0, size-2 and
// size-1 at a QP instant (always the 12th, 19th and 20th sample of the previous period), so those three samples
// are the persistent state (wg_herdt_mpc_state) and full 5 ms rows are an optional output.
#include "herdt_qp.cuh"
#include <algorithm>
#include <vector>

using herdt::N;

namespace {

constexpr int MPC_WARPS = 4;
constexpr int TPS = WG_HERDT_TICKS_PER_STEP;
constexpr double PI = 3.14159265358979323846;

struct MpcWarp {
  wg_herdt_mpc_state st;
  double yaw_s[TPS], dyaw_s[TPS];
  double support_angle0;
  int ss_branch;
};

struct Sup {  // support_state_t, privatepgtypes.hh:291-320
  int Phase, Foot, Changed;
  unsigned NbStepsLeft, StepNumber, NbInstants;
  double TimeLimit, StartTime, X, Y, Yaw;
};

// SupportFSM::update_vel_reference, SupportFSM.cpp:58-90
__device__ void update_vel_reference(wg_herdt_mpc_state &st)
{
  const double EPS = 1e-6;
  st.in_translation = (fabs(st.ref[0]) > 2 * EPS || fabs(st.ref[1]) > 2 * EPS);
  if (fabs(st.ref[2]) > EPS) {
    st.in_rotation = 1;
  } else {
    if (st.in_rotation && !st.in_translation) {
      st.ref[0] = 2 * EPS; st.ref[1] = 2 * EPS;
      if (!st.post_rotation) {
        st.fsm_support_foot = st.sup_foot; st.steps_after_rotation = 0; st.post_rotation = 1;
      } else {
        if (st.fsm_support_foot != st.sup_foot) { st.fsm_support_foot = st.sup_foot; ++st.steps_after_rotation; }
        if (st.steps_after_rotation > 2) { st.in_rotation = 0; st.post_rotation = 0; }
      }
    } else {
      st.in_rotation = 0;
    }
  }
}

// SupportFSM::set_support_state, SupportFSM.cpp:94-153
__device__ void set_support_state(const wg_herdt_mpc_params &M, const double *Ref, unsigned nb_ssds, double T,
                                  double time, unsigned pi, Sup &S)
{
  const double EPS = 1e-6;
  S.Changed = 0;
  S.NbInstants++;
  const bool given = (fabs(Ref[0]) > EPS || fabs(Ref[1]) > EPS || fabs(Ref[2]) > EPS);
  if (given && S.Phase == WG_DS && (S.TimeLimit - time - EPS) > M.dsss_period) {
    S.TimeLimit = time + M.dsss_period - T / 10.0;
    S.NbStepsLeft = nb_ssds;
  }
  if (time + EPS + pi * T >= S.TimeLimit) {
    if (S.Phase == WG_SS && !given && S.NbStepsLeft == 0) {
      S.Phase = WG_DS; S.TimeLimit = time + pi * T + M.ds_period - T / 10.0; S.Changed = 1; S.NbInstants = 0;
    } else if ((S.Phase == WG_DS && given) || (S.Phase == WG_DS && S.NbStepsLeft > 0)) {
      S.Phase = WG_SS; S.TimeLimit = time + pi * T + M.step_period - T / 10.0; S.NbStepsLeft = nb_ssds;
      S.Changed = 1; S.NbInstants = 0;
    } else if ((S.Phase == WG_SS && S.NbStepsLeft > 0) || (S.NbStepsLeft == 0 && given)) {
      S.Foot = (S.Foot == WG_LEFT) ? WG_RIGHT : WG_LEFT;
      S.Changed = 1; S.NbInstants = 0;
      S.TimeLimit = time + pi * T + M.step_period - T / 10.0;
      if (pi != 1) ++S.StepNumber;
      if (!given) S.NbStepsLeft = S.NbStepsLeft - 1;
      if (given) S.NbStepsLeft = nb_ssds;
    }
  }
}

__device__ inline void put_support(wg_herdt_qp_input &in, int i, const Sup &S)
{
  in.sup_x[i] = S.X; in.sup_y[i] = S.Y; in.sup_yaw[i] = S.Yaw;
  in.sup_foot[i] = (int8_t)S.Foot; in.sup_phase[i] = (int8_t)S.Phase;
  in.sup_step[i] = (int8_t)S.StepNumber; in.sup_changed[i] = (int8_t)S.Changed;
}

// GeneratorVelRef::preview_support_states, generator-vel-ref.cpp:71-134
__device__ void preview_support_states(const wg_herdt_mpc_params &M, double T, wg_herdt_mpc_state &st,
                                       wg_herdt_qp_input &in, double time)
{
  Sup cur;
  cur.Phase = st.sup_phase; cur.Foot = st.sup_foot; cur.Changed = st.sup_changed;
  cur.NbStepsLeft = (unsigned)st.sup_steps_left; cur.StepNumber = (unsigned)st.sup_step_number;
  cur.NbInstants = (unsigned)st.sup_nb_instants;
  cur.TimeLimit = st.sup_time_limit; cur.StartTime = st.sup_start_time;
  cur.X = st.sup_x; cur.Y = st.sup_y; cur.Yaw = st.sup_yaw;
  const unsigned nb = (unsigned)st.nb_steps_ssds;
  set_support_state(M, st.ref, nb, T, time, 0, cur);
  if (cur.Changed) {
    const wg_herdt_foot_sample &F = st.foot[cur.Foot][0];      // Final{Left,Right}FootTraj_deq.front()
    cur.X = F.x; cur.Y = F.y; cur.Yaw = F.theta * PI / 180.0; cur.StartTime = time;
  }
  st.sup_phase = cur.Phase; st.sup_foot = cur.Foot; st.sup_changed = cur.Changed;
  st.sup_steps_left = (int)cur.NbStepsLeft; st.sup_step_number = (int)cur.StepNumber;
  st.sup_nb_instants = (int)cur.NbInstants;
  st.sup_time_limit = cur.TimeLimit; st.sup_start_time = cur.StartTime;
  st.sup_x = cur.X; st.sup_y = cur.Y; st.sup_yaw = cur.Yaw;
  put_support(in, 0, cur);
  Sup prw = cur;
  prw.StepNumber = 0;
  for (unsigned pi = 1; pi <= (unsigned)N; ++pi) {
    set_support_state(M, st.ref, nb, T, time, pi, prw);
    if (prw.Changed) {
      if (pi == 1) {
        const wg_herdt_foot_sample &F = st.foot[prw.Foot][2];  // ...deq.back()
        prw.X = F.x; prw.Y = F.y; prw.Yaw = F.theta * PI / 180.0;
        prw.StartTime = time + pi * M.Ts;
      }
      if (prw.StepNumber > 0) { prw.X = 0.0; prw.Y = 0.0; }
    }
    put_support(in, (int)pi, prw);
  }
}

// OrientationsPreview::verify_angle_hip_joint, OrientationsPreview.cpp:271-300
__device__ bool verify_angle_hip_joint(const wg_herdt_mpc_params &M, double T, wg_herdt_mpc_state &st, int foot,
                                       double PrwTrunkAngleEnd, double CurrentSupportFootAngle, unsigned StepNumber)
{
  const double uJ = M.hip_upper[foot], lJ = M.hip_lower[foot];
  const double JointLimit = (st.trunk_t_yaw[1] < 0.0) ? lJ : uJ;
  if (fabs(PrwTrunkAngleEnd - CurrentSupportFootAngle) > fabs(JointLimit)) {
    st.trunk_t_yaw[1] = (CurrentSupportFootAngle + 0.9 * JointLimit - st.trunk_yaw[0] - st.trunk_yaw[1] * T / 2.0) /
                        (st.support_time_passed + StepNumber * M.step_period - T / 2.0);
    return false;
  }
  return true;
}

// OrientationsPreview::preview_orientations, OrientationsPreview.cpp:80-251.  Writes the previewed support
// yaws into in.sup_yaw[1..N]; returns SupportOrientations_deq[0].
__device__ double preview_orientations(const wg_herdt_mpc_params &M, double T, wg_herdt_mpc_state &st,
                                       wg_herdt_qp_input &in, double Time)
{
  const double SSP = M.step_period, EPSo = 0.00000001;
  double SupportAngles[8];
  int nsa = 0;
  const int cs_phase = st.sup_phase, cs_foot = st.sup_foot;
  const double cs_limit = st.sup_time_limit;
  // verify_acceleration_hip_joint, :254-268
  if (cs_phase != WG_DS) {
    if (fabs(st.ref[2] - st.trunk_yaw[1]) > 2.0 / 3.0 * T * M.hip_acc_limit) {
      const double sgn = (st.ref[2] - st.trunk_yaw[1] < 0.0) ? -1.0 : 1.0;
      st.trunk_t_yaw[1] = st.trunk_yaw[1] + sgn * 2.0 / 3.0 * T * M.hip_acc_limit;
    } else
      st.trunk_t_yaw[1] = st.ref[2];
  } else
    st.trunk_t_yaw[1] = 0.0;
  bool TrunkVelOK = false, TrunkAngleOK = false;
  double FirstFootPreviewed = 0.0;
  const double signRotVelTrunk = (st.trunk_t_yaw[1] < 0.0) ? -1.0 : 1.0;
  unsigned StepNumber = 0;
  double PreviewedTrunkAngleEnd = 0.0;
  const unsigned last_step = (unsigned)((int)ceil((N + 1) * T / M.step_period));
  int guard = 0;
  while (!TrunkVelOK) {
    if (++guard > 1000) break;
    const double CurrentSupportAngle = st.foot[cs_foot][0].theta * PI / 180.0;
    if (cs_phase != WG_DS) {
      TrunkAngleOK = false;
      int g2 = 0;
      while (!TrunkAngleOK) {
        if (++g2 > 1000) break;
        if (fabs(st.trunk_t_yaw[1] - st.trunk_yaw[1]) > EPSo) {
          const double a = st.trunk_yaw[0], b = st.trunk_yaw[1], c = 0.0;
          const double d = 3.0 * (st.trunk_t_yaw[1] - st.trunk_yaw[1]) / (T * T);
          const double e = -2.0 * d / (3.0 * T);
          st.trunk_t_yaw[0] = a + b * T + 1.0 / 2.0 * c * T * T + 1.0 / 3.0 * d * T * T * T + 1.0 / 4.0 * e * T * T * T * T;
        } else
          st.trunk_t_yaw[0] = st.trunk_yaw[0] + st.trunk_yaw[1] * T;
        st.support_time_passed = cs_limit - Time;
        PreviewedTrunkAngleEnd = st.trunk_t_yaw[0] + st.trunk_t_yaw[1] * (st.support_time_passed - T);
        TrunkAngleOK = verify_angle_hip_joint(M, T, st, cs_foot, PreviewedTrunkAngleEnd, CurrentSupportAngle, StepNumber);
      }
    } else {
      st.support_time_passed = cs_limit + SSP - Time;
      FirstFootPreviewed = 1;
      if (nsa < 8) SupportAngles[nsa++] = CurrentSupportAngle;
      st.trunk_t_yaw[0] = PreviewedTrunkAngleEnd = st.trunk_yaw[0];
    }
    double PreviousSupportAngle = CurrentSupportAngle;
    double PreviewedSupportFoot = (cs_foot == WG_LEFT) ? 1.0 : -1.0;
    for (StepNumber = (unsigned)FirstFootPreviewed; StepNumber <= last_step; StepNumber++) {
      PreviewedSupportFoot = -PreviewedSupportFoot;
      double PreviewedSupportAngle = PreviewedTrunkAngleEnd + st.trunk_t_yaw[1] * SSP / 2.0;
      // verify_velocity_hip_joint takes the angle BY VALUE in the reference (OrientationsPreview.hh): no effect
      if (PreviewedSupportFoot * (PreviousSupportAngle - PreviewedSupportAngle) - EPSo > M.feet_cross_limit)
        PreviewedSupportAngle = PreviousSupportAngle + signRotVelTrunk * M.feet_cross_limit;
      else if (fabs(PreviewedSupportAngle - PreviousSupportAngle) > M.foot_vel_limit * SSP)
        PreviewedSupportAngle = PreviousSupportAngle + PreviewedSupportFoot * M.foot_vel_limit * (SSP - T);
      TrunkAngleOK = verify_angle_hip_joint(M, T, st, cs_foot, PreviewedTrunkAngleEnd, CurrentSupportAngle, StepNumber);
      if (!TrunkAngleOK) { nsa = 0; TrunkVelOK = false; break; }
      if (nsa < 8) SupportAngles[nsa++] = PreviewedSupportAngle;
      PreviewedTrunkAngleEnd = PreviewedTrunkAngleEnd + SSP * st.trunk_t_yaw[1];
      PreviousSupportAngle = PreviewedSupportAngle;
      TrunkVelOK = true;
    }
  }
  int j = 0;
  double supportAngle = in.sup_yaw[0];
  for (int i = 1; i <= N; ++i) {
    if (in.sup_changed[i]) { supportAngle = (j < nsa) ? SupportAngles[j] : supportAngle; j++; }
    in.sup_yaw[i] = supportAngle;
  }
  return nsa > 0 ? SupportAngles[0] : 0.0;
}

// OrientationsPreview::interpolate_trunk_orientation, OrientationsPreview.cpp:369-418 (the condition inside the
// loop reads the trunk state the loop itself updates, hence serial)
__device__ void interpolate_trunk_orientation(const wg_herdt_mpc_params &M, double T, MpcWarp &w, double Time)
{
  wg_herdt_mpc_state &st = w.st;
  if (st.sup_phase == WG_SS && Time + 3.0 / 2.0 * T < st.sup_time_limit) {
    const double a = st.trunk_yaw[1];
    const double c = 3.0 * (st.trunk_t_yaw[1] - st.trunk_yaw[1]) / (T * T);
    const double d = -2.0 * c / (3.0 * T);
    const double Theta = st.trunk_yaw[0];
    for (int k = 0; k < TPS; k++) {
      const double tT = (double)(k + 1) * M.Ts;
      if (fabs(st.trunk_t_yaw[1] - st.trunk_yaw[1]) - 0.000001 > 0) {
        st.trunk_yaw[0] = (((1.0 / 4.0 * d * tT + 1.0 / 3.0 * c) * tT) * tT + a) * tT + Theta;
        st.trunk_yaw[1] = ((d * tT + c) * tT) * tT + a;
        st.trunk_yaw[2] = (3.0 * d * tT + 2.0 * c) * tT;
      } else
        st.trunk_yaw[0] += M.Ts * st.trunk_t_yaw[1];
      w.yaw_s[k] = st.trunk_yaw[0];
      w.dyaw_s[k] = st.trunk_yaw[1];
    }
  } else {
    for (int k = 0; k < TPS; k++) { w.yaw_s[k] = st.trunk_yaw[0]; w.dyaw_s[k] = st.trunk_yaw[1]; }
  }
}

// Polynome::Compute / ComputeDerivative / ComputeSecDerivative in ascending powers (Polynome.cpp:44-75)
template <int DEG> __device__ inline double pval(const double *c, double t)
{ double r = 0, pt = 1; for (int i = 0; i <= DEG; ++i) { r += c[i] * pt; pt *= t; } return r; }
template <int DEG> __device__ inline double pd1(const double *c, double t)
{ double r = 0, pt = 1; for (int i = 1; i <= DEG; ++i) { r += i * c[i] * pt; pt *= t; } return r; }
template <int DEG> __device__ inline double pd2(const double *c, double t)
{ double r = 0, pt = 1; for (int i = 2; i <= DEG; ++i) { r += i * (i - 1) * c[i] * pt; pt *= t; } return r; }

// Polynome5::SetParameters(FT, FP, InitPos, InitSpeed, InitAcc), PolynomeFoot.cpp:226-240
__device__ inline void poly5_set(double *c, double FT, double FP, double ip, double is, double ia)
{
  c[0] = ip; c[1] = is; c[2] = ia / 2.0;
  double tmp = FT * FT * FT;
  c[3] = (-3.0 / 2.0 * ia * FT * FT - 6.0 * is * FT - 10.0 * ip + 10.0 * FP) / tmp;
  tmp *= FT;
  c[4] = (3.0 / 2.0 * ia * FT * FT + 8.0 * is * FT + 15.0 * ip - 15.0 * FP) / tmp;
  tmp *= FT;
  c[5] = (-1.0 / 2.0 * ia * FT * FT - 3.0 * is * FT - 6.0 * ip + 6.0 * FP) / tmp;
}
// Polynome3::SetParametersWithInitPosInitSpeed, PolynomeFoot.cpp:57-78
__device__ inline void poly3_init(double *c, double FT, double FP, double ip, double is)
{
  c[0] = ip; c[1] = is;
  const double tmp = FT * FT;
  if (FT == 0.0) { c[2] = 0; c[3] = 0; }
  else { c[2] = (3 * FP - 3 * ip - 2 * is * FT) / tmp; c[3] = (is * FT + 2 * ip - 2 * FP) / (tmp * FT); }
}
// Polynome4::SetParameters, PolynomeFoot.cpp:100-121
__device__ inline void poly4_set(double *c, double FT, double MP)
{
  c[0] = 0; c[1] = 0;
  double tmp = FT * FT;
  if (MP == 0.0 || tmp == 0.0) { c[2] = c[3] = c[4] = 0; }
  else { c[2] = 16.0 * MP / tmp; tmp *= FT; c[3] = -32.0 * MP / tmp; tmp *= FT; c[4] = 16.0 * MP / tmp; }
}

__device__ inline void write_tick(wg_herdt_tick *row, const double *com11, const wg_herdt_foot_sample &L,
                                  const wg_herdt_foot_sample &R)
{
  double *d = reinterpret_cast<double *>(row);
#pragma unroll
  for (int i = 0; i < 11; ++i) d[i] = com11[i];
  d[11] = 0.0;
  row->left = L;
  row->right = R;
}

struct MpcState {
  wg_herdt_mpc_params h_params;
  wg_herdt_mpc_params *d_params = nullptr;
  bool ready = false;
  // staging for WG_MEM_HOST calls
  void *d_states = nullptr, *d_ref = nullptr, *d_ticks = nullptr, *d_steps = nullptr, *d_qpin = nullptr;
  size_t cap_states = 0, cap_ref = 0, cap_ticks = 0, cap_steps = 0, cap_qpin = 0;
  // per-period records (pre -> herdt_qp_kernel -> post)
  void *d_rec = nullptr, *d_out = nullptr, *d_scr = nullptr;
  size_t cap_rec = 0, cap_out = 0, cap_scr = 0;
};

// ---------------------------------------------------------------------------------------------------------------
// A period is three launches: "clock ticks + FSM + orientation preview + QP record" -> herdt_qp_kernel (the open-loop
// solver: 16 warps/SM, T in global memory) -> "jerk, LIPM, feet, state update".  The state and the QP records cross HBM
// once per period (2.7 KB per instance).
// ---------------------------------------------------------------------------------------------------------------
struct MpcScratch {
  double support_angle0;
  int fire, stopped;
};

// The QP record of a firing instance, part 1 (lane 0): VelRef_ from NewVelRef_, the support FSM and the previewed supports,
// the orientation preview and the CoM.  mpc_pre_kernel and online_tick_kernel both build their records with these two.
__device__ __forceinline__ void qp_record_fsm(const wg_herdt_mpc_params &M, double T, MpcWarp &w, wg_herdt_qp_input &in)
{
  wg_herdt_mpc_state &st = w.st;
  st.ref[0] = st.new_ref[0]; st.ref[1] = st.new_ref[1]; st.ref[2] = st.new_ref[2];
  update_vel_reference(st);
  // zero the input record's byte fields through put_support below
  preview_support_states(M, T, st, in, st.clock);
  w.support_angle0 = preview_orientations(M, T, st, in, st.clock);
  in.com_x[0] = st.com_x[0]; in.com_x[1] = st.com_x[1]; in.com_x[2] = st.com_x[2];
  in.com_y[0] = st.com_y[0]; in.com_y[1] = st.com_y[1]; in.com_y[2] = st.com_y[2];
  in.pad_[0] = in.pad_[1] = in.pad_[2] = in.pad_[3] = 0;
}

// Part 2 (lanes 0..N-1): compute_global_reference, generator-vel-ref.cpp:212-229 (TrunkOrientations_deq: current, next,
// then constant)
__device__ __forceinline__ void qp_record_reference(const wg_herdt_mpc_state &st, double T, int lane, wg_herdt_qp_input &in)
{
  if (lane < N) {
    const double yaw = (lane == 0) ? st.trunk_yaw[0]
                                   : (lane == 1 ? st.trunk_t_yaw[0] : st.trunk_t_yaw[0] + st.trunk_t_yaw[1] * T);
    double sn, cs;
    sincos(yaw, &sn, &cs);
    in.ref_x[lane] = st.ref[0] * cs - st.ref[1] * sn;
    in.ref_y[lane] = st.ref[1] * cs + st.ref[0] * sn;
  }
}

__global__ void __launch_bounds__(MPC_WARPS * 32)
mpc_pre_kernel(int B, int step, const herdt::Consts *__restrict__ Cp, const wg_herdt_mpc_params *__restrict__ Mp,
               wg_herdt_mpc_state *__restrict__ states, const double *__restrict__ vel_ref,
               wg_herdt_qp_input *__restrict__ qp_rec, MpcScratch *__restrict__ scratch)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  struct Pre { wg_herdt_qp_input in; };
  Pre *pres = reinterpret_cast<Pre *>(smem_raw);
  MpcWarp *mws = reinterpret_cast<MpcWarp *>(smem_raw + sizeof(Pre) * MPC_WARPS);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const herdt::Consts &C = *Cp;
  const wg_herdt_mpc_params &M = *Mp;
  Pre &s = pres[warp];
  MpcWarp &w = mws[warp];
  wg_herdt_mpc_state &st = w.st;
  const double T = C.P.T;
  constexpr int STW = (int)(sizeof(wg_herdt_mpc_state) / 8);
  for (int b = blockIdx.x * MPC_WARPS + warp; b < B; b += gridDim.x * MPC_WARPS) {
    {
      const double *src = reinterpret_cast<const double *>(states + b);
      double *dst = reinterpret_cast<double *>(&st);
      for (int e = lane; e < STW; e += 32) dst[e] = src[e];
    }
    __syncwarp();
    if (step == 0 && vel_ref && lane < 3 && st.online_mode) st.new_ref[lane] = vel_ref[3 * (size_t)b + lane];   // ended instances stay untouched
    __syncwarp();
    int stopped = (step == 0) ? 0 : scratch[b].stopped;
    int fire = 0;
    if (!stopped && st.online_mode) {
      // ---- control ticks until the QP fires: OnLine() runs every 5 ms and solves when
      // time + 0.00001 > UpperTimeLimitToUpdate_ (ZMPVelocityReferencedQP.cpp:346), i.e. at the first tick and then
      // at the LAST tick of every 20-tick period (clock = 0.1 k), when the deques still hold 9 samples
      if (lane == 0) {
        int n = 0;
        for (; n < 2 * TPS && st.online_mode; ++n) {
          st.clock += M.Ts;
          if (st.ending_phase && st.clock >= st.time_to_stop) st.online_mode = 0;   // this call still runs the test below
          if (st.clock + 0.00001 > st.upper_time_limit) { fire = 1; break; }
        }
        if (fire) {
          qp_record_fsm(M, T, w, s.in);
        } else if (st.online_mode) {
          st.last_fail = -1;                           // clock and QP cadence out of step: stop this instance
          st.online_mode = 0;
        }
      }
      fire = __shfl_sync(0xffffffffu, fire, 0);
      __syncwarp();
      qp_record_reference(st, T, lane, s.in);
      __syncwarp();
      if (fire) {
        const double *src = reinterpret_cast<const double *>(&s.in);
        double *dst = reinterpret_cast<double *>(qp_rec + b);
        for (int e = lane; e < (int)(sizeof(wg_herdt_qp_input) / 8); e += 32) dst[e] = src[e];
      }
    }
    if (!fire) stopped = 1;       // later periods of this call leave the instance alone
    if (lane == 0) { scratch[b].support_angle0 = w.support_angle0; scratch[b].fire = fire; scratch[b].stopped = stopped; }
    {
      double *dst = reinterpret_cast<double *>(states + b);
      const double *src = reinterpret_cast<const double *>(&st);
      for (int e = lane; e < STW; e += 32) dst[e] = src[e];
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(MPC_WARPS * 32)
mpc_post_kernel(int B, int step, int nsteps, const herdt::Consts *__restrict__ Cp, const wg_herdt_mpc_params *__restrict__ Mp,
                wg_herdt_mpc_state *__restrict__ states, const wg_herdt_qp_output *__restrict__ qp_out,
                const MpcScratch *__restrict__ scratch, wg_herdt_tick *__restrict__ ticks,
                wg_herdt_mpc_step *__restrict__ steps)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  MpcWarp *mws = reinterpret_cast<MpcWarp *>(smem_raw);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const herdt::Consts &C = *Cp;
  const wg_herdt_mpc_params &M = *Mp;
  MpcWarp &w = mws[warp];
  wg_herdt_mpc_state &st = w.st;
  const double T = C.P.T;
  constexpr int STW = (int)(sizeof(wg_herdt_mpc_state) / 8);
  for (int b = blockIdx.x * MPC_WARPS + warp; b < B; b += gridDim.x * MPC_WARPS) {
    if (!scratch[b].fire) continue;
    {
      const double *src = reinterpret_cast<const double *>(states + b);
      double *dst = reinterpret_cast<double *>(&st);
      for (int e = lane; e < STW; e += 32) dst[e] = src[e];
    }
    __syncwarp();
    if (lane == 0) w.support_angle0 = scratch[b].support_angle0;
    __syncwarp();
    {
      const wg_herdt_qp_output &o = qp_out[b];
      const int ns = (o.n_vars - 2 * N) / 2;
      const double qjx = o.x[0], qjy = o.x[N], qfx = ns > 0 ? o.x[2 * N] : 0.0, qfy = ns > 0 ? o.x[2 * N + ns] : 0.0;
      const int qfail = o.fail, qiter = o.iterations;
      int qact = 0;
      for (int e = lane; e < WG_HERDT_MAX_ROWS + 1; e += 32) qact += (o.lagr[e] != 0.0);
      qact = __reduce_add_sync(0xffffffffu, qact);
      const double Time = st.clock;
      // ---- jerk to apply (ZMPVelocityReferencedQP.cpp:404-431)
      double jx = qjx, jy = qjy;
      int running = 1;
      if (M.return_to_centre && st.sup_steps_left == 0) {
        jx = (st.foot[0][0].x + st.foot[1][0].x) / 2 - st.com_front[0];
        jy = (st.foot[0][0].y + st.foot[1][0].y) / 2 - st.com_front[3];
        running = st.running;
        if (fabs(jx) < 1e-3 && fabs(jy) < 1e-3) running = 0;
        const double tf = 0.75;
        jx = 6 / (tf * tf * tf) * (jx - tf * st.com_front[1] - (tf * tf / 2) * st.com_front[2]);
        jy = 6 / (tf * tf * tf) * (jy - tf * st.com_front[4] - (tf * tf / 2) * st.com_front[5]);
      }
      // ---- trunk yaw of the 20 samples (serial), feet polynomials (uniform)
      if (lane == 0) interpolate_trunk_orientation(M, T, w, Time);
      const int cs_foot = st.sup_foot, cs_phase = st.sup_phase;
      const bool ss_branch = (cs_phase == WG_SS && Time + 3.0 / 2.0 * T < st.sup_time_limit);
      const int swing = (cs_foot == WG_LEFT) ? WG_RIGHT : WG_LEFT;
      __syncwarp();

      // ---- the 20 samples: lane k-1 computes sample k
      const int k = lane + 1;
      double com11[11];
      {
        const double t = k * M.Ts;   // (lk + 1) * m_T
        const double *cx = st.com_x, *cy = st.com_y;
        com11[0] = cx[0] + t * cx[1] + 0.5 * t * t * cx[2] + t * t * t * jx / 6.0;
        com11[1] = cx[1] + t * cx[2] + 0.5 * t * t * jx;
        com11[2] = cx[2] + t * jx;
        com11[3] = cy[0] + t * cy[1] + 0.5 * t * t * cy[2] + t * t * t * jy / 6.0;
        com11[4] = cy[1] + t * cy[2] + 0.5 * t * t * jy;
        com11[5] = cy[2] + t * jy;
        com11[6] = st.com_height;
        com11[7] = (lane < TPS) ? w.yaw_s[lane] : 0.0;
        com11[8] = (lane < TPS) ? w.dyaw_s[lane] : 0.0;
        const double C2 = -st.com_height / 9.81;
        com11[9] = 1.0 * com11[0] + 0.0 * com11[1] + C2 * com11[2];
        com11[10] = 1.0 * com11[3] + 0.0 * com11[4] + C2 * com11[5];
      }
      wg_herdt_foot_sample fl, fr;       // this lane's sample of the left / right foot
      const wg_herdt_foot_sample old_back_l = st.foot[0][2], old_back_r = st.foot[1][2];
      wg_herdt_foot_sample back_l = old_back_l, back_r = old_back_r;   // deque element size-1 after this period's rewrite
      if (ss_branch) {
        // interpret_solution + interpolate_feet_positions, OnLineFootTrajectoryGeneration.cpp:203-346
        const double Sign = (cs_foot == WG_LEFT) ? 1.0 : -1.0;
        double FPx, FPy;
        if (st.sup_steps_left > 0 && ns > 0) { FPx = qfx; FPy = qfy; }
        else {
          FPx = st.sup_x + Sign * sin(st.sup_yaw) * C.P.ds_feet_distance;
          FPy = st.sup_y - Sign * cos(st.sup_yaw) * C.P.ds_feet_distance;
        }
        const double Local = Time - (st.sup_time_limit - (M.t_double + M.t_single));
        const double Unlocked = M.t_single * 0.9;
        const double EndOfLiftOff = (M.t_single - Unlocked) * 0.5;
        const double StartLanding = EndOfLiftOff + Unlocked;
        double SwingTimePassed = 0.0;
        if (Local > EndOfLiftOff) SwingTimePassed = Local - EndOfLiftOff;
        const wg_herdt_foot_sample Last = st.foot[swing][2];
        const wg_herdt_foot_sample Hold = st.foot[cs_foot][1];
        const double TimeInterval = Unlocked - SwingTimePassed;
        double PX[6], PY[6], PT[4];
        poly5_set(PX, TimeInterval, FPx, Last.x, Last.dx, Last.ddx);
        poly5_set(PY, TimeInterval, FPy, Last.y, Last.dy, Last.ddy);
        if (st.sup_changed && lane == 0) poly4_set(st.poly_z, M.t_single, M.step_height);
        __syncwarp();
        poly3_init(PT, TimeInterval, w.support_angle0 * 180.0 / PI, Last.theta, Last.dtheta);
        const double Interp = (double)k * M.Ts;
        const double tt = Local + Interp;
        wg_herdt_foot_sample sw;
        sw.x = sw.y = sw.z = sw.theta = sw.dx = sw.dy = sw.dz = sw.dtheta = sw.ddx = sw.ddy = 0.0;
        const bool hold = (tt <= EndOfLiftOff || tt >= StartLanding);
        if (!hold) {
          const double rt = (Local < EndOfLiftOff && tt > EndOfLiftOff) ? tt - EndOfLiftOff : Interp;
          sw.x = pval<5>(PX, rt); sw.dx = pd1<5>(PX, rt); sw.ddx = pd2<5>(PX, rt);
          sw.y = pval<5>(PY, rt); sw.dy = pd1<5>(PY, rt); sw.ddy = pd2<5>(PY, rt);
          sw.theta = pval<3>(PT, rt); sw.dtheta = pd1<3>(PT, rt);
        }
        // held samples copy (x, y, theta) of their predecessor: before lift-off that is the deque's last element,
        // after landing the last interpolated sample
        const unsigned nonhold = __ballot_sync(0xffffffffu, !hold && lane < TPS);
        int srcl = -1;
        if (hold) {
          const unsigned below = nonhold & ((1u << lane) - 1u);
          srcl = below ? 31 - __clz(below) : -1;
        }
        const double hx = __shfl_sync(0xffffffffu, sw.x, srcl < 0 ? 0 : srcl);
        const double hy = __shfl_sync(0xffffffffu, sw.y, srcl < 0 ? 0 : srcl);
        const double ht = __shfl_sync(0xffffffffu, sw.theta, srcl < 0 ? 0 : srcl);
        if (hold) {
          if (srcl < 0) { sw.x = Last.x; sw.y = Last.y; sw.theta = Last.theta; }
          else { sw.x = hx; sw.y = hy; sw.theta = ht; }
        }
        sw.z = pval<4>(st.poly_z, tt);
        sw.dz = pd1<4>(st.poly_z, tt);
        if (swing == WG_LEFT) { fl = sw; fr = Hold; } else { fr = sw; fl = Hold; }
      } else {
        // double support, or the landing margin of a single support: every new sample, and the deque's last element,
        // become copies of element size-2 (OnLineFootTrajectoryGeneration.cpp:331-343)
        fl = st.foot[0][1]; fr = st.foot[1][1];
        back_l = fl; back_r = fr;
      }
      __syncwarp();

      // ---- emit rows 7+20k .. 26+20k: the inherited last element (final now), then samples 1..19
      if (ticks) {
        wg_herdt_tick *row0 = ticks + ((size_t)b * nsteps + step) * TPS;
        if (lane == 0) write_tick(row0, st.com_back, back_l, back_r);
        if (lane < TPS - 1) write_tick(row0 + 1 + lane, com11, fl, fr);
      }
      __syncwarp();
      // ---- new persistent samples: deque elements 0, size-2, size-1 at the next QP = samples 12, 19, 20
      if (lane == 11) {
        st.foot[0][0] = fl; st.foot[1][0] = fr;
#pragma unroll
        for (int i = 0; i < 6; ++i) st.com_front[i] = com11[i];
      }
      if (lane == 18) { st.foot[0][1] = fl; st.foot[1][1] = fr; }
      if (lane == 19) {
        st.foot[0][2] = fl; st.foot[1][2] = fr;
#pragma unroll
        for (int i = 0; i < 11; ++i) st.com_back[i] = com11[i];
      }
      __syncwarp();
      if (lane == 0) {
        // LinearizedInvertedPendulum2D::OneIteration with T = QP_T_ (LinearizedInvertedPendulum2D.cpp:230-264)
        double nx[3], ny[3];
        const double A[3][3] = {{1.0, T, T * T / 2.0}, {0.0, 1.0, T}, {0.0, 0.0, 1.0}};
        const double Bv[3] = {T * T * T / 6.0, T * T / 2.0, T};
        for (int i = 0; i < 3; ++i) {
          double a = 0, bb = 0;
          for (int j = 0; j < 3; ++j) { a += A[i][j] * st.com_x[j]; bb += A[i][j] * st.com_y[j]; }
          nx[i] = a + jx * Bv[i]; ny[i] = bb + jy * Bv[i];
        }
        for (int i = 0; i < 3; ++i) { st.com_x[i] = nx[i]; st.com_y[i] = ny[i]; }
        st.running = running;
        st.qp_count++;
        st.last_fail = qfail;
        if (qfail) st.fail_count++;
        st.iterations_total += qiter;
        if (!st.ending_phase) st.time_to_stop = st.upper_time_limit + T * N;
        st.upper_time_limit = st.upper_time_limit + T;
        if (steps) {
          wg_herdt_mpc_step &o = steps[(size_t)b * nsteps + step];
          o.time = Time;
          for (int i = 0; i < 3; ++i) { o.com_x[i] = nx[i]; o.com_y[i] = ny[i]; }
          o.jerk_x = jx; o.jerk_y = jy;
          o.next_foot_x = ns > 0 ? qfx : 0.0; o.next_foot_y = ns > 0 ? qfy : 0.0;
          o.sup_x = st.sup_x; o.sup_y = st.sup_y; o.sup_yaw = st.sup_yaw;
          o.sup_foot = st.sup_foot; o.sup_phase = st.sup_phase; o.n_prw_steps = ns; o.fail = qfail;
          o.iterations = qiter; o.n_active = qact; o.pad_[0] = o.pad_[1] = 0;
        }
      }
      __syncwarp();
        }
    {
      double *dst = reinterpret_cast<double *>(states + b);
      const double *src = reinterpret_cast<const double *>(&st);
      for (int e = lane; e < STW; e += 32) dst[e] = src[e];
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------------------------
// The on-line generator (wg_herdt_online_*): one control tick is
//   online_tick_kernel -> herdt_qp_kernel -> mpc_post_kernel (nsteps = 1, rows staged per robot) -> online_merge_pop_kernel.
// Robots that do not fire this tick are skipped by the solver and the post kernel through MpcScratch::fire.
// ---------------------------------------------------------------------------------------------------------------
constexpr int QCAP = WG_HERDT_ONLINE_QUEUE;
constexpr int TICK_DOUBLES = (int)(sizeof(wg_herdt_tick) / 8);   // 32: one double per lane
static_assert(TICK_DOUBLES == 32, "a deque element is moved as one double per lane");

struct OnlineSlot {   // the deques of one robot: ring of QCAP rows from `head`, `count` rows; `running` = PGI m_Running
  int32_t head, count, running, pad_;
};

// Lane e's double of the row the state holds as the deques' not-yet-emitted back: com_back, then the feet at index 2.
__device__ inline double back_row_double(const wg_herdt_mpc_state &st, int e)
{
  if (e < 11) return st.com_back[e];
  if (e == 11) return 0.0;
  const double *f = reinterpret_cast<const double *>(e < 22 ? &st.foot[0][2] : &st.foot[1][2]);
  return f[e < 22 ? e - 12 : e - 22];
}

// :HerdtOnline for robots idx[0..n): the state record, and the TimeBuffer_/Ts buffered start samples as the deques
__global__ void __launch_bounds__(MPC_WARPS * 32)
online_start_kernel(int n, const int32_t *__restrict__ idx, const wg_herdt_mpc_state *__restrict__ init,
                    wg_herdt_mpc_state *__restrict__ states, wg_herdt_tick *__restrict__ queue, OnlineSlot *__restrict__ slots)
{
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int STW = (int)(sizeof(wg_herdt_mpc_state) / 8);
  for (int i = blockIdx.x * MPC_WARPS + warp; i < n; i += gridDim.x * MPC_WARPS) {
    const int b = idx[i];
    const double *src = reinterpret_cast<const double *>(init + i);
    double *dst = reinterpret_cast<double *>(states + b);
    for (int e = lane; e < STW; e += 32) dst[e] = src[e];
    const double v = back_row_double(init[i], lane);
    double *q = reinterpret_cast<double *>(queue + (size_t)b * QCAP);
    for (int k = 0; k < 8; ++k) q[k * TICK_DOUBLES + lane] = v;
    if (lane == 0) { OnlineSlot s; s.head = 0; s.count = 8; s.running = 1; s.pad_ = 0; slots[b] = s; }
  }
}

// Commands, clock, end-of-on-line test and QP instant of every running robot (lane = robot); then the QP record of each
// robot that fires, built by the whole warp exactly as mpc_pre_kernel builds it.
__global__ void __launch_bounds__(MPC_WARPS * 32)
online_tick_kernel(int B, const herdt::Consts *__restrict__ Cp, const wg_herdt_mpc_params *__restrict__ Mp,
                   wg_herdt_mpc_state *__restrict__ states, const OnlineSlot *__restrict__ slots,
                   const wg_herdt_command *__restrict__ cmd, wg_herdt_qp_input *__restrict__ qp_rec,
                   MpcScratch *__restrict__ scratch)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  wg_herdt_qp_input *ins = reinterpret_cast<wg_herdt_qp_input *>(smem_raw);
  MpcWarp *mws = reinterpret_cast<MpcWarp *>(smem_raw + sizeof(wg_herdt_qp_input) * MPC_WARPS);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const wg_herdt_mpc_params &M = *Mp;
  wg_herdt_qp_input &in = ins[warp];
  MpcWarp &w = mws[warp];
  wg_herdt_mpc_state &st = w.st;
  const double T = Cp->P.T;
  constexpr int STW = (int)(sizeof(wg_herdt_mpc_state) / 8);
  for (int base = (blockIdx.x * MPC_WARPS + warp) * 32; base < B; base += gridDim.x * MPC_WARPS * 32) {
    const int b = base + lane;
    int fire = 0;
    if (b < B && slots[b].running) {
      wg_herdt_mpc_state &g = states[b];
      if (cmd) {
        const wg_herdt_command &c = cmd[b];
        if (c.flags & WG_CMD_VEL) { g.new_ref[0] = c.vel[0]; g.new_ref[1] = c.vel[1]; g.new_ref[2] = c.vel[2]; }
        if (c.flags & WG_CMD_STOP) g.ending_phase = 1;
      }
      const double clock = g.clock + M.Ts;
      g.clock = clock;
      if (g.online_mode) {
        // ZMPVelocityReferencedQP.cpp:331-346, in the order of mpc_pre_kernel's tick loop: a QP instant whose end test
        // ends the on-line mode still solves
        if (g.ending_phase && clock >= g.time_to_stop) g.online_mode = 0;
        if (clock + 0.00001 > g.upper_time_limit) {
          if (slots[b].count + TPS <= QCAP) fire = 1;
          else { g.last_fail = -1; g.online_mode = 0; }   // the period would overflow the deques
        }
      }
    }
    if (b < B) scratch[b].fire = fire;
    unsigned todo = __ballot_sync(0xffffffffu, fire);
    __syncwarp();
    while (todo) {
      const int bf = base + __ffs(todo) - 1;
      todo &= todo - 1;
      {
        const double *src = reinterpret_cast<const double *>(states + bf);
        double *dst = reinterpret_cast<double *>(&st);
        for (int e = lane; e < STW; e += 32) dst[e] = src[e];
      }
      __syncwarp();
      if (lane == 0) qp_record_fsm(M, T, w, in);
      __syncwarp();
      qp_record_reference(st, T, lane, in);
      __syncwarp();
      {
        const double *src = reinterpret_cast<const double *>(&in);
        double *dst = reinterpret_cast<double *>(qp_rec + bf);
        for (int e = lane; e < (int)(sizeof(wg_herdt_qp_input) / 8); e += 32) dst[e] = src[e];
      }
      {
        double *dst = reinterpret_cast<double *>(states + bf);
        const double *src = reinterpret_cast<const double *>(&st);
        for (int e = lane; e < STW; e += 32) dst[e] = src[e];
      }
      if (lane == 0) scratch[bf].support_angle0 = w.support_angle0;
      __syncwarp();
    }
  }
}

// Merge the staged period into the deques of each robot that fired (walkgen_host.cpp:580-596: the inherited back element
// takes the new feet only, then samples 1..19, then the state's back sample), then pop one element of every running
// robot (walkgen_host_pgi.cpp:512-539).  One warp per robot, lane e moves double e of a row.
__global__ void __launch_bounds__(MPC_WARPS * 32)
online_merge_pop_kernel(int B, const wg_herdt_mpc_state *__restrict__ states, const MpcScratch *__restrict__ scratch,
                        const wg_herdt_tick *__restrict__ staged, wg_herdt_tick *__restrict__ queue,
                        OnlineSlot *__restrict__ slots, wg_herdt_tick *__restrict__ rows, int8_t *__restrict__ running)
{
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int b = blockIdx.x * MPC_WARPS + warp; b < B; b += gridDim.x * MPC_WARPS) {
    OnlineSlot s = slots[b];
    int popped = 0;
    if (s.running) {
      double *q = reinterpret_cast<double *>(queue + (size_t)b * QCAP);
      if (scratch[b].fire) {
        const double *src = reinterpret_cast<const double *>(staged + (size_t)b * TPS);
        if (s.count > 0 && lane >= 12) q[((s.head + s.count - 1) % QCAP) * TICK_DOUBLES + lane] = src[lane];
        for (int k = 1; k < TPS; ++k) q[((s.head + s.count + k - 1) % QCAP) * TICK_DOUBLES + lane] = src[k * TICK_DOUBLES + lane];
        q[((s.head + s.count + TPS - 1) % QCAP) * TICK_DOUBLES + lane] = back_row_double(states[b], lane);
        s.count += TPS;
      }
      if (s.count == 0) {
        s.running = 0;
      } else {
        if (rows) reinterpret_cast<double *>(rows + b)[lane] = q[s.head * TICK_DOUBLES + lane];
        s.head = (s.head + 1) % QCAP;
        s.count--;
        popped = 1;
      }
      __syncwarp();
      if (lane == 0) slots[b] = s;
    }
    if (running && lane == 0) running[b] = (int8_t)popped;
  }
}

}  // namespace

const herdt::Consts *wg_herdt_device_consts(wg_ctx *ctx);
const herdt::Consts *wg_herdt_host_consts(wg_ctx *ctx);
int wg_herdt_qp_solve_device(wg_ctx *ctx, int B, const wg_herdt_qp_input *in, wg_herdt_qp_output *out,
                             const herdt::LaunchOpts &opt);

void wg_herdt_mpc_release(wg_ctx *ctx)
{
  if (!ctx->herdt_mpc) return;
  MpcState *m = static_cast<MpcState *>(ctx->herdt_mpc);
  cudaFree(m->d_params); cudaFree(m->d_states); cudaFree(m->d_ref); cudaFree(m->d_ticks); cudaFree(m->d_steps);
  cudaFree(m->d_qpin); cudaFree(m->d_rec); cudaFree(m->d_out); cudaFree(m->d_scr);
  delete m;
  ctx->herdt_mpc = nullptr;
}

static MpcState *mpc_of(wg_ctx *ctx)
{
  if (!ctx->herdt_mpc) ctx->herdt_mpc = new MpcState();
  return static_cast<MpcState *>(ctx->herdt_mpc);
}

extern "C" {

void wg_herdt_mpc_default_params(wg_herdt_mpc_params *p)
{
  if (!p) return;
  std::memset(p, 0, sizeof *p);
  p->Ts = 0.005; p->time_buffer = 0.04;
  p->step_period = 0.8; p->ds_period = 1e9; p->dsss_period = 0.8;
  p->t_single = 0.7; p->t_double = 0.1; p->step_height = 0.05;
  // OrientationsPreview.cpp:52-53, :64-65: the defaults the reference falls back to when the model reports
  // equal bounds; the right hip reuses the left values (sic)
  p->hip_lower[0] = p->hip_lower[1] = -30.0 / 180.0 * PI;
  p->hip_upper[0] = p->hip_upper[1] = 45.0 / 180.0 * PI;
  p->foot_vel_limit = 3.54108;
  p->hip_acc_limit = 0.1;
  p->feet_cross_limit = 5.0 / 180.0 * PI;
  p->nb_steps_ssds = 2;
  p->return_to_centre = 1;
  p->warm_start = 0;   // measured on B200: 24.8 -> 23.5 active-set changes per QP, +8 % closed-loop rate (the guess is taken row by
                       // row, each row costs the two triangular products of a regular iteration); cold start stays the default
}

int wg_herdt_mpc_set_params(wg_ctx *ctx, const wg_herdt_mpc_params *params)
{
  if (!ctx || !params || !(params->Ts > 0.0)) return WG_ERR_INVALID;
  if (!wg_herdt_host_consts(ctx)) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_herdt_set_params not called");
  const double T = wg_herdt_host_consts(ctx)->P.T;
  if ((int)(T / params->Ts) != WG_HERDT_TICKS_PER_STEP)
    return wg_fail(ctx, WG_ERR_INVALID, "QP period / control period must be 20 (WG_HERDT_TICKS_PER_STEP)");
  if ((int)(params->time_buffer / params->Ts) != 8)
    return wg_fail(ctx, WG_ERR_INVALID, "time_buffer / Ts must be 8 samples");
  wg_device_guard guard(ctx->device);
  MpcState *m = mpc_of(ctx);
  m->h_params = *params;
  if (!m->d_params) WG_CUDA(ctx, cudaMalloc(&m->d_params, sizeof *params));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  WG_CUDA(ctx, cudaMemcpy(m->d_params, params, sizeof *params, cudaMemcpyHostToDevice));
  m->ready = true;
  return WG_OK;
}

static int mpc_init_impl(wg_ctx *ctx, int mem, int B, const double *init, int init_stride, wg_herdt_mpc_state *states, bool full);

int wg_herdt_mpc_init(wg_ctx *ctx, int mem, int B, const double *init9, int init_stride, wg_herdt_mpc_state *states)
{
  return mpc_init_impl(ctx, mem, B, init9, init_stride, states, false);
}

int wg_herdt_mpc_init15(wg_ctx *ctx, int mem, int B, const double *init15, int init_stride, wg_herdt_mpc_state *states)
{
  return mpc_init_impl(ctx, mem, B, init15, init_stride, states, true);
}

// qp_count, fail_count, iterations_total summed over the instances, and the number of instances still on line
__global__ void mpc_stats_kernel(int B, const wg_herdt_mpc_state *__restrict__ states, double *__restrict__ out4)
{
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    a0 += states[b].qp_count; a1 += states[b].fail_count; a2 += (double)states[b].iterations_total; a3 += states[b].online_mode ? 1.0 : 0.0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a0 += __shfl_xor_sync(0xffffffffu, a0, o); a1 += __shfl_xor_sync(0xffffffffu, a1, o);
    a2 += __shfl_xor_sync(0xffffffffu, a2, o); a3 += __shfl_xor_sync(0xffffffffu, a3, o);
  }
  if ((threadIdx.x & 31) == 0) { atomicAdd(out4, a0); atomicAdd(out4 + 1, a1); atomicAdd(out4 + 2, a2); atomicAdd(out4 + 3, a3); }
}

int wg_herdt_mpc_stats(wg_ctx *ctx, int B, const wg_herdt_mpc_state *d_states, double *d_out4)
{
  if (!ctx || B < 0 || !d_out4 || (B > 0 && !d_states)) return WG_ERR_INVALID;
  wg_device_guard guard(ctx->device);
  WG_CUDA(ctx, cudaMemsetAsync(d_out4, 0, sizeof(double) * 4, ctx->stream));
  if (B == 0) return WG_OK;
  mpc_stats_kernel<<<std::max(1, std::min((B + 255) / 256, ctx->sm_count * 4)), 256, 0, ctx->stream>>>(B, d_states, d_out4);
  WG_LAUNCHED(ctx);
  return WG_OK;
}

static int mpc_init_impl(wg_ctx *ctx, int mem, int B, const double *init9, int init_stride, wg_herdt_mpc_state *states, bool full)
{
  if (!ctx || B < 0 || (B > 0 && (!init9 || !states)) || init_stride < 0) return WG_ERR_INVALID;
  MpcState *m = mpc_of(ctx);
  if (!m->ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_herdt_mpc_set_params not called");
  if (B == 0) return WG_OK;
  wg_device_guard guard(ctx->device);
  // ZMPVelocityReferencedQP::InitOnLine, ZMPVelocityReferencedQP.cpp:213-319
  std::vector<wg_herdt_mpc_state> h((size_t)B);
  for (int b = 0; b < B; ++b) {
    const double *src = init9 + (size_t)b * init_stride;
    // init15 = {com x, dx, ddx, y, dy, ddy, z, trunk yaw, trunk yaw rate, left foot x, y, theta, right foot x, y, theta}
    double in[9];
    if (full) { in[0] = src[0]; in[1] = src[3]; in[2] = src[6]; for (int k = 0; k < 6; ++k) in[3 + k] = src[9 + k]; }
    else for (int k = 0; k < 9; ++k) in[k] = src[k];
    wg_herdt_mpc_state &s = h[b];
    std::memset(&s, 0, sizeof s);
    s.online_mode = 1; s.time_to_stop = -1.0;
    s.com_x[0] = in[0]; s.com_y[0] = in[1]; s.com_height = in[2];
    for (int f = 0; f < 2; ++f)
      for (int q = 0; q < 3; ++q) {
        s.foot[f][q].x = in[3 + 3 * f]; s.foot[f][q].y = in[4 + 3 * f]; s.foot[f][q].theta = in[5 + 3 * f];
      }
    s.com_front[0] = in[0]; s.com_front[3] = in[1];
    s.com_back[0] = in[0]; s.com_back[3] = in[1]; s.com_back[6] = in[2];   // ZMP of the buffered samples: (0, 0)
    s.trunk_yaw[0] = 0.0;
    s.sup_phase = WG_DS; s.sup_foot = WG_LEFT; s.sup_time_limit = 1000000000; s.sup_steps_left = 1;
    s.sup_x = in[3]; s.sup_y = in[4]; s.sup_yaw = in[5] * PI / 180.0;
    s.nb_steps_ssds = m->h_params.nb_steps_ssds;
    if (full) {
      // InitOnLine copies the whole lStartingCOMState into CoM_ and hands it to OrientPrw_->CurrentTrunkState
      // (ZMPVelocityReferencedQP.cpp:292-301): velocity, acceleration, trunk yaw and yaw rate of a start that is not at rest
      s.com_x[1] = src[1]; s.com_x[2] = src[2]; s.com_y[1] = src[4]; s.com_y[2] = src[5];
      s.com_front[1] = src[1]; s.com_front[2] = src[2]; s.com_front[4] = src[4]; s.com_front[5] = src[5];
      s.com_back[1] = src[1]; s.com_back[2] = src[2]; s.com_back[4] = src[4]; s.com_back[5] = src[5];
      s.trunk_yaw[0] = src[7]; s.trunk_yaw[1] = src[8];
      s.com_back[7] = src[7]; s.com_back[8] = src[8];
    }
  }
  if (mem == WG_MEM_HOST) { std::memcpy(states, h.data(), sizeof(wg_herdt_mpc_state) * (size_t)B); return WG_OK; }
  if (mem != WG_MEM_DEVICE) return WG_ERR_INVALID;
  WG_CUDA(ctx, cudaMemcpyAsync(states, h.data(), sizeof(wg_herdt_mpc_state) * (size_t)B, cudaMemcpyHostToDevice, ctx->stream));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return WG_OK;
}

// the per-period records of B instances (pre / tick kernel -> herdt_qp_kernel -> mpc_post_kernel)
static int mpc_grow_records(wg_ctx *ctx, MpcState *m, size_t nb)
{
  int rc;
  const size_t had = m->cap_rec;
  if ((rc = wgi_grow_scratch(ctx, &m->d_rec, &m->cap_rec, sizeof(wg_herdt_qp_input) * nb)) != WG_OK) return rc;
  if ((rc = wgi_grow_scratch(ctx, &m->d_out, &m->cap_out, sizeof(wg_herdt_qp_output) * nb)) != WG_OK) return rc;
  if ((rc = wgi_grow_scratch(ctx, &m->d_scr, &m->cap_scr, sizeof(MpcScratch) * nb)) != WG_OK) return rc;
  if (m->cap_rec != had)   // records of instances that do not fire are solved too: keep them well defined
    WG_CUDA(ctx, cudaMemsetAsync(m->d_rec, 0, sizeof(wg_herdt_qp_input) * nb, ctx->stream));
  return WG_OK;
}

// the QP solve of one period: instances whose MpcScratch::fire is 0 are skipped; warm start from / active set back into
// each instance's state
static int mpc_solve(wg_ctx *ctx, MpcState *m, int B, wg_herdt_mpc_state *states)
{
  herdt::LaunchOpts opt;
  MpcScratch *scr = static_cast<MpcScratch *>(m->d_scr);
  opt.fire = reinterpret_cast<const unsigned char *>(&scr->fire); opt.fire_stride = sizeof(MpcScratch);
  unsigned char *warm = reinterpret_cast<unsigned char *>(&states->warm);
  if (m->h_params.warm_start) { opt.guess = warm; opt.guess_stride = sizeof(wg_herdt_mpc_state); }
  opt.active_out = warm; opt.active_stride = sizeof(wg_herdt_mpc_state);
  opt.age = 1;
  return wg_herdt_qp_solve_device(ctx, B, static_cast<const wg_herdt_qp_input *>(m->d_rec),
                                  static_cast<wg_herdt_qp_output *>(m->d_out), opt);
}

static int mpc_launch(wg_ctx *ctx, MpcState *m, int B, int nsteps, wg_herdt_mpc_state *states, const double *vel_ref,
                      wg_herdt_tick *ticks, wg_herdt_mpc_step *steps, wg_herdt_qp_input *qp_in)
{
  const size_t nb = (size_t)B;
  int rc;
  if ((rc = mpc_grow_records(ctx, m, nb)) != WG_OK) return rc;
  wg_herdt_qp_input *rec = static_cast<wg_herdt_qp_input *>(m->d_rec);
  wg_herdt_qp_output *out = static_cast<wg_herdt_qp_output *>(m->d_out);
  MpcScratch *scr = static_cast<MpcScratch *>(m->d_scr);
  const int blocks = std::max(1, std::min((B + MPC_WARPS - 1) / MPC_WARPS, ctx->sm_count * 16));
  const size_t smem_pre = (sizeof(wg_herdt_qp_input) + sizeof(MpcWarp)) * MPC_WARPS, smem_post = sizeof(MpcWarp) * MPC_WARPS;
  for (int step = 0; step < nsteps; ++step) {
    wg_prof_start(ctx, WG_K_HERDT_MPC);
    mpc_pre_kernel<<<blocks, MPC_WARPS * 32, smem_pre, ctx->stream>>>(B, step, wg_herdt_device_consts(ctx), m->d_params, states,
                                                                      vel_ref, rec, scr);
    wg_prof_stop(ctx);
    WG_LAUNCHED(ctx);
    if ((rc = mpc_solve(ctx, m, B, states)) != WG_OK) return rc;
    wg_prof_start(ctx, WG_K_HERDT_MPC);
    mpc_post_kernel<<<blocks, MPC_WARPS * 32, smem_post, ctx->stream>>>(B, step, nsteps, wg_herdt_device_consts(ctx), m->d_params,
                                                                        states, out, scr, ticks, steps);
    wg_prof_stop(ctx);
    WG_LAUNCHED(ctx);
  }
  if (qp_in) WG_CUDA(ctx, cudaMemcpyAsync(qp_in, rec, sizeof(wg_herdt_qp_input) * nb, cudaMemcpyDeviceToDevice, ctx->stream));
  return WG_OK;
}

int wg_herdt_mpc_run_batch(wg_ctx *ctx, int mem, int B, int nsteps, wg_herdt_mpc_state *states, const double *vel_ref,
                           wg_herdt_tick *ticks, wg_herdt_mpc_step *steps, wg_herdt_qp_input *qp_in)
{
  if (!ctx || B < 0 || nsteps < 0 || (B > 0 && !states)) return WG_ERR_INVALID;
  MpcState *m = mpc_of(ctx);
  if (!m->ready || !wg_herdt_device_consts(ctx))
    return wg_fail(ctx, WG_ERR_NOT_READY, "wg_herdt_set_params / wg_herdt_mpc_set_params not called");
  if (B == 0 || nsteps == 0) return WG_OK;
  wg_device_guard guard(ctx->device);
  if (mem == WG_MEM_DEVICE) return mpc_launch(ctx, m, B, nsteps, states, vel_ref, ticks, steps, qp_in);
  if (mem != WG_MEM_HOST) return WG_ERR_INVALID;
  const size_t nb = (size_t)B, nt = nb * nsteps * TPS, nsx = nb * nsteps;
  int rc;
  if ((rc = wgi_grow_scratch(ctx, &m->d_states, &m->cap_states, sizeof(wg_herdt_mpc_state) * nb)) != WG_OK) return rc;
  if (vel_ref && (rc = wgi_grow_scratch(ctx, &m->d_ref, &m->cap_ref, sizeof(double) * 3 * nb)) != WG_OK) return rc;
  if (ticks && (rc = wgi_grow_scratch(ctx, &m->d_ticks, &m->cap_ticks, sizeof(wg_herdt_tick) * nt)) != WG_OK) return rc;
  if (steps && (rc = wgi_grow_scratch(ctx, &m->d_steps, &m->cap_steps, sizeof(wg_herdt_mpc_step) * nsx)) != WG_OK) return rc;
  if (qp_in && (rc = wgi_grow_scratch(ctx, &m->d_qpin, &m->cap_qpin, sizeof(wg_herdt_qp_input) * nb)) != WG_OK) return rc;
  WG_CUDA(ctx, cudaMemcpyAsync(m->d_states, states, sizeof(wg_herdt_mpc_state) * nb, cudaMemcpyHostToDevice, ctx->stream));
  if (vel_ref) WG_CUDA(ctx, cudaMemcpyAsync(m->d_ref, vel_ref, sizeof(double) * 3 * nb, cudaMemcpyHostToDevice, ctx->stream));
  if (ticks) WG_CUDA(ctx, cudaMemsetAsync(m->d_ticks, 0, sizeof(wg_herdt_tick) * nt, ctx->stream));
  if (steps) WG_CUDA(ctx, cudaMemsetAsync(m->d_steps, 0, sizeof(wg_herdt_mpc_step) * nsx, ctx->stream));
  if (qp_in) WG_CUDA(ctx, cudaMemsetAsync(m->d_qpin, 0, sizeof(wg_herdt_qp_input) * nb, ctx->stream));
  rc = mpc_launch(ctx, m, B, nsteps, static_cast<wg_herdt_mpc_state *>(m->d_states),
                  vel_ref ? static_cast<const double *>(m->d_ref) : nullptr,
                  ticks ? static_cast<wg_herdt_tick *>(m->d_ticks) : nullptr,
                  steps ? static_cast<wg_herdt_mpc_step *>(m->d_steps) : nullptr,
                  qp_in ? static_cast<wg_herdt_qp_input *>(m->d_qpin) : nullptr);
  if (rc != WG_OK) return rc;
  WG_CUDA(ctx, cudaMemcpyAsync(states, m->d_states, sizeof(wg_herdt_mpc_state) * nb, cudaMemcpyDeviceToHost, ctx->stream));
  if (ticks) WG_CUDA(ctx, cudaMemcpyAsync(ticks, m->d_ticks, sizeof(wg_herdt_tick) * nt, cudaMemcpyDeviceToHost, ctx->stream));
  if (steps) WG_CUDA(ctx, cudaMemcpyAsync(steps, m->d_steps, sizeof(wg_herdt_mpc_step) * nsx, cudaMemcpyDeviceToHost, ctx->stream));
  if (qp_in) WG_CUDA(ctx, cudaMemcpyAsync(qp_in, m->d_qpin, sizeof(wg_herdt_qp_input) * nb, cudaMemcpyDeviceToHost, ctx->stream));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return WG_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// wg_herdt_online_*
// ---------------------------------------------------------------------------------------------------------------
struct wg_herdt_online {
  wg_ctx *ctx = nullptr;
  int B = 0;
  wg_herdt_mpc_state *d_states = nullptr;
  wg_herdt_tick *d_queue = nullptr;    // [B][QCAP]
  OnlineSlot *d_slots = nullptr;       // [B]
  wg_herdt_tick *d_staged = nullptr;   // [B][20]: the rows mpc_post_kernel writes for a robot that fires
  // staging of start (init states, indices) and of WG_MEM_HOST ticks (commands, rows, running)
  void *d_init = nullptr, *d_idx = nullptr, *d_cmd = nullptr, *d_rows = nullptr, *d_run = nullptr;
  size_t cap_init = 0, cap_idx = 0, cap_cmd = 0, cap_rows = 0, cap_run = 0;
};

static void online_free(wg_herdt_online *h)
{
  cudaFree(h->d_states); cudaFree(h->d_queue); cudaFree(h->d_slots); cudaFree(h->d_staged);
  cudaFree(h->d_init); cudaFree(h->d_idx); cudaFree(h->d_cmd); cudaFree(h->d_rows); cudaFree(h->d_run);
  delete h;
}

static int online_ticks(wg_herdt_online *h, MpcState *m, int nticks, const wg_herdt_command *cmd, wg_herdt_tick *rows,
                        int8_t *running)
{
  wg_ctx *ctx = h->ctx;
  const int B = h->B;
  const size_t nb = (size_t)B;
  int rc;
  if ((rc = mpc_grow_records(ctx, m, nb)) != WG_OK) return rc;
  wg_herdt_qp_input *rec = static_cast<wg_herdt_qp_input *>(m->d_rec);
  wg_herdt_qp_output *out = static_cast<wg_herdt_qp_output *>(m->d_out);
  MpcScratch *scr = static_cast<MpcScratch *>(m->d_scr);
  const herdt::Consts *consts = wg_herdt_device_consts(ctx);
  const int blocks_tick = std::max(1, std::min((B + 32 * MPC_WARPS - 1) / (32 * MPC_WARPS), ctx->sm_count * 16));
  const int blocks = std::max(1, std::min((B + MPC_WARPS - 1) / MPC_WARPS, ctx->sm_count * 16));
  const size_t smem_tick = (sizeof(wg_herdt_qp_input) + sizeof(MpcWarp)) * MPC_WARPS, smem_post = sizeof(MpcWarp) * MPC_WARPS;
  for (int t = 0; t < nticks; ++t) {
    wg_prof_start(ctx, WG_K_HERDT_MPC);
    online_tick_kernel<<<blocks_tick, MPC_WARPS * 32, smem_tick, ctx->stream>>>(B, consts, m->d_params, h->d_states, h->d_slots,
                                                                                cmd ? cmd + (size_t)t * nb : nullptr, rec, scr);
    wg_prof_stop(ctx);
    WG_LAUNCHED(ctx);
    if ((rc = mpc_solve(ctx, m, B, h->d_states)) != WG_OK) return rc;
    wg_prof_start(ctx, WG_K_HERDT_MPC);
    mpc_post_kernel<<<blocks, MPC_WARPS * 32, smem_post, ctx->stream>>>(B, 0, 1, consts, m->d_params, h->d_states, out, scr,
                                                                        h->d_staged, nullptr);
    wg_prof_stop(ctx);
    WG_LAUNCHED(ctx);
    wg_prof_start(ctx, WG_K_HERDT_MPC);
    online_merge_pop_kernel<<<blocks, MPC_WARPS * 32, 0, ctx->stream>>>(B, h->d_states, scr, h->d_staged, h->d_queue, h->d_slots,
                                                                        rows ? rows + (size_t)t * nb : nullptr,
                                                                        running ? running + (size_t)t * nb : nullptr);
    wg_prof_stop(ctx);
    WG_LAUNCHED(ctx);
  }
  return WG_OK;
}

extern "C" {

int wg_herdt_online_create(wg_ctx *ctx, int B, wg_herdt_online **out)
{
  if (!ctx || B < 0 || !out) return WG_ERR_INVALID;
  *out = nullptr;
  wg_device_guard guard(ctx->device);
  wg_herdt_online *h = new wg_herdt_online();
  h->ctx = ctx;
  h->B = B;
  const size_t nb = std::max<size_t>(1, (size_t)B);
  cudaError_t e = cudaMalloc(&h->d_states, sizeof(wg_herdt_mpc_state) * nb);
  if (e == cudaSuccess) e = cudaMalloc(&h->d_queue, sizeof(wg_herdt_tick) * QCAP * nb);
  if (e == cudaSuccess) e = cudaMalloc(&h->d_slots, sizeof(OnlineSlot) * nb);
  if (e == cudaSuccess) e = cudaMalloc(&h->d_staged, sizeof(wg_herdt_tick) * TPS * nb);
  if (e == cudaSuccess) e = cudaMemsetAsync(h->d_states, 0, sizeof(wg_herdt_mpc_state) * nb, ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(h->d_slots, 0, sizeof(OnlineSlot) * nb, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) {
    online_free(h);
    return wg_fail(ctx, e == cudaErrorMemoryAllocation ? WG_ERR_ALLOC : WG_ERR_CUDA, "wg_herdt_online_create", e);
  }
  *out = h;
  return WG_OK;
}

int wg_herdt_online_destroy(wg_herdt_online *h)
{
  if (!h) return WG_ERR_INVALID;
  wg_device_guard guard(h->ctx->device);
  cudaStreamSynchronize(h->ctx->stream);
  online_free(h);
  return WG_OK;
}

wg_herdt_mpc_state *wg_herdt_online_states(wg_herdt_online *h)
{
  return h ? h->d_states : nullptr;
}

int wg_herdt_online_start(wg_herdt_online *h, int n, const int32_t *idx_host, const double *init15_host, int init_stride)
{
  if (!h || n < 0 || init_stride < 0 || (n > 0 && (!idx_host || !init15_host))) return WG_ERR_INVALID;
  wg_ctx *ctx = h->ctx;
  std::vector<char> seen((size_t)h->B, 0);
  for (int i = 0; i < n; ++i) {
    const int32_t b = idx_host[i];
    if (b < 0 || b >= h->B || seen[b]) return wg_fail(ctx, WG_ERR_INVALID, "wg_herdt_online_start: index out of range or repeated");
    seen[b] = 1;
  }
  MpcState *m = mpc_of(ctx);
  if (!m->ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_herdt_mpc_set_params not called");
  if (n == 0) return WG_OK;
  wg_device_guard guard(ctx->device);
  std::vector<wg_herdt_mpc_state> init((size_t)n);
  int rc = mpc_init_impl(ctx, WG_MEM_HOST, n, init15_host, init_stride, init.data(), true);
  if (rc != WG_OK) return rc;
  if ((rc = wgi_grow_scratch(ctx, &h->d_init, &h->cap_init, sizeof(wg_herdt_mpc_state) * (size_t)n)) != WG_OK) return rc;
  if ((rc = wgi_grow_scratch(ctx, &h->d_idx, &h->cap_idx, sizeof(int32_t) * (size_t)n)) != WG_OK) return rc;
  WG_CUDA(ctx, cudaMemcpyAsync(h->d_init, init.data(), sizeof(wg_herdt_mpc_state) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  WG_CUDA(ctx, cudaMemcpyAsync(h->d_idx, idx_host, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  const int blocks = std::max(1, std::min((n + MPC_WARPS - 1) / MPC_WARPS, ctx->sm_count * 16));
  online_start_kernel<<<blocks, MPC_WARPS * 32, 0, ctx->stream>>>(n, static_cast<const int32_t *>(h->d_idx),
                                                                  static_cast<const wg_herdt_mpc_state *>(h->d_init),
                                                                  h->d_states, h->d_queue, h->d_slots);
  WG_LAUNCHED(ctx);
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return WG_OK;
}

int wg_herdt_online_tick(wg_herdt_online *h, int mem, int nticks, const wg_herdt_command *commands, wg_herdt_tick *rows,
                         int8_t *running)
{
  if (!h || nticks < 0 || (mem != WG_MEM_HOST && mem != WG_MEM_DEVICE)) return WG_ERR_INVALID;
  wg_ctx *ctx = h->ctx;
  MpcState *m = mpc_of(ctx);
  if (!m->ready || !wg_herdt_device_consts(ctx))
    return wg_fail(ctx, WG_ERR_NOT_READY, "wg_herdt_set_params / wg_herdt_mpc_set_params not called");
  if (h->B == 0 || nticks == 0) return WG_OK;
  wg_device_guard guard(ctx->device);
  if (mem == WG_MEM_DEVICE) return online_ticks(h, m, nticks, commands, rows, running);
  const size_t n = (size_t)h->B * nticks;
  int rc;
  if (commands && (rc = wgi_grow_scratch(ctx, &h->d_cmd, &h->cap_cmd, sizeof(wg_herdt_command) * n)) != WG_OK) return rc;
  if (rows && (rc = wgi_grow_scratch(ctx, &h->d_rows, &h->cap_rows, sizeof(wg_herdt_tick) * n)) != WG_OK) return rc;
  if (running && (rc = wgi_grow_scratch(ctx, &h->d_run, &h->cap_run, sizeof(int8_t) * n)) != WG_OK) return rc;
  if (commands) WG_CUDA(ctx, cudaMemcpyAsync(h->d_cmd, commands, sizeof(wg_herdt_command) * n, cudaMemcpyHostToDevice, ctx->stream));
  if (rows) WG_CUDA(ctx, cudaMemsetAsync(h->d_rows, 0, sizeof(wg_herdt_tick) * n, ctx->stream));
  rc = online_ticks(h, m, nticks, commands ? static_cast<const wg_herdt_command *>(h->d_cmd) : nullptr,
                    rows ? static_cast<wg_herdt_tick *>(h->d_rows) : nullptr, running ? static_cast<int8_t *>(h->d_run) : nullptr);
  if (rc != WG_OK) return rc;
  if (rows) WG_CUDA(ctx, cudaMemcpyAsync(rows, h->d_rows, sizeof(wg_herdt_tick) * n, cudaMemcpyDeviceToHost, ctx->stream));
  if (running) WG_CUDA(ctx, cudaMemcpyAsync(running, h->d_run, sizeof(int8_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return WG_OK;
}

}  // extern "C"
