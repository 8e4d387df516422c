// kajita_online.cu - wg_kajita_online: the Kajita2003 on-line generator one 5 ms control tick at a time for B walks
// (PatternGeneratorInterface::RunOneStepOfTheControlLoop, Kajita branch), on top of wg_kajita_stream.
//
// No arithmetic of the walk lives here: every ZMP / feet sample and every CoM row comes from the stream's front-end and
// preview kernels.  This file plans the refills on the host (the tick rules only need counts, stacks and commands) and
// moves rows: a scatter kernel puts a run's new rows into each walk's queue ring, a gather kernel pops rows[t][b].
#include <algorithm>
#include <cmath>
#include <deque>
#include <new>
#include "wg_common.h"
#include "wg_records.cuh"

namespace {

constexpr int KO_WORDS = (int)(sizeof(wg_kajita_tick) / 16);   // 14 16-byte words per row
static_assert(sizeof(wg_kajita_tick) == 224 && sizeof(wg_kajita_command) == 64, "public layouts");
static_assert(offsetof(wg_kajita_tick, com_z) == 48 && offsetof(wg_kajita_tick, zmp_px) == 64 &&
              offsetof(wg_kajita_tick, zmp_theta) == 80 && offsetof(wg_kajita_tick, zmp_out) == 96 &&
              offsetof(wg_kajita_tick, left) == 112 && offsetof(wg_kajita_tick, right) == 160 &&
              offsetof(wg_kajita_tick, step_type) == 208, "wg_kajita_tick words");
constexpr int KO_WARPS = 8;

// One walk's share of a run: its new samples are rows [so, so + n) of the run's front-end outputs and walk samples
// [e0, e0 + n); its k new CoM rows are rows [co, co + k) of the run's preview outputs and walk samples [p0, p0 + k).
struct KoWork {
  int32_t b, start;
  int64_t e0, n, so, p0, k, co;
};

// The front-end and preview outputs of a run, in the handle's scratch.
struct KoRun {
  const double2 *zmpref;
  const double *theta;
  const wg_foot_sample *left, *right;
  const int32_t *types;
  const double *com, *zmp_out;
};

// Walk sample s lives in row s mod R of the walk's ring.  One warp per walk with new rows; lanes take samples.  The clock
// (ZMPPosition::time) is the sampling period accumulated sample by sample from the walk's start, as the reference's
// ZMPDiscretization accumulates it: every lane runs the same serial sum and keeps the value of its own sample.
__global__ void __launch_bounds__(KO_WARPS * 32)
kajita_online_scatter_kernel(int nwork, const KoWork *__restrict__ work, KoRun r, double T, double com_height, int R,
                             double2 *__restrict__ ring, double *__restrict__ clock)
{
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int j = blockIdx.x * KO_WARPS + warp; j < nwork; j += gridDim.x * KO_WARPS) {
    const KoWork w = work[j];
    double2 *rb = ring + (size_t)w.b * R * KO_WORDS;
    double t = w.start ? 0.0 : clock[w.b];
    for (int64_t i0 = 0; i0 < w.n; i0 += 32) {
      const int cnt = w.n - i0 < 32 ? (int)(w.n - i0) : 32;
      double mine = 0.0;
      for (int l = 0; l < cnt; ++l) {
        if (l == lane) mine = t;
        t += T;
      }
      if (lane < cnt) {
        const int64_t g = w.so + i0 + lane;
        double2 *row = rb + (size_t)((w.e0 + i0 + lane) % R) * KO_WORDS;
        const double th = r.theta[g];
        row[3] = make_double2(com_height, th);
        row[4] = r.zmpref[g];
        row[5] = make_double2(th, mine);
        const double2 *lf = reinterpret_cast<const double2 *>(r.left + g), *rf = reinterpret_cast<const double2 *>(r.right + g);
        row[7] = lf[0]; row[8] = lf[1]; row[9] = lf[2];
        row[10] = rf[0]; row[11] = rf[1]; row[12] = rf[2];
        const int32_t *ty = r.types + 3 * g;
        reinterpret_cast<int4 *>(row)[13] = make_int4(ty[0], ty[1], ty[2], 0);
      }
    }
    if (lane == 0) clock[w.b] = t;
    for (int64_t q = lane; q < w.k; q += 32) {
      double2 *row = rb + (size_t)((w.p0 + q) % R) * KO_WORDS;
      const double2 *c = reinterpret_cast<const double2 *>(r.com + 6 * (w.co + q));
      row[0] = c[0]; row[1] = c[1]; row[2] = c[2];
      row[6] = reinterpret_cast<const double2 *>(r.zmp_out)[w.co + q];
    }
  }
}

// rows[t][b] = the t-th row walk b pops in this chunk, for t < npop[b], its first at ring row first[b]; one thread per
// 16-byte word (the rows of one tick are contiguous across walks).  Other rows: zero when `zero`, else untouched.
__global__ void __launch_bounds__(256)
kajita_online_gather_kernel(int B, const int32_t *__restrict__ first, const int32_t *__restrict__ npop, int R,
                            const uint4 *__restrict__ ring, uint4 *__restrict__ rows, int8_t *__restrict__ running, int zero)
{
  const int j = blockIdx.x * blockDim.x + threadIdx.x, t = blockIdx.y;
  if (j >= B * KO_WORDS) return;
  const int b = j / KO_WORDS, w = j - b * KO_WORDS;
  const bool pop = t < npop[b];
  const size_t o = (size_t)t * B + b;
  if (running && w == 0) running[o] = pop ? 1 : 0;
  if (!rows) return;
  if (pop) {
    int s = first[b] + t;
    if (s >= R) s -= R;
    rows[o * KO_WORDS + w] = ring[((size_t)b * R + s) * KO_WORDS + w];
  } else if (zero) {
    rows[o * KO_WORDS + w] = make_uint4(0u, 0u, 0u, 0u);
  }
}

// ---- whole walks (wg_kajita_online_save / restore / copy) -------------------------------------------------------------
// One warp per walk, grid-stride; rows move as 16-byte words.  The stream part of a record (its first 36 words) is the
// stream's, moved by its own strided kernels (zmpdisc.cu); these kernels move the queue, the clock and the handle's words.
constexpr int KO_UNROLL = 8;
constexpr int KO_CTAS_PER_SM = 6;   // all resident at up to 40 registers (the kernels take 36 to 40): no second wave
constexpr int KO_STREAM_V4 = (int)(sizeof(wg_kajita_stream_walk) / 16);   // 36
constexpr int KO_WALK_V4 = (int)(sizeof(wg_kajita_online_walk) / 16);     // 39
static_assert(sizeof(wg_kajita_online_walk) == 624 && offsetof(wg_kajita_online_walk, popped) == 576 &&
              offsetof(wg_kajita_online_walk, clock) == 584 && offsetof(wg_kajita_online_walk, keep) == 592 &&
              offsetof(wg_kajita_online_walk, stacked) == 608, "wg_kajita_online_walk words");

// Walk b's queued span: q rows from ring row `first` on (wrapping at R), the first nc of them with their CoM.
struct KoSpan {
  int32_t b, first, q, nc;
};

// A save's host-side words of record i: its span, and record words 36..38 (word 36's clock half is the device's).
struct KoSave {
  KoSpan sp;
  uint4 tail[3];
};

// A copy of walk s's queued span and clock to walk d, at the same ring rows.
struct KoPair {
  int32_t d, s, first, q;
};

// Record words 36..38 and queue rows of walks in[i].sp.b, front first: the q queued rows, the CoM words (0..2 and 6) of
// rows nc..q-1 zero (the preview has not written them: they hold whatever an earlier walk left), rows past q zero.
__global__ void __launch_bounds__(KO_WARPS * 32)
kajita_online_save_kernel(int n, const KoSave *__restrict__ in, int R, const uint4 *__restrict__ ring,
                          const double *__restrict__ clock, uint4 *__restrict__ walks, uint4 *__restrict__ queue)
{
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = blockIdx.x * KO_WARPS + warp; i < n; i += gridDim.x * KO_WARPS) {
    const KoSpan sp = in[i].sp;
    if (lane < 3) {
      uint4 v = in[i].tail[lane];
      if (lane == 0) {
        const unsigned long long c = (unsigned long long)__double_as_longlong(clock[sp.b]);
        v.z = (unsigned)c; v.w = (unsigned)(c >> 32);
      }
      walks[(int64_t)i * KO_WALK_V4 + KO_STREAM_V4 + lane] = v;
    }
    const uint4 *rb = ring + (size_t)sp.b * R * KO_WORDS;
    uint4 *oq = queue + (size_t)i * R * KO_WORDS;
    const int a = min(sp.nc, R - sp.first);          // whole rows before the wrap
    wgi_warp_copy16<KO_UNROLL>(oq, rb + (size_t)sp.first * KO_WORDS, a * KO_WORDS, a * KO_WORDS, lane);
    wgi_warp_copy16<KO_UNROLL>(oq + (size_t)a * KO_WORDS, rb, (sp.nc - a) * KO_WORDS, (sp.nc - a) * KO_WORDS, lane);
    for (int e = sp.nc * KO_WORDS + lane; e < sp.q * KO_WORDS; e += 32) {
      const int j = e / KO_WORDS, w = e - j * KO_WORDS;
      int s = sp.first + j;
      if (s >= R) s -= R;
      oq[e] = (w < 3 || w == 6) ? make_uint4(0u, 0u, 0u, 0u) : rb[(size_t)s * KO_WORDS + w];
    }
    wgi_warp_copy16<KO_UNROLL>(oq + (size_t)sp.q * KO_WORDS, rb, (R - sp.q) * KO_WORDS, 0, lane);
  }
}

// Queue rows of record i -> ring rows first.. of walk sp[i].b (wrapping at R), its clock -> clock[b].  Ring rows past the
// queued span are left as they are: nothing reads them before a refill writes them.
__global__ void __launch_bounds__(KO_WARPS * 32)
kajita_online_restore_kernel(int n, const KoSpan *__restrict__ span, const wg_kajita_online_walk *__restrict__ walks,
                             const uint4 *__restrict__ queue, int R, uint4 *__restrict__ ring, double *__restrict__ clock)
{
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = blockIdx.x * KO_WARPS + warp; i < n; i += gridDim.x * KO_WARPS) {
    const KoSpan sp = span[i];
    if (lane == 0) clock[sp.b] = walks[i].clock;
    const uint4 *iq = queue + (size_t)i * R * KO_WORDS;
    uint4 *rb = ring + (size_t)sp.b * R * KO_WORDS;
    const int a = min(sp.q, R - sp.first);
    wgi_warp_copy16<KO_UNROLL>(rb + (size_t)sp.first * KO_WORDS, iq, a * KO_WORDS, a * KO_WORDS, lane);
    wgi_warp_copy16<KO_UNROLL>(rb, iq + (size_t)a * KO_WORDS, (sp.q - a) * KO_WORDS, (sp.q - a) * KO_WORDS, lane);
  }
}

// Walk pair[i].s of one handle -> walk pair[i].d of another (or of the same, the index sets disjoint): the queued span at
// the same ring rows, and the clock.
__global__ void __launch_bounds__(KO_WARPS * 32)
kajita_online_copy_kernel(int n, const KoPair *__restrict__ pair, int R, const uint4 *__restrict__ s_ring,
                          const double *__restrict__ s_clock, uint4 *__restrict__ d_ring, double *__restrict__ d_clock)
{
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = blockIdx.x * KO_WARPS + warp; i < n; i += gridDim.x * KO_WARPS) {
    const KoPair p = pair[i];
    if (lane == 0) d_clock[p.d] = s_clock[p.s];
    const uint4 *sb = s_ring + (size_t)p.s * R * KO_WORDS;
    uint4 *db = d_ring + (size_t)p.d * R * KO_WORDS;
    const int a = min(p.q, R - p.first);
    wgi_warp_copy16<KO_UNROLL>(db + (size_t)p.first * KO_WORDS, sb + (size_t)p.first * KO_WORDS, a * KO_WORDS, a * KO_WORDS, lane);
    wgi_warp_copy16<KO_UNROLL>(db, sb, (p.q - a) * KO_WORDS, (p.q - a) * KO_WORDS, lane);
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------------------------
struct KoWalk {                       // what the reference's PGI and StepStackHandler keep for one walk
  std::deque<wg_rel_step> stack;
  int64_t emitted = 0, popped = 0;    // samples since the start; queue = emitted - popped
  int32_t keep = 1;                   // m_KeepLastCorrectSupportFoot
  bool running = false, online = false, transition = false;   // m_Running, m_KajitaOnLine, m_TransitionFinishOnLine
};

struct wg_kajita_online {
  wg_ctx *ctx = nullptr;
  int B = 0, NL = 0, R = 0;
  wg_zmpdisc_params P;
  double com_height = 0.0;
  int max_seg = 0, n_end = 0;         // round(max_step_time / T); round(t_double / 2T) + 3 NL
  wg_kajita_stream *s = nullptr;
  std::vector<KoWalk> walks;
  double2 *d_ring = nullptr;          // [B][R] rows
  double *d_clock = nullptr;          // [B] time of the walk's next sample
  void *d_run = nullptr, *d_rows = nullptr, *d_flags = nullptr;   // run outputs; WG_MEM_HOST staging of rows, running
  void *d_io = nullptr;               // WG_MEM_HOST staging of whole walks: records, carry, queues
  size_t cap_run = 0, cap_rows = 0, cap_flags = 0, cap_io = 0;
  wgi_stage stage;                    // a chunk's scatter work, then first[B], npop[B]
  KoRun run;                          // where the last run's outputs are
  // the run being planned: per walk the steps it appends and its flags
  std::vector<int64_t> off;
  std::vector<wg_rel_step> steps;
  std::vector<int32_t> flags;
  std::vector<int32_t> first, npop;
  std::vector<double> feet;
};

static int ko_seg(const wg_zmpdisc_params &P, const wg_rel_step &s)
{
  const double ds = s.ds_time != 0.0 ? s.ds_time : P.t_double, ss = s.ds_time != 0.0 ? s.ss_time : P.t_single;
  return (int)(unsigned)std::round((ds + ss) / P.sampling_period);
}

// The step timing rules of the stream (wg_kajita_stream_append) and the handle's bound on the segment length.
static bool ko_step_ok(const wg_kajita_online *h, const wg_rel_step &s)
{
  const wg_zmpdisc_params &P = h->P;
  const double ds = s.ds_time != 0.0 ? s.ds_time : P.t_double, ss = s.ds_time != 0.0 ? s.ss_time : P.t_single;
  const int add = ko_seg(P, s);
  const int n1 = (int)(unsigned)std::round(ds / P.sampling_period), n2 = (int)(unsigned)std::round(ss / P.sampling_period);
  return n1 >= 1 && n1 + n2 <= add && add <= 2800 && add <= h->max_seg;
}

static wg_rel_step ko_standard(const wg_zmpdisc_params &P, double sx, double sy, double theta)
{
  wg_rel_step s;
  std::memset(&s, 0, sizeof s);
  s.sx = sx; s.sy = sy; s.theta = theta; s.ss_time = P.t_single; s.ds_time = P.t_double; s.step_type = 1;
  return s;
}

static void ko_free(wg_kajita_online *h)
{
  if (h->s) wg_kajita_stream_destroy(h->s);
  cudaFree(h->d_ring); cudaFree(h->d_clock); cudaFree(h->d_run); cudaFree(h->d_rows); cudaFree(h->d_flags); cudaFree(h->d_io);
  wgi_stage_free(&h->stage);
  delete h;
}

static size_t ko_align(size_t x) { return (x + 15) / 16 * 16; }

// Run the pending append of the handle's stream (front end and preview: two launches) with its outputs in the handle's
// scratch, and list the walks with new rows.  e0[b] is walk b's emitted count before the run; start[b] says it restarts.
static int ko_run(wg_kajita_online *h, const std::vector<int64_t> &e0, const std::vector<char> &start, KoWork *wk, int *nwork)
{
  wg_ctx *ctx = h->ctx;
  const int B = h->B;
  const int64_t *so = wg_kajita_stream_sample_offsets(h->s), *co = wg_kajita_stream_com_offsets(h->s);
  const int64_t *cnt = wg_kajita_stream_com_counts(h->s);
  const size_t ns = (size_t)so[B], nc = (size_t)co[B];
  const size_t o_th = ko_align(16 * ns), o_l = o_th + ko_align(8 * ns), o_r = o_l + 48 * ns, o_ty = o_r + 48 * ns;
  const size_t o_com = o_ty + ko_align(12 * ns), o_zo = o_com + 48 * nc, bytes = o_zo + 16 * nc;
  if (bytes > h->cap_run) {
    const int rc = wgi_grow_scratch(ctx, &h->d_run, &h->cap_run, std::max(bytes + bytes / 2, (size_t)256));
    if (rc != WG_OK) return rc;
  }
  unsigned char *base = static_cast<unsigned char *>(h->d_run);
  double2 *zr = reinterpret_cast<double2 *>(base);
  double *th = reinterpret_cast<double *>(base + o_th), *com = reinterpret_cast<double *>(base + o_com);
  double *zo = reinterpret_cast<double *>(base + o_zo);
  wg_foot_sample *l = reinterpret_cast<wg_foot_sample *>(base + o_l), *r = reinterpret_cast<wg_foot_sample *>(base + o_r);
  int32_t *ty = reinterpret_cast<int32_t *>(base + o_ty);
  const int rc = wg_kajita_stream_run(h->s, WG_MEM_DEVICE, reinterpret_cast<double *>(zr), th, l, r, ty, com, zo, 1);
  if (rc != WG_OK) return rc;
  h->run = KoRun{zr, th, l, r, ty, com, zo};
  const int NL1 = h->NL - 1;
  int n = 0;
  for (int b = 0; b < B; ++b) {
    const int64_t m = so[b + 1] - so[b];
    if (m == 0) continue;
    KoWork &w = wk[n++];
    w.b = b; w.start = start[b];
    w.e0 = start[b] ? 0 : e0[b];
    w.n = m; w.so = so[b];
    w.p0 = std::max<int64_t>(0, w.e0 - NL1);
    w.k = cnt[b]; w.co = co[b];
  }
  *nwork = n;
  return WG_OK;
}

// The last run's rows into the rings (one launch); d_work: its nwork entries on the device.
static int ko_scatter(wg_kajita_online *h, int nwork, const KoWork *d_work)
{
  wg_ctx *ctx = h->ctx;
  if (nwork == 0) return WG_OK;
  wg_prof_start(ctx, WG_K_ZMPDISC);
  kajita_online_scatter_kernel<<<wgi_grid(ctx, nwork, KO_WARPS, 8), KO_WARPS * 32, 0, ctx->stream>>>(
      nwork, d_work, h->run, h->P.sampling_period, h->com_height, h->R, h->d_ring, h->d_clock);
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  return WG_OK;
}

extern "C" {

int wg_kajita_online_create(wg_ctx *ctx, const wg_zmpdisc_params *p, int B, double com_height, double max_step_time,
                            wg_kajita_online **out)
{
  if (!ctx || !p || !out || B < 1) return WG_ERR_INVALID;
  *out = nullptr;
  const char *call = "wg_kajita_online_create";
  if (!ctx->preview_ready) return wg_fail(ctx, WG_ERR_NOT_READY, "wg_kajita_online_create: wg_preview_set_gains not called");
  if (!(p->sampling_period > 0) || !(max_step_time > 0) || !std::isfinite(max_step_time) || !std::isfinite(com_height))
    return wg_refuse(ctx, call, "sampling_period, max_step_time and com_height must be finite, the first two positive");
  wg_device_guard guard(ctx->device);
  wg_kajita_online *h = new (std::nothrow) wg_kajita_online();
  if (!h) return WG_ERR_ALLOC;
  h->ctx = ctx; h->B = B; h->P = *p; h->com_height = com_height;
  h->NL = ctx->preview_gains.NL;
  h->max_seg = (int)std::llround(max_step_time / p->sampling_period);
  h->n_end = (int)(unsigned)std::round(p->t_double / (2 * p->sampling_period)) + (int)(3.0 * p->preview_time / p->sampling_period);
  if (!ko_step_ok(h, ko_standard(*p, 0, 0, 0))) {
    delete h;
    return wg_refuse(ctx, call, "the default step (t_single, t_double) does not fit max_step_time or the stream's timing rules");
  }
  const int64_t R = 2 * (int64_t)h->NL + 1 + h->max_seg + h->n_end + WG_KAJITA_ONLINE_CHUNK - 1;
  if (R > (1 << 20)) { delete h; return wg_refuse(ctx, call, "max_step_time too long"); }
  h->R = (int)R;
  int rc = wg_kajita_stream_create(ctx, p, B, 1, &h->s);
  if (rc != WG_OK) { delete h; return rc; }
  h->walks.resize(B);
  h->off.assign(B + 1, 0); h->flags.assign(B, 0); h->first.assign(B, 0); h->npop.assign(B, 0); h->feet.assign(6 * (size_t)B, 0.0);
  cudaError_t e = cudaMalloc(&h->d_ring, sizeof(wg_kajita_tick) * (size_t)h->R * B);
  if (e == cudaSuccess) e = cudaMalloc(&h->d_clock, sizeof(double) * B);
  if (e == cudaSuccess) e = cudaMemsetAsync(h->d_clock, 0, sizeof(double) * B, ctx->stream);
  if (e != cudaSuccess) {
    ko_free(h);
    return wg_fail(ctx, e == cudaErrorMemoryAllocation ? WG_ERR_ALLOC : WG_ERR_CUDA, call, e);
  }
  *out = h;
  return WG_OK;
}

int wg_kajita_online_destroy(wg_kajita_online *h)
{
  if (!h) return WG_ERR_INVALID;
  wg_device_guard guard(h->ctx->device);
  cudaStreamSynchronize(h->ctx->stream);
  ko_free(h);
  return WG_OK;
}

int wg_kajita_online_ring_rows(const wg_kajita_online *h) { return h ? h->R : WG_ERR_INVALID; }

int wg_kajita_online_start(wg_kajita_online *h, int n, const int32_t *idx, const int64_t *step_off, const wg_rel_step *steps,
                           const double *init_feet, const int32_t *keep_last)
{
  if (!h) return WG_ERR_INVALID;
  wg_ctx *ctx = h->ctx;
  const char *call = "wg_kajita_online_start";
  const int B = h->B;
  if (n < 0) return wg_refuse(ctx, call, "n < 0");
  if (n > 0 && (!idx || !step_off || !steps || !init_feet)) return wg_refuse(ctx, call, "NULL array with n > 0");
  std::vector<char> mark((size_t)B, 0);
  if (!wgi_record_indices_ok(B, n, idx, true, mark)) return wg_refuse(ctx, call, "index out of range or repeated");
  if (n == 0) return WG_OK;
  if (!ctx->preview_ready || ctx->preview_gains.NL != h->NL)
    return wg_fail(ctx, WG_ERR_NOT_READY, "wg_kajita_online_start: the preview gains' NL changed since the handle was created");
  if (step_off[0] != 0) return wg_refuse(ctx, call, "step_offsets[0] must be 0");
  for (int i = 0; i < n; ++i) {
    const int64_t a = step_off[i], e = step_off[i + 1];
    if (e <= a) return wg_refuse(ctx, call, "every walk needs at least its support-foot step");
    if (keep_last && keep_last[i] != 1 && keep_last[i] != -1) return wg_refuse(ctx, call, "keep_last must be +1 or -1");
    int64_t q = 2 * (int64_t)h->NL;
    for (int64_t k = a + 1; k < e; ++k) {
      if (!ko_step_ok(h, steps[k]))
        return wg_refuse(ctx, call, "a step timing out of range or longer than max_step_time");
      q += ko_seg(h->P, steps[k]);
      if (q > h->R) return wg_refuse(ctx, call, "more start samples than the queue ring holds");
    }
  }
  // one append for the whole batch: START for the listed walks, nothing for the others
  std::vector<int64_t> off(B + 1, 0);
  std::vector<int32_t> flags(B, 0);
  std::vector<int> pos(B, -1);
  for (int i = 0; i < n; ++i) pos[idx[i]] = i;
  std::vector<wg_rel_step> st;
  st.reserve((size_t)step_off[n]);
  for (int b = 0; b < B; ++b) {
    const int i = pos[b];
    if (i >= 0) {
      st.insert(st.end(), steps + step_off[i], steps + step_off[i + 1]);
      flags[b] = WG_STREAM_START;
      std::copy(init_feet + 6 * (size_t)i, init_feet + 6 * (size_t)i + 6, h->feet.begin() + 6 * (size_t)b);
    }
    off[b + 1] = (int64_t)st.size();
  }
  wg_device_guard guard(ctx->device);
  int rc = wg_kajita_stream_append(h->s, off.data(), st.data(), flags.data(), h->feet.data());
  if (rc != WG_OK) return rc;
  std::vector<int64_t> e0(B, 0);
  std::vector<char> start(B, 0);
  for (int i = 0; i < n; ++i) start[idx[i]] = 1;
  std::vector<KoWork> work(n);
  int nwork = 0;
  if ((rc = ko_run(h, e0, start, work.data(), &nwork)) != WG_OK) return rc;
  unsigned char *hb;
  const size_t bytes = sizeof(KoWork) * (size_t)nwork;
  if ((rc = wgi_stage_reserve(ctx, &h->stage, bytes, &hb)) != WG_OK) return rc;
  std::memcpy(hb, work.data(), bytes);
  if ((rc = wgi_stage_send(ctx, &h->stage, bytes)) != WG_OK) return rc;
  if ((rc = ko_scatter(h, nwork, reinterpret_cast<const KoWork *>(h->stage.d))) != WG_OK) return rc;
  const int64_t *so = wg_kajita_stream_sample_offsets(h->s);
  for (int i = 0; i < n; ++i) {
    const int b = idx[i];
    KoWalk &w = h->walks[b];
    w.stack.clear();
    w.emitted = so[b + 1] - so[b];
    w.popped = 0;
    w.keep = keep_last ? keep_last[i] : 1;
    w.running = w.online = true;
    w.transition = false;
  }
  return WG_OK;
}

int wg_kajita_online_tick(wg_kajita_online *h, int mem, int nticks, const wg_kajita_command *cmd, wg_kajita_tick *rows,
                          int8_t *running)
{
  if (!h) return WG_ERR_INVALID;
  wg_ctx *ctx = h->ctx;
  const char *call = "wg_kajita_online_tick";
  const int B = h->B;
  if (nticks < 0) return wg_refuse(ctx, call, "nticks < 0");
  if (mem != WG_MEM_HOST && mem != WG_MEM_DEVICE) return wg_refuse(ctx, call, "unknown mem");
  if (mem == WG_MEM_DEVICE && (reinterpret_cast<uintptr_t>(rows) & 15)) return wg_refuse(ctx, call, "device rows must be 16-byte aligned");
  if (cmd)
    for (size_t i = 0; i < (size_t)nticks * B; ++i) {
      const int f = cmd[i].flags;
      if (f & ~(WG_KAJITA_PUSH | WG_KAJITA_STANDARD | WG_KAJITA_STOP)) return wg_refuse(ctx, call, "unknown command flags");
      if ((f & WG_KAJITA_STOP) && (f & (WG_KAJITA_PUSH | WG_KAJITA_STANDARD))) return wg_refuse(ctx, call, "STOP together with a step");
      if ((f & WG_KAJITA_PUSH) && (f & WG_KAJITA_STANDARD)) return wg_refuse(ctx, call, "PUSH together with STANDARD");
      if ((f & WG_KAJITA_PUSH) && !ko_step_ok(h, cmd[i].step))
        return wg_refuse(ctx, call, "a pushed step timing out of range or longer than max_step_time");
    }
  if (!ctx->preview_ready || ctx->preview_gains.NL != h->NL)
    return wg_fail(ctx, WG_ERR_NOT_READY, "wg_kajita_online_tick: the preview gains' NL changed since the handle was created");
  if (nticks == 0) return WG_OK;
  wg_device_guard guard(ctx->device);
  int rc;
  const size_t nrow = (size_t)nticks * B;
  wg_kajita_tick *d_rows = rows;
  int8_t *d_run = running;
  if (mem == WG_MEM_HOST) {
    if (rows && (rc = wgi_grow_scratch(ctx, &h->d_rows, &h->cap_rows, sizeof(wg_kajita_tick) * nrow)) != WG_OK) return rc;
    if (running && (rc = wgi_grow_scratch(ctx, &h->d_flags, &h->cap_flags, nrow)) != WG_OK) return rc;
    d_rows = rows ? static_cast<wg_kajita_tick *>(h->d_rows) : nullptr;
    d_run = running ? static_cast<int8_t *>(h->d_flags) : nullptr;
  }
  const int64_t lo = 2 * (int64_t)h->NL;      // the walk stops at <= 2 NL queued samples, refills at <= 2 NL + 1
  std::vector<int64_t> e0(B);
  const std::vector<char> no_start(B, 0);
  std::vector<KoWork> work;
  for (int t0 = 0; t0 < nticks; t0 += WG_KAJITA_ONLINE_CHUNK) {
    const int nt = std::min(WG_KAJITA_ONLINE_CHUNK, nticks - t0);
    // ---- replay the tick rules of every walk over the chunk on the host ----
    h->steps.clear();
    bool any = false;
    for (int b = 0; b < B; ++b) {
      KoWalk &w = h->walks[b];
      e0[b] = w.emitted;
      h->first[b] = (int32_t)(w.popped % h->R);
      h->flags[b] = 0;
      int np = 0;
      for (int t = 0; t < nt && w.running; ++t) {
        if (cmd && w.online) {
          const wg_kajita_command &c = cmd[(size_t)(t0 + t) * B + b];
          if (c.flags & WG_KAJITA_PUSH) w.stack.push_back(c.step);
          if (c.flags & WG_KAJITA_STANDARD) {
            w.stack.push_back(ko_standard(h->P, c.step.sx, c.step.sy + w.keep * 0.19, c.step.theta));
            w.keep = -w.keep;
          }
          if (c.flags & WG_KAJITA_STOP) {
            if (w.stack.size() % 2 == 0) w.keep = -w.keep;
            w.stack.clear();
            w.transition = true;
          }
        }
        if (w.online && w.emitted - w.popped <= lo + 1) {
          if (w.stack.empty()) {
            w.stack.push_back(ko_standard(h->P, 0.0, w.keep * 0.19, 0.0));
            w.keep = -w.keep;
          }
          const wg_rel_step f = w.stack.front();
          w.stack.pop_front();
          const bool last = w.stack.empty() && w.transition;
          h->steps.push_back(f);
          w.emitted += ko_seg(h->P, f);
          if (last) {
            w.emitted += h->n_end;
            w.online = w.transition = false;
            h->flags[b] = WG_STREAM_FINISH;
          }
        }
        if (w.emitted - w.popped <= lo) {
          w.running = false;
          break;
        }
        ++w.popped;
        ++np;
      }
      h->npop[b] = np;
      h->off[b + 1] = (int64_t)h->steps.size();
      // every row of the chunk is in the ring before its first pop: the rows queued at its start plus all it adds
      if (w.emitted - (w.popped - np) > h->R)
        return wg_fail(ctx, WG_ERR_INVALID, "wg_kajita_online_tick: queue ring bound exceeded");
      any = any || w.emitted > e0[b];
    }
    // ---- one run for all the refills of the chunk, the scatter, the gather ----
    int nwork = 0;
    if (any) {
      work.resize(B);
      if ((rc = wg_kajita_stream_append(h->s, h->off.data(), h->steps.data(), h->flags.data(), nullptr)) != WG_OK) return rc;
      if ((rc = ko_run(h, e0, no_start, work.data(), &nwork)) != WG_OK) return rc;
    }
    const size_t wbytes = ko_align(sizeof(KoWork) * (size_t)nwork), ib = sizeof(int32_t) * (size_t)B;
    const size_t bytes = wbytes + 2 * ib;
    unsigned char *hb;
    if ((rc = wgi_stage_reserve(ctx, &h->stage, bytes, &hb)) != WG_OK) return rc;
    if (nwork) std::memcpy(hb, work.data(), sizeof(KoWork) * (size_t)nwork);
    std::memcpy(hb + wbytes, h->first.data(), ib);
    std::memcpy(hb + wbytes + ib, h->npop.data(), ib);
    if ((rc = wgi_stage_send(ctx, &h->stage, bytes)) != WG_OK) return rc;
    if ((rc = ko_scatter(h, nwork, reinterpret_cast<const KoWork *>(h->stage.d))) != WG_OK) return rc;
    const dim3 grid((unsigned)((B * KO_WORDS + 255) / 256), (unsigned)nt);
    wg_prof_start(ctx, WG_K_ZMPDISC);
    kajita_online_gather_kernel<<<grid, 256, 0, ctx->stream>>>(
        B, reinterpret_cast<const int32_t *>(h->stage.d + wbytes), reinterpret_cast<const int32_t *>(h->stage.d + wbytes + ib),
        h->R, reinterpret_cast<const uint4 *>(h->d_ring), d_rows ? reinterpret_cast<uint4 *>(d_rows + (size_t)t0 * B) : nullptr,
        d_run ? d_run + (size_t)t0 * B : nullptr, mem == WG_MEM_HOST);
    wg_prof_stop(ctx);
    WG_LAUNCHED(ctx);
  }
  if (mem == WG_MEM_HOST) {
    if (rows) WG_CUDA(ctx, cudaMemcpyAsync(rows, d_rows, sizeof(wg_kajita_tick) * nrow, cudaMemcpyDeviceToHost, ctx->stream));
    if (running) WG_CUDA(ctx, cudaMemcpyAsync(running, d_run, nrow, cudaMemcpyDeviceToHost, ctx->stream));
    WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return WG_OK;
}

int wg_kajita_online_state(wg_kajita_online *h, int64_t *queued, int32_t *stacked, int32_t *running, int32_t *online)
{
  if (!h) return WG_ERR_INVALID;
  for (int b = 0; b < h->B; ++b) {
    const KoWalk &w = h->walks[b];
    if (queued) queued[b] = w.emitted - w.popped;
    if (stacked) stacked[b] = (int32_t)w.stack.size();
    if (running) running[b] = w.running;
    if (online) online[b] = w.online;
  }
  return WG_OK;
}

}  // extern "C"

// ---- whole walks ------------------------------------------------------------------------------------------------------
// The argument checks save and restore share: nullptr when the call may go on, else why it may not.
static const char *ko_io_refusal(const wg_kajita_online *h, int mem, int n, const void *walks, const void *carry, const void *queue)
{
  if (mem != WG_MEM_HOST && mem != WG_MEM_DEVICE) return "unknown mem";
  if (n < 0) return "n < 0";
  if (n > 0 && (!walks || !queue || (!carry && h->NL > 1))) return "NULL walks, carry or queue with n > 0";
  if (mem == WG_MEM_DEVICE &&
      ((reinterpret_cast<uintptr_t>(walks) | reinterpret_cast<uintptr_t>(carry) | reinterpret_cast<uintptr_t>(queue)) & 15))
    return "device arrays must be 16-byte aligned";
  return nullptr;
}

// The invariants every tick keeps, over a record from outside the program: nullptr when it keeps them, else which it breaks.
static const char *ko_record_refusal(const wg_kajita_online *h, const wg_kajita_online_walk &r)
{
  if (!wgi_kajita_stream_record_ok(h->s, &r.stream))
    return "a record breaks the stream's invariants of open, samples_emitted and steps_previewed";
  if ((r.running | r.online | r.transition) & ~1) return "running, online and transition must be 0 or 1";
  if (r.stream.open != r.online) return "stream.open differs from online";
  if ((r.online && !r.running) || (r.transition && !r.online) || (!r.online && r.stacked != 0))
    return "online without running, transition without online, or a stack on a walk off line";
  if (r.keep != 1 && r.keep != -1) return "keep must be +1 or -1";
  const int64_t q = r.stream.samples_emitted - r.popped;
  if (r.popped < 0 || q < 0 || q > h->R) return "popped out of [0, samples_emitted], or more queued rows than the ring holds";
  if (r.running && q < 2 * (int64_t)h->NL) return "a running walk with fewer than 2 NL queued samples";
  if (r.stacked < 0) return "stacked < 0";
  return nullptr;
}

// Device arrays of n records in the handle's WG_MEM_HOST staging: records, carry, queues.
static int ko_io(wg_kajita_online *h, int n, wg_kajita_online_walk **w, double **c, wg_kajita_tick **q)
{
  const size_t wb = sizeof(wg_kajita_online_walk) * (size_t)n, cb = ko_align(sizeof(double2) * (size_t)(h->NL - 1) * n);
  const int rc = wgi_grow_scratch(h->ctx, &h->d_io, &h->cap_io, wb + cb + sizeof(wg_kajita_tick) * (size_t)h->R * n);
  if (rc != WG_OK) return rc;
  unsigned char *base = static_cast<unsigned char *>(h->d_io);
  *w = reinterpret_cast<wg_kajita_online_walk *>(base);
  *c = reinterpret_cast<double *>(base + wb);
  *q = reinterpret_cast<wg_kajita_tick *>(base + wb + cb);
  return WG_OK;
}

extern "C" {

int wg_kajita_online_carry_rows(const wg_kajita_online *h) { return h ? h->NL - 1 : WG_ERR_INVALID; }

int wg_kajita_online_save(wg_kajita_online *h, int mem, int n, const int32_t *idx, wg_kajita_online_walk *walks, double *carry,
                          wg_kajita_tick *queue, wg_rel_step *stack_host, int64_t stack_cap, int64_t *stack_len)
{
  if (!h) return WG_ERR_INVALID;
  wg_ctx *ctx = h->ctx;
  const char *call = "wg_kajita_online_save";
  if (const char *why = ko_io_refusal(h, mem, n, walks, carry, queue)) return wg_refuse(ctx, call, why);
  std::vector<char> mark((size_t)h->B, 0);
  if (!wgi_record_indices_ok(h->B, n, idx, false, mark)) return wg_refuse(ctx, call, "index out of range, or n > B without indices");
  int64_t total = 0;
  for (int i = 0; i < n; ++i) total += (int64_t)h->walks[idx ? idx[i] : i].stack.size();
  if (total > stack_cap) return wg_refuse(ctx, call, "the stacks hold more than stack_cap steps");
  if (total > 0 && !stack_host) return wg_refuse(ctx, call, "NULL stack_host with steps to save");
  if (stack_len) *stack_len = total;
  if (n == 0) return WG_OK;
  wg_device_guard guard(ctx->device);
  // the stream's counters, then the handle's words and spans, in one H2D copy
  const size_t cb = ko_align(wgi_kajita_stream_counts(h->s, n, idx, nullptr)), bytes = cb + sizeof(KoSave) * (size_t)n;
  unsigned char *hb;
  int rc = wgi_stage_reserve(ctx, &h->stage, bytes, &hb);
  if (rc != WG_OK) return rc;
  wgi_kajita_stream_counts(h->s, n, idx, hb);
  KoSave *ks = reinterpret_cast<KoSave *>(hb + cb);
  const int64_t NL1 = h->NL - 1;
  int64_t at = 0;
  for (int i = 0; i < n; ++i) {
    const int b = idx ? idx[i] : i;
    const KoWalk &w = h->walks[b];
    const int64_t q = w.emitted - w.popped;
    KoSave &k = ks[i];
    k.sp = KoSpan{b, (int32_t)(w.popped % h->R), (int32_t)q, (int32_t)std::max<int64_t>(0, q - std::min(w.emitted, NL1))};
    k.tail[0] = make_uint4((unsigned)w.popped, (unsigned)((uint64_t)w.popped >> 32), 0u, 0u);
    k.tail[1] = make_uint4((unsigned)w.keep, w.running, w.online, w.transition);
    k.tail[2] = make_uint4((unsigned)w.stack.size(), 0u, 0u, 0u);
    std::copy(w.stack.begin(), w.stack.end(), stack_host + at);
    at += (int64_t)w.stack.size();
  }
  if ((rc = wgi_stage_send(ctx, &h->stage, bytes)) != WG_OK) return rc;
  wg_kajita_online_walk *d_w = walks;
  double *d_c = carry;
  wg_kajita_tick *d_q = queue;
  if (mem == WG_MEM_HOST && (rc = ko_io(h, n, &d_w, &d_c, &d_q)) != WG_OK) return rc;
  if ((rc = wgi_kajita_stream_save_strided(h->s, n, h->stage.d, d_w, sizeof(wg_kajita_online_walk), d_c)) != WG_OK) return rc;
  wg_prof_start(ctx, WG_K_ZMPDISC);
  kajita_online_save_kernel<<<wgi_grid(ctx, n, KO_WARPS, KO_CTAS_PER_SM), KO_WARPS * 32, 0, ctx->stream>>>(
      n, reinterpret_cast<const KoSave *>(h->stage.d + cb), h->R, reinterpret_cast<const uint4 *>(h->d_ring), h->d_clock,
      reinterpret_cast<uint4 *>(d_w), reinterpret_cast<uint4 *>(d_q));
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  if (mem == WG_MEM_DEVICE) return WG_OK;
  WG_CUDA(ctx, cudaMemcpyAsync(walks, d_w, sizeof(wg_kajita_online_walk) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
  if (NL1 > 0) WG_CUDA(ctx, cudaMemcpyAsync(carry, d_c, sizeof(double2) * NL1 * n, cudaMemcpyDeviceToHost, ctx->stream));
  WG_CUDA(ctx, cudaMemcpyAsync(queue, d_q, sizeof(wg_kajita_tick) * (size_t)h->R * n, cudaMemcpyDeviceToHost, ctx->stream));
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return WG_OK;
}

int wg_kajita_online_restore(wg_kajita_online *h, int mem, int n, const int32_t *idx, const wg_kajita_online_walk *walks,
                             const double *carry, const wg_kajita_tick *queue, const wg_rel_step *stack_host, int64_t stack_len)
{
  if (!h) return WG_ERR_INVALID;
  wg_ctx *ctx = h->ctx;
  const char *call = "wg_kajita_online_restore";
  if (const char *why = ko_io_refusal(h, mem, n, walks, carry, queue)) return wg_refuse(ctx, call, why);
  std::vector<char> mark((size_t)h->B, 0);
  if (!wgi_record_indices_ok(h->B, n, idx, true, mark))
    return wg_refuse(ctx, call, "index out of range or repeated, or n > B without indices");
  if (stack_len < 0 || (stack_len > 0 && !stack_host)) return wg_refuse(ctx, call, "stack_len < 0, or NULL stack_host with steps");
  if (n == 0) return stack_len == 0 ? WG_OK : wg_refuse(ctx, call, "the stacks hold other than stack_len steps");
  wg_device_guard guard(ctx->device);
  // blob: indices | spans | (device records) the records read back
  const size_t ib = ko_align(sizeof(int32_t) * (size_t)n), sb = ib + sizeof(KoSpan) * (size_t)n;
  const size_t bytes = sb + (mem == WG_MEM_DEVICE ? sizeof(wg_kajita_online_walk) * (size_t)n : 0);
  unsigned char *hb;
  int rc = wgi_stage_reserve(ctx, &h->stage, bytes, &hb);
  if (rc != WG_OK) return rc;
  const wg_kajita_online_walk *rec = walks;
  if (mem == WG_MEM_DEVICE) {       // the host replays the tick rules from these fields: read them back once
    WG_CUDA(ctx, cudaMemcpyAsync(hb + sb, walks, bytes - sb, cudaMemcpyDeviceToHost, ctx->stream));
    WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    rec = reinterpret_cast<const wg_kajita_online_walk *>(hb + sb);
  }
  int64_t total = 0;
  for (int i = 0; i < n; ++i) {
    if (const char *why = ko_record_refusal(h, rec[i])) return wg_refuse(ctx, call, why);
    total += rec[i].stacked;
  }
  if (total != stack_len) return wg_refuse(ctx, call, "the stacks hold other than stack_len steps");
  for (int64_t k = 0; k < stack_len; ++k)
    if (!ko_step_ok(h, stack_host[k])) return wg_refuse(ctx, call, "a stacked step timing out of range or longer than max_step_time");
  int32_t *hi = reinterpret_cast<int32_t *>(hb);
  KoSpan *hs = reinterpret_cast<KoSpan *>(hb + ib);
  for (int i = 0; i < n; ++i) {
    hi[i] = idx ? idx[i] : i;
    hs[i] = KoSpan{hi[i], (int32_t)(rec[i].popped % h->R), (int32_t)(rec[i].stream.samples_emitted - rec[i].popped), 0};
  }
  if ((rc = wgi_stage_send(ctx, &h->stage, sb)) != WG_OK) return rc;
  const wg_kajita_online_walk *d_w = walks;
  const double *d_c = carry;
  const wg_kajita_tick *d_q = queue;
  if (mem == WG_MEM_HOST) {
    wg_kajita_online_walk *w;
    double *c;
    wg_kajita_tick *q;
    if ((rc = ko_io(h, n, &w, &c, &q)) != WG_OK) return rc;
    WG_CUDA(ctx, cudaMemcpyAsync(w, walks, sizeof(wg_kajita_online_walk) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    if (h->NL > 1)
      WG_CUDA(ctx, cudaMemcpyAsync(c, carry, sizeof(double2) * (size_t)(h->NL - 1) * n, cudaMemcpyHostToDevice, ctx->stream));
    WG_CUDA(ctx, cudaMemcpyAsync(q, queue, sizeof(wg_kajita_tick) * (size_t)h->R * n, cudaMemcpyHostToDevice, ctx->stream));
    d_w = w; d_c = c; d_q = q;
  }
  wg_prof_start(ctx, WG_K_ZMPDISC);
  kajita_online_restore_kernel<<<wgi_grid(ctx, n, KO_WARPS, KO_CTAS_PER_SM), KO_WARPS * 32, 0, ctx->stream>>>(
      n, reinterpret_cast<const KoSpan *>(h->stage.d + ib), d_w, reinterpret_cast<const uint4 *>(d_q), h->R,
      reinterpret_cast<uint4 *>(h->d_ring), h->d_clock);
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  if ((rc = wgi_kajita_stream_restore_strided(h->s, n, hi, reinterpret_cast<const int32_t *>(h->stage.d), rec, d_w,
                                              sizeof(wg_kajita_online_walk), d_c)) != WG_OK)
    return rc;
  if (mem == WG_MEM_HOST) WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  int64_t at = 0;
  for (int i = 0; i < n; ++i) {
    const wg_kajita_online_walk &r = rec[i];
    KoWalk &w = h->walks[hi[i]];
    w.stack.assign(stack_host + at, stack_host + at + r.stacked);
    at += r.stacked;
    w.emitted = r.stream.samples_emitted;
    w.popped = r.popped;
    w.keep = r.keep;
    w.running = r.running; w.online = r.online; w.transition = r.transition;
  }
  return WG_OK;
}

int wg_kajita_online_copy(wg_kajita_online *dst, int n, const int32_t *dst_idx, const wg_kajita_online *src, const int32_t *src_idx)
{
  if (!dst || !src) return WG_ERR_INVALID;
  wg_ctx *ctx = dst->ctx;
  const char *call = "wg_kajita_online_copy";
  if (n < 0) return wg_refuse(ctx, call, "n < 0");
  if (src->ctx != ctx) return wg_refuse(ctx, call, "handles of two contexts");
  if (dst->NL != src->NL || dst->R != src->R) return wg_refuse(ctx, call, "NL or ring rows differ");
  if (const char *why = wgi_copy_indices_refusal(n, dst->B, dst_idx, src->B, src_idx, dst == src)) return wg_refuse(ctx, call, why);
  if (n == 0) return WG_OK;
  wg_device_guard guard(ctx->device);
  int rc = wg_kajita_stream_copy(dst->s, n, dst_idx, src->s, src_idx);
  if (rc != WG_OK) return rc;
  const size_t bytes = sizeof(KoPair) * (size_t)n;
  unsigned char *hb;
  if ((rc = wgi_stage_reserve(ctx, &dst->stage, bytes, &hb)) != WG_OK) return rc;
  KoPair *hp = reinterpret_cast<KoPair *>(hb);
  for (int i = 0; i < n; ++i) {
    const int d = dst_idx ? dst_idx[i] : i, s = src_idx ? src_idx[i] : i;
    const KoWalk &w = src->walks[s];
    hp[i] = KoPair{d, s, (int32_t)(w.popped % src->R), (int32_t)(w.emitted - w.popped)};
  }
  if ((rc = wgi_stage_send(ctx, &dst->stage, bytes)) != WG_OK) return rc;
  wg_prof_start(ctx, WG_K_ZMPDISC);
  kajita_online_copy_kernel<<<wgi_grid(ctx, n, KO_WARPS, KO_CTAS_PER_SM), KO_WARPS * 32, 0, ctx->stream>>>(
      n, reinterpret_cast<const KoPair *>(dst->stage.d), dst->R, reinterpret_cast<const uint4 *>(src->d_ring), src->d_clock,
      reinterpret_cast<uint4 *>(dst->d_ring), dst->d_clock);
  wg_prof_stop(ctx);
  WG_LAUNCHED(ctx);
  for (int i = 0; i < n; ++i)          // the index sets are disjoint when dst == src: no entry is read after it is written
    dst->walks[hp[i].d] = src->walks[hp[i].s];
  return WG_OK;
}

}  // extern "C"
