// wg_ctx.cu - context, memory and timing entry points of the C ABI (include/walkgen_b200.h).
#include "wg_common.h"
#include <algorithm>

extern "C" void wg_preview_release(wg_ctx *ctx);
extern void wg_herdt_release(wg_ctx *ctx);
extern void wg_herdt_mpc_release(wg_ctx *ctx);
extern void wg_pldp_release(wg_ctx *ctx);
extern void wg_dimitrov_release(wg_ctx *ctx);
extern void wg_qld_release(wg_ctx *ctx);
extern void wg_wieber_release(wg_ctx *ctx);

#include <map>
#include <mutex>
#include <utility>

namespace {
std::mutex g_attr_mutex;
std::map<std::pair<int, const void *>, size_t> g_attr_smem;   // largest dynamic shared memory size set per (device, kernel)
}

extern "C" int wgi_smem_attr(wg_ctx *ctx, const void *func, size_t bytes)
{
  if (bytes <= 48 * 1024) return WG_OK;   // the default limit needs no opt-in
  std::lock_guard<std::mutex> lock(g_attr_mutex);
  size_t &set = g_attr_smem[{ctx->device, func}];
  if (bytes > set) {
    WG_CUDA(ctx, cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    set = bytes;
  }
  return WG_OK;
}

extern "C" int wgi_grow_scratch(wg_ctx *ctx, void **buf, size_t *cap, size_t bytes)
{
  bytes = std::max<size_t>(bytes, 8);
  if (*buf && *cap >= bytes) return WG_OK;
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  cudaFree(*buf);
  *buf = nullptr; *cap = 0;
  WG_CUDA(ctx, cudaMalloc(buf, bytes));
  *cap = bytes;
  return WG_OK;
}

int wgi_stage_reserve(wg_ctx *ctx, wgi_stage *st, size_t bytes, unsigned char **host)
{
  if (!st->ev) WG_CUDA(ctx, cudaEventCreateWithFlags(&st->ev, cudaEventDisableTiming));
  else WG_CUDA(ctx, cudaEventSynchronize(st->ev));
  if (bytes > st->h_cap) {
    cudaFreeHost(st->h);
    st->h = nullptr; st->h_cap = 0;
    WG_CUDA(ctx, cudaMallocHost(&st->h, bytes + bytes / 2));
    st->h_cap = bytes + bytes / 2;
  }
  *host = st->h;
  return WG_OK;
}

int wgi_stage_send(wg_ctx *ctx, wgi_stage *st, size_t bytes, size_t room)
{
  const size_t need = std::max(bytes, room);
  int rc;
  if ((need > st->d_cap || !st->d) &&
      (rc = wgi_grow_scratch(ctx, reinterpret_cast<void **>(&st->d), &st->d_cap, std::max(need + need / 2, (size_t)256))) != WG_OK)
    return rc;
  if (bytes) WG_CUDA(ctx, cudaMemcpyAsync(st->d, st->h, bytes, cudaMemcpyHostToDevice, ctx->stream));
  WG_CUDA(ctx, cudaEventRecord(st->ev, ctx->stream));
  return WG_OK;
}

void wgi_stage_free(wgi_stage *st)
{
  if (st->ev) cudaEventDestroy(st->ev);
  cudaFreeHost(st->h);
  cudaFree(st->d);
}

bool wgi_record_indices_ok(int B, int n, const int32_t *idx, bool unique, std::vector<char> &mark)
{
  if (!idx) {
    if (n > B) return false;
    for (int i = 0; i < n; ++i) mark[i] = 1;
    return true;
  }
  for (int i = 0; i < n; ++i) {
    const int32_t b = idx[i];
    if (b < 0 || b >= B || (unique && mark[b])) return false;
    mark[b] = 1;
  }
  return true;
}

const char *wgi_copy_indices_refusal(int n, int dB, const int32_t *dst_idx, int sB, const int32_t *src_idx, bool same)
{
  std::vector<char> dmark((size_t)dB, 0), smark((size_t)sB, 0);
  if (!wgi_record_indices_ok(dB, n, dst_idx, true, dmark) || !wgi_record_indices_ok(sB, n, src_idx, false, smark))
    return "index out of range, repeated destination, or n > B without indices";
  if (same)
    for (int b = 0; b < dB; ++b)
      if (dmark[b] && smark[b]) return "an index is both a source and a destination";
  return nullptr;
}

extern "C" {

int wg_version(void) { return WG_VERSION; }

int wg_device_count(void)
{
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int wg_ctx_create(int device, wg_ctx **out)
{
  if (!out) return WG_ERR_INVALID;
  *out = nullptr;
  int n = wg_device_count();
  if (n <= 0 || device < 0 || device >= n) return WG_ERR_NO_DEVICE;  // no CPU fallback, by design
  wg_ctx *ctx = new (std::nothrow) wg_ctx();
  if (!ctx) return WG_ERR_ALLOC;
  ctx->device = device;
  cudaError_t e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev0);
  if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev1);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
  if (e != cudaSuccess) { delete ctx; return WG_ERR_CUDA; }
  *out = ctx;
  return WG_OK;
}

int wg_ctx_destroy(wg_ctx *ctx)
{
  if (!ctx) return WG_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  wg_preview_release(ctx);
  wg_herdt_mpc_release(ctx);
  wg_herdt_release(ctx);
  wg_dimitrov_release(ctx);
  wg_wieber_release(ctx);
  wg_qld_release(ctx);
  wg_pldp_release(ctx);
  for (cudaEvent_t e : ctx->prof.ev) cudaEventDestroy(e);
  cudaEventDestroy(ctx->ev0);
  cudaEventDestroy(ctx->ev1);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
  return WG_OK;
}

int wg_sync(wg_ctx *ctx)
{
  if (!ctx) return WG_ERR_INVALID;
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return WG_OK;
}

const char *wg_last_error(wg_ctx *ctx) { return ctx ? ctx->err : "null context"; }
void *wg_ctx_stream(wg_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

int wg_malloc_device(wg_ctx *ctx, size_t bytes, void **out)
{
  if (!ctx || !out) return WG_ERR_INVALID;
  wg_device_guard g(ctx->device);
  WG_CUDA(ctx, cudaMalloc(out, bytes ? bytes : 1));
  return WG_OK;
}
int wg_free_device(wg_ctx *ctx, void *p)
{
  if (!ctx) return WG_ERR_INVALID;
  wg_device_guard g(ctx->device);
  WG_CUDA(ctx, cudaFree(p));
  return WG_OK;
}
int wg_malloc_pinned(wg_ctx *ctx, size_t bytes, void **out)
{
  if (!ctx || !out) return WG_ERR_INVALID;
  wg_device_guard g(ctx->device);
  WG_CUDA(ctx, cudaMallocHost(out, bytes ? bytes : 1));
  return WG_OK;
}
int wg_free_pinned(wg_ctx *ctx, void *p)
{
  if (!ctx) return WG_ERR_INVALID;
  WG_CUDA(ctx, cudaFreeHost(p));
  return WG_OK;
}
int wg_memcpy_h2d(wg_ctx *ctx, void *dst, const void *src, size_t bytes)
{
  if (!ctx) return WG_ERR_INVALID;
  wg_device_guard g(ctx->device);
  WG_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return WG_OK;
}
int wg_memcpy_d2h(wg_ctx *ctx, void *dst, const void *src, size_t bytes)
{
  if (!ctx) return WG_ERR_INVALID;
  wg_device_guard g(ctx->device);
  WG_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  return WG_OK;
}
// 16 bytes per thread, grid-stride: small fills (the states of a batch) stay on the SMs, in order with the kernels around them
__global__ void __launch_bounds__(256) wg_fill_kernel(uint4 *__restrict__ p, unsigned v32, size_t n16)
{
  const uint4 v = make_uint4(v32, v32, v32, v32);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}
int wg_memset_device(wg_ctx *ctx, void *dst, int value, size_t bytes)
{
  if (!ctx) return WG_ERR_INVALID;
  wg_device_guard g(ctx->device);
  if (bytes == 0) return WG_OK;
  if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0 && (bytes & 15) == 0) {
    const unsigned b = (unsigned)value & 0xffu, v32 = b | (b << 8) | (b << 16) | (b << 24);
    const size_t n16 = bytes / 16;
    const int blocks = (int)std::min<size_t>((n16 + 255) / 256, (size_t)ctx->sm_count * 8);
    wg_fill_kernel<<<blocks, 256, 0, ctx->stream>>>(static_cast<uint4 *>(dst), v32, n16);
    WG_CUDA(ctx, cudaGetLastError());
    WG_LAUNCHED(ctx);
    return WG_OK;
  }
  WG_CUDA(ctx, cudaMemsetAsync(dst, value, bytes, ctx->stream));
  return WG_OK;
}

int wg_timer_start(wg_ctx *ctx)
{
  if (!ctx) return WG_ERR_INVALID;
  WG_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  return WG_OK;
}
int wg_timer_stop_ms(wg_ctx *ctx, float *ms)
{
  if (!ctx || !ms) return WG_ERR_INVALID;
  WG_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  WG_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
  WG_CUDA(ctx, cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
  return WG_OK;
}

int wg_prof_begin(wg_ctx *ctx, int capacity)
{
  if (!ctx || capacity < 0) return WG_ERR_INVALID;
  wg_device_guard g(ctx->device);
  wg_prof_state &p = ctx->prof;
  while (p.ev.size() < 2 * (size_t)capacity) {
    cudaEvent_t e;
    WG_CUDA(ctx, cudaEventCreate(&e));
    p.ev.push_back(e);
  }
  p.kid.assign(p.ev.size() / 2, 0);
  p.used = 0;
  for (int k = 0; k < WG_K_COUNT; ++k) { p.launches[k] = 0; p.total_ms[k] = 0.0; }
  p.on = true;
  return WG_OK;
}
int wg_prof_end(wg_ctx *ctx)
{
  if (!ctx) return WG_ERR_INVALID;
  wg_device_guard g(ctx->device);
  wg_prof_state &p = ctx->prof;
  p.on = false;
  WG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (size_t i = 0; i < p.used; ++i) {
    float ms = 0.f;
    WG_CUDA(ctx, cudaEventElapsedTime(&ms, p.ev[2 * i], p.ev[2 * i + 1]));
    p.launches[p.kid[i]]++;
    p.total_ms[p.kid[i]] += ms;
  }
  return WG_OK;
}
int wg_prof_get(wg_ctx *ctx, int kernel_id, long long *launches, double *total_ms)
{
  if (!ctx || kernel_id < 0 || kernel_id >= WG_K_COUNT) return WG_ERR_INVALID;
  if (launches) *launches = ctx->prof.launches[kernel_id];
  if (total_ms) *total_ms = ctx->prof.total_ms[kernel_id];
  return WG_OK;
}

long long wg_launch_count(wg_ctx *ctx) { return ctx ? ctx->launches : 0; }
void wg_launch_count_reset(wg_ctx *ctx) { if (ctx) ctx->launches = 0; }

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// FP64 peak: every thread runs 8 independent DFMA chains held in registers.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) wg_dfma_peak_kernel(double *out, int iters, double a, double b)
{
  double r0 = threadIdx.x, r1 = r0 + 1, r2 = r0 + 2, r3 = r0 + 3, r4 = r0 + 4, r5 = r0 + 5, r6 = r0 + 6, r7 = r0 + 7;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      r0 = fma(r0, a, b); r1 = fma(r1, a, b); r2 = fma(r2, a, b); r3 = fma(r3, a, b);
      r4 = fma(r4, a, b); r5 = fma(r5, a, b); r6 = fma(r6, a, b); r7 = fma(r7, a, b);
    }
  }
  double s = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
  if (s == 123.456) out[blockIdx.x * blockDim.x + threadIdx.x] = s;  // never true; keeps the chains live
}

extern "C" int wg_measure_fp64_peak(wg_ctx *ctx, double *tflops)
{
  if (!ctx || !tflops) return WG_ERR_INVALID;
  wg_device_guard g(ctx->device);
  double *d = nullptr;
  int blocks = ctx->sm_count * 8, threads = 256, iters = 4096;
  WG_CUDA(ctx, cudaMalloc(&d, sizeof(double) * blocks * threads));
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    WG_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    wg_dfma_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(d, iters, 0.999999, 1e-9);
    WG_LAUNCHED(ctx);
    WG_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    WG_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
    float ms = 0.f;
    WG_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    double flops = 2.0 * 64.0 * (double)iters * blocks * threads;
    double tf = flops / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaFree(d);
  *tflops = best;
  return WG_OK;
}
