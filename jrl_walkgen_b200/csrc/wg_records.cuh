// wg_records.cuh - device helpers of the whole-record kernels (save / restore / copy) of the on-line generators.
#pragma once
#include <cstdint>

// Words [0, nv) of dst from src, by one warp, UNROLL loads of a lane in flight before its stores; words from `keep` on are 0.
template <int UNROLL>
__device__ __forceinline__ void wgi_warp_copy16(uint4 *__restrict__ dst, const uint4 *__restrict__ src, int nv, int64_t keep, int lane)
{
  if (keep > nv) keep = nv;
  for (int e0 = 0; e0 < nv; e0 += 32 * UNROLL) {
    uint4 v[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const int e = e0 + 32 * u + lane;
      v[u] = (e < keep) ? src[e] : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const int e = e0 + 32 * u + lane;
      if (e < nv) dst[e] = v[u];
    }
  }
}
