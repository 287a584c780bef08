// fib_activation.cuh -- activation maps (fib_activation_watch): per cell, the threshold crossings of the
// diffusing variable between consecutive ODE-iteration samples, with linear interpolation -- the event rule
// of tests/test_spiral_statistics.py events(), evaluated at every cell on the device.
//
// Samples: s[0] = the plane when the map is armed, s[k] = the plane at the end of the k-th ODE iteration
// since.  In iteration k (prev = s[k-1], cur = s[k], k1 = (float)(k - 1), exact up to 2^24):
//   activation      prev < up <= cur     t = k1 + (up - prev) / (cur - prev)
//   repolarisation  prev >= down > cur   t = k1 + (prev - down) / (prev - cur)
// (exclusive: the first needs cur > prev, the second cur < prev).  One rounding per operation (__fsub_rn,
// __fdiv_rn, __fadd_rn; the library is built with -fmad=false), so oracle/activation_np.py reproduces the
// maps bit for bit.  A NaN sample compares false and produces no event.
//
// Five planes of the shard's row layout (rows x pitch, no halo), `plane` floats apart:
//   FIRST / LAST / PREV (the activation before LAST) / REPOL: NaN until set; COUNT: activations, as a float.
// A cell loads and stores the maps only when it has an event: 12 bytes per cell per iteration otherwise
// (read the plane and `prev`, write `prev`).
#pragma once
#include "fib_common.cuh"

namespace fib {

enum { kActFirst = 0, kActLast = 1, kActPrev = 2, kActRepol = 3, kActCount = 4, kActMaps = 5 };

__device__ __forceinline__ void act_cell(float prev, float cur, float k1, float up, float down,
                                         float* __restrict__ m, size_t plane) {
  if (prev < up && up <= cur) {
    const float t = __fadd_rn(k1, __fdiv_rn(__fsub_rn(up, prev), __fsub_rn(cur, prev)));
    if (isnan(m[kActFirst * plane])) m[kActFirst * plane] = t;
    m[kActPrev * plane] = m[kActLast * plane];
    m[kActLast * plane] = t;
    m[kActCount * plane] = __fadd_rn(m[kActCount * plane], 1.0f);
  } else if (prev >= down && down > cur) {
    m[kActRepol * plane] = __fadd_rn(k1, __fdiv_rn(__fsub_rn(prev, down), __fsub_rn(prev, cur)));
  }
}

// One sample of the whole shard: `x` = the owned rows of the diffusing variable, `prev` = the last sample
// (overwritten with this one), `*iter` = samples taken since arming, i.e. k - 1.  n4 = rows * pitch / 4.
__global__ void __launch_bounds__(256) activation_update_kernel(const float4* __restrict__ x,
                                                                float4* __restrict__ prev,
                                                                float* __restrict__ maps, size_t n4,
                                                                size_t plane,
                                                                const unsigned long long* __restrict__ iter,
                                                                float up, float down) {
  const float k1 = (float)*iter;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 b = x[i], a = prev[i];
    prev[i] = b;
    float* m = maps + 4 * i;
    act_cell(a.x, b.x, k1, up, down, m + 0, plane);
    act_cell(a.y, b.y, k1, up, down, m + 1, plane);
    act_cell(a.z, b.z, k1, up, down, m + 2, plane);
    act_cell(a.w, b.w, k1, up, down, m + 3, plane);
  }
}

// the iteration index of the next sample: a node of the iteration graph after the update (graph replays
// cannot take new kernel arguments)
__global__ void activation_advance_kernel(unsigned long long* __restrict__ iter) { *iter += 1; }

// arming: FIRST / LAST / PREV / REPOL := NaN, COUNT := 0
__global__ void activation_reset_kernel(float* __restrict__ maps, size_t plane) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < kActMaps * plane;
       i += (size_t)gridDim.x * blockDim.x)
    maps[i] = i >= kActCount * plane ? 0.0f : __int_as_float(0x7fc00000);
}

}  // namespace fib
