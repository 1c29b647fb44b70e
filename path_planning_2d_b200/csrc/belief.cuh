// belief.cuh -- device helpers shared by the planners, the simulator's
// filter and the closed-loop rollout kernels (rollout.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace pp2d {

// naive probability of slot i under action u (sim:459-495)
__device__ __forceinline__ float naive_prob(int u, int i) {
  if (u == 4) return i == 4 ? 1.0f : 0.0f;
  if (i == u) return 0.7f;
  if (i == 4) return 0.1f;
  // the two side slots of each action
  const int s0 = (u == 0) ? 1 : (u == 1) ? 0 : (u == 2) ? 1 : (u == 3) ? 0 :
                 (u == 5) ? 2 : (u == 6) ? 3 : (u == 7) ? 6 : 5;
  const int s1 = (u == 0) ? 3 : (u == 1) ? 2 : (u == 2) ? 5 : (u == 3) ? 6 :
                 (u == 5) ? 8 : (u == 6) ? 7 : (u == 7) ? 8 : 7;
  return (i == s0 || i == s1) ? 0.1f : 0.0f;
}

// MdpPathPlanning2d::beliefCallback (path_planning_2d.cu:168-189): index of
// the first strict maximum of the belief b[0 .. n) starting from (0.0f,
// index 0), valid in thread 0 of a 256-thread CTA.
__device__ __forceinline__ unsigned long long belief_mode(const float* __restrict__ b, size_t n) {
  float bm = 0.0f;
  unsigned long long bi = 0;
  for (size_t i = threadIdx.x; i < n; i += blockDim.x) {
    float v = b[i];
    if (v > bm) { bm = v; bi = i; }   // ascending i per thread: first max kept
  }
  // (value, index) reduction: larger value wins, ties -> smaller index.
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float ov = __shfl_xor_sync(0xffffffffu, bm, o);
    unsigned long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bm || (ov == bm && oi < bi)) { bm = ov; bi = oi; }
  }
  __shared__ float sv[8];
  __shared__ unsigned long long si[8];
  if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = bm; si[threadIdx.x >> 5] = bi; }
  __syncthreads();
  if (threadIdx.x == 0)
    for (int i = 1; i < 8; ++i)
      if (sv[i] > bm || (sv[i] == bm && si[i] < bi)) { bm = sv[i]; bi = si[i]; }
  // all beliefs <= 0: the reference keeps index 0.
  return bm > 0.0f ? bi : 0;
}

}  // namespace pp2d
