// belief.cuh -- device helpers shared by the planners, the simulator's
// filter and the closed-loop rollout kernels (rollout.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "philox.h"

namespace pp2d {

// naive probability of slot i under action u (sim:459-495)
__host__ __device__ __forceinline__ float naive_prob(int u, int i) {
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

// One step of the simulated world of the closed-loop rollouts (DESIGN.md
// section 7c), the same on the device (sim_rollout_kernel) and on the host
// (pp2d_sim_rollout_pomdp): from `cell` under action u, step t of episode e
// of `seed`.  Motion: the first slot whose running sum of naive_prob (from +0,
// each add rounded) exceeds r[0], else the last slot of non-zero probability;
// a blocked or out-of-map target keeps the cell and counts a collision.
// Sensors up, left, right, down of the new cell (out of the map reads as
// occupied), each flipped when its uniform is < 0.02; bit j = sensor j.
struct WorldStep { uint32_t cell, meas; bool collided; };
__host__ __device__ __forceinline__ WorldStep world_step(int H, int W, const uint8_t* map,
                                                         uint32_t cell, int u, uint64_t seed,
                                                         uint64_t e, uint32_t t) {
  float r[5];
  pp2d_step_uniforms(seed, e, t, r);
  int slot = -1, last = 4;
  float acc = 0.0f;
  for (int k = 0; k < 9; ++k) {
    const float pk = naive_prob(u, k);
    if (pk != 0.0f) last = k;
#ifdef __CUDA_ARCH__
    acc = __fadd_rn(acc, pk);
#else
    acc = acc + pk;                        // (SSE: one rounding to nearest)
#endif
    if (slot < 0 && r[0] < acc) slot = k;
  }
  if (slot < 0) slot = last;
  WorldStep w{0, 0, false};
  int x = (int)(cell % (uint32_t)W), y = (int)(cell / (uint32_t)W);
  if (slot != 4) {
    const int tx = x + slot % 3 - 1, ty = y + slot / 3 - 1;
    if (tx < 0 || tx >= W || ty < 0 || ty >= H || map[ty * W + tx] > 0) w.collided = true;
    else { x = tx; y = ty; }
  }
  const int ox[4] = {0, -1, 1, 0}, oy[4] = {-1, 0, 0, 1};
  for (int j = 0; j < 4; ++j) {
    const int mx = x + ox[j], my = y + oy[j];
    uint32_t v = (mx < 0 || mx >= W || my < 0 || my >= H) ? 1u : (map[my * W + mx] ? 1u : 0u);
    if (r[1 + j] < 0.02f) v ^= 1u;
    w.meas |= v << j;
  }
  w.cell = (uint32_t)(y * W + x);
  return w;
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
