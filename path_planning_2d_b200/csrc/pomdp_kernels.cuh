// pomdp_kernels.cuh -- sm_100a kernels of the QV-Tree half (SURVEY.md rows
// B1-B7).  Reference files, relative to /root/reference/path_planning_2d/:
//   model_gen = src/pomdp/model_generation_cuda.cu
//   pbvi      = src/pomdp/point_based_value_iteration_cuda.cu
//   fib       = src/pomdp/fast_informed_bound_cuda.cu
//   tree      = src/pomdp/search_tree_cuda.cu
//
// Layout: every belief of a batch is a COLUMN of a pool cut into blocks of 32
// slots (belief ids), inside a block cell-major:
//   bel[((slot / 32) * HW + s) * 32 + slot % 32]      s = cell (y*W+x)
// so that "one thread per belief, sequential over the cells" kernels are
// coalesced (32 neighbouring slots of a cell are one 128-byte line) AND a
// belief stays inside one HW * 128-byte region: with one [HW][cap] matrix the
// cells of a column were cap * 4 bytes apart -- 4 000 different pages for the
// 43 GB pool of a 1 250-query batch -- and every kernel that walks a column
// waited on the TLB.  That shape is what makes bit-exact parity possible: the
// reference normalises, prefix-sums and takes inner products with sequential
// single-accumulator float loops on the host (tree:226-229, 326-328,
// fib:289-292, pbvi:689-694).  Here each of those loops is run by one thread
// in the same order with the same roundings (separate multiply and add, IEEE
// division, subnormals kept), and the parallelism comes from the thousands of
// beliefs a batch of queries holds.  The device-side arithmetic of the
// reference (--use_fast_math: FFMA contraction, flush-to-zero) is reproduced
// with explicit .ftz PTX.
#pragma once
#include <cuda_runtime.h>
#include <curand_kernel.h>
#include <stdint.h>

#include "async_copy.cuh"
#include "fp_exact.cuh"
#include "pomdp_host.h"

namespace pp2d {

// ---------------------------------------------------------------- B1 -------
// model_gen:161-347: per cell trans_prob[9][9] (blocked mass moved to "stay"
// in ascending slot order, trapped override AFTER the naive copy),
// meas_prob[16] and stage_reward[9] (-1 free / -2 occupied over the naive
// probabilities; stay = -2, 0 at the goal).  Same table layout as the
// reference so that save_data / the FIB and PBVI solvers can consume them.
__global__ void pomdp_model_kernel(int H, int W, int gx, int gy,
                                   const uint8_t* __restrict__ map,
                                   float* __restrict__ trans_prob,
                                   float* __restrict__ meas_prob,
                                   float* __restrict__ stage_reward) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  if (x >= W || y >= H) return;
  const size_t idx = (size_t)y * W + x;
  uint8_t m[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    const int nx = x + i % 3 - 1, ny = y + i / 3 - 1;
    m[i] = (nx < 0 || nx >= W || ny < 0 || ny >= H) ? 1
           : (map[(size_t)ny * W + nx] == 1 ? 1 : 0);
  }
  // naive probabilities of action u: 0.7 at slot u, 0.1 at the two side
  // slots and at the centre (model_gen:175-211).
  const int side[9][2] = {{1, 3}, {0, 2}, {1, 5}, {0, 6}, {4, 4},
                          {2, 8}, {3, 7}, {6, 8}, {5, 7}};
  for (int u = 0; u < 9; ++u) {
    float tp[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) tp[i] = 0.0f;
    if (u == 4) {
      tp[4] = 1.0f;
    } else {
      tp[u] = 0.7f; tp[side[u][0]] = 0.1f; tp[side[u][1]] = 0.1f; tp[4] = 0.1f;
    }
    // stage reward over the naive probabilities (model_gen:287-290): the
    // reward is -1 / -2, so the product is exact and the chain is the
    // reference's FFMA chain.
    float r = 0.0f;
#pragma unroll
    for (int i = 0; i < 9; ++i) r = fma_ftz(m[i] ? -2.0f : -1.0f, tp[i], r);
    if (u == 4) r = (x != gx || y != gy) ? -2.0f : 0.0f;
    stage_reward[idx * 9 + u] = r;
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      if (m[i] && i != 4) { tp[4] = add_ftz(tp[4], tp[i]); tp[i] = 0.0f; }
    }
    if (m[4]) {
#pragma unroll
      for (int i = 0; i < 9; ++i) tp[i] = 0.0f;
      tp[4] = 1.0f;
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) trans_prob[idx * 81 + u * 9 + i] = tp[i];
  }
  // model_gen:235-263: 0.98 / 0.02 are double literals rounded to float.
  const float hit = (float)0.98, miss = (float)0.02;
  const uint8_t mm[4] = {m[1], m[3], m[5], m[7]};
  for (int z = 0; z < 16; ++z) {
    const float l0 = ((z >> 0) & 1) == mm[0] ? hit : miss;
    const float l1 = ((z >> 1) & 1) == mm[1] ? hit : miss;
    const float l2 = ((z >> 2) & 1) == mm[2] ? hit : miss;
    const float l3 = ((z >> 3) & 1) == mm[3] ? hit : miss;
    meas_prob[idx * 16 + z] = mul_ftz(mul_ftz(mul_ftz(l0, l1), l2), l3);
  }
}

// Cells no probability mass can ENTER: dead[s'] = 1 when P(s, u, s') == 0 for
// every action u and every neighbour s != s' inside the map (the only inflow
// of such a cell is from itself).  For the generated model these are the
// occupied cells (blocked mass is shifted to "stay", model_gen:213-233) plus
// free cells walled in on all sides; the mask is derived from the TABLES, so
// it also holds for tables loaded from a checkpoint.  A belief that is +0 on
// the dead cells keeps exact +0 there through every Bayes update
// (sum of +0 products, times the likelihood, divided by the sum), which is
// what lets the sequential inner products below skip those cells bit-exactly:
// acc + (+-0) == acc for an accumulator that starts at +0 (it can never become
// -0 under round-to-nearest).
__global__ void pomdp_dead_cells_kernel(int H, int W, const float* __restrict__ trans_prob,
                                        uint8_t* __restrict__ dead) {
  const int cell = blockIdx.x * blockDim.x + threadIdx.x;
  if (cell >= H * W) return;
  const int x = cell % W, y = cell / W;
  bool inflow = false;
  for (int s = 0; s < 9; ++s) {
    if (s == 4) continue;
    const int sx = x + s % 3 - 1, sy = y + s / 3 - 1;
    if (sx < 0 || sx >= W || sy < 0 || sy >= H) continue;
    const size_t sidx = (size_t)sy * W + sx;
    for (int u = 0; u < 9; ++u)
      inflow = inflow || (trans_prob[81 * sidx + 9 * u + (8 - s)] != 0.0f);
  }
  dead[cell] = inflow ? 0 : 1;
}

// ---------------------------------------------------------------- B2 -------
// pbvi:88-133 cudaBayesBeliefUpdate, batched: child c is made from belief
// column src[c] with action act[c] and observation obs[c] and written,
// un-normalised, to column dst[c].  threadIdx.x runs over children so that
// siblings (same source column) read the same addresses.
// (BayesItem is declared in pomdp_host.h)

__global__ void __launch_bounds__(256)
pomdp_bayes_kernel(int H, int W, const float* __restrict__ trans_prob,
                   const float* __restrict__ meas_prob,
                   const BayesItem* __restrict__ items, int n_items,
                   const float* bel_in, float* bel_out) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int cell = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (c >= n_items || cell >= H * W) return;
  const BayesItem it = items[c];
  const int x = cell % W, y = cell / W;
  // Arithmetic of the reference kernel as nvcc 12.9 compiles it for sm_100a
  // with --use_fast_math: FFMA.FTZ chain over slots 0..7, the last slot as a
  // rounded FMUL.FTZ product added with FADD.FTZ, then FMUL.FTZ by L.
  float p = 0.0f;
#pragma unroll
  for (int s = 0; s < 9; ++s) {
    const int sx = x + s % 3 - 1, sy = y + s / 3 - 1;
    if (sx < 0 || sx >= W || sy < 0 || sy >= H) continue;
    const size_t sidx = (size_t)sy * W + sx;
    const float tp = __ldg(trans_prob + 81 * sidx + 9 * it.act + (8 - s));
    const float b = bel_in[bel_off(H * W, (int)sidx, it.src)];
    if (s < 8) p = fma_ftz(tp, b, p);
    else p = add_ftz(p, mul_ftz(tp, b));
  }
  p = mul_ftz(p, __ldg(meas_prob + 16 * (size_t)cell + it.obs));
  bel_out[bel_off(H * W, cell, it.dst)] = p;
}

// The children of one Q node (same parent belief, same action) differ only in
// the observation: the predicted belief sum_s P(s,u,s') b(s) is computed once
// per (Q node, cell).  Bayes update, column sum and division of a round
// without ever storing the un-normalised children: the prediction of a Q node
// is written once to pred[row * ngp + g] (row = position of the cell in kidx);
// the sequential sum of a child and
// its normalised belief are both formed from pred * L on the fly.  Per element
// the operations are those of pomdp_bayes_kernel + pomdp_colsum_kernel +
// pomdp_scale_kernel (FMUL.FTZ by the likelihood, sequential rounded adds,
// IEEE division), so the bits are the same; the traffic drops from
// 4 x |children| to 2 x |Q nodes| + 1 x |children| belief-sized passes.
//
// Group g = 9 * i + a is action a of expanded node i (column slots[i]): one
// thread per (node, target cell) reads the 9 neighbour beliefs ONCE and runs
// the 9 action chains (pomdp_bayes_kernel's) on them.  Lanes run over nodes,
// so the transition probabilities are warp-uniform loads, one broadcast each
// (with one thread per (group, cell) and lanes over groups every load was 3-4
// wavefronts, the belief was read 9 times and the L1 pipe bounded the kernel).
// Only the K target cells listed in kidx are predicted: on the others (cells
// no mass can enter, belief +0) the prediction is +0 and nobody reads it --
// pomdp_child_sum_kernel walks the same list and pomdp_child_write_kernel
// writes those cells without it.  kidx = identity: every cell.
__global__ void __launch_bounds__(256)
pomdp_predict9_kernel(int H, int W, int K, const int* __restrict__ kidx, int ngp,
                      const float* __restrict__ trans_prob, const int* __restrict__ slots,
                      int n, const float* __restrict__ bel, float* __restrict__ pred) {
  const int i = blockIdx.x * 32 + (threadIdx.x & 31);
  const int kc = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (kc >= K) return;                             // warp-uniform
  const int cell = __ldg(kidx + kc);
  const int x = cell % W, y = cell / W;
  const float* col = bel + bel_off(H * W, 0, slots[min(i, n - 1)]);
  float b[9];
#pragma unroll
  for (int s = 0; s < 9; ++s) {
    const int sx = x + s % 3 - 1, sy = y + s / 3 - 1;
    const bool in = !(sx < 0 || sx >= W || sy < 0 || sy >= H);   // warp-uniform
    b[s] = in ? col[(size_t)(sy * W + sx) * kSlotBlock] : 0.0f;
  }
  float* out = pred + (size_t)kc * ngp + (size_t)i * 9;   // scratch rows = inner rows
#pragma unroll
  for (int a = 0; a < 9; ++a) {
    float p = 0.0f;
#pragma unroll
    for (int s = 0; s < 9; ++s) {
      const int sx = x + s % 3 - 1, sy = y + s / 3 - 1;
      if (sx < 0 || sx >= W || sy < 0 || sy >= H) continue;
      const float tp = __ldg(trans_prob + 81 * (size_t)(sy * W + sx) + 9 * a + (8 - s));
      if (s < 8) p = fma_ftz(tp, b[s], p);
      else p = add_ftz(p, mul_ftz(tp, b[s]));
    }
    if (i < n) out[a] = p;
  }
}

// sums[k] = accumulate over cells of pred * L(., z_k), in cell order.  Only
// the K cells listed in kidx (ascending) are visited: the prediction is +0 on
// the others and sum + (+0 * L) == sum (see pomdp_dead_cells_kernel); with
// kidx = identity this is the plain loop over all HW cells.
#ifndef PP2D_CS_BATCH
#define PP2D_CS_BATCH 32
#endif
// Register double buffer with ordered (volatile) loads: the operands of the
// NEXT kCsBatch rows are requested before the current ones are added, so
// 2 * kCsBatch loads per thread are in flight during every batch.  (Plain
// loads get interleaved with the adds by ptxas -- 40 registers, ~8 loads in
// flight, long-scoreboard stall 22 per issue, 289 us per launch; this version
// 132 us; batch 8 / 16 / 32 rows: 217 / 132 / 86 us.  Staging the operands of
// 128 children through shared memory with an 8-stage cp.async pipeline was
// measured twice -- per-lane ring: 297 us; CTA tile [16 rows][groups + 16
// likelihoods]: 70 us per launch but a slower batch, its 74 KB of shared
// memory keep it from sharing an SM with the values launch of another group
// -- and dropped.)  pred and mp_rows are indexed by inner row, not by cell:
// an index load in front of every operand load was a dependent round trip.
constexpr int kCsBatch = PP2D_CS_BATCH;
__device__ __forceinline__ float ldg_f32_ordered(const float* p) {
  float v;
  asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__global__ void __launch_bounds__(128)
pomdp_child_sum_kernel(int K, int ngp, const float* __restrict__ mp_rows,
                       const BayesItem* __restrict__ items, const int* __restrict__ kgroup,
                       int n, const float* __restrict__ pred, float* __restrict__ sums) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const float* pc = pred + kgroup[k];
  const float* L = mp_rows + items[k].obs;
  float v[2][kCsBatch], l[2][kCsBatch];
  auto request = [&](int buf, int c0) {
#pragma unroll
    for (int j = 0; j < kCsBatch; ++j) {
      const int s = min(c0 + j, K - 1);                      // clamped rows are not added
      v[buf][j] = ldg_f32_ordered(pc + (size_t)s * ngp);
      l[buf][j] = ldg_f32_ordered(L + (size_t)s * 16);
    }
  };
  float sum = 0.0f;
  request(0, 0);
  for (int c0 = 0; c0 < K; c0 += 2 * kCsBatch) {
    request(1, c0 + kCsBatch);
#pragma unroll
    for (int j = 0; j < kCsBatch; ++j)
      if (c0 + j < K) sum = __fadd_rn(sum, mul_ftz(v[0][j], l[0][j]));
    request(0, c0 + 2 * kCsBatch);
#pragma unroll
    for (int j = 0; j < kCsBatch; ++j)
      if (c0 + kCsBatch + j < K) sum = __fadd_rn(sum, mul_ftz(v[1][j], l[1][j]));
  }
  sums[k] = sum;
}
// child belief = (pred * L) / sum, written once into its pool column.
// kinv[cell] < 0: a cell whose prediction is +0 by construction and was not
// computed: (+0 * L) / sum.
constexpr int kCwCells = 8;      // cells per thread: their loads are in flight together
__global__ void __launch_bounds__(256)
pomdp_child_write_kernel(int HW, int ngp, const float* __restrict__ meas_prob,
                         const int* __restrict__ kinv,
                         const BayesItem* __restrict__ items, const int* __restrict__ kgroup,
                         int n, const float* __restrict__ pred, const float* __restrict__ sums,
                         float* __restrict__ bel) {
  const int k = blockIdx.x * 32 + (threadIdx.x & 31);
  const int cell0 = (blockIdx.y * 8 + (threadIdx.x >> 5)) * kCwCells;
  if (k >= n || cell0 >= HW) return;
  const BayesItem it = items[k];
  const float sum = sums[k];
  const float* pc = pred + kgroup[k];
  const float* L = meas_prob + it.obs;
  float p[kCwCells], l[kCwCells];
#pragma unroll
  for (int j = 0; j < kCwCells; ++j) {
    const int cell = min(cell0 + j, HW - 1);
    const int row = __ldg(kinv + cell);              // warp-uniform
    p[j] = row < 0 ? 0.0f : pc[(size_t)row * ngp];
    l[j] = __ldg(L + 16 * (size_t)cell);
  }
  // (+-0) / sum == +-0 for a sum > 0: the IEEE division (a dozen instructions)
  // is skipped on the cells outside the child's support -- the dead cells and
  // most of the map -- which whole warps share (a warp is 32 children of one or
  // two trees on one cell).
  const bool pos = sum > 0.0f;
#pragma unroll
  for (int j = 0; j < kCwCells; ++j) {
    if (cell0 + j >= HW) break;
    const float v = mul_ftz(p[j], l[j]);
    bel[bel_off(HW, cell0 + j, it.dst)] = (v == 0.0f && pos) ? v : __fdiv_rn(v, sum);
  }
}

// ---------------------------------------------------------------- B3 -------
// tree:226-229: sum = accumulate(b, 0.0f) sequentially, then b /= sum (IEEE
// division).  One thread per belief column.
// The sum is a serial chain of float adds by construction; the loads are
// issued 32 at a time so that memory latency overlaps.
__global__ void __launch_bounds__(128)
pomdp_colsum_kernel(int HW, const int* __restrict__ slots, int n,
                    const float* __restrict__ bel, float* __restrict__ sums) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* col = bel + bel_off(HW, 0, slots[i]);
  float sum = 0.0f;
  int s = 0;
  for (; s + 32 <= HW; s += 32) {
    float v[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = col[(size_t)(s + j) * kSlotBlock];
#pragma unroll
    for (int j = 0; j < 32; ++j) sum = __fadd_rn(sum, v[j]);
  }
  for (; s < HW; ++s) sum = __fadd_rn(sum, col[(size_t)s * kSlotBlock]);
  sums[i] = sum;
}

// b /= sum for every cell of every listed column (tree:228-229), IEEE division.
__global__ void __launch_bounds__(256)
pomdp_scale_kernel(int HW, const int* __restrict__ slots, int n,
                   const float* __restrict__ sums, float* __restrict__ bel) {
  const int i = blockIdx.x * 32 + (threadIdx.x & 31);
  const int s = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (i >= n || s >= HW) return;
  const size_t q = bel_off(HW, s, slots[i]);
  bel[q] = __fdiv_rn(bel[q], sums[i]);
}

// ---------------------------------------------------------------- B7 -------
// tree:326-328: distribution = partial_sum(belief) (sequential float adds).
// One WARP per expanded V node: the lanes fetch 32 consecutive cells (their
// addresses are a pool row apart, so all 32 loads are in flight together),
// then every lane replays the 32 adds in order from registers (shuffles) and
// keeps the partial sum of its own cell.  prefix[i * HW + s].
constexpr int kSeqDepth = 8;     // chunks of 32 cells requested ahead of the add chain
// (body shared with pomdp_expand_kernel; one warp, belief column `col`)
// The 32 values of a chunk reach every lane through the warp's 128 bytes of
// shared memory (one store, 8 broadcast LDS.128) rather than 32 shuffles: the
// shuffle unit, one per SM, was what bounded this kernel.
__device__ __forceinline__ void prefix_body(int HW, int lane, const float* __restrict__ col,
                                            float* __restrict__ out, float* __restrict__ sw) {
  float acc = 0.0f;
  // The chain of adds is serial by construction; what can overlap is the memory
  // latency: kSeqDepth chunks are in flight while one is summed.  Lanes past
  // the end hold +0 and acc + 0 == acc, so every chunk replays all 32 adds
  // (no trip count, fully unrolled: the dependent FADD is the only latency).
  float nxt[kSeqDepth];
#pragma unroll
  for (int d = 0; d < kSeqDepth; ++d) {
    const int sn = d * 32 + lane;
    nxt[d] = sn < HW ? col[(size_t)sn * kSlotBlock] : 0.0f;
  }
  for (int s0 = 0; s0 < HW; s0 += 32 * kSeqDepth) {
#pragma unroll
    for (int d = 0; d < kSeqDepth; ++d) {
      const int c0 = s0 + d * 32;
      if (c0 >= HW) break;                         // warp-uniform
      __syncwarp();                                // the previous chunk has been read
      sw[lane] = nxt[d];
      __syncwarp();
      const int sn = c0 + 32 * kSeqDepth + lane;
      nxt[d] = sn < HW ? col[(size_t)sn * kSlotBlock] : 0.0f;
      float mine = 0.0f;
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4) {
        const float4 t = *reinterpret_cast<const float4*>(sw + 4 * j4);
        acc = __fadd_rn(acc, t.x); mine = (4 * j4 + 0 == lane) ? acc : mine;
        acc = __fadd_rn(acc, t.y); mine = (4 * j4 + 1 == lane) ? acc : mine;
        acc = __fadd_rn(acc, t.z); mine = (4 * j4 + 2 == lane) ? acc : mine;
        acc = __fadd_rn(acc, t.w); mine = (4 * j4 + 3 == lane) ? acc : mine;
      }
      if (c0 + lane < HW) out[c0 + lane] = mine;
    }
  }
}

__global__ void __launch_bounds__(128)
pomdp_prefix_kernel(int HW, const int* __restrict__ slots, int n,
                    const float* __restrict__ bel, float* __restrict__ prefix) {
  __shared__ __align__(16) float sw[4][32];
  const int i = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (i >= n) return;
  prefix_body(HW, threadIdx.x & 31, bel + bel_off(HW, 0, slots[i]), prefix + (size_t)i * HW,
              sw[threadIdx.x >> 5]);
}

// The 2*n uniforms cudaForwardSampling consumes (tree:84-92, 117, 134):
// XORWOW, curand_init(1234, idx, 0), two curand_uniform draws.  The reference
// re-creates the states for every Q node, so these numbers never change.
__global__ void pomdp_uniforms_kernel(int n, float* out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n) return;
  curandState st;
  curand_init(1234, idx, 0, &st);
  out[2 * idx] = curand_uniform(&st);
  out[2 * idx + 1] = curand_uniform(&st);
}

// tree:331-337 (state sample by inverse CDF: first prefix >= draw) followed by
// tree:94-147 cudaForwardSampling.  One thread per (expanded node i, action
// a, sample k); draws[(i*9+a)*S + k] are the host rand() values already
// divided by RAND_MAX+1.  A draw beyond the last prefix sum is clamped to the
// last cell (the reference indexes one past the belief there).
// The binary search finds the same element as the linear search for every
// belief whose entries are >= 0, +inf or NaN (a class the Bayes update keeps):
// the prefix is non-decreasing up to its first NaN and NaN from there on, so
// "prefix >= draw or NaN" is monotone, and a search that stops on a NaN
// found no prefix >= draw before it.
__global__ void __launch_bounds__(128)
pomdp_sample_kernel(int H, int W, int n, int S,
                    const float* __restrict__ trans_prob,
                    const float* __restrict__ meas_prob,
                    const float* __restrict__ prefix,
                    const float* __restrict__ draws,
                    const float* __restrict__ uniforms,
                    uint8_t* __restrict__ observations) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * 9 * S) return;
  const int k = t % S, a = (t / S) % 9, i = t / (9 * S);
  const int HW = H * W;
  const float r = draws[t];
  const float* pre = prefix + (size_t)i * HW;
  int lo = 0, hi = HW;                       // first s with !(prefix[s] < r)
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (!(pre[mid] < r)) hi = mid; else lo = mid + 1;
  }
  const int s1 = lo < HW && pre[lo] >= r ? lo : HW - 1;
  float cum = 0.0f;
  const float r2 = uniforms[2 * k];
  int s2 = 0;
  bool found = false;
#pragma unroll
  for (int j = 0; j < 9; ++j) {
    const float tp = trans_prob[(size_t)s1 * 81 + a * 9 + j];
    cum = j == 0 ? tp : add_ftz(tp, cum);
    if (!found && r2 <= cum) { s2 = j; found = true; }
  }
  long long nxt = (long long)s1 + (long long)(s2 / 3 - 1) * W + (s2 % 3 - 1);
  if (nxt < 0) nxt = 0;
  if (nxt >= HW) nxt = HW - 1;
  const float r3 = uniforms[2 * k + 1];
  int z = 0;
  found = false;
  cum = 0.0f;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const float mp = meas_prob[(size_t)nxt * 16 + j];
    cum = j == 0 ? mp : add_ftz(mp, cum);
    if (!found && r3 <= cum) { z = j; found = true; }
  }
  observations[t] = (uint8_t)z;
}

// ------------------------------------------------------------ B4 / B5 ------
// Values of many beliefs against many alpha vectors:
//   out[i][j] = sum_s bel[s][slots[i]] * alpha[s][j]     (j < ncol)
// evaluated exactly like std::inner_product(b, b+HW, alpha, 0.0f) on the
// reference's host (fib:289-292, pbvi:689-694, tree:172): one accumulator per
// (i, j), cells in ascending order, float multiply rounded, then float add
// rounded (no FMA).  alpha is [HW][ld]: the bound matrix has the columns
//   0..8 FIB, 9..9+N-1 PBVI
// (509 -> 512 = two column tiles for the reference's 500 vectors); ld is a
// multiple of the column tile and the padding is zero.
// CTA tile 64 beliefs x 256 columns, 256 threads, 8x8 accumulators each
// (4 LDS.128 per 128 math instructions: the 4x4 version was bound by the
// shared-memory pipe), K chunks of 16 cells double-buffered with cp.async.
// (PP2D_EVM = 128 builds the square 128 x 128 tile: same speed per row walked,
// but a tile of 128 children is five trees wide and walks 1 175 cells per
// belief on the bench batch where the 64-wide tile walks 1 128 -- of 2 358 live
// cells, 4 000 in all: 58.5 vs 56.3 ms per 1 250 plans.)
#ifndef PP2D_EVM
#define PP2D_EVM 64
#endif
constexpr int kEvM = PP2D_EVM, kEvN = 128 * 128 / PP2D_EVM, kEvK = 16, kEvPad = 4;
static_assert(kEvM == 64 || kEvM == 128, "8x8 accumulators per thread, 256 threads");

// The inner dimension runs over the K cells listed in kidx (ascending cell
// order); alpha holds the K matching rows.  K = HW with kidx = identity is the
// dense product; with the live cells only (pomdp_dead_cells_kernel) every
// belief of the launch must be +0 on the cells left out, and the result is
// bit-identical: the skipped terms are acc + (+-0).
//
// TILED: every tile of kEvM beliefs walks its OWN ascending list of inner rows
// (pomdp_support_kernel: the rows on which at least one belief of the tile is
// non-zero; tlist[tile * tstride + i] = {cell, row of alpha}, tcount[tile]
// entries).  On a row left out all kEvM beliefs are +-0, the products are +-0
// for finite alpha and acc + (+-0) == acc -- an accumulator that starts at +0
// never becomes -0 under round-to-nearest -- so the bits do not change.  The
// beliefs of a tree are spatially compact (a Gaussian start belief widened by
// one cell per step) and a batch is planned in the order of the start
// beliefs' modes, so a tile touches about half of the live cells.
// Per-tile list of inner rows (see TILED above), two launches.
// pomdp_support_flags_kernel: CTA (tile, chunk of 256 rows): every warp tests
// 32 rows (all kEvM beliefs of the tile per row, kEvM / 32 per lane, 8 rows in
// flight) and writes one 32-bit mask: tmask[tile * mstride + chunk * 8 + warp].
__global__ void __launch_bounds__(256)
pomdp_support_flags_kernel(int HW, int K, const int* __restrict__ kidx,
                           const int* __restrict__ slots, int n,
                           const float* __restrict__ bel, uint32_t* __restrict__ tmask,
                           int mstride) {
  __shared__ int sslot[kEvM];
  const int tile = blockIdx.x, m0 = tile * kEvM;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // (the padding of the last tile repeats one of its members)
  if (tid < kEvM) sslot[tid] = slots[min(m0 + tid, n - 1)];
  __syncthreads();
  constexpr int kPer = kEvM / 32;                  // beliefs per lane
  const float* col[kPer];
#pragma unroll
  for (int q = 0; q < kPer; ++q) col[q] = bel + bel_off(HW, 0, sslot[lane + 32 * q]);
  const int r0 = blockIdx.y * 256 + warp * 32;     // this warp's 32 rows
  if (r0 >= K) return;                             // (warp-uniform; its mask word is never read)
  const int myrow = r0 + lane;
  const int mycell = myrow < K ? __ldg(kidx + myrow) : 0;
  uint32_t mask = 0;
#pragma unroll
  for (int j0 = 0; j0 < 32; j0 += 8) {
    float v[8][kPer];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int cell = __shfl_sync(0xffffffffu, mycell, j0 + j);
      const size_t off = (size_t)cell * kSlotBlock;
#pragma unroll
      for (int q = 0; q < kPer; ++q) v[j][q] = col[q][off];
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      bool nz = false;                             // (NaN != 0: a row holding a NaN is kept)
#pragma unroll
      for (int q = 0; q < kPer; ++q) nz = nz || v[j][q] != 0.0f;
      if (__any_sync(0xffffffffu, nz) && r0 + j0 + j < K) mask |= 1u << (j0 + j);
    }
  }
  if (lane == 0) tmask[(size_t)tile * mstride + (r0 >> 5)] = mask;
}

// pomdp_support_list_kernel: one CTA per tile turns its ceil(K/32) mask words
// into the ascending list tlist[tile * K + i] = {cell, row} and tcount[tile]
// (n = beliefs of the launch).
__global__ void __launch_bounds__(256)
pomdp_support_list_kernel(int K, const int* __restrict__ kidx,
                          const uint32_t* __restrict__ tmask, int mstride,
                          int2* __restrict__ tlist, int* __restrict__ tcount, int n,
                          unsigned long long* __restrict__ work) {
  __shared__ int wsum[8];
  const int tile = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nwords = (K + 31) / 32;
  int2* out = tlist + (size_t)tile * K;
  int base = 0;
  for (int w0 = 0; w0 < nwords; w0 += 256) {
    const int w = w0 + tid;
    const uint32_t m = w < nwords ? tmask[(size_t)tile * mstride + w] : 0u;
    const int cnt = __popc(m);
    int incl = cnt;                                // inclusive scan over the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    int off = base + incl - cnt, total = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (i < warp) off += wsum[i];
      total += wsum[i];
    }
    uint32_t rest = m;
    while (rest) {
      const int b = __ffs(rest) - 1;
      rest &= rest - 1;
      const int row = w * 32 + b;
      out[off++] = make_int2(__ldg(kidx + row), row);
    }
    base += total;
    __syncthreads();
  }
  if (tid == 0) {
    tcount[tile] = base;
    // (pp2d_pomdp_work_counters: rows x beliefs this tile's values CTAs walk)
    atomicAdd(work, (unsigned long long)base * (unsigned long long)min(kEvM, n - tile * kEvM));
  }
}

// Tiles in descending order of their row counts (ties: ascending tile):
// torder[rank] = tile.  The TILED values launch maps blockIdx.y = rank, so the
// longest tiles start first and the last wave of CTAs is made of the shortest
// ones (a launch is only ~1.4 waves long).
__global__ void __launch_bounds__(256)
pomdp_tile_order_kernel(int ntiles, const int* __restrict__ tcount, int* __restrict__ torder) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ntiles) return;
  const int ci = tcount[i];
  int rank = 0;
  for (int j = 0; j < ntiles; ++j) {
    const int cj = __ldg(tcount + j);
    rank += (cj > ci || (cj == ci && j < i)) ? 1 : 0;
  }
  torder[rank] = i;
}

// Grid: untiled (ceil(n / kEvM), column tiles); TILED (column tiles, ceil(n /
// kEvM)) with the belief tile = torder[blockIdx.y].
// Goals (DESIGN.md section 7e): every tile holds beliefs of one goal, and
// alpha is the goal-major stack [goals][rows][ld] with gstride floats per goal;
// the tile reads goal tile_goal[tile]'s matrix (tile_goal NULL: goal 0).
template <bool TILED>
__global__ void __launch_bounds__(256, 2)
pomdp_values_kernel(int HW, const int* __restrict__ kidx, int cells, int ld, int ncol,
                    const int* __restrict__ slots, int n,
                    const float* __restrict__ bel,
                    const float* __restrict__ alpha, float* __restrict__ out,
                    const int2* __restrict__ tlist, const int* __restrict__ tcount,
                    const int* __restrict__ torder, int tstride,
                    const int* __restrict__ tile_goal, size_t gstride) {
  const int mtile = TILED ? torder[blockIdx.y] : (int)blockIdx.x;
  const int ntile = TILED ? (int)blockIdx.x : (int)blockIdx.y;
  if (tile_goal) alpha += (size_t)tile_goal[mtile] * gstride;
  if constexpr (TILED) {
    // (HW is a by-value parameter: from here on it is this tile's row count)
    tlist += (size_t)mtile * tstride;
    HW = tcount[mtile];
  }
  __shared__ __align__(16) float sb[2][kEvK][kEvM + kEvPad];
  __shared__ __align__(16) float sa[2][kEvK][kEvN + kEvPad];
  __shared__ int sslot[kEvM];
  const int m0 = mtile * kEvM, n0 = ntile * kEvN;
  const int tid = threadIdx.x;
  if (tid < kEvM) sslot[tid] = (m0 + tid < n) ? slots[m0 + tid] : slots[0];
  __syncthreads();
  constexpr int kTM = kEvM / 8;                    // threads along the beliefs
  const int tx = tid % kTM, ty = tid / kTM;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;

  // Tile loaders (HW = the number K of inner-dimension rows of this launch).
  // Rows past it are clamped to the last row: they are never accumulated (the
  // k loop stops at HW), only kept in bounds.  Columns past ncol read the zero
  // padding of alpha (ld is a multiple of kEvN).
  // (tid + e * 256) % kEvM does not depend on e: every thread stages one belief
  static_assert(256 % kEvM == 0, "one belief column per thread");
  const float* bcol = bel + bel_off(cells, 0, sslot[tid % kEvM]);
  auto load_tiles = [&](int buf, int k0) {
#pragma unroll
    for (int e = 0; e < (kEvK * kEvM) / 256; ++e) {
      const int idx = tid + e * 256;
      const int kk = idx / kEvM, mm = idx % kEvM;
      const int s = TILED ? __ldg(tlist + min(k0 + kk, HW - 1)).x
                          : __ldg(kidx + min(k0 + kk, HW - 1));
      cp_async<4>((uint32_t)__cvta_generic_to_shared(&sb[buf][kk][mm]),
                  bcol + (size_t)s * kSlotBlock);
    }
#pragma unroll
    for (int e = 0; e < (kEvK * kEvN / 4) / 256; ++e) {
      const int idx = tid + e * 256;
      const int kk = idx / (kEvN / 4), nn = (idx % (kEvN / 4)) * 4;
      const int s = TILED ? __ldg(tlist + min(k0 + kk, HW - 1)).y : min(k0 + kk, HW - 1);
      cp_async<16>((uint32_t)__cvta_generic_to_shared(&sa[buf][kk][nn]),
                   alpha + (size_t)s * ld + n0 + nn);
    }
    cp_async_commit();
  };

  const int nchunks = (HW + kEvK - 1) / kEvK;
  if (nchunks > 0) load_tiles(0, 0);               // (a tile of all-zero beliefs has no rows)
  for (int c = 0; c < nchunks; ++c) {
    const int buf = c & 1;
    if (c + 1 < nchunks) {
      load_tiles(buf ^ 1, (c + 1) * kEvK);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const int kend = min(kEvK, HW - c * kEvK);
#pragma unroll 4
    for (int kk = 0; kk < kend; ++kk) {
      const float4 b0 = *reinterpret_cast<const float4*>(&sb[buf][kk][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&sb[buf][kk][kEvM / 2 + tx * 4]);
      const float4 a0 = *reinterpret_cast<const float4*>(&sa[buf][kk][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&sa[buf][kk][kEvN / 2 + ty * 4]);
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j)
          acc[i][j] = __fadd_rn(acc[i][j], __fmul_rn(bv[i], av[j]));
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int m = m0 + (i < 4 ? tx * 4 + i : kEvM / 2 + tx * 4 + (i - 4));
    if (m >= n) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = n0 + (j < 4 ? ty * 4 + j : kEvN / 2 + ty * 4 + (j - 4));
      if (col < ncol) out[(size_t)m * ncol + col] = acc[i][j];
    }
  }
}

// tree:168-173: reward[i][a] = inner_product(b_i, R(:,a), 0.0f) for the nodes
// being expanded: one WARP per (belief, 3 actions).  The lanes fetch and
// multiply 32 consecutive cells, then every lane replays the 32 rounded adds in
// order (the same sequential multiply-then-add chain as pomdp_values_kernel),
// three independent chains interleaved, the products broadcast through shared
// memory.  stage_reward is the reference table
// [HW][9].
// cells kidx[0..K) only (ascending): the belief is +0 on the others and
// acc + (+0 * r) == acc (see pomdp_dead_cells_kernel); lanes past the end hold
// +0 products for the same reason, so every chunk replays all 32 adds.
constexpr int kRewDepth = 4;     // chunks in flight
__device__ __forceinline__ void rewards_body(int K, const int* __restrict__ kidx,
                                             int lane, const float* __restrict__ col,
                                             const float* __restrict__ r3,
                                             float* __restrict__ out3,
                                             float* __restrict__ sw) {   // [3][32]
  float acc[3] = {0.0f, 0.0f, 0.0f};
  // (the cell index of a request is itself loaded one round of the ring
  // earlier: a dependent load inside the chunk loop stalls the in-order warp
  // for a full memory latency per chunk)
  float nb[kRewDepth], nr[kRewDepth][3];
  int sn[kRewDepth];
#pragma unroll
  for (int d = 0; d < kRewDepth; ++d) {
    const int cn = d * 32 + lane;
    const int s = cn < K ? __ldg(kidx + cn) : 0;
    nb[d] = cn < K ? col[(size_t)s * kSlotBlock] : 0.0f;
#pragma unroll
    for (int a = 0; a < 3; ++a) nr[d][a] = cn < K ? __ldg(r3 + (size_t)s * 9 + a) : 0.0f;
    const int c2 = cn + 32 * kRewDepth;
    sn[d] = c2 < K ? __ldg(kidx + c2) : 0;
  }
  for (int s0 = 0; s0 < K; s0 += 32 * kRewDepth) {
#pragma unroll
    for (int d = 0; d < kRewDepth; ++d) {
      const int c0 = s0 + d * 32;
      if (c0 >= K) break;                          // warp-uniform
      float p[3];
#pragma unroll
      for (int a = 0; a < 3; ++a) p[a] = __fmul_rn(nb[d], nr[d][a]);
      const int cn = c0 + 32 * kRewDepth + lane;
      const int s = sn[d];
      nb[d] = cn < K ? col[(size_t)s * kSlotBlock] : 0.0f;
#pragma unroll
      for (int a = 0; a < 3; ++a) nr[d][a] = cn < K ? __ldg(r3 + (size_t)s * 9 + a) : 0.0f;
      const int c2 = cn + 32 * kRewDepth;
      sn[d] = c2 < K ? __ldg(kidx + c2) : 0;
      // products to all lanes through shared memory (see prefix_body)
      __syncwarp();
#pragma unroll
      for (int a = 0; a < 3; ++a) sw[a * 32 + lane] = p[a];
      __syncwarp();
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4) {
        float4 t[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) t[a] = *reinterpret_cast<const float4*>(sw + a * 32 + 4 * j4);
#pragma unroll
        for (int a = 0; a < 3; ++a) acc[a] = __fadd_rn(acc[a], t[a].x);
#pragma unroll
        for (int a = 0; a < 3; ++a) acc[a] = __fadd_rn(acc[a], t[a].y);
#pragma unroll
        for (int a = 0; a < 3; ++a) acc[a] = __fadd_rn(acc[a], t[a].z);
#pragma unroll
        for (int a = 0; a < 3; ++a) acc[a] = __fadd_rn(acc[a], t[a].w);
      }
    }
  }
  if (lane < 3) out3[lane] = lane == 0 ? acc[0] : (lane == 1 ? acc[1] : acc[2]);
}

// Stage 1 of an expansion round in ONE launch: the prefix sums of the expanded
// nodes (blocks [0, ceil(n/4))) and their 9 reward dots (the blocks after
// them) do not depend on each other.  stage_reward is the goal-major stack
// [goals][HW][9]; node i reads goal goals[i]'s table.
__global__ void __launch_bounds__(128)
pomdp_expand_kernel(int HW, int K, const int* __restrict__ kidx,
                    const int* __restrict__ slots, const int* __restrict__ goals, int n,
                    const float* __restrict__ bel,
                    const float* __restrict__ stage_reward, float* __restrict__ prefix,
                    float* __restrict__ rewards) {
  __shared__ __align__(16) float sw[4][96];
  const int nbp = (n + 3) / 4;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if ((int)blockIdx.x < nbp) {
    const int i = blockIdx.x * 4 + warp;
    if (i >= n) return;
    prefix_body(HW, lane, bel + bel_off(HW, 0, slots[i]), prefix + (size_t)i * HW, sw[warp]);
  } else {
    const int w = (blockIdx.x - nbp) * 4 + warp;
    if (w >= n * 3) return;
    const int i = w / 3, a0 = (w % 3) * 3;
    rewards_body(K, kidx, lane, bel + bel_off(HW, 0, slots[i]),
                 stage_reward + (size_t)goals[i] * HW * 9 + a0, rewards + (size_t)i * 9 + a0,
                 sw[warp]);
  }
}

// Bounds of every evaluated belief from its row of values: first maximum over
// the FIB columns (upper, fib:294-296) and over the PBVI columns (lower,
// pbvi:696-698), as std::max_element does.  Packed per belief:
//   out[i*4 + 0] upper, [1] lower, [2] = fib index | pbvi index << 8 (as int
//   bits).
// max_element's rule `if (v[best] < v[a]) best = a` with NaN values: a NaN at
// index 0 is never replaced (NaN < x is false), so index 0 wins; otherwise a
// NaN is never taken (x < NaN is false) and the result is the first maximum
// of the other values.  +0 and -0 compare equal: the first of them wins.
__global__ void __launch_bounds__(128)
pomdp_bounds_kernel(int n, int ncol, int n_pbvi, const float* __restrict__ vals,
                    float* __restrict__ out) {
  // one warp per belief: lane-local first maximum over a strided subset of the
  // columns, then (value, index) reduction where ties keep the smaller index
  // -- the element std::max_element returns.  A NaN enters a lane's candidate
  // only at index 0, and a NaN candidate (index 0) beats every other one.
  const int i = blockIdx.x * 4 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= n) return;
  const float* v = vals + (size_t)i * ncol;
  float bu = 0.0f, bl = 0.0f;
  int iu = -1, il = -1;
  if (lane < 9) {
    bu = v[lane];
    if (lane == 0 || bu == bu) iu = lane;
  }
  for (int j = lane; j < n_pbvi; j += 32) {
    const float x = v[9 + j];
    if (il < 0 ? (j == 0 || x == x) : bl < x) { bl = x; il = j; }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const float ou = __shfl_xor_sync(0xffffffffu, bu, off);
    const int oiu = __shfl_xor_sync(0xffffffffu, iu, off);
    if (oiu >= 0 && (iu < 0 || bu < ou || (bu == ou && oiu < iu) || ou != ou)) {
      bu = ou; iu = oiu;
    }
    const float ol = __shfl_xor_sync(0xffffffffu, bl, off);
    const int oil = __shfl_xor_sync(0xffffffffu, il, off);
    if (oil >= 0 && (il < 0 || bl < ol || (bl == ol && oil < il) || ol != ol)) {
      bl = ol; il = oil;
    }
  }
  if (lane == 0) {
    float* o = out + (size_t)i * 4;
    o[0] = bu;
    o[1] = n_pbvi > 0 ? bl : 0.0f;
    o[2] = __int_as_float(iu | ((il < 0 ? 0 : il) << 8));
    o[3] = 0.0f;
  }
}

// ------------------------------------------------ FIB solver ("next" #1) ----
// fib:97-204 cudaFIBValueIteration: one sweep of the Fast Informed Bound
// backup on the 9 alpha vectors, alpha[s][a] layout.  One thread per
// (cell, action); same operation order as the reference kernel: per
// observation o, trans*meas (FMUL.FTZ), per next action an FFMA.FTZ chain over
// the 9 next states from 0, running max, FADD.FTZ into reward-to-go, and
// finally fma(gamma, reward_to_go, reward).
__global__ void __launch_bounds__(128)
pomdp_fib_kernel(int H, int W, float gamma, const float* __restrict__ trans_prob,
                 const float* __restrict__ meas_prob,
                 const float* __restrict__ stage_reward,
                 const float* __restrict__ prev, float* __restrict__ curr) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= H * W * 9) return;
  const int a = t % 9, cell = t / 9;
  const int x = cell % W, y = cell / W;
  float tp[9];
  int nidx[9];
#pragma unroll
  for (int sp = 0; sp < 9; ++sp) {
    const int nx = x + sp % 3 - 1, ny = y + sp / 3 - 1;
    nidx[sp] = (nx < 0 || nx >= W || ny < 0 || ny >= H) ? -1 : ny * W + nx;
    tp[sp] = __ldg(trans_prob + 81 * (size_t)cell + 9 * a + sp);
  }
  float rtg = 0.0f;
  for (int o = 0; o < 16; ++o) {
    float ltm[9];
#pragma unroll
    for (int sp = 0; sp < 9; ++sp)
      ltm[sp] = mul_ftz(tp[sp], nidx[sp] >= 0 ? __ldg(meas_prob + 16 * (size_t)nidx[sp] + o)
                                              : 0.0f);
    float best = -3.402823466e+38f;
    for (int ap = 0; ap < 9; ++ap) {
      float acc = 0.0f;
#pragma unroll
      for (int sp = 0; sp < 9; ++sp)
        acc = fma_ftz(ltm[sp], nidx[sp] >= 0 ? __ldg(prev + 9 * (size_t)nidx[sp] + ap) : 0.0f,
                      acc);
      if (best < acc) best = acc;
    }
    rtg = add_ftz(rtg, best);
  }
  curr[(size_t)cell * 9 + a] = fma_ftz(gamma, rtg, __ldg(stage_reward + (size_t)cell * 9 + a));
}

// max |a - b| over n floats (fib:245-251), atomicMax on the float bits.
__global__ void __launch_bounds__(256)
pomdp_maxdiff_kernel(const float* __restrict__ a, float* __restrict__ b_and_copy,
                     size_t n, unsigned int* result) {
  float m = 0.0f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (size_t)gridDim.x * blockDim.x) {
    const float v = a[i];
    m = fmaxf(m, fabsf(b_and_copy[i] - v));
    b_and_copy[i] = v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(result, __float_as_uint(m));
}

// Gather host-provided beliefs ([n][HW] row major) into belief columns.
__global__ void pomdp_scatter_kernel(int HW, const int* __restrict__ slots,
                                     int n, const float* __restrict__ rows,
                                     float* __restrict__ bel) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y;
  if (s >= HW || i >= n) return;
  bel[bel_off(HW, s, slots[i])] = rows[(size_t)i * HW + s];
}

// Belief columns back to [n][HW] rows.
__global__ void pomdp_gather_kernel(int HW, const int* __restrict__ slots,
                                    int n, const float* __restrict__ bel,
                                    float* __restrict__ rows) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y;
  if (s >= HW || i >= n) return;
  rows[(size_t)i * HW + s] = bel[bel_off(HW, s, slots[i])];
}

// Mode of each listed belief column as the sort key of the batched planners:
// column * H + row of the first maximum in cell order.  One warp per column.
__global__ void __launch_bounds__(128)
pomdp_root_mode_kernel(int H, int W, const int* __restrict__ slots, int n,
                       const float* __restrict__ bel, uint32_t* __restrict__ key) {
  const int i = blockIdx.x * 4 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= n) return;
  const int HW = H * W;
  const float* col = bel + bel_off(HW, 0, slots[i]);
  float bv = -INFINITY;
  int bi = INT_MAX;
  for (int s = lane; s < HW; s += 32) {
    const float v = col[(size_t)s * kSlotBlock];
    if (bi == INT_MAX || v > bv) { bv = v; bi = s; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  if (lane == 0) key[i] = (uint32_t)(bi % W) * (uint32_t)H + (uint32_t)(bi / W);
}

}  // namespace pp2d
