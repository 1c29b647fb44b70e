// pbvi.cu -- the offline Point-Based Value Iteration solver on the GPU
// (SURVEY.md section 8f "next" #2).  Replaces, for the reference's
// src/pomdp/point_based_value_iteration_cuda.cu:
//   generateBeliefSet   (165-293)  -> pp2d_pomdp_generate_belief_set
//   backupAlphaVectors  (344-641)  -> pp2d_pomdp_backup_alphas
//   pointBasedValueIteration (643-676) -> pp2d_pomdp_solve_pbvi
//
// The reference expands the belief set one belief and one action at a time
// (kernel launch + two 16 KB copies + an O(set * HW) host loop per candidate)
// and bounces 1.15 GB of Gamma_ao through host memory in every one of the 167
// backup iterations.  Here a whole expansion round (all beliefs x 9 actions)
// is a handful of launches on the belief pool, and the backup keeps
// everything in HBM.
//
// Arithmetic contract (what makes the results reproducible against the
// reference):
//   * host-side loops of the reference (partial_sum, accumulate, the L1
//     distance, inner_product) are sequential float chains without FMA: each
//     chain is evaluated in the same order with __fadd_rn / __fsub_rn /
//     __fmul_rn / __fdiv_rn;
//   * its device kernels are compiled with --use_fast_math: FFMA.FTZ chains,
//     reproduced with explicit PTX (fp_exact.cuh);
//   * rand() is glibc's TYPE_3 generator (GlibcRand), one global stream in the
//     reference's call order (belief-major, action-minor, three draws each);
//   * the one dense contraction, Gamma_ao^T * B (set x set x HW; cublasSgemm in
//     the reference, pbvi:505-513), is the hand-written pbvi_sgemm_tn_kernel
//     with a DEFINED summation order (one sequential FMA chain over the cells
//     per output).  Its result R only feeds an arg-max -- which Gamma_ao vector
//     each belief picks --; the alpha vectors are gathered from Gamma_ao, not
//     computed from R.  cuBLAS's blocking order is unspecified, so the
//     reference itself is only defined up to arg-max decisions between R
//     entries that agree to the last bits: against it the product path gives
//     identical alpha vectors wherever no such near-tie occurs, and otherwise
//     a lower-bound set of the same quality (tests/test_pbvi_gpu.py).  With
//     the order defined, the product path is bit-identical on ANY input to
//     the CPU oracle of this arithmetic (tests/pbvi_oracle.c,
//     tests/test_pbvi_kernel_gpu.py).  PP2D_PBVI_CUBLAS=1 switches to the
//     library call (bound at run time with dlopen) as a checker for tests: it
//     reproduces the reference's alpha vectors bit for bit on every fixture,
//     including the 500-belief bundled-map case.  Nothing else in the library
//     depends on cuBLAS.
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <vector>

#include <cublas_v2.h>
#include <dlfcn.h>

#include "async_copy.cuh"
#include "fp_exact.cuh"
#include "pomdp_host.h"

using namespace pp2d;

namespace {

// ---------------------------------------------------------------------------
// cuBLAS, bound at run time
struct Cublas {
  void* so = nullptr;
  decltype(&cublasCreate_v2) create = nullptr;
  decltype(&cublasDestroy_v2) destroy = nullptr;
  decltype(&cublasSetStream_v2) set_stream = nullptr;
  decltype(&cublasSgemm_v2) sgemm = nullptr;
  bool load() {
    if (so) return true;
    const char* names[] = {getenv("PP2D_CUBLAS"), "/usr/local/cuda/lib64/libcublas.so.12",
                           "libcublas.so.12", "libcublas.so"};
    for (const char* n : names) {
      if (!n || !*n) continue;
      so = dlopen(n, RTLD_NOW | RTLD_LOCAL);
      if (so) break;
    }
    if (!so) return false;
    create = (decltype(create))dlsym(so, "cublasCreate_v2");
    destroy = (decltype(destroy))dlsym(so, "cublasDestroy_v2");
    set_stream = (decltype(set_stream))dlsym(so, "cublasSetStream_v2");
    sgemm = (decltype(sgemm))dlsym(so, "cublasSgemm_v2");
    return create && destroy && set_stream && sgemm;
  }
};
Cublas g_cublas;

// ---------------------------------------------------------------------------
// belief-set expansion kernels (belief pool layout: bel_off of pomdp_kernels.cuh)

// pbvi:147-162 sampleFromProbDensity three times (pbvi:216-222): one thread
// per (belief i, action a).  prefix[i * HW + s] is partial_sum(b_i); draws are
// the host rand() values already divided by RAND_MAX+1.  find_if(x >= r) on a
// non-decreasing prefix = binary search for the first element >= r.  A draw
// beyond the last partial sum makes the reference index one past the array;
// here it is clamped to the last element.
__global__ void __launch_bounds__(128)
pbvi_sample_kernel(int H, int W, int n, const float* __restrict__ trans_prob,
                   const float* __restrict__ meas_prob, const float* __restrict__ prefix,
                   const float* __restrict__ draws, uint8_t* __restrict__ obs) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * 9) return;
  const int a = t % 9, i = t / 9;
  const int HW = H * W;
  const float r1 = draws[3 * t], r2 = draws[3 * t + 1], r3 = draws[3 * t + 2];
  int lo = 0, hi = HW;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (prefix[(size_t)i * HW + mid] >= r1) hi = mid; else lo = mid + 1;
  }
  const int s = lo < HW ? lo : HW - 1;
  float cum = 0.0f;
  int ns_local = 8;
  bool found = false;
  for (int j = 0; j < 9; ++j) {
    const float p = trans_prob[(size_t)s * 81 + a * 9 + j];
    cum = j == 0 ? p : __fadd_rn(cum, p);
    if (!found && cum >= r2) { ns_local = j; found = true; }
  }
  // pbvi:220: (s/width + ns_local/3 - 1)*width + (s%width + ns_local%3 - 1)
  long long ns = (long long)(s / W + ns_local / 3 - 1) * W + (s % W + ns_local % 3 - 1);
  if (ns < 0) ns = 0;
  if (ns >= HW) ns = HW - 1;
  int z = 15;
  found = false;
  cum = 0.0f;
  for (int j = 0; j < 16; ++j) {
    const float p = meas_prob[(size_t)ns * 16 + j];
    cum = j == 0 ? p : __fadd_rn(cum, p);
    if (!found && cum >= r3) { z = j; found = true; }
  }
  obs[t] = (uint8_t)z;
}

// pbvi:242-249: l1[c] = min_j sum_k |cand_c[k] - set_j[k]|, every sum a
// sequential float chain over k (subtract, abs, add -- no FMA).  CTA tile 64
// candidates x 64 set members, 4 x 4 chains per thread, 16 cells per stage.
// The minimum over j is exact in any order: atomicMin on the bits of the
// non-negative results (a NaN sum never replaces the minimum, as in `l1 <
// best`).
constexpr int kL1M = 64, kL1N = 64, kL1K = 16;
__global__ void __launch_bounds__(256)
pbvi_l1_kernel(int HW, const float* __restrict__ bel,
               const int* __restrict__ cand, int n_cand, const int* __restrict__ set,
               int n_set, unsigned int* __restrict__ l1_bits) {
  __shared__ __align__(16) float sa[kL1K][kL1M + 4];
  __shared__ __align__(16) float sb[kL1K][kL1N + 4];
  __shared__ int sca[kL1M], sse[kL1N];
  const int m0 = blockIdx.x * kL1M, n0 = blockIdx.y * kL1N;
  const int tid = threadIdx.x;
  if (tid < kL1M) sca[tid] = cand[min(m0 + tid, n_cand - 1)];
  else if (tid < kL1M + kL1N) sse[tid - kL1M] = set[min(n0 + tid - kL1M, n_set - 1)];
  __syncthreads();
  const int tm = (tid & 15) * 4, tn = (tid >> 4) * 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
  for (int k0 = 0; k0 < HW; k0 += kL1K) {
    for (int e = tid; e < kL1K * kL1M; e += 256) {
      const int kk = e / kL1M, mm = e % kL1M;
      const int s = min(k0 + kk, HW - 1);
      sa[kk][mm] = bel[bel_off(HW, s, sca[mm])];
      sb[kk][mm] = bel[bel_off(HW, s, sse[mm])];
    }
    __syncthreads();
    const int kend = min(kL1K, HW - k0);
    for (int kk = 0; kk < kend; ++kk) {
      const float4 a = *reinterpret_cast<const float4*>(&sa[kk][tm]);
      const float4 b = *reinterpret_cast<const float4*>(&sb[kk][tn]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
          acc[i][j] = __fadd_rn(acc[i][j], fabsf(__fsub_rn(av[i], bv[j])));
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + tm + i;
    if (m >= n_cand) continue;
    unsigned int best = 0xffffffffu;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (n0 + tn + j >= n_set) continue;
      const float v = acc[i][j];
      if (v == v) best = min(best, __float_as_uint(v));
    }
    if (best != 0xffffffffu) atomicMin(&l1_bits[m], best);
  }
}

__global__ void pbvi_fill_u32_kernel(unsigned int* p, int n, unsigned int v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// ---------------------------------------------------------------------------
// backup kernels (row-major [set][HW] layout, as the reference's device
// buffers, because that is what the GEMM consumes)

// pbvi:295-343 cudaComputeGammaOA for one action and ALL 16 observations:
//   G[o][i][s] = gamma * sum_k (T_a[s][k] * L[n_k][o]) * alpha_i[n_k]
// nvcc 12.9 / sm_100a compiles the reference kernel to: FMUL.FTZ for the
// T*L products, an FFMA.FTZ chain from +0 over the in-map neighbours in
// ascending k, FMUL.FTZ by gamma.  One thread per (cell, observation), a
// chunk of alpha vectors per blockIdx.z.
constexpr int kGammaChunk = 20;
__global__ void __launch_bounds__(128)
pbvi_gamma_ao_kernel(int H, int W, int n_set, float gamma, int a,
                     const float* __restrict__ trans_prob, const float* __restrict__ meas_prob,
                     const float* __restrict__ alphas, float* __restrict__ G) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  const int o = blockIdx.y;
  const int HW = H * W;
  if (s >= HW) return;
  const int x = s % W, y = s / W;
  float tm[9];
  int nidx[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    const int nx = x + k % 3 - 1, ny = y + k / 3 - 1;
    const bool in = !(nx < 0 || nx >= W || ny < 0 || ny >= H);
    nidx[k] = in ? ny * W + nx : -1;
    const float tp = __ldg(trans_prob + (size_t)s * 81 + a * 9 + k);
    tm[k] = in ? mul_ftz(tp, __ldg(meas_prob + (size_t)nidx[k] * 16 + o)) : tp;
  }
  const int i0 = blockIdx.z * kGammaChunk, i1 = min(n_set, i0 + kGammaChunk);
  for (int i = i0; i < i1; ++i) {
    const float* al = alphas + (size_t)i * HW;
    float acc = 0.0f;
#pragma unroll
    for (int k = 0; k < 9; ++k)
      if (nidx[k] >= 0) acc = fma_ftz(__ldg(al + nidx[k]), tm[k], acc);
    G[((size_t)o * n_set + i) * HW + s] = mul_ftz(acc, gamma);
  }
}

// pbvi:505-513: the one dense contraction of the reference, cublasSgemm(T, N):
//   R[o][b][i] = sum_s Gamma_ao[o][i][s] * B[b][s]        (n x n x HW, 16 of them)
// as a hand-written FP32 kernel.  R only feeds the arg-max over i below (which
// Gamma_ao vector a belief picks); the alpha vectors themselves are gathered
// from Gamma_ao and never see R.  Definition of the arithmetic (documented
// because it is NOT cuBLAS's unspecified blocking): every R[o][b][i] is ONE
// sequential FMA chain over the cells in ascending order, acc = fma(G, B, acc)
// from +0.  Cells on which every belief of the set is +0 (kidx lists the
// others) are skipped, which leaves the chain's value unchanged.
// Both operands are K-contiguous ("TN"); tiles are transposed on the way into
// shared memory with 4-byte cp.async (16 consecutive lanes = one 64-byte row
// segment).  CTA tile 128 x 128, 256 threads, 8 x 8 accumulators per thread,
// K chunks of 16 double-buffered.
constexpr int kGmM = 128, kGmN = 128, kGmK = 16, kGmPad = 4;

__global__ void __launch_bounds__(256, 2)
pbvi_sgemm_tn_kernel(int n, int HW, int K, const int* __restrict__ kidx,
                     const float* __restrict__ G, const float* __restrict__ B,
                     float* __restrict__ R) {
  __shared__ __align__(16) float sg[2][kGmK][kGmM + kGmPad];
  __shared__ __align__(16) float sb[2][kGmK][kGmN + kGmPad];
  const int o = blockIdx.z;
  const int i0 = blockIdx.x * kGmM, b0 = blockIdx.y * kGmN;
  const float* Go = G + (size_t)o * n * HW;
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;

  auto load_tiles = [&](int buf, int k0) {
#pragma unroll
    for (int e = 0; e < (kGmK * kGmM) / 256; ++e) {
      const int idx = tid + e * 256;
      const int kk = idx % kGmK, row = idx / kGmK;
      const int s = __ldg(kidx + min(k0 + kk, K - 1));     // clamped rows are never accumulated
      cp_async<4>((uint32_t)__cvta_generic_to_shared(&sg[buf][kk][row]),
                  Go + (size_t)min(i0 + row, n - 1) * HW + s);
      cp_async<4>((uint32_t)__cvta_generic_to_shared(&sb[buf][kk][row]),
                  B + (size_t)min(b0 + row, n - 1) * HW + s);
    }
    cp_async_commit();
  };

  const int nchunks = (K + kGmK - 1) / kGmK;
  load_tiles(0, 0);
  for (int c = 0; c < nchunks; ++c) {
    const int buf = c & 1;
    if (c + 1 < nchunks) {
      load_tiles(buf ^ 1, (c + 1) * kGmK);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const int kend = min(kGmK, K - c * kGmK);
#pragma unroll 4
    for (int kk = 0; kk < kend; ++kk) {
      const float4 g0 = *reinterpret_cast<const float4*>(&sg[buf][kk][tx * 4]);
      const float4 g1 = *reinterpret_cast<const float4*>(&sg[buf][kk][64 + tx * 4]);
      const float4 q0 = *reinterpret_cast<const float4*>(&sb[buf][kk][ty * 4]);
      const float4 q1 = *reinterpret_cast<const float4*>(&sb[buf][kk][64 + ty * 4]);
      const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
      const float bv[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = __fmaf_rn(gv[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  float* Ro = R + (size_t)o * n * n;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int b = b0 + (j < 4 ? ty * 4 + j : 64 + ty * 4 + (j - 4));
    if (b >= n) continue;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int a = i0 + (i < 4 ? tx * 4 + i : 64 + tx * 4 + (i - 4));
      if (a < n) Ro[(size_t)b * n + a] = acc[i][j];
    }
  }
}

// pbvi:531-537: for every belief i the FIRST maximum of row i of
// alphas_ao_reward (max_element).  R is [16][n][n]; one warp per row.
__global__ void __launch_bounds__(128)
pbvi_argmax_kernel(int n, int rows, const float* __restrict__ R, int* __restrict__ idx) {
  const int row = blockIdx.x * 4 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* r = R + (size_t)row * n;
  float best = 0.0f;
  int bj = -1;
  for (int j = lane; j < n; j += 32) {
    const float v = r[j];
    if (bj < 0 || best < v) { best = v; bj = j; }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, off);
    const int oj = __shfl_xor_sync(0xffffffffu, bj, off);
    if (oj >= 0 && (bj < 0 || best < ov || (best == ov && oj < bj))) { best = ov; bj = oj; }
  }
  if (lane == 0) idx[row] = bj < 0 ? 0 : bj;
}

// pbvi:476-482 + 539-558: Gamma_a[i] = R(:,a), then for o = 0..15 in order
// Gamma_a[i] += Gamma_ao[o][argmax_{o,i}] (cublasSgeam with alpha = beta = 1:
// a float add per element).
__global__ void __launch_bounds__(256)
pbvi_accumulate_kernel(int HW, int n_set, int a, const float* __restrict__ stage_reward,
                       const float* __restrict__ G, const int* __restrict__ idx,
                       float* __restrict__ GA) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y;
  if (s >= HW) return;
  float acc = __ldg(stage_reward + (size_t)s * 9 + a);
#pragma unroll 4
  for (int o = 0; o < 16; ++o) {
    const int j = idx[o * n_set + i];
    acc = __fadd_rn(G[((size_t)o * n_set + j) * HW + s], acc);
  }
  GA[((size_t)a * n_set + i) * HW + s] = acc;
}

// pbvi:595-596: inner_product(b_i, Gamma_a[a][i], 0.0f): a sequential chain of
// rounded multiply + rounded add.  One warp per (i, a): the lanes fetch and
// multiply 32 consecutive cells, then every lane replays the 32 adds in order
// from registers, so that the chain never waits for memory.
__global__ void __launch_bounds__(128)
pbvi_rewards_kernel(int HW, int n_set, const float* __restrict__ B,
                    const float* __restrict__ GA, float* __restrict__ rewards) {
  const int w = blockIdx.x * 4 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (w >= n_set * 9) return;
  const int a = w % 9, i = w / 9;
  const float* b = B + (size_t)i * HW;
  const float* g = GA + ((size_t)a * n_set + i) * HW;
  float acc = 0.0f;
  for (int s0 = 0; s0 < HW; s0 += 32) {
    const int s = s0 + lane;
    const float p = s < HW ? __fmul_rn(b[s], g[s]) : 0.0f;
    const int cnt = min(32, HW - s0);
    for (int j = 0; j < cnt; ++j)
      acc = __fadd_rn(acc, __shfl_sync(0xffffffffu, p, j));
  }
  if (lane == 0) rewards[i * 9 + a] = acc;
}

// pbvi:589-606: first action whose reward is > all earlier ones (from
// -FLT_MAX), alphas[i] = Gamma_a[action][i].  One block per belief.
__global__ void __launch_bounds__(256)
pbvi_select_kernel(int HW, int n_set, const float* __restrict__ rewards,
                   const float* __restrict__ GA, float* __restrict__ alphas,
                   uint8_t* __restrict__ actions) {
  const int i = blockIdx.x;
  float opt = -FLT_MAX;
  int oa = 0;
#pragma unroll
  for (int a = 0; a < 9; ++a) {
    const float r = rewards[i * 9 + a];
    if (r > opt) { opt = r; oa = a; }
  }
  const float* src = GA + ((size_t)oa * n_set + i) * HW;
  float* dst = alphas + (size_t)i * HW;
  for (int s = threadIdx.x; s < HW; s += blockDim.x) dst[s] = src[s];
  if (threadIdx.x == 0) actions[i] = (uint8_t)oa;
}

// ---------------------------------------------------------------------------
// generateBeliefSet (pbvi:165-293) on the belief pool; returns the pool slots
// of the set members in set order.
int expand_belief_set(pp2d_pomdp* h, const float* b0, uint32_t max_size, uint32_t rand_seed,
                      std::vector<int>& set) {
  const int HW = h->HW;
  GlibcRand rng;
  rng.seed(rand_seed ? rand_seed : 1);
  set.clear();
  PP2D_TRY(pool_reserve(h, (size_t)h->cap - h->free_slots.count() + 10 * (size_t)max_size + 32));
  int s0 = -1;
  PP2D_TRY(alloc_slot(h, &s0));
  set.push_back(s0);
  PP2D_TRY(launch_scatter(h, set, b0));
  DevBuf<float> d_draws;
  DevBuf<uint8_t> d_obs;
  DevBuf<int> d_cand, d_set;
  DevBuf<unsigned int> d_l1;
  int rc = [&]() -> int {
    while (set.size() < max_size) {
      const int n = (int)set.size();
      const int nc = n * 9;
      std::vector<float> draws((size_t)nc * 3);
      for (float& d : draws) d = (float)rng.next() / ((float)2147483647 + 1.0f);
      PP2D_TRY(d_draws.ensure(draws.size()));
      PP2D_TRY(d_obs.ensure(nc));
      PP2D_CUDA(cudaMemcpyAsync(d_draws.p, draws.data(), draws.size() * sizeof(float),
                                cudaMemcpyHostToDevice, h->stream));
      PP2D_TRY(launch_prefix(h, set));
      pbvi_sample_kernel<<<(nc + 127) / 128, 128, 0, h->stream>>>(
          h->H, h->W, n, h->d_tp, h->d_mp, h->d_prefix.p, d_draws.p, d_obs.p);
      count_launch();
      PP2D_CUDA(cudaGetLastError());
      std::vector<uint8_t> obs(nc);
      PP2D_CUDA(cudaMemcpyAsync(obs.data(), d_obs.p, nc, cudaMemcpyDeviceToHost, h->stream));
      PP2D_CUDA(cudaStreamSynchronize(h->stream));
      std::vector<int> cand(nc);
      std::vector<BayesItem> items(nc);
      for (int i = 0; i < n; ++i)
        for (int a = 0; a < 9; ++a) {
          PP2D_TRY(alloc_slot(h, &cand[i * 9 + a]));
          items[i * 9 + a] = BayesItem{set[i], cand[i * 9 + a], (uint8_t)a, obs[i * 9 + a]};
        }
      PP2D_TRY(launch_bayes(h, items));          // pbvi:227-232
      PP2D_TRY(launch_normalize(h, cand));       // pbvi:235-237
      PP2D_TRY(d_cand.ensure(nc));
      PP2D_TRY(d_set.ensure(n));
      PP2D_TRY(d_l1.ensure(nc));
      PP2D_CUDA(cudaMemcpyAsync(d_cand.p, cand.data(), nc * sizeof(int),
                                cudaMemcpyHostToDevice, h->stream));
      PP2D_CUDA(cudaMemcpyAsync(d_set.p, set.data(), n * sizeof(int), cudaMemcpyHostToDevice,
                                h->stream));
      pbvi_fill_u32_kernel<<<(nc + 255) / 256, 256, 0, h->stream>>>(
          d_l1.p, nc, 0x7f7fffffu /* FLT_MAX */);
      count_launch();
      dim3 grid((nc + kL1M - 1) / kL1M, (n + kL1N - 1) / kL1N);
      pbvi_l1_kernel<<<grid, 256, 0, h->stream>>>(HW, h->d_bel, d_cand.p, nc, d_set.p,
                                                  n, d_l1.p);
      count_launch();
      PP2D_CUDA(cudaGetLastError());
      std::vector<float> l1(nc);
      PP2D_CUDA(cudaMemcpyAsync(l1.data(), d_l1.p, nc * sizeof(float), cudaMemcpyDeviceToHost,
                                h->stream));
      PP2D_CUDA(cudaStreamSynchronize(h->stream));
      // pbvi:252-258: per belief the action whose new belief is farthest
      std::vector<int> new_bs(n);
      std::vector<float> new_bs_l1(n);
      std::vector<char> keep(nc, 0);
      for (int i = 0; i < n; ++i) {
        const float* r = l1.data() + (size_t)i * 9;
        const int best = (int)(std::max_element(r, r + 9) - r);
        new_bs[i] = cand[i * 9 + best];
        new_bs_l1[i] = r[best];
      }
      // pbvi:261-285
      std::vector<int> order;
      if (n < 100) {
        for (int i = 0; i < n; ++i) order.push_back(i);
      } else {
        std::vector<size_t> sorted_idx(n);
        std::iota(sorted_idx.begin(), sorted_idx.end(), 0);
        // NB the reference passes (begin, END, begin+100) -- middle and last
        // swapped (pbvi:272-276).  With libstdc++ that is make_heap +
        // sort_heap over the WHOLE range, i.e. a full heap sort; the same
        // two calls are made here so that ties come out in the same order.
        auto farther = [&new_bs_l1](const size_t& i, const size_t& j) {
          return new_bs_l1[i] > new_bs_l1[j];
        };
        std::make_heap(sorted_idx.begin(), sorted_idx.end(), farther);
        std::sort_heap(sorted_idx.begin(), sorted_idx.end(), farther);
        for (int i = 0; i < 100; ++i) order.push_back((int)sorted_idx[i]);
      }
      for (int i : order) {
        set.push_back(new_bs[i]);
        for (int a = 0; a < 9; ++a)
          if (cand[i * 9 + a] == new_bs[i]) keep[i * 9 + a] = 1;
        if (set.size() >= max_size) break;
      }
      for (int c = 0; c < nc; ++c)
        if (!keep[c]) h->free_slots.put(cand[c]);
    }
    return PP2D_OK;
  }();
  d_draws.release(); d_obs.release(); d_cand.release(); d_set.release(); d_l1.release();
  return rc;
}

// max_backup_iterations of pbvi:427-431 (float arithmetic, as written there).
// Defined only for 0 < gamma < 1: gamma = 1 gives -inf, gamma > 1 a negative
// count and gamma <= 0 or NaN a NaN, none of which converts to uint32_t.
bool reference_iterations_defined(float gamma) { return gamma > 0.0f && gamma < 1.0f; }
uint32_t reference_backup_iterations(float gamma) {
  return (uint32_t)ceilf(logf(1.0e-3f / 5.0f) / logf(gamma));
}

// backupAlphaVectors (pbvi:344-641) on device buffers: d_B [n][HW] beliefs,
// d_alphas [n][HW] (in: start vectors, out: result), d_actions [n].
int backup_on_device(pp2d_pomdp* h, int n, const float* d_B, float* d_alphas,
                     uint8_t* d_actions, uint32_t iterations,
                     bool beliefs_zero_on_dead_cells) {
  // PP2D_PBVI_CUBLAS=1 (tests only): the reference's library call instead of
  // pbvi_sgemm_tn_kernel, to show that both pick the same Gamma_ao vectors.
  const char* cb_env = getenv("PP2D_PBVI_CUBLAS");
  const bool use_cublas = cb_env && atoi(cb_env) != 0;
  if (use_cublas && !g_cublas.load())
    return fail(PP2D_ERR_STATE, "cuBLAS (libcublas.so.12) could not be loaded: %s", dlerror());
  const int HW = h->HW;
  // cells on which some belief of the set may be non-zero (the set grows from a
  // belief by Bayes updates, so normally the live cells)
  const bool dense = !h->skip_dead || !beliefs_zero_on_dead_cells;
  const int* kidx = dense ? h->d_kidx_all : h->d_kidx;
  const int K = dense ? HW : h->K;
  float *G = nullptr, *GA = nullptr, *R = nullptr, *rew = nullptr;
  int* idx = nullptr;
  cublasHandle_t cb = nullptr;
  int rc = [&]() -> int {
    PP2D_CUDA(cudaMalloc(&G, (size_t)16 * n * HW * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&GA, (size_t)9 * n * HW * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&R, (size_t)16 * n * n * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&rew, (size_t)9 * n * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&idx, (size_t)16 * n * sizeof(int)));
    if (use_cublas) {
      if (g_cublas.create(&cb) != CUBLAS_STATUS_SUCCESS)
        return fail(PP2D_ERR_CUDA, "cublasCreate failed");
      if (g_cublas.set_stream(cb, h->stream) != CUBLAS_STATUS_SUCCESS)
        return fail(PP2D_ERR_CUDA, "cublasSetStream failed");
    }
    const float one = 1.0f, zero = 0.0f;
    for (uint32_t it = 0; it < iterations; ++it) {
      for (int a = 0; a < 9; ++a) {
        dim3 ggrid((HW + 127) / 128, 16, (n + kGammaChunk - 1) / kGammaChunk);
        pbvi_gamma_ao_kernel<<<ggrid, 128, 0, h->stream>>>(h->H, h->W, n, h->gamma, a, h->d_tp,
                                                           h->d_mp, d_alphas, G);
        count_launch();
        if (use_cublas) {
          for (int o = 0; o < 16; ++o) {
            // pbvi:505-513, same call: C(n x n, col-major) = Gamma_ao^T * B
            if (g_cublas.sgemm(cb, CUBLAS_OP_T, CUBLAS_OP_N, n, n, HW, &one,
                               G + (size_t)o * n * HW, HW, d_B, HW, &zero,
                               R + (size_t)o * n * n, n) != CUBLAS_STATUS_SUCCESS)
              return fail(PP2D_ERR_CUDA, "cublasSgemm failed");
          }
        } else {
          dim3 mgrid((n + kGmM - 1) / kGmM, (n + kGmN - 1) / kGmN, 16);
          pbvi_sgemm_tn_kernel<<<mgrid, 256, 0, h->stream>>>(n, HW, K, kidx, G, d_B, R);
          count_launch();
        }
        pbvi_argmax_kernel<<<(16 * n + 3) / 4, 128, 0, h->stream>>>(n, 16 * n, R, idx);
        count_launch();
        dim3 agrid((HW + 255) / 256, n);
        pbvi_accumulate_kernel<<<agrid, 256, 0, h->stream>>>(HW, n, a, h->d_sr, G, idx, GA);
        count_launch();
      }
      pbvi_rewards_kernel<<<(9 * n + 3) / 4, 128, 0, h->stream>>>(HW, n, d_B, GA, rew);
      count_launch();
      pbvi_select_kernel<<<n, 256, 0, h->stream>>>(HW, n, rew, GA, d_alphas, d_actions);
      count_launch();
      PP2D_CUDA(cudaGetLastError());
    }
    PP2D_CUDA(cudaStreamSynchronize(h->stream));
    return PP2D_OK;
  }();
  if (cb) g_cublas.destroy(cb);
  cudaFree(G); cudaFree(GA); cudaFree(R); cudaFree(rew); cudaFree(idx);
  return rc;
}

}  // namespace

extern "C" {

int pp2d_pomdp_generate_belief_set(pp2d_pomdp* h, const float* initial_belief, uint32_t n,
                                   uint32_t rand_seed, float* belief_set) {
  if (!h || !initial_belief || !belief_set || n == 0)
    return fail(PP2D_ERR_INVALID, "NULL argument or empty set");
  std::vector<int> set;
  float* d_rows = nullptr;
  int rc = [&]() -> int {
    PP2D_TRY(expand_belief_set(h, initial_belief, n, rand_seed, set));
    PP2D_CUDA(cudaMalloc(&d_rows, (size_t)n * h->HW * sizeof(float)));
    PP2D_TRY(launch_gather(h, set, d_rows));
    PP2D_CUDA(cudaMemcpyAsync(belief_set, d_rows, (size_t)n * h->HW * sizeof(float),
                              cudaMemcpyDeviceToHost, h->stream));
    PP2D_CUDA(cudaStreamSynchronize(h->stream));
    return PP2D_OK;
  }();
  cudaFree(d_rows);
  for (int s : set) h->free_slots.put(s);
  return rc;
}

int pp2d_pomdp_backup_alphas(pp2d_pomdp* h, const float* belief_set, uint32_t n,
                             uint32_t iterations, float* alphas, uint8_t* actions) {
  if (!h || !belief_set || !alphas || n == 0)
    return fail(PP2D_ERR_INVALID, "NULL argument or empty set");
  if (iterations == 0) {
    if (!reference_iterations_defined(h->gamma))
      return fail(PP2D_ERR_INVALID, "iterations = 0 takes the reference's count, which needs "
                  "0 < gamma < 1 (gamma = %g); pass a count", (double)h->gamma);
    iterations = reference_backup_iterations(h->gamma);
  }
  const size_t bytes = (size_t)n * h->HW * sizeof(float);
  float *d_B = nullptr, *d_al = nullptr;
  uint8_t* d_ac = nullptr;
  int rc = [&]() -> int {
    PP2D_CUDA(cudaMalloc(&d_B, bytes));
    PP2D_CUDA(cudaMalloc(&d_al, bytes));
    PP2D_CUDA(cudaMalloc(&d_ac, n));
    PP2D_CUDA(cudaMemcpyAsync(d_B, belief_set, bytes, cudaMemcpyHostToDevice, h->stream));
    PP2D_CUDA(cudaMemsetAsync(d_al, 0, bytes, h->stream));     // pbvi:658-659
    PP2D_CUDA(cudaMemsetAsync(d_ac, 0, n, h->stream));
    bool zero = true;
    for (uint32_t i = 0; i < n && zero; ++i)
      zero = zero_on_dead_cells(h, belief_set + (size_t)i * h->HW);
    PP2D_TRY(backup_on_device(h, (int)n, d_B, d_al, d_ac, iterations, zero));
    PP2D_CUDA(cudaMemcpyAsync(alphas, d_al, bytes, cudaMemcpyDeviceToHost, h->stream));
    if (actions)
      PP2D_CUDA(cudaMemcpyAsync(actions, d_ac, n, cudaMemcpyDeviceToHost, h->stream));
    PP2D_CUDA(cudaStreamSynchronize(h->stream));
    return PP2D_OK;
  }();
  cudaFree(d_B); cudaFree(d_al); cudaFree(d_ac);
  return rc;
}

int pp2d_pomdp_solve_pbvi(pp2d_pomdp* h, const float* initial_belief, uint32_t n,
                          uint32_t rand_seed, uint32_t iterations, float* belief_set,
                          float* alphas, uint8_t* actions) {
  if (!h || !initial_belief || !alphas || n == 0)
    return fail(PP2D_ERR_INVALID, "NULL argument or empty set");
  if (iterations == 0) {
    if (!reference_iterations_defined(h->gamma))
      return fail(PP2D_ERR_INVALID, "iterations = 0 takes the reference's count, which needs "
                  "0 < gamma < 1 (gamma = %g); pass a count", (double)h->gamma);
    iterations = reference_backup_iterations(h->gamma);
  }
  const size_t bytes = (size_t)n * h->HW * sizeof(float);
  std::vector<int> set;
  float *d_B = nullptr, *d_al = nullptr;
  uint8_t* d_ac = nullptr;
  int rc = [&]() -> int {
    PP2D_TRY(expand_belief_set(h, initial_belief, n, rand_seed, set));
    PP2D_CUDA(cudaMalloc(&d_B, bytes));
    PP2D_CUDA(cudaMalloc(&d_al, bytes));
    PP2D_CUDA(cudaMalloc(&d_ac, n));
    PP2D_TRY(launch_gather(h, set, d_B));
    PP2D_CUDA(cudaMemsetAsync(d_al, 0, bytes, h->stream));
    PP2D_CUDA(cudaMemsetAsync(d_ac, 0, n, h->stream));
    // every belief of the set descends from initial_belief by Bayes updates
    PP2D_TRY(backup_on_device(h, (int)n, d_B, d_al, d_ac, iterations,
                              zero_on_dead_cells(h, initial_belief)));
    if (belief_set)
      PP2D_CUDA(cudaMemcpyAsync(belief_set, d_B, bytes, cudaMemcpyDeviceToHost, h->stream));
    PP2D_CUDA(cudaMemcpyAsync(alphas, d_al, bytes, cudaMemcpyDeviceToHost, h->stream));
    if (actions)
      PP2D_CUDA(cudaMemcpyAsync(actions, d_ac, n, cudaMemcpyDeviceToHost, h->stream));
    PP2D_CUDA(cudaStreamSynchronize(h->stream));
    return PP2D_OK;
  }();
  cudaFree(d_B); cudaFree(d_al); cudaFree(d_ac);
  for (int s : set) h->free_slots.put(s);
  return rc;
}

}  // extern "C"
