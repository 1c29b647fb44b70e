// sim.cu -- the dummy_simulator's histogram Bayes filter on the GPU
// (SURVEY.md section 8f row 4b): pp2d_sim_* of include/pp2d.h.
//
// Reference (a CPU loop in a peer ROS process):
//   /root/reference/dummy_simulator/src/dummy_simulator.cpp
//     440-522  transitionProbability   671-718  updateBelief(u)
//     720-773  updateBelief(meas)      162-195  controlCallback (u, then meas)
// The reference SCATTERS: for every source cell in row-major order it adds
// belief * P to its 9 targets.  A target cell therefore receives its (up to) 9
// contributions in ascending source order, which is DESCENDING slot order
// (slot 8 comes from the cell up-left, slot 0 from the cell down-right).  The
// kernel below gathers in exactly that order with separately rounded multiply
// and add (x86-64 host arithmetic, no FMA), so every cell gets the reference's
// bits.  Skipped sources (belief == 0) and zero probabilities contribute +-0,
// which leaves an accumulator that started at +0 unchanged.  The two sums are
// sequential float chains over the cells, replayed by one warp per belief.
// There is no CPU fallback.
#include "../../include/pp2d.h"

#include <cuda_runtime.h>

#include <cstring>
#include <new>
#include <vector>

#include "belief.cuh"
#include "handles.h"
#include "pomdp_host.h"

struct pp2d_sim {
  int H = 0, W = 0, HW = 0;
  uint8_t* d_map = nullptr;
  float *d_a = nullptr, *d_b = nullptr, *d_sum = nullptr;
  uint8_t* d_args = nullptr;
  std::vector<uint8_t> map_host;      // checks of the rollouts' starts
  size_t cap = 0;                     // beliefs the buffers hold
  cudaStream_t stream = nullptr;
};

namespace {
using namespace pp2d;

// updateBelief(u) without the normalisation: out[b][p] for every cell p.
__global__ void __launch_bounds__(256)
sim_predict_kernel(int H, int W, const uint8_t* __restrict__ map,
                   const uint8_t* __restrict__ actions, const float* __restrict__ in,
                   float* __restrict__ out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (p >= H * W) return;
  const int x = p % W, y = p / W;
  const int u = actions[b];
  const float* bel = in + (size_t)b * H * W;
  // P(p stays at p): the naive value plus the mass of every blocked slot, added
  // in ascending slot order (sim:503-519); out of the map counts as blocked.
  float stay = naive_prob(u, 4);
  bool occ_p = map[p] > 0;
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    if (i == 4) continue;
    const int px = x + i % 3 - 1, py = y + i / 3 - 1;
    const bool blocked = px < 0 || px >= W || py < 0 || py >= H || map[py * W + px] > 0;
    if (blocked) stay = __fadd_rn(stay, naive_prob(u, i));
  }
  float acc = 0.0f;
#pragma unroll
  for (int i = 8; i >= 0; --i) {
    // the source whose slot i is p
    const int sx = x - (i % 3 - 1), sy = y - (i / 3 - 1);
    if (sx < 0 || sx >= W || sy < 0 || sy >= H) continue;
    const float coef = (i == 4) ? stay : (occ_p ? 0.0f : naive_prob(u, i));
    acc = __fadd_rn(acc, __fmul_rn(bel[sy * W + sx], coef));
  }
  out[(size_t)b * H * W + p] = acc;
}

// updateBelief(meas) without the normalisation (sim:738-759).
__global__ void __launch_bounds__(256)
sim_correct_kernel(int H, int W, const uint8_t* __restrict__ map,
                   const uint8_t* __restrict__ meas, const float* __restrict__ in,
                   float* __restrict__ out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (p >= H * W) return;
  const int x = p % W, y = p / W;
  const int ox[4] = {0, -1, 1, 0}, oy[4] = {-1, 0, 0, 1};
  float l = 1.0f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int mx = x + ox[i], my = y + oy[i];
    const uint8_t m = (mx < 0 || mx >= W || my < 0 || my >= H) ? 1 : map[my * W + mx];
    l = __fmul_rn(l, m == meas[b * 4 + i] ? 0.98f : 0.02f);
  }
  const float v = in[(size_t)b * H * W + p];
  // belief == 0 -> 0 (sim:742-745); l * (+-0) would give the same +-0 except
  // for -0, which the reference replaces by +0
  out[(size_t)b * H * W + p] = (v == 0.0f) ? 0.0f : __fmul_rn(l, v);
}

// sum[b] = sequential float sum of the HW cells of belief b (sim:702-704,
// 757): one warp per belief, 32 loads in flight, the adds replayed in order.
__global__ void __launch_bounds__(128)
sim_sum_kernel(int HW, int n, const float* __restrict__ bel, float* __restrict__ sums) {
  const int b = blockIdx.x * 4 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= n) return;
  const float* col = bel + (size_t)b * HW;
  float acc = 0.0f;
  float nxt = lane < HW ? col[lane] : 0.0f;
  for (int s0 = 0; s0 < HW; s0 += 32) {
    const float v = nxt;
    const int sn = s0 + 32 + lane;
    nxt = sn < HW ? col[sn] : 0.0f;
    const int cnt = min(32, HW - s0);
    for (int j = 0; j < cnt; ++j) acc = __fadd_rn(acc, __shfl_sync(0xffffffffu, v, j));
  }
  if (lane == 0) sums[b] = acc;
}

__global__ void __launch_bounds__(256)
sim_scale_kernel(int HW, const float* __restrict__ sums, float* __restrict__ bel) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (p >= HW) return;
  const size_t q = (size_t)b * HW + p;
  bel[q] = __fdiv_rn(bel[q], sums[b]);
}

int ensure(pp2d_sim* s, size_t n) {
  if (n <= s->cap) return PP2D_OK;
  cudaFree(s->d_a); cudaFree(s->d_b); cudaFree(s->d_sum); cudaFree(s->d_args);
  s->d_a = s->d_b = s->d_sum = nullptr;
  s->d_args = nullptr;
  s->cap = 0;
  PP2D_CUDA(cudaMalloc(&s->d_a, n * s->HW * sizeof(float)));
  PP2D_CUDA(cudaMalloc(&s->d_b, n * s->HW * sizeof(float)));
  PP2D_CUDA(cudaMalloc(&s->d_sum, n * sizeof(float)));
  PP2D_CUDA(cudaMalloc(&s->d_args, n * 5));
  s->cap = n;
  return PP2D_OK;
}

// in d_a -> normalised result in d_b (predict) or d_a <- d_b ... see callers
int normalise(pp2d_sim* s, float* bel, uint32_t n) {
  sim_sum_kernel<<<(n + 3) / 4, 128, 0, s->stream>>>(s->HW, (int)n, bel, s->d_sum);
  count_launch();
  dim3 grid((s->HW + 255) / 256, n);
  sim_scale_kernel<<<grid, 256, 0, s->stream>>>(s->HW, s->d_sum, bel);
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  return PP2D_OK;
}

int run(pp2d_sim* s, float* beliefs, uint32_t n, const uint8_t* actions, const uint8_t* meas) {
  if (!s || !beliefs) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (n == 0) return PP2D_OK;
  if (actions)
    for (uint32_t i = 0; i < n; ++i)
      if (actions[i] >= 9) return fail(PP2D_ERR_INVALID, "belief %u: action %u out of range", i, actions[i]);
  PP2D_TRY(ensure(s, n));
  const size_t bytes = (size_t)n * s->HW * sizeof(float);
  PP2D_CUDA(cudaMemcpyAsync(s->d_a, beliefs, bytes, cudaMemcpyHostToDevice, s->stream));
  if (actions)
    PP2D_CUDA(cudaMemcpyAsync(s->d_args, actions, n, cudaMemcpyHostToDevice, s->stream));
  if (meas)
    PP2D_CUDA(cudaMemcpyAsync(s->d_args + n, meas, (size_t)n * 4, cudaMemcpyHostToDevice,
                              s->stream));
  dim3 grid((s->HW + 255) / 256, n);
  float* cur = s->d_a;
  float* other = s->d_b;
  if (actions) {
    sim_predict_kernel<<<grid, 256, 0, s->stream>>>(s->H, s->W, s->d_map, s->d_args, cur, other);
    count_launch();
    PP2D_TRY(normalise(s, other, n));
    float* t = cur; cur = other; other = t;
  }
  if (meas) {
    sim_correct_kernel<<<grid, 256, 0, s->stream>>>(s->H, s->W, s->d_map, s->d_args + n, cur,
                                                    other);
    count_launch();
    PP2D_TRY(normalise(s, other, n));
    float* t = cur; cur = other; other = t;
  }
  PP2D_CUDA(cudaGetLastError());
  PP2D_CUDA(cudaMemcpyAsync(beliefs, cur, bytes, cudaMemcpyDeviceToHost, s->stream));
  PP2D_CUDA(cudaStreamSynchronize(s->stream));
  return PP2D_OK;
}
}  // namespace

namespace pp2d {
SimView sim_view(const pp2d_sim* s) {
  SimView v;
  v.H = (uint32_t)s->H; v.W = (uint32_t)s->W;
  v.map_host = s->map_host.data();
  v.map = s->d_map;
  return v;
}
}  // namespace pp2d

extern "C" {

int pp2d_sim_create(uint32_t height, uint32_t width, const uint8_t* map, pp2d_sim** out) {
  if (!out) return fail(PP2D_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (!map || height == 0 || width == 0) return fail(PP2D_ERR_INVALID, "empty map");
  if ((uint64_t)height * width > (1u << 28)) return fail(PP2D_ERR_INVALID, "map too large");
  int dev_count = 0;
  PP2D_CUDA(cudaGetDeviceCount(&dev_count));
  if (dev_count == 0) return fail(PP2D_ERR_CUDA, "no CUDA device");
  int dev = 0;
  PP2D_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  PP2D_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10)
    return fail(PP2D_ERR_CUDA, "device %s is sm_%d%d; this library is sm_100a only", prop.name,
                prop.major, prop.minor);
  pp2d_sim* s = new (std::nothrow) pp2d_sim;
  if (!s) return fail(PP2D_ERR_INVALID, "out of host memory");
  s->H = (int)height; s->W = (int)width; s->HW = s->H * s->W;
  int rc = [&]() -> int {
    PP2D_CUDA(cudaMalloc(&s->d_map, (size_t)s->HW));
    PP2D_CUDA(cudaMemcpy(s->d_map, map, (size_t)s->HW, cudaMemcpyHostToDevice));
    s->map_host.assign(map, map + s->HW);
    return PP2D_OK;
  }();
  if (rc != PP2D_OK) { pp2d_sim_destroy(s); return rc; }
  *out = s;
  return PP2D_OK;
}

void pp2d_sim_destroy(pp2d_sim* s) {
  if (!s) return;
  cudaFree(s->d_map); cudaFree(s->d_a); cudaFree(s->d_b); cudaFree(s->d_sum);
  cudaFree(s->d_args);
  delete s;
}

int pp2d_sim_update_belief_action(pp2d_sim* s, float* beliefs, uint32_t n,
                                  const uint8_t* actions) {
  if (!actions) return fail(PP2D_ERR_INVALID, "NULL argument");
  return run(s, beliefs, n, actions, nullptr);
}

int pp2d_sim_update_belief_measurement(pp2d_sim* s, float* beliefs, uint32_t n,
                                       const uint8_t* measurements) {
  if (!measurements) return fail(PP2D_ERR_INVALID, "NULL argument");
  return run(s, beliefs, n, nullptr, measurements);
}

int pp2d_sim_step(pp2d_sim* s, float* beliefs, uint32_t n, const uint8_t* actions,
                  const uint8_t* measurements) {
  if (!actions || !measurements) return fail(PP2D_ERR_INVALID, "NULL argument");
  return run(s, beliefs, n, actions, measurements);
}

}  // extern "C"
