// rollout.cu -- closed-loop episodes of an MDP planner (pp2d_sim_rollout_mdp*)
// or of the QV-tree planner (pp2d_sim_rollout_pomdp) in the simulator
// (include/pp2d.h; contract in DESIGN.md sections 7c and 7d).
//
// MDP rollouts: one CTA runs one episode from its start to its stop, so an
// episode that has stopped costs nothing more (its CTA has exited and the next
// one takes the SM slot).  The belief and the prediction plane live in shared memory while
// both fit (2 * HW floats; 32 KB on the reference's 100x40 map); larger maps
// run the same code on two planes per episode in global memory.  Each step:
// belief_mode (the plan kernels' scan) -> action; thread 0 draws the motion
// and the four sensor flips from Philox; then the filter of sim.cu with the
// same bits: gather prediction (contributions in descending slot order, every
// product and sum rounded alone), one sequential sum, scale fused with the
// correction (__fdiv_rn then __fmul_rn, what two passes give), a second
// sequential sum and the final scale.  The two sums are chains of HW adds in
// cell order; one thread replays each from float4 loads, and they bound the
// step time.
#include "../../include/pp2d.h"

#include <cuda_runtime.h>

#include <cstring>
#include <vector>

#include "belief.cuh"
#include "handles.h"
#include "philox.h"
#include "pomdp_host.h"

namespace {
using namespace pp2d;

constexpr int kThreads = 256;   // belief_mode's CTA shape

struct Episode {              // one upload for all episodes
  const uint8_t* action;      // the planner's action grid [H][W]
  uint32_t start, goal;       // cells y*W+x
};

struct RolloutParams {
  int H, W, HW, plane;        // plane: HW rounded up to 4 floats
  const uint8_t* map;         // the simulator's (world) map
  const Episode* ep;
  const float* belief0;       // [n][HW] or nullptr: point mass at the start
  float* planes;              // [n][2][plane] in global memory, or nullptr
  uint32_t max_steps;
  uint64_t seed, first;
  uint32_t *steps, *collisions, *final_cell, *cells;
  uint8_t *reached, *actions, *meas;
  float* final_belief;
};

__device__ __forceinline__ bool blocked(const RolloutParams& p, int x, int y) {
  return x < 0 || x >= p.W || y < 0 || y >= p.H || p.map[y * p.W + x] > 0;
}

// Sequential float sum of v[0 .. n) from +0 in index order (v 16-byte aligned).
__device__ __forceinline__ float chain_sum(const float* v, int n) {
  float acc = 0.0f;
  int i = 0;
  for (; i + 4 <= n; i += 4) {
    const float4 q = *reinterpret_cast<const float4*>(v + i);
    acc = __fadd_rn(acc, q.x);
    acc = __fadd_rn(acc, q.y);
    acc = __fadd_rn(acc, q.z);
    acc = __fadd_rn(acc, q.w);
  }
  for (; i < n; ++i) acc = __fadd_rn(acc, v[i]);
  return acc;
}

template <bool kShared>
__global__ void __launch_bounds__(kThreads)
sim_rollout_kernel(const RolloutParams p) {
  extern __shared__ float4 smem4[];
  __shared__ uint32_t s_cell, s_act, s_meas, s_coll;
  __shared__ float s_sum;
  const uint32_t i = blockIdx.x;
  const int HW = p.HW;
  float* bel = kShared ? reinterpret_cast<float*>(smem4) : p.planes + (size_t)i * 2 * p.plane;
  float* pred = bel + p.plane;
  const Episode ep = p.ep[i];
  const uint64_t e = p.first + i;
  for (int q = threadIdx.x; q < HW; q += kThreads)
    bel[q] = p.belief0 ? p.belief0[(size_t)i * HW + q] : (q == (int)ep.start ? 1.0f : 0.0f);
  if (threadIdx.x == 0) {
    s_cell = ep.start;
    s_coll = 0;
    if (p.cells) p.cells[(size_t)i * ((size_t)p.max_steps + 1)] = ep.start;
  }
  __syncthreads();
  uint32_t t = 0;
  for (;; ++t) {
    const uint32_t cell = s_cell;
    if (cell == ep.goal || t == p.max_steps) break;
    // plan: the action at the belief mode
    const unsigned long long mode = belief_mode(bel, (size_t)HW);
    if (threadIdx.x == 0) {
      const int u = ep.action[mode];
      const WorldStep w = world_step(p.H, p.W, p.map, cell, u, p.seed, e, t);
      if (w.collided) ++s_coll;
      s_cell = w.cell; s_act = (uint32_t)u; s_meas = w.meas;
      if (p.cells) p.cells[(size_t)i * ((size_t)p.max_steps + 1) + t + 1] = w.cell;
      if (p.actions) p.actions[(size_t)i * p.max_steps + t] = (uint8_t)u;
      if (p.meas) p.meas[(size_t)i * p.max_steps + t] = (uint8_t)w.meas;
    }
    __syncthreads();
    const int u = (int)s_act;
    const uint32_t m = s_meas;
    // prediction (sim_predict_kernel): gather in descending slot order
    for (int q = threadIdx.x; q < HW; q += kThreads) {
      const int x = q % p.W, y = q / p.W;
      float stay = naive_prob(u, 4);
#pragma unroll
      for (int k = 0; k < 9; ++k) {
        if (k == 4) continue;
        if (blocked(p, x + k % 3 - 1, y + k / 3 - 1)) stay = __fadd_rn(stay, naive_prob(u, k));
      }
      const bool occ_q = p.map[q] > 0;
      float acc = 0.0f;
#pragma unroll
      for (int k = 8; k >= 0; --k) {
        const int sx = x - (k % 3 - 1), sy = y - (k / 3 - 1);
        if (sx < 0 || sx >= p.W || sy < 0 || sy >= p.H) continue;
        const float coef = (k == 4) ? stay : (occ_q ? 0.0f : naive_prob(u, k));
        acc = __fadd_rn(acc, __fmul_rn(bel[sy * p.W + sx], coef));
      }
      pred[q] = acc;
    }
    __syncthreads();
    if (threadIdx.x == 0) s_sum = chain_sum(pred, HW);
    __syncthreads();
    // normalisation fused with the correction (sim_correct_kernel)
    const float s1 = s_sum;
    for (int q = threadIdx.x; q < HW; q += kThreads) {
      const int x = q % p.W, y = q / p.W;
      const int ox[4] = {0, -1, 1, 0}, oy[4] = {-1, 0, 0, 1};
      float l = 1.0f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int mx = x + ox[j], my = y + oy[j];
        const uint32_t mv = (mx < 0 || mx >= p.W || my < 0 || my >= p.H) ? 1u : p.map[my * p.W + mx];
        l = __fmul_rn(l, mv == ((m >> j) & 1u) ? 0.98f : 0.02f);
      }
      const float v = __fdiv_rn(pred[q], s1);
      bel[q] = (v == 0.0f) ? 0.0f : __fmul_rn(l, v);
    }
    __syncthreads();
    if (threadIdx.x == 0) s_sum = chain_sum(bel, HW);
    __syncthreads();
    const float s2 = s_sum;
    for (int q = threadIdx.x; q < HW; q += kThreads) bel[q] = __fdiv_rn(bel[q], s2);
    __syncthreads();
  }
  const uint32_t cell = s_cell;
  if (threadIdx.x == 0) {
    if (p.steps) p.steps[i] = t;
    if (p.reached) p.reached[i] = cell == ep.goal ? 1 : 0;
    if (p.collisions) p.collisions[i] = s_coll;
    if (p.final_cell) p.final_cell[i] = cell;
  }
  if (p.final_belief)
    for (int q = threadIdx.x; q < HW; q += kThreads) p.final_belief[(size_t)i * HW + q] = bel[q];
}

// Device buffers of one call, freed on every return path.
struct DeviceBuffers {
  std::vector<void*> ptrs;
  ~DeviceBuffers() { for (void* q : ptrs) cudaFree(q); }
  template <class T>
  int alloc(T** out, size_t count) {
    *out = nullptr;
    if (count == 0) return PP2D_OK;
    void* q = nullptr;
    PP2D_CUDA(cudaMalloc(&q, count * sizeof(T)));
    ptrs.push_back(q);
    *out = static_cast<T*>(q);
    return PP2D_OK;
  }
};

// `views[i]` is the planner episode i follows; every argument is checked.
int rollout(pp2d_sim* s, const std::vector<PlannerView>& views, uint32_t n,
            const uint32_t* starts_xy, const float* beliefs, uint32_t max_steps, uint64_t seed,
            uint64_t first_episode, pp2d_rollout* out) {
  const SimView sv = sim_view(s);
  const size_t hw = (size_t)sv.H * sv.W;
  std::vector<Episode> eps(n);
  for (uint32_t i = 0; i < n; ++i) {
    eps[i].action = views[i].action;
    eps[i].start = starts_xy[2 * (size_t)i + 1] * sv.W + starts_xy[2 * (size_t)i];
    eps[i].goal = views[i].gy * sv.W + views[i].gx;
  }
  const cudaStream_t stream = views[0].stream;
  const int plane = (int)((hw + 3) / 4 * 4);
  const size_t smem = 2 * (size_t)plane * sizeof(float);
  int dev = 0, smem_max = 0;
  PP2D_CUDA(cudaGetDevice(&dev));
  PP2D_CUDA(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  // room for belief_mode's and the kernel's own static shared memory
  const bool shared = smem + 256 <= (size_t)smem_max;
  const size_t n_rec = out ? (size_t)n : 0;
  DeviceBuffers d;
  RolloutParams p{};
  Episode* d_ep = nullptr;
  float* d_b0 = nullptr;
  PP2D_TRY(d.alloc(&d_ep, n));
  PP2D_TRY(d.alloc(&d_b0, beliefs ? n * hw : 0));
  PP2D_TRY(d.alloc(&p.planes, shared ? 0 : (size_t)n * 2 * plane));
  // the records are copied per episode up to its last step, which needs the steps
  const bool records = out && (out->cells || out->actions || out->measurements);
  PP2D_TRY(d.alloc(&p.steps, out && (out->steps || records) ? n_rec : 0));
  PP2D_TRY(d.alloc(&p.reached, out && out->reached ? n_rec : 0));
  PP2D_TRY(d.alloc(&p.collisions, out && out->collisions ? n_rec : 0));
  PP2D_TRY(d.alloc(&p.final_cell, out && out->final_cell ? n_rec : 0));
  PP2D_TRY(d.alloc(&p.final_belief, out && out->final_belief ? n_rec * hw : 0));
  PP2D_TRY(d.alloc(&p.cells, out && out->cells ? n_rec * (max_steps + 1ull) : 0));
  PP2D_TRY(d.alloc(&p.actions, out && out->actions ? n_rec * max_steps : 0));
  PP2D_TRY(d.alloc(&p.meas, out && out->measurements ? n_rec * max_steps : 0));
  PP2D_CUDA(cudaMemcpyAsync(d_ep, eps.data(), n * sizeof(Episode), cudaMemcpyHostToDevice,
                            stream));
  if (beliefs)
    PP2D_CUDA(cudaMemcpyAsync(d_b0, beliefs, n * hw * sizeof(float), cudaMemcpyHostToDevice,
                              stream));
  p.H = (int)sv.H; p.W = (int)sv.W; p.HW = (int)hw; p.plane = plane;
  p.map = sv.map; p.ep = d_ep; p.belief0 = d_b0;
  p.max_steps = max_steps; p.seed = seed; p.first = first_episode;
  if (shared) {
    PP2D_CUDA(cudaFuncSetAttribute(sim_rollout_kernel<true>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    sim_rollout_kernel<true><<<n, kThreads, smem, stream>>>(p);
  } else {
    sim_rollout_kernel<false><<<n, kThreads, 0, stream>>>(p);
  }
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  auto down = [&](void* dst, const void* src, size_t bytes) -> int {
    if (dst && bytes)
      PP2D_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, stream));
    return PP2D_OK;
  };
  // Records go through host staging: entries past an episode's last step of
  // the caller's arrays are not written.
  std::vector<uint32_t> steps, cells;
  std::vector<uint8_t> acts, meas;
  if (out) {
    if (records) steps.resize(n);
    if (out->cells) cells.resize(n * (max_steps + 1ull));
    if (out->actions) acts.resize((size_t)n * max_steps);
    if (out->measurements) meas.resize((size_t)n * max_steps);
    PP2D_TRY(down(records ? steps.data() : out->steps, p.steps, n * sizeof(uint32_t)));
    PP2D_TRY(down(out->reached, p.reached, n));
    PP2D_TRY(down(out->collisions, p.collisions, n * sizeof(uint32_t)));
    PP2D_TRY(down(out->final_cell, p.final_cell, n * sizeof(uint32_t)));
    PP2D_TRY(down(out->final_belief, p.final_belief, n * hw * sizeof(float)));
    PP2D_TRY(down(cells.data(), p.cells, cells.size() * sizeof(uint32_t)));
    PP2D_TRY(down(acts.data(), p.actions, acts.size()));
    PP2D_TRY(down(meas.data(), p.meas, meas.size()));
  }
  PP2D_CUDA(cudaStreamSynchronize(stream));
  if (records) {
    for (uint32_t i = 0; i < n; ++i) {
      const size_t t = steps[i];
      if (out->cells)
        memcpy(out->cells + i * (max_steps + 1ull), cells.data() + i * (max_steps + 1ull),
               (t + 1) * sizeof(uint32_t));
      if (out->actions)
        memcpy(out->actions + (size_t)i * max_steps, acts.data() + (size_t)i * max_steps, t);
      if (out->measurements)
        memcpy(out->measurements + (size_t)i * max_steps, meas.data() + (size_t)i * max_steps, t);
    }
    if (out->steps) memcpy(out->steps, steps.data(), n * sizeof(uint32_t));
  }
  return PP2D_OK;
}

// Arguments every rollout shares; views[i] must already hold episode i's planner.
int check_common(pp2d_sim* s, const PlannerView& v, uint32_t n, const uint32_t* starts_xy) {
  if (!s) return fail(PP2D_ERR_INVALID, "NULL simulator");
  if (v.sharded)
    return fail(PP2D_ERR_STATE, "rollouts need an unsharded single-GPU planner");
  const SimView sv = sim_view(s);
  if (v.H != sv.H || v.W != sv.W)
    return fail(PP2D_ERR_INVALID, "planner map %ux%u differs from the simulator's %ux%u", v.W,
                v.H, sv.W, sv.H);
  if (n == 0) return PP2D_OK;
  if (!starts_xy) return fail(PP2D_ERR_INVALID, "NULL starts_xy");
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t x = starts_xy[2 * (size_t)i], y = starts_xy[2 * (size_t)i + 1];
    if (x >= sv.W || y >= sv.H)
      return fail(PP2D_ERR_INVALID, "episode %u: start (%u %u) outside the %ux%u map", i, x, y,
                  sv.W, sv.H);
    if (sv.map_host[(size_t)y * sv.W + x] > 0)
      return fail(PP2D_ERR_INVALID, "episode %u: start (%u %u) is occupied in the simulator's map",
                  i, x, y);
  }
  return PP2D_OK;
}
}  // namespace

extern "C" {

int pp2d_sim_rollout_mdp(pp2d_sim* s, pp2d_mdp* planner, uint32_t n, const uint32_t* starts_xy,
                         const float* beliefs, uint32_t max_steps, uint64_t seed,
                         uint64_t first_episode, pp2d_rollout* out) {
  if (!planner) return fail(PP2D_ERR_INVALID, "NULL planner");
  const PlannerView v = mdp_view(planner);
  PP2D_TRY(check_common(s, v, n, starts_xy));
  if (n == 0) return PP2D_OK;
  return rollout(s, std::vector<PlannerView>(n, v), n, starts_xy, beliefs, max_steps, seed,
                 first_episode, out);
}

int pp2d_sim_rollout_mdp_batch(pp2d_sim* s, pp2d_mdp_batch* planner, const uint32_t* instances,
                               uint32_t n, const uint32_t* starts_xy, const float* beliefs,
                               uint32_t max_steps, uint64_t seed, uint64_t first_episode,
                               pp2d_rollout* out) {
  if (!planner) return fail(PP2D_ERR_INVALID, "NULL planner");
  PP2D_TRY(check_common(s, mdp_batch_view(planner, 0), n, starts_xy));
  if (n == 0) return PP2D_OK;
  if (!instances) return fail(PP2D_ERR_INVALID, "NULL instances");
  const uint32_t count = mdp_batch_count(planner);
  std::vector<PlannerView> views(n);
  for (uint32_t i = 0; i < n; ++i) {
    if (instances[i] >= count)
      return fail(PP2D_ERR_INVALID, "episode %u names instance %u of a batch of %u", i,
                  instances[i], count);
    views[i] = mdp_batch_view(planner, instances[i]);
  }
  return rollout(s, views, n, starts_xy, beliefs, max_steps, seed, first_episode, out);
}

}  // extern "C"

namespace {
/* The loop of the MDP rollouts with the QV-tree as the planner (DESIGN.md
 * sections 7d, 7e): one persistent tree per episode, planned and updated
 * through a tree batch, the world stepped on the host by the function the
 * device rollouts use.  Episode i plans to goal goals[i] of the planner's goal
 * set (NULL: goal 0) and stops on that goal's cell. */
int rollout_pomdp(pp2d_sim* s, pp2d_pomdp* planner, const uint32_t* goals, uint32_t n,
                  const uint32_t* starts_xy, const float* beliefs, uint32_t max_steps,
                  uint32_t max_depth, uint32_t max_iter, uint64_t seed, uint64_t first_episode,
                  pp2d_rollout* out, const char* fn) {
  if (!planner) return fail(PP2D_ERR_INVALID, "NULL planner");
  PlannerView v;
  v.H = (uint32_t)planner->H; v.W = (uint32_t)planner->W;
  v.gx = (uint32_t)planner->gx; v.gy = (uint32_t)planner->gy;
  PP2D_TRY(check_common(s, v, n, starts_xy));
  // (every step updates the tree that planned it: its root must be expanded)
  if (max_depth == 0 || max_iter == 0)
    return fail(PP2D_ERR_INVALID, "%s: max_depth and max_iter must be > 0", fn);
  if (!goals && !planner->have_alphas)
    return fail(PP2D_ERR_STATE, "pp2d_pomdp_set_alphas not called");
  for (uint32_t i = 0; goals && i < n; ++i) {
    if (goals[i] > (uint32_t)planner->n_goals)
      return fail(PP2D_ERR_INVALID, "%s: episode %u names goal %u of a set of %d", fn, i,
                  goals[i], planner->n_goals + 1);
    if (!planner->goal_alphas[goals[i]])
      return fail(PP2D_ERR_STATE, "%s: episode %u: goal %u has no alpha vectors", fn, i, goals[i]);
  }
  if (n == 0) return PP2D_OK;
  const SimView sv = sim_view(s);
  const size_t hw = (size_t)sv.H * sv.W;
  // the goal cell of every episode, from the host copy of the goal set
  std::vector<uint32_t> goal(n);
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t g = goals ? goals[i] : 0;
    goal[i] = planner->goal_xy[2 * (size_t)g + 1] * sv.W + planner->goal_xy[2 * (size_t)g];
  }
  std::vector<float> point;
  if (!beliefs) {
    point.assign(n * hw, 0.0f);
    for (uint32_t i = 0; i < n; ++i)
      point[i * hw + starts_xy[2 * (size_t)i + 1] * sv.W + starts_xy[2 * (size_t)i]] = 1.0f;
  }
  pp2d_tree_batch* tb = nullptr;
  PP2D_TRY(pp2d_tree_batch_create_goals(planner, beliefs ? beliefs : point.data(), goals, n, &tb));
  struct Guard { pp2d_tree_batch* b; ~Guard() { pp2d_tree_batch_destroy(b); } } guard{tb};
  std::vector<uint32_t> cell(n), steps(n, 0), coll(n, 0), live(n);
  std::vector<uint8_t> act(n), meas(n);
  for (uint32_t i = 0; i < n; ++i) {
    cell[i] = starts_xy[2 * (size_t)i + 1] * sv.W + starts_xy[2 * (size_t)i];
    if (out && out->cells) out->cells[i * (max_steps + 1ull)] = cell[i];
  }
  for (uint32_t t = 0;; ++t) {
    uint32_t nl = 0;                             // episodes that take step t
    for (uint32_t i = 0; i < n; ++i)
      if (steps[i] == t && cell[i] != goal[i] && t < max_steps) live[nl++] = i;
    if (nl == 0) break;
    PP2D_TRY(pp2d_tree_batch_plan(tb, live.data(), nl, max_depth, max_iter, act.data(), nullptr,
                                  nullptr));
    for (uint32_t j = 0; j < nl; ++j) {
      const uint32_t i = live[j];
      const WorldStep w = world_step((int)sv.H, (int)sv.W, sv.map_host, cell[i], act[j], seed,
                                     first_episode + i, t);
      cell[i] = w.cell;
      coll[i] += w.collided ? 1 : 0;
      meas[j] = (uint8_t)w.meas;
      steps[i] = t + 1;
      if (out && out->cells) out->cells[i * (max_steps + 1ull) + t + 1] = w.cell;
      if (out && out->actions) out->actions[(size_t)i * max_steps + t] = act[j];
      if (out && out->measurements) out->measurements[(size_t)i * max_steps + t] = meas[j];
    }
    PP2D_TRY(pp2d_tree_batch_update(tb, live.data(), nl, act.data(), meas.data()));
  }
  if (!out) return PP2D_OK;
  if (out->final_belief) PP2D_TRY(tree_batch_root_beliefs(tb, out->final_belief));
  for (uint32_t i = 0; i < n; ++i) {
    if (out->steps) out->steps[i] = steps[i];
    if (out->reached) out->reached[i] = cell[i] == goal[i] ? 1 : 0;
    if (out->collisions) out->collisions[i] = coll[i];
    if (out->final_cell) out->final_cell[i] = cell[i];
  }
  return PP2D_OK;
}
}  // namespace

extern "C" {

int pp2d_sim_rollout_pomdp(pp2d_sim* s, pp2d_pomdp* planner, uint32_t n, const uint32_t* starts_xy,
                           const float* beliefs, uint32_t max_steps, uint32_t max_depth,
                           uint32_t max_iter, uint64_t seed, uint64_t first_episode,
                           pp2d_rollout* out) {
  return rollout_pomdp(s, planner, nullptr, n, starts_xy, beliefs, max_steps, max_depth, max_iter,
                       seed, first_episode, out, "pp2d_sim_rollout_pomdp");
}

int pp2d_sim_rollout_pomdp_goals(pp2d_sim* s, pp2d_pomdp* planner, const uint32_t* goals,
                                 uint32_t n, const uint32_t* starts_xy, const float* beliefs,
                                 uint32_t max_steps, uint32_t max_depth, uint32_t max_iter,
                                 uint64_t seed, uint64_t first_episode, pp2d_rollout* out) {
  if (n > 0 && !goals) return fail(PP2D_ERR_INVALID, "NULL goals");
  return rollout_pomdp(s, planner, goals, n, starts_xy, beliefs, max_steps, max_depth, max_iter,
                       seed, first_episode, out, "pp2d_sim_rollout_pomdp_goals");
}

}  // extern "C"
