// pomdp.cu -- host side of the QV-Tree C ABI (include/pp2d.h, pp2d_pomdp_* and
// pp2d_tree_*).  Replaces, for the reference's PomdpPathPlanning2d
// (/root/reference/path_planning_2d/src/pomdp/path_planning_2d.cu) and
// SearchTree (src/pomdp/search_tree_cuda.cu, include/.../search_tree.h):
//   generateModelData (model_generation_cuda.cu:349-375), the per-child
//   cudaMalloc / H2D / kernel / sync / D2H / host-normalise / host-bounds
//   sequence of QNode::QNode (search_tree_cuda.cu:161-242), forwardSampling
//   (311-366), evaluateFibCpu / evaluatePbviCpu (fast_informed_bound_cuda.cu:
//   278-297, point_based_value_iteration_cuda.cu:678-699) and the tree
//   bookkeeping (search_tree_cuda.cu:251-286, 397-450, 479-626).
// The tree bookkeeping stays on the host, as in the reference; everything
// that touches a belief runs on the GPU, batched over all the nodes that all
// the queries of a batch create in one expansion round.  No CPU fallback.
#include "../../include/pp2d.h"

#include <algorithm>
#include <atomic>
#include <cfloat>
#include <climits>
#include <cstdint>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <sched.h>
#include <chrono>
#include <vector>

#include "pomdp_host.h"
#include "pomdp_kernels.cuh"

using namespace pp2d;

namespace {

// Host-side tree nodes (search_tree.h:30-128), indices instead of pointers.
struct QNodeH {
  uint8_t action = 0;
  int parent = -1;
  std::vector<int> children;          // V node indices, ascending observation
  float upper = FLT_MAX, lower = -FLT_MAX, heuristic = FLT_MIN, reward = 0.f;
  int to_expand = -1;                 // vnode_to_expand (nullptr = -1)
  uint32_t depth = 1;
};
struct VNodeH {
  int slot = -1;
  uint8_t obs = 0;
  float weight = 0.f;
  int parent = -1;                    // Q node index, -1 for the root
  std::vector<int> children;          // 9 Q node indices once expanded
  float upper = FLT_MAX, lower = -FLT_MAX, heuristic = FLT_MIN;
  int to_expand = -1;
  uint32_t depth = 0;
};

struct Tree {
  std::vector<VNodeH> v;
  std::vector<QNodeH> q;
  int root = -1;
  GlibcRand rng;
  uint32_t expansions = 0;
  bool dead = false;                  // reference would dereference nullptr
  bool dense = false;                 // root belief not +0 on the dead cells: its
                                      // descendants need the dense inner products
  int goal = 0;                       // index in the handle's goal set
};

// search_tree_cuda.cu:251-286
void qnode_update(Tree& t, int qi, float gamma) {
  QNodeH& q = t.q[qi];
  float up = 0.0f, lo = 0.0f;
  for (int c : q.children) {
    up += t.v[c].upper * t.v[c].weight;
    lo += t.v[c].lower * t.v[c].weight;
  }
  q.upper = q.reward + gamma * up;
  q.lower = q.reward + gamma * lo;
  q.heuristic = 0.0f;
  for (int c : q.children) {
    const float h = gamma * t.v[c].weight * t.v[c].heuristic;
    if (h > q.heuristic) { q.heuristic = h; q.to_expand = t.v[c].to_expand; }
  }
  uint32_t child_depth = 0;
  for (int c : q.children)
    if (t.v[c].depth > child_depth) { child_depth = t.v[c].depth; q.depth = child_depth + 1; }
}

// search_tree_cuda.cu:397-435
void vnode_update(Tree& t, int vi) {
  VNodeH& v = t.v[vi];
  int umax = 0, lmax = 0;
  for (int i = 1; i < (int)v.children.size(); ++i) {
    if (t.q[v.children[umax]].upper < t.q[v.children[i]].upper) umax = i;
    if (t.q[v.children[lmax]].lower < t.q[v.children[i]].lower) lmax = i;
  }
  v.upper = t.q[v.children[umax]].upper;
  v.lower = t.q[v.children[lmax]].lower;
  v.heuristic = -FLT_MAX;
  for (int c : v.children) {
    const QNodeH& q = t.q[c];
    if (q.upper <= v.lower) continue;
    if (q.heuristic > v.heuristic) { v.heuristic = q.heuristic; v.to_expand = q.to_expand; }
  }
  uint32_t child_depth = 0;
  for (int c : v.children)
    if (t.q[c].depth > child_depth) { child_depth = t.q[c].depth; v.depth = child_depth + 1; }
}

}  // namespace

struct pp2d_tree {
  pp2d_pomdp* h = nullptr;
  Tree t;
};

namespace pp2d {

// Grow the belief pool (blocks of 32 slots, see bel_off) to at least
// slots_wanted slots.  Live beliefs keep their slot numbers: the blocks of the
// old pool are the first blocks of the new one, one contiguous copy.
int pool_reserve(pp2d_pomdp* h, size_t slots_wanted) {
  if ((size_t)h->cap >= slots_wanted && h->d_bel) return PP2D_OK;
  const size_t cap = (slots_wanted + 31) / 32 * 32;
  if (cap > (size_t)INT32_MAX)
    return fail(PP2D_ERR_INVALID, "belief pool of %zu slots is too large", cap);
  float* nb = nullptr;
  size_t old_cap = h->d_bel ? (size_t)h->cap : 0;
  if (old_cap && h->free_slots.count() == old_cap) {
    // No belief is live: release the old pool BEFORE asking for the new one (a
    // batch sizes the pool to half of the memory; old + new need not fit).
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaFree(h->d_bel);
    h->d_bel = nullptr;
    h->cap = 0;
    h->free_slots.clear();
    old_cap = 0;
    if (e != cudaSuccess)
      return fail(PP2D_ERR_CUDA, "CUDA error releasing the belief pool: %s", cudaGetErrorName(e));
  }
  PP2D_CUDA(cudaMalloc(&nb, cap * (size_t)h->HW * sizeof(float)));
  if (old_cap && h->free_slots.count() != old_cap) {
    cudaError_t e = cudaDeviceSynchronize();     // every stream that touches the pool
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(nb, h->d_bel, old_cap * (size_t)h->HW * sizeof(float),
                          cudaMemcpyDeviceToDevice, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) {
      cudaFree(nb);
      return fail(PP2D_ERR_CUDA, "CUDA error growing the belief pool: %s", cudaGetErrorName(e));
    }
  }
  if (h->d_bel) cudaFree(h->d_bel);
  h->d_bel = nb;
  h->cap = (int)cap;
  h->free_slots.grow(cap);
  return PP2D_OK;
}

int alloc_slot(pp2d_pomdp* h, int* out) {
  if (h->free_slots.empty())
    PP2D_TRY(pool_reserve(h, std::max<size_t>(4096, 2 * (size_t)h->cap)));
  *out = h->free_slots.take();
  return PP2D_OK;
}

int launch_bayes(pp2d_pomdp* h, const std::vector<BayesItem>& items) {
  const int n = (int)items.size();
  if (n == 0) return PP2D_OK;
  PP2D_TRY(h->d_items.ensure(n));
  PP2D_CUDA(cudaMemcpyAsync(h->d_items.p, items.data(), n * sizeof(BayesItem),
                            cudaMemcpyHostToDevice, h->stream));
  dim3 grid((n + 31) / 32, (h->HW + 7) / 8);
  pomdp_bayes_kernel<<<grid, 256, 0, h->stream>>>(h->H, h->W, h->d_tp, h->d_mp,
                                                  h->d_items.p, n, h->d_bel, h->d_bel);
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  h->n_bayes += n;
  return PP2D_OK;
}

// tree:226-229 on the listed columns: sequential sum, then divide.
int launch_normalize(pp2d_pomdp* h, const std::vector<int>& slots) {
  const int n = (int)slots.size();
  if (n == 0) return PP2D_OK;
  PP2D_TRY(h->d_slots.ensure(n));
  PP2D_TRY(h->d_sums.ensure(n));
  PP2D_CUDA(cudaMemcpyAsync(h->d_slots.p, slots.data(), n * sizeof(int),
                            cudaMemcpyHostToDevice, h->stream));
  pomdp_colsum_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(
      h->HW, h->d_slots.p, n, h->d_bel, h->d_sums.p);
  count_launch();
  dim3 grid((n + 31) / 32, (h->HW + 7) / 8);
  pomdp_scale_kernel<<<grid, 256, 0, h->stream>>>(h->HW, h->d_slots.p, n,
                                                  h->d_sums.p, h->d_bel);
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  return PP2D_OK;
}

// tree:326-328 for the listed columns into h->d_prefix[s * n + i].
int launch_prefix(pp2d_pomdp* h, const std::vector<int>& slots) {
  const int n = (int)slots.size();
  if (n == 0) return PP2D_OK;
  PP2D_TRY(h->d_slots.ensure(n));
  PP2D_TRY(h->d_prefix.ensure((size_t)n * h->HW));
  PP2D_CUDA(cudaMemcpyAsync(h->d_slots.p, slots.data(), n * sizeof(int),
                            cudaMemcpyHostToDevice, h->stream));
  pomdp_prefix_kernel<<<(n + 3) / 4, 128, 0, h->stream>>>(
      h->HW, h->d_slots.p, n, h->d_bel, h->d_prefix.p);
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  return PP2D_OK;
}

int launch_scatter(pp2d_pomdp* h, const std::vector<int>& slots, const float* host_rows) {
  const int n = (int)slots.size();
  if (n == 0) return PP2D_OK;
  PP2D_TRY(h->d_slots.ensure(n));
  PP2D_TRY(h->d_rows.ensure((size_t)n * h->HW));
  PP2D_CUDA(cudaMemcpyAsync(h->d_rows.p, host_rows, (size_t)n * h->HW * sizeof(float),
                            cudaMemcpyHostToDevice, h->stream));
  PP2D_CUDA(cudaMemcpyAsync(h->d_slots.p, slots.data(), n * sizeof(int),
                            cudaMemcpyHostToDevice, h->stream));
  dim3 grid((h->HW + 255) / 256, n);
  pomdp_scatter_kernel<<<grid, 256, 0, h->stream>>>(h->HW, h->d_slots.p, n,
                                                    h->d_rows.p, h->d_bel);
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  return PP2D_OK;
}

int launch_gather(pp2d_pomdp* h, const std::vector<int>& slots, float* dev_rows) {
  const int n = (int)slots.size();
  if (n == 0) return PP2D_OK;
  PP2D_TRY(h->d_slots.ensure(n));
  PP2D_CUDA(cudaMemcpyAsync(h->d_slots.p, slots.data(), n * sizeof(int),
                            cudaMemcpyHostToDevice, h->stream));
  dim3 grid((h->HW + 255) / 256, n);
  pomdp_gather_kernel<<<grid, 256, 0, h->stream>>>(h->HW, h->d_slots.p, n, h->d_bel,
                                                   dev_rows);
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  return PP2D_OK;
}

// Live-cell list and compacted bound matrix (see pomdp_host.h).
int refresh_live_cells(pp2d_pomdp* h) {
  const int HW = h->HW;
  if (!h->d_dead) PP2D_CUDA(cudaMalloc(&h->d_dead, HW));
  pomdp_dead_cells_kernel<<<(HW + 127) / 128, 128, 0, h->stream>>>(h->H, h->W, h->d_tp, h->d_dead);
  count_launch();
  h->dead.assign(HW, 0);
  PP2D_CUDA(cudaMemcpyAsync(h->dead.data(), h->d_dead, HW, cudaMemcpyDeviceToHost, h->stream));
  PP2D_CUDA(cudaStreamSynchronize(h->stream));
  std::vector<int> live, all(HW);
  for (int s = 0; s < HW; ++s) {
    all[s] = s;
    if (!h->dead[s]) live.push_back(s);
  }
  if (live.empty()) live.push_back(0);           // degenerate map: keep the kernels in bounds
  h->K = (int)live.size();
  if (!h->d_kidx) PP2D_CUDA(cudaMalloc(&h->d_kidx, HW * sizeof(int)));
  if (!h->d_kidx_all) PP2D_CUDA(cudaMalloc(&h->d_kidx_all, HW * sizeof(int)));
  PP2D_CUDA(cudaMemcpy(h->d_kidx, live.data(), live.size() * sizeof(int), cudaMemcpyHostToDevice));
  PP2D_CUDA(cudaMemcpy(h->d_kidx_all, all.data(), HW * sizeof(int), cudaMemcpyHostToDevice));
  // inverse list and the likelihood rows of the live cells (the Bayes kernels
  // of a round index their scratch by live row, not by cell)
  std::vector<int> kinv(HW, -1);
  for (int k = 0; k < h->K; ++k) kinv[live[k]] = k;
  if (!h->d_kinv) PP2D_CUDA(cudaMalloc(&h->d_kinv, HW * sizeof(int)));
  PP2D_CUDA(cudaMemcpy(h->d_kinv, kinv.data(), HW * sizeof(int), cudaMemcpyHostToDevice));
  if (!h->d_mp_live) PP2D_CUDA(cudaMalloc(&h->d_mp_live, (size_t)HW * 16 * sizeof(float)));
  for (int k = 0; k < h->K; ++k)
    PP2D_CUDA(cudaMemcpyAsync(h->d_mp_live + (size_t)k * 16, h->d_mp + (size_t)live[k] * 16,
                              16 * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
  PP2D_CUDA(cudaStreamSynchronize(h->stream));
  if (h->ld > 0) {                               // some goal has alpha vectors
    const size_t goals = (size_t)h->n_goals + 1;
    std::vector<float> rows(goals * h->K * h->ld);
    for (size_t g = 0; g < goals; ++g)
      for (int k = 0; k < h->K; ++k)
        memcpy(rows.data() + (g * h->K + k) * h->ld,
               h->alpha_host.data() + (g * HW + live[k]) * h->ld, (size_t)h->ld * sizeof(float));
    if (h->d_alpha_live) cudaFree(h->d_alpha_live);
    h->d_alpha_live = nullptr;
    PP2D_CUDA(cudaMalloc(&h->d_alpha_live, rows.size() * sizeof(float)));
    PP2D_CUDA(cudaMemcpy(h->d_alpha_live, rows.data(), rows.size() * sizeof(float),
                         cudaMemcpyHostToDevice));
  }
  return PP2D_OK;
}

bool zero_on_dead_cells(const pp2d_pomdp* h, const float* belief) {
  uint32_t any = 0;
  for (int s = 0; s < h->HW; ++s) {
    uint32_t bits;
    memcpy(&bits, belief + s, sizeof(bits));
    any |= h->dead[s] ? bits : 0u;               // -0 also forces the dense path
  }
  return any == 0;
}

}  // namespace pp2d

namespace {

// The inner dimension of the sequential products of one launch: the live
// cells, or all cells when some belief involved may be non-zero elsewhere.
// kinv: cell -> inner row (-1: left out); mp: the likelihood rows of the inner rows;
// gstride: floats from one goal's bound matrix to the next.
struct InnerDim {
  const int* kidx; int K; const float* alpha; const int* kinv; const float* mp; size_t gstride;
};
InnerDim inner_dim(const pp2d_pomdp* h, bool dense) {
  // (a non-finite bound makes 0 * alpha a NaN in the reference: nothing is skipped then)
  if (dense || !h->skip_dead || !h->alphas_finite)
    return {h->d_kidx_all, h->HW, h->d_alpha, h->d_kidx_all, h->d_mp, (size_t)h->HW * h->ld};
  return {h->d_kidx, h->K, h->d_alpha_live, h->d_kinv, h->d_mp_live, (size_t)h->K * h->ld};
}

// The entry list of the support, values and bounds launches over beliefs that
// come in runs of one goal (DESIGN.md section 7e).  Every run but the last is
// padded to whole tiles of kEvM entries by repeating its last slot, so that a
// tile holds beliefs of one goal; the goals of the tiles follow the entries
// (one upload).  A repeated belief adds no inner row to its tile and its values
// are never read.  With one goal the list is the beliefs' slots, unpadded.
struct GoalTiles {
  int* out = nullptr;                 // room() ints
  int n = 0, goal = -1;
  std::vector<int> tile_goal;
  std::vector<std::pair<int, int>> pads;   // (tile, repeated entries in it)
  // entries + tile goals of `beliefs` beliefs in at most `runs` runs
  static size_t room(size_t beliefs, size_t runs) {
    const size_t entries = beliefs + runs * (size_t)(kEvM - 1);
    return entries + entries / kEvM + 1;
  }
  void start(int* buf) { out = buf; n = 0; goal = -1; tile_goal.clear(); pads.clear(); }
  int add(int slot, int g) {          // -> the entry of this belief
    if (g != goal) {
      if (n % kEvM) {
        const int last = out[n - 1], first = n;
        while (n % kEvM) out[n++] = last;
        pads.push_back({first / kEvM, n - first});
      }
      goal = g;
    }
    if (n % kEvM == 0) tile_goal.push_back(g);
    out[n] = slot;
    return n++;
  }
  int finish() {                      // -> tiles; their goals now follow the entries
    std::copy(tile_goal.begin(), tile_goal.end(), out + n);
    return (int)tile_goal.size();
  }
};

// Host threads for the per-tree work of a batch: pp2d_set_host_threads, else
// PP2D_HOST_THREADS, else the CPUs this process may run on divided by the
// ranks sharing the node (LOCAL_WORLD_SIZE, set by torchrun), at most 8.
// (Set explicitly rather than left to OMP_NUM_THREADS, which torchrun forces
// to 1; more threads than cores makes OpenMP's spinning barriers crawl, and
// as many threads as cores leaves none for the thread that feeds the GPU:
// measured on a 16-core B200 box, 1 250 plans take 56-57 ms with 8 threads,
// 57-61 ms with 4 and 54-66 ms with occasional 160 ms outliers with 16.)
std::atomic<int> g_host_threads{0};
int host_threads() {
  const int forced = g_host_threads.load(std::memory_order_relaxed);
  if (forced > 0) return forced;
  static const int n = [] {
    const char* e = getenv("PP2D_HOST_THREADS");
    if (e && atoi(e) > 0) return atoi(e);
    cpu_set_t set;
    int c = 1;
    if (sched_getaffinity(0, sizeof(set), &set) == 0) c = CPU_COUNT(&set);
    const char* lw = getenv("LOCAL_WORLD_SIZE");
    if (lw && atoi(lw) > 1) c /= atoi(lw);
    return std::max(1, std::min(8, c));
  }();
  return n;
}

double now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// Evaluate the beliefs in `slots` against the bounds of their goals (`goals`
// per belief, NULL: goal 0): per belief 4 floats {upper, lower, packed
// indices, 0} into host `out` (B4, B5).  The beliefs are evaluated goal by
// goal (GoalTiles); every belief walks all inner rows, so its bits do not
// depend on which others share its tile.
int evaluate_slots(pp2d_pomdp* h, const std::vector<int>& slots, const int* goals, float* out,
                   bool dense) {
  const int n = (int)slots.size();
  if (n == 0) return PP2D_OK;
  std::vector<int> order(n);
  for (int i = 0; i < n; ++i) order[i] = i;
  if (goals)
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return goals[a] < goals[b]; });
  std::vector<int> list(GoalTiles::room(n, (size_t)h->n_goals + 1)), pos(n);
  GoalTiles gt;
  gt.start(list.data());
  for (int j = 0; j < n; ++j) pos[order[j]] = gt.add(slots[order[j]], goals ? goals[order[j]] : 0);
  const int np = gt.n, ntiles = gt.finish();
  PP2D_TRY(h->d_slots.ensure(np + ntiles));
  PP2D_TRY(h->d_vals.ensure((size_t)np * h->ncol));
  PP2D_TRY(h->d_out.ensure((size_t)np * 4));
  PP2D_CUDA(cudaMemcpyAsync(h->d_slots.p, list.data(), (np + ntiles) * sizeof(int),
                            cudaMemcpyHostToDevice, h->stream));
  dim3 grid(ntiles, (h->ncol + kEvN - 1) / kEvN);
  const InnerDim in = inner_dim(h, dense);
  pomdp_values_kernel<false><<<grid, 256, 0, h->stream>>>(
      in.K, in.kidx, h->HW, h->ld, h->ncol, h->d_slots.p, np, h->d_bel, in.alpha,
      h->d_vals.p, nullptr, nullptr, nullptr, 0, h->d_slots.p + np, in.gstride);
  h->work_rows += (uint64_t)in.K * (uint64_t)np;
  h->pad_entries += (uint64_t)(np - n);
  h->pad_rows += (uint64_t)in.K * (uint64_t)(np - n);
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  pomdp_bounds_kernel<<<(np + 3) / 4, 128, 0, h->stream>>>(
      np, h->ncol, h->n_pbvi, h->d_vals.p, h->d_out.p);
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  bool in_place = np == n;                       // entry i is belief i
  for (int i = 0; i < n && in_place; ++i) in_place = pos[i] == i;
  std::vector<float> res(in_place ? 0 : (size_t)np * 4);
  float* dst = in_place ? out : res.data();
  PP2D_CUDA(cudaMemcpyAsync(dst, h->d_out.p, (size_t)np * 4 * sizeof(float),
                            cudaMemcpyDeviceToHost, h->stream));
  PP2D_CUDA(cudaStreamSynchronize(h->stream));
  if (!in_place)
    for (int i = 0; i < n; ++i) memcpy(out + (size_t)i * 4, dst + (size_t)pos[i] * 4, 4 * sizeof(float));
  return PP2D_OK;
}

// tree:226-229 on the listed columns: sequential sum, then divide.
int normalize_slots(pp2d_pomdp* h, int n, float* sums_out_dev) {
  PP2D_TRY(h->d_sums.ensure(n));
  pomdp_colsum_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(
      h->HW, h->d_slots.p, n, h->d_bel, h->d_sums.p);
  count_launch();
  dim3 grid((n + 31) / 32, (h->HW + 7) / 8);
  pomdp_scale_kernel<<<grid, 256, 0, h->stream>>>(h->HW, h->d_slots.p, n,
                                                  h->d_sums.p, h->d_bel);
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  (void)sums_out_dev;
  return PP2D_OK;
}

// search_tree_cuda.cu:368-388 VNode::VNode for already-resident beliefs.
void init_vnode(VNodeH& v, int slot, uint8_t obs, float weight, int parent,
                const float* ev, int self) {
  v.slot = slot; v.obs = obs; v.weight = weight; v.parent = parent;
  v.upper = ev[0]; v.lower = ev[1];
  v.heuristic = v.upper - v.lower;
  v.to_expand = self;
  v.depth = 0;
}

// Upload host beliefs ([n][HW]) into fresh slots and create the root V nodes.
// mode_key (optional, n entries): column * H + row of the first maximum of
// every start belief (the order a batch is planned in, see pp2d_pomdp_plan_batch).
int make_roots(pp2d_pomdp* h, std::vector<Tree*>& trees, const float* beliefs,
               uint32_t* mode_key = nullptr) {
  const int n = (int)trees.size();
  std::vector<int> slots(n);
  for (int i = 0; i < n; ++i) PP2D_TRY(alloc_slot(h, &slots[i]));
  // A batch goes through page-locked staging: the caller's buffer is pageable
  // (a copy straight from it is staged by the driver at a fraction of the PCIe
  // rate, with the host blocked), and the host threads read every belief here
  // anyway.
  const size_t row = (size_t)h->HW;
  const bool staged = n >= 64;
  if (staged && h->pin_rows_cap < (size_t)n * row) {
    if (h->pin_rows) cudaFreeHost(h->pin_rows);
    h->pin_rows = nullptr;
    h->pin_rows_cap = 0;
    PP2D_CUDA(cudaHostAlloc((void**)&h->pin_rows, (size_t)n * row * sizeof(float),
                            cudaHostAllocDefault));
    h->pin_rows_cap = (size_t)n * row;
  }
  // Start beliefs that are not +0 on the dead cells (and everything grown from
  // them) are evaluated with the dense inner products.
  bool any_dense = false;
#pragma omp parallel for schedule(static) num_threads(host_threads()) reduction(|| : any_dense) \
    if (n >= 64)
  for (int i = 0; i < n; ++i) {
    const float* b = beliefs + (size_t)i * row;
    trees[i]->dense = !zero_on_dead_cells(h, b);
    any_dense = any_dense || trees[i]->dense;
    if (staged) memcpy(h->pin_rows + (size_t)i * row, b, row * sizeof(float));
    if (mode_key) {
      int best = 0;
      for (int s = 1; s < h->HW; ++s)
        if (b[s] > b[best]) best = s;
      mode_key[i] = (uint32_t)(best % h->W) * (uint32_t)h->H + (uint32_t)(best / h->W);
    }
  }
  PP2D_TRY(h->d_slots.ensure(n));
  PP2D_TRY(h->d_rows.ensure((size_t)n * h->HW));
  PP2D_CUDA(cudaMemcpyAsync(h->d_rows.p, staged ? h->pin_rows : beliefs,
                            (size_t)n * h->HW * sizeof(float), cudaMemcpyHostToDevice,
                            h->stream));
  PP2D_CUDA(cudaMemcpyAsync(h->d_slots.p, slots.data(), n * sizeof(int),
                            cudaMemcpyHostToDevice, h->stream));
  dim3 grid((h->HW + 255) / 256, n);
  pomdp_scatter_kernel<<<grid, 256, 0, h->stream>>>(h->HW, h->d_slots.p, n,
                                                    h->d_rows.p, h->d_bel);
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  std::vector<float> ev((size_t)n * 4);
  std::vector<int> goals(n);
  for (int i = 0; i < n; ++i) goals[i] = trees[i]->goal;
  PP2D_TRY(evaluate_slots(h, slots, goals.data(), ev.data(), any_dense));
  for (int i = 0; i < n; ++i) {
    Tree& t = *trees[i];
    t.v.emplace_back();
    t.root = (int)t.v.size() - 1;
    init_vnode(t.v.back(), slots[i], 0, 0.0f, -1, ev.data() + (size_t)i * 4, t.root);
    h->n_vnodes++;
  }
  return PP2D_OK;
}

// The belief slots of a subtree are appended to `freed` (the caller gives them
// back to the pool; trees of a batch are re-rooted on several host threads).
void free_subtree_v(Tree& t, int vi, std::vector<int>& freed);
void free_subtree_q(Tree& t, int qi, std::vector<int>& freed) {
  for (int c : t.q[qi].children) free_subtree_v(t, c, freed);
  t.q[qi].children.clear();
}
void free_subtree_v(Tree& t, int vi, std::vector<int>& freed) {
  for (int c : t.v[vi].children) free_subtree_q(t, c, freed);
  t.v[vi].children.clear();
  if (t.v[vi].slot >= 0) { freed.push_back(t.v[vi].slot); t.v[vi].slot = -1; }
}
void give_back(pp2d_pomdp* h, const std::vector<int>& freed) {
  for (int s : freed) h->free_slots.put(s);
}

// Page-locked host buffer: source / target of the asynchronous copies of a
// round (a pageable buffer would make cudaMemcpyAsync wait for the stream).
template <typename T>
struct PinnedBuf {
  T* p = nullptr;
  size_t cap = 0;
  int ensure(size_t n) {
    if (n <= cap) return PP2D_OK;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    const size_t want = n + n / 2 + 64;
    PP2D_CUDA(cudaHostAlloc((void**)&p, want * sizeof(T), cudaHostAllocDefault));
    cap = want;
    return PP2D_OK;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// Everything one expansion round of a group of trees needs, kept between
// rounds.  A batch is planned as TWO such groups in lock-step so that the host
// work of one (random draws, child lists, tree bookkeeping) overlaps the
// device work of the other.
struct RoundCtx {
  struct Job { Tree* t; int v; };
  struct Child { uint8_t a, z; float w; };
  std::vector<Job> jobs;
  int n = 0, nk = 0;
  bool dense = false;                // some tree of this round needs the dense products
  PinnedBuf<int> slots, kslots, kgroup;
  PinnedBuf<int> vlist;              // entries of the values launches (GoalTiles), tile goals
  std::vector<int> vpos;             // child k -> its entry
  GoalTiles tiles;
  PinnedBuf<int> tcount;             // rows per tile, read back when a tile has padding
  PinnedBuf<float> draws, rewards, ev;
  PinnedBuf<BayesItem> items;
  PinnedBuf<uint8_t> obs;
  std::vector<int> first;
  std::vector<Child> kids;
  bool tiled_pads = false;           // c.tcount holds this round's rows per tile
  DevBuf<int> d_jobslots, d_vlist, d_kgroup;
  DevBuf<float> d_pred;              // [HW][ngp] predictions of the Q nodes of a round
  DevBuf<float> d_prefix, d_draws, d_rew, d_sums, d_vals, d_out;
  DevBuf<uint8_t> d_obs;
  DevBuf<BayesItem> d_items;
  DevBuf<int2> d_tlist;              // per-tile inner rows of the values launch
  DevBuf<int> d_tcount, d_torder;
  DevBuf<uint32_t> d_tmask;
  cudaEvent_t e1 = nullptr, e2 = nullptr;
  cudaStream_t stream = nullptr;     // own stream: the tail of one group's launches
                                     // overlaps the other group's
  cudaStream_t stream_hi = nullptr;  // stage 1 (small sampling kernels): high priority, so
                                     // that it is not queued behind the other group's
                                     // values launch and the host can move on
  ~RoundCtx() {
    slots.release(); kslots.release(); kgroup.release(); draws.release();
    vlist.release(); tcount.release();
    rewards.release(); d_kgroup.release(); d_pred.release();
    ev.release(); items.release(); obs.release();
    d_jobslots.release(); d_vlist.release(); d_prefix.release();
    d_draws.release(); d_rew.release(); d_sums.release(); d_vals.release(); d_out.release();
    d_obs.release(); d_items.release(); d_tlist.release(); d_tcount.release(); d_torder.release(); d_tmask.release();
    if (e1) cudaEventDestroy(e1);
    if (e2) cudaEventDestroy(e2);
    if (stream) cudaStreamDestroy(stream);
    if (stream_hi) cudaStreamDestroy(stream_hi);
  }
};

constexpr int kMaxGroups = 4;          // = number of entries of pp2d_pomdp::round_ctx
RoundCtx* round_ctx(pp2d_pomdp* h, int which) {
  if (!h->round_ctx[which]) {
    RoundCtx* c = new RoundCtx;
    cudaEventCreateWithFlags(&c->e1, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->e2, cudaEventDisableTiming);
    cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    int lo_prio = 0, hi_prio = 0;
    cudaDeviceGetStreamPriorityRange(&lo_prio, &hi_prio);
    cudaStreamCreateWithPriority(&c->stream_hi, cudaStreamNonBlocking, hi_prio);
    h->round_ctx[which] = c;
  }
  return static_cast<RoundCtx*>(h->round_ctx[which]);
}

// Stage 1 of an expansion round (SearchTree::expand, search_tree_cuda.cu:490-508)
// for every tree in `trees`: the nodes to expand, their random draws, then
// -- enqueued, not waited for -- forward sampling (search_tree_cuda.cu:311-366)
// and the reward of the 9 new Q nodes (search_tree_cuda.cu:168-173).
int round_stage1(pp2d_pomdp* h, RoundCtx& c, const std::vector<Tree*>& trees) {
  double t0 = now_s();
  c.jobs.clear();
  c.dense = false;
  std::vector<int> freed;
  for (Tree* t : trees) {
    if (t->dead) continue;
    c.dense = c.dense || t->dense;
    const int v = t->v[t->root].to_expand;
    if (v < 0) { t->dead = true; continue; }
    if (!t->v[v].children.empty()) {            // re-expansion (leak in the ref)
      for (int q : t->v[v].children) free_subtree_q(*t, q, freed);
      t->v[v].children.clear();
    }
    c.jobs.push_back({t, v});
  }
  give_back(h, freed);
  const int n = c.n = (int)c.jobs.size();
  c.nk = 0;
  if (n == 0) return PP2D_OK;
  const int HW = h->HW;
  const size_t nd = (size_t)n * kActions * kSamples;
  PP2D_TRY(c.slots.ensure(2 * (size_t)n));     // slots, then goals
  PP2D_TRY(c.draws.ensure(nd));
  PP2D_TRY(c.obs.ensure(nd));
  PP2D_TRY(c.rewards.ensure((size_t)n * kActions));
#pragma omp parallel for schedule(static) num_threads(host_threads()) if (n >= 64)
  for (int i = 0; i < n; ++i) {
    c.slots.p[i] = c.jobs[i].t->v[c.jobs[i].v].slot;
    c.slots.p[n + i] = c.jobs[i].t->goal;
    float* d = c.draws.p + (size_t)i * kActions * kSamples;
    for (int k = 0; k < kActions * kSamples; ++k)
      d[k] = (float)c.jobs[i].t->rng.next() / ((float)2147483647 + 1.0f);
  }
  PP2D_TRY(c.d_jobslots.ensure(2 * (size_t)n));
  PP2D_TRY(c.d_prefix.ensure((size_t)n * HW));
  PP2D_TRY(c.d_draws.ensure(nd));
  PP2D_TRY(c.d_obs.ensure(nd));
  PP2D_TRY(c.d_rew.ensure((size_t)n * kActions));
  PP2D_CUDA(cudaMemcpyAsync(c.d_jobslots.p, c.slots.p, 2 * (size_t)n * sizeof(int),
                            cudaMemcpyHostToDevice, c.stream_hi));
  PP2D_CUDA(cudaMemcpyAsync(c.d_draws.p, c.draws.p, nd * sizeof(float),
                            cudaMemcpyHostToDevice, c.stream_hi));
  // prefix sums and reward dots of the expanded nodes in one launch, then the
  // sampling (which needs the prefix sums)
  const InnerDim in = inner_dim(h, c.dense);
  pomdp_expand_kernel<<<(n + 3) / 4 + (n * 3 + 3) / 4, 128, 0, c.stream_hi>>>(
      HW, in.K, in.kidx, c.d_jobslots.p, c.d_jobslots.p + n, n, h->d_bel, h->d_sr, c.d_prefix.p,
      c.d_rew.p);
  count_launch();
  const int nt = (int)nd;
  pomdp_sample_kernel<<<(nt + 127) / 128, 128, 0, c.stream_hi>>>(
      h->H, h->W, n, kSamples, h->d_tp, h->d_mp, c.d_prefix.p, c.d_draws.p,
      h->d_uniforms, c.d_obs.p);
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  PP2D_CUDA(cudaMemcpyAsync(c.obs.p, c.d_obs.p, nd, cudaMemcpyDeviceToHost, c.stream_hi));
  PP2D_CUDA(cudaMemcpyAsync(c.rewards.p, c.d_rew.p, (size_t)n * kActions * sizeof(float),
                            cudaMemcpyDeviceToHost, c.stream_hi));
  PP2D_CUDA(cudaEventRecord(c.e1, c.stream_hi));
  h->t_phase[0] += now_s() - t0;                 // host: draws, enqueue
  return PP2D_OK;
}

// Stage 2: unique observations per Q node (search_tree_cuda.cu:181-195), then
// -- enqueued -- the children beliefs (Bayes update + normalise,
// search_tree_cuda.cu:213-229) and their bounds (search_tree_cuda.cu:376-385).
int round_stage2(pp2d_pomdp* h, RoundCtx& c) {
  const int n = c.n;
  if (n == 0) return PP2D_OK;
  double t0 = now_s();
  PP2D_CUDA(cudaEventSynchronize(c.e1));
  h->t_phase[1] += now_s() - t0; t0 = now_s();   // wait: sampling + rewards on device
  const int HW = h->HW;
  c.first.assign(n + 1, 0);                      // children of job i: [first[i], first[i+1])
#pragma omp parallel for schedule(static) num_threads(host_threads()) if (n >= 64)
  for (int i = 0; i < n; ++i) {
    int cnt = 0;
    for (int a = 0; a < kActions; ++a) {
      const uint8_t* o = c.obs.p + ((size_t)i * kActions + a) * kSamples;
      uint32_t m = 0;
      for (int k = 0; k < kSamples; ++k) m |= 1u << (o[k] & 15);
      cnt += __builtin_popcount(m);
    }
    c.first[i + 1] = cnt;
  }
  for (int i = 0; i < n; ++i) c.first[i + 1] += c.first[i];
  const int nk = c.nk = c.first[n];
  PP2D_TRY(c.kslots.ensure(nk));
  PP2D_TRY(c.items.ensure(nk));
  PP2D_TRY(c.kgroup.ensure(nk));
  for (int k = 0; k < nk; ++k) PP2D_TRY(alloc_slot(h, &c.kslots.p[k]));
  c.kids.resize(nk);
#pragma omp parallel for schedule(static) num_threads(host_threads()) if (n >= 64)
  for (int i = 0; i < n; ++i) {
    int k = c.first[i];
    for (int a = 0; a < kActions; ++a) {
      const uint8_t* o = c.obs.p + ((size_t)i * kActions + a) * kSamples;
      int count[16] = {0};
      for (int s = 0; s < kSamples; ++s) count[o[s] & 15]++;
      for (int z = 0; z < 16; ++z) {
        if (!count[z]) continue;
        c.kids[k] = RoundCtx::Child{(uint8_t)a, (uint8_t)z, (float)count[z] / (float)kSamples};
        c.items.p[k] = BayesItem{c.slots.p[i], c.kslots.p[k], (uint8_t)a, (uint8_t)z};
        c.kgroup.p[k] = i * kActions + a;
        ++k;
      }
    }
  }
  // the children in runs of one goal (the jobs are in goal order, see
  // plan_trees), padded to whole tiles per goal
  size_t runs = n ? 1 : 0;
  for (int i = 1; i < n; ++i) runs += c.jobs[i].t->goal != c.jobs[i - 1].t->goal;
  PP2D_TRY(c.vlist.ensure(GoalTiles::room(nk, runs)));
  c.vpos.resize(nk);
  c.tiles.start(c.vlist.p);
  for (int i = 0; i < n; ++i)
    for (int k = c.first[i]; k < c.first[i + 1]; ++k)
      c.vpos[k] = c.tiles.add(c.kslots.p[k], c.jobs[i].t->goal);
  const int np = c.tiles.n, ntiles = c.tiles.finish();
  PP2D_TRY(c.ev.ensure((size_t)np * 4));
  const int ng = n * kActions;
  PP2D_TRY(c.d_items.ensure(nk));
  PP2D_TRY(c.d_vlist.ensure((size_t)np + ntiles));
  PP2D_TRY(c.d_sums.ensure(nk));
  PP2D_TRY(c.d_vals.ensure((size_t)np * h->ncol));
  PP2D_TRY(c.d_out.ensure((size_t)np * 4));
  PP2D_CUDA(cudaMemcpyAsync(c.d_items.p, c.items.p, nk * sizeof(BayesItem),
                            cudaMemcpyHostToDevice, c.stream));
  PP2D_CUDA(cudaMemcpyAsync(c.d_vlist.p, c.vlist.p, ((size_t)np + ntiles) * sizeof(int),
                            cudaMemcpyHostToDevice, c.stream));
  const int* d_tgoal = c.d_vlist.p + np;
  const int ngp = (ng + 31) / 32 * 32;
  PP2D_TRY(c.d_kgroup.ensure(nk));
  PP2D_TRY(c.d_pred.ensure((size_t)HW * ngp));
  PP2D_CUDA(cudaMemcpyAsync(c.d_kgroup.p, c.kgroup.p, nk * sizeof(int), cudaMemcpyHostToDevice,
                            c.stream));
  const InnerDim in = inner_dim(h, c.dense);
  // (group g = 9 * job + action; c.d_jobslots was uploaded in stage 1, which
  // this stream is behind: the host has waited for e1)
  dim3 bgrid((n + 31) / 32, (in.K + 7) / 8);
  pomdp_predict9_kernel<<<bgrid, 256, 0, c.stream>>>(h->H, h->W, in.K, in.kidx, ngp, h->d_tp,
                                                      c.d_jobslots.p, n, h->d_bel, c.d_pred.p);
  count_launch();
  h->n_bayes += nk;
  pomdp_child_sum_kernel<<<(nk + 127) / 128, 128, 0, c.stream>>>(
      in.K, ngp, in.mp, c.d_items.p, c.d_kgroup.p, nk, c.d_pred.p, c.d_sums.p);
  count_launch();
  dim3 sgrid((nk + 31) / 32, (HW + 8 * kCwCells - 1) / (8 * kCwCells));
  pomdp_child_write_kernel<<<sgrid, 256, 0, c.stream>>>(HW, ngp, h->d_mp, in.kinv,
                                                         c.d_items.p, c.d_kgroup.p, nk,
                                                         c.d_pred.p, c.d_sums.p, h->d_bel);
  count_launch();
  dim3 vgrid(ntiles, (h->ncol + kEvN - 1) / kEvN);
  const bool tiled = h->tile_support && h->alphas_finite;
  if (tiled) {
    // the inner rows each tile of kEvM children really needs (exact, see
    // pomdp_values_kernel<TILED>)
    const int mstride = (in.K + 31) / 32;
    PP2D_TRY(c.d_tlist.ensure((size_t)vgrid.x * in.K));
    PP2D_TRY(c.d_tcount.ensure(vgrid.x));
    PP2D_TRY(c.d_tmask.ensure((size_t)vgrid.x * mstride));
    dim3 fgrid(vgrid.x, (in.K + 255) / 256);
    pomdp_support_flags_kernel<<<fgrid, 256, 0, c.stream>>>(
        HW, in.K, in.kidx, c.d_vlist.p, np, h->d_bel, c.d_tmask.p, mstride);
    count_launch();
    pomdp_support_list_kernel<<<vgrid.x, 256, 0, c.stream>>>(in.K, in.kidx, c.d_tmask.p, mstride,
                                                             c.d_tlist.p, c.d_tcount.p, np,
                                                             h->d_work);
    count_launch();
    PP2D_TRY(c.d_torder.ensure(vgrid.x));
    pomdp_tile_order_kernel<<<(vgrid.x + 255) / 256, 256, 0, c.stream>>>(
        (int)vgrid.x, c.d_tcount.p, c.d_torder.p);
    count_launch();
    pomdp_values_kernel<true><<<dim3(vgrid.y, vgrid.x), 256, 0, c.stream>>>(
        in.K, in.kidx, h->HW, h->ld, h->ncol, c.d_vlist.p, np, h->d_bel, in.alpha, c.d_vals.p,
        c.d_tlist.p, c.d_tcount.p, c.d_torder.p, in.K, d_tgoal, in.gstride);
  } else {
    pomdp_values_kernel<false><<<vgrid, 256, 0, c.stream>>>(
        in.K, in.kidx, h->HW, h->ld, h->ncol, c.d_vlist.p, np, h->d_bel, in.alpha, c.d_vals.p,
        nullptr, nullptr, nullptr, 0, d_tgoal, in.gstride);
    h->work_rows += (uint64_t)in.K * (uint64_t)np;
  }
  count_launch();
  pomdp_bounds_kernel<<<(np + 3) / 4, 128, 0, c.stream>>>(np, h->ncol, h->n_pbvi,
                                                               c.d_vals.p, c.d_out.p);
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  PP2D_CUDA(cudaMemcpyAsync(c.ev.p, c.d_out.p, (size_t)np * 4 * sizeof(float),
                            cudaMemcpyDeviceToHost, c.stream));
  // the work spent on padding (pp2d_pomdp_padding_counters): rows of the
  // padded tiles, read back with the bounds
  h->pad_entries += (uint64_t)(np - nk);
  if (np != nk) {
    if (tiled) {
      PP2D_TRY(c.tcount.ensure(ntiles));
      PP2D_CUDA(cudaMemcpyAsync(c.tcount.p, c.d_tcount.p, ntiles * sizeof(int),
                                cudaMemcpyDeviceToHost, c.stream));
    } else {
      h->pad_rows += (uint64_t)in.K * (uint64_t)(np - nk);
    }
  }
  c.tiled_pads = tiled && np != nk;
  PP2D_CUDA(cudaEventRecord(c.e2, c.stream));
  h->t_phase[2] += now_s() - t0;                 // host: children lists, enqueue
  return PP2D_OK;
}

// Stage 3: the new nodes enter their trees; bounds, heuristics and depths are
// propagated to the roots (search_tree_cuda.cu:251-286, 397-450, 497-505).
int round_stage3(pp2d_pomdp* h, RoundCtx& c) {
  const int n = c.n;
  if (n == 0) return PP2D_OK;
  double t0 = now_s();
  PP2D_CUDA(cudaEventSynchronize(c.e2));
  h->t_phase[3] += now_s() - t0; t0 = now_s();   // wait: bayes + normalise + bounds on device
#pragma omp parallel for schedule(dynamic, 8) num_threads(host_threads()) if (n >= 64)
  for (int i = 0; i < n; ++i) {
    Tree& t = *c.jobs[i].t;
    const int vi = c.jobs[i].v;
    int kpos = c.first[i];
    const int kend = c.first[i + 1];
    // (room for whole rounds at once: an exact reserve would move every node
    // of the tree in every round)
    if (t.v.capacity() < t.v.size() + (size_t)(kend - kpos))
      t.v.reserve(std::max<size_t>(2 * t.v.capacity(), t.v.size() + 4 * (size_t)(kend - kpos)));
    if (t.q.capacity() < t.q.size() + kActions)
      t.q.reserve(std::max<size_t>(2 * t.q.capacity(), t.q.size() + 4 * kActions));
    t.v[vi].children.resize(kActions);
    for (int a = 0; a < kActions; ++a) {
      t.q.emplace_back();
      const int qi = (int)t.q.size() - 1;
      t.v[vi].children[a] = qi;
      t.q[qi].action = (uint8_t)a;
      t.q[qi].parent = vi;
      t.q[qi].reward = c.rewards.p[(size_t)i * kActions + a];
      while (kpos < kend && c.kids[kpos].a == a) {
        t.v.emplace_back();
        const int ci = (int)t.v.size() - 1;
        init_vnode(t.v[ci], c.kslots.p[kpos], c.kids[kpos].z, c.kids[kpos].w, qi,
                   c.ev.p + (size_t)c.vpos[kpos] * 4, ci);
        t.q[qi].children.push_back(ci);
        ++kpos;
      }
      qnode_update(t, qi, h->gamma);
    }
    vnode_update(t, vi);
    int v = vi;
    while (t.v[v].parent >= 0) {                 // search_tree_cuda.cu:497-505
      const int pq = t.v[v].parent;
      qnode_update(t, pq, h->gamma);
      const int pv = t.q[pq].parent;
      vnode_update(t, pv);
      v = pv;
    }
    t.expansions++;
  }
  h->n_vnodes += (uint64_t)c.nk;
  if (c.tiled_pads)
    for (const auto& p : c.tiles.pads) h->pad_rows += (uint64_t)c.tcount.p[p.first] * p.second;
  c.tiled_pads = false;
  c.n = 0;                                       // this round is absorbed
  h->t_phase[4] += now_s() - t0;                 // host: tree bookkeeping
  return PP2D_OK;
}

// One expansion round for every tree in `trees` (single group).
int expand_round(pp2d_pomdp* h, std::vector<Tree*>& trees) {
  RoundCtx& c = *round_ctx(h, 0);
  PP2D_TRY(round_stage1(h, c, trees));
  PP2D_TRY(round_stage2(h, c));
  return round_stage3(h, c);
}

void best_action(const Tree& t, uint8_t* a, float* r) {   // tree:510-524
  *a = 0;
  *r = -FLT_MAX;
  if (t.root < 0) return;
  for (int c : t.v[t.root].children)
    if (t.q[c].upper > *r) { *r = t.q[c].upper; *a = t.q[c].action; }
}

/* SearchTree::print (search_tree_cuda.cu:288-309, 452-473, 628-633) */
int64_t dump_tree(const Tree& t, float* out, uint64_t cap_nodes) {
  // pass 1: pre-order ids of the V nodes (V and Q nodes share one counter)
  std::vector<int> vid(t.v.size(), -1);
  struct Item { int idx; bool is_q; };
  std::vector<Item> order, stack{{t.root, false}};
  while (!stack.empty()) {
    const Item it = stack.back();
    stack.pop_back();
    if (!it.is_q) vid[it.idx] = (int)order.size();
    order.push_back(it);
    const std::vector<int>& ch = it.is_q ? t.q[it.idx].children : t.v[it.idx].children;
    for (size_t i = ch.size(); i-- > 0;) stack.push_back({ch[i], !it.is_q});
  }
  auto target = [&](int v) { return v >= 0 ? (float)vid[v] : -1.0f; };
  for (size_t k = 0; out && k < order.size() && k < cap_nodes; ++k) {
    float* o = out + 9 * k;
    if (order[k].is_q) {
      const QNodeH& q = t.q[order[k].idx];
      o[0] = 1.0f; o[1] = (float)q.action; o[2] = q.reward; o[3] = q.upper; o[4] = q.lower;
      o[5] = q.heuristic; o[6] = (float)q.depth; o[7] = (float)q.children.size();
      o[8] = target(q.to_expand);
    } else {
      const VNodeH& v = t.v[order[k].idx];
      o[0] = 0.0f; o[1] = (float)v.obs; o[2] = v.weight; o[3] = v.upper; o[4] = v.lower;
      o[5] = v.heuristic; o[6] = (float)v.depth; o[7] = (float)v.children.size();
      o[8] = target(v.to_expand);
    }
  }
  return (int64_t)order.size();
}

// The nodes SearchTree::update(a, z) keeps (search_tree_cuda.cu:548-555): the
// root's Q node for a, and its V child for z (-1: none, a new root is needed).
void kept_nodes(const Tree& t, uint8_t a, uint8_t z, int* root_q, int* root_v) {
  *root_q = *root_v = -1;
  for (int c : t.v[t.root].children)
    if (t.q[c].action == a) *root_q = c;
  if (*root_q < 0) return;
  for (int c : t.q[*root_q].children)
    if (t.v[c].obs == z) *root_v = c;
}

// The rest of SearchTree::update (search_tree_cuda.cu:556-626) once the new
// root's belief, if any, is resident: new_slot and its bounds ev when root_v
// is -1.  The beliefs of the dropped subtrees go to `freed`.
void reroot(Tree& t, int root_q, int root_v, int new_slot, const float* ev,
            std::vector<int>& freed) {
  for (int c : t.v[t.root].children)
    if (c != root_q) free_subtree_q(t, c, freed);
  for (int c : t.q[root_q].children)
    if (c != root_v) free_subtree_v(t, c, freed);
  VNodeH& old_root = t.v[t.root];
  if (old_root.slot >= 0) { freed.push_back(old_root.slot); old_root.slot = -1; }
  // Rebuild the node arrays from the kept subtree: a long-running planner
  // re-roots once per belief message, and dropped nodes must not accumulate.
  Tree fresh;
  fresh.goal = t.goal;
  fresh.rng = t.rng;
  fresh.expansions = t.expansions;
  fresh.dense = t.dense;
  if (root_v >= 0) {
    std::vector<int> vmap(t.v.size(), -1), qmap(t.q.size(), -1);
    struct Item { int idx; bool is_q; };
    std::vector<Item> stack{{root_v, false}};
    while (!stack.empty()) {                       // number the kept nodes
      const Item it = stack.back();
      stack.pop_back();
      if (it.is_q) {
        qmap[it.idx] = (int)fresh.q.size();
        fresh.q.push_back(t.q[it.idx]);
        for (int c : t.q[it.idx].children) stack.push_back({c, false});
      } else {
        vmap[it.idx] = (int)fresh.v.size();
        fresh.v.push_back(t.v[it.idx]);
        for (int c : t.v[it.idx].children) stack.push_back({c, true});
      }
    }
    auto mv = [&](int v) { return v >= 0 ? vmap[v] : -1; };
    for (VNodeH& v : fresh.v) {
      v.parent = v.parent >= 0 ? qmap[v.parent] : -1;
      v.to_expand = mv(v.to_expand);
      for (int& c : v.children) c = qmap[c];
    }
    for (QNodeH& q : fresh.q) {
      q.parent = vmap[q.parent];
      q.to_expand = mv(q.to_expand);
      for (int& c : q.children) c = vmap[c];
    }
    fresh.root = vmap[root_v];
    fresh.v[fresh.root].parent = -1;
  } else {
    fresh.v.emplace_back();
    fresh.root = 0;
    init_vnode(fresh.v[0], new_slot, 0, 0.0f, -1, ev, 0);
  }
  t = std::move(fresh);
}

// Belief slots a plan may hold: half of what is free once the current pool is
// counted as free (the pool must not ratchet up from call to call), or
// PP2D_POMDP_POOL_MB.
int pool_budget(pp2d_pomdp* h, size_t* max_slots) {
  size_t free_b = 0, total_b = 0;
  PP2D_CUDA(cudaMemGetInfo(&free_b, &total_b));
  size_t budget = (free_b + (size_t)h->cap * h->HW * sizeof(float)) / 2;
  const char* env = getenv("PP2D_POMDP_POOL_MB");
  if (env && *env) budget = (size_t)atol(env) << 20;
  *max_slots = budget / ((size_t)h->HW * sizeof(float));
  return PP2D_OK;
}

// Slots reserved up front per tree of a plan, of `worst` it may need.
// PP2D_POMDP_SLOTS_PER_QUERY: fewer; the pool then grows in place
// (pool_reserve) when the trees outgrow it.
size_t slots_per_tree(size_t worst) {
  const char* spq = getenv("PP2D_POMDP_SLOTS_PER_QUERY");
  if (spq && atol(spq) > 0) return std::min<size_t>(worst, (size_t)atol(spq));
  return worst;
}

// beliefCallback's loop (src/pomdp/path_planning_2d.cu:218-223) on every tree
// of `trees`: up to max_iter expansion rounds (<= 255) while its root is
// shallower than max_depth, the trees of a round batched.  `sorted`: `trees`
// is in the order of the roots' modes (see pp2d_pomdp_plan_batch).  The order
// and grouping change only how the work is batched: every tree owns its
// rand() stream, and no result of one tree depends on another.
int plan_trees(pp2d_pomdp* h, std::vector<Tree*>& trees, uint32_t max_depth, uint32_t max_iter,
               bool sorted) {
  const size_t n = trees.size();
  // Groups of trees a fraction of a round apart: while the device runs the
  // Bayes / bounds launches of one group, the host absorbs the previous round
  // of another and prepares its next one (all copies are asynchronous, each
  // group has its own streams).
  // (PP2D_POMDP_GROUPS overrides; measured at 1250 queries on a B200: 2 groups
  // 13.1e3 plans/s, 3 groups 14.4e3, 4 groups 13.1e3 -- more groups overlap
  // host and device better but launch smaller kernels)
  int G = n >= 384 ? 3 : (n >= 256 ? 2 : 1);
  if (const char* ge = getenv("PP2D_POMDP_GROUPS"))
    if (n >= 256 && atoi(ge) >= 1) G = std::min(atoi(ge), kMaxGroups);
  RoundCtx* ctx[kMaxGroups];
  bool more[kMaxGroups];
  size_t first_tree[kMaxGroups + 1];
  for (int g = 0; g < G; ++g) {
    ctx[g] = round_ctx(h, g);
    ctx[g]->n = 0;
    more[g] = true;
    first_tree[g] = n * (size_t)g / (size_t)G;
  }
  first_tree[G] = n;
  if (sorted && G > 1) {
    // Sorted trees are dealt to the groups in blocks of 16: every group then
    // spans the whole map (trees far from the goal grow more children than
    // those next to it; thirds of the sorted order would be unequal rounds)
    // while the neighbours inside a group stay neighbours.
    constexpr size_t kDeal = 16;
    std::vector<Tree*> dealt;
    dealt.reserve(n);
    for (int g = 0; g < G; ++g) {
      first_tree[g] = dealt.size();
      for (size_t b0 = (size_t)g * kDeal; b0 < n; b0 += (size_t)G * kDeal)
        for (size_t i = b0; i < std::min(n, b0 + kDeal); ++i) dealt.push_back(trees[i]);
    }
    trees.swap(dealt);
  }
  std::vector<Tree*> active;
  auto any_more = [&]() { for (int g = 0; g < G; ++g) if (more[g]) return true; return false; };
  for (uint32_t it = 0; it < max_iter && any_more(); ++it) {
    for (int g = 0; g < G; ++g) {
      if (!more[g]) continue;
      RoundCtx& c = *ctx[g];
      PP2D_TRY(round_stage3(h, c));            // previous round of this group
      active.clear();
      for (size_t i = first_tree[g]; i < first_tree[g + 1]; ++i) {
        Tree* t = trees[i];
        if (!t->dead && t->v[t->root].depth < max_depth) active.push_back(t);
      }
      if (active.empty()) { more[g] = false; continue; }
      PP2D_TRY(round_stage1(h, c, active));
      PP2D_TRY(round_stage2(h, c));
    }
  }
  for (int g = 0; g < G; ++g) PP2D_TRY(round_stage3(h, *ctx[g]));
  return PP2D_OK;
}

}  // namespace

extern "C" {

int pp2d_pomdp_create(uint32_t height, uint32_t width, const uint8_t* map,
                      uint32_t goal_x, uint32_t goal_y, float gamma,
                      pp2d_pomdp** out) {
  if (!out) return fail(PP2D_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (!map || height == 0 || width == 0) return fail(PP2D_ERR_INVALID, "empty map");
  if ((uint64_t)height * width > (1u << 26))
    return fail(PP2D_ERR_INVALID, "map too large for the POMDP path");
  if (goal_x >= width || goal_y >= height)
    return fail(PP2D_ERR_INVALID, "goal (%u %u) outside the %ux%u map", goal_x, goal_y,
                width, height);
  if (map[(size_t)goal_y * width + goal_x] > 0)   // pomdp path_planning_2d.cu:93-97
    return fail(PP2D_ERR_GOAL_OCCUPIED,
                "The assigned goal (%u %u) is at a occupied cell...", goal_x, goal_y);
  int dev_count = 0;
  PP2D_CUDA(cudaGetDeviceCount(&dev_count));
  if (dev_count == 0) return fail(PP2D_ERR_CUDA, "no CUDA device");
  int dev = 0;
  PP2D_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  PP2D_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10)
    return fail(PP2D_ERR_CUDA, "device %s is sm_%d%d; this library is sm_100a only",
                prop.name, prop.major, prop.minor);
  pp2d_pomdp* h = new (std::nothrow) pp2d_pomdp;
  if (!h) return fail(PP2D_ERR_INVALID, "out of host memory");
  h->H = (int)height; h->W = (int)width; h->HW = h->H * h->W;
  h->gx = (int)goal_x; h->gy = (int)goal_y; h->gamma = gamma;
  h->map_host.assign(map, map + (size_t)h->HW);
  h->goal_xy = {goal_x, goal_y};
  h->goal_alphas = {0};
  h->goal_finite = {1};
  int rc = [&]() -> int {
    const size_t n = (size_t)h->HW;
    PP2D_CUDA(cudaMalloc(&h->d_map, n));
    PP2D_CUDA(cudaMalloc(&h->d_tp, n * 81 * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&h->d_mp, n * 16 * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&h->d_sr, n * 9 * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&h->d_uniforms, 2 * kSamples * sizeof(float)));
    PP2D_CUDA(cudaMemcpy(h->d_map, map, n, cudaMemcpyHostToDevice));
    dim3 grid((h->W + 63) / 64, h->H);
    pomdp_model_kernel<<<grid, 64>>>(h->H, h->W, h->gx, h->gy, h->d_map, h->d_tp,
                                     h->d_mp, h->d_sr);
    count_launch();
    pomdp_uniforms_kernel<<<1, 64>>>(kSamples, h->d_uniforms);
    count_launch();
    PP2D_CUDA(cudaGetLastError());
    PP2D_CUDA(cudaDeviceSynchronize());
    const char* dense_env = getenv("PP2D_POMDP_DENSE");
    h->skip_dead = !(dense_env && atoi(dense_env) != 0);
    PP2D_CUDA(cudaMalloc(&h->d_work, sizeof(unsigned long long)));
    PP2D_CUDA(cudaMemset(h->d_work, 0, sizeof(unsigned long long)));
    const char* tile_env = getenv("PP2D_POMDP_TILE_SUPPORT");
    h->tile_support = !(tile_env && atoi(tile_env) == 0);
    const char* sort_env = getenv("PP2D_POMDP_SORT");
    h->sort_queries = !(sort_env && atoi(sort_env) == 0);
    return refresh_live_cells(h);
  }();
  if (rc != PP2D_OK) { pp2d_pomdp_destroy(h); return rc; }
  *out = h;
  return PP2D_OK;
}

void pp2d_pomdp_destroy(pp2d_pomdp* h) {
  if (!h) return;
  cudaFree(h->d_map); cudaFree(h->d_tp); cudaFree(h->d_mp); cudaFree(h->d_sr);
  cudaFree(h->d_uniforms); cudaFree(h->d_alpha); cudaFree(h->d_bel);
  cudaFree(h->d_kidx); cudaFree(h->d_kidx_all); cudaFree(h->d_alpha_live); cudaFree(h->d_dead);
  cudaFree(h->d_kinv); cudaFree(h->d_mp_live); cudaFree(h->d_work);
  if (h->pin_rows) cudaFreeHost(h->pin_rows);
  h->d_slots.release(); h->d_items.release(); h->d_prefix.release();
  h->d_draws.release(); h->d_vals.release(); h->d_rows.release();
  h->d_sums.release(); h->d_obs.release(); h->d_out.release(); h->d_keys.release();
  for (void*& c : h->round_ctx) { delete static_cast<RoundCtx*>(c); c = nullptr; }
  delete h;
}

int pp2d_pomdp_model_tables(pp2d_pomdp* h, float* trans_prob, float* meas_prob,
                            float* stage_reward) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  const size_t n = (size_t)h->HW;
  if (trans_prob)
    PP2D_CUDA(cudaMemcpy(trans_prob, h->d_tp, n * 81 * sizeof(float), cudaMemcpyDeviceToHost));
  if (meas_prob)
    PP2D_CUDA(cudaMemcpy(meas_prob, h->d_mp, n * 16 * sizeof(float), cudaMemcpyDeviceToHost));
  if (stage_reward)
    PP2D_CUDA(cudaMemcpy(stage_reward, h->d_sr, n * 9 * sizeof(float), cudaMemcpyDeviceToHost));
  return PP2D_OK;
}

int pp2d_pomdp_set_model_tables(pp2d_pomdp* h, const float* trans_prob,
                                const float* meas_prob, const float* stage_reward) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  const size_t n = (size_t)h->HW;
  // Trees keep beliefs that were propagated with the current tables (and were
  // classified against the current live-cell mask): like the reference, which
  // loads its tables once in initialize(), the tables are fixed before any tree.
  if (h->d_bel && h->free_slots.count() != (size_t)h->cap)
    return fail(PP2D_ERR_STATE, "pp2d_pomdp_set_model_tables: destroy the search trees of this "
                                "handle first (%zu beliefs are resident)",
                (size_t)h->cap - h->free_slots.count());
  // every stream that reads the tables (rounds of a batch in flight)
  PP2D_CUDA(cudaDeviceSynchronize());
  if (trans_prob)
    PP2D_CUDA(cudaMemcpy(h->d_tp, trans_prob, n * 81 * sizeof(float), cudaMemcpyHostToDevice));
  if (meas_prob)
    PP2D_CUDA(cudaMemcpy(h->d_mp, meas_prob, n * 16 * sizeof(float), cudaMemcpyHostToDevice));
  if (stage_reward)
    PP2D_CUDA(cudaMemcpy(h->d_sr, stage_reward, n * 9 * sizeof(float), cudaMemcpyHostToDevice));
  // the cells mass can enter are a property of the transition table
  return trans_prob ? refresh_live_cells(h) : PP2D_OK;
}

int pp2d_pomdp_sampling_uniforms(pp2d_pomdp* h, float* out100) {
  if (!h || !out100) return fail(PP2D_ERR_INVALID, "NULL argument");
  PP2D_CUDA(cudaMemcpy(out100, h->d_uniforms, 2 * kSamples * sizeof(float),
                       cudaMemcpyDeviceToHost));
  return PP2D_OK;
}

int pp2d_pomdp_set_alphas(pp2d_pomdp* h, const float* fib_alphas,
                          const uint8_t* fib_actions, const float* pbvi_alphas,
                          const uint8_t* pbvi_actions, uint32_t n_pbvi) {
  return pp2d_pomdp_set_goal_alphas(h, 0, fib_alphas, fib_actions, pbvi_alphas, pbvi_actions,
                                    n_pbvi);
}

int pp2d_pomdp_set_goal_alphas(pp2d_pomdp* h, uint32_t g, const float* fib_alphas,
                               const uint8_t* fib_actions, const float* pbvi_alphas,
                               const uint8_t* pbvi_actions, uint32_t n_pbvi) {
  if (!h || !fib_alphas) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (n_pbvi > 0 && !pbvi_alphas) return fail(PP2D_ERR_INVALID, "pbvi_alphas is NULL");
  if (g > (uint32_t)h->n_goals)
    return fail(PP2D_ERR_INVALID, "pp2d_pomdp_set_goal_alphas: goal %u of a set of %d", g,
                h->n_goals + 1);
  // All goals use one PBVI count (the bound matrices share ld and ncol).
  bool others = false;
  for (int j = 0; j <= h->n_goals; ++j) {
    if (j == (int)g || !h->goal_alphas[j]) continue;
    others = true;
    if ((uint32_t)h->n_pbvi != n_pbvi)
      return fail(PP2D_ERR_INVALID,
                  "goal %u: %u PBVI vectors, but goal %d holds %d (the goals of a handle share "
                  "one count)", g, n_pbvi, j, h->n_pbvi);
  }
  const int ncol = kColPbvi + (int)n_pbvi;
  const int ld = (ncol + kEvN - 1) / kEvN * kEvN;   // zero-padded to whole column tiles
  const size_t HW = (size_t)h->HW, goals = (size_t)h->n_goals + 1;
  // (a new ld only while no other goal holds bounds: their matrices are zero)
  if (!others && ld != h->ld) h->alpha_host.assign(goals * HW * ld, 0.0f);
  float* mat = h->alpha_host.data() + (size_t)g * HW * ld;
  bool finite = true;
  for (size_t s = 0; s < HW; ++s) {
    float* row = mat + s * ld;
    std::fill(row, row + ld, 0.0f);
    memcpy(row + kColFib, fib_alphas + s * 9, 9 * sizeof(float));
    for (uint32_t i = 0; i < n_pbvi; ++i) row[kColPbvi + i] = pbvi_alphas[(size_t)i * HW + s];
    for (int j = 0; j < ncol; ++j) finite = finite && std::isfinite(row[j]);
  }
  h->goal_alphas[g] = 1;
  h->goal_finite[g] = finite;
  // The exact skipping of zero belief entries (dead cells, per-tile inner rows)
  // needs 0 * alpha == 0, for every goal of a launch.
  h->alphas_finite = true;
  for (uint8_t f : h->goal_finite) h->alphas_finite = h->alphas_finite && f;
  if (h->d_alpha) cudaFree(h->d_alpha);
  h->d_alpha = nullptr;
  PP2D_CUDA(cudaMalloc(&h->d_alpha, h->alpha_host.size() * sizeof(float)));
  PP2D_CUDA(cudaMemcpy(h->d_alpha, h->alpha_host.data(), h->alpha_host.size() * sizeof(float),
                       cudaMemcpyHostToDevice));
  h->ld = ld; h->ncol = ncol; h->n_pbvi = (int)n_pbvi;
  PP2D_TRY(refresh_live_cells(h));
  if (g == 0) {
    h->fib_actions.assign(9, 0);
    for (int a = 0; a < 9; ++a) h->fib_actions[a] = fib_actions ? fib_actions[a] : (uint8_t)a;
    h->pbvi_actions.assign(n_pbvi, 0);
    if (pbvi_actions) memcpy(h->pbvi_actions.data(), pbvi_actions, n_pbvi);
    h->have_alphas = true;
  }
  return PP2D_OK;
}

int pp2d_pomdp_set_goals(pp2d_pomdp* h, const uint32_t* goals_xy, uint32_t n,
                         const float* stage_rewards) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  if (n > 0 && !goals_xy) return fail(PP2D_ERR_INVALID, "goals_xy is NULL");
  if (n > (1u << 20)) return fail(PP2D_ERR_INVALID, "pp2d_pomdp_set_goals: %u goals", n);
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t x = goals_xy[2 * (size_t)i], y = goals_xy[2 * (size_t)i + 1];
    if (x >= (uint32_t)h->W || y >= (uint32_t)h->H)
      return fail(PP2D_ERR_INVALID, "pp2d_pomdp_set_goals: goal %u (%u %u) outside the %dx%d map",
                  i + 1, x, y, h->W, h->H);
    if (h->map_host[(size_t)y * h->W + x] > 0)
      return fail(PP2D_ERR_GOAL_OCCUPIED,
                  "pp2d_pomdp_set_goals: goal %u (%u %u) is at an occupied cell", i + 1, x, y);
  }
  // as pp2d_pomdp_set_model_tables: trees hold rewards and bounds of their goals
  if (h->d_bel && h->free_slots.count() != (size_t)h->cap)
    return fail(PP2D_ERR_STATE, "pp2d_pomdp_set_goals: destroy the search trees of this "
                                "handle first (%zu beliefs are resident)",
                (size_t)h->cap - h->free_slots.count());
  PP2D_CUDA(cudaDeviceSynchronize());
  const size_t HW = (size_t)h->HW, tab = HW * 9;
  float* sr = nullptr;
  PP2D_CUDA(cudaMalloc(&sr, (n + 1) * tab * sizeof(float)));
  int rc = [&]() -> int {
    PP2D_CUDA(cudaMemcpy(sr, h->d_sr, tab * sizeof(float), cudaMemcpyDeviceToDevice));
    if (stage_rewards) {
      PP2D_CUDA(cudaMemcpy(sr + tab, stage_rewards, n * tab * sizeof(float),
                           cudaMemcpyHostToDevice));
      return PP2D_OK;
    }
    if (n == 0) return PP2D_OK;
    // the model rule of pp2d_pomdp_create per goal; its transition and
    // likelihood tables go to scratch (the handle's may have been replaced)
    float *tp = nullptr, *mp = nullptr;
    int r = [&]() -> int {
      PP2D_CUDA(cudaMalloc(&tp, HW * 81 * sizeof(float)));
      PP2D_CUDA(cudaMalloc(&mp, HW * 16 * sizeof(float)));
      dim3 grid((h->W + 63) / 64, h->H);
      for (uint32_t i = 0; i < n; ++i) {
        pomdp_model_kernel<<<grid, 64>>>(h->H, h->W, (int)goals_xy[2 * (size_t)i],
                                         (int)goals_xy[2 * (size_t)i + 1], h->d_map, tp, mp,
                                         sr + (i + 1) * tab);
        count_launch();
      }
      PP2D_CUDA(cudaGetLastError());
      PP2D_CUDA(cudaDeviceSynchronize());
      return PP2D_OK;
    }();
    cudaFree(tp);
    cudaFree(mp);
    return r;
  }();
  if (rc != PP2D_OK) { cudaFree(sr); return rc; }
  cudaFree(h->d_sr);
  h->d_sr = sr;
  h->n_goals = (int)n;
  h->goal_xy.assign({(uint32_t)h->gx, (uint32_t)h->gy});
  if (n) h->goal_xy.insert(h->goal_xy.end(), goals_xy, goals_xy + 2 * (size_t)n);
  h->goal_alphas.resize(n + 1);
  h->goal_finite.resize(n + 1);
  std::fill(h->goal_alphas.begin() + 1, h->goal_alphas.end(), 0);
  std::fill(h->goal_finite.begin() + 1, h->goal_finite.end(), 1);
  h->alphas_finite = h->goal_finite[0];
  if (h->ld == 0) return PP2D_OK;                  // no goal has alpha vectors
  // goal 0's bounds stay, the new goals have none (zero matrices)
  h->alpha_host.resize((n + 1) * HW * h->ld);
  std::fill(h->alpha_host.begin() + HW * h->ld, h->alpha_host.end(), 0.0f);
  if (h->d_alpha) cudaFree(h->d_alpha);
  h->d_alpha = nullptr;
  PP2D_CUDA(cudaMalloc(&h->d_alpha, h->alpha_host.size() * sizeof(float)));
  PP2D_CUDA(cudaMemcpy(h->d_alpha, h->alpha_host.data(), h->alpha_host.size() * sizeof(float),
                       cudaMemcpyHostToDevice));
  return refresh_live_cells(h);
}

int pp2d_pomdp_goals(pp2d_pomdp* h, uint32_t* count, uint32_t* goals_xy) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  if (count) *count = (uint32_t)h->n_goals + 1;
  if (goals_xy) memcpy(goals_xy, h->goal_xy.data(), h->goal_xy.size() * sizeof(uint32_t));
  return PP2D_OK;
}

int pp2d_pomdp_goal_reward(pp2d_pomdp* h, uint32_t g, float* stage_reward) {
  if (!h || !stage_reward) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (g > (uint32_t)h->n_goals)
    return fail(PP2D_ERR_INVALID, "pp2d_pomdp_goal_reward: goal %u of a set of %d", g,
                h->n_goals + 1);
  const size_t tab = (size_t)h->HW * 9;
  PP2D_CUDA(cudaMemcpy(stage_reward, h->d_sr + g * tab, tab * sizeof(float),
                       cudaMemcpyDeviceToHost));
  return PP2D_OK;
}

int pp2d_pomdp_solve_fib(pp2d_pomdp* h, float* alphas, uint8_t* actions,
                         uint32_t* sweeps_out, uint32_t max_sweeps) {
  if (!h || !alphas) return fail(PP2D_ERR_INVALID, "NULL argument");
  // The stopping rule is reached in useful time only for a contraction: with
  // |gamma| >= 1 the change per sweep stays around the rewards (or the values
  // reach -inf, whose NaN differences the inf-norm drops).
  if (max_sweeps == 0 && !(fabsf(h->gamma) < 1.0f))
    return fail(PP2D_ERR_INVALID,
                "pp2d_pomdp_solve_fib: without a sweep cap the stopping rule needs |gamma| < 1 "
                "(gamma = %g); pass max_sweeps", (double)h->gamma);
  const size_t n = (size_t)h->HW * 9;
  float *a1 = nullptr, *a2 = nullptr, *prev = nullptr;
  unsigned int* d_res = nullptr;
  int rc = [&]() -> int {
    PP2D_CUDA(cudaMalloc(&a1, n * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&a2, n * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&prev, n * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&d_res, sizeof(unsigned int)));
    PP2D_CUDA(cudaMemsetAsync(a1, 0, n * sizeof(float), h->stream));
    PP2D_CUDA(cudaMemsetAsync(a2, 0, n * sizeof(float), h->stream));
    PP2D_CUDA(cudaMemsetAsync(prev, 0, n * sizeof(float), h->stream));
    const int blocks = (int)((n + 127) / 128);
    uint32_t total = 0;
    float inf_norm = 0.0f;
    do {                                  // fast_informed_bound_cuda.cu:223-262
      for (int i = 0; i < 5; ++i) {
        pomdp_fib_kernel<<<blocks, 128, 0, h->stream>>>(h->H, h->W, h->gamma, h->d_tp,
                                                        h->d_mp, h->d_sr, a1, a2);
        count_launch();
        pomdp_fib_kernel<<<blocks, 128, 0, h->stream>>>(h->H, h->W, h->gamma, h->d_tp,
                                                        h->d_mp, h->d_sr, a2, a1);
        count_launch();
      }
      total += 10;
      PP2D_CUDA(cudaMemsetAsync(d_res, 0, sizeof(unsigned int), h->stream));
      pomdp_maxdiff_kernel<<<64, 256, 0, h->stream>>>(a1, prev, n, d_res);
      count_launch();
      PP2D_CUDA(cudaGetLastError());
      unsigned int bits = 0;
      PP2D_CUDA(cudaMemcpyAsync(&bits, d_res, sizeof(bits), cudaMemcpyDeviceToHost, h->stream));
      PP2D_CUDA(cudaStreamSynchronize(h->stream));
      memcpy(&inf_norm, &bits, sizeof(float));
    } while (inf_norm > 0.01f && (max_sweeps == 0 || total < max_sweeps));
    PP2D_CUDA(cudaMemcpy(alphas, a1, n * sizeof(float), cudaMemcpyDeviceToHost));
    if (actions) for (int a = 0; a < 9; ++a) actions[a] = (uint8_t)a;  // fib:75-77
    if (sweeps_out) *sweeps_out = total;
    return PP2D_OK;
  }();
  cudaFree(a1); cudaFree(a2); cudaFree(prev); cudaFree(d_res);
  return rc;
}

int pp2d_pomdp_live_cells(pp2d_pomdp* h, uint8_t* mask, uint32_t* count) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  uint32_t n = 0;
  for (int s = 0; s < h->HW; ++s) {
    const uint8_t live = h->dead[s] ? 0 : 1;
    n += live;
    if (mask) mask[s] = live;
  }
  if (count) *count = n;
  return PP2D_OK;
}

int pp2d_pomdp_work_counters(pp2d_pomdp* h, uint64_t out[3]) {
  if (!h || !out) return fail(PP2D_ERR_INVALID, "NULL argument");
  unsigned long long dev = 0;
  PP2D_CUDA(cudaDeviceSynchronize());
  PP2D_CUDA(cudaMemcpy(&dev, h->d_work, sizeof(dev), cudaMemcpyDeviceToHost));
  out[0] = h->n_vnodes;
  out[1] = h->n_bayes;
  out[2] = h->work_rows + (uint64_t)dev;
  return PP2D_OK;
}

int pp2d_pomdp_padding_counters(pp2d_pomdp* h, uint64_t out[2]) {
  if (!h || !out) return fail(PP2D_ERR_INVALID, "NULL argument");
  out[0] = h->pad_entries;
  out[1] = h->pad_rows;
  return PP2D_OK;
}

void pp2d_set_host_threads(int n) { g_host_threads.store(n > 0 ? n : 0); }

int pp2d_pomdp_reserve(pp2d_pomdp* h, uint32_t n_beliefs) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  return pool_reserve(h, n_beliefs);
}

int pp2d_pomdp_bayes_update(pp2d_pomdp* h, const float* beliefs_in, uint32_t n,
                            const uint8_t* actions, const uint8_t* observations,
                            int normalize, float* beliefs_out, float* sums) {
  if (!h || !beliefs_in || !actions || !observations || !beliefs_out)
    return fail(PP2D_ERR_INVALID, "NULL argument");
  if (n == 0) return PP2D_OK;
  for (uint32_t i = 0; i < n; ++i)
    if (actions[i] >= kActions || observations[i] >= 16)
      return fail(PP2D_ERR_INVALID, "item %u: action %u / observation %u out of range (9 / 16)",
                  i, actions[i], observations[i]);
  PP2D_TRY(pool_reserve(h, (size_t)h->cap - h->free_slots.count() + 2 * (size_t)n));
  const int HW = h->HW;
  std::vector<int> in(n), outs(n);
  std::vector<BayesItem> items(n);
  for (uint32_t i = 0; i < n; ++i) {
    PP2D_TRY(alloc_slot(h, &in[i]));
    PP2D_TRY(alloc_slot(h, &outs[i]));
    items[i] = BayesItem{in[i], outs[i], actions[i], observations[i]};
  }
  int rc = [&]() -> int {
    PP2D_TRY(h->d_slots.ensure(n));
    PP2D_TRY(h->d_rows.ensure((size_t)n * HW));
    PP2D_TRY(h->d_items.ensure(n));
    PP2D_TRY(h->d_sums.ensure(n));
    PP2D_CUDA(cudaMemcpyAsync(h->d_rows.p, beliefs_in, (size_t)n * HW * sizeof(float),
                              cudaMemcpyHostToDevice, h->stream));
    PP2D_CUDA(cudaMemcpyAsync(h->d_slots.p, in.data(), n * sizeof(int),
                              cudaMemcpyHostToDevice, h->stream));
    dim3 grid((HW + 255) / 256, n);
    pomdp_scatter_kernel<<<grid, 256, 0, h->stream>>>(HW, h->d_slots.p, n,
                                                      h->d_rows.p, h->d_bel);
    count_launch();
    PP2D_CUDA(cudaMemcpyAsync(h->d_items.p, items.data(), n * sizeof(BayesItem),
                              cudaMemcpyHostToDevice, h->stream));
    dim3 bgrid((n + 31) / 32, (HW + 7) / 8);
    pomdp_bayes_kernel<<<bgrid, 256, 0, h->stream>>>(h->H, h->W, h->d_tp, h->d_mp,
                                                     h->d_items.p, n, h->d_bel, h->d_bel);
    count_launch();
    h->n_bayes += n;
    PP2D_CUDA(cudaMemcpyAsync(h->d_slots.p, outs.data(), n * sizeof(int),
                              cudaMemcpyHostToDevice, h->stream));
    if (normalize) PP2D_TRY(normalize_slots(h, (int)n, nullptr));
    pomdp_gather_kernel<<<grid, 256, 0, h->stream>>>(HW, h->d_slots.p, n, h->d_bel,
                                                     h->d_rows.p);
    count_launch();
    PP2D_CUDA(cudaGetLastError());
    PP2D_CUDA(cudaMemcpyAsync(beliefs_out, h->d_rows.p, (size_t)n * HW * sizeof(float),
                              cudaMemcpyDeviceToHost, h->stream));
    if (sums && normalize)
      PP2D_CUDA(cudaMemcpyAsync(sums, h->d_sums.p, n * sizeof(float),
                                cudaMemcpyDeviceToHost, h->stream));
    PP2D_CUDA(cudaStreamSynchronize(h->stream));
    return PP2D_OK;
  }();
  for (uint32_t i = 0; i < n; ++i) {
    h->free_slots.put(in[i]);
    h->free_slots.put(outs[i]);
  }
  return rc;
}

int pp2d_pomdp_evaluate(pp2d_pomdp* h, const float* beliefs, uint32_t n,
                        float* upper, uint8_t* upper_action, float* lower,
                        uint8_t* lower_action) {
  if (!h || !beliefs) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (!h->have_alphas) return fail(PP2D_ERR_STATE, "pp2d_pomdp_set_alphas not called");
  if (n == 0) return PP2D_OK;
  PP2D_TRY(pool_reserve(h, (size_t)h->cap - h->free_slots.count() + n));
  const int HW = h->HW;
  std::vector<int> slots(n);
  for (uint32_t i = 0; i < n; ++i) PP2D_TRY(alloc_slot(h, &slots[i]));
  int rc = [&]() -> int {
    PP2D_TRY(h->d_slots.ensure(n));
    PP2D_TRY(h->d_rows.ensure((size_t)n * HW));
    PP2D_TRY(h->d_vals.ensure((size_t)n * h->ncol));
    PP2D_TRY(h->d_out.ensure((size_t)n * 4));
    PP2D_CUDA(cudaMemcpyAsync(h->d_rows.p, beliefs, (size_t)n * HW * sizeof(float),
                              cudaMemcpyHostToDevice, h->stream));
    PP2D_CUDA(cudaMemcpyAsync(h->d_slots.p, slots.data(), n * sizeof(int),
                              cudaMemcpyHostToDevice, h->stream));
    dim3 grid((HW + 255) / 256, n);
    pomdp_scatter_kernel<<<grid, 256, 0, h->stream>>>(HW, h->d_slots.p, n,
                                                      h->d_rows.p, h->d_bel);
    count_launch();
    dim3 vgrid((n + kEvM - 1) / kEvM, (h->ncol + kEvN - 1) / kEvN);
    bool dense = false;
    for (uint32_t i = 0; i < n && !dense; ++i)
      dense = !zero_on_dead_cells(h, beliefs + (size_t)i * HW);
    const InnerDim in = inner_dim(h, dense);
    pomdp_values_kernel<false><<<vgrid, 256, 0, h->stream>>>(in.K, in.kidx, h->HW, h->ld,
                                                             h->ncol, h->d_slots.p, n, h->d_bel,
                                                             in.alpha, h->d_vals.p, nullptr,
                                                             nullptr, nullptr, 0, nullptr, 0);
    h->work_rows += (uint64_t)in.K * (uint64_t)n;
    count_launch();
    pomdp_bounds_kernel<<<(n + 3) / 4, 128, 0, h->stream>>>(n, h->ncol, h->n_pbvi,
                                                                h->d_vals.p, h->d_out.p);
    count_launch();
    PP2D_CUDA(cudaGetLastError());
    std::vector<float> hres((size_t)n * 4);
    PP2D_CUDA(cudaMemcpyAsync(hres.data(), h->d_out.p, hres.size() * sizeof(float),
                              cudaMemcpyDeviceToHost, h->stream));
    PP2D_CUDA(cudaStreamSynchronize(h->stream));
    for (uint32_t i = 0; i < n; ++i) {
      int packed;
      memcpy(&packed, &hres[(size_t)i * 4 + 2], sizeof(int));
      if (upper) upper[i] = hres[(size_t)i * 4];
      if (lower) lower[i] = hres[(size_t)i * 4 + 1];
      if (upper_action) upper_action[i] = h->fib_actions[packed & 0xff];
      if (lower_action) lower_action[i] = h->n_pbvi ? h->pbvi_actions[packed >> 8] : 0;
    }
    return PP2D_OK;
  }();
  for (uint32_t i = 0; i < n; ++i) h->free_slots.put(slots[i]);
  return rc;
}

int pp2d_pomdp_plan_batch(pp2d_pomdp* h, const float* beliefs, uint32_t n,
                          uint32_t max_depth, uint32_t max_iter, uint8_t* actions,
                          float* values, uint32_t* stats) {
  if (!h || !beliefs || !actions) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (!h->have_alphas) return fail(PP2D_ERR_STATE, "pp2d_pomdp_set_alphas not called");
  if (n == 0) return PP2D_OK;
  if (max_iter > 255) max_iter = 255;           // uint8_t counter, pomdp:218-223
  // Worst case per query: root + max_iter * 9 * 16 children.
  const size_t per_query = slots_per_tree(1 + (size_t)max_iter * kActions * 16);
  size_t max_slots = 0;
  PP2D_TRY(pool_budget(h, &max_slots));
  if (max_slots < per_query)
    return fail(PP2D_ERR_STATE, "belief pool budget too small for one query");
  size_t group = std::min<size_t>(n, max_slots / per_query);
  if ((size_t)h->cap < group * per_query) PP2D_TRY(pool_reserve(h, group * per_query));
  group = std::min<size_t>(n, (size_t)h->cap / per_query);
  for (size_t g0 = 0; g0 < n; g0 += group) {
    const size_t gn = std::min<size_t>(group, n - g0);
    std::vector<Tree> store(gn);
    std::vector<Tree*> trees(gn);
    double tr = now_s();
    for (size_t i = 0; i < gn; ++i) { store[i].rng.seed(1); trees[i] = &store[i]; }
    const bool sorted = h->sort_queries && gn >= 2 * (size_t)kEvM;
    std::vector<uint32_t> key(sorted ? gn : 0);
    PP2D_TRY(make_roots(h, trees, beliefs + g0 * (size_t)h->HW, sorted ? key.data() : nullptr));
    // The trees are planned in the order of their start beliefs' modes (column,
    // then row): neighbours in that order have overlapping supports, which is
    // what makes the per-tile inner rows of the values launches short
    // (pomdp_support_flags_kernel).  Only the order of the work changes: every query
    // owns its rand() stream and its results land at its own index.
    if (sorted) {
      std::vector<int> order(gn);
      for (size_t i = 0; i < gn; ++i) order[i] = (int)i;
      std::stable_sort(order.begin(), order.end(),
                       [&](int a, int b) { return key[a] < key[b]; });
      for (size_t i = 0; i < gn; ++i) trees[i] = &store[order[i]];
    }
    h->t_phase[5] += now_s() - tr;               // roots: upload + bounds
    PP2D_TRY(plan_trees(h, trees, max_depth, max_iter, sorted));
    tr = now_s();
    const int gni = (int)gn;
#pragma omp parallel num_threads(host_threads()) if (gni >= 64)
    {
      std::vector<int> back;                       // belief slots of this thread's trees
#pragma omp for schedule(static) nowait
      for (int i = 0; i < gni; ++i) {
        float r;
        best_action(store[i], &actions[g0 + i], &r);
        if (values) values[g0 + i] = r;
        if (stats) {
          stats[(g0 + i) * 4 + 0] = (uint32_t)store[i].v.size();
          stats[(g0 + i) * 4 + 1] = (uint32_t)store[i].q.size();
          stats[(g0 + i) * 4 + 2] = store[i].v[store[i].root].depth;
          stats[(g0 + i) * 4 + 3] = store[i].expansions;
        }
        for (VNodeH& v : store[i].v)               // every node still holding a belief
          if (v.slot >= 0) { back.push_back(v.slot); v.slot = -1; }
      }
#pragma omp critical
      give_back(h, back);
    }
    h->t_phase[6] += now_s() - tr;               // actions out, slots back
  }
  if (getenv("PP2D_POMDP_PROFILE")) {
    fprintf(stderr, "pp2d pomdp host phases [s]: draws+enqueue %.4f  wait(sampling) %.4f  "
            "kids+enqueue %.4f  wait(bayes..bounds) %.4f  bookkeeping %.4f  roots %.4f  "
            "finish %.4f\n",
            h->t_phase[0], h->t_phase[1], h->t_phase[2], h->t_phase[3], h->t_phase[4],
            h->t_phase[5], h->t_phase[6]);
    for (double& t : h->t_phase) t = 0;
  }
  return PP2D_OK;
}

/* ---- single-query tree: SearchTree of search_tree.h:130-165 ------------- */
int pp2d_tree_create(pp2d_pomdp* h, const float* belief, pp2d_tree** out) {
  if (!h || !belief || !out) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (!h->have_alphas) return fail(PP2D_ERR_STATE, "pp2d_pomdp_set_alphas not called");
  *out = nullptr;
  if (h->cap == 0) PP2D_TRY(pool_reserve(h, 4096));
  pp2d_tree* t = new (std::nothrow) pp2d_tree;
  if (!t) return fail(PP2D_ERR_INVALID, "out of host memory");
  t->h = h;
  t->t.rng.seed(1);
  std::vector<Tree*> trees{&t->t};
  int rc = make_roots(h, trees, belief);
  if (rc != PP2D_OK) { delete t; return rc; }
  *out = t;
  return PP2D_OK;
}

void pp2d_tree_destroy(pp2d_tree* t) {
  if (!t) return;
  std::vector<int> freed;
  if (t->t.root >= 0) free_subtree_v(t->t, t->t.root, freed);
  give_back(t->h, freed);
  delete t;
}

int pp2d_tree_expand(pp2d_tree* t) {
  if (!t) return fail(PP2D_ERR_INVALID, "tree is NULL");
  if (t->t.dead || t->t.v[t->t.root].to_expand < 0)
    return fail(PP2D_ERR_STATE, "no V node to expand (the reference dereferences nullptr here)");
  std::vector<Tree*> trees{&t->t};
  return expand_round(t->h, trees);
}

uint32_t pp2d_tree_depth(const pp2d_tree* t) { return t ? t->t.v[t->t.root].depth : 0; }

int pp2d_tree_best_action(const pp2d_tree* t, uint8_t* action, float* value) {
  if (!t || !action) return fail(PP2D_ERR_INVALID, "NULL argument");
  float r;
  best_action(t->t, action, &r);
  if (value) *value = r;
  return PP2D_OK;
}

int pp2d_tree_root_bounds(const pp2d_tree* t, float* upper, float* lower) {
  if (!t) return fail(PP2D_ERR_INVALID, "tree is NULL");
  if (upper) *upper = t->t.v[t->t.root].upper;
  if (lower) *lower = t->t.v[t->t.root].lower;
  return PP2D_OK;
}

int64_t pp2d_tree_dump(const pp2d_tree* tt, float* out, uint64_t cap_nodes) {
  if (!tt || tt->t.root < 0) { fail(PP2D_ERR_INVALID, "tree is NULL"); return -1; }
  return dump_tree(tt->t, out, cap_nodes);
}

/* SearchTree::update(a, z), search_tree_cuda.cu:548-626 */
int pp2d_tree_update(pp2d_tree* tt, uint8_t a, uint8_t z) {
  if (!tt) return fail(PP2D_ERR_INVALID, "tree is NULL");
  if (a >= kActions || z >= 16)
    return fail(PP2D_ERR_INVALID, "action %u / observation %u out of range (9 / 16)", a, z);
  pp2d_pomdp* h = tt->h;
  Tree& t = tt->t;
  if (t.v[t.root].children.empty())
    return fail(PP2D_ERR_STATE, "update() on an unexpanded root (nullptr in the reference)");
  // Nothing is freed before the arguments are known to be usable.
  int root_q = -1, root_v = -1;
  kept_nodes(t, a, z, &root_q, &root_v);
  if (root_q < 0) return fail(PP2D_ERR_INVALID, "no Q node for action %u", a);
  int new_slot = -1;
  float ev[4] = {0, 0, 0, 0};
  if (root_v < 0) {
    // new root from one Bayes update of the old root belief (tree:586-614)
    PP2D_TRY(alloc_slot(h, &new_slot));
    int rc = [&]() -> int {
      BayesItem it{t.v[t.root].slot, new_slot, a, z};
      PP2D_TRY(h->d_items.ensure(1));
      PP2D_TRY(h->d_slots.ensure(1));
      PP2D_CUDA(cudaMemcpyAsync(h->d_items.p, &it, sizeof(it), cudaMemcpyHostToDevice, h->stream));
      dim3 bgrid(1, (h->HW + 7) / 8);
      pomdp_bayes_kernel<<<bgrid, 256, 0, h->stream>>>(h->H, h->W, h->d_tp, h->d_mp,
                                                       h->d_items.p, 1, h->d_bel, h->d_bel);
      count_launch();
      h->n_bayes++;
      PP2D_CUDA(cudaMemcpyAsync(h->d_slots.p, &new_slot, sizeof(int), cudaMemcpyHostToDevice,
                                h->stream));
      PP2D_TRY(normalize_slots(h, 1, nullptr));
      std::vector<int> s1{new_slot};
      return evaluate_slots(h, s1, nullptr, ev, t.dense);
    }();
    if (rc != PP2D_OK) { h->free_slots.put(new_slot); return rc; }
    h->n_vnodes++;
  }
  std::vector<int> freed;
  reroot(t, root_q, root_v, new_slot, ev, freed);
  give_back(h, freed);
  return PP2D_OK;
}

int pp2d_tree_plan(pp2d_tree* t, uint32_t max_depth, uint32_t max_iter,
                   uint8_t* action, float* value) {
  if (!t || !action) return fail(PP2D_ERR_INVALID, "NULL argument");
  uint8_t counter = 0;                          // pomdp path_planning_2d.cu:218-223
  while (pp2d_tree_depth(t) < max_depth && counter++ < max_iter) {
    if (t->t.v[t->t.root].to_expand < 0) break;
    PP2D_TRY(pp2d_tree_expand(t));
  }
  return pp2d_tree_best_action(t, action, value);
}

}  // extern "C"

/* ---- persistent tree batches: many SearchTrees planned together ---------- */
struct pp2d_tree_batch {
  pp2d_pomdp* h = nullptr;
  std::vector<Tree> trees;
};

namespace {

// A list of tree indices of a call: every entry < count, none twice.
int check_tree_list(const pp2d_tree_batch* b, const uint32_t* trees, uint32_t n,
                    const char* fn) {
  std::vector<uint8_t> seen(b->trees.size(), 0);
  for (uint32_t i = 0; i < n; ++i) {
    if (trees[i] >= b->trees.size())
      return fail(PP2D_ERR_INVALID, "%s: entry %u names tree %u of a batch of %zu", fn, i,
                  trees[i], b->trees.size());
    if (seen[trees[i]]++)
      return fail(PP2D_ERR_INVALID, "%s: tree %u is listed twice", fn, trees[i]);
  }
  return PP2D_OK;
}

// Sort keys of the listed roots (pomdp_root_mode_kernel), read from the pool.
int root_mode_keys(pp2d_pomdp* h, const std::vector<Tree*>& trees, std::vector<uint32_t>& key) {
  const int n = (int)trees.size();
  std::vector<int> slots(n);
  for (int i = 0; i < n; ++i) slots[i] = trees[i]->v[trees[i]->root].slot;
  PP2D_TRY(h->d_slots.ensure(n));
  PP2D_TRY(h->d_keys.ensure(n));
  PP2D_CUDA(cudaMemcpyAsync(h->d_slots.p, slots.data(), n * sizeof(int), cudaMemcpyHostToDevice,
                            h->stream));
  pomdp_root_mode_kernel<<<(n + 3) / 4, 128, 0, h->stream>>>(h->H, h->W, h->d_slots.p, n,
                                                             h->d_bel, h->d_keys.p);
  count_launch();
  PP2D_CUDA(cudaGetLastError());
  key.resize(n);
  PP2D_CUDA(cudaMemcpyAsync(key.data(), h->d_keys.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                            h->stream));
  PP2D_CUDA(cudaStreamSynchronize(h->stream));
  return PP2D_OK;
}

}  // namespace

extern "C" {

int pp2d_tree_batch_create(pp2d_pomdp* h, const float* beliefs, uint32_t n,
                           pp2d_tree_batch** out) {
  return pp2d_tree_batch_create_goals(h, beliefs, nullptr, n, out);
}

int pp2d_tree_batch_create_goals(pp2d_pomdp* h, const float* beliefs, const uint32_t* goals,
                                 uint32_t n, pp2d_tree_batch** out) {
  if (!h || !beliefs || !out) return fail(PP2D_ERR_INVALID, "NULL argument");
  *out = nullptr;
  if (!goals && !h->have_alphas) return fail(PP2D_ERR_STATE, "pp2d_pomdp_set_alphas not called");
  for (uint32_t k = 0; goals && k < n; ++k)
    if (goals[k] > (uint32_t)h->n_goals)
      return fail(PP2D_ERR_INVALID, "pp2d_tree_batch_create_goals: tree %u names goal %u of a "
                                    "set of %d", k, goals[k], h->n_goals + 1);
  for (uint32_t k = 0; goals && k < n; ++k)
    if (!h->goal_alphas[goals[k]])
      return fail(PP2D_ERR_STATE, "pp2d_tree_batch_create_goals: tree %u: goal %u has no alpha "
                                  "vectors", k, goals[k]);
  pp2d_tree_batch* b = new (std::nothrow) pp2d_tree_batch;
  if (!b) return fail(PP2D_ERR_INVALID, "out of host memory");
  b->h = h;
  int rc = [&]() -> int {
    b->trees.resize(n);
    std::vector<Tree*> trees(n);
    for (uint32_t i = 0; i < n; ++i) {
      b->trees[i].rng.seed(1);
      b->trees[i].goal = goals ? (int)goals[i] : 0;
      trees[i] = &b->trees[i];
    }
    if (n == 0) return PP2D_OK;
    PP2D_TRY(pool_reserve(h, (size_t)h->cap - h->free_slots.count() + n));
    return make_roots(h, trees, beliefs);
  }();
  if (rc != PP2D_OK) { pp2d_tree_batch_destroy(b); return rc; }
  *out = b;
  return PP2D_OK;
}

void pp2d_tree_batch_destroy(pp2d_tree_batch* b) {
  if (!b) return;
  std::vector<int> freed;
  for (Tree& t : b->trees)
    if (t.root >= 0) free_subtree_v(t, t.root, freed);
  give_back(b->h, freed);
  delete b;
}

int pp2d_tree_batch_update(pp2d_tree_batch* b, const uint32_t* trees, uint32_t n,
                           const uint8_t* actions, const uint8_t* observations) {
  if (!b) return fail(PP2D_ERR_INVALID, "batch is NULL");
  if (n == 0) return PP2D_OK;
  if (!trees || !actions || !observations) return fail(PP2D_ERR_INVALID, "NULL argument");
  PP2D_TRY(check_tree_list(b, trees, n, "pp2d_tree_batch_update"));
  pp2d_pomdp* h = b->h;
  std::vector<int> rq(n), rv(n);
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t k = trees[i];
    if (actions[i] >= kActions || observations[i] >= 16)
      return fail(PP2D_ERR_INVALID, "tree %u: action %u / observation %u out of range (9 / 16)",
                  k, actions[i], observations[i]);
    const Tree& t = b->trees[k];
    if (t.v[t.root].children.empty())
      return fail(PP2D_ERR_STATE, "tree %u: update() on an unexpanded root (nullptr in the "
                                  "reference)", k);
    kept_nodes(t, actions[i], observations[i], &rq[i], &rv[i]);
    if (rq[i] < 0) return fail(PP2D_ERR_INVALID, "tree %u: no Q node for action %u", k, actions[i]);
  }
  // Misses (an observation without a child): one Bayes update of the old root
  // each (tree:586-614), all in one set of launches.
  std::vector<uint32_t> miss;
  for (uint32_t i = 0; i < n; ++i)
    if (rv[i] < 0) miss.push_back(i);
  const size_t nm = miss.size();
  std::vector<int> slots(nm, -1);
  std::vector<float> ev(nm * 4, 0.0f);
  if (nm) {
    PP2D_TRY(pool_reserve(h, (size_t)h->cap - h->free_slots.count() + nm));
    std::vector<BayesItem> items(nm);
    std::vector<int> goals(nm);
    bool dense = false;
    for (size_t j = 0; j < nm; ++j) {
      const uint32_t i = miss[j];
      const Tree& t = b->trees[trees[i]];
      PP2D_TRY(alloc_slot(h, &slots[j]));            // (reserved: cannot fail)
      items[j] = BayesItem{t.v[t.root].slot, slots[j], actions[i], observations[i]};
      goals[j] = t.goal;
      dense = dense || t.dense;
    }
    int rc = [&]() -> int {
      PP2D_TRY(launch_bayes(h, items));
      PP2D_TRY(launch_normalize(h, slots));
      return evaluate_slots(h, slots, goals.data(), ev.data(), dense);
    }();
    if (rc != PP2D_OK) {
      for (int s : slots) h->free_slots.put(s);
      return rc;
    }
    h->n_vnodes += nm;
  }
  std::vector<int> slot_of(n, -1);
  std::vector<const float*> ev_of(n, nullptr);
  for (size_t j = 0; j < nm; ++j) { slot_of[miss[j]] = slots[j]; ev_of[miss[j]] = &ev[4 * j]; }
  const int ni = (int)n;
#pragma omp parallel num_threads(host_threads()) if (ni >= 64)
  {
    std::vector<int> freed;
#pragma omp for schedule(dynamic, 8) nowait
    for (int i = 0; i < ni; ++i)
      reroot(b->trees[trees[i]], rq[i], rv[i], slot_of[i], ev_of[i], freed);
#pragma omp critical
    give_back(h, freed);
  }
  return PP2D_OK;
}

int pp2d_tree_batch_plan(pp2d_tree_batch* b, const uint32_t* trees, uint32_t n,
                         uint32_t max_depth, uint32_t max_iter, uint8_t* actions, float* values,
                         uint32_t* stats) {
  if (!b) return fail(PP2D_ERR_INVALID, "batch is NULL");
  if (n == 0) return PP2D_OK;
  if (!trees || !actions) return fail(PP2D_ERR_INVALID, "NULL argument");
  PP2D_TRY(check_tree_list(b, trees, n, "pp2d_tree_batch_plan"));
  pp2d_pomdp* h = b->h;
  if (max_iter > 255) max_iter = 255;           // as pp2d_pomdp_plan_batch
  // live beliefs + the worst case of every listed tree (9 * 16 children per
  // expansion), within the budget of pp2d_pomdp_plan_batch; past it the pool
  // grows in place
  const size_t live = (size_t)h->cap - h->free_slots.count();
  size_t max_slots = 0;
  PP2D_TRY(pool_budget(h, &max_slots));
  const size_t want =
      std::min(live + (size_t)n * slots_per_tree((size_t)max_iter * kActions * 16),
               std::max(max_slots, live + n));
  if ((size_t)h->cap < want) PP2D_TRY(pool_reserve(h, want));
  std::vector<Tree*> list(n);
  for (uint32_t i = 0; i < n; ++i) list[i] = &b->trees[trees[i]];
  // goal by goal (a values tile holds children of one goal, DESIGN.md section
  // 7e), within a goal in the order of the roots' modes, as
  // pp2d_pomdp_plan_batch orders its queries, or else as listed
  const bool sorted = h->sort_queries && n >= 2 * (uint32_t)kEvM;
  std::vector<uint32_t> key;
  if (sorted) PP2D_TRY(root_mode_keys(h, list, key));
  std::vector<int> order(n);
  for (uint32_t i = 0; i < n; ++i) order[i] = (int)i;
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) {
    if (list[x]->goal != list[y]->goal) return list[x]->goal < list[y]->goal;
    return sorted && key[x] < key[y];
  });
  for (uint32_t i = 0; i < n; ++i) list[i] = &b->trees[trees[order[i]]];
  PP2D_TRY(plan_trees(h, list, max_depth, max_iter, sorted));
  for (uint32_t i = 0; i < n; ++i) {
    const Tree& t = b->trees[trees[i]];
    float r;
    best_action(t, &actions[i], &r);
    if (values) values[i] = r;
    if (stats) {
      stats[4 * (size_t)i + 0] = (uint32_t)t.v.size();
      stats[4 * (size_t)i + 1] = (uint32_t)t.q.size();
      stats[4 * (size_t)i + 2] = t.v[t.root].depth;
      stats[4 * (size_t)i + 3] = t.expansions;
    }
  }
  return PP2D_OK;
}

int64_t pp2d_tree_batch_dump(const pp2d_tree_batch* b, uint32_t k, float* out,
                             uint64_t cap_nodes) {
  if (!b) { fail(PP2D_ERR_INVALID, "batch is NULL"); return -1; }
  if (k >= b->trees.size()) {
    fail(PP2D_ERR_INVALID, "pp2d_tree_batch_dump: tree %u of a batch of %zu", k, b->trees.size());
    return -1;
  }
  return dump_tree(b->trees[k], out, cap_nodes);
}

}  // extern "C"

namespace pp2d {

int tree_batch_root_beliefs(pp2d_tree_batch* b, float* out) {
  pp2d_pomdp* h = b->h;
  const size_t n = b->trees.size();
  if (n == 0) return PP2D_OK;
  std::vector<int> slots(n);
  for (size_t i = 0; i < n; ++i) slots[i] = b->trees[i].v[b->trees[i].root].slot;
  PP2D_TRY(h->d_rows.ensure(n * h->HW));
  PP2D_TRY(launch_gather(h, slots, h->d_rows.p));
  PP2D_CUDA(cudaMemcpyAsync(out, h->d_rows.p, n * h->HW * sizeof(float), cudaMemcpyDeviceToHost,
                            h->stream));
  PP2D_CUDA(cudaStreamSynchronize(h->stream));
  return PP2D_OK;
}

}  // namespace pp2d
