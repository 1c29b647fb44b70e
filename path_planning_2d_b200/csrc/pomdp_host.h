// pomdp_host.h -- host-side state shared by pomdp.cu (QV-tree) and pbvi.cu
// (offline PBVI solver): the planner handle behind pp2d_pomdp, the belief
// pool helpers and the glibc rand() replica.
#pragma once
#include "../../include/pp2d.h"

#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <vector>

namespace pp2d {
int fail(int code, const char* fmt, ...);            // mdp.cu
extern std::atomic<uint64_t> g_launches;
inline void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

struct BayesItem { int src, dst; uint8_t act, obs; };

// Belief pool layout (see the header of pomdp_kernels.cuh): blocks of 32
// slots, inside a block cell-major.  Offset of (cell, slot); the column of
// `slot` is bel_off(HW, 0, slot) + cell * kSlotBlock.
constexpr int kSlotBlock = 32;
__host__ __device__ __forceinline__ size_t bel_off(int HW, int cell, int slot) {
  return ((size_t)(slot >> 5) * (size_t)HW + (size_t)cell) * kSlotBlock + (size_t)(slot & 31);
}
}  // namespace pp2d

#define PP2D_CUDA(expr)                                                      \
  do {                                                                       \
    cudaError_t e_ = (expr);                                                 \
    if (e_ != cudaSuccess)                                                   \
      return pp2d::fail(PP2D_ERR_CUDA, "CUDA error at %s:%d code=%d(%s) \"%s\"",   \
                  __FILE__, __LINE__, (int)e_, cudaGetErrorName(e_), #expr); \
  } while (0)
#define PP2D_TRY(expr)                 \
  do {                                 \
    int rc_ = (expr);                  \
    if (rc_ != PP2D_OK) return rc_;    \
  } while (0)

namespace pp2d {

constexpr int kSamples = 50;      // search_tree_cuda.cu:176
constexpr int kActions = 9;
constexpr int kColFib = 0, kColPbvi = 9;   // columns of the bound matrix

// glibc rand() (TYPE_3 additive feedback, what the planner's rand() is since
// it never calls srand(): search_tree_cuda.cu:332).  Every query owns one
// stream seeded like a fresh process.
struct GlibcRand {
  int32_t r[34];
  int k;
  void seed(uint32_t s) {
    int32_t t[344];
    if (s == 0) s = 1;
    t[0] = (int32_t)s;
    for (int i = 1; i < 31; ++i) {
      long long v = (16807LL * t[i - 1]) % 2147483647LL;
      if (v < 0) v += 2147483647LL;
      t[i] = (int32_t)v;
    }
    for (int i = 31; i < 34; ++i) t[i] = t[i - 31];
    for (int i = 34; i < 344; ++i)
      t[i] = (int32_t)((uint32_t)t[i - 31] + (uint32_t)t[i - 3]);
    for (int i = 0; i < 34; ++i) r[i] = t[310 + i];
    k = 0;
  }
  uint32_t next() {
    // (k + 3) % 34 and (k + 31) % 34 without the divisions: a batch draws
    // 450 numbers per expanded node on the host
    const int a = k + 3 >= 34 ? k + 3 - 34 : k + 3;
    const int b = k + 31 >= 34 ? k + 31 - 34 : k + 31;
    uint32_t v = (uint32_t)r[a] + (uint32_t)r[b];
    r[k] = (int32_t)v;
    k = k + 1 == 34 ? 0 : k + 1;
    return v >> 1;
  }
};

// Free slots of the belief pool, handed out lowest first.  The values launches
// load a tile's columns coalesced only when its beliefs share 32-slot blocks
// (bel_off): a fresh pool gives a round's children ascending slots, and so
// does this list after trees have given back scattered slots (re-rooting,
// finished batches).
struct FreeSlots {
  std::vector<uint64_t> bits;     // bit s: slot s is free
  size_t n = 0;
  size_t lo = 0;                  // no free slot in words below lo
  size_t cap = 0;
  size_t count() const { return n; }
  bool empty() const { return n == 0; }
  void clear() { bits.clear(); n = 0; lo = 0; cap = 0; }
  void grow(size_t new_cap) {     // slots [cap, new_cap) are new and free
    bits.resize((new_cap + 63) / 64, 0);
    for (size_t s = cap; s < new_cap;) {
      if ((s & 63) == 0 && s + 64 <= new_cap) { bits[s >> 6] = ~0ull; s += 64; }
      else { bits[s >> 6] |= 1ull << (s & 63); ++s; }
    }
    n += new_cap - cap;
    if (cap >> 6 < lo) lo = cap >> 6;
    cap = new_cap;
  }
  void put(int s) {
    bits[(size_t)s >> 6] |= 1ull << (s & 63);
    ++n;
    if ((size_t)s >> 6 < lo) lo = (size_t)s >> 6;
  }
  int take() {                    // n > 0
    while (!bits[lo]) ++lo;
    const int b = __builtin_ctzll(bits[lo]);
    bits[lo] &= bits[lo] - 1;
    --n;
    return (int)(lo * 64 + (size_t)b);
  }
};

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;
  int ensure(size_t n) {
    if (n <= cap) return PP2D_OK;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = n + n / 2 + 64;
    PP2D_CUDA(cudaMalloc(&p, want * sizeof(T)));
    cap = want;
    return PP2D_OK;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

}  // namespace pp2d

struct pp2d_pomdp {
  int H = 0, W = 0, HW = 0, gx = 0, gy = 0;
  float gamma = 0.f;
  uint8_t* d_map = nullptr;
  std::vector<uint8_t> map_host;           // [H][W] as given to pp2d_pomdp_create
  // Goal set (DESIGN.md section 7e): goal 0 is (gx, gy), goals 1..n_goals come
  // from pp2d_pomdp_set_goals.  Per-goal data is stored goal-major, goal 0
  // first: d_sr [n_goals+1][HW][9], the bound matrices below.
  int n_goals = 0;
  std::vector<uint32_t> goal_xy;           // [n_goals+1][2]
  std::vector<uint8_t> goal_alphas;        // [n_goals+1]: alpha vectors set
  std::vector<uint8_t> goal_finite;        // [n_goals+1]: every bound finite
  float *d_tp = nullptr, *d_mp = nullptr, *d_sr = nullptr, *d_uniforms = nullptr;
  // bound matrices [n_goals+1][HW][ld]: FIB | PBVI (zero padded to whole
  // column tiles; zero for a goal without alpha vectors)
  float* d_alpha = nullptr;
  int ld = 0, ncol = 9, n_pbvi = 0;
  // Live cells (pomdp_dead_cells_kernel): the cells probability mass can enter.
  // d_kidx lists them in ascending order (K of them), d_alpha_live holds the
  // matching rows of the bound matrix; d_kidx_all = 0..HW-1 is the dense case.
  // The sequential inner products of a launch run over the live cells only
  // when every belief of the launch is +0 elsewhere (roots are checked on
  // upload, see Tree::dense in pomdp.cu).
  std::vector<uint8_t> dead;               // host copy of the mask
  std::vector<float> alpha_host;           // dense bound matrices [n_goals+1][HW][ld] as uploaded
  int* d_kidx = nullptr;
  int* d_kidx_all = nullptr;
  uint8_t* d_dead = nullptr;               // device copy of the mask
  int* d_kinv = nullptr;                   // cell -> its position in d_kidx, -1 for a dead cell
  float* d_mp_live = nullptr;              // rows d_kidx[0..K) of the likelihood table [K][16]
  float* d_alpha_live = nullptr;           // [n_goals+1][K][ld]
  int K = 0;
  bool skip_dead = true;                   // PP2D_POMDP_DENSE=1 turns the skipping off
  bool alphas_finite = true;               // every bound of every goal finite (else nothing is skipped)
  // batched planner: per-tile inner rows of the values launches
  // (PP2D_POMDP_TILE_SUPPORT=0 off) and queries planned in the order of their
  // start beliefs' modes (PP2D_POMDP_SORT=0 off)
  bool tile_support = true, sort_queries = true;
  std::vector<uint8_t> fib_actions, pbvi_actions;   // goal 0's (pp2d_pomdp_evaluate)
  bool have_alphas = false;                // goal 0's alpha vectors are set
  // belief pool [HW][cap]
  float* d_bel = nullptr;
  int cap = 0;
  pp2d::FreeSlots free_slots;
  // scratch
  pp2d::DevBuf<int> d_slots;
  pp2d::DevBuf<pp2d::BayesItem> d_items;
  pp2d::DevBuf<float> d_prefix, d_draws, d_vals, d_rows, d_sums;
  pp2d::DevBuf<uint8_t> d_obs;
  pp2d::DevBuf<float> d_out;               // 4 floats per evaluated belief
  pp2d::DevBuf<uint32_t> d_keys;           // mode keys of a tree batch's roots
  float* pin_rows = nullptr;               // page-locked staging of a batch's start beliefs
  size_t pin_rows_cap = 0;
  void* round_ctx[4] = {nullptr, nullptr, nullptr, nullptr};   // RoundCtx of pomdp.cu (lazily created)
  cudaStream_t stream = nullptr;
  uint64_t n_bayes = 0, n_vnodes = 0;
  // belief x inner-row products of the values launches: counted on the host
  // for the launches over a fixed row list, on the device (d_work) for the
  // per-tile lists
  uint64_t work_rows = 0;
  unsigned long long* d_work = nullptr;
  // of which spent on the padding of goal segments (pp2d_pomdp_padding_counters):
  // padded entries and their belief x inner-row products
  uint64_t pad_entries = 0, pad_rows = 0;
  double t_phase[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // PP2D_POMDP_PROFILE=1: seconds per phase
};


namespace pp2d {
// belief pool [HW][cap] (pomdp.cu)
int pool_reserve(pp2d_pomdp* h, size_t slots_wanted);
int alloc_slot(pp2d_pomdp* h, int* out);
// the batched B2 / B3 / B7 launches on pool columns (pomdp.cu)
int launch_bayes(pp2d_pomdp* h, const std::vector<BayesItem>& items);
int launch_normalize(pp2d_pomdp* h, const std::vector<int>& slots);
int launch_prefix(pp2d_pomdp* h, const std::vector<int>& slots);   // -> h->d_prefix [i*HW+s]
int launch_scatter(pp2d_pomdp* h, const std::vector<int>& slots, const float* host_rows);
int launch_gather(pp2d_pomdp* h, const std::vector<int>& slots, float* dev_rows);
// (re)derive the live-cell list from the transition table on the device and
// rebuild the compacted bound matrix (pomdp.cu)
int refresh_live_cells(pp2d_pomdp* h);
// true when `belief` ([HW], host) is exactly +0 on every dead cell
bool zero_on_dead_cells(const pp2d_pomdp* h, const float* belief);
}  // namespace pp2d
