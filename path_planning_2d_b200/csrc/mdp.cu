// mdp.cu -- host side of the MDP value-iteration C ABI (include/pp2d.h).
//
// Replaces, for the reference's MdpPathPlanning2d
// (/root/reference/path_planning_2d/src/mdp/path_planning_2d.cu):
//   allocateDeviceMemory / freeDeviceMemory / the six global device pointers
//   (path_planning_2d_cuda.cu:26-74), the map upload and model generation
//   (path_planning_2d.cu:90-106), valueIteration() (207-269) and the result
//   download (118-126).
// There is no CPU fallback in this file: without a CUDA device every entry
// point fails with PP2D_ERR_CUDA.
#include "../../include/pp2d.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "handles.h"
#include "mdp_kernels.cuh"

namespace pp2d {

thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define PP2D_CUDA(expr)                                                      \
  do {                                                                       \
    cudaError_t e_ = (expr);                                                 \
    if (e_ != cudaSuccess)                                                   \
      return fail(PP2D_ERR_CUDA, "CUDA error at %s:%d code=%d(%s) \"%s\"",   \
                  __FILE__, __LINE__, (int)e_, cudaGetErrorName(e_), #expr); \
  } while (0)

#define PP2D_TRY_MDP(expr)             \
  do {                                 \
    int rc_ = (expr);                  \
    if (rc_ != PP2D_OK) return rc_;    \
  } while (0)

// ---------------------------------------------------------------------------
// Model numbers of one cell, restated from the reference for the table build:
// cudaTransitionProbability (path_planning_2d_cuda.cu:76-150) and
// cudaStageCost (152-172) for a FREE centre cell whose neighbour occupancy is
// `occ` (9 entries, slot 4 ignored).  Outputs per action u: the stage cost
// g[u] and the probability of staying P_u[4] after the blocked mass has been
// shifted to the centre.  The order of the float additions is the
// reference's (ascending slot index).
static void cell_model(const uint8_t occ[9], float g[9], float p4[9]) {
  static const float naive[9][9] = {
      {0.7f, 0.1f, 0.f, 0.1f, 0.1f, 0.f, 0.f, 0.f, 0.f},
      {0.1f, 0.7f, 0.1f, 0.f, 0.1f, 0.f, 0.f, 0.f, 0.f},
      {0.f, 0.1f, 0.7f, 0.f, 0.1f, 0.1f, 0.f, 0.f, 0.f},
      {0.1f, 0.f, 0.f, 0.7f, 0.1f, 0.f, 0.1f, 0.f, 0.f},
      {0.f, 0.f, 0.f, 0.f, 1.0f, 0.f, 0.f, 0.f, 0.f},
      {0.f, 0.f, 0.1f, 0.f, 0.1f, 0.7f, 0.f, 0.f, 0.1f},
      {0.f, 0.f, 0.f, 0.1f, 0.1f, 0.f, 0.7f, 0.1f, 0.f},
      {0.f, 0.f, 0.f, 0.f, 0.1f, 0.f, 0.1f, 0.7f, 0.1f},
      {0.f, 0.f, 0.f, 0.f, 0.1f, 0.1f, 0.f, 0.1f, 0.7f}};
  for (int u = 0; u < 9; ++u) {
    float stay = naive[u][4];
    float cost = 0.0f;
    for (int i = 0; i < 9; ++i) {
      const bool blocked = (i != 4) && occ[i];
      if (blocked) stay += naive[u][i];                 // cuda.cu:142-147
      // map_cost is 1 or 2: the product is exact, fmaf == the device FFMA.
      cost = fmaf(blocked ? 2.0f : 1.0f, naive[u][i], cost);  // cuda.cu:166-169
    }
    g[u] = cost;
    p4[u] = stay;
  }
}

// Ring position -> neighbour slot (see mdp_kernels.cuh).
static const int kRingSlot[10] = {0, 1, 2, 5, 8, 7, 6, 3, 0, 1};
// Action pair p reads ring bits 2p..2p+3; {first, second} action of the pair.
static const int kPairAction[4][2] = {{1, 2}, {5, 8}, {7, 6}, {3, 0}};

static void build_lut(float gamma, std::vector<float4>& lut) {
  lut.assign(kLutFloat4 / 8, make_float4(0, 0, 0, 0));   // one copy per row
  // row of action pair p for the 4-bit ring field f
  auto pair_row = [&](int p, int f) {
    uint8_t occ[9] = {0};
    for (int b = 0; b < 4; ++b)
      if (f >> b & 1) occ[kRingSlot[2 * p + b]] = 1;
    float g[9], p4[9];
    cell_model(occ, g, p4);
    const int u0 = kPairAction[p][0], u1 = kPairAction[p][1];
    // gamma*tp[i] is rounded to float before the FFMA (SASS of the
    // reference kernel: FMUL then FFMA).
    return make_float4(g[u0], gamma * p4[u0], g[u1], gamma * p4[u1]);
  };
  for (int p = 0; p < 4; ++p)
    for (int f = 0; f < 16; ++f) lut[p * 16 + f] = pair_row(p, f);
}

}  // namespace pp2d

using namespace pp2d;

struct pp2d_mdp {
  uint32_t Htot = 0, W = 0;        // whole grid
  uint32_t row_begin = 0, H = 0;   // owned rows
  uint32_t gx = 0, gy = 0;
  float gamma = 0.f;
  bool sharded = false;
  int pitch = 0;
  size_t plane = 0;                // elements of one padded plane
  float* j[2] = {nullptr, nullptr};
  float* jchk = nullptr;
  uint16_t* code = nullptr;
  uint8_t* action = nullptr;       // dense [H][W]
  uint8_t* occ = nullptr;          // dense rows [occ_row0, occ_row0+occ_rows)
  float* dense = nullptr;          // export staging [H][W]
  uint8_t* dense_action = nullptr; // action snapshot of an asynchronous download
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_snapshot = nullptr, ev_copied = nullptr;
  bool download_pending = false;
  // map of the NEXT reset, uploaded ahead of time (pp2d_mdp_stage_map)
  uint8_t* occ_next = nullptr;     // same size as occ
  cudaStream_t upload_stream = nullptr;
  cudaEvent_t ev_staged = nullptr, ev_code_built = nullptr;
  const uint8_t* staged_map = nullptr;   // host pointer the staged rows came from
  float4* lut = nullptr;
  uint32_t* resid = nullptr;       // device float bits
  uint32_t* resid_host = nullptr;  // pinned
  int cur = 0;                     // j[cur] holds J_n
  uint32_t n_sweeps = 0;
  uint32_t n_chk = 0;              // sweep count at the last residual call
  bool chk_is_zero = true;         // jchk stands for J_0 = 0 (not written since the reset)
  uint32_t action_sweep = 0;       // sweep count the action grid belongs to
  bool has_occupied = false;
  std::vector<float> trapped;      // trapped[n] = J_n of an occupied cell
  std::vector<uint8_t> action_host;
  bool action_host_valid = false;
  cudaStream_t stream = nullptr;
  bool async = false;
  int sm_count = 148;
  // peer-to-peer ghost rows (pp2d_mdp_ipc_connect)
  unsigned int* flags = nullptr;   // kFlagWords, IPC-shared
  bool p2p = false;
  float* up_j[2] = {nullptr, nullptr};     // mapped neighbour planes
  float* down_j[2] = {nullptr, nullptr};
  unsigned int* up_flags = nullptr;
  unsigned int* down_flags = nullptr;
  uint32_t up_H = 0;
  void* ipc_opened[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  unsigned int p2p_iter = 0, p2p_expect_top = 0, p2p_expect_bot = 0;
  int p2p_debug = 0;
  int p2p_edge_short = 20;         // rows the boundary row blocks are shorter (hand-shake cost)
  unsigned int p2p_spin_limit = 1u << 24;   // polls (32-256 ns apart) before kFlagError
  // ghost-row contract of a shard without peer-to-peer rows: sweeps that may
  // still run before the caller has to refresh the ghost rows (pp2d_mdp_halo)
  int halo_budget = kPadRows;
  // tuning knobs (environment overridable, read in make_handle)
  int cw2 = 2, cw1 = 4, rows_per_unit = 0;
  int linear_units = -1;      // -1 = choose per launch, 0 = row blocks, 1 = strip-major runs
  // policy iteration (pp2d_mdp_policy_iteration): evaluation sweeps since the
  // reset; occupied cells then follow J_n = (gamma*J_{n-1}) + 2
  bool pi_mode = false;
  std::vector<float> trapped_pi;
  // skipping of units whose two-sweep input is unchanged (PP2D_MDP_SKIP,
  // DESIGN.md section 4): three rotating unit masks of the fused row-block
  // launches.  need_valid: the mask the next such launch reads was written by
  // the launch right before it, on the same geometry; otherwise it runs every
  // unit.
  bool skip = true;
  uint32_t* need[3] = {nullptr, nullptr, nullptr};
  int need_words = 0, need_rot = 0;
  int need_units = 0, need_rows_per_unit = 0;
  bool need_valid = false;
  unsigned long long* work = nullptr;   // [0] units run, [1] units launched
  uint32_t* need_alloc = nullptr;
  int device = 0;                  // CUDA device the buffers live on
  bool owns_stream = false;
  // launch geometry cache (the occupancy query and the count of boundary units
  // cost microseconds per launch; a multi-GPU handle launches on N devices from
  // one host thread)
  struct LaunchCache {
    bool valid = false;
    int ctas_per_sm = 0;
    int y_rows = 0, lin_len = 0, rows_per_unit = 0, n_units = 0, rows_edge = 0, rows_inner = 0;
    int* d_unit_lo = nullptr;            // cost-balanced unit boundaries (P2P LIN kernels)
    std::vector<int> unit_lo_host;
    unsigned int top_segs = 0, bot_segs = 0;
  } launch_cache[2][3][2][2];      // [T-1][CW: 1,2,4 -> 0,1,2][POLICY][P2P]
  // ---- single-process multi-GPU container (pp2d_mdp_create_multi) ----------
  std::vector<pp2d_mdp*> parts;    // row shards, top to bottom; empty for ordinary handles
  std::vector<cudaEvent_t> ev_done, ev_pulled;   // one per part
  bool multi_p2p = false;          // ghost rows through the fused kernels' peer stores
  bool fused_pending = false;      // fused peer-to-peer launches since the last barrier
};

namespace pp2d {
struct DeviceGuard {               // restore the caller's current device on exit
  int prev = -1;
  DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
}  // namespace pp2d

namespace pp2d {

static float trapped_cost(pp2d_mdp* h, uint32_t n) {
  // Occupied cell: every action has P = e_4 and g = 2
  // (path_planning_2d_cuda.cu:131-134), so J_n = fma(gamma*1.0f, J_{n-1}, 2).
  while (h->trapped.size() <= n)
    h->trapped.push_back(fmaf(h->gamma, h->trapped.back(), 2.0f));
  return h->trapped[n];
}

// Occupied cell under policy evaluation: P = e_4, g = 2 for every action, so
// J_n = fma(fmul(gamma, J_{n-1}), 1, 2) = (gamma*J_{n-1}) + 2, two roundings.
static float trapped_cost_pi(pp2d_mdp* h, uint32_t n) {
  if (h->trapped_pi.empty()) h->trapped_pi.push_back(0.0f);
  while (h->trapped_pi.size() <= n)
    h->trapped_pi.push_back(h->gamma * h->trapped_pi.back() + 2.0f);
  return h->trapped_pi[n];
}
static float occupied_cost(pp2d_mdp* h, uint32_t n) {
  return h->pi_mode ? trapped_cost_pi(h, n) : trapped_cost(h, n);
}

// The reference's stopping rule (path_planning_2d.cu:219-263): sweeping goes
// on while the residual exceeds 1e-3 of the largest optimal cost.
static bool keeps_sweeping(double residual, float gamma) {
  const double max_optimal_cost = 5.0 / (1.0 - gamma);
  return residual > max_optimal_cost * 1e-3;
}

// The goal of a width x height map must lie inside it, on a free cell
// (path_planning_2d.cu:84-88).  instance >= 0: the batch instance the
// messages name.
static int check_goal(const uint8_t* map, uint32_t width, uint32_t height, uint32_t gx,
                      uint32_t gy, int64_t instance = -1) {
  char who[32] = "";
  if (instance >= 0) snprintf(who, sizeof(who), "instance %u: ", (uint32_t)instance);
  if (gx >= width || gy >= height)
    return fail(PP2D_ERR_INVALID, "%sgoal (%u %u) outside the %ux%u map", who, gx, gy, width,
                height);
  if (map[(size_t)gy * width + gx] > 0)
    return fail(PP2D_ERR_GOAL_OCCUPIED, "%sThe assigned goal (%u %u) is at a occupied cell...",
                who, gx, gy);
  return PP2D_OK;
}

// Occupancy rows [row0, row0 + rows) that a handle owning rows [row_begin,
// row_end) of a grid of `height` rows keeps on the device: the codes of its
// owned and ghost rows read up to 3 rows beyond them.
struct OccWindow {
  int row0, rows;
};
static OccWindow occ_window(uint32_t row_begin, uint32_t row_end, uint32_t height) {
  const int row0 = (int)row_begin - 3 < 0 ? 0 : (int)row_begin - 3;
  const int row1 = (int)row_end + 3 > (int)height ? (int)height : (int)row_end + 3;
  return {row0, row1 - row0};
}

// CodeParams of h's code plane built from the occupancy rows at `occ`, and the
// grid of a code or update kernel launch over it.
static CodeParams code_params(const pp2d_mdp* h, const uint8_t* occ) {
  const OccWindow ow = occ_window(h->row_begin, h->row_begin + h->H, h->Htot);
  CodeParams cp;
  cp.occ = occ; cp.code = h->code; cp.W = (int)h->W; cp.Htot = (int)h->Htot;
  cp.pitch = h->pitch; cp.rows_phys = (int)h->H + 2 * kPadRows;
  cp.row_begin = (int)h->row_begin; cp.occ_row0 = ow.row0; cp.occ_rows = ow.rows;
  cp.gx = (int)h->gx; cp.gy = (int)h->gy;
  return cp;
}
static dim3 code_grid(const CodeParams& cp) {
  return dim3((cp.pitch / 4 + kCodeThreads - 1) / kCodeThreads,
              (cp.rows_phys + kCodeRows - 1) / kCodeRows);
}

// The unit mask of h's next fused row-block launch, for a kernel that seeds or
// clears it.  Without a valid mask that launch runs every unit anyway, and
// `need` is NULL.
static UnitMask next_unit_mask(const pp2d_mdp* h) {
  UnitMask m = {nullptr, ((int)h->W + kUnitStrip - 1) / kUnitStrip, 1, 1};
  if (h->need_valid) {
    m.need = h->need[h->need_rot];
    m.rows_per_unit = h->need_rows_per_unit;
    m.n_rb = h->need_units / m.n_strips;
  }
  return m;
}

// CW == 1 kernels: rows ahead of the marching row touched with prefetch.global.L1
// (the slack rows below the plane bound how far ahead that may reach).
constexpr int kL1PrefetchRows = 6;
static_assert(kL1PrefetchRows >= kPrefetch && kL1PrefetchRows <= kSlackRows, "prefetch rows");
// P2P kernels: rows of a boundary unit marched before it publishes its flag.
constexpr int kP2pEdgeRows = 16;
static_assert(kP2pEdgeRows >= kPadRows, "edge rows");

template <int T, int CW, bool POLICY, bool P2P = false>
static int launch_sweep(pp2d_mdp* h) {
  // strip-major runs exist for the fused kernels at CW = 2 (the ones that
  // dominate a solve)
  constexpr bool kHasLin = (T == 2 && CW == 2);
  using G = StripGeom<T, CW>;
  SweepParams p;
  memset(&p, 0, sizeof(p));
  p.jin = h->j[h->cur];
  p.jout = h->j[h->cur ^ 1];
  p.code = h->code;
  p.action = h->action;
  p.lut = h->lut;
  p.W = (int)h->W;
  p.H = (int)h->H;
  p.pitch = h->pitch;
  p.n_strips = ((int)h->W + G::S - 1) / G::S;
  // A value-only single sweep also produces the first ghost row on each
  // side, so that a second sweep can follow without an exchange (the fused
  // kernel does the same in registers).  Outside the map those rows are
  // padding and stay 0.
  p.y_begin = (T == 1 && !POLICY) ? -1 : 0;
  p.y_end = (T == 1 && !POLICY) ? (int)h->H + 1 : (int)h->H;
  const int rows = p.y_end - p.y_begin;
  int rpu = h->rows_per_unit;
  p.lin_len = 0;
  pp2d_mdp::LaunchCache& lc =
      h->launch_cache[T - 1][CW == 1 ? 0 : (CW == 2 ? 1 : 2)][POLICY ? 1 : 0][P2P ? 1 : 0];
  if (lc.valid && lc.y_rows == rows) {
    p.lin_len = lc.lin_len;
    p.rows_per_unit = lc.rows_per_unit;
    p.n_units = lc.n_units;
    p.unit_lo = lc.d_unit_lo;
  } else if (rpu <= 0) {
    // Launch sized to exactly one full wave of resident CTAs (one unit per
    // warp); the units are equal runs of the strip-major row sequence.
    int ctas_per_sm = 0;
    PP2D_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(
        &ctas_per_sm, mdp_sweep_kernel<T, CW, POLICY, P2P>, kWarpsPerCta * 32, 0));
    if (ctas_per_sm < 1) ctas_per_sm = 1;
    lc.ctas_per_sm = ctas_per_sm;
    const long long slots = (long long)h->sm_count * ctas_per_sm * kWarpsPerCta;
    // (a) whole row blocks per strip: floor(slots / strips) blocks, no restart;
    long long rb = slots / p.n_strips;
    if (rb < 1) rb = 1;
    long long rpu_blocks = (rows + rb - 1) / rb;
    if (rpu_blocks < 8) rpu_blocks = 8;
    // (b) equal runs of the strip-major row sequence: every slot busy, but a
    // unit that crosses a strip boundary primes its pipeline twice (~4 rows).
    const long long total = (long long)p.n_strips * rows;
    long long len = (total + slots - 1) / slots;
    if (len < 8) len = 8;
    if (len > rows) len = rows;               // at most one strip boundary per unit
    const long long restart_rows = 4;
    if (kHasLin && h->linear_units != 0 &&
        (h->linear_units > 0 || len + restart_rows < rpu_blocks)) {
      p.lin_len = (int)len;
      p.rows_per_unit = (int)len;
      p.n_units = (int)((total + len - 1) / len);
    } else {
      p.rows_per_unit = (int)rpu_blocks;
      p.n_units = p.n_strips * (int)((rows + rpu_blocks - 1) / rpu_blocks);
    }
    if (P2P && p.lin_len > 0 && h->p2p_edge_short > 0 && rows >= 64) {
      // Cost-balanced units for the peer-to-peer kernels: rows cost 1, every
      // segment start ~3 rows of pipeline priming, every hand-shake (a segment
      // that touches the first / last two rows of a strip next to a neighbour)
      // p2p_edge_short rows.  Smallest cost target that fits the warp slots.
      const bool up = h->up_j[0] != nullptr, down = h->down_j[0] != nullptr;
      const double c_seg = 3.0, c_edge = (double)h->p2p_edge_short;
      std::vector<int>& lo_out = lc.unit_lo_host;
      auto build = [&](double target) -> long long {
        lo_out.clear();
        lo_out.push_back(0);
        double acc = 0.0;
        for (int k = 0; k < p.n_strips; ++k)
          for (int y = 0; y < rows; ++y) {
            double c = 1.0;
            if (y == 0 && up) c += c_edge;
            if (y == rows - 1 && down) c += c_edge;
            const bool may_cut = y != 1 && y != rows - 1;     // both edge rows stay together
            if (acc > 0.0 && may_cut && acc + c + (y == 0 ? c_seg : 0.0) > target) {
              lo_out.push_back(k * rows + y);
              acc = 0.0;
            }
            if (acc == 0.0 || y == 0) c += c_seg;
            acc += c;
          }
        lo_out.push_back(p.n_strips * rows);
        return (long long)lo_out.size() - 1;
      };
      // (one slot stays free for the warp that publishes the flags)
      const long long avail = slots - 1;
      double lo_t = (double)total / (double)slots, hi_t = 4.0 * lo_t + 4.0 * (c_edge + c_seg) + 16.0;
      for (int it = 0; it < 24; ++it) {
        const double mid = 0.5 * (lo_t + hi_t);
        if (build(mid) <= avail) hi_t = mid; else lo_t = mid;
      }
      const long long nu = build(hi_t);
      if (nu <= avail) {
        if (lc.d_unit_lo) cudaFree(lc.d_unit_lo);
        lc.d_unit_lo = nullptr;
        PP2D_CUDA(cudaMalloc(&lc.d_unit_lo, lo_out.size() * sizeof(int)));
        PP2D_CUDA(cudaMemcpy(lc.d_unit_lo, lo_out.data(), lo_out.size() * sizeof(int),
                             cudaMemcpyHostToDevice));
        p.unit_lo = lc.d_unit_lo;
        p.n_units = (int)nu;
        int longest = 1;
        for (size_t u = 0; u + 1 < lo_out.size(); ++u)
          longest = std::max(longest, lo_out[u + 1] - lo_out[u]);
        p.lin_len = longest;              // > 0 selects the LIN instantiation
        p.rows_per_unit = longest;
      }
    }
  } else {
    p.rows_per_unit = rpu;
    const int n_rb = (rows + rpu - 1) / rpu;
    p.n_units = p.n_strips * n_rb;
  }
  p.prefetch_rows = kL1PrefetchRows;
  p.gamma = h->gamma * 1.0f;
  p.ga = h->gamma * 0.7f;
  p.gb = h->gamma * 0.1f;
  if (P2P) {
    // Boundary units of this launch: those whose rows touch the first / last
    // two owned rows (they wait for and signal the neighbours).
    // (same enumeration of the segments as Sweeper::run)
    unsigned int top_segs = 0, bot_segs = 0;
    auto count = [&](int y0, int y1) {
      if (y0 < kPadRows) ++top_segs;
      if (y1 > (int)h->H - kPadRows) ++bot_segs;
    };
    if (lc.valid && lc.y_rows == rows) {
      top_segs = lc.top_segs;
      bot_segs = lc.bot_segs;
      p.rows_edge = lc.rows_edge;
      p.rows_inner = lc.rows_inner;
    } else if (p.unit_lo != nullptr) {
      const long long R = rows;
      for (int u = 0; u < p.n_units; ++u) {
        long long lo = lc.unit_lo_host[u];
        const long long hi = lc.unit_lo_host[u + 1];
        while (lo < hi) {
          const long long k = lo / R, a = lo - k * R, b = std::min(R, a + (hi - lo));
          count(p.y_begin + (int)a, p.y_begin + (int)b);
          lo += b - a;
        }
      }
    } else if (p.lin_len > 0) {
      const long long R = rows, total = (long long)p.n_strips * R;
      for (long long u = 0; u < p.n_units; ++u) {
        long long lo = u * p.lin_len;
        const long long hi = std::min(lo + (long long)p.lin_len, total);
        while (lo < hi) {
          const long long k = lo / R, a = lo - k * R, b = std::min(R, a + (hi - lo));
          count(p.y_begin + (int)a, p.y_begin + (int)b);
          lo += b - a;
        }
      }
    } else {
      const int n_rb = (rows + p.rows_per_unit - 1) / p.rows_per_unit;
      // Edge blocks pay for the hand-shake: make them shorter (same formulas as
      // Sweeper::run).  Needs interior blocks to take up the rows.
      p.rows_edge = p.rows_inner = 0;
      const int m = n_rb - 2, re = p.rows_per_unit - h->p2p_edge_short;
      if (h->p2p_edge_short > 0 && m >= 1 && re > m + 2 * kPadRows + 8 && 2 * re < rows) {
        p.rows_edge = re;
        p.rows_inner = (rows - 2 * re + m - 1) / m;
      }
      for (int rb = 0; rb < n_rb; ++rb) {
        int y0, y1;
        if (p.rows_edge > 0) {
          y0 = rb == 0 ? 0 : p.rows_edge + (rb - 1) * p.rows_inner;
          y1 = std::min(p.rows_edge + rb * p.rows_inner, (int)h->H);
        } else {
          y0 = rb * p.rows_per_unit;
          y1 = std::min(y0 + p.rows_per_unit, (int)h->H);
        }
        for (int k = 0; k < p.n_strips; ++k) count(y0, y1);
      }
    }
    lc.rows_edge = p.rows_edge;
    lc.rows_inner = p.rows_inner;
    lc.top_segs = top_segs;
    lc.bot_segs = bot_segs;
    h->p2p_iter += 1;
    const int nxt = h->cur ^ 1;
    if (h->up_j[nxt]) {
      h->p2p_expect_top += top_segs;
      p.peer_up_out = h->up_j[nxt] + (size_t)(h->up_H + kPadRows) * h->pitch;
      p.up_flag_remote = h->up_flags + kFlagFromDown;
    }
    if (h->down_j[nxt]) {
      h->p2p_expect_bot += bot_segs;
      p.peer_down_out = h->down_j[nxt];
      p.down_flag_remote = h->down_flags + kFlagFromUp;
    }
    p.flags = h->flags;
    p.iter = h->p2p_iter;
    p.expect_top = h->p2p_expect_top;
    p.expect_bot = h->p2p_expect_bot;
    p.p2p_debug = (unsigned int)h->p2p_debug;
    p.edge_rows = kP2pEdgeRows;
    p.spin_limit = h->p2p_spin_limit;
  }
  // P2P: a warp slot of the launch that has no rows publishes the flags (the
  // marching warps then never execute a system fence); without a free slot in
  // the last CTA the last boundary unit does it, as before.
  p.publisher_unit = -1;
  if (P2P && p.n_units % kWarpsPerCta != 0) p.publisher_unit = p.n_units;
  lc.valid = true;
  lc.y_rows = rows;
  lc.lin_len = p.lin_len;
  lc.rows_per_unit = p.rows_per_unit;
  lc.n_units = p.n_units;
  // Unit skipping: fused row-block launches only (not the strip-major runs,
  // not the peer-to-peer kernels); units of at least 2 rows, so that the 2-row
  // dependency cone of a unit lies inside its 3x3 unit neighbourhood.
  bool book = false;
  if constexpr (T == 2 && CW == 2 && !P2P) {
    p.work = h->work;
    book = h->skip && p.lin_len == 0 && p.rows_per_unit >= 2;
  }
  if (book) {
    const int words = (p.n_units + 31) / 32;
    if (p.n_units != h->need_units || p.rows_per_unit != h->need_rows_per_unit) {
      if (words > h->need_words) {
        cudaFree(h->need_alloc);
        h->need_alloc = nullptr;
        h->need_words = 0;
        PP2D_CUDA(cudaMalloc(&h->need_alloc, 3 * (size_t)words * sizeof(uint32_t)));
        h->need_words = words;
      }
      // (stream-ordered: a previous launch may still read the old masks)
      PP2D_CUDA(cudaMemsetAsync(h->need_alloc, 0, 3 * (size_t)h->need_words * sizeof(uint32_t),
                                h->stream));
      for (int i = 0; i < 3; ++i) h->need[i] = h->need_alloc + (size_t)i * h->need_words;
      h->need_units = p.n_units;
      h->need_rows_per_unit = p.rows_per_unit;
      h->need_rot = 0;
      h->need_valid = false;
    }
    p.need_in = h->need[h->need_rot];
    p.need_out = h->need[(h->need_rot + 1) % 3];
    p.need_clear = h->need[(h->need_rot + 2) % 3];
    // The arg-min launch runs every unit: the action grid is always complete.
    p.all_live = (POLICY || !h->need_valid) ? 1 : 0;
    // ghost rows of a shard with neighbours change under the row blocks next to them
    p.edge_live = (h->sharded && (h->row_begin > 0 || h->row_begin + h->H < h->Htot)) ? 1 : 0;
  }
  const int warps_per_cta = kWarpsPerCta;
  const int grid = (p.n_units + warps_per_cta - 1) / warps_per_cta;
  // Fused launches follow each other back to back: with programmatic dependent
  // launch the prologue of the next one overlaps the tail of this one.
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(warps_per_cta * 32);
  cfg.stream = h->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if constexpr (kHasLin) {
    if (p.lin_len > 0)
      PP2D_CUDA(cudaLaunchKernelEx(&cfg, mdp_sweep_kernel<T, CW, POLICY, P2P, true>, p));
    else
      PP2D_CUDA(cudaLaunchKernelEx(&cfg, mdp_sweep_kernel<T, CW, POLICY, P2P, false>, p));
  } else {
    PP2D_CUDA(cudaLaunchKernelEx(&cfg, mdp_sweep_kernel<T, CW, POLICY, P2P>, p));
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  PP2D_CUDA(cudaGetLastError());
  h->cur ^= 1;
  h->n_sweeps += T;
  // Any other launch changes J without change bits: the next one runs all.
  if (book) h->need_rot = (h->need_rot + 1) % 3;
  h->need_valid = book;
  return PP2D_OK;
}

template <int T, bool POLICY>
static int launch_sweep_cw(pp2d_mdp* h, int cw) {
  if (T == 2 && POLICY)      // fused pair whose second sweep is the arg-min one
    return h->p2p ? launch_sweep<2, 2, true, true>(h) : launch_sweep<2, 2, true, false>(h);
  if (T == 2 && !POLICY && h->p2p)
    return cw == 4 ? launch_sweep<2, 4, false, true>(h)
                   : launch_sweep<2, 2, false, true>(h);
  switch (cw) {
    case 1: return launch_sweep<T, 1, POLICY>(h);
    case 2: return launch_sweep<T, 2, POLICY>(h);
    default: return launch_sweep<T, 4, POLICY>(h);
  }
}

static int sync_if_needed(pp2d_mdp* h) {
  if (!h->async) PP2D_CUDA(cudaStreamSynchronize(h->stream));
  return PP2D_OK;
}

static int env_int(const char* name, int dflt) {
  const char* s = getenv(name);
  return (s && *s) ? atoi(s) : dflt;
}

// Zero J / action, upload the occupancy rows this handle needs and rebuild
// the code plane: allocateDeviceMemory's memsets + the map upload + the model
// generation of the reference (path_planning_2d_cuda.cu:55-61,
// path_planning_2d.cu:94-106).
static int upload_map(pp2d_mdp* h, const uint8_t* map) {
  const size_t owned = (size_t)h->H * h->W;
  PP2D_CUDA(cudaMemsetAsync(h->j[0], 0, h->plane * sizeof(float), h->stream));
  PP2D_CUDA(cudaMemsetAsync(h->j[1], 0, h->plane * sizeof(float), h->stream));
  h->chk_is_zero = true;          // Jchk = J_0 = 0: the first residual does not read it
  PP2D_CUDA(cudaMemsetAsync(h->action, 0, owned, h->stream));
  // a timed-out hand-shake of an earlier solve must not poison this one (the
  // launch counters in the flag block are cumulative and stay)
  PP2D_CUDA(cudaMemsetAsync(h->flags + kFlagError, 0, sizeof(unsigned int), h->stream));
  h->halo_budget = kPadRows;
  // The rows may already be on the device (pp2d_mdp_stage_map of this very
  // pointer): order the code kernel after that copy and swap the two buffers.
  const bool staged = h->staged_map != nullptr && h->staged_map == map;
  h->staged_map = nullptr;
  if (staged) {
    PP2D_CUDA(cudaStreamWaitEvent(h->stream, h->ev_staged, 0));
    std::swap(h->occ, h->occ_next);
  } else {
    const OccWindow ow = occ_window(h->row_begin, h->row_begin + h->H, h->Htot);
    PP2D_CUDA(cudaMemcpyAsync(h->occ, map + (size_t)ow.row0 * h->W, (size_t)ow.rows * h->W,
                              cudaMemcpyHostToDevice, h->stream));
  }
  const CodeParams cp = code_params(h, h->occ);
  mdp_code_kernel<<<code_grid(cp), kCodeThreads, 0, h->stream>>>(cp);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  PP2D_CUDA(cudaGetLastError());
  if (h->ev_code_built) PP2D_CUDA(cudaEventRecord(h->ev_code_built, h->stream));
  // (the caller may free `map` on return: wait for the copy; a staged map has
  // been waited for in stream order and the host is free to run ahead)
  if (!staged) PP2D_CUDA(cudaStreamSynchronize(h->stream));
  h->has_occupied =
      memchr(map + (size_t)h->row_begin * h->W, 1, owned) != nullptr;
  h->cur = 0;
  h->n_sweeps = h->n_chk = h->action_sweep = 0;
  h->action_host_valid = false;
  h->pi_mode = false;
  h->need_valid = false;
  return PP2D_OK;
}

// New map and goal (h->gx, h->gy already set) on a handle that keeps its J:
// codes rebuilt, J' and Jchk written by mdp_update_map_kernel, the sweep count
// kept.  The new rows always arrive through the staging buffer: a map that
// was not staged with pp2d_mdp_stage_map is staged here and waited for.
static int update_map(pp2d_mdp* h, const uint8_t* map) {
  const bool staged = h->staged_map != nullptr && h->staged_map == map;
  if (!staged) PP2D_TRY_MDP(pp2d_mdp_stage_map(h, map));
  h->staged_map = nullptr;
  PP2D_CUDA(cudaStreamWaitEvent(h->stream, h->ev_staged, 0));
  UpdateParams up;
  up.c = code_params(h, h->occ_next);
  up.j = h->j[h->cur];
  up.jchk = h->jchk;
  up.trapped = trapped_cost(h, h->n_sweeps);
  up.mask = next_unit_mask(h);
  up.H = (int)h->H;
  mdp_update_map_kernel<<<code_grid(up.c), kCodeThreads, 0, h->stream>>>(up);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  PP2D_CUDA(cudaGetLastError());
  PP2D_CUDA(cudaEventRecord(h->ev_code_built, h->stream));
  // (the caller may free `map` on return: wait for the copy)
  if (!staged) PP2D_CUDA(cudaStreamSynchronize(h->stream));
  std::swap(h->occ, h->occ_next);
  h->has_occupied =
      memchr(map + (size_t)h->row_begin * h->W, 1, (size_t)h->H * h->W) != nullptr;
  h->n_chk = h->n_sweeps;
  h->chk_is_zero = false;
  return PP2D_OK;
}

static int make_handle(uint32_t height, uint32_t width, float gamma, uint32_t row_begin,
                       uint32_t row_end, bool sharded, size_t occ_bytes, pp2d_mdp** out);

static int create_impl(uint32_t height, uint32_t width, const uint8_t* map,
                       uint32_t gx, uint32_t gy, float gamma,
                       uint32_t row_begin, uint32_t row_end, bool sharded,
                       pp2d_mdp** out) {
  if (!out) return fail(PP2D_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (!map || height == 0 || width == 0)
    return fail(PP2D_ERR_INVALID, "empty map");
  if (gx >= width || gy >= height)
    return fail(PP2D_ERR_INVALID, "goal (%u %u) outside the %ux%u map", gx, gy,
                width, height);
  if (row_begin >= row_end || row_end > height)
    return fail(PP2D_ERR_INVALID, "bad row range [%u, %u)", row_begin, row_end);
  if (sharded && row_end - row_begin < (uint32_t)kPadRows)
    return fail(PP2D_ERR_INVALID, "a shard needs at least %d rows", kPadRows);
  if ((uint64_t)height * width >= (1ull << 40))
    return fail(PP2D_ERR_INVALID, "map too large");
  PP2D_TRY_MDP(check_goal(map, width, height, gx, gy));
  pp2d_mdp* h = nullptr;
  PP2D_TRY_MDP(make_handle(height, width, gamma, row_begin, row_end, sharded,
                           (size_t)occ_window(row_begin, row_end, height).rows * width, &h));
  h->gx = gx; h->gy = gy;
  const int rc = upload_map(h, map);
  if (rc != PP2D_OK) { pp2d_mdp_destroy(h); return rc; }
  *out = h;
  return PP2D_OK;
}

// Device buffers, table and tuning knobs of a handle that owns rows
// [row_begin, row_end) of a height x width grid, with occ_bytes of occupancy
// storage; the map itself is uploaded by the caller.
static int make_handle(uint32_t height, uint32_t width, float gamma, uint32_t row_begin,
                       uint32_t row_end, bool sharded, size_t occ_bytes, pp2d_mdp** out) {
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

  pp2d_mdp* h = new (std::nothrow) pp2d_mdp;
  if (!h) return fail(PP2D_ERR_INVALID, "out of host memory");
  h->Htot = height; h->W = width; h->row_begin = row_begin;
  h->H = row_end - row_begin; h->gamma = gamma;
  h->sharded = sharded;
  h->device = dev;
  h->sm_count = prop.multiProcessorCount;
  h->pitch = (int)((kPadLeft + width + 128 + 31) / 32 * 32);
  h->plane = (size_t)(h->H + 2 * kPadRows + kSlackRows) * h->pitch;
  h->trapped.push_back(0.0f);
  h->cw2 = env_int("PP2D_MDP_CW2", 2);
  h->cw1 = env_int("PP2D_MDP_CW1", 4);
  h->linear_units = env_int("PP2D_MDP_LINEAR_UNITS", -1);
  h->skip = env_int("PP2D_MDP_SKIP", 1) != 0;
  h->rows_per_unit = env_int("PP2D_MDP_ROWS_PER_UNIT", 0);
  h->p2p_debug = env_int("PP2D_P2P_DEBUG", 0);
  {
    const int lim = env_int("PP2D_P2P_SPIN_LIMIT", 1 << 24);
    h->p2p_spin_limit = lim > 0 ? (unsigned int)lim : 1u;
  }
  h->p2p_edge_short = env_int("PP2D_P2P_EDGE_SHORT", 20);

  const size_t owned = (size_t)h->H * width;
  int rc = [&]() -> int {
    PP2D_CUDA(cudaMalloc(&h->j[0], h->plane * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&h->j[1], h->plane * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&h->jchk, h->plane * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&h->code, h->plane * sizeof(uint16_t)));
    PP2D_CUDA(cudaMalloc(&h->action, owned));
    PP2D_CUDA(cudaMalloc(&h->occ, occ_bytes));
    PP2D_CUDA(cudaMalloc(&h->lut, kLutFloat4 / 8 * sizeof(float4)));
    PP2D_CUDA(cudaMalloc(&h->resid, sizeof(uint32_t)));
    PP2D_CUDA(cudaMalloc(&h->flags, kFlagWords * sizeof(unsigned int)));
    PP2D_CUDA(cudaMemset(h->flags, 0, kFlagWords * sizeof(unsigned int)));
    PP2D_CUDA(cudaMalloc(&h->work, 2 * sizeof(unsigned long long)));
    PP2D_CUDA(cudaMemset(h->work, 0, 2 * sizeof(unsigned long long)));
    PP2D_CUDA(cudaMallocHost(&h->resid_host, sizeof(uint32_t)));
    std::vector<float4> lut;
    build_lut(gamma, lut);
    PP2D_CUDA(cudaMemcpy(h->lut, lut.data(), kLutFloat4 / 8 * sizeof(float4),
                         cudaMemcpyHostToDevice));
    return PP2D_OK;
  }();
  if (rc != PP2D_OK) { pp2d_mdp_destroy(h); return rc; }
  *out = h;
  return PP2D_OK;
}

// ---------------------------------------------------------------------------
// Single-process multi-GPU (pp2d_mdp_create_multi): a container handle whose
// `parts` are ordinary row shards, one per device, driven from the calling
// host thread.  Between neighbouring devices with peer access the ghost rows
// travel inside the fused kernel (direct peer pointers instead of the CUDA-IPC
// mappings of the one-process-per-GPU driver, same flag protocol); otherwise,
// and for single sweeps, they are pulled with cudaMemcpyPeerAsync between
// event-ordered streams.
static int multi_set_device(const pp2d_mdp* part) {
  PP2D_CUDA(cudaSetDevice(part->device));
  return PP2D_OK;
}

// Every part's stream waits for everything its neighbours have enqueued so far.
static int multi_barrier(pp2d_mdp* m) {
  const int n = (int)m->parts.size();
  for (int i = 0; i < n; ++i) {
    PP2D_TRY_MDP(multi_set_device(m->parts[i]));
    PP2D_CUDA(cudaEventRecord(m->ev_done[i], m->parts[i]->stream));
  }
  for (int i = 0; i < n; ++i) {
    PP2D_TRY_MDP(multi_set_device(m->parts[i]));
    if (i > 0) PP2D_CUDA(cudaStreamWaitEvent(m->parts[i]->stream, m->ev_done[i - 1], 0));
    if (i + 1 < n) PP2D_CUDA(cudaStreamWaitEvent(m->parts[i]->stream, m->ev_done[i + 1], 0));
  }
  m->fused_pending = false;
  return PP2D_OK;
}

// Ghost rows of every part pulled from its neighbours' current J planes.
static int multi_exchange(pp2d_mdp* m) {
  const int n = (int)m->parts.size();
  if (n == 1) return PP2D_OK;
  std::vector<pp2d_halo> halo(n);
  for (int i = 0; i < n; ++i) {
    int rc = pp2d_mdp_halo(m->parts[i], &halo[i]);
    if (rc != PP2D_OK) return rc;
    PP2D_TRY_MDP(multi_set_device(m->parts[i]));
    PP2D_CUDA(cudaEventRecord(m->ev_done[i], m->parts[i]->stream));
  }
  for (int i = 0; i < n; ++i) {
    pp2d_mdp* me = m->parts[i];
    PP2D_TRY_MDP(multi_set_device(me));
    if (i > 0) {       // rows H-2, H-1 of the upper neighbour -> my ghost rows -2, -1
      PP2D_CUDA(cudaStreamWaitEvent(me->stream, m->ev_done[i - 1], 0));
      PP2D_CUDA(cudaMemcpyPeerAsync(halo[i].recv_top, me->device, halo[i - 1].send_bottom,
                                    m->parts[i - 1]->device, halo[i].bytes, me->stream));
    }
    if (i + 1 < n) {   // rows 0, 1 of the lower neighbour -> my ghost rows H, H+1
      PP2D_CUDA(cudaStreamWaitEvent(me->stream, m->ev_done[i + 1], 0));
      PP2D_CUDA(cudaMemcpyPeerAsync(halo[i].recv_bottom, me->device, halo[i + 1].send_top,
                                    m->parts[i + 1]->device, halo[i].bytes, me->stream));
    }
    PP2D_CUDA(cudaEventRecord(m->ev_pulled[i], me->stream));
  }
  // nobody overwrites rows a neighbour is still pulling
  for (int i = 0; i < n; ++i) {
    PP2D_TRY_MDP(multi_set_device(m->parts[i]));
    if (i > 0) PP2D_CUDA(cudaStreamWaitEvent(m->parts[i]->stream, m->ev_pulled[i - 1], 0));
    if (i + 1 < n) PP2D_CUDA(cudaStreamWaitEvent(m->parts[i]->stream, m->ev_pulled[i + 1], 0));
  }
  m->fused_pending = false;
  return PP2D_OK;
}

static int multi_sync(pp2d_mdp* m) {
  for (pp2d_mdp* part : m->parts) {
    PP2D_TRY_MDP(multi_set_device(part));
    PP2D_CUDA(cudaStreamSynchronize(part->stream));
  }
  return PP2D_OK;
}

static int multi_sweeps(pp2d_mdp* m, uint32_t n, int want_action) {
  DeviceGuard guard;
  uint32_t left = n;
  while (left > 0) {
    const uint32_t k = left >= 2 ? 2 : 1;
    const bool last = left == k;
    const int wa = want_action && last;
    const bool fused = m->multi_p2p && k == 2;
    if (!fused && m->multi_p2p && m->fused_pending) PP2D_TRY_MDP(multi_barrier(m));
    for (pp2d_mdp* part : m->parts) {
      PP2D_TRY_MDP(multi_set_device(part));
      int rc = pp2d_mdp_sweeps_ex(part, k, wa);
      if (rc != PP2D_OK) return rc;
    }
    if (fused) m->fused_pending = true;
    else PP2D_TRY_MDP(multi_exchange(m));
    left -= k;
  }
  m->n_sweeps += n;
  if (want_action) m->action_sweep = m->n_sweeps;
  m->action_host_valid = false;
  return m->async ? PP2D_OK : multi_sync(m);
}

static int multi_residual(pp2d_mdp* m, float* inf_norm) {
  DeviceGuard guard;
  for (pp2d_mdp* part : m->parts) {
    PP2D_TRY_MDP(multi_set_device(part));
    int rc = pp2d_mdp_residual_device(part, nullptr);
    if (rc != PP2D_OK) return rc;
    PP2D_CUDA(cudaMemcpyAsync(part->resid_host, part->resid, sizeof(uint32_t),
                              cudaMemcpyDeviceToHost, part->stream));
  }
  PP2D_TRY_MDP(multi_sync(m));
  float r = 0.0f;
  for (pp2d_mdp* part : m->parts) {
    float v;
    memcpy(&v, part->resid_host, sizeof(float));
    r = v > r ? v : r;
  }
  *inf_norm = r;
  m->n_chk = m->n_sweeps;
  if (m->multi_p2p && std::isinf(r))
    return fail(PP2D_ERR_STATE, "peer-to-peer ghost-row hand-shake timed out on some device");
  return PP2D_OK;
}

static int multi_reset(pp2d_mdp* m, const uint8_t* map, uint32_t gx, uint32_t gy) {
  DeviceGuard guard;
  PP2D_TRY_MDP(multi_sync(m));               // no device may still write a neighbour's rows
  for (pp2d_mdp* part : m->parts) {
    PP2D_TRY_MDP(multi_set_device(part));
    part->gx = gx;
    part->gy = gy;
    int rc = upload_map(part, map);
    if (rc != PP2D_OK) return rc;
  }
  m->gx = gx;
  m->gy = gy;
  m->n_sweeps = m->n_chk = m->action_sweep = 0;
  m->action_host_valid = false;
  m->fused_pending = false;
  return PP2D_OK;
}

// Each part applies the update rule to its owned and ghost rows from its own
// occupancy rows; the rule is local, so the ghost rows stay equal to what the
// neighbour writes into its owned rows.
static int multi_update_map(pp2d_mdp* m, const uint8_t* map, uint32_t gx, uint32_t gy) {
  DeviceGuard guard;
  PP2D_TRY_MDP(multi_sync(m));               // no device may still write a neighbour's rows
  for (pp2d_mdp* part : m->parts) {
    PP2D_TRY_MDP(multi_set_device(part));
    part->gx = gx;
    part->gy = gy;
    int rc = update_map(part, map);
    if (rc != PP2D_OK) return rc;
  }
  m->gx = gx;
  m->gy = gy;
  m->n_chk = m->n_sweeps;
  m->fused_pending = false;
  return PP2D_OK;
}

static void multi_destroy(pp2d_mdp* m) {
  DeviceGuard guard;
  for (size_t i = 0; i < m->parts.size(); ++i) {
    pp2d_mdp* part = m->parts[i];
    cudaSetDevice(part->device);
    cudaStreamSynchronize(part->stream);
    if (i < m->ev_done.size() && m->ev_done[i]) cudaEventDestroy(m->ev_done[i]);
    if (i < m->ev_pulled.size() && m->ev_pulled[i]) cudaEventDestroy(m->ev_pulled[i]);
  }
  for (pp2d_mdp* part : m->parts) {
    cudaSetDevice(part->device);
    pp2d_mdp_destroy(part);
  }
  m->parts.clear();
}

}  // namespace pp2d

extern "C" {

const char* pp2d_last_error(void) { return g_err; }
int pp2d_abi_version(void) { return 2; }
uint64_t pp2d_kernel_launches(void) { return g_launches.load(); }

int pp2d_mdp_create(uint32_t height, uint32_t width, const uint8_t* map,
                    uint32_t goal_x, uint32_t goal_y, float gamma,
                    pp2d_mdp** out) {
  return create_impl(height, width, map, goal_x, goal_y, gamma, 0, height,
                     false, out);
}

int pp2d_mdp_create_shard(uint32_t height, uint32_t width, const uint8_t* map,
                          uint32_t goal_x, uint32_t goal_y, float gamma,
                          uint32_t row_begin, uint32_t row_end,
                          pp2d_mdp** out) {
  return create_impl(height, width, map, goal_x, goal_y, gamma, row_begin,
                     row_end, true, out);
}

int pp2d_mdp_create_multi(uint32_t height, uint32_t width, const uint8_t* map,
                          uint32_t goal_x, uint32_t goal_y, float gamma, uint32_t ngpus,
                          const int* devices, pp2d_mdp** out) {
  if (!out) return fail(PP2D_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (ngpus == 0) return fail(PP2D_ERR_INVALID, "ngpus must be >= 1");
  if (!map || height == 0 || width == 0) return fail(PP2D_ERR_INVALID, "empty map");
  if (ngpus > 1 && height < (uint32_t)kPadRows * ngpus)
    return fail(PP2D_ERR_INVALID, "%u rows cannot be split over %u devices (each shard needs "
                                  ">= %d rows)", height, ngpus, kPadRows);
  int dev_count = 0;
  PP2D_CUDA(cudaGetDeviceCount(&dev_count));
  if (dev_count == 0) return fail(PP2D_ERR_CUDA, "no CUDA device");
  for (uint32_t i = 0; i < ngpus; ++i) {
    const int d = devices ? devices[i] : (int)i;
    if (d < 0 || d >= dev_count)
      return fail(PP2D_ERR_INVALID, "shard %u wants CUDA device %d but only %d are visible", i, d,
                  dev_count);
  }
  DeviceGuard guard;
  pp2d_mdp* m = new (std::nothrow) pp2d_mdp;
  if (!m) return fail(PP2D_ERR_INVALID, "out of host memory");
  m->Htot = m->H = height; m->W = width; m->gx = goal_x; m->gy = goal_y; m->gamma = gamma;
  int rc = [&]() -> int {
    const uint32_t base = height / ngpus, extra = height % ngpus;
    uint32_t r0 = 0;
    for (uint32_t i = 0; i < ngpus; ++i) {
      const uint32_t r1 = r0 + base + (i < extra ? 1 : 0);
      PP2D_CUDA(cudaSetDevice(devices ? devices[i] : (int)i));
      pp2d_mdp* part = nullptr;
      int rc2 = create_impl(height, width, map, goal_x, goal_y, gamma, r0, r1, ngpus > 1, &part);
      if (rc2 != PP2D_OK) return rc2;
      m->parts.push_back(part);
      PP2D_CUDA(cudaStreamCreateWithFlags(&part->stream, cudaStreamNonBlocking));
      part->owns_stream = true;
      part->async = true;               // the container synchronises
      cudaEvent_t e0 = nullptr, e1 = nullptr;
      PP2D_CUDA(cudaEventCreateWithFlags(&e0, cudaEventDisableTiming));
      m->ev_done.push_back(e0);
      PP2D_CUDA(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
      m->ev_pulled.push_back(e1);
      r0 = r1;
    }
    // Peer-to-peer ghost rows need every neighbouring pair on two different
    // devices with peer access both ways (two shards on ONE device cannot
    // hand-shake inside their kernels: each launch fills the whole GPU, so the
    // neighbour it spins on may not be resident).
    bool p2p = ngpus > 1 && env_int("PP2D_P2P", 1) != 0;
    for (uint32_t i = 0; p2p && i + 1 < ngpus; ++i) {
      const int a = m->parts[i]->device, b = m->parts[i + 1]->device;
      int ab = 0, ba = 0;
      if (a == b) { p2p = false; break; }
      PP2D_CUDA(cudaDeviceCanAccessPeer(&ab, a, b));
      PP2D_CUDA(cudaDeviceCanAccessPeer(&ba, b, a));
      p2p = ab && ba;
    }
    if (p2p) {
      for (uint32_t i = 0; i + 1 < ngpus; ++i) {
        pp2d_mdp *up = m->parts[i], *down = m->parts[i + 1];
        const int pair[2][2] = {{up->device, down->device}, {down->device, up->device}};
        for (auto& pr : pair) {
          PP2D_CUDA(cudaSetDevice(pr[0]));
          cudaError_t e = cudaDeviceEnablePeerAccess(pr[1], 0);
          if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
          PP2D_CUDA(e);
        }
        for (int b = 0; b < 2; ++b) { up->down_j[b] = down->j[b]; down->up_j[b] = up->j[b]; }
        up->down_flags = down->flags;
        down->up_flags = up->flags;
        down->up_H = up->H;
        up->p2p = down->p2p = true;
      }
    }
    m->multi_p2p = p2p;
    return PP2D_OK;
  }();
  if (rc != PP2D_OK) { pp2d_mdp_destroy(m); return rc; }
  *out = m;
  return PP2D_OK;
}

int pp2d_mdp_device_count(const pp2d_mdp* h, int* peer_to_peer) {
  if (!h) return 0;
  if (peer_to_peer) *peer_to_peer = h->parts.empty() ? 0 : (h->multi_p2p ? 1 : 0);
  return h->parts.empty() ? 1 : (int)h->parts.size();
}

// Arguments of a new map and goal on an existing handle (reset, update).
static int check_map_goal(const pp2d_mdp* h, const uint8_t* map, uint32_t goal_x,
                          uint32_t goal_y) {
  if (!h || !map) return fail(PP2D_ERR_INVALID, "NULL argument");
  return check_goal(map, h->W, h->Htot, goal_x, goal_y);
}

int pp2d_mdp_reset(pp2d_mdp* h, const uint8_t* map, uint32_t goal_x,
                   uint32_t goal_y) {
  PP2D_TRY_MDP(check_map_goal(h, map, goal_x, goal_y));
  if (!h->parts.empty()) return multi_reset(h, map, goal_x, goal_y);
  h->gx = goal_x;
  h->gy = goal_y;
  return upload_map(h, map);
}

int pp2d_mdp_update_map(pp2d_mdp* h, const uint8_t* map, uint32_t goal_x, uint32_t goal_y) {
  PP2D_TRY_MDP(check_map_goal(h, map, goal_x, goal_y));
  if (h->pi_mode)
    return fail(PP2D_ERR_STATE, "pp2d_mdp_update_map continues value iteration: the handle "
                                "ran policy iteration, call pp2d_mdp_reset first");
  if (!h->parts.empty()) return multi_update_map(h, map, goal_x, goal_y);
  h->gx = goal_x;
  h->gy = goal_y;
  return update_map(h, map);
}

int pp2d_mdp_stage_map(pp2d_mdp* h, const uint8_t* map) {
  if (!h || !map) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (!h->parts.empty()) {
    DeviceGuard guard;
    for (pp2d_mdp* part : h->parts) {
      PP2D_TRY_MDP(multi_set_device(part));
      PP2D_TRY_MDP(pp2d_mdp_stage_map(part, map));
    }
    return PP2D_OK;
  }
  const OccWindow ow = occ_window(h->row_begin, h->row_begin + h->H, h->Htot);
  const size_t bytes = (size_t)ow.rows * h->W;
  if (!h->upload_stream) {
    PP2D_CUDA(cudaStreamCreateWithFlags(&h->upload_stream, cudaStreamNonBlocking));
    PP2D_CUDA(cudaEventCreateWithFlags(&h->ev_staged, cudaEventDisableTiming));
    PP2D_CUDA(cudaEventCreateWithFlags(&h->ev_code_built, cudaEventDisableTiming));
    PP2D_CUDA(cudaMalloc(&h->occ_next, bytes));
  } else {
    // occ_next was the occupancy buffer of an earlier reset: its code kernel
    // (on the solve stream) must have read it before it is overwritten
    PP2D_CUDA(cudaStreamWaitEvent(h->upload_stream, h->ev_code_built, 0));
  }
  PP2D_CUDA(cudaMemcpyAsync(h->occ_next, map + (size_t)ow.row0 * h->W, bytes,
                            cudaMemcpyHostToDevice, h->upload_stream));
  PP2D_CUDA(cudaEventRecord(h->ev_staged, h->upload_stream));
  h->staged_map = map;
  return PP2D_OK;
}

void pp2d_mdp_destroy(pp2d_mdp* h) {
  if (!h) return;
  if (!h->parts.empty()) multi_destroy(h);
  for (auto& a : h->launch_cache) for (auto& b : a) for (auto& c : b) for (auto& lc : c)
    if (lc.d_unit_lo) { cudaFree(lc.d_unit_lo); lc.d_unit_lo = nullptr; }
  if (h->download_pending) cudaEventSynchronize(h->ev_copied);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->ev_snapshot) cudaEventDestroy(h->ev_snapshot);
  if (h->ev_copied) cudaEventDestroy(h->ev_copied);
  cudaFree(h->dense_action);
  if (h->upload_stream) {
    cudaStreamSynchronize(h->upload_stream);
    cudaStreamDestroy(h->upload_stream);
  }
  if (h->ev_staged) cudaEventDestroy(h->ev_staged);
  if (h->ev_code_built) cudaEventDestroy(h->ev_code_built);
  cudaFree(h->occ_next);
  if (h->owns_stream && h->stream) cudaStreamDestroy(h->stream);
  cudaFree(h->j[0]); cudaFree(h->j[1]); cudaFree(h->jchk); cudaFree(h->code);
  cudaFree(h->action); cudaFree(h->occ); cudaFree(h->dense); cudaFree(h->lut);
  cudaFree(h->resid);
  for (void* q : h->ipc_opened) if (q) cudaIpcCloseMemHandle(q);
  cudaFree(h->flags);
  cudaFree(h->work);
  cudaFree(h->need_alloc);
  if (h->resid_host) cudaFreeHost(h->resid_host);
  delete h;
}

int pp2d_mdp_set_stream(pp2d_mdp* h, void* stream) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  if (!h->parts.empty())
    return fail(PP2D_ERR_STATE, "a multi-GPU handle runs on its own per-device streams");
  h->stream = (cudaStream_t)stream;
  return PP2D_OK;
}

int pp2d_mdp_set_async(pp2d_mdp* h, int async) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  h->async = async != 0;
  return PP2D_OK;
}

int pp2d_mdp_sweeps_ex(pp2d_mdp* h, uint32_t n, int want_action) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  if (n == 0) return PP2D_OK;
  if (!h->parts.empty()) return multi_sweeps(h, n, want_action);
  if (h->sharded && n > 2)
    return fail(PP2D_ERR_STATE,
                "a shard can advance at most 2 sweeps between halo exchanges");
  if (h->pi_mode)
    return fail(PP2D_ERR_STATE, "value-iteration sweeps after pp2d_mdp_policy_iteration "
                                "need a pp2d_mdp_reset first");
  // Ghost rows are good for kPadRows sweeps.  Fused peer-to-peer launches
  // refresh the neighbours' ghost rows themselves; everything else (shards
  // without peer mappings, single sweeps) consumes the budget until the caller
  // exchanges rows through pp2d_mdp_halo.
  const bool has_neighbour = h->sharded && (h->row_begin > 0 || h->row_begin + h->H < h->Htot);
  const bool p2p_fused = h->p2p && n == 2;
  if (has_neighbour && !p2p_fused) {
    if ((int)n > h->halo_budget)
      return fail(PP2D_ERR_STATE,
                  "%u sweep(s) requested but the ghost rows are only good for %d more: "
                  "exchange them first (pp2d_mdp_halo)", n, h->halo_budget);
    h->halo_budget -= (int)n;
  }
  // Value-only sweeps are fused in pairs; when the action grid is wanted the
  // last sweep is the arg-min variant, which leaves exactly what the
  // reference holds after n launches of cudaOneStepValueIteration.
  // With n >= 2 the arg-min sweep is the second half of a fused pair.
  const bool fused_tail = want_action && n >= 2;
  uint32_t plain = want_action ? n - (fused_tail ? 2 : 1) : n;
  int rc;
  while (plain >= 2) {
    if ((rc = launch_sweep_cw<2, false>(h, h->cw2)) != PP2D_OK) return rc;
    plain -= 2;
  }
  if (plain == 1)
    if ((rc = launch_sweep_cw<1, false>(h, h->cw1)) != PP2D_OK) return rc;
  if (want_action) {
    if (fused_tail) rc = launch_sweep_cw<2, true>(h, 2);
    else rc = launch_sweep_cw<1, true>(h, h->cw1);
    if (rc != PP2D_OK) return rc;
    h->action_sweep = h->n_sweeps;
  }
  h->action_host_valid = false;
  return sync_if_needed(h);
}

int pp2d_mdp_sweeps(pp2d_mdp* h, uint32_t n) {
  return pp2d_mdp_sweeps_ex(h, n, 1);
}

uint32_t pp2d_mdp_sweep_count(const pp2d_mdp* h) { return h ? h->n_sweeps : 0; }

int pp2d_mdp_work_counters(pp2d_mdp* h, uint64_t out[2]) {
  if (!h || !out) return fail(PP2D_ERR_INVALID, "NULL argument");
  out[0] = out[1] = 0;
  if (!h->parts.empty()) {
    DeviceGuard guard;
    for (pp2d_mdp* part : h->parts) {
      uint64_t c[2];
      PP2D_TRY_MDP(multi_set_device(part));
      PP2D_TRY_MDP(pp2d_mdp_work_counters(part, c));
      out[0] += c[0];
      out[1] += c[1];
    }
    return PP2D_OK;
  }
  unsigned long long c[2] = {0, 0};
  PP2D_CUDA(cudaMemcpyAsync(c, h->work, sizeof(c), cudaMemcpyDeviceToHost, h->stream));
  PP2D_CUDA(cudaStreamSynchronize(h->stream));
  out[0] = c[0];
  out[1] = c[1];
  return PP2D_OK;
}

int pp2d_mdp_residual_device(pp2d_mdp* h, void** dev_float_out) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  if (!h->parts.empty())
    return fail(PP2D_ERR_STATE, "pp2d_mdp_residual_device: use pp2d_mdp_residual on a "
                                "multi-GPU handle");
  PP2D_CUDA(cudaMemsetAsync(h->resid, 0, sizeof(uint32_t), h->stream));
  // Occupied cells are stored as 0; their change since the last check point
  // is the closed form and enters the reduction as a floor value.
  float floor_val = 0.0f;
  if (h->has_occupied)
    floor_val = fabsf(occupied_cost(h, h->n_sweeps) - occupied_cost(h, h->n_chk));
  uint32_t floor_bits;
  memcpy(&floor_bits, &floor_val, sizeof(floor_bits));
  // Owned rows only (ghost rows belong to the neighbours).
  const size_t off = (size_t)kPadRows * h->pitch;
  const size_t n4 = (size_t)h->H * h->pitch / 4;
  int grid = h->sm_count * 8;
  if ((size_t)grid * 256 > n4) grid = (int)((n4 + 255) / 256);
  if (grid < 1) grid = 1;
  if (h->chk_is_zero)
    mdp_residual_kernel<true><<<grid, 256, 0, h->stream>>>(
        reinterpret_cast<const float4*>(h->j[h->cur] + off),
        reinterpret_cast<float4*>(h->jchk + off), n4, floor_bits, h->resid,
        h->p2p ? h->flags + kFlagError : nullptr);
  else
    mdp_residual_kernel<false><<<grid, 256, 0, h->stream>>>(
        reinterpret_cast<const float4*>(h->j[h->cur] + off),
        reinterpret_cast<float4*>(h->jchk + off), n4, floor_bits, h->resid,
        h->p2p ? h->flags + kFlagError : nullptr);
  h->chk_is_zero = false;
  g_launches.fetch_add(1, std::memory_order_relaxed);
  PP2D_CUDA(cudaGetLastError());
  h->n_chk = h->n_sweeps;
  if (dev_float_out) *dev_float_out = h->resid;
  return sync_if_needed(h);
}

int pp2d_mdp_residual(pp2d_mdp* h, float* inf_norm) {
  if (!h || !inf_norm) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (!h->parts.empty()) return multi_residual(h, inf_norm);
  int rc = pp2d_mdp_residual_device(h, nullptr);
  if (rc != PP2D_OK) return rc;
  PP2D_CUDA(cudaMemcpyAsync(h->resid_host, h->resid, sizeof(uint32_t),
                            cudaMemcpyDeviceToHost, h->stream));
  PP2D_CUDA(cudaStreamSynchronize(h->stream));
  memcpy(inf_norm, h->resid_host, sizeof(float));
  if (h->p2p && std::isinf(*inf_norm))
    return fail(PP2D_ERR_STATE, "peer-to-peer ghost-row hand-shake timed out "
                                "(a neighbour shard did not run the same launches)");
  return PP2D_OK;
}

int pp2d_mdp_solve(pp2d_mdp* h, uint32_t* sweeps_out, double* residuals,
                   uint32_t max_residuals) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  if (h->sharded)
    return fail(PP2D_ERR_STATE, "pp2d_mdp_solve needs an unsharded handle");
  // path_planning_2d.cu:219-263.
  double cost_inf_norm = 0.0;
  uint32_t batch = 0, total = 0;
  do {
    int rc = pp2d_mdp_sweeps(h, 100);
    if (rc != PP2D_OK) return rc;
    total += 100;
    float r = 0.f;
    rc = pp2d_mdp_residual(h, &r);
    if (rc != PP2D_OK) return rc;
    cost_inf_norm = r;
    if (residuals && batch < max_residuals) residuals[batch] = cost_inf_norm;
    ++batch;
  } while (keeps_sweeping(cost_inf_norm, h->gamma));
  if (sweeps_out) *sweeps_out = total;
  return PP2D_OK;
}

int pp2d_mdp_policy_iteration(pp2d_mdp* h, uint32_t* evaluation_sweeps, double* residuals,
                              uint32_t* changed, uint32_t capacity, uint32_t max_rounds) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  if (h->sharded || !h->parts.empty())
    return fail(PP2D_ERR_STATE, "pp2d_mdp_policy_iteration needs an unsharded single-GPU handle");
  if (h->n_sweeps != 0)
    return fail(PP2D_ERR_STATE, "pp2d_mdp_policy_iteration starts from J = 0, action = 0: "
                                "call pp2d_mdp_reset first");
  h->pi_mode = true;
  h->need_valid = false;
  const size_t owned = (size_t)h->H * h->W;
  PolicyParams p;
  p.code = h->code; p.action = h->action;
  p.W = (int)h->W; p.H = (int)h->H; p.pitch = h->pitch; p.gamma = h->gamma;
  dim3 grid((h->W + 255) / 256, h->H);
  std::vector<uint8_t> a_prev(owned, 0), a_curr(owned);
  // path_planning_2d.cu:271-357
  double cost_inf_norm = 0.0;
  uint32_t round = 0;
  do {
    for (int i = 0; i < 50; ++i) {                     // 25 ping-pong pairs
      p.jin = h->j[h->cur];
      p.jout = h->j[h->cur ^ 1];
      mdp_policy_kernel<false><<<grid, 256, 0, h->stream>>>(p);
      g_launches.fetch_add(1, std::memory_order_relaxed);
      h->cur ^= 1;
      h->n_sweeps += 1;
    }
    PP2D_CUDA(cudaGetLastError());
    float r = 0.f;
    int rc = pp2d_mdp_residual(h, &r);
    if (rc != PP2D_OK) return rc;
    cost_inf_norm = r;
    p.jin = h->j[h->cur];
    p.jout = nullptr;
    mdp_policy_kernel<true><<<grid, 256, 0, h->stream>>>(p);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    PP2D_CUDA(cudaGetLastError());
    h->action_sweep = h->n_sweeps;
    h->action_host_valid = false;
    if (changed) {                                      // "# of changed actions", :343-347
      PP2D_CUDA(cudaMemcpyAsync(a_curr.data(), h->action, owned, cudaMemcpyDeviceToHost,
                                h->stream));
      PP2D_CUDA(cudaStreamSynchronize(h->stream));
      uint32_t diff = 0;
      for (size_t i = 0; i < owned; ++i) diff += a_prev[i] != a_curr[i];
      a_prev.swap(a_curr);
      if (round < capacity) changed[round] = diff;
    }
    if (residuals && round < capacity) residuals[round] = cost_inf_norm;
    ++round;
    if (max_rounds > 0 && round >= max_rounds) break;
  } while (keeps_sweeping(cost_inf_norm, h->gamma));
  if (evaluation_sweeps) *evaluation_sweeps = h->n_sweeps;
  return sync_if_needed(h);
}

int pp2d_mdp_download_begin(pp2d_mdp* h, float* cost, uint8_t* action) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  if (!h->parts.empty()) {
    DeviceGuard guard;
    if (h->multi_p2p && h->fused_pending) PP2D_TRY_MDP(multi_barrier(h));
    for (pp2d_mdp* part : h->parts) {
      PP2D_TRY_MDP(multi_set_device(part));
      const size_t off = (size_t)part->row_begin * h->W;
      int rc = pp2d_mdp_download_begin(part, cost ? cost + off : nullptr,
                                       action ? action + off : nullptr);
      if (rc != PP2D_OK) return rc;
    }
    return PP2D_OK;
  }
  const size_t owned = (size_t)h->H * h->W;
  if (!h->copy_stream) {
    PP2D_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    PP2D_CUDA(cudaEventCreateWithFlags(&h->ev_snapshot, cudaEventDisableTiming));
    PP2D_CUDA(cudaEventCreateWithFlags(&h->ev_copied, cudaEventDisableTiming));
  }
  // the staging buffers may still be feeding an earlier download
  if (h->download_pending) PP2D_CUDA(cudaStreamWaitEvent(h->stream, h->ev_copied, 0));
  if (cost) {
    if (!h->dense) PP2D_CUDA(cudaMalloc(&h->dense, owned * sizeof(float)));
    if ((h->W & 3) == 0 && (kPadLeft & 3) == 0) {
      dim3 grid((h->W / 4 + 255) / 256, h->H);
      mdp_export_kernel<true><<<grid, 256, 0, h->stream>>>(
          h->j[h->cur], h->code, h->dense, (int)h->W, (int)h->H, h->pitch,
          occupied_cost(h, h->n_sweeps));
    } else {
      dim3 grid((h->W + 255) / 256, h->H);
      mdp_export_kernel<false><<<grid, 256, 0, h->stream>>>(
          h->j[h->cur], h->code, h->dense, (int)h->W, (int)h->H, h->pitch,
          occupied_cost(h, h->n_sweeps));
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    PP2D_CUDA(cudaGetLastError());
  }
  if (action) {
    if (!h->dense_action) PP2D_CUDA(cudaMalloc(&h->dense_action, owned));
    PP2D_CUDA(cudaMemcpyAsync(h->dense_action, h->action, owned, cudaMemcpyDeviceToDevice,
                              h->stream));
  }
  PP2D_CUDA(cudaEventRecord(h->ev_snapshot, h->stream));
  PP2D_CUDA(cudaStreamWaitEvent(h->copy_stream, h->ev_snapshot, 0));
  if (cost)
    PP2D_CUDA(cudaMemcpyAsync(cost, h->dense, owned * sizeof(float), cudaMemcpyDeviceToHost,
                              h->copy_stream));
  if (action)
    PP2D_CUDA(cudaMemcpyAsync(action, h->dense_action, owned, cudaMemcpyDeviceToHost,
                              h->copy_stream));
  PP2D_CUDA(cudaEventRecord(h->ev_copied, h->copy_stream));
  h->download_pending = true;
  return PP2D_OK;
}

int pp2d_mdp_download_wait(pp2d_mdp* h) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  if (!h->parts.empty()) {
    DeviceGuard guard;
    for (pp2d_mdp* part : h->parts) {
      PP2D_TRY_MDP(multi_set_device(part));
      int rc = pp2d_mdp_download_wait(part);
      if (rc != PP2D_OK) return rc;
    }
    return PP2D_OK;
  }
  if (h->download_pending) {
    PP2D_CUDA(cudaEventSynchronize(h->ev_copied));
    h->download_pending = false;
  }
  if (h->p2p) {
    int timed_out = 0;
    int rc = pp2d_mdp_p2p_status(h, &timed_out);
    if (rc != PP2D_OK) return rc;
    if (timed_out)
      return fail(PP2D_ERR_STATE, "peer-to-peer ghost-row hand-shake timed out: J and the "
                                  "action grid of this shard are invalid");
  }
  return PP2D_OK;
}

int pp2d_mdp_download(pp2d_mdp* h, float* cost, uint8_t* action) {
  int rc = pp2d_mdp_download_begin(h, cost, action);
  if (rc != PP2D_OK) return rc;
  return pp2d_mdp_download_wait(h);
}

int pp2d_mdp_plan_batch(pp2d_mdp* h, const float* beliefs, uint32_t n_beliefs,
                        uint8_t* actions) {
  if (!h || !beliefs || !actions) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (h->sharded)
    return fail(PP2D_ERR_STATE, "pp2d_mdp_plan needs an unsharded handle");
  if (n_beliefs == 0) return PP2D_OK;
  const size_t n = (size_t)h->H * h->W;
  const bool multi = !h->parts.empty();
  DeviceGuard guard;
  cudaStream_t stream = h->stream;
  if (multi) {
    // the belief scan runs on the first device; the action grid is spread over
    // the devices, so the host copy (downloaded once per solve) is consulted
    if (!h->action_host_valid) {
      h->action_host.resize(n);
      int rc = pp2d_mdp_download(h, nullptr, h->action_host.data());
      if (rc != PP2D_OK) return rc;
      h->action_host_valid = true;
    }
    PP2D_CUDA(cudaSetDevice(h->parts[0]->device));
    stream = h->parts[0]->stream;
  }
  float* d_b = nullptr;
  uint8_t* d_a = nullptr;
  unsigned long long* d_i = nullptr;
  PP2D_CUDA(cudaMalloc(&d_b, n * n_beliefs * sizeof(float)));
  cudaError_t e = multi ? cudaMalloc(&d_i, n_beliefs * sizeof(unsigned long long))
                        : cudaMalloc(&d_a, n_beliefs);
  if (e != cudaSuccess) { cudaFree(d_b); PP2D_CUDA(e); }
  int rc = [&]() -> int {
    PP2D_CUDA(cudaMemcpyAsync(d_b, beliefs, n * n_beliefs * sizeof(float),
                              cudaMemcpyHostToDevice, stream));
    mdp_plan_kernel<<<n_beliefs, 256, 0, stream>>>(d_b, n, multi ? nullptr : h->action, d_a, d_i);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    PP2D_CUDA(cudaGetLastError());
    if (multi) {
      std::vector<unsigned long long> idx(n_beliefs);
      PP2D_CUDA(cudaMemcpyAsync(idx.data(), d_i, n_beliefs * sizeof(unsigned long long),
                                cudaMemcpyDeviceToHost, stream));
      PP2D_CUDA(cudaStreamSynchronize(stream));
      for (uint32_t i = 0; i < n_beliefs; ++i) actions[i] = h->action_host[idx[i]];
    } else {
      PP2D_CUDA(cudaMemcpyAsync(actions, d_a, n_beliefs, cudaMemcpyDeviceToHost, stream));
      PP2D_CUDA(cudaStreamSynchronize(stream));
    }
    return PP2D_OK;
  }();
  cudaFree(d_b);
  cudaFree(d_a);
  cudaFree(d_i);
  return rc;
}

int pp2d_mdp_plan(pp2d_mdp* h, const float* belief, uint8_t* action) {
  return pp2d_mdp_plan_batch(h, belief, 1, action);
}

// Greedy rollout of a dense H x W action grid from (sx, sy): follow
// (u%3-1, u/3-1) until action 4 (stay), the map border or max_len cells;
// returns the number of cells written.
static uint32_t rollout(const uint8_t* action, uint32_t W, uint32_t H, uint32_t sx, uint32_t sy,
                        uint32_t* cells, uint32_t max_len) {
  uint32_t n = 0;
  int64_t x = sx, y = sy;
  while (n < max_len && x >= 0 && x < (int64_t)W && y >= 0 && y < (int64_t)H) {
    cells[n++] = (uint32_t)(y * W + x);
    const uint8_t u = action[(size_t)y * W + x];
    if (u == 4) break;
    x += (int)(u % 3) - 1;   // path_planning_2d_cuda.cu:83-88
    y += (int)(u / 3) - 1;
  }
  return n;
}

int pp2d_mdp_waypoints(pp2d_mdp* h, uint32_t sx, uint32_t sy, uint32_t* cells,
                       uint32_t max_len, uint32_t* n_out) {
  if (!h || !cells || !n_out) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (h->sharded)
    return fail(PP2D_ERR_STATE, "pp2d_mdp_waypoints needs an unsharded handle");
  if (sx >= h->W || sy >= h->H)
    return fail(PP2D_ERR_INVALID, "start (%u %u) outside the map", sx, sy);
  if (!h->action_host_valid) {
    h->action_host.resize((size_t)h->H * h->W);
    int rc = pp2d_mdp_download(h, nullptr, h->action_host.data());
    if (rc != PP2D_OK) return rc;
    h->action_host_valid = true;
  }
  *n_out = rollout(h->action_host.data(), h->W, h->H, sx, sy, cells, max_len);
  return PP2D_OK;
}

namespace {
struct IpcDesc {
  cudaIpcMemHandle_t j[2];
  cudaIpcMemHandle_t flags;
  uint32_t H, pitch, W, magic;
};
static_assert(sizeof(IpcDesc) <= PP2D_IPC_DESC_BYTES, "IPC descriptor too large");
}  // namespace

int pp2d_mdp_ipc_export(pp2d_mdp* h, void* desc) {
  if (!h || !desc) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (!h->parts.empty()) return fail(PP2D_ERR_STATE, "not a shard handle");
  IpcDesc d;
  memset(&d, 0, sizeof(d));
  PP2D_CUDA(cudaIpcGetMemHandle(&d.j[0], h->j[0]));
  PP2D_CUDA(cudaIpcGetMemHandle(&d.j[1], h->j[1]));
  PP2D_CUDA(cudaIpcGetMemHandle(&d.flags, h->flags));
  d.H = h->H; d.pitch = (uint32_t)h->pitch; d.W = h->W; d.magic = 0x70703264u;
  memset(desc, 0, PP2D_IPC_DESC_BYTES);
  memcpy(desc, &d, sizeof(d));
  return PP2D_OK;
}

int pp2d_mdp_ipc_connect(pp2d_mdp* h, const void* up_desc, const void* down_desc) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  if (!h->sharded) return fail(PP2D_ERR_STATE, "peer-to-peer needs a shard handle");
  if (h->p2p) return fail(PP2D_ERR_STATE, "already connected");
  if (h->n_sweeps != 0) return fail(PP2D_ERR_STATE, "connect before the first sweep");
  int slot = 0;
  auto open = [&](const void* src, float** j, unsigned int** flags, uint32_t* H) -> int {
    IpcDesc d;
    memcpy(&d, src, sizeof(d));
    if (d.magic != 0x70703264u || d.pitch != (uint32_t)h->pitch || d.W != h->W)
      return fail(PP2D_ERR_INVALID, "neighbour descriptor does not match this shard");
    for (int b = 0; b < 2; ++b) {
      void* q = nullptr;
      PP2D_CUDA(cudaIpcOpenMemHandle(&q, d.j[b], cudaIpcMemLazyEnablePeerAccess));
      h->ipc_opened[slot++] = q;
      j[b] = static_cast<float*>(q);
    }
    void* q = nullptr;
    PP2D_CUDA(cudaIpcOpenMemHandle(&q, d.flags, cudaIpcMemLazyEnablePeerAccess));
    h->ipc_opened[slot++] = q;
    *flags = static_cast<unsigned int*>(q);
    if (H) *H = d.H;
    return PP2D_OK;
  };
  if (up_desc) {
    int rc = open(up_desc, h->up_j, &h->up_flags, &h->up_H);
    if (rc != PP2D_OK) return rc;
  }
  if (down_desc) {
    int rc = open(down_desc, h->down_j, &h->down_flags, nullptr);
    if (rc != PP2D_OK) return rc;
  }
  h->p2p = (up_desc != nullptr) || (down_desc != nullptr);
  return PP2D_OK;
}

int pp2d_mdp_p2p_status(pp2d_mdp* h, int* timed_out) {
  if (!h || !timed_out) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (!h->parts.empty()) {
    DeviceGuard guard;
    *timed_out = 0;
    for (pp2d_mdp* part : h->parts) {
      int t = 0;
      PP2D_CUDA(cudaSetDevice(part->device));
      int rc = pp2d_mdp_p2p_status(part, &t);
      if (rc != PP2D_OK) return rc;
      *timed_out |= t;
    }
    return PP2D_OK;
  }
  unsigned int e = 0;
  PP2D_CUDA(cudaMemcpyAsync(&e, h->flags + kFlagError, sizeof(e), cudaMemcpyDeviceToHost,
                            h->stream));
  PP2D_CUDA(cudaStreamSynchronize(h->stream));
  *timed_out = (int)e;
  return PP2D_OK;
}

int pp2d_mdp_halo(pp2d_mdp* h, pp2d_halo* out) {
  if (!h || !out) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (!h->parts.empty()) return fail(PP2D_ERR_STATE, "not a shard handle");
  float* j = h->j[h->cur];
  const size_t row = (size_t)h->pitch;
  out->recv_top = j;                                       // rows -2, -1
  out->send_top = j + kPadRows * row;                      // rows 0, 1
  out->send_bottom = j + (size_t)h->H * row;               // rows H-2, H-1
  out->recv_bottom = j + (size_t)(h->H + kPadRows) * row;  // rows H, H+1
  out->bytes = kPadRows * row * sizeof(float);
  h->halo_budget = kPadRows;     // the caller is about to refresh the ghost rows
  return PP2D_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------
// Batches of equal-size instances (pp2d_mdp_batch_*, DESIGN.md section 4): the
// instances are stacked into one tall grid with an occupied separator row
// between neighbours, and an ordinary handle (`grid`) runs its fused sweeps
// unchanged.  The batch adds the per-instance codes, residuals, stopping and
// results around it.
struct pp2d_mdp_batch {
  pp2d_mdp* grid = nullptr;        // the tall grid; grid->occ holds the maps
  uint32_t H = 0, W = 0, count = 0;
  size_t map_stride = 0;           // device: H*W, or 0 for one shared map
  uint32_t* goals = nullptr;       // device [count][2]
  std::vector<uint32_t> goals_host;
  std::vector<uint8_t> has_occ;    // instance k's own map has an occupied cell
  uint8_t* frozen_dev = nullptr;   // device [count]
  std::vector<uint8_t> frozen;     // instance k met the stopping rule in solve
  uint32_t n_frozen = 0;
  std::vector<uint32_t> stop_sweeps;   // sweep count of a frozen instance
  // Sweep count and check point of a live instance minus the grid's
  // n_sweeps and n_chk (mod 2^32): 0 until an update re-activates an instance
  // that stopped at another count, or gives one a new check point.
  std::vector<uint32_t> sweep_off, chk_off;
  // device [3][count]: instances of the next kernel, then up to two arrays of
  // one 32-bit value per listed instance (upload_list)
  uint32_t* list = nullptr;
  std::vector<uint32_t> list_host;
  uint32_t* resid = nullptr;       // device [count] float bits
  std::vector<uint32_t> resid_host;
  float* res_cost = nullptr;       // device [count][H][W]: snapshots and downloads
  uint8_t* res_action = nullptr;   // device [count][H][W]
};

namespace pp2d {

// Arguments of a batch (create and reset).  The size check comes first: it
// reads neither the maps nor the goals.
static int batch_check(uint32_t height, uint32_t width, uint32_t count, const uint8_t* maps,
                       size_t map_stride, const uint32_t* goals) {
  if (!maps || !goals) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (height == 0 || width == 0) return fail(PP2D_ERR_INVALID, "empty map");
  if (count == 0) return fail(PP2D_ERR_INVALID, "a batch needs at least one instance");
  const uint64_t hw = (uint64_t)height * width;
  if (map_stride != 0 && map_stride < hw)
    return fail(PP2D_ERR_INVALID, "map_stride %zu is below height*width = %llu", map_stride,
                (unsigned long long)hw);
  // the kernels index rows, units and plane elements of the tall grid with int
  const uint64_t rows = (uint64_t)count * (height + 1ull) - 1;
  const uint64_t pitch = (kPadLeft + (uint64_t)width + 128 + 31) / 32 * 32;
  const uint64_t plane = (rows + 2 * kPadRows + kSlackRows) * pitch;
  if (rows > (uint64_t)INT32_MAX || plane > (uint64_t)INT32_MAX)
    return fail(PP2D_ERR_INVALID, "%u instances of %ux%u stack to a grid of %llu rows x %llu "
                                  "columns: too large for one batch", count, width, height,
                (unsigned long long)rows, (unsigned long long)pitch);
  for (uint32_t k = 0; k < count; ++k)
    PP2D_TRY_MDP(check_goal(maps + k * map_stride, width, height, goals[2 * (size_t)k],
                            goals[2 * (size_t)k + 1], k));
  return PP2D_OK;
}

// Maps i = 0 .. n-1 at maps + i * map_stride (map_stride 0: one map) to the
// front of g->occ, back to back; a shared map is copied once.
static int upload_maps(pp2d_mdp* g, const uint8_t* maps, size_t map_stride, size_t hw,
                       uint32_t n) {
  if (map_stride == 0 || map_stride == hw)
    PP2D_CUDA(cudaMemcpyAsync(g->occ, maps, (map_stride ? n : 1) * hw, cudaMemcpyHostToDevice,
                              g->stream));
  else
    PP2D_CUDA(cudaMemcpy2DAsync(g->occ, hw, maps, map_stride, hw, n, cudaMemcpyHostToDevice,
                                g->stream));
  return PP2D_OK;
}

// Maps, goals and codes of a checked batch; J = 0, actions = 0, sweep count 0.
static int batch_upload(pp2d_mdp_batch* b, const uint8_t* maps, size_t map_stride,
                        const uint32_t* goals) {
  pp2d_mdp* g = b->grid;
  const size_t hw = (size_t)b->H * b->W;
  PP2D_CUDA(cudaMemsetAsync(g->j[0], 0, g->plane * sizeof(float), g->stream));
  PP2D_CUDA(cudaMemsetAsync(g->j[1], 0, g->plane * sizeof(float), g->stream));
  PP2D_CUDA(cudaMemsetAsync(g->jchk, 0, g->plane * sizeof(float), g->stream));
  PP2D_CUDA(cudaMemsetAsync(g->action, 0, (size_t)g->H * g->W, g->stream));
  PP2D_TRY_MDP(upload_maps(g, maps, map_stride, hw, b->count));
  b->map_stride = map_stride ? hw : 0;
  b->goals_host.assign(goals, goals + 2 * (size_t)b->count);
  PP2D_CUDA(cudaMemcpyAsync(b->goals, goals, 2 * sizeof(uint32_t) * b->count,
                            cudaMemcpyHostToDevice, g->stream));
  for (uint32_t k = 0; k < b->count; ++k)
    b->has_occ[k] = (map_stride == 0 && k > 0)
                        ? b->has_occ[0]
                        : memchr(maps + k * map_stride, 1, hw) != nullptr;
  std::fill(b->frozen.begin(), b->frozen.end(), 0);
  b->n_frozen = 0;
  std::fill(b->stop_sweeps.begin(), b->stop_sweeps.end(), 0);
  std::fill(b->sweep_off.begin(), b->sweep_off.end(), 0);
  std::fill(b->chk_off.begin(), b->chk_off.end(), 0);
  PP2D_CUDA(cudaMemsetAsync(b->frozen_dev, 0, b->count, g->stream));
  BatchCodeParams cp;
  cp.maps = g->occ; cp.map_stride = b->map_stride; cp.goals = b->goals; cp.code = g->code;
  cp.W = (int)b->W; cp.H = (int)b->H; cp.count = (int)b->count; cp.pitch = g->pitch;
  cp.rows_phys = (int)g->H + 2 * kPadRows;
  const int row_groups = (cp.rows_phys + kCodeRows - 1) / kCodeRows;
  dim3 grid((g->pitch / 4 + kCodeThreads - 1) / kCodeThreads, std::min(row_groups, 65535));
  mdp_batch_code_kernel<<<grid, kCodeThreads, 0, g->stream>>>(cp);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  PP2D_CUDA(cudaGetLastError());
  // (the caller may free the maps on return)
  PP2D_CUDA(cudaStreamSynchronize(g->stream));
  g->cur = 0;
  g->n_sweeps = g->n_chk = g->action_sweep = 0;
  g->action_host_valid = false;
  g->pi_mode = false;
  g->need_valid = false;
  return PP2D_OK;
}

// Sweep count and check point of instance k.
static uint32_t batch_sweeps_of(const pp2d_mdp_batch* b, uint32_t k) {
  return b->frozen[k] ? b->stop_sweeps[k] : b->grid->n_sweeps + b->sweep_off[k];
}
static uint32_t batch_chk_of(const pp2d_mdp_batch* b, uint32_t k) {
  return b->grid->n_chk + b->chk_off[k];
}
// Instance k's action grid (H*W bytes): its snapshot once frozen, else its
// rows of the live grid.
static const uint8_t* batch_actions_of(const pp2d_mdp_batch* b, uint32_t k) {
  return b->frozen[k] ? b->res_action + k * (size_t)b->H * b->W
                      : b->grid->action + (size_t)k * (b->H + 1) * b->W;
}
static uint32_t word_of(float v) {
  uint32_t w;
  memcpy(&w, &v, sizeof(w));
  return w;
}

// Host side of b->list: the n instances of the next kernel, then `arrays`
// arrays of one 32-bit value per listed instance (array a at (a + 1) * n,
// filled by the caller), all sent by one upload_list.
static uint32_t* stage_list(pp2d_mdp_batch* b, const std::vector<uint32_t>& list, int arrays) {
  const size_t n = list.size();
  b->list_host.resize((size_t)(arrays + 1) * n);
  std::copy(list.begin(), list.end(), b->list_host.begin());
  return b->list_host.data();
}
static int upload_list(pp2d_mdp_batch* b) {
  PP2D_CUDA(cudaMemcpyAsync(b->list, b->list_host.data(), b->list_host.size() * sizeof(uint32_t),
                            cudaMemcpyHostToDevice, b->grid->stream));
  return PP2D_OK;
}

// Residuals of the instances in `list` into b->resid_host (one launch, one
// round trip).
static int batch_residual(pp2d_mdp_batch* b, const std::vector<uint32_t>& list) {
  pp2d_mdp* g = b->grid;
  const size_t n = list.size();
  uint32_t* words = stage_list(b, list, 1);
  for (size_t i = 0; i < n; ++i) {
    const uint32_t k = list[i];
    words[n + i] = word_of(b->has_occ[k] ? fabsf(trapped_cost(g, batch_sweeps_of(b, k)) -
                                                 trapped_cost(g, batch_chk_of(b, k)))
                                         : 0.0f);
  }
  PP2D_TRY_MDP(upload_list(b));
  PP2D_CUDA(cudaMemsetAsync(b->resid, 0, b->count * sizeof(uint32_t), g->stream));
  const size_t n4 = (size_t)b->H * g->pitch / 4;
  const size_t fill = std::max<size_t>(1, (size_t)g->sm_count * 8 / n);
  const int blocks_per = (int)std::min((n4 + 255) / 256, fill);
  mdp_batch_residual_kernel<<<(unsigned)(n * blocks_per), 256, 0, g->stream>>>(
      g->j[g->cur], g->jchk, b->list, reinterpret_cast<const float*>(b->list + n), blocks_per,
      (int)b->H, g->pitch, b->resid);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  PP2D_CUDA(cudaGetLastError());
  g->n_chk = g->n_sweeps;
  for (uint32_t k : list) b->chk_off[k] = b->sweep_off[k];
  PP2D_CUDA(cudaMemcpyAsync(b->resid_host.data(), b->resid, b->count * sizeof(uint32_t),
                            cudaMemcpyDeviceToHost, g->stream));
  PP2D_CUDA(cudaStreamSynchronize(g->stream));
  return PP2D_OK;
}

// Snapshot of the instances in `list` into their result slots; FREEZE: they
// just stopped (b->frozen already says so) and leave the live grid.
template <bool FREEZE>
static int batch_snapshot(pp2d_mdp_batch* b, const std::vector<uint32_t>& list) {
  pp2d_mdp* g = b->grid;
  const size_t n = list.size();
  uint32_t* words = stage_list(b, list, 1);
  for (size_t i = 0; i < n; ++i)
    words[n + i] = word_of(trapped_cost(g, batch_sweeps_of(b, list[i])));
  PP2D_TRY_MDP(upload_list(b));
  BatchFreezeParams p;
  memset(&p, 0, sizeof(p));
  p.j[0] = g->j[0]; p.j[1] = g->j[1]; p.cur = g->cur;
  p.code = g->code; p.action = g->action;
  p.res_cost = b->res_cost; p.res_action = b->res_action;
  p.list = b->list; p.n_list = (int)n;
  p.trapped = reinterpret_cast<const float*>(b->list + n);
  p.W = (int)b->W; p.H = (int)b->H; p.pitch = g->pitch;
  if (FREEZE) {
    PP2D_CUDA(cudaMemcpyAsync(b->frozen_dev, b->frozen.data(), b->count,
                              cudaMemcpyHostToDevice, g->stream));
    p.frozen = b->frozen_dev;
    p.count = (int)b->count;
    p.Htot = (int)g->H;
    // (seeded by the arg-min launch that ended the batch)
    p.mask = next_unit_mask(g);
  }
  const size_t work = std::max<size_t>((size_t)list.size() * b->H * b->W, (size_t)p.mask.n_rb);
  const int grid = (int)std::min<size_t>((work + 255) / 256, (size_t)g->sm_count * 16);
  mdp_batch_freeze_kernel<FREEZE><<<std::max(grid, 1), 256, 0, g->stream>>>(p);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  PP2D_CUDA(cudaGetLastError());
  return PP2D_OK;
}

// Accessors of handles.h (the closed-loop rollouts of rollout.cu).
PlannerView mdp_view(const pp2d_mdp* h) {
  PlannerView v;
  v.H = h->H; v.W = h->W;
  v.sharded = h->sharded || !h->parts.empty();
  v.action = h->action;
  v.gx = h->gx; v.gy = h->gy;
  v.stream = h->stream;
  return v;
}
uint32_t mdp_batch_count(const pp2d_mdp_batch* b) { return b->count; }
PlannerView mdp_batch_view(const pp2d_mdp_batch* b, uint32_t k) {
  PlannerView v;
  v.H = b->H; v.W = b->W;
  v.action = batch_actions_of(b, k);
  v.gx = b->goals_host[2 * (size_t)k]; v.gy = b->goals_host[2 * (size_t)k + 1];
  v.stream = b->grid->stream;
  return v;
}

}  // namespace pp2d

extern "C" {

int pp2d_mdp_batch_create(uint32_t height, uint32_t width, uint32_t count, const uint8_t* maps,
                          size_t map_stride, const uint32_t* goals_xy, float gamma,
                          pp2d_mdp_batch** out) {
  if (!out) return fail(PP2D_ERR_INVALID, "out is NULL");
  *out = nullptr;
  PP2D_TRY_MDP(batch_check(height, width, count, maps, map_stride, goals_xy));
  const uint32_t rows = count * (height + 1) - 1;
  const size_t hw = (size_t)height * width;
  pp2d_mdp* g = nullptr;
  // room for one map per instance whatever this call passes: a later reset
  // may switch from a shared map to per-instance maps
  PP2D_TRY_MDP(make_handle(rows, width, gamma, 0, rows, false, (size_t)count * hw, &g));
  pp2d_mdp_batch* b = new (std::nothrow) pp2d_mdp_batch;
  if (!b) { pp2d_mdp_destroy(g); return fail(PP2D_ERR_INVALID, "out of host memory"); }
  b->grid = g;
  b->H = height; b->W = width; b->count = count;
  b->has_occ.assign(count, 0);
  b->frozen.assign(count, 0);
  b->stop_sweeps.assign(count, 0);
  b->sweep_off.assign(count, 0);
  b->chk_off.assign(count, 0);
  b->resid_host.assign(count, 0);
  int rc = [&]() -> int {
    PP2D_CUDA(cudaMalloc(&b->goals, 2 * sizeof(uint32_t) * count));
    PP2D_CUDA(cudaMalloc(&b->frozen_dev, count));
    PP2D_CUDA(cudaMalloc(&b->list, 3 * (size_t)count * sizeof(uint32_t)));
    PP2D_CUDA(cudaMalloc(&b->resid, count * sizeof(uint32_t)));
    PP2D_CUDA(cudaMalloc(&b->res_cost, count * hw * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&b->res_action, count * hw));
    return batch_upload(b, maps, map_stride, goals_xy);
  }();
  if (rc != PP2D_OK) { pp2d_mdp_batch_destroy(b); return rc; }
  *out = b;
  return PP2D_OK;
}

int pp2d_mdp_batch_reset(pp2d_mdp_batch* h, const uint8_t* maps, size_t map_stride,
                         const uint32_t* goals_xy) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  PP2D_TRY_MDP(batch_check(h->H, h->W, h->count, maps, map_stride, goals_xy));
  return batch_upload(h, maps, map_stride, goals_xy);
}

void pp2d_mdp_batch_destroy(pp2d_mdp_batch* h) {
  if (!h) return;
  if (h->grid) cudaStreamSynchronize(h->grid->stream);
  cudaFree(h->goals); cudaFree(h->frozen_dev); cudaFree(h->list);
  cudaFree(h->resid); cudaFree(h->res_cost); cudaFree(h->res_action);
  pp2d_mdp_destroy(h->grid);
  delete h;
}

int pp2d_mdp_batch_set_stream(pp2d_mdp_batch* h, void* stream) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  return pp2d_mdp_set_stream(h->grid, stream);
}

int pp2d_mdp_batch_sweeps(pp2d_mdp_batch* h, uint32_t n) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  if (h->n_frozen)
    return fail(PP2D_ERR_STATE, "the batch was solved (its instances stopped at their own "
                                "sweep counts): call pp2d_mdp_batch_reset first");
  return pp2d_mdp_sweeps(h->grid, n);
}

int pp2d_mdp_batch_residual(pp2d_mdp_batch* h, float* out) {
  if (!h || !out) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (h->n_frozen)
    return fail(PP2D_ERR_STATE, "the batch was solved: call pp2d_mdp_batch_reset first");
  std::vector<uint32_t> all(h->count);
  for (uint32_t k = 0; k < h->count; ++k) all[k] = k;
  PP2D_TRY_MDP(batch_residual(h, all));
  memcpy(out, h->resid_host.data(), h->count * sizeof(float));
  return PP2D_OK;
}

int pp2d_mdp_batch_solve(pp2d_mdp_batch* h, uint32_t* sweeps_out, double* residuals,
                         uint32_t max_residuals) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  if (h->n_frozen == h->count)
    return fail(PP2D_ERR_STATE, "the batch was solved: call pp2d_mdp_batch_reset or "
                                "pp2d_mdp_batch_update first");
  // pp2d_mdp_solve per instance (path_planning_2d.cu:219-263), all active
  // instances in the same launches; an instance leaves after its first batch
  // of 100 sweeps whose residual meets the rule.
  pp2d_mdp* g = h->grid;
  std::vector<uint32_t> active, still, stopped;
  for (uint32_t k = 0; k < h->count; ++k)
    if (!h->frozen[k]) active.push_back(k);
  uint32_t batch = 0, total = 0;
  while (!active.empty()) {
    PP2D_TRY_MDP(pp2d_mdp_sweeps(g, 100));
    total += 100;
    PP2D_TRY_MDP(batch_residual(h, active));
    still.clear();
    stopped.clear();
    for (uint32_t k : active) {
      float r;
      memcpy(&r, &h->resid_host[k], sizeof(float));
      const double cost_inf_norm = r;
      if (residuals && batch < max_residuals)
        residuals[(size_t)k * max_residuals + batch] = cost_inf_norm;
      if (keeps_sweeping(cost_inf_norm, g->gamma)) {
        still.push_back(k);
      } else {
        stopped.push_back(k);
        h->stop_sweeps[k] = batch_sweeps_of(h, k);
        h->frozen[k] = 1;
        ++h->n_frozen;
        if (sweeps_out) sweeps_out[k] = total;
      }
    }
    if (!stopped.empty()) PP2D_TRY_MDP(batch_snapshot<true>(h, stopped));
    active.swap(still);
    ++batch;
  }
  PP2D_CUDA(cudaStreamSynchronize(g->stream));
  return PP2D_OK;
}

int pp2d_mdp_batch_update(pp2d_mdp_batch* h, const uint32_t* instances, uint32_t n,
                          const uint8_t* maps, size_t map_stride, const uint32_t* goals_xy) {
  if (!h || !instances || !maps || !goals_xy) return fail(PP2D_ERR_INVALID, "NULL argument");
  const size_t hw = (size_t)h->H * h->W;
  if (map_stride != 0 && map_stride < hw)
    return fail(PP2D_ERR_INVALID, "map_stride %zu is below height*width = %zu", map_stride, hw);
  std::vector<uint8_t> listed(h->count, 0);
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t k = instances[i];
    if (k >= h->count)
      return fail(PP2D_ERR_INVALID, "entry %u names instance %u of a batch of %u", i, k, h->count);
    if (listed[k]) return fail(PP2D_ERR_INVALID, "instance %u is listed twice", k);
    listed[k] = 1;
  }
  for (uint32_t i = 0; i < n; ++i)
    PP2D_TRY_MDP(check_goal(maps + i * map_stride, h->W, h->H, goals_xy[2 * (size_t)i],
                            goals_xy[2 * (size_t)i + 1], instances[i]));
  if (n == 0) return PP2D_OK;
  pp2d_mdp* g = h->grid;
  // Per listed instance: its trapped(n_k) and whether a solve froze it.
  const std::vector<uint32_t> list(instances, instances + n);
  uint32_t* words = stage_list(h, list, 2);
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t k = list[i];
    words[n + i] = word_of(trapped_cost(g, batch_sweeps_of(h, k)));
    words[2 * n + i] = h->frozen[k];
  }
  PP2D_TRY_MDP(upload_list(h));
  // The device maps are read only while codes are built: the new maps go to
  // the front of g->occ in list order, and no instance reads its map again
  // before the next reset or update.
  PP2D_TRY_MDP(upload_maps(g, maps, map_stride, hw, n));
  for (uint32_t i = 0; i < n; ++i) {
    h->goals_host[2 * (size_t)list[i]] = goals_xy[2 * (size_t)i];
    h->goals_host[2 * (size_t)list[i] + 1] = goals_xy[2 * (size_t)i + 1];
  }
  PP2D_CUDA(cudaMemcpyAsync(h->goals, h->goals_host.data(), 2 * sizeof(uint32_t) * h->count,
                            cudaMemcpyHostToDevice, g->stream));
  BatchUpdateParams p;
  memset(&p, 0, sizeof(p));
  p.c.goals = h->goals; p.c.code = g->code;
  p.c.W = (int)h->W; p.c.H = (int)h->H; p.c.count = (int)h->count; p.c.pitch = g->pitch;
  p.c.rows_phys = (int)g->H + 2 * kPadRows;
  p.maps = g->occ;
  p.map_stride = map_stride ? hw : 0;
  p.list = h->list;
  p.trapped = reinterpret_cast<const float*>(h->list + n);
  p.thaw = h->list + 2 * (size_t)n;
  p.n_list = (int)n;
  p.groups = ((int)h->H + kCodeRows - 1) / kCodeRows;
  p.j = g->j[g->cur];
  p.jchk = g->jchk;
  p.action = g->action;
  p.res_cost = h->res_cost;
  p.res_action = h->res_action;
  p.mask = next_unit_mask(g);
  const size_t groups = (size_t)n * p.groups;
  dim3 grid((g->pitch / 4 + kCodeThreads - 1) / kCodeThreads,
            (unsigned)std::min<size_t>(groups, 65535));
  mdp_batch_update_kernel<<<grid, kCodeThreads, 0, g->stream>>>(p);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  PP2D_CUDA(cudaGetLastError());
  // (the caller may free the maps on return)
  PP2D_CUDA(cudaStreamSynchronize(g->stream));
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t k = list[i];
    const uint32_t nk = batch_sweeps_of(h, k);
    if (h->frozen[k]) {
      h->frozen[k] = 0;
      --h->n_frozen;
    }
    h->sweep_off[k] = nk - g->n_sweeps;
    h->chk_off[k] = nk - g->n_chk;        // the next residual measures the change from J'
    h->has_occ[k] = memchr(maps + i * map_stride, 1, hw) != nullptr;
  }
  return PP2D_OK;
}

int pp2d_mdp_batch_download(pp2d_mdp_batch* h, uint32_t first, uint32_t n, float* cost,
                            uint8_t* action) {
  if (!h) return fail(PP2D_ERR_INVALID, "handle is NULL");
  if (first >= h->count || n > h->count - first)
    return fail(PP2D_ERR_INVALID, "instances [%u, %llu) outside the batch of %u", first,
                (unsigned long long)first + n, h->count);
  if (n == 0 || (!cost && !action)) return PP2D_OK;
  pp2d_mdp* g = h->grid;
  // instances still in the live grid are exported into their result slots;
  // the slots of frozen instances hold their snapshots
  std::vector<uint32_t> live;
  for (uint32_t k = first; k < first + n; ++k)
    if (!h->frozen[k]) live.push_back(k);
  if (!live.empty()) PP2D_TRY_MDP(batch_snapshot<false>(h, live));
  const size_t hw = (size_t)h->H * h->W;
  if (cost)
    PP2D_CUDA(cudaMemcpyAsync(cost, h->res_cost + first * hw, n * hw * sizeof(float),
                              cudaMemcpyDeviceToHost, g->stream));
  if (action)
    PP2D_CUDA(cudaMemcpyAsync(action, h->res_action + first * hw, n * hw,
                              cudaMemcpyDeviceToHost, g->stream));
  PP2D_CUDA(cudaStreamSynchronize(g->stream));
  return PP2D_OK;
}

int pp2d_mdp_batch_plan(pp2d_mdp_batch* h, const uint32_t* instance, const float* beliefs,
                        uint32_t n, uint8_t* actions) {
  if (!h || !instance || !beliefs || !actions) return fail(PP2D_ERR_INVALID, "NULL argument");
  for (uint32_t i = 0; i < n; ++i)
    if (instance[i] >= h->count)
      return fail(PP2D_ERR_INVALID, "belief %u names instance %u of a batch of %u", i,
                  instance[i], h->count);
  if (n == 0) return PP2D_OK;
  pp2d_mdp* g = h->grid;
  const size_t hw = (size_t)h->H * h->W;
  std::vector<const uint8_t*> bases(n);
  for (uint32_t i = 0; i < n; ++i) bases[i] = batch_actions_of(h, instance[i]);
  float* d_b = nullptr;
  const uint8_t** d_base = nullptr;
  uint8_t* d_a = nullptr;
  int rc = [&]() -> int {
    PP2D_CUDA(cudaMalloc(&d_b, hw * n * sizeof(float)));
    PP2D_CUDA(cudaMalloc(&d_base, n * sizeof(uint8_t*)));
    PP2D_CUDA(cudaMalloc(&d_a, n));
    PP2D_CUDA(cudaMemcpyAsync(d_b, beliefs, hw * n * sizeof(float), cudaMemcpyHostToDevice,
                              g->stream));
    PP2D_CUDA(cudaMemcpyAsync(d_base, bases.data(), n * sizeof(uint8_t*),
                              cudaMemcpyHostToDevice, g->stream));
    mdp_batch_plan_kernel<<<n, 256, 0, g->stream>>>(d_b, hw, d_base, d_a);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    PP2D_CUDA(cudaGetLastError());
    PP2D_CUDA(cudaMemcpyAsync(actions, d_a, n, cudaMemcpyDeviceToHost, g->stream));
    PP2D_CUDA(cudaStreamSynchronize(g->stream));
    return PP2D_OK;
  }();
  cudaFree(d_b);
  cudaFree(d_base);
  cudaFree(d_a);
  return rc;
}

int pp2d_mdp_batch_waypoints(pp2d_mdp_batch* h, uint32_t k, uint32_t sx, uint32_t sy,
                             uint32_t* cells, uint32_t max_len, uint32_t* n_out) {
  if (!h || !cells || !n_out) return fail(PP2D_ERR_INVALID, "NULL argument");
  if (k >= h->count)
    return fail(PP2D_ERR_INVALID, "instance %u outside the batch of %u", k, h->count);
  if (sx >= h->W || sy >= h->H)
    return fail(PP2D_ERR_INVALID, "start (%u %u) outside the map", sx, sy);
  const size_t hw = (size_t)h->H * h->W;
  std::vector<uint8_t> a(hw);
  PP2D_CUDA(cudaMemcpyAsync(a.data(), batch_actions_of(h, k), hw, cudaMemcpyDeviceToHost, h->grid->stream));
  PP2D_CUDA(cudaStreamSynchronize(h->grid->stream));
  *n_out = rollout(a.data(), h->W, h->H, sx, sy, cells, max_len);
  return PP2D_OK;
}

int pp2d_mdp_batch_sweep_counts(const pp2d_mdp_batch* h, uint32_t* out) {
  if (!h || !out) return fail(PP2D_ERR_INVALID, "NULL argument");
  for (uint32_t k = 0; k < h->count; ++k)
    out[k] = batch_sweeps_of(h, k);
  return PP2D_OK;
}

int pp2d_mdp_batch_work_counters(pp2d_mdp_batch* h, uint64_t out[2]) {
  if (!h || !out) return fail(PP2D_ERR_INVALID, "NULL argument");
  return pp2d_mdp_work_counters(h->grid, out);
}

}  // extern "C"
