// mdp_kernels.cuh -- sm_100a kernels of the MDP value-iteration hot path.
//
// Reference behaviour being reproduced (paths relative to
// /root/reference/path_planning_2d/):
//   src/mdp/path_planning_2d_cuda.cu:76-213  model tables (P, g) per cell
//   src/mdp/path_planning_2d_cuda.cu:215-264 one Jacobi Bellman backup
//
// Design (see DESIGN.md for the derivation):
//   * The reference's 360 B/cell tables are never materialised.  Everything a
//     backup needs is a function of the 3x3 occupancy, stored as one 16-bit
//     code per cell ("ring code": the 8 neighbours in ring order
//     s0 s1 s2 s5 s8 s7 s6 s3 s0 s1, so that the three neighbour slots every
//     action can move into are 3 consecutive bits).
//   * J of occupied cells, of the goal and of out-of-map padding is stored as
//     0.  A blocked neighbour then contributes fma(coef, 0, cost) = cost,
//     exactly what the reference's zero probability does, with no select.
//     Occupied cells follow the closed form J_n = fma(gamma, J_{n-1}, 2) and
//     are filled in on download.
//   * Per action the only occupancy-dependent numbers are the stage cost g_u
//     and the centre coefficient gamma*P_u[4]; both come from an 8 KB
//     shared-memory table indexed by 4 ring bits (two actions per 16-byte
//     row, replicated 8x so that a quarter-warp LDS.128 never bank-conflicts).
//   * Each lane owns CW consecutive columns and marches down its rows; the
//     3-row window of J lives in registers, horizontal neighbours come from
//     warp shuffles, so there is no shared-memory tile and every global load
//     is a coalesced row segment.
//   * T = 2 fuses two sweeps: J^1 of row y is produced in registers, shuffled
//     to the neighbours and consumed for J^2 of row y-1 while the LUT rows of
//     row y-1 are still in registers (register-level temporal blocking).  A
//     warp recomputes HL lanes of halo on each side.
//   * min over the 9 actions uses FMNMX3; the arg-min (POLICY) variant is
//     only run for the last sweep of a pp2d_mdp_sweeps call.
//
// Bit-exactness: each action cost is the reference's chain
//   cost = g_u; for k ascending: cost = fma(gamma*P_u[k], J[n_k], cost)
// with gamma*0.7f, gamma*0.1f and gamma*P_u[4] rounded once (FMUL) before the
// FFMA, as in the SASS of the reference kernel (SURVEY.md section 7).  Terms
// whose probability is 0 are skipped: fma(0, J, c) == c for finite J.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "async_copy.cuh"
#include "belief.cuh"
#include "fp_exact.cuh"

namespace pp2d {

constexpr int kPadRows = 2;   // ghost rows above and below the owned rows
constexpr int kSlackRows = 8; // extra rows at the bottom: prefetch may overrun
constexpr int kPrefetch = 2;  // CW == 1 path: rows held in registers ahead of use
constexpr int kRing = 3;      // CW >= 2 path: cp.async ring slots per lane (divides the 6-step unroll)
constexpr int kPadLeft = 8;   // zero columns left of x = 0
// Table: 4 tables (one per action pair) x 16 rows (4 ring bits) x 8 lane
// replicas of one float4 = 8 KB; a cell needs 4 row addresses.
constexpr int kLutFloat4 = 4 * 16 * 8;
constexpr int kLutAlign = 2048;
// Fused kernel: 8 warps per CTA, 2 resident CTAs per SM (the other occupancies
// that were timed are in DESIGN.md section 4).
constexpr int kWarpsPerCta = 8;

// Code bits.
constexpr uint32_t kCodeRingMask = 0x3FFu;   // bits 0..9
constexpr uint32_t kCodeOccBit = 1u << 13;   // occupied or padding
constexpr uint32_t kCodeLiveBit = 1u << 14;  // free, in map, not the goal

struct SweepParams {
  const float* jin;      // padded plane, element (y, x) at [(y+2)*pitch + x+8]
  float* jout;
  const uint16_t* code;  // same geometry as J
  uint8_t* action;       // dense [H][W] (POLICY only)
  const float4* lut;     // kLutFloat4 / 8 rows (the kernel writes the 8 lane replicas)
  int W, H, pitch;
  int n_strips, rows_per_unit, n_units;
  int y_begin, y_end;    // rows to produce (may extend 1 row into the ghosts)
  int prefetch_rows;     // rows ahead touched with prefetch.global.L1 (>= kPrefetch)
  float gamma, ga, gb;   // gamma*1.0f, gamma*0.7f, gamma*0.1f
  // --- peer-to-peer ghost rows (P2P kernels only, see P2pParams) ---
  float* peer_up_out;    // up neighbour's jout plane at ITS ghost row H_up, col 0
  float* peer_down_out;  // down neighbour's jout plane at ITS ghost row -2, col 0
  unsigned int* flags;   // this shard's flag block (kFlag*)
  unsigned int* up_flag_remote;    // &up.flags[kFlagFromDown]
  unsigned int* down_flag_remote;  // &down.flags[kFlagFromUp]
  unsigned int iter;               // 1-based count of fused P2P launches
  unsigned int expect_top, expect_bot;  // cumulative boundary-unit counts
  unsigned int p2p_debug;               // bit0 no waits, bit1 no peer stores, bit2 no signals
  int edge_rows;                        // rows of a boundary unit processed first
  int lin_len;           // LIN kernels: units are runs of lin_len rows of the strip-major sequence
  unsigned int spin_limit;  // P2P: polls of a neighbour flag before giving up (kFlagError)
  // P2P LIN kernels: unit u covers rows [unit_lo[u], unit_lo[u+1]) of the
  // strip-major sequence.  The host balances COST, not rows: a unit that
  // touches the first / last two rows of a strip also does the hand-shake
  // (system fences wait for NVLink write acknowledgements) and gets fewer rows,
  // so that it does not finish after everybody else.  NULL: runs of lin_len.
  const int* unit_lo;
  // P2P row-block units: the same idea with two numbers: the first and last
  // row block of a strip get rows_edge < rows_per_unit rows, the blocks between
  // them rows_inner; rows_edge == 0: all blocks have rows_per_unit rows.
  int rows_edge, rows_inner;
  // P2P: index of the warp that publishes this launch's flags to the
  // neighbours (see publish_flags), -1: the last boundary unit to finish its
  // edge rows does it itself.
  int publisher_unit;
  // --- skipping of unchanged units (fused row-block kernels, DESIGN.md 4) ---
  // need_out == NULL: every unit runs on its own warp, no bookkeeping.
  // Otherwise bit u of need_in says unit u must run; a unit whose output
  // differs from its input sets the bits of its 3x3 unit neighbourhood in
  // need_out (the mask of the next launch), and need_clear (the mask of the
  // launch after that) is cleared.
  const uint32_t* need_in;
  uint32_t* need_out;
  uint32_t* need_clear;
  unsigned long long* work;  // [0] += units run, [1] += units of the launch (may be NULL)
  int all_live;              // need_in is not read: every unit runs
  int edge_live;             // the row blocks next to the ghost rows of a shard always run
};

// Shortest row segment a live unit is split into when few units are live:
// every segment pays 2 priming steps of the T = 2 march.
constexpr int kMinSegRows = 8;

// Flag block of a shard (uint32 each, cudaMalloc'ed, IPC-shared).
constexpr int kFlagFromUp = 0;     // written by the up neighbour: its launch #
constexpr int kFlagFromDown = 1;   // written by the down neighbour
constexpr int kFlagCountTop = 2;   // local: finished top-boundary units
constexpr int kFlagCountBot = 3;   // local: finished bottom-boundary units
constexpr int kFlagError = 4;      // local: a wait timed out
constexpr int kFlagWords = 8;

__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned int ld_relaxed_gpu(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

__device__ __forceinline__ float min3(float a, float b, float c) {
  float d;
  asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// One Bellman backup of one cell.  j0..j8: J of the 3x3 neighbourhood in the
// reference's slot order (row-major, slot 4 = the cell), blocked slots = 0.
// t[0]={g1,c1,g2,c2} t[1]={g5,c5,g8,c8} t[2]={g7,c7,g6,c6} t[3]={g3,c3,g0,c0}
// (g = stage cost, c = gamma*P[4] of that action), g4 = stage cost of "stay".
template <bool POLICY>
__device__ __forceinline__ float backup(float j0, float j1, float j2, float j3,
                                        float j4, float j5, float j6, float j7,
                                        float j8, const float4 (&t)[4],
                                        float g4, float gam, float ga,
                                        float gb, uint32_t& act) {
  // Slot order of the non-zero probabilities of each action
  // (path_planning_2d_cuda.cu:89-125), centre coefficient from the table.
  float c0 = fmaf(t[3].w, j4, fmaf(gb, j3, fmaf(gb, j1, fmaf(ga, j0, t[3].z))));
  float c1 = fmaf(t[0].y, j4, fmaf(gb, j2, fmaf(ga, j1, fmaf(gb, j0, t[0].x))));
  float c2 = fmaf(gb, j5, fmaf(t[0].w, j4, fmaf(ga, j2, fmaf(gb, j1, t[0].z))));
  float c3 = fmaf(gb, j6, fmaf(t[3].y, j4, fmaf(ga, j3, fmaf(gb, j0, t[3].x))));
  float c4 = fmaf(gam, j4, g4);
  float c5 = fmaf(gb, j8, fmaf(ga, j5, fmaf(t[1].y, j4, fmaf(gb, j2, t[1].x))));
  float c6 = fmaf(gb, j7, fmaf(ga, j6, fmaf(t[2].w, j4, fmaf(gb, j3, t[2].z))));
  float c7 = fmaf(gb, j8, fmaf(ga, j7, fmaf(gb, j6, fmaf(t[2].y, j4, t[2].x))));
  float c8 = fmaf(ga, j8, fmaf(gb, j7, fmaf(gb, j5, fmaf(t[1].w, j4, t[1].z))));
  if (POLICY) {
    // path_planning_2d_cuda.cu:244-258: first strict minimum, u ascending.
    // (A compare-and-keep chain: the equality form -- FMNMX3 minimum, then the
    // lowest index whose cost equals it -- took 236 against 245 instructions
    // per marching step of the fused arg-min kernel, but the P2P strip-major
    // instantiation spilled two registers with it.)
    float best = c0;
    uint32_t a = 0;
    if (c1 < best) { best = c1; a = 1; }
    if (c2 < best) { best = c2; a = 2; }
    if (c3 < best) { best = c3; a = 3; }
    if (c4 < best) { best = c4; a = 4; }
    if (c5 < best) { best = c5; a = 5; }
    if (c6 < best) { best = c6; a = 6; }
    if (c7 < best) { best = c7; a = 7; }
    if (c8 < best) { best = c8; a = 8; }
    act = a;
    return best;
  } else {
    return min3(min3(c0, c1, c2), min3(c3, c4, c5), min3(c6, c7, c8));
  }
}

// Row loads are volatile asm on purpose: a plain __ldg() is sunk by the
// compiler to just before its first use, which collapses the kPrefetch-deep
// software pipeline (seen in the ncu source view: long-scoreboard stalls on
// the first use of every prefetched register).
// NC: the non-coherent (read-only) path.  It is only legal for data nobody
// writes while the kernel runs, so the P2P instantiations -- whose ghost rows
// of jin are written by the neighbour GPU during the launch, ordered by the
// flag hand-shake -- use ordinary weak loads, which the acquire of the flag
// wait does order.
template <int CW, bool NC = true>
__device__ __forceinline__ void load_own(const float* __restrict__ p,
                                         float (&o)[CW]) {
  if constexpr (!NC) {
    if constexpr (CW == 1) {
      asm volatile("ld.global.f32 %0, [%1];" : "=f"(o[0]) : "l"(p) : "memory");
    } else if constexpr (CW == 2) {
      asm volatile("ld.global.v2.f32 {%0, %1}, [%2];"
                   : "=f"(o[0]), "=f"(o[1]) : "l"(p) : "memory");
    } else {
      asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];"
                   : "=f"(o[0]), "=f"(o[1]), "=f"(o[2]), "=f"(o[3]) : "l"(p) : "memory");
    }
  } else if constexpr (CW == 1) {
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(o[0]) : "l"(p));
  } else if constexpr (CW == 2) {
    asm volatile("ld.global.nc.v2.f32 {%0, %1}, [%2];"
                 : "=f"(o[0]), "=f"(o[1]) : "l"(p));
  } else {
    asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(o[0]), "=f"(o[1]), "=f"(o[2]), "=f"(o[3]) : "l"(p));
  }
}

template <int CW>
__device__ __forceinline__ void store_own(float* p, const float (&o)[CW]) {
  if constexpr (CW == 1) {
    *p = o[0];
  } else if constexpr (CW == 2) {
    *reinterpret_cast<float2*>(p) = make_float2(o[0], o[1]);
  } else {
    *reinterpret_cast<float4*>(p) = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// Codes of the lane's CW cells, packed two per 32-bit word.
template <int CW>
__device__ __forceinline__ void load_codes(const uint16_t* __restrict__ p,
                                           uint32_t (&c)[(CW + 1) / 2]) {
  if constexpr (CW == 1) {
    uint16_t v;
    asm volatile("ld.global.nc.u16 %0, [%1];" : "=h"(v) : "l"(p));
    c[0] = v;
  } else if constexpr (CW == 2) {
    asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(c[0]) : "l"(p));
  } else {
    asm volatile("ld.global.nc.v2.u32 {%0, %1}, [%2];"
                 : "=r"(c[0]), "=r"(c[1]) : "l"(p));
  }
}

// own[CW] -> row[CW+2] with the left/right neighbours taken from the
// adjacent lanes (lane 0 / lane 31 get their own value: those lanes are halo).
template <int CW>
__device__ __forceinline__ void fill_row(const float (&own)[CW],
                                         float (&row)[CW + 2]) {
  row[0] = __shfl_up_sync(0xffffffffu, own[CW - 1], 1);
  row[CW + 1] = __shfl_down_sync(0xffffffffu, own[0], 1);
#pragma unroll
  for (int j = 0; j < CW; ++j) row[1 + j] = own[j];
}

// Fetch the 4 table rows of one cell.  `word` holds two 16-bit codes; HI
// selects the upper one.  lane_base = shared address of the table (8 KB
// aligned) | (lane & 7) * 16, so the row offset can be OR-ed in: one shift
// and one LOP3 per row.
template <int IMM>
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+%5];"
      : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
      : "r"(addr), "n"(IMM));
  return v;
}

template <bool HI, int P>
__device__ __forceinline__ float4 lut_row(uint32_t lane_base, uint32_t word) {
  const uint32_t sh = HI ? (word >> (9 + 2 * P)) : (word << (7 - 2 * P));
  return lds128<P * 2048>((sh & 0x780u) | lane_base);
}

template <bool HI>
__device__ __forceinline__ void lut_fetch(uint32_t lane_base, uint32_t word,
                                          float4 (&t)[4], float& g4) {
  t[0] = lut_row<HI, 0>(lane_base, word);
  t[1] = lut_row<HI, 1>(lane_base, word);
  t[2] = lut_row<HI, 2>(lane_base, word);
  t[3] = lut_row<HI, 3>(lane_base, word);
  // live bit (14 of the code) -> 2.0f (0x40000000); goal, occupied cells and
  // padding -> 0.0f, which makes "stay" cost exactly 0 there (their J is 0).
  g4 = __uint_as_float((HI ? word : (word << 16)) & 0x40000000u);
}

// ---- cp.async staging (CW >= 2) --------------------------------------------
// Every lane copies its own CW floats of J and CW codes of a row into its
// private slot of a per-warp shared-memory ring, kRing rows ahead, and reads
// them back itself: cp.async.wait_group is per thread, so no warp or block
// synchronisation is needed.  Unlike register loads (which ptxas sinks to
// their first use, sharing a scoreboard with younger loads) the copies are
// issued where they are written and waited for with a counting barrier
// (LDGDEPBAR / DEPBAR.LE in SASS).
template <int CW, int OFF>
__device__ __forceinline__ void lds_row(uint32_t saddr, float (&o)[CW]) {
  if constexpr (CW == 2) {
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2+%3];"
                 : "=f"(o[0]), "=f"(o[1]) : "r"(saddr), "n"(OFF) : "memory");
  } else {
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+%5];"
                 : "=f"(o[0]), "=f"(o[1]), "=f"(o[2]), "=f"(o[3])
                 : "r"(saddr), "n"(OFF) : "memory");
  }
}
template <int CW, int OFF>
__device__ __forceinline__ void lds_codes(uint32_t saddr,
                                          uint32_t (&c)[(CW + 1) / 2]) {
  if constexpr (CW == 2) {
    asm volatile("ld.shared.u32 %0, [%1+%2];"
                 : "=r"(c[0]) : "r"(saddr), "n"(OFF) : "memory");
  } else {
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2+%3];"
                 : "=r"(c[0]), "=r"(c[1]) : "r"(saddr), "n"(OFF) : "memory");
  }
}

template <int T, int CW>
struct StripGeom {
  static constexpr int HL = (T + CW - 1) / CW;          // halo lanes per side
  static constexpr int S = (32 - 2 * HL) * CW;          // valid columns/strip
  static constexpr int XOFF = -HL * CW;                 // x of lane 0, cell 0
  // cp.async ring: per warp and slot, 32 lanes x (CW floats + CW codes).
  static constexpr int kSlotBytes = 32 * CW * 6;
  static constexpr int kCodeOff = 32 * CW * 4;
  static constexpr int kRingBytesPerWarp = (CW >= 2) ? kRing * kSlotBytes : 0;
};

// LIN: units are runs of the strip-major row sequence (see run()); a separate
// instantiation because the loop around the marching code costs registers the
// row-block scheme cannot spare (126 of 128).
template <int T, int CW, bool POLICY, bool P2P = false, bool LIN = false>
struct Sweeper {
  using G = StripGeom<T, CW>;
  // the instantiations that can skip units: they OR the bit difference between
  // J^2 and J^0 of every produced cell into `diff`
  static constexpr bool kSkip = T == 2 && CW == 2 && !P2P && !LIN;
  uint32_t diff = 0;
  float A[3][CW + 2];        // J^0 rows y-1, y, y+1 (rotating)
  float B[3][CW + 2];        // J^1 rows y-2, y-1, y (T == 2)
  float4 L[2][CW][4];        // LUT rows of row y (cur) and y-1 (prev)
  float G4[2][CW];
  float nxt[kPrefetch][CW];              // prefetched raw J^0 rows
  uint32_t cnx[kPrefetch][(CW + 1) / 2]; // prefetched code rows
  uint32_t cprev[(CW + 1) / 2];          // codes of row y-1 (T == 2 && POLICY)

  const SweepParams& p;
  uint32_t lane_base;        // shared address of this lane's table replica
  const float* pin;          // next J^0 row to prefetch (row y+1+kPrefetch)
  const uint16_t* pcode;     // next code row to prefetch (row y+kPrefetch)
  float* pout;               // row written at step y (y for T=1, y-1 for T=2)
  uint8_t* pact;             // action row y (POLICY)
  float *pup, *pdn;          // P2P: this lane's column in the neighbours' ghost rows
  bool peer_top, peer_bot;   // P2P: this segment feeds the upper / lower neighbour (warp-uniform)
  int yout;                  // P2P: row index of pout
  size_t l1_ahead;           // CW == 1: rows ahead for prefetch.global.L1
  uint32_t ring_j, ring_c;   // CW >= 2: shared addresses of this lane's ring slots
  int x0;                    // map x of the lane's first cell
  bool valid;

  __device__ __forceinline__ Sweeper(const SweepParams& p_, uint32_t lb,
                                     uint32_t ring_warp)
      : p(p_), lane_base(lb), ring_j(ring_warp), ring_c(ring_warp) {}

  // One marching step on row y.  I: rotation index (compile time).  J2: also
  // produce the second sweep of row y-1 (steady state of T == 2).
  template <int I, bool J2, bool PEER = false>
  __device__ __forceinline__ void step() {
    constexpr int a0 = I % 3, a1 = (I + 1) % 3, a2 = (I + 2) % 3;
    constexpr int lc = I % 2, lp = (I + 1) % 2;
    uint32_t cc[(CW + 1) / 2];
    if constexpr (CW >= 2) {
      constexpr int slot = I % kRing;
      // The oldest of the kRing groups in flight (row y+1, codes of row y)
      // has landed in this lane's slot.
      cp_async_wait<kRing - 1>();
      float own[CW];
      lds_row<CW, slot * G::kSlotBytes>(ring_j, own);
      lds_codes<CW, slot * G::kSlotBytes + G::kCodeOff>(ring_c, cc);
      fill_row<CW>(own, A[a2]);
      // Refill the slot with row y+1+kRing / codes of row y+kRing (the planes
      // have kSlackRows spare rows, so the last steps may run past the end).
      // (Issued here, right after the slot was read.  Refilling at the END of
      // the step was tried: it saved the three predicated-off LDS ptxas puts in
      // front of the LDGSTS pair -- 193 instead of 195 instructions per step --
      // but ran slower, 64.8 vs 63.4 us per launch: the copy had one step less
      // to land.)
      cp_async<CW * 4>(ring_j + slot * G::kSlotBytes, pin);
      cp_async<CW * 2>(ring_c + slot * G::kSlotBytes + G::kCodeOff, pcode);
      cp_async_commit();
    } else {
      constexpr int q = I % kPrefetch;
      fill_row<CW>(nxt[q], A[a2]);
      cc[0] = cnx[q][0];
      load_own<CW, !P2P>(pin, nxt[q]);
      load_codes<CW>(pcode, cnx[q]);
      asm volatile("prefetch.global.L1 [%0];" :: "l"(pin + l1_ahead));
      asm volatile("prefetch.global.L1 [%0];" :: "l"(pcode + l1_ahead));
    }
    pin += p.pitch;
    pcode += p.pitch;
    // Table rows of row y.
#pragma unroll
    for (int j = 0; j < CW; ++j) {
      if (j & 1) lut_fetch<true>(lane_base, cc[j >> 1], L[lc][j], G4[lc][j]);
      else lut_fetch<false>(lane_base, cc[j >> 1], L[lc][j], G4[lc][j]);
    }
    float v1[CW];
    uint32_t act[CW];
#pragma unroll
    for (int j = 0; j < CW; ++j) {
      v1[j] = backup<(POLICY && T == 1)>(A[a0][j], A[a0][j + 1], A[a0][j + 2],
                             A[a1][j], A[a1][j + 1], A[a1][j + 2],
                             A[a2][j], A[a2][j + 1], A[a2][j + 2],
                             L[lc][j], G4[lc][j], p.gamma, p.ga, p.gb, act[j]);
    }
    if constexpr (T == 1) {
      if (valid) {
        store_own<CW>(pout, v1);
        if constexpr (POLICY) {
#pragma unroll
          for (int j = 0; j < CW; ++j) {
            if (x0 + j < p.W) {
              const uint32_t cj = (j & 1) ? (cc[j >> 1] >> 16) : cc[j >> 1];
              // Occupied cells tie on every action in the reference -> 0.
              pact[j] = (cj & kCodeOccBit) ? 0 : (uint8_t)act[j];
            }
          }
        }
      }
      pout += p.pitch;
      if constexpr (POLICY) pact += p.W;
    } else {
      fill_row<CW>(v1, B[a2]);
      if constexpr (J2) {
        float v2[CW];
        uint32_t act2[CW];
#pragma unroll
        for (int j = 0; j < CW; ++j) {
          // the arg-min of a fused launch belongs to its SECOND sweep
          v2[j] = backup<POLICY>(B[a0][j], B[a0][j + 1], B[a0][j + 2],
                                 B[a1][j], B[a1][j + 1], B[a1][j + 2],
                                 B[a2][j], B[a2][j + 1], B[a2][j + 2],
                                 L[lp][j], G4[lp][j], p.gamma, p.ga, p.gb,
                                 act2[j]);
        }
        if (valid) store_own<CW>(pout, v2);
        if constexpr (kSkip) {
          // J^0 of row y-1 is still in the window: one LOP3 per cell
#pragma unroll
          for (int j = 0; j < CW; ++j)
            asm("lop3.b32 %0, %1, %2, %0, 0xBE;"      // (a ^ b) | diff
                : "+r"(diff) : "r"(__float_as_uint(v2[j])), "r"(__float_as_uint(A[a0][j + 1])));
        }
        if constexpr (POLICY) {
          // (single predicated stores: no divergent region inside the marching loop)
#pragma unroll
          for (int j = 0; j < CW; ++j) {
            const uint32_t occ_bit = (j & 1) ? (kCodeOccBit << 16) : kCodeOccBit;
            // Occupied cells tie on every action in the reference -> 0.
            const uint32_t a = (cprev[j >> 1] & occ_bit) ? 0u : act2[j];
            if (valid && x0 + j < p.W) pact[j] = (uint8_t)a;
          }
        }
        if constexpr (PEER) {
          // The first / last two owned rows are also the neighbours' ghost
          // rows: written straight into their HBM over NVLink.  peer_top /
          // peer_bot and yout are warp-uniform, `valid` only predicates the
          // store (no divergent region in front of the next shuffle).
          if (peer_top && yout < kPadRows) {
            if (valid) store_own<CW>(pup + (size_t)yout * p.pitch, v2);
          }
          if (peer_bot && yout >= p.H - kPadRows) {
            if (valid) store_own<CW>(pdn + (size_t)(yout - (p.H - kPadRows)) * p.pitch, v2);
          }
        }
        if constexpr (POLICY) pact += p.W;
        if constexpr (PEER) ++yout;
        pout += p.pitch;
      }
      if constexpr (POLICY) {
#pragma unroll
        for (int j = 0; j < (CW + 1) / 2; ++j) cprev[j] = cc[j];
      }
    }
  }

  // March over rows [y0, y1) of this lane's columns.  PEER: rows 0,1 / H-2,H-1
  // are also stored into the neighbours' ghost rows.
  template <bool PEER>
  __device__ __forceinline__ void march(int y0, int y1, size_t col) {
    const size_t pitch = (size_t)p.pitch;
    // First row stepped on: y0-1 for T=2 (J^1 of the row above), y0 for T=1.
    const int ys = (T == 2) ? y0 - 1 : y0;
    int steps = y1 - ys + (T == 2 ? 1 : 0);               // rows ys .. ye
    if constexpr (PEER) yout = y0;
    const float* jin = p.jin + col + (size_t)(ys - 1 + kPadRows) * pitch;
    {
      float r[CW];
      load_own<CW, !P2P>(jin, r);
      fill_row<CW>(r, A[0]);
      load_own<CW, !P2P>(jin + pitch, r);
      fill_row<CW>(r, A[1]);
    }
    pin = jin + 2 * pitch;                                  // row ys+1
    pcode = p.code + col + (size_t)(ys + kPadRows) * pitch; // row ys
    if constexpr (CW >= 2) {
#pragma unroll
      for (int d = 0; d < kRing; ++d) {
        cp_async<CW * 4>(ring_j + d * G::kSlotBytes, pin);
        cp_async<CW * 2>(ring_c + d * G::kSlotBytes + G::kCodeOff, pcode);
        cp_async_commit();
        pin += pitch;
        pcode += pitch;
      }
    } else {
#pragma unroll
      for (int d = 0; d < kPrefetch; ++d) {
        load_own<CW, !P2P>(pin, nxt[d]);
        load_codes<CW>(pcode, cnx[d]);
        pin += pitch;
        pcode += pitch;
      }
    }
    pout = p.jout + col + (size_t)(y0 + kPadRows) * pitch;
    if constexpr (POLICY) pact = p.action + (size_t)y0 * p.W + x0;
    if constexpr (T == 2) {
      // Two priming steps (rows y0-1 and y0) produce J^1 only.
      step<0, false, PEER>();
      step<1, false, PEER>();
      steps -= 2;
      while (true) {
        step<2, true, PEER>(); if (--steps == 0) break;
        step<3, true, PEER>(); if (--steps == 0) break;
        step<4, true, PEER>(); if (--steps == 0) break;
        step<5, true, PEER>(); if (--steps == 0) break;
        step<0, true, PEER>(); if (--steps == 0) break;
        step<1, true, PEER>(); if (--steps == 0) break;
      }
    } else {
      while (true) {
        step<0, false>(); if (--steps == 0) break;
        step<1, false>(); if (--steps == 0) break;
        step<2, false>(); if (--steps == 0) break;
        step<3, false>(); if (--steps == 0) break;
        step<4, false>(); if (--steps == 0) break;
        step<5, false>(); if (--steps == 0) break;
      }
    }
    // Do not leave the slot ring with copies in flight.
    if constexpr (CW >= 2) cp_async_wait<0>();
  }

  // A unit is a run of `lin_len` rows of the strip-major sequence (strip 0 rows
  // y_begin..y_end-1, strip 1 rows ..., ...): every warp of the one-wave launch
  // gets the same number of rows whatever W and H are (with whole row blocks
  // per strip, 274 strips x 8 blocks fill only 92.6 % of the 2368 warp slots at
  // W = 16384).  A unit that crosses a strip boundary marches twice.
  __device__ __forceinline__ void run(int unit, int lane) {
    if constexpr (LIN) {
      l1_ahead = (size_t)(p.prefetch_rows - kPrefetch) * (size_t)p.pitch;
      if constexpr (CW >= 2) {
        ring_j += lane * (CW * 4);
        ring_c += lane * (CW * 2);
      }
      const int R = p.y_end - p.y_begin;
      int lo, hi;
      if (P2P && p.unit_lo != nullptr) {
        // (through lane 0: the compiler must keep seeing warp-uniform bounds)
        lo = __shfl_sync(0xffffffffu, __ldg(p.unit_lo + unit), 0);
        hi = __shfl_sync(0xffffffffu, __ldg(p.unit_lo + unit + 1), 0);
      } else {
        lo = unit * p.lin_len;
        hi = min(lo + p.lin_len, p.n_strips * R);
      }
      while (lo < hi) {
        const int k = lo / R;
        const int a = lo - k * R;
        const int b = min(R, a + (hi - lo));
        run_segment(k, p.y_begin + a, p.y_begin + b, lane);
        lo += b - a;
      }
    } else {
      const int k = unit % p.n_strips;
      const int rb = unit / p.n_strips;
      int y0, y1;                                             // rows [y0, y1)
      if (P2P && p.rows_edge > 0) {
        y0 = rb == 0 ? p.y_begin : p.y_begin + p.rows_edge + (rb - 1) * p.rows_inner;
        y1 = min(p.y_begin + p.rows_edge + rb * p.rows_inner, p.y_end);
      } else {
        y0 = p.y_begin + rb * p.rows_per_unit;
        y1 = min(y0 + p.rows_per_unit, p.y_end);
      }
      run_segment(k, y0, y1, lane);
    }
  }

  // Rows [y0, y1) of strip k.
  __device__ __forceinline__ void run_segment(const int k, const int y0, const int y1,
                                              const int lane) {
    x0 = k * G::S + G::XOFF + lane * CW;
    valid = (lane >= G::HL) && (lane < 32 - G::HL) && (x0 < p.W);
    const size_t col = (size_t)(x0 + kPadLeft);
    if constexpr (!LIN) {
      l1_ahead = (size_t)(p.prefetch_rows - kPrefetch) * (size_t)p.pitch;
      if constexpr (CW >= 2) {
        ring_j += lane * (CW * 4);
        ring_c += lane * (CW * 2);
      }
    }
    int r0 = y0, r1 = y1;            // rows marched without peer stores
    if constexpr (P2P) {
      // Units that touch the first / last two owned rows read ghost rows and
      // write the neighbours' ghost rows.  They process the `edge_rows` rows
      // next to the boundary FIRST and publish their flag right after, so the
      // hand-shake is off the critical path of the launch.
      const bool top = p.peer_up_out != nullptr && y0 < kPadRows;
      const bool bot = p.peer_down_out != nullptr && y1 > p.H - kPadRows;
      if (top || bot) {
        pup = p.peer_up_out + col;       // only dereferenced under peer_top / peer_bot
        pdn = p.peer_down_out + col;
        peer_top = top && !(p.p2p_debug & 2u);
        peer_bot = bot && !(p.p2p_debug & 2u);
        int e0 = y0, e1 = y1;
        const int e = p.edge_rows;
        if (top != bot && y1 - y0 > e) {
          if (top) { e1 = y0 + e; r0 = e1; }
          else     { e0 = y1 - e; r1 = e0; }
        } else {
          r1 = r0;                     // the whole unit is the edge segment
        }
        if (!(p.p2p_debug & 1u)) {
          // Wait until the neighbour's previous launch has (a) written my
          // ghost rows of this buffer parity and (b) finished reading its own
          // ghost rows that I am about to overwrite; both are implied by its
          // flag, published after ALL its edge segments facing me are done.
          // Every lane polls (one broadcast transaction per poll) and the
          // value is taken from lane 0 through a shuffle: the loop exit is
          // then warp-uniform FOR THE COMPILER, which keeps the marching code
          // below free of divergence guards (a lane-0-only spin loop cost the
          // whole kernel its uniformity: 63 -> 82 us per launch).
          const unsigned int want = p.iter - 1;
#pragma unroll
          for (int side = 0; side < 2; ++side) {
            if (!(side == 0 ? top : bot)) continue;
            const unsigned int* f = p.flags + (side == 0 ? kFlagFromUp : kFlagFromDown);
            // A neighbour that never shows up (crashed rank, mismatched launch
            // counts) must not hang the GPU: after spin_limit polls the error
            // word is set.  The rows this launch produces from stale ghost rows
            // are wrong from here on; mdp_residual_kernel turns the error word
            // into an infinite residual and every host entry point that returns
            // results checks it, so the failure cannot pass silently.
            unsigned int spins = 0;
            while (true) {
              const unsigned int v = __shfl_sync(0xffffffffu, ld_acquire_sys(f), 0);
              if ((int)(v - want) >= 0) break;
              if (++spins > p.spin_limit) {
                if (lane == 0) atomicExch(p.flags + kFlagError, 1u);
                break;
              }
              __nanosleep(spins < 64u ? 32u : 256u);
            }
          }
        }
        march<true>(e0, e1, col);
        // Publish: the last edge segment on each side to finish writes this
        // launch's number into the neighbour's flag.  (All lanes fence; lane 0
        // counts; the count comes back through a shuffle so that the decision
        // is warp-uniform.)
        if (!(p.p2p_debug & 4u)) {
          // Release of this unit's peer stores into the local count.  A system
          // fence waits for the flush of EVERY egress port of the GPU, PCIe
          // included: while a download is on its way to the host it takes tens
          // of microseconds, and a marching warp that executes it becomes the
          // tail of the launch (measured: +17 us per launch at 2 GPUs).  So the
          // marching warps only order their stores at GPU scope (barrier, then
          // fence, then lane 0's atomic: the release pattern of the PTX memory
          // model, cumulative over the whole warp's stores); the one system
          // fence per side and launch is executed by whoever publishes the
          // flag -- a warp without rows (publish_flags) when there is one.
          const bool gpu_scope = p.publisher_unit >= 0 || (p.p2p_debug & 8u);
          if (gpu_scope) {
            __syncwarp();
            __threadfence();
          } else {
            __threadfence_system();        // every lane: its peer stores before the count
            __syncwarp();                  // ... and all of them before lane 0 counts
          }
#pragma unroll
          for (int side = 0; side < 2; ++side) {
            if (!(side == 0 ? top : bot)) continue;
            unsigned int c = 0;
            if (lane == 0)
              c = atomicAdd(p.flags + (side == 0 ? kFlagCountTop : kFlagCountBot), 1u) + 1u;
            c = __shfl_sync(0xffffffffu, c, 0);
            if (p.publisher_unit < 0 && c == (side == 0 ? p.expect_top : p.expect_bot)) {
              __threadfence_system();      // (acquires the other units' counts, too)
              if (lane == 0)
                st_release_sys(side == 0 ? p.up_flag_remote : p.down_flag_remote, p.iter);
            }
          }
        }
      }
    }
    if (r1 > r0) march<false>(r0, r1, col);
  }
};

// The publisher warp of a P2P launch (SweepParams::publisher_unit): waits until
// every boundary unit of a side has counted itself in (their peer stores happen
// before their count, the fence after the last poll acquires it), executes the system fence
// and writes this launch's number into the neighbour's flag.  The counts are
// cumulative over launches.  Lane 0 serves the upper, lane 1 the lower side.
__device__ __forceinline__ void publish_flags(const SweepParams& p, int lane) {
  if (p.p2p_debug & 4u) return;
  if (lane < 2) {
    unsigned int* remote = lane == 0 ? p.up_flag_remote : p.down_flag_remote;
    const bool feeds = (lane == 0 ? p.peer_up_out : p.peer_down_out) != nullptr;
    if (feeds && remote != nullptr) {
      const unsigned int* cnt = p.flags + (lane == 0 ? kFlagCountTop : kFlagCountBot);
      const unsigned int expect = lane == 0 ? p.expect_top : p.expect_bot;
      unsigned int spins = 0;
      bool ok = true;
      // (relaxed polls: an acquire load invalidates the L1 of the SM on every
      // poll, which the marching warps of this SM pay for -- 68.0 against 65.8
      // us per launch; the fence below is the acquire)
      while ((int)(ld_relaxed_gpu(cnt) - expect) < 0) {
        if (++spins > p.spin_limit) {       // a unit never finished: do not publish
          atomicExch(p.flags + kFlagError, 1u);
          ok = false;
          break;
        }
        __nanosleep(200u);
      }
      if (ok) {
        __threadfence_system();             // acquire of the counts + release of the flag
        st_release_sys(remote, p.iter);
      }
    }
  }
}

// Bits of word i of a unit mask that stand for the units [lo, hi).
__device__ __forceinline__ uint32_t unit_range_bits(int i, int lo, int hi) {
  const int a = min(max(lo - 32 * i, 0), 32), b = min(max(hi - 32 * i, 0), 32);
  const uint32_t m = b - a >= 32 ? 0xffffffffu : (1u << max(b - a, 0)) - 1u;
  return m << (a & 31);
}

// Word i of the units this launch must run.
__device__ __forceinline__ uint32_t need_word(const SweepParams& p, int i, int n_words) {
  if (i >= n_words) return 0u;
  uint32_t m = p.need_in[i];
  if (p.edge_live) {
    // every row block with a row whose 2-row cone reaches a ghost row: rows
    // 0, 1 (block 0, blocks have >= 2 rows) and rows H-2, H-1 (the last block,
    // and the one before it when the last block has 1 row)
    const int rb_bot = max(0, (p.y_end - p.y_begin - 2) / p.rows_per_unit);
    m |= unit_range_bits(i, 0, p.n_strips) |
         unit_range_bits(i, rb_bot * p.n_strips, p.n_units);
  }
  return m;
}

// Work of warp w of a fused row-block launch: unit `unit`, rows [y0, y1).
// Without bookkeeping (need_out == NULL) warp w runs unit w, as it always
// did.  Otherwise the n_live units that must run share the launch's warps:
// s = max(1, warps / n_live) warps per live unit, warp w takes live unit w / s
// and row segment w % s of it (segments of at least kMinSegRows rows).  Every
// lane computes the same values (lane-0 shuffles and ballots): the march that
// follows stays warp-uniform.  Returns false when the warp has nothing to do.
__device__ __forceinline__ bool unit_plan(const SweepParams& p, int w, int lane, int& unit,
                                          int& y0, int& y1) {
  const bool book = p.need_out != nullptr;
  const int n_words = (p.n_units + 31) >> 5;
  const int per = (n_words + 31) >> 5;          // mask words per lane
  int n_live = p.n_units, cnt = 0, incl = 0;
  if (book && !p.all_live) {
#pragma unroll 1
    for (int i = 0; i < per; ++i) cnt += __popc(need_word(p, lane * per + i, n_words));
    incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      incl += lane >= o ? t : 0;
    }
    n_live = __shfl_sync(0xffffffffu, incl, 31);
  }
  if (p.work != nullptr && w == 0 && lane == 0) {
    atomicAdd(p.work, (unsigned long long)n_live);
    atomicAdd(p.work + 1, (unsigned long long)p.n_units);
  }
  const int s = book ? max(1, (int)(gridDim.x * kWarpsPerCta) / max(n_live, 1)) : 1;
  const int li = w / s;
  if (li >= n_live) return false;
  if (book && !p.all_live) {
    // the lane whose words hold live unit number li finds its index
    int r = li - (incl - cnt), u = -1;
#pragma unroll 1
    for (int i = 0; i < per; ++i) {
      const uint32_t m = need_word(p, lane * per + i, n_words);
      const int c = __popc(m);
      if (u < 0 && r >= 0 && r < c) u = (lane * per + i) * 32 + (int)__fns(m, 0u, r + 1);
      r -= c;
    }
    const uint32_t owner = __ballot_sync(0xffffffffu, u >= 0);
    unit = __shfl_sync(0xffffffffu, u, __ffs(owner) - 1);
  } else {
    unit = li;
  }
  const int rb = unit / p.n_strips;
  const int uy0 = p.y_begin + rb * p.rows_per_unit;
  const int rows = min(uy0 + p.rows_per_unit, p.y_end) - uy0;
  const int nseg = min(s, max(1, rows / kMinSegRows));
  const int seg = w - li * s;
  if (seg >= nseg) return false;
  y0 = uy0 + seg * rows / nseg;
  y1 = uy0 + (seg + 1) * rows / nseg;
  return true;
}

// One warp per (column strip, row block) unit; kWarpsPerCta warps per CTA.
template <int T, int CW, bool POLICY, bool P2P = false, bool LIN = false>
__global__ void __launch_bounds__(kWarpsPerCta * 32, (T == 2 && CW == 2) ? 2 : 1)
mdp_sweep_kernel(const SweepParams p) {
  // The table must start on a 2 KB boundary of the shared window so that the
  // row offset (bits 7..10) and the lane replica (bits 4..6) can be OR-ed
  // into the base.  The window itself starts at 1 KB (system reserved), so
  // the alignment is done at run time on an over-allocated buffer.
  using G = StripGeom<T, CW>;
  constexpr int kWarps = kWarpsPerCta;
  // Programmatic dependent launch: the next launch of the stream may start its
  // prologue (the table copy below, which reads nothing a sweep writes) while
  // this one is still running; it blocks in griddepcontrol.wait until this grid
  // has completed and its writes are visible.  Both are no-ops for a launch
  // without the attribute.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  __shared__ __align__(16) unsigned char
      lut_raw[kLutFloat4 * 16 + kLutAlign + kWarps * G::kRingBytesPerWarp];
  const uint32_t raw_addr = (uint32_t)__cvta_generic_to_shared(lut_raw);
  const uint32_t lut_addr = (raw_addr + (uint32_t)(kLutAlign - 1)) & ~(uint32_t)(kLutAlign - 1);
  float4* lut_s = reinterpret_cast<float4*>(lut_raw + (lut_addr - raw_addr));
  // p.lut holds ONE copy of every row (kLutFloat4 / 8 rows); the 8 lane
  // replicas are written here: one global load and 8 shared stores per row.
  for (int i = threadIdx.x; i < kLutFloat4 / 8; i += blockDim.x) {
    const float4 row = p.lut[i];
#pragma unroll
    for (int c = 0; c < 8; ++c) lut_s[i * 8 + c] = row;
  }
  __syncthreads();
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int lane = threadIdx.x & 31;
  // The warp index is read through a shuffle from lane 0, which tells the
  // compiler it is warp-uniform (unit, row counts and loop exits then are, too:
  // no divergence guard in front of the shuffles of the marching loop).
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int unit = blockIdx.x * (blockDim.x >> 5) + warp;
  using Sw = Sweeper<T, CW, POLICY, P2P, LIN>;
  if constexpr (P2P) {
    if (unit == p.publisher_unit) {
      publish_flags(p, lane);
      return;
    }
  }
  int run_unit = unit, y0 = 0, y1 = 0;
  if constexpr (Sw::kSkip) {
    // The mask the launch after next reads: the previous launch read it and
    // has completed (griddepcontrol.wait above).  (Reductions, not stores.)
    if (p.need_out != nullptr && blockIdx.x == 0)
      for (int i = threadIdx.x; i < (p.n_units + 31) >> 5; i += blockDim.x)
        atomicAnd(p.need_clear + i, 0u);
    if (!unit_plan(p, unit, lane, run_unit, y0, y1)) return;
  } else {
    if (unit >= p.n_units) return;
  }
  // Produced by a volatile asm after the barrier: the table loads (plain asm,
  // free to be scheduled) depend on it and so cannot move above the barrier.
  uint32_t lane_base;
  asm volatile("or.b32 %0, %1, %2;"
               : "=r"(lane_base) : "r"(lut_addr), "r"((lane & 7) << 4) : "memory");
  const uint32_t ring_warp =
      lut_addr + kLutFloat4 * 16 + warp * G::kRingBytesPerWarp;
  Sw s(p, lane_base, ring_warp);
  if constexpr (Sw::kSkip) {
    const int k = run_unit % p.n_strips;
    s.run_segment(k, y0, y1, lane);
    // Output of the segment differs from its input somewhere: the 3x3 unit
    // neighbourhood must run in the next launch (lanes 0..8, one unit each).
    const bool changed = __any_sync(0xffffffffu, s.valid && s.diff != 0u);
    if (p.need_out != nullptr && changed && lane < 9) {
      const int rb = run_unit / p.n_strips + lane / 3 - 1, kk = k + lane % 3 - 1;
      if (rb >= 0 && rb < p.n_units / p.n_strips && kk >= 0 && kk < p.n_strips) {
        const int v = rb * p.n_strips + kk;
        atomicOr(p.need_out + (v >> 5), 1u << (v & 31));
      }
    }
  } else {
    s.run(unit, lane);
  }
}

// ---------------------------------------------------------------------------
// Code plane from the occupancy grid (replaces cudaGenerateModelData's crop of
// the 3x3 neighbourhood, path_planning_2d_cuda.cu:185-196: out of map =
// occupied).  occ holds global rows [occ_row0, occ_row0 + occ_rows).
struct CodeParams {
  const uint8_t* occ;
  uint16_t* code;
  int W, Htot, pitch;
  int rows_phys;       // owned rows + 2*kPadRows
  int row_begin;       // global row of local y = 0
  int occ_row0, occ_rows;
  int gx, gy;
};

// Occupancy of the 6 columns x0-1 .. x0+4 of global row gy as a bit mask (bit i
// = column x0-1+i; out of map = occupied, a cell is occupied iff its byte is
// exactly 1).  FAST: x0 is 4-aligned, inside the map with 3 columns to spare
// and W % 4 == 0, so the 4 own bytes are one aligned 32-bit load.
template <bool FAST>
__device__ __forceinline__ uint32_t occ_mask6(const CodeParams& p, int x0, int gy) {
  const int r = gy - p.occ_row0;
  if (gy < 0 || gy >= p.Htot || r < 0 || r >= p.occ_rows) return 0x3Fu;
  const uint8_t* __restrict__ q = p.occ + (size_t)r * p.W;
  uint32_t m = 0;
  if (FAST) {
    const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(q + x0));
    m |= ((w & 0xFFu) == 1u) << 1;
    m |= (((w >> 8) & 0xFFu) == 1u) << 2;
    m |= (((w >> 16) & 0xFFu) == 1u) << 3;
    m |= ((w >> 24) == 1u) << 4;
    m |= (x0 > 0 ? (uint32_t)(__ldg(q + x0 - 1) == 1) : 1u);
    m |= (x0 + 4 < p.W ? (uint32_t)(__ldg(q + x0 + 4) == 1) : 1u) << 5;
  } else {
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const int gx = x0 - 1 + i;
      m |= ((gx < 0 || gx >= p.W) ? 1u : (uint32_t)(__ldg(q + gx) == 1)) << i;
    }
  }
  return m;
}

// One thread builds the codes of 4 consecutive cells and marches kCodeRows rows
// down with the three 6-column occupancy masks of rows y-1, y, y+1 in
// registers: 3 loads (1 word + 2 bytes) and one 8-byte store per 4 cells
// instead of 9 byte loads and a 2-byte store per cell.
constexpr int kCodeRows = 16;
constexpr int kCodeThreads = 128;

// Codes of the 4 cells x0 .. x0+3 of global row gy from the occupancy masks
// m0, m1, m2 of rows gy-1, gy, gy+1 (occ_mask6).  Used by the code kernel and
// the map-update kernel, so that both build the same bits.
__device__ __forceinline__ void cell_codes4(const CodeParams& p, int x0, int gy, uint32_t m0,
                                            uint32_t m1, uint32_t m2, uint32_t (&code)[4]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int x = x0 + j;
    uint32_t cd = kCodeOccBit;   // padding
    if (x >= 0 && x < p.W && gy >= 0 && gy < p.Htot) {
      // slots: 0 1 2 / 3 4 5 / 6 7 8 ; ring: s0 s1 s2 s5 s8 s7 s6 s3 s0 s1
      const uint32_t t = m0 >> j, c = m1 >> j, b = m2 >> j;
      const uint32_t s0 = t & 1u, s1 = (t >> 1) & 1u, s2 = (t >> 2) & 1u, s3 = c & 1u,
                     s4 = (c >> 1) & 1u, s5 = (c >> 2) & 1u, s6 = b & 1u,
                     s7 = (b >> 1) & 1u, s8 = (b >> 2) & 1u;
      cd = s0 | (s1 << 1) | (s2 << 2) | (s5 << 3) | (s8 << 4) | (s7 << 5) |
           (s6 << 6) | (s3 << 7) | (s0 << 8) | (s1 << 9);
      if (s4) cd |= kCodeOccBit;
      else if (!(x == p.gx && gy == p.gy)) cd |= kCodeLiveBit;
    }
    code[j] = cd;
  }
}

// The CodeParams grid row gy is built from, and its row ly in them: the row
// itself on a single grid (batch_row below on the tall grid of a batch).
__device__ __forceinline__ const CodeParams& row_of(const CodeParams& p, int gy, int& ly) {
  ly = gy;
  return p;
}
__device__ __forceinline__ int first_row(const CodeParams& p) { return p.row_begin; }

// P: CodeParams or BatchCodeParams (code, pitch, rows_phys, row_of, first_row)
template <bool FAST, class P>
__device__ __forceinline__ void code_march(const P& p, int c0, int r0) {
  const int x0 = c0 - kPadLeft;
  const int r1 = min(r0 + kCodeRows, p.rows_phys);
  int gy = first_row(p) + r0 - kPadRows;
  int ly;
  uint32_t m0 = occ_mask6<FAST>(row_of(p, gy - 1, ly), x0, ly);
  uint32_t m1 = occ_mask6<FAST>(row_of(p, gy, ly), x0, ly);
  for (int r = r0; r < r1; ++r, ++gy) {
    const uint32_t m2 = occ_mask6<FAST>(row_of(p, gy + 1, ly), x0, ly);
    uint32_t code[4];
    cell_codes4(row_of(p, gy, ly), x0, ly, m0, m1, m2, code);
    // pitch is a multiple of 32 and c0 of 4: the 4 codes are 8-byte aligned
    *reinterpret_cast<uint2*>(p.code + (size_t)r * p.pitch + c0) =
        make_uint2(code[0] | (code[1] << 16), code[2] | (code[3] << 16));
    m0 = m1;
    m1 = m2;
  }
}

// grid: (ceil(pitch / 4 / kCodeThreads), ceil(rows_phys / kCodeRows))
__global__ void __launch_bounds__(kCodeThreads) mdp_code_kernel(const CodeParams p) {
  const int c0 = 4 * (blockIdx.x * kCodeThreads + threadIdx.x);
  const int r0 = blockIdx.y * kCodeRows;
  if (c0 >= p.pitch || r0 >= p.rows_phys) return;
  const int x0 = c0 - kPadLeft;
  const bool fast = (p.W & 3) == 0 && (x0 & 3) == 0 && x0 >= 0 && x0 + 3 < p.W &&
                    (reinterpret_cast<uintptr_t>(p.occ) & 3u) == 0;
  if (fast) code_march<true>(p, c0, r0);
  else code_march<false>(p, c0, r0);
}

// ---------------------------------------------------------------------------
// New map on a solved handle (pp2d_mdp_update_map, DESIGN.md section 4): the
// codes of the new map and goal, and J' in place of J_n:
//   newly occupied cell -> stored 0 (occupied cells are stored as 0);
//   newly freed cell    -> trapped(n), the value it was reported with;
//   the new goal        -> 0;
// every other cell keeps its value.  Jchk <- J' on the owned rows (the next
// residual measures the change since the update).  A cell whose code or
// stored J changed is dirty; every dirty unit of the fused row-block launch
// geometry sets the bits of its 3x3 unit neighbourhood in `need`, the mask the
// next fused launch reads.

// The unit mask of the next fused row-block launch; unit = row_block *
// n_strips + strip.  need == NULL: no valid mask (that launch runs every unit).
struct UnitMask {
  uint32_t* need;
  int n_strips, rows_per_unit, n_rb;
};

struct UpdateParams {
  CodeParams c;          // occupancy of the new map, code plane, new goal
  float* j;              // current J plane (ghost rows included)
  float* jchk;           // residual snapshot
  float trapped;         // J_n of an occupied cell, n = sweep count
  UnitMask mask;         // seeded with the dirty units
  int H;                 // owned rows
};

__device__ __forceinline__ void mark_unit_neighbourhood(const UnitMask& m, int rb, int k) {
#pragma unroll 1
  for (int i = 0; i < 9; ++i) {
    const int r = rb + i / 3 - 1, kk = k + i % 3 - 1;
    if (r >= 0 && r < m.n_rb && kk >= 0 && kk < m.n_strips) {
      const int v = r * m.n_strips + kk;
      atomicOr(m.need + (v >> 5), 1u << (v & 31));
    }
  }
}

// Strip width of the fused row-block launches: a 4-cell group from column x0
// lies in strip k_lo = max(x0, 0) / kUnitStrip or in the next one.
constexpr int kUnitStrip = StripGeom<2, 2>::S;

// Warp-wide: the units of row block rb that hold a dirty cell of this row
// (dirty_lo: strip k_lo, dirty_hi: strip k_lo + 1) mark their 3x3 unit
// neighbourhoods in m.need, one lane per unit.  All 32 lanes call it.
__device__ __forceinline__ void seed_dirty_units(const UnitMask& m, int rb, int k_lo,
                                                 bool dirty_lo, bool dirty_hi, int lane) {
#pragma unroll
  for (int side = 0; side < 2; ++side) {
    const bool d = side ? dirty_hi : dirty_lo;
    const uint32_t b = __ballot_sync(0xffffffffu, d);
    if (d) {
      const int k = k_lo + side;
      const uint32_t peers = __match_any_sync(b, k);
      if (__ffs(peers) - 1 == lane) mark_unit_neighbourhood(m, rb, k);
    }
  }
}

// The update rule on the 4 cells of plane index q (columns x0 .. x0+3), given
// their new codes: reads the old codes and J, writes the codes and J that
// changed, and J' into jchk unless it is NULL.  A newly freed cell takes
// `trapped`, or its entry of the result-slot row `slot` (indexed by column)
// when slot is not NULL.  Returns whether a cell of strip k_lo (or left of the
// map) and of strip k_lo + 1 is dirty.
__device__ __forceinline__ void replan_cells4(uint16_t* code_plane, float* j, float* jchk,
                                              size_t q, int x0, int k_lo,
                                              const uint32_t (&code)[4], float trapped,
                                              const float* slot, bool& dirty_lo, bool& dirty_hi) {
  const uint2 oc2 = *reinterpret_cast<const uint2*>(code_plane + q);
  const uint32_t old[4] = {oc2.x & 0xFFFFu, oc2.x >> 16, oc2.y & 0xFFFFu, oc2.y >> 16};
  const float4 jv = *reinterpret_cast<const float4*>(j + q);
  const float jo[4] = {jv.x, jv.y, jv.z, jv.w};
  float jn[4];
  bool code_changed = false, j_changed = false;
  dirty_lo = dirty_hi = false;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool occ_new = code[i] & kCodeOccBit, occ_old = old[i] & kCodeOccBit;
    jn[i] = jo[i];
    if (occ_new && !occ_old) jn[i] = 0.0f;
    if (!occ_new && occ_old) jn[i] = slot ? __ldg(slot + x0 + i) : trapped;
    if (!(code[i] & (kCodeOccBit | kCodeLiveBit))) jn[i] = 0.0f;   // the goal
    const bool cc = code[i] != old[i];
    const bool jc = __float_as_uint(jn[i]) != __float_as_uint(jo[i]);
    code_changed |= cc;
    j_changed |= jc;
    if (cc || jc) {
      if ((x0 + i) / kUnitStrip == k_lo || x0 + i < 0) dirty_lo = true;
      else dirty_hi = true;
    }
  }
  if (code_changed)
    *reinterpret_cast<uint2*>(code_plane + q) =
        make_uint2(code[0] | (code[1] << 16), code[2] | (code[3] << 16));
  const float4 jw = make_float4(jn[0], jn[1], jn[2], jn[3]);
  if (j_changed) *reinterpret_cast<float4*>(j + q) = jw;
  if (jchk != nullptr) *reinterpret_cast<float4*>(jchk + q) = jw;
}

// Same thread shape as mdp_code_kernel (4 cells per thread, kCodeRows rows
// marched with the occupancy masks in registers), but every lane of a warp
// runs the whole march: the dirty units are aggregated per warp.
__global__ void __launch_bounds__(kCodeThreads) mdp_update_map_kernel(const UpdateParams p) {
  const CodeParams& cp = p.c;
  const int lane = threadIdx.x & 31;
  const int c0 = 4 * (blockIdx.x * kCodeThreads + threadIdx.x);
  const int r0 = blockIdx.y * kCodeRows;
  if (r0 >= cp.rows_phys) return;                 // uniform over the block
  const bool active = c0 < cp.pitch;
  const int x0 = c0 - kPadLeft;
  const bool fast = (cp.W & 3) == 0 && (x0 & 3) == 0 && x0 >= 0 && x0 + 3 < cp.W &&
                    (reinterpret_cast<uintptr_t>(cp.occ) & 3u) == 0;
  auto mask = [&](int gy) {
    return fast ? occ_mask6<true>(cp, x0, gy) : occ_mask6<false>(cp, x0, gy);
  };
  const int k_lo = max(x0, 0) / kUnitStrip;
  const int r1 = min(r0 + kCodeRows, cp.rows_phys);
  int gy = cp.row_begin + r0 - kPadRows;
  uint32_t m0 = mask(gy - 1), m1 = mask(gy);
  for (int r = r0; r < r1; ++r, ++gy) {
    const uint32_t m2 = mask(gy + 1);
    uint32_t code[4];
    cell_codes4(cp, x0, gy, m0, m1, m2, code);
    m0 = m1;
    m1 = m2;
    bool dirty_lo = false, dirty_hi = false;
    if (active) {
      const bool owned = r >= kPadRows && r < kPadRows + p.H;
      replan_cells4(cp.code, p.j, owned ? p.jchk : nullptr, (size_t)r * cp.pitch + c0, x0, k_lo,
                    code, p.trapped, nullptr, dirty_lo, dirty_hi);
    }
    if (p.mask.need != nullptr && __any_sync(0xffffffffu, dirty_lo || dirty_hi)) {
      // ghost rows belong to the row block next to them
      const int y = min(max(r - kPadRows, 0), p.H - 1);
      seed_dirty_units(p.mask, min(y / p.mask.rows_per_unit, p.mask.n_rb - 1), k_lo, dirty_lo,
                       dirty_hi, lane);
    }
  }
}

// ---------------------------------------------------------------------------
// Maximum of m over a CTA of 256 threads into *result, as float bits:
// atomicMax on uint is order preserving for non-negative floats.
__device__ __forceinline__ void block_max_to(float m, uint32_t* result) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  __shared__ float wm[8];
  if ((threadIdx.x & 31) == 0) wm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; ++i) m = fmaxf(m, wm[i]);
    atomicMax(result, __float_as_uint(m));
  }
}

// max |J - Jchk| over the owned rows, then Jchk = J
// (path_planning_2d.cu:243-251), into *result (block_max_to).
// CHK_ZERO: first check after a reset -- Jchk is J_0 = 0 by definition and is
// not read (the reset then does not have to zero it).
template <bool CHK_ZERO>
__global__ void __launch_bounds__(256)
mdp_residual_kernel(const float4* __restrict__ j, float4* __restrict__ chk,
                    size_t n4, uint32_t floor_bits, uint32_t* result,
                    const unsigned int* p2p_error) {
  float m = __uint_as_float(floor_bits);
  // a ghost-row hand-shake timed out: J is not to be trusted, and the
  // stopping rule must never be satisfied by it
  if (p2p_error != nullptr && *p2p_error != 0u) m = __uint_as_float(0x7f800000u);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
       i += (size_t)gridDim.x * blockDim.x) {
    const float4 a = j[i];
    const float4 b = CHK_ZERO ? make_float4(0.f, 0.f, 0.f, 0.f) : chk[i];
    m = fmaxf(m, fmaxf(fmaxf(fabsf(a.x - b.x), fabsf(a.y - b.y)),
                       fmaxf(fabsf(a.z - b.z), fabsf(a.w - b.w))));
    chk[i] = a;
  }
  block_max_to(m, result);
}

// ---------------------------------------------------------------------------
// Policy iteration (path_planning_2d_cuda.cu:266-355, called from the
// reference's policyIteration(), path_planning_2d.cu:271-357 -- dead code
// there, SURVEY.md section 8f row 4).  Not a hot path: one thread per cell,
// the model of the cell rebuilt from its code word.
//   evaluation:  J'(s) = g(s,u) + sum_k P(s,u,k) * (gamma * J(n_k)),  u = pi(s)
//   improvement: pi(s) = first arg-min over u of the same expression
// Arithmetic of the reference kernels (nvcc 12.9, sm_100a): t_k = FMUL(J_k,
// gamma) once per neighbour, cost = FFMA(P_k, t_k, cost) for k = 0..8 --
// (gamma*J)*P, NOT the (gamma*P)*J of the value-iteration kernel, all with
// flush-to-zero (J of the goal decays into the denormal range).  Zero
// probabilities contribute fma(0, t, c) = c and are skipped.  Occupied cells
// (stored as 0, see the header of this file) follow J_n = (gamma*J_{n-1}) + 2
// and keep action 0; unlike in value iteration the goal is an ordinary cell
// here (its J is only 0 once the policy says "stay").
struct PolicyParams {
  const float* jin;
  float* jout;             // evaluation only
  const uint16_t* code;
  uint8_t* action;
  int W, H, pitch;
  float gamma;
};

// P(s,u,.) and g(s,u) of one action from the ring code of the cell
// (path_planning_2d_cuda.cu:76-172).  blocked: bit i = slot i occupied or out
// of map (bit 4 unused: the cell itself is free here).
__device__ __forceinline__ void policy_model(uint32_t blocked, bool is_goal, int u,
                                             float (&P)[9], float& g) {
  // slots with non-zero naive probability, ascending; side[u] as in the
  // reference's switch
  const int s0[9] = {0, 0, 1, 0, 4, 2, 3, 4, 4};
  const int s1[9] = {1, 1, 2, 3, 4, 4, 4, 6, 5};
  const int s2[9] = {3, 2, 4, 4, 4, 5, 6, 7, 7};
  const int s3[9] = {4, 4, 5, 6, 4, 8, 7, 8, 8};
#pragma unroll
  for (int i = 0; i < 9; ++i) P[i] = 0.0f;
  if (u == 4) {
    P[4] = 1.0f;
    g = is_goal ? 0.0f : 2.0f;                       // cuda.cu:171
    return;
  }
  const int sl[4] = {s0[u], s1[u], s2[u], s3[u]};
  float naive[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) naive[j] = (sl[j] == u) ? 0.7f : 0.1f;
  // stage cost over the NAIVE probabilities, ascending slot (cuda.cu:166-169)
  g = 0.0f;
#pragma unroll
  for (int j = 0; j < 4; ++j)
    g = fmaf(((blocked >> sl[j]) & 1u) && sl[j] != 4 ? 2.0f : 1.0f, naive[j], g);
  // blocked mass moves to "stay", ascending slot (cuda.cu:142-147)
  float stay = 0.1f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (sl[j] == 4) continue;
    if ((blocked >> sl[j]) & 1u) stay += naive[j];
    else P[sl[j]] = naive[j];
  }
  P[4] = stay;
}

// ring bit r of the code -> neighbour slot: s0 s1 s2 s5 s8 s7 s6 s3
__device__ __forceinline__ uint32_t blocked_slots(uint32_t code) {
  return ((code >> 0) & 1u) << 0 | ((code >> 1) & 1u) << 1 | ((code >> 2) & 1u) << 2 |
         ((code >> 3) & 1u) << 5 | ((code >> 4) & 1u) << 8 | ((code >> 5) & 1u) << 7 |
         ((code >> 6) & 1u) << 6 | ((code >> 7) & 1u) << 3;
}

template <bool IMPROVE>
__global__ void __launch_bounds__(256)
mdp_policy_kernel(const PolicyParams p) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  if (x >= p.W || y >= p.H) return;
  const size_t q = (size_t)(y + kPadRows) * p.pitch + x + kPadLeft;
  const uint32_t code = p.code[q];
  const size_t dense = (size_t)y * p.W + x;
  if (code & kCodeOccBit) {                // trapped: closed form on download
    if (IMPROVE) p.action[dense] = 0;
    else p.jout[q] = 0.0f;
    return;
  }
  const bool is_goal = !(code & kCodeLiveBit);
  const uint32_t blocked = blocked_slots(code);
  float t[9];
#pragma unroll
  for (int i = 0; i < 9; ++i)
    t[i] = mul_ftz(p.jin[q + (size_t)((i / 3 - 1) * p.pitch) + (i % 3 - 1)], p.gamma);
  if (IMPROVE) {
    float opt = 3.402823466e+38f;
    int oa = 0;
    for (int u = 0; u < 9; ++u) {
      float P[9], g;
      policy_model(blocked, is_goal, u, P, g);
      float cost = g;
#pragma unroll
      for (int i = 0; i < 9; ++i)
        if (P[i] != 0.0f) cost = fma_ftz(P[i], t[i], cost);
      if (cost < opt) { opt = cost; oa = u; }
    }
    p.action[dense] = (uint8_t)oa;
  } else {
    float P[9], g;
    policy_model(blocked, is_goal, p.action[dense], P, g);
    float cost = g;
#pragma unroll
    for (int i = 0; i < 9; ++i)
      if (P[i] != 0.0f) cost = fma_ftz(P[i], t[i], cost);
    p.jout[q] = cost;
  }
}

// Dense J for download: occupied cells get the closed-form trapped cost.
// VEC: 4 cells per thread (W % 4 == 0 and 4-aligned pad columns: 16-byte loads
// and stores); otherwise one cell per thread.
template <bool VEC>
__global__ void mdp_export_kernel(const float* __restrict__ j,
                                  const uint16_t* __restrict__ code,
                                  float* __restrict__ out, int W, int H,
                                  int pitch, float occupied_cost) {
  const int x = (blockIdx.x * blockDim.x + threadIdx.x) * (VEC ? 4 : 1);
  const int y = blockIdx.y;
  if (x >= W || y >= H) return;
  const size_t q = (size_t)(y + kPadRows) * pitch + x + kPadLeft;
  if (VEC) {
    float4 v = *reinterpret_cast<const float4*>(j + q);
    const uint2 c = *reinterpret_cast<const uint2*>(code + q);
    if (c.x & kCodeOccBit) v.x = occupied_cost;
    if (c.x & (kCodeOccBit << 16)) v.y = occupied_cost;
    if (c.y & kCodeOccBit) v.z = occupied_cost;
    if (c.y & (kCodeOccBit << 16)) v.w = occupied_cost;
    *reinterpret_cast<float4*>(out + (size_t)y * W + x) = v;
  } else {
    out[(size_t)y * W + x] = (code[q] & kCodeOccBit) ? occupied_cost : j[q];
  }
}

// The action at the belief mode.  One CTA per belief.
__global__ void __launch_bounds__(256)
mdp_plan_kernel(const float* __restrict__ beliefs, size_t n,
                const uint8_t* __restrict__ action, uint8_t* __restrict__ out,
                unsigned long long* __restrict__ out_index) {
  const unsigned long long mode = belief_mode(beliefs + (size_t)blockIdx.x * n, n);
  if (threadIdx.x == 0) {
    // (a multi-GPU handle keeps the action grid spread over its devices: the
    // cell index goes back and the host looks the action up)
    if (action != nullptr) out[blockIdx.x] = action[mode];
    else out_index[blockIdx.x] = mode;
  }
}

// ---------------------------------------------------------------------------
// Batches of equal-size instances (pp2d_mdp_batch_*, DESIGN.md section 4).
// Instance k owns rows [k*(H+1), k*(H+1)+H) of one tall grid of
// count*(H+1)-1 rows; the row between two instances is an occupied separator
// whose J stays +0, so the fused sweep kernel runs the tall grid unchanged.
struct BatchCodeParams {
  const uint8_t* maps;   // count maps of H*W bytes back to back, or one shared map
  size_t map_stride;     // H*W, or 0 for the shared map
  const uint32_t* goals; // [count][2]: (x, y) of each instance
  uint16_t* code;        // code plane of the tall grid
  int W, H, count, pitch, rows_phys;
};

// CodeParams of the instance that owns tall row gy, and gy's row ly in it.
// Rows above the first instance belong to instance 0 and rows below the last
// one to the last instance; like a separator (ly == H) they lie outside the
// instance's rows [0, H) and so read as out of map = occupied.
__device__ __forceinline__ CodeParams batch_row(const BatchCodeParams& p, int gy, int& ly) {
  const int k = min(gy < 0 ? 0 : gy / (p.H + 1), p.count - 1);
  ly = gy - k * (p.H + 1);
  CodeParams c;
  c.occ = p.maps + (size_t)k * p.map_stride;
  c.code = p.code;
  c.W = p.W;
  c.Htot = p.H;
  c.pitch = p.pitch;
  c.rows_phys = p.rows_phys;
  c.row_begin = 0;
  c.occ_row0 = 0;
  c.occ_rows = p.H;
  c.gx = (int)__ldg(p.goals + 2 * k);
  c.gy = (int)__ldg(p.goals + 2 * k + 1);
  return c;
}

// code_march on the tall grid: every row is built from the map and goal of
// its own instance.
__device__ __forceinline__ CodeParams row_of(const BatchCodeParams& p, int gy, int& ly) {
  return batch_row(p, gy, ly);
}
__device__ __forceinline__ int first_row(const BatchCodeParams&) { return 0; }

// grid: (ceil(pitch / 4 / kCodeThreads), any); blocks stride over the
// kCodeRows row groups.
__global__ void __launch_bounds__(kCodeThreads) mdp_batch_code_kernel(const BatchCodeParams p) {
  const int c0 = 4 * (blockIdx.x * kCodeThreads + threadIdx.x);
  if (c0 >= p.pitch) return;
  const int x0 = c0 - kPadLeft;
  // instance bases are H*W apart: 4-aligned whenever W is
  const bool fast = (p.W & 3) == 0 && (x0 & 3) == 0 && x0 >= 0 && x0 + 3 < p.W &&
                    (reinterpret_cast<uintptr_t>(p.maps) & 3u) == 0;
  for (int r0 = blockIdx.y * kCodeRows; r0 < p.rows_phys; r0 += gridDim.y * kCodeRows) {
    if (fast) code_march<true>(p, c0, r0);
    else code_march<false>(p, c0, r0);
  }
}

// Per-instance max |J - Jchk| over the rows of the instances in `list` (the
// separators are not read), then Jchk = J there: mdp_residual_kernel
// segmented by instance.  blocks_per CTAs serve one instance: block b takes
// instance list[b / blocks_per].  floor[i] is list[i]'s floor: the change of
// the occupied cells' closed form between its own check point and sweep
// count, or 0 when its map has no occupied cell.
__global__ void __launch_bounds__(256)
mdp_batch_residual_kernel(const float* __restrict__ j, float* __restrict__ chk,
                          const uint32_t* __restrict__ list, const float* __restrict__ floor,
                          int blocks_per, int H, int pitch, uint32_t* result) {
  const uint32_t i = blockIdx.x / blocks_per;
  const uint32_t k = list[i];
  const int part = (int)(blockIdx.x % blocks_per);
  const size_t off = ((size_t)k * (H + 1) + kPadRows) * pitch;
  const float4* __restrict__ a4 = reinterpret_cast<const float4*>(j + off);
  float4* __restrict__ b4 = reinterpret_cast<float4*>(chk + off);
  const size_t n4 = (size_t)H * pitch / 4;
  float m = floor[i];
  for (size_t i = (size_t)part * blockDim.x + threadIdx.x; i < n4;
       i += (size_t)blocks_per * blockDim.x) {
    const float4 a = a4[i];
    const float4 b = b4[i];
    m = fmaxf(m, fmaxf(fmaxf(fabsf(a.x - b.x), fabsf(a.y - b.y)),
                       fmaxf(fabsf(a.z - b.z), fabsf(a.w - b.w))));
    b4[i] = a;
  }
  block_max_to(m, result + k);
}

struct BatchFreezeParams {
  float* j[2];             // both J planes of the tall grid; j[cur] holds J_n
  int cur;
  uint16_t* code;
  const uint8_t* action;   // dense action grid of the tall grid
  float* res_cost;         // [count][H][W]
  uint8_t* res_action;     // [count][H][W]
  const uint32_t* list;    // instances to snapshot
  const float* trapped;    // [n_list]: J of an occupied cell at list[i]'s sweep count
  int n_list;
  int W, H, pitch;
  UnitMask mask;           // FREEZE: the mask to clear
  const uint8_t* frozen;   // [count]: 1 = instance stopped
  int count, Htot;
};

// Snapshot of the instances in `list` into their result slots: J with the
// occupied cells at `trapped`, and the action grid (the dense export of
// mdp_export_kernel, one slot per instance).  FREEZE (instances that just met
// the stopping rule):
//   (a) after the snapshot their rows of the tall grid become occupied rows:
//       code = padding, J = 0 in both planes.  Their live values are never
//       read again, and a unit made of such rows and separators computes
//       +0 from +0, so it never marks its neighbours when it runs;
//   (b) the bits of every unit whose rows all lie in stopped instances and
//       separators are cleared in mask.need.
// One thread per cell, then one thread per row block (grid-stride loops).
template <bool FREEZE>
__global__ void __launch_bounds__(256) mdp_batch_freeze_kernel(const BatchFreezeParams p) {
  const size_t hw = (size_t)p.H * p.W;
  const size_t cells = hw * (size_t)p.n_list;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (size_t t = t0; t < cells; t += stride) {
    const size_t i = t / hw;
    const uint32_t k = p.list[i];
    const size_t c = t % hw;
    const int y = (int)(c / p.W), x = (int)(c - (size_t)y * p.W);
    const size_t ty = (size_t)k * (p.H + 1) + y;     // row in the tall grid
    const size_t q = (ty + kPadRows) * p.pitch + x + kPadLeft;
    const size_t dst = (size_t)k * hw + c;
    p.res_cost[dst] = (p.code[q] & kCodeOccBit) ? p.trapped[i] : p.j[p.cur][q];
    p.res_action[dst] = p.action[ty * p.W + x];
    if (FREEZE) {
      p.code[q] = (uint16_t)kCodeOccBit;
      p.j[0][q] = 0.0f;
      p.j[1][q] = 0.0f;
    }
  }
  const UnitMask& m = p.mask;
  if (!FREEZE || m.need == nullptr) return;
  for (size_t rb = t0; rb < (size_t)m.n_rb; rb += stride) {
    const int y0 = (int)rb * m.rows_per_unit;
    const int y1 = min(y0 + m.rows_per_unit, p.Htot);
    // instances with a row in [y0, y1): a separator row belongs to none
    int k0 = y0 / (p.H + 1), k1 = (y1 - 1) / (p.H + 1);
    if (y0 - k0 * (p.H + 1) == p.H) ++k0;
    if ((y1 - 1) - k1 * (p.H + 1) == p.H) --k1;
    bool all_frozen = true;
    for (int k = k0; k <= k1 && all_frozen; ++k) all_frozen = p.frozen[k] != 0;
    if (!all_frozen) continue;
    const int u0 = (int)rb * m.n_strips;
    for (int w = u0 >> 5; w <= (u0 + m.n_strips - 1) >> 5; ++w)
      atomicAnd(m.need + w, ~unit_range_bits(w, u0, u0 + m.n_strips));
  }
}

// New maps and goals for the instances in `list` (pp2d_mdp_batch_update,
// DESIGN.md section 4): mdp_update_map_kernel on their rows of the tall grid
// only, with each instance's own trapped(n_k).  An instance that a solve froze
// (thaw[i] != 0) has padding codes and J = +0 in its rows: its J comes from
// its result slot, where the occupied cells already hold trapped(n_k), and
// its action rows are restored from the slot, so that plan and way-points
// return what they returned before the update.
struct BatchUpdateParams {
  BatchCodeParams c;       // goals (the new ones), code plane and sizes; maps unused
  const uint8_t* maps;     // the new map of list[i] at maps + i * map_stride (0: one map)
  size_t map_stride;
  const uint32_t* list;    // [n_list] instances
  const float* trapped;    // [n_list] J of an occupied cell at list[i]'s sweep count
  const uint32_t* thaw;    // [n_list] 1: list[i] is frozen
  int n_list, groups;      // groups: kCodeRows row groups per instance
  float* j;                // j[cur]
  float* jchk;
  uint8_t* action;         // dense action grid of the tall grid
  const float* res_cost;   // [count][H][W]
  const uint8_t* res_action;
  UnitMask mask;           // seeded with the dirty units
};

// grid: (ceil(pitch / 4 / kCodeThreads), any); blocks stride over the row
// groups of the listed instances.  Thread shape and dirty-unit seeding as in
// mdp_update_map_kernel.
__global__ void __launch_bounds__(kCodeThreads) mdp_batch_update_kernel(const BatchUpdateParams p) {
  const int lane = threadIdx.x & 31;
  const int c0 = 4 * (blockIdx.x * kCodeThreads + threadIdx.x);
  const bool active = c0 < p.c.pitch;
  const int x0 = c0 - kPadLeft;
  const int W = p.c.W, H = p.c.H;
  const size_t hw = (size_t)H * W;
  // the maps are H*W bytes apart: 4-aligned whenever W is
  const bool fast = (W & 3) == 0 && (x0 & 3) == 0 && x0 >= 0 && x0 + 3 < W &&
                    (reinterpret_cast<uintptr_t>(p.maps) & 3u) == 0;
  const int k_lo = max(x0, 0) / kUnitStrip;
  for (int g = blockIdx.y; g < p.n_list * p.groups; g += gridDim.y) {   // uniform over the block
    const int i = g / p.groups;
    const int ly0 = (g - i * p.groups) * kCodeRows;
    const int ly1 = min(ly0 + kCodeRows, H);
    const uint32_t k = __ldg(p.list + i);
    const float trapped = __ldg(p.trapped + i);
    const bool thaw = __ldg(p.thaw + i) != 0;
    // batch_row over a one-map view: every row of instance k reads map i
    BatchCodeParams bp = p.c;
    bp.maps = p.maps + (size_t)i * p.map_stride;
    bp.map_stride = 0;
    auto mask = [&](int gy) {
      int ly;
      const CodeParams c = batch_row(bp, gy, ly);
      return fast ? occ_mask6<true>(c, x0, ly) : occ_mask6<false>(c, x0, ly);
    };
    int ty = (int)k * (H + 1) + ly0;              // row of the tall grid
    uint32_t m0 = mask(ty - 1), m1 = mask(ty);
    for (int ly = ly0; ly < ly1; ++ly, ++ty) {
      const uint32_t m2 = mask(ty + 1);
      int cy;
      const CodeParams c = batch_row(bp, ty, cy);
      uint32_t code[4];
      cell_codes4(c, x0, cy, m0, m1, m2, code);
      m0 = m1;
      m1 = m2;
      bool dirty_lo = false, dirty_hi = false;
      if (active) {
        // row ly of k's result slot; a frozen row's codes are all padding:
        // every free cell takes its slot value
        const size_t slot = (size_t)k * hw + (size_t)ly * W;
        replan_cells4(p.c.code, p.j, p.jchk, (size_t)(ty + kPadRows) * p.c.pitch + c0, x0, k_lo,
                      code, trapped, thaw ? p.res_cost + slot : nullptr, dirty_lo, dirty_hi);
        if (thaw) {
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (x0 + e >= 0 && x0 + e < W)
              p.action[(size_t)ty * W + x0 + e] = __ldg(p.res_action + slot + x0 + e);
        }
      }
      if (p.mask.need != nullptr && __any_sync(0xffffffffu, dirty_lo || dirty_hi))
        seed_dirty_units(p.mask, min(ty / p.mask.rows_per_unit, p.mask.n_rb - 1), k_lo, dirty_lo,
                         dirty_hi, lane);
    }
  }
}

// mdp_plan_kernel with an action grid per belief (H*W bytes at bases[i]).
__global__ void __launch_bounds__(256)
mdp_batch_plan_kernel(const float* __restrict__ beliefs, size_t n,
                      const uint8_t* const* __restrict__ bases, uint8_t* __restrict__ out) {
  const unsigned long long mode = belief_mode(beliefs + (size_t)blockIdx.x * n, n);
  if (threadIdx.x == 0) out[blockIdx.x] = bases[blockIdx.x][mode];
}

}  // namespace pp2d
