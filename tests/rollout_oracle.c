/*
 * tests/rollout_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU restatement of one closed-loop episode of pp2d_sim_rollout_mdp*
 * (DESIGN.md section 7, "Closed-loop rollouts"), built from the filter oracle
 * oracle/sim_oracle.c (included unchanged: transition_probability and the two
 * oracle_sim_update_* steps) and the generator of philox.h.  The planner is a
 * dense action grid; its action is taken at a plain-C belief mode.  Compiled
 * by tests/rollout_oracle_py.py with -ffp-contract=off like the other oracles.
 */
#include "../oracle/sim_oracle.c"
#include "../path_planning_2d_b200/csrc/philox.h"

void oracle_philox(uint32_t c[4], uint32_t k0, uint32_t k1) { pp2d_philox4x32_10(c, k0, k1); }

void oracle_step_uniforms(uint64_t seed, uint64_t e, uint32_t t, float r[5]) {
  pp2d_step_uniforms(seed, e, t, r);
}

/* MdpPathPlanning2d::beliefCallback: first strict maximum from (0.0f, 0). */
static int32_t belief_mode(const float* b, int32_t n) {
  float bm = 0.0f;
  int32_t bi = 0;
  for (int32_t i = 0; i < n; ++i)
    if (b[i] > bm) { bm = b[i]; bi = i; }
  return bi;
}

/* Motion slot of action u for the uniform r: the naive probabilities (the
 * motion model of a cell with nothing blocked) summed in ascending slot order
 * with separate roundings; the first slot whose sum exceeds r, else the last
 * slot of non-zero probability. */
int32_t oracle_motion_slot(uint8_t u, float r) {
  static const uint8_t open3[9] = {0};
  float tp[9], acc = 0.0f;
  int32_t last = 4;
  transition_probability(3, 3, open3, 1, 1, u, tp);
  for (int32_t i = 0; i < 9; ++i) {
    if (tp[i] != 0.0f) last = i;
    acc += tp[i];
    if (r < acc) return i;
  }
  return last;
}

static uint8_t occupied(int32_t h, int32_t w, const uint8_t* grid, int32_t x, int32_t y) {
  return (x < 0 || x >= w || y < 0 || y >= h) ? 1 : (grid[y * w + x] > 0);
}

/* One episode e on world map `grid`: planner action grid `act` [h][w], goal
 * (gx, gy), start (sx, sy), belief (updated in place; the final belief).  The
 * recording arrays may be NULL. */
void oracle_rollout_episode(int32_t h, int32_t w, const uint8_t* grid, const uint8_t* act,
                            uint32_t gx, uint32_t gy, uint32_t sx, uint32_t sy, float* belief,
                            uint32_t max_steps, uint64_t seed, uint64_t e, uint32_t stats[4],
                            uint32_t* cells, uint8_t* actions, uint8_t* meas) {
  static const int8_t ox[4] = {0, -1, 1, 0};
  static const int8_t oy[4] = {-1, 0, 0, 1};
  int32_t x = (int32_t)sx, y = (int32_t)sy;
  uint32_t t = 0, collisions = 0;
  if (cells) cells[0] = (uint32_t)(y * w + x);
  for (;; ++t) {
    if ((uint32_t)x == gx && (uint32_t)y == gy) break;
    if (t == max_steps) break;
    const uint8_t u = act[belief_mode(belief, h * w)];
    float r[5];
    pp2d_step_uniforms(seed, e, t, r);
    const int32_t slot = oracle_motion_slot(u, r[0]);
    if (slot != 4) {
      const int32_t tx = x + slot % 3 - 1, ty = y + slot / 3 - 1;
      if (occupied(h, w, grid, tx, ty)) ++collisions;
      else { x = tx; y = ty; }
    }
    uint8_t m4[4], bits = 0;
    for (int j = 0; j < 4; ++j) {
      m4[j] = occupied(h, w, grid, x + ox[j], y + oy[j]);
      if (r[1 + j] < 0.02f) m4[j] ^= 1;
      bits |= (uint8_t)(m4[j] << j);
    }
    oracle_sim_update_action(h, w, grid, belief, u);
    oracle_sim_update_measurement(h, w, grid, belief, m4);
    if (cells) cells[t + 1] = (uint32_t)(y * w + x);
    if (actions) actions[t] = u;
    if (meas) meas[t] = bits;
  }
  stats[0] = t;
  stats[1] = ((uint32_t)x == gx && (uint32_t)y == gy) ? 1 : 0;
  stats[2] = collisions;
  stats[3] = (uint32_t)(y * w + x);
}
