// Test driver for the goal sets of PomdpPathPlanning2d and SearchTreeBatch with
// goals (include/pp2d/planners.hpp):
//   pomdp_goals_main <map.png> <goal_x> <goal_y> <gamma> <dir0> <n_pbvi> <iters>
//                    <goals.bin> <beliefs.bin> <tree_goals.bin> <dir1> [<dir2> ...]
// dir0: goal 0's checkpoint (the seven text files), dir1.. the checkpoints of
// goals 1.. (goals.bin: uint32 (x, y) per goal); beliefs.bin: float32 [n][HW];
// tree_goals.bin: uint32 per tree.  Plans every tree, updates each with its
// action and observation 0, plans again, and prints per tree the two actions
// and the bits of the two values.
#include <cinttypes>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "pp2d/planners.hpp"

using namespace path_planning_2d;

int main(int argc, char** argv) {
  if (argc < 12) return 2;
  Params p{{"map_path", argv[1]}, {"goal_x", argv[2]}, {"goal_y", argv[3]},
           {"discount_factor", argv[4]}, {"map_resolution", "0.2"},
           {"read_data_from_file", "true"}, {"data_dir", argv[5]},
           {"belief_set_size", argv[6]}, {"max_search_tree_depth", "50"},
           {"max_online_iteration", argv[7]}};
  PomdpPathPlanning2d planner(p);
  if (!planner.initialize()) { std::printf("INIT_FAILED\n"); return 0; }
  std::vector<uint8_t> graw, braw, traw;
  if (!pp2d::read_file(argv[8], graw) || !pp2d::read_file(argv[9], braw) ||
      !pp2d::read_file(argv[10], traw))
    return 1;
  std::vector<std::array<uint32_t, 2>> goals(graw.size() / 8);
  std::memcpy(goals.data(), graw.data(), goals.size() * 8);
  std::vector<std::string> dirs(argv + 11, argv + argc);
  if (!planner.loadGoalsFromFiles(goals, dirs)) { std::printf("LOAD_FAILED\n"); return 0; }
  std::vector<float> beliefs(braw.size() / 4);
  std::memcpy(beliefs.data(), braw.data(), beliefs.size() * 4);
  std::vector<uint32_t> tree_goals(traw.size() / 4);
  std::memcpy(tree_goals.data(), traw.data(), tree_goals.size() * 4);
  SearchTreeBatch batch(planner.handle(), beliefs.data(), tree_goals);
  std::vector<uint32_t> all(tree_goals.size());
  for (uint32_t k = 0; k < all.size(); ++k) all[k] = k;
  const uint32_t iters = (uint32_t)atoi(argv[7]);
  std::vector<float> v0, v1;
  const std::vector<uint8_t> a0 = batch.plan(all, 50, iters, &v0);
  batch.update(all, a0, std::vector<uint8_t>(all.size(), 0));
  const std::vector<uint8_t> a1 = batch.plan(all, 50, iters, &v1);
  for (uint32_t k = 0; k < all.size(); ++k) {
    uint32_t r0, r1;
    std::memcpy(&r0, &v0[k], 4);
    std::memcpy(&r1, &v1[k], 4);
    std::printf("RESULT k=%u a0=%u r0=%08x a1=%u r1=%08x\n", k, a0[k], r0, a1[k], r1);
  }
  return 0;
}
