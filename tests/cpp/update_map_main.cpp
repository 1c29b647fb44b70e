// Test driver for MdpPathPlanning2d::updateMap (include/pp2d/planners.hpp):
//   update_map <map.png> <goal_x> <goal_y> <gamma> <new_map.bin> <new_goal_x> <new_goal_y>
// initialize() on the PNG, then updateMap() with the raw height*width bytes of
// new_map.bin; prints the sweep counts and FNV-1a hashes of J and the actions.
#include <cinttypes>
#include <cstdio>
#include <cstdlib>
#include <string>

#include "pp2d/planners.hpp"

using namespace path_planning_2d;

static uint64_t fnv(const void* p, size_t n) {
  const uint8_t* b = static_cast<const uint8_t*>(p);
  uint64_t h = 1469598103934665603ull;
  for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 1099511628211ull; }
  return h;
}

int main(int argc, char** argv) {
  if (argc < 8) return 2;
  Params p{{"map_path", argv[1]}, {"goal_x", argv[2]}, {"goal_y", argv[3]},
           {"discount_factor", argv[4]}, {"map_resolution", "0.2"}};
  MdpPathPlanning2d planner(p);
  if (!planner.initialize()) { std::printf("INIT_FAILED\n"); return 0; }
  const int first = planner.total_iterations;
  std::vector<uint8_t> next;
  if (!pp2d::read_file(argv[5], next)) return 1;
  if (!planner.updateMap(next, atoi(argv[6]), atoi(argv[7]))) {
    std::printf("UPDATE_FAILED\n");
    return 0;
  }
  std::printf("RESULT sweeps0=%d sweeps=%d cost=%016" PRIx64 " action=%016" PRIx64 "\n", first,
              planner.total_iterations,
              fnv(planner.optimal_cost.data(), planner.optimal_cost.size() * 4),
              fnv(planner.optimal_action.data(), planner.optimal_action.size()));
  return 0;
}
