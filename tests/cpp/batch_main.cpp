// Test driver for MdpBatchPathPlanning2d (include/pp2d/planners.hpp):
//   batch_main <maps.bin> <height> <width> <goals.bin> <gamma>
// maps.bin: one shared height*width map or one map per goal, back to back;
// goals.bin: uint32 (x, y) per instance.  Runs valueIteration() and prints,
// per instance, its sweep count, residual count and FNV-1a hashes of J and
// the actions.
#include <cinttypes>
#include <cstdio>
#include <cstdlib>
#include <cstring>
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
  if (argc < 6) return 2;
  std::vector<uint8_t> maps, graw;
  if (!pp2d::read_file(argv[1], maps) || !pp2d::read_file(argv[4], graw)) return 1;
  const uint32_t height = (uint32_t)atoi(argv[2]), width = (uint32_t)atoi(argv[3]);
  std::vector<std::array<uint32_t, 2>> goals(graw.size() / 8);
  std::memcpy(goals.data(), graw.data(), goals.size() * 8);
  MdpBatchPathPlanning2d batch(height, width, maps, goals, (float)atof(argv[5]));
  batch.valueIteration();
  for (uint32_t k = 0; k < batch.count(); ++k) {
    const std::vector<float> cost = batch.optimalCost(k);
    const std::vector<uint8_t> action = batch.optimalAction(k);
    std::printf("RESULT k=%u sweeps=%u batches=%zu cost=%016" PRIx64 " action=%016" PRIx64 "\n",
                k, batch.sweeps[k], batch.residuals[k].size(),
                fnv(cost.data(), cost.size() * 4), fnv(action.data(), action.size()));
  }
  return 0;
}
