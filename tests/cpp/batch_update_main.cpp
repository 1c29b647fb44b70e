// Test driver for MdpBatchPathPlanning2d::updateMap (include/pp2d/planners.hpp):
//   batch_update_main <maps.bin> <height> <width> <goals.bin> <gamma>
//                     <instances.bin> <maps2.bin> <goals2.bin>
// maps.bin / goals.bin as for batch_main; instances.bin: uint32 instance
// indices; maps2.bin: one shared map or one map per listed instance;
// goals2.bin: uint32 (x, y) per listed instance.  Runs valueIteration(),
// updateMap() and prints, per instance, the sweep count and residual count of
// the solve after the update and FNV-1a hashes of J and the actions.
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

static std::vector<std::array<uint32_t, 2>> pairs(const std::vector<uint8_t>& raw) {
  std::vector<std::array<uint32_t, 2>> out(raw.size() / 8);
  std::memcpy(out.data(), raw.data(), out.size() * 8);
  return out;
}

int main(int argc, char** argv) {
  if (argc < 9) return 2;
  std::vector<uint8_t> maps, graw, iraw, maps2, graw2;
  if (!pp2d::read_file(argv[1], maps) || !pp2d::read_file(argv[4], graw) ||
      !pp2d::read_file(argv[6], iraw) || !pp2d::read_file(argv[7], maps2) ||
      !pp2d::read_file(argv[8], graw2))
    return 1;
  const uint32_t height = (uint32_t)atoi(argv[2]), width = (uint32_t)atoi(argv[3]);
  std::vector<uint32_t> instances(iraw.size() / 4);
  std::memcpy(instances.data(), iraw.data(), instances.size() * 4);
  MdpBatchPathPlanning2d batch(height, width, maps, pairs(graw), (float)atof(argv[5]));
  batch.valueIteration();
  if (!batch.updateMap(instances, maps2, pairs(graw2))) return 3;
  for (uint32_t k = 0; k < batch.count(); ++k) {
    const std::vector<float> cost = batch.optimalCost(k);
    const std::vector<uint8_t> action = batch.optimalAction(k);
    std::printf("RESULT k=%u sweeps=%u batches=%zu cost=%016" PRIx64 " action=%016" PRIx64 "\n",
                k, batch.sweeps[k], batch.residuals[k].size(),
                fnv(cost.data(), cost.size() * 4), fnv(action.data(), action.size()));
  }
  return 0;
}
