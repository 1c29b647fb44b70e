// handles.h -- what the closed-loop rollouts (rollout.cu) read from the
// planner and simulator handles.  The structs stay in mdp.cu and sim.cu; these
// accessors are defined next to them.
#pragma once
#include "../../include/pp2d.h"

#include <cuda_runtime.h>

#include <cstdint>

namespace pp2d {

// A planner as the belief-mode plan kernels read it.
struct PlannerView {
  uint32_t H = 0, W = 0;
  bool sharded = false;            // a shard or a multi-GPU container
  const uint8_t* action = nullptr; // device [H][W]
  uint32_t gx = 0, gy = 0;
  cudaStream_t stream = nullptr;   // the stream the action grid is written on
};

PlannerView mdp_view(const pp2d_mdp* h);                                   // mdp.cu
uint32_t mdp_batch_count(const pp2d_mdp_batch* b);                         // mdp.cu
// Instance k < count: its goal and its action grid (the snapshot once frozen).
PlannerView mdp_batch_view(const pp2d_mdp_batch* b, uint32_t k);           // mdp.cu

// The root beliefs of trees 0 .. count-1 of a tree batch, [count][HW] into
// host memory (pomdp.cu).
int tree_batch_root_beliefs(pp2d_tree_batch* b, float* out);               // pomdp.cu

struct SimView {
  uint32_t H = 0, W = 0;
  const uint8_t* map_host = nullptr;   // [H][W], 1 = occupied
  const uint8_t* map = nullptr;        // device copy
};
SimView sim_view(const pp2d_sim* s);                                       // sim.cu

}  // namespace pp2d
