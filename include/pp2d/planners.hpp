// pp2d/planners.hpp -- C++ host side above the C ABI: ROS-free mirrors of the
// reference's planner classes, same names, members and error behaviour.
//
//   reference                                           here
//   include/path_planning_2d/path_planning_2d_base.h    PathPlanning2dBase
//   include/path_planning_2d/mdp_path_planning_2d.h     MdpPathPlanning2d
//   include/path_planning_2d/pomdp_path_planning_2d.h   PomdpPathPlanning2d
//   include/path_planning_2d/search_tree.h              SearchTree
//
// What changes against the reference: ros::NodeHandle parameters become a
// string map (`Params`), dummy_simulator::Belief becomes the plain struct
// `Belief`, publishers become return values, cv::imread becomes
// pp2d/map_io.hpp, and every device-side call goes through include/pp2d.h.
// CUDA failures keep the reference's print-and-exit behaviour
// (helper_cuda.h:984-999) through PP2D_CHECK.
#pragma once
#include <algorithm>
#include <array>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../pp2d.h"
#include "map_io.hpp"

#define PP2D_CHECK(call)                                                    \
  do {                                                                      \
    int rc_ = (call);                                                       \
    if (rc_ != PP2D_OK) {                                                   \
      std::fprintf(stderr, "pp2d error at %s:%d code=%d \"%s\" : %s\n",    \
                   __FILE__, __LINE__, rc_, #call, pp2d_last_error());      \
      std::exit(EXIT_FAILURE);                                              \
    }                                                                       \
  } while (0)

namespace path_planning_2d {

typedef std::map<std::string, std::string> Params;   // ~ private ROS params

struct Belief {                       // dummy_simulator/msg/Belief.msg
  uint8_t action = 0;
  uint8_t measurement[4] = {0, 0, 0, 0};
  std::vector<float> belief;
};

class PathPlanning2dBase {            // path_planning_2d_base.h:29-79
 public:
  explicit PathPlanning2dBase(const Params& n) : nh(n) {}
  virtual ~PathPlanning2dBase() {}
  virtual bool initialize() = 0;

 protected:
  virtual bool loadParameters() = 0;
  bool getParam(const std::string& k, std::string& v) const {
    auto it = nh.find(k);
    if (it == nh.end()) return false;
    v = it->second;
    return true;
  }
  bool getParam(const std::string& k, int32_t& v) const {
    std::string s;
    if (!getParam(k, s)) return false;
    v = (int32_t)std::strtol(s.c_str(), nullptr, 10);
    return true;
  }
  bool getParam(const std::string& k, float& v) const {
    std::string s;
    if (!getParam(k, s)) return false;
    v = (float)std::strtod(s.c_str(), nullptr);   // double param -> float member
    return true;
  }
  bool getParam(const std::string& k, bool& v) const {
    std::string s;
    if (!getParam(k, s)) return false;
    v = (s == "true" || s == "1");
    return true;
  }
  // loadMapFromFile (src/mdp/path_planning_2d.cu:191-205)
  virtual bool loadMapFromFile() {
    return pp2d::load_occupancy(map_path, map_width, map_height, grid_map);
  }

  Params nh;
  std::string map_path;
  uint32_t map_width = 0, map_height = 0;
  double map_resolution = 0.0;
  std::vector<uint8_t> grid_map;
  int32_t goal[2] = {0, 0};
  float discount_factor = 0.0f;

 public:
  uint32_t width() const { return map_width; }
  uint32_t height() const { return map_height; }
  const std::vector<uint8_t>& map() const { return grid_map; }
};

// ---------------------------------------------------------------------------
class MdpPathPlanning2d : public PathPlanning2dBase {
 public:
  explicit MdpPathPlanning2d(const Params& n) : PathPlanning2dBase(n) {}
  ~MdpPathPlanning2d() override { pp2d_mdp_destroy(mdp_); }

  // src/mdp/path_planning_2d.cu:72-140
  bool initialize() override {
    if (!loadParameters()) {
      std::fprintf(stderr, "Cannot load all required parameters...\n");
      return false;
    }
    if (!loadMapFromFile()) {
      std::fprintf(stderr, "Cannot load the map %s\n", map_path.c_str());
      return false;
    }
    // One ROS process, `num_gpus` GPUs (optional parameters, not in the
    // reference: num_gpus, default 1, and gpu_devices, a comma-separated list
    // of CUDA device ordinals, one per row shard): the same handle type, the
    // same calls below, bit-identical results.
    int rc;
    if (num_gpus > 1 || !gpu_devices.empty())
      rc = pp2d_mdp_create_multi(map_height, map_width, grid_map.data(), goal[0], goal[1],
                                 discount_factor,
                                 gpu_devices.empty() ? (uint32_t)num_gpus
                                                     : (uint32_t)gpu_devices.size(),
                                 gpu_devices.empty() ? nullptr : gpu_devices.data(), &mdp_);
    else
      rc = pp2d_mdp_create(map_height, map_width, grid_map.data(), goal[0], goal[1],
                           discount_factor, &mdp_);
    if (rc == PP2D_ERR_GOAL_OCCUPIED || rc == PP2D_ERR_INVALID) {
      std::fprintf(stderr, "The assigned goal (%d %d) is at a occupied cell...\n", goal[0],
                   goal[1]);
      return false;
    }
    PP2D_CHECK(rc);
    std::printf("Solve MDP with value iteration...\n");
    valueIteration();
    optimal_cost.resize((size_t)map_height * map_width);
    optimal_action.resize((size_t)map_height * map_width);
    PP2D_CHECK(pp2d_mdp_download(mdp_, optimal_cost.data(), optimal_action.data()));
    std::printf("Initialization finished...\n");
    return true;
  }

  // src/mdp/path_planning_2d.cu:168-189: the action at the belief mode.
  uint8_t beliefCallback(const Belief& belief) const {
    float belief_mode = 0.0f;
    int32_t belief_mode_idx = 0;
    for (size_t i = 0; i < belief.belief.size(); ++i)
      if (belief.belief[i] > belief_mode) {
        belief_mode_idx = (int32_t)i;
        belief_mode = belief.belief[i];
      }
    return optimal_action[belief_mode_idx];
  }

  // Way-points of the greedy policy (row W of SURVEY.md section 8a).
  std::vector<uint32_t> waypoints(uint32_t sx, uint32_t sy) const {
    std::vector<uint32_t> cells((size_t)map_height * map_width);
    uint32_t n = 0;
    PP2D_CHECK(pp2d_mdp_waypoints(mdp_, sx, sy, cells.data(), (uint32_t)cells.size(), &n));
    cells.resize(n);
    return cells;
  }

  // Units run / launched by the fused sweeps so far (pp2d_mdp_work_counters).
  std::array<uint64_t, 2> workCounters() {
    std::array<uint64_t, 2> c{};
    PP2D_CHECK(pp2d_mdp_work_counters(mdp_, c.data()));
    return c;
  }

  std::vector<float> optimal_cost;
  std::vector<uint8_t> optimal_action;
  int total_iterations = 0;
  std::vector<double> residuals;

 private:
  bool loadParameters() override {          // src/mdp/path_planning_2d.cu:142-154
    if (!getParam("map_path", map_path)) return false;
    if (!getParam("goal_x", goal[0])) return false;
    if (!getParam("goal_y", goal[1])) return false;
    if (!getParam("discount_factor", discount_factor)) return false;
    float res = 0.f;
    if (!getParam("map_resolution", res)) return false;
    map_resolution = res;
    getParam("num_gpus", num_gpus);
    std::string list;
    if (getParam("gpu_devices", list)) {
      gpu_devices.clear();
      const char* c = list.c_str();
      while (*c) {
        char* end = nullptr;
        const long d = std::strtol(c, &end, 10);
        if (end == c) break;
        gpu_devices.push_back((int)d);
        c = (*end == ',') ? end + 1 : end;
      }
    }
    return true;
  }

  // Not in the reference (one map per process): re-plan on a changed map of
  // the same size and/or a new goal from the current solution
  // (pp2d_mdp_update_map), then valueIteration() from there and the download,
  // as initialize() does.  total_iterations and residuals carry on.  Returns
  // false and changes nothing when the goal is occupied or out of the map.
 public:
  bool updateMap(const std::vector<uint8_t>& map, int32_t goal_x, int32_t goal_y) {
    if (map.size() != (size_t)map_width * map_height) return false;
    const int rc = pp2d_mdp_update_map(mdp_, map.data(), (uint32_t)goal_x, (uint32_t)goal_y);
    if (rc == PP2D_ERR_GOAL_OCCUPIED || rc == PP2D_ERR_INVALID) {
      std::fprintf(stderr, "The assigned goal (%d %d) is at a occupied cell...\n", goal_x,
                   goal_y);
      return false;
    }
    PP2D_CHECK(rc);
    grid_map = map;
    goal[0] = goal_x;
    goal[1] = goal_y;
    valueIteration();
    PP2D_CHECK(pp2d_mdp_download(mdp_, optimal_cost.data(), optimal_action.data()));
    return true;
  }

 private:
  // src/mdp/path_planning_2d.cu:207-269 (imshow windows dropped)
  void valueIteration() {
    float cost_inf_norm = 0.0f;
    const double max_optimal_cost = 5.0 / (1.0 - discount_factor);
    do {
      PP2D_CHECK(pp2d_mdp_sweeps(mdp_, 100));
      total_iterations += 100;
      PP2D_CHECK(pp2d_mdp_residual(mdp_, &cost_inf_norm));
      residuals.push_back(cost_inf_norm);
      std::printf("Inf-norm: %f\n", cost_inf_norm);
    } while (cost_inf_norm > max_optimal_cost * 1e-3);
  }

  // src/mdp/path_planning_2d.cu:271-357.  As in the reference it is not called
  // by initialize() (the call is commented out there, :115-116); it needs the
  // state initialize() starts from (J = 0, action = 0), i.e. a reset handle.
  void policyIteration() {
    std::vector<double> res(4096);
    std::vector<uint32_t> changed(4096);
    uint32_t sweeps = 0;
    PP2D_CHECK(pp2d_mdp_policy_iteration(mdp_, &sweeps, res.data(), changed.data(),
                                         (uint32_t)res.size(), 0));
    total_iterations += (int)sweeps;
    for (uint32_t r = 0; r < sweeps / 50 && r < res.size(); ++r) {
      std::printf("Inf-norm: %f\n", res[r]);
      std::printf("# of changed actions: %u\n", changed[r]);
    }
  }

  pp2d_mdp* mdp_ = nullptr;
  int32_t num_gpus = 1;
  std::vector<int> gpu_devices;
};

// Not in the reference (one goal per process): many goals or maps of one size
// solved together on one GPU (pp2d_mdp_batch_*), e.g. one goal per robot of a
// fleet.  maps: height*width bytes shared by every goal, or one map per goal
// back to back; goals: one (x, y) per instance.  Instance k's results equal
// those of MdpPathPlanning2d on its map and goal bit for bit.
class MdpBatchPathPlanning2d {
 public:
  MdpBatchPathPlanning2d(uint32_t height, uint32_t width, const std::vector<uint8_t>& maps,
                         const std::vector<std::array<uint32_t, 2>>& goals, float gamma)
      : height_(height), width_(width), count_((uint32_t)goals.size()) {
    const size_t hw = (size_t)height * width;
    if (maps.size() != hw && maps.size() != hw * goals.size()) {
      std::fprintf(stderr, "MdpBatchPathPlanning2d: one shared map or one map per goal\n");
      std::exit(EXIT_FAILURE);
    }
    PP2D_CHECK(pp2d_mdp_batch_create(height, width, count_, maps.data(),
                                     maps.size() == hw ? 0 : hw, goals.data()->data(), gamma,
                                     &batch_));
  }
  MdpBatchPathPlanning2d(const MdpBatchPathPlanning2d&) = delete;
  MdpBatchPathPlanning2d& operator=(const MdpBatchPathPlanning2d&) = delete;
  ~MdpBatchPathPlanning2d() { pp2d_mdp_batch_destroy(batch_); }

  // valueIteration() of every instance (src/mdp/path_planning_2d.cu:207-269);
  // sweeps[k] and residuals[k] are instance k's.
  void valueIteration() {
    const uint32_t cap = 64;
    std::vector<double> res((size_t)count_ * cap);
    sweeps.assign(count_, 0);
    PP2D_CHECK(pp2d_mdp_batch_solve(batch_, sweeps.data(), res.data(), cap));
    residuals.assign(count_, {});
    for (uint32_t k = 0; k < count_; ++k)
      residuals[k].assign(res.begin() + (size_t)k * cap,
                          res.begin() + (size_t)k * cap + std::min(cap, sweeps[k] / 100));
  }

  // Re-plan the listed instances on new maps and goals from their current
  // solutions (pp2d_mdp_batch_update), then valueIteration() of the instances
  // that are active; sweeps[k] and residuals[k] of the others are 0 and empty.
  // maps: one height*width map shared by the listed instances, or one per
  // instance back to back.  Returns false and changes nothing on a bad
  // argument or an occupied goal.
  bool updateMap(const std::vector<uint32_t>& instances, const std::vector<uint8_t>& maps,
                 const std::vector<std::array<uint32_t, 2>>& goals) {
    const size_t hw = (size_t)height_ * width_;
    if (goals.size() != instances.size() ||
        (maps.size() != hw && maps.size() != hw * instances.size()))
      return false;
    if (instances.empty()) return true;
    const int rc = pp2d_mdp_batch_update(batch_, instances.data(), (uint32_t)instances.size(),
                                         maps.data(), maps.size() == hw ? 0 : hw,
                                         goals.data()->data());
    if (rc == PP2D_ERR_GOAL_OCCUPIED || rc == PP2D_ERR_INVALID) {
      std::fprintf(stderr, "%s\n", pp2d_last_error());
      return false;
    }
    PP2D_CHECK(rc);
    valueIteration();
    return true;
  }

  std::vector<float> optimalCost(uint32_t k) const {
    std::vector<float> c((size_t)height_ * width_);
    PP2D_CHECK(pp2d_mdp_batch_download(batch_, k, 1, c.data(), nullptr));
    return c;
  }
  std::vector<uint8_t> optimalAction(uint32_t k) const {
    std::vector<uint8_t> a((size_t)height_ * width_);
    PP2D_CHECK(pp2d_mdp_batch_download(batch_, k, 1, nullptr, a.data()));
    return a;
  }
  std::vector<uint32_t> waypoints(uint32_t k, uint32_t sx, uint32_t sy) const {
    std::vector<uint32_t> cells((size_t)height_ * width_);
    uint32_t n = 0;
    PP2D_CHECK(pp2d_mdp_batch_waypoints(batch_, k, sx, sy, cells.data(), (uint32_t)cells.size(),
                                        &n));
    cells.resize(n);
    return cells;
  }

  uint32_t count() const { return count_; }
  std::vector<uint32_t> sweeps;
  std::vector<std::vector<double>> residuals;

 private:
  uint32_t height_, width_, count_;
  pp2d_mdp_batch* batch_ = nullptr;
};

// ---------------------------------------------------------------------------
class SearchTree {                     // search_tree.h:130-165
 public:
  SearchTree(pp2d_pomdp* h, const float* b) { PP2D_CHECK(pp2d_tree_create(h, b, &t_)); }
  SearchTree(const SearchTree&) = delete;
  SearchTree& operator=(const SearchTree&) = delete;
  ~SearchTree() { pp2d_tree_destroy(t_); }
  void expand() { PP2D_CHECK(pp2d_tree_expand(t_)); }
  void getOptimalAction(uint8_t& a, float& r) { PP2D_CHECK(pp2d_tree_best_action(t_, &a, &r)); }
  void update(const uint8_t a, const uint8_t z) { PP2D_CHECK(pp2d_tree_update(t_, a, z)); }
  uint32_t getDepth() { return pp2d_tree_depth(t_); }

 private:
  pp2d_tree* t_ = nullptr;
};

// Not in the reference (one tree per process): many SearchTrees on one
// planner handle that live across belief callbacks, e.g. one per robot of a
// fleet, updated and planned together (pp2d_tree_batch_*).  Tree k behaves bit
// for bit like SearchTree(h, beliefs + k * HW) fed the same calls.  With
// `goals`, tree k plans to goal goals[k] of the planner's goal set
// (PomdpPathPlanning2d::setGoals), bit for bit like a SearchTree on a planner
// created with that goal.
class SearchTreeBatch {
 public:
  SearchTreeBatch(pp2d_pomdp* h, const float* beliefs, uint32_t n) {
    PP2D_CHECK(pp2d_tree_batch_create(h, beliefs, n, &b_));
  }
  SearchTreeBatch(pp2d_pomdp* h, const float* beliefs, const std::vector<uint32_t>& goals) {
    PP2D_CHECK(pp2d_tree_batch_create_goals(h, beliefs, goals.data(), (uint32_t)goals.size(), &b_));
  }
  SearchTreeBatch(const SearchTreeBatch&) = delete;
  SearchTreeBatch& operator=(const SearchTreeBatch&) = delete;
  ~SearchTreeBatch() { pp2d_tree_batch_destroy(b_); }
  // update(actions[i], observations[i]) of tree trees[i]
  void update(const std::vector<uint32_t>& trees, const std::vector<uint8_t>& actions,
              const std::vector<uint8_t>& observations) {
    if (actions.size() != trees.size() || observations.size() != trees.size()) {
      std::fprintf(stderr, "SearchTreeBatch::update: one action and observation per tree\n");
      std::exit(EXIT_FAILURE);
    }
    PP2D_CHECK(pp2d_tree_batch_update(b_, trees.data(), (uint32_t)trees.size(), actions.data(),
                                      observations.data()));
  }
  // beliefCallback's loop + getOptimalAction of every listed tree
  std::vector<uint8_t> plan(const std::vector<uint32_t>& trees, uint32_t max_depth,
                            uint32_t max_iter, std::vector<float>* values = nullptr) {
    std::vector<uint8_t> a(trees.size());
    if (values) values->resize(trees.size());
    PP2D_CHECK(pp2d_tree_batch_plan(b_, trees.data(), (uint32_t)trees.size(), max_depth, max_iter,
                                    a.data(), values ? values->data() : nullptr, nullptr));
    return a;
  }

 private:
  pp2d_tree_batch* b_ = nullptr;
};

class PomdpPathPlanning2d : public PathPlanning2dBase {
 public:
  explicit PomdpPathPlanning2d(const Params& n) : PathPlanning2dBase(n) {}
  ~PomdpPathPlanning2d() override {
    delete search_tree;
    pp2d_pomdp_destroy(pomdp_);
  }

  // src/pomdp/path_planning_2d.cu:80-166.  read_data_from_file = false: the
  // model is generated and the FIB and PBVI offline solvers run on the GPU
  // (path_planning_2d.cu:109-125); true (the launch-file default): model
  // tables AND alpha vectors come from the text files the reference's
  // save_data service writes (model_data_trans_prob, model_data_meas_prob,
  // model_data_stage_reward, fib_alphas, fib_actions, pbvi_alphas,
  // pbvi_actions) in `data_dir` (path_planning_2d.cu:127-143), or, with
  // data_format = "binary", from the lossless pp2d_data.bin.
  bool initialize() override {
    if (!loadParameters()) {
      std::fprintf(stderr, "Cannot load all required parameters...\n");
      return false;
    }
    if (!loadMapFromFile()) return false;
    int rc = pp2d_pomdp_create(map_height, map_width, grid_map.data(), goal[0], goal[1],
                               discount_factor, &pomdp_);
    if (rc == PP2D_ERR_GOAL_OCCUPIED || rc == PP2D_ERR_INVALID) {
      std::fprintf(stderr, "The assigned goal (%d %d) is at a occupied cell...\n", goal[0],
                   goal[1]);
      return false;
    }
    PP2D_CHECK(rc);
    // uniform initial belief over the free cells (path_planning_2d.cu:99-107)
    float sum = 0.0f;
    for (size_t i = 0; i < grid_map.size(); ++i) sum += 1.0f - grid_map[i];
    initial_belief.resize(grid_map.size());
    for (size_t i = 0; i < grid_map.size(); ++i) initial_belief[i] = (1.0f - grid_map[i]) / sum;
    if (!read_from_file) {
      const size_t n = (size_t)map_height * map_width;
      // fastInformedBound (fast_informed_bound_cuda.cu:206-276)
      fib_alphas.resize(n * 9);
      fib_actions.resize(9);
      PP2D_CHECK(pp2d_pomdp_solve_fib(pomdp_, fib_alphas.data(), fib_actions.data(),
                                      &fib_sweeps, 0));
      // pointBasedValueIteration (point_based_value_iteration_cuda.cu:643-676);
      // rand() of a fresh process, as in the reference node
      pbvi_alphas.resize((size_t)belief_set_size * n);
      pbvi_actions.resize(belief_set_size);
      PP2D_CHECK(pp2d_pomdp_solve_pbvi(pomdp_, initial_belief.data(), belief_set_size, 1, 0,
                                       nullptr, pbvi_alphas.data(), pbvi_actions.data()));
    } else if (data_format == "binary") {
      if (!loadDataBinary(data_dir)) return false;
    } else if (!loadModelDataFromFile() || !loadFibDataFromFile() || !loadPbviDataFromFile()) {
      // path_planning_2d.cu:127-143: the default launch starts from the seven
      // text files; the model tables it plans with are the ROUNDED ones
      return false;
    }
    PP2D_CHECK(pp2d_pomdp_set_alphas(pomdp_, fib_alphas.data(), fib_actions.data(),
                                     pbvi_alphas.data(), pbvi_actions.data(),
                                     belief_set_size));
    return true;
  }

  // src/pomdp/path_planning_2d.cu:199-241
  uint8_t beliefCallback(const Belief& msg) {
    const uint8_t action = msg.action;
    const uint8_t observation = (uint8_t)((msg.measurement[3] << 3) + (msg.measurement[2] << 2) +
                                          (msg.measurement[1] << 1) + msg.measurement[0]);
    if (search_tree == nullptr) search_tree = new SearchTree(pomdp_, msg.belief.data());
    else search_tree->update(action, observation);
    uint8_t update_counter = 0;
    while (search_tree->getDepth() < (uint32_t)max_search_tree_depth &&
           update_counter++ < max_online_iteration)
      search_tree->expand();
    uint8_t new_action = 0;
    float new_reward = 0.0f;
    search_tree->getOptimalAction(new_action, new_reward);
    last_reward = new_reward;
    return new_action;
  }

  void resetSearchTreeCallback() { delete search_tree; search_tree = nullptr; }

  // Not in the reference (one goal per node): goals 1..n of this planner's
  // goal set (DESIGN.md section 7e), which trees of a SearchTreeBatch can plan
  // to; goal 0 is the launch file's goal.  stage_rewards [n][HW][9] as read
  // from checkpoint files, or nullptr: generated by the model rule.
  void setGoals(const std::vector<std::array<uint32_t, 2>>& goals,
                const float* stage_rewards = nullptr) {
    PP2D_CHECK(pp2d_pomdp_set_goals(pomdp_, goals.empty() ? nullptr : goals[0].data(),
                                    (uint32_t)goals.size(), stage_rewards));
  }
  // setAlphas of goal g (alphas as the solvers or the checkpoint files give them)
  void setGoalAlphas(uint32_t g, const std::vector<float>& fib, const std::vector<uint8_t>& fib_acts,
                     const std::vector<float>& pbvi, const std::vector<uint8_t>& pbvi_acts) {
    PP2D_CHECK(pp2d_pomdp_set_goal_alphas(pomdp_, g, fib.data(), fib_acts.data(), pbvi.data(),
                                          pbvi_acts.data(), (uint32_t)pbvi_acts.size()));
  }
  // Goals 1..n with their checkpoints: dirs[i] holds what the reference's
  // save_data writes for a planner with goal goals[i] (the text files; only
  // model_data_stage_reward of the model is read: the transition and
  // likelihood tables do not depend on the goal).  belief_set_size vectors
  // per goal, as for goal 0.
  bool loadGoalsFromFiles(const std::vector<std::array<uint32_t, 2>>& goals,
                          const std::vector<std::string>& dirs) {
    if (dirs.size() != goals.size()) return false;
    const size_t n = (size_t)map_height * map_width;
    std::vector<float> sr(goals.size() * n * 9), fib(n * 9), pbvi((size_t)belief_set_size * n);
    std::vector<uint8_t> fa(9), pa(belief_set_size);
    for (size_t i = 0; i < goals.size(); ++i) {
      std::vector<float> one(n * 9);
      if (!readFloats(dirs[i] + "/model_data_stage_reward", one)) return false;
      std::copy(one.begin(), one.end(), sr.begin() + i * n * 9);
    }
    setGoals(goals, sr.data());
    for (size_t i = 0; i < goals.size(); ++i) {
      if (!readFloats(dirs[i] + "/fib_alphas", fib) || !readBytes(dirs[i] + "/fib_actions", fa) ||
          !readFloats(dirs[i] + "/pbvi_alphas", pbvi) || !readBytes(dirs[i] + "/pbvi_actions", pa))
        return false;
      setGoalAlphas((uint32_t)i + 1, fib, fa, pbvi, pa);
    }
    return true;
  }

  // saveDataCallback's model half (model_generation_cuda.cu:74-115), "%15.8f".
  bool saveModelDataToFile(const std::string& dir) {
    const size_t n = (size_t)map_height * map_width;
    std::vector<float> tp(n * 81), mp(n * 16), sr(n * 9);
    PP2D_CHECK(pp2d_pomdp_model_tables(pomdp_, tp.data(), mp.data(), sr.data()));
    return saveRows(dir + "/model_data_trans_prob", tp, 9) &&
           saveRows(dir + "/model_data_meas_prob", mp, 16) &&
           saveRows(dir + "/model_data_stage_reward", sr, 9);
  }

  // saveFibDataToFile / savePbviDataToFile (fast_informed_bound_cuda.cu:343-360,
  // point_based_value_iteration_cuda.cu:747-766): "%15.8f" rows, "%10u" actions.
  bool saveFibDataToFile(const std::string& dir) {
    return saveRows(dir + "/fib_alphas", fib_alphas, 9) &&
           saveBytes(dir + "/fib_actions", fib_actions);
  }
  bool savePbviDataToFile(const std::string& dir) {
    return saveRows(dir + "/pbvi_alphas", pbvi_alphas, (int)((size_t)map_height * map_width)) &&
           saveBytes(dir + "/pbvi_actions", pbvi_actions);
  }
  // saveDataCallback (src/pomdp/path_planning_2d.cu:259-273)
  bool saveDataCallback(const std::string& dir) {
    if (data_format == "binary") return saveDataBinary(dir);
    return saveModelDataToFile(dir) && saveFibDataToFile(dir) && savePbviDataToFile(dir);
  }

  // Lossless variant of the checkpoint (SURVEY.md section 8f row 3): one file,
  // raw little-endian float32 / uint8 arrays in the order of the seven text
  // files, so that a planner restarted from it plans with the bits it saved.
  struct BinaryHeader {
    char magic[8];                      // "PP2DCKP1"
    uint32_t height, width, belief_set_size, reserved;
  };
  bool saveDataBinary(const std::string& dir) {
    const size_t n = (size_t)map_height * map_width;
    std::vector<float> tp(n * 81), mp(n * 16), sr(n * 9);
    PP2D_CHECK(pp2d_pomdp_model_tables(pomdp_, tp.data(), mp.data(), sr.data()));
    FILE* f = std::fopen((dir + "/pp2d_data.bin").c_str(), "wb");
    if (!f) return false;
    BinaryHeader hd = {{'P', 'P', '2', 'D', 'C', 'K', 'P', '1'}, map_height, map_width,
                       belief_set_size, 0};
    bool ok = std::fwrite(&hd, sizeof(hd), 1, f) == 1;
    auto put = [&](const void* p, size_t bytes) {
      ok = ok && (bytes == 0 || std::fwrite(p, 1, bytes, f) == bytes);
    };
    put(tp.data(), tp.size() * 4); put(mp.data(), mp.size() * 4); put(sr.data(), sr.size() * 4);
    put(fib_alphas.data(), fib_alphas.size() * 4); put(fib_actions.data(), fib_actions.size());
    put(pbvi_alphas.data(), pbvi_alphas.size() * 4); put(pbvi_actions.data(), pbvi_actions.size());
    return std::fclose(f) == 0 && ok;
  }
  bool loadDataBinary(const std::string& dir) {
    FILE* f = std::fopen((dir + "/pp2d_data.bin").c_str(), "rb");
    if (!f) { std::fprintf(stderr, "cannot open %s/pp2d_data.bin\n", dir.c_str()); return false; }
    BinaryHeader hd;
    bool ok = std::fread(&hd, sizeof(hd), 1, f) == 1 &&
              std::memcmp(hd.magic, "PP2DCKP1", 8) == 0 && hd.height == map_height &&
              hd.width == map_width && hd.belief_set_size == belief_set_size;
    if (!ok) {
      std::fprintf(stderr, "Data dimension is not set properly\n");
      std::fclose(f);
      return false;
    }
    const size_t n = (size_t)map_height * map_width;
    std::vector<float> tp(n * 81), mp(n * 16), sr(n * 9);
    fib_alphas.resize(n * 9); fib_actions.resize(9);
    pbvi_alphas.resize((size_t)belief_set_size * n); pbvi_actions.resize(belief_set_size);
    auto get = [&](void* p, size_t bytes) {
      ok = ok && (bytes == 0 || std::fread(p, 1, bytes, f) == bytes);
    };
    get(tp.data(), tp.size() * 4); get(mp.data(), mp.size() * 4); get(sr.data(), sr.size() * 4);
    get(fib_alphas.data(), fib_alphas.size() * 4); get(fib_actions.data(), fib_actions.size());
    get(pbvi_alphas.data(), pbvi_alphas.size() * 4); get(pbvi_actions.data(), pbvi_actions.size());
    std::fclose(f);
    if (!ok) { std::fprintf(stderr, "Data dimension is not set properly\n"); return false; }
    PP2D_CHECK(pp2d_pomdp_set_model_tables(pomdp_, tp.data(), mp.data(), sr.data()));
    return true;
  }

  std::vector<float> initial_belief;
  uint32_t fib_sweeps = 0;
  const std::vector<float>& fibAlphas() const { return fib_alphas; }
  const std::vector<float>& pbviAlphas() const { return pbvi_alphas; }
  const std::vector<uint8_t>& pbviActions() const { return pbvi_actions; }
  float last_reward = 0.0f;
  pp2d_pomdp* handle() { return pomdp_; }

 private:
  bool loadParameters() override {          // src/pomdp/path_planning_2d.cu:168-184
    if (!getParam("map_path", map_path)) return false;
    if (!getParam("goal_x", goal[0])) return false;
    if (!getParam("goal_y", goal[1])) return false;
    if (!getParam("discount_factor", discount_factor)) return false;
    float res = 0.f;
    if (!getParam("map_resolution", res)) return false;
    map_resolution = res;
    if (!getParam("read_data_from_file", read_from_file)) return false;
    if (!getParam("max_search_tree_depth", max_search_tree_depth)) return false;
    if (!getParam("max_online_iteration", max_online_iteration)) return false;
    getParam("data_dir", data_dir);
    getParam("data_format", data_format);     // "text" (reference) | "binary" (lossless)
    int32_t n = 500;                        // belief_set_size, path_planning_2d.cu:122
    if (getParam("belief_set_size", n)) belief_set_size = (uint32_t)n;
    return true;
  }

  static bool readFloats(const std::string& path, std::vector<float>& v) {
    FILE* f = std::fopen(path.c_str(), "r");
    if (!f) { std::fprintf(stderr, "cannot open %s\n", path.c_str()); return false; }
    for (float& x : v)
      if (std::fscanf(f, "%f", &x) != 1) {
        std::fprintf(stderr, "Data dimension is not set properly\n");
        std::fclose(f);
        return false;
      }
    std::fclose(f);
    return true;
  }
  static bool readBytes(const std::string& path, std::vector<uint8_t>& v) {
    FILE* f = std::fopen(path.c_str(), "r");
    if (!f) { std::fprintf(stderr, "cannot open %s\n", path.c_str()); return false; }
    for (uint8_t& x : v) {
      unsigned u = 0;
      if (std::fscanf(f, "%u", &u) != 1) { std::fclose(f); return false; }
      x = (uint8_t)u;
    }
    std::fclose(f);
    return true;
  }
  static bool saveBytes(const std::string& path, const std::vector<uint8_t>& v) {
    FILE* f = std::fopen(path.c_str(), "w");
    if (!f) return false;
    for (uint8_t x : v) std::fprintf(f, "%10u\n", (unsigned)x);
    std::fclose(f);
    return true;
  }
  static bool saveRows(const std::string& path, const std::vector<float>& v, int per_row) {
    FILE* f = std::fopen(path.c_str(), "w");
    if (!f) return false;
    for (size_t i = 0; i < v.size(); ++i) {
      std::fprintf(f, "%15.8f", v[i]);
      if ((i + 1) % per_row == 0) std::fprintf(f, "\n");
    }
    std::fclose(f);
    return true;
  }
  // model_generation_cuda.cu:109-159: the three "%15.8f" tables, then upload.
  bool loadModelDataFromFile() {
    const size_t n = (size_t)map_height * map_width;
    std::vector<float> tp(n * 81), mp(n * 16), sr(n * 9);
    if (!readFloats(data_dir + "/model_data_trans_prob", tp) ||
        !readFloats(data_dir + "/model_data_meas_prob", mp) ||
        !readFloats(data_dir + "/model_data_stage_reward", sr))
      return false;
    PP2D_CHECK(pp2d_pomdp_set_model_tables(pomdp_, tp.data(), mp.data(), sr.data()));
    return true;
  }
  // fast_informed_bound_cuda.cu:361-394
  bool loadFibDataFromFile() {
    fib_alphas.resize((size_t)map_height * map_width * 9);
    fib_actions.resize(9);
    return readFloats(data_dir + "/fib_alphas", fib_alphas) &&
           readBytes(data_dir + "/fib_actions", fib_actions);
  }
  // point_based_value_iteration_cuda.cu:768-800
  bool loadPbviDataFromFile() {
    pbvi_alphas.resize((size_t)belief_set_size * map_height * map_width);
    pbvi_actions.resize(belief_set_size);
    return readFloats(data_dir + "/pbvi_alphas", pbvi_alphas) &&
           readBytes(data_dir + "/pbvi_actions", pbvi_actions);
  }

  pp2d_pomdp* pomdp_ = nullptr;
  SearchTree* search_tree = nullptr;
  bool read_from_file = true;
  int32_t max_search_tree_depth = 50, max_online_iteration = 15;
  uint32_t belief_set_size = 500;
  std::string data_dir = ".", data_format = "text";
  std::vector<float> fib_alphas, pbvi_alphas;
  std::vector<uint8_t> fib_actions, pbvi_actions;
};

}  // namespace path_planning_2d
