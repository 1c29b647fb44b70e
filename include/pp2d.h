/*
 * pp2d.h -- C ABI of the B200-native hot path of path_planning_2d.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has no
 * FFI: its host classes share C++-linkage symbols, global device pointers and
 * raw kernel launches with the .cu files.  Each entry point below names the
 * reference call sites it replaces (paths relative to
 * /root/reference/path_planning_2d/); INTEGRATION.md shows the mechanical
 * edit of the reference classes that binds them.
 *
 * Conventions kept from the reference:
 *   - the caller owns every host buffer; inputs are copied, never retained;
 *   - every call is synchronous on return (the reference synchronises after
 *     every launch: src/mdp/path_planning_2d.cu:231,236);
 *   - row-major cells, idx = y*width + x; map value 1 = occupied, 0 = free
 *     (src/mdp/path_planning_2d.cu:191-205);
 *   - 9 actions, action u moves by (u%3-1, u/3-1)
 *     (src/mdp/path_planning_2d_cuda.cu:83-88).
 * Errors: the reference prints and exit()s inside checkCudaErrors
 * (include/path_planning_2d/helper_cuda/helper_cuda.h:984-999).  A library
 * must not exit: every function returns PP2D_OK (0) or a negative code and
 * pp2d_last_error() returns the message; the reference-side shim keeps the
 * print-and-exit behaviour (INTEGRATION.md).
 *
 * There is no CPU fallback: every entry point needs a CUDA device of compute
 * capability 10.x and fails with PP2D_ERR_CUDA otherwise.
 */
#ifndef PP2D_H_
#define PP2D_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PP2D_OK 0
#define PP2D_ERR_INVALID (-1) /* bad argument (null, zero size, goal outside) */
#define PP2D_ERR_GOAL_OCCUPIED (-2) /* src/mdp/path_planning_2d.cu:84-88 */
#define PP2D_ERR_CUDA (-3)    /* CUDA runtime error, see pp2d_last_error() */
#define PP2D_ERR_STATE (-4)   /* call order violated */

/* Message of the last failure on the calling thread ("" if none). */
const char* pp2d_last_error(void);
/* ABI version of this library (bumped on any signature change). */
int pp2d_abi_version(void);
/* Number of CUDA kernels this library has launched in this process so far
 * (all handles).  bench.py reports the delta over its timed region. */
uint64_t pp2d_kernel_launches(void);

/* ------------------------------------------------------------------------
 * MDP value iteration (SURVEY.md rows A1-A8, W)
 * ------------------------------------------------------------------------ */
typedef struct pp2d_mdp pp2d_mdp;

/*
 * Replaces allocateDeviceMemory + map upload + cudaGenerateModelData
 * (src/mdp/path_planning_2d_cuda.cu:40-64,174-213;
 *  src/mdp/path_planning_2d.cu:84-106).
 * map: height*width bytes, 1 = occupied.  (goal_x, goal_y) must be a free
 * cell, otherwise PP2D_ERR_GOAL_OCCUPIED (the reference's initialize() fails
 * the same way).  J is initialised to 0 and the action grid to 0 exactly as
 * the reference's cudaMemset does.  The per-cell 360-byte tables of the
 * reference are never materialised: the model is a pure function of the 3x3
 * occupancy and is stored as a 2-byte code per cell.
 */
int pp2d_mdp_create(uint32_t height, uint32_t width, const uint8_t* map,
                    uint32_t goal_x, uint32_t goal_y, float gamma,
                    pp2d_mdp** out);

/*
 * Row-sharded variant for one-process-per-GPU runs (SURVEY.md section 8e).
 * The handle owns rows [row_begin, row_end) of a height x width grid; `map`
 * is still the whole grid (only rows row_begin-3 .. row_end+2 are read).
 * Ghost rows of J are exchanged by the caller between pp2d_mdp_sweeps calls
 * through the pointers of pp2d_mdp_halo (NCCL send/recv in
 * path_planning_2d_b200/distributed.py).
 */
int pp2d_mdp_create_shard(uint32_t height, uint32_t width, const uint8_t* map,
                          uint32_t goal_x, uint32_t goal_y, float gamma,
                          uint32_t row_begin, uint32_t row_end,
                          pp2d_mdp** out);

/*
 * Single-process multi-GPU variant: what MdpPathPlanning2d::initialize (ONE ROS
 * process, src/mdp/path_planning_2d.cu:72-140) can bind to reach 2, 4 or 8
 * GPUs.  The grid is cut into `ngpus` contiguous row blocks; shard i lives on
 * CUDA device devices[i] (NULL: devices 0 .. ngpus-1) and all of them are
 * driven from the calling host thread on per-device streams.  The handle
 * behaves like the one pp2d_mdp_create returns: pp2d_mdp_sweeps(_ex),
 * pp2d_mdp_residual, pp2d_mdp_solve, pp2d_mdp_download (whole grid),
 * pp2d_mdp_reset, pp2d_mdp_plan(_batch), pp2d_mdp_waypoints,
 * pp2d_mdp_sweep_count, pp2d_mdp_p2p_status and pp2d_mdp_destroy work on it,
 * and the results are bit-identical to the single-GPU solve (Jacobi sweeps do
 * not depend on the partition).  Between neighbouring shards on different
 * devices with peer access, ghost rows are written by the fused sweep kernel
 * straight into the neighbour's memory (NVLink stores + device flags, no
 * host involvement between launches); otherwise -- including several shards
 * on one device, e.g. devices = {0, 0} -- they are copied between
 * event-ordered streams after every launch.  The current device of the
 * calling thread is preserved by every call.
 */
int pp2d_mdp_create_multi(uint32_t height, uint32_t width, const uint8_t* map,
                          uint32_t goal_x, uint32_t goal_y, float gamma, uint32_t ngpus,
                          const int* devices, pp2d_mdp** out);
/* Number of row shards of a handle (1 for pp2d_mdp_create / _create_shard);
 * peer_to_peer (may be NULL): 1 when the ghost rows of a multi-GPU handle travel
 * inside the fused kernel. */
int pp2d_mdp_device_count(const pp2d_mdp* h, int* peer_to_peer);

/*
 * Start over on the same handle with a new map (same height/width/rows) and
 * goal: J = 0, action = 0, sweep count 0, codes rebuilt.  Same checks as
 * pp2d_mdp_create; lets a long-running planner re-solve without paying the
 * device allocations again (the reference allocates once per process,
 * src/mdp/path_planning_2d.cu:91).
 */
int pp2d_mdp_reset(pp2d_mdp* h, const uint8_t* map, uint32_t goal_x,
                   uint32_t goal_y);

/*
 * Upload the map of the NEXT pp2d_mdp_reset ahead of time: the rows this handle
 * needs start travelling to a second device buffer on a separate upload stream
 * and the call returns at once, so the copy overlaps the solve that is still
 * running (page-locked host memory is needed for that).  A following
 * pp2d_mdp_reset(h, map, ...) with the SAME pointer uses the staged rows (it
 * waits for them in stream order, skips its own copy and does not block the
 * host); with any other pointer the staged rows are dropped.  The host buffer
 * must stay unchanged until that reset has been called.  No counterpart in the
 * reference (one map per process, src/mdp/path_planning_2d.cu:94); for a
 * planner that re-plans on a stream of maps.
 */
int pp2d_mdp_stage_map(pp2d_mdp* h, const uint8_t* map);

/*
 * Re-plan on a changed map (same height/width/rows) and/or goal from the
 * current solution instead of from J = 0.  Same checks and error codes as
 * pp2d_mdp_reset; on an error the handle is unchanged.  Afterwards:
 *   - J' = what pp2d_mdp_download returned just before the call, except that
 *     every cell occupied in the new map gets trapped(n) (the value every
 *     occupied cell has after n sweeps, n = pp2d_mdp_sweep_count) and the new
 *     goal gets 0.  Everything else keeps its value, including newly freed
 *     cells (they keep the trapped(n) they were reported with) and the old goal
 *     (it stays 0).
 *   - the model (codes) is that of the new map and goal;
 *   - pp2d_mdp_sweep_count is unchanged and keeps counting;
 *   - the next pp2d_mdp_residual measures the change since this call;
 *   - the action grid is left as it was: it belongs to the old map until the
 *     next sweep that writes actions, which rewrites all of it.
 * So "update, then k sweeps" equals k of the reference's sweeps on the new
 * map started from J', and pp2d_mdp_solve after it runs the reference's
 * stopping rule from J'.  Only the units the change reaches are recomputed by
 * the following fused sweeps while the rest of the grid stays at its fixed
 * point (DESIGN.md section 4).  A map staged with pp2d_mdp_stage_map is used
 * when the same pointer is passed (the call then does not block the host);
 * otherwise the call returns once the map has been copied.  Works on every
 * handle kind (a shard applies the rule to its own and its ghost rows).
 * After pp2d_mdp_policy_iteration: PP2D_ERR_STATE.
 */
int pp2d_mdp_update_map(pp2d_mdp* h, const uint8_t* map, uint32_t goal_x,
                        uint32_t goal_y);


/* Replaces freeDeviceMemory (src/mdp/path_planning_2d_cuda.cu:66-74). */
void pp2d_mdp_destroy(pp2d_mdp* h);

/* Run the library's kernels on `stream` (a cudaStream_t; NULL = default
 * stream) from now on.  Calls still synchronise that stream before
 * returning unless pp2d_mdp_set_async(h, 1) was called. */
int pp2d_mdp_set_stream(pp2d_mdp* h, void* stream);
/* async != 0: pp2d_mdp_sweeps / pp2d_mdp_residual_begin only enqueue work
 * (used by the multi-GPU driver to overlap with NCCL on the same stream). */
int pp2d_mdp_set_async(pp2d_mdp* h, int async);

/*
 * n Jacobi Bellman backups of every owned cell; replaces n launches of
 * cudaOneStepValueIteration (src/mdp/path_planning_2d_cuda.cu:215-264,
 * call sites src/mdp/path_planning_2d.cu:226-237).  After the call J and the
 * greedy action grid are exactly those the reference holds after the same n
 * launches (the action grid is produced by the last backup only, which is
 * all that is observable).  For a shard, n must not exceed the halo depth
 * the caller refreshed (pp2d_mdp_halo: depth 2), i.e. n <= 2 between
 * exchanges; for an unsharded handle any n.
 */
int pp2d_mdp_sweeps(pp2d_mdp* h, uint32_t n);
/* Same, but with want_action == 0 the greedy action grid is left untouched
 * (all n backups are value-only; the multi-GPU driver uses this between
 * ghost-row exchanges and asks for the action only on the last sweep). */
int pp2d_mdp_sweeps_ex(pp2d_mdp* h, uint32_t n, int want_action);

/*
 * Inf-norm of the change of J since the previous call (or since creation),
 * max_s |J_now(s) - J_then(s)| over the owned cells, as the reference
 * computes it on the host every 100 sweeps
 * (src/mdp/path_planning_2d.cu:243-251).
 */
int pp2d_mdp_residual(pp2d_mdp* h, float* inf_norm);

/*
 * The reference's valueIteration() loop (src/mdp/path_planning_2d.cu:207-269):
 * batches of 100 sweeps until the residual of a batch is
 * <= 5.0/(1.0-gamma)*1e-3 (double arithmetic on the float gamma).
 * sweeps_out receives the total number of sweeps; residuals (optional,
 * capacity max_residuals) one inf-norm per batch.  Unsharded handles only.
 */
int pp2d_mdp_solve(pp2d_mdp* h, uint32_t* sweeps_out, double* residuals,
                   uint32_t max_residuals);

/* policyIteration() (src/mdp/path_planning_2d.cu:271-357; dead code in the
 * reference, its call is commented out at :115-116) on a freshly created or
 * reset, unsharded handle: rounds of 50 evaluation sweeps
 * (cudaOneStepPolicyEvaluation, path_planning_2d_cuda.cu:266-306), the
 * inf-norm of the change of J over the round, one policy improvement
 * (cudaPolicyImprovment, :308-355), until the inf-norm is <=
 * 5/(1-gamma)*1e-3.  residuals / changed (optional, `capacity` entries each)
 * receive one entry per round, rounds beyond `capacity` are not recorded;
 * max_rounds = 0 runs to the stopping rule. */
int pp2d_mdp_policy_iteration(pp2d_mdp* h, uint32_t* evaluation_sweeps, double* residuals,
                              uint32_t* changed, uint32_t capacity, uint32_t max_rounds);

/*
 * Replaces the two result cudaMemcpy calls
 * (src/mdp/path_planning_2d.cu:118-126).  cost: rows*width floats,
 * action: rows*width bytes (rows = owned rows); either may be NULL.
 */
int pp2d_mdp_download(pp2d_mdp* h, float* cost, uint8_t* action);
/*
 * The same download in two halves, for a planner that re-solves while the
 * previous solution is still on its way to the host: _begin snapshots J (cost
 * of occupied cells filled in) and the action grid into device staging buffers
 * in stream order and starts the device-to-host copies on a separate copy
 * stream, then returns; the handle may be swept or reset immediately.  _wait
 * blocks until the host buffers are complete (page-locked host buffers are
 * needed for the copies to overlap device work).  A second _begin before the
 * _wait of the first waits for it on the device.
 */
int pp2d_mdp_download_begin(pp2d_mdp* h, float* cost, uint8_t* action);
int pp2d_mdp_download_wait(pp2d_mdp* h);

/*
 * MdpPathPlanning2d::beliefCallback (src/mdp/path_planning_2d.cu:168-189):
 * the action at the first strict maximum of `belief` (height*width floats,
 * host memory).  Unsharded handles only.
 */
int pp2d_mdp_plan(pp2d_mdp* h, const float* belief, uint8_t* action);
/* Batched form: n_beliefs beliefs laid out [n][height*width]. */
int pp2d_mdp_plan_batch(pp2d_mdp* h, const float* beliefs, uint32_t n_beliefs,
                        uint8_t* actions);

/*
 * Row W of SURVEY.md section 8a: greedy rollout of the action grid from
 * (start_x, start_y): follow (u%3-1, u/3-1) until action 4 (stay), the map
 * border, or max_len cells.  Writes cell indices y*width+x (start included)
 * and their count.  Unsharded handles only.
 */
int pp2d_mdp_waypoints(pp2d_mdp* h, uint32_t start_x, uint32_t start_y,
                       uint32_t* cells, uint32_t max_len, uint32_t* n_out);

/* Number of sweeps applied so far. */
uint32_t pp2d_mdp_sweep_count(const pp2d_mdp* h);

/*
 * Work of the fused two-sweep row-block launches so far (cumulative, counted
 * on the device; summed over the devices of a multi-GPU handle):
 * out[0] = units run, out[1] = units launched.  A unit whose 3x3 unit
 * neighbourhood did not change in the previous launch is skipped: its output
 * is already in the buffer the launch writes (DESIGN.md section 4).
 * PP2D_MDP_SKIP=0 at handle creation turns skipping off (then out[0] ==
 * out[1]).  Measurement only, no reference counterpart.
 */
int pp2d_mdp_work_counters(pp2d_mdp* h, uint64_t out[2]);

/*
 * Ghost-row exchange for shards.  depth = 2 rows.  After any
 * pp2d_mdp_sweeps call the caller copies `bytes` bytes
 *   from this rank's send_top  to the upper neighbour's recv_bottom,
 *   from this rank's send_bottom to the lower neighbour's recv_top
 * (device pointers into the CURRENT J buffer; they change after every
 * pp2d_mdp_sweeps call, so query them again).  Pointers for a missing
 * neighbour (first/last shard) are still valid memory and may be ignored.
 */
typedef struct pp2d_halo {
  void* send_top;
  void* send_bottom;
  void* recv_top;
  void* recv_bottom;
  size_t bytes;
} pp2d_halo;
int pp2d_mdp_halo(pp2d_mdp* h, pp2d_halo* out);

/*
 * Peer-to-peer ghost rows over NVLink (same node, one process per GPU).
 * Each rank exports a descriptor (CUDA IPC handles of its two J planes and
 * its flag block), the ranks swap descriptors (any transport; distributed.py
 * uses all_gather_object) and connect to their upper / lower neighbour (NULL
 * where there is none) before the first sweep.  From then on every fused
 * 2-sweep launch (pp2d_mdp_sweeps_ex(h, 2, 0)) writes its first / last two
 * rows straight into the neighbours' ghost rows and synchronises with them
 * through flags in device memory: no exchange call, no collective.  Single
 * sweeps and arg-min sweeps still need the pp2d_mdp_halo exchange, preceded by
 * a stream-ordered cross-rank barrier (any NCCL collective).
 */
#define PP2D_IPC_DESC_BYTES 256
int pp2d_mdp_ipc_export(pp2d_mdp* h, void* desc /* PP2D_IPC_DESC_BYTES */);
int pp2d_mdp_ipc_connect(pp2d_mdp* h, const void* up_desc, const void* down_desc);
/* timed_out != 0: a flag wait gave up after PP2D_P2P_SPIN_LIMIT polls (default
 * 2^24, a few seconds: the neighbour is missing or did not run the same
 * launches); J of this shard is invalid from then on.  The failure is also
 * reported without this call: the residual of the shard becomes +inf
 * (pp2d_mdp_residual fails with PP2D_ERR_STATE, a caller that reduces
 * pp2d_mdp_residual_device itself sees inf) and pp2d_mdp_download fails with
 * PP2D_ERR_STATE.  pp2d_mdp_reset clears the condition. */
int pp2d_mdp_p2p_status(pp2d_mdp* h, int* timed_out);

/* Device-side residual for shards: enqueue the reduction, then read it. */
int pp2d_mdp_residual_device(pp2d_mdp* h, void** dev_float_out);

/* ------------------------------------------------------------------------
 * MDP batches: many goals or maps of one size solved together
 * ------------------------------------------------------------------------ */
typedef struct pp2d_mdp_batch pp2d_mdp_batch;

/*
 * `count` independent value-iteration instances of one height x width size on
 * the current device: a fleet with one goal per robot, cost-to-go fields for
 * every docking station of a map, a sweep over maps.  No counterpart in the
 * reference (one goal per process).  The instances are stacked into one tall
 * grid with an occupied separator row between neighbours (DESIGN.md section
 * 4, "Batches"), so every instance computes bit for bit what pp2d_mdp_create on its map
 * and goal computes, while all of them share the launches.
 * maps: `count` maps of height*width bytes, `map_stride` bytes apart;
 * map_stride == 0: one map shared by all instances (only goals differ).
 * goals_xy: uint32_t[count][2], (x, y) per instance.  The checks of
 * pp2d_mdp_create apply per instance; an occupied goal gives
 * PP2D_ERR_GOAL_OCCUPIED with the instance index in the message.
 * PP2D_ERR_INVALID for count == 0, map_stride below height*width, or a
 * stacked grid (count*(height+1)-1 rows) too large for int row and element
 * indices.  J = 0, actions = 0, sweep count 0.  Not sharded, one device.
 */
int pp2d_mdp_batch_create(uint32_t height, uint32_t width, uint32_t count, const uint8_t* maps,
                          size_t map_stride, const uint32_t* goals_xy, float gamma,
                          pp2d_mdp_batch** out);
/* New maps and goals (same size and count) on the same allocations, as
 * pp2d_mdp_reset; map_stride may differ from the one given at creation (a
 * shared map may become one map per instance and back).  On an error the
 * handle is unchanged. */
int pp2d_mdp_batch_reset(pp2d_mdp_batch* h, const uint8_t* maps, size_t map_stride,
                         const uint32_t* goals_xy);
void pp2d_mdp_batch_destroy(pp2d_mdp_batch* h);
/* As pp2d_mdp_set_stream; calls still synchronise before they return. */
int pp2d_mdp_batch_set_stream(pp2d_mdp_batch* h, void* stream);

/* n sweeps of every instance, as pp2d_mdp_sweeps (the action grids come
 * from the last one).  PP2D_ERR_STATE after pp2d_mdp_batch_solve until
 * pp2d_mdp_batch_reset. */
int pp2d_mdp_batch_sweeps(pp2d_mdp_batch* h, uint32_t n);
/* out[count]: per instance, what pp2d_mdp_residual returns for it: the
 * inf-norm of the change since the previous call, with the occupied-cell
 * floor when its own map has an occupied cell.  PP2D_ERR_STATE after
 * pp2d_mdp_batch_solve. */
int pp2d_mdp_batch_residual(pp2d_mdp_batch* h, float* out);
/*
 * pp2d_mdp_solve per instance: batches of 100 sweeps, instance k stops after
 * its first batch whose residual is <= 5/(1-gamma)*1e-3.  sweeps_out[count]
 * (optional) and residuals (optional, [count][max_residuals], entries past an
 * instance's last batch are not written) are exactly what pp2d_mdp_solve
 * returns for each instance alone.  Returns once every instance has stopped;
 * each then holds its J and actions at its own stopping point.  A stopped
 * instance is frozen: its results are kept aside and its rows stop costing
 * work in the launches that the others still need.  Afterwards sweeps,
 * residual and solve return PP2D_ERR_STATE until pp2d_mdp_batch_reset.
 * After pp2d_mdp_batch_update, solve runs the instances that are active
 * (never frozen, or re-activated by the update); sweeps_out[k] and residual
 * row k are written for those only, and solve returns PP2D_ERR_STATE when
 * none is active.  sweeps and residual return PP2D_ERR_STATE while any
 * instance is frozen.
 */
int pp2d_mdp_batch_solve(pp2d_mdp_batch* h, uint32_t* sweeps_out, double* residuals,
                         uint32_t max_residuals);
/*
 * pp2d_mdp_update_map on the instances instances[0 .. n) (distinct indices):
 * instance instances[i] gets the map at maps + i*map_stride (map_stride == 0:
 * one map for all n) and the goal (goals_xy[2i], goals_xy[2i+1]), and keeps
 * its solution.  With n_k its sweep count (pp2d_mdp_batch_sweep_counts), J'
 * is its download just before the call with every occupied cell of the new
 * map at trapped(n_k) and the new goal at 0.  n_k carries on, the next
 * residual of the instance measures the change since the update, and its
 * action grid (plan, way-points) stays as it was until its next sweep.  An
 * instance frozen by a solve becomes active again from its result.  Instances
 * not listed are left bit for bit as they were; frozen ones stay frozen.
 * PP2D_ERR_INVALID for NULL pointers, an index >= count or listed twice, a
 * non-zero map_stride below height*width or a goal outside the map;
 * PP2D_ERR_GOAL_OCCUPIED for an occupied goal (messages name the instance).
 * On an error the handle is unchanged; n == 0 does nothing.
 */
int pp2d_mdp_batch_update(pp2d_mdp_batch* h, const uint32_t* instances, uint32_t n,
                          const uint8_t* maps, size_t map_stride, const uint32_t* goals_xy);
/* Results of instances [first, first+n): cost [n][height][width] floats
 * (occupied cells filled in as by pp2d_mdp_download), action
 * [n][height][width] bytes; either may be NULL. */
int pp2d_mdp_batch_download(pp2d_mdp_batch* h, uint32_t first, uint32_t n, float* cost,
                            uint8_t* action);
/* pp2d_mdp_plan_batch where belief i ([n][height*width] floats) reads the
 * action grid of instance instance[i]. */
int pp2d_mdp_batch_plan(pp2d_mdp_batch* h, const uint32_t* instance, const float* beliefs,
                        uint32_t n, uint8_t* actions);
/* pp2d_mdp_waypoints on instance k. */
int pp2d_mdp_batch_waypoints(pp2d_mdp_batch* h, uint32_t k, uint32_t start_x,
                             uint32_t start_y, uint32_t* cells, uint32_t max_len,
                             uint32_t* n_out);
/* out[count]: sweeps applied to each instance (a frozen instance keeps the
 * count it stopped at). */
int pp2d_mdp_batch_sweep_counts(const pp2d_mdp_batch* h, uint32_t* out);
/* As pp2d_mdp_work_counters, over the launches of the whole batch. */
int pp2d_mdp_batch_work_counters(pp2d_mdp_batch* h, uint64_t out[2]);

/* ------------------------------------------------------------------------
 * POMDP model, belief propagation, bounds and QV-Tree Search
 * (SURVEY.md rows B1-B10)
 * ------------------------------------------------------------------------ */
typedef struct pp2d_pomdp pp2d_pomdp;
typedef struct pp2d_tree pp2d_tree;

/*
 * Replaces allocateDeviceMemoryOfModel + generateModelData
 * (src/pomdp/model_generation_cuda.cu:41-59, 349-375; call site
 * src/pomdp/path_planning_2d.cu:109-112): uploads the map and builds
 * trans_prob f32[HW][9][9], meas_prob f32[HW][16], stage_reward f32[HW][9] on
 * the device in the reference's layout.  Goal on an occupied cell ->
 * PP2D_ERR_GOAL_OCCUPIED (src/pomdp/path_planning_2d.cu:93-97).
 */
int pp2d_pomdp_create(uint32_t height, uint32_t width, const uint8_t* map,
                      uint32_t goal_x, uint32_t goal_y, float gamma,
                      pp2d_pomdp** out);
/* Replaces freeDeviceMemoryOfModel / ...OfFIB / ...OfPBVI. */
void pp2d_pomdp_destroy(pp2d_pomdp* h);
/* The host mirrors host_trans_prob / host_meas_prob / host_stage_reward
 * (model_generation_cuda.cu:366-371); any pointer may be NULL. */
int pp2d_pomdp_model_tables(pp2d_pomdp* h, float* trans_prob, float* meas_prob,
                            float* stage_reward);
/*
 * Replaces the upload half of loadModelDataFromFile
 * (src/pomdp/model_generation_cuda.cu:109-159, the three cudaMemcpy at
 * :150-156; call site src/pomdp/path_planning_2d.cu:131): the reference's
 * DEFAULT launch (read_data_from_file=true) does not generate the model, it
 * reads the "%15.8f" text tables back and uploads those -- rounded to 8
 * decimals, so e.g. 0.02^4 becomes 0.00000016.  The tables replace the ones
 * pp2d_pomdp_create generated (layouts as in pp2d_pomdp_model_tables); any
 * pointer may be NULL (that table is kept).  Parsing the files stays on the
 * host side (include/pp2d/planners.hpp: loadModelDataFromFile).  Call it
 * before any search tree exists on the handle (PP2D_ERR_STATE otherwise), as
 * the reference loads its tables once in initialize().
 */
int pp2d_pomdp_set_model_tables(pp2d_pomdp* h, const float* trans_prob,
                                const float* meas_prob, const float* stage_reward);
/* The 100 curand_uniform values cudaForwardSampling consumes for its 50
 * samples (search_tree_cuda.cu:84-92,117,134; XORWOW, seed 1234, subsequence
 * = sample index, re-initialised per call, hence constant). */
int pp2d_pomdp_sampling_uniforms(pp2d_pomdp* h, float* out100);
/*
 * The alpha vectors the tree reads: replaces host_fib_alphas f32[HW][9] +
 * host_fib_actions u8[9] (fast_informed_bound_cuda.cu:36-52) and
 * host_pbvi_alphas f32[n][HW] + host_pbvi_actions u8[n]
 * (point_based_value_iteration_cuda.cu:44-58), however they were produced
 * (solvers or loadFibDataFromFile / loadPbviDataFromFile).  fib_actions /
 * pbvi_actions may be NULL (identity / zeros).
 */
int pp2d_pomdp_set_alphas(pp2d_pomdp* h, const float* fib_alphas,
                          const uint8_t* fib_actions, const float* pbvi_alphas,
                          const uint8_t* pbvi_actions, uint32_t n_pbvi);
/*
 * fastInformedBound (fast_informed_bound_cuda.cu:97-276): value iteration on
 * the 9 FIB alpha vectors, 10 sweeps per convergence check, stop when the
 * inf-norm of the change is <= 0.01 (or after max_sweeps > 0; a cap is
 * rounded up to whole 10-sweep checks).  max_sweeps = 0 needs |gamma| < 1:
 * for a NaN gamma or |gamma| >= 1 that rule is not reached in useful time, and
 * the call returns PP2D_ERR_INVALID before any device work.  alphas:
 * f32[HW][9] (host), actions: u8[9] = identity (may be NULL).  The result is
 * what pp2d_pomdp_set_alphas takes as fib_alphas.
 */
int pp2d_pomdp_solve_fib(pp2d_pomdp* h, float* alphas, uint8_t* actions,
                         uint32_t* sweeps_out, uint32_t max_sweeps);
/* Size the device belief pool for n_beliefs resident beliefs (optional). */
/* ---- offline PBVI solver (point_based_value_iteration_cuda.cu) ----------- */
/* generateBeliefSet (pbvi:165-293): expands {initial_belief} to n beliefs
 * (rand() stream seeded with rand_seed, 1 = a fresh process; 0 is taken as 1).
 * belief_set: [n][HW] host, row-major, in set order. */
int pp2d_pomdp_generate_belief_set(pp2d_pomdp* h, const float* initial_belief,
                                   uint32_t n, uint32_t rand_seed, float* belief_set);
/* backupAlphaVectors (pbvi:344-641) from alpha = 0: `iterations` point-based
 * backups of all n alpha vectors (0 = the reference's count,
 * ceil(log(1e-3/5)/log(gamma)), pbvi:427-431; defined only for 0 < gamma < 1,
 * PP2D_ERR_INVALID otherwise).  alphas [n][HW], actions [n]. */
int pp2d_pomdp_backup_alphas(pp2d_pomdp* h, const float* belief_set, uint32_t n,
                             uint32_t iterations, float* alphas, uint8_t* actions);
/* pointBasedValueIteration (pbvi:643-676): both steps without the round trip
 * through the host; belief_set (optional) and alphas are [n][HW]. */
int pp2d_pomdp_solve_pbvi(pp2d_pomdp* h, const float* initial_belief, uint32_t n,
                          uint32_t rand_seed, uint32_t iterations, float* belief_set,
                          float* alphas, uint8_t* actions);

int pp2d_pomdp_reserve(pp2d_pomdp* h, uint32_t n_beliefs);
/* The cells probability mass can enter under the current transition table
 * (some P(s, u, s') != 0 with s != s'); for the generated model: the free cells
 * that are not walled in.  A belief that is +0 on all other cells stays +0
 * there through every Bayes update, and the sequential inner products of the
 * QV-tree path (evaluateFibCpu / evaluatePbviCpu, the reward dot, the
 * normalisation sum) skip those cells bit-exactly; beliefs that are not (checked
 * when a start belief is uploaded) take the dense products.  mask: HW bytes,
 * 1 = live (may be NULL); count: number of live cells (may be NULL). */
int pp2d_pomdp_live_cells(pp2d_pomdp* h, uint8_t* mask, uint32_t* count);
/* Work done on this handle so far (cumulative): out[0] = V nodes created,
 * out[1] = Bayes updates, out[2] = belief x inner-row products of the bound
 * evaluations (each one is `ncol` separately rounded multiply-adds; the
 * launches of pp2d_pomdp_plan_batch walk per tile only the rows on which some
 * belief of the tile is non-zero, so this is what a FLOP count must use).
 * Measurement only, no reference counterpart. */
int pp2d_pomdp_work_counters(pp2d_pomdp* h, uint64_t out[3]);
/* Host threads used for the per-tree work of pp2d_pomdp_plan_batch (random
 * draws, child lists, tree bookkeeping; the trees of a batch are independent).
 * 0 = default: PP2D_HOST_THREADS, else min(8, CPUs of the process /
 * LOCAL_WORLD_SIZE).  The reference is single-threaded (ros::spin). */
void pp2d_set_host_threads(int n);
/*
 * Batched cudaBayesBeliefUpdate (point_based_value_iteration_cuda.cu:88-133;
 * call sites search_tree_cuda.cu:217, 601): out[i] = update(in[i], actions[i],
 * observations[i]), beliefs laid out [n][HW] in host memory.  normalize != 0
 * also applies the host normalisation of search_tree_cuda.cu:226-229 and
 * returns the pre-normalisation sums (may be NULL).
 */
int pp2d_pomdp_bayes_update(pp2d_pomdp* h, const float* beliefs_in, uint32_t n,
                            const uint8_t* actions, const uint8_t* observations,
                            int normalize, float* beliefs_out, float* sums);
/*
 * Batched evaluateFibCpu / evaluatePbviCpu
 * (fast_informed_bound_cuda.cu:278-297,
 * point_based_value_iteration_cuda.cu:678-699): upper = max_a <b, fib_a>,
 * lower = max_i <b, pbvi_i> and the action attached to the maximiser, same
 * summation order and roundings as the reference.  The maximiser is the one
 * std::max_element picks, also with non-finite alphas or beliefs: index 0 if
 * its value is NaN, else the first maximum of the values that are not NaN
 * (ties, +0 and -0 included, go to the smaller index).  Outputs may be NULL.
 */
int pp2d_pomdp_evaluate(pp2d_pomdp* h, const float* beliefs, uint32_t n,
                        float* upper, uint8_t* upper_action, float* lower,
                        uint8_t* lower_action);
/*
 * n independent PomdpPathPlanning2d::beliefCallback first calls
 * (src/pomdp/path_planning_2d.cu:199-241): per belief a fresh SearchTree,
 * up to max_iter expansions while depth < max_depth, then the action with the
 * largest upper bound and that bound.  Every query uses its own rand()
 * stream seeded like a fresh process (the planner never calls srand()).
 * stats (optional): 4 values per query {V nodes, Q nodes, depth, expansions}.
 */
int pp2d_pomdp_plan_batch(pp2d_pomdp* h, const float* beliefs, uint32_t n,
                          uint32_t max_depth, uint32_t max_iter,
                          uint8_t* actions, float* values, uint32_t* stats);

/* SearchTree (include/path_planning_2d/search_tree.h:130-165). */
int pp2d_tree_create(pp2d_pomdp* h, const float* belief, pp2d_tree** out);
void pp2d_tree_destroy(pp2d_tree* t);
int pp2d_tree_expand(pp2d_tree* t);                       /* expand() */
uint32_t pp2d_tree_depth(const pp2d_tree* t);             /* getDepth() */
int pp2d_tree_best_action(const pp2d_tree* t, uint8_t* action, float* value);
int pp2d_tree_update(pp2d_tree* t, uint8_t action, uint8_t observation);
int pp2d_tree_root_bounds(const pp2d_tree* t, float* upper, float* lower);
/* beliefCallback's loop + getOptimalAction on an existing tree.  Its
 * iteration counter is a uint8_t as in the reference, so max_iter > 255 runs
 * until the depth limit or a tree without a node to expand
 * (pp2d_pomdp_plan_batch and pp2d_tree_batch_plan clamp max_iter to 255). */
int pp2d_tree_plan(pp2d_tree* t, uint32_t max_depth, uint32_t max_iter,
                   uint8_t* action, float* value);
/* SearchTree::print (search_tree_cuda.cu:288-309, 452-473, 628-633) into a
 * buffer instead of stdout: pre-order walk from the root, 9 floats per node =
 * kind (0 = V node, 1 = Q node), observation | action, weight | reward,
 * upper bound, lower bound, heuristic, depth, number of children, pre-order
 * id of vnode_to_expand (-1 = nullptr).  Writes at most cap_nodes nodes,
 * returns the number of nodes in the tree (negative on error). */
int64_t pp2d_tree_dump(const pp2d_tree* t, float* out, uint64_t cap_nodes);

/*
 * Persistent tree batches: n SearchTrees on one planner handle that live
 * across belief callbacks (one per robot of a fleet) and are updated and
 * planned together.  Tree k behaves bit for bit like a pp2d_tree created from
 * beliefs[k] and fed the same calls: its own rand() stream, seeded like a
 * fresh process at creation and kept through updates, its own expansion count.
 * The trees' beliefs stay resident in the handle's belief pool until the
 * batch is destroyed (pp2d_pomdp_set_model_tables refuses meanwhile).
 *
 * create: pp2d_tree_create for every belief ([n][HW], host), one upload and
 * one bounds launch for all roots.
 * update: pp2d_tree_update(actions[i], observations[i]) on tree trees[i]; the
 * new roots that need a Bayes update share one set of launches.  Every listed
 * tree is checked before any changes: NULL pointers, an index >= n, an index
 * listed twice, an action >= 9 or an observation >= 16 give PP2D_ERR_INVALID,
 * an unexpanded root PP2D_ERR_STATE (messages name the tree).  Unlisted trees
 * are untouched.
 * plan: pp2d_tree_plan on every listed tree, the trees' expansion rounds
 * batched as in pp2d_pomdp_plan_batch (max_iter clamped to 255).  actions,
 * values (may be NULL) and stats (may be NULL; [n][4] = {V nodes, Q nodes,
 * root depth, expansions since creation}) are indexed like `trees`.  Results
 * do not depend on which other trees a call lists or on their order.
 * dump: pp2d_tree_dump of tree k (negative for a bad k).
 */
typedef struct pp2d_tree_batch pp2d_tree_batch;
int pp2d_tree_batch_create(pp2d_pomdp* h, const float* beliefs, uint32_t n,
                           pp2d_tree_batch** out);
void pp2d_tree_batch_destroy(pp2d_tree_batch* b);
int pp2d_tree_batch_update(pp2d_tree_batch* b, const uint32_t* trees, uint32_t n,
                           const uint8_t* actions, const uint8_t* observations);
int pp2d_tree_batch_plan(pp2d_tree_batch* b, const uint32_t* trees, uint32_t n,
                         uint32_t max_depth, uint32_t max_iter, uint8_t* actions, float* values,
                         uint32_t* stats);
int64_t pp2d_tree_batch_dump(const pp2d_tree_batch* b, uint32_t k, float* out,
                             uint64_t cap_nodes);

/*
 * Goal sets (DESIGN.md section 7e): one planner handle for many goals of one
 * map.  The goal enters the model only through the stage reward (0 instead of
 * -2 for staying on the goal cell); the transition and likelihood tables, the
 * live cells and the belief pool are shared.  Goal 0 is the goal the handle
 * was created with: its reward table is the one pp2d_pomdp_model_tables
 * returns and pp2d_pomdp_set_model_tables replaces, its bounds the ones
 * pp2d_pomdp_set_alphas sets, and every entry point without a goal argument
 * works on goal 0 alone.  A tree with goal g behaves bit for bit like a tree on
 * a handle created with goal g, with the same tables and goal g's alpha
 * vectors, fed the same calls.
 *
 * set_goals: goals_xy [n][2] = (x, y) replace goals 1..n (n = 0 removes them;
 * the new goals have no alpha vectors).  stage_rewards NULL: each goal's table
 * is generated by the model rule from the handle's map (the table
 * pp2d_pomdp_model_tables returns on a handle created with that goal);
 * otherwise stage_rewards [n][HW][9] is uploaded as given (tables read back
 * from text files differ in their bits from generated ones).  A goal outside
 * the map gives PP2D_ERR_INVALID, an occupied one PP2D_ERR_GOAL_OCCUPIED (the
 * message names the goal index); while any belief is resident PP2D_ERR_STATE,
 * as pp2d_pomdp_set_model_tables.  A refused call changes nothing.
 * goals: count = goals in the set, goal 0 included; goals_xy [count][2] (each
 * may be NULL).  goal_reward: goal g's stage reward table [HW][9].
 * set_goal_alphas: pp2d_pomdp_set_alphas for goal g (g = 0: the same call).
 * All goals of a handle use one PBVI count: a call that would give a goal
 * another count than a goal already holding alpha vectors is refused with
 * PP2D_ERR_INVALID (pp2d_pomdp_set_alphas too).  fib_actions / pbvi_actions of
 * goals >= 1 are not kept: only pp2d_pomdp_evaluate reads actions, on goal 0.
 * tree_batch_create_goals: pp2d_tree_batch_create, tree k planning to goal
 * goals[k] (goals NULL: goal 0 for every tree, = pp2d_tree_batch_create).  A
 * goal index above the set gives PP2D_ERR_INVALID, a goal without alpha
 * vectors PP2D_ERR_STATE (messages name the tree).  The other pp2d_tree_batch_*
 * calls work on such batches unchanged.
 * padding_counters: of the work out[2] of pp2d_pomdp_work_counters, what went
 * to the padding of goal segments: out[0] = padded entries evaluated, out[1] =
 * their belief x inner-row products.  Measurement only.
 */
int pp2d_pomdp_set_goals(pp2d_pomdp* h, const uint32_t* goals_xy, uint32_t n,
                         const float* stage_rewards);
int pp2d_pomdp_goals(pp2d_pomdp* h, uint32_t* count, uint32_t* goals_xy);
int pp2d_pomdp_goal_reward(pp2d_pomdp* h, uint32_t g, float* stage_reward);
int pp2d_pomdp_set_goal_alphas(pp2d_pomdp* h, uint32_t g, const float* fib_alphas,
                               const uint8_t* fib_actions, const float* pbvi_alphas,
                               const uint8_t* pbvi_actions, uint32_t n_pbvi);
int pp2d_tree_batch_create_goals(pp2d_pomdp* h, const float* beliefs, const uint32_t* goals,
                                 uint32_t n, pp2d_tree_batch** out);
int pp2d_pomdp_padding_counters(pp2d_pomdp* h, uint64_t out[2]);

/* ------------------------------------------------------------------------
 * dummy_simulator's Bayes filter (SURVEY.md section 8f row 4b)
 * ------------------------------------------------------------------------ */
typedef struct pp2d_sim pp2d_sim;

/* The simulator's own copy of the map (dummy_simulator.cpp:399-410: the same
 * threshold as the planners, 1 = occupied). */
int pp2d_sim_create(uint32_t height, uint32_t width, const uint8_t* map, pp2d_sim** out);
void pp2d_sim_destroy(pp2d_sim* s);
/*
 * DummySimulator::updateBelief(const uint8_t& u) (dummy_simulator.cpp:671-718,
 * with transitionProbability, :440-522): prediction with the motion model --
 * blocked and out-of-map mass stays, NO trapped-cell override, unlike the
 * planners' tables -- then the sequential-sum normalisation.  n independent
 * beliefs [n][HW] in host memory, updated in place, belief i with actions[i].
 * Same bits as the reference's scatter loop (summation order per target cell
 * reproduced).
 */
int pp2d_sim_update_belief_action(pp2d_sim* s, float* beliefs, uint32_t n,
                                  const uint8_t* actions);
/*
 * DummySimulator::updateBelief(const std::vector<uint8_t>& meas)
 * (dummy_simulator.cpp:720-773): likelihood of the four cell measurements
 * {up, left, right, down} (0.98 / 0.02, out of map = occupied) times the prior,
 * normalised.  measurements: [n][4] bytes.
 */
int pp2d_sim_update_belief_measurement(pp2d_sim* s, float* beliefs, uint32_t n,
                                       const uint8_t* measurements);
/* controlCallback's filter part (dummy_simulator.cpp:174-181): action update,
 * then measurement update, one round trip. */
int pp2d_sim_step(pp2d_sim* s, float* beliefs, uint32_t n, const uint8_t* actions,
                  const uint8_t* measurements);

/* ------------------------------------------------------------------------
 * Closed-loop episodes: planner + simulator in one device loop (DESIGN.md
 * section 7, "Closed-loop rollouts")
 * ------------------------------------------------------------------------
 * Episode i (global id e = first_episode + i) starts at cell starts_xy[2i],
 * starts_xy[2i+1] (free in the simulator's map) with belief beliefs[i] ([n][HW];
 * NULL: a point mass of 1.0f at the start).  Each step t: stop when the true
 * cell is the planner's goal (reached = 1) or t == max_steps (reached = 0);
 * u = the planner's action at the belief mode; move by the simulator's motion
 * model (blocked or out-of-map targets: stay, collisions += 1); read the four
 * cell sensors {up, left, right, down} of the simulator's map, each flipped
 * with probability 0.02; filter the belief as pp2d_sim_step.  Random numbers:
 * Philox4x32-10, key (seed & 0xffffffff, seed >> 32), step t of episode e uses
 * the blocks of counters (t, e_lo, e_hi, 0) and (t, e_lo, e_hi, 1); a word w
 * is the uniform (w >> 8) * 2^-24.  Results depend only on (maps, planner,
 * start, belief, seed, e), not on the other episodes of the call.
 *
 * Every output pointer may be NULL; entries past an episode's last step are
 * not written.  PP2D_ERR_INVALID (messages name the episode) for NULL handles
 * or starts_xy, a world / planner size mismatch, a start outside the map or
 * occupied in the simulator's map, an instance index >= count;
 * PP2D_ERR_STATE for a shard or multi-GPU planner.  All checks come before any
 * device work; n == 0 does nothing. */
typedef struct pp2d_rollout {   /* every pointer may be NULL */
  uint32_t* steps;          /* [n] steps taken */
  uint8_t*  reached;        /* [n] 1: stopped on the goal */
  uint32_t* collisions;     /* [n] moves into a blocked or out-of-map cell */
  uint32_t* final_cell;     /* [n] y*W+x */
  float*    final_belief;   /* [n][HW] */
  uint32_t* cells;          /* [n][max_steps+1], start included */
  uint8_t*  actions;        /* [n][max_steps] */
  uint8_t*  measurements;   /* [n][max_steps], bit j = sensor j */
} pp2d_rollout;
/* Every episode follows the single-GPU handle `planner` (its goal, its action
 * grid as pp2d_mdp_plan reads it). */
int pp2d_sim_rollout_mdp(pp2d_sim* s, pp2d_mdp* planner, uint32_t n, const uint32_t* starts_xy,
                         const float* beliefs, uint32_t max_steps, uint64_t seed,
                         uint64_t first_episode, pp2d_rollout* out);
/* Episode i follows batch instance instances[i] (its goal, and its action
 * grid as pp2d_mdp_batch_plan reads it: the snapshot of a frozen instance). */
int pp2d_sim_rollout_mdp_batch(pp2d_sim* s, pp2d_mdp_batch* planner, const uint32_t* instances,
                               uint32_t n, const uint32_t* starts_xy, const float* beliefs,
                               uint32_t max_steps, uint64_t seed, uint64_t first_episode,
                               pp2d_rollout* out);
/* Every episode follows the QV-tree planner `planner` (its goal; its alpha
 * vectors must be set, PP2D_ERR_STATE otherwise) as PomdpPathPlanning2d's
 * beliefCallback does (DESIGN.md section 7d): episode i keeps one search tree,
 * created from beliefs[i] (NULL: the point mass at its start); step t plans it
 * (pp2d_tree_plan with max_depth, max_iter), u = the best action, the world
 * moves and senses as above, and the tree is updated with (u, z), z = the
 * measurement byte.  The simulator's filter is not run: final_belief is the
 * tree's root belief after the last update (the start belief if no step was
 * taken).  max_depth == 0 or max_iter == 0 give PP2D_ERR_INVALID (a step must
 * leave an expanded root to update).  Each step plans only the episodes still
 * running, together, through one tree batch; the world steps on the host. */
int pp2d_sim_rollout_pomdp(pp2d_sim* s, pp2d_pomdp* planner, uint32_t n, const uint32_t* starts_xy,
                           const float* beliefs, uint32_t max_steps, uint32_t max_depth,
                           uint32_t max_iter, uint64_t seed, uint64_t first_episode,
                           pp2d_rollout* out);
/* pp2d_sim_rollout_pomdp with a goal per episode (DESIGN.md section 7e):
 * episode i plans to goal goals[i] of the planner's goal set and stops on that
 * goal's cell.  It is bit for bit episode i (same id) of
 * pp2d_sim_rollout_pomdp on a handle created with that goal, with the same
 * tables and that goal's alpha vectors.  Checks as pp2d_sim_rollout_pomdp,
 * plus NULL goals or an index above the set (PP2D_ERR_INVALID) and a goal
 * without alpha vectors (PP2D_ERR_STATE), all before any device work. */
int pp2d_sim_rollout_pomdp_goals(pp2d_sim* s, pp2d_pomdp* planner, const uint32_t* goals,
                                 uint32_t n, const uint32_t* starts_xy, const float* beliefs,
                                 uint32_t max_steps, uint32_t max_depth, uint32_t max_iter,
                                 uint64_t seed, uint64_t first_episode, pp2d_rollout* out);

#ifdef __cplusplus
}
#endif
#endif /* PP2D_H_ */
