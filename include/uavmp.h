/* uavmp.h — C-ABI of the B200-native batched trajectory front-end / back-end.
 *
 * The reference has no plugin/FFI layer: the two hot paths are plain C++ classes called from ROS test nodes
 * (SURVEY.md §8(b)).  A maintainer swaps them by calling these entry points from thin C++ shims that keep the
 * reference signatures (include/uavmp/kino_astar.hpp, include/uavmp/minimum_control.hpp, INTEGRATION.md):
 *
 *   uavmp_kino_search_batch      replaces  path_searching::KinoAstar::search
 *                                (src/planner/path_searching/include/path_searching/kino_astar.h:197-198,
 *                                 src/planner/path_searching/src/kino_astar.cpp:81-272), B queries at once
 *   uavmp_kino_set_params        replaces  KinoAstar::setParam            (kino_astar.cpp:6-36)
 *   uavmp_map_set                replaces  KinoAstar::setGridMap + init + localCloudCallback
 *                                (kino_astar.cpp:38-79) and the GridMap lookups it reads
 *                                (src/planner/plan_env/include/plan_env/grid_map.h:257-260,350-359,370-385,400-404)
 *   uavmp_minctrl_solve_batch    replaces  traj_optimization::MinimumControl::solve + getCoef1d
 *                                (src/planner/traj_optimization/include/traj_optimization/minimum_control.h:34-41,
 *                                 src/planner/traj_optimization/src/minimum_control.cpp:127-202), B 1-D QPs at once
 *   uavmp_minctrl_solve_ragged_batch  the same for problems with a different segment count each, in one call
 *   uavmp_rrt_plan_batch         the reference's own RRTStar::search -> MinimumControl::solve flow (test_minimum_jerk.cpp:40-75),
 *                                B queries at once
 *   uavmp_plan_batch             the search -> waypoints -> 3 x QP pipeline (an extension; the reference never
 *                                chains the two, SURVEY.md §0)
 *
 * Conventions: plain pointers and sizes, no exceptions, return 0 on success or a negative UAVMP_E* code
 * (uavmp_last_error gives the text).  A context is bound to one CUDA device and one stream and is not thread-safe.
 * Unless a function says otherwise, pointers are HOST memory and the call copies in / out and synchronises.
 */
#ifndef UAVMP_H
#define UAVMP_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define UAVMP_OK 0
#define UAVMP_EINVAL (-1)
#define UAVMP_ECUDA (-2)
#define UAVMP_ENOMEM (-3)
#define UAVMP_ESTATE (-4) /* e.g. search before uavmp_map_set */
#define UAVMP_ECAP (-5)   /* an output capacity was too small */

/* search return codes, kino_astar.h:155-159 */
#define UAVMP_REACH_END 1
#define UAVMP_NO_PATH_FOUND 2

typedef struct uavmp_ctx uavmp_ctx;

/* ROS parameters of KinoAstar::setParam (kino_astar.cpp:8-19), same names */
typedef struct {
  int allocated_node_num;
  int collision_check_type; /* 1: inflated grid, then (switch fall-through) ellipsoid; 2: ellipsoid only */
  double rou_time;
  double lambda_heu;
  double goal_tolerance;
  double time_step_size;
  double max_velocity;
  double max_accelration; /* sic — the reference's parameter name */
  double acc_resolution;
  double sample_tau;
  double robot_r; /* kino_se3/robot_r */
  double robot_h; /* kino_se3/robot_h */
} uavmp_kino_params;

/* OSQP settings that MinimumControl::solve leaves at their defaults or overrides
 * (minimum_control.cpp:160-162; 3rd/osqp/include/public/osqp_api_constants.h:96-153) */
typedef struct {
  double rho, sigma, alpha;
  double eps_abs, eps_rel, eps_prim_inf, eps_dual_inf;
  int max_iter;
  int check_termination;
  int scaling;               /* Ruiz iterations */
  int adaptive_rho;
  int adaptive_rho_interval; /* 0 = 4 x check_termination (the deterministic, profiling-off rule) */
  double adaptive_rho_tolerance;
} uavmp_osqp_settings;

/* per-call device timings, milliseconds, CUDA events on the context's stream */
typedef struct {
  float h2d_ms, search_ms, path_ms, qp_ms, d2h_ms, total_ms;
  int search_launches, qp_launches, aux_launches;
} uavmp_timings;

/* counters the search kernel accumulates (summed over the batch); feed SURVEY.md §8(d)'s byte formula */
typedef struct {
  long long n_pop, n_occ_lookup, n_cloud_pts_tested, n_hash_probe, n_insert, n_update, n_heuristic, n_shot;
} uavmp_kino_counters;

/* what uavmp_plan_wait reports about one batch of the asynchronous pipeline */
typedef struct {
  int error_flags; /* 0, or bits: 1 voxel index outside the key range, 2 path with too many nodes, 4 path longer than path_cap */
  uavmp_kino_counters counters;
  uavmp_timings timings; /* CUDA events on the batch's own stream; batches in flight overlap, so their durations do too */
} uavmp_plan_info;

/* ---- context ------------------------------------------------------------------------------------- */
int uavmp_ctx_create(uavmp_ctx** out, int device);
void uavmp_ctx_destroy(uavmp_ctx* ctx);
const char* uavmp_last_error(const uavmp_ctx* ctx);
/* the cudaStream_t every kernel of this context is launched on (for external CUDA events) */
void* uavmp_ctx_stream(uavmp_ctx* ctx);
/* waits for everything issued so far, batches in flight included; returns the error of an asynchronous batch, if any */
int uavmp_ctx_sync(uavmp_ctx* ctx);
const char* uavmp_version(void);

/* ---- parameters ------------------------------------------------------------------------------------ */
void uavmp_kino_params_default(uavmp_kino_params* p); /* the C++ defaults, kino_astar.cpp:8-19 */
void uavmp_kino_params_launch(uavmp_kino_params* p);  /* test_kino_astar_searching.launch:44-57 */
void uavmp_osqp_settings_default(uavmp_osqp_settings* s); /* what MinimumControl::solve ends up running with */
int uavmp_kino_set_params(uavmp_ctx* ctx, const uavmp_kino_params* p);

/* ---- map -------------------------------------------------------------------------------------------- */
/* occ_inflate: GridMap::md_.occupancy_buffer_inflate_, address = x*ny*nz + y*nz + z (grid_map.h:257-260).
 * origin / map_size: mp_.map_origin_ / mp_.map_size_ (grid_map.cpp:52-54).  cloud_xyz: the PointCloud2 the
 * planner subscribed to ("local_cloud", kino_astar.cpp:38-55), n_cloud x 3 float32; may be NULL/0 only when no
 * search uses the ellipsoid test. */
int uavmp_map_set(uavmp_ctx* ctx, const int8_t* occ_inflate, int nx, int ny, int nz, const double origin[3],
                  const double map_size[3], double resolution, const float* cloud_xyz, int n_cloud);

/* the same, with GridMap::cloudCallback's inflation (src/planner/plan_env/src/grid_map.cpp:733-785: every point stamps its
 * (2s+1) x (2s+1) x 3 voxel neighbourhood, s = ceil(obstacles_inflation / resolution)) done on the device: only the cloud
 * crosses PCIe.  uavmp_map_get_occupancy returns the resulting occupancy_buffer_inflate_ (nx*ny*nz bytes). */
int uavmp_map_set_from_cloud(uavmp_ctx* ctx, const float* cloud_xyz, int n_cloud, int nx, int ny, int nz, const double origin[3],
                             const double map_size[3], double resolution, double obstacles_inflation);
int uavmp_map_get_occupancy(uavmp_ctx* ctx, int8_t* occ_inflate, long long cap);

/* ---- hot path (a): batched KinoAstar::search -------------------------------------------------------- */
/* start_pt/start_vel/end_pt/end_vel: B x 3 f64.  status: 1|2 per query.  use_node_num: KinoAstar::use_node_num_
 * at return.  path_offsets: B+1 prefix sums of path point counts (the points search() push_back's into `path`).
 * pop_hash / n_pop (nullable): digest and length of the ordered expansion sequence, for parity checks.
 * Returns the total number of path points (>= 0) or a negative error.  Fetch the points with uavmp_kino_get_paths. */
long long uavmp_kino_search_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* start_vel,
                                  const double* end_pt, const double* end_vel, int* status, int* use_node_num,
                                  long long* path_offsets, uint64_t* pop_hash, int* n_pop);
int uavmp_kino_get_paths(uavmp_ctx* ctx, double* path_xyz, long long cap_points);
/* ordered popped voxel indices of query q of the last batch (B*pop_cap*3 ints kept on device when tracing is on) */
int uavmp_kino_set_trace(uavmp_ctx* ctx, int pop_cap);
int uavmp_kino_get_trace(uavmp_ctx* ctx, int q, int32_t* pop_idx_xyz, int cap);
/* counters of the most recently completed batch */
int uavmp_kino_get_counters(uavmp_ctx* ctx, uavmp_kino_counters* out);
/* capacity of the per-query path staging, in sampled points (default 1024; a longer path fails its batch with UAVMP_ECAP) */
int uavmp_kino_set_path_cap(uavmp_ctx* ctx, int points);

/* ---- the other grid front-end: batched Astar::search (SURVEY.md §8(f) row 4) ------------------------------ */
/* replaces path_searching::Astar::setParam / search (src/planner/path_searching/src/a_star.cpp:6-11,48-154,
 * include/path_searching/a_star.h:142-147) on the map given to uavmp_map_set: 26-connected grid A* whose nodes are keyed by their
 * exact position, diagonal heuristic, in-place g updates, libstdc++ heap order.  lambda_heu / allocated_node_num: the ROS
 * parameters astar/lambda_heu, astar/allocated_node_num (astar/resolution is overwritten by the grid map's, a_star.cpp:31);
 * path_cap_nodes: capacity of a returned path (a longer one fails the call with UAVMP_ECAP). */
int uavmp_astar_set_params(uavmp_ctx* ctx, double lambda_heu, int allocated_node_num, int path_cap_nodes);
/* start_pt / end_pt: B x 3.  status 1 REACH_END | 2 NO_PATH_FOUND; use_node_num = use_node_num_ at return; path_offsets: B + 1 prefix
 * sums of path node counts (start ... last popped node, retrievePath a_star.cpp:180-190); pop_hash / n_pop (nullable): digest and
 * length of the ordered expansion sequence.  Returns the total number of path nodes or a negative error. */
long long uavmp_astar_search_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* end_pt, int* status,
                                   int* use_node_num, long long* path_offsets, uint64_t* pop_hash, int* n_pop);
int uavmp_astar_get_paths(uavmp_ctx* ctx, double* path_xyz, long long cap_points);

/* ---- the sampling front-end: batched RRTStar::search (SURVEY.md §8(f) row 4; the reference's QP front-end, test_minimum_jerk.cpp:40-75) -- */
/* replaces path_searching::RRTStar::setParam / search / getOptimalPath (src/planner/path_searching/src/rrt_star.cpp:5-11,304-429,
 * :299-302; include/path_searching/rrt_star.h:84-93) and the kd-tree it calls (src/kdtree/kdtree.cpp).  The reference draws every sample
 * from a fresh std::random_device (one 32-bit value seeds a std::mt19937_64 per sample, rrt_star.cpp:104-116) and stops on wall-clock time;
 * the deterministic form here: the 32-bit seed of query q's sample i is uavmp_rrt_sample_seed(query_seed[q], i), and
 * `rrt_star/max_tolerance_time` is `sample_budget`, a number of drawn samples (the search returns REACH_END at the first accepted sample
 * i with i + 1 >= sample_budget once the goal is connected, else after max_tree_node_num samples).  With that, the tree (every node's
 * position, parent and g_cost) is the one the reference's own code builds from the same seeds (oracle/_ref/librrt_ref.so).
 * max_tree_node_num / step_length / search_radius / collision_check_resolution: the ROS parameters of the same names. */
int uavmp_rrt_set_params(uavmp_ctx* ctx, int max_tree_node_num, double step_length, double search_radius,
                         double collision_check_resolution, double sample_budget, int path_cap_nodes);
uint32_t uavmp_rrt_sample_seed(uint64_t query_seed, long long i);
/* start_pt / end_pt: B x 3; query_seed: B.  status 1 REACH_END | 2 NO_PATH_FOUND; use_node_num = use_node_num_; n_samples = samples drawn;
 * goal_g_cost = the goal node's g_cost (1 << 30 if never connected); tree_digest: order-free digest over (index, position, g_cost, parent)
 * of every node; path_offsets: B + 1 prefix sums over getOptimalPath() — which the reference only fills when a LATER sample improves on the
 * first feasible cost (rrt_star.cpp:396-404), so it may be empty with status 1.  Nullable outputs: all but status.  Returns the total number
 * of path points or a negative error. */
long long uavmp_rrt_search_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* end_pt, const uint64_t* query_seed,
                                 int* status, int* use_node_num, long long* n_samples, double* goal_g_cost, uint64_t* tree_digest,
                                 long long* path_offsets);
int uavmp_rrt_get_paths(uavmp_ctx* ctx, double* path_xyz, long long cap_points);

/* ---- hot path (b): batched MinimumControl::solve ---------------------------------------------------- */
/* order: 5 (minimum jerk, the reference) or 7 (minimum snap, extension §9.3).  S segments.
 * pos_1d: B x (S+1) waypoints; bound_vel / bound_acc (/ bound_jerk, order 7 only, else NULL): B x 2 start,end
 * derivatives; time_vec: B x S.  coef: B x (order+1)*S, segment-major, ascending power, local time
 * (== MinimumControl::getCoef1d).  solved[b] = 1 iff OSQP status == SOLVED (== the bool solve() returns);
 * osqp_status / iters are OSQP's status_val / iter. */
int uavmp_minctrl_solve_batch(uavmp_ctx* ctx, int order, int S, int B, const double* pos_1d,
                              const double* bound_vel, const double* bound_acc, const double* bound_jerk,
                              const double* time_vec, const uavmp_osqp_settings* settings, double* coef,
                              int* solved, int* osqp_status, int* iters);

/* The same with corridor (inequality) rows — an EXTENSION (SURVEY.md §9.3; the reference's rows are all equalities,
 * minimum_control.cpp:98-125): for every segment s and every j < n_corridor, the position at the interior time
 * (j + 1) / (n_corridor + 1) * T_s must lie in [corridor_lo[b][s], corridor_hi[b][s]] (B x S each).  These are true
 * inequality rows of the OSQP problem: rho = settings->rho on them (1e3 rho on the equality rows, auxil.c:75-104) and the
 * z-projection clip(., l, u) of update_z (auxil.c:188-203) is active.  n_corridor = 0 is uavmp_minctrl_solve_batch. */
int uavmp_minctrl_solve_corridor_batch(uavmp_ctx* ctx, int order, int S, int n_corridor, int B, const double* pos_1d,
                                       const double* bound_vel, const double* bound_acc, const double* bound_jerk,
                                       const double* time_vec, const double* corridor_lo, const double* corridor_hi,
                                       const uavmp_osqp_settings* settings, double* coef, int* solved, int* osqp_status,
                                       int* iters);

/* B one-dimensional MinimumControl::solve problems, problem b with its own S[b] >= 1 segments (order 5 or 7, no corridor rows).
 * Packed inputs / outputs, problems in order: problem b's waypoints start at pos_1d[sum_{i<b}(S[i]+1)], its segment times at
 * time_vec[sum_{i<b} S[i]], its coefficients at coef[(order+1) * sum_{i<b} S[i]].  bound_vel / bound_acc (/ bound_jerk, order 7
 * only): B x 2.  solved / osqp_status / iters (nullable): B.  settings NULL = defaults.  Per problem, every output is bit-identical
 * to uavmp_minctrl_solve_batch(order, S[b], 1, ...) on the same inputs: the problems whose warp workspace fits in shared memory
 * (order 5 up to S = 103, order 7 up to S = 70) are solved by ONE grouped launch whatever their S, the others by the thread-per-problem
 * kernel, one launch per such S (uavmp_get_timings: qp_launches). */
int uavmp_minctrl_solve_ragged_batch(uavmp_ctx* ctx, int order, int B, const int* S, const double* pos_1d, const double* bound_vel,
                                     const double* bound_acc, const double* bound_jerk, const double* time_vec,
                                     const uavmp_osqp_settings* settings, double* coef, int* solved, int* osqp_status, int* iters);

/* ---- the reference's RRT* -> minimum-jerk flow, batched (test_minimum_jerk.cpp:28-173 GoalCallback) ---------------------------- */
/* For every query: RRTStar::search (as uavmp_rrt_search_batch, same parameters, seeds and results); then, if it returned REACH_END
 * and getOptimalPath() has n >= 2 points, S = n - 1 segments with EVERY optimal-path point a waypoint, T_s = seg_time,
 * bound_vel = (start_vel, 0), bound_acc = (0, 0) (bound_jerk = 0 for order 7), one QP per axis (test_minimum_jerk.cpp:40-75), all
 * of the batch's QPs solved as one ragged batch (uavmp_minctrl_solve_ragged_batch) whose waypoints never leave the device.
 * n_segments[q] = S, or 0 when no QP was posed: status 2, or REACH_END with an empty optimal path (getOptimalPath() is only written
 * when a later sample improves the first feasible cost).  There the reference node would reuse its stale optimal_path_ (reset()
 * does not clear it) or resize time_vec to -1; this call poses no QP instead: n_segments = 0, qp_solved = 0, no coefficients.
 * qp_solved[q] = all three axes SOLVED.  coef_offsets (B + 1): prefix sums of 3 (order+1) S_q; query q's coefficients are axis-major
 * [3][(order+1) S_q] (== uavmp_plan_batch's per-query layout).  Nullable: start_vel (zero), coef_offsets, osqp_status / iters (B x 3,
 * 0 where no QP was posed).  Returns the total number of coefficients or a negative error (path longer than path_cap_nodes:
 * UAVMP_ECAP; no map: UAVMP_ESTATE); fetch them with uavmp_rrt_plan_get_coef.  uavmp_rrt_get_paths afterwards returns the optimal
 * paths (the waypoints).  Synchronous on the context's stream.  uavmp_get_timings: search_ms, path_ms (QP input packing), qp_ms. */
long long uavmp_rrt_plan_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* start_vel, const double* end_pt,
                               const uint64_t* query_seed, int order, double seg_time, const uavmp_osqp_settings* settings,
                               int* search_status, int* n_segments, int* qp_solved, long long* coef_offsets,
                               int* osqp_status, int* iters);
int uavmp_rrt_plan_get_coef(uavmp_ctx* ctx, double* coef, long long cap);

/* ---- pipeline: search -> waypoints -> QP (extension) ------------------------------------------------ */
/* For every query whose search reaches the goal, S+1 waypoints are taken from the sampled path at indices
 * floor(k*(n-1)/S), T_i = seg_time (the reference's convention is 1.0, test_minimum_jerk.cpp:66-71), boundary
 * derivatives = start_vel / end_vel and zero.  coef: B x 3 x (order+1)*S. */
int uavmp_plan_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* start_vel, const double* end_pt,
                     const double* end_vel, int order, int S, double seg_time, const uavmp_osqp_settings* settings,
                     int* search_status, int* qp_solved, double* coef);
/* same, every pointer already in device memory (inputs resident in HBM; outputs stay there).  Asynchronous: ordered after the
 * work already on the context's stream, and the context's stream waits for it; an error flag raised by the batch is returned by
 * the next uavmp_plan_batch_dev / uavmp_ctx_sync / uavmp_get_timings call. */
int uavmp_plan_batch_dev(uavmp_ctx* ctx, int B, const double* d_start_pt, const double* d_start_vel,
                         const double* d_end_pt, const double* d_end_vel, int order, int S, double seg_time,
                         const uavmp_osqp_settings* settings, int* d_search_status, int* d_qp_solved, double* d_coef);

/* What the pipeline builds between the search and the QP (all of it an extension: the reference never chains the two).
 * With n sampled path points (one every time_step_size along the searched trajectory) and idx_k = floor(k (n - 1) / S):
 *   waypoint k = path[idx_k];
 *   time_alloc 0: T_s = seg_time (the reference's convention, test_minimum_jerk.cpp:66-71);
 *   time_alloc 1: T_s = max(idx_{s+1} - idx_s, 1) * time_step_size — the searched trajectory's own timing;
 *   corridor_samples > 0: per segment and axis the box [min - margin, max + margin] over path[idx_s .. idx_{s+1}], imposed
 *   at corridor_samples interior times (uavmp_minctrl_solve_corridor_batch). */
typedef struct {
  int order; /* 5 or 7 */
  int S;
  double seg_time;
  int time_alloc;
  int corridor_samples;
  double corridor_margin;
} uavmp_plan_options;
void uavmp_plan_options_default(uavmp_plan_options* o); /* order 7, S 8, seg_time 1.0, no time allocation, no corridor */

/* Asynchronous form with several batches in flight.  A batch is ONE kernel (the CTA that finishes a query also solves its three
 * QPs), each batch runs on its own stream and its CTAs take search arenas from a shared pool, so the CTAs of batch k + 1 fill the
 * SMs the long tail of batch k leaves idle.  uavmp_plan_submit returns at once with a ticket; the outputs (and, for host
 * pointers, the copies into them) are complete when uavmp_plan_wait(ticket) returns.  At most uavmp_plan_max_in_flight()
 * tickets may be outstanding.  Host buffers should be page-locked, otherwise the copies serialise the batches.
 * flags: UAVMP_PLAN_DEVICE_IO = every pointer is device memory and the inputs are ordered after the work already on the
 * context's stream; uavmp_plan_stream_wait makes a CUDA stream of the caller wait for the batch without blocking the host. */
#define UAVMP_PLAN_DEVICE_IO 1u
int uavmp_plan_submit(uavmp_ctx* ctx, int B, const double* start_pt, const double* start_vel, const double* end_pt,
                      const double* end_vel, int order, int S, double seg_time, const uavmp_osqp_settings* settings,
                      unsigned flags, int* search_status, int* qp_solved, double* coef, long long* ticket);
/* uavmp_plan_submit with the full option block (time allocation, corridor rows) */
int uavmp_plan_submit_opt(uavmp_ctx* ctx, int B, const double* start_pt, const double* start_vel, const double* end_pt,
                          const double* end_vel, const uavmp_plan_options* opt, const uavmp_osqp_settings* settings,
                          unsigned flags, int* search_status, int* qp_solved, double* coef, long long* ticket);
int uavmp_plan_wait(uavmp_ctx* ctx, long long ticket, uavmp_plan_info* info /* nullable */);
int uavmp_plan_stream_wait(uavmp_ctx* ctx, long long ticket, void* cuda_stream);
int uavmp_plan_max_in_flight(void);

/* ---- consumer of the coefficients: PolyTraj::evaluatePos / Vel / Acc (traj_utils/poly_traj.hpp:74-168), batched ------- */
/* coef: B x 3 x S x (order+1) (axis-major per trajectory == uavmp_plan_batch's layout); times: B x S segment durations;
 * t: n_t sample times shared by all trajectories; deriv 0 position, 1 velocity, 2 acceleration; out: B x n_t x 3. */
int uavmp_polytraj_eval_batch(uavmp_ctx* ctx, int B, int order, int S, const double* coef, const double* times, int n_t,
                              const double* t, int deriv, double* out);

int uavmp_get_timings(uavmp_ctx* ctx, uavmp_timings* out);
/* optional in-kernel profile of the search: SM cycles per phase (0 pop, 1 shot/path, 2 primitive evaluation, 3 dedup +
 * table probe, 4 heuristic + id scan, 5 node/hash writes, 6 ordered heap commit, 7 query setup/epilogue) summed over the
 * CTAs (entries 8..15: diagnostics: cloud staging cycles, staged expansions, cycles of the ordered heap replay, staged points,
 * flagged primitives, closure staging / slow key updates / deferred writes of the commit),
 * the cycles every query kept its CTA busy, and the grid size of the last launch */
int uavmp_kino_set_profile(uavmp_ctx* ctx, int on);
int uavmp_kino_get_profile(uavmp_ctx* ctx, unsigned long long phase_cycles[16], long long* query_cycles, int cap, int* grid);

/* ---- test support ------------------------------------------------------------------------------------ */
/* device-evaluated csrc/fpmath.h (op 0 cbrt, 1 acos, 2 cos, 3 powi) for host/device bit-parity tests */
int uavmp_fpmath_eval(uavmp_ctx* ctx, int op, int n_pow, const double* x, double* y, long long n);

#ifdef __cplusplus
}
#endif
#endif /* UAVMP_H */
