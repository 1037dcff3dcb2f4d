// uavmp_internal.h — shared declarations of the CUDA library (not installed; include/uavmp.h is the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "uavmp.h"

#define UAVMP_MAXPRIM 736   // (2*acc_resolution+1)^3 <= 729  (acc_resolution <= 4), padded to 23 warps
#define UAVMP_MAXK 16       // checkpoints per primitive: floor(sample_tau/time_step_size)+1
#define UAVMP_MAXNA 9       // lattice values per axis: 2*acc_resolution+1
#define UAVMP_NONE 0xffffffffu

// ---- device-side views ---------------------------------------------------------------------------
struct KinoParamsDev {
  int allocated, ctype, K, nprim, na;
  double ua[UAVMP_MAXNA];  // the per-axis acceleration values (the lattice is their tensor product, ax outer / az inner)
  double rou, lambda, goal_tol, step, vmax, tau, tie;
  double robot_r, robot_h;
  double box_r;     // conservative half-extent of the ellipsoid bounding cube
  float kd_r2;      // (float)(robot_r + 0.1) squared: the KD-tree radius filter of kino_astar.cpp:744
  double cull2;     // (max semi-axis * 1.001 + 1e-6)^2: farther points cannot be inside the ellipsoid
  float cullf;      // the same with a 2 mm margin, for the float pre-cull
  double inv_r2, inv_h2;
  float inv_r2f, inv_h2f;
  double tk[UAVMP_MAXK];  // i * step_size
  double hk[UAVMP_MAXK];  // 0.5 * t * t
  double htau;            // 0.5 * tau * tau
};

// per-primitive tables (global memory, read-only)
struct LatticeDev {
  const double* ux; const double* uy; const double* uz;  // acceleration lattice in the reference's loop order
  const double* ginc;                                    // (u.u + rou) * tau
  const double* Einv;                                    // nprim x 9, row-major inverse of Rot diag(r,r,h) Rot^T
  const double* b3;                                      // nprim x 3, body z axis (thrust direction)
  const float4* b3f;                                     // the same in float (w unused), for the float slab pre-test
};

struct MapDev {
  const uint8_t* flags;  // bit0: inflate==1, bit1: inflate!=0, bit2: a cloud point may lie within the ellipsoid box
                         // layout [nx][nzp / 16][ny][16] (16-voxel z blocks innermost), nzp = nz rounded up to 16
  int nx, ny, nz, nzp;
  double ox, oy, oz;                    // mp_.map_origin_
  double lox, loy, loz, hix, hiy, hiz;  // map_min_boundary_ + 1e-4, map_max_boundary_ - 1e-4
  double inv_res;
  // uniform cell list over the cloud (float4-padded points sorted by cell)
  const int* cell_start;
  const float4* pts;
  double cox, coy, coz, inv_cell;
  int cnx, cny, cnz, n_cloud;
};

struct __align__(8) KinoNode {
  double px, py, pz, vx, vy, vz, g;
  uint32_t parent;    // node id or UAVMP_NONE
  uint32_t hslot;     // this node's slot in the arena's hash table
  uint16_t input;     // lattice id of the primitive that produced this state
  uint8_t closed;
  uint8_t pad0;
  uint32_t pad1;
};
static_assert(sizeof(KinoNode) == 72, "node record is 72 B");

struct __align__(16) HeapSlot {
  double f;      // cached key; kept equal to the live f_cost (in-place mutations write through the slot's heap_pos)
  uint32_t id;
  uint32_t hs;   // hash slot of node `id` (bit 31: dirty marker while staged in shared memory)
};
// One 32 B sector answers everything the successor classification needs: exists? closed? g? where in the open list?
struct __align__(32) HashSlot {
  unsigned long long key;  // (packed voxel index << 10) | epoch
  uint32_t id;
  uint32_t heap_pos;       // 0-based slot in the open-list array (valid while the node is open)
  double g;
  uint32_t closed;
  uint32_t pad;
};
static_assert(sizeof(HashSlot) == 32, "hash slot is one sector");

struct KinoArena {           // one per resident CTA, reused across queries
  KinoNode* nodes;           // allocated
  HeapSlot* heap;            // allocated + 2 (slot i lives at heap[i+1] so both children share a 32 B sector)
  HashSlot* table;           // table_size
  uint32_t* epoch;           // 1 word
};

struct KinoBatchDev {
  int B;
  const double* start_pt; const double* start_vel; const double* end_pt; const double* end_vel;
  const int* order;          // processing order (longest straight-line distance first) or nullptr
  int* status; int* use_node_num; int* n_pop; unsigned long long* pop_hash;
  int* n_path;               // points per query
  double* path_stage;        // B x path_cap x 3
  int path_cap;
  int* pop_trace; int pop_cap;  // optional B x pop_cap x 3
  int* error_flag;
  unsigned long long* counters;  // 8 words
  int* next_query;           // work counter
  unsigned long long* phase_cycles;  // optional profiling: 8 words, SM cycles per phase summed over CTAs
  long long* query_cycles;           // optional profiling: B words, SM cycles each query occupied its CTA
  unsigned long long* query_phase;   // optional profiling: B x 16 words, the phase cycles of every query
};

// In-kernel QP of the plan pipeline: the CTA that finished a query also solves its three 1-D problems (one warp per problem,
// workspace in the shared memory the search no longer needs), so a batch is ONE kernel with no second stream and no
// cross-kernel flag polling.  Problem id = 3 * query + axis.
struct KinoQpDev {
  int enabled;               // 0: search only
  int warps;                 // problems solved concurrently per round (how many workspaces fit in the overlay)
  int Sg, n;                 // segments, coefficients per axis ((order + 1) * S)
  double seg_time;
  int time_alloc;            // 1: T_s = max(idx_{s+1} - idx_s, 1) * step (uavmp_plan_options)
  double step;               // time_step_size: spacing of the sampled path points
  int Kc;                    // corridor samples per segment (0: none)
  double margin;             // corridor box = bounding box of the segment's path points +- margin
  double* lo; double* hi;    // per-problem corridor boxes (3 B x S), Kc > 0 only
  double* pos; double* bv; double* ba; double* bj; double* T;  // per-problem inputs of qp_warp_solve_one (3 B problems)
  double* coef;              // B x 3 x n, the caller-visible layout (problem id * n)
  int* solved3; int* status3; int* iters3;                     // per problem
  int* qp_solved;            // per query: search reached the goal AND all three axes solved
};

// ---- host-side context -----------------------------------------------------------------------------
struct QpPlan;  // qp_kernel.cu
struct AstarState;  // astar_kernel.cu
struct RrtState;    // rrt_kernel.cu

#define UAVMP_NSLOT 7  // slot 0: the synchronous entry points; 1..6: batches in flight (uavmp_plan_submit) — the tail of a batch
                       // spans ~3 batch times

// device scratch of the stand-alone QP kernels (one per user of qp_solve_batch_dev: the context and every slot)
struct QpScratch {
  void* ws = nullptr; size_t ws_bytes = 0;       // batch-interleaved workspace of the thread-per-problem kernel
  void* tab = nullptr; size_t tab_bytes = 0;     // ragged batches: chunk counter | group table | segment offsets | problem ids
  void* tmp = nullptr; size_t tmp_bytes = 0;     // ragged batches: contiguous copy of one thread-kernel group (inputs, outputs)
};

// One ragged batch of 1-D problems (qp_solve_ragged_dev): problem p has S_p segments; with so_p = sum_{i<p} S_i its waypoints start
// at pos[so_p + p], its segment times at T[so_p], its coefficients at coef[(order + 1) so_p]; bv / ba / bj (B x 2) and the per-problem
// outputs are indexed by p.  seg_off (so_p, device) is filled in by qp_solve_ragged_dev.
struct QpRaggedIo {
  const double *pos, *bv, *ba, *bj, *T;
  double* coef; int *solved, *status, *iters;
  const long long* seg_off;
  int order;
};

// Everything ONE batch in flight owns.  Slot 0 runs on the context's stream and serves the synchronous entry points.
struct PlanSlot {
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[5];               // 0 start, 1 inputs on the device, 2 after the kernels, 3 outputs copied, 4 done (info copied)
  bool in_flight = false;
  long long ticket = -1;
  int B = 0;
  bool host_io = false;
  // search batch buffers
  int cap = 0, path_cap = 0, pop_cap = 0;
  double* d_q = nullptr;           // 4 x B x 3 (host-input calls)
  int* d_order = nullptr;          // idx | idx_sorted | key | key_sorted
  int* d_status = nullptr; int* d_use = nullptr; int* d_npop = nullptr; unsigned long long* d_hash = nullptr;
  int* d_npath = nullptr; double* d_path_stage = nullptr; int* d_trace = nullptr; long long* d_offsets = nullptr;
  int* d_misc = nullptr;           // [0] error flag, [1] work counter
  unsigned long long* d_counters = nullptr;
  void* d_cub_tmp = nullptr; size_t cub_tmp_bytes = 0;
  // plan pipeline
  double* d_wp = nullptr; size_t wp_bytes = 0;         // per-problem QP inputs (3 B problems)
  int* d_qp_int = nullptr; size_t qp_int_bytes = 0;    // solved | status | iters per problem
  double* d_qp_out = nullptr; size_t qp_out_bytes = 0; // sequential fallback only: axis-major coefficients
  double* d_plan_out = nullptr; size_t plan_out_bytes = 0;  // host-output calls: B x 3 x n staging
  int* d_plan_io = nullptr; size_t plan_io_bytes = 0;       // host-output calls: status | qp_solved
  QpScratch qp_scr;
  // pinned host mirror of the error flag and the counters, written by the stream at the end of the batch
  struct HostInfo { int flag; int pad; unsigned long long counters[8]; }* h_info = nullptr;
  int launches_search = 0, launches_qp = 0, launches_aux = 0;
};

struct uavmp_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  int sm_count = 0;

  // params
  uavmp_kino_params kp;
  bool params_dirty = true;
  KinoParamsDev* d_kparams = nullptr;
  double* d_lattice = nullptr;  // ux|uy|uz|ginc|Einv|b3
  float4* d_b3f = nullptr;
  int nprim = 0;
  int path_cap = 1024, pop_cap = 0;

  // map
  bool have_map = false;
  int nx = 0, ny = 0, nz = 0;
  double origin[3], map_size[3], resolution = 0;
  int8_t* d_occ = nullptr;
  uint8_t* d_flags = nullptr;
  uint8_t* d_tmp = nullptr;
  float* d_cloud = nullptr;
  int n_cloud = 0;
  int* d_cell_start = nullptr;
  float4* d_pts = nullptr;
  MapDev map_host;
  MapDev* d_map = nullptr;
  uint8_t* d_flags_pad = nullptr;   // [nx][nzp / 16][ny][16]
  unsigned char tmap_bytes[128] __attribute__((aligned(64)));  // CUtensorMap over d_flags_pad, box 32 x 32 x 48
  bool have_tmap = false;
  bool flags_dirty = true;

  // search arenas: a pool shared by every search kernel in flight; a CTA takes a free one when it starts (arena_busy)
  int n_arenas = 0, arena_nodes = 0, table_size = 0;
  void* d_arena_mem = nullptr;
  KinoArena* d_arenas = nullptr;
  int* d_arena_busy = nullptr;

  // batches
  PlanSlot slots[UAVMP_NSLOT];
  long long next_ticket = 0;
  int last_slot = 0;               // slot of the most recently completed batch (what the legacy getters read)
  long long last_total_path = 0;
  double* d_path_packed = nullptr; long long path_packed_cap = 0;
  bool profile_phases = false;
  unsigned long long* d_phase = nullptr; long long* d_query_cycles = nullptr; int query_cycles_cap = 0;
  int last_grid = 0;
  uavmp_kino_counters last_counters;
  int last_error_flag = 0;

  // qp (stand-alone uavmp_minctrl_solve_batch, on the context's stream)
  std::vector<QpPlan*> qp_plans;
  QpScratch qp_scr;
  double* d_qp_in = nullptr; size_t qp_in_bytes = 0;
  double* d_qp_out = nullptr; size_t qp_out_bytes = 0;
  int* d_qp_int = nullptr; size_t qp_int_bytes = 0;

  // batched grid A* (astar_kernel.cu): parameters of Astar::setParam (a_star.cpp:6-11) and the lazily built device state
  AstarState* astar = nullptr;
  int astar_allocated = 100000, astar_path_cap = 4096;
  double astar_lambda = 1.0;
  // batched RRT* (rrt_kernel.cu): parameters of RRTStar::setParam (rrt_star.cpp:7-11; the time budget is a budget of drawn samples)
  RrtState* rrt = nullptr;
  int rrt_max_nodes = 100000, rrt_path_cap = 4096;
  double rrt_step = 0.5, rrt_radius = 0.5, rrt_ccres = 0.05, rrt_budget = 100000.0;

  // timings of the last completed call
  cudaEvent_t ev[8];
  uavmp_timings tm;
};

int uavmp_fail(uavmp_ctx* ctx, int code, const char* fmt, ...);
#define UAVMP_CUDA(ctx, call)                                                                  \
  do {                                                                                         \
    cudaError_t e_ = (call);                                                                   \
    if (e_ != cudaSuccess) return uavmp_fail(ctx, UAVMP_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
  } while (0)

int ensure_bytes(uavmp_ctx* ctx, void** p, size_t* have, size_t want);
int drain_all(uavmp_ctx* ctx);  // capi.cu: wait for every batch in flight
int uavmp_map_check_geometry(uavmp_ctx* ctx, int nx, int ny, int nz, const double origin[3], const double map_size[3], double resolution);

// kino_kernel.cu
int kino_upload_params(uavmp_ctx* ctx);
int kino_build_map(uavmp_ctx* ctx);
int kino_ensure_arenas(uavmp_ctx* ctx);
int kino_ensure_slot(uavmp_ctx* ctx, PlanSlot& sl, int B);
void kino_free_slot(PlanSlot& sl);
int kino_qp_overlay_bytes();  // shared memory of the search CTA the in-kernel QP may overlay
struct QpPlanDev;
int kino_launch_search(uavmp_ctx* ctx, PlanSlot& sl, int B, const double* d_start_pt, const double* d_start_vel,
                       const double* d_end_pt, const double* d_end_vel, bool sort_order, bool profile,
                       const KinoQpDev* qp, const QpPlanDev* plan, const uavmp_osqp_settings* settings);
int kino_pack_paths(uavmp_ctx* ctx, PlanSlot& sl, int B);

// astar_kernel.cu
long long astar_search_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* end_pt, int* status, int* use_node_num,
                             long long* path_offsets, uint64_t* pop_hash, int* n_pop);
int astar_get_paths(uavmp_ctx* ctx, double* path_xyz, long long cap_points);
void astar_destroy(uavmp_ctx* ctx);
// rrt_kernel.cu
long long rrt_search_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* end_pt, const uint64_t* query_seed, int* status,
                           int* use_node_num, long long* n_samples, double* goal_g_cost, uint64_t* tree_digest, long long* path_offsets);
int rrt_get_paths(uavmp_ctx* ctx, double* path_xyz, long long cap_points);
long long rrt_plan_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* start_vel, const double* end_pt, const uint64_t* query_seed,
                         int order, double seg_time, const uavmp_osqp_settings* settings, int* search_status, int* n_segments,
                         int* qp_solved, long long* coef_offsets, int* osqp_status, int* iters);
int rrt_plan_get_coef(uavmp_ctx* ctx, double* coef, long long cap);
// qp_kernel.cu: B problems with S_host[p] segments each (order 5 / 7, no corridor rows) in one grouped launch plus one thread-kernel
// launch per S whose warp workspace does not fit in shared memory; asynchronous on `st`
int qp_solve_ragged_dev(uavmp_ctx* ctx, cudaStream_t st, QpScratch& scr, int order, int B, const int* S_host, QpRaggedIo r,
                        const uavmp_osqp_settings* settings, int* qp_launches, int* aux_launches, int* n_groups, int* n_thread_groups);
void rrt_destroy(uavmp_ctx* ctx);
uint32_t rrt_sample_seed_host(unsigned long long query_seed, long long i);
