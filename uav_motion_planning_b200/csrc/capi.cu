// capi.cu — the extern "C" boundary declared in include/uavmp.h.  No torch types, plain pointers and sizes.
#include <math.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "qp_plan.h"
#include "uavmp_internal.h"

int kino_fpmath_eval(uavmp_ctx* ctx, int op, int npow, const double* x, double* y, long long n);
// qp_kernel.cu
int qp_solve_batch_dev(uavmp_ctx* ctx, cudaStream_t stream, QpScratch& scr, int* launches, int order, int S, int Kc, int B,
                       const double* d_pos, const double* d_bv, const double* d_ba, const double* d_bj, const double* d_T,
                       const double* d_lo, const double* d_hi, const uavmp_osqp_settings* st, double* d_coef, int* d_solved,
                       int* d_status, int* d_iters);
int qp_waypoints_from_paths(uavmp_ctx* ctx, PlanSlot& sl, int B, const uavmp_plan_options& o, const double* d_sv, const double* d_ev,
                            double** d_pos, double** d_bv, double** d_ba, double** d_bj, double** d_T, double** d_lo, double** d_hi);
int qp_scatter_plan_outputs(uavmp_ctx* ctx, PlanSlot& sl, int B, int order, int S, const int* d_solved3, const double* d_coef3,
                            int* d_qp_solved, double* d_coef);
int qp_get_plan_dev(uavmp_ctx* ctx, int order, int S, int Kc, const QpPlanDev** out);
void qp_free_plans(uavmp_ctx* ctx);

int ensure_bytes(uavmp_ctx* ctx, void** p, size_t* have, size_t want) {
  if (*have >= want) return UAVMP_OK;
  if (*p) cudaFree(*p);
  *p = nullptr; *have = 0;
  UAVMP_CUDA(ctx, cudaMalloc(p, want));
  *have = want;
  return UAVMP_OK;
}

// ---- batches in flight -------------------------------------------------------------------------------------------------
static int error_from_flag(uavmp_ctx* ctx, int flag) {
  if (flag & 1) return uavmp_fail(ctx, UAVMP_ECAP, "voxel index outside the 18-bit key range");
  if (flag & 2) return uavmp_fail(ctx, UAVMP_ECAP, "path has more than %d nodes", UAVMP_MAXPRIM);
  if (flag & 4) return uavmp_fail(ctx, UAVMP_ECAP, "path longer than path_cap=%d points (uavmp_kino_set_path_cap)", ctx->path_cap);
  return UAVMP_OK;
}

// block until the batch of `sl` is complete, publish its info as "the last call" and free the slot
static int slot_finish(uavmp_ctx* ctx, PlanSlot& sl, uavmp_plan_info* info) {
  if (!sl.in_flight) return UAVMP_OK;
  UAVMP_CUDA(ctx, cudaEventSynchronize(sl.ev[4]));
  sl.in_flight = false;
  uavmp_timings& t = ctx->tm;
  memset(&t, 0, sizeof(t));
  cudaEventElapsedTime(&t.h2d_ms, sl.ev[0], sl.ev[1]);
  cudaEventElapsedTime(&t.search_ms, sl.ev[1], sl.ev[2]);
  cudaEventElapsedTime(&t.d2h_ms, sl.ev[2], sl.ev[3]);
  cudaEventElapsedTime(&t.total_ms, sl.ev[0], sl.ev[4]);
  t.search_launches = sl.launches_search; t.qp_launches = sl.launches_qp; t.aux_launches = sl.launches_aux;
  const unsigned long long* c = sl.h_info->counters;
  uavmp_kino_counters& k = ctx->last_counters;
  k.n_pop = c[0]; k.n_occ_lookup = c[1]; k.n_cloud_pts_tested = c[2]; k.n_hash_probe = c[3];
  k.n_insert = c[4]; k.n_update = c[5]; k.n_heuristic = c[6]; k.n_shot = c[7];
  ctx->last_error_flag = sl.h_info->flag;
  ctx->last_slot = (int)(&sl - ctx->slots);
  if (info) { info->error_flags = sl.h_info->flag; info->counters = k; info->timings = t; }
  return error_from_flag(ctx, sl.h_info->flag);
}

// every batch complete (results of un-waited tickets are in the caller's buffers; their info is dropped)
int drain_all(uavmp_ctx* ctx) {
  int rc = UAVMP_OK;
  for (PlanSlot& sl : ctx->slots) { int r = slot_finish(ctx, sl, nullptr); if (r && !rc) rc = r; }
  return rc;
}

// d_occ / d_cloud are in place: record the geometry and build the derived structures (flag grid, cell list, tensor map)
int uavmp_map_commit(uavmp_ctx* ctx, int nx, int ny, int nz, const double origin[3], const double map_size[3], double resolution,
                     int n_cloud) {
  ctx->nx = nx; ctx->ny = ny; ctx->nz = nz; ctx->n_cloud = n_cloud; ctx->resolution = resolution;
  for (int i = 0; i < 3; i++) { ctx->origin[i] = origin[i]; ctx->map_size[i] = map_size[i]; }
  ctx->have_map = true;
  ctx->flags_dirty = true;
  if (ctx->params_dirty) { int r = kino_upload_params(ctx); if (r) return r; }
  return kino_build_map(ctx);
}

// geometry the lookups rely on: in_map() bounds positions by origin + map_size, indexing uses nx / ny / nz
int uavmp_map_check_geometry(uavmp_ctx* ctx, int nx, int ny, int nz, const double origin[3], const double map_size[3], double resolution) {
  if (!origin || !map_size) return uavmp_fail(ctx, UAVMP_EINVAL, "origin / map_size is NULL");
  const int n[3] = {nx, ny, nz};
  for (int i = 0; i < 3; i++) {
    if (!(map_size[i] > 0)) return uavmp_fail(ctx, UAVMP_EINVAL, "map_size must be > 0");
    // the reference derives voxel_num = ceil(map_size / resolution) (grid_map.cpp:56-58): fewer voxels than that would let an
    // in-map position index past the grid
    if (map_size[i] > n[i] * resolution * (1.0 + 1e-9))
      return uavmp_fail(ctx, UAVMP_EINVAL, "axis %d: %d voxels of %g m do not cover map_size %g (expect ceil(map_size / resolution))", i,
                        n[i], resolution, map_size[i]);
  }
  return UAVMP_OK;
}

extern "C" {

const char* uavmp_version(void) { return "uavmp-b200 0.2 (sm_100a)"; }

void uavmp_kino_params_default(uavmp_kino_params* p) {  // kino_astar.cpp:8-19
  p->allocated_node_num = 100000; p->collision_check_type = 1; p->rou_time = 1.0; p->lambda_heu = 2.0;
  p->goal_tolerance = 2.0; p->time_step_size = 0.1; p->max_velocity = 5.0; p->max_accelration = 7.0;
  p->acc_resolution = 2.0; p->sample_tau = 0.5; p->robot_r = 0.2; p->robot_h = 0.1;
}
void uavmp_kino_params_launch(uavmp_kino_params* p) {  // test_kino_astar_searching.launch:44-57
  p->allocated_node_num = 100000; p->collision_check_type = 1; p->rou_time = 50.0; p->lambda_heu = 3.0;
  p->goal_tolerance = 2.0; p->time_step_size = 0.075; p->max_velocity = 7.0; p->max_accelration = 10.0;
  p->acc_resolution = 4.0; p->sample_tau = 0.3; p->robot_r = 0.4; p->robot_h = 0.1;
}
void uavmp_osqp_settings_default(uavmp_osqp_settings* s) {
  // osqp_api_constants.h:96-153 with minimum_control.cpp:160-162's overrides
  s->rho = 0.1; s->sigma = 1e-6; s->alpha = 1.6; s->eps_abs = 1e-3; s->eps_rel = 1e-3; s->eps_prim_inf = 1e-3;
  s->eps_dual_inf = 1e-4; s->max_iter = 1000; s->check_termination = 25; s->scaling = 10; s->adaptive_rho = 1;
  s->adaptive_rho_interval = 0; s->adaptive_rho_tolerance = 5.0;
}

int uavmp_ctx_create(uavmp_ctx** out, int device) {
  if (!out) return UAVMP_EINVAL;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0) {
    fprintf(stderr, "uavmp: no CUDA device (%s) — this library has no CPU fallback\n", cudaGetErrorString(e));
    return UAVMP_ECUDA;
  }
  if (device < 0 || device >= ndev) return UAVMP_EINVAL;
  if (cudaSetDevice(device) != cudaSuccess) return UAVMP_ECUDA;
  uavmp_ctx* ctx = new uavmp_ctx();
  ctx->device = device;
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  ctx->sm_count = prop.multiProcessorCount;
  bool ok = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) == cudaSuccess;
  for (PlanSlot& sl : ctx->slots) {
    ok = ok && cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; i < 5; i++) ok = ok && cudaEventCreate(&sl.ev[i]) == cudaSuccess;
  }
  for (int i = 0; i < 8; i++) ok = ok && cudaEventCreate(&ctx->ev[i]) == cudaSuccess;
  if (!ok) { fprintf(stderr, "uavmp: cannot create CUDA streams / events\n"); delete ctx; return UAVMP_ECUDA; }
  uavmp_kino_params_launch(&ctx->kp);
  memset(&ctx->tm, 0, sizeof(ctx->tm));
  memset(&ctx->last_counters, 0, sizeof(ctx->last_counters));
  memset(&ctx->map_host, 0, sizeof(ctx->map_host));
  *out = ctx;
  return UAVMP_OK;
}

void uavmp_ctx_destroy(uavmp_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  for (PlanSlot& sl : ctx->slots) cudaStreamSynchronize(sl.stream);
  cudaStreamSynchronize(ctx->stream);
  void* ptrs[] = {ctx->d_kparams, ctx->d_lattice, ctx->d_occ, ctx->d_flags, ctx->d_tmp, ctx->d_cloud, ctx->d_cell_start,
                  ctx->d_pts, ctx->d_map, ctx->d_arena_mem, ctx->d_arenas, ctx->d_arena_busy, ctx->d_path_packed,
                  ctx->qp_scr.ws, ctx->qp_scr.tab, ctx->qp_scr.tmp, ctx->d_qp_in, ctx->d_qp_out, ctx->d_qp_int, ctx->d_phase, ctx->d_query_cycles,
                  ctx->d_flags_pad, ctx->d_b3f};
  for (void* p : ptrs) if (p) cudaFree(p);
  for (PlanSlot& sl : ctx->slots) {
    kino_free_slot(sl);
    if (sl.h_info) cudaFreeHost(sl.h_info);
    for (int i = 0; i < 5; i++) cudaEventDestroy(sl.ev[i]);
    cudaStreamDestroy(sl.stream);
  }
  qp_free_plans(ctx);
  astar_destroy(ctx);
  rrt_destroy(ctx);
  for (int i = 0; i < 8; i++) cudaEventDestroy(ctx->ev[i]);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* uavmp_last_error(const uavmp_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
void* uavmp_ctx_stream(uavmp_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
int uavmp_ctx_sync(uavmp_ctx* ctx) {
  // everything issued so far — including batches still in flight — is complete when this returns; an error flag raised by
  // an asynchronous batch (uavmp_plan_batch_dev / an un-waited uavmp_plan_submit ticket) is reported here
  if (!ctx) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  int rc = drain_all(ctx);
  UAVMP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return rc;
}

int uavmp_kino_set_params(uavmp_ctx* ctx, const uavmp_kino_params* p) {
  if (!ctx || !p) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  drain_all(ctx);  // the parameter block and the lattice tables are shared by every batch in flight
  ctx->kp = *p;
  ctx->params_dirty = true;
  return kino_upload_params(ctx);
}

int uavmp_kino_set_path_cap(uavmp_ctx* ctx, int points) {
  if (!ctx || points < 16) return UAVMP_EINVAL;
  drain_all(ctx);
  ctx->path_cap = points;  // the slots re-allocate their path stage on the next call
  return UAVMP_OK;
}

int uavmp_map_set(uavmp_ctx* ctx, const int8_t* occ, int nx, int ny, int nz, const double origin[3],
                  const double map_size[3], double resolution, const float* cloud_xyz, int n_cloud) {
  if (!ctx || !occ || nx <= 0 || ny <= 0 || nz <= 0 || !(resolution > 0) || n_cloud < 0) return UAVMP_EINVAL;
  if (n_cloud > 0 && !cloud_xyz) return UAVMP_EINVAL;
  if (nx >= (1 << 17) || ny >= (1 << 17) || nz >= (1 << 17)) return uavmp_fail(ctx, UAVMP_EINVAL, "grid dimension too large");
  int r = uavmp_map_check_geometry(ctx, nx, ny, nz, origin, map_size, resolution);
  if (r) return r;
  cudaSetDevice(ctx->device);
  drain_all(ctx);
  const size_t nvox = (size_t)nx * ny * nz;
  if (ctx->d_occ) { cudaFree(ctx->d_occ); ctx->d_occ = nullptr; }
  if (ctx->d_flags) { cudaFree(ctx->d_flags); ctx->d_flags = nullptr; }
  if (ctx->d_tmp) { cudaFree(ctx->d_tmp); ctx->d_tmp = nullptr; }
  if (ctx->d_cloud) { cudaFree(ctx->d_cloud); ctx->d_cloud = nullptr; }
  ctx->have_map = false;
  UAVMP_CUDA(ctx, cudaMalloc(&ctx->d_occ, nvox));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(ctx->d_occ, occ, nvox, cudaMemcpyHostToDevice, ctx->stream));
  if (n_cloud > 0) {
    UAVMP_CUDA(ctx, cudaMalloc(&ctx->d_cloud, (size_t)n_cloud * 3 * sizeof(float)));
    UAVMP_CUDA(ctx, cudaMemcpyAsync(ctx->d_cloud, cloud_xyz, (size_t)n_cloud * 3 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  }
  return uavmp_map_commit(ctx, nx, ny, nz, origin, map_size, resolution, n_cloud);
}

static int prepare_search(uavmp_ctx* ctx) {
  if (!ctx->have_map) return uavmp_fail(ctx, UAVMP_ESTATE, "uavmp_map_set has not been called");
  if (ctx->params_dirty) { drain_all(ctx); int r = kino_upload_params(ctx); if (r) return r; }
  if (ctx->flags_dirty) { drain_all(ctx); int r = kino_build_map(ctx); if (r) return r; }
  if (ctx->kp.collision_check_type == 2 && ctx->n_cloud == 0)
    return uavmp_fail(ctx, UAVMP_ESTATE, "collision_check_type 2 needs a cloud");
  return kino_ensure_arenas(ctx);
}

// the batch's error flag and counters travel to pinned host memory at the end of the slot's stream work
static int slot_record_info(uavmp_ctx* ctx, PlanSlot& sl) {
  UAVMP_CUDA(ctx, cudaMemcpyAsync(&sl.h_info->flag, sl.d_misc, sizeof(int), cudaMemcpyDeviceToHost, sl.stream));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(sl.h_info->counters, sl.d_counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, sl.stream));
  UAVMP_CUDA(ctx, cudaEventRecord(sl.ev[4], sl.stream));
  return UAVMP_OK;
}

long long uavmp_kino_search_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* start_vel,
                                  const double* end_pt, const double* end_vel, int* status, int* use_node_num,
                                  long long* path_offsets, uint64_t* pop_hash, int* n_pop) {
  if (!ctx || B <= 0 || !start_pt || !start_vel || !end_pt || !end_vel || !status) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  int r = prepare_search(ctx);
  if (r) return r;
  PlanSlot& sl = ctx->slots[0];
  slot_finish(ctx, sl, nullptr);
  r = kino_ensure_slot(ctx, sl, B);
  if (r) return r;
  cudaStream_t st = sl.stream;
  const size_t nb = (size_t)B * 3 * sizeof(double);
  double* d = sl.d_q;
  cudaEventRecord(sl.ev[0], st);
  UAVMP_CUDA(ctx, cudaMemcpyAsync(d, start_pt, nb, cudaMemcpyHostToDevice, st));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(d + 3 * (size_t)B, start_vel, nb, cudaMemcpyHostToDevice, st));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(d + 6 * (size_t)B, end_pt, nb, cudaMemcpyHostToDevice, st));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(d + 9 * (size_t)B, end_vel, nb, cudaMemcpyHostToDevice, st));
  cudaEventRecord(sl.ev[1], st);
  sl.launches_qp = 0;
  r = kino_launch_search(ctx, sl, B, d, d + 3 * (size_t)B, d + 6 * (size_t)B, d + 9 * (size_t)B, true, ctx->profile_phases,
                         nullptr, nullptr, nullptr);
  if (r) return r;
  cudaEventRecord(sl.ev[2], st);
  cudaEventRecord(ctx->ev[0], st);
  r = kino_pack_paths(ctx, sl, B);
  if (r) return r;
  cudaEventRecord(ctx->ev[1], st);
  UAVMP_CUDA(ctx, cudaMemcpyAsync(status, sl.d_status, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  if (use_node_num) UAVMP_CUDA(ctx, cudaMemcpyAsync(use_node_num, sl.d_use, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  if (path_offsets) UAVMP_CUDA(ctx, cudaMemcpyAsync(path_offsets, sl.d_offsets, (size_t)(B + 1) * sizeof(long long), cudaMemcpyDeviceToHost, st));
  if (pop_hash) UAVMP_CUDA(ctx, cudaMemcpyAsync(pop_hash, sl.d_hash, (size_t)B * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
  if (n_pop) UAVMP_CUDA(ctx, cudaMemcpyAsync(n_pop, sl.d_npop, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  cudaEventRecord(sl.ev[3], st);
  r = slot_record_info(ctx, sl);
  if (r) return r;
  sl.in_flight = true; sl.B = B; sl.ticket = -1;
  r = slot_finish(ctx, sl, nullptr);
  cudaEventElapsedTime(&ctx->tm.path_ms, ctx->ev[0], ctx->ev[1]);
  if (r) return r;
  return ctx->last_total_path;
}

int uavmp_kino_get_paths(uavmp_ctx* ctx, double* path_xyz, long long cap_points) {
  if (!ctx || !path_xyz) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  if (cap_points < ctx->last_total_path) return uavmp_fail(ctx, UAVMP_ECAP, "path buffer too small");
  cudaStream_t st = ctx->slots[0].stream;
  if (ctx->last_total_path > 0)
    UAVMP_CUDA(ctx, cudaMemcpyAsync(path_xyz, ctx->d_path_packed, (size_t)ctx->last_total_path * 3 * sizeof(double), cudaMemcpyDeviceToHost, st));
  UAVMP_CUDA(ctx, cudaStreamSynchronize(st));
  return UAVMP_OK;
}

int uavmp_kino_set_trace(uavmp_ctx* ctx, int pop_cap) {
  if (!ctx || pop_cap < 0) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  drain_all(ctx);
  ctx->pop_cap = pop_cap;  // the slots re-allocate their buffers on the next call
  return UAVMP_OK;
}

int uavmp_kino_get_trace(uavmp_ctx* ctx, int q, int32_t* pop_idx_xyz, int cap) {
  if (!ctx || !pop_idx_xyz) return UAVMP_EINVAL;
  PlanSlot& sl = ctx->slots[0];
  if (q < 0 || q >= sl.B) return UAVMP_EINVAL;
  if (!sl.d_trace || sl.pop_cap <= 0) return uavmp_fail(ctx, UAVMP_ESTATE, "tracing is off");
  cudaSetDevice(ctx->device);
  int n = std::min(cap, sl.pop_cap);
  UAVMP_CUDA(ctx, cudaMemcpyAsync(pop_idx_xyz, sl.d_trace + (size_t)q * sl.pop_cap * 3, (size_t)n * 3 * sizeof(int), cudaMemcpyDeviceToHost, sl.stream));
  UAVMP_CUDA(ctx, cudaStreamSynchronize(sl.stream));
  return UAVMP_OK;
}

int uavmp_kino_get_counters(uavmp_ctx* ctx, uavmp_kino_counters* out) {
  // counters of the most recently COMPLETED batch (a synchronous call, or the last ticket uavmp_plan_wait returned)
  if (!ctx || !out) return UAVMP_EINVAL;
  *out = ctx->last_counters;
  return UAVMP_OK;
}

int uavmp_kino_set_profile(uavmp_ctx* ctx, int on) {
  if (!ctx) return UAVMP_EINVAL;
  ctx->profile_phases = on != 0;
  return UAVMP_OK;
}

int uavmp_kino_get_profile(uavmp_ctx* ctx, unsigned long long phase_cycles[16], long long* query_cycles, int cap, int* grid) {
  if (!ctx || !phase_cycles) return UAVMP_EINVAL;
  if (!ctx->d_phase) return uavmp_fail(ctx, UAVMP_ESTATE, "profiling was off for the last search");
  cudaSetDevice(ctx->device);
  PlanSlot& sl = ctx->slots[0];
  UAVMP_CUDA(ctx, cudaMemcpyAsync(phase_cycles, ctx->d_phase, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, sl.stream));
  // cap >= 17 * B: the B per-query totals followed by the B x 16 per-query phase cycles; else only the totals
  if (query_cycles && cap > 0) {
    const size_t nq = (cap >= 17 * sl.B) ? (size_t)17 * sl.B : (size_t)std::min(cap, sl.B);
    UAVMP_CUDA(ctx, cudaMemcpyAsync(query_cycles, ctx->d_query_cycles, nq * sizeof(long long), cudaMemcpyDeviceToHost, sl.stream));
  }
  UAVMP_CUDA(ctx, cudaStreamSynchronize(sl.stream));
  if (grid) *grid = ctx->last_grid;
  return UAVMP_OK;
}

int uavmp_get_timings(uavmp_ctx* ctx, uavmp_timings* out) {
  if (!ctx || !out) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  // uavmp_plan_batch_dev is asynchronous: its batch (slot 0) is resolved here
  if (ctx->slots[0].in_flight && ctx->slots[0].ticket < 0) slot_finish(ctx, ctx->slots[0], nullptr);
  *out = ctx->tm;
  return UAVMP_OK;
}

int uavmp_fpmath_eval(uavmp_ctx* ctx, int op, int n_pow, const double* x, double* y, long long n) {
  if (!ctx || !x || !y || n <= 0) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  return kino_fpmath_eval(ctx, op, n_pow, x, y, n);
}

// ---- grid A* ---------------------------------------------------------------------------------------------
int uavmp_astar_set_params(uavmp_ctx* ctx, double lambda_heu, int allocated_node_num, int path_cap_nodes) {
  if (!ctx || allocated_node_num < 2 || path_cap_nodes < 2 || !(lambda_heu >= 0.0)) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  ctx->astar_lambda = lambda_heu; ctx->astar_allocated = allocated_node_num; ctx->astar_path_cap = path_cap_nodes;
  return UAVMP_OK;
}

long long uavmp_astar_search_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* end_pt, int* status,
                                   int* use_node_num, long long* path_offsets, uint64_t* pop_hash, int* n_pop) {
  if (!ctx || B <= 0 || !start_pt || !end_pt || !status) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  if (!ctx->have_map) return uavmp_fail(ctx, UAVMP_ESTATE, "uavmp_map_set has not been called");
  drain_all(ctx);
  return astar_search_batch(ctx, B, start_pt, end_pt, status, use_node_num, path_offsets, pop_hash, n_pop);
}

int uavmp_astar_get_paths(uavmp_ctx* ctx, double* path_xyz, long long cap_points) {
  if (!ctx || !path_xyz) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  return astar_get_paths(ctx, path_xyz, cap_points);
}

int uavmp_rrt_set_params(uavmp_ctx* ctx, int max_tree_node_num, double step_length, double search_radius,
                         double collision_check_resolution, double sample_budget, int path_cap_nodes) {
  if (!ctx || max_tree_node_num < 1 || path_cap_nodes < 2 || !(step_length > 0.0) || !(search_radius > 0.0) ||
      !(collision_check_resolution > 0.0) || !(sample_budget >= 0.0))
    return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  ctx->rrt_max_nodes = max_tree_node_num; ctx->rrt_step = step_length; ctx->rrt_radius = search_radius;
  ctx->rrt_ccres = collision_check_resolution; ctx->rrt_budget = sample_budget; ctx->rrt_path_cap = path_cap_nodes;
  return UAVMP_OK;
}

uint32_t uavmp_rrt_sample_seed(uint64_t query_seed, long long i) { return rrt_sample_seed_host(query_seed, i); }

long long uavmp_rrt_search_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* end_pt, const uint64_t* query_seed,
                                 int* status, int* use_node_num, long long* n_samples, double* goal_g_cost, uint64_t* tree_digest,
                                 long long* path_offsets) {
  if (!ctx || B <= 0 || !start_pt || !end_pt || !query_seed || !status) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  if (!ctx->have_map) return uavmp_fail(ctx, UAVMP_ESTATE, "uavmp_map_set has not been called");
  drain_all(ctx);
  return rrt_search_batch(ctx, B, start_pt, end_pt, query_seed, status, use_node_num, n_samples, goal_g_cost, tree_digest, path_offsets);
}

int uavmp_rrt_get_paths(uavmp_ctx* ctx, double* path_xyz, long long cap_points) {
  if (!ctx || !path_xyz) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  return rrt_get_paths(ctx, path_xyz, cap_points);
}

// ---- hot path (b) --------------------------------------------------------------------------------------

int uavmp_minctrl_solve_batch(uavmp_ctx* ctx, int order, int S, int B, const double* pos_1d, const double* bound_vel,
                              const double* bound_acc, const double* bound_jerk, const double* time_vec,
                              const uavmp_osqp_settings* settings, double* coef, int* solved, int* osqp_status,
                              int* iters) {
  return uavmp_minctrl_solve_corridor_batch(ctx, order, S, 0, B, pos_1d, bound_vel, bound_acc, bound_jerk, time_vec, nullptr, nullptr,
                                            settings, coef, solved, osqp_status, iters);
}

int uavmp_minctrl_solve_corridor_batch(uavmp_ctx* ctx, int order, int S, int Kc, int B, const double* pos_1d,
                                       const double* bound_vel, const double* bound_acc, const double* bound_jerk,
                                       const double* time_vec, const double* corridor_lo, const double* corridor_hi,
                                       const uavmp_osqp_settings* settings, double* coef, int* solved, int* osqp_status,
                                       int* iters) {
  if (!ctx || B <= 0 || S <= 0 || !pos_1d || !bound_vel || !bound_acc || !time_vec || !coef) return UAVMP_EINVAL;
  if (Kc < 0 || Kc > 8) return uavmp_fail(ctx, UAVMP_EINVAL, "n_corridor must be in [0, 8]");
  if (Kc > 0 && (!corridor_lo || !corridor_hi)) return uavmp_fail(ctx, UAVMP_EINVAL, "n_corridor > 0 needs corridor_lo / corridor_hi");
  if (Kc > 0)  // osqp_setup rejects l > u (auxil.c:856-921): "solver init failed" for the whole call, like validate_data
    for (size_t i = 0; i < (size_t)B * S; i++)
      if (!(corridor_lo[i] <= corridor_hi[i])) return uavmp_fail(ctx, UAVMP_EINVAL, "corridor_lo > corridor_hi at entry %zu", i);
  if (order != 5 && order != 7) return uavmp_fail(ctx, UAVMP_EINVAL, "order must be 5 (jerk) or 7 (snap)");
  if (order == 7 && !bound_jerk) return uavmp_fail(ctx, UAVMP_EINVAL, "order 7 needs bound_jerk");
  cudaSetDevice(ctx->device);
  uavmp_osqp_settings def;
  if (!settings) { uavmp_osqp_settings_default(&def); settings = &def; }
  cudaStream_t st = ctx->stream;
  const int n = (order + 1) * S;
  const size_t in_d = (size_t)B * ((S + 1) + 6 + S + 2 * S);
  int r = ensure_bytes(ctx, (void**)&ctx->d_qp_in, &ctx->qp_in_bytes, in_d * sizeof(double)); if (r) return r;
  r = ensure_bytes(ctx, (void**)&ctx->d_qp_out, &ctx->qp_out_bytes, (size_t)B * n * sizeof(double)); if (r) return r;
  r = ensure_bytes(ctx, (void**)&ctx->d_qp_int, &ctx->qp_int_bytes, (size_t)B * 3 * sizeof(int)); if (r) return r;
  double* d_pos = ctx->d_qp_in; double* d_bv = d_pos + (size_t)B * (S + 1); double* d_ba = d_bv + 2 * (size_t)B;
  double* d_bj = d_ba + 2 * (size_t)B; double* d_T = d_bj + 2 * (size_t)B;
  double* d_lo = d_T + (size_t)B * S; double* d_hi = d_lo + (size_t)B * S;
  cudaEventRecord(ctx->ev[0], st);
  UAVMP_CUDA(ctx, cudaMemcpyAsync(d_pos, pos_1d, (size_t)B * (S + 1) * sizeof(double), cudaMemcpyHostToDevice, st));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(d_bv, bound_vel, (size_t)B * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(d_ba, bound_acc, (size_t)B * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
  if (order == 7) UAVMP_CUDA(ctx, cudaMemcpyAsync(d_bj, bound_jerk, (size_t)B * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(d_T, time_vec, (size_t)B * S * sizeof(double), cudaMemcpyHostToDevice, st));
  if (Kc > 0) {
    UAVMP_CUDA(ctx, cudaMemcpyAsync(d_lo, corridor_lo, (size_t)B * S * sizeof(double), cudaMemcpyHostToDevice, st));
    UAVMP_CUDA(ctx, cudaMemcpyAsync(d_hi, corridor_hi, (size_t)B * S * sizeof(double), cudaMemcpyHostToDevice, st));
  }
  cudaEventRecord(ctx->ev[1], st);
  int* d_solved = ctx->d_qp_int; int* d_stat = d_solved + B; int* d_it = d_stat + B;
  int launches = 0;
  r = qp_solve_batch_dev(ctx, st, ctx->qp_scr, &launches, order, S, Kc, B, d_pos, d_bv, d_ba, order == 7 ? d_bj : nullptr, d_T,
                         d_lo, d_hi, settings, ctx->d_qp_out, d_solved, d_stat, d_it);
  if (r) return r;
  cudaEventRecord(ctx->ev[2], st);
  UAVMP_CUDA(ctx, cudaMemcpyAsync(coef, ctx->d_qp_out, (size_t)B * n * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (solved) UAVMP_CUDA(ctx, cudaMemcpyAsync(solved, d_solved, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  if (osqp_status) UAVMP_CUDA(ctx, cudaMemcpyAsync(osqp_status, d_stat, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  if (iters) UAVMP_CUDA(ctx, cudaMemcpyAsync(iters, d_it, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  cudaEventRecord(ctx->ev[3], st);
  UAVMP_CUDA(ctx, cudaStreamSynchronize(st));
  memset(&ctx->tm, 0, sizeof(ctx->tm));
  cudaEventElapsedTime(&ctx->tm.h2d_ms, ctx->ev[0], ctx->ev[1]);
  cudaEventElapsedTime(&ctx->tm.qp_ms, ctx->ev[1], ctx->ev[2]);
  cudaEventElapsedTime(&ctx->tm.d2h_ms, ctx->ev[2], ctx->ev[3]);
  cudaEventElapsedTime(&ctx->tm.total_ms, ctx->ev[0], ctx->ev[3]);
  ctx->tm.qp_launches = launches;
  return UAVMP_OK;
}

int uavmp_minctrl_solve_ragged_batch(uavmp_ctx* ctx, int order, int B, const int* S, const double* pos_1d, const double* bound_vel,
                                     const double* bound_acc, const double* bound_jerk, const double* time_vec,
                                     const uavmp_osqp_settings* settings, double* coef, int* solved, int* osqp_status, int* iters) {
  if (!ctx || B <= 0 || !S || !pos_1d || !bound_vel || !bound_acc || !time_vec || !coef) return UAVMP_EINVAL;
  if (order != 5 && order != 7) return uavmp_fail(ctx, UAVMP_EINVAL, "order must be 5 (jerk) or 7 (snap)");
  if (order == 7 && !bound_jerk) return uavmp_fail(ctx, UAVMP_EINVAL, "order 7 needs bound_jerk");
  long long sumS = 0;
  for (int b = 0; b < B; b++) {
    if (S[b] < 1) return uavmp_fail(ctx, UAVMP_EINVAL, "S[%d] = %d: every problem needs at least one segment", b, S[b]);
    sumS += S[b];
  }
  uavmp_osqp_settings def;
  if (!settings) { uavmp_osqp_settings_default(&def); settings = &def; }
  if (settings->max_iter <= 0 || settings->check_termination < 0 || settings->scaling < 0)
    return uavmp_fail(ctx, UAVMP_EINVAL, "bad OSQP settings");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  const size_t n_pos = (size_t)(sumS + B), n_coef = (size_t)(order + 1) * sumS;
  int r = ensure_bytes(ctx, (void**)&ctx->d_qp_in, &ctx->qp_in_bytes, (n_pos + 6 * (size_t)B + sumS) * sizeof(double)); if (r) return r;
  r = ensure_bytes(ctx, (void**)&ctx->d_qp_out, &ctx->qp_out_bytes, n_coef * sizeof(double)); if (r) return r;
  r = ensure_bytes(ctx, (void**)&ctx->d_qp_int, &ctx->qp_int_bytes, (size_t)B * 3 * sizeof(int)); if (r) return r;
  double* d_pos = ctx->d_qp_in; double* d_bv = d_pos + n_pos; double* d_ba = d_bv + 2 * (size_t)B; double* d_bj = d_ba + 2 * (size_t)B;
  double* d_T = d_bj + 2 * (size_t)B;
  int* d_solved = ctx->d_qp_int; int* d_stat = d_solved + B; int* d_it = d_stat + B;
  cudaEventRecord(ctx->ev[0], st);
  UAVMP_CUDA(ctx, cudaMemcpyAsync(d_pos, pos_1d, n_pos * sizeof(double), cudaMemcpyHostToDevice, st));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(d_bv, bound_vel, (size_t)B * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(d_ba, bound_acc, (size_t)B * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
  if (order == 7) UAVMP_CUDA(ctx, cudaMemcpyAsync(d_bj, bound_jerk, (size_t)B * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(d_T, time_vec, (size_t)sumS * sizeof(double), cudaMemcpyHostToDevice, st));
  cudaEventRecord(ctx->ev[1], st);
  QpRaggedIo io;
  io.pos = d_pos; io.bv = d_bv; io.ba = d_ba; io.bj = order == 7 ? d_bj : nullptr; io.T = d_T;
  io.coef = ctx->d_qp_out; io.solved = d_solved; io.status = d_stat; io.iters = d_it; io.seg_off = nullptr; io.order = order;
  int launches = 0, aux = 0;
  r = qp_solve_ragged_dev(ctx, st, ctx->qp_scr, order, B, S, io, settings, &launches, &aux, nullptr, nullptr);
  if (r) return r;
  cudaEventRecord(ctx->ev[2], st);
  UAVMP_CUDA(ctx, cudaMemcpyAsync(coef, ctx->d_qp_out, n_coef * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (solved) UAVMP_CUDA(ctx, cudaMemcpyAsync(solved, d_solved, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  if (osqp_status) UAVMP_CUDA(ctx, cudaMemcpyAsync(osqp_status, d_stat, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  if (iters) UAVMP_CUDA(ctx, cudaMemcpyAsync(iters, d_it, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  cudaEventRecord(ctx->ev[3], st);
  UAVMP_CUDA(ctx, cudaStreamSynchronize(st));
  memset(&ctx->tm, 0, sizeof(ctx->tm));
  cudaEventElapsedTime(&ctx->tm.h2d_ms, ctx->ev[0], ctx->ev[1]);
  cudaEventElapsedTime(&ctx->tm.qp_ms, ctx->ev[1], ctx->ev[2]);
  cudaEventElapsedTime(&ctx->tm.d2h_ms, ctx->ev[2], ctx->ev[3]);
  cudaEventElapsedTime(&ctx->tm.total_ms, ctx->ev[0], ctx->ev[3]);
  ctx->tm.qp_launches = launches;
  ctx->tm.aux_launches = aux;
  return UAVMP_OK;
}

// ---- RRT* -> minimum jerk (test_minimum_jerk.cpp GoalCallback, batched) ------------------------------------------------------
long long uavmp_rrt_plan_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* start_vel, const double* end_pt,
                               const uint64_t* query_seed, int order, double seg_time, const uavmp_osqp_settings* settings,
                               int* search_status, int* n_segments, int* qp_solved, long long* coef_offsets, int* osqp_status,
                               int* iters) {
  if (!ctx || B <= 0 || !start_pt || !end_pt || !query_seed || !search_status || !n_segments || !qp_solved) return UAVMP_EINVAL;
  if (order != 5 && order != 7) return uavmp_fail(ctx, UAVMP_EINVAL, "order must be 5 (jerk) or 7 (snap)");
  if (!(seg_time > 0.0)) return uavmp_fail(ctx, UAVMP_EINVAL, "seg_time must be > 0");
  uavmp_osqp_settings def;
  if (!settings) { uavmp_osqp_settings_default(&def); settings = &def; }
  if (settings->max_iter <= 0 || settings->check_termination < 0 || settings->scaling < 0)
    return uavmp_fail(ctx, UAVMP_EINVAL, "bad OSQP settings");
  cudaSetDevice(ctx->device);
  if (!ctx->have_map) return uavmp_fail(ctx, UAVMP_ESTATE, "uavmp_map_set has not been called");
  drain_all(ctx);
  return rrt_plan_batch(ctx, B, start_pt, start_vel, end_pt, query_seed, order, seg_time, settings, search_status, n_segments, qp_solved,
                        coef_offsets, osqp_status, iters);
}

int uavmp_rrt_plan_get_coef(uavmp_ctx* ctx, double* coef, long long cap) {
  if (!ctx || !coef) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  return rrt_plan_get_coef(ctx, coef, cap);
}

// ---- pipeline ---------------------------------------------------------------------------------------------
// Issue one batch of the search -> waypoints -> 3 x QP pipeline on slot `sl` (asynchronous).  host_io: the pointers are host
// memory and the copies are part of the batch; otherwise they are device memory and the batch is ordered after everything
// submitted to the context's stream so far.
static int plan_issue(uavmp_ctx* ctx, PlanSlot& sl, int B, const double* sp, const double* sv, const double* ep, const double* ev,
                      const uavmp_plan_options& opt, const uavmp_osqp_settings* settings, bool host_io, int* status,
                      int* qp_solved, double* coef) {
  const int order = opt.order, S = opt.S, Kc = opt.corridor_samples;
  if (order != 5 && order != 7) return uavmp_fail(ctx, UAVMP_EINVAL, "order must be 5 or 7");
  if (S <= 0) return uavmp_fail(ctx, UAVMP_EINVAL, "S must be > 0");
  if (Kc < 0 || Kc > 8 || !(opt.corridor_margin >= 0.0)) return uavmp_fail(ctx, UAVMP_EINVAL, "corridor_samples must be in [0, 8] and corridor_margin >= 0");
  if (!opt.time_alloc && !(opt.seg_time > 0.0)) return uavmp_fail(ctx, UAVMP_EINVAL, "seg_time must be > 0");
  uavmp_osqp_settings def;
  if (!settings) { uavmp_osqp_settings_default(&def); settings = &def; }
  if (settings->max_iter <= 0 || settings->check_termination < 0 || settings->scaling < 0)
    return uavmp_fail(ctx, UAVMP_EINVAL, "bad OSQP settings");
  int r = prepare_search(ctx);
  if (r) return r;
  r = kino_ensure_slot(ctx, sl, B);
  if (r) return r;
  const QpPlanDev* plan = nullptr;
  r = qp_get_plan_dev(ctx, order, S, Kc, &plan);
  if (r) return r;
  const int n = (order + 1) * S;
  const size_t nB = (size_t)3 * B;
  r = ensure_bytes(ctx, (void**)&sl.d_wp, &sl.wp_bytes, nB * ((S + 1) + 6 + S + 2 * S) * sizeof(double)); if (r) return r;
  r = ensure_bytes(ctx, (void**)&sl.d_qp_int, &sl.qp_int_bytes, nB * 3 * sizeof(int)); if (r) return r;
  if (host_io) {
    r = ensure_bytes(ctx, (void**)&sl.d_plan_out, &sl.plan_out_bytes, (size_t)B * 3 * n * sizeof(double)); if (r) return r;
    r = ensure_bytes(ctx, (void**)&sl.d_plan_io, &sl.plan_io_bytes, (size_t)B * 2 * sizeof(int)); if (r) return r;
  }
  // in-kernel QP: how many warp workspaces fit in the shared memory the search gives up between two queries
  const int ws_bytes = plan->ws_warp * (int)sizeof(double);
  const int idx_bytes = plan->n_sidx * (int)sizeof(unsigned short);  // the solves' index block, staged once per round
  int warps = plan->n_sidx > 0 ? std::min(8, (kino_qp_overlay_bytes() - idx_bytes) / ws_bytes) : 0;
  if (warps < 0) warps = 0;
  if (getenv("UAVMP_NO_FUSE")) warps = 0;
  if (warps == 0) { r = ensure_bytes(ctx, (void**)&sl.d_qp_out, &sl.qp_out_bytes, nB * n * sizeof(double)); if (r) return r; }

  cudaStream_t st = sl.stream;
  const double *d_sp = sp, *d_sv = sv, *d_ep = ep, *d_ev = ev;
  double* d_coef = coef; int* d_solved = qp_solved;
  cudaEventRecord(sl.ev[0], st);
  if (host_io) {
    const size_t nb = (size_t)B * 3 * sizeof(double);
    double* d = sl.d_q;
    UAVMP_CUDA(ctx, cudaMemcpyAsync(d, sp, nb, cudaMemcpyHostToDevice, st));
    UAVMP_CUDA(ctx, cudaMemcpyAsync(d + 3 * (size_t)B, sv, nb, cudaMemcpyHostToDevice, st));
    UAVMP_CUDA(ctx, cudaMemcpyAsync(d + 6 * (size_t)B, ep, nb, cudaMemcpyHostToDevice, st));
    UAVMP_CUDA(ctx, cudaMemcpyAsync(d + 9 * (size_t)B, ev, nb, cudaMemcpyHostToDevice, st));
    d_sp = d; d_sv = d + 3 * (size_t)B; d_ep = d + 6 * (size_t)B; d_ev = d + 9 * (size_t)B;
    d_coef = sl.d_plan_out; d_solved = sl.d_plan_io + B;
  } else {
    // device inputs: ordered after the work already submitted to the context's stream
    UAVMP_CUDA(ctx, cudaEventRecord(ctx->ev[7], ctx->stream));
    UAVMP_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev[7], 0));
  }
  cudaEventRecord(sl.ev[1], st);
  double* pos = sl.d_wp; double* bv = pos + nB * (S + 1); double* ba = bv + nB * 2; double* bj = ba + nB * 2; double* T = bj + nB * 2;
  double* lo = T + nB * S; double* hi = lo + nB * S;
  int* d_solved3 = sl.d_qp_int; int* d_stat3 = d_solved3 + nB; int* d_it3 = d_stat3 + nB;
  if (warps > 0) {
    KinoQpDev qp;
    qp.enabled = 1; qp.warps = warps; qp.Sg = S; qp.n = n; qp.seg_time = opt.seg_time;
    qp.time_alloc = opt.time_alloc; qp.step = ctx->kp.time_step_size; qp.Kc = Kc; qp.margin = opt.corridor_margin; qp.lo = lo; qp.hi = hi;
    qp.pos = pos; qp.bv = bv; qp.ba = ba; qp.bj = bj; qp.T = T;
    qp.coef = d_coef; qp.solved3 = d_solved3; qp.status3 = d_stat3; qp.iters3 = d_it3; qp.qp_solved = d_solved;
    r = kino_launch_search(ctx, sl, B, d_sp, d_sv, d_ep, d_ev, true, ctx->profile_phases && &sl == &ctx->slots[0], &qp, plan, settings);
    if (r) return r;
    sl.launches_qp = 0;  // the QP runs inside the search kernel
  } else {
    // sequential fallback (the QP workspace does not fit next to the search, or UAVMP_NO_FUSE): three more kernels on the stream
    r = kino_launch_search(ctx, sl, B, d_sp, d_sv, d_ep, d_ev, true, false, nullptr, nullptr, nullptr);
    if (r) return r;
    double *w_pos, *w_bv, *w_ba, *w_bj, *w_T, *w_lo, *w_hi;
    r = qp_waypoints_from_paths(ctx, sl, B, opt, d_sv, d_ev, &w_pos, &w_bv, &w_ba, &w_bj, &w_T, &w_lo, &w_hi);
    if (r) return r;
    int launches = 0;
    r = qp_solve_batch_dev(ctx, st, sl.qp_scr, &launches, order, S, Kc, 3 * B, w_pos, w_bv, w_ba, order == 7 ? w_bj : nullptr, w_T,
                           w_lo, w_hi, settings, sl.d_qp_out, d_solved3, d_stat3, d_it3);
    if (r) return r;
    r = qp_scatter_plan_outputs(ctx, sl, B, order, S, d_solved3, sl.d_qp_out, d_solved, d_coef);
    if (r) return r;
    sl.launches_qp = launches; sl.launches_aux += 2;  // k_waypoints, k_scatter_plan
  }
  cudaEventRecord(sl.ev[2], st);
  if (host_io) {
    UAVMP_CUDA(ctx, cudaMemcpyAsync(status, sl.d_status, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
    UAVMP_CUDA(ctx, cudaMemcpyAsync(qp_solved, d_solved, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
    UAVMP_CUDA(ctx, cudaMemcpyAsync(coef, d_coef, (size_t)B * 3 * n * sizeof(double), cudaMemcpyDeviceToHost, st));
  } else {
    UAVMP_CUDA(ctx, cudaMemcpyAsync(status, sl.d_status, (size_t)B * sizeof(int), cudaMemcpyDeviceToDevice, st));
  }
  cudaEventRecord(sl.ev[3], st);
  r = slot_record_info(ctx, sl);
  if (r) return r;
  sl.in_flight = true; sl.B = B; sl.host_io = host_io;
  return UAVMP_OK;
}

int uavmp_plan_max_in_flight(void) { return UAVMP_NSLOT - 1; }

void uavmp_plan_options_default(uavmp_plan_options* o) {
  o->order = 7; o->S = 8; o->seg_time = 1.0; o->time_alloc = 0; o->corridor_samples = 0; o->corridor_margin = 0.0;
}
static uavmp_plan_options plain_options(int order, int S, double seg_time) {
  uavmp_plan_options o;
  uavmp_plan_options_default(&o);
  o.order = order; o.S = S; o.seg_time = seg_time;
  return o;
}

int uavmp_plan_submit_opt(uavmp_ctx* ctx, int B, const double* start_pt, const double* start_vel, const double* end_pt,
                          const double* end_vel, const uavmp_plan_options* opt, const uavmp_osqp_settings* settings,
                          unsigned flags, int* search_status, int* qp_solved, double* coef, long long* ticket) {
  if (!ctx || B <= 0 || !start_pt || !start_vel || !end_pt || !end_vel || !opt || !search_status || !qp_solved || !coef || !ticket) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  PlanSlot& sl = ctx->slots[1 + ctx->next_ticket % (UAVMP_NSLOT - 1)];  // slot 0 serves the synchronous entry points
  if (sl.in_flight)
    return uavmp_fail(ctx, UAVMP_ESTATE, "%d batches are in flight: collect the oldest ticket with uavmp_plan_wait first", UAVMP_NSLOT - 1);
  int r = plan_issue(ctx, sl, B, start_pt, start_vel, end_pt, end_vel, *opt, settings, !(flags & UAVMP_PLAN_DEVICE_IO), search_status,
                     qp_solved, coef);
  if (r) return r;
  sl.ticket = ctx->next_ticket++;
  *ticket = sl.ticket;
  return UAVMP_OK;
}

int uavmp_plan_submit(uavmp_ctx* ctx, int B, const double* start_pt, const double* start_vel, const double* end_pt,
                      const double* end_vel, int order, int S, double seg_time, const uavmp_osqp_settings* settings,
                      unsigned flags, int* search_status, int* qp_solved, double* coef, long long* ticket) {
  const uavmp_plan_options o = plain_options(order, S, seg_time);
  return uavmp_plan_submit_opt(ctx, B, start_pt, start_vel, end_pt, end_vel, &o, settings, flags, search_status, qp_solved, coef, ticket);
}

static PlanSlot* find_ticket(uavmp_ctx* ctx, long long ticket) {
  if (ticket < 0) return nullptr;
  PlanSlot& sl = ctx->slots[1 + ticket % (UAVMP_NSLOT - 1)];
  return (sl.in_flight && sl.ticket == ticket) ? &sl : nullptr;
}

int uavmp_plan_wait(uavmp_ctx* ctx, long long ticket, uavmp_plan_info* info) {
  if (!ctx) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  PlanSlot* sl = find_ticket(ctx, ticket);
  if (!sl) return uavmp_fail(ctx, UAVMP_EINVAL, "unknown or already collected ticket %lld", ticket);
  return slot_finish(ctx, *sl, info);
}

int uavmp_plan_stream_wait(uavmp_ctx* ctx, long long ticket, void* cuda_stream) {
  if (!ctx) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  PlanSlot* sl = find_ticket(ctx, ticket);
  if (!sl) return uavmp_fail(ctx, UAVMP_EINVAL, "unknown or already collected ticket %lld", ticket);
  UAVMP_CUDA(ctx, cudaStreamWaitEvent((cudaStream_t)cuda_stream, sl->ev[4], 0));
  return UAVMP_OK;
}

int uavmp_plan_batch_dev(uavmp_ctx* ctx, int B, const double* d_sp, const double* d_sv, const double* d_ep,
                         const double* d_ev, int order, int S, double seg_time, const uavmp_osqp_settings* settings,
                         int* d_search_status, int* d_qp_solved, double* d_coef) {
  if (!ctx || B <= 0 || !d_sp || !d_sv || !d_ep || !d_ev || !d_search_status || !d_qp_solved || !d_coef) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  PlanSlot& sl = ctx->slots[0];
  int r = slot_finish(ctx, sl, nullptr);  // surfaces the error flag of the previous asynchronous batch on this slot
  if (r) return r;
  r = plan_issue(ctx, sl, B, d_sp, d_sv, d_ep, d_ev, plain_options(order, S, seg_time), settings, false, d_search_status, d_qp_solved, d_coef);
  if (r) return r;
  sl.ticket = -1;
  // everything submitted to the context's stream after this call sees the results
  UAVMP_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, sl.ev[4], 0));
  return UAVMP_OK;
}

int uavmp_plan_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* start_vel, const double* end_pt,
                     const double* end_vel, int order, int S, double seg_time, const uavmp_osqp_settings* settings,
                     int* search_status, int* qp_solved, double* coef) {
  if (!ctx || B <= 0 || !start_pt || !start_vel || !end_pt || !end_vel || !search_status || !qp_solved || !coef) return UAVMP_EINVAL;
  cudaSetDevice(ctx->device);
  PlanSlot& sl = ctx->slots[0];
  slot_finish(ctx, sl, nullptr);
  int r = plan_issue(ctx, sl, B, start_pt, start_vel, end_pt, end_vel, plain_options(order, S, seg_time), settings, true, search_status, qp_solved, coef);
  if (r) return r;
  sl.ticket = -1;
  return slot_finish(ctx, sl, nullptr);
}

}  // extern "C"
