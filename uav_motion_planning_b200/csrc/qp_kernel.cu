// qp_kernel.cu — K2: batched minimum-jerk / minimum-snap QP, one thread per 1-D problem, for sm_100a.
//
// Replaces traj_optimization::MinimumControl::solve (reference: src/planner/traj_optimization/src/
// minimum_control.cpp:127-192) INCLUDING the OSQP solve it delegates to, restated from the algorithm of the
// vendored OSQP 1.0.0.beta0 C sources:
//   osqp_setup  3rd/osqp/src/osqp_api.c:149-425   (Ruiz scaling scaling.c:49-165, rho vector auxil.c:75-104,
//                                                   KKT assembly algebra/_common/kkt.c, LDL' qdldl_interface.c:85-134)
//   osqp_solve  3rd/osqp/src/osqp_api.c:430-814   (ADMM steps auxil.c:135-228, residuals :247-397, infeasibility
//                                                   :399-528, termination :736-851, adaptive rho :14-73 + refactor
//                                                   osqp_api.c:1178-1228, unscale scaling.c:195-209)
// with the deterministic build settings the CPU oracle uses (profiling off => adaptive-rho interval = 4 x
// check_termination; no polishing; cold start because the reference tears the solver down after every solve).
//
// Data layout.  All problems of a batch share one sparsity pattern (qp_symbolic.cpp), so every thread walks the same
// index lists (uniform, read-only loads) while its own numbers live in a batch-interleaved workspace:
// element e of problem b is ws[e * stride + b].  A warp therefore touches 32 consecutive doubles per access
// (fully coalesced 256 B) and never diverges on structure — only on the data-dependent iteration count.
// The fill-reducing order is the one the reference's own AMD returns for this pattern (csrc/amd_perm_table.inc: order 5 with
// S <= 80, order 7 with S <= 40), so the ADMM iterates are bit-identical to the reference's OSQP; other (order, S) fall back to a plain
// minimum-degree order and agree to rounding only (the parity gate there is 1e-5 relative + identical status / iterations).
//
// Three executions of the same restatement: qp_solve_kernel (one thread per problem, batch-interleaved workspace),
// qp_solve_warp_kernel (one warp per problem, workspace in shared memory; qp_solve_grouped_kernel runs the same warp body over
// problems of different S in one launch) and — for the search -> QP pipeline — the same warp body called from inside
// kino_search_kernel by the CTA that finished the query (kino_kernel.cu: qp_round).
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <vector>

#include "fpmath.h"
#include "qp_body.h"
#include "qp_body_warp.h"
#include "qp_plan.h"
#include "uavmp_internal.h"


struct QpPlan {
  QpPlanHost* host = nullptr;
  QpPlanDev dev;
  int* d_ints = nullptr;
  double* d_dbls = nullptr;
  unsigned short* d_sidx = nullptr;
  unsigned int* d_sch = nullptr;
};

namespace {

__global__ void __launch_bounds__(QP_TPB) qp_solve_kernel(QpPlanDev pl, QpIo io, uavmp_osqp_settings S, double* ws, int use_smem) {
  extern __shared__ __align__(16) double qp_sv[];  // [2 N][QP_TPB]: bp | xz of every thread's problem
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= io.B) return;
  qp_solve_one(pl, io, S, ws, b, use_smem ? qp_sv : nullptr);
}

// ---- K2w: one warp per problem, workspace in shared memory (qp_body_warp.h) ------------------------------------------------------
__global__ void qp_solve_warp_kernel(QpPlanDev pl, QpIo io, uavmp_osqp_settings S, int warps_per_cta) {
  extern __shared__ __align__(16) double qpw_sm[];
  // the index block of the triangular solves, shared by the CTA's warps, behind their workspaces
  unsigned short* sx = reinterpret_cast<unsigned short*>(qpw_sm + (size_t)warps_per_cta * pl.ws_warp);
  for (int i = threadIdx.x; i < pl.n_sidx / 2; i += blockDim.x) reinterpret_cast<uint32_t*>(sx)[i] = reinterpret_cast<const uint32_t*>(pl.Sidx)[i];
  __syncthreads();
  const int warp = threadIdx.x >> 5;
  const int b = blockIdx.x * warps_per_cta + warp;
  if (b >= io.B) return;  // whole warps leave together
  qp_warp_solve_one(pl, io, S, qpw_sm + (size_t)warp * pl.ws_warp, b, sx);
}

// warps per CTA of the warp-per-problem kernel: whatever keeps the most problems resident per SM — one big CTA (up to 227 KB of
// shared memory) or two of up to 113 KB; 0 = a problem's workspace does not fit (or UAVMP_QP_THREAD asks for the thread kernel)
static int qpw_warps_per_cta(const QpPlanDev& pl, int B) {
  if (getenv("UAVMP_QP_THREAD")) return 0;
  (void)B;
  const size_t per = (size_t)pl.ws_warp * sizeof(double);
  const size_t idx = (size_t)pl.n_sidx * sizeof(unsigned short);
  if (pl.n_sidx == 0 || per + idx > 226 * 1024) return 0;
  int w1 = (int)((226 * 1024 - idx) / per), w2 = (per + idx <= 112 * 1024) ? (int)((112 * 1024 - idx) / per) : 0;
  if (w1 > 16) w1 = 16;
  if (w2 > 8) w2 = 8;
  return (2 * w2 >= w1) ? w2 : w1;
}

// ---- K2g: grouped warp-per-problem kernel — one launch for problems of different S (ragged batches) ------------------------------
// A chunk is up to `wps` problems of one group (one S, one plan).  One persistent CTA per SM pulls chunks from a global counter,
// stages the group's plan view and index block, and its warps run qp_warp_solve_one unchanged: the same body with the same plan as
// qp_solve_warp_kernel, so every problem's result is bit-identical to a per-S launch.  Only the scheduling differs.
struct QpChunkGroup {
  QpPlanDev pl;
  const int* pid;  // the group's problems (indices into the ragged batch)
  int count;       // problems in the group
  int wps;         // problems per chunk = warp workspaces that fit next to the index block
  int chunk0;      // first chunk of the group (groups are stored in processing order)
};

__global__ void qp_solve_grouped_kernel(const QpChunkGroup* __restrict__ groups, int n_groups, int n_chunks, QpRaggedIo r,
                                        uavmp_osqp_settings S, int* next_chunk) {
  extern __shared__ __align__(16) double qpg_sm[];
  __shared__ __align__(16) QpPlanDev s_pl;
  __shared__ int s_chunk, s_group;
  static_assert(sizeof(QpPlanDev) % 4 == 0, "plan view copied as words");
  const int warp = threadIdx.x >> 5;
  for (;;) {
    if (threadIdx.x == 0) {
      const int c = atomicAdd(next_chunk, 1);
      int lo = 0, hi = n_groups - 1;  // last group with chunk0 <= c
      while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (groups[mid].chunk0 <= c) lo = mid; else hi = mid - 1; }
      s_chunk = c; s_group = lo;
    }
    __syncthreads();
    const int c = s_chunk;
    if (c >= n_chunks) return;  // uniform: the whole CTA leaves
    const QpChunkGroup& G = groups[s_group];
    for (int i = threadIdx.x; i < (int)(sizeof(QpPlanDev) / 4); i += blockDim.x)
      reinterpret_cast<uint32_t*>(&s_pl)[i] = reinterpret_cast<const uint32_t*>(&G.pl)[i];
    const int wps = G.wps, ws_warp = G.pl.ws_warp, n_sidx = G.pl.n_sidx;
    unsigned short* sx = reinterpret_cast<unsigned short*>(qpg_sm + (size_t)wps * ws_warp);
    const uint32_t* gsx = reinterpret_cast<const uint32_t*>(G.pl.Sidx);
    for (int i = threadIdx.x; i < n_sidx / 2; i += blockDim.x) reinterpret_cast<uint32_t*>(sx)[i] = gsx[i];
    __syncthreads();
    const int j = (c - G.chunk0) * wps + warp;
    if (warp < wps && j < G.count) {
      const int p = G.pid[j];
      const long long so = r.seg_off[p];
      QpIo io;
      io.pos = r.pos + so + p; io.bv = r.bv + 2 * (size_t)p; io.ba = r.ba + 2 * (size_t)p; io.bj = r.bj + 2 * (size_t)p;
      io.T = r.T + so; io.lo = nullptr; io.hi = nullptr;
      io.coef = r.coef + (size_t)(r.order + 1) * so; io.solved = r.solved + p; io.status = r.status + p; io.iters = r.iters + p;
      io.B = 1; io.stride = 0;
      qp_warp_solve_one(s_pl, io, S, qpg_sm + (size_t)warp * ws_warp, 0, sx);
    }
    __syncthreads();  // the next chunk may restage the plan and the index block
  }
}

// problems of a group whose warp workspace does not fit in shared memory: copied to / from a contiguous batch for qp_solve_kernel
__global__ void k_ragged_gather(QpRaggedIo r, const int* pid, int S, double* pos, double* bv, double* ba, double* bj, double* T) {
  const int j = blockIdx.x, p = pid[j];
  const long long so = r.seg_off[p];
  for (int i = threadIdx.x; i <= S; i += blockDim.x) pos[(size_t)j * (S + 1) + i] = r.pos[so + p + i];
  for (int i = threadIdx.x; i < S; i += blockDim.x) T[(size_t)j * S + i] = r.T[so + i];
  if (threadIdx.x < 2) {
    bv[2 * j + threadIdx.x] = r.bv[2 * (size_t)p + threadIdx.x];
    ba[2 * j + threadIdx.x] = r.ba[2 * (size_t)p + threadIdx.x];
    bj[2 * j + threadIdx.x] = r.bj[2 * (size_t)p + threadIdx.x];
  }
}

__global__ void k_ragged_scatter(QpRaggedIo r, const int* pid, int n, const double* coef, const int* solved, const int* status,
                                 const int* iters) {
  const int j = blockIdx.x, p = pid[j];
  double* out = r.coef + (size_t)(r.order + 1) * r.seg_off[p];
  for (int i = threadIdx.x; i < n; i += blockDim.x) out[i] = coef[(size_t)j * n + i];
  if (threadIdx.x == 0) { r.solved[p] = solved[j]; r.status[p] = status[j]; r.iters[p] = iters[j]; }
}

// ---- pipeline glue: waypoints from the searched paths, outputs back to per-plan layout --------------------------------------
__global__ void k_waypoints(int B, int S, double seg_time, int time_alloc, double step, int Kc, double margin, const int* n_path,
                            const double* path_stage, int path_cap, const int* search_status, const double* sv, const double* ev,
                            double* pos, double* bv, double* ba, double* bj, double* T, double* lo, double* hi) {
  // axis-major batch of 3B one-dimensional problems: problem id = axis * B + q (the rule of uavmp_plan_options, see uavmp.h)
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= B) return;
  const int np = n_path[q];
  const bool ok = (search_status[q] == UAVMP_REACH_END) && np >= 1;
  const double* path = path_stage + (size_t)q * path_cap * 3;
  for (int ax = 0; ax < 3; ax++) {
    const size_t id = (size_t)ax * B + q;
    for (int k = 0; k <= S; k++) {
      double v = 0.0;
      if (ok) {
        const long long idx = ((long long)k * (np - 1)) / S;
        v = path[3 * idx + ax];
      }
      pos[id * (S + 1) + k] = v;
    }
    bv[id * 2] = ok ? sv[3 * q + ax] : 0.0;
    bv[id * 2 + 1] = ok ? ev[3 * q + ax] : 0.0;
    ba[id * 2] = 0.0; ba[id * 2 + 1] = 0.0;
    bj[id * 2] = 0.0; bj[id * 2 + 1] = 0.0;
    for (int s = 0; s < S; s++) {
      const long long i0 = ok ? ((long long)s * (np - 1)) / S : 0, i1 = ok ? ((long long)(s + 1) * (np - 1)) / S : 0;
      T[id * S + s] = (time_alloc && ok) ? (double)(i1 > i0 ? i1 - i0 : 1) * step : seg_time;
      if (Kc > 0) {
        double mn = 0.0, mx = 0.0;
        if (ok) {
          mn = mx = path[3 * i0 + ax];
          for (long long i = i0 + 1; i <= i1; i++) { const double v = path[3 * i + ax]; mn = fmin(mn, v); mx = fmax(mx, v); }
        }
        lo[id * S + s] = mn - margin;
        hi[id * S + s] = mx + margin;
      }
    }
  }
}

__global__ void k_scatter_plan(int B, int n, const int* search_status, const int* solved3, const double* coef3,
                               int* qp_solved, double* coef) {
  const int q = blockIdx.x;
  const bool ok = search_status[q] == UAVMP_REACH_END;
  if (threadIdx.x == 0) qp_solved[q] = ok ? (solved3[q] & solved3[B + q] & solved3[2 * B + q]) : 0;
  for (int i = threadIdx.x; i < 3 * n; i += blockDim.x) {
    const int ax = i / n, j = i % n;
    coef[(size_t)q * 3 * n + i] = ok ? coef3[((size_t)ax * B + q) * n + j] : 0.0;
  }
}

}  // namespace

// =============================================================================================================
static QpPlan* get_plan(uavmp_ctx* ctx, int order, int S, int Kc) {
  for (QpPlan* p : ctx->qp_plans)
    if (p->host->order == order && p->host->S == S && p->host->Kc == Kc) return p;
  QpPlan* p = new QpPlan();
  p->host = qp_plan_build(order, S, Kc);
  const QpPlanHost& H = *p->host;
  std::vector<int> ints;
  std::vector<double> dbl;
  QpPlanOffsets off;
  qp_plan_pack(H, ints, dbl, off);
  if (cudaMalloc(&p->d_ints, ints.size() * sizeof(int)) != cudaSuccess) return nullptr;
  if (cudaMalloc(&p->d_dbls, dbl.size() * sizeof(double)) != cudaSuccess) return nullptr;
  cudaMemcpyAsync(p->d_ints, ints.data(), ints.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream);
  cudaMemcpyAsync(p->d_dbls, dbl.data(), dbl.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
  if (!H.Sidx.empty()) {
    if (cudaMalloc(&p->d_sidx, H.Sidx.size() * sizeof(unsigned short)) != cudaSuccess) return nullptr;
    cudaMemcpyAsync(p->d_sidx, H.Sidx.data(), H.Sidx.size() * sizeof(unsigned short), cudaMemcpyHostToDevice, ctx->stream);
  }
  if (!H.Sch.empty()) {
    if (cudaMalloc(&p->d_sch, H.Sch.size() * sizeof(unsigned int)) != cudaSuccess) return nullptr;
    cudaMemcpyAsync(p->d_sch, H.Sch.data(), H.Sch.size() * sizeof(unsigned int), cudaMemcpyHostToDevice, ctx->stream);
  }
  cudaStreamSynchronize(ctx->stream);
  qp_plan_bind(H, off, p->d_ints, p->d_dbls, p->dev);
  p->dev.Sidx = p->d_sidx;
  p->dev.Sch = p->d_sch;
  ctx->qp_plans.push_back(p);
  return p;
}

void qp_free_plans(uavmp_ctx* ctx) {
  for (QpPlan* p : ctx->qp_plans) {
    if (p->d_ints) cudaFree(p->d_ints);
    if (p->d_dbls) cudaFree(p->d_dbls);
    if (p->d_sidx) cudaFree(p->d_sidx);
    if (p->d_sch) cudaFree(p->d_sch);
    delete p->host;
    delete p;
  }
  ctx->qp_plans.clear();
}

// device view of the (order, S) plan, for the in-kernel QP of the search kernel
int qp_get_plan_dev(uavmp_ctx* ctx, int order, int S, int Kc, const QpPlanDev** out) {
  QpPlan* p = get_plan(ctx, order, S, Kc);
  if (!p) return uavmp_fail(ctx, UAVMP_ECUDA, "cannot build the QP plan");
  *out = &p->dev;
  return UAVMP_OK;
}

int qp_plan_stats(uavmp_ctx* ctx, int order, int S, int* out6) {
  QpPlan* p = get_plan(ctx, order, S, 0);
  if (!p) return UAVMP_ECUDA;
  out6[0] = p->host->n; out6[1] = p->host->m; out6[2] = p->host->nnzP; out6[3] = p->host->nnzA; out6[4] = p->host->nnzK;
  out6[5] = p->host->nnzL;
  return UAVMP_OK;
}

int qp_solve_batch_dev(uavmp_ctx* ctx, cudaStream_t stream, QpScratch& scr, int* launches, int order, int S, int Kc, int B,
                       const double* d_pos, const double* d_bv, const double* d_ba, const double* d_bj, const double* d_T,
                       const double* d_lo, const double* d_hi, const uavmp_osqp_settings* st, double* d_coef, int* d_solved,
                       int* d_status, int* d_iters) {
  QpPlan* p = get_plan(ctx, order, S, Kc);
  if (!p) return uavmp_fail(ctx, UAVMP_ECUDA, "cannot build the QP plan");
  if (st->max_iter <= 0 || st->check_termination < 0 || st->scaling < 0)
    return uavmp_fail(ctx, UAVMP_EINVAL, "bad OSQP settings");
  const int stride = (B + 31) & ~31;
  QpIo io;
  io.pos = d_pos; io.bv = d_bv; io.ba = d_ba; io.bj = d_bj ? d_bj : d_ba; io.T = d_T; io.lo = d_lo; io.hi = d_hi;
  io.coef = d_coef; io.solved = d_solved; io.status = d_status; io.iters = d_iters; io.B = B; io.stride = stride;
  if (launches) *launches = 1;
  if (const int wpc = qpw_warps_per_cta(p->dev, B)) {
    // one warp per problem, everything in shared memory: no global workspace at all
    const size_t smem = (size_t)wpc * p->dev.ws_warp * sizeof(double) + (size_t)p->dev.n_sidx * sizeof(unsigned short);
    if (smem > 48 * 1024) cudaFuncSetAttribute(qp_solve_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    qp_solve_warp_kernel<<<(B + wpc - 1) / wpc, 32 * wpc, smem, stream>>>(p->dev, io, *st, wpc);
    UAVMP_CUDA(ctx, cudaGetLastError());
    return UAVMP_OK;
  }
  {
    const size_t need = (size_t)p->dev.ws_doubles * stride * sizeof(double);
    int r = ensure_bytes(ctx, &scr.ws, &scr.ws_bytes, need);
    if (r) return r;
  }
  const int threads = QP_TPB;
  // bp and xz in shared memory when they fit (2 N doubles per thread); otherwise everything stays in the workspace
  size_t smem = (size_t)2 * p->dev.N * sizeof(double) * threads;
  const int use_smem = smem <= 200 * 1024 ? 1 : 0;
  if (!use_smem) smem = 0;
  if (smem > 48 * 1024) cudaFuncSetAttribute(qp_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  qp_solve_kernel<<<(B + threads - 1) / threads, threads, smem, stream>>>(p->dev, io, *st, (double*)scr.ws, use_smem);
  UAVMP_CUDA(ctx, cudaGetLastError());
  return UAVMP_OK;
}

int qp_waypoints_from_paths(uavmp_ctx* ctx, PlanSlot& sl, int B, const uavmp_plan_options& o, const double* d_sv, const double* d_ev,
                            double** d_pos, double** d_bv, double** d_ba, double** d_bj, double** d_T, double** d_lo, double** d_hi) {
  const size_t nB = (size_t)3 * B;
  const int S = o.S;
  double* pos = sl.d_wp; double* bv = pos + nB * (S + 1); double* ba = bv + nB * 2; double* bj = ba + nB * 2;
  double* T = bj + nB * 2; double* lo = T + nB * S; double* hi = lo + nB * S;
  k_waypoints<<<(B + 127) / 128, 128, 0, sl.stream>>>(B, S, o.seg_time, o.time_alloc, ctx->kp.time_step_size, o.corridor_samples,
                                                      o.corridor_margin, sl.d_npath, sl.d_path_stage, sl.path_cap, sl.d_status,
                                                      d_sv, d_ev, pos, bv, ba, bj, T, lo, hi);
  UAVMP_CUDA(ctx, cudaGetLastError());
  *d_pos = pos; *d_bv = bv; *d_ba = ba; *d_bj = bj; *d_T = T; *d_lo = lo; *d_hi = hi;
  return UAVMP_OK;
}

int qp_scatter_plan_outputs(uavmp_ctx* ctx, PlanSlot& sl, int B, int order, int S, const int* d_solved3, const double* d_coef3,
                            int* d_qp_solved, double* d_coef) {
  const int n = (order + 1) * S;
  k_scatter_plan<<<B, 128, 0, sl.stream>>>(B, n, sl.d_status, d_solved3, d_coef3, d_qp_solved, d_coef);
  UAVMP_CUDA(ctx, cudaGetLastError());
  return UAVMP_OK;
}

// ---- ragged batches: problems with different S in one grouped launch ------------------------------------------------------------
// Groups whose warp workspace fits in shared memory (qpw_warps_per_cta != 0, the same test qp_solve_batch_dev applies) are cut into
// chunks of W_S problems, W_S = warp workspaces that fit next to the group's index block in one 226 KB CTA (at most 16), and solved
// by ONE qp_solve_grouped_kernel launch, longest S first.  The other groups run through qp_solve_batch_dev's thread-per-problem
// kernel, one launch per S, exactly as uavmp_minctrl_solve_batch runs them.  UAVMP_QP_RAGGED_CTAS=2: two 112 KB CTAs per SM
// instead (used only when every grouped S fits; measured, see DESIGN.md §4); UAVMP_QP_RAGGED_ASC=1: chunks by increasing S.
int qp_solve_ragged_dev(uavmp_ctx* ctx, cudaStream_t st, QpScratch& scr, int order, int B, const int* S_host, QpRaggedIo r,
                        const uavmp_osqp_settings* settings, int* qp_launches, int* aux_launches, int* n_groups_out, int* n_thread_out) {
  if (settings->max_iter <= 0 || settings->check_termination < 0 || settings->scaling < 0)
    return uavmp_fail(ctx, UAVMP_EINVAL, "bad OSQP settings");
  // problems by S (counting sort over the distinct values)
  std::vector<int> Svals(S_host, S_host + B);
  std::sort(Svals.begin(), Svals.end());
  Svals.erase(std::unique(Svals.begin(), Svals.end()), Svals.end());
  const bool ascending = getenv("UAVMP_QP_RAGGED_ASC") != nullptr;
  if (!ascending) std::reverse(Svals.begin(), Svals.end());
  const int nS = (int)Svals.size();
  std::vector<QpPlan*> plans(nS);
  std::vector<int> cnt(nS, 0), start(nS + 1, 0), wps(nS, 0);
  for (int g = 0; g < nS; g++) {
    plans[g] = get_plan(ctx, order, Svals[g], 0);
    if (!plans[g]) return uavmp_fail(ctx, UAVMP_ECUDA, "cannot build the QP plan");
  }
  auto group_of = [&](int S) {
    return ascending ? (int)(std::lower_bound(Svals.begin(), Svals.end(), S) - Svals.begin())
                     : (int)(std::lower_bound(Svals.begin(), Svals.end(), S, std::greater<int>()) - Svals.begin());
  };
  std::vector<int> grp(B);
  for (int p = 0; p < B; p++) cnt[grp[p] = group_of(S_host[p])]++;
  for (int g = 0; g < nS; g++) start[g + 1] = start[g] + cnt[g];
  // shared-memory budget of one CTA
  bool two = getenv("UAVMP_QP_RAGGED_CTAS") && atoi(getenv("UAVMP_QP_RAGGED_CTAS")) == 2;
  auto fit = [](const QpPlanDev& pl, size_t budget, int cap) {
    const size_t per = (size_t)pl.ws_warp * sizeof(double), idx = (size_t)pl.n_sidx * sizeof(unsigned short);
    if (pl.n_sidx == 0 || per + idx > budget) return 0;
    return std::min(cap, (int)((budget - idx) / per));
  };
  for (int g = 0; g < nS; g++)
    if (qpw_warps_per_cta(plans[g]->dev, cnt[g]) && two && fit(plans[g]->dev, 112 * 1024, 8) == 0) two = false;
  const size_t budget = two ? 112 * 1024 : 226 * 1024;
  // host image of the table: counter | groups | seg_off[B] | pid[B]
  std::vector<long long> seg_off(B);
  long long so = 0;
  for (int p = 0; p < B; p++) { seg_off[p] = so; so += S_host[p]; }
  const size_t o_groups = 256, o_seg = o_groups + ((sizeof(QpChunkGroup) * nS + 255) & ~(size_t)255), o_pid = o_seg + (size_t)B * 8;
  const size_t tab_bytes = o_pid + (size_t)B * 4;
  int r0 = ensure_bytes(ctx, &scr.tab, &scr.tab_bytes, tab_bytes);
  if (r0) return r0;
  char* d_tab = (char*)scr.tab;
  std::vector<char> img(tab_bytes, 0);
  int* pid = (int*)(img.data() + o_pid);
  {
    std::vector<int> fill(start.begin(), start.end() - 1);
    for (int p = 0; p < B; p++) pid[fill[grp[p]]++] = p;
  }
  memcpy(img.data() + o_seg, seg_off.data(), (size_t)B * 8);
  std::vector<QpChunkGroup> tab;
  std::vector<int> thread_groups;
  int n_chunks = 0, max_w = 0;
  size_t smem = 0;
  for (int g = 0; g < nS; g++) {
    const QpPlanDev& pl = plans[g]->dev;
    const int w = qpw_warps_per_cta(pl, cnt[g]) ? fit(pl, budget, two ? 8 : 16) : 0;
    if (w == 0) { thread_groups.push_back(g); continue; }
    QpChunkGroup G;
    G.pl = pl; G.pid = (const int*)(d_tab + o_pid) + start[g]; G.count = cnt[g]; G.wps = w; G.chunk0 = n_chunks;
    n_chunks += (cnt[g] + w - 1) / w;
    max_w = std::max(max_w, w);
    smem = std::max(smem, (size_t)w * pl.ws_warp * sizeof(double) + (size_t)pl.n_sidx * sizeof(unsigned short));
    tab.push_back(G);
  }
  if (!tab.empty()) memcpy(img.data() + o_groups, tab.data(), sizeof(QpChunkGroup) * tab.size());
  UAVMP_CUDA(ctx, cudaMemcpyAsync(d_tab, img.data(), tab_bytes, cudaMemcpyHostToDevice, st));
  r.seg_off = (const long long*)(d_tab + o_seg);
  if (!r.bj) r.bj = r.ba;
  int qp_l = 0, aux_l = 0;
  if (!tab.empty()) {
    UAVMP_CUDA(ctx, cudaFuncSetAttribute(qp_solve_grouped_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = std::min(n_chunks, ctx->sm_count * (two ? 2 : 1));
    qp_solve_grouped_kernel<<<grid, 32 * max_w, smem, st>>>((const QpChunkGroup*)(d_tab + o_groups), (int)tab.size(), n_chunks, r,
                                                           *settings, (int*)d_tab);
    UAVMP_CUDA(ctx, cudaGetLastError());
    qp_l++;
  }
  for (int g : thread_groups) {
    const int S = Svals[g], nb = cnt[g], n = (order + 1) * S;
    const size_t nd = (size_t)nb * ((S + 1) + 6 + S + n), ni = (size_t)nb * 3;
    int rr = ensure_bytes(ctx, &scr.tmp, &scr.tmp_bytes, nd * sizeof(double) + ni * sizeof(int));
    if (rr) return rr;
    double* pos = (double*)scr.tmp; double* bv = pos + (size_t)nb * (S + 1); double* ba = bv + 2 * (size_t)nb; double* bj = ba + 2 * (size_t)nb;
    double* T = bj + 2 * (size_t)nb; double* coef = T + (size_t)nb * S;
    int* solved = (int*)(coef + (size_t)nb * n); int* status = solved + nb; int* iters = status + nb;
    const int* gp = (const int*)(d_tab + o_pid) + start[g];
    k_ragged_gather<<<nb, 128, 0, st>>>(r, gp, S, pos, bv, ba, bj, T);
    UAVMP_CUDA(ctx, cudaGetLastError());
    int l = 0;
    rr = qp_solve_batch_dev(ctx, st, scr, &l, order, S, 0, nb, pos, bv, ba, order == 7 ? bj : nullptr, T, nullptr, nullptr, settings, coef,
                            solved, status, iters);
    if (rr) return rr;
    k_ragged_scatter<<<nb, 128, 0, st>>>(r, gp, n, coef, solved, status, iters);
    UAVMP_CUDA(ctx, cudaGetLastError());
    qp_l += l; aux_l += 2;
  }
  if (qp_launches) *qp_launches = qp_l;
  if (aux_launches) *aux_launches = aux_l;
  if (n_groups_out) *n_groups_out = nS;
  if (n_thread_out) *n_thread_out = (int)thread_groups.size();
  return UAVMP_OK;
}
