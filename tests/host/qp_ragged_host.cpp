// tests/host/qp_ragged_host.cpp — TEST HARNESS (never part of libuavmp.so): the schedule of qp_solve_grouped_kernel (qp_kernel.cu) run
// on the host with the product's warp body (qp_body_warp.h as "one lane") and symbolic plans (qp_symbolic.cpp).
//
// One CTA's shared-memory arena (226 KB) is reused by every chunk, as on the device: chunks of W_S problems of one S, groups by S
// descending, the group's index block staged behind its W_S workspaces.  Between chunks the whole arena is poisoned with NaN, so a
// body that read anything a previous chunk (of another plan) left behind would produce NaN or different bits.  Problems are
// addressed exactly as the kernel does it: the ragged layout, pointers offset to the problem and b = 0.
// Build: g++ -O2 -ffp-contract=off -shared -fPIC (tests/test_rrt_plan_host.py does it on demand).
#include <string.h>

#include <algorithm>
#include <functional>
#include <map>
#include <vector>

#define QPW_HOST 1
#include "../../uav_motion_planning_b200/csrc/qp_body_warp.h"

static const size_t kArena = 226 * 1024;

// warp workspaces of one chunk: what fits next to the index block in the arena, at most 16 (0: the group takes the thread kernel)
static int chunk_warps(const QpPlanDev& D) {
  const size_t per = (size_t)D.ws_warp * sizeof(double), idx = (size_t)D.n_sidx * sizeof(unsigned short);
  if (D.n_sidx == 0 || per + idx > kArena) return 0;
  return (int)std::min<size_t>(16, (kArena - idx) / per);
}

extern "C" int host_qp_chunk_warps(int order, int S) {
  QpPlanHost* H = qp_plan_build(order, S, 0);
  std::vector<int> ints;
  std::vector<double> dbls;
  QpPlanOffsets off;
  QpPlanDev D;
  qp_plan_pack(*H, ints, dbls, off);
  qp_plan_bind(*H, off, ints.data(), dbls.data(), D);
  const int w = chunk_warps(D);
  delete H;
  return w;
}

// B problems, problem p with S[p] segments, ragged layout of uavmp_minctrl_solve_ragged_batch.  Returns the number of chunks run,
// or -(1 + p) when problem p's workspace does not fit in the arena.
extern "C" int host_qp_solve_grouped(int order, int B, const int* S, const double* pos, const double* bv, const double* ba, const double* bj,
                                     const double* T, const uavmp_osqp_settings* st, double* coef, int* solved, int* status, int* iters) {
  struct Plan { QpPlanHost* H; std::vector<int> ints; std::vector<double> dbls; QpPlanDev D; };
  std::map<int, std::vector<int>, std::greater<int>> groups;  // S descending -> problems in order
  std::vector<long long> seg_off(B);
  long long so = 0;
  for (int p = 0; p < B; p++) { groups[S[p]].push_back(p); seg_off[p] = so; so += S[p]; }
  std::vector<double> arena(kArena / sizeof(double));
  const double nan = fpm::from_bits(0x7ff8000000000000ull);
  int chunks = 0;
  for (auto& g : groups) {
    Plan P;
    P.H = qp_plan_build(order, g.first, 0);
    QpPlanOffsets off;
    qp_plan_pack(*P.H, P.ints, P.dbls, off);
    qp_plan_bind(*P.H, off, P.ints.data(), P.dbls.data(), P.D);
    P.D.Sidx = P.H->Sidx.data(); P.D.Sch = P.H->Sch.data();
    const int w = chunk_warps(P.D);
    if (w == 0) { delete P.H; return -(1 + g.second[0]); }
    const std::vector<int>& pid = g.second;
    for (size_t c0 = 0; c0 < pid.size(); c0 += w, chunks++) {
      std::fill(arena.begin(), arena.end(), nan);
      unsigned short* sx = reinterpret_cast<unsigned short*>(arena.data() + (size_t)w * P.D.ws_warp);
      memcpy(sx, P.H->Sidx.data(), P.H->Sidx.size() * sizeof(unsigned short));
      for (int k = 0; k < w && c0 + k < pid.size(); k++) {
        const int p = pid[c0 + k];
        const long long s = seg_off[p];
        QpIo io;
        io.pos = pos + s + p; io.bv = bv + 2 * (size_t)p; io.ba = ba + 2 * (size_t)p; io.bj = (bj ? bj : ba) + 2 * (size_t)p;
        io.T = T + s; io.lo = nullptr; io.hi = nullptr;
        io.coef = coef + (size_t)(order + 1) * s; io.solved = solved + p; io.status = status + p; io.iters = iters + p;
        io.B = 1; io.stride = 0;
        qp_warp_solve_one(P.D, io, *st, arena.data() + (size_t)k * P.D.ws_warp, 0, sx);
      }
    }
    delete P.H;
  }
  return chunks;
}

// one problem alone: fresh poisoned workspace, plan-owned index block (what qp_solve_warp_kernel does per problem)
extern "C" int host_qp_solve_single(int order, int S, const double* pos, const double* bv, const double* ba, const double* bj, const double* T,
                                    const uavmp_osqp_settings* st, double* coef, int* solved, int* status, int* iters) {
  QpPlanHost* H = qp_plan_build(order, S, 0);
  std::vector<int> ints;
  std::vector<double> dbls;
  QpPlanOffsets off;
  QpPlanDev D;
  qp_plan_pack(*H, ints, dbls, off);
  qp_plan_bind(*H, off, ints.data(), dbls.data(), D);
  D.Sidx = H->Sidx.data(); D.Sch = H->Sch.data();
  QpIo io;
  io.pos = pos; io.bv = bv; io.ba = ba; io.bj = bj ? bj : ba; io.T = T; io.lo = nullptr; io.hi = nullptr;
  io.coef = coef; io.solved = solved; io.status = status; io.iters = iters; io.B = 1; io.stride = 0;
  std::vector<double> w((size_t)D.ws_warp, fpm::from_bits(0x7ff8000000000000ull));
  qp_warp_solve_one(D, io, *st, w.data(), 0, H->Sidx.data());
  delete H;
  return 0;
}
