// rrt_kernel.cu — batched RRT* (SURVEY.md §8(f) row 4, second half): one warp per query.
//
// Replaces path_searching::RRTStar::search and its callees
// (reference: src/planner/path_searching/src/rrt_star.cpp:104-116 getRandomNode, :118-123 Step, :125-137 isCollisionFree,
//  :139-172 ChooseParent, :174-226 ReWireTree, :228-238 retrievePath, :304-429 search; and the kd-tree library it calls,
//  src/planner/path_searching/src/kdtree/kdtree.cpp:117-149 kd_insert, :152-182 find_nearest, :231-344 kd_nearest,
//  :474-496 rlist_insert; plan_env/grid_map.h:350-385 the occupancy lookup).
//
// The reference search is not reproducible as written: getRandomNode builds a std::mt19937_64 from ONE 32-bit draw of a fresh
// std::random_device for every sample, and the loop ends on wall-clock time (`max_tolerance_time`, :413-418).  The deterministic
// form built here (and pinned to the reference's own sources by oracle/_ref/librrt_ref.so): the 32-bit seed of sample i is
// uavmp_rrt_sample_seed(query_seed, i), and the time budget is a budget of drawn samples.  Given that, the tree is reproduced
// exactly — which needs the reference's own kd-tree, because the order in which kd_nearest_range hands out the neighbours (reverse
// visiting order of an unbalanced tree in insertion order, results prepended) decides ties in ChooseParent and the order of the
// rewires, and every rewire changes the costs the next one compares.  Quirks kept: see oracle/rrt_star_ref.cpp's header (the
// 1 m collision walk along the normalised direction, out-of-map x_new accepted, the goal node linked into several children
// lists, getOptimalPath() written only by a later improvement, `inf` = 1 << 30).
//
// Execution model: the 32 lanes of a warp run the scalar algorithm REDUNDANTLY (same loads, same stores of the same values to the
// same addresses: one transaction each, and every lane only ever reads what it wrote itself, so no intra-warp fences are needed),
// and split up where the work is wide: the ~20 occupancy lookups of a collision walk (one per lane), the sample stream (lane l
// runs the mt19937_64 seeding recurrence for sample base + l, once per 32 samples) and the tree digest.  The tree walks stay
// dependent chains of L2 / HBM round trips; this is a correctness-first "next row" like K3, not a tuned kernel.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "uavmp_internal.h"

#define RW 4  // warps (queries in flight) per CTA
#define RFULL 0xffffffffu
#define R_STACK_CAP 4096
#define R_NBR_CAP 2048
#define R_INF 1073741824.0  // `#define inf (1 << 30)` (rrt_star.h:14)

namespace {

struct __align__(16) RNode {  // 64 B: RRTStarNode (rrt_star.h:16-28) + its kdnode (kdtree.h) + its place in the parent's children vector
  double px, py, pz, g;
  int parent, kl, kr, dir;
  int ch_head, ch_tail, sib_next, sib_prev;  // children in push_back order: list of cells; cell c < NCAP is node c, else a goal link
};
struct __align__(16) RFrame { int node, stage; double keep; };
struct RArena { RNode* nodes; int2* gcell; int* queue; RFrame* frames; int* stack; int* nbr; };

struct RParams {
  int max_nodes, nx, ny, nz, path_cap;
  double step, radius, ccres, budget, ox, oy, oz, msx, msy, msz, inv_res, lox, loy, loz, hix, hiy, hiz;
};
struct RBatch {
  int B;
  const double* start; const double* end; const unsigned long long* seeds;
  int* status; int* use_num; int* n_opt; long long* n_samples; double* goal_g; unsigned long long* digest;
  double* path_stage; int* next_query; int* error_flag;
};

__device__ __forceinline__ unsigned long long rfold(unsigned long long h, unsigned long long v) {
  h ^= v; h *= 0x100000001b3ull; h ^= h >> 29; return h;
}
__host__ __device__ __forceinline__ uint32_t rrt_seed32(unsigned long long query_seed, long long i) {
  unsigned long long z = query_seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(i + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (uint32_t)(z >> 32);
}

// The first three outputs of std::mt19937_64(seed) through std::uniform_real_distribution<>(0, 1) (libstdc++ bits/random.tcc:
// seed() x[i] = 6364136223846793005 (x[i-1] ^ x[i-1] >> 62) + i; _M_gen_rand twists x[k] from x[k], x[k+1], x[k+156];
// generate_canonical<double, 53> of a 64-bit engine takes ONE draw: double(u) / 2^64, clamped below 1).
__device__ __forceinline__ unsigned long long mt_temper(unsigned long long z) {
  z ^= (z >> 29) & 0x5555555555555555ull;
  z ^= (z << 17) & 0x71D67FFFEDA60000ull;
  z ^= (z << 37) & 0xFFF7EEE000000000ull;
  z ^= z >> 43;
  return z;
}
__device__ __forceinline__ double mt_canonical(unsigned long long u) {
  const double r = (double)u / 18446744073709551616.0;
  return r >= 1.0 ? 0.99999999999999989 : r;  // nextafter(1, 0)
}
__device__ void rrt_sample3(uint32_t seed, double& u0, double& u1, double& u2) {
  unsigned long long x = seed, lo0 = 0, lo1 = 0, lo2 = 0, lo3 = 0, hi0 = 0, hi1 = 0, hi2 = 0;
  lo0 = x;
  for (int i = 1; i <= 158; i++) {
    x = 6364136223846793005ull * (x ^ (x >> 62)) + (unsigned long long)i;
    if (i == 1) lo1 = x;
    if (i == 2) lo2 = x;
    if (i == 3) lo3 = x;
    if (i == 156) hi0 = x;
    if (i == 157) hi1 = x;
    if (i == 158) hi2 = x;
  }
  const unsigned long long UP = ~0ull << 31, LOW = ~UP, MA = 0xB5026F5AA96619E9ull;
  unsigned long long y;
  y = (lo0 & UP) | (lo1 & LOW); u0 = mt_canonical(mt_temper(hi0 ^ (y >> 1) ^ ((y & 1) ? MA : 0ull)));
  y = (lo1 & UP) | (lo2 & LOW); u1 = mt_canonical(mt_temper(hi1 ^ (y >> 1) ^ ((y & 1) ? MA : 0ull)));
  y = (lo2 & UP) | (lo3 & LOW); u2 = mt_canonical(mt_temper(hi2 ^ (y >> 1) ^ ((y & 1) ? MA : 0ull)));
}

__device__ __forceinline__ double sel3(double a0, double a1, double a2, int k) { return k == 0 ? a0 : (k == 1 ? a1 : a2); }
__device__ __forceinline__ void set3(double& a0, double& a1, double& a2, int k, double v) {
  if (k == 0) a0 = v; else if (k == 1) a1 = v; else a2 = v;
}
__device__ __forceinline__ double sq3(double a, double b, double c) { return (a * a + b * b) + c * c; }  // Eigen's 3-vector reduction order

// GridMap::getInflateOccupancy (grid_map.h:350-359): -1 outside the map (isInMap :370-385), else the inflated byte
__device__ __forceinline__ int r_lookup(const RParams& P, const int8_t* __restrict__ occ, double x, double y, double z) {
  if (x < P.lox || y < P.loy || z < P.loz) return -1;
  if (x > P.hix || y > P.hiy || z > P.hiz) return -1;
  const int ix = (int)floor((x - P.ox) * P.inv_res), iy = (int)floor((y - P.oy) * P.inv_res), iz = (int)floor((z - P.oz) * P.inv_res);
  return occ[((size_t)ix * P.ny + iy) * P.nz + iz];
}

// RRTStar::isCollisionFree (rrt_star.cpp:125-137): the direction is normalised and t runs over [0, |dir|) — about 1 m whatever the
// distance — by repeated addition of the check resolution; lane l takes the l-th point of each block of 32
__device__ bool r_collision_free(const RParams& P, const int8_t* __restrict__ occ, int lane, double fx, double fy, double fz,
                                 double tx, double ty, double tz) {
  double dx = tx - fx, dy = ty - fy, dz = tz - fz;
  const double n2 = sq3(dx, dy, dz);
  if (n2 > 0.0) { const double s = sqrt(n2); dx = dx / s; dy = dy / s; dz = dz / s; }
  const double len = sqrt(sq3(dx, dy, dz));
  double tbase = 0.0;
  for (;;) {
    double t = tbase;
    for (int k = 0; k < lane; k++) t += P.ccres;
    const bool valid = t < len;
    int o = 0;
    if (valid) o = r_lookup(P, occ, fx + t * dx, fy + t * dy, fz + t * dz);
    const unsigned hit = __ballot_sync(RFULL, valid && o != 0), vm = __ballot_sync(RFULL, valid);
    if (hit) return false;
    if (vm != RFULL) return true;
    tbase = __shfl_sync(RFULL, t, 31) + P.ccres;
  }
}

struct RQuery {
  RNode* N; int2* gcell; int NCAP;
  __device__ __forceinline__ int cell_next(int c) const { return c < NCAP ? N[c].sib_next : gcell[c - NCAP].x; }
  __device__ __forceinline__ void set_next(int c, int v) { if (c < NCAP) N[c].sib_next = v; else gcell[c - NCAP].x = v; }
  __device__ __forceinline__ void set_prev(int c, int v) { if (c < NCAP) N[c].sib_prev = v; else gcell[c - NCAP].y = v; }
  // children.push_back
  __device__ __forceinline__ void append(int parent, int c) {
    const int tail = N[parent].ch_tail;
    set_prev(c, tail); set_next(c, -1);
    if (tail >= 0) set_next(tail, c); else N[parent].ch_head = c;
    N[parent].ch_tail = c;
  }
  // std::remove + erase of one regular node, order of the others kept (rrt_star.cpp:196-198)
  __device__ __forceinline__ void unlink(int parent, int c) {
    const int pv = N[c].sib_prev, nx = N[c].sib_next;
    if (pv >= 0) set_next(pv, nx); else N[parent].ch_head = nx;
    if (nx >= 0) set_prev(nx, pv); else N[parent].ch_tail = pv;
  }
};

template <int MINB>
__global__ void __launch_bounds__(RW * 32, MINB) rrt_star_kernel(RParams P, const int8_t* __restrict__ occ, const RArena* arenas, RBatch bt) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const RArena A = arenas[blockIdx.x * RW + warp];
  RNode* N = A.nodes;
  RQuery Q; Q.N = N; Q.gcell = A.gcell; Q.NCAP = P.max_nodes + 2;
  const int NCAP = Q.NCAP;
  const double r2 = P.radius * P.radius;

  for (;;) {
    int q = 0;
    if (lane == 0) q = atomicAdd(bt.next_query, 1);
    q = __shfl_sync(RFULL, q, 0);
    if (q >= bt.B) break;
    const double sx = bt.start[3 * q], sy = bt.start[3 * q + 1], sz = bt.start[3 * q + 2];
    const double ex = bt.end[3 * q], ey = bt.end[3 * q + 1], ez = bt.end[3 * q + 2];
    const unsigned long long qseed = bt.seeds[q];
    {
      RNode a; a.px = sx; a.py = sy; a.pz = sz; a.g = 0.0; a.parent = -1; a.kl = a.kr = -1; a.dir = 0; a.ch_head = a.ch_tail = a.sib_next = a.sib_prev = -1;
      N[0] = a;  // start node, kd_insert'ed as the root (rrt_star.cpp:307-322)
      a.px = ex; a.py = ey; a.pz = ez; a.g = R_INF;
      N[1] = a;  // global goal node: never in the kd-tree
    }
    int use = 2, n_gc = 0, status = 0, n_opt = 0, err = 0;
    bool reach = false;
    double feasible = R_INF;
    long long samples = 0;
    double rlo0 = sx, rlo1 = sy, rlo2 = sz, rhi0 = sx, rhi1 = sy, rhi2 = sz;  // the tree's bounding hyperrect (kd_insert :141-147)
    double bx = 0, by = 0, bz = 0;                                            // this lane's sample of the current block of 32

    for (int it = 0; it < P.max_nodes && !status && !err; it++) {
      if ((it & 31) == 0) {
        double u0, u1, u2;
        rrt_sample3(rrt_seed32(qseed, (long long)it + lane), u0, u1, u2);
        bx = u0 * P.msx + P.ox; by = u1 * P.msy + P.oy; bz = u2 * P.msz + P.oz;  // getRandomNode :111-113
      }
      const double xr = __shfl_sync(RFULL, bx, it & 31), yr = __shfl_sync(RFULL, by, it & 31), zr = __shfl_sync(RFULL, bz, it & 31);
      samples++;

      // ---- kd_nearest (kdtree.cpp:231-344), recursion unrolled onto A.frames ----
      int best = 0;
      double bd2 = sq3(N[0].px - xr, N[0].py - yr, N[0].pz - zr);
      {
        double lo0 = rlo0, lo1 = rlo1, lo2 = rlo2, hi0 = rhi0, hi1 = rhi1, hi2 = rhi2;
        int sp = 0, cur = 0, state = 0;  // 0 enter, 1 after the nearer subtree, 2 return
        for (;;) {
          if (state == 2) {
            if (sp == 0) break;
            const RFrame f = A.frames[--sp];
            cur = f.node;
            const int dir = N[cur].dir;
            const bool neg = (sel3(xr, yr, zr, dir) - sel3(N[cur].px, N[cur].py, N[cur].pz, dir)) <= 0;
            if (f.stage == 1) { if (neg) set3(hi0, hi1, hi2, dir, f.keep); else set3(lo0, lo1, lo2, dir, f.keep); state = 1; }
            else { if (neg) set3(lo0, lo1, lo2, dir, f.keep); else set3(hi0, hi1, hi2, dir, f.keep); state = 2; continue; }
          }
          const RNode t = N[cur];
          const int dir = t.dir;
          const double pd = sel3(t.px, t.py, t.pz, dir);
          const bool neg = (sel3(xr, yr, zr, dir) - pd) <= 0;
          if (state == 0) {
            const int nearer = neg ? t.kl : t.kr;
            if (nearer >= 0) {
              if (sp >= R_STACK_CAP) { err = 1; break; }
              RFrame f; f.node = cur; f.stage = 1;
              if (neg) { f.keep = sel3(hi0, hi1, hi2, dir); set3(hi0, hi1, hi2, dir, pd); }
              else { f.keep = sel3(lo0, lo1, lo2, dir); set3(lo0, lo1, lo2, dir, pd); }
              A.frames[sp++] = f;
              cur = nearer; state = 0;
              continue;
            }
          }
          // the node itself, then the farther subtree if its sliced hyperrect can still hold something closer
          const double d2 = sq3(t.px - xr, t.py - yr, t.pz - zr);
          if (d2 < bd2) { best = cur; bd2 = d2; }
          const int farther = neg ? t.kr : t.kl;
          state = 2;
          if (farther >= 0) {
            double keep;
            if (neg) { keep = sel3(lo0, lo1, lo2, dir); set3(lo0, lo1, lo2, dir, pd); }
            else { keep = sel3(hi0, hi1, hi2, dir); set3(hi0, hi1, hi2, dir, pd); }
            double rd = 0;
            if (xr < lo0) rd += (lo0 - xr) * (lo0 - xr); else if (xr > hi0) rd += (hi0 - xr) * (hi0 - xr);
            if (yr < lo1) rd += (lo1 - yr) * (lo1 - yr); else if (yr > hi1) rd += (hi1 - yr) * (hi1 - yr);
            if (zr < lo2) rd += (lo2 - zr) * (lo2 - zr); else if (zr > hi2) rd += (hi2 - zr) * (hi2 - zr);
            if (rd < bd2) {
              if (sp >= R_STACK_CAP) { err = 1; break; }
              RFrame f; f.node = cur; f.stage = 2; f.keep = keep;
              A.frames[sp++] = f;
              cur = farther; state = 0;
            } else {
              if (neg) set3(lo0, lo1, lo2, dir, keep); else set3(hi0, hi1, hi2, dir, keep);
            }
          }
        }
        if (err) break;
      }

      // ---- Step (:118-123) and the occupancy test of x_new (:341: `!= true`, so -1 = outside the map passes) ----
      double nx_, ny_, nz_;
      {
        const double px = N[best].px, py = N[best].py, pz = N[best].pz;
        double dx = xr - px, dy = yr - py, dz = zr - pz;
        const double n2 = sq3(dx, dy, dz);
        if (n2 > 0.0) { const double s = sqrt(n2); dx = dx / s; dy = dy / s; dz = dz / s; }
        nx_ = px + dx * P.step; ny_ = py + dy * P.step; nz_ = pz + dz * P.step;
      }
      if (r_lookup(P, occ, nx_, ny_, nz_) == 1) continue;

      // ---- kd_nearest_range (find_nearest, kdtree.cpp:152-182): visiting order into A.nbr, walked backwards (results are prepended) ----
      auto range = [&](double qx, double qy, double qz) -> int {
        int cnt = 0, sp = 0;
        A.stack[sp++] = 0;
        while (sp > 0) {
          const int id = A.stack[--sp];
          const RNode t = N[id];
          if (sq3(t.px - qx, t.py - qy, t.pz - qz) <= r2) {
            if (cnt >= R_NBR_CAP) { err = 2; return 0; }
            A.nbr[cnt++] = id;
          }
          const double dxx = sel3(qx, qy, qz, t.dir) - sel3(t.px, t.py, t.pz, t.dir);
          const int near = dxx <= 0.0 ? t.kl : t.kr, far = dxx <= 0.0 ? t.kr : t.kl;
          if (sp + 2 > R_STACK_CAP) { err = 1; return 0; }
          if (fabs(dxx) < P.radius && far >= 0) A.stack[sp++] = far;
          if (near >= 0) A.stack[sp++] = near;
        }
        return cnt;
      };

      // ---- ChooseParent (:139-172) ----
      int cnt = range(nx_, ny_, nz_);
      if (err) break;
      double compare = R_INF;
      int parent = -1;
      for (int j = cnt - 1; j >= 0; j--) {
        const int nb = A.nbr[j];
        const double npx = N[nb].px, npy = N[nb].py, npz = N[nb].pz;
        const double g_new = N[nb].g + sqrt(sq3(npx - nx_, npy - ny_, npz - nz_));
        if (g_new < compare && r_collision_free(P, occ, lane, npx, npy, npz, nx_, ny_, nz_)) { compare = g_new; parent = nb; }
      }
      if (compare == R_INF) continue;
      const int nw = use++;
      {
        RNode a; a.px = nx_; a.py = ny_; a.pz = nz_; a.g = compare; a.parent = parent; a.kl = a.kr = -1; a.dir = 0;
        a.ch_head = a.ch_tail = a.sib_next = a.sib_prev = -1;
        N[nw] = a;
      }
      Q.append(parent, nw);

      // ---- kd_insert (:117-149) ----
      {
        int cur = 0;
        for (;;) {
          const int dir = N[cur].dir;
          const bool left = sel3(nx_, ny_, nz_, dir) < sel3(N[cur].px, N[cur].py, N[cur].pz, dir);
          const int child = left ? N[cur].kl : N[cur].kr;
          if (child < 0) {
            N[nw].dir = (dir + 1) % 3;
            if (left) N[cur].kl = nw; else N[cur].kr = nw;
            break;
          }
          cur = child;
        }
        if (nx_ < rlo0) rlo0 = nx_;
        if (nx_ > rhi0) rhi0 = nx_;
        if (ny_ < rlo1) rlo1 = ny_;
        if (ny_ > rhi1) rhi1 = ny_;
        if (nz_ < rlo2) rlo2 = nz_;
        if (nz_ > rhi2) rhi2 = nz_;
      }

      // ---- ReWireTree (:174-226) ----
      cnt = range(nx_, ny_, nz_);
      if (err) break;
      for (int j = cnt - 1; j >= 0; j--) {
        const int nb = A.nbr[j];
        const double npx = N[nb].px, npy = N[nb].py, npz = N[nb].pz;
        const double g_new = N[nw].g + sqrt(sq3(npx - nx_, npy - ny_, npz - nz_));
        if (g_new < N[nb].g && r_collision_free(P, occ, lane, nx_, ny_, nz_, npx, npy, npz)) {
          Q.unlink(N[nb].parent, nb);
          N[nb].parent = nw; N[nb].g = g_new;
          Q.append(nw, nb);
          // cost propagation over the children vectors, in queue order (a goal link may be stale: :207-219 does not look at ->parent)
          int head = 0, tail = 0;
          A.queue[tail++] = nb;
          while (head < tail) {
            const int cur = A.queue[head++];
            const double cg = N[cur].g, cx = N[cur].px, cy = N[cur].py, cz = N[cur].pz;
            for (int c = N[cur].ch_head; c >= 0; c = Q.cell_next(c)) {
              const int child = c < NCAP ? c : 1;
              N[child].g = cg + sqrt(sq3(N[child].px - cx, N[child].py - cy, N[child].pz - cz));
              A.queue[tail++] = child;
            }
          }
        }
      }

      // ---- the goal (:348-391) ----
      const double gd = sqrt(sq3(nx_ - ex, ny_ - ey, nz_ - ez));
      if (gd <= P.radius) {
        if (!r_collision_free(P, occ, lane, nx_, ny_, nz_, ex, ey, ez)) continue;
        const double via = N[nw].g + sqrt(sq3(ex - nx_, ey - ny_, ez - nz_));
        if (!reach) {
          reach = true;
          Q.append(nw, NCAP + n_gc++);
          N[1].parent = nw; N[1].g = via; feasible = via;
        } else if (via < feasible) {
          N[1].parent = nw;
          Q.append(nw, NCAP + n_gc++);
          N[1].g = via;
        }
      }
      if (reach) {
        const double tmp = N[1].g;
        if (tmp < feasible) {  // getOptimalPath() is (re)written only here (:396-404)
          feasible = tmp;
          int len = 0;
          for (int t = 1; t >= 0; t = N[t].parent) len++;
          n_opt = len;
          if (len > P.path_cap) err = 4;
          else {
            double* out = bt.path_stage + (size_t)q * P.path_cap * 3;
            int k = len - 1;
            for (int t = 1; t >= 0; t = N[t].parent, k--) { out[3 * k] = N[t].px; out[3 * k + 1] = N[t].py; out[3 * k + 2] = N[t].pz; }
          }
        }
        if ((double)samples >= P.budget) status = 1;  // `max_tolerance_time` as a sample budget (:413-418)
      }
    }
    if (!status) status = reach ? 1 : 2;

    unsigned long long h = 0;
    for (int i = lane; i < use; i += 32) {
      unsigned long long hn = 0xcbf29ce484222325ull ^ (0x9E3779B97F4A7C15ull * (unsigned long long)(i + 1));
      hn = rfold(hn, (unsigned long long)__double_as_longlong(N[i].px));
      hn = rfold(hn, (unsigned long long)__double_as_longlong(N[i].py));
      hn = rfold(hn, (unsigned long long)__double_as_longlong(N[i].pz));
      hn = rfold(hn, (unsigned long long)__double_as_longlong(N[i].g));
      hn = rfold(hn, N[i].parent >= 0 ? (unsigned long long)N[i].parent : 0xffffffffull);
      h += hn;
    }
    for (int o = 16; o; o >>= 1) h += __shfl_xor_sync(RFULL, h, o);
    if (lane == 0) {
      bt.status[q] = err ? 0 : status; bt.use_num[q] = use; bt.n_opt[q] = err ? 0 : n_opt; bt.n_samples[q] = samples;
      bt.goal_g[q] = N[1].g; bt.digest[q] = h;
      if (err) atomicOr(bt.error_flag, err);
    }
    __syncwarp();
  }
}

}  // namespace

// =====================================================================================================
struct RrtState {
  int ctas = 8;
  int max_nodes = 0, n_arenas = 0;
  void* mem = nullptr;
  RArena* d_arenas = nullptr;
  int cap = 0, path_cap = 0;
  double* d_q = nullptr;
  unsigned long long *d_seeds = nullptr, *d_digest = nullptr;
  int *d_status = nullptr, *d_use = nullptr, *d_nopt = nullptr, *d_misc = nullptr;
  long long *d_nsamples = nullptr, *d_offsets = nullptr;
  double *d_goal_g = nullptr, *d_path_stage = nullptr, *d_packed = nullptr;
  long long packed_cap = 0, last_total = 0;
  // uavmp_rrt_plan_batch: ragged QP inputs / coefficients, per-problem results, per-QP-query packing table
  double* d_plan = nullptr; size_t plan_bytes = 0;
  int* d_plan_i = nullptr; size_t plan_i_bytes = 0;
  long long* d_plan_q = nullptr; size_t plan_q_bytes = 0;
  double* d_plan_coef = nullptr; long long plan_total = -1;
};

static void rrt_free_batch(RrtState* a) {
  void* ptrs[] = {a->d_q, a->d_seeds, a->d_digest, a->d_status, a->d_use, a->d_nopt, a->d_misc, a->d_nsamples, a->d_offsets, a->d_goal_g,
                  a->d_path_stage};
  for (void* p : ptrs) if (p) cudaFree(p);
  a->d_q = nullptr; a->d_seeds = a->d_digest = nullptr; a->d_status = a->d_use = a->d_nopt = a->d_misc = nullptr;
  a->d_nsamples = a->d_offsets = nullptr; a->d_goal_g = a->d_path_stage = nullptr; a->cap = 0;
}
static void rrt_free(RrtState* a) {
  rrt_free_batch(a);
  if (a->mem) cudaFree(a->mem);
  if (a->d_arenas) cudaFree(a->d_arenas);
  if (a->d_packed) cudaFree(a->d_packed);
  if (a->d_plan) cudaFree(a->d_plan);
  if (a->d_plan_i) cudaFree(a->d_plan_i);
  if (a->d_plan_q) cudaFree(a->d_plan_q);
  *a = RrtState();
}
void rrt_destroy(uavmp_ctx* ctx) {
  if (ctx->rrt) { rrt_free(ctx->rrt); delete ctx->rrt; ctx->rrt = nullptr; }
}
uint32_t rrt_sample_seed_host(unsigned long long query_seed, long long i) { return rrt_seed32(query_seed, i); }

static int rrt_ensure(uavmp_ctx* ctx, int B) {
  if (!ctx->rrt) ctx->rrt = new RrtState();
  RrtState& a = *ctx->rrt;
  const int max_nodes = ctx->rrt_max_nodes;
  if (a.max_nodes != max_nodes) {
    rrt_free(&a);
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t ncap = (size_t)max_nodes + 2;
    const size_t sz_nodes = up(ncap * sizeof(RNode)), sz_gc = up(ncap * sizeof(int2)), sz_queue = up(2 * ncap * sizeof(int)),
                 sz_frames = up((size_t)R_STACK_CAP * sizeof(RFrame)), sz_stack = up((size_t)R_STACK_CAP * sizeof(int)),
                 sz_nbr = up((size_t)R_NBR_CAP * sizeof(int)), per = sz_nodes + sz_gc + sz_queue + sz_frames + sz_stack + sz_nbr;
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    const char* env = getenv("UAVMP_RRT_CTAS");  // resident CTAs per SM: 8 (64 registers, some spills) measured 1.46x over 4 — latency bound
    a.ctas = (env && atoi(env) == 4) ? 4 : 8;
    int want = ctx->sm_count * a.ctas * RW;
    const long long fit = (long long)((free_b / 2) / per);
    if (fit < RW) return uavmp_fail(ctx, UAVMP_ENOMEM, "not enough device memory for RRT* arenas of %d nodes", max_nodes);
    if (want > fit) want = (int)(fit / RW) * RW;
    UAVMP_CUDA(ctx, cudaMalloc(&a.mem, per * (size_t)want));
    std::vector<RArena> ha(want);
    for (int i = 0; i < want; i++) {
      char* b = (char*)a.mem + per * (size_t)i;
      ha[i].nodes = (RNode*)b; b += sz_nodes;
      ha[i].gcell = (int2*)b; b += sz_gc;
      ha[i].queue = (int*)b; b += sz_queue;
      ha[i].frames = (RFrame*)b; b += sz_frames;
      ha[i].stack = (int*)b; b += sz_stack;
      ha[i].nbr = (int*)b;
    }
    UAVMP_CUDA(ctx, cudaMalloc(&a.d_arenas, sizeof(RArena) * want));
    UAVMP_CUDA(ctx, cudaMemcpyAsync(a.d_arenas, ha.data(), sizeof(RArena) * want, cudaMemcpyHostToDevice, ctx->stream));
    UAVMP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    a.max_nodes = max_nodes; a.n_arenas = want;
  }
  if (B > a.cap || a.path_cap != ctx->rrt_path_cap) {
    rrt_free_batch(&a);
    const int cap = B;
    UAVMP_CUDA(ctx, cudaMalloc(&a.d_q, (size_t)cap * 6 * sizeof(double)));
    UAVMP_CUDA(ctx, cudaMalloc(&a.d_seeds, (size_t)cap * sizeof(unsigned long long)));
    UAVMP_CUDA(ctx, cudaMalloc(&a.d_digest, (size_t)cap * sizeof(unsigned long long)));
    UAVMP_CUDA(ctx, cudaMalloc(&a.d_status, (size_t)cap * sizeof(int)));
    UAVMP_CUDA(ctx, cudaMalloc(&a.d_use, (size_t)cap * sizeof(int)));
    UAVMP_CUDA(ctx, cudaMalloc(&a.d_nopt, (size_t)cap * sizeof(int)));
    UAVMP_CUDA(ctx, cudaMalloc(&a.d_misc, 64));
    UAVMP_CUDA(ctx, cudaMalloc(&a.d_nsamples, (size_t)cap * sizeof(long long)));
    UAVMP_CUDA(ctx, cudaMalloc(&a.d_offsets, (size_t)(cap + 1) * sizeof(long long)));
    UAVMP_CUDA(ctx, cudaMalloc(&a.d_goal_g, (size_t)cap * sizeof(double)));
    UAVMP_CUDA(ctx, cudaMalloc(&a.d_path_stage, (size_t)cap * ctx->rrt_path_cap * 3 * sizeof(double)));
    a.cap = cap; a.path_cap = ctx->rrt_path_cap;
  }
  return UAVMP_OK;
}

namespace {
__global__ void k_rrt_offsets(const int* n_path, int B, long long* offsets) {
  long long acc = 0;
  for (int i = 0; i < B; i++) { offsets[i] = acc; acc += n_path[i]; }
  offsets[B] = acc;
}
__global__ void k_rrt_pack(const double* stage, const int* n_path, const long long* offsets, int path_cap, double* out) {
  const int q = blockIdx.x, n = n_path[q];
  const double* src = stage + (size_t)q * path_cap * 3;
  double* dst = out + offsets[q] * 3;
  for (int i = threadIdx.x; i < 3 * n; i += blockDim.x) dst[i] = src[i];
}
// QP inputs of uavmp_rrt_plan_batch, straight from the optimal paths: query k of the QP set (source query kq[3k], S = kq[3k+1]
// segments, sum of S over the QP queries before it kq[3k+2] = Q) owns problems 3k + axis of the ragged batch (QpRaggedIo layout:
// segment offset 3 Q + axis S); every optimal-path point is a waypoint and every T_s = seg_time
__global__ void k_rrt_plan_inputs(const long long* kq, const double* stage, int path_cap, double seg_time, double* pos, double* T) {
  const int k = blockIdx.x;
  const long long q = kq[3 * k], S = kq[3 * k + 1], Q = kq[3 * k + 2];
  const double* path = stage + (size_t)q * path_cap * 3;
  for (int ax = 0; ax < 3; ax++) {
    const long long p = 3 * (long long)k + ax, so = 3 * Q + ax * S;
    for (long long i = threadIdx.x; i <= S; i += blockDim.x) pos[so + p + i] = path[3 * i + ax];
    for (long long i = threadIdx.x; i < S; i += blockDim.x) T[so + i] = seg_time;
  }
}
}  // namespace

// the search itself, shared by uavmp_rrt_search_batch and uavmp_rrt_plan_batch: inputs up, kernel, path offsets, the post-search
// sync with its capacity checks, and the packing of the optimal paths (what uavmp_rrt_get_paths returns).  Returns the total number
// of path points or an error; per-query results stay on the device.
static long long rrt_search_run(uavmp_ctx* ctx, int B, const double* start_pt, const double* end_pt, const uint64_t* query_seed) {
  int r = rrt_ensure(ctx, B);
  if (r) return r;
  RrtState& a = *ctx->rrt;
  cudaStream_t st = ctx->stream;
  const size_t nb = (size_t)B * 3 * sizeof(double);
  UAVMP_CUDA(ctx, cudaMemcpyAsync(a.d_q, start_pt, nb, cudaMemcpyHostToDevice, st));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(a.d_q + 3 * (size_t)B, end_pt, nb, cudaMemcpyHostToDevice, st));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(a.d_seeds, query_seed, (size_t)B * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  UAVMP_CUDA(ctx, cudaMemsetAsync(a.d_misc, 0, 64, st));
  RParams P;
  P.max_nodes = a.max_nodes; P.nx = ctx->nx; P.ny = ctx->ny; P.nz = ctx->nz; P.path_cap = a.path_cap;
  P.step = ctx->rrt_step; P.radius = ctx->rrt_radius; P.ccres = ctx->rrt_ccres; P.budget = ctx->rrt_budget;
  P.ox = ctx->origin[0]; P.oy = ctx->origin[1]; P.oz = ctx->origin[2];
  P.msx = ctx->map_size[0]; P.msy = ctx->map_size[1]; P.msz = ctx->map_size[2];
  P.inv_res = 1.0 / ctx->resolution;
  P.lox = ctx->origin[0] + 1e-4; P.loy = ctx->origin[1] + 1e-4; P.loz = ctx->origin[2] + 1e-4;
  P.hix = (ctx->origin[0] + ctx->map_size[0]) - 1e-4; P.hiy = (ctx->origin[1] + ctx->map_size[1]) - 1e-4; P.hiz = (ctx->origin[2] + ctx->map_size[2]) - 1e-4;
  RBatch bt;
  bt.B = B; bt.start = a.d_q; bt.end = a.d_q + 3 * (size_t)B; bt.seeds = a.d_seeds;
  bt.status = a.d_status; bt.use_num = a.d_use; bt.n_opt = a.d_nopt; bt.n_samples = a.d_nsamples; bt.goal_g = a.d_goal_g; bt.digest = a.d_digest;
  bt.path_stage = a.d_path_stage; bt.next_query = a.d_misc + 1; bt.error_flag = a.d_misc;
  const int grid = std::min(a.n_arenas / RW, (B + RW - 1) / RW);
  if (a.ctas == 8) rrt_star_kernel<8><<<grid, RW * 32, 0, st>>>(P, ctx->d_occ, a.d_arenas, bt);
  else rrt_star_kernel<4><<<grid, RW * 32, 0, st>>>(P, ctx->d_occ, a.d_arenas, bt);
  UAVMP_CUDA(ctx, cudaGetLastError());
  k_rrt_offsets<<<1, 1, 0, st>>>(a.d_nopt, B, a.d_offsets);
  long long total = 0;
  int flag = 0;
  UAVMP_CUDA(ctx, cudaMemcpyAsync(&total, a.d_offsets + B, sizeof(long long), cudaMemcpyDeviceToHost, st));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(&flag, a.d_misc, sizeof(int), cudaMemcpyDeviceToHost, st));
  UAVMP_CUDA(ctx, cudaStreamSynchronize(st));
  if (flag & 4) return uavmp_fail(ctx, UAVMP_ECAP, "RRT* path longer than %d nodes (uavmp_rrt_set_params: path_cap_nodes)", a.path_cap);
  if (flag & 3) return uavmp_fail(ctx, UAVMP_ECAP, "RRT* kd-tree walk exceeded its fixed capacity (depth %d / %d neighbours in range)", R_STACK_CAP, R_NBR_CAP);
  if (total > a.packed_cap) {
    if (a.d_packed) cudaFree(a.d_packed);
    a.d_packed = nullptr; a.packed_cap = 0;
    const long long cap = std::max(total, (long long)1024);
    UAVMP_CUDA(ctx, cudaMalloc(&a.d_packed, (size_t)cap * 3 * sizeof(double)));
    a.packed_cap = cap;
  }
  if (total > 0) k_rrt_pack<<<B, 128, 0, st>>>(a.d_path_stage, a.d_nopt, a.d_offsets, a.path_cap, a.d_packed);
  a.last_total = total;
  return total;
}

long long rrt_search_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* end_pt, const uint64_t* query_seed, int* status,
                           int* use_node_num, long long* n_samples, double* goal_g_cost, uint64_t* tree_digest, long long* path_offsets) {
  const long long total = rrt_search_run(ctx, B, start_pt, end_pt, query_seed);
  if (total < 0) return total;
  RrtState& a = *ctx->rrt;
  cudaStream_t st = ctx->stream;
  UAVMP_CUDA(ctx, cudaMemcpyAsync(status, a.d_status, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  if (use_node_num) UAVMP_CUDA(ctx, cudaMemcpyAsync(use_node_num, a.d_use, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  if (n_samples) UAVMP_CUDA(ctx, cudaMemcpyAsync(n_samples, a.d_nsamples, (size_t)B * sizeof(long long), cudaMemcpyDeviceToHost, st));
  if (goal_g_cost) UAVMP_CUDA(ctx, cudaMemcpyAsync(goal_g_cost, a.d_goal_g, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (tree_digest) UAVMP_CUDA(ctx, cudaMemcpyAsync(tree_digest, a.d_digest, (size_t)B * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
  if (path_offsets) UAVMP_CUDA(ctx, cudaMemcpyAsync(path_offsets, a.d_offsets, (size_t)(B + 1) * sizeof(long long), cudaMemcpyDeviceToHost, st));
  UAVMP_CUDA(ctx, cudaStreamSynchronize(st));
  return total;
}

int rrt_get_paths(uavmp_ctx* ctx, double* path_xyz, long long cap_points) {
  if (!ctx->rrt) return uavmp_fail(ctx, UAVMP_ESTATE, "no RRT* batch has run");
  RrtState& a = *ctx->rrt;
  if (cap_points < a.last_total) return uavmp_fail(ctx, UAVMP_ECAP, "path buffer too small");
  if (a.last_total > 0) UAVMP_CUDA(ctx, cudaMemcpyAsync(path_xyz, a.d_packed, (size_t)a.last_total * 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  UAVMP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return UAVMP_OK;
}

// RRTStar::search, then the reference node's minimum-jerk step (test_minimum_jerk.cpp:40-75) for every query that reached the goal
// with an optimal path of n >= 2 points: S = n - 1, one 1-D QP per axis, solved as ONE ragged batch (qp_solve_ragged_dev) whose
// inputs are written on the device from the staged paths.  Query k of the QP set = problems 3k .. 3k+2, so its coefficients come out
// axis-major [3][(order+1) S] and contiguous: the ragged coefficient array IS the per-query output.
long long rrt_plan_batch(uavmp_ctx* ctx, int B, const double* start_pt, const double* start_vel, const double* end_pt, const uint64_t* query_seed,
                         int order, double seg_time, const uavmp_osqp_settings* settings, int* search_status, int* n_segments,
                         int* qp_solved, long long* coef_offsets, int* osqp_status, int* iters) {
  cudaStream_t st = ctx->stream;
  if (ctx->rrt) ctx->rrt->plan_total = -1;
  cudaEventRecord(ctx->ev[0], st);
  const long long total = rrt_search_run(ctx, B, start_pt, end_pt, query_seed);
  if (total < 0) return total;
  RrtState& a = *ctx->rrt;
  cudaEventRecord(ctx->ev[1], st);
  std::vector<int> nopt(B);
  UAVMP_CUDA(ctx, cudaMemcpyAsync(search_status, a.d_status, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  UAVMP_CUDA(ctx, cudaMemcpyAsync(nopt.data(), a.d_nopt, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  UAVMP_CUDA(ctx, cudaStreamSynchronize(st));
  // the QP set: REACH_END with at least two optimal-path points (the node would otherwise reuse a stale / empty path)
  std::vector<long long> kq;
  std::vector<int> Sp;
  long long Q = 0;
  for (int q = 0; q < B; q++) {
    const int S = (search_status[q] == UAVMP_REACH_END && nopt[q] >= 2) ? nopt[q] - 1 : 0;
    n_segments[q] = S;
    if (!S) continue;
    kq.push_back(q); kq.push_back(S); kq.push_back(Q);
    for (int ax = 0; ax < 3; ax++) Sp.push_back(S);
    Q += S;
  }
  const int M = (int)(kq.size() / 3), P = 3 * M, n1 = order + 1;
  const long long sumS = 3 * Q;
  // device: pos (sumS + P) | bv (2P) | ba = bj (2P, zero) | T (sumS) | coef (n1 sumS);  ints: solved | status | iters (P each)
  const size_t o_bv = (size_t)(sumS + P), o_ba = o_bv + 2 * (size_t)P, o_T = o_ba + 2 * (size_t)P, o_coef = o_T + (size_t)sumS;
  int qp_l = 0, aux_l = 0;
  std::vector<int> pint(3 * (size_t)P);
  if (M > 0) {
    int r = ensure_bytes(ctx, (void**)&a.d_plan, &a.plan_bytes, (o_coef + (size_t)n1 * sumS) * sizeof(double)); if (r) return r;
    r = ensure_bytes(ctx, (void**)&a.d_plan_i, &a.plan_i_bytes, 3 * (size_t)P * sizeof(int)); if (r) return r;
    r = ensure_bytes(ctx, (void**)&a.d_plan_q, &a.plan_q_bytes, kq.size() * sizeof(long long)); if (r) return r;
    std::vector<double> bv(2 * (size_t)P, 0.0);
    for (int k = 0; k < M; k++)
      for (int ax = 0; ax < 3; ax++) bv[2 * (3 * (size_t)k + ax)] = start_vel ? start_vel[3 * kq[3 * k] + ax] : 0.0;
    double* d = a.d_plan;
    UAVMP_CUDA(ctx, cudaMemcpyAsync(a.d_plan_q, kq.data(), kq.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
    UAVMP_CUDA(ctx, cudaMemcpyAsync(d + o_bv, bv.data(), bv.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    UAVMP_CUDA(ctx, cudaMemsetAsync(d + o_ba, 0, 2 * (size_t)P * sizeof(double), st));
    k_rrt_plan_inputs<<<M, 128, 0, st>>>(a.d_plan_q, a.d_path_stage, a.path_cap, seg_time, d, d + o_T);
    UAVMP_CUDA(ctx, cudaGetLastError());
    cudaEventRecord(ctx->ev[2], st);
    QpRaggedIo io;
    io.pos = d; io.bv = d + o_bv; io.ba = d + o_ba; io.bj = d + o_ba; io.T = d + o_T;
    io.coef = d + o_coef; io.solved = a.d_plan_i; io.status = a.d_plan_i + P; io.iters = a.d_plan_i + 2 * P; io.seg_off = nullptr;
    io.order = order;
    r = qp_solve_ragged_dev(ctx, st, ctx->qp_scr, order, P, Sp.data(), io, settings, &qp_l, &aux_l, nullptr, nullptr);
    if (r) return r;
    cudaEventRecord(ctx->ev[3], st);
    UAVMP_CUDA(ctx, cudaMemcpyAsync(pint.data(), a.d_plan_i, pint.size() * sizeof(int), cudaMemcpyDeviceToHost, st));
    cudaEventRecord(ctx->ev[4], st);
    UAVMP_CUDA(ctx, cudaStreamSynchronize(st));
    a.d_plan_coef = d + o_coef;
  }
  // per-query outputs
  long long off = 0;
  int k = 0;
  for (int q = 0; q < B; q++) {
    if (coef_offsets) coef_offsets[q] = off;
    int ok = 0;
    for (int ax = 0; ax < 3; ax++) {
      if (osqp_status) osqp_status[3 * q + ax] = 0;
      if (iters) iters[3 * q + ax] = 0;
    }
    if (n_segments[q]) {
      ok = 1;
      for (int ax = 0; ax < 3; ax++) {
        const int p = 3 * k + ax;
        ok &= pint[p];
        if (osqp_status) osqp_status[3 * q + ax] = pint[P + p];
        if (iters) iters[3 * q + ax] = pint[2 * P + p];
      }
      off += 3 * (long long)n1 * n_segments[q];
      k++;
    }
    qp_solved[q] = ok;
  }
  if (coef_offsets) coef_offsets[B] = off;
  a.plan_total = off;
  uavmp_timings& t = ctx->tm;
  memset(&t, 0, sizeof(t));
  cudaEventElapsedTime(&t.search_ms, ctx->ev[0], ctx->ev[1]);
  if (M > 0) {
    cudaEventElapsedTime(&t.path_ms, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&t.qp_ms, ctx->ev[2], ctx->ev[3]);
    cudaEventElapsedTime(&t.d2h_ms, ctx->ev[3], ctx->ev[4]);
    cudaEventElapsedTime(&t.total_ms, ctx->ev[0], ctx->ev[4]);
  } else {
    t.total_ms = t.search_ms;
  }
  t.search_launches = 1; t.qp_launches = qp_l; t.aux_launches = 1 + (total > 0 ? 1 : 0) + (M > 0 ? 1 : 0) + aux_l;
  return off;
}

int rrt_plan_get_coef(uavmp_ctx* ctx, double* coef, long long cap) {
  if (!ctx->rrt || ctx->rrt->plan_total < 0) return uavmp_fail(ctx, UAVMP_ESTATE, "no uavmp_rrt_plan_batch call has completed");
  RrtState& a = *ctx->rrt;
  if (cap < a.plan_total) return uavmp_fail(ctx, UAVMP_ECAP, "coefficient buffer too small (%lld < %lld)", cap, a.plan_total);
  if (a.plan_total > 0)
    UAVMP_CUDA(ctx, cudaMemcpyAsync(coef, a.d_plan_coef, (size_t)a.plan_total * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  UAVMP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return UAVMP_OK;
}
