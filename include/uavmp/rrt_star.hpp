// include/uavmp/rrt_star.hpp — C++ shim with the reference's class interface over the C-ABI (include/uavmp.h).
//
// Drop-in for path_searching::RRTStar (reference: src/planner/path_searching/include/path_searching/rrt_star.h:30-101): same method
// names, argument meaning and return codes (REACH_END = 1, NO_PATH_FOUND = 2, :62-65).  As in the reference, search() leaves `path`
// empty (rrt_star.cpp:366,403 clear it) and the result is getOptimalPath(), which keeps its previous value when a search does not
// rewrite it (reset() does not clear optimal_path_).  Two things the reference leaves to chance are explicit: setQuerySeed() (the
// reference seeds every sample from std::random_device) and the sample budget that stands for `max_tolerance_time` (uavmp.h).
// Compiled only where Eigen exists; nothing in this repository includes it except the compile check in tests/host/shim_check.cpp.
#pragma once
#include <Eigen/Eigen>
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <vector>

#include "../uavmp.h"

namespace uavmp {

class RRTStar {
 public:
  typedef std::shared_ptr<RRTStar> Ptr;
  enum { REACH_END = 1, NO_PATH_FOUND = 2 };

  explicit RRTStar(uavmp_ctx* shared = nullptr, int device = 0) : ctx_(shared), owned_(shared == nullptr) {
    if (owned_ && uavmp_ctx_create(&ctx_, device) != UAVMP_OK) throw std::runtime_error("uavmp: no CUDA device (no CPU fallback)");
  }
  ~RRTStar() { if (owned_) uavmp_ctx_destroy(ctx_); }
  RRTStar(const RRTStar&) = delete;
  RRTStar& operator=(const RRTStar&) = delete;

  // void setParam(ros::NodeHandle& nh): rrt_star/max_tree_node_num, step_length, search_radius, collision_check_resolution (rrt_star.cpp:7-10);
  // rrt_star/max_tolerance_time (:11) becomes a budget of drawn samples
  void setParam(int max_tree_node_num = 100000, double step_length = 0.5, double search_radius = 0.5,
                double collision_check_resolution = 0.05, double sample_budget = 100000.0, int path_cap_nodes = 4096) {
    check(uavmp_rrt_set_params(ctx_, max_tree_node_num, step_length, search_radius, collision_check_resolution, sample_budget, path_cap_nodes));
  }
  void setQuerySeed(uint64_t seed) { seed_ = seed; }
  void setGridMap(const std::vector<char>& occupancy_buffer_inflate, const Eigen::Vector3i& map_voxel_num,
                  const Eigen::Vector3d& map_origin, const Eigen::Vector3d& map_size, double resolution) {
    check(uavmp_map_set(ctx_, reinterpret_cast<const int8_t*>(occupancy_buffer_inflate.data()), map_voxel_num(0),
                        map_voxel_num(1), map_voxel_num(2), map_origin.data(), map_size.data(), resolution, nullptr, 0));
  }
  void init() {}   // node pools and kd-trees are per-warp arenas on the device (rrt_star.cpp:66-84)
  void reset() {}  // (rrt_star.cpp:86-101)

  // int search(Eigen::Vector3d start, Eigen::Vector3d end, std::vector<Eigen::Vector3d>& path)   (rrt_star.h:93)
  int search(Eigen::Vector3d start, Eigen::Vector3d end, std::vector<Eigen::Vector3d>& path) {
    (void)path;
    int status = 0;
    long long off[2] = {0, 0};
    long long n = uavmp_rrt_search_batch(ctx_, 1, start.data(), end.data(), &seed_, &status, nullptr, nullptr, nullptr, nullptr, off);
    if (n < 0) throw std::runtime_error(uavmp_last_error(ctx_));
    if (n > 0) {
      std::vector<double> xyz(3 * (size_t)n);
      check(uavmp_rrt_get_paths(ctx_, xyz.data(), n));
      optimal_path_.clear();
      for (long long i = 0; i < n; i++) optimal_path_.push_back(Eigen::Vector3d(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]));
    }
    return status;
  }
  std::vector<Eigen::Vector3d> getOptimalPath() { return optimal_path_; }
  long long searchBatch(int B, const double* start, const double* end, const uint64_t* query_seed, int* status, long long* path_offsets) {
    return uavmp_rrt_search_batch(ctx_, B, start, end, query_seed, status, nullptr, nullptr, nullptr, nullptr, path_offsets);
  }
  // test_minimum_jerk.cpp's GoalCallback for B queries at once (uavmp_rrt_plan_batch): search, then every optimal-path point a
  // waypoint, T_s = seg_time, one QP per axis.  n_segments[q] = S_q (0: no QP posed); query q's coefficients are
  // coef[coef_offsets[q] .. coef_offsets[q + 1]), axis-major [3][(order+1) S_q], each axis in MinimumControl::getCoef1d's layout.
  // start_vel may be NULL (zero).  Returns the total number of coefficients.
  long long planMinimumJerkBatch(int B, const double* start, const double* start_vel, const double* end, const uint64_t* query_seed,
                                 int* status, int* n_segments, int* qp_solved, std::vector<long long>& coef_offsets,
                                 std::vector<double>& coef, int order = 5, double seg_time = 1.0,
                                 const uavmp_osqp_settings* settings = nullptr) {
    coef_offsets.assign((size_t)B + 1, 0);
    long long n = uavmp_rrt_plan_batch(ctx_, B, start, start_vel, end, query_seed, order, seg_time, settings, status, n_segments, qp_solved,
                                       coef_offsets.data(), nullptr, nullptr);
    if (n < 0) throw std::runtime_error(uavmp_last_error(ctx_));
    coef.resize((size_t)n);
    if (n > 0) check(uavmp_rrt_plan_get_coef(ctx_, coef.data(), n));
    return n;
  }
  uavmp_ctx* context() { return ctx_; }

 private:
  void check(int rc) { if (rc < 0) throw std::runtime_error(uavmp_last_error(ctx_)); }
  uavmp_ctx* ctx_ = nullptr;
  bool owned_;
  uint64_t seed_ = 0;
  std::vector<Eigen::Vector3d> optimal_path_;
};

}  // namespace uavmp
