// include/uavmp/minimum_control.hpp — C++ shim with the reference's class interface over the C-ABI (include/uavmp.h).
//
// Drop-in for traj_optimization::MinimumControl (reference: src/planner/traj_optimization/include/traj_optimization/
// minimum_control.h:10-49): bool solve(VectorXd& pos_1d, Vector2d& bound_vel, Vector2d& bound_acc, VectorXd& time_vec), one axis
// per call, true only when OSQP reports SOLVED (3rd/osqp-eigen/src/Solver.cpp:181-187); getCoef1d() returns the 6S coefficients,
// segment-major, ascending power, local time; a failed solve leaves the previous coefficients in place (minimum_control.cpp:182).
// Compiled only where Eigen exists.
#pragma once
#include <Eigen/Eigen>
#include <algorithm>
#include <iostream>
#include <stdexcept>
#include <vector>

#include "../uavmp.h"

namespace uavmp {

class MinimumControl {
 public:
  explicit MinimumControl(uavmp_ctx* ctx, int order = 5) : ctx_(ctx), order_(order) { uavmp_osqp_settings_default(&settings_); }

  bool solve(Eigen::VectorXd& pos_1d, Eigen::Vector2d& bound_vel, Eigen::Vector2d& bound_acc, Eigen::VectorXd& time_vec) {
    const int S = (int)time_vec.size();
    Eigen::VectorXd coef((order_ + 1) * S);
    double bj[2] = {0.0, 0.0};
    int solved = 0;
    int rc = uavmp_minctrl_solve_batch(ctx_, order_, S, 1, pos_1d.data(), bound_vel.data(), bound_acc.data(),
                                       order_ == 7 ? bj : nullptr, time_vec.data(), &settings_, coef.data(), &solved, nullptr,
                                       nullptr);
    if (rc < 0) throw std::runtime_error(uavmp_last_error(ctx_));
    if (!solved) { std::cout << "solver solve failed!" << std::endl; return false; }
    coef_1d_ = coef;
    return true;
  }
  // B problems with a different segment count each, in one call (uavmp_minctrl_solve_ragged_batch): pos_1d[b] has S_b + 1 waypoints,
  // time_vec[b] S_b durations; coef[b] receives (order+1) S_b coefficients (getCoef1d's layout), solved[b] what solve() would return.
  // Results are bit-identical to calling solve() per problem; coef_1d_ is not touched.
  void solveBatchRagged(const std::vector<Eigen::VectorXd>& pos_1d, const std::vector<Eigen::Vector2d>& bound_vel,
                        const std::vector<Eigen::Vector2d>& bound_acc, const std::vector<Eigen::VectorXd>& time_vec,
                        std::vector<Eigen::VectorXd>& coef, std::vector<bool>& solved) {
    const int B = (int)time_vec.size();
    std::vector<int> S(B);
    std::vector<double> pos, T, bv(2 * (size_t)B), ba(2 * (size_t)B), bj(2 * (size_t)B, 0.0);
    size_t n_coef = 0;
    for (int b = 0; b < B; b++) {
      S[b] = (int)time_vec[b].size();
      pos.insert(pos.end(), pos_1d[b].data(), pos_1d[b].data() + pos_1d[b].size());
      T.insert(T.end(), time_vec[b].data(), time_vec[b].data() + S[b]);
      bv[2 * b] = bound_vel[b](0); bv[2 * b + 1] = bound_vel[b](1);
      ba[2 * b] = bound_acc[b](0); ba[2 * b + 1] = bound_acc[b](1);
      n_coef += (size_t)(order_ + 1) * S[b];
    }
    std::vector<double> out(n_coef);
    std::vector<int> ok(B);
    int rc = uavmp_minctrl_solve_ragged_batch(ctx_, order_, B, S.data(), pos.data(), bv.data(), ba.data(), order_ == 7 ? bj.data() : nullptr,
                                              T.data(), &settings_, out.data(), ok.data(), nullptr, nullptr);
    if (rc < 0) throw std::runtime_error(uavmp_last_error(ctx_));
    coef.resize(B);
    solved.resize(B);
    size_t o = 0;
    for (int b = 0; b < B; b++) {
      const int n = (order_ + 1) * S[b];
      coef[b] = Eigen::VectorXd(n);
      std::copy(out.data() + o, out.data() + o + n, coef[b].data());
      solved[b] = ok[b] != 0;
      o += n;
    }
  }
  Eigen::VectorXd getCoef1d() { return coef_1d_; }
  void reset() { coef_1d_.setZero(); }
  uavmp_osqp_settings& settings() { return settings_; }

 private:
  uavmp_ctx* ctx_;
  int order_;
  uavmp_osqp_settings settings_;
  Eigen::VectorXd coef_1d_;
};

}  // namespace uavmp
