// mpc_b200.hpp -- C++ host side above the C-ABI (include/mpc_b200.h): a controller class with the
// reference's interface
//     class MPC { MPC(); vector<double> solve(VectorXd &state, double target_velocity,
//                 vector<double>* x_trajectory, vector<double>* y_trajectory, double dir);
//                 vector<double> run(Vehicle&, vector<double>& ptsx, vector<double>& ptsy, ...); }
//     /root/reference/src/control/MPC.h:11-56, MPC.cpp:160-382
// with the same argument meaning, return vectors and failure behaviour, minus the global mutable
// Config statics (the configuration is a value held by the object) and minus Eigen/CppAD (the state
// is anything indexable, so Eigen::VectorXd works unchanged).  Header-only; link libmpc_b200.so.
#ifndef MPC_B200_HPP
#define MPC_B200_HPP

#include <iostream>
#include <stdexcept>
#include <string>
#include <vector>

#include "mpc_b200.h"

namespace mpcb200 {

// what MPC::run reads from the reference's Vehicle (getX .. getSteering, Vehicle.h)
struct VehiclePose {
  double x, y, psi, v, steering, accel;
};

class MPC {
  mpc_handle *h_;
  mpc_config cfg_;
  double coeffs_[MPC_NCOEF];
  double yaw_lo_, yaw_hi_;       // Config::yawLow / yawHigh of the reference, zero until run()/setRoad()
  int status_, iters_;
  mpc_run_aux aux_;

 public:
  // replaces MPC::MPC() (MPC.cpp:160-179) + the Config statics it reads
  explicit MPC(const mpc_config &cfg, int device = 0) : h_(0), cfg_(cfg), yaw_lo_(0), yaw_hi_(0), status_(0), iters_(0) {
    for (int i = 0; i < MPC_NCOEF; i++) coeffs_[i] = 0.0;
    const int rc = mpc_create(&cfg_, device, &h_);
    if (rc != MPC_OK) throw std::runtime_error(std::string("mpc_create failed (") + std::to_string(rc) + "): " + mpc_last_error());
  }
  MPC(const MPC &) = delete;
  MPC &operator=(const MPC &) = delete;
  virtual ~MPC() { mpc_destroy(h_); }

  // the fitted centre line and yaw bounds that run() leaves in MPC::roadGeometry / Config (MPC.cpp:330,345-352)
  void setRoad(const double *coeffs, int n, double yaw_lo, double yaw_hi) {
    for (int i = 0; i < MPC_NCOEF; i++) coeffs_[i] = i < n ? coeffs[i] : 0.0;
    yaw_lo_ = yaw_lo; yaw_hi_ = yaw_hi;
  }
  const double *polynomial() const { return coeffs_; }
  double yawLow() const { return yaw_lo_; }
  double yawHigh() const { return yaw_hi_; }
  int lastStatus() const { return status_; }     // CppAD::ipopt::solve_result::status_type integer
  int lastIters() const { return iters_; }
  const mpc_config &config() const { return cfg_; }
  // Config::load on a live controller: the handle (device workspace, stream) is kept
  void setConfig(const mpc_config &cfg) {
    const int rc = mpc_set_config(h_, &cfg);
    if (rc != MPC_OK) throw std::runtime_error(std::string("mpc_set_config failed (") + std::to_string(rc) + ")");
    cfg_ = cfg;
  }

  // Opt-in warm start of solve() (off by default, so a drop-in MPC behaves as the reference): the previous solution
  // stays on the device and each solve starts from it moved one stage on (mpc_set_warm_start_one); mu_init is the
  // initial barrier parameter of those solves (0 = Ipopt's 0.1; a start point near the solution helps with a small one).
  void setWarmStart(bool on, double mu_init = 0.0) {
    const int rc = mpc_set_warm_start_one(h_, on ? 1 : 0, mu_init);
    if (rc != MPC_OK) throw std::runtime_error(std::string("mpc_set_warm_start_one failed (") + std::to_string(rc) + ")");
  }

  // MPC::solve, MPC.cpp:183-325.  Returns {x1, y1, psi1, v1, cte1, epsi1, delta0, a0, cost}; appends the N
  // predicted points (stage 0 included) to *x_trajectory / *y_trajectory.  target_velocity and dir are
  // accepted and ignored, as in the reference (MPC.cpp:43-47,87,152).
  template <class Vec>
  std::vector<double> solve(const Vec &state, double target_velocity, std::vector<double> *x_trajectory = 0,
                            std::vector<double> *y_trajectory = 0, double dir = 1) {
    (void)target_velocity; (void)dir;
    double st[6], res[9];
    for (int i = 0; i < 6; i++) st[i] = state[i];
    std::vector<double> tx(cfg_.N), ty(cfg_.N);
    const int rc = mpc_solve_one(h_, st, coeffs_, yaw_lo_, yaw_hi_, res, tx.data(), ty.data(), &status_, &iters_);
    if (rc != MPC_OK) throw std::runtime_error(std::string("mpc_solve_one failed (") + std::to_string(rc) + "): " + mpc_last_error());
    if (status_ != MPC_STATUS_SUCCESS) {   // MPC.cpp:295-303
#ifdef EXIT_ON_IPOPT_FAILURE
      throw std::string("Ipopt failed with ") + std::to_string(status_);
#else
      std::cout << "Ipopt failed with " + std::to_string(status_) << std::endl;
#endif
    }
    if (x_trajectory) {   // MPC.cpp:306-311 (y_trajectory is dereferenced unconditionally there too)
      for (int i = 0; i < cfg_.N; i++) { x_trajectory->push_back(tx[i]); y_trajectory->push_back(ty[i]); }
    }
    return std::vector<double>(res, res + 9);
  }

  // MPC::run, MPC.cpp:327-382.  ptsx/ptsy are transformed to the vehicle frame in place.
  // Returns {x1, y1, psi1, v1, steer in [-1, 1], accel, cte1, epsi1}.
  std::vector<double> run(const VehiclePose &vehicle, std::vector<double> &ptsx, std::vector<double> &ptsy,
                          std::vector<double> *x_trajectory = 0, std::vector<double> *y_trajectory = 0) {
    const double pose[4] = {vehicle.x, vehicle.y, vehicle.psi, vehicle.v};
    double state[6];
    const int rc = mpc_run_prepare(&cfg_, pose, vehicle.steering, ptsx.data(), ptsy.data(), (int)ptsx.size(), state,
                                   coeffs_, &yaw_lo_, &yaw_hi_, &aux_);
    if (rc != MPC_OK) throw std::runtime_error("mpc_run_prepare failed (" + std::to_string(rc) + ")");
    std::vector<double> r = solve(state, aux_.target_speed, x_trajectory, y_trajectory);
    double out[8];
    mpc_run_finish(&cfg_, &aux_, vehicle.v, r.data(), out);
    return std::vector<double>(out, out + 8);
  }
  const mpc_run_aux &lastRun() const { return aux_; }
};

}  // namespace mpcb200
#endif
