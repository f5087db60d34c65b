// fcc_qp.hpp -- C++ host class with the reference's surface, over the CUDA C ABI.
//
// Drop-in for the reference header `src/fcc_qp.hpp` (class fcc_qp::FCCQP,
// FCCQPOptions, FCCQPDetails, FCCQPSolution, FCCQPSolveStatus): same names,
// same constructor / setter / Solve / GetSolution signatures and meaning.  The
// arithmetic runs on a B200 through libfccqp_b200.so (include/fccqp.h); there
// is no CPU fallback -- construction throws std::runtime_error without a GPU.
//
// Header-only on purpose: when <Eigen/Dense> has been included BEFORE this
// header, the Eigen-typed overloads of the reference (Ref<const MatrixXd>, ...,
// FCCQPSolution::z as VectorXd) are enabled, so a C++ caller of the reference
// recompiles unchanged; without Eigen the same methods take the light views
// below (plain pointers + strides) and z is a std::vector<double>.
#pragma once

#include <cmath>
#include <cstddef>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "fccqp.h"

#if defined(EIGEN_CORE_H) || defined(EIGEN_CORE_MODULE_H)
#define FCC_QP_HAVE_EIGEN 1
#endif

namespace fcc_qp {

// src/fcc_qp.hpp:14-17 (+ kNumericalIssue: the GPU path reports a broken KKT solve
// instead of returning NaNs silently)
enum FCCQPSolveStatus { kSuccess = 0, kMaxIterations = 1, kNumericalIssue = 2 };

// src/fcc_qp.hpp:19-28
struct FCCQPDetails {
  int n_iter{};
  double admm_residual_bounds{};
  double admm_residual_friction_cone{};
  double solve_time{};
  double factorization_time{};
  double bounds_viol{};
  double friction_cone_viol{};
  FCCQPSolveStatus solve_status{kSuccess};
};

// src/fcc_qp.hpp:30-35
struct FCCQPOptions {
  int max_iter = 1000;
  double rho = 1e-6;
  double eps_fcone = 1e-3;
  double eps_bound = 1e-6;
  double relaxation = 1.0;   // extension, not in the reference: ADMM over-relaxation (fccqp_options::relaxation)
  int adapt_rho_interval = 0;  // extension, not in the reference: adaptive rho every so many iterations (0 = off)
};

// src/fcc_qp.hpp:37-40
struct FCCQPSolution {
  FCCQPDetails details{};
#ifdef FCC_QP_HAVE_EIGEN
  Eigen::VectorXd z;
#else
  std::vector<double> z;
#endif
};

// Non-owning views used when Eigen is not available (and by the pybind module).
struct ConstMatrixView {
  const double* data;
  int rows, cols;
  std::ptrdiff_t row_stride, col_stride;  // element (i,j) at data[i*row_stride + j*col_stride]
};
struct ConstVectorView {
  const double* data;
  int size;
};

class FCCQP {
 public:
  // src/fcc_qp.hpp:73 / src/fcc_qp.cpp:24-55.  `device` is an extension (CUDA ordinal).
  FCCQP(int num_vars, int num_equality_constraints, int nc, int lambda_c_start, int device = 0)
      : n_vars_(num_vars), n_eq_(num_equality_constraints), nc_(nc), lambda_c_start_(lambda_c_start) {
    check(fccqp_create(num_vars, num_equality_constraints, nc, lambda_c_start, device, &h_));
  }
  ~FCCQP() { fccqp_destroy(h_); }
  FCCQP(const FCCQP&) = delete;
  FCCQP& operator=(const FCCQP&) = delete;
  FCCQP(FCCQP&& o) noexcept
      : h_(o.h_), n_vars_(o.n_vars_), n_eq_(o.n_eq_), nc_(o.nc_), lambda_c_start_(o.lambda_c_start_) {
    o.h_ = nullptr;
  }

  // src/fcc_qp.hpp:75-91.  The reference asserts rho > 0 / n > 0 (compiled out in Release);
  // here the same conditions throw std::invalid_argument.
  void set_rho(double rho) { check(fccqp_set_rho(h_, rho)); }
  void set_max_iter(int n) { check(fccqp_set_max_iter(h_, n)); }
  void set_options(FCCQPOptions opt) {
    fccqp_options o;
    o.max_iter = opt.max_iter; o.adapt_rho_interval = opt.adapt_rho_interval; o.rho = opt.rho; o.relaxation = opt.relaxation;
    o.eps_fcone = opt.eps_fcone; o.eps_bound = opt.eps_bound;
    check(fccqp_set_options(h_, &o));
  }
  void set_warm_start(bool warm_start) { check(fccqp_set_warm_start(h_, warm_start ? 1 : 0)); }

  // src/fcc_qp.hpp:114-117.  Shape mismatches (asserts in the reference, UB in Release)
  // throw std::invalid_argument; too few friction coefficients throws std::out_of_range
  // like the reference's friction_coeffs.at(i) (src/constraint_utils.cpp:32).
  void Solve(ConstMatrixView Q, ConstVectorView b, ConstMatrixView A_eq, ConstVectorView b_eq,
             const std::vector<double>& friction_coeffs, ConstVectorView lb, ConstVectorView ub) {
    if (Q.rows != n_vars_ || Q.cols != n_vars_) throw std::invalid_argument("Q must be num_vars x num_vars");
    if (b.size != n_vars_) throw std::invalid_argument("b must have num_vars entries");
    if (A_eq.cols != n_vars_ && !(n_eq_ == 0 && A_eq.rows == 0))
      throw std::invalid_argument("A_eq must have num_vars columns");
    if (A_eq.rows != n_eq_ || b_eq.size != n_eq_)
      throw std::invalid_argument("A_eq / b_eq must have num_equality_constraints rows");
    if (lb.size != n_vars_ || ub.size != n_vars_) throw std::invalid_argument("lb / ub must have num_vars entries");
    if (static_cast<int>(friction_coeffs.size()) < nc_ / 3)
      throw std::out_of_range("friction_coeffs has fewer than nc/3 entries");
    for (int i = 0; i < n_vars_; ++i)
      if (lb.data[i] > ub.data[i]) throw std::invalid_argument("lb > ub (validate_bounds, src/constraint_utils.cpp:67-75)");
    check(fccqp_solve(h_, Q.data, Q.row_stride, Q.col_stride, b.data, A_eq.data, A_eq.row_stride,
                      A_eq.col_stride, b_eq.data, friction_coeffs.data(),
                      static_cast<int>(friction_coeffs.size()), lb.data, ub.data));
  }

#ifdef FCC_QP_HAVE_EIGEN
  // The reference's exact signature (column-major Refs, arbitrary outer stride).
  void Solve(const Eigen::Ref<const Eigen::MatrixXd>& Q, const Eigen::Ref<const Eigen::VectorXd>& b,
             const Eigen::Ref<const Eigen::MatrixXd>& A_eq, const Eigen::Ref<const Eigen::VectorXd>& b_eq,
             const std::vector<double>& friction_coeffs, const Eigen::Ref<const Eigen::VectorXd>& lb,
             const Eigen::Ref<const Eigen::VectorXd>& ub) {
    Solve(ConstMatrixView{Q.data(), (int)Q.rows(), (int)Q.cols(), 1, (std::ptrdiff_t)Q.outerStride()},
          ConstVectorView{b.data(), (int)b.size()},
          ConstMatrixView{A_eq.data(), (int)A_eq.rows(), (int)A_eq.cols(), 1, (std::ptrdiff_t)A_eq.outerStride()},
          ConstVectorView{b_eq.data(), (int)b_eq.size()}, friction_coeffs,
          ConstVectorView{lb.data(), (int)lb.size()}, ConstVectorView{ub.data(), (int)ub.size()});
  }
#endif

  // src/fcc_qp.cpp:194-207
  FCCQPSolution GetSolution() const {
    FCCQPSolution out;
    out.z.resize(n_vars_);
    fccqp_details d;
    check(fccqp_get_solution(h_, out.z.data(), &d));
    out.details.n_iter = d.n_iter;
    out.details.admm_residual_bounds = d.admm_residual_bounds;
    out.details.admm_residual_friction_cone = d.admm_residual_friction_cone;
    out.details.solve_time = d.solve_time;
    out.details.factorization_time = d.factorization_time;
    out.details.bounds_viol = d.bounds_viol;
    out.details.friction_cone_viol = d.friction_cone_viol;
    out.details.solve_status = static_cast<FCCQPSolveStatus>(d.solve_status);
    return out;
  }

  int contact_vars_start() const { return lambda_c_start_; }  // src/fcc_qp.hpp:121

  // Extensions: the warm-start state the reference keeps private (src/fcc_qp.hpp:147-153).
  void GetWarmState(double* x, double* mu_x, double* mu_lambda_c) const {
    check(fccqp_get_warm_state(h_, x, mu_x, mu_lambda_c));
  }
  void SetWarmState(const double* x, const double* mu_x, const double* mu_lambda_c) {
    check(fccqp_set_warm_state(h_, x, mu_x, mu_lambda_c));
  }
  int num_vars() const { return n_vars_; }
  int num_equality_constraints() const { return n_eq_; }
  int num_contact_vars() const { return nc_; }

 private:
  static void check(int rc) {
    if (rc == FCCQP_OK) return;
    const std::string msg = fccqp_last_error();
    if (rc == FCCQP_E_INVALID) throw std::invalid_argument(msg);
    throw std::runtime_error(msg);
  }
  fccqp_handle h_ = nullptr;
  const int n_vars_, n_eq_, nc_, lambda_c_start_;
};

// ---------------------------------------------------------------------------
// Batched solver (extension; the reference solves one QP per call): B QPs of identical dimensions per
// Solve through fccqp_batch_solve.  Same option / warm-start semantics as FCCQP, applied lane-wise;
// the carried state (x, mu_x, mu_lambda_c) of every lane lives in this object.
// ---------------------------------------------------------------------------
struct FCCQPBatchProblem {
  // dense row-major stacks: Q [B,n,n], b [B,n], A_eq [B,m,n], b_eq [B,m], friction_coeffs [B,nc/3], lb/ub [B,n]
  const double* Q = nullptr;
  const double* b = nullptr;
  const double* A_eq = nullptr;
  const double* b_eq = nullptr;
  const double* friction_coeffs = nullptr;
  const double* lb = nullptr;
  const double* ub = nullptr;
  bool shared_structure = false;   // Q is [n,n] and A_eq is [m,n]: one pair for the whole batch
  bool shared_bounds = false;      // lb / ub are [n]
  bool shared_friction = false;    // friction_coeffs is [nc/3]
};

// Device-resident batch (extension): every pointer is DEVICE memory of `device`, strides in elements (batch stride 0 =
// one array shared by all QPs), outputs / carried state caller-owned ([B,n] [B,n] [B,nc], [B] ints, [B] doubles; the
// four per-QP scalars may be null).  What DLPack-able tensors (torch CUDA, cupy) boil down to.
struct FCCQPBatchDeviceIO {
  const double* Q = nullptr;      std::ptrdiff_t q_batch_stride = 0, q_row_stride = 0, q_col_stride = 1;
  const double* b = nullptr;      std::ptrdiff_t b_batch_stride = 0;
  const double* A_eq = nullptr;   std::ptrdiff_t a_batch_stride = 0, a_row_stride = 0, a_col_stride = 1;
  const double* b_eq = nullptr;   std::ptrdiff_t beq_batch_stride = 0;
  const double* friction_coeffs = nullptr;  std::ptrdiff_t mu_batch_stride = 0;
  const double* lb = nullptr;     std::ptrdiff_t lb_batch_stride = 0;
  const double* ub = nullptr;     std::ptrdiff_t ub_batch_stride = 0;
  double *x = nullptr, *mu_x = nullptr, *mu_lambda_c = nullptr;
  int *n_iter = nullptr, *solve_status = nullptr;
  double *admm_residual_bounds = nullptr, *admm_residual_friction_cone = nullptr, *bounds_viol = nullptr, *friction_cone_viol = nullptr;
  void* stream = nullptr;         // cudaStream_t the solve is enqueued on (asynchronous unless `device_seconds` is asked for)
  int device = 0;
};

struct FCCQPBatchSolution {
  int batch = 0;
  std::vector<double> z;                       // [B,n]
  std::vector<int> n_iter, solve_status;       // [B]
  std::vector<double> admm_residual_bounds, admm_residual_friction_cone, bounds_viol, friction_cone_viol;  // [B]
  double solve_time = 0.0;                     // wall seconds of the whole call
};

class FCCQPBatch {
 public:
  FCCQPBatch(int num_vars, int num_equality_constraints, int nc, int lambda_c_start, int device = 0)
      : n_(num_vars), m_(num_equality_constraints), nc_(nc), lcs_(lambda_c_start), device_(device) {
    if (nc % 3 != 0) throw std::invalid_argument("nc must be a multiple of 3 (src/fcc_qp.cpp:32)");
    if (lambda_c_start < 0 || lambda_c_start + nc > num_vars)
      throw std::invalid_argument("lambda_c_start + nc must be <= num_vars (src/fcc_qp.cpp:33)");
    fccqp_default_options(&opt_);
  }
  // Several devices of one box: every Solve() is split into contiguous shards, one per device, inside one call
  // (fccqp_batch_solve_multi).
  FCCQPBatch(int num_vars, int num_equality_constraints, int nc, int lambda_c_start, std::vector<int> devices)
      : FCCQPBatch(num_vars, num_equality_constraints, nc, lambda_c_start, devices.empty() ? 0 : devices[0]) {
    if (devices.empty()) throw std::invalid_argument("device list is empty");
    devices_.assign(devices.begin(), devices.end());
  }
  // fccqp_structure (| FCCQP_STRUCTURE_REFINE) of the batched calls; default FCCQP_STRUCTURE_AUTO
  void set_structure(int structure) { structure_ = structure; }
  // One rho for every lane (clears a per-lane rho), as on FCCQP.
  void set_rho(double rho) {
    if (!(rho > 0)) throw std::invalid_argument("rho must be > 0");
    opt_.rho = rho;
    rho_lanes_.clear();
  }
  // Per lane (fccqp_batch_solve_rho): lane i of the next host Solve is solved as an FCCQP after set_rho(rho_lanes[i]),
  // and the vector, owned by this object, then holds the rho each lane ended with (rho_lanes()): with adaptive rho the
  // next warm Solve continues from it.  One entry per lane of that Solve, each finite and > 0.
  void set_rho(const std::vector<double>& rho_lanes) {
    if (rho_lanes.empty()) throw std::invalid_argument("rho_lanes is empty");
    for (double r : rho_lanes)
      if (!(r > 0 && std::isfinite(r))) throw std::invalid_argument("every per-lane rho must be finite and > 0");
    rho_lanes_ = rho_lanes;
  }
  const std::vector<double>& rho_lanes() const { return rho_lanes_; }
  void set_max_iter(int n) { if (n <= 0) throw std::invalid_argument("max_iter must be > 0"); opt_.max_iter = n; }
  void set_options(FCCQPOptions o) {
    opt_.max_iter = o.max_iter; opt_.rho = o.rho; opt_.eps_fcone = o.eps_fcone; opt_.eps_bound = o.eps_bound;
    opt_.relaxation = o.relaxation; opt_.adapt_rho_interval = o.adapt_rho_interval;
  }
  void set_warm_start(bool warm_start) { warm_ = warm_start; warm_lanes_.clear(); }
  // Per lane (fccqp_batch_desc::warm_lanes): lane i of the next host Solve is solved as an FCCQP after
  // set_warm_start(warm_lanes[i] != 0).  The vector must hold one entry per lane of that Solve.
  void set_warm_start(const std::vector<uint8_t>& warm_lanes) {
    if (warm_lanes.empty()) throw std::invalid_argument("warm_lanes is empty");
    warm_ = true;
    warm_lanes_ = warm_lanes;
  }

  // Host pointers; blocks until the results are back.
  void Solve(int batch, const FCCQPBatchProblem& p) {
    const size_t B = (size_t)batch, n = (size_t)n_, m = (size_t)m_, nc = (size_t)nc_;
    if (!warm_lanes_.empty() && warm_lanes_.size() != B)
      throw std::invalid_argument("warm_lanes has " + std::to_string(warm_lanes_.size()) + " entries, the batch " +
                                  std::to_string(batch));
    if (!rho_lanes_.empty() && rho_lanes_.size() != B)
      throw std::invalid_argument("rho_lanes has " + std::to_string(rho_lanes_.size()) + " entries, the batch " +
                                  std::to_string(batch));
    const bool carry = warm_ && sol_.batch == batch;    // like a never-solved FCCQP, a fresh lane starts from zero
    if (!carry) { sol_.z.assign(B * n, 0.0); mu_x_.assign(B * n, 0.0); mu_c_.assign(B * nc, 0.0); }
    sol_.batch = batch;
    sol_.n_iter.resize(B); sol_.solve_status.resize(B);
    sol_.admm_residual_bounds.resize(B); sol_.admm_residual_friction_cone.resize(B);
    sol_.bounds_viol.resize(B); sol_.friction_cone_viol.resize(B);
    fccqp_batch_desc d{};
    d.abi_version = FCCQP_ABI_VERSION; d.batch = batch; d.n = n_; d.m = m_; d.nc = nc_; d.lambda_c_start = lcs_;
    d.device = device_; d.memory_space = FCCQP_MEM_HOST; d.precision = FCCQP_PRECISION_FP64; d.warm_start = warm_ ? 1 : 0;
    d.options = opt_;
    d.Q = p.Q; d.q_batch_stride = p.shared_structure ? 0 : (int64_t)(n * n); d.q_row_stride = n_; d.q_col_stride = 1;
    d.b = p.b; d.b_batch_stride = n_;
    d.A_eq = p.A_eq; d.a_batch_stride = p.shared_structure ? 0 : (int64_t)(m * n); d.a_row_stride = n_; d.a_col_stride = 1;
    d.b_eq = p.b_eq; d.beq_batch_stride = m_;
    d.friction_coeffs = p.friction_coeffs; d.mu_batch_stride = p.shared_friction ? 0 : nc_ / 3;
    d.lb = p.lb; d.lb_batch_stride = p.shared_bounds ? 0 : n_;
    d.ub = p.ub; d.ub_batch_stride = p.shared_bounds ? 0 : n_;
    d.x = sol_.z.data(); d.mu_x = mu_x_.data(); d.mu_lambda_c = mu_c_.data();
    d.n_iter = sol_.n_iter.data(); d.status = sol_.solve_status.data();
    d.res_bounds = sol_.admm_residual_bounds.data(); d.res_fcone = sol_.admm_residual_friction_cone.data();
    d.bounds_viol = sol_.bounds_viol.data(); d.fcone_viol = sol_.friction_cone_viol.data();
    double secs = 0.0;
    d.device_seconds = &secs;
    d.structure = structure_;
    d.warm_lanes = warm_lanes_.empty() ? nullptr : warm_lanes_.data();
    double* rho = rho_lanes_.empty() ? nullptr : rho_lanes_.data();
    const int rc = devices_.size() > 1 ? fccqp_batch_solve_multi_rho(&d, rho, devices_.data(), (int32_t)devices_.size())
                                       : fccqp_batch_solve_rho(&d, rho);
    if (rc == FCCQP_E_INVALID) throw std::invalid_argument(fccqp_last_error());
    if (rc != FCCQP_OK) throw std::runtime_error(fccqp_last_error());
    sol_.solve_time = secs;
  }
  const FCCQPBatchSolution& GetSolution() const { return sol_; }

  // Device pointers; enqueued on io.stream and NOT waited for unless device_seconds is given (then the call
  // returns after the kernels and *device_seconds holds their time).  io.x / mu_x / mu_lambda_c are the carried
  // state when set_warm_start(true).  warm_lanes: optional DEVICE [batch] mask, one byte per lane, that replaces
  // set_warm_start for this call (lane i warm where warm_lanes[i] != 0; read by the kernels when they run).  rho:
  // optional DEVICE [batch] per-lane rho that replaces the options' rho for this call, read and overwritten in place
  // with the rho each lane ended with (fccqp_batch_solve_rho).
  void SolveDevice(int batch, const FCCQPBatchDeviceIO& io, double* device_seconds = nullptr,
                   const uint8_t* warm_lanes = nullptr) {
    SolveDevice(batch, io, device_seconds, warm_lanes, nullptr);
  }
  void SolveDevice(int batch, const FCCQPBatchDeviceIO& io, double* device_seconds, const uint8_t* warm_lanes,
                   double* rho) {
    fccqp_batch_desc d{};
    d.abi_version = FCCQP_ABI_VERSION; d.batch = batch; d.n = n_; d.m = m_; d.nc = nc_; d.lambda_c_start = lcs_;
    d.device = io.device; d.memory_space = FCCQP_MEM_DEVICE; d.precision = FCCQP_PRECISION_FP64; d.warm_start = warm_ ? 1 : 0;
    d.options = opt_;
    d.Q = io.Q; d.q_batch_stride = io.q_batch_stride; d.q_row_stride = io.q_row_stride; d.q_col_stride = io.q_col_stride;
    d.b = io.b; d.b_batch_stride = io.b_batch_stride;
    d.A_eq = io.A_eq; d.a_batch_stride = io.a_batch_stride; d.a_row_stride = io.a_row_stride; d.a_col_stride = io.a_col_stride;
    d.b_eq = io.b_eq; d.beq_batch_stride = io.beq_batch_stride;
    d.friction_coeffs = io.friction_coeffs; d.mu_batch_stride = io.mu_batch_stride;
    d.lb = io.lb; d.lb_batch_stride = io.lb_batch_stride;
    d.ub = io.ub; d.ub_batch_stride = io.ub_batch_stride;
    d.x = io.x; d.mu_x = io.mu_x; d.mu_lambda_c = io.mu_lambda_c;
    d.n_iter = io.n_iter; d.status = io.solve_status;
    d.res_bounds = io.admm_residual_bounds; d.res_fcone = io.admm_residual_friction_cone;
    d.bounds_viol = io.bounds_viol; d.fcone_viol = io.friction_cone_viol;
    d.stream = io.stream;
    d.device_seconds = device_seconds;
    d.structure = structure_;
    d.warm_lanes = warm_lanes;
    const int rc = fccqp_batch_solve_rho(&d, rho);
    if (rc == FCCQP_E_INVALID) throw std::invalid_argument(fccqp_last_error());
    if (rc != FCCQP_OK) throw std::runtime_error(fccqp_last_error());
  }
  int num_vars() const { return n_; }
  int num_equality_constraints() const { return m_; }
  int num_contact_vars() const { return nc_; }
  int contact_vars_start() const { return lcs_; }

 private:
  const int n_, m_, nc_, lcs_, device_;
  fccqp_options opt_{};
  bool warm_ = false;
  std::vector<uint8_t> warm_lanes_;   // per-lane warm start of the host Solve (empty: warm_ for every lane)
  std::vector<double> rho_lanes_;     // per-lane rho of the host Solve, written back by it (empty: opt_.rho for every lane)
  int structure_ = FCCQP_STRUCTURE_AUTO;
  std::vector<int32_t> devices_;
  FCCQPBatchSolution sol_;
  std::vector<double> mu_x_, mu_c_;
};

}  // namespace fcc_qp
