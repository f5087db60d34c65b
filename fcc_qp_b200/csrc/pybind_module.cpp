// pybind11 module `fcc_qp_solver`: the reference's Python surface (src/main.cpp:19-56)
// over the B200 host class in include/fcc_qp.hpp.  Same class names, same attribute
// names (eps_bounds / eps_friction_cone renames included), same keyword arguments.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <cstdint>
#include <string>
#include <vector>

#include "fcc_qp.hpp"

namespace py = pybind11;

using fcc_qp::FCCQPBatch;
using fcc_qp::FCCQPBatchDeviceIO;
using fcc_qp::FCCQPBatchProblem;
using fcc_qp::FCCQPBatchSolution;
using fcc_qp::ConstMatrixView;
using fcc_qp::ConstVectorView;
using fcc_qp::FCCQP;
using fcc_qp::FCCQPDetails;
using fcc_qp::FCCQPOptions;
using fcc_qp::FCCQPSolution;

namespace {

// Any-layout float64 matrix (dtype conversions are copies, like pybind's Eigen caster;
// C- or F-ordered float64 arrays are consumed in place -- the reference's caster copies
// C-ordered ones, pybind11/eigen/matrix.h:516-533).
using Mat = py::array_t<double, py::array::forcecast>;
using Vec = py::array_t<double, py::array::c_style | py::array::forcecast>;

ConstMatrixView mat_view(const Mat& a, const char* name) {
  if (a.ndim() != 2) throw py::type_error(std::string(name) + " must be a 2-D array");
  return ConstMatrixView{a.data(), (int)a.shape(0), (int)a.shape(1),
                         (std::ptrdiff_t)(a.strides(0) / (py::ssize_t)sizeof(double)),
                         (std::ptrdiff_t)(a.strides(1) / (py::ssize_t)sizeof(double))};
}
ConstVectorView vec_view(const Vec& a, const char* name) {
  if (a.ndim() != 1) throw py::type_error(std::string(name) + " must be a 1-D array");
  return ConstVectorView{a.data(), (int)a.shape(0)};
}

// ---- batched entry point: contiguous float64 host stacks (numpy) ...
using Stack = py::array_t<double, py::array::c_style | py::array::forcecast>;

// ... or device tensors through the DLPack protocol (any object with __dlpack__: torch CUDA tensors, cupy arrays).
// Minimal restatement of the DLPack C structs (dlpack.h, ABI-stable since v0.2).
struct DLDevice_ { int32_t device_type; int32_t device_id; };
struct DLDataType_ { uint8_t code; uint8_t bits; uint16_t lanes; };
struct DLTensor_ { void* data; DLDevice_ device; int32_t ndim; DLDataType_ dtype; int64_t* shape; int64_t* strides; uint64_t byte_offset; };
struct DLManagedTensor_ { DLTensor_ dl_tensor; void* manager_ctx; void (*deleter)(DLManagedTensor_*); };
constexpr int kDLCUDA = 2, kDLInt = 0, kDLUInt = 1, kDLFloat = 2, kDLBool = 6;

struct DevView {
  void* data = nullptr;
  int ndim = 0, device = 0;
  int64_t shape[3] = {0, 0, 0}, stride[3] = {0, 0, 0};
};

// Consumes the capsule at once (pointer, shape and strides are copied out; the caller keeps the tensor object alive).
// code kDLUInt with bits 8 also takes kDLBool (one byte per element): the per-lane warm-start mask.
DevView dev_view(const py::object& obj, const char* name, int code, int bits, int max_ndim) {
  if (!py::hasattr(obj, "__dlpack__")) throw py::type_error(std::string(name) + ": expected an object with __dlpack__ (device tensor)");
  py::capsule cap = obj.attr("__dlpack__")();
  if (std::string(cap.name() ? cap.name() : "") != "dltensor") throw py::type_error(std::string(name) + ": not a fresh DLPack capsule");
  auto* mt = static_cast<DLManagedTensor_*>(PyCapsule_GetPointer(cap.ptr(), "dltensor"));
  const DLTensor_& t = mt->dl_tensor;
  DevView v;
  std::string err;
  if (t.device.device_type != kDLCUDA) err = ": must live in CUDA device memory (no CPU solve path; pass numpy arrays to Solve for host data)";
  else if (!(t.dtype.code == code || (code == kDLUInt && t.dtype.code == kDLBool)) || t.dtype.bits != bits || t.dtype.lanes != 1)
    err = std::string(": must be ") + (code == kDLFloat ? "float64" : code == kDLInt ? "int32" : "bool or uint8");
  else if (t.ndim < 1 || t.ndim > max_ndim) err = ": wrong number of dimensions";
  if (err.empty()) {
    v.data = static_cast<char*>(t.data) + t.byte_offset;
    v.ndim = t.ndim; v.device = t.device.device_id;
    int64_t run = 1;
    for (int i = t.ndim - 1; i >= 0; --i) {
      v.shape[i] = t.shape[i];
      v.stride[i] = t.strides ? t.strides[i] : run;
      run *= t.shape[i];
    }
  }
  PyCapsule_SetName(cap.ptr(), "used_dltensor");
  if (mt->deleter) mt->deleter(mt);
  if (!err.empty()) throw py::type_error(std::string(name) + err);
  return v;
}

// [B, d] (or [d] shared by all QPs) vector stack: pointer + batch stride; the last dimension must be unit-stride
void vec_io(const DevView& v, int B, int d, const char* name, const double*& ptr, std::ptrdiff_t& bs, bool allow_longer = false) {
  const int last = v.ndim - 1;
  const bool ok_len = allow_longer ? v.shape[last] >= d : v.shape[last] == d;
  if (v.ndim > 2 || !ok_len || (v.ndim == 2 && v.shape[0] != B))
    throw py::value_error(std::string(name) + " must be [B," + std::to_string(d) + "] or [" + std::to_string(d) + "]");
  if (v.shape[last] > 1 && v.stride[last] != 1) throw py::value_error(std::string(name) + ": last dimension must be contiguous");
  ptr = static_cast<const double*>(v.data);
  bs = v.ndim == 2 ? (std::ptrdiff_t)v.stride[0] : 0;
}

template <class T>
T* out_io(const DevView& v, int64_t rows, int64_t cols, const char* name) {
  const bool ok = cols == 0 ? (v.ndim == 1 && v.shape[0] == rows)
                            : (v.ndim == 2 && v.shape[0] == rows && v.shape[1] == cols && (cols <= 1 || v.stride[1] == 1) &&
                               (rows <= 1 || v.stride[0] == cols));
  if (!ok) throw py::value_error(std::string(name) + ": expected a contiguous output of the documented shape");
  return static_cast<T*>(v.data);
}

}  // namespace

PYBIND11_MODULE(fcc_qp_solver, m) {
  m.doc() = "B200-native FCCQP solver with the Python surface of Brian-Acosta/fcc_qp";

  py::class_<FCCQPDetails>(m, "FCCQPDetails")
      .def_readwrite("n_iter", &FCCQPDetails::n_iter)
      .def_readwrite("eps_bounds", &FCCQPDetails::admm_residual_bounds)
      .def_readwrite("eps_friction_cone", &FCCQPDetails::admm_residual_friction_cone)
      .def_readwrite("bounds_viol", &FCCQPDetails::bounds_viol)
      .def_readwrite("friction_cone_viol", &FCCQPDetails::friction_cone_viol)
      .def_readwrite("solve_time", &FCCQPDetails::solve_time)
      .def_readwrite("factorization_time", &FCCQPDetails::factorization_time)
      // superset of the reference binding: status is computed there but not exposed
      .def_property_readonly("solve_status", [](const FCCQPDetails& d) { return (int)d.solve_status; });

  py::class_<FCCQPOptions>(m, "FCCQPOptions")
      .def(py::init<>())
      .def_readwrite("max_iter", &FCCQPOptions::max_iter)
      .def_readwrite("rho", &FCCQPOptions::rho)
      .def_readwrite("eps_fcone", &FCCQPOptions::eps_fcone)
      .def_readwrite("eps_bound", &FCCQPOptions::eps_bound)
      .def_readwrite("relaxation", &FCCQPOptions::relaxation)    // extension, default 1.0 = the reference
      .def_readwrite("adapt_rho_interval", &FCCQPOptions::adapt_rho_interval);   // extension, default 0 = the reference's fixed rho

  py::class_<FCCQPSolution>(m, "FCCQPSolution")
      .def_readwrite("details", &FCCQPSolution::details)
      .def_property(
          "z",
          [](const FCCQPSolution& s) { return py::array_t<double>((py::ssize_t)s.z.size(), s.z.data()); },
          [](FCCQPSolution& s, const std::vector<double>& v) { s.z = v; });

  py::class_<FCCQP>(m, "FCCQP")
      .def(py::init<int, int, int, int, int>(), py::arg("num_vars"), py::arg("num_equality_constraints"),
           py::arg("nc"), py::arg("lambda_c_start"), py::arg("device") = 0)
      .def("set_rho", &FCCQP::set_rho)
      .def("set_max_iter", &FCCQP::set_max_iter)
      .def("set_warm_start", &FCCQP::set_warm_start)
      .def("set_options", &FCCQP::set_options)
      .def("contact_vars_start", &FCCQP::contact_vars_start)
      .def(
          "Solve",
          [](FCCQP& self, const Mat& Q, const Vec& b, const Mat& A_eq, const Vec& b_eq,
             const std::vector<double>& friction_coeffs, const Vec& lb, const Vec& ub) {
            const ConstMatrixView q = mat_view(Q, "Q");
            ConstMatrixView a = mat_view(A_eq, "A_eq");
            const ConstVectorView bv = vec_view(b, "b"), beq = vec_view(b_eq, "b_eq");
            const ConstVectorView l = vec_view(lb, "lb"), u = vec_view(ub, "ub");
            py::gil_scoped_release release;  // the reference holds the GIL for the whole Solve
            self.Solve(q, bv, a, beq, friction_coeffs, l, u);
          },
          py::arg("Q"), py::arg("b"), py::arg("A_eq"), py::arg("b_eq"), py::arg("friction_coeffs"),
          py::arg("lb"), py::arg("ub"))
      .def("GetSolution", &FCCQP::GetSolution)
      .def("GetWarmState",
           [](const FCCQP& self) {
             py::array_t<double> x(self.num_vars()), mx(self.num_vars()), mc(self.num_contact_vars());
             self.GetWarmState(x.mutable_data(), mx.mutable_data(), mc.mutable_data());
             return py::make_tuple(x, mx, mc);
           })
      .def("SetWarmState", [](FCCQP& self, const Vec& x, const Vec& mx, const Vec& mc) {
        if (x.size() != self.num_vars() || mx.size() != self.num_vars() || mc.size() != self.num_contact_vars())
          throw py::value_error("warm state arrays must be [num_vars], [num_vars], [nc]");
        self.SetWarmState(x.data(), mx.data(), mc.data());
      });

  // ---- batched extension: fcc_qp::FCCQPBatch (include/fcc_qp.hpp) -- B QPs per Solve, lane-wise warm start
  py::class_<FCCQPBatchSolution>(m, "FCCQPBatchSolution")
      .def_readonly("batch", &FCCQPBatchSolution::batch)
      .def_readonly("solve_time", &FCCQPBatchSolution::solve_time)
      .def_property_readonly("z", [](const FCCQPBatchSolution& s) {
        const py::ssize_t B = s.batch, n = B ? (py::ssize_t)s.z.size() / B : 0;
        return py::array_t<double>({B, n}, s.z.data());
      })
      .def_property_readonly("n_iter", [](const FCCQPBatchSolution& s) { return py::array_t<int>((py::ssize_t)s.n_iter.size(), s.n_iter.data()); })
      .def_property_readonly("solve_status", [](const FCCQPBatchSolution& s) { return py::array_t<int>((py::ssize_t)s.solve_status.size(), s.solve_status.data()); })
      .def_property_readonly("eps_bounds", [](const FCCQPBatchSolution& s) { return py::array_t<double>((py::ssize_t)s.admm_residual_bounds.size(), s.admm_residual_bounds.data()); })
      .def_property_readonly("eps_friction_cone", [](const FCCQPBatchSolution& s) { return py::array_t<double>((py::ssize_t)s.admm_residual_friction_cone.size(), s.admm_residual_friction_cone.data()); })
      .def_property_readonly("bounds_viol", [](const FCCQPBatchSolution& s) { return py::array_t<double>((py::ssize_t)s.bounds_viol.size(), s.bounds_viol.data()); })
      .def_property_readonly("friction_cone_viol", [](const FCCQPBatchSolution& s) { return py::array_t<double>((py::ssize_t)s.friction_cone_viol.size(), s.friction_cone_viol.data()); });

  py::class_<FCCQPBatch>(m, "FCCQPBatch")
      .def(py::init<int, int, int, int, int>(), py::arg("num_vars"), py::arg("num_equality_constraints"),
           py::arg("nc"), py::arg("lambda_c_start"), py::arg("device") = 0)
      .def(py::init<int, int, int, int, std::vector<int>>(), py::arg("num_vars"), py::arg("num_equality_constraints"),
           py::arg("nc"), py::arg("lambda_c_start"), py::arg("devices"))
      // a float for every lane, or a per-lane sequence for the host Solve (written back: rho_lanes)
      .def("set_rho",
           [](FCCQPBatch& self, const py::object& r) {
             if (!py::isinstance<py::sequence>(r) && !py::isinstance<py::array>(r)) { self.set_rho(r.cast<double>()); return; }
             const auto a = py::array_t<double, py::array::c_style | py::array::forcecast>::ensure(r);
             if (!a || a.ndim() != 1) throw py::value_error("a per-lane rho must be a 1-D sequence");
             self.set_rho(std::vector<double>(a.data(), a.data() + a.size()));
           },
           py::arg("rho"))
      .def_property_readonly("rho_lanes", [](const FCCQPBatch& self) {
        return py::array_t<double>((py::ssize_t)self.rho_lanes().size(), self.rho_lanes().data());
      })
      .def("set_max_iter", &FCCQPBatch::set_max_iter)
      // a bool for every lane, or a per-lane sequence (list, numpy bool / uint8 array) for the host Solve
      .def("set_warm_start",
           [](FCCQPBatch& self, const py::object& w) {
             if (!py::isinstance<py::sequence>(w)) { self.set_warm_start(w.cast<bool>()); return; }
             const auto a = py::array_t<uint8_t, py::array::c_style | py::array::forcecast>::ensure(w);
             if (!a || a.ndim() != 1) throw py::value_error("a warm-start mask must be a 1-D sequence");
             self.set_warm_start(std::vector<uint8_t>(a.data(), a.data() + a.size()));
           },
           py::arg("warm_start"))
      .def("set_options", &FCCQPBatch::set_options)
      .def("set_structure", &FCCQPBatch::set_structure)
      .def("contact_vars_start", &FCCQPBatch::contact_vars_start)
      // host stacks: Q [B,n,n] (or [n,n] with A_eq [m,n]: shared structure), b [B,n], A_eq [B,m,n], b_eq [B,m],
      // friction_coeffs [B,nc/3] or [nc/3], lb / ub [B,n] or [n]
      .def(
          "Solve",
          [](FCCQPBatch& self, const Stack& Q, const Stack& b, const Stack& A_eq, const Stack& b_eq, const Stack& mu,
             const Stack& lb, const Stack& ub) {
            const py::ssize_t n = self.num_vars(), mm = self.num_equality_constraints(), nc3 = self.num_contact_vars() / 3;
            if (b.ndim() != 2 || b.shape(1) != n) throw py::value_error("b must be [B,n]");
            const py::ssize_t B = b.shape(0);
            FCCQPBatchProblem p;
            p.shared_structure = Q.ndim() == 2;
            if (p.shared_structure ? !(Q.shape(0) == n && Q.shape(1) == n && A_eq.ndim() == 2 && A_eq.shape(0) == mm && A_eq.shape(1) == n)
                                   : !(Q.ndim() == 3 && Q.shape(0) == B && Q.shape(1) == n && Q.shape(2) == n && A_eq.size() == B * mm * n))
              throw py::value_error("expected Q [B,n,n] and A_eq [B,m,n] (or Q [n,n] and A_eq [m,n] shared by the batch)");
            if (b_eq.size() != B * mm) throw py::value_error("b_eq must be [B,m]");
            p.shared_friction = mu.ndim() <= 1;
            if (p.shared_friction ? mu.size() != nc3 : !(mu.ndim() == 2 && mu.shape(0) == B && mu.shape(1) == nc3)) {
              if (mu.ndim() >= 1 && mu.shape(mu.ndim() - 1) < nc3) throw py::index_error("friction_coeffs too short (reference: std::out_of_range)");
              throw py::value_error("friction_coeffs must be [B,nc/3] or [nc/3]");
            }
            p.shared_bounds = lb.ndim() == 1;
            if (lb.ndim() != ub.ndim() || (p.shared_bounds ? !(lb.size() == n && ub.size() == n)
                                                           : !(lb.ndim() == 2 && lb.shape(0) == B && lb.shape(1) == n && ub.shape(0) == B && ub.shape(1) == n)))
              throw py::value_error("lb / ub must both be [B,n] or both [n]");
            p.Q = Q.data(); p.b = b.data(); p.A_eq = A_eq.data(); p.b_eq = b_eq.data(); p.friction_coeffs = mu.data();
            p.lb = lb.data(); p.ub = ub.data();
            py::gil_scoped_release release;
            self.Solve((int)B, p);
          },
          py::arg("Q"), py::arg("b"), py::arg("A_eq"), py::arg("b_eq"), py::arg("friction_coeffs"), py::arg("lb"), py::arg("ub"))
      .def("GetSolution", &FCCQPBatch::GetSolution, py::return_value_policy::reference_internal)
      // device tensors through DLPack (torch CUDA tensors, cupy arrays): inputs as above, outputs / carried state
      // caller-owned: x, mu_x [B,n], mu_lambda_c [B,nc] float64, n_iter, solve_status [B] int32, details [4,B]
      // float64 (eps_bounds, eps_friction_cone, bounds_viol, friction_cone_viol).  Enqueued on `stream` (a
      // cudaStream_t as an integer) and not waited for unless time_kernel, which returns the kernel seconds.
      .def(
          "SolveDLPack",
          [](FCCQPBatch& self, const py::object& Q, const py::object& b, const py::object& A_eq, const py::object& b_eq,
             const py::object& mu, const py::object& lb, const py::object& ub, const py::object& x, const py::object& mu_x,
             const py::object& mu_lambda_c, const py::object& n_iter, const py::object& solve_status, const py::object& details,
             std::uintptr_t stream, bool time_kernel, const py::object& warm_lanes, const py::object& rho) {
            const int n = self.num_vars(), mm = self.num_equality_constraints(), nc = self.num_contact_vars();
            const DevView vb = dev_view(b, "b", kDLFloat, 64, 2);
            if (vb.ndim != 2 || vb.shape[1] != n) throw py::value_error("b must be [B,n]");
            const int B = (int)vb.shape[0];
            FCCQPBatchDeviceIO io;
            io.device = vb.device;
            vec_io(vb, B, n, "b", io.b, io.b_batch_stride);
            const DevView vq = dev_view(Q, "Q", kDLFloat, 64, 3), va = dev_view(A_eq, "A_eq", kDLFloat, 64, 3);
            const int qd = vq.ndim - 2, ad = va.ndim - 2;
            if (qd < 0 || vq.shape[qd] != n || vq.shape[qd + 1] != n || (qd == 1 && vq.shape[0] != B)) throw py::value_error("Q must be [B,n,n] or [n,n]");
            if (ad < 0 || va.shape[ad] != mm || va.shape[ad + 1] != n || (ad == 1 && va.shape[0] != B)) throw py::value_error("A_eq must be [B,m,n] or [m,n]");
            io.Q = static_cast<const double*>(vq.data); io.q_batch_stride = qd ? vq.stride[0] : 0;
            io.q_row_stride = vq.stride[qd]; io.q_col_stride = vq.stride[qd + 1];
            io.A_eq = static_cast<const double*>(va.data); io.a_batch_stride = ad ? va.stride[0] : 0;
            io.a_row_stride = mm ? va.stride[ad] : n; io.a_col_stride = mm ? va.stride[ad + 1] : 1;
            vec_io(dev_view(b_eq, "b_eq", kDLFloat, 64, 2), B, mm, "b_eq", io.b_eq, io.beq_batch_stride);
            vec_io(dev_view(mu, "friction_coeffs", kDLFloat, 64, 2), B, nc / 3, "friction_coeffs", io.friction_coeffs, io.mu_batch_stride, true);
            vec_io(dev_view(lb, "lb", kDLFloat, 64, 2), B, n, "lb", io.lb, io.lb_batch_stride);
            vec_io(dev_view(ub, "ub", kDLFloat, 64, 2), B, n, "ub", io.ub, io.ub_batch_stride);
            io.x = out_io<double>(dev_view(x, "x", kDLFloat, 64, 2), B, n, "x");
            io.mu_x = out_io<double>(dev_view(mu_x, "mu_x", kDLFloat, 64, 2), B, n, "mu_x");
            io.mu_lambda_c = out_io<double>(dev_view(mu_lambda_c, "mu_lambda_c", kDLFloat, 64, 2), B, nc, "mu_lambda_c");
            io.n_iter = out_io<int>(dev_view(n_iter, "n_iter", kDLInt, 32, 1), B, 0, "n_iter");
            io.solve_status = out_io<int>(dev_view(solve_status, "solve_status", kDLInt, 32, 1), B, 0, "solve_status");
            double* det = out_io<double>(dev_view(details, "details", kDLFloat, 64, 2), 4, B, "details");
            io.admm_residual_bounds = det; io.admm_residual_friction_cone = det + B; io.bounds_viol = det + 2 * (size_t)B;
            io.friction_cone_viol = det + 3 * (size_t)B;
            io.stream = reinterpret_cast<void*>(stream);
            const uint8_t* mask = nullptr;   // per-lane warm start of this call, [B] bool / uint8 on the same device
            if (!warm_lanes.is_none()) {
              const DevView vm = dev_view(warm_lanes, "warm_lanes", kDLUInt, 8, 1);
              if (vm.shape[0] != B || (B > 1 && vm.stride[0] != 1) || vm.device != io.device)
                throw py::value_error("warm_lanes must be a contiguous [B] tensor on the device of the batch");
              mask = static_cast<const uint8_t*>(vm.data);
            }
            double* rho_lanes = nullptr;   // per-lane rho of this call, [B] float64 on the same device, written back
            if (!rho.is_none()) {
              const DevView vr = dev_view(rho, "rho", kDLFloat, 64, 1);
              if (vr.ndim != 1 || vr.shape[0] != B || (B > 1 && vr.stride[0] != 1) || vr.device != io.device)
                throw py::value_error("rho must be a contiguous [B] float64 tensor on the device of the batch");
              rho_lanes = static_cast<double*>(vr.data);
            }
            double secs = 0.0;
            {
              py::gil_scoped_release release;
              self.SolveDevice(B, io, time_kernel ? &secs : nullptr, mask, rho_lanes);
            }
            return secs;
          },
          py::arg("Q"), py::arg("b"), py::arg("A_eq"), py::arg("b_eq"), py::arg("friction_coeffs"), py::arg("lb"), py::arg("ub"),
          py::arg("x"), py::arg("mu_x"), py::arg("mu_lambda_c"), py::arg("n_iter"), py::arg("solve_status"), py::arg("details"),
          py::arg("stream") = 0, py::arg("time_kernel") = false, py::arg("warm_lanes") = py::none(), py::arg("rho") = py::none());
}
