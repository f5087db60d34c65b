/*
 * fccqp.h -- C ABI of the B200-native batched FCCQP solver (libfccqp_b200.so).
 *
 * This is the drop-in boundary for the one hot path of Brian-Acosta/fcc_qp:
 * the ADMM whole-body-control QP solve
 *
 *     minimize   1/2 x'Qx + b'x
 *     subject to A_eq x = b_eq,  lb <= x <= ub,
 *                x[lambda_c_start : lambda_c_start+nc] in a product of nc/3 Coulomb cones
 *
 * (reference: src/fcc_qp.hpp:43-53).  Plain pointers and sizes only -- no C++
 * or torch types -- so it can be bound from C++, ctypes, cgo, JNI, ...
 * Every entry point cites the reference interface it replaces (file:line is
 * relative to the reference repository root).
 *
 * There is NO CPU fallback: every solve runs on a CUDA device (sm_100a);
 * fccqp_create / fccqp_batch_solve fail with FCCQP_E_CUDA when none is usable.
 *
 * Return convention: 0 (FCCQP_OK) on success, negative fccqp_error otherwise;
 * fccqp_last_error() returns a thread-local human-readable message.
 */
#ifndef FCCQP_H
#define FCCQP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FCCQP_ABI_VERSION 5

typedef enum fccqp_error {
  FCCQP_OK = 0,
  FCCQP_E_INVALID = -1,     /* bad dimensions / null pointers / too few friction coefficients */
  FCCQP_E_CUDA = -2,        /* CUDA runtime failure (message has the CUDA error string)      */
  FCCQP_E_UNSUPPORTED = -3  /* problem too large for the device kernels, unknown precision   */
} fccqp_error;
/* Largest problem: the padded KKT matrix of one QP (n and m each rounded up to a multiple of 8) lives in the opt-in
 * shared memory of one thread block.  On a B200 (227 KB per block) that allows padded n + m <= 224 for every problem
 * with m <= n (e.g. n = 140, m = 76); fccqp_create and the batch calls return FCCQP_E_UNSUPPORTED for a problem with
 * m <= n whose padded n + m is 232 or more.  (Only problems with more equality rows than variables, n <= 16, fit at 232.) */

/* Per-QP solve status.  0/1 are the reference's FCCQPSolveStatus
 * (src/fcc_qp.hpp:14-17; derived at src/fcc_qp.cpp:203-204).  2 is an
 * extension: the KKT solve broke down (a non-finite iterate, a pivot of the
 * wrong sign or of rounding-noise size that is not explained by dependent
 * constraint rows, or dependent rows that contradict each other) -- the
 * reference would return garbage/NaN silently.
 * Rank-deficient A_eq: the factorizations here are unpivoted.  A dependent
 * constraint row is detected by its pivot (wrong sign, or below 1e-12 of the
 * largest constraint pivot), gets -1e-10 x that largest pivot on its diagonal
 * and the factorization is redone (up to 4 such rows per QP); the x that comes
 * out is the minimiser of the QP whenever the dependent rows are CONSISTENT --
 * what the reference's COD fall-back returns when its LDLT notices the
 * singularity (src/fcc_qp.cpp:164-177), and the right answer where it does not
 * (the reference then returns a point that violates A_eq x = b_eq under status
 * 0).  A_eq x = b_eq is verified on the result; contradicting rows give 2.
 * Conditioning limit: the unpivoted factorization works on the Schur
 * complement A (Q + sigma A'A)^-1 A', which squares the condition number of a
 * square or nearly square A_eq (measured: 1.2e-6 .. 4.4e-6 relative error at
 * cond(A_eq) = 2.7e5 with m = n). */
typedef enum fccqp_solve_status {
  FCCQP_STATUS_SUCCESS = 0,
  FCCQP_STATUS_MAX_ITERATIONS = 1,
  FCCQP_STATUS_NUMERICAL_ISSUE = 2
} fccqp_solve_status;

/* FCCQPOptions, src/fcc_qp.hpp:30-35 (same defaults via fccqp_default_options). */
typedef struct fccqp_options {
  int32_t max_iter;  /* 1000 */
  /* Extension (SURVEY.md 8f row 4), NOT in the reference: adaptive rho.  Every adapt_rho_interval ADMM iterations the
   * primal residual r_p = max(|x_hat - x_bar|, |lambda_hat - lambda_bar|) and the dual residual r_d = rho |z_k - z_{k-1}|
   * (infinity norms, scaled duals) are compared; when they are more than a factor 5 apart, rho moves by sqrt(r_p / r_d)
   * (at most 10x per update, kept inside [1e-9, 1e9]), the scaled duals are rescaled so that y = rho mu stays put, and the
   * rho-KKT matrix is factored again.  0 (the default) = off = the reference's fixed rho.  Measured with interval 5 on the
   * walking log: QPs ending at max_iter 1.29 % -> 0, mean iterations of the QPs that iterate 66 -> 18; multi-contact
   * humanoid set 16.8 % -> 3.1 %.  All three kernels implement it.  A shared-structure batch (Q and A_eq with batch stride 0) that sets
   * it runs on the per-QP kernels instead of the cached-factorization path.  (This field was
   * `reserved`, always 0, up to ABI version 3.) */
  int32_t adapt_rho_interval; /* 0 */
  double rho;        /* 1e-6 */
  double eps_fcone;  /* 1e-3 */
  double eps_bound;  /* 1e-6 */
  /* Extension (SURVEY.md 8f row 4), NOT in the reference: over-relaxation of the ADMM iterates,
   *   x_hat = alpha x + (1 - alpha) x_bar_prev;  x_bar = proj(x_hat + mu);  mu += x_hat - x_bar
   * (residuals and the exit test on x_hat - x_bar; the returned primal is still the KKT solve x).
   * alpha in (0, 2); 1.0 -- or 0.0 = unset -- is exactly the reference's iteration.  alpha = 1.5 cuts the
   * iterations of the QPs that iterate by 30-70 % on the walking log and the synthetic sets. */
  double relaxation; /* 1.0 */
} fccqp_options;

/* FCCQPDetails, src/fcc_qp.hpp:19-28.  Times are seconds; for the device path
 * solve_time is host wall time of the call and factorization_time the device
 * time spent in the KKT factorizations (clock64-derived, 0 if not profiled). */
typedef struct fccqp_details {
  int32_t n_iter;
  int32_t solve_status; /* fccqp_solve_status */
  double admm_residual_bounds;
  double admm_residual_friction_cone;
  double solve_time;
  double factorization_time;
  double bounds_viol;
  double friction_cone_viol;
} fccqp_details;

void fccqp_default_options(fccqp_options* opt);
const char* fccqp_last_error(void);
int fccqp_abi_version(void);
/* number of usable CUDA devices (0 if none / no driver) */
int fccqp_device_count(void);

/* ------------------------------------------------------------------------- *
 * Single-problem object: replaces class fcc_qp::FCCQP (src/fcc_qp.hpp:54-171)
 * ------------------------------------------------------------------------- */
typedef struct fccqp_solver* fccqp_handle;

/* FCCQP::FCCQP(num_vars, num_equality_constraints, nc, lambda_c_start),
 * src/fcc_qp.hpp:73, src/fcc_qp.cpp:24-55.  Requires nc % 3 == 0 and
 * lambda_c_start + nc <= n (asserted there, checked here).  `device` is the
 * CUDA ordinal that owns the workspace and the warm-start state. */
int fccqp_create(int n, int m, int nc, int lambda_c_start, int device, fccqp_handle* out);
int fccqp_destroy(fccqp_handle h);
/* set_options / set_rho / set_max_iter / set_warm_start, src/fcc_qp.hpp:75-91 */
int fccqp_set_options(fccqp_handle h, const fccqp_options* opt);
int fccqp_get_options(fccqp_handle h, fccqp_options* opt);
int fccqp_set_rho(fccqp_handle h, double rho);
int fccqp_set_max_iter(fccqp_handle h, int max_iter);
int fccqp_set_warm_start(fccqp_handle h, int warm_start);
/* Extension: fccqp_structure for this object's solves (AUTO classifies each QP on the host -- its data is
 * host memory -- and sizes the reduced kernel for it; DENSE always runs the general kernel). */
int fccqp_set_structure(fccqp_handle h, int structure);
/* contact_vars_start(), src/fcc_qp.hpp:121 */
int fccqp_contact_vars_start(fccqp_handle h);

/* FCCQP::Solve, src/fcc_qp.hpp:114-117 / src/fcc_qp.cpp:114-191.
 * HOST pointers.  Q is n x n and A_eq is m x n with element (i,j) at
 * base[i*row_stride + j*col_stride] (Eigen column-major with outer stride ld:
 * row_stride = 1, col_stride = ld; C-ordered numpy: row_stride = n, col_stride = 1).
 * friction_coeffs must hold at least nc/3 values (the reference throws
 * std::out_of_range, src/constraint_utils.cpp:32,55) -> FCCQP_E_INVALID. */
int fccqp_solve(fccqp_handle h, const double* Q, ptrdiff_t q_row_stride, ptrdiff_t q_col_stride,
                const double* b, const double* A_eq, ptrdiff_t a_row_stride,
                ptrdiff_t a_col_stride, const double* b_eq, const double* friction_coeffs,
                int n_friction_coeffs, const double* lb, const double* ub);
/* FCCQP::GetSolution, src/fcc_qp.cpp:194-207: copies z (n doubles) + details. */
int fccqp_get_solution(fccqp_handle h, double* z, fccqp_details* details);
/* Warm-start state x_, mu_x_, mu_lambda_c_ (src/fcc_qp.hpp:147-153) -- private in
 * the reference, exposed here so callers can checkpoint / migrate it. */
int fccqp_get_warm_state(fccqp_handle h, double* x, double* mu_x, double* mu_lambda_c);
int fccqp_set_warm_state(fccqp_handle h, const double* x, const double* mu_x,
                         const double* mu_lambda_c);

/* ------------------------------------------------------------------------- *
 * Batched entry point: B independent QPs of identical dimensions per call.
 * Semantically B calls of FCCQP::Solve + GetSolution (src/fcc_qp.cpp:114-207)
 * on B solver objects, one launch.
 * ------------------------------------------------------------------------- */
typedef enum fccqp_memory_space { FCCQP_MEM_HOST = 0, FCCQP_MEM_DEVICE = 1 } fccqp_memory_space;
/* FCCQP_PRECISION_FP64: everything IEEE double, like the reference (parity bar 1e-6 relative on z and the
 * objective, identical iteration counts).
 * FCCQP_PRECISION_FP32_DATA: the PROBLEM DATA (Q, b, A_eq, b_eq, friction_coeffs, lb, ub) are float32 arrays
 * (same element strides); they are widened on the way into the solver, and all arithmetic, the warm-start
 * state and every output stay FP64.  Halves the bytes moved per QP (PCIe and HBM).  Stated bound: 2e-3
 * relative on z, 1e-5 relative on the objective (measured on the walking log: p50 1e-7, max 7.7e-4 on z --
 * the ill-conditioned, nearly cost-free force directions -- and 1e-8 on the objective; iteration counts
 * unchanged).
 * FCCQP_PRECISION_FP32: float32 problem data as above AND FP32 ARITHMETIC -- KKT matrix, factorization, solves,
 * projections, duals, residuals and the exit test all in float -- where a kernel for it exists: problems with
 * n + m <= 32 (the warp-per-QP kernel).  Larger problems run as FCCQP_PRECISION_FP32_DATA (FP64 arithmetic): plain
 * FP32 factors lose the answers of whole-body QPs at cond ~ 1e8 (SURVEY.md section 7).  Warm state and outputs stay
 * FP64 arrays.  Stated bound: 1e-4 relative on z (max |dz| / max(1, max |z|)) and on the objective against the
 * FP64 reference for problems whose rho-KKT matrix [[Q + rho I, A'], [A, 0]] has cond <= 1e3, with tolerances eps_fcone,
 * eps_bound >= 1e-4 (the exit test cannot resolve residuals below ~1e-6 |x| in float).  Measured on random QPs
 * (profiles/r02_fp32_mode.jsonl): max 2.7e-5 on z, 9.3e-5 on the objective at cond <= 80, max 6.9e-6 on z at
 * 1e2 < cond <= 1e3 (rows of A_eq scaled apart), same status and iteration count for every QP; 1.5-1.9 x the FP64 rate.
 * Beyond cond ~ 1e3 the float factorization of the pre-solve system breaks down on some QPs (it squares the conditioning
 * of A_eq): most of those are reported as FCCQP_STATUS_NUMERICAL_ISSUE by the pivot test, NOT all -- use FP32_DATA or
 * FP64 there. */
typedef enum fccqp_precision {
  FCCQP_PRECISION_FP64 = 0, FCCQP_PRECISION_FP32_DATA = 1, FCCQP_PRECISION_FP32 = 2
} fccqp_precision;

/* Problem structure (SURVEY.md 8f row 3).  Whole-body-control QPs are mostly made of variables that enter the
 * cost only through their own square (torques, constraint forces, slacks: diagonal-only rows of Q).  The
 * solver detects them PER QP on the device and factors a reduced KKT system without them (src/fcc_qp.cpp:141-150
 * assembles, and :62-71 / :159-178 factor, the full (n+m) x (n+m) matrix); QPs without such structure, or whose
 * reduced system fails its inertia check, run on the general kernel in the same call.  Results are those of
 * FCCQP::Solve either way (parity bar unchanged).
 *   FCCQP_STRUCTURE_AUTO   size the reduced kernel from a probe of up to 128 QPs of the batch (device memory:
 *                          one small extra launch and ONE stream synchronisation inside the call; host memory:
 *                          classified on the host, no synchronisation)
 *   FCCQP_STRUCTURE_DENSE  never reduce (the general kernel only; fully asynchronous, graph-capturable)
 *   FCCQP_STRUCTURE_CAPS   struct_caps = upper bounds {variables with off-diagonal cost entries, separable
 *                          variables whose A_eq column has >= 2 entries, zero-cost separable variables} valid for
 *                          the batch (e.g. from fccqp_last_struct_info after an AUTO call on the same kind of
 *                          data): no probe, no synchronisation; QPs beyond the caps still run, on the general kernel
 *   FCCQP_STRUCTURE_REFINE flag, OR-ed into any of the above: one step of iterative refinement of the reduced cold
 *                          pre-solve against the ORIGINAL Q and A_eq.  Eliminating a variable whose cost is h puts
 *                          1/h-sized terms into the reduced system; measured against the compiled reference on the
 *                          walking log (smallest cost 1e-6) the reduced pre-solve alone is within 1.2e-7 relative on z
 *                          with identical iteration counts -- inside the 1e-6 bar, the default -- and the refined one
 *                          within 7e-11, the level of the general kernel, for about 25 % more time per cold QP.
 *                          Set it when costs far below 1e-6 are eliminated.
 *   FCCQP_SCHEDULE_LPT     flag, OR-ed into any of the above (FCCQP_MEM_DEVICE only): the n_iter array of the call HOLDS THE
 *                          ITERATION COUNTS OF AN EARLIER SOLVE of the same lanes (a control loop re-solving a slowly changing
 *                          batch into the same arrays).  Lanes that ran long then are pulled from the work queue first
 *                          (longest-processing-time-first with the previous count as the prediction), so the few QPs that
 *                          run to max_iter no longer finish after everything else: 5-8 % of a 2^16 launch on the walking
 *                          log.  Only the ORDER in which QPs are processed changes, never a result. */
typedef enum fccqp_structure {
  FCCQP_STRUCTURE_AUTO = 0, FCCQP_STRUCTURE_DENSE = 1, FCCQP_STRUCTURE_CAPS = 2, FCCQP_STRUCTURE_REFINE = 256,
  FCCQP_SCHEDULE_LPT = 512
} fccqp_structure;

typedef struct fccqp_batch_desc {
  int32_t abi_version;     /* FCCQP_ABI_VERSION */
  int32_t batch;           /* B >= 0 */
  int32_t n, m, nc, lambda_c_start;
  int32_t device;          /* CUDA ordinal */
  int32_t memory_space;    /* fccqp_memory_space: where EVERY pointer below lives */
  int32_t precision;       /* fccqp_precision */
  int32_t warm_start;      /* 0: cold (pre-solve, duals zeroed; fcc_qp.cpp:136-139,159-178)
                              1: warm: x/mu_x/mu_lambda_c are read as the carried state
                              (ignored when warm_lanes is set)                                */
  fccqp_options options;

  /* inputs (float32 arrays behind the same pointer types when precision = FCCQP_PRECISION_FP32_DATA);
   * *_batch_stride in elements between consecutive QPs (0 = shared by all).  A cold batch
   * whose Q and A_eq are BOTH shared (stride 0) is solved with the KKT factorizations cached per
   * thread block (two launches) -- same results as B separate FCCQP::Solve calls. */
  const double* Q;        int64_t q_batch_stride, q_row_stride, q_col_stride;
  const double* b;        int64_t b_batch_stride;
  const double* A_eq;     int64_t a_batch_stride, a_row_stride, a_col_stride;
  const double* b_eq;     int64_t beq_batch_stride;
  const double* friction_coeffs; int64_t mu_batch_stride; /* nc/3 per QP */
  const double* lb;       int64_t lb_batch_stride;
  const double* ub;       int64_t ub_batch_stride;

  /* in/out state, dense [B,n] / [B,n] / [B,nc].  x is also the solution z.
   * mu_x / mu_lambda_c may be NULL for cold solves (warm_start = 0, no warm_lanes) whose duals are not needed. */
  double* x;
  double* mu_x;
  double* mu_lambda_c;

  /* outputs, dense [B]; any may be NULL */
  int32_t* n_iter;
  int32_t* status;         /* fccqp_solve_status */
  double* res_bounds;      /* admm_residual_bounds        */
  double* res_fcone;       /* admm_residual_friction_cone */
  double* bounds_viol;
  double* fcone_viol;

  void* stream;            /* cudaStream_t for FCCQP_MEM_DEVICE (NULL = default stream).
                              Device calls are asynchronous on this stream. */
  double* device_seconds;  /* optional HOST pointer: kernel time by CUDA events (forces a sync) */
  int32_t structure;       /* enum fccqp_structure, optionally | FCCQP_STRUCTURE_REFINE; 0 = AUTO */
  int32_t struct_caps[3];  /* FCCQP_STRUCTURE_CAPS only */

  /* Per-lane cold or warm start (ABI version 5): NULL = warm_start decides for every lane.  Otherwise a dense [B]
   * array, one byte per lane in the call's memory_space, and it alone decides: lane i is solved exactly as a reference
   * object after set_warm_start(warm_lanes[i] != 0) -- a warm lane from its carried x / mu_x / mu_lambda_c (pre-solve only
   * when equality-constrained, fcc_qp.cpp:159), a cold lane with the pre-solve and zero duals, its state ignored on
   * input -- and no lane's result depends on the other lanes.  x, mu_x and mu_lambda_c (nc > 0) must then be non-NULL.
   * FCCQP_MEM_DEVICE: read on the device when the call runs (no synchronisation), so a captured CUDA graph sees the
   * values written into it before each replay (environments of a vectorised simulation that reset at different
   * steps).  FCCQP_MEM_HOST: staged with every chunk of the batch.  One small kernel splits the lanes into a cold and
   * a warm list; the call then runs the launches of a cold call of the whole batch over the cold list and those of a
   * warm call over the warm list, with the same kernels, so every lane returns the bits of a uniform call (on the
   * shared-structure path up to the last bits that already depend there on which QPs a thread block solves first). */
  const uint8_t* warm_lanes;
} fccqp_batch_desc;

int fccqp_batch_solve(const fccqp_batch_desc* desc);
/* The same call spread over several devices of one box (FCCQP_MEM_HOST only; desc->device is ignored): the batch is
 * cut into contiguous slabs (multiples of 4096 QPs; guided sizes: half an equal share of what is left, at least 8192) and every device -- on its own host
 * thread with its own streams and staging buffers -- takes the next slab when it has finished its own, so a device
 * behind a slower host link takes fewer.  QPs are independent: there is no exchange step, and a result does not depend
 * on which device produced it.  Outputs land in the caller's arrays exactly as with one device; device_seconds is the
 * wall time of the whole call.
 * (Device-resident data lives on ONE device: shard it yourself and call fccqp_batch_solve per device.) */
int fccqp_batch_solve_multi(const fccqp_batch_desc* desc, const int32_t* devices, int32_t n_devices);

/* Per-lane rho (next to warm_lanes; the descriptor and FCCQP_ABI_VERSION are unchanged): fccqp_batch_solve and
 * fccqp_batch_solve_multi are these calls with rho = NULL, which is today's behaviour bit for bit.  Otherwise rho is a
 * dense [B] FP64 array in the call's memory_space that the call both reads and writes:
 *   - lane i is solved exactly as a reference object on which set_rho(rho[i]) was called before Solve, cold or warm,
 *     with or without warm_lanes (both index the same lanes); options.rho is not used;
 *   - on return rho[i] holds the rho lane i ended with.  With options.adapt_rho_interval = 0 that is rho[i] unchanged.
 *     With adaptive rho the returned mu_x / mu_lambda_c are scaled for that rho (y = rho mu), so feeding x, mu_x,
 *     mu_lambda_c AND rho back into the next warm call continues every lane's ADMM from a consistent state.  (Without
 *     the array each warm call restarts at options.rho and reads the duals as if they were scaled for it: y is off by
 *     the factor rho_end / options.rho, and rho has to adapt again from scratch.)
 *   - FCCQP_MEM_DEVICE: read and written in place by the kernels (no synchronisation), so CUDA-graph replays carry rho
 *     from step to step.  An entry that is not finite or not > 0 ends its lane with FCCQP_STATUS_NUMERICAL_ISSUE and
 *     n_iter = 0; the entry is left as it was, the lane's other outputs are unspecified, no other lane is affected.
 *   - FCCQP_MEM_HOST: staged with every chunk (in and out); an array with such an entry is refused with FCCQP_E_INVALID
 *     before anything runs.
 * Calls with the array run the kernel instances that keep rho per QP (those of adaptive rho), and a shared-structure
 * batch (Q and A_eq with batch stride 0) runs on the per-QP kernels, as it does under adaptive rho: a cached
 * factorization has one rho. */
int fccqp_batch_solve_rho(const fccqp_batch_desc* desc, double* rho);
int fccqp_batch_solve_multi_rho(const fccqp_batch_desc* desc, double* rho, const int32_t* devices, int32_t n_devices);
/* Page-locked host memory for FCCQP_MEM_HOST callers: inputs and outputs that live in
 * memory from here (or from cudaHostAlloc / torch pin_memory) move by asynchronous DMA that
 * overlaps the solve; pageable outputs go through an internal pinned bounce buffer. */
int fccqp_alloc_pinned(size_t bytes, void** out);
int fccqp_free_pinned(void* ptr);
/* Frees the cached per-device staging buffers used by FCCQP_MEM_HOST calls. */
int fccqp_release_workspaces(void);

/* ------------------------------------------------------------------------- *
 * On-device assembly of whole-body-control QPs from robot quantities (SURVEY.md 8f row 2:
 * the step BEFORE Solve in an operational-space-control / sampling-MPC loop; fccqp.pdf
 * section 4, eq. 10).  The reference has no such function -- its callers (fcc_qp_test.py's log,
 * the DAIRLab OSC) hand FCCQP::Solve finished Q, b, A_eq, b_eq (src/fcc_qp.hpp:114-117) -- so a
 * batch that is assembled on the GPU moves nv^2 + (nh+nc+ny) nv + ... doubles per QP over PCIe
 * instead of n^2 + m n.  Decision vector x = [vdot(nv) u(nu) lambda_h(nh) lambda_c(nc) eps(nc)],
 * n = nv+nu+nh+2nc, m = nv+nh+nc, lambda_c_start = nv+nu+nh:
 *     Q    = blkdiag(Jy' diag(W) Jy + w_vdot I, w_u I, 0, w_lambda_c I, w_eps I)
 *     b    = [-Jy' (W .* ydd_cmd); 0]
 *     A_eq = [[M, -S, -Jh', -Jc', 0], [Jh, 0, 0, 0, 0], [Jc, 0, 0, 0, I]],  S = [0; I_nu]
 *     b_eq = [-bias; -gamma_h; -gamma_c]
 * All pointers are DEVICE pointers to dense row-major FP64 arrays with the batch as the leading
 * dimension (inputs: a *_batch_stride of 0 shares one array across the batch); outputs are the
 * dense [B,n,n], [B,n], [B,m,n], [B,m] arrays fccqp_batch_solve takes.  Asynchronous on `stream`.
 * ------------------------------------------------------------------------- */
typedef struct fccqp_wbc_desc {
  int32_t abi_version;     /* FCCQP_ABI_VERSION */
  int32_t batch;
  int32_t nv, nu, nh, nc, ny;
  int32_t device;
  double w_vdot, w_u, w_lambda_c, w_eps;   /* diagonal cost weights (1e-5, 1e-4, 1e-6, 80 on the walking log) */
  const double* M;        int64_t M_batch_stride;      /* [B,nv,nv] mass matrix              */
  const double* Jh;       int64_t Jh_batch_stride;     /* [B,nh,nv] holonomic Jacobian       */
  const double* Jc;       int64_t Jc_batch_stride;     /* [B,nc,nv] contact Jacobian         */
  const double* Jy;       int64_t Jy_batch_stride;     /* [B,ny,nv] task Jacobian            */
  const double* W;        int64_t W_batch_stride;      /* [B,ny]    task weights             */
  const double* ydd_cmd;  int64_t ydd_batch_stride;    /* [B,ny]    commanded task accel.    */
  const double* bias;     int64_t bias_batch_stride;   /* [B,nv]    Coriolis + gravity       */
  const double* gamma_h;  int64_t gh_batch_stride;     /* [B,nh]    Jh_dot v                 */
  const double* gamma_c;  int64_t gc_batch_stride;     /* [B,nc]    Jc_dot v                 */
  double* Q; double* b; double* A_eq; double* b_eq;    /* outputs */
  void* stream;
} fccqp_wbc_desc;

int fccqp_wbc_assemble(const fccqp_wbc_desc* desc);

/* ------------------------------------------------------------------------- *
 * Opt-in solution polish (SURVEY.md 8f row 4).  NOT part of the reference: src/fcc_qp.cpp returns the ADMM iterate as it
 * is (fccqp.pdf Table 2 lists polish among the OSQP features FCCQP lacks), so nothing here is covered by the parity bar.
 * The active set is guessed from the solver's own state: a bounded variable outside the contact block with
 * x + mu_x at or beyond a bound sits on it; a contact is classified by the branch of project_to_friction_cone
 * (src/constraint_utils.cpp:5-25) its argument x_c + mu_c takes: inside (free), polar cone (lambda_c = 0), otherwise on the
 * boundary, free in the tangent plane of the cone at the projection o (lambda_c = alpha o/|o| + beta t1, t1 the horizontal
 * tangent; the plane leaves the cone only to second order in beta).  fccqp_polish_prepare writes the resulting
 * equality-constrained QP -- SAME n and m: boundary contacts rotated into (alpha, beta, normal = 0), fixed variables decoupled
 * with their coupling moved to the right-hand sides -- which the caller solves with fccqp_batch_solve as a QP with nc = 0 and
 * infinite bounds (the pre-solve is the KKT solve, src/fcc_qp.cpp:159-178).  fccqp_polish_finish rotates that answer back
 * and ACCEPTS it per QP only if the solve returned FCCQP_STATUS_SUCCESS, the point satisfies A_eq z = b_eq (1e-7 relative to
 * the magnitude of the terms plus a rounding-level floor: a guess that fixes too much leaves an inconsistent system), every bound to eps_bound and
 * every friction cone to eps_fcone, and its objective is not above the ADMM iterate's by more than eps_objective relative
 * (f_p <= f_admm + eps_objective max(1, |f_admm|): a feasible point of a wrong guess is optimal for the wrong problem; the
 * ADMM iterate's objective is a lower estimate of the optimum).  z, bounds_viol, fcone_viol of accepted QPs are overwritten,
 * polished[i] = 1 / 0.
 * Device memory only; Q / A_eq dense row-major per QP (batch strides in elements, 0 = shared).  Bounds on contact
 * variables are not part of the guess (they still gate acceptance).  Python: FCCQPBatch.Polish().
 * ------------------------------------------------------------------------- */
typedef struct fccqp_polish_desc {
  int32_t abi_version;
  int32_t batch, n, m, nc, lambda_c_start;
  int32_t device;
  int32_t reserved;
  double eps_fcone, eps_bound, eps_objective;
  const double* Q;               int64_t q_batch_stride;     /* [B,n,n] */
  const double* b;               int64_t b_batch_stride;
  const double* A_eq;            int64_t a_batch_stride;     /* [B,m,n] */
  const double* b_eq;            int64_t beq_batch_stride;
  const double* friction_coeffs; int64_t mu_batch_stride;
  const double* lb;              int64_t lb_batch_stride;
  const double* ub;              int64_t ub_batch_stride;
  const double* x;               /* [B,n]  ADMM result (prepare) */
  const double* mu_x;            /* [B,n]  */
  const double* mu_lambda_c;     /* [B,nc] */
  double* Qp; double* bp; double* Ap; double* beqp;          /* polished QP, contiguous [B,n,n] [B,n] [B,m,n] [B,m] */
  double* rot;                   /* [B, nc/3, 4] scratch written by prepare, read by finish */
  const double* y;               /* [B,n]  solution of the polished QP (finish) */
  const int32_t* y_status;       /* [B]    its status */
  double* z;                     /* [B,n]  overwritten where accepted (may be the x array) */
  double* bounds_viol; double* fcone_viol;                   /* [B] overwritten where accepted */
  int32_t* polished;             /* [B] out */
  void* stream;
} fccqp_polish_desc;

int fccqp_polish_prepare(const fccqp_polish_desc* desc);
int fccqp_polish_finish(const fccqp_polish_desc* desc);

/* Introspection used by bench.py for the roofline line: kernel launches issued
 * by this library since load, and the launch geometry of the last batch call. */
int64_t fccqp_kernel_launch_count(void);
/* Vector-FP64 FMA peak of `device` in TFLOP/s, MEASURED with a ~50 ms register-only DFMA kernel (the FP64 tensor-core
 * instruction the solver uses shares that pipe): the denominator of bench.py's roofline_fp64. */
int fccqp_measure_fp64_peak(int device, double* tflops);
int fccqp_last_launch_info(int* grid, int* block, int* smem_bytes, int* ctas_per_sm);
/* What the last batch launch did about problem structure: used = 1 if the reduced kernel ran; caps[3] = the
 * structure bounds its layout was sized for (pass them back as FCCQP_STRUCTURE_CAPS); rows / rows_dense = padded
 * KKT rows factored per QP by the reduced and by the general kernel; deferred = QPs the reduced kernel handed to
 * the general one (valid once the stream of that call has been synchronised).  Any pointer may be NULL. */
int fccqp_last_struct_info(int* used, int* caps, int* rows, int* rows_dense, int* deferred);

#ifdef __cplusplus
}
#endif
#endif /* FCCQP_H */
