// fccqp_kernel.cuh -- sm_100a device code of the batched FCCQP solve (FP64 tensor-core tiles).
//
// One CTA solves one QP at a time; persistent CTAs pull QP indices from a global
// work counter, so the 1-2 % of QPs that run to max_iter do not stall the rest of
// the batch.  Everything between stage-in and the final store lives in shared
// memory / registers.  Stages (reference code they replace):
//
//   K0 stage-in          Solve assembly            src/fcc_qp.cpp:141-150
//   K1 cold pre-solve    LDLT -> COD fallback      src/fcc_qp.cpp:159-178
//   K2 rho-KKT factor    LDLT.compute              src/fcc_qp.cpp:62-71
//   K3 x-update          LDLT.solve                src/fcc_qp.cpp:81-87
//   K4 z-update          clamp + cone projection   src/fcc_qp.cpp:90-92, src/constraint_utils.cpp:5-46
//   K5 residuals / duals / exit                    src/fcc_qp.cpp:95-109
//   K6 epilogue          violations + details      src/fcc_qp.cpp:184-186,194-207
//
// This is NOT a port of the Eigen code paths.  The linear algebra is re-derived so that it is
// pivot-free, symmetric, and made of 8x8 tiles that map onto the FP64 tensor-core instruction
// (DMMA, mma.sync.m8n8k4.f64):
//
//   * K1.  The reference solves the indefinite system [[Q,A'],[A,0]] s = [-b; b_eq] whose (1,1)
//     block is singular (zero-cost force variables) through a failed LDLT and a complete
//     orthogonal decomposition.  Here the SAME solution comes from the augmented-Lagrangian
//     form [[Q + sigma A'A, A'],[A,0]] with right-hand side [-b + sigma A' b_eq; b_eq]: on
//     {Ax = b_eq} the added term is constant, so x is unchanged, while Q + sigma A'A is positive
//     definite exactly when the KKT matrix is nonsingular.  That matrix is quasi-definite, so an
//     unpivoted LDL^T exists.  x-update 0 of a cold solve is then the identity (x0 minimises the
//     proximal problem anchored at itself), so the 98 % of QPs that pass the exit test at x0 never
//     factor the rho-KKT matrix; the others factor it lazily at iteration 1.
//   * K2 is the same unpivoted blocked LDL^T on [[Q + rho I, A'],[A,0]].
//   * factor_tiles: blocked LEFT-looking LDL^T on 8x8 tiles, one tile column at a time.  One warp
//     runs the critical path (ONE thread factors the diagonal tile in registers and inverts its
//     unit-lower factor; the warp forms the tile below it and updates the next diagonal tile), the
//     helper warps own the tile rows i = w (mod #helpers) and stay one column behind:
//     (B) L_ij = C_ij inv(L_jj)' inv(D_j), (A) C_i,j+1 -= sum_{k<=j} L_ik D_k L_j+1,k' for up to four
//     tiles at a time with one shared scaled operand, accumulators in registers, nothing written
//     back in between.  sigma A'A (K1) is formed beforehand in tile-row chunks, rho I (K2) is a
//     diagonal add.
//   * K3, kkt_solve.  The 8x8 inverses are composed (again with DMMAs) into explicit inverses of
//     the 32x32 diagonal blocks of L, stored in place.  A triangular solve is then ceil(N/32) steps
//     of "one warp applies a 32x32 inverse, the others subtract a 32-column slab" instead of N
//     dependent scalar steps.
//   * K3 for long-running QPs (complete_inverse, kkt_solve_full, form_g, g_apply): after
//     full_inverse_at ADMM iterations W = inv(L) is completed in place by recursive doubling and
//     G = [K^-1]_xx replaces its top-left tiles; every later x-update is
//     x = x_base + rho G (x_bar - mu), one symmetric matrix-vector product.
//
// Storage: the lower triangle of the padded KKT matrix as dense 8x8 tiles (512 B each),
// tile (I,J) at index I(I+1)/2+J.  Variables are padded to a multiple of 8 (n8) before the
// constraint rows start (pads are decoupled unit pivots).  Inside a tile element (r,c) lives at
// r*8 + (((c/2) ^ (r/2)) & 3)*2 + (c&1): the 16-byte chunks of a row are XOR-swizzled by r/2
// (the TMA SWIZZLE_64B pattern), which makes the tensor-core fragment access (row = lane/4,
// column pair = lane%4), the row-per-thread access of the forward solve and the
// column-per-thread access of the backward solve bank-conflict-free within a tile.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace fccqp {

// Shared-memory carve-up (offsets in doubles).  Computed on the host, passed by value in the
// kernel parameters (constant bank), so the kernel never recomputes it.
struct Layout {
  int n, m, nc;
  int n8, m8, N8;   // padded sizes (multiples of 8)
  int NB, NBx;      // number of 8-tiles per side; tiles covering the variable rows
  int NB32, NT;     // 32-row solve blocks; padded vector length (NB32 * 32)
  int NBT;          // number of stored tiles
  int off_M, off_dinv, off_dneg, off_tbuf, off_ybuf, off_xs, off_lcbar, off_muc, off_mu;
  int off_red, off_int;
  int doubles_total;
  static inline int up2(int v) { return (v + 1) & ~1; }
  Layout() = default;
  Layout(int n_, int m_, int nc_) {
    n = n_; m = m_; nc = nc_;
    n8 = (n + 7) & ~7; m8 = (m + 7) & ~7; N8 = n8 + m8;
    NB = N8 >> 3; NBx = n8 >> 3;
    NB32 = (N8 + 31) >> 5; NT = NB32 * 32;
    NBT = NB * (NB + 1) / 2;
    int o = 0;
    off_M = o;     o += NBT * 64;
    off_dinv = o;  o += NT;
    off_dneg = o;  o += NT;
    off_tbuf = o;  o += NT;
    off_ybuf = o;  o += NT;
    off_xs = o;    o += n8 + 8;
    off_lcbar = o; o += up2(nc + 2);
    off_muc = o;   o += up2(nc + 2);
    off_mu = o;    o += up2(nc / 3 + 2);
    off_red = o;   o += 4 * 32;   // block_reduce2 scratch: 2 buffers x 2 values x 32 warps
    off_int = o;   o += 32;       // ints: work index, profiling slots
    doubles_total = o;
  }
  size_t bytes() const { return (size_t)doubles_total * sizeof(double); }
};

// Shared-memory carve-up of the structure-exploiting kernel (fccqp_struct.cuh), sized by CAPS on the
// per-QP structure: nr (variables whose Q row has off-diagonal entries -- they stay in the KKT
// system), ndp (separable variables, i.e. diagonal-only Q rows with positive cost, whose A_eq column has
// two or more entries -- eliminated analytically, column kept as tiles), nd0 (separable variables
// with zero cost -- kept as the trailing block of the KKT system).  Separable variables with an
// empty or one-entry A_eq column cost no storage at all.  QPs that exceed the caps are handed to the
// general kernel.
struct StructLayout {
  int n, m, nc;
  int n8, m8, mt;
  int nr8c, ndp8c, dptc, nd08c;
  int N8c, NBc, NB32c, NTc, NBTc;
  int off_M, off_AP, off_dinv, off_dneg, off_tbuf, off_ybuf, off_sred, off_rf, off_vd, off_hinv, off_d1c, off_beq;
  int off_qd, off_xs, off_lcbar, off_muc, off_mu, off_red, off_int;
  int off_part;    // [warps][n8] per-warp partial column sums (iterative refinement of the register front end)
  // int region (offsets in ints from off_int)
  int io_vtype, io_vpos, io_rlist, io_dplist, io_d0list, io_d1var, io_rowcnt, io_wtot, io_nzflag, io_colcnt, io_colk, ints_total;
  int stage_cap;   // doubles of the [M | AP] region: staging space of the classification (>= 4 rows of Q)
  int doubles_total;
  static inline int up2(int v) { return (v + 1) & ~1; }
  static inline int up8(int v) { return (v + 7) & ~7; }
  StructLayout() = default;
  StructLayout(int n_, int m_, int nc_, int nr_cap, int ndp_cap, int nd0_cap) {
    n = n_; m = m_; nc = nc_;
    n8 = up8(n); m8 = up8(m); mt = m8 >> 3;
    nr8c = up8(nr_cap); ndp8c = up8(ndp_cap); dptc = ndp8c >> 3; nd08c = up8(nd0_cap);
    N8c = nr8c + m8 + nd08c; NBc = N8c >> 3;
    NB32c = (N8c + 31) >> 5; NTc = NB32c * 32;
    NBTc = NBc * (NBc + 1) / 2;
    int o = 0;
    off_M = o;     o += NBTc * 64;
    off_AP = o;    o += mt * dptc * 64;
    if (o < 4 * n8) o = 4 * n8;     // (tiny reduced systems: keep room to stage a few rows of Q)
    stage_cap = o;
    off_dinv = o;  o += NTc;
    off_dneg = o;  o += NTc;
    off_tbuf = o;  o += NTc;
    off_ybuf = o;  o += NTc;
    off_sred = o;  o += NTc;
    off_rf = o;    o += n8;
    {
      const int need = n > N8c ? n : N8c;   // thread count of the kernel instance (pick_struct_kernel)
      const int warps = need <= 64 ? 2 : (need <= 96 ? 3 : (need <= 128 ? 4 : 8));
      off_part = o;  o += warps * n8;
    }
    off_vd = o;    o += ndp8c + 8;
    off_hinv = o;  o += ndp8c + 8;
    off_d1c = o;   o += m8 + 8;
    off_beq = o;   o += m8 + 8;
    off_qd = o;    o += n8;
    off_xs = o;    o += n8 + 8;
    off_lcbar = o; o += up2(nc + 2);
    off_muc = o;   o += up2(nc + 2);
    off_mu = o;    o += up2(nc / 3 + 2);
    off_red = o;   o += 4 * 32 + 16;   // + 16: developer phase counters
    off_int = o;
    int io = 8;                      // [0] work index, [1..7] spare
    io_vtype = io;  io += n8;
    io_vpos = io;   io += n8;
    io_rlist = io;  io += nr8c + 8;
    io_dplist = io; io += ndp8c + 8;
    io_d0list = io; io += nd08c + 8;
    io_d1var = io;  io += m8 + 8;
    io_rowcnt = io; io += m8 + 8;
    io_wtot = io;   io += 32 * 3;
    io_nzflag = io; io += n8;
    io_colcnt = io; io += n8;
    io_colk = io;   io += n8;
    ints_total = io;
    o += (io + 1) / 2;
    doubles_total = o;
  }
  size_t bytes() const { return (size_t)doubles_total * sizeof(double); }
};

struct SolveParams {
  int B, n, m, nc, lcs;
  int max_iter, warm;
  // Shared-structure batches (Q and A_eq common to all QPs, only the vectors vary -- sampling-based MPC;
  // SURVEY 8f row 3): 0 = off; 1 = pre-solve launch (every CTA factors the pre-solve KKT matrix ONCE,
  // completes inv(L) and streams QPs through it; QPs that need ADMM iterations park x0 and their
  // index in pending_list); 2 = ADMM launch over index_list / count_dev with the rho-KKT factors cached
  // the same way.
  int shared_mode;
  const int* index_list;          // mode 2: QP indices to process
  const unsigned int* count_dev;  // mode 2: how many (device memory, written by the mode-1 launch)
  int* pending_list;              // mode 1: output list
  unsigned int* pending_count;    // mode 1: its length
  int full_inverse_at;        // ADMM iteration from which x-updates use the completed inverse of L (launch_solve)
  double rho, eps_fcone, eps_bound;
  double alpha;               // over-relaxation (fccqp_options::relaxation); 1.0 = the reference's iteration
  int adapt_k;                // adaptive rho (fccqp_options::adapt_rho_interval): rebalance every adapt_k iterations; 0 = off
  const double* Q;   long long q_bs, q_rs, q_cs;
  const double* b;   long long b_bs;
  const double* A;   long long a_bs, a_rs, a_cs;
  const double* beq; long long beq_bs;
  const double* mu;  long long mu_bs;
  const double* lb;  long long lb_bs;
  const double* ub;  long long ub_bs;
  double* x; double* mu_x; double* mu_c;
  int* n_iter; int* status;
  double* res_b; double* res_f; double* bviol; double* fviol;
  unsigned int* work_counter;
  unsigned long long* cycles;  // optional [2]: summed factorization / total cycles
  unsigned long long* prof;    // optional [16]: per-phase cycle counters (developer profiling)
  Layout lay;                  // filled in by launch_solve
  StructLayout slay;           // structure-exploiting kernel (fccqp_struct.cuh); filled in by launch_solve
  int struct_refine;           // that kernel: one step of iterative refinement on the cold pre-solve
  double* op_scratch;          // that kernel: per-CTA global scratch of the full-space operator of long-running QPs
  long long op_stride;         //   doubles per CTA
  int* resume_list;            // its first stage (kStructFirst): QPs that keep iterating
  unsigned int* resume_count;  //   their count
};

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide reduction of two values (max or sum).  `red` holds 2 x 2 x 32 doubles;
// `parity` alternates between the two halves so one barrier per call suffices.  Inlined and
// by value: the two shuffle chains interleave and nothing goes through local memory.
template <bool kSum>
__device__ __forceinline__ void block_reduce2(double& a, double& b, double* red, int& parity) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  double va = a, vb = b;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double oa = __shfl_xor_sync(0xffffffffu, va, o), ob = __shfl_xor_sync(0xffffffffu, vb, o);
    if (kSum) { va += oa; vb += ob; } else { va = fmax(va, oa); vb = fmax(vb, ob); }
  }
  double* r = red + parity * 64;
  if (lane == 0) { r[warp] = va; r[32 + warp] = vb; }
  __syncthreads();
  double ra = r[0], rb = r[32];
#pragma unroll 1
  for (int w = 1; w < nw; ++w) {
    if (kSum) { ra += r[w]; rb += r[32 + w]; } else { ra = fmax(ra, r[w]); rb = fmax(rb, r[32 + w]); }
  }
  a = ra; b = rb;
  parity ^= 1;
}

// Smallest pivot, relative to the largest pivot of the same class, that the unpivoted LDL^T still trusts.
constexpr double kPivotRatio = 1e-12;
// Regularisation of the constraint block on the retry after a failed factorization, relative to its largest pivot.
constexpr double kRegDelta = 1e-10;
constexpr int kRegTries = 4;

// 1/d to full double precision: MUFU seed x0 (relative error e <= 2^-23) and ONE third-order step
// x0 (1 + e + e^2) = (1/d)(1 - e^3): three dependent FMAs behind the MUFU instead of the four of two
// Newton steps, and far shorter than the IEEE division sequence.  d is a factorization pivot
// (finite, non-denormal); this reciprocal sits on the pivot chain of every tile column.
__device__ __forceinline__ double fast_rcp(double d) {
  double x;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
  const double e = fma(-d, x, 1.0);
  const double t = fma(e, e, e);
  return fma(x, t, x);
}

__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gsrc) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async16(double* smem_dst, const double* gsrc) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// constraint_utils.cpp:5-25, including the f_z == 0 quirk (zero cone_ray is not normalised).
__device__ __forceinline__ void project_cone3(double f0, double f1, double f2, double mu,
                                              double& o0, double& o1, double& o2) {
  const double r = sqrt(f0 * f0 + f1 * f1);
  if (mu * f2 >= r) { o0 = f0; o1 = f1; o2 = f2; return; }
  if (f2 < -mu * r) { o0 = 0.0; o1 = 0.0; o2 = 0.0; return; }
  const double ratio = mu * f2 / r;
  double r0 = ratio * f0, r1 = ratio * f1, r2 = f2;
  const double sq = r0 * r0 + r1 * r1 + r2 * r2;
  if (sq > 0.0) { const double nr = sqrt(sq); r0 /= nr; r1 /= nr; r2 /= nr; }
  const double d = r0 * f0 + r1 * f1 + r2 * f2;
  o0 = d * r0; o1 = d * r1; o2 = d * r2;
}

template <typename T>
__device__ __forceinline__ T clampd(T x, T lb, T ub) {
  const T t = x < ub ? x : ub;  // std::min(x, ub)
  return t > lb ? t : lb;       // std::max(., lb)   constraint_utils.cpp:43
}

// ---------------------------------------------------------------------------
// The ADMM step after each x-update (fcc_qp.cpp:88-109), shared by the solve kernels.  T = float: the FP32 warp kernel.
// `relax`: the over-relaxation extension, x_hat = alpha x + (1 - alpha) x_bar_prev in place of x.  kDz (adaptive rho):
// dz gets |z_k - z_{k-1}| of the entries updated.
// ---------------------------------------------------------------------------
// z-update and scaled-dual update of one bounded variable; returns |r|, its residual.
template <typename T, bool kDz>
__device__ __forceinline__ T box_step(const T val, const T alpha, const bool relax, const T lb, const T ub, T& xbar,
                                      T& mux, T& dz) {
  const T xh = relax ? fma(alpha, val, (T(1) - alpha) * xbar) : val;
  const T xb = clampd(xh + mux, lb, ub);
  if (kDz) dz = fabs(xb - xbar);
  xbar = xb;
  const T r = xh - xb;
  mux += r;
  return fabs(r);
}
// The same for one contact triple: x0..x2 its x entries, lcb / mc its slack and scaled duals (updated in place);
// returns the triple's max |r|.
template <bool kDz>
__device__ __forceinline__ double cone_step(double x0, double x1, double x2, const double mu, const double alpha,
                                            const bool relax, double* lcb, double* mc, double& dz) {
  if (relax) {
    x0 = fma(alpha, x0, (1.0 - alpha) * lcb[0]);
    x1 = fma(alpha, x1, (1.0 - alpha) * lcb[1]);
    x2 = fma(alpha, x2, (1.0 - alpha) * lcb[2]);
  }
  double o0, o1, o2;
  project_cone3(x0 + mc[0], x1 + mc[1], x2 + mc[2], mu, o0, o1, o2);
  if (kDz) dz = fmax(dz, fmax(fabs(o0 - lcb[0]), fmax(fabs(o1 - lcb[1]), fabs(o2 - lcb[2]))));
  lcb[0] = o0; lcb[1] = o1; lcb[2] = o2;
  const double r0 = x0 - o0, r1 = x1 - o1, r2 = x2 - o2;
  mc[0] += r0; mc[1] += r1; mc[2] += r2;
  return fmax(fabs(r0), fmax(fabs(r1), fabs(r2)));
}
// Adaptive rho (extension, fccqp_options::adapt_rho_interval; restated in oracle/fccqp_oracle.c, do_admm): with scaled
// duals the primal residual is rp = max(|x_hat - x_bar|, |lambda_hat - lambda_bar|), the dual one rho dz; more than a
// factor 5 apart, rho moves by sqrt(rp / (rho dz)), at most 10x.  Returns the new rho, or rho when it stays.
template <typename T>
__device__ __forceinline__ T rebalance_rho(const T rp, const T dz, const T rho) {
  constexpr T tiny = sizeof(T) == sizeof(double) ? T(1e-300) : T(1e-30f);
  const T rd = rho * dz;
  T ratio = sqrt(rp / (rd > tiny ? rd : tiny));
  ratio = fmin(fmax(ratio, T(0.1)), T(10));
  if (ratio > T(5) || ratio < T(0.2)) return fmin(fmax(rho * ratio, T(1e-9)), T(1e9));
  return rho;
}
// The CTA kernels' side of it: block-wide rp and dz, and on a change the scaled duals of this thread's variable (mux)
// and contact (mc, when `contact`) rescaled so that y = rho mu stays put.  The caller has the rho-KKT system
// factored again.
__device__ __forceinline__ double cta_rebalance_rho(const double rx, const double rc, const double dz, const double rho,
                                                    double& mux, double* mc, const bool contact, double* red,
                                                    int& parity) {
  double rp = fmax(rx, rc), rd = dz;
  block_reduce2<false>(rp, rd, red, parity);
  const double rho_new = rebalance_rho(rp, rd, rho);
  if (rho_new != rho) {
    const double sc = rho / rho_new;
    mux *= sc;
    if (contact) { mc[0] *= sc; mc[1] *= sc; mc[2] *= sc; }
    __syncthreads();
  }
  return rho_new;
}

// K6 of the CTA kernels: the squared box violation of this thread's variable and the cone violation of its contact
// (constraint_utils.cpp:48-65), summed over the block into bv / fv.  Returns 1 when x is not finite.
__device__ __forceinline__ int cta_violations(const bool is_x, const double x, const double lb, const double ub,
                                              const double* xs, const double* vmu, const int nc, const int lcs,
                                              double* red, int& parity, double& bv, double& fv) {
  const int tid = threadIdx.x;
  __syncthreads();
  bv = 0.0; fv = 0.0;
  int bad = 0;
  if (is_x) {
    const double d = x - clampd(x, lb, ub);
    bv = d * d;
    if (!isfinite(x)) bad = 1;
  }
  if (tid < nc / 3) {
    const int o = lcs + 3 * tid;
    const double r = sqrt(xs[o] * xs[o] + xs[o + 1] * xs[o + 1]) - vmu[tid] * xs[o + 2];
    fv = r > 0.0 ? r : 0.0;
  }
  block_reduce2<true>(bv, fv, red, parity);
  return bad;
}

// The per-QP details of every solve kernel (fcc_qp.cpp:194-207), stored by one thread; bv is the summed square.
template <typename T>
__device__ __forceinline__ void store_details(const SolveParams& p, const int qp, const int n_iter, const bool bad,
                                              const T res_x, const T res_c, const T bv, const T fv,
                                              const unsigned long long fact_cycles, const long long t_start) {
  if (p.n_iter) p.n_iter[qp] = n_iter;
  if (p.status) p.status[qp] = bad ? 2 : (n_iter == p.max_iter ? 1 : 0);  // fcc_qp.cpp:203-204
  if (p.res_b) p.res_b[qp] = (double)res_x;
  if (p.res_f) p.res_f[qp] = (double)res_c;
  if (p.bviol) p.bviol[qp] = (double)sqrt(bv);
  if (p.fviol) p.fviol[qp] = (double)fv;
  if (p.cycles) {
    atomicAdd(p.cycles, fact_cycles);
    atomicAdd(p.cycles + 1, (unsigned long long)(clock64() - t_start));
  }
}

// ---------------------------------------------------------------------------
// Tile storage
// ---------------------------------------------------------------------------
__host__ __device__ __forceinline__ int tile_off(int I, int J) { return (((I * (I + 1)) >> 1) + J) << 6; }
// element (r,c) inside a tile (16-byte chunks XOR-swizzled by r/2)
__host__ __device__ __forceinline__ int el_off(int r, int c) {
  return (r << 3) + ((((c >> 1) ^ (r >> 1)) & 3) << 1) + (c & 1);
}
// element (i,j), i >= j in tile terms, of the packed matrix
__host__ __device__ __forceinline__ int mat_off(int i, int j) { return tile_off(i >> 3, j >> 3) + el_off(i & 7, j & 7); }

// FP64 tensor-core step: C(8x8) += A(8x4) B(4x8).  Fragments (PTX ISA, m8n8k4 .f64): lane l holds
// A[l/4][l%4], B[l%4][l/4], C[l/4][2(l%4)], C[l/4][2(l%4)+1].
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
      : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
// C(8x8) += Aop(8x8) Bop(8x8) with the contraction index split as k = 2(l%4)+s over two DMMAs:
//   a = (Aop[l/4][2q], Aop[l/4][2q+1]),  b = (Bop[2q][l/4], Bop[2q+1][l/4]),  q = l%4.
// With "fragC(X)" = (X[l/4][2q], X[l/4][2q+1]) (one 16-byte load) and
//      "fragT(X)" = (X[2q][l/4], X[2q+1][l/4]) (two 8-byte loads):
//   X Y'  : a = fragC(X), b = fragC(Y)        X Y  : a = fragC(X), b = fragT(Y)
//   X' Y  : a = fragT(X), b = fragT(Y)        X' Y': a = fragT(X), b = fragC(Y)
// and a product held in registers as fragC(P) is fragT(P') for the next product.
__device__ __forceinline__ void mma8(double2& c, const double2 a, const double2 b) {
  dmma(c.x, c.y, a.x, b.x);
  dmma(c.x, c.y, a.y, b.y);
}
__device__ __forceinline__ double2 ld2(const double* p) { return *reinterpret_cast<const double2*>(p); }
__device__ __forceinline__ void st2(double* p, double2 v) { *reinterpret_cast<double2*>(p) = v; }

// LDL^T of one 8x8 tile by ONE thread, all in registers, plus the in-place inverse of its
// unit-lower factor.  Writes inv(L11) (zeros above, ones on the diagonal) back into the tile, 1/d
// and -d into dinv / dneg.  A warp issues in order, so the statement order below IS the schedule:
// the pivot chain (reciprocal -> first multiplier -> next pivot) goes first in every column and
// the independent work (remaining multipliers, trailing updates, the row of the inverse that just
// became computable, its stores) is placed right behind it to fill the reciprocal's latency.
__device__ __forceinline__ void factor_diag_tile(double* __restrict__ tile, double* __restrict__ dinv,
                                                 double* __restrict__ dneg) {
  double a[8][8];
  // lower triangle incl. diagonal: 16-byte chunks 0..r/2 of row r
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int cc = 0; cc <= (r >> 1); ++cc) {
      const double2 v = ld2(tile + el_off(r, 2 * cc));
      a[r][2 * cc] = v.x;
      if (2 * cc + 1 <= r) a[r][2 * cc + 1] = v.y;
    }
  double rd[8], dg[8];
  rd[0] = fast_rcp(a[0][0]);
  dg[0] = a[0][0];
  st2(tile + el_off(0, 0), make_double2(1.0, 0.0));
#pragma unroll
  for (int cc = 1; cc < 4; ++cc) st2(tile + el_off(0, 2 * cc), make_double2(0.0, 0.0));
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    // --- chain: row c+1 gets its multiplier and its pivot, then the next reciprocal starts
    if (c + 1 < 8) {
      const double arc = a[c + 1][c];
      const double l = arc * rd[c];
      a[c + 1][c + 1] -= arc * l;
      a[c + 1][c] = l;
      dg[c + 1] = a[c + 1][c + 1];
      rd[c + 1] = fast_rcp(a[c + 1][c + 1]);
    }
    // --- off the chain: rows r >= c+2 (a[r][c] still unscaled = l_rc d_c; rows c2 < r hold l_{c2,c})
#pragma unroll
    for (int r = c + 2; r < 8; ++r) {
      const double arc = a[r][c];
      const double l = arc * rd[c];
#pragma unroll
      for (int c2 = c + 1; c2 < r; ++c2) a[r][c2] -= arc * a[c2][c];
      a[r][r] -= arc * l;
      a[r][c] = l;
    }
    // --- row c+1 of L is final: row c+1 of X = inv(L):  X[i][j] = -(L[i][j] + sum_{j<k<i} L[i][k] X[k][j])
    if (c + 1 < 8) {
      const int i = c + 1;
      double x[8];
#pragma unroll
      for (int j = 0; j < i; ++j) {
        double sm = a[i][j];
#pragma unroll
        for (int k = j + 1; k < i; ++k) sm += a[i][k] * a[k][j];
        x[j] = -sm;
      }
#pragma unroll
      for (int j = 0; j < i; ++j) a[i][j] = x[j];
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        const int c0 = 2 * cc, c1 = 2 * cc + 1;
        const double v0 = c0 < i ? a[i][c0] : (c0 == i ? 1.0 : 0.0);
        const double v1 = c1 < i ? a[i][c1] : (c1 == i ? 1.0 : 0.0);
        st2(tile + el_off(i, c0), make_double2(v0, v1));
      }
    }
  }
#pragma unroll
  for (int c = 0; c < 8; c += 2) {
    st2(dinv + c, make_double2(rd[c], rd[c + 1]));
    st2(dneg + c, make_double2(-dg[c], -dg[c + 1]));
  }
}

// Named barriers (ids 1..15; 0 is __syncthreads): producer warps arrive, consumer warps sync,
// `count` = all threads taking part either way.  The fence makes the producer's shared-memory
// writes visible before the arrival is counted.
// The barrier id is an IMMEDIATE (kBase or kBase + 1, picked by `odd`): with a register operand ptxas has
// to assume that all 16 hardware barriers of the CTA are in use, and the SM runs out of barriers at
// 4 resident CTAs whatever the shared-memory and register budget says.
template <int kBase>
__device__ __forceinline__ void bar_arrive(int odd, int count) {
  __threadfence_block();
  if (odd) asm volatile("bar.arrive %0, %1;" ::"n"(kBase + 1), "r"(count) : "memory");
  else asm volatile("bar.arrive %0, %1;" ::"n"(kBase), "r"(count) : "memory");
}
template <int kBase>
__device__ __forceinline__ void bar_sync(int odd, int count) {
  if (odd) asm volatile("bar.sync %0, %1;" ::"n"(kBase + 1), "r"(count) : "memory");
  else asm volatile("bar.sync %0, %1;" ::"n"(kBase), "r"(count) : "memory");
}

// Developer phase counters of the CTA kernels (-DFCCQP_DEV, FCCQP_PROFILE; slot names: PhaseProfile, fccqp_capi.cu).
// FCCQP_PROF_BEGIN(slots) puts the 16 counters at `slots` (shared memory) and zeroes them; FCCQP_PROF(slot) has thread 0
// add the cycles since its previous mark to a slot, FCCQP_PROF_COUNT(slot) add one; FCCQP_PROF_END() sums them into p.prof.
#ifdef FCCQP_DEV
#define FCCQP_PROF_BEGIN(slots)                                            \
  unsigned long long* const s_prof = (slots);                              \
  long long t_prof = 0;                                                    \
  if (p.prof && tid == 0) { for (int i = 0; i < 16; ++i) s_prof[i] = 0; t_prof = clock64(); }
#define FCCQP_PROF(slot)                                                   \
  do {                                                                     \
    if (p.prof && tid == 0) {                                              \
      const long long t_now = clock64();                                   \
      s_prof[slot] += (unsigned long long)(t_now - t_prof);                \
      t_prof = t_now;                                                      \
    }                                                                      \
  } while (0)
#define FCCQP_PROF_COUNT(slot) do { if (p.prof && tid == 0) s_prof[slot] += 1; } while (0)
#define FCCQP_PROF_END() \
  do { if (p.prof && tid == 0) for (int i = 0; i < 16; ++i) atomicAdd(p.prof + i, s_prof[i]); } while (0)
#else
#define FCCQP_PROF_BEGIN(slots)
#define FCCQP_PROF(slot) do { } while (0)
#define FCCQP_PROF_COUNT(slot) do { } while (0)
#define FCCQP_PROF_END() do { } while (0)
#endif

// One helper step of the left-looking LDL^T for up to T tile rows i_t = i0 + t*stride owned by
// this warp (all >= j+2):
//   (B) L_{i,j}    = C_{i,j} inv(L_jj)' inv(D_j)                      (stored; kept in registers)
//   (A) C_{i,j+1} -= sum_{k<=j} L_{i,k} D_k L_{j+1,k}'                 (in place)
//       C_{i,i}   -= sum_{k<=j} L_{i,k} D_k L_{i,k}'   for i == j+2   (the next-but-one diagonal tile)
// All T tiles advance together: the scaled B operand D_k L_{j+1,k}' is loaded once per k and
// shared, every tile has two independent DMMA chains, so a warp has 2T (+2) DMMAs in flight
// instead of two, and the k = j term comes straight from the registers of step (B).
// Tiles of one tile row are contiguous (64 doubles apart), so the operand pointers just advance.
template <int T>
__device__ __forceinline__ void helper_step(double* __restrict__ M, const double* __restrict__ dneg, int i0,
                                            int stride, int j, const double2 li, const double2 di,
                                            int fragC, int fq, const int cnt) {
  int rowoff[T];
  double2 l[T], ca[T], cb[T];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const int i = t < cnt ? i0 + t * stride : i0;     // unused slots alias the first tile row (never stored)
    rowoff[t] = tile_off(i, 0) + fragC;
    l[t] = ld2(M + rowoff[t] + 64 * j);
    ca[t] = ld2(M + rowoff[t] + 64 * (j + 1));
    cb[t] = make_double2(0.0, 0.0);
  }
  const bool diag = i0 == j + 2;  // warp-uniform
  double* const dgp = M + tile_off(i0, i0) + fragC;
  double2 da = make_double2(0.0, 0.0), db = make_double2(0.0, 0.0);
  if (diag) da = ld2(dgp);
  // (B)
#pragma unroll
  for (int t = 0; t < T; ++t) {
    double2 wa = make_double2(0.0, 0.0), wb = make_double2(0.0, 0.0);
    dmma(wa.x, wa.y, l[t].x, li.x);
    dmma(wb.x, wb.y, l[t].y, li.y);
    l[t] = make_double2((wa.x + wb.x) * di.x, (wa.y + wb.y) * di.y);
    if (t < cnt) st2(M + rowoff[t] + 64 * j, l[t]);
  }
  // (A), terms k < j from shared memory
  const double* bp = M + tile_off(j + 1, 0) + fragC;
  const double* dp = dneg + 2 * fq;
  int ko = 0;
#pragma unroll 1
  for (int k = 0; k < j; ++k, ko += 64, bp += 64, dp += 8) {
    const double2 b = ld2(bp), d = ld2(dp);
    const double bx = b.x * d.x, by = b.y * d.y;
    double2 a[T];
#pragma unroll
    for (int t = 0; t < T; ++t) a[t] = ld2(M + rowoff[t] + ko);
#pragma unroll
    for (int t = 0; t < T; ++t) {
      dmma(ca[t].x, ca[t].y, a[t].x, bx);
      dmma(cb[t].x, cb[t].y, a[t].y, by);
    }
    if (diag) {
      dmma(da.x, da.y, a[0].x, a[0].x * d.x);
      dmma(db.x, db.y, a[0].y, a[0].y * d.y);
    }
  }
  // term k = j from registers
  {
    const double2 b = ld2(bp), d = ld2(dp);
    const double bx = b.x * d.x, by = b.y * d.y;
#pragma unroll
    for (int t = 0; t < T; ++t) {
      dmma(ca[t].x, ca[t].y, l[t].x, bx);
      dmma(cb[t].x, cb[t].y, l[t].y, by);
    }
    if (diag) {
      dmma(da.x, da.y, l[0].x, l[0].x * d.x);
      dmma(db.x, db.y, l[0].y, l[0].y * d.y);
    }
  }
#pragma unroll
  for (int t = 0; t < T; ++t)
    if (t < cnt) st2(M + rowoff[t] + 64 * (j + 1), make_double2(ca[t].x + cb[t].x, ca[t].y + cb[t].y));
  if (diag) st2(dgp, make_double2(da.x + db.x, da.y + db.y));
}

// sigma A'A for T consecutive tiles (I, J0..J0+T-1) of the variable block (cold pre-solve):
//   C_IJ += sigma sum_kb A_{kb,I}' A_{kb,J},  kb over the constraint tile rows.
// The A_{kb,I} operand is shared by the T tiles, each tile has two independent DMMA chains.
template <int T>
__device__ __forceinline__ void ata_chunk(double* __restrict__ M, int NBx, int NB, int I, int J0, double sigma,
                                          int fragC, int fragT) {
  double2 sa[T], sb[T];
#pragma unroll
  for (int t = 0; t < T; ++t) { sa[t] = make_double2(0.0, 0.0); sb[t] = make_double2(0.0, 0.0); }
  // X'Y products take both operands as "fragT" (element (2q+s, l/4), s = 0/1: two 8-byte loads).  Lanes
  // with odd q take s = 1 first: the two loads of a warp then cover all shared-memory banks instead
  // of half of them (2 wavefronts instead of 4), and each DMMA still contracts every k exactly once
  // (k = 2q+s with the same s rule for both operands).
  const int s0 = (fragT >> 4 & 1) << 3, s1 = 8 - s0;   // fragT = (2q) * 8 + ...: bit 4 is q & 1
  const double* ai = M + tile_off(NBx, I) + fragT;
  const double* aj = M + tile_off(NBx, J0) + fragT;
#pragma unroll 1
  for (int kb = NBx; kb < NB; ++kb) {
    const double a0 = ai[s0], a1 = ai[s1];
    double b0[T], b1[T];
#pragma unroll
    for (int t = 0; t < T; ++t) { b0[t] = aj[64 * t + s0]; b1[t] = aj[64 * t + s1]; }
#pragma unroll
    for (int t = 0; t < T; ++t) {
      dmma(sa[t].x, sa[t].y, a0, b0[t]);
      dmma(sb[t].x, sb[t].y, a1, b1[t]);
    }
    ai += 64 * (kb + 1); aj += 64 * (kb + 1);
  }
  double* cp = M + tile_off(I, J0) + fragC;
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const double2 c = ld2(cp + 64 * t);
    st2(cp + 64 * t, make_double2(c.x + sigma * (sa[t].x + sb[t].x), c.y + sigma * (sa[t].y + sb[t].y)));
  }
}

// Row-per-thread dot product over one tile: sum_c T[row][c] * v[c]   (trow = tile + row*8, tf = row/2)
__device__ __forceinline__ double row_dot8(const double* __restrict__ trow, int tf, const double* __restrict__ v) {
  const double2 x0 = ld2(trow + 2 * (0 ^ tf)), x1 = ld2(trow + 2 * (1 ^ tf));
  const double2 x2 = ld2(trow + 2 * (2 ^ tf)), x3 = ld2(trow + 2 * (3 ^ tf));
  const double2 v0 = ld2(v), v1 = ld2(v + 2), v2 = ld2(v + 4), v3 = ld2(v + 6);
  return ((x0.x * v0.x + x0.y * v0.y) + (x1.x * v1.x + x1.y * v1.y)) +
         ((x2.x * v2.x + x2.y * v2.y) + (x3.x * v3.x + x3.y * v3.y));
}
// Column-per-thread dot product over one tile: sum_r T[r][col] * v[r]   (tcol = tile + (col&1), colc = col/2).
// flip (0/1) swaps the rows of every row pair: odd tile columns start on the other half of the banks.
__device__ __forceinline__ double col_dot8(const double* __restrict__ tcol, int colc, int flip,
                                           const double* __restrict__ v) {
  double s0 = 0.0, s1 = 0.0;
  const int f8 = flip << 3;
#pragma unroll
  for (int r = 0; r < 8; r += 2) {
    const int sw = ((colc ^ (r >> 1)) & 3) << 1;
    s0 += tcol[r * 8 + f8 + sw] * v[r + flip];
    s1 += tcol[(r + 1) * 8 - f8 + sw] * v[r + 1 - flip];
  }
  return s0 + s1;
}

// Thread t's part of a product with a lower-stored symmetric tile matrix M, two interleaved partial sums s0 / s1:
//   sym_lower_rows: row t%8 of the tiles (tb, 0..tb), left of and on the diagonal, by rows;
//   sym_lower_cols: column t%8 of the tiles (ib0..NB-1, tb) below it, by columns.
// (tb is the thread's tile row t/8, clamped by the caller where rows past the matrix take part.)
__device__ __forceinline__ void sym_lower_rows(const double* __restrict__ M, const double* __restrict__ v, const int tb,
                                               double& s0, double& s1) {
  const int tr = threadIdx.x & 7, tf = tr >> 1;
  const double* lrow = M + tile_off(tb, 0) + tr * 8;
  int jb = 0;
#pragma unroll 1
  for (; jb + 1 <= tb; jb += 2) {
    s0 += row_dot8(lrow + 64 * jb, tf, v + jb * 8);
    s1 += row_dot8(lrow + 64 * jb + 64, tf, v + jb * 8 + 8);
  }
  if (jb <= tb) s0 += row_dot8(lrow + 64 * jb, tf, v + jb * 8);
}
__device__ __forceinline__ void sym_lower_cols(const double* __restrict__ M, const double* __restrict__ v, const int tb,
                                               int ib, const int NB, double& s0, double& s1) {
  const int tr = threadIdx.x & 7, colo = tr & 1, colc = tr >> 1;
  const int flip = (threadIdx.x >> 3) & 1;   // odd tile columns walk row pairs swapped (bank spread)
#pragma unroll 1
  for (; ib + 1 < NB; ib += 2) {
    s0 += col_dot8(M + tile_off(ib, tb) + colo, colc, flip, v + ib * 8);
    s1 += col_dot8(M + tile_off(ib + 1, tb) + colo, colc, flip, v + ib * 8 + 8);
  }
  if (ib < NB) s0 += col_dot8(M + tile_off(ib, tb) + colo, colc, flip, v + ib * 8);
}
// Row t of the symmetric matrix (NB tile rows) times v.
__device__ __forceinline__ double sym_row_dot(const double* __restrict__ M, const double* __restrict__ v, const int NB) {
  const int tb = threadIdx.x >> 3;
  double s0 = 0.0, s1 = 0.0;
  sym_lower_rows(M, v, tb, s0, s1);
  sym_lower_cols(M, v, tb, tb + 1, NB, s0, s1);
  return s0 + s1;
}


// ---------------------------------------------------------------------------
// Factorization of the assembled tile matrix, in place: unpivoted blocked left-looking LDL^T,
// then the explicit 32x32 diagonal-block inverses the triangular solves use.  Deliberately NOT
// inlined: the call parks the caller's per-row state (bounds, duals, right-hand sides) in
// local memory, so the DMMA loops get the whole register file and ptxas can keep the operand
// loads of several tiles in flight instead of recycling two registers.
// ---------------------------------------------------------------------------
template <int kThreads>
__device__ __noinline__ void factor_tiles(double* __restrict__ M, double* __restrict__ dinv, double* __restrict__ dneg,
                                          const int NB, const int NB32) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kThreads / 32;
  constexpr int kHelpers = kWarps - 1;
  const int fr = lane >> 2, fq = lane & 3;
  const int fragC = (fr << 3) + (((fq ^ (fr >> 1)) & 3) << 1);
  const int fragT = ((2 * fq) << 3) + ((((fr >> 1) ^ fq) & 3) << 1) + (fr & 1);
  // ---------------- unpivoted blocked left-looking LDL^T on 8x8 tiles ----------------
  // Warp 0 runs the critical path: factor the diagonal tile (one thread, registers), turn the
  // tile below it into L, bring the next diagonal tile up to date, signal.  The helper warps
  // stay one tile column behind: they finish the L tiles of column j, then accumulate column
  // j+1 (and the part of the diagonal tile j+2 that does not need column j+1) in place.
  if (warp == 0) {
#pragma unroll 1
    for (int j = 0; j < NB; ++j) {
      double* dt = M + tile_off(j, j);
      if (lane == 0) factor_diag_tile(dt, dinv + 8 * j, dneg + 8 * j);
      __syncwarp();
      if (j > 0) bar_sync<3>((j - 1) & 1, kThreads);   // helpers finished step j-1
      if (j + 1 < NB) {
        const double2 li = ld2(dt + fragC), di = ld2(dinv + 8 * j + 2 * fq);
        double* lp = M + tile_off(j + 1, j) + fragC;
        const double2 c = ld2(lp);
        double2 t1 = ld2(lp + 64);                       // tile (j+1, j+1)
        double2 wa = make_double2(0.0, 0.0), wb = make_double2(0.0, 0.0);
        dmma(wa.x, wa.y, c.x, li.x);
        dmma(wb.x, wb.y, c.y, li.y);
        const double wx = wa.x + wb.x, wy = wa.y + wb.y;   // L D
        const double2 l = make_double2(wx * di.x, wy * di.y);
        st2(lp, l);
        double2 t2 = make_double2(0.0, 0.0);
        dmma(t1.x, t1.y, -wx, l.x);
        dmma(t2.x, t2.y, -wy, l.y);
        st2(lp + 64, make_double2(t1.x + t2.x, t1.y + t2.y));
      }
      bar_arrive<1>(j & 1, kThreads);                     // column j: inv(L_jj), D_j, L_{j+1,j} ready
    }
    bar_sync<3>((NB - 1) & 1, kThreads);
  } else {
#pragma unroll 1
    for (int j = 0; j < NB; ++j) {
      bar_sync<1>(j & 1, kThreads);
      const double2 li = ld2(M + tile_off(j, j) + fragC), di = ld2(dinv + 8 * j + 2 * fq);
      // own tile rows i >= j+2, i = warp-1 (mod kHelpers), four at a time
      int i0 = j + 2;
      i0 += (warp - 1 - i0 % kHelpers + kHelpers) % kHelpers;
#pragma unroll 1
      for (; i0 < NB; i0 += 4 * kHelpers) {
        const int cnt = (NB - i0 + kHelpers - 1) / kHelpers;
        if (cnt > 2) helper_step<4>(M, dneg, i0, kHelpers, j, li, di, fragC, fq, cnt);
        else helper_step<2>(M, dneg, i0, kHelpers, j, li, di, fragC, fq, cnt);
      }
      bar_arrive<3>(j & 1, kThreads);
    }
  }
  __syncthreads();
  // ---------------- explicit inverses of the 32x32 diagonal blocks of L, in place ----------------
  // level 1: 16x16 = [[X1,0],[-X2 L21 X1, X2]] from the 8x8 inverses left by the factorization
#pragma unroll 1
  for (int a = warp; 2 * a + 1 < NB; a += kWarps) {
    const double* x1 = M + tile_off(2 * a, 2 * a) + fragT;
    double* l21 = M + tile_off(2 * a + 1, 2 * a) + fragC;
    const double2 x2 = ld2(M + tile_off(2 * a + 1, 2 * a + 1) + fragC);
    double2 tt = make_double2(0.0, 0.0);                 // fragC((L21 X1)') = fragT(L21 X1)
    mma8(tt, make_double2(x1[0], x1[8]), ld2(l21));      // X1' L21'
    double2 r = make_double2(0.0, 0.0);
    mma8(r, x2, tt);                                     // X2 (L21 X1)
    st2(l21, make_double2(-r.x, -r.y));
  }
  __syncthreads();
  // level 2: 32x32 = [[A,0],[-B L A, B]] with 16x16 A, B; one warp per (block, tile column).
  // Both columns of a block read tiles the other one overwrites: all products first, one
  // barrier, then the stores (the two columns of a block always share a round).
#pragma unroll 1
  for (int base = 0; base < 2 * NB32; base += kWarps) {
    const int w = base + warp;
    const int q4 = (w >> 1) * 4, col = w & 1;
    const bool act = w < 2 * NB32 && q4 + 2 < NB;
    const bool two = q4 + 3 < NB;  // second tile row of the lower-left 16x16 exists
    double2 r0 = make_double2(0.0, 0.0), r1 = make_double2(0.0, 0.0);
    if (act) {
      // T(:,col) = L A(:,col), kept transposed in registers
      double2 t0 = make_double2(0.0, 0.0), t1 = make_double2(0.0, 0.0);
      const double2 l01 = ld2(M + tile_off(q4 + 2, q4 + 1) + fragC);
      double2 l11 = make_double2(0.0, 0.0);
      if (two) l11 = ld2(M + tile_off(q4 + 3, q4 + 1) + fragC);
      if (col == 0) {
        const double2 l00 = ld2(M + tile_off(q4 + 2, q4) + fragC);
        const double* a00 = M + tile_off(q4, q4) + fragT;
        const double* a10 = M + tile_off(q4 + 1, q4) + fragT;
        const double2 f00 = make_double2(a00[0], a00[8]), f10 = make_double2(a10[0], a10[8]);
        mma8(t0, f00, l00); mma8(t0, f10, l01);          // T00' = A00' L00' + A10' L01'
        if (two) {
          const double2 l10 = ld2(M + tile_off(q4 + 3, q4) + fragC);
          mma8(t1, f00, l10); mma8(t1, f10, l11);        // T10'
        }
      } else {
        const double* a11 = M + tile_off(q4 + 1, q4 + 1) + fragT;
        const double2 f11 = make_double2(a11[0], a11[8]);
        mma8(t0, f11, l01);                              // T01' = A11' L01'
        if (two) mma8(t1, f11, l11);                     // T11'
      }
      // R(:,col) = B T(:,col)
      mma8(r0, ld2(M + tile_off(q4 + 2, q4 + 2) + fragC), t0);
      if (two) {
        mma8(r1, ld2(M + tile_off(q4 + 3, q4 + 2) + fragC), t0);
        mma8(r1, ld2(M + tile_off(q4 + 3, q4 + 3) + fragC), t1);
      }
    }
    __syncthreads();
    if (act) {
      st2(M + tile_off(q4 + 2, q4 + col) + fragC, make_double2(-r0.x, -r0.y));
      if (two) st2(M + tile_off(q4 + 3, q4 + col) + fragC, make_double2(-r1.x, -r1.y));
    }
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------
// x = K^{-1} rhs with the factors left by factor_tiles: L y = rhs, D^{-1}, L' x = y, 32 rows per
// step (one warp applies the explicit inverse of a 32x32 diagonal block, the others subtract the
// 32-column slab).  Thread t owns row t: `acc` is its right-hand-side entry, the return value its
// solution entry (rows >= N8 return 0).  Not inlined, for the same reason as factor_tiles.
// ---------------------------------------------------------------------------
__device__ __noinline__ double kkt_solve(const double* __restrict__ M, const double* __restrict__ dinv,
                                         double* __restrict__ tbuf, double* __restrict__ ybuf, double acc,
                                         const int NB, const int NB32, const int N8) {
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const bool is_row = t < N8;
  const int tb = t >> 3, tr = t & 7, tf = tr >> 1;
  const int colo = tr & 1, colc = tr >> 1;
  const int flip = tb & 1;
  const int tbe = tb < NB ? tb : NB - 1;
  double val = 0.0;
  (void)lane;
  // ---- forward: L y = rhs, 32 rows per step (warp J applies inv(L_JJ), later warps subtract).
  // Tiles of a tile row are contiguous; tiles beyond the diagonal are clamped and masked.
  const double* lrow = M + tile_off(tbe, 0) + tr * 8;
#pragma unroll 1
  for (int J = 0; J < NB32; ++J) {
    const int Jb0 = J * 4;
    if (warp == J) {
      tbuf[t] = acc;
      __syncwarp();
      double s = 0.0;
#pragma unroll 1
      for (int jb = Jb0; jb <= tbe; ++jb) s += row_dot8(lrow + 64 * jb, tf, tbuf + jb * 8);
      val = is_row ? s : 0.0;
      ybuf[t] = val;
    }
    __syncthreads();
    if (warp > J && is_row) {
      double s = 0.0;
#pragma unroll 2
      for (int jb = Jb0; jb < Jb0 + 4; ++jb) s += row_dot8(lrow + 64 * jb, tf, ybuf + jb * 8);
      acc -= s;
    }
  }
  // ---- D^{-1}
  acc = is_row ? val * dinv[t] : 0.0;
  // ---- backward: L' x = y (column-per-thread reads; odd tile columns take row pairs swapped)
#pragma unroll 1
  for (int J = NB32 - 1; J >= 0; --J) {
    const int Jb0 = J * 4, Jb1 = min(Jb0 + 4, NB);
    if (warp == J) {
      tbuf[t] = acc;
      __syncwarp();
      double s = 0.0;
#pragma unroll 1
      for (int ib = tbe; ib < Jb1; ++ib) s += col_dot8(M + tile_off(ib, tbe) + colo, colc, flip, tbuf + ib * 8);
      val = is_row ? s : 0.0;
      ybuf[t] = val;
    }
    __syncthreads();
    if (warp < J) {
      double s = 0.0;
#pragma unroll 2
      for (int ib = Jb0; ib < Jb1; ++ib) s += col_dot8(M + tile_off(ib, tb) + colo, colc, flip, ybuf + ib * 8);
      acc -= s;
    }
  }
  return val;
}

// ---------------------------------------------------------------------------
// Long-running QPs (the 1-2 % that iterate towards max_iter dominate both the mean and the tail of
// a batch): after SolveParams::full_inverse_at ADMM iterations the factor is completed to
// W = inv(L), in place (complete_inverse), x_base = [K^{-1} (-b; b_eq)]_x is formed with two triangular
// matrix-vector products (kkt_solve_full) and G = [K^{-1}]_xx replaces the top-left tiles of W
// (form_g); every later x-update is x = x_base + rho G (x_bar - mu) (g_apply): one symmetric
// n x n matrix-vector product and one barrier instead of 2 x N/32 dependent block steps.
//
// complete_inverse: recursive doubling from the 32x32 diagonal-block inverses factor_tiles left.
// For block sizes s = 4, 8, 16 tiles, neighbouring diagonal blocks A (tiles [q, q+s)) and B (tiles
// [q+s, q+2s), clipped) whose inverses are in place absorb the block C below A / left of B:
//     inv([[A, 0], [C, B]]) = [[inv A, 0], [-inv(B) C inv(A), inv B]].
// Phase 0: C <- C inv(A), phase 1: C <- -inv(B) C.  A task is one tile row (phase 0) or tile
// column (phase 1) of C in chunks of up to four tiles sharing one operand.  In-place hazards
// (a chunk overwrites tiles that chunks to its left / above still read) are covered by the task
// order (phase 0: left chunks first, phase 1: bottom chunks first) and by "all products,
// barrier, all stores, barrier" within a round.
// ---------------------------------------------------------------------------
template <int kThreads>
__device__ __noinline__ void complete_inverse(double* __restrict__ M, const int NB) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int kWarps = kThreads / 32;
  const int fr = lane >> 2, fq = lane & 3;
  const int fragC = (fr << 3) + (((fq ^ (fr >> 1)) & 3) << 1);
  const int fragT = ((2 * fq) << 3) + ((((fr >> 1) ^ fq) & 3) << 1) + (fr & 1);
#pragma unroll 1
  for (int s = 4; s < NB; s <<= 1) {
    const int nchunk = (s + 3) >> 2;
    const int npair = (NB + 2 * s - 1) / (2 * s);
    const int ntask = npair * s;               // (pair, line): line = row of C (phase 0) / column of C (phase 1)
#pragma unroll 1
    for (int phase = 0; phase < 2; ++phase) {
#pragma unroll 1
      for (int c = 0; c < nchunk; ++c) {
#pragma unroll 1
        for (int base = 0; base < ntask; base += kWarps) {
          const int task = base + warp;
          const int pr = task / s, ln = task - pr * s;
          const int q = pr * 2 * s;            // A = [q, q+s), B = [q+s, qe)
          const int qe = min(q + 2 * s, NB);
          const int nb = qe - (q + s);         // tile rows of C (<= 0: no B block)
          bool act = task < ntask && nb > 0;
          double2 r[4], rb[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) { r[u] = make_double2(0.0, 0.0); rb[u] = make_double2(0.0, 0.0); }
          int cnt = 0, i = 0, j = 0;
          if (phase == 0) {
            // row i of C, columns j..j+cnt-1 of A:  T_ij = sum_{k=j}^{q+s-1} C_ik Ainv_kj
            act = act && ln < nb;
            i = q + s + ln; j = q + 4 * c; cnt = min(4, q + s - j);
            if (act && cnt > 0) {
#pragma unroll 1
              for (int k = j; k < q + s; ++k) {
                const double2 a = ld2(M + tile_off(i, k) + fragC);
                const double* bp = M + tile_off(k, j) + fragT;
#pragma unroll
                for (int u = 0; u < 4; ++u)
                  if (u < cnt && j + u <= k) {
                    dmma(r[u].x, r[u].y, a.x, bp[64 * u]);
                    dmma(rb[u].x, rb[u].y, a.y, bp[64 * u + 8]);
                  }
              }
#pragma unroll
              for (int u = 0; u < 4; ++u) { r[u].x += rb[u].x; r[u].y += rb[u].y; }
            }
          } else {
            // column j of C, rows i..i+cnt-1 of B, bottom chunk first:  R_ij = -sum_{k=q+s}^{i} Binv_ik T_kj
            j = q + ln;
            const int cc = ((nb + 3) >> 2) - 1 - c;
            act = act && cc >= 0;
            i = q + s + 4 * cc; cnt = min(4, qe - i);
            if (act && cnt > 0) {
#pragma unroll 1
              for (int k = q + s; k < i + cnt; ++k) {
                const double* bp = M + tile_off(k, j) + fragT;
                const double b0 = bp[0], b1 = bp[8];
#pragma unroll
                for (int u = 0; u < 4; ++u)
                  if (u < cnt && i + u >= k) {
                    const double2 a = ld2(M + tile_off(i + u, k) + fragC);
                    dmma(r[u].x, r[u].y, a.x, b0);
                    dmma(rb[u].x, rb[u].y, a.y, b1);
                  }
              }
#pragma unroll
              for (int u = 0; u < 4; ++u) { r[u].x = -(r[u].x + rb[u].x); r[u].y = -(r[u].y + rb[u].y); }
            }
          }
          __syncthreads();
          if (act && cnt > 0) {
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (u < cnt) {
                if (phase == 0) st2(M + tile_off(i, j + u) + fragC, r[u]);
                else st2(M + tile_off(i + u, j) + fragC, r[u]);
              }
          }
          __syncthreads();
        }
      }
    }
  }
}

// x = W' D^{-1} W rhs with the full inverse W = inv(L) of complete_inverse.  Thread t owns row t of
// the forward product (tiles (tb, 0..tb), contiguous) and column t of the backward one (tiles
// (tb..NB-1, tb)): NB + 1 tile-vector products per thread whatever its row, two barriers per solve.
__device__ __noinline__ double kkt_solve_full(const double* __restrict__ M, const double* __restrict__ dinv,
                                              double* __restrict__ tbuf, double* __restrict__ ybuf, double acc,
                                              const int NB, const int N8) {
  const int t = threadIdx.x;
  const bool is_row = t < N8;
  const int tb = t >> 3;
  const int tbe = tb < NB ? tb : NB - 1;
  if (is_row) tbuf[t] = acc;
  __syncthreads();
  {
    double s0 = 0.0, s1 = 0.0;
    sym_lower_rows(M, tbuf, tbe, s0, s1);
    if (is_row) ybuf[t] = (s0 + s1) * dinv[t];
  }
  __syncthreads();
  double s0 = 0.0, s1 = 0.0;
  sym_lower_cols(M, ybuf, tbe, tbe, NB, s0, s1);
  return is_row ? s0 + s1 : 0.0;
}

// G = [K^{-1}]_xx = sum_K W_{K,:n8}' D_K^{-1} W_{K,:n8}, written over the top-left NBx x NBx tile triangle of
// W (W is not needed afterwards): with x_base = [K^{-1} (-b; b_eq)]_x every later x-update is
//     x = x_base + rho G (x_bar - mu)        (one symmetric matrix-vector product, one barrier).
// One chunk of up to four tiles (I, J..J+3) per warp and round; chunks in ascending row order, so a
// round only overwrites W rows that no later chunk reads (row I' > I needs W_{K,.} for K >= I' only;
// the K = I term of a later chunk of the SAME row reads tile (I,I) and its own columns, which are
// stored with that chunk).  All products of a round, barrier, all stores, barrier.
template <int kThreads>
__device__ __noinline__ void form_g(double* __restrict__ M, const double* __restrict__ dinv, const int NB, const int NBx,
                                    const int NBr) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int kWarps = kThreads / 32;
  const int fr = lane >> 2, fq = lane & 3;
  const int fragC = (fr << 3) + (((fq ^ (fr >> 1)) & 3) << 1);
  const int fragT = ((2 * fq) << 3) + ((((fr >> 1) ^ fq) & 3) << 1) + (fr & 1);
  // NBr = NBx: G itself.  NBr = NB: the rows [K^{-1}]_cx below it as well (tiles (I >= NBx, J < NBx)), so that
  // [K^{-1}]_{x,:} rhs is one product over the lower-stored block column (shared-structure batches).
  int I = 0, J = 0;               // chunk cursor: row I, first column J
  bool more = NBr > 0;
#pragma unroll 1
  while (more) {
    // this warp's chunk = cursor advanced by `warp` chunks; then the cursor moves kWarps chunks on
    int ci = I, cj = J;
    bool act = true;
#pragma unroll 1
    for (int k = 0; k < warp && act; ++k) { cj += 4; if (cj > min(ci, NBx - 1)) { ++ci; cj = 0; } act = ci < NBr; }
    double2 r[4], rb[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { r[u] = make_double2(0.0, 0.0); rb[u] = make_double2(0.0, 0.0); }
    const int cnt = act ? min(4, min(ci, NBx - 1) + 1 - cj) : 0;
    if (act) {
#pragma unroll 1
      for (int K = ci; K < NB; ++K) {
        const double* ap = M + tile_off(K, ci) + fragT;
        const double2 d = ld2(dinv + 8 * K + 2 * fq);
        const double a0 = ap[0] * d.x, a1 = ap[8] * d.y;
        const double* bp = M + tile_off(K, cj) + fragT;
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (u < cnt) {
            dmma(r[u].x, r[u].y, a0, bp[64 * u]);
            dmma(rb[u].x, rb[u].y, a1, bp[64 * u + 8]);
          }
      }
    }
    __syncthreads();
    if (act) {
      double* cp = M + tile_off(ci, cj) + fragC;
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (u < cnt) st2(cp + 64 * u, make_double2(r[u].x + rb[u].x, r[u].y + rb[u].y));
    }
    __syncthreads();
#pragma unroll 1
    for (int k = 0; k < kWarps && more; ++k) { J += 4; if (J > min(I, NBx - 1)) { ++I; J = 0; } more = I < NBr; }
  }
}

// (G w)_t for the variable rows t < n8 (0 elsewhere): row part over tiles (tb, 0..tb), column part over
// tiles (tb+1.., tb) of the lower-stored symmetric G.
__device__ __noinline__ double g_apply(const double* __restrict__ M, double* __restrict__ tbuf, double w,
                                       const int NBr, const int n8) {
  const int t = threadIdx.x;
  if (t < 8 * NBr) tbuf[t] = w;      // NBr tile rows of the operand take part (NBx: w; NB: a full KKT right-hand side)
  __syncthreads();
  if (t >= n8) return 0.0;
  return sym_row_dot(M, tbuf, NBr);
}

// ---------------------------------------------------------------------------
// The fused solve kernel.  kThreads >= padded KKT size N8 (one thread per KKT row in the
// triangular solves and all vector work).  Warp 0 is the factorization's critical-path warp,
// warps 1.. are its helpers.
// ---------------------------------------------------------------------------
template <int kThreads, int kMinBlocks, bool kShared, bool kF32, bool kAdapt = false>
__global__ void __launch_bounds__(kThreads, kMinBlocks) fccqp_solve_kernel(const SolveParams p) {
  // kAdapt: the adaptive-rho extension compiled in (separate instances: the default path carries none of it)
  // kF32: the problem data (Q, b, A_eq, b_eq, friction_coeffs, lb, ub) are float32 arrays (same element
  // strides); they are widened on the way into shared memory / registers, everything else is FP64.
  // kShared = false compiles the shared-structure logic out of the general kernel
  const int shared_mode = kShared ? p.shared_mode : 0;
  extern __shared__ __align__(16) double smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kThreads / 32;
  const int n = p.n, m = p.m, nc = p.nc, lcs = p.lcs;
  const int n8 = p.lay.n8, N8 = p.lay.N8, NB = p.lay.NB, NBx = p.lay.NBx, NB32 = p.lay.NB32;

  double* const M = smem + p.lay.off_M;
  double* const dinv = smem + p.lay.off_dinv;
  double* const dneg = smem + p.lay.off_dneg;
  double* const tbuf = smem + p.lay.off_tbuf;
  double* const ybuf = smem + p.lay.off_ybuf;
  double* const xs = smem + p.lay.off_xs;
  double* const lcbar = smem + p.lay.off_lcbar;
  double* const muc = smem + p.lay.off_muc;
  double* const vmu = smem + p.lay.off_mu;
  double* const red = smem + p.lay.off_red;
  int* const ibuf = reinterpret_cast<int*>(smem + p.lay.off_int);
  int* const s_work = ibuf;  // [1]
  FCCQP_PROF_BEGIN(reinterpret_cast<unsigned long long*>(ibuf + 2));

  int parity = 0;
  // thread-per-row identity: rows [0,n) variables, [n,n8) pads, [n8,n8+m) constraints, rest pads
  const int t = tid;
  const bool is_x = t < n;
  const bool is_c = t >= n8 && t < n8 + m;
  const bool is_row = t < N8;
  const bool in_cone = is_x && t >= lcs && t < lcs + nc;
  const int tb = t >> 3, tr = t & 7, tf = tr >> 1;  // tile row, row in tile, row swizzle
  const int colo = tr & 1, colc = tr >> 1;          // column-per-thread access: element (r, tr) of a tile
  const int flip = tb & 1;                          // odd tile columns walk row pairs swapped (bank spread)
  // tensor-core fragment coordinates of this lane
  const int fr = lane >> 2, fq = lane & 3;
  const int fragC = (fr << 3) + (((fq ^ (fr >> 1)) & 3) << 1);                       // (fr, 2fq..2fq+1)
  const int fragT = ((2 * fq) << 3) + ((((fr >> 1) ^ fq) & 3) << 1) + (fr & 1);      // (2fq, fr); +8 for (2fq+1, fr)

  // Q is symmetric: walk it along whichever stride is contiguous.
  auto ldin = [](const double* base, size_t idx) -> double {
    return kF32 ? (double)reinterpret_cast<const float*>(base)[idx] : base[idx];
  };
  const long long q_slow = p.q_cs <= p.q_rs ? p.q_rs : p.q_cs;
  const long long q_fast = p.q_cs <= p.q_rs ? p.q_cs : p.q_rs;

  const int Btot = p.count_dev ? (int)*p.count_dev : p.B;
  // cold ADMM launch of a shared-structure batch: x0 of the pre-solve launch is in p.x, pass 0 is done.
  // (A WARM batch launched directly in mode 2 has had no pre-solve launch: equality-constrained QPs still
  // take pass 0 there, fcc_qp.cpp:159.)
  const bool resume = shared_mode == 2 && !p.warm;
  int cached_pass = -1;                     // shared-structure modes: which KKT factorization sits in M
  int factor_flag = 0;                      // 2: the factorization in M had the wrong inertia / a non-finite pivot
  double sigma_cached = 1.0;
  for (;;) {
    __syncthreads();  // previous QP fully retired (smem reuse) before taking new work
    if (tid == 0) *s_work = (int)atomicAdd(p.work_counter, 1u);
    __syncthreads();
    const int qslot = *s_work;
    if (qslot >= Btot) break;
    const int qp = p.index_list ? p.index_list[qslot] : qslot;

    const double* Qg = p.Q + (size_t)qp * p.q_bs;
    const double* Ag = p.A + (size_t)qp * p.a_bs;
    // 16-byte copies need contiguous rows, 16-byte aligned row starts and an even n
    const bool q_vec = q_fast == 1 && (n & 1) == 0 &&
                       ((reinterpret_cast<uintptr_t>(Qg) | (uintptr_t)(q_slow * 8)) & 15) == 0;
    const bool a_vec = p.a_cs == 1 && (n & 1) == 0 &&
                       ((reinterpret_cast<uintptr_t>(Ag) | (uintptr_t)(p.a_rs * 8)) & 15) == 0;

    // ---------------- K0: vectors (one register per row and vector) ----------------
    double v_b = 0.0;       // b (variable rows) or b_eq (constraint rows)
    double v_lb = 0.0, v_ub = 0.0, v_mux = 0.0, v_xbar = 0.0, v_x = 0.0;
    int finite_bounds = 0;
    if (is_x) {
      v_b = ldin(p.b, (size_t)qp * p.b_bs + t);
      v_lb = ldin(p.lb, (size_t)qp * p.lb_bs + t);
      v_ub = ldin(p.ub, (size_t)qp * p.ub_bs + t);
      if (!isinf(v_lb) || !isinf(v_ub)) finite_bounds = 1;
      if (p.warm || resume) v_x = p.x[(size_t)qp * n + t];
      if (p.warm) v_mux = p.mu_x[(size_t)qp * n + t];
    } else if (is_c) {
      v_b = ldin(p.beq, (size_t)qp * p.beq_bs + (t - n8));
    }
    if (t < n8) xs[t] = v_x;
    if (t < nc / 3) vmu[t] = ldin(p.mu, (size_t)qp * p.mu_bs + t);
    if (t < nc) muc[t] = p.warm ? p.mu_c[(size_t)qp * nc + t] : 0.0;
    // equality-constrained (fcc_qp.cpp:132-133) needs nc == 0 AND no finite bound: with contacts the block-wide
    // vote -- and the stall on the bound loads it implies -- is skipped (nothing below reads another thread's
    // K0 shared-memory writes before the next barrier)
    const bool eqc = (nc == 0) && (__syncthreads_or(finite_bounds) == 0);
    const bool presolve = eqc || !p.warm;                                  // fcc_qp.cpp:159

    const long long t_start = clock64();
    unsigned long long fact_cycles = 0;
    int status_flag = 0;
    bool reg_used = false;   // a factorization of this QP needed the regularised retry (rank-deficient A_eq)
    bool reg_mine = false;   //   ... and this thread's constraint row is one of the regularised ones
    double reg_delta = 0.0;  //   ... with -reg_delta on its diagonal
    int reg_tries = 0;
    int n_iter = 0;
    double res_x = 0.0, res_c = 0.0;
    FCCQP_PROF(0);

    // pass 0: cold pre-solve on [[Q + sigma A'A, A'],[A,0]];  pass 1: ADMM on [[Q + rho I, A'],[A,0]].
    // A KKT matrix is assembled and factored lazily, right before the first solve that needs it.
    // Cold solves never need pass 1's for their first x-update: ADMM starts from x_bar = x0 and
    // zero duals (fcc_qp.cpp:74-75,136-139), so x-update 0 minimises
    //   1/2 x'Qx + b'x + rho/2 |x - x0|^2   s.t.  A x = b_eq,
    // whose minimiser is x0 itself (x0 minimises the first two terms on the same set).  The kernel
    // takes that x-update as the identity: a QP whose pre-solve point already passes the exit test
    // (98 % of the walking log) finishes without the second factorization; the others factor and
    // carry on from iteration 1.
    bool defer = false;   // shared_mode 1: this QP needs ADMM iterations, hand it to the second launch
    for (int pass = (presolve && !resume) ? 0 : 1; pass < 2 && !defer; ++pass) {
      if (pass == 1 && eqc) break;
      if (pass == 1) {
        // ADMM initial slack (fcc_qp.cpp:74-75): x_bar = x, lambda_c_bar = x[lambda_c segment]
        v_xbar = v_x;
        if (in_cone) lcbar[t - lcs] = v_x;
        __syncthreads();
        n_iter = p.max_iter;
      }
      const int iters = pass == 0 ? 1 : p.max_iter;
      bool factored = false;
      bool full_inverse = false;   // long-running QP: x-updates through G = [K^{-1}]_xx
      double v_xbase = 0.0;        // its x_base entry of row t
      double rhs0 = 0.0;   // pass-0 right-hand side of row t
      double rho_cur = p.rho;      // (changes only with the adaptive-rho extension, SolveParams::adapt_k)

#pragma unroll 1
      for (int iter = 0; iter < iters; ++iter) {
      double val = v_x;    // solution component of row t (t < N8)
      if (!(pass == 1 && iter == 0 && presolve)) {
      while (!factored) {   // (a second trip only for a rank-deficient A_eq, see reg_delta below)
      factored = true;
      const long long t_f0 = clock64();
      if (shared_mode != 0 && cached_pass == pass) {
        // shared structure: the factors (and inv(L)) of an earlier QP of this CTA are still in M; only the
        // pre-solve right-hand side -b + sigma A' b_eq is new (A from global memory: shared, L2-resident)
        if (pass == 0) {
          // (b_eq staged in ybuf: the operator product below refills tbuf while slower threads still read)
          if (t >= n8 && t < N8) ybuf[t] = is_c ? v_b : 0.0;
          __syncthreads();
          if (is_x) {
            double s0 = 0.0;
            const double* acol = Ag + (long long)t * p.a_cs;
#pragma unroll 4
            for (int k = 0; k < m; ++k) s0 = fma(acol[(long long)k * p.a_rs], ybuf[n8 + k], s0);
            rhs0 = fma(sigma_cached, s0, -v_b);
          } else if (is_c) {
            rhs0 = v_b;
          }
        }
      } else {

      // ---------------- assemble the lower tiles of the padded KKT matrix ----------------
      // one warp per tile, lane = (row fr, column pair 2fq): 8 x 64-byte row segments from HBM/L2.
      // Tile rows outer, warps strided over the tile columns.
      if constexpr (kF32) {
        // float32 problem data: stage 0 copies each tile's 8 x 8 floats asynchronously into the first
        // 256 bytes of its own 512-byte slot, stage 1 widens them in place (all lanes of the owning
        // warp read their pair, __syncwarp, write the FP64 pair / the pad value at its final place)
        const float* Qf = reinterpret_cast<const float*>(p.Q) + (size_t)qp * p.q_bs;
        const float* Af = reinterpret_cast<const float*>(p.A) + (size_t)qp * p.a_bs;
        const bool q_v2 = q_fast == 1 && (n & 1) == 0 && ((reinterpret_cast<uintptr_t>(Qf) | (uintptr_t)(q_slow * 4)) & 7) == 0;
        const bool a_v2 = p.a_cs == 1 && (n & 1) == 0 && ((reinterpret_cast<uintptr_t>(Af) | (uintptr_t)(p.a_rs * 4)) & 7) == 0;
        const int gc0 = 2 * fq;
        const int stg = fr * 4 + fq;   // staging slot of this lane inside a tile (in doubles = float pairs)
#pragma unroll 1
        for (int stage = 0; stage < 2; ++stage) {
          const float* qrow = Qf + fr * q_slow + gc0 * q_fast;
#pragma unroll 1
          for (int I = 0; I < NBx; ++I, qrow += 8 * q_slow) {
            const int gi = 8 * I + fr;
#pragma unroll 1
            for (int J = warp; J <= I; J += kWarps) {
              const int gc = 8 * J + gc0;
              double* tile = M + tile_off(I, J);
              const float* src = qrow + (8 * J) * q_fast;
              const bool d0 = gi < n && gc < n, d1 = gi < n && gc + 1 < n;
              if (stage == 0) {
                if (q_v2) { if (d0) cp_async8(tile + stg, reinterpret_cast<const double*>(src)); }
                else {
                  if (d0) cp_async4(reinterpret_cast<float*>(tile + stg), src);
                  if (d1) cp_async4(reinterpret_cast<float*>(tile + stg) + 1, src + q_fast);
                }
              } else {
                const float2 v = *reinterpret_cast<const float2*>(tile + stg);
                __syncwarp();
                st2(tile + fragC, make_double2(d0 ? (double)v.x : (gi == gc ? 1.0 : 0.0),
                                               d1 ? (double)v.y : (gi == gc + 1 ? 1.0 : 0.0)));
              }
            }
          }
          const float* arow = Af + (long long)fr * p.a_rs + gc0 * p.a_cs;
#pragma unroll 1
          for (int I = NBx; I < NB; ++I, arow += 8 * p.a_rs) {
            const int k = 8 * (I - NBx) + fr;
#pragma unroll 1
            for (int J = warp; J < NBx; J += kWarps) {
              const int gc = 8 * J + gc0;
              double* tile = M + tile_off(I, J);
              const float* src = arow + (8 * J) * p.a_cs;
              const bool d0 = k < m && gc < n, d1 = k < m && gc + 1 < n;
              if (stage == 0) {
                if (a_v2) { if (d0) cp_async8(tile + stg, reinterpret_cast<const double*>(src)); }
                else {
                  if (d0) cp_async4(reinterpret_cast<float*>(tile + stg), src);
                  if (d1) cp_async4(reinterpret_cast<float*>(tile + stg) + 1, src + p.a_cs);
                }
              } else {
                const float2 v = *reinterpret_cast<const float2*>(tile + stg);
                __syncwarp();
                st2(tile + fragC, make_double2(d0 ? (double)v.x : 0.0, d1 ? (double)v.y : 0.0));
              }
            }
            if (stage == 0) {
              // (2,2) block: zero; decoupled unit pivots on the constraint pads
              double* dst = M + tile_off(I, NBx + warp) + fragC;
#pragma unroll 1
              for (int J = NBx + warp; J <= I; J += kWarps, dst += 64 * kWarps) {
                const bool dg = J == I && k >= m;
                st2(dst, make_double2((dg && fr == gc0) ? 1.0 : 0.0, (dg && fr == gc0 + 1) ? 1.0 : 0.0));
              }
            }
          }
          if (stage == 0) { cp_async_wait_all(); __syncthreads(); }
        }
      } else {
        const int gc0 = 2 * fq;
        // Q (symmetric; row read along the contiguous direction), unit pivots on the pads
        const double* qrow = Qg + fr * q_slow + gc0 * q_fast;
#pragma unroll 1
        for (int I = 0; I < NBx; ++I, qrow += 8 * q_slow) {
          const int gi = 8 * I + fr;
          double* dst = M + tile_off(I, warp) + fragC;
          const double* src = qrow + (8 * warp) * q_fast;
#pragma unroll 1
          for (int J = warp; J <= I; J += kWarps, dst += 64 * kWarps, src += 8 * kWarps * q_fast) {
            const int gc = 8 * J + gc0;
            if (q_vec) {
              if (gi < n && gc < n) cp_async16(dst, src);
              else st2(dst, make_double2(gi == gc ? 1.0 : 0.0, gi == gc + 1 ? 1.0 : 0.0));
            } else {
              if (gi < n && gc < n) cp_async8(dst, src); else dst[0] = (gi == gc) ? 1.0 : 0.0;
              if (gi < n && gc + 1 < n) cp_async8(dst + 1, src + q_fast); else dst[1] = (gi == gc + 1) ? 1.0 : 0.0;
            }
          }
        }
        // A rows below it
        const double* arow = Ag + (long long)fr * p.a_rs + gc0 * p.a_cs;
#pragma unroll 1
        for (int I = NBx; I < NB; ++I, arow += 8 * p.a_rs) {
          const int k = 8 * (I - NBx) + fr;
          double* dst = M + tile_off(I, warp) + fragC;
          const double* src = arow + (8 * warp) * p.a_cs;
#pragma unroll 1
          for (int J = warp; J < NBx; J += kWarps, dst += 64 * kWarps, src += 8 * kWarps * p.a_cs) {
            const int gc = 8 * J + gc0;
            if (a_vec) {
              if (k < m && gc < n) cp_async16(dst, src); else st2(dst, make_double2(0.0, 0.0));
            } else {
              if (k < m && gc < n) cp_async8(dst, src); else dst[0] = 0.0;
              if (k < m && gc + 1 < n) cp_async8(dst + 1, src + p.a_cs); else dst[1] = 0.0;
            }
          }
          // (2,2) block: zero; decoupled unit pivots on the constraint pads
          dst = M + tile_off(I, NBx + warp) + fragC;
#pragma unroll 1
          for (int J = NBx + warp; J <= I; J += kWarps, dst += 64 * kWarps) {
            const bool dg = J == I && k >= m;
            st2(dst, make_double2((dg && fr == gc0) ? 1.0 : 0.0, (dg && fr == gc0 + 1) ? 1.0 : 0.0));
          }
        }
      }
      cp_async_wait_all();
      __syncthreads();
      FCCQP_PROF(1);

      // retry after a failed factorization: -delta on the (so far zero) diagonal entry of the dependent constraint rows
      if (reg_mine) M[mat_off(t, t)] = -reg_delta;
      if (pass == 1) {
        if (is_x) M[mat_off(t, t)] += rho_cur;
      } else {
        // sigma = trace(Q) / ||A||_F^2 balances the two terms of Q + sigma A'A
        double trq = is_x ? M[mat_off(t, t)] : 0.0, fro = 0.0;
        if (t >= n8 && t < N8) tbuf[t] = is_c ? v_b : 0.0;
        if (is_c) {
          double f1 = 0.0, f2 = 0.0, f3 = 0.0;
#pragma unroll 2
          for (int jb = 0; jb < NBx; ++jb) {
            const double* row = M + tile_off(tb, jb) + tr * 8;
            const double2 v0 = ld2(row + 2 * (0 ^ tf)), v1 = ld2(row + 2 * (1 ^ tf));
            const double2 v2 = ld2(row + 2 * (2 ^ tf)), v3 = ld2(row + 2 * (3 ^ tf));
            fro = fma(v0.x, v0.x, fma(v0.y, v0.y, fro)); f1 = fma(v1.x, v1.x, fma(v1.y, v1.y, f1));
            f2 = fma(v2.x, v2.x, fma(v2.y, v2.y, f2)); f3 = fma(v3.x, v3.x, fma(v3.y, v3.y, f3));
          }
          fro = (fro + f1) + (f2 + f3);
        }
        block_reduce2<true>(trq, fro, red, parity);
        const double sigma = (trq > 0.0 && fro > 0.0 && isfinite(trq / fro)) ? trq / fro : 1.0;
        sigma_cached = sigma;
        // rhs_x = -b + sigma A' b_eq (needs A before the factorization overwrites it)
        if (is_x) {
          double s = 0.0;
#pragma unroll 1
          for (int ib = NBx; ib < NB; ++ib) s += col_dot8(M + tile_off(ib, tb) + colo, colc, flip, tbuf + ib * 8);
          rhs0 = -v_b + sigma * s;
        } else if (is_c) {
          rhs0 = v_b;
        }
        // H += sigma A'A on the tiles of the variable block, in place: chunks of up to four tiles of
        // one tile row (shared A operand, 2 x cnt independent DMMA chains), round-robin over the warps
        {
          int ch = 0;
#pragma unroll 1
          for (int I = 0; I < NBx; ++I) {
#pragma unroll 1
            for (int J0 = 0; J0 <= I; J0 += 4, ++ch) {
              if (ch % kWarps != warp) continue;
              const int cnt = I + 1 - J0;
              if (cnt >= 4) ata_chunk<4>(M, NBx, NB, I, J0, sigma, fragC, fragT);
              else if (cnt == 3) ata_chunk<3>(M, NBx, NB, I, J0, sigma, fragC, fragT);
              else if (cnt == 2) ata_chunk<2>(M, NBx, NB, I, J0, sigma, fragC, fragT);
              else ata_chunk<1>(M, NBx, NB, I, J0, sigma, fragC, fragT);
            }
          }
        }
      }
      __syncthreads();
      FCCQP_PROF(2);

      factor_tiles<kThreads>(M, dinv, dneg, NB, NB32);
      FCCQP_PROF(3);
      fact_cycles += (unsigned long long)(clock64() - t_f0);
      {
        // Inertia of the quasi-definite KKT matrix: positive pivots on the variable rows (and all pads),
        // negative ones on the constraint rows.  Anything else means Q + sigma A'A (or Q + rho I) is not
        // positive definite on this QP or A_eq lost row rank -- the unpivoted factors are meaningless even
        // when x comes out finite (the reference pivots / falls back to COD there): NUMERICAL_ISSUE.
        // A pivot of the right sign that is pure rounding noise (nearly dependent rows of A_eq; Q + sigma A'A
        // singular to working precision) is caught by its size: below kPivotRatio times the largest pivot of its
        // own class (variable rows / constraint rows) -- legitimate scale differences inside one class stay
        // many orders of magnitude above that (fccqp.h, "conditioning limit").
        bool badp = false;
        double pa = 0.0, pc = 0.0;
        const double dn = is_row ? dneg[t] : 0.0;   // -d_t
        if (is_row) {
          badp = !isfinite(dn) || (is_c ? !(dn > 0.0) : !(dn < 0.0));
          if (is_c) pc = fabs(dn); else if (pass == 0) pa = fabs(dn);   // (Q + rho I: any spread of scales is legitimate)
        }
        block_reduce2<false>(pa, pc, red, parity);
        if (is_row && fabs(dn) < kPivotRatio * (is_c ? pc : pa)) badp = true;
        factor_flag = __syncthreads_or(badp) ? 2 : 0;
        // Rank-deficient A_eq (dependent constraint rows): the reference's LDLT fails there too and its COD fall-back
        // returns the minimum-norm solution of the singular KKT system (src/fcc_qp.cpp:164-177) -- whose x part, for
        // CONSISTENT constraints, is the unique minimiser of the QP.  The same x comes out of the quasi-definite
        // factorization when the dependent row gets -delta on its diagonal (delta = kRegDelta x the largest constraint
        // pivot): the rows it depends on are still enforced exactly, so the constraint it states holds by itself and
        // its multiplier comes out as (rounding) / delta.  Only the FIRST failing row of an attempt is touched (pivots
        // behind a broken one are not to be trusted), up to kRegTries dependent rows per QP; the rows found in the
        // pre-solve stay regularised in the rho-KKT system.  Whether the constraints were consistent is checked on
        // the final x (epilogue): if not, the status stays NUMERICAL_ISSUE.
        if (kShared == false && factor_flag != 0 && m > 0 && reg_tries < kRegTries && isfinite(pc) && pc > 0.0) {
          double first = badp ? (double)(N8 - t) : 0.0, unused = 0.0;    // largest value = smallest failing row index
          block_reduce2<false>(first, unused, red, parity);
          const int row = N8 - (int)first;
          if (row >= n8 && row < n8 + m) {        // a constraint row (a failing variable row is a genuine breakdown)
            if (reg_delta == 0.0) reg_delta = kRegDelta * pc;
            if (t == row) reg_mine = true;
            reg_used = true;
            ++reg_tries;
            factored = false;
          }
        }
      }
      if (shared_mode != 0) {
        // shared structure: [K^{-1}]_{x,:} as an explicit operator, kept for every later QP of this CTA
        complete_inverse<kThreads>(M, NB);
        form_g<kThreads>(M, dinv, NB, NBx, NB);
        cached_pass = pass;
      }
      FCCQP_PROF(6);
      }
      }  // lazy factorization
      if (factor_flag) status_flag = 2;

        // ---- K3 right-hand side
        double acc = 0.0;
        if (pass == 0) {
          acc = rhs0;
        } else if (is_x) {
          // -(b + q_rho), q_rho = -rho (xbar - mu_x) with the cone segment overwritten (fcc_qp.cpp:81-83)
          const double w = in_cone ? (lcbar[t - lcs] - muc[t - lcs]) : (v_xbar - v_mux);
          const double q_rho = -rho_cur * w;
          acc = -(v_b + q_rho);
        } else if (is_c) {
          acc = v_b;
        }
        if (shared_mode != 0) {
          const double gx = g_apply(M, tbuf, is_row ? acc : 0.0, NB, n8);   // x = [K^{-1}]_{x,:} rhs, cached operator
          val = is_x ? gx : 0.0;
        } else {
        if (!full_inverse && pass == 1 && iter >= p.full_inverse_at) {
          // long-running QP: W = inv(L), x_base = [K^{-1} (-b; b_eq)]_x, G = [K^{-1}]_xx (see form_g)
          __syncthreads();
          complete_inverse<kThreads>(M, NB);
          v_xbase = kkt_solve_full(M, dinv, tbuf, ybuf, is_x ? -v_b : (is_c ? v_b : 0.0), NB, N8);
          __syncthreads();
          form_g<kThreads>(M, dinv, NB, NBx, NBx);
          full_inverse = true;
          FCCQP_PROF(4);
        }
        if (full_inverse) {
          // rhs_x = -b + rho w, rhs_c = b_eq  =>  x = x_base + rho G w
          const double w = is_x ? (in_cone ? (lcbar[t - lcs] - muc[t - lcs]) : (v_xbar - v_mux)) : 0.0;
          const double gw = g_apply(M, tbuf, w, NBx, n8);
          val = is_x ? fma(rho_cur, gw, v_xbase) : 0.0;
        } else {
          val = kkt_solve(M, dinv, tbuf, ybuf, acc, NB, NB32, N8);
        }
        }
        FCCQP_PROF(7);
        // val = solution component of row t (t < N8)

        }  // x-update solve

        if (pass == 0) {
          v_x = val;
          if (t < n8) xs[t] = is_x ? val : 0.0;
          __syncthreads();
          FCCQP_PROF(8);
          continue;
        }

        // ---- K4 + K5 (pass 1)
        if (is_x) { xs[t] = val; v_x = val; }
        __syncthreads();
        double rx = 0.0, rc = 0.0;
        double dz = 0.0;                     // |z_k - z_{k-1}| of this thread's entries (adaptive rho only)
        const bool relax = p.alpha != 1.0;
        if (is_x) rx = box_step<double, kAdapt>(val, p.alpha, relax, v_lb, v_ub, v_xbar, v_mux, dz);
        if (t < nc / 3) {  // lane per contact
          const int o = lcs + 3 * t;
          rc = cone_step<kAdapt>(xs[o], xs[o + 1], xs[o + 2], vmu[t], p.alpha, relax, lcbar + 3 * t, muc + 3 * t, dz);
        }
        // fmax drops NaNs, so flag them separately
        if (rx != rx || rc != rc) status_flag = 2;
        // exit test (fcc_qp.cpp:105-109) as one hardware barrier-reduction; the infinity norms
        // themselves are only needed for the iteration that ends the loop
        const int conv = __syncthreads_and((rc < p.eps_fcone) && (rx < p.eps_bound));
        FCCQP_PROF(9);
        FCCQP_PROF_COUNT(15);
        if (conv || iter + 1 == iters) {
          block_reduce2<false>(rx, rc, red, parity);
          res_x = rx; res_c = rc;
          if (conv) { n_iter = iter; break; }
        } else if (shared_mode == 1) {
          defer = true;   // iteration 0 (the identity x-update) did not pass the exit test
          break;
        } else if (kAdapt && shared_mode == 0 && p.adapt_k > 0 && (iter + 1) % p.adapt_k == 0) {
          // adaptive rho (rebalance_rho): on a change the rho-KKT matrix is assembled and factored again (the
          // lazy-factorization block at the top of the next iteration; the operator of a long-running QP with it)
          const double rho_new = cta_rebalance_rho(rx, rc, dz, rho_cur, v_mux, muc + 3 * t, t < nc / 3, red, parity);
          if (rho_new != rho_cur) {
            rho_cur = rho_new;
            factored = false;
            full_inverse = false;
          }
        }
      }
    }

    if (defer) {
      // park x0 and the index; the ADMM launch redoes iteration 0 from x0 (same arithmetic) and carries on
      if (is_x) p.x[(size_t)qp * n + t] = xs[t];
      if (tid == 0) p.pending_list[atomicAdd(p.pending_count, 1u)] = qp;
      continue;
    }
    // ---------------- K6: epilogue ----------------
    double bv, fv;
    int bad = cta_violations(is_x, v_x, v_lb, v_ub, xs, vmu, nc, lcs, red, parity, bv, fv);
    if (reg_used && is_c) {
      // rank-deficient A_eq handled through the regularised retry: the answer is the reference's only if the dependent
      // constraints were consistent, i.e. if A_eq x = b_eq still holds to rounding on the x returned
      const size_t arow = (size_t)qp * p.a_bs + (size_t)(t - n8) * p.a_rs;   // element index (float32 or float64 data)
      double ax = 0.0, mag = fabs(v_b);
      for (int j = 0; j < n; ++j) {
        const double term = ldin(p.A, arow + (size_t)j * p.a_cs) * xs[j];
        ax += term; mag += fabs(term);
      }
      if (!(fabs(ax - v_b) <= 1e-7 * mag + 1e-300)) bad = 1;
    }
    bad = __syncthreads_or(bad | (status_flag == 2));
    if (is_x) {
      p.x[(size_t)qp * n + t] = v_x;
      if (p.mu_x) p.mu_x[(size_t)qp * n + t] = v_mux;
    }
    if (p.mu_c && t < nc) p.mu_c[(size_t)qp * nc + t] = muc[t];
    if (tid == 0) store_details(p, qp, n_iter, bad, res_x, res_c, bv, fv, fact_cycles, t_start);
    FCCQP_PROF(10);
    FCCQP_PROF_COUNT(14);
  }
  FCCQP_PROF_END();
}

// ---------------------------------------------------------------------------
// WBC assembly (include/fccqp.h, fccqp_wbc_assemble): one CTA per QP writes Q, b, A_eq, b_eq from
// the robot quantities.  HBM-write bound (8 (n^2 + m n + n + m) bytes per QP, every output element
// written exactly once, coalesced); the only arithmetic is the nv x nv task Hessian Jy' W Jy and
// the gradient, formed from a shared-memory copy of Jy (lower triangle computed, mirrored, so Q is
// exactly symmetric).
// ---------------------------------------------------------------------------
struct WbcParams {
  int B, nv, nu, nh, nc, ny;
  double w_vdot, w_u, w_lc, w_eps;
  const double* M; long long M_bs;
  const double* Jh; long long Jh_bs;
  const double* Jc; long long Jc_bs;
  const double* Jy; long long Jy_bs;
  const double* W; long long W_bs;
  const double* ydd; long long ydd_bs;
  const double* bias; long long bias_bs;
  const double* gh; long long gh_bs;
  const double* gc; long long gc_bs;
  double* Q; double* b; double* A; double* beq;
};

__global__ void __launch_bounds__(256) wbc_assemble_kernel(const WbcParams p) {
  extern __shared__ __align__(16) double sm[];
  const int nv = p.nv, nu = p.nu, nh = p.nh, nc = p.nc, ny = p.ny;
  const int n = nv + nu + nh + 2 * nc, m = nv + nh + nc;
  const int o_u = nv, o_h = nv + nu, o_c = nv + nu + nh, o_e = o_c + nc;
  double* const sJ = sm;                 // [ny][nv]
  double* const sW = sm + ny * nv;       // [ny]
  double* const sH = sW + ny;            // [nv][nv] task Hessian
  for (int qp = blockIdx.x; qp < p.B; qp += gridDim.x) {
    const double* Jy = p.Jy + (size_t)qp * p.Jy_bs;
    const double* W = p.W + (size_t)qp * p.W_bs;
    const double* ydd = p.ydd + (size_t)qp * p.ydd_bs;
    const double* Mq = p.M + (size_t)qp * p.M_bs;
    const double* Jh = p.Jh + (size_t)qp * p.Jh_bs;
    const double* Jc = p.Jc + (size_t)qp * p.Jc_bs;
    double* Q = p.Q + (size_t)qp * n * n;
    double* A = p.A + (size_t)qp * m * n;
    double* b = p.b + (size_t)qp * n;
    double* beq = p.beq + (size_t)qp * m;
    __syncthreads();
    for (int e = threadIdx.x; e < ny * nv; e += blockDim.x) sJ[e] = Jy[e];
    for (int e = threadIdx.x; e < ny; e += blockDim.x) sW[e] = W[e];
    __syncthreads();
    // task Hessian, lower triangle (k ascending: the summation order of the numpy restatement)
    for (int e = threadIdx.x; e < nv * nv; e += blockDim.x) {
      const int i = e / nv, j = e - i * nv;
      if (j <= i) {
        double s = 0.0;
        for (int k = 0; k < ny; ++k) s += sJ[k * nv + i] * sW[k] * sJ[k * nv + j];
        sH[i * nv + j] = s;
        sH[j * nv + i] = s;
      }
    }
    // gradient and constraint right-hand side
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      double s = 0.0;
      if (i < nv) {
        for (int k = 0; k < ny; ++k) s += sJ[k * nv + i] * (sW[k] * ydd[k]);
        s = -s;
      }
      b[i] = s;
    }
    for (int r = threadIdx.x; r < m; r += blockDim.x)
      beq[r] = r < nv ? -p.bias[(size_t)qp * p.bias_bs + r]
                      : (r < nv + nh ? -p.gh[(size_t)qp * p.gh_bs + (r - nv)] : -p.gc[(size_t)qp * p.gc_bs + (r - nv - nh)]);
    __syncthreads();
    // Q and A_eq: one warp per matrix row, lanes along the row (no index division, coalesced stores)
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int i = wid; i < n; i += nw) {
      const double dg = i < o_u ? p.w_vdot : (i < o_h ? p.w_u : (i < o_c ? 0.0 : (i < o_e ? p.w_lc : p.w_eps)));
      double* qrow = Q + (size_t)i * n;
      const double* hrow = sH + i * nv;
      for (int j = lane; j < n; j += 32) {
        double v = (i < nv && j < nv) ? hrow[j] : 0.0;
        if (i == j) v += dg;
        qrow[j] = v;
      }
    }
    for (int r = wid; r < m; r += nw) {
      double* arow = A + (size_t)r * n;
      if (r < nv) {
        const double* mrow = Mq + r * nv;
        for (int c = lane; c < n; c += 32) {
          double v = 0.0;
          if (c < o_u) v = mrow[c];
          else if (c < o_h) v = (r - (nv - nu) == c - o_u) ? -1.0 : 0.0;       // -S, S = [0; I_nu]
          else if (c < o_c) v = -Jh[(c - o_h) * nv + r];                         // -Jh'
          else if (c < o_e) v = -Jc[(c - o_c) * nv + r];                         // -Jc'
          arow[c] = v;
        }
      } else {
        const bool hol = r < nv + nh;
        const double* jrow = hol ? Jh + (r - nv) * nv : Jc + (r - nv - nh) * nv;
        const int one = hol ? -1 : o_e + (r - nv - nh);                          // identity on the slack columns
        for (int c = lane; c < n; c += 32) arow[c] = c < o_u ? jrow[c] : (c == one ? 1.0 : 0.0);
      }
    }
  }
}

// FP64 FMA peak of this device, measured (bench.py's roofline denominator): 8 independent DFMA chains per thread,
// 4 x 256 threads per SM, no memory traffic.  2 * fmas / time is what the vector FP64 pipe (which the DMMA
// instruction shares, profiles/r01_fp64_ubench.log) can do at the clocks of the moment.
// Processing order for FCCQP_SCHEDULE_LPT: lanes whose earlier solve took >= `long_at` iterations first (from the front of
// `order`), everybody else from the back; counters zeroed by the caller.  The order inside the two groups is whatever the
// atomics give -- results do not depend on it.
__global__ void __launch_bounds__(256) lpt_order_kernel(const int* __restrict__ prev_n_iter, const int B, const int long_at,
                                                        int* __restrict__ order, unsigned int* __restrict__ n_long,
                                                        unsigned int* __restrict__ n_short) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  if (prev_n_iter[i] >= long_at) order[atomicAdd(n_long, 1u)] = i;
  else order[B - 1 - (int)atomicAdd(n_short, 1u)] = i;
}

__global__ void __launch_bounds__(256) fp64_peak_kernel(double* out, const int iters, const double seed) {
  double a[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) a[k] = seed + threadIdx.x * 1e-9 + k;
  const double m1 = 1.0 - 1e-12, c1 = 1e-13;
#pragma unroll 1
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u)
#pragma unroll
      for (int k = 0; k < 8; ++k) a[k] = fma(a[k], m1, c1);
  }
  double s = 0.0;
#pragma unroll
  for (int k = 0; k < 8; ++k) s += a[k];
  if (s == 12345.678) out[0] = s;   // never true: keeps the chains alive
}

}  // namespace fccqp
