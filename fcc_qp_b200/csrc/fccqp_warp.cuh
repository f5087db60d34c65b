// fccqp_warp.cuh -- one QP per WARP: the mapping for small problems (n + m <= 32).
//
// Same contract as fccqp_solve_kernel (fccqp_kernel.cuh): FCCQP::Solve + GetSolution of the reference
// (src/fcc_qp.cpp:114-207) per QP, FP64 throughout, same pre-solve (augmented-Lagrangian quasi-definite KKT matrix,
// unpivoted LDL^T), same lazy rho-KKT factorization, same order of operations in the z-update / residuals / duals /
// exit test.  What changes is the mapping: a CTA-per-QP kernel spends a 5-variable QP's time in block-wide barriers
// and 8x8-tile bookkeeping for a matrix that is smaller than one tile row.  Here lane i of a warp owns row i of the
// (n + m) x (n + m) KKT matrix and every per-row scalar (bounds, duals, right-hand side, pivot) in registers; the matrix
// itself sits in shared memory, one private slab per warp with an odd row stride (row-per-lane and column-per-lane
// accesses are both conflict-free, reads of the pivot row are broadcasts); lanes talk through shuffles; nothing but
// __syncwarp orders anything, so the warps of a CTA -- and of an SM -- run fully decoupled, each pulling QPs from the
// work counter on its own.
//
//   factorization   right-looking LDL^T on the full symmetric square: step k scales column k below the pivot and
//                   updates rows k+1.. with the (untouched) pivot row -- no divergence, (N-k) fused multiply-adds per lane
//   solves          forward / backward substitution, one shuffle broadcast per step
//   long-running    after SolveParams::full_inverse_at iterations the x-block of the inverse, G = [K^-1]_xx, replaces the
//   QPs             factors (n solves for unit vectors, lanes keep one ROW of G each): every later x-update is
//                   x = x_base + rho G (x_bar - mu), n shuffle-broadcast multiply-adds with no dependent chain
//
// The kernel is a template over the scalar type T.  T = double is the contract above.  T = float is the FP32 ARITHMETIC mode
// (FCCQP_PRECISION_FP32, include/fccqp.h): float32 problem data, KKT matrix, factorization, solves, projections, duals and
// residuals all in float (one shuffle per broadcast instead of two, MUFU-based division / square root in the cone projection,
// half the shared memory per warp); warm state and outputs stay the caller's double arrays, converted at the boundary.  Its
// results carry the stated FP32 bound of the header, not the 1e-6 of FP64 mode.
#pragma once
#include "fccqp_kernel.cuh"

namespace fccqp {

constexpr unsigned kFullMask = 0xffffffffu;
template <typename T> __device__ __forceinline__ T shfl_t(T v, int src) { return __shfl_sync(kFullMask, v, src); }
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// the float twin of project_cone3 (fccqp_kernel.cuh; constraint_utils.cpp:5-25) -- same branches, same order
__device__ __forceinline__ void project_cone3(float f0, float f1, float f2, float mu, float& o0, float& o1, float& o2) {
  const float r = sqrtf(f0 * f0 + f1 * f1);
  if (mu * f2 >= r) { o0 = f0; o1 = f1; o2 = f2; return; }
  if (f2 < -mu * r) { o0 = 0.0f; o1 = 0.0f; o2 = 0.0f; return; }
  const float ratio = mu * f2 / r;
  float r0 = ratio * f0, r1 = ratio * f1, r2 = f2;
  const float sq = r0 * r0 + r1 * r1 + r2 * r2;
  if (sq > 0.0f) { const float nr = rsqrtf(sq); r0 *= nr; r1 *= nr; r2 *= nr; }
  const float d = r0 * f0 + r1 * f1 + r2 * f2;
  o0 = d * r0; o1 = d * r1; o2 = d * r2;
}
// working-precision constants of the pivot tests (fccqp_kernel.cuh: kPivotRatio, kRegDelta) and of the consistency check
template <typename T> struct WarpTol;
template <> struct WarpTol<double> {
  static constexpr double pivot_ratio = kPivotRatio, reg_delta = kRegDelta, incons = 1e-7, tiny = 1e-300;
};
template <> struct WarpTol<float> {
  static constexpr float pivot_ratio = 2e-6f, reg_delta = 1e-4f, incons = 1e-3f, tiny = 1e-30f;
};

// LDL^T of the N x N symmetric matrix in K (row stride ld), in place: strictly-lower part = L, diagonal = D.
template <typename T>
__device__ __forceinline__ void warp_ldlt(T* __restrict__ K, const int N, const int ld, const int lane) {
  T* const Krow = K + lane * ld;
#pragma unroll 1
  for (int k = 0; k + 1 < N; ++k) {
    const T* const prow = K + k * ld;
    const T rk = T(1.0) / prow[k];
    if (lane > k && lane < N) {
      const T l = Krow[k] * rk;
#pragma unroll 4
      for (int j = k + 1; j < N; ++j) Krow[j] = fma(-l, prow[j], Krow[j]);
      Krow[k] = l;
    }
    __syncwarp();
  }
}

// x = K^-1 rhs with the factors of warp_ldlt; lane i holds rhs_i / returns x_i (lanes >= N: 0).
// (Not inlined: called from three places, 32 times over when the inverse of a long-running QP is formed.)
template <typename T>
__device__ __noinline__ T warp_solve(const T* __restrict__ K, const int N, const int ld, const int lane, const T dinv, T y) {
  const T* const Krow = K + lane * ld;
#pragma unroll 4
  for (int k = 0; k + 1 < N; ++k) {
    const T yk = shfl_t(y, k);
    if (lane > k && lane < N) y = fma(-Krow[k], yk, y);
  }
  y *= dinv;
#pragma unroll 4
  for (int k = N - 1; k > 0; --k) {
    const T xk = shfl_t(y, k);
    if (lane < k) y = fma(-K[k * ld + lane], xk, y);
  }
  return y;
}

// kRhoLanes: the per-lane rho of SolveParams::rho_lanes compiled in (a separate instance: the default path carries none of it)
template <int kWarps, int kMinBlocks, typename T, bool kRhoLanes = false>
__global__ void __launch_bounds__(32 * kWarps, kMinBlocks) fccqp_warp_kernel(const SolveParams p) {
  extern __shared__ __align__(16) double smem_d[];
  T* const smem = reinterpret_cast<T*>(smem_d);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n = p.n, m = p.m, nc = p.nc, lcs = p.lcs, N = n + m;
  const int ld = N | 1;
  T* const K = smem + (size_t)warp * (size_t)(N * ld);
  T* const Krow = K + (lane < N ? lane : 0) * ld;
  const bool is_x = lane < n, is_c = lane >= n && lane < N;
  const bool in_cone = is_x && lane >= lcs && lane < lcs + nc;
  const int ck = in_cone ? (lane - lcs) % 3 : 0;     // component inside the contact triple
  const int cbase = in_cone ? lane - ck : 0;         // first lane of the triple
  const long long q_slow = p.q_cs <= p.q_rs ? p.q_rs : p.q_cs;
  const long long q_fast = p.q_cs <= p.q_rs ? p.q_cs : p.q_rs;

  for (;;) {
    int qp = 0;
    if (lane == 0) {
      qp = (int)atomicAdd(p.work_counter, 1u);
      if (p.index_list && qp < p.B) qp = p.index_list[qp];    // processing order (FCCQP_SCHEDULE_LPT)
    }
    qp = __shfl_sync(kFullMask, qp, 0);
    if (qp >= p.B) break;
    const long long t_start = clock64();
    // (T = float: float32 arrays behind the double-typed pointers of SolveParams, strides in elements)
    const T* Qg = reinterpret_cast<const T*>(p.Q) + (size_t)qp * p.q_bs;
    const T* Ag = reinterpret_cast<const T*>(p.A) + (size_t)qp * p.a_bs;
    const T* const bg = reinterpret_cast<const T*>(p.b), *const beqg = reinterpret_cast<const T*>(p.beq);
    const T* const lbg = reinterpret_cast<const T*>(p.lb), *const ubg = reinterpret_cast<const T*>(p.ub);
    const T* const mug = reinterpret_cast<const T*>(p.mu);
    const T rho0 = (T)p.rho, alpha = (T)p.alpha, eps_fcone = (T)p.eps_fcone, eps_bound = (T)p.eps_bound;
    // per-lane rho: an entry the solve cannot take ends the lane here with NUMERICAL_ISSUE, its state and the entry
    // untouched (fccqp_solve_kernel); the others start pass 1 below, converted to T at the boundary
    if constexpr (kRhoLanes) {
      if (!rho_valid(p.rho_lanes[qp])) {
        if (lane == 0) store_details(p, qp, 0, true, T(0), T(0), T(0), T(0), 0ull, t_start);
        continue;
      }
    }

    // ---------------- vectors: one register per row and vector ----------------
    T v_b = 0, v_lb = 0, v_ub = 0, v_mux = 0, v_xbar = 0, v_x = 0;
    T v_muc = 0, v_lcbar = 0, v_fric = 0;
    int finite_bounds = 0;
    if (is_x) {
      v_b = bg[(size_t)qp * p.b_bs + lane];
      v_lb = lbg[(size_t)qp * p.lb_bs + lane];
      v_ub = ubg[(size_t)qp * p.ub_bs + lane];
      if (p.warm) { v_x = (T)p.x[(size_t)qp * n + lane]; v_mux = (T)p.mu_x[(size_t)qp * n + lane]; }
      if (!isinf(v_lb) || !isinf(v_ub)) finite_bounds = 1;
    } else if (is_c) {
      v_b = beqg[(size_t)qp * p.beq_bs + (lane - n)];
    }
    if (in_cone) {
      v_fric = mug[(size_t)qp * p.mu_bs + (lane - lcs) / 3];
      if (p.warm) v_muc = (T)p.mu_c[(size_t)qp * nc + (lane - lcs)];
    }
    const bool eqc = (nc == 0) && !__any_sync(kFullMask, finite_bounds);   // fcc_qp.cpp:132-133
    const bool presolve = eqc || !p.warm;                                  // fcc_qp.cpp:159

    int status_flag = 0, n_iter = 0;
    bool reg_used = false, reg_mine = false;   // regularised retry for dependent constraint rows (fccqp_kernel.cuh)
    T reg_delta = 0;
    int reg_tries = 0;
    T res_x = 0, res_c = 0;
    unsigned long long fact_cycles = 0;

    for (int pass = presolve ? 0 : 1; pass < 2; ++pass) {
      if (pass == 1 && eqc) break;
      if (pass == 1) {
        v_xbar = v_x;            // fcc_qp.cpp:74-75
        v_lcbar = v_x;
        n_iter = p.max_iter;
      }
      const int iters = pass == 0 ? 1 : p.max_iter;
      bool factored = false, have_g = false;
      T dinv = 0, rhs0 = 0, v_xbase = 0;
      T rho_cur = rho0;   // (changes only with the adaptive-rho extension)
      if constexpr (kRhoLanes) rho_cur = (T)p.rho_lanes[qp];

#pragma unroll 1
      for (int iter = 0; iter < iters; ++iter) {
        T val = v_x;
        // x-update 0 of a cold solve is the identity (x_bar = x0, zero duals; fccqp_kernel.cuh): the rho-KKT system is
        // only factored for QPs that go on iterating
        if (!(pass == 1 && iter == 0 && presolve)) {
          while (!factored) {
            factored = true;
            const long long t_f0 = clock64();
            __syncwarp();
            // ---- assemble [[Q (+ rho I), A'], [A, 0]]: coalesced rows of Q and A_eq, A_eq also transposed
#pragma unroll 2
            for (int i = 0; i < n; ++i)
              if (is_x) K[i * ld + lane] = Qg[(long long)i * q_slow + (long long)lane * q_fast];
#pragma unroll 2
            for (int r = 0; r < m; ++r) {
              if (is_x) {
                const T a = Ag[(long long)r * p.a_rs + (long long)lane * p.a_cs];
                K[(n + r) * ld + lane] = a;
                Krow[n + r] = a;
              } else if (is_c) {
                K[(n + r) * ld + lane] = 0;
              }
            }
            __syncwarp();
            if (reg_mine) Krow[lane] = -reg_delta;
            if (pass == 1) {
              if (is_x) Krow[lane] += rho_cur;
            } else {
              // sigma = trace(Q) / ||A||_F^2 balances the two terms of Q + sigma A'A (fccqp_kernel.cuh, pre-solve)
              T trq = is_x ? Krow[lane] : T(0), fro = 0;
              if (is_c)
                for (int j = 0; j < n; ++j) fro = fma(Krow[j], Krow[j], fro);
              trq = warp_sum(trq); fro = warp_sum(fro);
              const T sigma = (trq > 0 && fro > 0 && isfinite(trq / fro)) ? trq / fro : T(1);
              // rhs_x = -b + sigma A' b_eq, rhs_c = b_eq; Q += sigma A'A
              T s = 0;
              for (int r = 0; r < m; ++r) {
                const T br = shfl_t(v_b, n + r);
                if (is_x) s = fma(Krow[n + r], br, s);
              }
              rhs0 = is_x ? fma(sigma, s, -v_b) : (is_c ? v_b : T(0));
              if (is_x) {
#pragma unroll 1
                for (int j = 0; j < n; ++j) {
                  const T* cj = K + j * ld + n;      // column j of A_eq = row j of the transposed copy (broadcast)
                  T t = 0;
                  for (int r = 0; r < m; ++r) t = fma(Krow[n + r], cj[r], t);
                  Krow[j] = fma(sigma, t, Krow[j]);
                }
              }
            }
            __syncwarp();
            warp_ldlt<T>(K, N, ld, lane);
            const T d = lane < N ? Krow[lane] : T(1);
            dinv = T(1) / d;
            {
              // inertia (+ on the variable rows, - on the constraint rows) and pivot size (kPivotRatio), as in the
              // CTA kernels: anything else is FCCQP_STATUS_NUMERICAL_ISSUE
              bool badp = lane < N && (!isfinite(d) || (is_c ? !(d < 0) : !(d > 0)));
              const T pa = warp_max((is_x && pass == 0) ? fabs(d) : T(0)), pc = warp_max(is_c ? fabs(d) : T(0));
              if (lane < N && fabs(d) < WarpTol<T>::pivot_ratio * (is_c ? pc : pa)) badp = true;
              const unsigned fmask = __ballot_sync(kFullMask, badp);
              const int row = fmask ? __ffs(fmask) - 1 : -1;       // first failing row
              if (fmask && row >= n && row < N && reg_tries < kRegTries && isfinite(pc) && pc > 0) {
                // a dependent constraint row: -delta on its diagonal and one more attempt (fccqp_kernel.cuh)
                if (reg_delta == 0) reg_delta = WarpTol<T>::reg_delta * pc;
                if (lane == row) reg_mine = true;
                reg_used = true;
                ++reg_tries;
                factored = false;
              } else if (fmask) {
                status_flag = 2;
              }
            }
            fact_cycles += (unsigned long long)(clock64() - t_f0);
          }

          const T w = (pass == 1 && is_x) ? (in_cone ? (v_lcbar - v_muc) : (v_xbar - v_mux)) : T(0);
          if (pass == 1 && !have_g && iter >= p.full_inverse_at) {
            // long-running QP: x_base = [K^-1 (-b; b_eq)]_x, then G = [K^-1]_xx column by column (one solve per unit
            // vector; lane i keeps G[i][c], which is G[c][i]).  The solves read all of L, so G cannot be built in
            // place: it is collected in registers (n <= 32 columns) and written over the factors afterwards.
            v_xbase = warp_solve<T>(K, N, ld, lane, dinv, is_x ? -v_b : (is_c ? v_b : T(0)));
            T g[32];
#pragma unroll
            for (int c = 0; c < 32; ++c) g[c] = 0;
#pragma unroll
            for (int c = 0; c < 32; ++c)
              if (c < n) g[c] = warp_solve<T>(K, N, ld, lane, dinv, lane == c ? T(1) : T(0));   // column c of K^-1; keeps G[lane][c]
            __syncwarp();
#pragma unroll
            for (int c = 0; c < 32; ++c)
              if (c < n && is_x) Krow[c] = g[c];
            __syncwarp();
            have_g = true;
          }
          if (have_g) {
            // x = x_base + rho G w
            T s0 = 0, s1 = 0;
            int c = 0;
#pragma unroll 2
            for (; c + 1 < n; c += 2) {
              s0 = fma(Krow[c], shfl_t(w, c), s0);
              s1 = fma(Krow[c + 1], shfl_t(w, c + 1), s1);
            }
            if (c < n) s0 = fma(Krow[c], shfl_t(w, c), s0);
            val = is_x ? fma(rho_cur, s0 + s1, v_xbase) : T(0);
          } else {
            // -(b + q_rho), q_rho = -rho (xbar - mu_x) with the cone segment overwritten (fcc_qp.cpp:81-83)
            const T acc = pass == 0 ? rhs0 : (is_x ? -(v_b - rho_cur * w) : (is_c ? v_b : T(0)));
            val = warp_solve<T>(K, N, ld, lane, dinv, acc);
            if (!is_x) val = 0;
          }
        }

        if (pass == 0) {
          v_x = val;
          continue;
        }

        // ---- z-update, residuals, duals (fcc_qp.cpp:88-103), exit test (:105-109)
        v_x = val;
        T rx = 0, rc = 0, dz = 0;
        const bool relax = alpha != T(1);
        if (is_x) rx = box_step<T, true>(val, alpha, relax, v_lb, v_ub, v_xbar, v_mux, dz);
        {
          // every lane of a contact triple projects the whole triple and keeps its own component
          const T xk = relax ? fma(alpha, val, (T(1) - alpha) * v_lcbar) : val;
          const T fk = xk + v_muc;
          const T f0 = shfl_t(fk, cbase), f1 = shfl_t(fk, cbase + 1), f2 = shfl_t(fk, cbase + 2);
          if (in_cone) {
            T o0, o1, o2;
            project_cone3(f0, f1, f2, v_fric, o0, o1, o2);
            const T o = ck == 0 ? o0 : (ck == 1 ? o1 : o2);
            dz = fmax(dz, fabs(o - v_lcbar));
            v_lcbar = o;
            const T r = xk - o;
            v_muc += r;
            rc = fabs(r);
          }
        }
        if (rx != rx || rc != rc) status_flag = 2;   // (ballot below: any lane)
        const bool conv = __all_sync(kFullMask, (rc < eps_fcone) && (rx < eps_bound));
        if (conv || iter + 1 == iters) {
          res_x = warp_max(rx); res_c = warp_max(rc);
          if (conv) { n_iter = iter; break; }
        } else if (p.adapt_k > 0 && (iter + 1) % p.adapt_k == 0) {
          // adaptive rho (rebalance_rho, fccqp_kernel.cuh)
          const T rho_new = rebalance_rho(warp_max(fmax(rx, rc)), warp_max(dz), rho_cur);
          if (rho_new != rho_cur) {
            const T sc = rho_cur / rho_new;
            v_mux *= sc; v_muc *= sc;
            rho_cur = rho_new;
            // (the lane's entry follows each move, so it ends with the final rho; an entry that never moves is not
            // written, which T = float would round)
            if constexpr (kRhoLanes) { if (lane == 0) p.rho_lanes[qp] = (double)rho_new; }
            factored = false;
            have_g = false;
          }
        }
      }
    }

    // ---------------- epilogue: violations (constraint_utils.cpp:48-65), outputs ----------------
    T bv = 0, fv = 0;
    if (is_x) { const T d = v_x - clampd(v_x, v_lb, v_ub); bv = d * d; }
    {
      const T x1 = shfl_t(v_x, cbase + 1), x2 = shfl_t(v_x, cbase + 2);
      if (in_cone && ck == 0) {
        const T r = sqrt(v_x * v_x + x1 * x1) - v_fric * x2;
        fv = r > 0 ? r : T(0);
      }
    }
    bv = warp_sum(bv); fv = warp_sum(fv);
    bool incons = false;
    if (reg_used) {
      // regularised retry taken: the answer is the reference's only if A_eq x = b_eq still holds (consistent dependent rows)
      T ax = 0, mag = fabs(v_b);
      for (int j = 0; j < n; ++j) {
        const T xj = shfl_t(v_x, j);
        if (is_c) { const T term = Ag[(long long)(lane - n) * p.a_rs + (long long)j * p.a_cs] * xj; ax += term; mag += fabs(term); }
      }
      incons = is_c && !(fabs(ax - v_b) <= WarpTol<T>::incons * mag + WarpTol<T>::tiny);
    }
    const bool bad = __any_sync(kFullMask, (is_x && !isfinite(v_x)) || status_flag == 2 || incons);
    if (is_x) {
      p.x[(size_t)qp * n + lane] = (double)v_x;
      if (p.mu_x) p.mu_x[(size_t)qp * n + lane] = (double)v_mux;
    }
    if (p.mu_c && in_cone) p.mu_c[(size_t)qp * nc + (lane - lcs)] = (double)v_muc;
    if (lane == 0) store_details(p, qp, n_iter, bad, res_x, res_c, bv, fv, fact_cycles, t_start);
  }
}

}  // namespace fccqp
