// fccqp_struct.cuh -- structure-exploiting variant of the fused FCCQP solve (SURVEY 8f row 3).
//
// Same contract as fccqp_solve_kernel (fccqp_kernel.cuh): one CTA solves one QP at a time,
// FCCQP::Solve + GetSolution of the reference (src/fcc_qp.cpp:114-207), FP64 throughout.  What
// changes is the KKT system that gets factored.  Whole-body-control QPs are mostly made of
// variables that appear in the cost only through their own square -- torques, constraint forces,
// slacks: the rows of Q that belong to them are diagonal (fccqp.pdf eq. 10; 38-40 of the 60
// variables of the walking log) -- and the reference assembles and factors the full
// (n + m) x (n + m) matrix regardless (src/fcc_qp.cpp:141-150, 62-71).  Here every QP is classified ON
// THE DEVICE while it is staged (nothing is assumed about the layout of x, nothing is declared by
// the caller):
//
//   R   variables whose Q row has an off-diagonal entry                      -> stay in the system
//   D+  separable (diagonal-only Q row), cost q_j > 0, A_eq column with >= 2 entries
//                                                                            -> eliminated, column kept
//   D1  separable, q_j > 0, A_eq column with 0 or 1 entries (actuator selection, slack identity,
//       forces of contacts that are off)                                    -> eliminated, O(1) each
//   D0  separable, q_j = 0 (zero-cost constraint forces)                     -> trailing block
//
// With h_j = q_j (+ rho in the ADMM pass) the separable variables satisfy
//   x_j = (r_j - a_j' y) / h_j,
// and the remaining unknowns (x_R, y, x_D0) solve the REDUCED symmetric system
//
//   [ Q_RR (+rho I)   A_R'            0        ] [x_R ]   [ r_R                          ]
//   [ A_R            -C               A_D0     ] [ y  ] = [ r_y - sum_j a_j r_j / h_j    ]
//   [ 0               A_D0'           (rho I)  ] [x_D0]   [ r_D0                         ]
//
//   C = sum_{j in D+ u D1} a_j a_j' / h_j   (D1 columns only touch one diagonal entry).
//
// In this order -- positive block, negative block, zero-cost block last -- the matrix has an
// unpivoted LDL^T whenever Qbar = blkdiag(Q_RR, diag q_D) > 0 and A_eq keeps full row rank without
// the D0 columns; the pivots then come out (+, -, +).  The inertia is checked after every
// factorization and a QP that fails it (or whose structure exceeds the caps the shared-memory
// layout was sized for) is handed to the general kernel through a device-side list, never to the
// CPU.  Cassie log: 72 padded KKT rows instead of 104 (45 tiles instead of 91, 9 tile columns
// instead of 13, no sigma A'A product), humanoid 88 instead of 144, quadruped 56 instead of 88,
// multi-contact humanoid 120 instead of 192.
//
// Accuracy.  Eliminating variables whose cost is 1e-6 puts 1e6-sized terms into C; measured against
// the compiled reference on the walking log (tools/proto/struct_full_check.py, the numpy model of
// this kernel) the unpivoted reduced solve alone is within 2e-7 relative with identical iteration
// counts on all 2019 QPs, and ONE step of iterative refinement of the cold pre-solve against the
// ORIGINAL Q and A_eq (SolveParams::struct_refine, on when the caller asks for it) brings it back to 7e-11 -- the level of
// the general kernel.  The ADMM pass needs none (h_j >= rho).
#pragma once
#include "fccqp_kernel.cuh"

namespace fccqp {

enum : int { VT_R = 0, VT_DP = 1, VT_D1 = 2, VT_D0 = 3, VT_NONE = 4 };

// Per-thread view of "its" variable (thread j < n owns variable j in all vector work).
struct VarClass {
  int type, pos, krow, nnz;
  double aval, qd;
};

// Pointers into the int scratch region of StructLayout.
struct StructInts {
  int *vtype, *vpos, *rlist, *dplist, *d0list, *d1var, *rowcnt, *wtot, *nzflag, *colcnt, *colk;
};

// ---- bulk-async (TMA) staging: one thread issues ONE cp.async.bulk for a whole matrix (or as many rows of it as
// fit), completion is signalled on an mbarrier every thread then waits on.  No per-thread address
// arithmetic, no registers, nothing to unroll.
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async8_s(unsigned smem_dst, const double* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  // (generic-proxy accesses to the destination by this CTA are ordered before by the caller's __syncthreads)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "MBAR_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra MBAR_DONE_%=;\n"
      "bra MBAR_WAIT_%=;\n"
      "MBAR_DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// Classification of one QP (all threads of the CTA).  Reads ALL of Q and A_eq once (the algorithmic
// read of the path: they are inputs, every entry matters); what the assembly reads again afterwards
// comes from L1/L2.  Returns nonzero when the QP does not fit (caps) or is structurally singular
// (a zero-cost variable that no constraint touches).
//
// The matrices are STAGED into `stg` -- the tile region of the KKT matrix, idle until the assembly -- as
// many rows at a time as fit: ONE bulk-async copy (TMA, cp.async.bulk + mbarrier) per chunk when the
// matrix is a dense contiguous block, per-row cp.async otherwise; every byte is in flight at once and
// no register is held.  The staged rows are then walked column-wise: thread groups take interleaved
// rows, a thread owns a column pair (16-byte shared loads).  (Q is symmetric: column j has an
// off-diagonal entry iff row j has.)  Compact rolled loops on purpose: this runs once per QP, and
// straight-line unrolled load batches cost more in instruction fetch than they save.
struct StageCtl {
  unsigned long long* bar;   // mbarrier of the bulk copies
  unsigned phase;            // its parity (flips with every completed copy)
  bool q_bulk, a_bulk;       // dense contiguous 16-byte aligned blocks
};

// Second half of the classification, common to both front ends: the per-column findings (off-diagonal flag and
// diagonal entry of Q; entry count, row and value of the last entry of the A_eq column) become a class and a position per
// variable.  All threads of the CTA.
template <int kThreads>
__device__ __forceinline__ int struct_classify_finish(const int n, const int m8, const double* __restrict__ qd_s,
                                                      const double* __restrict__ colv, const StructInts& I, const int capR,
                                                      const int capP, const int cap0, VarClass& vc, int& nr, int& ndp, int& nd0) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kThreads / 32;
  __syncthreads();
  int type = VT_NONE, nnz = 0, kr = 0;
  double qd = 0.0, av = 0.0;
  if (tid < n) {
    nnz = I.colcnt[tid];
    if (nnz == 1) { kr = I.colk[tid]; av = colv[tid]; }
    qd = qd_s[tid];
    if (I.nzflag[tid] || !(qd >= 0.0)) type = VT_R;          // (NaN or negative curvature: leave it to the dense block)
    else if (qd < 1e-200) type = VT_D0;
    else type = nnz <= 1 ? VT_D1 : VT_DP;
    if (type == VT_D1 && nnz == 1) atomicAdd(&I.rowcnt[kr], 1);
  }
  __syncthreads();
  // two one-entry columns on the same constraint row: keep them as general columns
  if (type == VT_D1 && nnz == 1 && I.rowcnt[kr] > 1) type = VT_DP;
  const unsigned bR = __ballot_sync(0xffffffffu, type == VT_R);
  const unsigned bP = __ballot_sync(0xffffffffu, type == VT_DP);
  const unsigned b0 = __ballot_sync(0xffffffffu, type == VT_D0);
  if (lane == 0) { I.wtot[3 * warp] = __popc(bR); I.wtot[3 * warp + 1] = __popc(bP); I.wtot[3 * warp + 2] = __popc(b0); }
  __syncthreads();
  int oR = 0, oP = 0, o0 = 0;
  nr = 0; ndp = 0; nd0 = 0;
#pragma unroll
  for (int w = 0; w < kWarps; ++w) {
    const int a = I.wtot[3 * w], b = I.wtot[3 * w + 1], c = I.wtot[3 * w + 2];
    if (w < warp) { oR += a; oP += b; o0 += c; }
    nr += a; ndp += b; nd0 += c;
  }
  const unsigned lt = (1u << lane) - 1u;
  const int nr8 = (nr + 7) & ~7;
  int bad = (nr > capR || ndp + nd0 > capP || nd0 > cap0) ? 1 : 0;   // block-uniform (capP covers pass 1: D+ and D0)
  int pos = 0;
  if (!bad && tid < n) {
    if (type == VT_R) { pos = oR + __popc(bR & lt); I.rlist[pos] = tid; }
    else if (type == VT_DP) { pos = oP + __popc(bP & lt); I.dplist[pos] = tid; }
    else if (type == VT_D0) { const int q = o0 + __popc(b0 & lt); I.d0list[q] = tid; pos = nr8 + m8 + q; }
    else { pos = kr; if (nnz == 1) I.d1var[kr] = tid; }
    I.vtype[tid] = type;
    I.vpos[tid] = pos;
  }
  bad |= __syncthreads_or(type == VT_D0 && nnz == 0);
  vc.type = type; vc.pos = pos; vc.krow = kr; vc.nnz = nnz; vc.aval = av; vc.qd = qd;
  return bad;
}

template <int kThreads>
__device__ __forceinline__ int struct_classify(const int n, const int m, const int n8, const int m8,
                                               const double* __restrict__ Qg, const long long q_slow, const long long q_fast,
                                               const bool q_vec, const double* __restrict__ Ag, const long long a_rs,
                                               const long long a_cs, const bool a_vec, double* __restrict__ stg,
                                               const int stg_cap, StageCtl& sc, double* __restrict__ qd_s,
                                               double* __restrict__ colv, const StructInts& I, const int capR, const int capP,
                                               const int cap0, VarClass& vc, int& nr, int& ndp, int& nd0) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kThreads / 32;
  const int rpc = stg_cap / n;   // rows per chunk (>= 1 by construction of the layout)
  // column pairs and row groups of the scans (n even: thread -> (group, pair); n odd: thread -> column, one group)
  const bool pairs = (n & 1) == 0;
  const int npair = pairs ? (n >> 1) : n;
  const int ngrp = max(1, kThreads / npair);
  const int grp = tid / npair, cp = tid - grp * npair;
  const bool scan = grp < ngrp;
  for (int e = tid; e < m8 + 8; e += kThreads) { I.rowcnt[e] = 0; I.d1var[e] = -1; }
  for (int e = tid; e < n8; e += kThreads) { I.nzflag[e] = 0; I.colcnt[e] = 0; }
  // ---- Q: separable <=> no off-diagonal entry in column j; diagonal entry
  bool nzx = false, nzy = false;
#pragma unroll 1
  for (int row0 = 0; row0 < n; row0 += rpc) {
    const int rows = min(rpc, n - row0);
    if (sc.q_bulk) {
      if (tid == 0) bulk_g2s(stg, Qg + (size_t)row0 * n, (unsigned)(rows * n * sizeof(double)), sc.bar);
      mbar_wait(sc.bar, sc.phase);
      sc.phase ^= 1u;
    } else {
      if (q_vec) {
#pragma unroll 1
        for (int i = warp; i < rows; i += kWarps) {
          const double* src = Qg + (size_t)(row0 + i) * q_slow;
          for (int c = 2 * lane; c < n; c += 64) cp_async16(stg + i * n + c, src + c);
        }
      } else {
#pragma unroll 1
        for (int i = warp; i < rows; i += kWarps) {
          const double* src = Qg + (long long)(row0 + i) * q_slow;
          for (int c = lane; c < n; c += 32) cp_async8(stg + i * n + c, src + (long long)c * q_fast);
        }
      }
      cp_async_wait_all();
      __syncthreads();
    }
    if (scan) {
      if (pairs) {
        const int c0 = 2 * cp;
#pragma unroll 2
        for (int i = grp; i < rows; i += ngrp) {
          const double2 v = ld2(stg + i * n + c0);
          const int gi = row0 + i;
          if (gi == c0) qd_s[gi] = v.x; else nzx = nzx || (v.x != 0.0);
          if (gi == c0 + 1) qd_s[gi] = v.y; else nzy = nzy || (v.y != 0.0);
        }
      } else {
#pragma unroll 2
        for (int i = grp; i < rows; i += ngrp) {
          const double v = stg[i * n + cp];
          if (row0 + i == cp) qd_s[cp] = v; else nzx = nzx || (v != 0.0);
        }
      }
    }
    __syncthreads();
  }
  if (scan) {
    if (pairs) { if (nzx) atomicOr(&I.nzflag[2 * cp], 1); if (nzy) atomicOr(&I.nzflag[2 * cp + 1], 1); }
    else if (nzx) atomicOr(&I.nzflag[cp], 1);
  }
  // ---- A_eq: entry count of every column, and its entry if there is only one
  int cx = 0, cy = 0, kx = 0, ky = 0;
  double vx = 0.0, vy = 0.0;
#pragma unroll 1
  for (int row0 = 0; row0 < m; row0 += rpc) {
    const int rows = min(rpc, m - row0);
    if (sc.a_bulk) {
      if (tid == 0) bulk_g2s(stg, Ag + (size_t)row0 * n, (unsigned)(rows * n * sizeof(double)), sc.bar);
      mbar_wait(sc.bar, sc.phase);
      sc.phase ^= 1u;
    } else {
      if (a_vec) {
#pragma unroll 1
        for (int k = warp; k < rows; k += kWarps) {
          const double* src = Ag + (size_t)(row0 + k) * a_rs;
          for (int c = 2 * lane; c < n; c += 64) cp_async16(stg + k * n + c, src + c);
        }
      } else {
#pragma unroll 1
        for (int k = warp; k < rows; k += kWarps) {
          const double* src = Ag + (long long)(row0 + k) * a_rs;
          for (int c = lane; c < n; c += 32) cp_async8(stg + k * n + c, src + (long long)c * a_cs);
        }
      }
      cp_async_wait_all();
      __syncthreads();
    }
    if (scan) {
      if (pairs) {
#pragma unroll 2
        for (int k = grp; k < rows; k += ngrp) {
          const double2 v = ld2(stg + k * n + 2 * cp);
          if (v.x != 0.0) { ++cx; kx = row0 + k; vx = v.x; }
          if (v.y != 0.0) { ++cy; ky = row0 + k; vy = v.y; }
        }
      } else {
#pragma unroll 2
        for (int k = grp; k < rows; k += ngrp) {
          const double v = stg[k * n + cp];
          if (v != 0.0) { ++cx; kx = row0 + k; vx = v; }
        }
      }
    }
    __syncthreads();
  }
  // (several groups with entries in one column: the count says >= 2 and the entry is not used)
  if (scan) {
    const int c0 = pairs ? 2 * cp : cp;
    // (atomic exchanges: two groups may both write here -- then the count is >= 2 and nobody reads the entry)
    if (cx) {
      atomicAdd(&I.colcnt[c0], cx); atomicExch(&I.colk[c0], kx);
      atomicExch(reinterpret_cast<unsigned long long*>(colv + c0), (unsigned long long)__double_as_longlong(vx));
    }
    if (cy) {
      atomicAdd(&I.colcnt[c0 + 1], cy); atomicExch(&I.colk[c0 + 1], ky);
      atomicExch(reinterpret_cast<unsigned long long*>(colv + c0 + 1), (unsigned long long)__double_as_longlong(vy));
    }
  }
  return struct_classify_finish<kThreads>(n, m8, qd_s, colv, I, capR, capP, cap0, vc, nr, ndp, nd0);
}

// ---- coalesced row sweeps (iterative refinement) ------------------------------------------------------
// For row-major, 16-byte aligned Q and A_eq with an even number of columns (what numpy / torch callers hand
// over) a warp reads whole matrix rows with one 16-byte load per lane and column pair, kRows rows in flight.
// (A register front end built on the same sweeps -- classification and scatter straight from registers, no
// staging -- was measured against the staged one and lost: profiles/r02_front_end_ldg_vs_staged.log.)
__device__ __forceinline__ double2 ldg2(const double* p) { return __ldg(reinterpret_cast<const double2*>(p)); }
// pairs of columns per lane (lane + 32 u), rows in flight per warp: kPairs * kRows = 8 loads of 16 bytes per lane
template <int kThreads> struct FrontGeom {
  static constexpr int kPairs = (kThreads / 2 + 31) / 32;
  static constexpr int kRows = kPairs >= 4 ? 2 : (kPairs == 2 ? 4 : 8);
};

// Probe: classifies `ns` QPs spread evenly over the batch and reports the largest structure seen
// (out[0..2] = max nr, ndp, nd0; out[3] = QPs that are structurally singular) -- the host sizes the
// shared-memory layout of the solve kernel from it.
template <int kThreads>
__global__ void __launch_bounds__(kThreads) fccqp_struct_probe_kernel(const SolveParams p, const int ns, int* __restrict__ out) {
  constexpr int kStage = 3072;   // staged doubles: >= 12 rows of the widest supported matrix
  __shared__ __align__(16) double stg[kStage];
  __shared__ __align__(16) double qd_s[kThreads];
  __shared__ __align__(16) double colv[kThreads];
  __shared__ __align__(8) unsigned long long bar;
  __shared__ int ints[8 * kThreads + 2 * (kThreads + 16) + 96];
  StructInts I;
  int* q = ints;
  I.vtype = q; q += kThreads;
  I.vpos = q; q += kThreads;
  I.rlist = q; q += kThreads;
  I.dplist = q; q += kThreads;
  I.d0list = q; q += kThreads;
  I.nzflag = q; q += kThreads;
  I.colcnt = q; q += kThreads;
  I.colk = q; q += kThreads;
  I.d1var = q; q += kThreads + 16;
  I.rowcnt = q; q += kThreads + 16;
  I.wtot = q;
  const int s = blockIdx.x;
  const long long qp = ns > 1 ? (long long)s * (p.B - 1) / (ns - 1) : 0;
  const long long q_slow = p.q_cs <= p.q_rs ? p.q_rs : p.q_cs;
  const long long q_fast = p.q_cs <= p.q_rs ? p.q_cs : p.q_rs;
  const int n8 = (p.n + 7) & ~7, m8 = (p.m + 7) & ~7;
  const double* Qg = p.Q + (size_t)qp * p.q_bs;
  const double* Ag = p.A + (size_t)qp * p.a_bs;
  const bool q_vec = q_fast == 1 && (p.n & 1) == 0 && (q_slow & 1) == 0 && (reinterpret_cast<uintptr_t>(Qg) & 15) == 0;
  const bool a_vec = p.a_cs == 1 && (p.n & 1) == 0 && (p.a_rs & 1) == 0 && (reinterpret_cast<uintptr_t>(Ag) & 15) == 0;
  StageCtl sc;
  sc.bar = &bar; sc.phase = 0;
  sc.q_bulk = q_vec && q_slow == p.n;
  sc.a_bulk = a_vec && p.a_rs == p.n;
  if (threadIdx.x == 0) mbar_init(&bar, 1);
  __syncthreads();
  VarClass vc;
  int nr, ndp, nd0;
  const int bad = struct_classify<kThreads>(p.n, p.m, n8, m8, Qg, q_slow, q_fast, q_vec, Ag, p.a_rs, p.a_cs, a_vec, stg, kStage, sc,
                                            qd_s, colv, I, 1 << 30, 1 << 30, 1 << 30, vc, nr, ndp, nd0);
  if (threadIdx.x == 0) {
    atomicMax(out, nr); atomicMax(out + 1, ndp); atomicMax(out + 2, nd0);
    if (bad) atomicAdd(out + 3, 1);
  }
}

// L2 prefetch of a contiguous global range (16-byte granules inside [ptr, ptr + bytes)): one bulk-async
// instruction, no shared memory, no completion to wait for.
__device__ __forceinline__ void l2_prefetch(const void* ptr, size_t bytes) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(ptr);
  const uintptr_t lo = (a + 15) & ~(uintptr_t)15, hi = (a + bytes) & ~(uintptr_t)15;
  if (hi > lo)
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(lo), "r"((unsigned)(hi - lo)) : "memory");
}

// x-update through the reduced system.  r = this thread's entry of the full-space right-hand side
// (variable rows; the constraint rows' b_eq is in shared memory, left out when `homog`).  Returns x_j
// for variable threads.  use_op: the factors have been replaced by the explicit inverse of the
// reduced matrix (long-running QPs).  refine: one step of iterative refinement against the original
// Q and A_eq (cold pre-solve).
struct StructQP {
  int nr, nr8, ndp, dpt, nd0, NB, NB32, N8;
};

template <int kThreads>
__device__ __forceinline__ double struct_xsolve(const SolveParams& p, const StructLayout& L, double* __restrict__ smem,
                                                const StructInts& I, const StructQP& S, const VarClass& vc,
                                                const double* __restrict__ Qg, const double* __restrict__ Ag,
                                                const long long q_slow, const long long q_fast, const double r,
                                                const double hi, const double shift, const bool use_op, const bool homog,
                                                const bool refine, const bool coal
#ifdef FCCQP_DEV
                                                , unsigned long long* s_prof, long long& t_prof
#endif
                                                ) {
  const int t = threadIdx.x;
#ifdef FCCQP_DEV
  const int tid = t;   // (FCCQP_PROF)
#endif
  const int n = p.n, m = p.m;
  double* const M = smem + L.off_M;
  const double* const AP = smem + L.off_AP;
  double* const dinv = smem + L.off_dinv;
  double* const tbuf = smem + L.off_tbuf;
  double* const ybuf = smem + L.off_ybuf;
  double* const sred = smem + L.off_sred;
  double* const rf = smem + L.off_rf;
  double* const vd = smem + L.off_vd;
  double* const d1c = smem + L.off_d1c;
  const double* const beqs = smem + L.off_beq;
  const double* const qd_s = smem + L.off_qd;
  double* const xs = smem + L.off_xs;
  const bool is_x = t < n;
  const int m8 = L.m8, dptc = L.dptc;
  const int yrow = t - S.nr8;                       // constraint index of this thread's reduced row
  const bool row_R = t < S.nr, row_y = yrow >= 0 && yrow < m;
  const int zrow = t - S.nr8 - m8;
  const bool row_0 = zrow >= 0 && zrow < S.nd0;
  // ---- reduced right-hand side
  if (is_x) {
    rf[t] = r;
    if (vc.type == VT_DP) vd[vc.pos] = r * hi;
    else if (vc.type == VT_D1 && vc.nnz == 1) d1c[vc.krow] = vc.aval * (r * hi);
  }
  __syncthreads();
  double acc = 0.0;
  if (row_R) acc = rf[I.rlist[t]];
  else if (row_y) {
    const double* arow = AP + (size_t)((yrow >> 3) * dptc) * 64 + (yrow & 7) * 8;
    double s = 0.0;
#pragma unroll 1
    for (int kt = 0; kt < S.dpt; ++kt) s += row_dot8(arow + 64 * kt, (yrow & 7) >> 1, vd + 8 * kt);
    acc = (homog ? 0.0 : beqs[yrow]) - s;
    if (I.d1var[yrow] >= 0) acc -= d1c[yrow];
  } else if (row_0) acc = rf[I.d0list[zrow]];
  FCCQP_PROF(6);
  double val;
  if (use_op) val = g_apply(M, tbuf, acc, S.NB, S.N8);
  else val = kkt_solve(M, dinv, tbuf, ybuf, acc, S.NB, S.NB32, S.N8);
  FCCQP_PROF(7);
  if (t < S.N8) sred[t] = val;
  __syncthreads();
  const double* ys = sred + S.nr8;
  auto recover = [&]() -> double {
    double x = 0.0;
    if (is_x) {
      if (vc.type == VT_R || vc.type == VT_D0) x = sred[vc.pos];
      else if (vc.type == VT_DP) {
        const double* tcol = AP + (size_t)(vc.pos >> 3) * 64 + (vc.pos & 1);
        const int colc = (vc.pos & 7) >> 1;
        double s = 0.0;
#pragma unroll 1
        for (int It = 0; It < L.mt; ++It) s += col_dot8(tcol + (size_t)It * dptc * 64, colc, 0, ys + 8 * It);
        x = (r - s) * hi;
      } else {
        x = vc.nnz == 1 ? (r - vc.aval * ys[vc.krow]) * hi : r * hi;
      }
    }
    return x;
  };
  if (refine) {
    // Residual of the ORIGINAL KKT system at (x, y): it vanishes on the eliminated variables by construction,
    // so its R / constraint / D0 entries are the residual of the reduced system.  Q and A_eq come from
    // L1/L2 (this CTA read them a moment ago); threads [0, m) take the constraint rows, the others the R and D0
    // variables, kLB loads in flight each.
    constexpr int kLB = 4;
    const double x = recover();
    if (is_x) xs[t] = x;
    __syncthreads();
    double acc2 = 0.0;
    if (coal) {
      // Row-major aligned data: a warp takes whole rows (one 16-byte load per lane and column pair, kRows rows in
      // flight, L2 hits): row k of A_eq gives the constraint residual b_eq,k - a_k x (warp reduction) and, in the same
      // sweep, this warp's share of A_eq' y (per-lane column sums, combined across warps in a fixed order below);
      // row i of an R variable gives (Q x)_i (separable columns are zero in such a row).
      constexpr int kWarps = kThreads / 32;
      constexpr int kPairs = FrontGeom<kThreads>::kPairs, kRows = FrontGeom<kThreads>::kRows;
      const int lane = t & 31, warp = t >> 5;
      const int npair = n >> 1;
      double* const part = smem + L.off_part + warp * L.n8;
      double2 xv[kPairs], cs[kPairs];
#pragma unroll
      for (int u = 0; u < kPairs; ++u) {
        const int cp = lane + 32 * u;
        xv[u] = cp < npair ? ld2(xs + 2 * cp) : make_double2(0.0, 0.0);
        cs[u] = make_double2(0.0, 0.0);
      }
#pragma unroll 1
      for (int k0 = warp; k0 < m; k0 += kWarps * kRows) {
        double2 v[kRows][kPairs];
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
          const int k = k0 + r * kWarps;
#pragma unroll
          for (int u = 0; u < kPairs; ++u) {
            const int cp = lane + 32 * u;
            v[r][u] = (k < m && cp < npair) ? ldg2(Ag + (size_t)k * p.a_rs + 2 * cp) : make_double2(0.0, 0.0);
          }
        }
        double dot[kRows];
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
          const int k = k0 + r * kWarps;
          const double yk = k < m ? ys[k] : 0.0;
          double d = 0.0;
#pragma unroll
          for (int u = 0; u < kPairs; ++u) {
            d = fma(v[r][u].x, xv[u].x, d); d = fma(v[r][u].y, xv[u].y, d);
            cs[u].x = fma(v[r][u].x, yk, cs[u].x); cs[u].y = fma(v[r][u].y, yk, cs[u].y);
          }
          dot[r] = d;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
          for (int r = 0; r < kRows; ++r) dot[r] += __shfl_xor_sync(0xffffffffu, dot[r], o);
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
          const int k = k0 + r * kWarps;
          if (lane == 0 && k < m) d1c[k] = beqs[k] - dot[r];
        }
      }
#pragma unroll
      for (int u = 0; u < kPairs; ++u) {
        const int cp = lane + 32 * u;
        if (cp < npair) st2(part + 2 * cp, cs[u]);
      }
#pragma unroll 1
      for (int a0 = warp; a0 < S.nr; a0 += kWarps * kRows) {
        double2 v[kRows][kPairs];
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
          const int a = a0 + r * kWarps;
          const int i = a < S.nr ? I.rlist[a] : -1;
#pragma unroll
          for (int u = 0; u < kPairs; ++u) {
            const int cp = lane + 32 * u;
            v[r][u] = (i >= 0 && cp < npair) ? ldg2(Qg + (size_t)i * q_slow + 2 * cp) : make_double2(0.0, 0.0);
          }
        }
        double dot[kRows];
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
          double d = 0.0;
#pragma unroll
          for (int u = 0; u < kPairs; ++u) { d = fma(v[r][u].x, xv[u].x, d); d = fma(v[r][u].y, xv[u].y, d); }
          dot[r] = d;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
          for (int r = 0; r < kRows; ++r) dot[r] += __shfl_xor_sync(0xffffffffu, dot[r], o);
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
          const int a = a0 + r * kWarps;
          if (lane == 0 && a < S.nr) tbuf[a] = dot[r];
        }
      }
      __syncthreads();
      if (row_R || row_0) {
        const int j = row_R ? I.rlist[t] : I.d0list[zrow];
        double s = row_R ? fma(shift, xs[j], tbuf[t]) : (qd_s[j] + shift) * xs[j];
        const double* pp = smem + L.off_part + j;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) s += pp[w * L.n8];
        acc2 = rf[j] - s;
      } else if (row_y) acc2 = d1c[yrow];
    } else {
      if (t < m) {
        const double* arow = Ag + (long long)t * p.a_rs;
        double sa = 0.0;
#pragma unroll 1
        for (int j0 = 0; j0 < n; j0 += kLB) {
          double v[kLB];
#pragma unroll
          for (int u = 0; u < kLB; ++u) v[u] = j0 + u < n ? arow[(long long)(j0 + u) * p.a_cs] : 0.0;
#pragma unroll
          for (int u = 0; u < kLB; ++u) sa = fma(v[u], j0 + u < n ? xs[j0 + u] : 0.0, sa);
        }
        d1c[t] = beqs[t] - sa;
      } else {
        const int stride = kThreads - m > 0 ? kThreads - m : 1;
#pragma unroll 1
        for (int idx = t - m; idx < S.nr + S.nd0; idx += stride) {
          const bool isR = idx < S.nr;
          const int j = isR ? I.rlist[idx] : I.d0list[idx - S.nr];
          double s0 = (isR ? shift : qd_s[j] + shift) * xs[j], s1 = 0.0;
          if (isR) {
            const double* qcol = Qg + (long long)j * q_fast;
#pragma unroll 1
            for (int a0 = 0; a0 < S.nr; a0 += kLB) {
              double v[kLB];
#pragma unroll
              for (int u = 0; u < kLB; ++u) v[u] = a0 + u < S.nr ? qcol[(long long)I.rlist[a0 + u] * q_slow] : 0.0;
#pragma unroll
              for (int u = 0; u < kLB; ++u) s0 = fma(v[u], a0 + u < S.nr ? sred[a0 + u] : 0.0, s0);
            }
          }
          const double* acol = Ag + (long long)j * p.a_cs;
#pragma unroll 1
          for (int k0 = 0; k0 < m; k0 += kLB) {
            double v[kLB];
#pragma unroll
            for (int u = 0; u < kLB; ++u) v[u] = k0 + u < m ? acol[(long long)(k0 + u) * p.a_rs] : 0.0;
#pragma unroll
            for (int u = 0; u < kLB; ++u) s1 = fma(v[u], k0 + u < m ? ys[k0 + u] : 0.0, s1);
          }
          rf[j] -= s0 + s1;   // rf[j] held r_j
        }
      }
      __syncthreads();
      if (row_R) acc2 = rf[I.rlist[t]];
      else if (row_y) acc2 = d1c[yrow];
      else if (row_0) acc2 = rf[I.d0list[zrow]];
    }
    const double dv = kkt_solve(M, dinv, tbuf, ybuf, acc2, S.NB, S.NB32, S.N8);
    if (t < S.N8) sred[t] = val + dv;
    __syncthreads();
    FCCQP_PROF(10);
  }
  const double xr = recover();
  FCCQP_PROF(11);
  return xr;
}

// ---------------------------------------------------------------------------------------------------
// Full-space operator of long-running QPs.  Once the explicit inverse G = inv(K_red) of the reduced rho-KKT
// matrix sits in M (complete_inverse + form_g), an x-update through it still costs a right-hand-side reduction
// (A_P H^-1 r_P), the product with G, and the recovery of the eliminated variables -- five barriers.  With
//   B = A_E H_E^-1  (m x ne; E = every eliminated variable: D+, former D0 and the one-entry columns D1),
// the x-part of the solution for a right-hand side r that is zero on the constraint rows is
//   x_R = G_RR r_R - G_Ry B r_E,      x_E = H^-1 r_E - B' y = -B' G_yR r_R + (H^-1 + B' G_yy B) r_E,
// i.e. x = F r with the symmetric n x n matrix, in class order [R | E],
//   F = [[ G_RR, . ], [ X, Y ]],   X = -B' G_yR,   Y = H^-1 + B' G_yy B.
// F replaces the constraint rows of G in M (the tile rows after R), and every later x-update is
// x = x_base + F (rho w): one symmetric matrix-vector product in the space of the variables, permuted on the way in
// and out.  The products are formed OUT of place through a per-CTA scratch slab in global memory (L2-resident, used
// once per long-running QP): B, Z = G_yy B, X and Y are written there tile by tile (one output tile per warp and
// round, all operands read-only), then copied over M.  Tiles keep the chunk swizzle, so the fragment offsets of the
// factorization apply to the scratch tiles as well.
struct FullOpDims {
  int NBr, mt, dptc, dpt, ne, neT, NBF, NF;
};

template <int kThreads>
__device__ __noinline__ void build_full_op(double* __restrict__ M, const double* __restrict__ AP, const double* __restrict__ hinv,
                                           double* __restrict__ scr, const FullOpDims d, const int etype, const int epos,
                                           const int krow, const int nnz, const double aval, const double hi) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kThreads / 32;
  const int fr = lane >> 2, fq = lane & 3;
  const int fragC = (fr << 3) + (((fq ^ (fr >> 1)) & 3) << 1);
  const int fragT = ((2 * fq) << 3) + ((((fr >> 1) ^ fq) & 3) << 1) + (fr & 1);
  double* const Bs = scr;                              // [mt][neT] tiles
  double* const Zs = Bs + (size_t)d.mt * d.neT * 64;   // [mt][neT] tiles
  double* const Xs = Zs + (size_t)d.mt * d.neT * 64;   // [neT][NBr] tiles
  double* const Ys = Xs + (size_t)d.neT * d.NBr * 64;  // lower [neT][neT] tiles, (E, E') at E(E+1)/2 + E'
  double* const hE = Ys + (size_t)((d.neT * (d.neT + 1)) >> 1) * 64;   // [8 neT]: 1/h of the eliminated variables
  // ---- B = A_E H^-1 and 1/h, in class order of the eliminated variables
  for (int e = tid; e < d.mt * d.neT * 64; e += kThreads) {
    const int tile = e >> 6, off = e & 63;
    const int K = tile / d.neT, E = tile - K * d.neT;
    double v = 0.0;
    if (E < d.dpt) {
      const int r = off >> 3, c = ((((off >> 1) & 3) ^ (r >> 1)) & 3) * 2 + (off & 1);
      v = AP[(size_t)(K * d.dptc + E) * 64 + off] * hinv[8 * E + c];
    }
    Bs[e] = v;
  }
  for (int e = tid; e < 8 * d.neT; e += kThreads) hE[e] = 0.0;
  __syncthreads();
  if (etype == VT_DP || etype == VT_D1) {
    hE[epos] = hi;
    if (etype == VT_D1 && nnz == 1) Bs[(size_t)((krow >> 3) * d.neT + (epos >> 3)) * 64 + el_off(krow & 7, epos & 7)] = aval * hi;
  }
  __syncthreads();
  // ---- Z = G_yy B (G_yy symmetric, lower tiles of M at tile rows / columns NBr..) and X = -B' G_yR
  // The B / Z operands come from the global scratch slab (L2 hits, ~700 cycles each): every contraction loop below
  // loads the operands of kU steps first and multiplies afterwards, so a tile costs ceil(mt / kU) round trips, not mt.
  constexpr int kU = 4;
  const int nz = d.mt * d.neT, nx = d.neT * d.NBr;
#pragma unroll 1
  for (int w = warp; w < nz + nx; w += kWarps) {
    double2 ca = make_double2(0.0, 0.0), cb = make_double2(0.0, 0.0);
    if (w < nz) {
      const int K = w / d.neT, E = w - K * d.neT;
#pragma unroll 1
      for (int K0 = 0; K0 < d.mt; K0 += kU) {
        double b0[kU], b1[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          const double* bt = Bs + (size_t)(min(K0 + u, d.mt - 1) * d.neT + E) * 64 + fragT;
          b0[u] = bt[0]; b1[u] = bt[8];
        }
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          const int K2 = K0 + u;
          if (K2 < d.mt) {
            double2 a;
            if (K >= K2) a = ld2(M + tile_off(d.NBr + K, d.NBr + K2) + fragC);
            else { const double* gt = M + tile_off(d.NBr + K2, d.NBr + K) + fragT; a = make_double2(gt[0], gt[8]); }
            dmma(ca.x, ca.y, a.x, b0[u]);
            dmma(cb.x, cb.y, a.y, b1[u]);
          }
        }
      }
      st2(Zs + (size_t)w * 64 + fragC, make_double2(ca.x + cb.x, ca.y + cb.y));
    } else {
      const int wi = w - nz, E = wi / d.NBr, J = wi - E * d.NBr;
#pragma unroll 1
      for (int K0 = 0; K0 < d.mt; K0 += kU) {
        double a0[kU], a1[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          const double* at = Bs + (size_t)(min(K0 + u, d.mt - 1) * d.neT + E) * 64 + fragT;
          a0[u] = at[0]; a1[u] = at[8];
        }
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          const int K = K0 + u;
          if (K < d.mt) {
            const double* gt = M + tile_off(d.NBr + K, J) + fragT;
            dmma(ca.x, ca.y, a0[u], gt[0]);
            dmma(cb.x, cb.y, a1[u], gt[8]);
          }
        }
      }
      st2(Xs + (size_t)wi * 64 + fragC, make_double2(-(ca.x + cb.x), -(ca.y + cb.y)));
    }
  }
  __syncthreads();
  // ---- Y = H^-1 + B' Z (lower tiles)
  const int ny = (d.neT * (d.neT + 1)) >> 1;
#pragma unroll 1
  for (int w = warp; w < ny; w += kWarps) {
    int E = 0;
    while (((E + 1) * (E + 2)) >> 1 <= w) ++E;
    const int E2 = w - ((E * (E + 1)) >> 1);
    double2 ca = make_double2(0.0, 0.0), cb = make_double2(0.0, 0.0);
#pragma unroll 1
    for (int K0 = 0; K0 < d.mt; K0 += kU) {
      double a0[kU], a1[kU], z0[kU], z1[kU];
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const int K = min(K0 + u, d.mt - 1);
        const double* at = Bs + (size_t)(K * d.neT + E) * 64 + fragT;
        const double* zt = Zs + (size_t)(K * d.neT + E2) * 64 + fragT;
        a0[u] = at[0]; a1[u] = at[8]; z0[u] = zt[0]; z1[u] = zt[8];
      }
#pragma unroll
      for (int u = 0; u < kU; ++u)
        if (K0 + u < d.mt) {
          dmma(ca.x, ca.y, a0[u], z0[u]);
          dmma(cb.x, cb.y, a1[u], z1[u]);
        }
    }
    double2 y = make_double2(ca.x + cb.x, ca.y + cb.y);
    if (E == E2) {   // element (fr, 2 fq) and (fr, 2 fq + 1) of the tile
      if (2 * fq == fr) y.x += hE[8 * E + fr];
      if (2 * fq + 1 == fr) y.y += hE[8 * E + fr];
    }
    st2(Ys + (size_t)w * 64 + fragC, y);
  }
  __syncthreads();
  // ---- F over the constraint rows of G
#pragma unroll 1
  for (int I = d.NBr; I < d.NBF; ++I) {
    const int E = I - d.NBr;
    double* dst = M + tile_off(I, 0);
    const double* sx = Xs + (size_t)E * d.NBr * 64;
    const double* sy = Ys + (size_t)((E * (E + 1)) >> 1) * 64;
#pragma unroll 4
    for (int e = tid; e < (I + 1) * 32; e += kThreads) {
      const int j2 = e - d.NBr * 32;
      st2(dst + 2 * e, j2 < 0 ? ld2(sx + 2 * e) : ld2(sy + 2 * j2));
    }
  }
  __syncthreads();
}

// x = x_base + F (rho w): thread `t` owns variable t with class-order index ci (-1: no variable); row t of F is
// thread t's as well.  tbuf: operand, xb: x_base in class order, out: result in class order.
__device__ __noinline__ double full_op_apply(const double* __restrict__ M, double* __restrict__ tbuf, const double* __restrict__ xb,
                                             double* __restrict__ out, const int ci, const double w, const int NBF, const int NF) {
  const int t = threadIdx.x;
  if (ci >= 0) tbuf[ci] = w;
  __syncthreads();
  if (t < NF) out[t] = xb[t] + sym_row_dot(M, tbuf, NBF);
  __syncthreads();
  return ci >= 0 ? out[ci] : 0.0;
}

// ---------------------------------------------------------------------------
// The ADMM iterations of a long-running QP once the full-space operator F is in place (build_full_op), as ONE compact loop
// with its own registers: x = x_base + F (rho w), z-update, dual update, exit test (fcc_qp.cpp:81-109; the same
// arithmetic in the same order as the iteration body of the kernel -- results are bit-identical to taking these
// iterations there).  Two block barriers per iteration instead of four: the z-update stores the operand rho w of the NEXT
// product straight into the operand buffer (the contact lanes store the cone entries through cidx, variable -> class
// order), the exit-test barrier publishes it; x stays in the product's output buffer in class order and the contact lanes
// read it there.  1.3 % of the walking log's QPs and 17 % of the multi-contact set spend > 90 iterations here.
// Returns the iteration at which the loop stopped; th.conv tells whether the exit test passed there.
// ---------------------------------------------------------------------------
struct OpLoopArgs {   // buffers as OFFSETS into the dynamic shared memory (doubles): pointers rebuilt from the extern array
  int M, tbuf, xb, out, xs, lcbar, muc, vmu, ints, cidx;   // in the function are known to be shared (LDS / STS, not generic LD / ST)
  int NBF, NF, nc, lcs, iter0, iters;
  double shift, alpha, eps_fcone, eps_bound;
};
struct OpLoopThread {
  double xbar, mux, lb, ub, x, rx, rc;
  int ci, conv, nan_seen;
};

__device__ __noinline__ int full_op_loop(const OpLoopArgs& a, OpLoopThread& th, const bool is_x, const bool in_cone) {
  const int t = threadIdx.x;
  extern __shared__ __align__(16) double smem[];
  const double* const M = smem + a.M;
  double* const tbuf = smem + a.tbuf;
  double* const out = smem + a.out;
  double* const lcbar = smem + a.lcbar;
  double* const muc = smem + a.muc;
  int* const cidx = reinterpret_cast<int*>(smem + a.ints) + a.cidx;   // (cidx: offset in ints inside the int region)
  const int NBF = a.NBF;
  const bool row = t < a.NF;
  const bool contact = t < a.nc / 3;
  const bool relax = a.alpha != 1.0;
  const double shift = a.shift, alpha = a.alpha;
  const int ci = th.ci;
  double xbar = th.xbar, mux = th.mux;
  const double lb = th.lb, ub = th.ub;
  const double xbt = row ? smem[a.xb + t] : 0.0;
  const double mu_t = contact ? smem[a.vmu + t] : 0.0;
  // operand of the first product, and the class-order index of every variable for the contact lanes
  if (is_x) {
    cidx[t] = ci;
    tbuf[ci] = shift * (in_cone ? (lcbar[t - a.lcs] - muc[t - a.lcs]) : (xbar - mux));
  }
  __syncthreads();
  int c0 = 0, c1 = 0, c2 = 0;
  if (contact) { const int o = a.lcs + 3 * t; c0 = cidx[o]; c1 = cidx[o + 1]; c2 = cidx[o + 2]; }
  double val = 0.0, rx = 0.0, rc = 0.0, dz = 0.0;
  int iter = a.iter0, conv = 0, nan_seen = 0;
#pragma unroll 1
  for (;; ++iter) {
    if (row) out[t] = xbt + sym_row_dot(M, tbuf, NBF);   // row t of the symmetric F (full_op_apply)
    __syncthreads();
    rx = 0.0; rc = 0.0;
    if (is_x) {
      val = out[ci];
      rx = box_step<double, false>(val, alpha, relax, lb, ub, xbar, mux, dz);
      if (!in_cone) tbuf[ci] = shift * (xbar - mux);
    }
    if (contact) {
      double* const lcb = lcbar + 3 * t;
      double* const mc = muc + 3 * t;
      rc = cone_step<false>(out[c0], out[c1], out[c2], mu_t, alpha, relax, lcb, mc, dz);
      const double n0 = shift * (lcb[0] - mc[0]), n1 = shift * (lcb[1] - mc[1]), n2 = shift * (lcb[2] - mc[2]);
      tbuf[c0] = n0; tbuf[c1] = n1; tbuf[c2] = n2;
    }
    if (rx != rx || rc != rc) nan_seen = 1;
    conv = __syncthreads_and((rc < a.eps_fcone) && (rx < a.eps_bound));   // fcc_qp.cpp:105-109
    if (conv || iter + 1 == a.iters) break;
  }
  if (is_x) smem[a.xs + t] = val;   // the epilogue reads the cone variables from xs (behind its barrier)
  th.xbar = xbar; th.mux = mux; th.x = val; th.rx = rx; th.rc = rc; th.conv = conv; th.nan_seen = nan_seen;
  return iter;
}

// Which part of a solve an instance of fccqp_struct_kernel runs.  Cold batches large enough to fill the GPU twice over
// run in two stages (launch_struct): nearly every QP of a whole-body-control batch passes the exit test at iteration 0,
// so the first stage stops there and carries none of the code of the QPs that keep iterating (rho-KKT factorization,
// explicit inverse, full-space operator, adaptive rho); the full kernel then resumes the others.
//   kStructFull          the whole solve; with p.count_dev set (the resume launch) the QPs of that list, each from ADMM
//                        iteration 0 at the pre-solve point the first stage left in p.x (mu_x = mu_c = 0, as in any cold
//                        solve): iteration 0 is redone from the same values.  (One instance for both: a separately
//                        compiled resume instance rounds differently -- the resumed QPs would no longer be bit-identical
//                        to a single launch.)
//   kStructFirst(Refine) cold solves through the exit test of iteration 0, without (with) the refinement step of the
//                        pre-solve; a QP that needs more iterations leaves its pre-solve point in p.x and its index on
//                        p.resume_list
enum : int { kStructFull = 0, kStructFirst = 1, kStructFirstRefine = 2 };

// kAdapt: the adaptive-rho extension compiled in (a separate instance: the default path carries none of it)
template <int kThreads, int kMinBlocks, bool kAdapt, int kStage = kStructFull>
__global__ void __launch_bounds__(kThreads, kMinBlocks) fccqp_struct_kernel(const SolveParams p) {
  constexpr bool kFirst = kStage != kStructFull;
  static_assert(!(kFirst && kAdapt), "the first stage stops before adaptive rho can act");
  extern __shared__ __align__(16) double smem[];
  const StructLayout& L = p.slay;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kThreads / 32;
  const int n = p.n, m = p.m, nc = p.nc, lcs = p.lcs;
  const int n8 = L.n8, m8 = L.m8, mt = L.mt, dptc = L.dptc;

  double* const M = smem + L.off_M;
  double* const AP = smem + L.off_AP;
  double* const dinv = smem + L.off_dinv;
  double* const dneg = smem + L.off_dneg;
  double* const vd = smem + L.off_vd;
  double* const hinv = smem + L.off_hinv;
  double* const beqs = smem + L.off_beq;
  double* const qd_s = smem + L.off_qd;
  double* const xs = smem + L.off_xs;
  double* const lcbar = smem + L.off_lcbar;
  double* const muc = smem + L.off_muc;
  double* const vmu = smem + L.off_mu;
  double* const red = smem + L.off_red;
  int* const ibuf = reinterpret_cast<int*>(smem + L.off_int);
  int* const s_work = ibuf;   // [0] this QP, [1] the next one (already being prefetched into L2)
  StructInts I;
  I.vtype = ibuf + L.io_vtype; I.vpos = ibuf + L.io_vpos; I.rlist = ibuf + L.io_rlist; I.dplist = ibuf + L.io_dplist;
  I.d0list = ibuf + L.io_d0list; I.d1var = ibuf + L.io_d1var; I.rowcnt = ibuf + L.io_rowcnt; I.wtot = ibuf + L.io_wtot;
  I.nzflag = ibuf + L.io_nzflag; I.colcnt = ibuf + L.io_colcnt; I.colk = ibuf + L.io_colk;
  double* const rf = smem + L.off_rf;
  StageCtl sc;
  sc.bar = reinterpret_cast<unsigned long long*>(ibuf + 2);   // 8-byte aligned slot of the int region
  sc.phase = 0;
  if (tid == 0) mbar_init(sc.bar, 1);

  FCCQP_PROF_BEGIN(reinterpret_cast<unsigned long long*>(smem + L.off_red + 4 * 32));   // [16], the layout pads red for it
  int parity = 0;
  const int t = tid;
  const bool is_x = t < n;
  const bool in_cone = is_x && t >= lcs && t < lcs + nc;
  const int fr = lane >> 2, fq = lane & 3;
  const int fragC = (fr << 3) + (((fq ^ (fr >> 1)) & 3) << 1);
  const long long q_slow = p.q_cs <= p.q_rs ? p.q_rs : p.q_cs;
  const long long q_fast = p.q_cs <= p.q_rs ? p.q_cs : p.q_rs;
  // dense per-QP blocks can be prefetched with one bulk instruction each
  const bool q_dense = q_fast == 1 && q_slow == n;
  const bool a_dense = (p.a_cs == 1 && p.a_rs == n) || (p.a_rs == 1 && p.a_cs == m);

  // Work indices are fetched one QP ahead (thread 0 keeps the next one in a register): the atomic's round trip
  // hides behind the QP in flight, and the index is known early enough to pull that QP's data into L2.
  // (p.index_list: a processing order -- FCCQP_SCHEDULE_LPT, or the p.count_dev QPs the first stage left -- the queue
  // slot is mapped through it, one QP ahead as well; p.B: the queue is drained)
  int w_next = 0;
  if (tid == 0) {
    w_next = (int)atomicAdd(p.work_counter, 1u);
    if (!kFirst && p.count_dev && w_next >= (int)*p.count_dev) w_next = p.B;
    if (p.index_list && w_next < p.B) w_next = p.index_list[w_next];
  }
  for (;;) {
    __syncthreads();  // previous QP fully retired (smem reuse) before taking new work
    if (tid == 0) {
      s_work[0] = w_next;
      if (w_next < p.B) {
        w_next = (int)atomicAdd(p.work_counter, 1u);
        if (!kFirst && p.count_dev && w_next >= (int)*p.count_dev) w_next = p.B;
        if (p.index_list && w_next < p.B) w_next = p.index_list[w_next];
      }
    }
    __syncthreads();
    const int qp = s_work[0];
    if (qp >= p.B) break;
    const bool resume = !kFirst && p.count_dev != nullptr;
    // per-lane rho (kAdapt instances only; the first stage never reaches the rho-KKT system): as in fccqp_solve_kernel
    double rho_qp = p.rho;
    if constexpr (kAdapt) {
      if (p.rho_lanes) {
        rho_qp = p.rho_lanes[qp];
        if (!rho_valid(rho_qp)) {
          if (tid == 0) store_details(p, qp, 0, true, 0.0, 0.0, 0.0, 0.0, 0ull, clock64());
          continue;
        }
      }
    }
    const double* Qg = p.Q + (size_t)qp * p.q_bs;
    const double* Ag = p.A + (size_t)qp * p.a_bs;
    FCCQP_PROF(0);

    // ---------------- K0: vectors ----------------
    double v_b = 0.0, v_lb = 0.0, v_ub = 0.0, v_mux = 0.0, v_xbar = 0.0, v_x = 0.0;
    int finite_bounds = 0;
    if (is_x) {
      v_b = p.b[(size_t)qp * p.b_bs + t];
      v_lb = p.lb[(size_t)qp * p.lb_bs + t];
      v_ub = p.ub[(size_t)qp * p.ub_bs + t];
      if (p.warm || resume) v_x = p.x[(size_t)qp * n + t];
      if (p.warm) v_mux = p.mu_x[(size_t)qp * n + t];
    }
    if (t < m) beqs[t] = p.beq[(size_t)qp * p.beq_bs + t];
    if (t < nc / 3) vmu[t] = p.mu[(size_t)qp * p.mu_bs + t];
    if (t < nc) muc[t] = p.warm ? p.mu_c[(size_t)qp * nc + t] : 0.0;
    for (int e = t; e < L.ndp8c + 8; e += kThreads) { vd[e] = 0.0; hinv[e] = 0.0; }

    const long long t_start = clock64();
    unsigned long long fact_cycles = 0;
    int status_flag = 0;
    int n_iter = 0;
    double res_x = 0.0, res_c = 0.0;

    // ---------------- classification (reads all of Q and A_eq; the vector loads above are still in flight) ----------------
    VarClass vc;
    StructQP S;
    const bool q_vec = q_fast == 1 && (n & 1) == 0 && (q_slow & 1) == 0 && (reinterpret_cast<uintptr_t>(Qg) & 15) == 0;
    const bool a_vec = p.a_cs == 1 && (n & 1) == 0 && (p.a_rs & 1) == 0 && (reinterpret_cast<uintptr_t>(Ag) & 15) == 0;
    sc.q_bulk = q_vec && q_slow == n;
    sc.a_bulk = a_vec && p.a_rs == n;
    bool defer = struct_classify<kThreads>(n, m, n8, m8, Qg, q_slow, q_fast, q_vec, Ag, p.a_rs, p.a_cs, a_vec, M, L.stage_cap, sc,
                                           qd_s, rf, I, L.nr8c, L.ndp8c, L.nd08c, vc, S.nr, S.ndp, S.nd0) != 0;
    FCCQP_PROF(1);
    if (tid == 0 && w_next < p.B) {
      // the next QP of this CTA: start pulling its Q and A_eq into L2 (one bulk-async instruction each); by the
      // time the CTA gets to it, its stage-in reads are L2 hits
      if (q_dense) l2_prefetch(p.Q + (size_t)w_next * p.q_bs, (size_t)n * n * sizeof(double));
      if (a_dense) l2_prefetch(p.A + (size_t)w_next * p.a_bs, (size_t)m * n * sizeof(double));
    }
    S.nr8 = (S.nr + 7) & ~7;
    const int NBr = S.nr8 >> 3;
    const int yrow = t - S.nr8;
    if (is_x && (!isinf(v_lb) || !isinf(v_ub))) finite_bounds = 1;
    if (t < n8) xs[t] = v_x;
    const bool eqc = (nc == 0) && (__syncthreads_or(finite_bounds) == 0);   // fcc_qp.cpp:132-133
    const bool presolve = eqc || !p.warm;                                      // fcc_qp.cpp:159

    // pass 0: cold pre-solve (shift 0);  pass 1: ADMM (shift rho).  Same lazy scheme as the general kernel:
    // x-update 0 of a cold solve is the identity, the rho-KKT system is only factored for QPs that iterate.
    bool survive = false;   // first stage: iteration 0 did not end the solve
    for (int pass = (presolve && !resume) ? 0 : 1; pass < 2 && !defer; ++pass) {
      if (pass == 1 && eqc) break;
      if (pass == 1) {
        v_xbar = v_x;                             // fcc_qp.cpp:74-75
        if (in_cone) lcbar[t - lcs] = v_x;
        __syncthreads();
        n_iter = p.max_iter;
      }
      const int iters = pass == 0 ? 1 : p.max_iter;
      double shift = pass == 0 ? 0.0 : p.rho;   // (rho of pass 1 changes only with the adaptive-rho extension)
      if constexpr (kAdapt) shift = pass == 0 ? 0.0 : rho_qp;
      // In the ADMM pass the zero-cost variables have h = rho > 0 like everybody else: they are eliminated too
      // (keeping them as a trailing block with a rho-sized pivot costs three digits; tools/proto), so the
      // reduced system of pass 1 is [R, constraints] only.
      VarClass ve = vc;
      StructQP Se = S;
      if (pass == 1 && S.nd0 > 0) {
        if (vc.type == VT_D0) { ve.type = VT_DP; ve.pos = S.ndp + (vc.pos - S.nr8 - m8); }
        Se.ndp = S.ndp + S.nd0;
        Se.nd0 = 0;
      }
      Se.dpt = (Se.ndp + 7) >> 3;
      Se.N8 = S.nr8 + m8 + ((Se.nd0 + 7) & ~7);
      Se.NB = Se.N8 >> 3;
      Se.NB32 = (Se.N8 + 31) >> 5;
      double hi = (ve.type == VT_DP || ve.type == VT_D1) ? 1.0 / (ve.qd + shift) : 0.0;
      bool factored = false;
      bool full_inverse = false;
      bool full_op = false;          // the full-space operator F sits in M (build_full_op)
      int ci = -1, NBF = 0, NF = 0;  //   this thread's variable in class order [R | E]; tile rows / rows of F
      double v_xbase = 0.0;

#pragma unroll 1
      for (int iter = 0; iter < iters; ++iter) {
        double val = v_x;
        // (the first stage stops at iteration 0 of pass 1, whose x-update is the identity: it solves in pass 0 only)
        if (kFirst ? pass == 0 : !(pass == 1 && iter == 0 && presolve)) {
          if (!factored) {
            factored = true;
            const long long t_f0 = clock64();
            // ---------------- assemble the reduced KKT matrix (lower tiles) and the D+ columns ----------------
            {
              const int nbt = (Se.NB * (Se.NB + 1)) >> 1;
              const double2 z2 = make_double2(0.0, 0.0);
              for (int e = t; e < nbt * 32; e += kThreads) st2(M + 2 * e, z2);
              for (int e = t; e < mt * dptc * 32; e += kThreads) st2(AP + 2 * e, z2);
            }
            if (is_x) { I.vtype[t] = ve.type; I.vpos[t] = ve.pos; }
            __syncthreads();
            // Q_RR -> top-left tiles; A_eq: R columns -> constraint rows of the matrix, D0 columns -> transposed into
            // the trailing rows, D+ columns -> AP tiles (row tile I, column tile kt at (I * dptc + kt) * 64).  Second
            // read of the data (L1/L2), element-wise asynchronous copies straight to their tile positions; a lane
            // keeps the same columns (lane, lane + 32, ...) for every row, so their class and position are loop
            // invariants.  Row-major A_eq walks rows per warp, column-major A_eq (Eigen callers) columns per warp.
            {
              constexpr int kCol = kThreads / 32;
              const unsigned mS = smem_u32(M), apS = smem_u32(AP);
              // per owned column: kind (0 R, 1 D+, 2 D0, 3 nothing to copy), the 16-byte chunk it sits in (XOR-swizzled with
              // the other index below) and the row-independent part of its destination: R / D+ columns: byte offset inside a
              // tile row (tile column * 512 + (c & 1) * 8); D0 columns (stored TRANSPOSED, the variable is the row): the
              // shared address of that row.  Branch-free inner loops: lanes of one warp hold columns of every kind.
              int ckind[kCol], cps[kCol], chf[kCol];
              unsigned cof[kCol];
#pragma unroll
              for (int u = 0; u < kCol; ++u) {
                const int j = lane + 32 * u;
                const int ty = j < n ? I.vtype[j] : VT_NONE;
                const int ps = j < n ? I.vpos[j] : 0;
                ckind[u] = ty == VT_R ? 0 : (ty == VT_DP ? 1 : (ty == VT_D0 ? 2 : 3));
                cps[u] = ps;
                chf[u] = (ps & 7) >> 1;
                cof[u] = ty == VT_D0 ? mS + (unsigned)tile_off(ps >> 3, 0) * 8u + ((ps & 7) << 6)
                                     : (unsigned)(((ps >> 3) << 9) + ((ps & 1) << 3));
              }
#pragma unroll 1
              for (int a = warp; a < S.nr; a += kWarps) {
                const double* qrow = Qg + (long long)I.rlist[a] * q_slow;
                const unsigned rowS = mS + (unsigned)tile_off(a >> 3, 0) * 8u + ((a & 7) << 6);
                const int rh = (a & 7) >> 1;
#pragma unroll
                for (int u = 0; u < kCol; ++u)
                  if (ckind[u] == 0 && cps[u] <= a)
                    cp_async8_s(rowS + cof[u] + (((chf[u] ^ rh) & 3) << 4), qrow + (long long)(lane + 32 * u) * q_fast);
              }
              if (p.a_cs == 1 || p.a_rs != 1) {
#pragma unroll 1
                for (int k = warp; k < m; k += kWarps) {
                  const double* arow = Ag + (long long)k * p.a_rs;
                  const int yr = S.nr8 + k, rh = (k & 7) >> 1;
                  const unsigned rowM = mS + (unsigned)tile_off(yr >> 3, 0) * 8u + ((k & 7) << 6);
                  const unsigned rowP = apS + (unsigned)((k >> 3) * dptc) * 512u + ((k & 7) << 6);
                  const unsigned colT = (unsigned)(((yr >> 3) << 9) + ((yr & 1) << 3));   // this row as a COLUMN of a D0 row
#pragma unroll
                  for (int u = 0; u < kCol; ++u) {
                    const int kd = ckind[u];
                    const unsigned base = kd == 0 ? rowM : (kd == 1 ? rowP : colT);
                    if (kd < 3) cp_async8_s(base + cof[u] + (((chf[u] ^ rh) & 3) << 4), arow + (long long)(lane + 32 * u) * p.a_cs);
                  }
                }
              } else {
#pragma unroll 1
                for (int j = warp; j < n; j += kWarps) {
                  const int ty = I.vtype[j], ps = I.vpos[j];
                  if (ty == VT_D1) continue;
                  const double* acol = Ag + (long long)j * p.a_cs;
                  for (int k = lane; k < m; k += 32) {
                    const int yr = S.nr8 + k;
                    if (ty == VT_R) cp_async8(M + mat_off(yr, ps), acol + k);
                    else if (ty == VT_D0) cp_async8(M + mat_off(ps, yr), acol + k);
                    else cp_async8(AP + (size_t)((k >> 3) * dptc + (ps >> 3)) * 64 + el_off(k & 7, ps & 7), acol + k);
                  }
                }
              }
            }
            // decoupled unit pivots on the pads, cost of the zero-cost block, 1/h of the D+ columns
            if (t < Se.N8) {
              const bool pad = (t >= S.nr && t < S.nr8) || (yrow >= m && yrow < m8) || (t >= S.nr8 + m8 + Se.nd0);
              if (pad) M[mat_off(t, t)] = 1.0;
            }
            if (ve.type == VT_D0) M[mat_off(ve.pos, ve.pos)] = ve.qd + shift;
            if (ve.type == VT_DP) hinv[ve.pos] = hi;
            FCCQP_PROF(2);
            cp_async_wait_all();
            __syncthreads();
            FCCQP_PROF(3);
            if (t < S.nr && shift != 0.0) M[mat_off(t, t)] += shift;
            // -C on the constraint block: C_IJ = sum_kt AP_I,kt diag(1/h) AP_J,kt'  (one tile per warp and round)
            {
              const int ntile = (mt * (mt + 1)) >> 1;
#pragma unroll 1
              for (int w = warp; w < ntile; w += kWarps) {
                // (Ic, Jc) of the w-th lower tile
                int Ic = 0;
                while (((Ic + 1) * (Ic + 2)) >> 1 <= w) ++Ic;
                const int Jc = w - ((Ic * (Ic + 1)) >> 1);
                double2 ca = make_double2(0.0, 0.0), cb = make_double2(0.0, 0.0);
                const double* ai = AP + (size_t)(Ic * dptc) * 64 + fragC;
                const double* aj = AP + (size_t)(Jc * dptc) * 64 + fragC;
#pragma unroll 1
                for (int kt = 0; kt < Se.dpt; ++kt) {
                  const double2 a = ld2(ai + 64 * kt), b = ld2(aj + 64 * kt), h = ld2(hinv + 8 * kt + 2 * fq);
                  dmma(ca.x, ca.y, a.x * h.x, b.x);
                  dmma(cb.x, cb.y, a.y * h.y, b.y);
                }
                st2(M + tile_off(NBr + Ic, NBr + Jc) + fragC, make_double2(-(ca.x + cb.x), -(ca.y + cb.y)));
              }
            }
            __syncthreads();
            // one-entry columns: a^2 / h on one diagonal entry each (at most one such column per row); the pad
            // rows of the constraint block get their unit pivot back (the tile store above overwrote it)
            if (ve.type == VT_D1 && ve.nnz == 1) M[mat_off(S.nr8 + ve.krow, S.nr8 + ve.krow)] -= ve.aval * ve.aval * hi;
            if (yrow >= m && yrow < m8) M[mat_off(t, t)] = 1.0;
            __syncthreads();
            FCCQP_PROF(4);
            factor_tiles<kThreads>(M, dinv, dneg, Se.NB, Se.NB32);
            FCCQP_PROF(5);
            fact_cycles += (unsigned long long)(clock64() - t_f0);
            // inertia (+ on R and D0 rows and all pads, - on the constraint rows): anything else goes to the general kernel
            {
              // (and a constraint pivot that is rounding noise next to the others -- nearly dependent rows of A_eq --
              // goes the same way: kPivotRatio, fccqp_kernel.cuh)
              bool badp = false;
              const bool neg = yrow >= 0 && yrow < m;
              const double dn = t < Se.N8 ? dneg[t] : 0.0;
              if (t < Se.N8) badp = !isfinite(dn) || (neg ? !(dn > 0.0) : !(dn < 0.0));
              double pc = neg ? fabs(dn) : 0.0, pu = 0.0;
              block_reduce2<false>(pc, pu, red, parity);
              if (neg && fabs(dn) < kPivotRatio * pc) badp = true;
              if (__syncthreads_or(badp)) { defer = true; break; }
            }
          }  // lazy factorization

          // -(b + q_rho), q_rho = -rho (xbar - mu_x) with the cone segment overwritten (fcc_qp.cpp:81-83); w = 0 in pass 0
          const double w = (pass == 1 && is_x) ? (in_cone ? (lcbar[t - lcs] - muc[t - lcs]) : (v_xbar - v_mux)) : 0.0;
          // Long-running QP (iteration full_inverse_at): first x_base = the solve for w = 0 through the factors
          // (rep 0), then the explicit inverse of the reduced matrix; every later x-update is
          // x_base + (one symmetric product with the rho w part).  One call site: the solve is inlined once.
          const bool make_op = !kFirst && pass == 1 && !full_inverse && iter >= p.full_inverse_at;
          const bool refine = kFirst ? kStage == kStructFirstRefine : (pass == 0 && p.struct_refine != 0);
#pragma unroll 1
          for (int rep = make_op ? 0 : 1; rep < 2; ++rep) {
            const bool base_solve = rep == 0;
            if (!kFirst && !base_solve && full_op) {
              val = full_op_apply(M, smem + L.off_tbuf, smem + L.off_ybuf, smem + L.off_sred, ci, shift * w, NBF, NF);
              break;
            }
            const bool op = !kFirst && !base_solve && full_inverse;
            double r = 0.0;
            if (is_x) r = (base_solve || pass == 0) ? -v_b : (op ? shift * w : -(v_b - shift * w));
#ifdef FCCQP_DEV
            const double res = struct_xsolve<kThreads>(p, L, smem, I, Se, ve, Qg, Ag, q_slow, q_fast, r, hi, shift, op, op,
                                                       refine, q_vec && a_vec, s_prof, t_prof);
#else
            const double res = struct_xsolve<kThreads>(p, L, smem, I, Se, ve, Qg, Ag, q_slow, q_fast, r, hi, shift, op, op,
                                                       refine, q_vec && a_vec);
#endif
            if constexpr (kFirst) {
              val = res;
            } else if (base_solve) {
              v_xbase = res;
              __syncthreads();
              FCCQP_PROF(12);
              complete_inverse<kThreads>(M, Se.NB);
              FCCQP_PROF(13);
              form_g<kThreads>(M, dinv, Se.NB, Se.NB, Se.NB);
              FCCQP_PROF(15);
              full_inverse = true;
              // full-space operator (build_full_op) when it fits: rows of F <= threads and vector buffers, tiles of F
              // within the [M | AP] region (AP is not needed afterwards).  launch_struct always allocates the operator
              // scratch, so op_stride > 0 holds; the test stays because without it CUDA 12.9 spills more in the
              // <64, 8, true> instance.
              if (p.op_stride > 0) {
                FullOpDims fd;
                fd.NBr = NBr; fd.mt = mt; fd.dptc = dptc; fd.dpt = Se.dpt;
                fd.ne = n - S.nr; fd.neT = (fd.ne + 7) >> 3; fd.NBF = NBr + fd.neT; fd.NF = fd.NBF * 8;
                if (fd.NF <= kThreads && fd.NF <= L.NTc && tile_off(fd.NBF, 0) <= L.stage_cap) {
                  // class order of the eliminated variables: the D+ columns (position in AP), then the one-entry columns
                  const bool is_d1 = is_x && ve.type == VT_D1;
                  const unsigned b1 = __ballot_sync(0xffffffffu, is_d1);
                  if (lane == 0) I.wtot[warp] = __popc(b1);
                  __syncthreads();
                  int o1 = 0;
  #pragma unroll
                  for (int w2 = 0; w2 < kWarps; ++w2) if (w2 < warp) o1 += I.wtot[w2];
                  int epos = -1;
                  if (is_x && ve.type == VT_DP) epos = ve.pos;
                  else if (is_d1) epos = Se.ndp + o1 + __popc(b1 & ((1u << lane) - 1u));
                  ci = is_x ? (ve.type == VT_R ? ve.pos : S.nr8 + epos) : -1;
                  NBF = fd.NBF; NF = fd.NF;
                  build_full_op<kThreads>(M, AP, hinv, p.op_scratch + (size_t)blockIdx.x * p.op_stride, fd, is_x ? ve.type : VT_NONE,
                                          epos, ve.krow, ve.nnz, ve.aval, hi);
                  FCCQP_PROF(10);
                  double* const tb2 = smem + L.off_tbuf;
                  double* const xb2 = smem + L.off_ybuf;
                  if (t < NF) { tb2[t] = 0.0; xb2[t] = 0.0; }
                  __syncthreads();
                  if (ci >= 0) xb2[ci] = v_xbase;
                  full_op = true;   // (the barrier inside full_op_apply orders the write above)
                }
              }
            } else {
              val = op ? v_xbase + res : res;
            }
          }
        }  // x-update solve
        FCCQP_PROF(12);

        if (pass == 0) {
          v_x = val;
          if (t < n8) xs[t] = is_x ? val : 0.0;
          __syncthreads();
          continue;
        }

        // ---- K4 + K5
        if (is_x) { xs[t] = val; v_x = val; }
        __syncthreads();
        double rx = 0.0, rc = 0.0, dz = 0.0;
        const bool relax = p.alpha != 1.0;
        if (is_x) rx = box_step<double, kAdapt>(val, p.alpha, relax, v_lb, v_ub, v_xbar, v_mux, dz);
        if (t < nc / 3) {  // lane per contact
          const int o = lcs + 3 * t;
          rc = cone_step<kAdapt>(xs[o], xs[o + 1], xs[o + 2], vmu[t], p.alpha, relax, lcbar + 3 * t, muc + 3 * t, dz);
        }
        if (rx != rx || rc != rc) status_flag = 2;
        const int conv = __syncthreads_and((rc < p.eps_fcone) && (rx < p.eps_bound));   // fcc_qp.cpp:105-109
        if (conv || iter + 1 == iters) {
          block_reduce2<false>(rx, rc, red, parity);
          res_x = rx; res_c = rc;
          if (conv) { n_iter = iter; FCCQP_PROF(8); break; }
        } else if (kFirst) {
          survive = true;
          break;
        } else if (!kAdapt && kThreads > 64 && full_op) {
          // every further iteration of this QP in the compact operator loop (full_op_loop).  Not in the two-warp instance:
          // a barrier between two warps costs little, and the call cost that instance 3.5 % on the quadruped shape
          // (profiles/r02_op_loop_ab.log).
          OpLoopArgs oa;
          oa.M = (int)(M - smem); oa.tbuf = L.off_tbuf; oa.xb = L.off_ybuf; oa.out = L.off_sred; oa.xs = (int)(xs - smem);
          oa.lcbar = L.off_lcbar; oa.muc = L.off_muc; oa.vmu = L.off_mu;
          oa.ints = L.off_int; oa.cidx = L.io_colk;          // (the front end is done with colk)
          oa.NBF = NBF; oa.NF = NF; oa.nc = nc; oa.lcs = lcs; oa.iter0 = iter + 1; oa.iters = iters;
          oa.shift = shift; oa.alpha = p.alpha; oa.eps_fcone = p.eps_fcone; oa.eps_bound = p.eps_bound;
          OpLoopThread th;
          th.xbar = v_xbar; th.mux = v_mux; th.lb = v_lb; th.ub = v_ub; th.x = v_x; th.ci = ci;
          const int it_end = full_op_loop(oa, th, is_x, in_cone);
          v_xbar = th.xbar; v_mux = th.mux;
          if (is_x) v_x = th.x;
          if (th.nan_seen) status_flag = 2;
          rx = th.rx; rc = th.rc;
          block_reduce2<false>(rx, rc, red, parity);
          res_x = rx; res_c = rc;
          if (th.conv) n_iter = it_end;
          FCCQP_PROF(8);
          break;
        } else if (kAdapt && p.adapt_k > 0 && (iter + 1) % p.adapt_k == 0) {
          // adaptive rho (rebalance_rho, fccqp_kernel.cuh): on a change the reduced rho-KKT system (h = q + rho of every
          // eliminated variable included) is assembled and factored again at the top of the next iteration
          const double rho_new = cta_rebalance_rho(rx, rc, dz, shift, v_mux, muc + 3 * t, t < nc / 3, red, parity);
          if (rho_new != shift) {
            shift = rho_new;
            rho_qp = rho_new;
            hi = (ve.type == VT_DP || ve.type == VT_D1) ? 1.0 / (ve.qd + shift) : 0.0;
            factored = false; full_inverse = false; full_op = false;
          }
        }
        FCCQP_PROF(8);
      }
    }

    if (defer) {
      // not reducible within the caps / wrong inertia: the general kernel takes this QP (device-side list)
      if (tid == 0) p.pending_list[atomicAdd(p.pending_count, 1u)] = qp;
      continue;
    }
    if (kFirst && survive) {
      // the full kernel resumes this QP at iteration 0 from its pre-solve point
      if (is_x) p.x[(size_t)qp * n + t] = v_x;
      if (tid == 0) p.resume_list[atomicAdd(p.resume_count, 1u)] = qp;
      continue;
    }
    // ---------------- K6: epilogue ----------------
    double bv, fv;
    const int bad = __syncthreads_or(cta_violations(is_x, v_x, v_lb, v_ub, xs, vmu, nc, lcs, red, parity, bv, fv) |
                                     (status_flag == 2));
    if (is_x) {
      p.x[(size_t)qp * n + t] = v_x;
      if (p.mu_x) p.mu_x[(size_t)qp * n + t] = v_mux;
    }
    if (p.mu_c && t < nc) p.mu_c[(size_t)qp * nc + t] = muc[t];
    if (tid == 0) store_details(p, qp, n_iter, bad, res_x, res_c, bv, fv, fact_cycles, t_start);
    if constexpr (kAdapt) {
      if (p.rho_lanes && tid == 0) p.rho_lanes[qp] = rho_qp;
    }
    FCCQP_PROF(9);
    FCCQP_PROF_COUNT(14);
  }
  FCCQP_PROF_END();
}

}  // namespace fccqp
