// fccqp_capi.cu -- host side of libfccqp_b200.so: the C ABI declared in
// include/fccqp.h over the sm_100a kernels in fccqp_kernel.cuh.
//
// No CPU fallback: every entry point that computes needs a CUDA device and
// returns FCCQP_E_CUDA otherwise.
#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "../../include/fccqp.h"
#include "fccqp_kernel.cuh"
#include "fccqp_struct.cuh"
#include "fccqp_warp.cuh"
#include "fccqp_polish.cuh"

namespace {

thread_local std::string g_err;
std::atomic<long long> g_launches{0};
struct LaunchInfo { int grid = 0, block = 0, smem = 0, ctas_per_sm = 0; };
LaunchInfo g_last_launch;
// what the last batch launch did about problem structure (fccqp_last_struct_info)
struct StructInfo { int used = 0, nr = 0, ndp = 0, nd0 = 0, rows = 0, rows_dense = 0, device = 0; };
StructInfo g_last_struct;
std::mutex g_info_mu;

// How launch_solve decides about the structure-exploiting kernel (fccqp_batch_desc::structure).
struct StructHint {
  int mode = FCCQP_STRUCTURE_AUTO;   // AUTO: probe on the device (one tiny kernel + a stream sync); DENSE: never; CAPS: given
  int caps[3] = {0, 0, 0};           // nr, ndp, nd0
  int refine = 0;                    // FCCQP_STRUCTURE_REFINE: one step of iterative refinement on the reduced cold pre-solve
  int lpt = 0;                       // FCCQP_SCHEDULE_LPT: p.n_iter holds earlier iteration counts; long lanes first
  void set(int structure) {
    mode = structure & ~(FCCQP_STRUCTURE_REFINE | FCCQP_SCHEDULE_LPT);
    refine = (structure & FCCQP_STRUCTURE_REFINE) != 0;
    lpt = (structure & FCCQP_SCHEDULE_LPT) != 0;
  }
};

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                       \
  do {                                                                                       \
    cudaError_t e__ = (expr);                                                                \
    if (e__ != cudaSuccess)                                                                  \
      return fail(FCCQP_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__),     \
                  __FILE__, __LINE__);                                                       \
  } while (0)

// Per-device context: properties, work counters, global scratch, host-path staging.
struct DeviceCtx {
  int device = -1;
  int num_sms = 0;
  int max_smem_optin = 0;
  int clock_khz = 0;
  // host-path staging (grow only)
  char* stage = nullptr;
  size_t stage_bytes = 0;
  cudaStream_t streams[3] = {nullptr, nullptr, nullptr};
  // pinned bounce buffer for outputs whose destination is pageable host memory (grow only)
  char* hstage = nullptr;
  size_t hstage_bytes = 0;
  cudaEvent_t chunk_ev[16] = {};
  unsigned int* h_deferred = nullptr;   // pinned [2]: QPs the structure-exploiting kernel handed to the general one in
                                        // the last structure call, per lane set
  int* h_probe = nullptr;               // pinned [4]: result of the structure probe
  std::mutex mu;       // guards counters / gscratch / occupancy cache
  std::mutex host_mu;  // serialises FCCQP_MEM_HOST calls (they share the staging buffer)
  std::map<std::pair<const void*, size_t>, int> occupancy;  // (kernel, smem) -> CTAs/SM
};

std::mutex g_ctx_mu;
std::map<int, std::unique_ptr<DeviceCtx>> g_ctx;

int get_ctx(int device, DeviceCtx** out) {
  std::lock_guard<std::mutex> lk(g_ctx_mu);
  auto it = g_ctx.find(device);
  if (it != g_ctx.end()) { *out = it->second.get(); return FCCQP_OK; }
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(FCCQP_E_CUDA, "no usable CUDA device (%s); this library has no CPU fallback",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  if (device < 0 || device >= count) return fail(FCCQP_E_INVALID, "device %d out of range [0,%d)", device, count);
  CUDA_TRY(cudaSetDevice(device));
  auto ctx = std::make_unique<DeviceCtx>();
  ctx->device = device;
  CUDA_TRY(cudaDeviceGetAttribute(&ctx->num_sms, cudaDevAttrMultiProcessorCount, device));
  CUDA_TRY(cudaDeviceGetAttribute(&ctx->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  CUDA_TRY(cudaDeviceGetAttribute(&ctx->clock_khz, cudaDevAttrClockRate, device));
  {
    // stream-ordered scratch (cudaMallocAsync in the shared-structure path) stays in the pool across
    // synchronisation points instead of going back to the OS after every call
    cudaMemPool_t pool = nullptr;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess && pool) {
      unsigned long long keep = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
  }
  for (auto& s : ctx->streams) CUDA_TRY(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  for (auto& e : ctx->chunk_ev) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  CUDA_TRY(cudaMallocHost(&ctx->h_deferred, 2 * sizeof(unsigned int)));
  ctx->h_deferred[0] = ctx->h_deferred[1] = 0;
  CUDA_TRY(cudaMallocHost(&ctx->h_probe, 4 * sizeof(int)));
  *out = ctx.get();
  g_ctx[device] = std::move(ctx);
  return FCCQP_OK;
}

using KernelFn = void (*)(const fccqp::SolveParams);

// Developer switches, read from the environment once per process: tests and tools/ compare kernel paths with them.
struct DevSwitches {
  bool no_warp = false;     // FCCQP_NO_WARP: FP64 problems with n + m <= 32 take the CTA-per-QP kernels
  bool no_shared = false;   // FCCQP_NO_SHARED: shared-structure batches take the structure-exploiting / general kernels
  int full_inverse_at = 0;  // FCCQP_FULL_INVERSE_AT (>= 1): ADMM iteration from which long-running QPs use the completed
                            // inverse of L; 0 = unset: 8 for n + m <= 32 (tuned on the warp kernel), 6 above
                            // (8 until the compact operator loop; sweep: profiles/r02_full_inverse_at_sweep.log)
  int cta_cap = 0;          // FCCQP_CTAS_PER_SM: at most this many CTAs per SM (0: as many as fit)
#ifdef FCCQP_DEV
  bool profile = false;     // FCCQP_PROFILE: phase cycle counters of the structure-exploiting and general kernels
#endif
};

const DevSwitches& dev_switches() {
  static const DevSwitches s = [] {
    DevSwitches d;
    d.no_warp = getenv("FCCQP_NO_WARP") != nullptr;
    d.no_shared = getenv("FCCQP_NO_SHARED") != nullptr;
    if (const char* v = getenv("FCCQP_FULL_INVERSE_AT")) d.full_inverse_at = atoi(v) < 1 ? 1 : atoi(v);
    if (const char* v = getenv("FCCQP_CTAS_PER_SM")) d.cta_cap = atoi(v);
#ifdef FCCQP_DEV
    d.profile = getenv("FCCQP_PROFILE") != nullptr;
#endif
    return d;
  }();
  return s;
}

// Whether the CTA-per-QP kernels take the shape: one thread per padded KKT row, at most 256 rows, the packed matrix in
// shared memory.  The shared memory binds first: on a B200 (227 KB) padded n + m <= 224 when m <= n.
int check_shape(const DeviceCtx& ctx, int n, int m, int nc) {
  const int N = n + m;
  if (N < 1) return fail(FCCQP_E_INVALID, "n + m must be >= 1");
  const fccqp::Layout l(n, m, nc);
  if (l.N8 > 256 || l.bytes() > (size_t)ctx.max_smem_optin)
    return fail(FCCQP_E_UNSUPPORTED,
                "n + m = %d (padded %d) needs %zu B of shared memory per QP, the device allows %d B (a B200 takes "
                "padded n + m <= 224 when m <= n): too large for the shared-memory-resident kernels", N, l.N8, l.bytes(),
                ctx.max_smem_optin);
  return FCCQP_OK;
}

// CTA-per-QP kernel instances (fccqp_kernel.cuh): 4 CTAs/SM for the <= 128-row shapes (Cassie, quadruped), 2 above.
// The shared-structure instance has no adaptive-rho variant: launch_solve sends stride-0 batches with adaptive rho to the
// other kernels.
template <int kThreads, int kMinBlocks>
KernelFn solve_instance(bool shared, bool f32, bool adapt) {
  using fccqp::fccqp_solve_kernel;
  if (shared) return fccqp_solve_kernel<kThreads, kMinBlocks, true, false>;
  if (f32) return adapt ? fccqp_solve_kernel<kThreads, kMinBlocks, false, true, true> : fccqp_solve_kernel<kThreads, kMinBlocks, false, true>;
  return adapt ? fccqp_solve_kernel<kThreads, kMinBlocks, false, false, true> : fccqp_solve_kernel<kThreads, kMinBlocks, false, false>;
}
KernelFn pick_kernel(int threads, bool shared, bool f32, bool adapt) {
  return threads == 128 ? solve_instance<128, 4>(shared, f32, adapt) : solve_instance<256, 2>(shared, f32, adapt);
}

template <int kThreads, int kMinBlocks>
KernelFn struct_instance(bool adapt) {
  return adapt ? fccqp::fccqp_struct_kernel<kThreads, kMinBlocks, true> : fccqp::fccqp_struct_kernel<kThreads, kMinBlocks, false>;
}
template <int kThreads, int kMinBlocks>
KernelFn struct_first_instance(bool refine) {
  using fccqp::fccqp_struct_kernel;
  return refine ? fccqp_struct_kernel<kThreads, kMinBlocks, false, fccqp::kStructFirstRefine>
                : fccqp_struct_kernel<kThreads, kMinBlocks, false, fccqp::kStructFirst>;
}

// Host-side twin of fccqp::struct_classify for callers whose data is in host memory (no probe launch,
// no stream sync): counts of one QP.  Returns false for a structurally singular QP.
bool host_classify(int n, int m, const double* Q, long long q_rs, long long q_cs, const double* A, long long a_rs,
                   long long a_cs, int* nr, int* ndp, int* nd0) {
  std::vector<int> rowcnt(m > 0 ? m : 1, 0), one_row(n, -1);
  std::vector<char> type(n, 0);
  bool ok = true;
  for (int j = 0; j < n; ++j) {
    bool sep = true;
    for (int i = 0; i < n && sep; ++i)
      if (i != j && (Q[i * q_rs + j * q_cs] != 0.0 || Q[j * q_rs + i * q_cs] != 0.0)) sep = false;
    const double qd = Q[j * q_rs + j * q_cs];
    int nnz = 0, kr = 0;
    for (int k = 0; k < m; ++k) if (A[k * a_rs + j * a_cs] != 0.0) { ++nnz; kr = k; }
    if (!sep || !(qd >= 0.0)) type[j] = fccqp::VT_R;
    else if (qd < 1e-200) { type[j] = fccqp::VT_D0; if (nnz == 0) ok = false; }
    else if (nnz <= 1) { type[j] = fccqp::VT_D1; if (nnz == 1) { one_row[j] = kr; ++rowcnt[kr]; } }
    else type[j] = fccqp::VT_DP;
  }
  *nr = *ndp = *nd0 = 0;
  for (int j = 0; j < n; ++j) {
    if (type[j] == fccqp::VT_D1 && one_row[j] >= 0 && rowcnt[one_row[j]] > 1) type[j] = fccqp::VT_DP;
    if (type[j] == fccqp::VT_R) ++*nr; else if (type[j] == fccqp::VT_DP) ++*ndp; else if (type[j] == fccqp::VT_D0) ++*nd0;
  }
  return ok;
}

// Launch geometry of fn: as many CTAs per SM as fit (occupancy calculator, cached per device; at most
// FCCQP_CTAS_PER_SM), and no more CTAs than the batch fills at qps_per_cta QPs each.
int geometry(DeviceCtx& ctx, KernelFn fn, int threads, size_t smem, int B, int qps_per_cta, LaunchInfo* li) {
  int c = 0;
  {
    std::lock_guard<std::mutex> lk(ctx.mu);
    const auto key = std::make_pair((const void*)fn, smem);
    auto it = ctx.occupancy.find(key);
    if (it != ctx.occupancy.end()) c = it->second;
    else {
      // the attribute is per kernel, the smem size per problem shape: raise it to the device maximum once
      CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx.max_smem_optin));
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c, fn, threads, smem));
      if (c < 1) return fail(FCCQP_E_UNSUPPORTED, "kernel does not fit on an SM (smem %zu B)", smem);
      ctx.occupancy[key] = c;
    }
  }
  const int cap = dev_switches().cta_cap;
  if (cap > 0 && cap < c) c = cap;
  const int need = (B + qps_per_cta - 1) / qps_per_cta;
  *li = {c * ctx.num_sms < need ? c * ctx.num_sms : need, threads, (int)smem, c};
  return FCCQP_OK;
}

// One uniform set of QPs, run by a path launcher with exactly the launches a uniform call of its kind runs: the whole
// batch, or the cold or the warm QPs of a call with a per-lane mask.  Its counters and lists are its own.
struct LaneSet {
  int warm = 0;
  const int* order = nullptr;            // processing order: nullptr (0..B-1), the LPT order, or a kNoQP-padded list
  const unsigned int* count = nullptr;   // device-side length of a list; nullptr: the order ends at B or at its padding
  unsigned int* work = nullptr;          // [3] work counters: first or single launch, general kernel, resume launch
  unsigned int* handover_count = nullptr;  // QPs handed to a later launch: structure -> general kernel, shared-structure
  int* handover = nullptr;                 //   pre-solve -> ADMM launch
  unsigned int* resume_count = nullptr;    // QPs the first stage of a two-stage structure solve leaves to the resume
  int* resume = nullptr;                   //   launch
};

// Stream-ordered scratch of one launch_solve call: one allocation and one memset of its header, so that any number of
// calls may be in flight on any number of streams.  Offsets in 32-bit words.
struct Scratch {
  static constexpr size_t kProbe = 0;          // [0, 4): structure probe (atomicMax)
  static constexpr size_t kLpt = 4;            // [4, 6): counters of lpt_order_kernel
  static constexpr size_t kListCount = 6;      // [6, 8): lengths of the cold and the warm list (warm_split_kernel)
  static constexpr size_t kHandoverCount = 8;  // [8, 10): hand-over count of lane set 0 and of lane set 1, adjacent
  static constexpr size_t kResumeCount = 10;   // [10, 12): resume count of each lane set
  static constexpr size_t kWork = 12;          // [12, 18): three work counters of each lane set
  static constexpr size_t kHeader = 18;        // then [B] arrays: the hand-over and the resume list of set 0, the LPT
                                               // order; with a per-lane mask also the cold list, the warm list and the
                                               // hand-over and the resume list of set 1
  unsigned int* w = nullptr;
  size_t B = 0;
  int sets = 1;                                // 2 with a per-lane mask: set[0] its cold QPs, set[1] its warm ones
  LaneSet set[2];
  int* array(int i) const { return reinterpret_cast<int*>(w + kHeader + i * B); }
  LaneSet lanes(int k, int warm, const int* order, const unsigned int* count) const {
    return {warm, order, count, w + kWork + 3 * k, w + kHandoverCount + k, array(k ? 5 : 0), w + kResumeCount + k,
            array(k ? 6 : 1)};
  }
};

// Per-lane warm start (fccqp_batch_desc::warm_lanes): the processing order (`order`, or 0..B-1) split into the cold and the
// warm QPs, in that order within every warp of 32 slots; counts[0] / counts[1] = the lengths (zeroed by the caller).  The
// lists are pre-filled with kNoQP (>= B) bytes: the warp and structure-exploiting kernels stop at an index >= B and need no
// count; the general and shared-structure kernels take the count (SolveParams::count_dev).
constexpr unsigned char kNoQPByte = 0x7f;
__global__ void __launch_bounds__(256) warm_split_kernel(const uint8_t* __restrict__ warm_lanes, const int* __restrict__ order,
                                                         const int B, int* __restrict__ cold_list, int* __restrict__ warm_list,
                                                         unsigned int* __restrict__ counts) {
  const int slot = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31;
  const int qp = slot < B ? (order ? order[slot] : slot) : -1;
  const bool warm = qp >= 0 && warm_lanes[qp] != 0, cold = qp >= 0 && !warm;
  const unsigned int bw = __ballot_sync(0xffffffffu, warm), bc = __ballot_sync(0xffffffffu, cold);
  unsigned int base_c = 0, base_w = 0;
  if (lane == 0) {
    if (bc) base_c = atomicAdd(counts, (unsigned int)__popc(bc));
    if (bw) base_w = atomicAdd(counts + 1, (unsigned int)__popc(bw));
  }
  base_c = __shfl_sync(0xffffffffu, base_c, 0);
  base_w = __shfl_sync(0xffffffffu, base_w, 0);
  const unsigned int below = (1u << lane) - 1u;
  if (cold) cold_list[base_c + __popc(bc & below)] = qp;
  if (warm) warm_list[base_w + __popc(bw & below)] = qp;
}

// Per-lane rho (SolveParams::rho_lanes) and a two-stage structure solve: the first stage never reads rho, so a cold lane
// whose entry the solve cannot take may finish there.  Its n_iter and status are set here, after the launches, to what
// every other kernel path reports for it.
__global__ void __launch_bounds__(256) rho_invalid_kernel(const double* __restrict__ rho_lanes, const int B,
                                                          int* __restrict__ n_iter, int* __restrict__ status) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B || fccqp::rho_valid(rho_lanes[i])) return;
  if (n_iter) n_iter[i] = 0;
  if (status) status[i] = FCCQP_STATUS_NUMERICAL_ISSUE;
}

// Allocates the scratch of a call and sets out its lane sets.  FCCQP_SCHEDULE_LPT, when the batch holds at least two QPs
// for each of the `slots` that run at once: QPs whose previous solve ran long go to the front of the processing order.
// warm_lanes (device memory): the processing order is split into a cold and a warm list, one lane set each.
int begin_call(const fccqp::SolveParams& p, cudaStream_t stream, bool lpt_hint, long long slots, const uint8_t* warm_lanes,
               Scratch* s) {
  const bool lpt = lpt_hint && p.n_iter != nullptr && p.B >= 2 * slots;
  s->B = (size_t)p.B;
  const size_t arrays = warm_lanes ? 7 : (lpt ? 3 : 2);
  CUDA_TRY(cudaMallocAsync(&s->w, (Scratch::kHeader + arrays * s->B) * sizeof(unsigned int), stream));
  CUDA_TRY(cudaMemsetAsync(s->w, 0, Scratch::kHeader * sizeof(unsigned int), stream));
  int* order = nullptr;
  if (lpt) {
    order = s->array(2);
    fccqp::lpt_order_kernel<<<(p.B + 255) / 256, 256, 0, stream>>>(p.n_iter, p.B, p.full_inverse_at, order,
                                                                   s->w + Scratch::kLpt, s->w + Scratch::kLpt + 1);
    CUDA_TRY(cudaGetLastError());
  }
  if (!warm_lanes) {
    s->set[0] = s->lanes(0, p.warm, order, nullptr);
    return FCCQP_OK;
  }
  int *cold = s->array(3), *warm = s->array(4);
  CUDA_TRY(cudaMemsetAsync(cold, kNoQPByte, 2 * s->B * sizeof(int), stream));
  warm_split_kernel<<<(p.B + 255) / 256, 256, 0, stream>>>(warm_lanes, order, p.B, cold, warm, s->w + Scratch::kListCount);
  CUDA_TRY(cudaGetLastError());
  s->sets = 2;
  s->set[0] = s->lanes(0, 0, cold, s->w + Scratch::kListCount);
  s->set[1] = s->lanes(1, 1, warm, s->w + Scratch::kListCount + 1);
  return FCCQP_OK;
}

// p over a lane set: its warm flag, processing order and count, and its first work counter.
fccqp::SolveParams over(fccqp::SolveParams p, const LaneSet& l) {
  p.warm = l.warm;
  p.index_list = l.order;
  p.count_dev = l.count;
  p.work_counter = l.work;
  return p;
}

// Every solve launch: launched, checked and counted (fccqp_kernel_launch_count).
int launch(KernelFn fn, const LaunchInfo& li, const fccqp::SolveParams& p, cudaStream_t stream) {
  fn<<<li.grid, li.block, li.smem, stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return FCCQP_OK;
}

// Frees the scratch (stream-ordered) and records the call for fccqp_last_launch_info and fccqp_last_struct_info.
int end_call(const Scratch& s, cudaStream_t stream, const LaunchInfo& li, const StructInfo& si) {
  CUDA_TRY(cudaFreeAsync(s.w, stream));
  std::lock_guard<std::mutex> lk(g_info_mu);
  g_last_launch = li;
  g_last_struct = si;
  return FCCQP_OK;
}

StructInfo dense_info(const DeviceCtx& ctx, int rows) {
  StructInfo si;
  si.rows = si.rows_dense = rows;
  si.device = ctx.device;
  return si;
}

#ifdef FCCQP_DEV
// FCCQP_PROFILE: per-phase cycle counters of one launch (SolveParams::prof), summed over its CTAs and printed per QP
// to stderr.  Slot 14 counts the QPs; slot 15, when it has no name, the ADMM iterations.
struct PhaseProfile {
  unsigned long long* d = nullptr;
  int start(cudaStream_t stream, fccqp::SolveParams* p) {
    if (!dev_switches().profile) return FCCQP_OK;
    CUDA_TRY(cudaMalloc(&d, 16 * sizeof(unsigned long long)));
    CUDA_TRY(cudaMemsetAsync(d, 0, 16 * sizeof(unsigned long long), stream));
    p->prof = d;
    return FCCQP_OK;
  }
  int report(cudaStream_t stream, const char* kernel, const char* const (&names)[16], int B, int grid) {
    if (!d) return FCCQP_OK;
    unsigned long long h[16];
    CUDA_TRY(cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    CUDA_TRY(cudaFree(d));
    const double qps = (double)h[14];
    double tot = 0;
    for (int i = 0; i < 16; ++i) if (names[i]) tot += (double)h[i];
    fprintf(stderr, "[fccqp %s profile] B=%d grid=%d qps=%llu", kernel, B, grid, h[14]);
    if (!names[15]) fprintf(stderr, " iters=%llu", h[15]);
    fprintf(stderr, " cycles/QP=%.0f\n", qps > 0 ? tot / qps : 0.0);
    for (int i = 0; i < 16; ++i)
      if (names[i])
        fprintf(stderr, "   %-14s %10.0f cyc/QP  %5.1f%%\n", names[i], qps > 0 ? (double)h[i] / qps : 0.0,
                tot > 0 ? 100.0 * (double)h[i] / tot : 0.0);
    return FCCQP_OK;
  }
};
const char* const kStructPhases[16] = {"fetch+vectors", "classify", "zero+scatter", "wait-copies", "C+diag", "factor",
                                       "x: rhs", "x: solve", "project/exit", "epilogue", "x: refine | op: F", "x: recover",
                                       "x: rest", "op: inv(L)", nullptr, "op: G"};
const char* const kGeneralPhases[16] = {"stage-in", "assemble", "sigma/rhs0", "ldlt-acc+diag", "full-inverse", "-",
                                        "xinv32", "kkt-solve", "presolve-tail", "admm-project", "epilogue",
                                        "B-work-w0w2", "B-work-w1w3", "B-barrier-w0", nullptr, nullptr};
#endif

// Shared-structure batch (one Q and one A_eq for the whole batch): every CTA caches its KKT factorization
// (SolveParams::shared_mode).  Cold: a pre-solve launch hands the QPs that need ADMM iterations to an ADMM launch.
// Warm (an MPC loop re-solving around one linearisation with carried duals): no pre-solve, the ADMM launch alone.
int launch_shared(KernelFn fn, const LaunchInfo& li, const fccqp::SolveParams& p, const LaneSet& l, cudaStream_t stream) {
  fccqp::SolveParams a = over(p, l);
  if (!l.warm) {
    fccqp::SolveParams pre = a;
    pre.shared_mode = 1;
    pre.pending_count = l.handover_count;
    pre.pending_list = l.handover;
    if (int rc = launch(fn, li, pre, stream)) return rc;
    a.count_dev = l.handover_count;
    a.index_list = l.handover;
    a.work_counter = l.work + 1;
  }
  a.shared_mode = 2;
  return launch(fn, li, a, stream);
}

constexpr int kNotApplicable = 1;

// Structure-exploiting kernel (fccqp_struct.cuh): QPs whose separable variables can be eliminated analytically run on
// a reduced KKT system; the others (if any) are appended to a device-side list that the general kernel takes in a last
// launch.  plan_struct decides once per call what launch_struct runs for each lane set.
struct StructPlan {
  StructInfo info;
  fccqp::StructLayout sl;
  KernelFn first = nullptr, full = nullptr;   // the first stage; the single or the resume launch
  LaunchInfo fli, li;                          // their geometry
  bool two_stage = false;                      // a cold lane set runs in two stages
  double* op_scratch = nullptr;                // per-CTA global scratch of the full-space operator of long-running QPs
  long long op_stride = 0;                     //   (build_full_op), doubles per CTA
};

// The caps (probed on the device, or given), the reduced layout, the instances and their geometry, and op_scratch.
// Returns kNotApplicable, with nothing launched but the probe, when the reduction does not pay.
int plan_struct(DeviceCtx& ctx, const fccqp::SolveParams& p, cudaStream_t stream, const Scratch& s, const StructHint& hint,
                StructPlan* sp) {
  int caps[3] = {hint.caps[0], hint.caps[1], hint.caps[2]};
  if (hint.mode != FCCQP_STRUCTURE_CAPS) {
    // probe: classify up to 128 QPs spread over the batch, take the largest structure seen
    const int ns = p.B < 128 ? p.B : 128;
    int* d_probe = reinterpret_cast<int*>(s.w + Scratch::kProbe);
    if (p.n <= 128 && p.m <= 128) fccqp::fccqp_struct_probe_kernel<128><<<ns, 128, 0, stream>>>(p, ns, d_probe);
    else fccqp::fccqp_struct_probe_kernel<256><<<ns, 256, 0, stream>>>(p, ns, d_probe);
    CUDA_TRY(cudaGetLastError());
    int h[4];
    {
      std::lock_guard<std::mutex> lk(ctx.mu);   // the pinned landing pad is per device
      CUDA_TRY(cudaMemcpyAsync(ctx.h_probe, d_probe, sizeof(h), cudaMemcpyDeviceToHost, stream));
      CUDA_TRY(cudaStreamSynchronize(stream));
      memcpy(h, ctx.h_probe, sizeof(h));
    }
    g_launches.fetch_add(1);
    if (h[3] != 0) return kNotApplicable;   // a structurally singular QP in the sample
    caps[0] = h[0]; caps[1] = h[1]; caps[2] = h[2];
  }
  if (caps[0] < 0 || caps[0] > p.n || caps[1] < 0 || caps[2] < 0 || caps[0] + caps[1] + caps[2] > p.n) return kNotApplicable;
  const fccqp::StructLayout sl(p.n, p.m, p.nc, caps[0], caps[1] + caps[2], caps[2]);   // D+ store: pass 1 eliminates D0 too
  // worth it when at least one tile row of the KKT matrix goes away
  if (sl.N8c + 8 > p.lay.N8 || sl.bytes() > (size_t)ctx.max_smem_optin) return kNotApplicable;
  // threads >= max(n, padded reduced KKT size), at most 256 since the reduced size is below p.lay.N8
  const int need = p.n > sl.N8c ? p.n : sl.N8c;
  const bool adapt = p.adapt_k > 0 || p.rho_lanes, refine = p.struct_refine != 0;
  int threads;
  if (need <= 64) { threads = 64; sp->first = struct_first_instance<64, 8>(refine); sp->full = struct_instance<64, 8>(adapt); }
  else if (need <= 96) { threads = 96; sp->first = struct_first_instance<96, 5>(refine); sp->full = struct_instance<96, 5>(adapt); }
  else if (need <= 128) { threads = 128; sp->first = struct_first_instance<128, 4>(refine); sp->full = struct_instance<128, 4>(adapt); }
  else { threads = 256; sp->first = struct_first_instance<256, 2>(refine); sp->full = struct_instance<256, 2>(adapt); }
  int rc;
  if ((rc = geometry(ctx, sp->first, threads, sl.bytes(), p.B, 1, &sp->fli)) ||
      (rc = geometry(ctx, sp->full, threads, sl.bytes(), p.B, 1, &sp->li)))
    return rc;
  // Cold batches of at least 8 QPs per resident CTA run in two stages: the first-stage kernel takes every QP through the
  // exit test of iteration 0 (where nearly all whole-body-control QPs stop) and lists the others, which the full kernel
  // resumes from there.  Smaller batches and warm solves keep the single launch.  The rule looks at the whole batch,
  // also when a per-lane mask leaves only some of its QPs cold.
  sp->two_stage = p.B >= 8LL * sp->fli.ctas_per_sm * ctx.num_sms;
  sp->sl = sl;
  // B, Z, X, Y tiles and 1/h sized for every variable eliminated
  const long long neT = sl.n8 >> 3, NBr = sl.nr8c >> 3, mt = sl.mt;
  sp->op_stride = (2 * mt * neT + neT * NBr + neT * (neT + 1) / 2) * 64 + 8 * neT;
  CUDA_TRY(cudaMallocAsync(&sp->op_scratch, (size_t)sp->li.grid * sp->op_stride * sizeof(double), stream));
  StructInfo& si = sp->info;
  si.used = 1; si.nr = caps[0]; si.ndp = caps[1]; si.nd0 = caps[2]; si.rows = sl.N8c; si.rows_dense = p.lay.N8; si.device = ctx.device;
  return FCCQP_OK;
}

// One lane set on the structure path: the single launch, or a cold set in two stages; then the general kernel (geometry
// gli) over the QPs handed over.
int launch_struct(const StructPlan& sp, KernelFn general, const LaunchInfo& gli, const fccqp::SolveParams& p, const LaneSet& l,
                  cudaStream_t stream) {
  const bool split = !l.warm && sp.two_stage;
  fccqp::SolveParams a = over(p, l);
  a.count_dev = nullptr;   // to the structure kernel a count marks the resume launch; a list's padding ends this one
  a.slay = sp.sl;
  a.pending_count = l.handover_count;
  a.pending_list = l.handover;
  int rc;
  if (split) {
    fccqp::SolveParams f = a;
    f.resume_list = l.resume;
    f.resume_count = l.resume_count;
#ifdef FCCQP_DEV
    PhaseProfile prof;
    if ((rc = prof.start(stream, &f))) return rc;
#endif
    if ((rc = launch(sp.first, sp.fli, f, stream))) return rc;
#ifdef FCCQP_DEV
    if ((rc = prof.report(stream, "struct first stage", kStructPhases, p.B, sp.fli.grid))) return rc;
#endif
    a.count_dev = l.resume_count;
    a.index_list = l.resume;
    a.work_counter = l.work + 2;
  }
  a.op_scratch = sp.op_scratch;
  a.op_stride = sp.op_stride;
#ifdef FCCQP_DEV
  PhaseProfile prof;
  if ((rc = prof.start(stream, &a))) return rc;
#endif
  if ((rc = launch(sp.full, sp.li, a, stream))) return rc;
#ifdef FCCQP_DEV
  if ((rc = prof.report(stream, split ? "struct resume" : "struct", kStructPhases, p.B, sp.li.grid))) return rc;
#endif
  if (split && p.rho_lanes) {
    rho_invalid_kernel<<<(p.B + 255) / 256, 256, 0, stream>>>(p.rho_lanes, p.B, p.n_iter, p.status);
    CUDA_TRY(cudaGetLastError());
    g_launches.fetch_add(1);
  }
  fccqp::SolveParams b = over(p, l);
  b.count_dev = l.handover_count;
  b.index_list = l.handover;
  b.work_counter = l.work + 1;
  return launch(general, gli, b, stream);
}

int launch_general(KernelFn fn, const LaunchInfo& li, fccqp::SolveParams p, cudaStream_t stream) {
#ifdef FCCQP_DEV
  PhaseProfile prof;
  int rc = prof.start(stream, &p);
  if (!rc) rc = launch(fn, li, p, stream);
  return rc ? rc : prof.report(stream, "general", kGeneralPhases, p.B, li.grid);
#else
  return launch(fn, li, p, stream);
#endif
}

// Launches the solve on `stream` for device-resident data described by p (scratch allocated here, stream-ordered).
// precision: fccqp_precision of the call (FP32_DATA and FP32: float32 problem data behind the pointers of p; FP32: FP32
// arithmetic too where a kernel for it exists -- the warp kernel -- and FP32_DATA's FP64 arithmetic otherwise)
// warm_lanes: optional per-lane mask in device memory (fccqp_batch_desc::warm_lanes); p.warm is then ignored, and the
// path runs twice: as a uniform cold call over the cold QPs, then as a uniform warm call over the warm ones.
// p.rho_lanes: optional per-lane rho in device memory (fccqp_batch_solve_rho); such calls run the instances that keep rho
// per QP (kAdapt, and kRhoLanes of the warp kernel), never the shared-structure path (its cached factorization has one rho).
int launch_solve(DeviceCtx& ctx, fccqp::SolveParams p, cudaStream_t stream, int precision, const StructHint& hint,
                 const uint8_t* warm_lanes = nullptr) {
  if (p.B == 0) return FCCQP_OK;
  int rc = check_shape(ctx, p.n, p.m, p.nc);
  if (rc) return rc;
  const DevSwitches& sw = dev_switches();
  const bool f32 = precision != FCCQP_PRECISION_FP64;
  const bool small = p.n + p.m <= 32;   // the KKT matrix fits one row per lane
  p.lay = fccqp::Layout(p.n, p.m, p.nc);
  p.full_inverse_at = sw.full_inverse_at ? sw.full_inverse_at : (small ? 8 : 6);
  p.struct_refine = hint.refine;
  enum { kWarp, kShared, kStruct, kGeneral } path;
  KernelFn fn, general = nullptr;
  LaunchInfo li, gli;   // geometry of fn, and of the general kernel
  long long slots;      // QPs that run at once
  int rows = p.lay.N8;
  if (small && (precision == FCCQP_PRECISION_FP32 || (!f32 && !sw.no_warp))) {
    // Small problems (n + m <= 32): one QP per warp (fccqp_warp.cuh), four warps per CTA, each pulling QPs from the work
    // counter on its own; shared memory per CTA = 4 private (n + m) x ((n + m) | 1) slabs.  FCCQP_PRECISION_FP32: the FP32
    // arithmetic instance (float32 problem data, float slabs).
    constexpr int kW = 4;
    const bool f32a = precision == FCCQP_PRECISION_FP32;
    rows = p.n + p.m;
    const size_t smem = (size_t)kW * rows * (rows | 1) * (f32a ? sizeof(float) : sizeof(double));
    using fccqp::fccqp_warp_kernel;
    fn = p.rho_lanes ? (f32a ? (KernelFn)fccqp_warp_kernel<kW, 6, float, true> : (KernelFn)fccqp_warp_kernel<kW, 6, double, true>)
                     : (f32a ? (KernelFn)fccqp_warp_kernel<kW, 6, float> : (KernelFn)fccqp_warp_kernel<kW, 6, double>);
    // (measured, tools/bench_small.py: 6 CTAs x 4 warps at 80 registers beats 8 x 4 at 64 and 4 x 4 at 128 on every shape but n = 6;
    //  float instance, tools/fp32_occ.py: 6 / 8 / 10 / 12 CTAs -> 82.7 / 78.5 / 71.4 / 70.5 M QP/s at n = 6, 22.4 / 23.1 / 21.1 / 21.7 at n = 24)
    path = kWarp;
    rc = geometry(ctx, fn, 32 * kW, smem, p.B, kW, &li);
    slots = (long long)kW * li.ctas_per_sm * ctx.num_sms;
  } else {
    // one CTA per QP; float32 problem data take the general kernel's widening instance, same geometry
    const int threads = p.lay.N8 <= 128 ? 128 : 256;
    general = pick_kernel(threads, false, f32, p.adapt_k > 0 || p.rho_lanes);
    if ((rc = geometry(ctx, general, threads, p.lay.bytes(), p.B, 1, &gli))) return rc;
    slots = (long long)gli.ctas_per_sm * ctx.num_sms;
    // one Q and one A_eq for the whole batch: caching the factorization pays once every CTA sees several QPs.  Not with
    // adaptive or per-lane rho: a lane with its own rho needs its own rho-KKT factorization, so those batches take the
    // structure-exploiting or general kernel (both read Q and A_eq through the batch stride).
    if (!sw.no_shared && !f32 && p.adapt_k == 0 && !p.rho_lanes && p.q_bs == 0 && (p.m == 0 || p.a_bs == 0) &&
        p.B >= 4 * gli.ctas_per_sm * ctx.num_sms) {
      path = kShared;
      fn = pick_kernel(threads, true, false, false);
      rc = geometry(ctx, fn, threads, p.lay.bytes(), p.B, 1, &li);
    } else {
      path = !f32 && hint.mode != FCCQP_STRUCTURE_DENSE && p.m > 0 ? kStruct : kGeneral;
      fn = general;
      li = gli;
    }
  }
  Scratch s;
  if (rc || (rc = begin_call(p, stream, hint.lpt, slots, warm_lanes, &s))) return rc;
  StructPlan sp;
  if (path == kStruct && (rc = plan_struct(ctx, p, stream, s, hint, &sp))) {
    if (rc != kNotApplicable) return rc;
    path = kGeneral;
    rc = FCCQP_OK;
  }
  for (int k = 0; k < s.sets && !rc; ++k) {
    const LaneSet& l = s.set[k];
    if (path == kWarp) rc = launch(fn, li, over(p, l), stream);
    else if (path == kShared) rc = launch_shared(fn, li, p, l, stream);
    else if (path == kStruct) rc = launch_struct(sp, general, gli, p, l, stream);
    else rc = launch_general(fn, li, over(p, l), stream);
  }
  if (rc) return rc;
  if (path != kStruct) return end_call(s, stream, li, dense_info(ctx, rows));
  CUDA_TRY(cudaFreeAsync(sp.op_scratch, stream));
  CUDA_TRY(cudaMemcpyAsync(ctx.h_deferred, s.w + Scratch::kHandoverCount, 2 * sizeof(unsigned int), cudaMemcpyDeviceToHost,
                           stream));
  // the geometry of the cold sequence: its first stage when it ran in two stages
  return end_call(s, stream, sp.two_stage && !s.set[0].warm ? sp.fli : sp.li, sp.info);
}

int check_dims(int n, int m, int nc, int lcs) {
  if (n < 0 || m < 0 || nc < 0) return fail(FCCQP_E_INVALID, "negative dimension");
  if (nc % 3 != 0) return fail(FCCQP_E_INVALID, "nc = %d must be a multiple of 3 (src/fcc_qp.cpp:32)", nc);
  if (lcs < 0 || lcs + nc > n)
    return fail(FCCQP_E_INVALID, "lambda_c_start + nc = %d exceeds num_vars = %d (src/fcc_qp.cpp:33)", lcs + nc, n);
  if (n < 1) return fail(FCCQP_E_INVALID, "num_vars must be >= 1");
  return FCCQP_OK;
}

int check_options(const fccqp_options& o) {
  if (o.max_iter < 0) return fail(FCCQP_E_INVALID, "max_iter must be >= 0");
  if (!(o.rho > 0.0)) return fail(FCCQP_E_INVALID, "rho must be > 0 (src/fcc_qp.hpp:76)");
  if (o.relaxation != 0.0 && !(o.relaxation > 0.0 && o.relaxation < 2.0))
    return fail(FCCQP_E_INVALID, "relaxation must be in (0, 2) (0 = unset = 1)");
  if (o.adapt_rho_interval < 0) return fail(FCCQP_E_INVALID, "adapt_rho_interval must be >= 0 (0 = off)");
  return FCCQP_OK;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// The solve parameters every path needs; the data pointers are left to the caller.
fccqp::SolveParams solve_params(int B, int n, int m, int nc, int lcs, const fccqp_options& o, bool warm) {
  fccqp::SolveParams p{};
  p.B = B; p.n = n; p.m = m; p.nc = nc; p.lcs = lcs;
  p.max_iter = o.max_iter; p.rho = o.rho; p.eps_fcone = o.eps_fcone; p.eps_bound = o.eps_bound;
  p.alpha = o.relaxation > 0.0 ? o.relaxation : 1.0;
  p.adapt_k = o.adapt_rho_interval;
  p.warm = warm;
  return p;
}

}  // namespace

// ---------------------------------------------------------------------------
// single-problem object
// ---------------------------------------------------------------------------
struct fccqp_solver {
  int n, m, nc, lcs, device;
  fccqp_options opt;
  int warm = 0;
  int structure = FCCQP_STRUCTURE_AUTO;
  bool has_state = false;  // a Solve has happened (x_ is meaningful)
  DeviceCtx* ctx = nullptr;
  cudaStream_t stream = nullptr;
  // device: inputs packed [Q n*n | A m*n | b n | beq m | mu nc/3 | lb n | ub n], state, outputs
  double* d_in = nullptr;
  double* d_x = nullptr; double* d_mux = nullptr; double* d_muc = nullptr;
  double* d_out = nullptr;   // [4] res_b res_f bviol fviol ; then ints
  int* d_iout = nullptr;     // [2] n_iter status
  unsigned long long* d_cycles = nullptr;
  // pinned host mirrors
  double* h_in = nullptr;
  double* h_out = nullptr;   // [n + 4] z + scalars
  int* h_iout = nullptr;
  unsigned long long* h_cycles = nullptr;
  unsigned long long prev_fact_cycles = 0;   // the device counter accumulates across solves
  size_t in_doubles = 0;
  fccqp_details details{};
};

extern "C" {

void fccqp_default_options(fccqp_options* opt) {
  if (!opt) return;
  opt->max_iter = 1000; opt->adapt_rho_interval = 0; opt->rho = 1e-6; opt->eps_fcone = 1e-3; opt->eps_bound = 1e-6;
  opt->relaxation = 1.0;
}
const char* fccqp_last_error(void) { return g_err.c_str(); }
int fccqp_abi_version(void) { return FCCQP_ABI_VERSION; }
int fccqp_device_count(void) {
  int c = 0;
  if (cudaGetDeviceCount(&c) != cudaSuccess) { cudaGetLastError(); return 0; }
  return c;
}
int64_t fccqp_kernel_launch_count(void) { return g_launches.load(); }

int fccqp_measure_fp64_peak(int device, double* tflops) {
  if (!tflops) return fail(FCCQP_E_INVALID, "tflops is null");
  DeviceCtx* ctx = nullptr;
  int rc = get_ctx(device, &ctx);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(device));
  double* d_out = nullptr;
  CUDA_TRY(cudaMalloc(&d_out, sizeof(double)));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  const int grid = ctx->num_sms * 4, iters = 60000;   // ~50 ms on a B200
  double best = 0.0;
  for (int rep = 0; rep < 3; ++rep) {   // first launch warms the clocks up
    CUDA_TRY(cudaEventRecord(e0, 0));
    fccqp::fp64_peak_kernel<<<grid, 256>>>(d_out, iters, 1.0);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(e1, 0));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    const double fl = 2.0 * 64.0 * (double)iters * 256.0 * (double)grid;
    const double tf = fl / (1e-3 * ms) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  g_launches.fetch_add(3);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  CUDA_TRY(cudaFree(d_out));
  *tflops = best;
  return FCCQP_OK;
}
int fccqp_last_struct_info(int* used, int* caps, int* rows, int* rows_dense, int* deferred) {
  StructInfo si;
  { std::lock_guard<std::mutex> lk(g_info_mu); si = g_last_struct; }
  if (used) *used = si.used;
  if (caps) { caps[0] = si.nr; caps[1] = si.ndp; caps[2] = si.nd0; }
  if (rows) *rows = si.rows;
  if (rows_dense) *rows_dense = si.rows_dense;
  if (deferred) {
    *deferred = 0;
    if (si.used) {
      std::lock_guard<std::mutex> lk(g_ctx_mu);
      auto it = g_ctx.find(si.device);
      if (it != g_ctx.end() && it->second->h_deferred)
        *deferred = (int)it->second->h_deferred[0] + (int)it->second->h_deferred[1];
    }
  }
  return FCCQP_OK;
}
int fccqp_last_launch_info(int* grid, int* block, int* smem_bytes, int* ctas_per_sm) {
  std::lock_guard<std::mutex> lk(g_info_mu);
  if (grid) *grid = g_last_launch.grid;
  if (block) *block = g_last_launch.block;
  if (smem_bytes) *smem_bytes = g_last_launch.smem;
  if (ctas_per_sm) *ctas_per_sm = g_last_launch.ctas_per_sm;
  return FCCQP_OK;
}

int fccqp_create(int n, int m, int nc, int lcs, int device, fccqp_handle* out) {
  if (!out) return fail(FCCQP_E_INVALID, "out is null");
  *out = nullptr;
  int rc = check_dims(n, m, nc, lcs);
  if (rc) return rc;
  DeviceCtx* ctx = nullptr;
  rc = get_ctx(device, &ctx);
  if (rc) return rc;
  rc = check_shape(*ctx, n, m, nc);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(device));
  auto* h = new fccqp_solver();
  h->n = n; h->m = m; h->nc = nc; h->lcs = lcs; h->device = device; h->ctx = ctx;
  fccqp_default_options(&h->opt);
  h->in_doubles = (size_t)n * n + (size_t)m * n + n + m + nc / 3 + n + n;
  auto cleanup_fail = [&](cudaError_t e, const char* what) {
    int r = fail(FCCQP_E_CUDA, "%s failed: %s", what, cudaGetErrorString(e));
    fccqp_destroy(h);
    return r;
  };
  cudaError_t e;
  if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking))) return cleanup_fail(e, "cudaStreamCreate");
  if ((e = cudaMalloc(&h->d_in, (h->in_doubles + 2) * sizeof(double)))) return cleanup_fail(e, "cudaMalloc");
  // outputs packed in one device buffer so that ONE D2H copy brings everything back:
  //   [x (n doubles) | res_b res_f bviol fviol | cycles (2 x u64) | n_iter status (2 x i32)]
  if ((e = cudaMalloc(&h->d_x, (size_t)(n + 8) * sizeof(double)))) return cleanup_fail(e, "cudaMalloc");
  h->d_out = h->d_x + n;
  h->d_cycles = reinterpret_cast<unsigned long long*>(h->d_x + n + 4);
  h->d_iout = reinterpret_cast<int*>(h->d_x + n + 6);
  if ((e = cudaMalloc(&h->d_mux, (size_t)(n + 1) * sizeof(double)))) return cleanup_fail(e, "cudaMalloc");
  if ((e = cudaMalloc(&h->d_muc, (size_t)(nc + 1) * sizeof(double)))) return cleanup_fail(e, "cudaMalloc");
  if ((e = cudaMallocHost(&h->h_in, (h->in_doubles + 2) * sizeof(double)))) return cleanup_fail(e, "cudaMallocHost");
  if ((e = cudaMallocHost(&h->h_out, (size_t)(n + 8) * sizeof(double)))) return cleanup_fail(e, "cudaMallocHost");
  h->h_cycles = reinterpret_cast<unsigned long long*>(h->h_out + n + 4);
  h->h_iout = reinterpret_cast<int*>(h->h_out + n + 6);
  if ((e = cudaMemset(h->d_x, 0, (size_t)(n + 8) * sizeof(double)))) return cleanup_fail(e, "cudaMemset");
  if ((e = cudaMemset(h->d_mux, 0, (size_t)(n + 1) * sizeof(double)))) return cleanup_fail(e, "cudaMemset");
  if ((e = cudaMemset(h->d_muc, 0, (size_t)(nc + 1) * sizeof(double)))) return cleanup_fail(e, "cudaMemset");
  memset(h->h_out, 0, (size_t)(n + 8) * sizeof(double));
  *out = h;
  return FCCQP_OK;
}

int fccqp_destroy(fccqp_handle h) {
  if (!h) return FCCQP_OK;
  cudaSetDevice(h->device);
  if (h->stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); }
  cudaFree(h->d_in); cudaFree(h->d_x); cudaFree(h->d_mux); cudaFree(h->d_muc);
  cudaFreeHost(h->h_in); cudaFreeHost(h->h_out);
  delete h;
  return FCCQP_OK;
}

int fccqp_set_options(fccqp_handle h, const fccqp_options* opt) {
  if (!h || !opt) return fail(FCCQP_E_INVALID, "null argument");
  int rc = check_options(*opt);
  if (rc) return rc;
  h->opt = *opt;
  return FCCQP_OK;
}
int fccqp_get_options(fccqp_handle h, fccqp_options* opt) {
  if (!h || !opt) return fail(FCCQP_E_INVALID, "null argument");
  *opt = h->opt;
  return FCCQP_OK;
}
int fccqp_set_rho(fccqp_handle h, double rho) {
  if (!h) return fail(FCCQP_E_INVALID, "null handle");
  if (!(rho > 0.0)) return fail(FCCQP_E_INVALID, "rho must be > 0 (src/fcc_qp.hpp:76)");
  h->opt.rho = rho;
  return FCCQP_OK;
}
int fccqp_set_max_iter(fccqp_handle h, int max_iter) {
  if (!h) return fail(FCCQP_E_INVALID, "null handle");
  if (max_iter <= 0) return fail(FCCQP_E_INVALID, "max_iter must be > 0 (src/fcc_qp.hpp:81)");
  h->opt.max_iter = max_iter;
  return FCCQP_OK;
}
int fccqp_set_warm_start(fccqp_handle h, int warm) {
  if (!h) return fail(FCCQP_E_INVALID, "null handle");
  h->warm = warm != 0;
  return FCCQP_OK;
}
int fccqp_set_structure(fccqp_handle h, int structure) {
  if (!h) return fail(FCCQP_E_INVALID, "null handle");
  StructHint hint;
  hint.set(structure);
  if (hint.mode != FCCQP_STRUCTURE_AUTO && hint.mode != FCCQP_STRUCTURE_DENSE)
    return fail(FCCQP_E_INVALID, "structure must be FCCQP_STRUCTURE_AUTO or FCCQP_STRUCTURE_DENSE (optionally | FCCQP_STRUCTURE_REFINE)");
  h->structure = structure;
  return FCCQP_OK;
}
int fccqp_contact_vars_start(fccqp_handle h) { return h ? h->lcs : -1; }

int fccqp_solve(fccqp_handle h, const double* Q, ptrdiff_t q_rs, ptrdiff_t q_cs, const double* b,
                const double* A, ptrdiff_t a_rs, ptrdiff_t a_cs, const double* b_eq,
                const double* mu, int n_mu, const double* lb, const double* ub) {
  if (!h) return fail(FCCQP_E_INVALID, "null handle");
  const int n = h->n, m = h->m, nc = h->nc;
  if (!Q || !b || (m > 0 && (!A || !b_eq)) || !lb || !ub || (nc > 0 && !mu))
    return fail(FCCQP_E_INVALID, "null input pointer");
  if (n_mu < nc / 3)
    return fail(FCCQP_E_INVALID, "friction_coeffs has %d entries, need %d (src/constraint_utils.cpp:32)", n_mu, nc / 3);
  const auto t0 = std::chrono::steady_clock::now();
  CUDA_TRY(cudaSetDevice(h->device));
  // pack into pinned staging: Q row-major n x n (symmetric), A in its cheaper traversal order
  double* s = h->h_in;
  double* sQ = s; s += (size_t)n * n;
  double* sA = s; s += (size_t)m * n;
  double* sb = s; s += n;
  double* sbeq = s; s += m;
  double* smu = s; s += nc / 3;
  double* slb = s; s += n;
  double* sub = s;
  // Q: copy along the contiguous direction when there is one
  if (q_cs == 1) for (int i = 0; i < n; ++i) memcpy(sQ + (size_t)i * n, Q + i * q_rs, sizeof(double) * n);
  else if (q_rs == 1) for (int j = 0; j < n; ++j) memcpy(sQ + (size_t)j * n, Q + j * q_cs, sizeof(double) * n);  // symmetric
  else for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) sQ[(size_t)i * n + j] = Q[i * q_rs + j * q_cs];
  // A_eq: always packed row-major (a column-major Eigen matrix is transposed here, m x n is small): the kernels'
  // row-wise 16-byte passes then apply whatever the caller's layout
  const long long k_a_rs = n, k_a_cs = 1;
  for (int i = 0; i < m; ++i)
    for (int j = 0; j < n; ++j) sA[(size_t)i * n + j] = A[i * a_rs + j * a_cs];
  memcpy(sb, b, sizeof(double) * n);
  if (m) memcpy(sbeq, b_eq, sizeof(double) * m);
  if (nc) memcpy(smu, mu, sizeof(double) * (nc / 3));
  memcpy(slb, lb, sizeof(double) * n);
  memcpy(sub, ub, sizeof(double) * n);
  CUDA_TRY(cudaMemcpyAsync(h->d_in, h->h_in, h->in_doubles * sizeof(double), cudaMemcpyHostToDevice, h->stream));

  // warm with no earlier Solve starts from the zero state, like the reference object
  fccqp::SolveParams p = solve_params(1, n, m, nc, h->lcs, h->opt, h->warm != 0);
  double* d = h->d_in;
  p.Q = d; p.q_bs = 0; p.q_rs = n; p.q_cs = 1; d += (size_t)n * n;
  p.A = d; p.a_bs = 0; p.a_rs = k_a_rs; p.a_cs = k_a_cs; d += (size_t)m * n;
  p.b = d; p.b_bs = 0; d += n;
  p.beq = d; p.beq_bs = 0; d += m;
  p.mu = d; p.mu_bs = 0; d += nc / 3;
  p.lb = d; p.lb_bs = 0; d += n;
  p.ub = d; p.ub_bs = 0;
  p.x = h->d_x; p.mu_x = h->d_mux; p.mu_c = h->d_muc;
  p.n_iter = h->d_iout; p.status = h->d_iout + 1;
  p.res_b = h->d_out; p.res_f = h->d_out + 1; p.bviol = h->d_out + 2; p.fviol = h->d_out + 3;
  p.cycles = h->d_cycles;
  // the data is right here on the host: classify it here (no probe launch, no extra synchronisation)
  StructHint hint;
  hint.set(h->structure);
  const bool want_struct = hint.mode == FCCQP_STRUCTURE_AUTO;
  hint.mode = FCCQP_STRUCTURE_DENSE;
  if (want_struct && m > 0 &&
      host_classify(n, m, sQ, n, 1, sA, k_a_rs, k_a_cs, &hint.caps[0], &hint.caps[1], &hint.caps[2]))
    hint.mode = FCCQP_STRUCTURE_CAPS;
  int rc = launch_solve(*h->ctx, p, h->stream, FCCQP_PRECISION_FP64, hint);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(h->h_out, h->d_x, sizeof(double) * (n + 8), cudaMemcpyDeviceToHost, h->stream));   // packed outputs
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  h->has_state = true;
  h->details.n_iter = h->h_iout[0];
  h->details.solve_status = h->h_iout[1];
  h->details.admm_residual_bounds = h->h_out[n];
  h->details.admm_residual_friction_cone = h->h_out[n + 1];
  h->details.bounds_viol = h->h_out[n + 2];
  h->details.friction_cone_viol = h->h_out[n + 3];
  h->details.factorization_time =
      h->ctx->clock_khz > 0 ? (double)(h->h_cycles[0] - h->prev_fact_cycles) / (1e3 * h->ctx->clock_khz) : 0.0;
  h->prev_fact_cycles = h->h_cycles[0];
  h->details.solve_time = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  return FCCQP_OK;
}

int fccqp_get_solution(fccqp_handle h, double* z, fccqp_details* details) {
  if (!h) return fail(FCCQP_E_INVALID, "null handle");
  if (z) memcpy(z, h->h_out, sizeof(double) * h->n);
  if (details) *details = h->details;
  return FCCQP_OK;
}

int fccqp_get_warm_state(fccqp_handle h, double* x, double* mu_x, double* mu_c) {
  if (!h) return fail(FCCQP_E_INVALID, "null handle");
  CUDA_TRY(cudaSetDevice(h->device));
  if (x) CUDA_TRY(cudaMemcpy(x, h->d_x, sizeof(double) * h->n, cudaMemcpyDeviceToHost));
  if (mu_x) CUDA_TRY(cudaMemcpy(mu_x, h->d_mux, sizeof(double) * h->n, cudaMemcpyDeviceToHost));
  if (mu_c && h->nc) CUDA_TRY(cudaMemcpy(mu_c, h->d_muc, sizeof(double) * h->nc, cudaMemcpyDeviceToHost));
  return FCCQP_OK;
}
int fccqp_set_warm_state(fccqp_handle h, const double* x, const double* mu_x, const double* mu_c) {
  if (!h) return fail(FCCQP_E_INVALID, "null handle");
  CUDA_TRY(cudaSetDevice(h->device));
  if (x) CUDA_TRY(cudaMemcpy(h->d_x, x, sizeof(double) * h->n, cudaMemcpyHostToDevice));
  if (mu_x) CUDA_TRY(cudaMemcpy(h->d_mux, mu_x, sizeof(double) * h->n, cudaMemcpyHostToDevice));
  if (mu_c && h->nc) CUDA_TRY(cudaMemcpy(h->d_muc, mu_c, sizeof(double) * h->nc, cudaMemcpyHostToDevice));
  h->has_state = true;
  return FCCQP_OK;
}

// Structure bounds of a HOST batch from a sample of up to 64 of its QPs (FCCQP_STRUCTURE_AUTO); other modes pass through.
static void host_struct_hint(const fccqp_batch_desc& d, StructHint* out) {
  StructHint hint;
  hint.set(d.structure);
  hint.caps[0] = d.struct_caps[0]; hint.caps[1] = d.struct_caps[1]; hint.caps[2] = d.struct_caps[2];
  const int B = d.batch, n = d.n, m = d.m;
  const bool q_shared = d.q_batch_stride == 0, a_shared = d.a_batch_stride == 0;
  if (hint.mode == FCCQP_STRUCTURE_AUTO) {
    hint.mode = FCCQP_STRUCTURE_DENSE;
    if (d.precision == FCCQP_PRECISION_FP64 && m > 0 && !(q_shared && a_shared) && B > 0) {
      const int ns = B < 64 ? B : 64;
      bool ok = true;
      for (int sidx = 0; sidx < ns && ok; ++sidx) {
        const long long qp = ns > 1 ? (long long)sidx * (B - 1) / (ns - 1) : 0;
        int c[3];
        ok = host_classify(n, m, d.Q + (q_shared ? 0 : qp * (long long)n * n), d.q_row_stride, d.q_col_stride,
                           d.A_eq + (a_shared ? 0 : qp * (long long)m * n), d.a_row_stride, d.a_col_stride, &c[0], &c[1], &c[2]);
        for (int k = 0; k < 3; ++k) if (c[k] > hint.caps[k]) hint.caps[k] = c[k];
      }
      if (ok) hint.mode = FCCQP_STRUCTURE_CAPS;
    }
  }
  *out = hint;
}

// ---------------------------------------------------------------------------
// batched entry point
// ---------------------------------------------------------------------------
static int validate_desc(const fccqp_batch_desc* d) {
  if (!d) return fail(FCCQP_E_INVALID, "desc is null");
  if (d->abi_version != FCCQP_ABI_VERSION)
    return fail(FCCQP_E_INVALID, "abi_version %d != %d", d->abi_version, FCCQP_ABI_VERSION);
  if (d->batch < 0) return fail(FCCQP_E_INVALID, "batch < 0");
  int rc = check_dims(d->n, d->m, d->nc, d->lambda_c_start);
  if (rc) return rc;
  rc = check_options(d->options);
  if (rc) return rc;
  if (d->precision != FCCQP_PRECISION_FP64 && d->precision != FCCQP_PRECISION_FP32_DATA && d->precision != FCCQP_PRECISION_FP32)
    return fail(FCCQP_E_UNSUPPORTED, "precision must be FCCQP_PRECISION_FP64, FCCQP_PRECISION_FP32_DATA or FCCQP_PRECISION_FP32");
  if (d->memory_space != FCCQP_MEM_HOST && d->memory_space != FCCQP_MEM_DEVICE)
    return fail(FCCQP_E_INVALID, "bad memory_space");
  if (d->batch == 0) return FCCQP_OK;
  if (!d->Q || !d->b || !d->lb || !d->ub || !d->x) return fail(FCCQP_E_INVALID, "null Q/b/lb/ub/x");
  if (d->m > 0 && (!d->A_eq || !d->b_eq)) return fail(FCCQP_E_INVALID, "null A_eq/b_eq with m > 0");
  if (d->nc > 0 && !d->friction_coeffs) return fail(FCCQP_E_INVALID, "null friction_coeffs with nc > 0");
  if (d->warm_start && (!d->mu_x || (d->nc > 0 && !d->mu_lambda_c)))
    return fail(FCCQP_E_INVALID, "warm_start needs mu_x and mu_lambda_c");
  if (d->warm_lanes && (!d->mu_x || (d->nc > 0 && !d->mu_lambda_c)))
    return fail(FCCQP_E_INVALID, "warm_lanes needs mu_x and mu_lambda_c");
  return FCCQP_OK;
}

// A host-memory per-lane rho array is checked before anything runs (a device one lane by lane in the kernels).
static int validate_rho(const fccqp_batch_desc* d, const double* rho) {
  if (!rho || d->memory_space != FCCQP_MEM_HOST) return FCCQP_OK;
  for (int i = 0; i < d->batch; ++i)
    if (!(rho[i] > 0.0 && std::isfinite(rho[i])))
      return fail(FCCQP_E_INVALID, "rho[%d] = %g: every per-lane rho must be finite and > 0", i, rho[i]);
  return FCCQP_OK;
}

int fccqp_batch_solve(const fccqp_batch_desc* desc) { return fccqp_batch_solve_rho(desc, nullptr); }

int fccqp_batch_solve_rho(const fccqp_batch_desc* desc, double* rho) {
  int rc = validate_desc(desc);
  if (!rc) rc = validate_rho(desc, rho);
  if (rc) return rc;
  const fccqp_batch_desc& d = *desc;
  DeviceCtx* ctx = nullptr;
  rc = get_ctx(d.device, &ctx);
  if (rc) return rc;
  if (d.batch == 0) { if (d.device_seconds) *d.device_seconds = 0.0; return FCCQP_OK; }
  CUDA_TRY(cudaSetDevice(d.device));
  const int n = d.n, m = d.m, nc = d.nc, B = d.batch;

  if (d.memory_space == FCCQP_MEM_DEVICE) {
    fccqp::SolveParams p = solve_params(B, n, m, nc, d.lambda_c_start, d.options, d.warm_start != 0);
    p.Q = d.Q; p.q_bs = d.q_batch_stride; p.q_rs = d.q_row_stride; p.q_cs = d.q_col_stride;
    p.b = d.b; p.b_bs = d.b_batch_stride;
    p.A = d.A_eq; p.a_bs = d.a_batch_stride; p.a_rs = d.a_row_stride; p.a_cs = d.a_col_stride;
    p.beq = d.b_eq; p.beq_bs = d.beq_batch_stride;
    p.mu = d.friction_coeffs; p.mu_bs = d.mu_batch_stride;
    p.lb = d.lb; p.lb_bs = d.lb_batch_stride;
    p.ub = d.ub; p.ub_bs = d.ub_batch_stride;
    p.x = d.x; p.mu_x = d.mu_x; p.mu_c = d.mu_lambda_c;
    p.n_iter = d.n_iter; p.status = d.status;
    p.res_b = d.res_bounds; p.res_f = d.res_fcone; p.bviol = d.bounds_viol; p.fviol = d.fcone_viol;
    p.rho_lanes = rho;
    cudaStream_t st = (cudaStream_t)d.stream;
    StructHint hint;
    hint.set(d.structure);
    hint.caps[0] = d.struct_caps[0]; hint.caps[1] = d.struct_caps[1]; hint.caps[2] = d.struct_caps[2];
    // timing events are per call: concurrent callers on one device must not share them
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    if (d.device_seconds) {
      CUDA_TRY(cudaEventCreate(&ev0));
      CUDA_TRY(cudaEventCreate(&ev1));
      CUDA_TRY(cudaEventRecord(ev0, st));
    }
    rc = launch_solve(*ctx, p, st, d.precision, hint, d.warm_lanes);
    if (rc) { if (ev0) { cudaEventDestroy(ev0); cudaEventDestroy(ev1); } return rc; }
    if (d.device_seconds) {
      float ms = 0.f;
      cudaError_t e = cudaEventRecord(ev1, st);
      if (e == cudaSuccess) e = cudaEventSynchronize(ev1);
      if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, ev0, ev1);
      cudaEventDestroy(ev0); cudaEventDestroy(ev1);
      if (e != cudaSuccess) return fail(FCCQP_E_CUDA, "event timing failed: %s", cudaGetErrorString(e));
      *d.device_seconds = 1e-3 * ms;
    }
    return FCCQP_OK;
  }

  // ---- host memory: stage through device buffers, chunked over 3 streams so that the
  // H2D copy of chunk c+1 overlaps the solve of chunk c and the D2H of chunk c-1.
  std::lock_guard<std::mutex> lk(ctx->host_mu);  // one host-path call per device at a time
  struct Seg { size_t off; size_t per_qp; bool shared; };
  auto seg = [&](size_t& cur, size_t per_qp, bool shared) {
    Seg s{cur, per_qp, shared};
    cur += align_up((shared ? per_qp : per_qp * (size_t)B) * sizeof(double), 256);
    return s;
  };
  // dense (packed) per-QP sizes on the device
  size_t cur = 0;
  const bool q_shared = d.q_batch_stride == 0, a_shared = d.a_batch_stride == 0;
  const bool b_shared = d.b_batch_stride == 0, beq_shared = d.beq_batch_stride == 0;
  const bool mu_shared = d.mu_batch_stride == 0, lb_shared = d.lb_batch_stride == 0, ub_shared = d.ub_batch_stride == 0;
  // The host path requires each QP's Q / A block to be a dense n*n / m*n slab (either order).
  const bool q_dense = (d.q_row_stride == n && d.q_col_stride == 1) || (d.q_row_stride == 1 && d.q_col_stride == n);
  const bool a_dense = m == 0 || (d.a_row_stride == n && d.a_col_stride == 1) || (d.a_row_stride == 1 && d.a_col_stride == m);
  if (!q_dense || !a_dense) return fail(FCCQP_E_UNSUPPORTED, "host path needs dense per-QP Q and A_eq blocks");
  if ((!q_shared && d.q_batch_stride != (int64_t)n * n) || (!a_shared && m > 0 && d.a_batch_stride != (int64_t)m * n) ||
      (!b_shared && d.b_batch_stride != n) || (!beq_shared && m > 0 && d.beq_batch_stride != m) ||
      (!mu_shared && nc > 0 && d.mu_batch_stride != nc / 3) || (!lb_shared && d.lb_batch_stride != n) ||
      (!ub_shared && d.ub_batch_stride != n))
    return fail(FCCQP_E_UNSUPPORTED, "host path needs densely stacked inputs (batch stride 0 or the per-QP size)");
  Seg sQ = seg(cur, (size_t)n * n, q_shared), sA = seg(cur, (size_t)m * n, a_shared);
  Seg sb = seg(cur, n, b_shared), sbeq = seg(cur, m, beq_shared), smu = seg(cur, nc / 3, mu_shared);
  Seg slb = seg(cur, n, lb_shared), sub = seg(cur, n, ub_shared);
  Seg sx = seg(cur, n, false), smx = seg(cur, n, false), smc = seg(cur, nc, false);
  Seg sres = seg(cur, 4, false);
  Seg sint = seg(cur, 1, false);  // 2 ints per QP packed in one double slot
  const Seg smask{cur, 1, false};  // per-lane warm mask: one byte per QP
  if (d.warm_lanes) cur += align_up((size_t)B, 256);
  const Seg srho{cur, 1, false};   // per-lane rho: in and out
  if (rho) cur += align_up((size_t)B * sizeof(double), 256);
  if (cur > ctx->stage_bytes) {
    if (ctx->stage) CUDA_TRY(cudaFree(ctx->stage));
    ctx->stage = nullptr; ctx->stage_bytes = 0;
    CUDA_TRY(cudaMalloc(&ctx->stage, cur));
    ctx->stage_bytes = cur;
  }
  char* base = ctx->stage;
  auto dp = [&](const Seg& s) { return reinterpret_cast<double*>(base + s.off); };
  int* d_niter = reinterpret_cast<int*>(base + sint.off);
  int* d_status = d_niter + B;

  const auto t0 = std::chrono::steady_clock::now();
  // shared inputs once
  cudaStream_t s0 = ctx->streams[0];
  // problem data are float32 in FCCQP_PRECISION_FP32_DATA (es = 4): half the bytes over PCIe; the staging
  // segments keep their FP64 size, state and outputs are always FP64
  const size_t es = d.precision != FCCQP_PRECISION_FP64 ? sizeof(float) : sizeof(double);
  auto h2d_shared = [&](const Seg& s, const double* src) -> int {
    if (s.shared && s.per_qp && src)
      CUDA_TRY(cudaMemcpyAsync(dp(s), src, s.per_qp * es, cudaMemcpyHostToDevice, s0));
    return FCCQP_OK;
  };
  if ((rc = h2d_shared(sQ, d.Q)) || (rc = h2d_shared(sA, d.A_eq)) || (rc = h2d_shared(sb, d.b)) ||
      (rc = h2d_shared(sbeq, d.b_eq)) || (rc = h2d_shared(smu, d.friction_coeffs)) ||
      (rc = h2d_shared(slb, d.lb)) || (rc = h2d_shared(sub, d.ub)))
    return rc;
  CUDA_TRY(cudaStreamSynchronize(s0));

  // where do the outputs go?  (page-locked destination: direct DMA; pageable: pinned bounce buffer)
  void* outs[10] = {d.x, d.mu_x, d.mu_lambda_c, d.n_iter, d.status, d.res_bounds, d.res_fcone, d.bounds_viol, d.fcone_viol,
                    rho};
  const size_t out_elem[10] = {n * sizeof(double), n * sizeof(double), nc * sizeof(double), sizeof(int), sizeof(int),
                               sizeof(double), sizeof(double), sizeof(double), sizeof(double), sizeof(double)};
  bool out_pinned[10];
  size_t out_off[10], hneed = 0;
  for (int i = 0; i < 10; ++i) {
    out_pinned[i] = true;
    out_off[i] = 0;
    if (!outs[i] || !out_elem[i]) continue;
    cudaPointerAttributes at{};
    const bool pinned = cudaPointerGetAttributes(&at, outs[i]) == cudaSuccess && at.type == cudaMemoryTypeHost;
    cudaGetLastError();
    out_pinned[i] = pinned;
    if (!pinned) { out_off[i] = hneed; hneed += align_up((size_t)B * out_elem[i], 256); }
  }
  if (hneed > ctx->hstage_bytes) {
    if (ctx->hstage) CUDA_TRY(cudaFreeHost(ctx->hstage));
    ctx->hstage = nullptr; ctx->hstage_bytes = 0;
    CUDA_TRY(cudaMallocHost(&ctx->hstage, hneed));
    ctx->hstage_bytes = hneed;
  }
  struct Pending { int chunk; void* dst; const void* src; size_t bytes; };
  std::vector<Pending> pending;

  // structure of the batch, from the host copy of the data (a sample of up to 64 QPs; no device probe,
  // no synchronisation inside the chunk pipeline)
  StructHint hint;
  host_struct_hint(d, &hint);

  int nchunks = (B + 4095) / 4096;
  if (nchunks > 16) nchunks = 16;
  if (nchunks < 1) nchunks = 1;
  for (int c = 0; c < nchunks; ++c) {
    const long long lo = (long long)B * c / nchunks, hi = (long long)B * (c + 1) / nchunks;
    const size_t cnt = (size_t)(hi - lo);
    if (!cnt) continue;
    cudaStream_t st = ctx->streams[c % 3];
    auto h2d = [&](const Seg& s, const void* src, size_t esz) -> int {
      if (!s.shared && s.per_qp && src)
        CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(dp(s)) + (size_t)lo * s.per_qp * esz,
                                 static_cast<const char*>(src) + (size_t)lo * s.per_qp * esz, cnt * s.per_qp * esz,
                                 cudaMemcpyHostToDevice, st));
      return FCCQP_OK;
    };
    if ((rc = h2d(sQ, d.Q, es)) || (rc = h2d(sA, d.A_eq, es)) || (rc = h2d(sb, d.b, es)) || (rc = h2d(sbeq, d.b_eq, es)) ||
        (rc = h2d(smu, d.friction_coeffs, es)) || (rc = h2d(slb, d.lb, es)) || (rc = h2d(sub, d.ub, es)))
      return rc;
    if (d.warm_start || d.warm_lanes) {
      if ((rc = h2d(sx, d.x, 8)) || (rc = h2d(smx, d.mu_x, 8)) || (rc = h2d(smc, d.mu_lambda_c, 8))) return rc;
    }
    if (d.warm_lanes && (rc = h2d(smask, d.warm_lanes, 1))) return rc;
    if (rho && (rc = h2d(srho, rho, sizeof(double)))) return rc;
    fccqp::SolveParams p = solve_params((int)cnt, n, m, nc, d.lambda_c_start, d.options, d.warm_start != 0);
    auto off = [&](const Seg& s) { return s.shared ? dp(s) : dp(s) + lo * s.per_qp; };
    auto offi = [&](const Seg& s) {   // problem data: element size es
      return s.shared ? dp(s) : reinterpret_cast<double*>(reinterpret_cast<char*>(dp(s)) + (size_t)lo * s.per_qp * es);
    };
    p.Q = offi(sQ); p.q_bs = q_shared ? 0 : (long long)n * n; p.q_rs = d.q_row_stride; p.q_cs = d.q_col_stride;
    p.A = offi(sA); p.a_bs = a_shared ? 0 : (long long)m * n; p.a_rs = d.a_row_stride; p.a_cs = d.a_col_stride;
    p.b = offi(sb); p.b_bs = b_shared ? 0 : n;
    p.beq = offi(sbeq); p.beq_bs = beq_shared ? 0 : m;
    p.mu = offi(smu); p.mu_bs = mu_shared ? 0 : nc / 3;
    p.lb = offi(slb); p.lb_bs = lb_shared ? 0 : n;
    p.ub = offi(sub); p.ub_bs = ub_shared ? 0 : n;
    p.x = off(sx); p.mu_x = off(smx); p.mu_c = off(smc);
    p.n_iter = d_niter + lo; p.status = d_status + lo;
    double* res = dp(sres);
    p.res_b = res + lo; p.res_f = res + (size_t)B + lo; p.bviol = res + 2 * (size_t)B + lo; p.fviol = res + 3 * (size_t)B + lo;
    p.rho_lanes = rho ? dp(srho) + lo : nullptr;
    rc = launch_solve(*ctx, p, st, d.precision, hint,
                      d.warm_lanes ? reinterpret_cast<const uint8_t*>(base + smask.off) + lo : nullptr);
    if (rc) return rc;
    // D2H: straight into the caller's buffer when it is page-locked (a true asynchronous DMA);
    // otherwise into the pinned bounce buffer, copied out below once the chunk's event has fired
    // (a cudaMemcpyAsync into pageable memory would block the host and serialise the chunks).
    auto d2h = [&](int slot, void* dst, const void* src, size_t elem_bytes) -> int {
      if (!dst || !cnt) return FCCQP_OK;
      const size_t bytes = cnt * elem_bytes;
      void* to = (char*)dst + (size_t)lo * elem_bytes;
      if (!out_pinned[slot]) {
        to = ctx->hstage + out_off[slot] + (size_t)lo * elem_bytes;
        pending.push_back({c, (char*)dst + (size_t)lo * elem_bytes, to, bytes});
      }
      CUDA_TRY(cudaMemcpyAsync(to, src, bytes, cudaMemcpyDeviceToHost, st));
      return FCCQP_OK;
    };
    if ((rc = d2h(0, d.x, p.x, n * sizeof(double))) ||
        (rc = d2h(1, d.mu_x, p.mu_x, n * sizeof(double))) ||
        (rc = d2h(2, d.mu_lambda_c, p.mu_c, nc * sizeof(double))) ||
        (rc = d2h(3, d.n_iter, p.n_iter, sizeof(int))) ||
        (rc = d2h(4, d.status, p.status, sizeof(int))) ||
        (rc = d2h(5, d.res_bounds, p.res_b, sizeof(double))) ||
        (rc = d2h(6, d.res_fcone, p.res_f, sizeof(double))) ||
        (rc = d2h(7, d.bounds_viol, p.bviol, sizeof(double))) ||
        (rc = d2h(8, d.fcone_viol, p.fviol, sizeof(double))) ||
        (rc = d2h(9, rho, p.rho_lanes, sizeof(double))))
      return rc;
    CUDA_TRY(cudaEventRecord(ctx->chunk_ev[c], st));
  }
  // drain the bounce buffer chunk by chunk while later chunks are still in flight
  {
    int waited = -1;
    for (const Pending& pe : pending) {
      if (pe.chunk != waited) { CUDA_TRY(cudaEventSynchronize(ctx->chunk_ev[pe.chunk])); waited = pe.chunk; }
      memcpy(pe.dst, pe.src, pe.bytes);
    }
  }
  for (auto& s : ctx->streams) CUDA_TRY(cudaStreamSynchronize(s));
  if (d.device_seconds)
    *d.device_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  return FCCQP_OK;
}

// One call, several devices (SURVEY 8e: "one host thread + stream set per device, host-side scatter and gather").
// The batch shards trivially -- QPs are independent, there is no exchange step -- so device r of W takes the
// contiguous range [B r / W, B (r+1) / W) of every stacked array (shared arrays, batch stride 0, go to every device)
// and runs the single-device host path on its own host thread: staging buffers, streams, H2D / solve / D2H
// pipeline and structure classification are per device.
int fccqp_batch_solve_multi(const fccqp_batch_desc* desc, const int32_t* devices, int32_t n_devices) {
  return fccqp_batch_solve_multi_rho(desc, nullptr, devices, n_devices);
}

int fccqp_batch_solve_multi_rho(const fccqp_batch_desc* desc, double* rho, const int32_t* devices, int32_t n_devices) {
  int rc = validate_desc(desc);
  if (!rc) rc = validate_rho(desc, rho);
  if (rc) return rc;
  if (!devices || n_devices < 1) return fail(FCCQP_E_INVALID, "devices / n_devices");
  if (desc->memory_space != FCCQP_MEM_HOST)
    return fail(FCCQP_E_UNSUPPORTED, "fccqp_batch_solve_multi takes host memory (device pointers live on ONE device: call fccqp_batch_solve per device)");
  for (int i = 0; i < n_devices; ++i)
    for (int j = 0; j < i; ++j)
      if (devices[i] == devices[j]) return fail(FCCQP_E_INVALID, "device %d listed twice", devices[i]);
  for (int i = 0; i < n_devices; ++i) {
    DeviceCtx* ctx = nullptr;
    if ((rc = get_ctx(devices[i], &ctx))) return rc;
  }
  const fccqp_batch_desc& d = *desc;
  const auto t0 = std::chrono::steady_clock::now();
  const int W = n_devices;
  std::vector<int> rcs(W, FCCQP_OK);
  std::vector<std::string> errs(W);
  // Dynamic split: the batch is cut into slabs and every device thread pulls the next slab when it is done with its
  // own, so a device behind a slower or shared PCIe link simply takes fewer of them (measured on an 8-GPU box:
  // 24 GB/s for GPUs 0-3 against 46-56 GB/s for GPUs 4-7 under load, profiles/r02_h2d_scaling_8gpu.log).  Results do
  // not depend on which device solved a QP.
  // Guided sizes: a slab is half of an equal share of what is LEFT (multiples of the 4096-QP chunk, at least two chunks):
  // few, large slabs while there is plenty of work -- every slab pays one pipeline fill and drain, ~1 ms -- and small
  // ones at the end, so that the slowest device finishes at most one small slab after the others.
  const long long Btot = d.batch;
  auto slab_at = [&](long long lo) -> long long {
    if (W == 1) return Btot - lo;
    long long sz = ((Btot - lo) / (2LL * W) + 4095) / 4096 * 4096;
    if (sz < 8192) sz = 8192;
    return sz < Btot - lo ? sz : Btot - lo;
  };
  // (the structure bounds are worked out once, from a sample of the whole batch, and handed to every slab)
  StructHint mh;
  host_struct_hint(d, &mh);
  std::atomic<long long> next{0};
  auto run_range = [&](int r, long long lo, long long hi) -> int {
    fccqp_batch_desc s = d;
    s.device = devices[r];
    s.batch = (int32_t)(hi - lo);
    s.device_seconds = nullptr;
    s.structure = mh.mode | (mh.refine ? FCCQP_STRUCTURE_REFINE : 0);
    s.struct_caps[0] = mh.caps[0]; s.struct_caps[1] = mh.caps[1]; s.struct_caps[2] = mh.caps[2];
    const size_t es = d.precision != FCCQP_PRECISION_FP64 ? sizeof(float) : sizeof(double);
    auto adv = [&](const double* p, int64_t stride) -> const double* {   // problem data: element size es
      return p ? reinterpret_cast<const double*>(reinterpret_cast<const char*>(p) + (size_t)lo * (size_t)stride * es) : p;
    };
    s.Q = adv(d.Q, d.q_batch_stride); s.b = adv(d.b, d.b_batch_stride); s.A_eq = adv(d.A_eq, d.a_batch_stride);
    s.b_eq = adv(d.b_eq, d.beq_batch_stride); s.friction_coeffs = adv(d.friction_coeffs, d.mu_batch_stride);
    s.lb = adv(d.lb, d.lb_batch_stride); s.ub = adv(d.ub, d.ub_batch_stride);
    if (d.x) s.x = d.x + lo * d.n;
    if (d.mu_x) s.mu_x = d.mu_x + lo * d.n;
    if (d.mu_lambda_c) s.mu_lambda_c = d.mu_lambda_c + lo * d.nc;
    if (d.warm_lanes) s.warm_lanes = d.warm_lanes + lo;
    if (d.n_iter) s.n_iter = d.n_iter + lo;
    if (d.status) s.status = d.status + lo;
    if (d.res_bounds) s.res_bounds = d.res_bounds + lo;
    if (d.res_fcone) s.res_fcone = d.res_fcone + lo;
    if (d.bounds_viol) s.bounds_viol = d.bounds_viol + lo;
    if (d.fcone_viol) s.fcone_viol = d.fcone_viol + lo;
    return fccqp_batch_solve_rho(&s, rho ? rho + lo : nullptr);
  };
  auto shard = [&](int r) {
    for (;;) {
      long long lo = next.load();
      long long sz = 0;
      do {
        if (lo >= Btot) return;
        sz = slab_at(lo);
      } while (!next.compare_exchange_weak(lo, lo + sz));
      const long long hi = lo + sz;
      rcs[r] = run_range(r, lo, hi);
      if (rcs[r]) { errs[r] = g_err; return; }   // (thread-local: carried back to the caller's thread below)
    }
  };
  if (W == 1) shard(0);
  else {
    std::vector<std::thread> th;
    th.reserve(W);
    for (int r = 0; r < W; ++r) th.emplace_back(shard, r);
    for (auto& t : th) t.join();
  }
  for (int r = 0; r < W; ++r)
    if (rcs[r]) return fail(rcs[r], "device %d: %s", devices[r], errs[r].c_str());
  if (d.device_seconds)
    *d.device_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  return FCCQP_OK;
}

int fccqp_wbc_assemble(const fccqp_wbc_desc* d) {
  if (!d) return fail(FCCQP_E_INVALID, "desc is null");
  if (d->abi_version != FCCQP_ABI_VERSION) return fail(FCCQP_E_INVALID, "abi_version %d != %d", d->abi_version, FCCQP_ABI_VERSION);
  if (d->batch < 0 || d->nv < 1 || d->nu < 0 || d->nu > d->nv || d->nh < 0 || d->nc < 0 || d->ny < 0)
    return fail(FCCQP_E_INVALID, "bad WBC dimensions (need nv >= 1, 0 <= nu <= nv, nh, nc, ny >= 0)");
  if (d->nc % 3 != 0) return fail(FCCQP_E_INVALID, "nc = %d must be a multiple of 3 (src/fcc_qp.cpp:32)", d->nc);
  DeviceCtx* ctx = nullptr;
  int rc = get_ctx(d->device, &ctx);
  if (rc) return rc;
  if (d->batch == 0) return FCCQP_OK;
  if (!d->M || !d->bias || !d->Q || !d->b || !d->A_eq || !d->b_eq || (d->nh > 0 && (!d->Jh || !d->gamma_h)) ||
      (d->nc > 0 && (!d->Jc || !d->gamma_c)) || (d->ny > 0 && (!d->Jy || !d->W || !d->ydd_cmd)))
    return fail(FCCQP_E_INVALID, "null WBC input/output pointer");
  CUDA_TRY(cudaSetDevice(d->device));
  fccqp::WbcParams p{};
  p.B = d->batch; p.nv = d->nv; p.nu = d->nu; p.nh = d->nh; p.nc = d->nc; p.ny = d->ny;
  p.w_vdot = d->w_vdot; p.w_u = d->w_u; p.w_lc = d->w_lambda_c; p.w_eps = d->w_eps;
  p.M = d->M; p.M_bs = d->M_batch_stride; p.Jh = d->Jh; p.Jh_bs = d->Jh_batch_stride;
  p.Jc = d->Jc; p.Jc_bs = d->Jc_batch_stride; p.Jy = d->Jy; p.Jy_bs = d->Jy_batch_stride;
  p.W = d->W; p.W_bs = d->W_batch_stride; p.ydd = d->ydd_cmd; p.ydd_bs = d->ydd_batch_stride;
  p.bias = d->bias; p.bias_bs = d->bias_batch_stride; p.gh = d->gamma_h; p.gh_bs = d->gh_batch_stride;
  p.gc = d->gamma_c; p.gc_bs = d->gc_batch_stride;
  p.Q = d->Q; p.b = d->b; p.A = d->A_eq; p.beq = d->b_eq;
  const size_t smem = sizeof(double) * ((size_t)d->ny * d->nv + d->ny + (size_t)d->nv * d->nv);
  if (smem > (size_t)ctx->max_smem_optin) return fail(FCCQP_E_UNSUPPORTED, "WBC terms need %zu B of shared memory", smem);
  static std::mutex attr_mu;
  {
    std::lock_guard<std::mutex> lk(attr_mu);
    CUDA_TRY(cudaFuncSetAttribute(fccqp::wbc_assemble_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->max_smem_optin));
  }
  int grid = ctx->num_sms * 8;
  if (grid > d->batch) grid = d->batch;
  fccqp::wbc_assemble_kernel<<<grid, 256, smem, (cudaStream_t)d->stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return FCCQP_OK;
}

namespace {
int polish_params(const fccqp_polish_desc* d, fccqp::PolishParams* out, DeviceCtx** ctx, bool finish) {
  if (!d) return fail(FCCQP_E_INVALID, "desc is null");
  if (d->abi_version != FCCQP_ABI_VERSION) return fail(FCCQP_E_INVALID, "abi_version %d != %d", d->abi_version, FCCQP_ABI_VERSION);
  int rc = check_dims(d->n, d->m, d->nc, d->lambda_c_start);
  if (rc) return rc;
  if (d->batch < 0) return fail(FCCQP_E_INVALID, "batch < 0");
  if ((rc = get_ctx(d->device, ctx))) return rc;
  if (d->batch == 0) return FCCQP_OK;
  if (!d->lb || !d->ub || !d->rot || (d->nc > 0 && !d->friction_coeffs))
    return fail(FCCQP_E_INVALID, "null polish pointer (lb, ub, rot, friction_coeffs)");
  if (!finish && (!d->Q || !d->b || (d->m > 0 && (!d->A_eq || !d->b_eq)) || !d->x || !d->mu_x || (d->nc > 0 && !d->mu_lambda_c) ||
                  !d->Qp || !d->bp || (d->m > 0 && (!d->Ap || !d->beqp))))
    return fail(FCCQP_E_INVALID, "null polish pointer (prepare needs the QP, x, mu_x, mu_lambda_c, Qp, bp, Ap, beqp)");
  if (finish && (!d->Q || !d->b || (d->m > 0 && (!d->A_eq || !d->b_eq)) || !d->y || !d->y_status || !d->z || !d->bounds_viol || !d->fcone_viol || !d->polished))
    return fail(FCCQP_E_INVALID, "null polish pointer (finish needs Q, b, A_eq, b_eq, y, y_status, z, bounds_viol, fcone_viol, polished)");
  fccqp::PolishParams p{};
  p.B = d->batch; p.n = d->n; p.m = d->m; p.nc = d->nc; p.lcs = d->lambda_c_start;
  p.eps_fcone = d->eps_fcone; p.eps_bound = d->eps_bound; p.eps_objective = d->eps_objective;
  p.Q = d->Q; p.q_bs = d->q_batch_stride; p.b = d->b; p.b_bs = d->b_batch_stride;
  p.A = d->A_eq; p.a_bs = d->a_batch_stride; p.beq = d->b_eq; p.beq_bs = d->beq_batch_stride;
  p.mu = d->friction_coeffs; p.mu_bs = d->mu_batch_stride;
  p.lb = d->lb; p.lb_bs = d->lb_batch_stride; p.ub = d->ub; p.ub_bs = d->ub_batch_stride;
  p.x = d->x; p.mu_x = d->mu_x; p.mu_c = d->mu_lambda_c;
  p.Qp = d->Qp; p.bp = d->bp; p.Ap = d->Ap; p.beqp = d->beqp; p.rot = d->rot;
  p.y = d->y; p.y_status = d->y_status; p.z = d->z; p.bviol = d->bounds_viol; p.fviol = d->fcone_viol; p.polished = d->polished;
  *out = p;
  return FCCQP_OK;
}
}  // namespace

int fccqp_polish_prepare(const fccqp_polish_desc* d) {
  fccqp::PolishParams p{};
  DeviceCtx* ctx = nullptr;
  int rc = polish_params(d, &p, &ctx, false);
  if (rc || d->batch == 0) return rc;
  CUDA_TRY(cudaSetDevice(d->device));
  const size_t smem = (size_t)d->n * (5 * sizeof(double) + 3 * sizeof(int));
  int grid = ctx->num_sms * 8;
  if (grid > d->batch) grid = d->batch;
  fccqp::polish_prepare_kernel<<<grid, 128, smem, (cudaStream_t)d->stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return FCCQP_OK;
}

int fccqp_polish_finish(const fccqp_polish_desc* d) {
  fccqp::PolishParams p{};
  DeviceCtx* ctx = nullptr;
  int rc = polish_params(d, &p, &ctx, true);
  if (rc || d->batch == 0) return rc;
  CUDA_TRY(cudaSetDevice(d->device));
  int grid = (d->batch + 3) / 4;
  if (grid > ctx->num_sms * 16) grid = ctx->num_sms * 16;
  fccqp::polish_finish_kernel<<<grid, 128, (size_t)4 * 2 * d->n * sizeof(double), (cudaStream_t)d->stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return FCCQP_OK;
}

int fccqp_alloc_pinned(size_t bytes, void** out) {
  if (!out) return fail(FCCQP_E_INVALID, "out is null");
  *out = nullptr;
  if (bytes == 0) return FCCQP_OK;
  CUDA_TRY(cudaMallocHost(out, bytes));
  return FCCQP_OK;
}
int fccqp_free_pinned(void* ptr) {
  if (ptr) CUDA_TRY(cudaFreeHost(ptr));
  return FCCQP_OK;
}

int fccqp_release_workspaces(void) {
  std::lock_guard<std::mutex> lk(g_ctx_mu);
  for (auto& kv : g_ctx) {
    DeviceCtx& c = *kv.second;
    std::lock_guard<std::mutex> lk2(c.host_mu);
    std::lock_guard<std::mutex> lk3(c.mu);
    cudaSetDevice(c.device);
    if (c.stage) { cudaFree(c.stage); c.stage = nullptr; c.stage_bytes = 0; }
    if (c.hstage) { cudaFreeHost(c.hstage); c.hstage = nullptr; c.hstage_bytes = 0; }
  }
  return FCCQP_OK;
}

}  // extern "C"
