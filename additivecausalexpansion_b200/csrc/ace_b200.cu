// ace_b200.cu -- C ABI (include/ace_b200.h) of the B200-native ACE hot path: device-resident fit
// handle + per-function entry points.  Host code here only sequences kernels; all arithmetic of the
// path runs in the hand-written sm_100a kernels of dgemm_nt.cuh / chol.cuh / gp_kernels.cuh /
// pred_kernels.cuh.  No cuBLAS / cuSOLVER, no CPU fallback.
#include "../../include/ace_b200.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "chol.cuh"
#include "nccl_dyn.h"
#include "shard_dense.cuh"
#include "gp_kernels.cuh"
#include "pair_kernels.cuh"
#include "grad2_kernel.cuh"
#include "grad3_kernel.cuh"
#include "kernmat2_kernel.cuh"
#include "pred_kernels.cuh"
#include "prep_kernels.cuh"

namespace ace {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }

static int usage(const std::string& m) {
  set_error(m);
  return ACE_ERR_USAGE;
}

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// ---------------------------------------------------------------------------------------------
// small RAII device buffer
// ---------------------------------------------------------------------------------------------
template <typename T>
struct DBuf {
  T* p = nullptr;
  size_t count = 0;
  DBuf() = default;
  DBuf(const DBuf&) = delete;
  DBuf& operator=(const DBuf&) = delete;
  ~DBuf() { release(); }
  int alloc(size_t n) {
    release();
    if (n == 0) n = 1;
    cudaError_t e = cudaMalloc(&p, n * sizeof(T));
    if (e != cudaSuccess) {
      p = nullptr;
      set_error(std::string("cudaMalloc of ") + std::to_string(n * sizeof(T)) + " bytes: " + cudaGetErrorString(e));
      return -(int)e - 1000;
    }
    count = n;
    return 0;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    count = 0;
  }
};

static int check_device() {
  int cnt = 0;
  cudaError_t e = cudaGetDeviceCount(&cnt);
  if (e != cudaSuccess || cnt <= 0) {
    set_error(std::string("no CUDA device available (") + cudaGetErrorString(e) +
              "); this library has no CPU fallback");
    return ACE_ERR_NO_DEVICE;
  }
  return 0;
}

static int configure_kernels_once() {
  // per device: opt in to large dynamic shared memory for every kernel that needs it
  static std::mutex mu;
  static std::vector<int> done;
  int dev = 0;
  ACE_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(mu);
  if (std::find(done.begin(), done.end(), dev) != done.end()) return 0;
  ACE_TRY(configure_dense_kernels());
  done.push_back(dev);
  return 0;
}

// host (ld = rows) -> device (ld = ld_dev), zero padded
static int upload_matrix(double* dst, long ld_dev, int rows_pad, const double* src, int rows, int cols,
                         cudaStream_t st) {
  ACE_CUDA(cudaMemsetAsync(dst, 0, sizeof(double) * (size_t)ld_dev * (size_t)std::max(cols, 1), st));
  (void)rows_pad;
  if (rows > 0 && cols > 0)
    ACE_CUDA(cudaMemcpy2DAsync(dst, sizeof(double) * ld_dev, src, sizeof(double) * rows, sizeof(double) * rows,
                               cols, cudaMemcpyHostToDevice, st));
  return 0;
}

static int download_matrix(double* dst, int rows, int cols, const double* src, long ld_dev, cudaStream_t st) {
  if (rows > 0 && cols > 0)
    ACE_CUDA(cudaMemcpy2DAsync(dst, sizeof(double) * rows, src, sizeof(double) * ld_dev, sizeof(double) * rows,
                               cols, cudaMemcpyDeviceToHost, st));
  return 0;
}

__global__ void pad_identity_kernel(double* A, long ld, int n, int n_pad) {
  // rows/cols >= n of a freshly uploaded (zero padded) matrix become an identity block
  const int i = n + blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_pad) A[i + (size_t)i * ld] = 1.0;
}

__global__ void add_diag_kernel(double* A, long ld, int n, double v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) A[i + (size_t)i * ld] += v;
}

__global__ void synth_spd_kernel(double* A, long ld, int n) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)n * n) return;
  const int i = (int)(idx % n), j = (int)(idx / n);
  const double t = 8.0 * (double)(i - j) / (double)n;
  A[i + (size_t)j * ld] = exp(-t * t) + (i == j ? 0.5 : 0.0);
}

// ---------------------------------------------------------------------------------------------
// kernel dispatch
// ---------------------------------------------------------------------------------------------
// The exact-shape pair kernels (grad3_kernel.cuh, kernmat2_kernel.cuh) read lambda_b and the length-scale weights from
// a __constant__ table, one per module: [wait for the previous user's kernel] -> copy -> kernel -> [record], enqueued
// under a per-device lock, serialises the launches of different fit handles that use the same table on one device (all
// other work of the handles still overlaps).  Inside a stream capture the wait / record become external event nodes,
// so graph replays of different handles are ordered the same way.
struct ConstChain {
  std::mutex mu;
  cudaEvent_t ev = nullptr;
  bool recorded = false;
};
static ConstChain& const_chain(int which, int dev) {
  static ConstChain chains[2][64];
  return chains[which][dev & 63];
}
template <class F>
static int with_const_chain(int which, cudaStream_t st, F&& launch) {
  int dev = 0;
  ACE_CUDA(cudaGetDevice(&dev));
  ConstChain& ch = const_chain(which, dev);
  std::lock_guard<std::mutex> lk(ch.mu);
  if (ch.ev == nullptr) ACE_CUDA(cudaEventCreateWithFlags(&ch.ev, cudaEventDisableTiming));
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  ACE_CUDA(cudaStreamIsCapturing(st, &cs));
  const bool cap = cs != cudaStreamCaptureStatusNone;
  if (ch.recorded) ACE_CUDA(cudaStreamWaitEvent(st, ch.ev, cap ? cudaEventWaitExternal : cudaEventWaitDefault));
  ACE_TRY(launch());
  ACE_CUDA(cudaEventRecordWithFlags(ch.ev, st, cap ? cudaEventRecordExternal : cudaEventRecordDefault));
  ch.recorded = true;
  return 0;
}

// launchers exported by the pair_kernmat2.cu objects (one per kernel kind)
int launch_kernmat2_k0(const KernArgs&, unsigned, size_t, cudaStream_t);
int launch_kernmat2_k1(const KernArgs&, unsigned, size_t, cudaStream_t);

// launchers exported by the pair_widep.cu object (p > PMAX: dimensions streamed through shared memory)
int launch_kernmat_wide(const KernArgs&, int, unsigned, cudaStream_t);
int grad_wide_slab(int B, int kind);
int launch_grad_wide(const GradArgs&, int, int, int, cudaStream_t);

// Which kernel builds K for a (p, B, symmetric) shape.  launch_kernmat launches what this selects, and
// ace_dbg_kernel_plan reports it, so that tests can check which kernel a shape runs.
struct BuildPlan {
  enum { GENERIC, EXACT, WIDE } family = GENERIC;  // kernmat_kernel, kernmat2_kernel, kernmat_wide_kernel
  int bc = 0;       // kernmat_kernel: terms per chunk (4, 8 or 12)
  size_t smem = 0;  // dynamic shared memory (not used by the wide kernel)
};

static int plan_kernmat(int p, int B, int sym, BuildPlan* bp) {
  if (B < 1 || B > BMAXT || p < 1) {
    set_error("kernel build supports p >= 1 and B = Bz+1 <= 32");
    return ACE_ERR_UNSUPPORTED;
  }
  if (p > PMAX) {
    bp->family = BuildPlan::WIDE;
    return 0;
  }
  bp->smem = kb::smem_bytes(p, B - 1, sym != 0);
  if (bp->smem > 227 * 1024) {
    set_error("kernel build: p and Bz too large for one shared-memory tile");
    return ACE_ERR_UNSUPPORTED;
  }
  // kernmat2_kernel: exact number of terms, weights in constant memory, lock-step sqrt / exp (B <= 16, p <= 32).
  // ACE_KERNMAT_IMPL is read once per process.
  static const int impl = [] {
    const char* e = std::getenv("ACE_KERNMAT_IMPL");
    return e ? std::atoi(e) : 2;
  }();
  if (impl == 2 && B <= G3_LAM && p <= G3_PD) {
    bp->family = BuildPlan::EXACT;
    bp->smem = kb2::smem_bytes(p, B - 1, sym != 0);
    return 0;
  }
  bp->bc = kb::chunk_terms(B);  // terms per chunk x columns per step: 16 or 24 accumulators per thread
  return 0;
}

static int launch_kernmat(const KernArgs& a, int kind, cudaStream_t st) {
  BuildPlan bp;
  ACE_TRY(plan_kernmat(a.p, a.B, a.sym, &bp));
  unsigned grid;
  if (a.sym) {
    const long T = a.n1_pad / kb::T;
    grid = (unsigned)(T * (T + 1) / 2);
  } else {
    grid = (unsigned)((a.n1_pad / kb::T) * (a.n2_pad / kb::T));
  }
  if (bp.family == BuildPlan::WIDE) return launch_kernmat_wide(a, kind, grid, st);
  if (bp.family == BuildPlan::EXACT) {
    return with_const_chain(1, st, [&]() -> int {
      return kind == 0 ? launch_kernmat2_k0(a, grid, bp.smem, st) : launch_kernmat2_k1(a, grid, bp.smem, st);
    });
  }
  const size_t smem = bp.smem;
  auto go = [&](auto kern) -> int {
    ACE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, 256, smem, st>>>(a);
    return 0;
  };
  const int bc = bp.bc;
  if (kind == 0) {
    if (bc == 4) ACE_TRY(go(kernmat_kernel<0, 4, 4>));
    else if (bc == 8) ACE_TRY(go(kernmat_kernel<0, 8, 2>));
    else ACE_TRY(go(kernmat_kernel<0, 12, 2>));
  } else {
    if (bc == 4) ACE_TRY(go(kernmat_kernel<1, 4, 4>));
    else if (bc == 8) ACE_TRY(go(kernmat_kernel<1, 8, 2>));
    else ACE_TRY(go(kernmat_kernel<1, 12, 2>));
  }
  ACE_CUDA(cudaGetLastError());
  return 0;
}

struct GradPlan {
  int PD = 0, BT = 0, groups = 0, gy = 0, threads = 0, gx = 0;
  size_t smem = 0;
  int v2 = 0, PD8 = 0, BD8 = 0;  // second-generation kernel (grad2_kernel.cuh) when the shape is instantiated
  int nw2 = 8;                   // its warps per CTA: 8 (<= 255 registers) or 16 (128 registers)
  int cw3 = 1;                   // grad3: weights in __constant__ memory (0: shared memory; ACE_GRAD3_CW)
  int v3 = 0, NT3 = 0;           // third-generation kernel (grad3_kernel.cuh, exact-shape instantiations in pair_grad3.cu)
  int wide_sw = 0;               // p > PMAX: grad_wide_kernel (widep_kernels.cuh) with slabs of this many columns
};

// launchers exported by the pair_grad3.cu objects (one per kernel kind and p tile count)
int launch_grad3_k0_nt1(const GradArgs&, int, size_t, int, cudaStream_t);
int launch_grad3_k0_nt2(const GradArgs&, int, size_t, int, cudaStream_t);
int launch_grad3_k0_nt3(const GradArgs&, int, size_t, int, cudaStream_t);
int launch_grad3_k0_nt4(const GradArgs&, int, size_t, int, cudaStream_t);
int launch_grad3_k1_nt1(const GradArgs&, int, size_t, int, cudaStream_t);
int launch_grad3_k1_nt2(const GradArgs&, int, size_t, int, cudaStream_t);
int launch_grad3_k1_nt3(const GradArgs&, int, size_t, int, cudaStream_t);
int launch_grad3_k1_nt4(const GradArgs&, int, size_t, int, cudaStream_t);

static int plan_grad(int p, int B, int kind, int sms, GradPlan* pl) {
  if (p > PMAX && B <= BMAXT) {
    pl->wide_sw = grad_wide_slab(B, kind);
    if (pl->wide_sw == 0) {
      set_error("gradient pass: Bz too large for one shared-memory stage");
      return ACE_ERR_UNSUPPORTED;
    }
    pl->gx = sms; pl->gy = 1;
    return 0;
  }
  static const int table[][2] = {{4, 16}, {8, 8}, {12, 5}, {16, 4}, {20, 3}, {24, 2}, {32, 2}, {48, 1}, {64, 1}};
  for (auto& t : table) {
    if (p <= t[0]) {
      pl->PD = t[0];
      pl->BT = t[1];
      break;
    }
  }
  if (pl->PD == 0 || B > BMAXT) {
    set_error("gradient pass supports B = Bz+1 <= 32");
    return ACE_ERR_UNSUPPORTED;
  }
  int gpc_max = gk::GROUPS_PER_CTA;
  if (pl->PD == 20) {  // tuning knobs for the headline shape (p <= 20): terms per thread, b-groups per CTA
    if (const char* e = std::getenv("ACE_GRAD_BT")) pl->BT = (std::atoi(e) == 2) ? 2 : 3;
  }
  if (const char* e = std::getenv("ACE_GRAD_GPC")) gpc_max = std::max(1, std::min(4, std::atoi(e)));
  pl->groups = (B + pl->BT - 1) / pl->BT;
  const int gpc = std::min(pl->groups, gpc_max);
  pl->gy = (pl->groups + gpc - 1) / gpc;
  pl->threads = 64 * gpc;
  pl->smem = gk::smem_bytes(pl->PD, B - 1, pl->BT, kind);
  if (pl->smem > 227 * 1024) {
    set_error("gradient pass: p and Bz too large for one shared-memory tile");
    return ACE_ERR_UNSUPPORTED;
  }
  pl->gx = 2 * sms;
  // grad2_kernel: one thread per pair for all terms, length-scale sums on the tensor pipe
  const int PD8 = (p + 7) / 8 * 8, BD8 = (B + 7) / 8 * 8;
  const char* impl = std::getenv("ACE_GRAD_IMPL");
  // measured (profiles/r02/grad_sweep2.log, gemv + gradient + finalize phase, ms): with 16 warps per CTA at 128
  // registers grad2 wins at every BASELINE shape -- C3 (n=8192) 4.91 -> 4.51, C2 0.90 -> 0.61, C5 1.68 -> 1.33,
  // C4 (n=8192) 2.27 -> 1.23; with 8 warps (<= 255 registers) it only won for p <= 16 (profiles/r01)
  const int want = impl ? std::atoi(impl) : 3;
  const bool want2 = want >= 2;
  // grad3_kernel: the same decomposition with the exact number of terms compiled in and lock-step exp / sqrt / rcp
  if (want == 3 && p <= 32 && B <= 16) {
    const int NT = (p + 7) / 8;
    const size_t sm3 = g3::smem_bytes(NT, B, kind, 16);
    if (sm3 <= 227 * 1024) {
      pl->v3 = 1; pl->NT3 = NT; pl->smem = sm3; pl->gy = 1; pl->threads = 512;
      if (const char* e = std::getenv("ACE_GRAD3_CW")) pl->cw3 = std::atoi(e) != 0;
      return 0;
    }
  }
  if (PD8 <= 32 && BD8 <= 16 && want2) {
    int nw = 16;
    if (const char* e = std::getenv("ACE_GRAD2_WARPS")) nw = (std::atoi(e) == 8) ? 8 : 16;
    size_t sm2 = g2::smem_bytes(PD8, BD8, B - 1, nw, kind);
    if (sm2 > 227 * 1024 && nw == 16) {
      nw = 8;
      sm2 = g2::smem_bytes(PD8, BD8, B - 1, nw, kind);
    }
    if (sm2 <= 227 * 1024) {
      pl->v2 = 1; pl->PD8 = PD8; pl->BD8 = BD8; pl->smem = sm2; pl->gy = 1; pl->threads = 32 * nw; pl->nw2 = nw;
    }
  }
  return 0;
}

template <int PD8, int BD8, int KIND, int NW>
static int launch_grad2_k(const GradArgs& a, const GradPlan& pl, cudaStream_t st) {
  ACE_CUDA(cudaFuncSetAttribute(grad2_kernel<PD8, BD8, KIND, NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
  grad2_kernel<PD8, BD8, KIND, NW><<<pl.gx, NW * 32, pl.smem, st>>>(a);
  ACE_CUDA(cudaGetLastError());
  return 0;
}

template <int PD8, int BD8>
static int launch_grad2_t(const GradArgs& a, int kind, const GradPlan& pl, cudaStream_t st) {
  if (pl.nw2 == 16) return kind == 0 ? launch_grad2_k<PD8, BD8, 0, 16>(a, pl, st) : launch_grad2_k<PD8, BD8, 1, 16>(a, pl, st);
  return kind == 0 ? launch_grad2_k<PD8, BD8, 0, 8>(a, pl, st) : launch_grad2_k<PD8, BD8, 1, 8>(a, pl, st);
}

static int launch_grad2(const GradArgs& a, int kind, const GradPlan& pl, cudaStream_t st) {
  const int key = pl.PD8 * 100 + pl.BD8;
  switch (key) {
    case 808: return launch_grad2_t<8, 8>(a, kind, pl, st);
    case 816: return launch_grad2_t<8, 16>(a, kind, pl, st);
    case 1608: return launch_grad2_t<16, 8>(a, kind, pl, st);
    case 1616: return launch_grad2_t<16, 16>(a, kind, pl, st);
    case 2408: return launch_grad2_t<24, 8>(a, kind, pl, st);
    case 2416: return launch_grad2_t<24, 16>(a, kind, pl, st);
    case 3208: return launch_grad2_t<32, 8>(a, kind, pl, st);
    default: return launch_grad2_t<32, 16>(a, kind, pl, st);
  }
}

template <int PD, int BT>
static int launch_grad_t(const GradArgs& a, int kind, const GradPlan& pl, cudaStream_t st) {
  dim3 grid(pl.gx, pl.gy);
  if (kind == 0) {
    ACE_CUDA(cudaFuncSetAttribute(grad_kernel<PD, BT, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    grad_kernel<PD, BT, 0><<<grid, pl.threads, pl.smem, st>>>(a);
  } else {
    ACE_CUDA(cudaFuncSetAttribute(grad_kernel<PD, BT, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    grad_kernel<PD, BT, 1><<<grid, pl.threads, pl.smem, st>>>(a);
  }
  ACE_CUDA(cudaGetLastError());
  return 0;
}

static int launch_grad2(const GradArgs& a, int kind, const GradPlan& pl, cudaStream_t st);

static int launch_grad(const GradArgs& a, int kind, const GradPlan& pl, cudaStream_t st) {
  if (pl.wide_sw) return launch_grad_wide(a, kind, pl.wide_sw, pl.gx, st);
  if (pl.v3) {
    auto go = [&](int cw) -> int {
      switch (kind * 10 + pl.NT3) {
        case 1: return launch_grad3_k0_nt1(a, pl.gx, pl.smem, cw, st);
        case 2: return launch_grad3_k0_nt2(a, pl.gx, pl.smem, cw, st);
        case 3: return launch_grad3_k0_nt3(a, pl.gx, pl.smem, cw, st);
        case 4: return launch_grad3_k0_nt4(a, pl.gx, pl.smem, cw, st);
        case 11: return launch_grad3_k1_nt1(a, pl.gx, pl.smem, cw, st);
        case 12: return launch_grad3_k1_nt2(a, pl.gx, pl.smem, cw, st);
        case 13: return launch_grad3_k1_nt3(a, pl.gx, pl.smem, cw, st);
        default: return launch_grad3_k1_nt4(a, pl.gx, pl.smem, cw, st);
      }
    };
    if (!pl.cw3) return go(0);
    return with_const_chain(0, st, [&]() -> int { return go(1); });
  }
  if (pl.v2) return launch_grad2(a, kind, pl, st);
  switch (pl.PD) {
    case 4: return launch_grad_t<4, 16>(a, kind, pl, st);
    case 8: return launch_grad_t<8, 8>(a, kind, pl, st);
    case 12: return launch_grad_t<12, 5>(a, kind, pl, st);
    case 16: return launch_grad_t<16, 4>(a, kind, pl, st);
    case 20: return pl.BT == 2 ? launch_grad_t<20, 2>(a, kind, pl, st) : launch_grad_t<20, 3>(a, kind, pl, st);
    case 24: return launch_grad_t<24, 2>(a, kind, pl, st);
    case 32: return launch_grad_t<32, 2>(a, kind, pl, st);
    case 48: return launch_grad_t<48, 1>(a, kind, pl, st);
    default: return launch_grad_t<64, 1>(a, kind, pl, st);
  }
}

// ---------------------------------------------------------------------------------------------
// Core: everything a GP step needs on one device.  Used by the fit handle and, transiently, by the
// per-function entry points.
// ---------------------------------------------------------------------------------------------
struct Core {
  int device = 0, sms = 148;
  int n = 0, n_pad = 0, p = 0, Bz = 0, B = 0, P = 0, kind = 0;
  cudaStream_t st = nullptr, side = nullptr, aux = nullptr, bgst = nullptr;
  cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  DBuf<double> Wp0, Wp1, Wsmall;  // fused panel TRSM workspaces (chol.cuh)
  DBuf<double> diag_ws;           // scratch of the fused diagonal-block kernel (diag_block.cuh)
  DBuf<int8_t> oz_planes;         // INT8 U U^T engine (uut_i8.cuh): residue planes, row maxima, row exponents
  DBuf<unsigned long long> oz_rowmax;
  DBuf<int> oz_ex;
  int uut_engine = 0;             // debug pin (ace_dbg_fit_set_uut_engine): 0 by size, 1 DMMA, 2 INT8
  int panel_blocks = 4;
  cudaEvent_t tev[8] = {};
  DBuf<double> X, Z, LZ, y, theta, m, v, grad, tab, sc, A, Bf, DX, DU, dvec, alpha, uvec, svec, Ka, pu, ps, partials;
  DBuf<int> info;
  double* h_sc = nullptr;  // pinned: SC_COUNT doubles + info
  GradPlan gp;
  int nchunks = 0;
  // multi-GPU sharding of ONE fit (ace_fit_shard): rank/world of the communicator, and `red` = [P partial
  // sums | n_pad entries of K*alpha], the vector that is all-reduced each iteration
  int shard_rank = 0, shard_world = 1;
  DBuf<double> red;
  double* ka() { return red.p ? red.p + P : Ka.p; }
  // sharded dense phases (shard_dense.cuh): triangular inverse split by levels, K^-1 tiles dealt round-robin
  bool shard_dense = false;    // on by default for a sharded fit (ACE_SHARD_DENSE=0: redundant dense phases)
  bool shard_emulate = false;  // one process plays all ranks in turn (single-GPU tests), no NCCL
  int shard_hmin = 16;
  bool kinv_partial = false;   // Bf does not hold the complete stored inverse (U is complete in A): rebuilt on demand
  bool u_valid = false;        // A / DX / DU hold U = L^-T, X = L^-1 of the stored inverse (after an iteration)
  DBuf<double> tvy, tv1, pdg, kdg;
  bool shard_incr = true;      // inverse grown behind the panels, column panels per rank (ACE_SHARD_INCR=0: split merge tree)
  bool shard_potrf = false;    // panel-cyclic Cholesky with panel broadcasts (ACE_SHARD_POTRF=0: redundant potrf)
  std::vector<cudaEvent_t> shard_events;
  DBuf<double> head0, head1;   // packed panel heads (shard_dense.cuh)
  cudaStream_t bulk = nullptr; // bulk panel pieces: own stream (and communicator)
  int rank_lo() const { return shard_emulate ? 0 : shard_rank; }
  int rank_hi() const { return shard_emulate ? shard_world : shard_rank + 1; }
  DBuf<double> chain_ws;       // split-K partials of the chain's small GEMMs (shard_dense.cuh: chain_gemm)
  DBuf<double> mid0, mid1;     // early copies of the first bulk block (shard_dense.cuh: mid)
  cudaStream_t mids = nullptr;
  ShardCtx shard_ctx(ncclComm_t comm, ncclComm_t comm2, ncclComm_t comm3 = nullptr) const {
    ShardCtx cx;
    cx.rank = shard_rank; cx.world = shard_world; cx.emulate = shard_emulate; cx.comm = comm; cx.h_min = shard_hmin;
    cx.comm2 = comm2;
    cx.events = const_cast<cudaEvent_t*>(shard_events.data());
    cx.head[0] = head0.p; cx.head[1] = head1.p; cx.bulk_stream = bulk;
    cx.chain_ws = chain_ws.p;
    cx.comm3 = comm3; cx.mid[0] = mid0.p; cx.mid[1] = mid1.p; cx.mid_stream = mids;
    cx.incr = shard_incr;
    return cx;
  }
  int alloc_shard() {
    ACE_TRY(red.alloc((size_t)P + n_pad));
    ACE_CUDA(cudaMemsetAsync(red.p, 0, sizeof(double) * ((size_t)P + n_pad), st));
    const char* e = std::getenv("ACE_SHARD_DENSE");
    shard_dense = e ? (std::atoi(e) != 0) : true;
    if (const char* h = std::getenv("ACE_SHARD_HMIN")) shard_hmin = std::max(1, std::atoi(h));
    if (shard_dense) {
      const char* sp = std::getenv("ACE_SHARD_POTRF");
      const bool pow2 = (panel_blocks & (panel_blocks - 1)) == 0;
      if ((sp ? std::atoi(sp) != 0 : true) && pow2 && panel_blocks >= 2) {
        const size_t N = (size_t)n_pad;
        if (!Wp0.p) {  // packed panel buffers (the fused-TRSM workspaces of the single-GPU path, if it has them)
          ACE_TRY(Wp0.alloc(N * panel_blocks * TB));
          ACE_TRY(Wp1.alloc(N * panel_blocks * TB));
          ACE_TRY(Wsmall.alloc((size_t)(panel_blocks * TB / 2) * (panel_blocks * TB / 2)));
        }
        const size_t pw = (size_t)panel_blocks * TB;
        ACE_TRY(head0.alloc(2 * pw * pw));
        ACE_TRY(head1.alloc(2 * pw * pw));
        if (!bulk) {
          // priorities (numerically lower = more urgent): side (diagonal block, head) > mid > bulk > main (trailing
          // updates); the bulk GEMMs are large, at the side stream's priority they would sit in front of the small
          // kernels of the serial chain
          int lo = 0, hi = 0;
          ACE_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
          int pb_ = (hi + lo) / 2;
          if (const char* e = std::getenv("ACE_SHARD_BULK_PRIO")) pb_ = std::max(hi, std::min(lo, std::atoi(e)));
          ACE_CUDA(cudaStreamCreateWithPriority(&bulk, cudaStreamNonBlocking, pb_));
        }
        {
          const char* sk = std::getenv("ACE_SHARD_SPLITK");
          if (!(sk && std::atoi(sk) == 0)) ACE_TRY(chain_ws.alloc(4 * pw * pw));
        }
        {
          const char* sm = std::getenv("ACE_SHARD_MID");
          if (!(sm && std::atoi(sm) == 0)) {
            ACE_TRY(mid0.alloc(pw * pw));
            ACE_TRY(mid1.alloc(pw * pw));
            if (!mids) {
              int lo = 0, hi = 0;
              ACE_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
              ACE_CUDA(cudaStreamCreateWithPriority(&mids, cudaStreamNonBlocking, std::min(lo, hi + 1)));
            }
          }
        }
        const int NP = shard_panels(n_pad / TB, panel_blocks);
        while ((int)shard_events.size() < SHARD_EVENT_KINDS * NP) {
          cudaEvent_t e;
          ACE_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
          shard_events.push_back(e);
        }
        shard_potrf = true;
        // Inverse grown behind the panels (incremental) vs. split merge tree after the factorisation: the first
        // wins while the Cholesky is bound by its serial panel chain (~0.85 ms per panel), i.e. while the GPUs have
        // idle time to fill (C3: 47.3 -> 42.6 ms on 8 GPUs); when the trailing updates dominate, background work
        // only competes with them (C4, n = 65536, 8 GPUs: 1.20 s split tree vs 1.25 s incremental).
        {
          const double nn = (double)n_pad;
          const double chain_s = NP * 0.85e-3, update_s = nn * nn * nn / (3.0 * shard_world * 3.5e13);
          shard_incr = 2.0 * chain_s >= update_s;
        }
        if (const char* si = std::getenv("ACE_SHARD_INCR")) shard_incr = std::atoi(si) != 0;
      }
    }
    return 0;
  }
  // the full inverse from the replicated U (consumers outside the iteration: invKmatn download, posterior)
  int ensure_full_inverse() {
    if (!kinv_partial) return 0;
    DenseWork w = dense(A.p, Bf.p);
    ACE_TRY(uut_inverse(w));
    kinv_partial = false;
    return 0;
  }

  ~Core() {
    if (h_sc) cudaFreeHost(h_sc);
    for (auto& e : ev)
      if (e) cudaEventDestroy(e);
    for (auto& e : tev)
      if (e) cudaEventDestroy(e);
    for (auto& e : shard_events) cudaEventDestroy(e);
    if (bulk) cudaStreamDestroy(bulk);
    if (mids) cudaStreamDestroy(mids);
    if (st) cudaStreamDestroy(st);
    if (side) cudaStreamDestroy(side);
    if (aux) cudaStreamDestroy(aux);
    if (bgst) cudaStreamDestroy(bgst);
  }

  int init(int dev, int n_, int p_, int Bz_, int kind_, bool need_dense, bool need_grad) {
    ACE_TRY(check_device());
    device = dev;
    ACE_CUDA(cudaSetDevice(dev));
    ACE_TRY(configure_kernels_once());
    cudaDeviceProp prop;
    ACE_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (prop.major < 10) {
      set_error("this library is built for sm_100a (B200) only");
      return ACE_ERR_NO_DEVICE;
    }
    sms = prop.multiProcessorCount;
    n = n_; p = p_; Bz = Bz_; B = Bz_ + 1; P = 2 + B + B * p; kind = kind_;
    n_pad = round_up(n, TB);
    ACE_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    int lo = 0, hi = 0;
    ACE_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    ACE_CUDA(cudaStreamCreateWithPriority(&side, cudaStreamNonBlocking, hi));  // panel stream: high priority
    ACE_CUDA(cudaStreamCreateWithPriority(&aux, cudaStreamNonBlocking, lo));   // filler work: lowest priority
    ACE_CUDA(cudaStreamCreateWithPriority(&bgst, cudaStreamNonBlocking, lo));  // incremental inverse behind the panels
    for (auto& e : ev) ACE_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto& e : tev) ACE_CUDA(cudaEventCreate(&e));
    ACE_CUDA(cudaMallocHost(&h_sc, sizeof(double) * (SC_COUNT + 2)));
    const size_t N = (size_t)n_pad;
    ACE_TRY(X.alloc(N * p));
    ACE_TRY(Z.alloc(N * std::max(Bz, 1)));
    ACE_TRY(LZ.alloc(N * std::max(Bz, 1)));
    ACE_TRY(y.alloc(N));
    ACE_TRY(theta.alloc(P));
    ACE_TRY(m.alloc(P));
    ACE_TRY(v.alloc(P));
    ACE_TRY(grad.alloc(P));
    ACE_TRY(tab.alloc(tab_doubles(p)));
    ACE_TRY(sc.alloc(SC_COUNT));
    ACE_TRY(info.alloc(1));
    ACE_CUDA(cudaMemsetAsync(sc.p, 0, sizeof(double) * SC_COUNT, st));
    ACE_CUDA(cudaMemsetAsync(m.p, 0, sizeof(double) * P, st));
    ACE_CUDA(cudaMemsetAsync(v.p, 0, sizeof(double) * P, st));
    ACE_CUDA(cudaMemsetAsync(grad.p, 0, sizeof(double) * P, st));
    ACE_CUDA(cudaMemsetAsync(info.p, 0, sizeof(int), st));
    if (need_dense) {
      ACE_TRY(A.alloc(N * N));
      ACE_TRY(Bf.alloc(N * N));
      ACE_TRY(DX.alloc(N * TB));
      ACE_TRY(DU.alloc(N * TB));
      ACE_TRY(dvec.alloc(N));
      if (const char* e = std::getenv("ACE_PANEL_BLOCKS")) {  // tuning knob (128-blocks per look-ahead panel)
        const int v = std::atoi(e);
        if (v >= 1 && v <= 64) panel_blocks = v;
      }
      const char* fu = std::getenv("ACE_FUSED_TRSM");
      const bool pow2 = (panel_blocks & (panel_blocks - 1)) == 0;
      // The fused panel TRSM (early X_JJ) also enables the incremental inverse behind the panels (chol.cuh); together
      // they pay off at every size measured: C2 (n=4096) 8.65 -> 7.87 ms, C5 (n=8192) 27.0 -> 23.5 ms, C3 (n=16384)
      // 164.9 -> 158.3 ms per iteration.  ACE_FUSED_TRSM=0 switches both off.
      const bool want = fu ? (std::atoi(fu) != 0) : true;
      ACE_TRY(alloc_uut_engine());
      if (pow2 && panel_blocks >= 2 && want) {
        ACE_TRY(Wp0.alloc(N * panel_blocks * TB));
        ACE_TRY(Wp1.alloc(N * panel_blocks * TB));
        ACE_TRY(Wsmall.alloc((size_t)(panel_blocks * TB / 2) * (panel_blocks * TB / 2)));
        // one cluster launch per diagonal block instead of ~16 small launches (ACE_DIAG_FUSED=0: the leaf recursion)
        const char* df = std::getenv("ACE_DIAG_FUSED");
        if (!(df && std::atoi(df) == 0)) ACE_TRY(diag_ws.alloc(dg::ws_doubles(panel_blocks)));
      }
    }
    if (need_grad) {
      ACE_TRY(plan_grad(p, B, kind, sms, &gp));
      nchunks = (n + gv::CHUNK - 1) / gv::CHUNK;
      ACE_TRY(alpha.alloc(N));
      ACE_TRY(uvec.alloc(N));
      ACE_TRY(svec.alloc(N));
      ACE_TRY(Ka.alloc(N));
      ACE_TRY(pu.alloc(N * nchunks));
      ACE_TRY(ps.alloc(N * nchunks));
      ACE_TRY(partials.alloc((size_t)gp.gx * gp.gy * P));
      if (!dvec.p) ACE_TRY(dvec.alloc(N));
      ACE_TRY(tvy.alloc(N));  // U^T y, U^T 1, diag(K^-1) partials: posterior in factor form, alpha in factor form
      ACE_TRY(tv1.alloc(N));
      ACE_TRY(pdg.alloc(N * nchunks));
      ACE_TRY(kdg.alloc(N));
    }
    return 0;
  }

  // the residue-plane workspace, when the U U^T of this size runs on the INT8 engine
  int alloc_uut_engine() {
    if (uut_engine == 2 && n_pad > oz::MAX_N) {
      set_error("the INT8 U U^T engine covers n_pad <= " + std::to_string(oz::MAX_N) + " (CRT range bound)");
      return ACE_ERR_UNSUPPORTED;
    }
    if (!uut_uses_i8(n_pad, uut_engine)) {  // pinned to DMMA: the planes are not needed
      oz_planes.release();
      oz_rowmax.release();
      oz_ex.release();
      return 0;
    }
    if (oz_planes.p) return 0;
    ACE_TRY(oz_planes.alloc(oz::plane_bytes(n_pad / TB)));
    ACE_TRY(oz_rowmax.alloc(n_pad));
    ACE_TRY(oz_ex.alloc(n_pad));
    return 0;
  }

  int upload_data(const double* hy, const double* hX, const double* hZ) {
    if (hX) ACE_TRY(upload_matrix(X.p, n_pad, n_pad, hX, n, p, st));
    if (hZ) {
      ACE_TRY(upload_matrix(Z.p, n_pad, n_pad, hZ, n, Bz, st));
      const size_t cnt = (size_t)n_pad * Bz;
      if (cnt) logabs_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>(Z.p, LZ.p, cnt);
      ACE_CUDA(cudaGetLastError());
    }
    if (hy) ACE_TRY(upload_matrix(y.p, n_pad, n_pad, hy, n, 1, st));
    return 0;
  }

  int upload_theta(const double* hpar) {
    ACE_CUDA(cudaMemcpyAsync(theta.p, hpar, sizeof(double) * P, cudaMemcpyHostToDevice, st));
    return 0;
  }

  DenseWork dense(double* Abuf, double* Bbuf, bool allow_fused = true) {
    DenseWork w;
    w.panel_blocks = panel_blocks;
    if (allow_fused && Wp0.p) {
      w.Wp[0] = Wp0.p; w.Wp[1] = Wp1.p; w.Wsmall = Wsmall.p; w.ev_copy[0] = ev[6]; w.ev_copy[1] = ev[7];
      w.diag_ws = diag_ws.p;
    }
    w.A = Abuf; w.ld = n_pad; w.nb = n_pad / TB; w.DX = DX.p; w.DU = DU.p; w.dvec = dvec.p; w.info = info.p;
    w.Bf = Bbuf; w.main = st; w.side = side; w.aux = aux; w.bg = bgst; w.ev_half = ev[4]; w.ev_aux = ev[5];
    w.ev_panel[0] = ev[0]; w.ev_panel[1] = ev[1]; w.ev_upd[0] = ev[2]; w.ev_upd[1] = ev[3];
    w.oz.planes = oz_planes.p; w.oz.rowmax = oz_rowmax.p; w.oz.ex = oz_ex.p; w.uut_engine = uut_engine;

    return w;
  }

  int enqueue_prep() {
    prep_tables_kernel<<<1, 256, 0, st>>>(theta.p, p, B, tab.p);
    ACE_CUDA(cudaGetLastError());
    return 0;
  }

  // K (+ e^sigma on the diagonal, identity padding) of the training points into `out`
  int enqueue_build_sym(double* out, int add_noise, double* cube, long cube_slice) {
    KernArgs a{};
    a.X1 = a.X2 = X.p; a.Z1 = a.Z2 = Z.p; a.LZ1 = a.LZ2 = LZ.p; a.ld1 = a.ld2 = n_pad;
    a.n1 = a.n2 = n; a.n1_pad = a.n2_pad = n_pad; a.p = p; a.B = B; a.tab = tab.p;
    a.K = out; a.ldk = n_pad; a.cube = cube; a.cube_slice = cube_slice;
    a.sym = 1; a.add_noise = add_noise; a.pad_identity = add_noise;
    return launch_kernmat(a, kind, st);
  }

  // Multi-GPU: this rank's two column blocks of K + e^sigma I (rows >= first column of the block only)
  int enqueue_build_blocks(double* out) {
    const int w = shard_block_width(n_pad, shard_world);
    for (int blk = 0; blk < 2 * shard_world; ++blk) {
      const int owner = shard_block_owner(blk, shard_world);
      if (owner < rank_lo() || owner >= rank_hi()) continue;
      const int c0 = blk * w, r0 = c0;
      KernArgs a{};
      a.X1 = X.p + r0; a.Z1 = Z.p + r0; a.LZ1 = LZ.p + r0; a.ld1 = n_pad;
      a.X2 = X.p + c0; a.Z2 = Z.p + c0; a.LZ2 = LZ.p + c0; a.ld2 = n_pad;
      a.n1 = std::max(0, n - r0); a.n2 = std::max(0, std::min(w, n - c0));
      a.n1_pad = n_pad - r0; a.n2_pad = w; a.p = p; a.B = B; a.tab = tab.p;
      a.K = out + r0 + (size_t)c0 * n_pad; a.ldk = n_pad;
      a.sym = 0; a.add_noise = 1; a.pad_identity = 1; a.row_off = r0; a.col_off = c0;
      ACE_TRY(launch_kernmat(a, kind, st));
    }
    return 0;
  }

  // Multi-GPU with the panel-cyclic Cholesky: the column panels this rank owns (rows >= first column of the panel)
  int enqueue_build_panels(double* out) {
    const int nb = n_pad / TB, NP = shard_panels(nb, panel_blocks);
    for (int c = 0; c < NP; ++c) {
      if (!(shard_emulate || c % shard_world == shard_rank)) continue;
      const int c0 = c * panel_blocks * TB, w = std::min(panel_blocks * TB, n_pad - c0), r0 = c0;
      KernArgs a{};
      a.X1 = X.p + r0; a.Z1 = Z.p + r0; a.LZ1 = LZ.p + r0; a.ld1 = n_pad;
      a.X2 = X.p + c0; a.Z2 = Z.p + c0; a.LZ2 = LZ.p + c0; a.ld2 = n_pad;
      a.n1 = std::max(0, n - r0); a.n2 = std::max(0, std::min(w, n - c0));
      a.n1_pad = n_pad - r0; a.n2_pad = w; a.p = p; a.B = B; a.tab = tab.p;
      a.K = out + r0 + (size_t)c0 * n_pad; a.ldk = n_pad;
      a.sym = 0; a.add_noise = 1; a.pad_identity = 1; a.row_off = r0; a.col_off = c0;
      ACE_TRY(launch_kernmat(a, kind, st));
    }
    return 0;
  }

  // u = Kinv y, s = Kinv 1, alpha = u - mu s (mu closed form first when asked and iter == 1)
  int enqueue_alpha(const double* Kinv, int set_mu_first_iter) {
    dim3 grid((n_pad + gv::ROWS - 1) / gv::ROWS, nchunks);
    gemv2_kernel<<<grid, gv::ROWS, 0, st>>>(Kinv, n_pad, n, y.p, pu.p, ps.p, n_pad);
    ACE_CUDA(cudaGetLastError());
    alpha_kernel<<<1, 1024, 0, st>>>(pu.p, ps.p, nchunks, n, n_pad, theta.p, uvec.p, svec.p, alpha.p, ka(), sc.p,
                                     set_mu_first_iter);
    ACE_CUDA(cudaGetLastError());
    return 0;
  }

  // u = U (U^T y), s = U (U^T 1), diag(K^-1) into kdg, all from the factor (upper(Afac) + DUfac tiles): alpha, mu
  // and the evidence then do not depend on how K^-1 itself was formed (sharded tiles, INT8 engine)
  int enqueue_alpha_tri(const double* Afac, int set_mu_first_iter, const double* DUfac = nullptr) {
    if (!DUfac) DUfac = DU.p;
    utv2_kernel<<<(n_pad + 7) / 8, 256, 0, st>>>(Afac, n_pad, DUfac, n, n_pad, y.p, tvy.p, tv1.p);
    ACE_CUDA(cudaGetLastError());
    dim3 grid((n_pad + gv::ROWS - 1) / gv::ROWS, nchunks);
    uv2_kernel<<<grid, gv::ROWS, 0, st>>>(Afac, n_pad, DUfac, n_pad, tvy.p, tv1.p, pu.p, ps.p, pdg.p);
    ACE_CUDA(cudaGetLastError());
    alpha_kernel<<<1, 1024, 0, st>>>(pu.p, ps.p, nchunks, n, n_pad, theta.p, uvec.p, svec.p, alpha.p, ka(), sc.p,
                                     set_mu_first_iter, pdg.p, kdg.p);
    ACE_CUDA(cudaGetLastError());
    return 0;
  }

  // alpha, mu, diag(K^-1) of an unsharded inverse: from the factor when K^-1 comes from the INT8 engine (so that the
  // evidence, alpha and the mu refresh do not see its rounding), from the DMMA K^-1 in Kinv otherwise (one pass over
  // K^-1 is the cheaper read: C2 5.08 vs 5.11 ms per iteration with the factor form)
  bool alpha_from_factor() const { return uut_uses_i8(n_pad, uut_engine); }
  int enqueue_alpha_any(const double* Afac, int set_mu_first_iter, const double* DUfac = nullptr,
                        const double* Kinv = nullptr) {
    if (alpha_from_factor()) return enqueue_alpha_tri(Afac, set_mu_first_iter, DUfac);
    return enqueue_alpha(Kinv ? Kinv : Bf.p, set_mu_first_iter);
  }

  // tile_world 1: all lower tiles.  Otherwise every world-th tile; tile_mode 1 follows the ownership of the
  // sharded U U^T launch (the rank only reads entries of K^-1 it computed itself).
  int enqueue_grad(const double* Kinv, int tile_rank = 0, int tile_world = 1, int tile_mode = 0) {
    GradArgs g{};
    g.X = X.p; g.Z = Z.p; g.LZ = LZ.p; g.ldx = n_pad; g.Kinv = Kinv; g.ld = n_pad; g.alpha = alpha.p; g.Ka = ka();
    g.tab = tab.p; g.partials = partials.p; g.n = n; g.p = p; g.B = B; g.P = P;
    g.ntiles_side = (n + gk::T - 1) / gk::T;
    g.tile_rank = tile_rank; g.tile_world = tile_world; g.tile_mode = tile_mode; g.gemm_rows = n_pad / TB;
    return launch_grad(g, kind, gp, st);
  }

  int enqueue_finalize(const double* Kinv, const ace_fit_config& c, int do_update, bool reduced = false,
                       const double* kdiag = nullptr, const double* dvec_alt = nullptr) {
    FinalizeArgs f{};
    f.partials = partials.p; f.nparts = gp.gx * gp.gy; f.y = y.p; f.alpha = alpha.p; f.Ka = ka();
    f.dvec = dvec_alt ? dvec_alt : dvec.p;
    if (reduced) {  // sharded iteration: the all-reduced sums live in red[0..P)
      f.partials = red.p;
      f.nparts = 1;
    }
    f.kdiag = kdiag;
    f.Kinv = Kinv; f.ld = n_pad; f.tab = tab.p; f.theta = theta.p; f.m = m.p; f.v = v.p; f.grad = grad.p; f.sc = sc.p;
    f.n = n; f.p = p; f.B = B; f.P = P; f.kind = kind; f.optimizer = c.optimizer; f.lr = c.learning_rate;
    f.beta1 = c.beta1; f.beta2 = c.beta2; f.eps = 1e-8; f.momentum = c.momentum; f.std_y = c.std_y;
    f.clip_at = c.clip_at; f.norm_clip = c.norm_clip; f.do_update = do_update;
    finalize_kernel<<<1, 1024, 0, st>>>(f);
    ACE_CUDA(cudaGetLastError());
    return 0;
  }

  int fetch_scalars() {
    ACE_CUDA(cudaMemcpyAsync(h_sc, sc.p, sizeof(double) * SC_COUNT, cudaMemcpyDeviceToHost, st));
    ACE_CUDA(cudaMemcpyAsync(h_sc + SC_COUNT, info.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    ACE_CUDA(cudaStreamSynchronize(st));
    return 0;
  }
  int h_info() const { return *reinterpret_cast<const int*>(h_sc + SC_COUNT); }
};

}  // namespace ace

using namespace ace;

// =============================================================================================
// fit handle
// =============================================================================================
struct ace_fit {
  Core c;
  ace_fit_config cfg;
  cudaEvent_t sw0 = nullptr, sw1 = nullptr;  // stopwatch
  int launches = -1;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t gexec = nullptr;
  double iter_dev = 0.0;  // host shadow of sc[SC_ITER]
  double ms[6] = {0, 0, 0, 0, 0, 0};
  ncclComm_t comm = nullptr, comm2 = nullptr, comm3 = nullptr;  // multi-GPU sharded mode
  ~ace_fit() {
    if (comm2 && nccl_api().ok) nccl_api().CommDestroy(comm2);
    if (comm3 && nccl_api().ok) nccl_api().CommDestroy(comm3);
    if (comm && nccl_api().ok) nccl_api().CommDestroy(comm);
    if (sw0) cudaEventDestroy(sw0);
    if (sw1) cudaEventDestroy(sw1);
    if (gexec) cudaGraphExecDestroy(gexec);
    if (graph) cudaGraphDestroy(graph);
  }
};

static int enqueue_iteration(ace_fit* f, bool timed) {
  Core& c = f->c;
  DenseWork w = c.dense(c.A.p, c.Bf.p);
  if (timed) ACE_CUDA(cudaEventRecord(c.tev[0], c.st));
  ACE_TRY(c.enqueue_prep());
  const bool sharded = c.shard_world > 1;
  const bool comm = sharded && !c.shard_emulate;
  const bool spotrf = sharded && c.shard_dense && c.shard_potrf;
  if (!sharded) {
    ACE_TRY(c.enqueue_build_sym(c.A.p, 1, nullptr, 0));
  } else if (spotrf) {
    // panel-cyclic Cholesky: a rank only ever needs the K columns of the panels it owns -- no exchange
    ACE_TRY(c.enqueue_build_panels(c.A.p));
  } else {
    // every rank builds its two column blocks, then the blocks are exchanged over NVLink (one grouped
    // NCCL broadcast per block)
    ACE_TRY(c.enqueue_build_blocks(c.A.p));
    if (comm) {
      NcclApi& nc = nccl_api();
      const int wdt = shard_block_width(c.n_pad, c.shard_world);
      const size_t cnt = (size_t)wdt * c.n_pad;
      ACE_NCCL(nc.GroupStart());
      for (int blk = 0; blk < 2 * c.shard_world; ++blk) {
        double* ptr = c.A.p + (size_t)blk * cnt;
        ACE_NCCL(nc.Broadcast(ptr, ptr, cnt, ncclFloat64, shard_block_owner(blk, c.shard_world), f->comm, c.st));
      }
      ACE_NCCL(nc.GroupEnd());
    }
  }
  if (timed) ACE_CUDA(cudaEventRecord(c.tev[1], c.st));
  const bool sdense = sharded && c.shard_dense;
  if (!sdense) {
    // Cholesky and triangular inverse overlap (potrf_trtri), so they are timed as one phase: ms[1] = both, ms[2] = 0
    ACE_TRY(potrf_trtri(w));
    if (timed) ACE_CUDA(cudaEventRecord(c.tev[2], c.st));
    if (timed) ACE_CUDA(cudaEventRecord(c.tev[3], c.st));
    ACE_TRY(uut_inverse(w));
    if (timed) ACE_CUDA(cudaEventRecord(c.tev[4], c.st));
    ACE_TRY(c.enqueue_alpha_any(c.A.p, 1));
  } else {
    // redundant Cholesky (ms[1]), then the split triangular inverse (ms[2]) and this rank's tiles of U U^T (ms[3])
    const ShardCtx cx = c.shard_ctx(f->comm, f->comm2, f->comm3);
    if (spotrf) {
      static const bool host_time = std::getenv("ACE_SHARD_HOSTTIME") != nullptr;
      const auto h0 = std::chrono::steady_clock::now();
      ACE_TRY(potrf_sharded(w, cx));
      if (host_time)
        std::fprintf(stderr, "[rank %d] potrf_sharded: host enqueue %.3f ms\n", c.shard_rank,
                     std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - h0).count());
    } else {
      const int s = potrf_blocked(w);
      if (s < 0) return s;
    }
    if (timed) ACE_CUDA(cudaEventRecord(c.tev[2], c.st));
    if (spotrf && cx.incr)
      ACE_TRY(gather_inverse_sharded(w, cx));
    else
      ACE_TRY(trtri_merge_sharded(w, cx));
    if (timed) ACE_CUDA(cudaEventRecord(c.tev[3], c.st));
    ACE_TRY(uut_inverse_sharded(w, cx));
    if (timed) ACE_CUDA(cudaEventRecord(c.tev[4], c.st));
    ACE_TRY(c.enqueue_alpha_tri(c.A.p, 1));
  }
  if (!sharded) {
    ACE_TRY(c.enqueue_grad(c.Bf.p));
  } else {
    // each rank takes every world-th tile: sum its CTA partials, then all-reduce [P sums | K*alpha] so that
    // every rank finalises with bit-identical inputs (parameters stay in lock-step without a broadcast)
    for (int r = c.rank_lo(); r < c.rank_hi(); ++r) {
      ACE_TRY(c.enqueue_grad(c.Bf.p, r, c.shard_world, sdense ? 1 : 0));
      partials_reduce_kernel<<<1, 1024, 0, c.st>>>(c.partials.p, c.gp.gx * c.gp.gy, c.P, c.red.p, r > c.rank_lo());
      ACE_CUDA(cudaGetLastError());
    }
    if (comm)
      ACE_NCCL(nccl_api().AllReduce(c.red.p, c.red.p, (size_t)c.P + c.n_pad, ncclFloat64, ncclSum, f->comm, c.st));
  }
  ACE_TRY(c.enqueue_finalize(c.Bf.p, f->cfg, 1, sharded, (sdense || c.alpha_from_factor()) ? c.kdg.p : nullptr));
  if (timed) ACE_CUDA(cudaEventRecord(c.tev[5], c.st));
  return 0;
}

extern "C" {

const char* ace_last_error(void) { return g_err.c_str(); }
const char* ace_version(void) { return "ace_b200 0.1 (sm_100a; FP64 DMMA; TMA bulk)"; }

int ace_device_count(void) {
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return cnt;
}

static thread_local int g_device = 0;
int ace_set_device(int device) {
  ACE_TRY(check_device());
  ACE_CUDA(cudaSetDevice(device));
  g_device = device;
  return 0;
}

void ace_fit_default_config(ace_fit_config* cfg) {
  cfg->kernel = ACE_KERNEL_SE;
  cfg->optimizer = ACE_OPT_NADAM;
  cfg->learning_rate = 0.01;
  cfg->beta1 = 0.9;
  cfg->beta2 = 0.999;
  cfg->momentum = 0.0;
  cfg->norm_clip = 1;
  cfg->clip_at = 1.0;
  cfg->std_y = 1.0;
  cfg->device = 0;
  cfg->use_graph = 1;
}

int ace_fit_create(ace_fit** out, const double* y, const double* X, const double* Z, int n, int p, int Bz,
                   const double* parameters, const ace_fit_config* cfg) {
  if (!out || !y || !X || (Bz > 0 && !Z) || !parameters || !cfg) return usage("ace_fit_create: null argument");
  if (n < 1 || p < 1 || Bz < 0) return usage("ace_fit_create: need n >= 1, p >= 1, Bz >= 0");
  *out = nullptr;
  ace_fit* f = new (std::nothrow) ace_fit();
  if (!f) return usage("out of host memory");
  f->cfg = *cfg;
  int s = f->c.init(cfg->device, n, p, Bz, cfg->kernel, true, true);
  if (s == 0) s = f->c.upload_data(y, X, Z);
  if (s == 0) s = f->c.upload_theta(parameters);
  if (s == 0) {
    cudaError_t e = cudaStreamSynchronize(f->c.st);
    if (e != cudaSuccess) {
      set_error(std::string("ace_fit_create: ") + cudaGetErrorString(e));
      s = -(int)e - 1000;
    }
  }
  if (s != 0) {
    delete f;
    return s;
  }
  *out = f;
  return 0;
}

int ace_fit_destroy(ace_fit* fit) {
  if (!fit) return 0;
  cudaSetDevice(fit->c.device);
  cudaDeviceSynchronize();
  delete fit;
  return 0;
}

int ace_fit_para_update(ace_fit* f, int iter, double* stats, double* gnorm) {
  if (!f) return usage("null handle");
  Core& c = f->c;
  ACE_CUDA(cudaSetDevice(c.device));
  if ((double)iter != f->iter_dev) {
    c.h_sc[SC_COUNT + 1] = (double)iter;
    ACE_CUDA(cudaMemcpyAsync(c.sc.p + SC_ITER, c.h_sc + SC_COUNT + 1, sizeof(double), cudaMemcpyHostToDevice, c.st));
    f->iter_dev = (double)iter;
  }
  // a fit sharded over real ranks launches eagerly: its iteration contains NCCL collectives on several streams
  const bool use_graph = f->cfg.use_graph && !(c.shard_world > 1 && !c.shard_emulate);
  if (use_graph) {
    if (!f->gexec) {
      ACE_CUDA(cudaStreamBeginCapture(c.st, cudaStreamCaptureModeThreadLocal));
      int s = enqueue_iteration(f, false);
      cudaGraph_t g = nullptr;
      cudaError_t e = cudaStreamEndCapture(c.st, &g);
      if (s != 0) {
        if (g) cudaGraphDestroy(g);
        return s;
      }
      ACE_CUDA(e);
      f->graph = g;
      ACE_CUDA(cudaGraphInstantiate(&f->gexec, f->graph, 0));
    }
    ACE_CUDA(cudaEventRecord(c.tev[6], c.st));
    ACE_CUDA(cudaGraphLaunch(f->gexec, c.st));
    ACE_CUDA(cudaEventRecord(c.tev[7], c.st));
  } else {
    ACE_CUDA(cudaEventRecord(c.tev[6], c.st));
    ACE_TRY(enqueue_iteration(f, true));
    ACE_CUDA(cudaEventRecord(c.tev[7], c.st));
  }
  // state of the buffers after this iteration (set here, not while enqueueing: a captured graph is replayed
  // without re-running the enqueue code, and counting launches captures without executing)
  c.u_valid = true;  // A / DX / DU hold the factor of the stored inverse
  c.kinv_partial = c.shard_world > 1 && c.shard_dense && !c.shard_emulate;  // only this rank's tiles of K^-1 in Bf
  ACE_TRY(c.fetch_scalars());
  f->iter_dev = c.h_sc[SC_ITER];
  float t = 0;
  ACE_CUDA(cudaEventElapsedTime(&t, c.tev[6], c.tev[7]));
  f->ms[5] = t;
  if (!use_graph) {
    for (int k = 0; k < 5; ++k) {
      ACE_CUDA(cudaEventElapsedTime(&t, c.tev[k], c.tev[k + 1]));
      f->ms[k] = t;
    }
  }
  if (stats) {
    stats[0] = c.h_sc[SC_RMSE];
    stats[1] = c.h_sc[SC_EVID];
  }
  if (gnorm) *gnorm = c.h_sc[SC_GNORM];
  if (c.h_info() > 0) {
    set_error("matrix not positive definite at pivot " + std::to_string(c.h_info()));
    return c.h_info();
  }
  if (c.h_sc[SC_FINITE] == 0.0) {
    set_error("Some gradients are not finite, NaN, or NA. Often this is due to too large learning rates.");
    return ACE_ERR_NOT_FINITE;
  }
  return 0;
}

int ace_fit_run(ace_fit* f, int iter_start, int max_iter, double tol, double prev_evidence, double* stats_out,
                int* iters_done) {
  if (!f || !iters_done) return usage("null argument");
  double prev = prev_evidence;
  int done = 0;
  for (int k = 0; k < max_iter; ++k) {
    const int iter = iter_start + k;
    double st[2];
    int s = ace_fit_para_update(f, iter, st, nullptr);
    if (s != 0) {
      *iters_done = done;
      return s;
    }
    ++done;
    if (stats_out) {
      stats_out[2 * k] = st[0];
      stats_out[2 * k + 1] = st[1];
    }
    const double change = std::fabs(st[1] - prev);  // R/main_ace.R:221
    prev = st[1];
    if (change < tol && iter > 3) break;
  }
  *iters_done = done;
  return 0;
}

int ace_dbg_kernel_plan(int p, int B, int kind, int sym, char* build, int build_len, char* grad, int grad_len) {
  if (kind != 0 && kind != 1) return usage("dbg_kernel_plan: kind must be 0 (SE) or 1 (Matern-3/2)");
  if (!build || !grad || build_len < 1 || grad_len < 1) return usage("dbg_kernel_plan: null or empty output buffer");
  BuildPlan bp;
  ACE_TRY(plan_kernmat(p, B, sym, &bp));
  GradPlan gp;
  ACE_TRY(plan_grad(p, B, kind, 148, &gp));  // the SM count only sets gridDim.x, which selects no code
  const char* shape = sym ? "sym" : "rect";
  int nb;
  if (bp.family == BuildPlan::WIDE) nb = std::snprintf(build, build_len, "kernmat_wide_kernel<%d> %s", kind, shape);
  else if (bp.family == BuildPlan::EXACT) nb = std::snprintf(build, build_len, "kernmat2_kernel<%d,%d> %s", kind, B, shape);
  else nb = std::snprintf(build, build_len, "kernmat_kernel<%d,%d,%d> %s", kind, bp.bc, bp.bc == 4 ? 4 : 2, shape);
  int ng;
  if (gp.wide_sw) ng = std::snprintf(grad, grad_len, "grad_wide_kernel<%d,%d>", kind, gp.wide_sw);
  else if (gp.v3) ng = std::snprintf(grad, grad_len, "grad3_kernel<%d,%d,%d> weights=%s", B, gp.NT3, kind,
                                     gp.cw3 ? "const" : "shared");
  else if (gp.v2) ng = std::snprintf(grad, grad_len, "grad2_kernel<%d,%d,%d,%d>", gp.PD8, gp.BD8, kind, gp.nw2);
  else ng = std::snprintf(grad, grad_len, "grad_kernel<%d,%d,%d> gpc=%d gy=%d", gp.PD, gp.BT, kind, gp.threads / 64,
                          gp.gy);
  if (nb >= build_len || ng >= grad_len) return usage("dbg_kernel_plan: output buffer too small");
  return 0;
}

int ace_dbg_fit_set_uut_engine(ace_fit* f, int engine) {
  if (!f) return usage("null handle");
  if (engine < 0 || engine > 2) return usage("dbg_fit_set_uut_engine: engine must be 0 (by size), 1 (DMMA) or 2 (INT8)");
  Core& c = f->c;
  ACE_CUDA(cudaSetDevice(c.device));
  ACE_CUDA(cudaStreamSynchronize(c.st));
  c.uut_engine = engine;
  ACE_TRY(c.alloc_uut_engine());
  // the captured iteration holds the old engine's launches
  if (f->gexec) cudaGraphExecDestroy(f->gexec);
  if (f->graph) cudaGraphDestroy(f->graph);
  f->gexec = nullptr;
  f->graph = nullptr;
  return 0;
}

int ace_fit_get_train_stats(ace_fit* f, double* stats) {
  if (!f || !stats) return usage("null argument");
  Core& c = f->c;
  ACE_CUDA(cudaSetDevice(c.device));
  // Local factorisation of K(theta_final): the STORED inverse must stay as it is (quirk Q6).  It is kept in factor
  // form -- U, X in A with the DX / DU tiles, which the posterior uses directly -- so this runs in other buffers:
  // Bf takes the new factor (the stored K^-1 is rebuilt from U on demand), B2 its workspace / inverse.
  DBuf<double> B2, DX2, DU2, dv2;
  ACE_TRY(B2.alloc((size_t)c.n_pad * c.n_pad));
  double* Fac = c.Bf.p;
  DenseWork w = c.dense(Fac, B2.p);
  if (c.u_valid) {
    ACE_TRY(DX2.alloc((size_t)c.n_pad * TB));
    ACE_TRY(DU2.alloc((size_t)c.n_pad * TB));
    ACE_TRY(dv2.alloc(c.n_pad));
    w.DX = DX2.p; w.DU = DU2.p; w.dvec = dv2.p;
    c.kinv_partial = true;
  } else {  // nothing stored yet: plain buffers
    Fac = c.A.p;
    w = c.dense(Fac, B2.p);
  }
  ACE_TRY(c.enqueue_prep());
  ACE_TRY(c.enqueue_build_sym(Fac, 1, nullptr, 0));
  ACE_TRY(spd_inverse(w));
  ACE_TRY(c.enqueue_alpha_any(Fac, 0, w.DU, B2.p));
  ACE_TRY(c.enqueue_grad(B2.p));
  ACE_TRY(c.enqueue_finalize(B2.p, f->cfg, 0, false, c.alpha_from_factor() ? c.kdg.p : nullptr, w.dvec));
  ACE_TRY(c.fetch_scalars());
  stats[0] = c.h_sc[SC_RMSE];
  stats[1] = c.h_sc[SC_EVID];
  if (c.h_info() > 0) return c.h_info();
  return 0;
}

int ace_comm_unique_id(char* id128) {
  if (!id128) return usage("null argument");
  NcclApi& nc = nccl_api();
  if (!nc.ok) {
    set_error(nc.why);
    return ACE_ERR_UNSUPPORTED;
  }
  ncclUniqueId id;
  ACE_NCCL(nc.GetUniqueId(&id));
  static_assert(sizeof(id) == 128, "ncclUniqueId is 128 bytes");
  std::memcpy(id128, &id, 128);
  return 0;
}

int ace_shard_plan(int n, int world, int rank, int* blocks2, int* width) {
  if (!blocks2 || !width || world < 1 || rank < 0 || rank >= world) return usage("ace_shard_plan: bad argument");
  const int n_pad = round_up(n, TB);
  *width = shard_block_width(n_pad, world);
  if (*width == 0) {
    set_error("sharding needs ceil(n/128)*128 divisible by 128*world");
    return ACE_ERR_UNSUPPORTED;
  }
  blocks2[0] = rank;
  blocks2[1] = 2 * world - 1 - rank;
  return 0;
}

int ace_fit_shard(ace_fit* f, const char* id128, int rank, int world) {
  if (!f || !id128 || world < 1 || rank < 0 || rank >= world) return usage("ace_fit_shard: bad argument");
  if (world == 1) return 0;
  Core& c = f->c;
  ACE_CUDA(cudaSetDevice(c.device));
  if (shard_block_width(c.n_pad, world) == 0) {
    set_error("sharding needs ceil(n/128)*128 divisible by 128*world");
    return ACE_ERR_UNSUPPORTED;
  }
  NcclApi& nc = nccl_api();
  if (!nc.ok) {
    set_error(nc.why);
    return ACE_ERR_UNSUPPORTED;
  }
  ncclUniqueId id;
  std::memcpy(&id, id128, 128);
  ACE_NCCL(nc.CommInitRank(&f->comm, world, id, rank));
  {  // second communicator (bulk panel broadcasts): its id is created on rank 0 and travels over the first one
    ncclUniqueId id2;
    DBuf<double> box;
    ACE_TRY(box.alloc(16));
    if (rank == 0) {
      ACE_NCCL(nc.GetUniqueId(&id2));
      ACE_CUDA(cudaMemcpyAsync(box.p, &id2, 128, cudaMemcpyHostToDevice, c.st));
    }
    ACE_NCCL(nc.Broadcast(box.p, box.p, 16, ncclFloat64, 0, f->comm, c.st));
    ACE_CUDA(cudaMemcpyAsync(&id2, box.p, 128, cudaMemcpyDeviceToHost, c.st));
    ACE_CUDA(cudaStreamSynchronize(c.st));
    ACE_NCCL(nc.CommInitRank(&f->comm2, world, id2, rank));
  }
  {  // third communicator (early first bulk block), same way
    ncclUniqueId id3;
    DBuf<double> box;
    ACE_TRY(box.alloc(16));
    if (rank == 0) {
      ACE_NCCL(nc.GetUniqueId(&id3));
      ACE_CUDA(cudaMemcpyAsync(box.p, &id3, 128, cudaMemcpyHostToDevice, c.st));
    }
    ACE_NCCL(nc.Broadcast(box.p, box.p, 16, ncclFloat64, 0, f->comm, c.st));
    ACE_CUDA(cudaMemcpyAsync(&id3, box.p, 128, cudaMemcpyDeviceToHost, c.st));
    ACE_CUDA(cudaStreamSynchronize(c.st));
    ACE_NCCL(nc.CommInitRank(&f->comm3, world, id3, rank));
  }
  c.shard_rank = rank;
  c.shard_world = world;
  ACE_TRY(c.alloc_shard());
  if (f->gexec) {  // a graph captured before sharding is stale
    cudaGraphExecDestroy(f->gexec);
    cudaGraphDestroy(f->graph);
    f->gexec = nullptr;
    f->graph = nullptr;
  }
  f->launches = -1;
  return 0;
}

int ace_fit_shard_emulate(ace_fit* f, int world) {
  if (!f || world < 1) return usage("ace_fit_shard_emulate: bad argument");
  Core& c = f->c;
  if (world == 1) return 0;
  ACE_CUDA(cudaSetDevice(c.device));
  if (shard_block_width(c.n_pad, world) == 0) {
    set_error("sharding needs ceil(n/128)*128 divisible by 128*world");
    return ACE_ERR_UNSUPPORTED;
  }
  c.shard_rank = 0;
  c.shard_world = world;
  c.shard_emulate = true;
  ACE_TRY(c.alloc_shard());
  if (f->gexec) {
    cudaGraphExecDestroy(f->gexec);
    cudaGraphDestroy(f->graph);
    f->gexec = nullptr;
    f->graph = nullptr;
  }
  f->launches = -1;
  return 0;
}

int ace_dbg_shard_trace_dump(int rank) {
  shard_trace_dump(rank);
  return 0;
}

int ace_fit_upload_data(ace_fit* f, const double* y, const double* X, const double* Z) {
  if (!f) return usage("null handle");
  ACE_CUDA(cudaSetDevice(f->c.device));
  return f->c.upload_data(y, X, Z);  // stream ordered before the next para_update
}

static int count_kernel_nodes(cudaGraph_t g, int* out) {
  size_t nn = 0;
  ACE_CUDA(cudaGraphGetNodes(g, nullptr, &nn));
  std::vector<cudaGraphNode_t> nodes(nn);
  if (nn) ACE_CUDA(cudaGraphGetNodes(g, nodes.data(), &nn));
  int k = 0;
  for (size_t i = 0; i < nn; ++i) {
    cudaGraphNodeType t;
    ACE_CUDA(cudaGraphNodeGetType(nodes[i], &t));
    if (t == cudaGraphNodeTypeKernel) ++k;
  }
  *out = k;
  return 0;
}

int ace_fit_kernel_launches(ace_fit* f, int* launches) {
  if (!f || !launches) return usage("null argument");
  Core& c = f->c;
  ACE_CUDA(cudaSetDevice(c.device));
  if (f->launches < 0) {
    if (f->graph) {
      ACE_TRY(count_kernel_nodes(f->graph, &f->launches));
    } else {  // capture once just to count; nothing is executed
      ACE_CUDA(cudaStreamBeginCapture(c.st, cudaStreamCaptureModeThreadLocal));
      int s = enqueue_iteration(f, false);
      cudaGraph_t g = nullptr;
      cudaError_t e = cudaStreamEndCapture(c.st, &g);
      if (s != 0 || e != cudaSuccess) {
        if (g) cudaGraphDestroy(g);
        return s != 0 ? s : -(int)e - 1000;
      }
      s = count_kernel_nodes(g, &f->launches);
      cudaGraphDestroy(g);
      ACE_TRY(s);
    }
  }
  *launches = f->launches;
  return 0;
}

int ace_fit_timer_start(ace_fit* f) {
  if (!f) return usage("null handle");
  ACE_CUDA(cudaSetDevice(f->c.device));
  if (!f->sw0) {
    ACE_CUDA(cudaEventCreate(&f->sw0));
    ACE_CUDA(cudaEventCreate(&f->sw1));
  }
  ACE_CUDA(cudaEventRecord(f->sw0, f->c.st));
  return 0;
}

int ace_fit_timer_stop(ace_fit* f, double* ms) {
  if (!f || !ms || !f->sw0) return usage("timer not started");
  ACE_CUDA(cudaSetDevice(f->c.device));
  ACE_CUDA(cudaEventRecord(f->sw1, f->c.st));
  ACE_CUDA(cudaEventSynchronize(f->sw1));
  float t = 0;
  ACE_CUDA(cudaEventElapsedTime(&t, f->sw0, f->sw1));
  *ms = t;
  return 0;
}

int ace_fit_get_parameters(ace_fit* f, double* par) {
  if (!f || !par) return usage("null argument");
  ACE_CUDA(cudaSetDevice(f->c.device));
  ACE_CUDA(cudaMemcpyAsync(par, f->c.theta.p, sizeof(double) * f->c.P, cudaMemcpyDeviceToHost, f->c.st));
  ACE_CUDA(cudaStreamSynchronize(f->c.st));
  return 0;
}

int ace_fit_set_parameters(ace_fit* f, const double* par) {
  if (!f || !par) return usage("null argument");
  ACE_CUDA(cudaSetDevice(f->c.device));
  ACE_TRY(f->c.upload_theta(par));
  ACE_CUDA(cudaStreamSynchronize(f->c.st));
  return 0;
}

int ace_fit_get_gradients(ace_fit* f, double* g) {
  if (!f || !g) return usage("null argument");
  ACE_CUDA(cudaSetDevice(f->c.device));
  ACE_CUDA(cudaMemcpyAsync(g, f->c.grad.p, sizeof(double) * f->c.P, cudaMemcpyDeviceToHost, f->c.st));
  ACE_CUDA(cudaStreamSynchronize(f->c.st));
  return 0;
}

int ace_fit_get_optimizer_state(ace_fit* f, double* m, double* v) {
  if (!f) return usage("null argument");
  ACE_CUDA(cudaSetDevice(f->c.device));
  if (m) ACE_CUDA(cudaMemcpyAsync(m, f->c.m.p, sizeof(double) * f->c.P, cudaMemcpyDeviceToHost, f->c.st));
  if (v) ACE_CUDA(cudaMemcpyAsync(v, f->c.v.p, sizeof(double) * f->c.P, cudaMemcpyDeviceToHost, f->c.st));
  ACE_CUDA(cudaStreamSynchronize(f->c.st));
  return 0;
}

int ace_fit_get_invKmatn(ace_fit* f, double* inv) {
  if (!f || !inv) return usage("null argument");
  ACE_CUDA(cudaSetDevice(f->c.device));
  ACE_TRY(f->c.ensure_full_inverse());
  ACE_TRY(download_matrix(inv, f->c.n, f->c.n, f->c.Bf.p, f->c.n_pad, f->c.st));
  ACE_CUDA(cudaStreamSynchronize(f->c.st));
  return 0;
}

int ace_fit_get_alpha(ace_fit* f, double* a) {
  if (!f || !a) return usage("null argument");
  ACE_CUDA(cudaSetDevice(f->c.device));
  ACE_CUDA(cudaMemcpyAsync(a, f->c.alpha.p, sizeof(double) * f->c.n, cudaMemcpyDeviceToHost, f->c.st));
  ACE_CUDA(cudaStreamSynchronize(f->c.st));
  return 0;
}

int ace_fit_dims(ace_fit* f, int* n, int* p, int* B, int* P) {
  if (!f) return usage("null argument");
  if (n) *n = f->c.n;
  if (p) *p = f->c.p;
  if (B) *B = f->c.B;
  if (P) *P = f->c.P;
  return 0;
}

int ace_fit_last_timing(ace_fit* f, double* ms6) {
  if (!f || !ms6) return usage("null argument");
  for (int k = 0; k < 6; ++k) ms6[k] = f->ms[k];
  return 0;
}

}  // extern "C"

// =============================================================================================
// posterior (shared by the handle and the per-function entry points)
// =============================================================================================
namespace ace {

// T = Kx * Kinv (Kinv symmetric), then map / var rows.  Kx: nx_pad x n_pad (ld nx_pad, zero padded),
// kdiag: nx (diag of K_xx).  noise: e^sigma added to the variance (pred_cpp) or 0 (marginal).
struct PostOut {
  DBuf<double> T, map, var, p1, p2;
};

static int posterior_rows(Core& c, const double* Kinv, const double* Kx, const double* kdiag, int nx, int nx_pad,
                          double mu, double noise, PostOut& o) {
  const int n = c.n, n_pad = c.n_pad;
  ACE_TRY(o.T.alloc((size_t)nx_pad * n_pad));
  GemmNT g{};
  g.A = Kx; g.lda = nx_pad; g.B = Kinv; g.ldb = n_pad; g.C = o.T.p; g.ldc = nx_pad;
  g.M = nx_pad; g.N = n_pad; g.K = n_pad; g.alpha = 1.0; g.beta = 0.0;
  ACE_TRY(launch_gemm_nt(g, c.st));
  const int chunks = (n + pk::CHUNK - 1) / pk::CHUNK;
  ACE_TRY(o.p1.alloc((size_t)nx_pad * chunks));
  ACE_TRY(o.p2.alloc((size_t)nx_pad * chunks));
  ACE_TRY(o.map.alloc(nx_pad));
  ACE_TRY(o.var.alloc(nx_pad));
  dim3 grid((nx_pad + pk::ROWS - 1) / pk::ROWS, chunks);
  rowdot2_kernel<<<grid, pk::ROWS, 0, c.st>>>(o.T.p, Kx, nx_pad, nx_pad, n, c.y.p, mu, o.p1.p, o.p2.p);
  ACE_CUDA(cudaGetLastError());
  post_finish_kernel<<<(nx_pad + 255) / 256, 256, 0, c.st>>>(o.p1.p, o.p2.p, chunks, nx, nx_pad, kdiag, noise,
                                                            o.map.p, o.var.p);
  ACE_CUDA(cudaGetLastError());
  return 0;
}

// The same rows from the factor: W = Kx * U (ONE triangular product, half the flops of Kx * K^-1 and no K^-1 at
// all), mean = W (U^T (y - mu)), T Kx^T = rowsum(W^2).  Afac: lower = X = L^-1, diagonal tiles in DX; upper = U, DU.
static int posterior_rows_tri(Core& c, const double* Kx, const double* kdiag, int nx, int nx_pad, double mu,
                              double noise, PostOut& o) {
  const int n = c.n, n_pad = c.n_pad;
  ACE_TRY(o.T.alloc((size_t)nx_pad * n_pad));
  GemmNT g{};
  g.A = Kx; g.lda = nx_pad; g.B = c.A.p; g.ldb = n_pad; g.b_tri = 2; g.Bdiag = c.DX.p;
  g.C = o.T.p; g.ldc = nx_pad;
  g.M = nx_pad; g.N = n_pad; g.K = n_pad; g.alpha = 1.0; g.beta = 0.0;
  ACE_TRY(launch_gemm_nt(g, c.st));
  utv2_kernel<<<(n_pad + 7) / 8, 256, 0, c.st>>>(c.A.p, n_pad, c.DU.p, n, n_pad, c.y.p, c.tvy.p, c.tv1.p);
  ACE_CUDA(cudaGetLastError());
  const int chunks = (n + pk::CHUNK - 1) / pk::CHUNK;
  ACE_TRY(o.p1.alloc((size_t)nx_pad * chunks));
  ACE_TRY(o.p2.alloc((size_t)nx_pad * chunks));
  ACE_TRY(o.map.alloc(nx_pad));
  ACE_TRY(o.var.alloc(nx_pad));
  dim3 grid((nx_pad + pk::ROWS - 1) / pk::ROWS, chunks);
  rowdot_tri_kernel<<<grid, pk::ROWS, 0, c.st>>>(o.T.p, nx_pad, nx_pad, n, c.tvy.p, c.tv1.p, mu, o.p1.p, o.p2.p);
  ACE_CUDA(cudaGetLastError());
  post_finish_kernel<<<(nx_pad + 255) / 256, 256, 0, c.st>>>(o.p1.p, o.p2.p, chunks, nx, nx_pad, kdiag, noise,
                                                            o.map.p, o.var.p);
  ACE_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace ace

extern "C" {

int ace_fit_predict(ace_fit* f, const double* X2, const double* Z2, int nx, double mean_y, double std_y,
                    double* map, double* ci, double* var) {
  if (!f || !X2 || (f->c.Bz > 0 && !Z2) || !map || !ci || !var || nx < 1) return usage("ace_fit_predict: bad argument");
  Core& c = f->c;
  ACE_CUDA(cudaSetDevice(c.device));
  // A sharded fit blocks the test points over the ranks (SURVEY 8e: the factor is replicated, rows are independent);
  // the raw mean / variance rows are all-gathered, so every rank returns the complete result.  Collective call.
  const bool split = c.shard_world > 1 && !c.shard_emulate && c.u_valid && f->comm != nullptr;
  const int G = split ? c.shard_world : 1, r = split ? c.shard_rank : 0;
  const int chunk = round_up((nx + G - 1) / G, TB);  // rows per rank, on the 128 grid
  const int nx_all = chunk * G;                       // padded length of the gathered vectors
  // lo stays on the 128 grid (16-byte aligned TMA sources) and inside the nx_all-sized buffers even when this
  // rank's block lies entirely beyond nx: such a rank computes cnt = 0 rows of zero-padded inputs
  const int lo = r * chunk, cnt = std::max(0, std::min(nx, lo + chunk) - lo);
  DBuf<double> dX2, dZ2, dLZ2, Kx, kd, res;
  ACE_TRY(dX2.alloc((size_t)nx_all * c.p));
  ACE_TRY(dZ2.alloc((size_t)nx_all * std::max(c.Bz, 1)));
  ACE_TRY(dLZ2.alloc((size_t)nx_all * std::max(c.Bz, 1)));
  ACE_TRY(Kx.alloc((size_t)chunk * c.n_pad));
  ACE_TRY(kd.alloc(chunk));
  ACE_TRY(res.alloc((size_t)2 * nx_all));  // [map of all ranks | var of all ranks]
  ACE_TRY(upload_matrix(dX2.p, nx_all, nx_all, X2, nx, c.p, c.st));
  ACE_TRY(upload_matrix(dZ2.p, nx_all, nx_all, Z2, nx, c.Bz, c.st));
  if (c.Bz > 0)
    logabs_kernel<<<(unsigned)(((size_t)nx_all * c.Bz + 255) / 256), 256, 0, c.st>>>(dZ2.p, dLZ2.p, (size_t)nx_all * c.Bz);
  ACE_CUDA(cudaGetLastError());
  ACE_TRY(c.enqueue_prep());  // kernels built from the CURRENT parameters (R/kernel_SE_R6.R:78-79)
  KernArgs a{};
  a.X1 = dX2.p + lo; a.Z1 = dZ2.p + lo; a.LZ1 = dLZ2.p + lo; a.ld1 = nx_all;
  a.X2 = c.X.p; a.Z2 = c.Z.p; a.LZ2 = c.LZ.p; a.ld2 = c.n_pad;
  a.n1 = cnt; a.n2 = c.n; a.n1_pad = chunk; a.n2_pad = c.n_pad; a.p = c.p; a.B = c.B; a.tab = c.tab.p;
  a.K = Kx.p; a.ldk = chunk;
  ACE_TRY(launch_kernmat(a, c.kind, c.st));
  kdiag_kernel<<<(chunk + 255) / 256, 256, 0, c.st>>>(dZ2.p + lo, dLZ2.p + lo, nx_all, cnt, c.B, c.kind, c.tab.p, 0, kd.p);
  ACE_CUDA(cudaGetLastError());
  double hpar[2];
  ACE_CUDA(cudaMemcpyAsync(hpar, c.theta.p, sizeof(double) * 2, cudaMemcpyDeviceToHost, c.st));
  ACE_CUDA(cudaStreamSynchronize(c.st));
  PostOut o;
  if (c.u_valid) {
    ACE_TRY(posterior_rows_tri(c, Kx.p, kd.p, cnt, chunk, hpar[1], std::exp(hpar[0]), o));
  } else {
    ACE_TRY(c.ensure_full_inverse());
    ACE_TRY(posterior_rows(c, c.Bf.p, Kx.p, kd.p, cnt, chunk, hpar[1], std::exp(hpar[0]), o));
  }
  ACE_CUDA(cudaMemcpyAsync(res.p + (size_t)r * chunk, o.map.p, sizeof(double) * chunk, cudaMemcpyDeviceToDevice, c.st));
  ACE_CUDA(cudaMemcpyAsync(res.p + nx_all + (size_t)r * chunk, o.var.p, sizeof(double) * chunk, cudaMemcpyDeviceToDevice,
                           c.st));
  if (split) {
    NcclApi& nc = nccl_api();
    ACE_NCCL(nc.GroupStart());
    ACE_NCCL(nc.AllGather(res.p + (size_t)r * chunk, res.p, chunk, ncclFloat64, f->comm, c.st));
    ACE_NCCL(nc.AllGather(res.p + nx_all + (size_t)r * chunk, res.p + nx_all, chunk, ncclFloat64, f->comm, c.st));
    ACE_NCCL(nc.GroupEnd());
  }
  std::vector<double> h((size_t)2 * nx_all);
  ACE_CUDA(cudaMemcpyAsync(h.data(), res.p, sizeof(double) * 2 * nx_all, cudaMemcpyDeviceToHost, c.st));
  ACE_CUDA(cudaStreamSynchronize(c.st));
  for (int i = 0; i < nx; ++i) {  // src/pred_cpp.cpp:20,26-29; point i sits at i (rank block i / chunk, offset i % chunk)
    map[i] = mean_y + std_y * (h[i] + hpar[1]);
    const double sd = std_y * std::sqrt(std::fabs(h[(size_t)nx_all + i]));
    ci[i] = map[i] - 1.96 * sd;
    ci[i + nx] = map[i] + 1.96 * sd;
    var[i] = sd * sd;
  }
  return 0;
}

}  // extern "C"

#include "api_functions.inl"
