// chol.cuh -- blocked FP64 Cholesky, triangular inverse and SPD inverse on the 128-block grid.
//
// Replaces invkernel_cpp's eigendecomposition route (src/kernel_SE_cpp.cpp:137-157:
// K + e^sigma I = V L V', inv = (V L^-1/2)(V L^-1/2)', logdet = sum log lambda) by
//   phase 1  potrf   A = L L'            right-looking, panel width 512 with one-panel look-ahead
//   phase 2  trtri   U = L^-T            bottom-up pairwise merge, strided-batched per level
//   phase 3  U U'    (K + e^sigma I)^-1  ONE triangular SYRK launch, mirrored on the fly: DMMA, or from
//                    n_pad >= UUT_I8_MIN_N the INT8 Ozaki (CRT) engine of uut_i8.cuh
// with logdet = 2 sum log L_ii.  Phases 1 and 2 run every O(n^3) flop in dgemm_nt_kernel (DMMA); the only
// other kernels are the two 128-wide leaf kernels below.  n^3 flops in total (n^3/3 per phase).
//
// Storage (column-major, ld = n_pad, n_pad a multiple of 128, padding = identity):
//   lower(A)  : L, later X = L^-1 (needed as operands while merging)
//   upper(A)  : U = L^-T (strictly-upper 128-blocks)
//   DX, DU    : dense 128x128 tiles holding the diagonal blocks of X (lower) and U (upper)
//   dvec      : diag(L)
//   Bf        : workspace during phase 2, receives the full symmetric inverse in phase 3
#pragma once
#include "dgemm_nt.cuh"
#include "fastmath.cuh"
#include "diag_block.cuh"
#include "uut_i8.cuh"

#include <cstdlib>
#include <vector>

namespace ace {

// ---------------------------------------------------------------------------------------------
// Leaf: Cholesky of one 128x128 diagonal tile + inverse of its factor, one CTA.
// The tile lives in registers (16x16 threads, cyclic 8x8 elements each); one __syncthreads per
// column thanks to double-buffered pivot columns/rows.
// ---------------------------------------------------------------------------------------------
namespace leaf {
constexpr int LD = 129;
constexpr size_t SMEM_BYTES = (size_t)(128 * LD + 2 * 128 + 2 * 128 + 128 + 128) * 8;
}  // namespace leaf

template <int JB>
__device__ __forceinline__ void leaf_chol_block(double (&r)[8][8], double* Ls, double* colbuf, double* dg, double* idg,
                                                int tx, int ty, int* info, int blk) {
  using namespace leaf;
#pragma unroll 1
  for (int jx = 0; jx < 16; ++jx) {
    const int j = 16 * JB + jx;
    double* cb = colbuf + (j & 1) * 128;
    if (tx == jx) {
#pragma unroll
      for (int a = JB; a < 8; ++a) {
        const int i = 16 * a + ty;
        if (i >= j) cb[i] = r[a][JB];
      }
    }
    __syncthreads();
    const double pj = cb[j];
    // one MUFU-seeded reciprocal square root serves everything on the critical path of this column:
    // 1/L_jj = y, L_jj = p y, 1/p = y^2 (no IEEE division / sqrt: their latency was ~2/3 of a step)
    const double inv = fast_rsqrt(pj);
    if (tx == jx) {
#pragma unroll
      for (int a = JB; a < 8; ++a) {
        const int i = 16 * a + ty;
        if (i > j) Ls[i + j * LD] = r[a][JB] * inv;
        if (i == j) {
          double s = pj * inv;
          s = fma(fma(-s, s, pj), 0.5 * inv, s);
          dg[j] = s;
          idg[j] = inv;
          if (!(pj > 0.0)) atomicCAS(info, 0, blk * 128 + j + 1);
        }
      }
    }
    const double invp = inv * inv;
    // Branch-free rank-1 update of the trailing part held in registers.  Only the block row a == JB and
    // the block column b == JB straddle the pivot, so only those need a mask; entries above the diagonal
    // inside diagonal blocks are never read, so no k <= i test at all.
    double lm[8], cm[8];
#pragma unroll
    for (int a = JB; a < 8; ++a) {
      lm[a] = cb[16 * a + ty] * invp;
      cm[a] = cb[16 * a + tx];
    }
    lm[JB] = (ty > jx) ? lm[JB] : 0.0;
    cm[JB] = (tx > jx) ? cm[JB] : 0.0;
#pragma unroll
    for (int a = JB; a < 8; ++a)
#pragma unroll
      for (int b = JB; b <= a; ++b) r[a][b] = fma(-lm[a], cm[b], r[a][b]);
  }
}

template <int JB>
__device__ __forceinline__ void leaf_inv_block(double (&r)[8][8], double* Ls, double* rowbuf, const double* idg,
                                               int tx, int ty) {
  using namespace leaf;
#pragma unroll 1
  for (int jx = 0; jx < 16; ++jx) {
    const int j = 16 * JB + jx;
    double* rb = rowbuf + (j & 1) * 128;
    if (ty == jx) {  // owners of row j (a == JB)
      const double dj = idg[j];
#pragma unroll
      for (int b = 0; b <= JB; ++b) {
        const int k = 16 * b + tx;
        if (k <= j) {
          const double x = r[JB][b] * dj;
          rb[k] = x;
          if (k < j) Ls[k + j * LD] = x;  // U(k,j) = X(j,k) into the (still unused) upper triangle
        }
      }
    }
    __syncthreads();
    // branch-free: rows i <= j (only possible for a == JB) and columns k > j (only for b == JB) get a zero
    double lm[8], xm[8];
#pragma unroll
    for (int a = JB; a < 8; ++a) lm[a] = Ls[16 * a + ty + j * LD];
    lm[JB] = (ty > jx) ? lm[JB] : 0.0;
#pragma unroll
    for (int b = 0; b <= JB; ++b) xm[b] = rb[16 * b + tx];
    xm[JB] = (tx <= jx) ? xm[JB] : 0.0;
#pragma unroll
    for (int a = JB; a < 8; ++a)
#pragma unroll
      for (int b = 0; b <= JB; ++b) r[a][b] = fma(-lm[a], xm[b], r[a][b]);
  }
}

// A: matrix base, tile blk on its diagonal.  Writes L (lower of the tile), DX/DU tiles, dvec, info.
__global__ void __launch_bounds__(256, 1) potrf_leaf_kernel(double* __restrict__ A, long ld, int blk,
                                                            double* __restrict__ DX, double* __restrict__ DU,
                                                            double* __restrict__ dvec, int* info) {
  using namespace leaf;
  extern __shared__ __align__(16) double sm[];
  double* Ls = sm;
  double* colbuf = Ls + 128 * LD;
  double* rowbuf = colbuf + 256;
  double* dg = rowbuf + 256;
  double* idg = dg + 128;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  double* At = A + (size_t)blk * 128 * (ld + 1);

  for (int idx = threadIdx.x; idx < 128 * 128; idx += 256) {
    const int i = idx & 127, k = idx >> 7;
    Ls[i + k * LD] = At[i + (size_t)k * ld];
  }
  __syncthreads();
  double r[8][8];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      const int i = 16 * a + ty, k = 16 * b + tx;
      r[a][b] = (k <= i) ? Ls[i + k * LD] : 0.0;
    }
  __syncthreads();

  leaf_chol_block<0>(r, Ls, colbuf, dg, idg, tx, ty, info, blk);
  leaf_chol_block<1>(r, Ls, colbuf, dg, idg, tx, ty, info, blk);
  leaf_chol_block<2>(r, Ls, colbuf, dg, idg, tx, ty, info, blk);
  leaf_chol_block<3>(r, Ls, colbuf, dg, idg, tx, ty, info, blk);
  leaf_chol_block<4>(r, Ls, colbuf, dg, idg, tx, ty, info, blk);
  leaf_chol_block<5>(r, Ls, colbuf, dg, idg, tx, ty, info, blk);
  leaf_chol_block<6>(r, Ls, colbuf, dg, idg, tx, ty, info, blk);
  leaf_chol_block<7>(r, Ls, colbuf, dg, idg, tx, ty, info, blk);
  __syncthreads();
  // idg = 1/diag(L) was filled column by column above
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) r[a][b] = (16 * a + ty == 16 * b + tx) ? 1.0 : 0.0;
  __syncthreads();

  leaf_inv_block<0>(r, Ls, rowbuf, idg, tx, ty);
  leaf_inv_block<1>(r, Ls, rowbuf, idg, tx, ty);
  leaf_inv_block<2>(r, Ls, rowbuf, idg, tx, ty);
  leaf_inv_block<3>(r, Ls, rowbuf, idg, tx, ty);
  leaf_inv_block<4>(r, Ls, rowbuf, idg, tx, ty);
  leaf_inv_block<5>(r, Ls, rowbuf, idg, tx, ty);
  leaf_inv_block<6>(r, Ls, rowbuf, idg, tx, ty);
  leaf_inv_block<7>(r, Ls, rowbuf, idg, tx, ty);
  __syncthreads();

  double* DXt = DX + (size_t)blk * 128 * 128;
  double* DUt = DU + (size_t)blk * 128 * 128;
  for (int idx = threadIdx.x; idx < 128 * 128; idx += 256) {
    const int i = idx & 127, k = idx >> 7;  // i fast: coalesced global writes
    if (i > k) {
      At[i + (size_t)k * ld] = Ls[i + k * LD];
      DXt[idx] = Ls[k + i * LD];
      DUt[idx] = 0.0;
    } else if (i == k) {
      At[i + (size_t)k * ld] = dg[i];
      DXt[idx] = idg[i];
      DUt[idx] = idg[i];
    } else {
      DXt[idx] = 0.0;
      DUt[idx] = Ls[i + k * LD];
    }
  }
  if (threadIdx.x < 128) dvec[blk * 128 + threadIdx.x] = dg[threadIdx.x];
}

// ---------------------------------------------------------------------------------------------
// Panel x 128-wide triangular block, in place:  P <- P * DX^T  (the leaf of the blocked TRSM
// X L^T = P, with DX = L_kk^-1).  One CTA owns 64 full rows, so in-place is race free.
// ---------------------------------------------------------------------------------------------
namespace trsml {
constexpr int ROWS = 64, LDA = ROWS + 4, LDB = 128 + 4, KH = 64;
// A tile (all 128 k) + HALF of DX at a time: 137 KB, so that the kernel can take the slot next to a resident
// dgemm_nt CTA (77 KB) instead of waiting for a completely empty SM behind the trailing update
constexpr size_t SMEM_BYTES = (size_t)(128 * LDA + KH * LDB) * 8 + 16;
constexpr uint32_t TX0_BYTES = (128 * ROWS + KH * 128) * 8, TX1_BYTES = KH * 128 * 8;
}  // namespace trsml

__global__ void __launch_bounds__(128, 1) trsm_leaf_kernel(double* __restrict__ P, long ld,
                                                           const double* __restrict__ DXt) {
  using namespace trsml;
  extern __shared__ __align__(128) unsigned char smraw[];
  double* As = reinterpret_cast<double*>(smraw);
  double* Bs = As + 128 * LDA;
  uint64_t* bar = reinterpret_cast<uint64_t*>(Bs + KH * LDB);  // bar[0]: A + DX[:, 0:64), bar[1]: DX[:, 64:128)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* Pr = P + (size_t)blockIdx.x * ROWS;
  if (threadIdx.x == 0) {
    mbar_init(&bar[0], 1);
    mbar_init(&bar[1], 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (warp == 0) {
    if (lane == 0) mbar_arrive_expect_tx(&bar[0], TX0_BYTES);
    __syncwarp();
    for (int kk = lane; kk < 128; kk += 32) tma_bulk_g2s(As + kk * LDA, Pr + (size_t)kk * ld, ROWS * 8, &bar[0]);
    for (int kk = lane; kk < KH; kk += 32) tma_bulk_g2s(Bs + kk * LDB, DXt + (size_t)kk * 128, 128 * 8, &bar[0]);
  }
  mbar_wait(&bar[0], 0);

  const int g = lane >> 2, tq = lane & 3;
  double acc[8][4][2];
#pragma unroll
  for (int mt = 0; mt < 8; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
  const double* as = As + g;
  const double* bs = Bs + warp * 32 + g;
  const int ks_end = 8 * (warp + 1);  // DX lower triangular: column j only needs k <= j
#pragma unroll 1
  for (int half = 0; half < 2; ++half) {
    if (half == 1) {
      __syncthreads();  // everybody is done with DX[:, 0:64) before it is overwritten
      if (warp == 0) {
        if (lane == 0) mbar_arrive_expect_tx(&bar[1], TX1_BYTES);
        __syncwarp();
        for (int kk = lane; kk < KH; kk += 32)
          tma_bulk_g2s(Bs + kk * LDB, DXt + (size_t)(KH + kk) * 128, 128 * 8, &bar[1]);
      }
      if (ks_end <= KH / 4) break;  // warps 0 and 1 only need k < 64 (uniform per warp; no later barrier)
      mbar_wait(&bar[1], 0);
    }
    const int ks_lo = half * (KH / 4), ks_hi = min(ks_end, (half + 1) * (KH / 4));
#pragma unroll 2
    for (int ks = ks_lo; ks < ks_hi; ++ks) {
      const int k = ks * 4 + tq;
      double a[8], b[4];
#pragma unroll
      for (int mt = 0; mt < 8; ++mt) a[mt] = as[k * LDA + mt * 8];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) b[nt] = bs[(k - half * KH) * LDB + nt * 8];
#pragma unroll
      for (int mt = 0; mt < 8; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) dmma884(acc[mt][nt][0], acc[mt][nt][1], a[mt], b[nt]);
    }
  }
  const int col0 = warp * 32 + 2 * tq;
#pragma unroll
  for (int nt = 0; nt < 4; ++nt)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      double* cc = Pr + (size_t)(col0 + nt * 8 + e) * ld + g;
#pragma unroll
      for (int mt = 0; mt < 8; ++mt) cc[mt * 8] = acc[mt][nt][e];
    }
}

// ---------------------------------------------------------------------------------------------
// Host-side drivers
// ---------------------------------------------------------------------------------------------
// optional poor-man's timeline of the look-ahead schedule (ACE_POTRF_TRACE=1 in ace_bench_dense)
struct PotrfTrace {
  std::vector<cudaEvent_t> panel_begin, panel_end, upd_begin, upda_end, updb_end;
  cudaEvent_t t0 = nullptr;
};

struct DenseWork {
  double* A = nullptr;     // n_pad x n_pad
  long ld = 0;
  int nb = 0;              // n_pad / 128
  double* DX = nullptr;    // nb tiles
  double* DU = nullptr;    // nb tiles
  double* dvec = nullptr;  // n_pad
  int* info = nullptr;     // device int: 0, or 1-based index of the first non-positive pivot
  double* Bf = nullptr;    // n_pad x n_pad: workspace, then the inverse
  cudaStream_t main = nullptr, side = nullptr, aux = nullptr;
  cudaStream_t bg = nullptr;  // background stream of the incremental inverse (lowest priority)
  cudaEvent_t ev_panel[2] = {nullptr, nullptr}, ev_upd[2] = {nullptr, nullptr};
  cudaEvent_t ev_half = nullptr, ev_aux = nullptr;  // overlap of the leading block's inverse with the potrf tail
  int panel_blocks = 4;    // look-ahead panel width in 128-blocks (512 columns)
  PotrfTrace* trace = nullptr;
  // fused panel TRSM (production path): after a diagonal block is factored its inverse X_JJ is formed at once
  // (the first log2(panel) merge levels of phase 2, done early) and the rows below are solved by ONE GEMM
  // P X_JJ^T into Wp[J&1] instead of a chain of 7 slot-starved 128-wide kernels; the trailing update reads the
  // panel from Wp, a copy back into A follows off the critical path (aux stream).
  double* Wp[2] = {nullptr, nullptr};  // n_pad x (panel_blocks*128) each, ld = n_pad
  double* Wsmall = nullptr;            // (panel_blocks*128/2)^2 doubles: workspace of the early merges
  cudaEvent_t ev_copy[2] = {nullptr, nullptr};
  // fused diagonal-block kernel (diag_block.cuh): scratch of dg::ws_doubles(panel_blocks) doubles; nullptr = the
  // recursion of 128-wide leaf kernels + early merge levels (ACE_DIAG_FUSED=0)
  double* diag_ws = nullptr;
  long long* diag_dbg = nullptr;  // debug: phase clock stamps of the diagonal-block kernel
  OzWork oz;                      // residue planes of the INT8 U U^T engine (allocated when uut_uses_i8 selects it)
  int uut_engine = 0;             // debug pin of the U U^T engine: 0 by size, 1 DMMA, 2 INT8
};

inline int configure_dense_kernels() {
  ACE_CUDA(cudaFuncSetAttribute(dgemm_nt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)gemm::SMEM_BYTES));
  ACE_CUDA(cudaFuncSetAttribute(potrf_leaf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)leaf::SMEM_BYTES));
  ACE_CUDA(cudaFuncSetAttribute(trsm_leaf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)trsml::SMEM_BYTES));
  ACE_TRY(configure_diag_kernel());
  ACE_TRY(configure_uut_i8_kernel());
  return 0;
}

inline double* blkptr(const DenseWork& w, int rb, int cb) { return w.A + (size_t)rb * TB + (size_t)cb * TB * w.ld; }

inline int gemm_plain(const DenseWork& w, const double* A, const double* B, double* C, int M, int N, int K,
                      double alpha, double beta, int lower_only, cudaStream_t st) {
  GemmNT p{};
  p.A = A; p.lda = w.ld; p.B = B; p.ldb = w.ld; p.C = C; p.ldc = w.ld;
  p.M = M; p.N = N; p.K = K; p.alpha = alpha; p.beta = beta; p.lower_only = lower_only;
  return launch_gemm_nt(p, st);
}

// rows [r0,r1) x tri [a,c):  A[r0:r1, a:c] <- A[r0:r1, a:c] * L[a:c,a:c]^-T   (recursive TRSM)
inline int trsm_rec(const DenseWork& w, int r0, int r1, int a, int c, cudaStream_t st) {
  if (r1 <= r0) return 0;
  if (c - a == 1) {
    trsm_leaf_kernel<<<(unsigned)((r1 - r0) * TB / trsml::ROWS), 128, trsml::SMEM_BYTES, st>>>(
        blkptr(w, r0, a), w.ld, w.DX + (size_t)a * TB * TB);
    ACE_CUDA(cudaGetLastError());
    return 0;
  }
  const int m = a + (c - a + 1) / 2;
  ACE_TRY(trsm_rec(w, r0, r1, a, m, st));
  ACE_TRY(gemm_plain(w, blkptr(w, r0, a), blkptr(w, m, a), blkptr(w, r0, m), (r1 - r0) * TB, (c - m) * TB,
                     (m - a) * TB, -1.0, 1.0, 0, st));
  return trsm_rec(w, r0, r1, m, c, st);
}

// Cholesky of the diagonal block range [a,b) (small, runs on one stream)
inline int potrf_rec(const DenseWork& w, int a, int b, cudaStream_t st) {
  if (b - a == 1) {
    potrf_leaf_kernel<<<1, 256, leaf::SMEM_BYTES, st>>>(w.A, w.ld, a, w.DX, w.DU, w.dvec, w.info);
    ACE_CUDA(cudaGetLastError());
    return 0;
  }
  const int c = a + (b - a + 1) / 2;
  ACE_TRY(potrf_rec(w, a, c, st));
  ACE_TRY(trsm_rec(w, c, b, a, c, st));
  ACE_TRY(gemm_plain(w, blkptr(w, c, a), blkptr(w, c, a), blkptr(w, c, c), (b - c) * TB, (b - c) * TB,
                     (c - a) * TB, -1.0, 1.0, 1, st));
  return potrf_rec(w, c, b, st);
}

inline int trtri_merge_range(const DenseWork& w, int lo, int hi, cudaStream_t st, double* ws, int h_min = 1);

// Diagonal block [j0, j1) of the panel schedule: L_JJ, X_JJ = L_JJ^-1 (lower 128-blocks), U_JJ (upper), DX / DU tiles,
// dvec.  One cluster launch (diag_block.cuh), or the leaf recursion followed by the early merge levels.
// `share` = how many ranks split the trailing work (1 on a single GPU): the 16-CTA cluster halves the block's latency
// but has to gather 16 free SMs of one GPC, which costs throughput while the trailing updates still fill the GPU
// (C3 on one GPU: 89.1 ms with 8 CTAs, 90.5 with 16); it is used once the remaining trailing matrix per rank is
// small enough for the chain of diagonal blocks to bound the factorisation.
inline int diag_block_factor_invert(const DenseWork& w, int j0, int j1, cudaStream_t st, int share = 1) {
  if (w.diag_ws != nullptr) {
    DiagArgs a{};
    a.A = w.A; a.ld = w.ld; a.blk0 = j0; a.nblk = j1 - j0; a.DX = w.DX; a.DU = w.DU; a.dvec = w.dvec; a.info = w.info;
    a.S = w.diag_ws;
    a.W = w.diag_ws + (size_t)w.panel_blocks * TB * w.panel_blocks * TB;
    a.dbg = w.diag_dbg;
    const long rest = (long)(w.nb - j1) * TB;  // rows below this block
    return launch_diag_block(a, st, rest <= 6144L * share);
  }
  ACE_TRY(potrf_rec(w, j0, j1, st));
  return trtri_merge_range(w, j0, j1, st, w.Wsmall);
}

// Phase 1: right-looking blocked Cholesky with one-panel look-ahead on two streams.
//   panel(J)  : factor the diagonal block + TRSM of the rows below it        (side stream)
//   upd_a(J)  : trailing update restricted to the next panel's block column  (main stream)
//   upd_b(J)  : the rest of the trailing update                              (main stream)
// panel(J+1) only waits for upd_a(J), so it overlaps upd_b(J).
// fork_at > 0: as soon as the leading fork_at block rows/columns of L are final, their triangular inverse is
// started on the aux stream (it only touches A[0:fork_at, 0:fork_at], which potrf never reads again); the
// caller joins on ev_aux.  The tail of a Cholesky is latency bound (a chain of 128-wide leaf kernels with
// almost no trailing work), so this fills otherwise idle SMs.
inline int potrf_blocked(const DenseWork& w, int fork_at = 0, int fork_when = 0, bool incremental = false) {
  const int nb = w.nb, pb = w.panel_blocks;
  bool forked = false;
  ACE_CUDA(cudaMemsetAsync(w.info, 0, sizeof(int), w.main));
  // fork: side stream joins after everything already queued on main
  ACE_CUDA(cudaEventRecord(w.ev_upd[1], w.main));
  ACE_CUDA(cudaStreamWaitEvent(w.side, w.ev_upd[1], 0));
  int J = 0;
  for (int j0 = 0; j0 < nb; j0 += pb, ++J) {
    const int j1 = min(j0 + pb, nb), j2 = min(j1 + pb, nb);
    // ---- panel(J) on the side stream
    auto mark = [&](std::vector<cudaEvent_t>* v, cudaStream_t st) {
      if (!v) return;
      cudaEvent_t e;
      cudaEventCreate(&e);
      cudaEventRecord(e, st);
      v->push_back(e);
    };
    mark(w.trace ? &w.trace->panel_begin : nullptr, w.side);
    const bool fused = (w.Wp[0] != nullptr);
    const double* panel = blkptr(w, j1 < nb ? j1 : j0, j0);  // operand of the trailing update
    if (!fused) {
      ACE_TRY(potrf_rec(w, j0, j1, w.side));
      ACE_TRY(trsm_rec(w, j1, nb, j0, j1, w.side));
    } else {
      ACE_TRY(diag_block_factor_invert(w, j0, j1, w.side));  // L_JJ, X_JJ (lower blocks of the diagonal block), U_JJ
      if (j1 < nb) {
        if (J >= 2) ACE_CUDA(cudaStreamWaitEvent(w.side, w.ev_copy[J & 1], 0));  // Wp[J&1] free again
        GemmNT t{};
        t.A = blkptr(w, j1, j0); t.lda = w.ld;
        t.B = blkptr(w, j0, j0); t.ldb = w.ld; t.b_tri = 2; t.Bdiag = w.DX + (size_t)j0 * TB * TB;
        t.C = w.Wp[J & 1] + (size_t)j1 * TB; t.ldc = w.ld;
        t.M = (nb - j1) * TB; t.N = (j1 - j0) * TB; t.K = (j1 - j0) * TB; t.alpha = 1.0; t.beta = 0.0;
        ACE_TRY(launch_gemm_nt(t, w.side));
        panel = w.Wp[J & 1] + (size_t)j1 * TB;
      }
    }
    mark(w.trace ? &w.trace->panel_end : nullptr, w.side);
    ACE_CUDA(cudaEventRecord(w.ev_panel[J & 1], w.side));
    if (fused && j1 < nb) {  // solved panel back into A (phase 2 reads it as L21), off the critical path
      ACE_CUDA(cudaStreamWaitEvent(w.aux, w.ev_panel[J & 1], 0));
      ACE_CUDA(cudaMemcpy2DAsync(blkptr(w, j1, j0), sizeof(double) * w.ld, w.Wp[J & 1] + (size_t)j1 * TB,
                                 sizeof(double) * w.ld, sizeof(double) * (size_t)(nb - j1) * TB, (size_t)(j1 - j0) * TB,
                                 cudaMemcpyDeviceToDevice, w.aux));
      ACE_CUDA(cudaEventRecord(w.ev_copy[J & 1], w.aux));
    }
    if (incremental && fused && J >= 1) {
      // Incremental inverse: as soon as block row J of L is final and X_JJ is known, the rows X[J, 0:j0] follow
      // from the leading inverse -- the merge of [0,j0) with [j0,j1) -- on the low-priority stream, filling the
      // SM time the latency-bound panel chain leaves idle.  In stream order after all earlier merges and copies.
      cudaStream_t bg = w.bg ? w.bg : w.aux;
      ACE_CUDA(cudaStreamWaitEvent(bg, w.ev_panel[J & 1], 0));        // X_JJ
      ACE_CUDA(cudaStreamWaitEvent(bg, w.ev_copy[(J - 1) & 1], 0));   // block row J of L is in A (copies are in order)
      const int s1 = j0 * TB, s2 = (j1 - j0) * TB;
      GemmNT p{};
      p.A = w.A; p.lda = w.ld; p.a_tri = 1; p.Adiag = w.DU;
      p.B = blkptr(w, j0, 0); p.ldb = w.ld;
      p.C = w.Bf; p.ldc = s1;
      p.M = s1; p.N = s2; p.K = s1; p.alpha = 1.0; p.beta = 0.0;
      ACE_TRY(launch_gemm_nt(p, bg));
      GemmNT r{};
      r.A = blkptr(w, j0, j0); r.lda = w.ld; r.a_tri = 2; r.Adiag = w.DX + (size_t)j0 * TB * TB;
      r.B = w.Bf; r.ldb = s1;
      r.C = blkptr(w, j0, 0); r.ldc = w.ld;
      r.Ct = blkptr(w, 0, j0); r.ldct = w.ld;
      r.M = s2; r.N = s1; r.K = s2; r.alpha = -1.0; r.beta = 0.0;
      ACE_TRY(launch_gemm_nt(r, bg));
      ACE_CUDA(cudaEventRecord(w.ev_aux, bg));
      forked = true;
    }
    if (fork_at > 0 && !forked && j1 >= fork_at && j1 >= fork_when && j1 < nb) {
      ACE_CUDA(cudaEventRecord(w.ev_half, w.side));
      ACE_CUDA(cudaStreamWaitEvent(w.aux, w.ev_half, 0));
      ACE_TRY(trtri_merge_range(w, 0, fork_at, w.aux, w.Bf, w.Wp[0] ? w.panel_blocks : 1));
      ACE_CUDA(cudaEventRecord(w.ev_aux, w.aux));
      forked = true;
    }
    if (j1 >= nb) break;
    // ---- trailing update on the main stream
    ACE_CUDA(cudaStreamWaitEvent(w.main, w.ev_panel[J & 1], 0));
    const int K = (j1 - j0) * TB;
    mark(w.trace ? &w.trace->upd_begin : nullptr, w.main);
    // upd_a: rows [j1,nb) x cols [j1,j2)
    ACE_TRY(gemm_plain(w, panel, panel, blkptr(w, j1, j1), (nb - j1) * TB, (j2 - j1) * TB, K, -1.0, 1.0, 0, w.main));
    mark(w.trace ? &w.trace->upda_end : nullptr, w.main);
    ACE_CUDA(cudaEventRecord(w.ev_upd[J & 1], w.main));
    ACE_CUDA(cudaStreamWaitEvent(w.side, w.ev_upd[J & 1], 0));
    // upd_b: square block [j2,nb) lower tiles
    if (j2 < nb)
      ACE_TRY(gemm_plain(w, panel + (size_t)(j2 - j1) * TB, panel + (size_t)(j2 - j1) * TB, blkptr(w, j2, j2),
                         (nb - j2) * TB, (nb - j2) * TB, K, -1.0, 1.0, 1, w.main));
    mark(w.trace ? &w.trace->updb_end : nullptr, w.main);
  }
  // join
  ACE_CUDA(cudaStreamWaitEvent(w.main, w.ev_panel[J & 1], 0));
  if (w.Wp[0] != nullptr && J >= 1) {
    ACE_CUDA(cudaStreamWaitEvent(w.main, w.ev_copy[0], 0));
    if (J >= 2) ACE_CUDA(cudaStreamWaitEvent(w.main, w.ev_copy[1], 0));
  }
  return forked ? 1 : 0;
}

// Phase 2: U = L^-T into upper(A) (and X = L^-1 into lower(A)) by bottom-up pairwise merging.
// For a node with children [a,c) and [c,b):   X21 = -X22 * L21 * X11, done as two NT GEMMs
//   Wt  = U11 * L21^T              (A operand upper triangular, diagonal tiles from DU)
//   X21 = -X22 * Wt^T, U12 = X21^T (A operand lower triangular, diagonal tiles from DX; dual store)
// Wt lives in Bf.  All nodes of one level are independent; equal-shaped ones go in one batched launch.
inline int& dbg_trtri_max_h() {
  static int v = 1 << 30;
  return v;
}

// one level (child size h) of the merges lying inside the block range [lo, lo + len)
inline int trtri_level(const DenseWork& w, int lo, int len, int h, cudaStream_t st, double* ws) {
  const int nodes = (len + 2 * h - 1) / (2 * h);
  const int s1 = h * TB;
  // regular nodes (full right child) q = 0 .. nreg-1 in one strided-batched launch, ragged last node alone
  int nreg = 0;
  while (nreg < nodes && (nreg * 2 * h + 2 * h) <= len) ++nreg;
  for (int pass = 0; pass < 2; ++pass) {
    int q0, cnt, s2;
    if (pass == 0) {
      q0 = 0; cnt = nreg; s2 = s1;
    } else {
      q0 = nreg; cnt = nodes - nreg;  // 0 or 1
      if (cnt == 0) break;
      const int c_local = q0 * 2 * h + h;
      if (c_local >= len) break;  // lone left child, nothing to merge
      s2 = (len - c_local) * TB;
    }
    if (cnt == 0) continue;
    const int a = lo + q0 * 2 * h, c = a + h;
    const long node_stride = (long)2 * h * TB * (w.ld + 1);
    double* Wt = ws + (size_t)q0 * s1 * s1;
    GemmNT p{};
    p.A = blkptr(w, a, a); p.lda = w.ld; p.a_tri = 1; p.Adiag = w.DU + (size_t)a * TB * TB;
    p.B = blkptr(w, c, a); p.ldb = w.ld;
    p.C = Wt; p.ldc = s1;
    p.M = s1; p.N = s2; p.K = s1; p.alpha = 1.0; p.beta = 0.0;
    p.batch = cnt; p.sA = node_stride; p.sB = node_stride; p.sC = (long)s1 * s1;
    p.sAdiag = (long)2 * h * TB * TB;
    ACE_TRY(launch_gemm_nt(p, st));
    GemmNT r{};
    r.A = blkptr(w, c, c); r.lda = w.ld; r.a_tri = 2; r.Adiag = w.DX + (size_t)c * TB * TB;
    r.B = Wt; r.ldb = s1;
    r.C = blkptr(w, c, a); r.ldc = w.ld;
    r.Ct = blkptr(w, a, c); r.ldct = w.ld;
    r.M = s2; r.N = s1; r.K = s2; r.alpha = -1.0; r.beta = 0.0;
    r.batch = cnt; r.sA = node_stride; r.sB = (long)s1 * s1; r.sC = node_stride; r.sCt = node_stride;
    r.sAdiag = (long)2 * h * TB * TB;
    ACE_TRY(launch_gemm_nt(r, st));
  }
  return 0;
}

// all levels of the merges inside [lo, hi); workspace need <= ((hi - lo) * 128 / 2)^2 doubles
inline int trtri_merge_range(const DenseWork& w, int lo, int hi, cudaStream_t st, double* ws, int h_min) {
  for (int h = h_min; h < hi - lo && h <= dbg_trtri_max_h(); h *= 2) ACE_TRY(trtri_level(w, lo, hi - lo, h, st, ws));
  return 0;
}

// levels below the panel width were already merged panel by panel when the fused panel TRSM is on
inline int trtri_hmin(const DenseWork& w) { return w.Wp[0] ? w.panel_blocks : 1; }

inline int trtri_merge(const DenseWork& w) { return trtri_merge_range(w, 0, w.nb, w.main, w.Bf, trtri_hmin(w)); }

// Phases 1 + 2 with the inverse of the leading h_top x h_top block (h_top = largest power of two < nb, the
// left child of the top-level merge) overlapped with the latency-bound tail of the Cholesky.
inline int potrf_trtri(const DenseWork& w) {
  const int nb = w.nb;
  int h_top = 1;
  while (2 * h_top < nb) h_top *= 2;
  if (nb < 8 || w.aux == nullptr || dbg_trtri_max_h() < (1 << 30)) {
    int s = potrf_blocked(w);
    if (s < 0) return s;
    return trtri_merge(w);
  }
  // default: incremental inverse behind the panels whenever the fused panel path (early X_JJ) is on; measured at
  // n = 16384: potrf + trtri 95.5 -> 88.4 ms (ACE_INCR_TRTRI=0 restores the fork-at-3/4 schedule below)
  static const int incr = std::getenv("ACE_INCR_TRTRI") ? std::atoi(std::getenv("ACE_INCR_TRTRI")) : 1;
  if (incr && w.Wp[0] != nullptr) {
    const int forked = potrf_blocked(w, 0, 0, true);
    if (forked < 0) return forked;
    if (forked) ACE_CUDA(cudaStreamWaitEvent(w.main, w.ev_aux, 0));
    return 0;  // X, U complete: every merge ran behind its panel
  }
  // the leading block is final after panel h_top/pb, but its inverse is only released once the trailing
  // updates have become small (last ~quarter of the columns): released earlier it merely competes with them
  double frac = 0.75;
  if (const char* e = std::getenv("ACE_FORK_FRAC")) frac = std::atof(e);
  const int forked = potrf_blocked(w, h_top, (int)(frac * nb));
  if (forked < 0) return forked;
  const size_t left_ws = (size_t)(h_top * TB / 2) * (h_top * TB / 2);
  if (!forked) ACE_TRY(trtri_merge_range(w, 0, h_top, w.main, w.Bf, trtri_hmin(w)));
  ACE_TRY(trtri_merge_range(w, h_top, nb, w.main, w.Bf + left_ws, trtri_hmin(w)));   // right child, own workspace region
  if (forked) ACE_CUDA(cudaStreamWaitEvent(w.main, w.ev_aux, 0));
  return trtri_level(w, 0, nb, h_top, w.main, w.Bf);                   // top-level merge
}

// n_pad from which U U^T runs on the INT8 engine (B200 timings and why 8192: DESIGN section 3.2c).
constexpr int UUT_I8_MIN_N = 8192;

// The one place that chooses the U U^T engine.  engine: 0 by size, 1 DMMA, 2 INT8 (debug pins).
inline bool uut_uses_i8(int n_pad, int engine) {
  if (engine != 0) return engine == 2;
  return n_pad >= UUT_I8_MIN_N && n_pad <= oz::MAX_N;
}

// Phase 3: inverse = U * U^T into Bf (both triangles), one launch (the INT8 engine: split, one product per
// modulus, CRT).
inline int uut_inverse(const DenseWork& w) {
  if (uut_uses_i8(w.nb * TB, w.uut_engine)) return launch_uut_i8(w.oz, w.A, w.DU, w.nb, w.Bf, w.main);
  GemmNT p{};
  p.A = w.A; p.lda = w.ld; p.a_tri = 1; p.Adiag = w.DU;
  p.B = w.A; p.ldb = w.ld; p.Bdiag = w.DU;
  p.C = w.Bf; p.ldc = w.ld; p.Ct = w.Bf; p.ldct = w.ld;
  p.M = p.N = p.K = w.nb * TB;
  p.alpha = 1.0; p.beta = 0.0; p.lower_only = 1;
  return launch_gemm_nt(p, w.main);
}

inline int spd_inverse(const DenseWork& w) {
  ACE_TRY(potrf_trtri(w));
  return uut_inverse(w);
}

}  // namespace ace
