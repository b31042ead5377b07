// diag_block.cuh -- Cholesky factor AND triangular inverse of one diagonal block (<= 512 x 512) of the blocked
// factorisation in ONE launch: a thread-block cluster of 8 CTAs.
//
// Why: the diagonal blocks are the serial chain of the right-looking Cholesky (chol.cuh).  Done as a recursion
// of 128-wide leaf kernels (4 x potrf_leaf + 4 x trsm_leaf + 8 small GEMM launches, ~0.6 ms per 512-block:
// profiles/r01) the chain bounds the tail of the factorisation on one GPU, all of C2 (n = 4096) and the sharded
// fit.  Here the block is cut into 32 x 32 tiles and processed by the 64 warps of the cluster:
//
//   factor   right-looking over the 16 tile columns:  one warp factors the diagonal tile in registers
//            (column broadcast through shared memory, MUFU-seeded rsqrt) and inverts it;  every warp then solves
//            tiles of the column as a product with that inverse (DMMA) and updates trailing tiles (DMMA).  The warp
//            that factors tile k+1 updates it first and factors it while the others finish the trailing update
//            of step k (look-ahead): two cluster barriers per tile column.
//   inverse  X = L^-1 right-looking and in place, as single 32^3 tile products dealt to the warps that would otherwise
//            wait for the serial chain (see the kernel body): no separate phase, no extra barriers.
//   output   the layout the rest of the dense engine expects from potrf_rec + trtri_merge_range: L in the
//            diagonal 128-tiles of A, X / U in the off-diagonal 128-blocks of the block (lower / upper), dense
//            DX / DU tiles, diag(L) in dvec, the first non-positive pivot in info.
//
// All exchange between CTAs goes through global memory (the 2 MB block stays in L2) ordered by
// barrier.cluster (release / acquire at cluster scope); operands reach the tensor pipe through a warp-private
// shared-memory stage filled by TMA bulk copies (cp.async.bulk, L2 -> smem) on a per-warp mbarrier.  Replaces the eigendecomposition
// route of invkernel_cpp for the diagonal blocks (src/kernel_SE_cpp.cpp:137-157).
#pragma once
#include <cstdlib>
#include "common.cuh"
#include "fastmath.cuh"

namespace ace {

struct DiagArgs {
  double* A;       // matrix base (column-major, ld)
  long ld;
  int blk0, nblk;  // first 128-block on the diagonal, number of 128-blocks (<= 4 by default)
  double* DX;      // dense diagonal tiles of X = L^-1 (lower), tile t at + t * 128 * 128
  double* DU;      // dense diagonal tiles of U = L^-T (upper)
  double* dvec;    // diag(L)
  int* info;       // 0, or 1-based global index of the first non-positive pivot
  double* S;       // scratch (nblk*128)^2: X below / U above the diagonal while the inverse is built
  double* W;       // scratch (nblk*128/2)^2: the W^T = U11 L21^T products of one merge level
  long long* dbg;  // optional (debug): SM clock stamps of the phases, see ace_dbg_diag_block_timeline
};

namespace dg {
constexpr int TS = 32;                    // tile edge
// CTAs per cluster: 8 (portable maximum) or 16 (opt-in, cudaFuncAttributeNonPortableClusterSizeAllowed): template
// parameter of the kernel.  With 8 the first tile columns of a 512-block are bound by the 56 worker warps (13-15 us of
// trailing update against a 13 us serial chain, profiles/r02/diag_block_timeline.md); 16 CTAs halve that.
constexpr int WARPS = 8, THREADS = WARPS * 32;
constexpr int LDT = 36;                   // stride of a staged tile: rows 16-byte aligned, DMMA fragment loads conflict free
constexpr int STAGE = 2 * TS * LDT + 2;   // doubles per warp: one A tile + one B tile (+ 2 spare)
constexpr int COLBARS = 32;               // one mbarrier per column of the diagonal tile: leader -> follower hand-over
constexpr size_t SMEM_BYTES = (size_t)(WARPS * STAGE + COLBARS) * 8;
constexpr int KEEP_ALL = 0, KEEP_UPPER = 1, KEEP_LOWER = 2;
inline size_t ws_doubles(int panel_blocks) {
  const size_t N = (size_t)panel_blocks * 128;
  return N * N + (N / 2) * (N / 2);
}
}  // namespace dg

__device__ __forceinline__ unsigned cluster_ctarank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}

// all threads of all CTAs of the cluster; orders global (and shared) memory accesses at cluster scope
__device__ __forceinline__ void cluster_barrier() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// split form: a warp that has published its part may go on and collect the barrier later
__device__ __forceinline__ void cluster_arrive() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait() {
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Two 32 x 32 tiles (column c at src + c * ld) -> the warp's stage (column c at dst + c * LDT) with 16-byte loads
// through L2 (ld.global.cg): 16 lanes per column, 32 loads per lane in flight, ~0.4 us.  (The first version used one
// 256-byte TMA bulk copy per lane and tile: 64 serialised UBLKCP issues cost ~3 us per tile pair, more than the tile
// product itself -- profiles/r02/diag_block_timeline.md.)  Operands must be 16-byte aligned with even strides.
__device__ __forceinline__ void dg_stage_pair(double* stage, const double* A, long lda, const double* B, long ldb,
                                              int lane) {
  using namespace dg;
  const int r2 = 2 * (lane & 15), c0 = lane >> 4;
  double2 va[16], vb[16];
#pragma unroll
  for (int q = 0; q < 16; ++q) va[q] = __ldcg(reinterpret_cast<const double2*>(A + r2 + (size_t)(2 * q + c0) * lda));
#pragma unroll
  for (int q = 0; q < 16; ++q) vb[q] = __ldcg(reinterpret_cast<const double2*>(B + r2 + (size_t)(2 * q + c0) * ldb));
#pragma unroll
  for (int q = 0; q < 16; ++q) *reinterpret_cast<double2*>(stage + r2 + (2 * q + c0) * LDT) = va[q];
#pragma unroll
  for (int q = 0; q < 16; ++q) *reinterpret_cast<double2*>(stage + TS * LDT + r2 + (2 * q + c0) * LDT) = vb[q];
  __syncwarp();
}

// One warp:  C = beta * C + alpha * sum_{t < nk} A_t B_t^T  on 32 x 32 tiles (A_t at A + t * sa, B_t at B + t * sb),
// optional transposed copy Ct.  Tile ma_t of the A sequence / mb_t of the B sequence is triangular and stored with
// the other triangle occupied by something else: only its upper (KEEP_UPPER: row <= col) or lower part is used.
// C may alias A_0 when nk == 1 (the operands are staged completely before anything is stored).
__device__ __noinline__ void dg_tile_gemm(double* stage, int lane, const double* A, long lda, long sa, int ma_t,
                                             int ma_kind, const double* B, long ldb, long sb, int mb_t, int mb_kind,
                                             int nk, double alpha, double beta, double* C, long ldc, double* Ct,
                                             long ldct, long long* tdbg = nullptr) {
  using namespace dg;
  const int g = lane >> 2, tq = lane & 3;
  double acc[4][4][2];
  if (tdbg != nullptr && lane == 0) tdbg[0] = clock64();
  double* sA = stage;
  double* sB = stage + TS * LDT;
#pragma unroll 1
  for (int t = 0; t < nk; ++t) {
    __syncwarp();  // everybody is done reading the previous tiles
    dg_stage_pair(stage, A + (size_t)t * sa, lda, B + (size_t)t * sb, ldb, lane);
    if (t == 0) {
      if (beta != 0.0) {  // acc = (beta / alpha) C, so that alpha * acc ends as beta C + alpha sum
        const double sc = beta / alpha;
#pragma unroll
        for (int mt = 0; mt < 4; ++mt)
#pragma unroll
          for (int nt = 0; nt < 4; ++nt)
#pragma unroll
            for (int e = 0; e < 2; ++e)
              acc[mt][nt][e] = sc * __ldcg(C + (mt * 8 + g) + (size_t)(nt * 8 + 2 * tq + e) * ldc);
      } else {
#pragma unroll
        for (int mt = 0; mt < 4; ++mt)
#pragma unroll
          for (int nt = 0; nt < 4; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
      }
    }
    if (tdbg != nullptr && lane == 0) tdbg[1] = clock64();
    const int ka = (t == ma_t) ? ma_kind : KEEP_ALL, kb = (t == mb_t) ? mb_kind : KEEP_ALL;
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      const int k = ks * 4 + tq;
      double a[4], b[4];
#pragma unroll
      for (int mt = 0; mt < 4; ++mt) {
        const int row = mt * 8 + g;
        double v = sA[row + k * LDT];
        if (ka == KEEP_UPPER) v = (row <= k) ? v : 0.0;
        if (ka == KEEP_LOWER) v = (row >= k) ? v : 0.0;
        a[mt] = v;
      }
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const int row = nt * 8 + g;
        double v = sB[row + k * LDT];
        if (kb == KEEP_UPPER) v = (row <= k) ? v : 0.0;
        if (kb == KEEP_LOWER) v = (row >= k) ? v : 0.0;
        b[nt] = v;
      }
#pragma unroll
      for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) dmma884(acc[mt][nt][0], acc[mt][nt][1], a[mt], b[nt]);
    }
  }
  if (tdbg != nullptr && lane == 0) tdbg[2] = clock64();
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const double v = alpha * acc[mt][nt][e];
        acc[mt][nt][e] = v;
        __stcg(C + (mt * 8 + g) + (size_t)(nt * 8 + 2 * tq + e) * ldc, v);
      }
  if (tdbg != nullptr && lane == 0) tdbg[3] = clock64();
  if (Ct != nullptr) {
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt)
        __stcg(reinterpret_cast<double2*>(Ct + (nt * 8 + 2 * tq) + (size_t)(mt * 8 + g) * ldct),
               make_double2(acc[mt][nt][0], acc[mt][nt][1]));
  }
}

// ---------------------------------------------------------------------------------------------
// One warp: Cholesky of a 32 x 32 diagonal tile and the inverse of its factor.
// The tile lives in registers in a 2-D cyclic layout -- lane (ty, tx) = (lane / 8, lane % 8) owns the elements
// (4a + ty, 8b + tx), a < 8, b < 4 -- so that "which column" is a lane predicate, not a register index: the column
// loops are ROLLED (4 columns per template instance), the code stays a few KB (a fully unrolled row-per-lane
// version was instruction-fetch bound: 12 us per tile), and all 32 lanes share the rank-1 updates.
// ---------------------------------------------------------------------------------------------
// Running pointers of the column loop (kept explicitly: recomputed per column they were a third of the loop body).
struct DgCholState {
  double* cbc;     // half of the column buffer that holds the published column j
  double* cbn;     // the other half: column j+1 is published there
  double* lsw;     // Ls + ty + 33 j: this lane's rows of column j of L
  double* dgj;     // dgl + j (L_jj); 1 / L_jj at dgj + 32
  uint64_t* bar;   // colbar + j - 1
  int j;
};

// Columns 8 JB + 4 H .. + 3.  Software-pipelined: column j+1 is published to the column buffer as soon as its block
// column has received the update of column j; the rest of the update and the stores of column j then overlap the
// STS -> __syncwarp -> LDS round trip of the hand-over.
template <int JB, int H>
__device__ __forceinline__ void dg_chol_cols(double (&r)[8][4], DgCholState& st, int tx, int ty, int* info, int gidx0) {
  constexpr int A0 = 2 * JB + H;  // row block of the pivots of these 4 columns
#pragma unroll 1
  for (int jj = 0; jj < 4; ++jj) {
    const int jx = 4 * H + jj;
    __syncwarp();  // column j is in st.cbc (published at the end of the previous iteration / before the first)
    // column j-1 of L and 1/L_(j-1)(j-1) are in shared memory (stored in the previous iteration, ordered by the
    // __syncwarp above): hand them to the follower.  mbarrier.arrive has release semantics at CTA scope and costs one
    // instruction (the MEMBAR.SC.CTA of a fence + flag store was ~3 us per tile on the critical path).
    if (tx == 0 && ty == 0 && st.j > 0) mbar_arrive(st.bar);
    const double pj = st.cbc[st.j];
    // one MUFU-seeded reciprocal square root serves the whole column: 1/L_jj = y, L_jj = p y.  One cubic step on the
    // ~2^-23 seed leaves ~2^-60: the second step of fast_rsqrt is off this chain.
    double inv;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(inv) : "d"(pj));
    {
      const double e = fma(-pj * inv, inv, 1.0);
      inv = fma(inv * e, fma(0.375, e, 0.5), inv);
    }
    double lm[8], cm[4];
    const double* cl = st.cbc + ty;
    const double* cc = st.cbc + tx;
#pragma unroll
    for (int a = A0; a < 8; ++a) lm[a] = cl[4 * a] * inv;
#pragma unroll
    for (int b = JB; b < 4; ++b) cm[b] = cc[8 * b] * inv;
    lm[A0] = (ty > jj) ? lm[A0] : 0.0;   // rows <= j (only block A0 straddles the pivot)
    cm[JB] = (tx > jx) ? cm[JB] : 0.0;   // columns <= j (only block JB straddles it)
    double* cn = st.cbn + ty;
    // the block column that holds the next pivot column first (entries above the diagonal: never read)
#pragma unroll
    for (int a = A0; a < 8; ++a) r[a][JB] = fma(-lm[a], cm[JB], r[a][JB]);
    if (H == 0 || jj < 3) {
      if (tx == jx + 1) {
#pragma unroll
        for (int a = A0; a < 8; ++a) cn[4 * a] = r[a][JB];
      }
      // keep the rest of the update BEHIND the hand-over (the compiler otherwise hoists these independent DFMAs above
      // the divergent store block and the pipelining is lost)
#pragma unroll
      for (int b = JB + 1; b < 4; ++b) asm volatile("" : "+d"(cm[b]) : : "memory");
#pragma unroll
      for (int b = JB + 1; b < 4; ++b)
#pragma unroll
        for (int a = A0; a < 8; ++a) r[a][b] = fma(-lm[a], cm[b], r[a][b]);
    } else if (JB < 3) {  // the next column opens block column JB + 1
      constexpr int JN = (JB < 3) ? JB + 1 : 3;
#pragma unroll
      for (int a = A0; a < 8; ++a) r[a][JN] = fma(-lm[a], cm[JN], r[a][JN]);
      if (tx == 0) {
#pragma unroll
        for (int a = A0; a < 8; ++a) cn[4 * a] = r[a][JN];
      }
#pragma unroll
      for (int b = JN + 1; b < 4; ++b) asm volatile("" : "+d"(cm[b]) : : "memory");
#pragma unroll
      for (int b = JN + 1; b < 4; ++b)
#pragma unroll
        for (int a = A0; a < 8; ++a) r[a][b] = fma(-lm[a], cm[b], r[a][b]);
    }
    // column j of L (the owners' copy of column j is untouched by the update: their cm[JB] is masked to zero) goes to
    // shared memory for the follower, which also writes it out
    if (tx == jx) {
      if (ty > jj) st.lsw[4 * A0] = lm[A0];  // the pivot's row block: rows below the pivot only
#pragma unroll
      for (int a = A0 + 1; a < 8; ++a) st.lsw[4 * a] = lm[a];
      if (ty == jj) {  // the pivot itself (one lane): L_jj by one Newton step on p y, 1 / L_jj, positivity check
        double sq = pj * inv;
        sq = fma(fma(-sq, sq, pj), 0.5 * inv, sq);
        st.dgj[0] = sq;
        st.dgj[32] = inv;
        if (!(pj > 0.0)) atomicCAS(info, 0, gidx0 + st.j + 1);
      }
    }
    double* t = st.cbc;
    st.cbc = st.cbn;
    st.cbn = t;
    st.lsw += 33;
    st.dgj += 1;
    st.bar = st.bar + 1;
    st.j += 1;
  }
}

// The diagonal tile is factored by TWO warps of one CTA: the leader runs the Cholesky (and writes L, diag(L)), the
// follower computes X = L^-1 one column behind it -- row j of X only needs columns <= j of L -- and writes the X / U
// tile.  Both work on the leader's shared-memory stage `sm0` (columns of L below the diagonal, rows of U above it);
// column j is handed over on the mbarrier colbar[j] (phase parity = how often this CTA has factored a tile, mod 2).
// SRC_SMEM: the tile is taken from shared memory (`tile`, element (i, c) at tile[i + 33 c]) instead of from At.
template <bool SRC_SMEM>
__device__ __noinline__ void dg_chol_lead(double* sm0, int lane, double* At, long ld, const double* tile, double* dv,
                                          int* info, int gidx0, uint64_t* colbar) {
  double* Ls = sm0;                 // [32][33]: strictly lower = L, strictly upper = U (filled by the follower)
  double* colbuf = sm0 + 32 * 33;   // 2 x 32: pivot column, double buffered
  double* dgl = colbuf + 64;        // L_jj
  double* idg = dgl + 32;           // 1 / L_jj
  const int tx = lane & 7, ty = lane >> 3;
  double r[8][4];
#pragma unroll
  for (int b = 0; b < 4; ++b)
#pragma unroll
    for (int a = 0; a < 8; ++a)
      r[a][b] = SRC_SMEM ? tile[(4 * a + ty) + (8 * b + tx) * 33] : __ldcg(At + (4 * a + ty) + (size_t)(8 * b + tx) * ld);
  __syncwarp();  // SRC_SMEM: `tile` overlaps idg, which the first column writes
  DgCholState st;
  st.cbc = colbuf;
  st.cbn = colbuf + 32;
  st.lsw = Ls + ty;
  st.dgj = dgl;
  st.bar = colbar - 1;
  st.j = 0;
  if (tx == 0) {  // publish column 0
#pragma unroll
    for (int a = 0; a < 8; ++a) st.cbc[4 * a + ty] = r[a][0];
  }
  dg_chol_cols<0, 0>(r, st, tx, ty, info, gidx0);
  dg_chol_cols<0, 1>(r, st, tx, ty, info, gidx0);
  dg_chol_cols<1, 0>(r, st, tx, ty, info, gidx0);
  dg_chol_cols<1, 1>(r, st, tx, ty, info, gidx0);
  dg_chol_cols<2, 0>(r, st, tx, ty, info, gidx0);
  dg_chol_cols<2, 1>(r, st, tx, ty, info, gidx0);
  dg_chol_cols<3, 0>(r, st, tx, ty, info, gidx0);
  dg_chol_cols<3, 1>(r, st, tx, ty, info, gidx0);
  __syncwarp();
  if (lane == 0) mbar_arrive(colbar + 31);
}

// Follower: X = L^-1, one COLUMN of X per lane (lane c solves L x = e_c), right-looking and fully unrolled: when column
// k of L is published, x_k = (delta_kc - acc_k) / L_kk is final and acc_i += L(i, k) x_k for i > k -- 31 - k independent
// DFMAs fed by broadcast reads of the leader's shared-memory copy of L, accumulators in registers, no cross-lane traffic
// at all: ~1.5 us of work per tile against the leader's ~6 us, so the inverse is complete right after the last column of
// the factorisation.  (The first version mirrored the factorisation -- a right-looking update of a register tile with
// a shared-memory broadcast per row -- and fell 3 us per tile behind once the leader was pipelined; a rolled
// dot-product form was latency bound on its loads: 6 us behind.)  It also writes the outputs: column k of L and L_kk
// (coalesced), row k of X into the X (lower) / U (upper) tile.
__device__ __noinline__ void dg_inv_follow(double* sm0, int lane, double* St, long lds, uint64_t* colbar, uint32_t parity,
                                           double* At, long ld, double* dv) {
  const double* Ls = sm0;
  const double* dgl = sm0 + 32 * 33 + 64;
  const double* idg = dgl + 32;
  double acc[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) acc[i] = 0.0;
  double* gl = At + lane;         // column k of L at gl + k ld
  double* gu = St + lane;         // U(c, k) at gu + k lds
  double* gx = St + (size_t)lane * lds;  // X(k, c) at gx + k
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    mbar_wait(colbar + k, parity);  // column k of L and 1 / L_kk published by the factoring warp (acquire)
    const double* lk = Ls + 33 * k;  // L(i, k) at lk[i]
    {  // column k of L out
      const double v = (lane > k) ? lk[lane] : dgl[k];
      if (lane >= k) __stcg(gl + (size_t)k * ld, v);
      if (lane == k) dv[k] = v;
    }
    const double x = (((lane == k) ? 1.0 : 0.0) - acc[k]) * idg[k];
    if (lane <= k) __stcg(gu + (size_t)k * lds, x);  // U(c, k) = X(k, c), and the diagonal
    if (lane < k) __stcg(gx + k, x);                 // X(k, c)
#pragma unroll
    for (int i = k + 1; i < 32; ++i) acc[i] = fma(lk[i], x, acc[i]);
  }
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// The serial chain of one tile column, run by FOUR warps of the CTA that will factor tile k+1 (one per SM sub-partition:
// the leader = warp 0, and three helpers that would otherwise idle) right after the barrier that publishes L_kk / X_kk --
// they do not wait for the rest of the column solve:
//   L_(k+1)k = A_(k+1)k X_kk^T            (stored for everybody else; each warp arrives at the step's second barrier)
//   A_(k+1)(k+1) -= L_(k+1)k L_(k+1)k^T   (operand straight from shared memory, result handed over in shared memory)
//   Cholesky of the updated tile          (leader only: dg_chol_lead; the follower warp runs one column behind)
// Each of the four warps owns 8 columns of both products (32 DMMA per product instead of 128 on one warp); operands are
// staged cooperatively, the three hand-overs are named barriers of 128 threads.  History (profiles/r02/
// diag_block_timeline.md): update + factorisation after the second barrier, through global memory: 21.5 us per tile
// column; one warp running this chain: 14.4 us.
// h = 0 (leader) .. 3.  sA / sB: the leader's stage; sL: a helper's stage.
__device__ __noinline__ void dg_chain_step(double* stage0, double* sL, int h, int lane, double* Lk1k, const double* Xkk,
                                           long ldx, double* Adiag, long ld, double* dv, int* info, int gidx0,
                                           uint64_t* colbar, long long* dbg) {
  using namespace dg;
  const int g = lane >> 2, tq = lane & 3;
  double* sA = stage0;
  double* sB = stage0 + TS * LDT;
  // this warp's 8 columns of the diagonal tile (all updates of earlier columns were complete at the first barrier)
  double c[4][2];
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int e = 0; e < 2; ++e) c[mt][e] = __ldcg(Adiag + (mt * 8 + g) + (size_t)(8 * h + 2 * tq + e) * ld);
  {  // cooperative staging: 128 lanes, 4 + 4 16-byte loads each
    const int tid = h * 32 + lane;
    double2 va[4], vb[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int idx = q * 128 + tid, col = idx >> 4, r2 = 2 * (idx & 15);
      va[q] = __ldcg(reinterpret_cast<const double2*>(Lk1k + r2 + (size_t)col * ld));
      vb[q] = __ldcg(reinterpret_cast<const double2*>(Xkk + r2 + (size_t)col * ldx));
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int idx = q * 128 + tid, col = idx >> 4, r2 = 2 * (idx & 15);
      *reinterpret_cast<double2*>(sA + r2 + col * LDT) = va[q];
      *reinterpret_cast<double2*>(sB + r2 + col * LDT) = vb[q];
    }
  }
  named_bar_sync(1, 128);
  double acc[4][2];
#pragma unroll
  for (int mt = 0; mt < 4; ++mt) acc[mt][0] = acc[mt][1] = 0.0;
#pragma unroll
  for (int ks = 0; ks < 8; ++ks) {
    const int k = ks * 4 + tq;
    const int row = 8 * h + g;
    const double bv = sB[row + k * LDT];
    const double b = (row >= k) ? bv : 0.0;  // X_kk is lower triangular; its upper part holds U
#pragma unroll
    for (int mt = 0; mt < 4; ++mt) dmma884(acc[mt][0], acc[mt][1], sA[mt * 8 + g + k * LDT], b);
  }
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int row = mt * 8 + g, col = 8 * h + 2 * tq + e;
      __stcg(Lk1k + row + (size_t)col * ld, acc[mt][e]);
      sL[row + col * LDT] = acc[mt][e];
    }
  cluster_arrive();  // second barrier of the step: this warp's part of L_(k+1)k is published; collected at the end
  named_bar_sync(2, 128);
#pragma unroll
  for (int ks = 0; ks < 8; ++ks) {
    const int k = ks * 4 + tq;
    const double b = sL[8 * h + g + k * LDT];
#pragma unroll
    for (int mt = 0; mt < 4; ++mt) dmma884(c[mt][0], c[mt][1], -sL[mt * 8 + g + k * LDT], b);
  }
  // hand the updated tile to the factorisation's register layout through the B half of the stage (stride 33)
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int e = 0; e < 2; ++e) sB[(mt * 8 + g) + (8 * h + 2 * tq + e) * 33] = c[mt][e];
  if (h == 0) {
    named_bar_sync(3, 128);
    if (dbg != nullptr && lane == 0) dbg[1] = clock64();
    dg_chol_lead<true>(stage0, lane, Adiag, ld, sB, dv, info, gidx0, colbar);
    if (dbg != nullptr && lane == 0) dbg[2] = clock64();
  } else {
    named_bar_arrive(3, 128);
  }
  cluster_wait();
}

template <int NC>
__device__ __forceinline__ void diag_block_body(const DiagArgs& a) {
  using namespace dg;
  constexpr int GW = NC * WARPS;  // warps in the cluster
  extern __shared__ __align__(128) unsigned char smraw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int crank = (int)cluster_ctarank();
  // warp index inside the cluster, CTA index fastest: consecutive tasks go to different SMs (a tile product is
  // bound by the SM's FP64 tensor rate: eight of them on one SM take four times as long as two)
  const int gw = warp * NC + crank;
  double* stage = reinterpret_cast<double*>(smraw) + warp * STAGE;
  uint64_t* colbar = reinterpret_cast<uint64_t*>(reinterpret_cast<double*>(smraw) + WARPS * STAGE);
  if (warp == 0) {
    mbar_init(colbar + lane, 1);  // column hand-over barriers of the tile factorisation
    fence_mbar_init();
  }
  __syncthreads();
  double* stage0 = reinterpret_cast<double*>(smraw);  // warp 0's stage: the tile factorisation lives there
  const int nt = a.nblk * 4;            // 32-tiles per side
  const long N = (long)nt * TS;
  const long ld = a.ld;
  double* Ab = a.A + (size_t)a.blk0 * 128 * (ld + 1);
  double* dv = a.dvec + (size_t)a.blk0 * 128;
  auto At = [&](int i, int j) { return Ab + (size_t)i * TS + (size_t)j * TS * ld; };
  auto St = [&](int i, int j) { return a.S + (size_t)i * TS + (size_t)j * TS * N; };
  auto fw = [&](int k) { return k % NC; };  // the warp that factors diagonal tile k: warp 0 of CTA k mod NC
  // debug stamps: T(k, s) by warp 0 of CTA 0 (s = 0..4: before B1, after B1, after its column solves, after B2, after
  // its trailing tiles), F(k, s) by the factoring warp of tile k (0: start of its diagonal update, 1: after it, 2:
  // after the factorisation); 8 slots per tile column, then 4 per merge level, then the end
  auto stampT = [&](int k, int sidx) {
    if (a.dbg != nullptr && gw == 0 && lane == 0) a.dbg[8 * k + sidx] = clock64();
  };
  auto stampF = [&](int k, int sidx) {
    if (a.dbg != nullptr && lane == 0) a.dbg[8 * k + 5 + sidx] = clock64();
  };

  // ------------------------------------------------------------------ factorisation + inverse, interleaved
  // Serial chain per tile column k:  Cholesky of the diagonal tile (its inverse follows on a second warp) -> barrier -> column solve
  // L_ik = A_ik X_kk^T (every warp one tile product) -> barrier -> update of the next diagonal tile (the warp that will
  // factor it).  Everything else hides behind it:
  //   * trailing update A_ij -= L_ik L_jk^T, dealt over the warps of the other CTAs;
  //   * the inverse X = L^-1, right-looking and in place in S: the upper tile (j, i), j < i, first accumulates
  //     AccT(j, i) = sum_{t = j}^{i-1} U(j, t) L(i, t)^T (one term per tile column t, as soon as row t of X is final)
  //     and is then replaced by U(j, i) = X(i, j)^T with X(i, j) = -X_ii AccT(j, i)^T.
  // Every task is ONE 32^3 tile product: no separate inverse phase, no long K loops, no extra barriers.
  // (Measured alternatives, profiles/r02/diag_block_timeline.md: a bottom-up merge tree after the factorisation
  // costs +140 us; solving the column by substitution against L_kk with X_kk computed one slot later takes the tile
  // inverse off the chain but the rolled substitution is slower than the tile product: 433 vs 379 us per block.)
  // tile k is factored by warp 0 (Cholesky) and warp 1 (inverse, one column behind) of CTA k mod NC
  if (gw == fw(0)) {
    stampF(0, 1);
    dg_chol_lead<false>(stage0, lane, At(0, 0), ld, nullptr, dv, a.info, a.blk0 * 128, colbar);
    stampF(0, 2);
  } else if (gw == fw(0) + NC) {
    dg_inv_follow(stage0, lane, St(0, 0), N, colbar, 0u, At(0, 0), ld, dv);
  }
#pragma unroll 1
  for (int k = 0; k < nt; ++k) {
    stampT(k, 0);
    cluster_barrier();  // L_kk, X_kk visible; trailing update and accumulations of step k-1 complete
    stampT(k, 1);
    const bool more = (k + 1 < nt);
    const int f = fw(k + 1);  // CTA rank of the warps that factor tile k+1 (warp 0: Cholesky, warp 1: inverse)
    if (more && crank == f) {
      // the serial chain: warps 0, 5, 2, 3 of the factoring CTA (one per SM sub-partition) solve L_(k+1)k and update
      // tile k+1, warp 0 factors it, warp 1 inverts it one column behind; all of them arrive at the second barrier on
      // the way and collect it when they are done
      const int h = (warp == 0) ? 0 : (warp == 5) ? 1 : (warp == 2) ? 2 : (warp == 3) ? 3 : -1;
      if (h >= 0) {
        if (h == 0) stampF(k + 1, 0);
        dg_chain_step(stage0, stage0 + 2 * STAGE, h, lane, At(k + 1, k), St(k, k), N, At(k + 1, k + 1), ld,
                      dv + (k + 1) * TS, a.info, a.blk0 * 128 + (k + 1) * TS, colbar,
                      a.dbg ? a.dbg + 8 * (k + 1) + 5 : nullptr);
        continue;
      }
      if (warp == 1) {
        cluster_arrive();
        dg_inv_follow(stage0, lane, St(k + 1, k + 1), N, colbar, (uint32_t)(((k + 1) / NC) & 1),
                      At(k + 1, k + 1), ld, dv + (k + 1) * TS);
        cluster_wait();
        continue;
      }
    }
    // column k of L: L_ik = A_ik X_kk^T (in place), i > k+1, and row k of X: X(k, j) = -X_kk AccT(j, k)^T,
    // U(j, k) = X(k, j)^T -- dealt over the warps that are not on the chain
    {
      constexpr int NWK = (NC - 1) * WARPS;        // warps of the other CTAs
      const int skip = more ? 1 : 0;               // tile (k+1, k) belongs to the chain
      const int nsolve = nt - 1 - k - skip;
      const int nw = more ? NWK + 3 : GW;
      int me = gw;
      if (more) {
        if (crank != f) me = warp * (NC - 1) + (crank - f - 1 + NC) % NC;  // CTA index fastest
        else me = NWK + ((warp == 4) ? 0 : (warp == 6) ? 1 : 2);           // warps 4, 6, 7 of the chain CTA
      }
      for (int u = me; u < nsolve + k; u += nw) {
        if (u < nsolve) {
          const int i = k + 1 + skip + u;
          dg_tile_gemm(stage, lane, At(i, k), ld, 0, -1, KEEP_ALL, St(k, k), N, 0, 0, KEEP_LOWER, 1, 1.0, 0.0, At(i, k), ld,
                       nullptr, 0);
        } else {
          const int j = u - nsolve;
          dg_tile_gemm(stage, lane, St(k, k), N, 0, 0, KEEP_LOWER, St(j, k), N, 0, -1, KEEP_ALL, 1, -1.0, 0.0, St(k, j), N,
                       St(j, k), N);
        }
      }
    }
    stampT(k, 2);
    cluster_barrier();  // column k of L and row k of X / column k of U visible
    stampT(k, 3);
    if (!more) break;
    // The warps of the CTAs that do not hold the chain share
    //   trailing update  A_ij -= L_ik L_jk^T           for k < j <= i        (column-major order, without (k+1, k+1))
    //   accumulation     AccT(j, i) (+)= U(j, k) L_ik^T  for j <= k < i
    // (the factoring CTA stays out of it: its SM's FP64 pipe belongs to the serial chain).
    if (crank != f) {
      constexpr int NWK = (NC - 1) * WARPS;                        // worker warps
      const int me = warp * (NC - 1) + (crank - f - 1 + NC) % NC;  // 0 .. NWK-1, CTA index fastest
      const int m = nt - 1 - k;                                    // trailing tile rows / columns
      const int nupd = m * (m + 1) / 2 - 1;                        // without (k+1, k+1)
      const int nacc = m * (k + 1);
      for (int u = me; u < nupd + nacc; u += NWK) {
        if (u < nupd) {
          // task u+1 of the column-major enumeration (jj, ii), 0 <= jj <= ii < m: column jj holds m - jj tiles
          int rest = u + 1, jj = 0;
          while (rest >= m - jj) {
            rest -= m - jj;
            ++jj;
          }
          const int i = k + 1 + jj + rest, j = k + 1 + jj;
          dg_tile_gemm(stage, lane, At(i, k), ld, 0, -1, KEEP_ALL, At(j, k), ld, 0, -1, KEEP_ALL, 1, -1.0, 1.0, At(i, j), ld,
                       nullptr, 0, (a.dbg != nullptr && u == 0) ? a.dbg + 8 * (20 + k) : nullptr);
        } else {
          const int v = u - nupd, i = k + 1 + v % m, j = v / m;
          dg_tile_gemm(stage, lane, St(j, k), N, 0, (j == k) ? 0 : -1, KEEP_UPPER, At(i, k), ld, 0, -1, KEEP_ALL, 1, 1.0,
                       (j == k) ? 0.0 : 1.0, St(j, i), N, nullptr, 0);
        }
      }
      stampT(k, 4);
    }
  }
  const int lvl = 0;

  // ------------------------------------------------------------------ output layout of the dense engine
  for (int j = crank * WARPS + warp; j < (int)N; j += GW) {
    const int bj = j >> 7;
    const double* src = a.S + (size_t)j * N;
#pragma unroll 1
    for (int i0 = 0; i0 < (int)N; i0 += 256) {
      double v[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) v[q] = (i0 + 32 * q < (int)N) ? __ldcg(src + i0 + 32 * q + lane) : 0.0;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int i = i0 + 32 * q + lane;
        if (i0 + 32 * q >= (int)N) break;
        if ((i >> 7) == bj) {
          const size_t o = (size_t)(a.blk0 + bj) * 128 * 128 + (size_t)(j & 127) * 128 + (i & 127);
          a.DX[o] = (i >= j) ? v[q] : 0.0;
          a.DU[o] = (i <= j) ? v[q] : 0.0;
        } else {
          Ab[i + (size_t)j * ld] = v[q];
        }
      }
    }
  }
  stampT(nt, 4 * lvl);
}

template <int NC>
__global__ void __launch_bounds__(dg::THREADS, 2) diag_block_kernel(const DiagArgs a) {
  diag_block_body<NC>(a);
}

// Batched fit (ace_fit_batch): one cluster per member q = blockIdx.y, each with its own matrix, tiles, diag(L), pivot
// slot and scratch (strides in elements); members with active[q] == 0 are left untouched.
struct DiagStrides {
  const int* active;
  long A, tiles, vec, ws;
};

template <int NC>
__global__ void __launch_bounds__(dg::THREADS, 2) diag_block_batch_kernel(const DiagArgs a, const DiagStrides m) {
  const long q = blockIdx.y;
  if (m.active != nullptr && m.active[q] == 0) return;  // uniform over the cluster
  DiagArgs b = a;
  b.A += q * m.A;
  b.DX += q * m.tiles;
  b.DU += q * m.tiles;
  b.dvec += q * m.vec;
  b.info += q;
  b.S += q * m.ws;
  b.W += q * m.ws;
  diag_block_body<NC>(b);
}

// cluster size in use on this device: 16 when the opt-in size is accepted and can be co-scheduled, else 8
inline int& diag_cluster_size() {
  static int nc = 0;
  return nc;
}

template <int NC>
inline int launch_diag_block_nc(const DiagArgs& a, cudaStream_t st) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(NC, 1, 1);
  cfg.blockDim = dim3(dg::THREADS, 1, 1);
  cfg.dynamicSmemBytes = dg::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = NC;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  ACE_CUDA(cudaLaunchKernelEx(&cfg, diag_block_kernel<NC>, a));
  return 0;
}

inline int configure_diag_kernel() {
  ACE_CUDA(cudaFuncSetAttribute(diag_block_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dg::SMEM_BYTES));
  ACE_CUDA(cudaFuncSetAttribute(diag_block_batch_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)dg::SMEM_BYTES));
  int want = 16;
  if (const char* e = std::getenv("ACE_DIAG_CLUSTER")) want = (std::atoi(e) == 8) ? 8 : 16;
  int nc = 8;
  if (want == 16 &&
      cudaFuncSetAttribute(diag_block_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dg::SMEM_BYTES) ==
          cudaSuccess &&
      cudaFuncSetAttribute(diag_block_kernel<16>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(16, 1, 1);
    cfg.blockDim = dim3(dg::THREADS, 1, 1);
    cfg.dynamicSmemBytes = dg::SMEM_BYTES;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 16;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    int ncl = 0;
    if (cudaOccupancyMaxActiveClusters(&ncl, diag_block_kernel<16>, &cfg) == cudaSuccess && ncl >= 1) nc = 16;
  }
  (void)cudaGetLastError();  // a refused opt-in is not an error: the portable size is used
  diag_cluster_size() = nc;
  return 0;
}

// S members (blockIdx.y), 8-CTA clusters: the portable size, so that as many members as possible are in flight at once
constexpr int DIAG_BATCH_NC = 8;
inline int launch_diag_block_batch(const DiagArgs& a, const DiagStrides& m, int S, cudaStream_t st) {
  constexpr int NC = DIAG_BATCH_NC;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(NC, (unsigned)S, 1);
  cfg.blockDim = dim3(dg::THREADS, 1, 1);
  cfg.dynamicSmemBytes = dg::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = NC;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  ACE_CUDA(cudaLaunchKernelEx(&cfg, diag_block_batch_kernel<NC>, a, m));
  return 0;
}

// wide: use the 16-CTA cluster when the device accepts it (ACE_DIAG_CLUSTER=8 / 16 forces one size)
inline int launch_diag_block(const DiagArgs& a, cudaStream_t st, bool wide = true) {
  if (diag_cluster_size() == 0) ACE_TRY(configure_diag_kernel());
  static const int forced = [] {
    const char* e = std::getenv("ACE_DIAG_CLUSTER");
    return e ? std::atoi(e) : 0;
  }();
  const bool use16 = diag_cluster_size() == 16 && (forced == 16 || (forced == 0 && wide));
  return use16 ? launch_diag_block_nc<16>(a, st) : launch_diag_block_nc<8>(a, st);
}

}  // namespace ace
