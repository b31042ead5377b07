// uut_i8.cuh -- K^-1 = U U^T on the INT8 tensor cores (tcgen05.mma kind::i8) by Ozaki splitting (scheme I).
//
// Every row of U gets a power-of-two scale 2^e_i > 2 max_k |U(i,k)| and is split, exactly, into S signed 8-bit
// digit planes:   U(i,k) = 2^e_i sum_{t<S} 2^(-7(t+1)) D_t(i,k) + r(i,k),   |D_t| <= 64,  |r| <= 2^(e_i-7S-1).
// The product keeps the digit pairs with a + b <= S - 1 (S(S+1)/2 products); pairs of equal a + b carry the same
// weight and share one INT32 accumulator, so a 128 x 64 output tile holds S accumulators (S * 64 TMEM columns).
// The epilogue folds them in a fixed order:  C_ij = 2^(e_i+e_j-14) sum_g 2^(-7g) acc_g(i,j).  The integer sums
// are exact and acc_g(i,j) = acc_g(j,i), so the result is exactly symmetric; the only rounding is the FP64 fold.
//
// Splitting is error free: x = U * 2^-e (exact), then per digit x <- 128 x (exact), d = rint(x), x <- x - d
// (exact by Sterbenz, |x - d| <= 1/2), so |d| <= 64 at every step.
//
// INT32 headroom: group g has at most S pairs, each |D_a D_b| <= 2^12, so after K products of k an accumulator is
// bounded by S * 2^12 * K.  K <= KMAX = floor((2^31 - 1) / (S * 2^12)) keeps it exact without an intermediate fold:
// 65535 for S = 8, i.e. every n_pad <= MAX_N = 65408.  Larger problems (C4, n = 65536) use the DMMA engine.
//
// Plane layout (what the UMMA shared-memory descriptor reads, no swizzle, K-major): per plane, per 128-row block rb,
// per 32-deep k chunk c >= 4 rb (U is upper triangular: earlier chunks are never read and not stored), one 4 KB
// block; inside it, core matrix (8 rows x 16 bytes, 128 contiguous bytes) (row group r/8, k half kk/16) sits at
// (r/8) * 256 + (kk/16) * 128.  A 64-row half of a block is then 2 KB contiguous, so every operand of a pipeline
// stage is ONE cp.async.bulk behind an mbarrier.
#pragma once
#include "common.cuh"

namespace ace {

namespace oz {
constexpr int S = 8;           // digit planes (error study: DESIGN section 3.2c)
constexpr int DMAX = 64;       // |digit| bound
constexpr int BM = 128, BN = 64, BK = 32;  // BK = int8 k values per stage = the K of one kind::i8 MMA
constexpr int CPB = TB / BK;   // k chunks per 128-block
constexpr int STAGES = 4;
constexpr int A_PLANE = BM * BK, B_PLANE = BN * BK;  // bytes per plane and stage
constexpr int STAGE_BYTES = S * (A_PLANE + B_PLANE);
constexpr size_t SMEM_BYTES = 1024 + (size_t)STAGES * STAGE_BYTES + 128;  // 193 KB: one CTA per SM
static_assert(SMEM_BYTES <= 227 * 1024, "pipeline exceeds the shared memory of one block");
constexpr int TMEM_COLS = 512;
constexpr int THREADS = 192;   // warp 0: bulk-copy producer, warp 1: MMA issuer + TMEM owner, warps 2-5: epilogue
constexpr long KMAX = 2147483647L / ((long)S * DMAX * DMAX);
constexpr int MAX_N = (int)(KMAX / TB) * TB;
static_assert(S * BN <= TMEM_COLS, "S accumulators of BN columns must fit the 512 TMEM columns");
static_assert((long)S * DMAX * DMAX * MAX_N <= 2147483647L, "INT32 accumulators may overflow");
// instruction descriptor: D s32 (bits 4-5 = 2), A and B signed 8-bit (bits 7-9, 10-12 = 1), both K-major,
// N >> 3 at bits 17-22, M >> 4 at bits 24-28
constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

// byte offset of the (plane t, row block rb, k chunk c) block; c >= CPB * rb
__host__ __device__ inline size_t block_off(int nb, int t, int rb, int c) {
  const long nc = (long)nb * CPB;
  const long per_plane = (long)nb * nc - (long)CPB * nb * (nb - 1) / 2;
  const long off = (long)rb * nc - (long)CPB * rb * (rb - 1) / 2 + (c - (long)CPB * rb);
  return ((size_t)t * per_plane + off) * (size_t)(BM * BK);
}
inline size_t plane_bytes(int nb) { return block_off(nb, S, 0, 0); }
}  // namespace oz

// ---------------------------------------------------------------------------------------------
// tcgen05 wrappers
// ---------------------------------------------------------------------------------------------
// shared-memory matrix descriptor, no swizzle: LBO = 128 B between the two K-adjacent core matrices, SBO = 256 B
// between 8-row groups, bits 46-48 = 0b001 (sm_100 descriptor version)
__device__ __forceinline__ uint64_t oz_smem_desc(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) |
         (1ull << 46);
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tc_mma_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(oz::IDESC), "r"(accumulate)
      : "memory");
}

// arrives on the mbarrier once every MMA issued so far by this thread has completed
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

// ---------------------------------------------------------------------------------------------
// Split: row maxima, then digit planes + row exponents.  U(i,k) = upper(A)[i + k*ld] off the diagonal 128-blocks,
// DU tile rb on it (the operand dgemm_nt reads for the DMMA product).  CTA = (column block cb, row block rb),
// cb >= rb, one thread per row: every k step reads 128 contiguous doubles.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double oz_u(const double* A, long ld, const double* DU, int rb, int cb, int r, int kk) {
  return (cb == rb) ? DU[(size_t)rb * TB * TB + r + (size_t)kk * TB] : A[(size_t)rb * TB + r + (size_t)(cb * TB + kk) * ld];
}

__global__ void __launch_bounds__(128) oz_rowmax_kernel(const double* __restrict__ A, long ld,
                                                        const double* __restrict__ DU,
                                                        unsigned long long* __restrict__ rowmax) {
  const int cb = blockIdx.x, rb = blockIdx.y, r = threadIdx.x;
  if (cb < rb) return;
  double m = 0.0;
#pragma unroll 8
  for (int kk = 0; kk < TB; ++kk) m = fmax(m, fabs(oz_u(A, ld, DU, rb, cb, r, kk)));
  // non-negative doubles order like their bit patterns
  atomicMax(rowmax + rb * TB + r, (unsigned long long)__double_as_longlong(m));
}

__global__ void __launch_bounds__(128) oz_split_kernel(const double* __restrict__ A, long ld,
                                                       const double* __restrict__ DU,
                                                       const unsigned long long* __restrict__ rowmax, int nb,
                                                       int8_t* __restrict__ planes, int* __restrict__ ex) {
  using namespace oz;
  const int cb = blockIdx.x, rb = blockIdx.y, r = threadIdx.x;
  if (cb < rb) return;
  const double m = __longlong_as_double((long long)rowmax[rb * TB + r]);
  int e = 0;
  if (m > 0.0) {
    frexp(m, &e);  // m < 2^e
    ++e;           // |U| * 2^-e < 1/2: every digit within [-64, 64]
  }
  if (cb == rb) ex[rb * TB + r] = e;
  const double scale = ldexp(1.0, -e);
#pragma unroll 1
  for (int q = 0; q < TB / 16; ++q) {  // 16 k values = one core-matrix row of every plane
    uint32_t w[S][4];
#pragma unroll
    for (int t = 0; t < S; ++t) w[t][0] = w[t][1] = w[t][2] = w[t][3] = 0u;
#pragma unroll
    for (int x16 = 0; x16 < 16; ++x16) {
      double x = oz_u(A, ld, DU, rb, cb, r, q * 16 + x16) * scale;
#pragma unroll
      for (int t = 0; t < S; ++t) {
        x *= 128.0;
        const double d = rint(x);
        x -= d;
        w[t][x16 >> 2] |= ((uint32_t)(int)d & 0xffu) << (8 * (x16 & 3));
      }
    }
    const int c = cb * CPB + q / 2;
    const size_t in_blk = (size_t)(r >> 3) * 256 + (q & 1) * 128 + (r & 7) * 16;
#pragma unroll
    for (int t = 0; t < S; ++t)
      *reinterpret_cast<uint4*>(planes + block_off(nb, t, rb, c) + in_blk) = make_uint4(w[t][0], w[t][1], w[t][2], w[t][3]);
  }
}

// ---------------------------------------------------------------------------------------------
// Product: one CTA per lower 128 x 64 tile (the tile order of dgemm_nt's lower_only), k from the tile's row block.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(oz::THREADS, 1) uut_i8_kernel(const int8_t* __restrict__ planes,
                                                                const int* __restrict__ ex, int nb,
                                                                double* __restrict__ C, long ldc) {
  using namespace oz;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* sm = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(sm + (size_t)STAGES * STAGE_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* done = empty + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  int ti, tj;
  {
    const long L = blockIdx.x;
    long t = (long)((sqrt(4.0 * (double)L + 1.0) - 1.0) * 0.5);
    while (t * (t + 1) > L) --t;
    while ((t + 1) * (t + 2) <= L) ++t;
    ti = (int)t;
    tj = (int)(L - t * (t + 1));
  }
  const int i0 = ti * BM, j0 = tj * BN, jb = tj >> 1, jh = tj & 1;
  const int c_begin = ti * CPB, nchunks = nb * CPB - c_begin;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(done, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ================================ bulk-copy producer ======================================
    if (lane == 0) {
      for (int it = 0; it < nchunks; ++it) {
        const int s = it % STAGES;
        mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
        mbar_arrive_expect_tx(&full[s], STAGE_BYTES);
        unsigned char* st = sm + (size_t)s * STAGE_BYTES;
        const int c = c_begin + it;
#pragma unroll
        for (int t = 0; t < S; ++t)
          tma_bulk_g2s(st + t * A_PLANE, planes + block_off(nb, t, ti, c), A_PLANE, &full[s]);
#pragma unroll
        for (int t = 0; t < S; ++t)
          tma_bulk_g2s(st + S * A_PLANE + t * B_PLANE, planes + block_off(nb, t, jb, c) + jh * B_PLANE, B_PLANE,
                       &full[s]);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================================ single MMA issuer =======================================
    if (lane == 0) {
      for (int it = 0; it < nchunks; ++it) {
        const int s = it % STAGES;
        mbar_wait(&full[s], (it / STAGES) & 1);
        tc_fence_after();
        const uint32_t a0 = smem_u32(sm + (size_t)s * STAGE_BYTES), b0 = a0 + S * A_PLANE;
#pragma unroll
        for (int a = 0; a < S; ++a)
#pragma unroll
          for (int b = 0; a + b < S; ++b)  // group a + b; a == 0 opens every group
            tc_mma_i8(tmem + (uint32_t)((a + b) * BN), oz_smem_desc(a0 + a * A_PLANE), oz_smem_desc(b0 + b * B_PLANE),
                      (it > 0 || a > 0) ? 1u : 0u);
        tc_commit(&empty[s]);  // stage free once its MMAs have read it
      }
      tc_commit(done);
    }
    __syncwarp();
  } else {
    // ================================ epilogue: fold + mirrored store ==========================
    mbar_wait(done, 0);
    tc_fence_after();
    const int q = warp & 3;  // TMEM lane quadrant this warp may access
    const int r = q * 32 + lane, i = i0 + r;
    const int ei = ex[i] - 14;
    const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
    for (int jc = 0; jc < BN / 16; ++jc) {
      uint32_t v[S][16];
#pragma unroll
      for (int g = 0; g < S; ++g) tc_ld16(trow + (uint32_t)(g * BN + jc * 16), v[g]);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      double out[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        double acc = (double)(int)v[S - 1][j];
#pragma unroll
        for (int g = S - 2; g >= 0; --g) acc = fma(acc, 0x1p-7, (double)(int)v[g][j]);
        const int col = j0 + jc * 16 + j;
        out[j] = ldexp(acc, ei + ex[col]);
        C[(size_t)col * ldc + i] = out[j];
      }
      double2* ct = reinterpret_cast<double2*>(C + (size_t)i * ldc + j0 + jc * 16);
#pragma unroll
      for (int j = 0; j < 8; ++j) ct[j] = make_double2(out[2 * j], out[2 * j + 1]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS) : "memory");
  }
}

struct OzWork {
  int8_t* planes = nullptr;           // oz::plane_bytes(nb)
  unsigned long long* rowmax = nullptr;  // n_pad
  int* ex = nullptr;                  // n_pad
};

inline int configure_uut_i8_kernel() {
  ACE_CUDA(cudaFuncSetAttribute(uut_i8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)oz::SMEM_BYTES));
  return 0;
}

// C (ld = n_pad = nb * 128, both triangles) = U U^T from U = upper(A) with the diagonal tiles in DU
inline int launch_uut_i8(const OzWork& o, const double* A, const double* DU, int nb, double* C, cudaStream_t st) {
  using namespace oz;
  if ((long)nb * TB > MAX_N) {
    set_error("uut_i8: n_pad beyond the INT32 accumulator bound");
    return -2;
  }
  if (!o.planes || !o.rowmax || !o.ex) {
    set_error("uut_i8: digit-plane workspace not allocated");
    return -2;
  }
  const long ld = (long)nb * TB;
  ACE_CUDA(cudaMemsetAsync(o.rowmax, 0, sizeof(unsigned long long) * (size_t)ld, st));
  const dim3 g2(nb, nb);
  oz_rowmax_kernel<<<g2, TB, 0, st>>>(A, ld, DU, o.rowmax);
  ACE_CUDA(cudaGetLastError());
  oz_split_kernel<<<g2, TB, 0, st>>>(A, ld, DU, o.rowmax, nb, o.planes, o.ex);
  ACE_CUDA(cudaGetLastError());
  const long tiles = (long)nb * (nb + 1);
  uut_i8_kernel<<<(unsigned)tiles, THREADS, SMEM_BYTES, st>>>(o.planes, o.ex, nb, C, ld);
  ACE_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace ace
