// uut_i8.cuh -- K^-1 = U U^T on the INT8 tensor cores (tcgen05.mma kind::i8) by modular Ozaki splitting (scheme II).
//
// Every row of U gets a power-of-two scale 2^e_i > max_k |U(i,k)| and becomes an integer row
//     a'(i,k) = rint(U(i,k) * 2^(b - e_i)),   |a'| <= 2^b,   |U(i,k) - 2^(e_i - b) a'(i,k)| <= 2^(e_i - b - 1),
// b = crt_bits(n_pad) (55 up to n_pad = 16384, 54 up to MAX_N).  The exact integer product C' = a' a'^T is formed by
// the Chinese Remainder Theorem over the NMOD = 16 pairwise-coprime moduli m_t of MOD below (256 and the 15 largest
// odd ones <= 255 that stay coprime), M = prod m_t ~ 2^125.4:
//   split     a' mod m_t as a signed residue, [-128, 127] for 256 and [-(m-1)/2, (m-1)/2] for the odd moduli, one
//             INT8 plane per modulus;
//   product   per modulus, C'_t = A_t A_t^T on the lower 128 x 256 tiles: one exact INT32 accumulator (|residue
//             product| <= 2^14, K <= MAX_N < 2^17 terms), reduced by the epilogue to a signed residue mod m_t;
//   CRT       Garner's mixed radix with signed digits, radix 256 first (digit sums as exact FP32 FMAs), recovers the
//             unique C' in [-M/2, M/2), which holds every |C'| <= n_pad 2^(2b) < M/2 (static_asserts below).  C' is
//             formed exactly (two 64-bit Horner halves joined in 128 bits) and rounded to FP64 ONCE (round to
//             nearest even); the scale 2^(e_i + e_j - 2b) is exact.
// So C_ij is the correctly rounded value of 2^(e_i+e_j-2b) sum_k a'(i,k) a'(j,k) (bar underflow to subnormals): the
// only errors are the row truncation above (2^-55 of the row maximum at C3, as the 8-plane scheme-I split had) and
// that one rounding; no cross term is dropped.  C'_ij = C'_ji exactly, so the result is exactly symmetric and
// deterministic.
//
// Workspace (OzWork::planes, NMOD + 1 slots of slot_bytes(nb) = nb (nb + 1) / 2 * 16 KB each; 2.28 GB at n_pad =
// 16384, against 1.07 GB for the earlier 8-plane engine): operand plane t lives in slot t + 1.  The product of modulus t reads slot t + 1 and writes the residues of
// its lower 128 x 128 blocks into slot t, whose operand plane (t - 1) the previous launch has consumed (a slot holds
// nb (nb + 1) / 2 blocks of 16 KB in either layout): the 16 output residue planes cost one slot beyond the 16
// operand planes.  Slot 0 is that extra slot.
//
// Operand layout (what the UMMA shared-memory descriptor reads, no swizzle, K-major): per slot, per 128-row block rb,
// per 32-deep k chunk c >= 4 rb (U is upper triangular: earlier chunks are never read and not stored), one 4 KB block;
// inside it, core matrix (8 rows x 16 bytes, 128 contiguous bytes) (row group r/8, k half kk/16) sits at
// (r/8) * 256 + (kk/16) * 128.  The 256 B operand of a stage is two such blocks, back to back in shared memory.
// Residue layout: per slot, lower 128 x 128 block (ti, tj <= ti) at (ti (ti + 1) / 2 + tj) * 16 KB, row-major.
#pragma once
#include "common.cuh"

namespace ace {

namespace oz {
constexpr int NMOD = 16;
constexpr int MOD[NMOD] = {256, 255, 253, 251, 247, 241, 239, 233, 229, 227, 223, 217, 211, 199, 197, 193};
constexpr int BM = 128, BN = 256, BK = 32;  // BK = int8 k values per stage = the K of one kind::i8 MMA
constexpr int CPB = TB / BK;                // k chunks per 128-block
constexpr int STAGES = 8;
constexpr int A_BYTES = BM * BK, B_BYTES = BN * BK;
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
// 99 KB: two CTAs per SM (their 2 x 256 TMEM columns fill the 512), so one tile's epilogue overlaps the other's MMAs;
// a third would not fit the shared memory, and could not allocate tensor memory
constexpr size_t SMEM_BYTES = 1024 + (size_t)STAGES * STAGE_BYTES + 128;
static_assert(2 * SMEM_BYTES <= 227 * 1024 && 3 * SMEM_BYTES > 228 * 1024, "exactly two CTAs per SM");
constexpr int TMEM_COLS = BN;
constexpr int THREADS = 192;  // warp 0: bulk-copy producer, warp 1: MMA issuer + TMEM owner, warps 2-5: epilogue
constexpr int MAX_N = 65408;  // n_pad bound of the CRT range at b = 54 (below); larger problems use DMMA
static_assert((long)128 * 128 * MAX_N <= 2147483647L, "INT32 accumulators may overflow");
// instruction descriptor: D s32 (bits 4-5 = 2), A and B signed 8-bit (bits 7-9, 10-12 = 1), both K-major,
// N >> 3 at bits 17-22, M >> 4 at bits 24-28
constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

// bits of the integer rows: the largest b with n_pad 2^(2b) < M/2 over each range
constexpr int crt_bits(int n_pad) { return n_pad <= 16384 ? 55 : 54; }
constexpr unsigned __int128 crt_half_range() {
  unsigned __int128 p = 1;
  for (int t = 0; t < NMOD; ++t) p *= (unsigned)MOD[t];
  return p / 2;
}
static_assert(((unsigned __int128)16384 << (2 * 55)) < crt_half_range(), "CRT range at b = 55");
static_assert(((unsigned __int128)MAX_N << (2 * 54)) < crt_half_range(), "CRT range at b = 54");

// byte offset of the (slot t, row block rb, k chunk c) operand block; c >= CPB * rb
__host__ __device__ inline size_t block_off(int nb, int t, int rb, int c) {
  const long nc = (long)nb * CPB;
  const long per_plane = (long)nb * nc - (long)CPB * nb * (nb - 1) / 2;
  const long off = (long)rb * nc - (long)CPB * rb * (rb - 1) / 2 + (c - (long)CPB * rb);
  return ((size_t)t * per_plane + off) * (size_t)(BM * BK);
}
__host__ __device__ inline size_t slot_bytes(int nb) { return block_off(nb, 1, 0, 0); }
inline size_t plane_bytes(int nb) { return block_off(nb, NMOD + 1, 0, 0); }
// byte offset of lower residue block (ti, tj) inside a slot: the same bytes as the operand blocks of row block ti
__host__ __device__ inline size_t res_off(int ti, int tj) { return ((size_t)ti * (ti + 1) / 2 + tj) * (size_t)(TB * TB); }
// lower 128 x 256 product tiles: row block ti holds ti / 2 + 1 of them
inline long product_tiles(int nb) { return (long)(nb / 2) * (nb / 2 + 1) + (nb & 1) * (nb / 2 + 1); }

// Constants of the three kernels, built once on the host and passed by value (kernel parameter space: a loop
// unrolled over t reads them as constant-bank operands).  x mod m for 0 <= x < 2^24 is x - m umulhi(x, magic) with
// magic = ceil(2^32 / m): the quotient estimate is exact while x < 2^32 / m.
struct Tables {
  int m[NMOD];
  unsigned magic[NMOD];
  int c14[NMOD], c28[NMOD], c42[NMOD];  // 2^14, 2^28, 2^42 mod m (split)
  // Garner, in FP32: every operand and partial sum is an integer below 2^20 in magnitude, so each FMA is exact
  float mf[NMOD], rcp[NMOD];            // m_k, 1 / m_k rounded
  float inv[NMOD];                      // (m_0 ... m_{k-1})^-1 mod m_k
  float w[NMOD][NMOD];                  // w[k][j] = (m_0 ... m_{j-1}) inv[k] mod m_k, j < k
  unsigned long long p8;                // m_0 ... m_7 < 2^64: joins the two 8-digit halves
};

inline Tables make_tables() {
  Tables T{};
  for (int k = 0; k < NMOD; ++k) {
    const long m = MOD[k];
    T.m[k] = (int)m;
    T.magic[k] = (unsigned)(((1ull << 32) + (unsigned long long)m - 1) / (unsigned long long)m);
    T.c14[k] = (int)((1L << 14) % m);
    T.c28[k] = (int)((1L << 28) % m);
    T.c42[k] = (int)((1L << 42) % m);
    T.mf[k] = (float)m;
    T.rcp[k] = 1.0f / (float)m;
    long pk = 1;  // m_0 ... m_{k-1} mod m_k
    for (int j = 0; j < k; ++j) pk = pk * MOD[j] % m;
    long inv = 1;
    while (k > 0 && pk * inv % m != 1) ++inv;
    T.inv[k] = (float)inv;
    long pj = 1;
    for (int j = 0; j < k; ++j) {
      T.w[k][j] = (float)(pj * inv % m);
      pj = pj * MOD[j] % m;
    }
  }
  T.p8 = 1;
  for (int j = 0; j < 8; ++j) T.p8 *= (unsigned long long)MOD[j];
  return T;
}
}  // namespace oz

// signed residue of 0 <= x < 2^24 modulo the odd modulus t: [-(m-1)/2, (m-1)/2]
__device__ __forceinline__ int oz_smod(unsigned x, const oz::Tables& T, int t) {
  const int r = (int)(x - (unsigned)T.m[t] * __umulhi(x, T.magic[t]));
  return r > (T.m[t] >> 1) ? r - T.m[t] : r;
}

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
// Split: row maxima, then residue planes + row exponents.  U(i,k) = upper(A)[i + k*ld] off the diagonal 128-blocks,
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
                                                       const unsigned long long* __restrict__ rowmax, int nb, int b,
                                                       const __grid_constant__ oz::Tables T,
                                                       int8_t* __restrict__ planes, int* __restrict__ ex) {
  using namespace oz;
  const int cb = blockIdx.x, rb = blockIdx.y, r = threadIdx.x;
  if (cb < rb) return;
  const double m = __longlong_as_double((long long)rowmax[rb * TB + r]);
  int e = 0;
  if (m > 0.0) frexp(m, &e);  // m < 2^e
  if (cb == rb) ex[rb * TB + r] = e;
  const double scale = ldexp(1.0, b - e);
#pragma unroll 1
  for (int q = 0; q < TB / 16; ++q) {  // 16 k values = one core-matrix row of every plane
    uint32_t w[NMOD][4];
#pragma unroll
    for (int t = 0; t < NMOD; ++t) w[t][0] = w[t][1] = w[t][2] = w[t][3] = 0u;
#pragma unroll
    for (int x16 = 0; x16 < 16; ++x16) {
      // |U| 2^(b-e) < 2^b exactly; its rint is an integer-valued double, converted exactly
      const long long a = __double2ll_rn(rint(oz_u(A, ld, DU, rb, cb, r, q * 16 + x16) * scale));
      const unsigned long long ua = (unsigned long long)(a < 0 ? -a : a);
      const unsigned q0 = (unsigned)ua & 0x3FFFu, q1 = (unsigned)(ua >> 14) & 0x3FFFu,
                     q2 = (unsigned)(ua >> 28) & 0x3FFFu, q3 = (unsigned)(ua >> 42);  // |a| <= 2^55: q3 <= 2^13
      const int sh = 8 * (x16 & 3);
      w[0][x16 >> 2] |= ((uint32_t)a & 0xffu) << sh;  // two's complement low byte = residue mod 256 in [-128, 127]
#pragma unroll
      for (int t = 1; t < NMOD; ++t) {
        // |a| mod m from 14-bit chunks: the sum stays below 2^14 (1 + 3 * 254) < 2^24
        const int s = oz_smod(q0 + q1 * (unsigned)T.c14[t] + q2 * (unsigned)T.c28[t] + q3 * (unsigned)T.c42[t], T, t);
        w[t][x16 >> 2] |= ((uint32_t)(a < 0 ? -s : s) & 0xffu) << sh;
      }
    }
    const int c = cb * CPB + q / 2;
    const size_t in_blk = (size_t)(r >> 3) * 256 + (q & 1) * 128 + (r & 7) * 16;
#pragma unroll
    for (int t = 0; t < NMOD; ++t)
      *reinterpret_cast<uint4*>(planes + block_off(nb, t + 1, rb, c) + in_blk) =
          make_uint4(w[t][0], w[t][1], w[t][2], w[t][3]);
  }
}

// ---------------------------------------------------------------------------------------------
// Product of one modulus: one CTA per lower 128 x 256 tile (ti, column blocks 2 tj2 and 2 tj2 + 1 <= ti when it
// exists), k from the tile's row block; tiles in order of ti, the longest first.  Reads operand slot `slot + 1`,
// writes the residues of C'_t into slot `slot`.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(oz::THREADS, 2) uut_i8_mod_kernel(int8_t* __restrict__ planes, int nb, int slot,
                                                                    int m, double inv_m) {
  using namespace oz;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* sm = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(sm + (size_t)STAGES * STAGE_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* done = empty + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  int ti, tj2;
  {
    // row blocks 2q and 2q + 1 hold q + 1 tiles each: q(q + 1) tiles precede row block 2q
    const long L = blockIdx.x;
    long q = (long)((sqrt(4.0 * (double)L + 1.0) - 1.0) * 0.5);
    while (q * (q + 1) > L) --q;
    while ((q + 1) * (q + 2) <= L) ++q;
    const long rem = L - q * (q + 1);
    ti = (int)(2 * q + rem / (q + 1));
    tj2 = (int)(rem % (q + 1));
  }
  const int jb0 = 2 * tj2;
  const bool has1 = jb0 + 1 <= ti;            // the second column block is lower (and exists)
  const int jb1 = has1 ? jb0 + 1 : jb0;       // otherwise its half of the tile repeats the first and is not stored
  const int c_begin = ti * CPB, nchunks = nb * CPB - c_begin;
  const int8_t* src = planes;

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
        tma_bulk_g2s(st, src + block_off(nb, slot + 1, ti, c), A_BYTES, &full[s]);
        tma_bulk_g2s(st + A_BYTES, src + block_off(nb, slot + 1, jb0, c), A_BYTES, &full[s]);
        tma_bulk_g2s(st + 2 * A_BYTES, src + block_off(nb, slot + 1, jb1, c), A_BYTES, &full[s]);
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
        const uint32_t a0 = smem_u32(sm + (size_t)s * STAGE_BYTES);
        tc_mma_i8(tmem, oz_smem_desc(a0), oz_smem_desc(a0 + A_BYTES), it > 0 ? 1u : 0u);
        tc_commit(&empty[s]);  // stage free once its MMA has read it
      }
      tc_commit(done);
    }
    __syncwarp();
  } else {
    // ================================ epilogue: residues mod m ================================
    mbar_wait(done, 0);
    tc_fence_after();
    const int q = warp & 3;  // TMEM lane quadrant this warp may access
    const int r = q * 32 + lane;
    const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16);
    int8_t* dst = planes + block_off(nb, slot, 0, 0) + (size_t)r * TB;
#pragma unroll 1
    for (int jc = 0; jc < (has1 ? BN : TB) / 32; ++jc) {
      uint32_t v[2][16];
      tc_ld16(trow + (uint32_t)(jc * 32), v[0]);
      tc_ld16(trow + (uint32_t)(jc * 32 + 16), v[1]);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      uint32_t pk[8];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int x = (int)v[j >> 4][j & 15];
        int res;
        if (m == 256) {
          res = x;  // the low byte is the residue in [-128, 127]
        } else {
          // |x| < 2^31: x / m is never within 1/(2m) of a half-integer (m odd), far above the rounding of x * inv_m
          res = x - m * (int)rint((double)x * inv_m);
        }
        if ((j & 3) == 0) pk[j >> 2] = 0u;
        pk[j >> 2] |= ((uint32_t)res & 0xffu) << (8 * (j & 3));
      }
      uint4* o = reinterpret_cast<uint4*>(dst + res_off(ti, jb0 + (jc >> 2)) + (jc & 3) * 32);
      o[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      o[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------
// CRT: one CTA per lower 128 x 128 block (ti, tj), 32 rows per pass.  Every entry: 16 residues -> signed Garner
// digits -> C' exactly (64-bit halves, 128-bit join) -> one rounding to FP64 -> exact scale; then the block and its mirror are written
// through shared memory, both coalesced (the diagonal block once).
// ---------------------------------------------------------------------------------------------
// exact conversions between FP32 and int32 for |x| < 2^22 on the FP32 / integer pipes (the converters are slower)
__device__ __forceinline__ float oz_i2f(int x) { return __int_as_float(0x4B400000 + x) - 0x1.8p23f; }
__device__ __forceinline__ int oz_f2i(float x) { return __float_as_int(x + 0x1.8p23f) - 0x4B400000; }

__device__ __forceinline__ double oz_crt(const int (&res)[oz::NMOD], const oz::Tables& T, int scale_exp) {
  using namespace oz;
  float v[NMOD];
  v[0] = oz_i2f(res[0]);
#pragma unroll
  for (int k = 1; k < NMOD; ++k) {
    // v_k = (r_k - sum_{j<k} v_j m_0..m_{j-1}) (m_0..m_{k-1})^-1 mod m_k, with |v_j| <= 128, w < 256:
    // |s| < 2^15 + 15 * 2^15 < 2^20, every FMA exact
    float s = oz_i2f(res[k]) * T.inv[k];
#pragma unroll
    for (int j = 0; j < k; ++j) s = fmaf(-v[j], T.w[k][j], s);
    // the quotient estimate is off by at most one (|s / m| < 2^13, relative error < 2^-22): r exact, then centred
    float r = fmaf(-T.mf[k], rintf(s * T.rcp[k]), s);
    const float h = 0.5f * T.mf[k];
    r = r > h ? r - T.mf[k] : r;
    r = r < -h ? r + T.mf[k] : r;
    v[k] = r;
  }
  // C' = v_0 + m_0 (v_1 + m_1 (v_2 + ...)): the signed digits span exactly [-M/2, M/2).  Each 8-digit half by
  // Horner in 64 bits (|half| < 2^63, wrapping arithmetic), joined once in 128 bits.
  unsigned long long ulo = (unsigned long long)(long long)oz_f2i(v[7]);
  unsigned long long uhi = (unsigned long long)(long long)oz_f2i(v[NMOD - 1]);
#pragma unroll
  for (int k = 6; k >= 0; --k) ulo = ulo * (unsigned)T.m[k] + (unsigned long long)(long long)oz_f2i(v[k]);
#pragma unroll
  for (int k = NMOD - 2; k >= 8; --k) uhi = uhi * (unsigned)T.m[k] + (unsigned long long)(long long)oz_f2i(v[k]);
  const __int128 x = (__int128)(long long)uhi * (__int128)T.p8 + (__int128)(long long)ulo;
  const bool neg = x < 0;
  const unsigned __int128 u = neg ? (unsigned __int128)(-x) : (unsigned __int128)x;
  const unsigned long long hi = (unsigned long long)(u >> 64), lo = (unsigned long long)u;
  double d;
  if (hi == 0) {
    d = ldexp(__ull2double_rn(lo), scale_exp);
  } else {
    // the leading 64 bits with a sticky bit for the rest round to 53 bits exactly as the whole would
    const int z = __clzll((long long)hi);
    const unsigned long long top = z ? (hi << z) | (lo >> (64 - z)) : hi;
    const unsigned long long rest = lo << z;
    d = ldexp(__ull2double_rn(top | (rest != 0 ? 1ull : 0ull)), scale_exp + 64 - z);
  }
  return neg ? -d : d;
}

__global__ void __launch_bounds__(256) oz_crt_kernel(const int8_t* __restrict__ planes, const int* __restrict__ ex,
                                                     int nb, int b, const __grid_constant__ oz::Tables T,
                                                     double* __restrict__ C, long ldc) {
  using namespace oz;
  __shared__ double tile[32][TB + 1];
  int ti, tj;
  {
    const long L = blockIdx.x;
    long t = (long)((sqrt(8.0 * (double)L + 1.0) - 1.0) * 0.5);
    while (t * (t + 1) / 2 > L) --t;
    while ((t + 1) * (t + 2) / 2 <= L) ++t;
    ti = (int)t;
    tj = (int)(L - t * (t + 1) / 2);
  }
  const size_t sb = slot_bytes(nb);
  const int8_t* blk = planes + res_off(ti, tj);
  const int tid = threadIdx.x, rr = tid >> 3, c0 = (tid & 7) * 16;
  const int i0 = ti * TB, j0 = tj * TB;
#pragma unroll 1
  for (int r0 = 0; r0 < TB; r0 += 32) {
    const int r = r0 + rr;
    uint4 rv[NMOD];
#pragma unroll
    for (int t = 0; t < NMOD; ++t) rv[t] = *reinterpret_cast<const uint4*>(blk + t * sb + (size_t)r * TB + c0);
    const int ei = ex[i0 + r];
#pragma unroll 1
    for (int j = 0; j < 16; ++j) {
      int res[NMOD];
#pragma unroll
      for (int t = 0; t < NMOD; ++t) {
        const uint32_t wv = j < 4 ? rv[t].x : j < 8 ? rv[t].y : j < 12 ? rv[t].z : rv[t].w;
        res[t] = (int)(int8_t)(wv >> (8 * (j & 3)));
      }
      tile[rr][c0 + j] = oz_crt(res, T, ei + ex[j0 + c0 + j] - 2 * b);
    }
    __syncthreads();
#pragma unroll 4
    for (int k = tid; k < 32 * TB; k += 256) {  // rows of the block: C[(i0 + r) * ldc + j0 + c]
      const int a = k >> 7, c = k & (TB - 1);
      C[(size_t)(i0 + r0 + a) * ldc + j0 + c] = tile[a][c];
    }
    if (ti != tj) {
#pragma unroll 4
      for (int k = tid; k < 32 * TB; k += 256) {  // the mirror: C[(j0 + c) * ldc + i0 + r]
        const int c = k >> 5, a = k & 31;
        C[(size_t)(j0 + c) * ldc + i0 + r0 + a] = tile[a][c];
      }
    }
    __syncthreads();
  }
}

struct OzWork {
  int8_t* planes = nullptr;              // oz::plane_bytes(nb): NMOD + 1 slots
  unsigned long long* rowmax = nullptr;  // n_pad
  int* ex = nullptr;                     // n_pad
};

inline int configure_uut_i8_kernel() {
  ACE_CUDA(cudaFuncSetAttribute(uut_i8_mod_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)oz::SMEM_BYTES));
  return 0;
}

// C (ld = n_pad = nb * 128, both triangles) = U U^T from U = upper(A) with the diagonal tiles in DU
inline int launch_uut_i8(const OzWork& o, const double* A, const double* DU, int nb, double* C, cudaStream_t st) {
  using namespace oz;
  if ((long)nb * TB > MAX_N) {
    set_error("uut_i8: n_pad beyond the CRT range bound");
    return -2;
  }
  if (!o.planes || !o.rowmax || !o.ex) {
    set_error("uut_i8: residue-plane workspace not allocated");
    return -2;
  }
  static const Tables T = make_tables();
  const long ld = (long)nb * TB;
  const int b = crt_bits((int)ld);
  ACE_CUDA(cudaMemsetAsync(o.rowmax, 0, sizeof(unsigned long long) * (size_t)ld, st));
  const dim3 g2(nb, nb);
  oz_rowmax_kernel<<<g2, TB, 0, st>>>(A, ld, DU, o.rowmax);
  ACE_CUDA(cudaGetLastError());
  oz_split_kernel<<<g2, TB, 0, st>>>(A, ld, DU, o.rowmax, nb, b, T, o.planes, o.ex);
  ACE_CUDA(cudaGetLastError());
  const long tiles = product_tiles(nb);
  for (int t = 0; t < NMOD; ++t) {
    uut_i8_mod_kernel<<<(unsigned)tiles, THREADS, SMEM_BYTES, st>>>(o.planes, nb, t, MOD[t], 1.0 / MOD[t]);
    ACE_CUDA(cudaGetLastError());
  }
  oz_crt_kernel<<<(unsigned)((long)nb * (nb + 1) / 2), 256, 0, st>>>(o.planes, o.ex, nb, b, T, C, ld);
  ACE_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace ace
