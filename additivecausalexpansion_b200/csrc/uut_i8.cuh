// uut_i8.cuh -- NT products C = +-A B^T on the INT8 tensor cores (tcgen05.mma kind::i8) by modular Ozaki splitting
// (scheme II): K^-1 = U U^T, and the two products of the top-level merge of the triangular inverse (chol.cuh).
//
// Every row of A and of B gets a power-of-two scale 2^e_i > max_k |X(i,k)| and becomes an integer row
//     a'(i,k) = rint(X(i,k) * 2^(b - e_i)),   |a'| <= 2^b,   |X(i,k) - 2^(e_i - b) a'(i,k)| <= 2^(e_i - b - 1),
// b = crt_bits(K) (55 up to K = 16384, 54 up to MAX_N), K the contraction length.  The exact integer product
// C' = a' b'^T is formed by the Chinese Remainder Theorem over the NMOD = 16 pairwise-coprime moduli m_t of MOD below
// (256 and the 15 largest odd ones <= 255 that stay coprime), M = prod m_t ~ 2^125.4:
//   split     a' mod m_t as a signed residue, [-128, 127] for 256 and [-(m-1)/2, (m-1)/2] for the odd moduli, one
//             INT8 plane per modulus;
//   product   per modulus, C'_t = A_t B_t^T on 128 x 256 tiles: one exact INT32 accumulator (|residue product| <=
//             2^14, K <= MAX_N < 2^17 terms), reduced by the epilogue to a signed residue mod m_t;
//   CRT       Garner's mixed radix with signed digits, radix 256 first (digit sums as exact FP32 FMAs), recovers the
//             unique C' in [-M/2, M/2), which holds every |C'| <= K 2^(2b) < M/2 (static_asserts below).  C' is
//             formed exactly (two 64-bit Horner halves joined in 128 bits) and rounded to FP64 ONCE (round to
//             nearest even); the scale 2^(e_i + e_j - 2b) and the sign are exact.
// So C_ij is the correctly rounded value of +-2^(e_i+e_j-2b) sum_k a'(i,k) b'(j,k) (bar underflow to subnormals): the
// only errors are the row truncation above (2^-55 of the row maximum at K <= 16384) and that one rounding; no cross
// term is dropped.  The result is deterministic, and in the symmetric mode (B = A) exactly symmetric.
//
// Operands (OzNT): each is dense, upper triangular (row block rb has k >= 128 rb; its diagonal tiles come from a
// separate array of dense 128 x 128 tiles, DU as potrf_trtri leaves it) or lower triangular (k < 128 (rb + 1), diagonal
// tiles likewise, DX).  The split stores only the k chunks an operand can have nonzero, and a tile's product runs
// over the intersection of the k ranges of its rows.  A triangular B is only read in the symmetric mode, where every
// tile is lower (column blocks <= ti) and B's k ranges hold A's.  Outputs: the symmetric mode writes the lower tiles
// and their mirror into C; the dense mode writes the M x N block C = +-A B^T and, optionally, its transpose into Ct.
//
// Workspace (OzWork::planes, NMOD + 1 slots of max(operand bytes, residue bytes) of one modulus; U U^T at n_pad =
// 16384: 17 x 135 MB = 2.28 GB): operand planes of modulus t (A, then B unless symmetric) live in slot t + 1.  The
// product of modulus t reads slot t + 1 and writes the residues of its 128 x 128 output blocks into slot t, whose
// operand plane (t - 1) the previous launch has consumed: the 16 output residue planes cost one slot beyond the 16
// operand planes.  Slot 0 is that extra slot.
//
// Operand layout (what the UMMA shared-memory descriptor reads, no swizzle, K-major): per operand, per 128-row block
// rb, per 32-deep k chunk c of its range, one 4 KB block; inside it, core matrix (8 rows x 16 bytes, 128 contiguous
// bytes) (row group r/8, k half kk/16) sits at (r/8) * 256 + (kk/16) * 128.  The 256 B operand of a stage is two such
// blocks, back to back in shared memory.  Residue layout: 128 x 128 blocks of 16 KB, row-major; lower block (ti, tj)
// at ti (ti + 1) / 2 + tj (symmetric), block (ti, tj) at ti * (N / 128) + tj (dense).
#pragma once
#include "common.cuh"

#include <algorithm>

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
constexpr int MAX_N = 65408;  // K bound of the CRT range at b = 54 (below); longer contractions use DMMA
static_assert((long)128 * 128 * MAX_N <= 2147483647L, "INT32 accumulators may overflow");
// instruction descriptor: D s32 (bits 4-5 = 2), A and B signed 8-bit (bits 7-9, 10-12 = 1), both K-major,
// N >> 3 at bits 17-22, M >> 4 at bits 24-28
constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

// bits of the integer rows: the largest b with K 2^(2b) < M/2 over each range of the contraction length K
constexpr int crt_bits(int K) { return K <= 16384 ? 55 : 54; }
constexpr unsigned __int128 crt_half_range() {
  unsigned __int128 p = 1;
  for (int t = 0; t < NMOD; ++t) p *= (unsigned)MOD[t];
  return p / 2;
}
static_assert(((unsigned __int128)16384 << (2 * 55)) < crt_half_range(), "CRT range at K = 16384, b = 55");
static_assert(((unsigned __int128)MAX_N << (2 * 54)) < crt_half_range(), "CRT range at K = MAX_N, b = 54");

enum Shape { DENSE = 0, UPPER = 1, LOWER = 2 };
// k chunks [chunk_lo, chunk_hi) of row block rb of an operand with nck chunks per row (triangular: square, rows = K)
__host__ __device__ inline int chunk_lo(int shape, int rb) { return shape == UPPER ? CPB * rb : 0; }
__host__ __device__ inline int chunk_hi(int shape, int rb, int nck) { return shape == LOWER ? CPB * (rb + 1) : nck; }
// 4 KB blocks stored before row block rb
__host__ __device__ inline long blocks_before(int shape, int rb, int nck) {
  if (shape == UPPER) return (long)rb * nck - (long)CPB * rb * (rb - 1) / 2;
  if (shape == LOWER) return (long)CPB * rb * (rb + 1) / 2;
  return (long)rb * nck;
}
// byte offset of the (row block rb, k chunk c) block inside an operand plane; chunk_lo <= c < chunk_hi
__host__ __device__ inline size_t op_off(int shape, int nck, int rb, int c) {
  return (size_t)(blocks_before(shape, rb, nck) + c - chunk_lo(shape, rb)) * (BM * BK);
}
inline size_t op_bytes(int shape, int rows, int K) { return op_off(shape, K / BK, rows / TB, chunk_lo(shape, rows / TB)); }
// lower residue block (ti, tj) of the symmetric mode: the same bytes as the operand blocks of row block ti of U
__host__ __device__ inline size_t res_off(int ti, int tj) { return ((size_t)ti * (ti + 1) / 2 + tj) * (size_t)(TB * TB); }
// U U^T at n_pad = 128 nb: one slot per modulus plus one
inline size_t plane_bytes(int nb) { return (size_t)(NMOD + 1) * op_bytes(UPPER, nb * TB, nb * TB); }

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
// Split: row maxima, then residue planes + row exponents of one operand.  X(i,k) = X[i + k*ld] off the diagonal
// 128-blocks, or everywhere when dense; diagonal tile rb from D when triangular (the operands dgemm_nt reads for the
// DMMA product).  CTA = (column block cb, row block rb) inside the operand's range, one thread per row: every k step
// reads 128 contiguous doubles.
// ---------------------------------------------------------------------------------------------
struct OzOperand {
  const double* X;
  long ld;
  const double* D;  // diagonal 128 x 128 tiles (triangular shapes)
  int shape;
  int nck;          // k chunks per row (K / BK)
};

__device__ __forceinline__ bool oz_in_range(const OzOperand& o, int rb, int cb) {
  return o.shape == oz::UPPER ? cb >= rb : o.shape == oz::LOWER ? cb <= rb : true;
}

__device__ __forceinline__ double oz_x(const OzOperand& o, int rb, int cb, int r, int kk) {
  return (o.shape != oz::DENSE && cb == rb) ? o.D[(size_t)rb * TB * TB + r + (size_t)kk * TB]
                                            : o.X[(size_t)rb * TB + r + (size_t)(cb * TB + kk) * o.ld];
}

__global__ void __launch_bounds__(128) oz_rowmax_kernel(const OzOperand o, unsigned long long* __restrict__ rowmax) {
  const int cb = blockIdx.x, rb = blockIdx.y, r = threadIdx.x;
  if (!oz_in_range(o, rb, cb)) return;
  double m = 0.0;
#pragma unroll 8
  for (int kk = 0; kk < TB; ++kk) m = fmax(m, fabs(oz_x(o, rb, cb, r, kk)));
  // non-negative doubles order like their bit patterns
  atomicMax(rowmax + rb * TB + r, (unsigned long long)__double_as_longlong(m));
}

// residues of modulus t at planes + (t + 1) * slot + base
__global__ void __launch_bounds__(128) oz_split_kernel(const OzOperand o,
                                                       const unsigned long long* __restrict__ rowmax, int b,
                                                       const __grid_constant__ oz::Tables T, int8_t* __restrict__ planes,
                                                       size_t slot, size_t base, int* __restrict__ ex) {
  using namespace oz;
  const int cb = blockIdx.x, rb = blockIdx.y, r = threadIdx.x;
  if (!oz_in_range(o, rb, cb)) return;
  const double m = __longlong_as_double((long long)rowmax[rb * TB + r]);
  int e = 0;
  if (m > 0.0) frexp(m, &e);  // m < 2^e
  if (cb * CPB == chunk_lo(o.shape, rb)) ex[rb * TB + r] = e;
  const double scale = ldexp(1.0, b - e);
#pragma unroll 1
  for (int q = 0; q < TB / 16; ++q) {  // 16 k values = one core-matrix row of every plane
    uint32_t w[NMOD][4];
#pragma unroll
    for (int t = 0; t < NMOD; ++t) w[t][0] = w[t][1] = w[t][2] = w[t][3] = 0u;
#pragma unroll
    for (int x16 = 0; x16 < 16; ++x16) {
      // |X| 2^(b-e) < 2^b exactly; its rint is an integer-valued double, converted exactly
      const long long a = __double2ll_rn(rint(oz_x(o, rb, cb, r, q * 16 + x16) * scale));
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
    const size_t off = base + op_off(o.shape, o.nck, rb, c) + in_blk;
#pragma unroll
    for (int t = 0; t < NMOD; ++t)
      *reinterpret_cast<uint4*>(planes + (size_t)(t + 1) * slot + off) = make_uint4(w[t][0], w[t][1], w[t][2], w[t][3]);
  }
}

// ---------------------------------------------------------------------------------------------
// Product of one modulus: one CTA per 128 x 256 tile (row block ti, column blocks jb0 = 2 tj2 and jb0 + 1 when it
// exists; in the symmetric mode only lower tiles, jb0 + 1 <= ti), k over the intersection of the ranges of its rows;
// tiles with the longest k range first.  Reads operand slot `slot + 1`, writes the residues of C'_t into slot `slot`.
// ---------------------------------------------------------------------------------------------
struct OzGeo {
  size_t slot;    // bytes per slot
  size_t b_base;  // offset of B's plane inside a slot (B = A in the symmetric mode)
  int a_shape, b_shape;
  int nck;        // k chunks
  int mb, nbn;    // 128-row blocks of A and of B
  int sym;
};

__host__ __device__ inline long oz_tiles(const OzGeo& g) {
  if (g.sym) return (long)(g.mb / 2) * (g.mb / 2 + 1) + (g.mb & 1) * (g.mb / 2 + 1);  // row block ti: ti / 2 + 1 tiles
  return (long)g.mb * ((g.nbn + 1) / 2);
}
__host__ __device__ inline size_t oz_out_off(const OzGeo& g, int ti, int tj) {
  return g.sym ? oz::res_off(ti, tj) : ((size_t)ti * g.nbn + tj) * (size_t)(TB * TB);
}

__global__ void __launch_bounds__(oz::THREADS, 2) oz_mod_kernel(int8_t* __restrict__ planes, const OzGeo g, int slot,
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
  if (g.sym) {
    // row blocks 2q and 2q + 1 hold q + 1 tiles each: q(q + 1) tiles precede row block 2q
    const long L = blockIdx.x;
    long q = (long)((sqrt(4.0 * (double)L + 1.0) - 1.0) * 0.5);
    while (q * (q + 1) > L) --q;
    while ((q + 1) * (q + 2) <= L) ++q;
    const long rem = L - q * (q + 1);
    ti = (int)(2 * q + rem / (q + 1));
    tj2 = (int)(rem % (q + 1));
  } else {
    const int nt2 = (g.nbn + 1) / 2, rq = (int)(blockIdx.x / nt2);
    ti = g.a_shape == LOWER ? g.mb - 1 - rq : rq;  // lower rows grow with ti, upper ones shrink
    tj2 = (int)(blockIdx.x % nt2);
  }
  const int jb0 = 2 * tj2;
  const bool has1 = g.sym ? jb0 + 1 <= ti : jb0 + 1 < g.nbn;  // the second column block exists (and is lower)
  const int jb1 = has1 ? jb0 + 1 : jb0;  // otherwise its half of the tile repeats the first and is not stored
  const int c_begin = max(chunk_lo(g.a_shape, ti), max(chunk_lo(g.b_shape, jb0), chunk_lo(g.b_shape, jb1)));
  const int c_end = min(chunk_hi(g.a_shape, ti, g.nck), min(chunk_hi(g.b_shape, jb0, g.nck), chunk_hi(g.b_shape, jb1, g.nck)));
  const int nchunks = c_end - c_begin;
  // a row block's chunks are contiguous: the producer only steps three pointers
  const int8_t* srcA = planes + (size_t)(slot + 1) * g.slot;
  const int8_t* pa = srcA + op_off(g.a_shape, g.nck, ti, c_begin);
  const int8_t* pb0 = srcA + g.b_base + op_off(g.b_shape, g.nck, jb0, c_begin);
  const int8_t* pb1 = srcA + g.b_base + op_off(g.b_shape, g.nck, jb1, c_begin);

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
        const size_t o = (size_t)it * A_BYTES;
        tma_bulk_g2s(st, pa + o, A_BYTES, &full[s]);
        tma_bulk_g2s(st + A_BYTES, pb0 + o, A_BYTES, &full[s]);
        tma_bulk_g2s(st + 2 * A_BYTES, pb1 + o, A_BYTES, &full[s]);
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
    int8_t* dst = planes + (size_t)slot * g.slot + (size_t)r * TB;
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
      uint4* o = reinterpret_cast<uint4*>(dst + oz_out_off(g, ti, jb0 + (jc >> 2)) + (jc & 3) * 32);
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

// Every entry of block (ti, tj) goes to P[(i0 + r) * ldp + j0 + c] (when P) and to Q[(j0 + c) * ldq + i0 + r] (when
// Q), both coalesced: symmetric mode P = C and Q = C off the diagonal (the mirror); dense mode Q = C (column-major
// M x N), P = Ct (its transpose).  neg: the entries are negated after the rounding, exactly.
__global__ void __launch_bounds__(256) oz_crt_kernel(const int8_t* __restrict__ planes, const OzGeo g,
                                                     const int* __restrict__ exA, const int* __restrict__ exB, int b,
                                                     const __grid_constant__ oz::Tables T, double* __restrict__ P,
                                                     long ldp, double* __restrict__ Q, long ldq, int neg) {
  using namespace oz;
  __shared__ double tile[32][TB + 1];
  int ti, tj;
  const long L = blockIdx.x;
  if (g.sym) {
    long t = (long)((sqrt(8.0 * (double)L + 1.0) - 1.0) * 0.5);
    while (t * (t + 1) / 2 > L) --t;
    while ((t + 1) * (t + 2) / 2 <= L) ++t;
    ti = (int)t;
    tj = (int)(L - t * (t + 1) / 2);
    if (ti == tj) Q = nullptr;
  } else {
    ti = (int)(L / g.nbn);
    tj = (int)(L % g.nbn);
  }
  const int8_t* blk = planes + oz_out_off(g, ti, tj);
  const int tid = threadIdx.x, rr = tid >> 3, c0 = (tid & 7) * 16;
  const int i0 = ti * TB, j0 = tj * TB;
#pragma unroll 1
  for (int r0 = 0; r0 < TB; r0 += 32) {
    const int r = r0 + rr;
    uint4 rv[NMOD];
#pragma unroll
    for (int t = 0; t < NMOD; ++t) rv[t] = *reinterpret_cast<const uint4*>(blk + t * g.slot + (size_t)r * TB + c0);
    const int ei = exA[i0 + r];
#pragma unroll 1
    for (int j = 0; j < 16; ++j) {
      int res[NMOD];
#pragma unroll
      for (int t = 0; t < NMOD; ++t) {
        const uint32_t wv = j < 4 ? rv[t].x : j < 8 ? rv[t].y : j < 12 ? rv[t].z : rv[t].w;
        res[t] = (int)(int8_t)(wv >> (8 * (j & 3)));
      }
      const double v = oz_crt(res, T, ei + exB[j0 + c0 + j] - 2 * b);
      tile[rr][c0 + j] = neg ? -v : v;
    }
    __syncthreads();
    if (P) {
#pragma unroll 4
      for (int k = tid; k < 32 * TB; k += 256) {
        const int a = k >> 7, c = k & (TB - 1);
        P[(size_t)(i0 + r0 + a) * ldp + j0 + c] = tile[a][c];
      }
    }
    if (Q) {
#pragma unroll 4
      for (int k = tid; k < 32 * TB; k += 256) {
        const int c = k >> 5, a = k & 31;
        Q[(size_t)(j0 + c) * ldq + i0 + r0 + a] = tile[a][c];
      }
    }
    __syncthreads();
  }
}

struct OzWork {
  int8_t* planes = nullptr;              // NMOD + 1 slots (oz::plane_bytes(n_pad / 128) in a fit)
  size_t plane_bytes = 0;
  unsigned long long* rowmax = nullptr;  // rows: one per row of A and of B
  int* ex = nullptr;                     // rows
  int rows = 0;
};

inline int configure_uut_i8_kernel() {
  ACE_CUDA(cudaFuncSetAttribute(oz_mod_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)oz::SMEM_BYTES));
  return 0;
}

// One product of the engine, in the spirit of GemmNT: C = sign A B^T, A M x K, B N x K, column-major.
struct OzNT {
  const double* A = nullptr;
  long lda = 0;
  const double* Adiag = nullptr;  // diagonal tiles of a triangular A (DU for upper, DX for lower)
  int a_shape = oz::DENSE;
  const double* B = nullptr;      // ignored in the symmetric mode (B = A)
  long ldb = 0;
  int M = 0, N = 0, K = 0;        // multiples of 128; a triangular A has M = K
  int sym = 0;                    // C = A A^T, A upper: lower tiles and their mirror into C (M = N = K)
  double* C = nullptr;
  long ldc = 0;
  double* Ct = nullptr;           // dense mode: optional transposed store Ct = C^T
  long ldct = 0;
  int neg = 0;                    // dense mode: C = -A B^T
};

inline OzGeo oz_geo(const OzNT& p) {
  using namespace oz;
  OzGeo g{};
  g.a_shape = p.a_shape; g.nck = p.K / BK; g.mb = p.M / TB; g.nbn = p.N / TB; g.sym = p.sym;
  g.b_shape = p.sym ? p.a_shape : DENSE;
  const size_t a_bytes = op_bytes(p.a_shape, p.M, p.K);
  g.b_base = p.sym ? 0 : a_bytes;
  const size_t out_bytes = p.sym ? oz::res_off(g.mb, 0) : (size_t)p.M * p.N;
  g.slot = std::max(g.b_base + (p.sym ? a_bytes : op_bytes(DENSE, p.N, p.K)), out_bytes);
  return g;
}
// workspace of one product: NMOD + 1 slots
inline size_t oz_plane_bytes(const OzNT& p) { return (size_t)(oz::NMOD + 1) * oz_geo(p).slot; }

inline int launch_oz_nt(const OzWork& o, const OzNT& p, cudaStream_t st) {
  using namespace oz;
  if (p.M <= 0 || p.N <= 0 || p.K <= 0 || p.M % TB || p.N % TB || p.K % TB || !p.A || !p.C ||
      (p.a_shape != DENSE && (p.M != p.K || !p.Adiag)) || (p.sym && (p.a_shape != UPPER || p.N != p.M || p.Ct || p.neg)) ||
      (!p.sym && !p.B)) {
    set_error("oz_nt: bad descriptor");
    return -2;
  }
  if (p.K > MAX_N) {
    set_error("oz_nt: K beyond the CRT range bound");
    return -2;
  }
  const OzGeo g = oz_geo(p);
  const int rows = p.sym ? p.M : p.M + p.N;
  if (!o.planes || !o.rowmax || !o.ex || o.plane_bytes < oz_plane_bytes(p) || o.rows < rows) {
    set_error("oz_nt: residue-plane workspace not allocated or too small");
    return -2;
  }
  static const Tables T = make_tables();
  const int b = crt_bits(p.K);
  ACE_CUDA(cudaMemsetAsync(o.rowmax, 0, sizeof(unsigned long long) * (size_t)rows, st));
  const OzOperand a{p.A, p.lda, p.Adiag, p.a_shape, g.nck};
  const dim3 ga(p.K / TB, p.M / TB);
  oz_rowmax_kernel<<<ga, TB, 0, st>>>(a, o.rowmax);
  ACE_CUDA(cudaGetLastError());
  oz_split_kernel<<<ga, TB, 0, st>>>(a, o.rowmax, b, T, o.planes, g.slot, 0, o.ex);
  ACE_CUDA(cudaGetLastError());
  if (!p.sym) {
    const OzOperand bo{p.B, p.ldb, nullptr, DENSE, g.nck};
    const dim3 gb(p.K / TB, p.N / TB);
    oz_rowmax_kernel<<<gb, TB, 0, st>>>(bo, o.rowmax + p.M);
    ACE_CUDA(cudaGetLastError());
    oz_split_kernel<<<gb, TB, 0, st>>>(bo, o.rowmax + p.M, b, T, o.planes, g.slot, g.b_base, o.ex + p.M);
    ACE_CUDA(cudaGetLastError());
  }
  const long tiles = oz_tiles(g);
  for (int t = 0; t < NMOD; ++t) {
    oz_mod_kernel<<<(unsigned)tiles, THREADS, SMEM_BYTES, st>>>(o.planes, g, t, MOD[t], 1.0 / MOD[t]);
    ACE_CUDA(cudaGetLastError());
  }
  const long blocks = p.sym ? (long)g.mb * (g.mb + 1) / 2 : (long)g.mb * g.nbn;
  const int* exB = p.sym ? o.ex : o.ex + p.M;
  if (p.sym)
    oz_crt_kernel<<<(unsigned)blocks, 256, 0, st>>>(o.planes, g, o.ex, exB, b, T, p.C, p.ldc, p.C, p.ldc, 0);
  else
    oz_crt_kernel<<<(unsigned)blocks, 256, 0, st>>>(o.planes, g, o.ex, exB, b, T, p.Ct, p.ldct, p.C, p.ldc, p.neg);
  ACE_CUDA(cudaGetLastError());
  return 0;
}

// C (ld = n_pad = nb * 128, both triangles) = U U^T from U = upper(A) with the diagonal tiles in DU
inline int launch_uut_i8(const OzWork& o, const double* A, const double* DU, int nb, double* C, cudaStream_t st) {
  OzNT p;
  p.A = A; p.lda = (long)nb * TB; p.Adiag = DU; p.a_shape = oz::UPPER; p.sym = 1;
  p.M = p.N = p.K = nb * TB;
  p.C = C; p.ldc = p.lda;
  return launch_oz_nt(o, p, st);
}

}  // namespace ace
