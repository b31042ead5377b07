// pair_common.cuh -- definitions shared by the pair kernels (kernel build, gradient passes) and by the
// translation units that hold them: table layout, one additive term for one pair, the gradient pass's
// arguments and its tile enumeration.  No __global__ functions here (the header is included by several TUs).
#pragma once
#include "fastmath.cuh"

namespace ace {

constexpr int PMAX = 64;   // max confounder columns supported by the fused kernels
constexpr int BMAXT = 32;  // max additive terms (B = Bz + 1)

// derived-table layout (doubles) in the device buffer `tab`
constexpr int TAB_ESIG = 0;                       // exp(theta[0])
constexpr int TAB_LAM = 8;                        // lambda_b            [BMAXT]
// Extended length-scale table we[d][c] = exp(-theta[1 + B + B*d + c]), c = 0..B  [PMAX][WSTRIDE].
// The kernel BUILD reads the length-scale of (d, b) at theta[1 + b + B*(d+1)] = we[d][b] (quirk Q1), the
// GRADIENT differentiates theta[2 + B + b + B*d] = we[d][b+1]: one table, shifted by one column.
constexpr int WSTRIDE = 36;
constexpr int TAB_WE = TAB_LAM + BMAXT;
// Compact copy for the constant-memory gradient kernels (grad3_kernel.cuh): lambda_b [G3_LAM] followed by
// we[d][c] as [G3_PD][G3_WS] -- one contiguous block, copied into __constant__ memory before the gradient launch.
constexpr int G3_LAM = 16, G3_PD = 32, G3_WS = 18;
constexpr int G3_SIZE = G3_LAM + G3_PD * G3_WS;
constexpr int TAB_G3 = TAB_WE + PMAX * WSTRIDE;
constexpr int TAB_SIZE = TAB_G3 + G3_SIZE;
// p > PMAX only: the extended table for all p dimensions, [p][WSTRIDE], appended after the fixed block (read from
// global memory by widep_kernels.cuh and by the gradient assembly)
constexpr int TAB_WIDE = TAB_SIZE;
inline size_t tab_doubles(int p) { return TAB_SIZE + (p > PMAX ? (size_t)p * WSTRIDE : 0); }
// where the gradient assembly finds we[d][c] for this p
__host__ __device__ __forceinline__ int tab_we(int p) { return p > PMAX ? TAB_WIDE : TAB_WE; }

__device__ __forceinline__ double sgn(double x) { return (double)((0.0 < x) - (x < 0.0)); }

constexpr double SQRT3 = 1.7320508075688772;

// One additive term for one pair.  `first`/`second` follow the reference's evaluation order:
// SE: sign * exp(lambda - D + log|z_first| + log|z_second|)      (src/kernel_SE_cpp.cpp:53,119)
// Matern: (1 + sqrt3 r) exp(lambda - sqrt3 r) * z_first * z_second (src/kernel_Matern_cpp.cpp:86,227)
// For Matern `r` = sqrt(D) is passed in (the gradient kernel shares the square roots between terms).
template <int KIND>
__device__ __forceinline__ double term_value(int b, double lam, double D_or_r, double z1, double z2, double lz1,
                                             double lz2) {
  if (KIND == 0) {
    if (b == 0) return fast_exp(lam - D_or_r);
    if (z1 == 0.0 || z2 == 0.0) return 0.0;
    return (sgn(z1) * sgn(z2)) * fast_exp(lam - D_or_r + lz1 + lz2);
  } else {
    const double sr = SQRT3 * D_or_r;
    const double base = (1.0 + sr) * fast_exp(lam - sr);
    if (b == 0) return base;
    return base * z1 * z2;  // exactly (+-)0 when a basis value is 0: base is finite, no test needed
  }
}

struct KernArgs {
  const double *X1, *Z1, *LZ1;  // row points    (n1, ld1)
  const double *X2, *Z2, *LZ2;  // column points (n2, ld2)
  long ld1, ld2;
  int n1, n2, n1_pad, n2_pad, p, B;
  const double* tab;
  double* K;        // n1_pad x n2_pad, ldk
  long ldk;
  double* cube;     // optional: B slices of (ldk x n2_pad)
  long cube_slice;
  int sym;          // 1: X1 == X2, lower tiles computed and mirrored, exactly symmetric output
  int add_noise;    // sym: K_ii += e^sigma for i < n
  int pad_identity; // sym: rows/cols >= n form an identity block
  int skip0;        // 1: leave the nuisance term b = 0 out of the sum (marginal kernels, src/pred_cpp.cpp:55-63)
  // rectangular blocks of the TRAINING kernel (multi-GPU column-block sharding): global index of the
  // block's first row / column, so that the noise diagonal and the identity padding land where they
  // belong.  Both 0 and add_noise = pad_identity = 0 for ordinary cross kernels.
  int row_off, col_off;
};

struct GradArgs {
  const double *X, *Z, *LZ;  // n_pad x p, n_pad x Bz (ld = ldx)
  long ldx;
  const double* Kinv;
  long ld;
  const double* alpha;
  double* Ka;        // K * alpha accumulated with atomics (RMSE statistic only)
  const double* tab;
  double* partials;  // [gridDim.y * gridDim.x][P]
  int n, p, B, P;
  int ntiles_side;   // ceil(n / 64)
  int tile_rank, tile_world;  // multi-GPU: this rank takes tiles L = tile_rank (mod tile_world); 0, 1 otherwise
  // tile_mode 1 (sharded inverse): ownership follows the 128 x 64 tiles of the sharded U U^T launch
  // (dgemm_nt lower_only order over gemm_rows = n_pad / 128 tile rows, tile L owned by rank L mod world), so
  // that a rank only reads the entries of K^-1 it has computed itself; each such tile holds two 64 x 64 tiles
  int tile_mode, gemm_rows;
};

// Batched fit (ace_fit_batch): member q = blockIdx.z of a batched launch finds its operands at every pointer advanced
// by q times the array's stride (elements; 0 = one copy shared by all members), and does nothing while active[q] == 0.
struct MemberStrides {
  const int* active;
  long x, z;    // X (X1 and X2 of a symmetric build), Z and LZ
  long tab;     // derived tables
  long mat;     // K (build) / K^-1 (gradient)
  long vec;     // alpha, K alpha
  long part;    // gradient partials
};

__device__ __forceinline__ bool member_active(const MemberStrides& m) {
  return m.active == nullptr || m.active[blockIdx.z] != 0;
}

__device__ __forceinline__ KernArgs member_args(KernArgs a, const MemberStrides& m) {
  const long q = blockIdx.z;
  a.X1 += q * m.x; a.X2 += q * m.x;
  a.Z1 += q * m.z; a.Z2 += q * m.z; a.LZ1 += q * m.z; a.LZ2 += q * m.z;
  a.tab += q * m.tab;
  a.K += q * m.mat;
  return a;
}

__device__ __forceinline__ GradArgs member_args(GradArgs a, const MemberStrides& m) {
  const long q = blockIdx.z;
  a.X += q * m.x; a.Z += q * m.z; a.LZ += q * m.z;
  a.tab += q * m.tab;
  a.Kinv += q * m.mat;
  a.alpha += q * m.vec; a.Ka += q * m.vec;
  a.partials += q * m.part;
  return a;
}

// work item w of this launch -> lower 64 x 64 tile (ti, tj); false: nothing to do for this item
__device__ __forceinline__ long grad_work_items(const GradArgs& a) {
  if (a.tile_mode == 0) {
    const long ntiles = (long)a.ntiles_side * (a.ntiles_side + 1) / 2;
    return (ntiles - a.tile_rank + a.tile_world - 1) / a.tile_world;
  }
  const long ng = (long)a.gemm_rows * (a.gemm_rows + 1);
  return 2 * ((ng - a.tile_rank + a.tile_world - 1) / a.tile_world);
}
__device__ __forceinline__ bool grad_work_tile(const GradArgs& a, long w, int& ti, int& tj) {
  if (a.tile_mode == 0) {
    const long L = w * a.tile_world + a.tile_rank;
    long tt = (long)((sqrt(8.0 * (double)L + 1.0) - 1.0) * 0.5);
    while (tt * (tt + 1) / 2 > L) --tt;
    while ((tt + 1) * (tt + 2) / 2 <= L) ++tt;
    ti = (int)tt;
    tj = (int)(L - tt * (tt + 1) / 2);
    return true;
  }
  const long L = (w >> 1) * a.tile_world + a.tile_rank;
  long t = (long)((sqrt(4.0 * (double)L + 1.0) - 1.0) * 0.5);
  while (t * (t + 1) > L) --t;
  while ((t + 1) * (t + 2) <= L) ++t;
  ti = 2 * (int)t + (int)(w & 1);
  tj = (int)(L - t * (t + 1));
  return tj <= ti && ti < a.ntiles_side;
}

}  // namespace ace
