// pair_kernels.cuh -- the two O(n^2 * B * p) kernels of the GP step (sm_100a):
//   kernmat_kernel   fused additive kernel build (SE / Matern-3/2; symmetric or rectangular)
//   grad_kernel      fused trace-gradient pass: reads K^-1 once, rebuilds k_b and D^2_d per pair
// Both stage X / Z / log|Z| tiles in shared memory with TMA bulk copies (cp.async.bulk, SASS UBLKCP) and
// are FP64-pipe / issue bound (arithmetic intensity B(3p+4)/16 flop/B >> the 5.7 flop/B ridge), so the
// design goal is few instructions per (pair, term) and enough independent work per thread.
//
// Reference semantics (paths relative to /root/reference), including its quirks (SURVEY.md 8a-Q):
//   build     src/kernel_SE_cpp.cpp:9-134, src/kernel_Matern_cpp.cpp:52-93,190-240
//   gradient  src/kernel_SE_cpp.cpp:161-243, src/kernel_Matern_cpp.cpp:340-377,420-467
// The reference materialises an n x n x B cube (two for Matern); nothing here does, except the optional
// API-compat cube output of kernmat_kernel.
#pragma once
#include "pair_common.cuh"
#include "gp_kernels.cuh"

namespace ace {

// ---------------------------------------------------------------------------------------------
// Fused kernel build.  64 x 64 pair tile per CTA; a thread owns one row and 16 columns, processed 4
// columns at a time; the additive terms are processed in chunks of 4 (rolled loop: small code, 16
// accumulators), each chunk re-deriving D^2_d from the staged X tiles.
// ---------------------------------------------------------------------------------------------
namespace kb {
constexpr int T = 64;        // tile edge
constexpr int LDT = T + 1;   // staging tile stride
// additive terms per chunk: every chunk re-derives D^2_d from the staged X tiles, so ONE chunk for B <= 12 (C3: B = 12,
// C2: B = 8) instead of three / two chunks of 4 saves 2 * (chunks - 1) FP64 instructions per pair and dimension
inline int chunk_terms(int B) { return B <= 4 ? 4 : (B <= 8 ? 8 : 12); }
inline int bpad(int B) {
  const int bc = chunk_terms(B);
  return (B + bc - 1) / bc * bc;
}
inline size_t smem_bytes(int p, int Bz, bool sym) {
  const int B = Bz + 1;
  size_t d = (size_t)(2 * p + 4 * Bz) * T + (size_t)p * bpad(B) + bpad(B) + (sym ? (size_t)T * LDT : 0);
  return d * 8 + 16;
}
}  // namespace kb

// BC additive terms per chunk, QC columns per step (BC * QC accumulators per thread)
template <int KIND, int BC, int QC>
__device__ __forceinline__ void kernmat_body(const KernArgs& a) {
  using namespace kb;
  extern __shared__ __align__(128) unsigned char smraw[];
  const int p = a.p, B = a.B, Bz = a.B - 1;
  const int BP = (B + BC - 1) / BC * BC;
  double* Xi = reinterpret_cast<double*>(smraw);
  double* Xj = Xi + p * T;
  double* Zi = Xj + p * T;
  double* Zj = Zi + Bz * T;
  double* LZi = Zj + Bz * T;
  double* LZj = LZi + Bz * T;
  double* wb = LZj + Bz * T;        // [p][BP]
  double* lam = wb + p * BP;        // [BP]
  double* Tt = lam + BP;            // [T][LDT] (sym only)
  uint64_t* bar = reinterpret_cast<uint64_t*>(Tt + (a.sym ? T * LDT : 0));

  int ti, tj;
  if (a.sym) {
    const long L = blockIdx.x;
    long t = (long)((sqrt(8.0 * (double)L + 1.0) - 1.0) * 0.5);
    while (t * (t + 1) / 2 > L) --t;
    while ((t + 1) * (t + 2) / 2 <= L) ++t;
    ti = (int)t;
    tj = (int)(L - t * (t + 1) / 2);
  } else {
    const int tm = a.n1_pad / T;
    ti = blockIdx.x % tm;
    tj = blockIdx.x / tm;
  }
  const int i0 = ti * T, j0 = tj * T;

  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    if (lane == 0) mbar_arrive_expect_tx(bar, (uint32_t)((2 * p + 4 * Bz) * T * 8));
    __syncwarp();
    for (int c = lane; c < p; c += 32) {
      tma_bulk_g2s(Xi + c * T, a.X1 + i0 + (size_t)c * a.ld1, T * 8, bar);
      tma_bulk_g2s(Xj + c * T, a.X2 + j0 + (size_t)c * a.ld2, T * 8, bar);
    }
    for (int c = lane; c < Bz; c += 32) {
      tma_bulk_g2s(Zi + c * T, a.Z1 + i0 + (size_t)c * a.ld1, T * 8, bar);
      tma_bulk_g2s(Zj + c * T, a.Z2 + j0 + (size_t)c * a.ld2, T * 8, bar);
      tma_bulk_g2s(LZi + c * T, a.LZ1 + i0 + (size_t)c * a.ld1, T * 8, bar);
      tma_bulk_g2s(LZj + c * T, a.LZ2 + j0 + (size_t)c * a.ld2, T * 8, bar);
    }
  }
  for (int idx = threadIdx.x; idx < p * BP; idx += 256) {
    const int d = idx / BP, b = idx % BP;
    wb[idx] = (b < B) ? a.tab[TAB_WE + d * WSTRIDE + b] : 0.0;  // build column of the extended table
  }
  if (threadIdx.x < BP) lam[threadIdx.x] = (threadIdx.x < B) ? a.tab[TAB_LAM + threadIdx.x] : 0.0;
  const double esig = a.tab[TAB_ESIG];
  __syncthreads();
  mbar_wait(bar, 0);

  const int li = threadIdx.x & 63, cg = threadIdx.x >> 6;
  const int gi = i0 + li;
#pragma unroll 1
  for (int step = 0; step < 16 / QC; ++step) {
    const int jj0 = cg * 16 + step * QC;
    double ksum[QC];
#pragma unroll
    for (int q = 0; q < QC; ++q) ksum[q] = 0.0;
#pragma unroll 1
    for (int b0 = 0; b0 < B; b0 += BC) {
      double acc[QC][BC];
#pragma unroll
      for (int q = 0; q < QC; ++q)
#pragma unroll
        for (int t = 0; t < BC; ++t) acc[q][t] = 0.0;
#pragma unroll 4
      for (int d = 0; d < p; ++d) {
        const double xi = Xi[d * T + li];
        double d2[QC];
#pragma unroll
        for (int q = 0; q < QC; q += 2) {
          const double2 xa = *reinterpret_cast<const double2*>(Xj + d * T + jj0 + q);
          d2[q] = (xi - xa.x) * (xi - xa.x);
          d2[q + 1] = (xi - xa.y) * (xi - xa.y);
        }
#pragma unroll
        for (int t = 0; t < BC; t += 2) {
          const double2 w = *reinterpret_cast<const double2*>(wb + d * BP + b0 + t);
#pragma unroll
          for (int q = 0; q < QC; ++q) {
            acc[q][t] = fma(d2[q], w.x, acc[q][t]);
            acc[q][t + 1] = fma(d2[q], w.y, acc[q][t + 1]);
          }
        }
      }
#pragma unroll
      for (int t = 0; t < BC; ++t) {
        const int b = b0 + t;
        if (b < B) {
          const double lb = lam[b];
          double zi = 1.0, lzi = 0.0;
          if (b > 0) {
            zi = Zi[(b - 1) * T + li];
            lzi = LZi[(b - 1) * T + li];
          }
#pragma unroll
          for (int q = 0; q < QC; ++q) {
            const int jj = jj0 + q, gj = j0 + jj;
            double zj = 1.0, lzj = 0.0;
            if (b > 0) {
              zj = Zj[(b - 1) * T + jj];
              lzj = LZj[(b - 1) * T + jj];
            }
            const double dv = KIND ? fast_sqrt(acc[q][t]) : acc[q][t];
            // symmetric build: the reference evaluates the r <= c half, so the smaller index (our column
            // point in a lower tile) comes first; rectangular build: row point first.
            const double kv = a.sym ? term_value<KIND>(b, lb, dv, zj, zi, lzj, lzi)
                                    : term_value<KIND>(b, lb, dv, zi, zj, lzi, lzj);
            if (!(a.skip0 && b == 0)) ksum[q] += kv;
            if (a.cube != nullptr && gi < a.n1 && gj < a.n2) {
              if (!a.sym) {
                a.cube[(size_t)b * a.cube_slice + gi + (size_t)gj * a.ldk] = kv;
              } else if (gi >= gj) {
                a.cube[(size_t)b * a.cube_slice + gi + (size_t)gj * a.ldk] = kv;
                a.cube[(size_t)b * a.cube_slice + gj + (size_t)gi * a.ldk] = kv;
              }
            }
          }
        }
      }
    }
#pragma unroll
    for (int q = 0; q < QC; ++q) {
      const int jj = jj0 + q, gj = j0 + jj;
      if (a.sym) {
        Tt[li * LDT + jj] = ksum[q];
      } else {
        double v = (gi < a.n1 && gj < a.n2) ? ksum[q] : 0.0;
        if (a.row_off + gi == a.col_off + gj) {
          if (gi < a.n1 && gj < a.n2) v += a.add_noise ? esig : 0.0;
          else if (a.pad_identity) v = 1.0;
        }
        a.K[gi + (size_t)gj * a.ldk] = v;
      }
    }
  }
  if (!a.sym) return;
  __syncthreads();
  const bool diag_tile = (ti == tj);
  // pass 1: K[i0+ii, j0+jj]  (ii fastest -> coalesced)
  for (int idx = threadIdx.x; idx < T * T; idx += 256) {
    const int ii = idx & 63, jj = idx >> 6;
    const int gr = i0 + ii, gc = j0 + jj;
    double v = (diag_tile && ii < jj) ? Tt[jj * LDT + ii] : Tt[ii * LDT + jj];
    if (gr >= a.n1 || gc >= a.n1) v = (a.pad_identity && gr == gc) ? 1.0 : 0.0;
    else if (a.add_noise && gr == gc) v += esig;
    a.K[gr + (size_t)gc * a.ldk] = v;
  }
  if (diag_tile) return;
  // pass 2: mirror K[j0+jj, i0+ii]  (jj fastest)
  for (int idx = threadIdx.x; idx < T * T; idx += 256) {
    const int jj = idx & 63, ii = idx >> 6;
    const int gr = j0 + jj, gc = i0 + ii;
    double v = Tt[ii * LDT + jj];
    if (gr >= a.n1 || gc >= a.n1) v = 0.0;
    a.K[gr + (size_t)gc * a.ldk] = v;
  }
}

template <int KIND, int BC, int QC>
__global__ void __launch_bounds__(256, 2) kernmat_kernel(const KernArgs a) {
  kernmat_body<KIND, BC, QC>(a);
}

// batched fit: member blockIdx.z
template <int KIND, int BC, int QC>
__global__ void __launch_bounds__(256, 2) kernmat_batch_kernel(const KernArgs a, const MemberStrides m) {
  if (!member_active(m)) return;
  kernmat_body<KIND, BC, QC>(member_args(a, m));
}

// ---------------------------------------------------------------------------------------------
// Fused trace-gradient pass.  Persistent CTAs stride over the lower 64x64 pair tiles; a thread owns one
// row of the tile and BT of the additive terms (its warp's b-group), and keeps the PD*BT length-scale
// sums + BT scale sums in registers across all tiles.  Per pair it reads K^-1(i,j) once and rebuilds
// D^2_d and k_b in registers.  For Matern the build distance of term b and the gradient distance of
// term b-1 are the same sum (extended table, gp_kernels.cuh), so a group needs BT+1 sums, not 2*BT.
// Two columns are processed per iteration for instruction-level parallelism when registers allow.
// Partial sums leave through warp shuffles -> smem -> one row of `partials` per CTA (no atomics).
// ---------------------------------------------------------------------------------------------
namespace gk {
constexpr int T = 64;
constexpr int GROUPS_PER_CTA = 4;
constexpr int nw(int BT, int kind) { return kind ? BT + 1 : BT; }
constexpr int wp(int BT, int kind) { return 2 * ((nw(BT, kind) + 1) / 2); }
inline size_t smem_bytes(int PD, int Bz, int BT, int kind) {
  size_t d = (size_t)2 * PD * T + (size_t)4 * Bz * T + 2 * T + (size_t)GROUPS_PER_CTA * PD * wp(BT, kind) + BMAXT +
             (size_t)8 * (PD * BT + BT);
  return d * 8 + 16;
}
}  // namespace gk

template <int PD, int BT, int KIND>
__device__ __forceinline__ void grad_body(const GradArgs& a) {
  using namespace gk;
  static_assert(BT <= 16, "BT too large");
  constexpr int NW = nw(BT, KIND);          // distance sums per thread
  constexpr int WP = wp(BT, KIND);          // padded to a multiple of 2 for 16-byte loads
  constexpr int Q = (PD * (BT + 2) <= 80 && BT <= 5) ? 2 : 1;  // columns per iteration (register budget)
  extern __shared__ __align__(128) unsigned char smraw[];
  const int p = a.p, B = a.B, Bz = a.B - 1;
  const int ngroups_cta = blockDim.x / 64;  // b-groups handled by this CTA (<= 4)
  double* Xi = reinterpret_cast<double*>(smraw);
  double* Xj = Xi + PD * T;
  double* Zi = Xj + PD * T;
  double* Zj = Zi + Bz * T;
  double* LZi = Zj + Bz * T;
  double* LZj = LZi + Bz * T;
  double* ai = LZj + Bz * T;  // alpha rows
  double* aj = ai + T;        // alpha cols
  double* wgrp = aj + T;      // [GROUPS_PER_CTA][PD][WP] weights packed per b-group
  double* lam = wgrp + GROUPS_PER_CTA * PD * WP;
  double* red = lam + BMAXT;  // [8 warps][PD*BT + BT]
  uint64_t* bar = reinterpret_cast<uint64_t*>(red + 8 * (PD * BT + BT));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pw = warp & 1;             // which half of the 64 rows
  const int gl = warp >> 1;            // local b-group
  const int bg = blockIdx.y * ngroups_cta + gl;     // global b-group
  const int b0 = bg * BT;
  const int li = pw * 32 + lane;

  for (int idx = threadIdx.x; idx < ngroups_cta * PD * WP; idx += blockDim.x) {
    const int g = idx / (PD * WP), r = idx % (PD * WP), d = r / WP, t = r % WP;
    const int c = (blockIdx.y * ngroups_cta + g) * BT + t;  // column of the extended table
    const bool ok = (t < NW) && (c <= B) && (d < p);
    wgrp[idx] = ok ? a.tab[TAB_WE + d * WSTRIDE + c] : 0.0;
  }
  for (int b = threadIdx.x; b < BMAXT; b += blockDim.x) lam[b] = a.tab[TAB_LAM + b];
  // zero the padded d rows of the X tiles once (TMA only ever writes rows d < p)
  for (int idx = threadIdx.x; idx < (PD - p) * T; idx += blockDim.x) {
    Xi[p * T + idx] = 0.0;
    Xj[p * T + idx] = 0.0;
  }
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  __syncthreads();

  double S[PD][BT];
  double Sb[BT];
#pragma unroll
  for (int d = 0; d < PD; ++d)
#pragma unroll
    for (int t = 0; t < BT; ++t) S[d][t] = 0.0;
#pragma unroll
  for (int t = 0; t < BT; ++t) Sb[t] = 0.0;

  const double* w_mine = wgrp + gl * PD * WP;
  const long nwork = grad_work_items(a);
  uint32_t phase = 0;
  for (long wk = blockIdx.x; wk < nwork; wk += gridDim.x) {
    int ti, tj;
    if (!grad_work_tile(a, wk, ti, tj)) continue;  // uniform over the CTA
    const int i0 = ti * T, j0 = tj * T;
    const bool diag_tile = (ti == tj);
    const double wt = diag_tile ? 1.0 : 2.0;

    __syncthreads();  // previous tile fully consumed before the TMA overwrites the staging tiles
    if (warp == 0) {
      if (lane == 0) mbar_arrive_expect_tx(bar, (uint32_t)((2 * p + 4 * Bz + 2) * T * 8));
      __syncwarp();
      for (int c = lane; c < p; c += 32) {
        tma_bulk_g2s(Xi + c * T, a.X + i0 + (size_t)c * a.ldx, T * 8, bar);
        tma_bulk_g2s(Xj + c * T, a.X + j0 + (size_t)c * a.ldx, T * 8, bar);
      }
      for (int c = lane; c < Bz; c += 32) {
        tma_bulk_g2s(Zi + c * T, a.Z + i0 + (size_t)c * a.ldx, T * 8, bar);
        tma_bulk_g2s(Zj + c * T, a.Z + j0 + (size_t)c * a.ldx, T * 8, bar);
        tma_bulk_g2s(LZi + c * T, a.LZ + i0 + (size_t)c * a.ldx, T * 8, bar);
        tma_bulk_g2s(LZj + c * T, a.LZ + j0 + (size_t)c * a.ldx, T * 8, bar);
      }
      if (lane == 0) {
        tma_bulk_g2s(ai, a.alpha + i0, T * 8, bar);
        tma_bulk_g2s(aj, a.alpha + j0, T * 8, bar);
      }
    }
    mbar_wait(bar, phase);
    phase ^= 1;

    const int gi = i0 + li;
    const double alpha_i = ai[li];
    const double* kcol = a.Kinv + gi + (size_t)j0 * a.ld;
    double rowacc = 0.0;
    double knext[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) knext[q] = kcol[(size_t)q * a.ld];
#pragma unroll 1
    for (int jj = 0; jj < T; jj += Q) {
      double kinv[Q];
#pragma unroll
      for (int q = 0; q < Q; ++q) kinv[q] = knext[q];
      if (jj + Q < T) {
#pragma unroll
        for (int q = 0; q < Q; ++q) knext[q] = kcol[(size_t)(jj + Q + q) * a.ld];
      }
      double d2[Q][PD];
      double E[Q][NW];
#pragma unroll
      for (int q = 0; q < Q; ++q)
#pragma unroll
        for (int t = 0; t < NW; ++t) E[q][t] = 0.0;
#pragma unroll
      for (int d = 0; d < PD; ++d) {
        const double xi = Xi[d * T + li];
        if (Q == 2) {
          const double2 xj = *reinterpret_cast<const double2*>(Xj + d * T + jj);
          const double f0 = xi - xj.x, f1 = xi - xj.y;
          d2[0][d] = f0 * f0;
          d2[Q - 1][d] = f1 * f1;
        } else {
          const double f0 = xi - Xj[d * T + jj];
          d2[0][d] = f0 * f0;
        }
        double w[WP];
#pragma unroll
        for (int t = 0; t < WP; t += 2) {
          const double2 v = *reinterpret_cast<const double2*>(w_mine + d * WP + t);
          w[t] = v.x;
          w[t + 1] = v.y;
        }
#pragma unroll
        for (int q = 0; q < Q; ++q)
#pragma unroll
          for (int t = 0; t < NW; ++t) E[q][t] = fma(d2[q][d], w[t], E[q][t]);
      }
      if (KIND) {
#pragma unroll
        for (int q = 0; q < Q; ++q)
#pragma unroll
          for (int t = 0; t < NW; ++t) E[q][t] = fast_sqrt(E[q][t]);
      }
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int gj = j0 + jj + q;
        const double alpha_j = aj[jj + q];
        const bool valid = (gi < a.n) && (gj < a.n);
        const double W = valid ? wt * (kinv[q] - alpha_i * alpha_j) : 0.0;
        double kpart = 0.0;
#pragma unroll
        for (int t = 0; t < BT; ++t) {
          const int b = b0 + t;
          if (b < B) {
            double zi = 1.0, zj = 1.0, lzi = 0.0, lzj = 0.0;
            if (b > 0) {
              zi = Zi[(b - 1) * T + li];
              zj = Zj[(b - 1) * T + jj + q];
              lzi = LZi[(b - 1) * T + li];
              lzj = LZj[(b - 1) * T + jj + q];
            }
            const double kv = term_value<KIND>(b, lam[b], E[q][t], zj, zi, lzj, lzi);
            kpart += kv;
            Sb[t] = fma(W, kv, Sb[t]);
            // SE: dK_b/dL = K_b * D2_d * exp(-L).  Matern as written in the reference:
            // K_b / (1 + sqrt(3 D_grad)) * D2_d * exp(-L), D_grad = sum with the GRADIENT's length-scales
            // = the next column of the extended table (sqrt(3 D) = sqrt3 * sqrt(D) up to rounding).
            double tv = W * kv;
            if (KIND) tv *= fast_rcp(1.0 + SQRT3 * E[q][t + (KIND ? 1 : 0)]);
#pragma unroll
            for (int d = 0; d < PD; ++d) S[d][t] = fma(tv, d2[q][d], S[d][t]);
          }
        }
        // K*alpha for the RMSE statistic (src/kernel_SE_cpp.cpp:238): row part in a register, column part
        // (mirror tile) reduced over the 32 rows of this warp
        rowacc = fma(kpart, alpha_j, rowacc);
        if (!diag_tile) {
          const double cpart = warp_sum(kpart * alpha_i);
          if (lane == 0) atomicAdd(a.Ka + gj, cpart);
        }
      }
    }
    atomicAdd(a.Ka + gi, rowacc);
  }

  // ---- CTA reduction: lanes -> warps -> one partial row per CTA -----------------------------
  constexpr int NV = PD * BT + BT;
  __syncthreads();
#pragma unroll
  for (int d = 0; d < PD; ++d)
#pragma unroll
    for (int t = 0; t < BT; ++t) {
      const double v = warp_sum(S[d][t]);
      if (lane == 0) red[warp * NV + d * BT + t] = v;
    }
#pragma unroll
  for (int t = 0; t < BT; ++t) {
    const double v = warp_sum(Sb[t]);
    if (lane == 0) red[warp * NV + PD * BT + t] = v;
  }
  __syncthreads();
  double* out = a.partials + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * a.P;
  for (int idx = threadIdx.x; idx < a.P; idx += blockDim.x) out[idx] = 0.0;
  __syncthreads();
  for (int idx = threadIdx.x; idx < ngroups_cta * NV; idx += blockDim.x) {
    const int g = idx / NV, r = idx % NV;
    const double v = red[(2 * g) * NV + r] + red[(2 * g + 1) * NV + r];
    const int gb0 = (blockIdx.y * ngroups_cta + g) * BT;
    if (r < PD * BT) {
      const int d = r / BT, b = gb0 + r % BT;
      if (d < p && b < B) out[2 + B + b + B * d] = v;
    } else {
      const int b = gb0 + (r - PD * BT);
      if (b < B) out[2 + b] = v;
    }
  }
}

template <int PD, int BT, int KIND>
__global__ void __launch_bounds__(256, 1) grad_kernel(const GradArgs a) {
  grad_body<PD, BT, KIND>(a);
}

// batched fit: member blockIdx.z (gridDim.y stays the b-groups)
template <int PD, int BT, int KIND>
__global__ void __launch_bounds__(256, 1) grad_batch_kernel(const GradArgs a, const MemberStrides m) {
  if (!member_active(m)) return;
  grad_body<PD, BT, KIND>(member_args(a, m));
}

}  // namespace ace
