// grad3_kernel.cuh -- third-generation fused trace-gradient pass (sm_100a), exact-shape instantiations.
//
// Same decomposition as grad2_kernel (one thread owns a pair for ALL additive terms; D^2_d and the distance sums in
// registers; the length-scale sums S[b][d] += t_b D^2_d on the FP64 tensor pipe through a warp-private stage), but
// the instruction stream is cut down to what the FP64 pipe must execute (ncu r02 of grad2 at C3: 2249 warp
// instructions per 32 pairs, 0.48 IPC, FP64 pipe 37 % busy, top stalls `wait` and `short_scoreboard`):
//   * the number of additive terms BX is a template parameter: the B+1 distance sums, the term loop and the scale
//     sums have exactly the size of the problem (grad2 pads B to a multiple of 8: 17 sums instead of 13 at C3) and
//     no uniform `b < B` branches are left in the loop body;
//   * exp / sqrt / reciprocal run in lock step over G terms (fastmath.cuh: fast_*_n), so the schedule has G
//     independent dependency chains where the scalar calls were issued back to back;
//   * the gradient's square roots and reciprocals skip the last rounding-cleanup step (<= 2 ulp instead of <= 1);
//   * CW = 1: the length-scale weights and lambda_b live in __constant__ memory (copied there from the device table
//     before the launch) and the distance loop is fully unrolled, so every weight is a c[3][imm] operand of its DFMA
//     -- the 7 LDS.128 per (pair, dimension) of the shared-memory version (ncu r02: the distance loop took 37 % of the
//     samples for 28 % of the FP64 work, stalled on short_scoreboard / mio_throttle) disappear.  One table per
//     module: launches that use it are serialised per device by the caller (ace_b200.cu: G3Chain).  CW = 0 keeps the
//     table in shared memory (no serialisation needed).
// Reference semantics: src/kernel_SE_cpp.cpp:161-243 (grad_SE_cpp), src/kernel_Matern_cpp.cpp:340-377,420-467.
#pragma once
#include "pair_common.cuh"

namespace ace {

// lambda_b and we[d][c] of the launch in flight (layout: pair_common.cuh G3_*); one copy per translation unit
static __constant__ double cG3[G3_SIZE];

namespace g3 {
constexpr int T = 64;      // tile edge
constexpr int LDS_ = 36;   // stage row stride (32 pairs + 4): conflict-free DMMA fragment loads
constexpr int ne(int BX, int kind) { return kind ? BX + 1 : BX; }     // distance sums per pair
constexpr int ws(int BX, int kind) { return (ne(BX, kind) + 1) / 2 * 2; }  // weight-row stride (16-byte loads)
constexpr int mt8(int BX) { return (BX + 7) / 8 * 8; }
inline size_t smem_bytes(int NT, int BX, int kind, int nwarps) {
  const int PD8 = 8 * NT, Bz = BX - 1;
  size_t d = (size_t)2 * PD8 * T + (size_t)(kind ? 2 : 4) * Bz * T + 2 * T + (size_t)PD8 * ws(BX, kind) + mt8(BX) +
             (size_t)nwarps * (mt8(BX) + PD8) * LDS_;
  return d * 8 + 16;
}
}  // namespace g3

// BX additive terms (exact), NT = ceil(p / 8) tiles of length-scale dimensions, G terms per lock-step group
template <int BX, int NT, int KIND, int NWARPS, int G, int CW>
__device__ __forceinline__ void grad3_body(const GradArgs& a) {
  static_assert(BX <= G3_LAM && g3::ne(BX, KIND) <= G3_WS && 8 * NT <= G3_PD, "shape exceeds the constant table");
  using namespace g3;
  constexpr int NTHR = NWARPS * 32;
  constexpr int JCOLS = 128 / NWARPS;  // columns of the 64 x 64 tile per warp
  constexpr int PD8 = 8 * NT, BD8 = mt8(BX), MT = BD8 / 8;
  constexpr int NE = ne(BX, KIND), WS = ws(BX, KIND), Bz = BX - 1;
  extern __shared__ __align__(128) unsigned char smraw[];
  const int p = a.p;
  const int p4 = (p + 3) / 4 * 4;  // <= PD8
  double* Xi = reinterpret_cast<double*>(smraw);
  double* Xj = Xi + PD8 * T;
  double* Zi = Xj + PD8 * T;
  double* Zj = Zi + Bz * T;
  double* LZi = Zj + Bz * T;                      // Matern: not staged (its terms do not read log|z|)
  double* LZj = LZi + (KIND ? 0 : Bz * T);
  double* ai = LZj + (KIND ? 0 : Bz * T);
  double* aj = ai + T;
  double* wt_s = aj + T;            // [PD8][WS] extended weight table rows (columns 0..NE-1)
  double* lam = wt_s + PD8 * WS;    // [BD8]
  double* stage = lam + BD8;        // [NWARPS][(BD8 + PD8)][LDS_]
  uint64_t* bar = reinterpret_cast<uint64_t*>(stage + NWARPS * (BD8 + PD8) * LDS_);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, tq = lane & 3;
  const int li = (warp & 1) * 32 + lane;   // row of the tile owned by this thread
  const int jbase = (warp >> 1) * JCOLS;   // this warp's columns of the tile
  double* Ts = stage + warp * (BD8 + PD8) * LDS_;  // [BD8][LDS_]  t_b of the warp's 32 pairs
  double* Ds = Ts + BD8 * LDS_;                    // [PD8][LDS_]  D^2_d of the warp's 32 pairs

  for (int idx = threadIdx.x; idx < PD8 * WS; idx += NTHR) {
    const int d = idx / WS, c = idx % WS;
    wt_s[idx] = (d < p && c < NE) ? a.tab[TAB_WE + d * WSTRIDE + c] : 0.0;
  }
  for (int b = threadIdx.x; b < BD8; b += NTHR) lam[b] = (b < BX) ? a.tab[TAB_LAM + b] : 0.0;
  for (int idx = threadIdx.x; idx < (PD8 - p) * T; idx += NTHR) {  // padded d rows stay zero (TMA never writes them)
    Xi[p * T + idx] = 0.0;
    Xj[p * T + idx] = 0.0;
  }
  for (int idx = threadIdx.x; idx < NWARPS * (BD8 + PD8) * LDS_; idx += NTHR) stage[idx] = 0.0;  // rows b >= BX, d >= p4
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  __syncthreads();

  double acc[MT][NT][2];   // S[b = 8 mt + g][d = 8 nt + 2 tq + e], summed over this warp's pairs
  double Sb[BX];           // sum W k_b over this thread's pairs
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
#pragma unroll
  for (int b = 0; b < BX; ++b) Sb[b] = 0.0;

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
      if (lane == 0) mbar_arrive_expect_tx(bar, (uint32_t)((2 * p + (KIND ? 2 : 4) * Bz + 2) * T * 8));
      __syncwarp();
      for (int c = lane; c < p; c += 32) {
        tma_bulk_g2s(Xi + c * T, a.X + i0 + (size_t)c * a.ldx, T * 8, bar);
        tma_bulk_g2s(Xj + c * T, a.X + j0 + (size_t)c * a.ldx, T * 8, bar);
      }
      for (int c = lane; c < Bz; c += 32) {
        tma_bulk_g2s(Zi + c * T, a.Z + i0 + (size_t)c * a.ldx, T * 8, bar);
        tma_bulk_g2s(Zj + c * T, a.Z + j0 + (size_t)c * a.ldx, T * 8, bar);
        if (KIND == 0) {
          tma_bulk_g2s(LZi + c * T, a.LZ + i0 + (size_t)c * a.ldx, T * 8, bar);
          tma_bulk_g2s(LZj + c * T, a.LZ + j0 + (size_t)c * a.ldx, T * 8, bar);
        }
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
    const double* kcol = a.Kinv + gi + (size_t)(j0 + jbase) * a.ld;
    double rowacc = 0.0;
    double knext = kcol[0];
#pragma unroll 1
    for (int jc = 0; jc < JCOLS; ++jc) {
      const int jj = jbase + jc;
      const int gj = j0 + jj;
      const double kinv = knext;
      if (jc + 1 < JCOLS) knext = kcol[(size_t)(jc + 1) * a.ld];
      const double alpha_j = aj[jj];
      const bool valid = (gi < a.n) && (gj < a.n);
      const double W = valid ? wt * (kinv - alpha_i * alpha_j) : 0.0;

      // ---- phase 1: D^2_d -> stage, distance sums E_c = sum_d we[d][c] D^2_d ------------------------
      double E[NE];
#pragma unroll
      for (int c = 0; c < NE; ++c) E[c] = 0.0;
      if (CW) {
        const double* xi = Xi + li;
        const double* xj = Xj + jj;
        double* ds = Ds + lane;
#pragma unroll
        for (int d0 = 0; d0 < PD8; d0 += 4) {
          if (d0 >= p4) break;  // uniform
#pragma unroll
          for (int dd = 0; dd < 4; ++dd) {
            const int d = d0 + dd;
            const double df = xi[d * T] - xj[d * T];
            const double d2 = df * df;
            ds[d * LDS_] = d2;
#pragma unroll
            for (int c = 0; c < NE; ++c) E[c] = fma(d2, cG3[G3_LAM + d * G3_WS + c], E[c]);
          }
        }
      } else {
        const double* xi = Xi + li;
        const double* xj = Xj + jj;
        double* ds = Ds + lane;
        const double* wr = wt_s;
#pragma unroll 1
        for (int d0 = 0; d0 < p4; d0 += 4) {
#pragma unroll
          for (int dd = 0; dd < 4; ++dd) {
            const double df = xi[dd * T] - xj[dd * T];
            const double d2 = df * df;
            ds[dd * LDS_] = d2;
#pragma unroll
            for (int c = 0; c < NE; c += 2) {
              const double2 wv = *reinterpret_cast<const double2*>(wr + dd * WS + c);
              E[c] = fma(d2, wv.x, E[c]);
              if (c + 1 < NE) E[c + 1] = fma(d2, wv.y, E[c + 1]);
            }
          }
          xi += 4 * T;
          xj += 4 * T;
          ds += 4 * LDS_;
          wr += 4 * WS;
        }
      }
      if (KIND) {  // r_c = sqrt(E_c), in lock-step chunks
        constexpr int CH = (NE % 5 == 0 || NE % 5 >= 3) ? 5 : 4;
#pragma unroll
        for (int c0 = 0; c0 < NE; c0 += CH) {
          if (c0 + CH <= NE) {
            double v[CH];
#pragma unroll
            for (int k = 0; k < CH; ++k) v[k] = E[c0 + k];
            fast_sqrt_n<CH, false>(v);
#pragma unroll
            for (int k = 0; k < CH; ++k) E[c0 + k] = v[k];
          } else {
            constexpr int R = NE % CH == 0 ? 1 : NE % CH;
            double v[R];
#pragma unroll
            for (int k = 0; k < R; ++k) v[k] = E[c0 + k];
            fast_sqrt_n<R, false>(v);
#pragma unroll
            for (int k = 0; k < R; ++k) E[c0 + k] = v[k];
          }
        }
      }
      // ---- phase 2: the BX terms, G at a time in lock step -------------------------------------------
      double kpart = 0.0;
#pragma unroll
      for (int b0 = 0; b0 < BX; b0 += G) {
        double ex[G], zz[G], den[G];
        bool live[G];
#pragma unroll
        for (int k = 0; k < G; ++k) {
          const int b = (b0 + k < BX) ? b0 + k : BX - 1;  // the tail group repeats the last term (results unused)
          double zi = 1.0, zj = 1.0;
          if (b > 0) {
            zi = Zi[(b - 1) * T + li];
            zj = Zj[(b - 1) * T + jj];
          }
          if (KIND == 0) {
            // sign(z_first) sign(z_second) exp(lambda - D + log|z_first| + log|z_second|), first = column point
            // (the smaller index of a lower-triangle pair; src/kernel_SE_cpp.cpp:103-119)
            double arg = (CW ? cG3[b] : lam[b]) - E[b];
            if (b > 0) arg = arg + LZj[(b - 1) * T + jj] + LZi[(b - 1) * T + li];
            ex[k] = arg;
            live[k] = (b == 0) || !(zj == 0.0 || zi == 0.0);
            zz[k] = (b == 0) ? 1.0 : sgn(zj) * sgn(zi);
          } else {
            // (1 + sqrt3 r) exp(lambda - sqrt3 r) z_first z_second (src/kernel_Matern_cpp.cpp:217,227)
            const double sr = SQRT3 * E[b];
            ex[k] = (CW ? cG3[b] : lam[b]) - sr;
            den[k] = 1.0 + sr;
            zz[k] = zj;
            live[k] = true;
            if (b > 0) zz[k] = zj * zi;  // grouping (base z_first) z_second = base (z_first z_second) up to rounding
            else zz[k] = 1.0;
          }
        }
        fast_exp_n<G>(ex);
        double tv[G];
#pragma unroll
        for (int k = 0; k < G; ++k) {
          double kv;
          if (KIND == 0) kv = live[k] ? zz[k] * ex[k] : 0.0;
          else kv = (den[k] * ex[k]) * zz[k];
          if (b0 + k < BX) kpart += kv;
          tv[k] = W * kv;
          if (b0 + k < BX) Sb[b0 + k] += tv[k];
        }
        if (KIND) {
          // dK_b/dL as the reference writes it: K_b / (1 + sqrt(3 D_grad)), D_grad = the NEXT column of the extended
          // table (src/kernel_Matern_cpp.cpp:362-364; quirk Q2)
#pragma unroll
          for (int k = 0; k < G; ++k) {
            const int b = (b0 + k < BX) ? b0 + k : BX - 1;
            den[k] = fma(SQRT3, E[b + 1], 1.0);
          }
          fast_rcp_n<G>(den);
#pragma unroll
          for (int k = 0; k < G; ++k) tv[k] *= den[k];
        }
#pragma unroll
        for (int k = 0; k < G; ++k)
          if (b0 + k < BX) Ts[(b0 + k) * LDS_ + lane] = tv[k];
      }
      rowacc = fma(kpart, alpha_j, rowacc);
      if (!diag_tile) {
        const double cpart = warp_sum(kpart * alpha_i);
        if (lane == 0) atomicAdd(a.Ka + gj, cpart);
      }
      __syncwarp();
      // ---- phase 3: S[b][d] += sum over the warp's 32 pairs of t_b * D^2_d  (FP64 tensor pipe) -------
#pragma unroll
      for (int s = 0; s < 8; ++s) {
        double af[MT], bf[NT];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) af[mt] = Ts[(8 * mt + g) * LDS_ + 4 * s + tq];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) bf[nt] = Ds[(8 * nt + g) * LDS_ + 4 * s + tq];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
          for (int nt = 0; nt < NT; ++nt) dmma884(acc[mt][nt][0], acc[mt][nt][1], af[mt], bf[nt]);
      }
      __syncwarp();
    }
    atomicAdd(a.Ka + gi, rowacc);
  }

  // ---- CTA reduction: per-warp fragments / lane sums -> smem -> one partial row per CTA -------------
  constexpr int NV = BD8 * PD8 + BD8;
  __syncthreads();           // everybody is done with the stage buffers; reuse them as red[NWARPS][NV]
  double* red = stage;       // NV = BD8 (PD8 + 1) <= (BD8 + PD8) * 36 for every shape
  static_assert(NV <= (BD8 + PD8) * LDS_, "reduction buffer does not fit the stage");
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) red[warp * NV + (8 * mt + g) * PD8 + 8 * nt + 2 * tq + e] = acc[mt][nt][e];
#pragma unroll
  for (int b = 0; b < BX; ++b) {
    const double v = warp_sum(Sb[b]);
    if (lane == 0) red[warp * NV + BD8 * PD8 + b] = v;
  }
  __syncthreads();
  double* out = a.partials + (size_t)blockIdx.x * a.P;
  for (int idx = threadIdx.x; idx < a.P; idx += NTHR) out[idx] = 0.0;
  __syncthreads();
  for (int r = threadIdx.x; r < NV; r += NTHR) {
    const bool is_len = r < BD8 * PD8;
    const int b = is_len ? r / PD8 : r - BD8 * PD8;
    const int d = is_len ? r % PD8 : 0;
    if (b >= BX || d >= p) continue;
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < NWARPS; ++w) v += red[w * NV + r];
    if (is_len) out[2 + BX + b + BX * d] = v;
    else out[2 + b] = v;
  }
}

template <int BX, int NT, int KIND, int NWARPS, int G, int CW>
__global__ void __launch_bounds__(NWARPS * 32, 1) grad3_kernel(const GradArgs a) {
  grad3_body<BX, NT, KIND, NWARPS, G, CW>(a);
}

// batched fit: member blockIdx.z; weights from shared memory (the constant table is one per module)
template <int BX, int NT, int KIND, int NWARPS, int G>
__global__ void __launch_bounds__(NWARPS * 32, 1) grad3_batch_kernel(const GradArgs a, const MemberStrides m) {
  if (!member_active(m)) return;
  grad3_body<BX, NT, KIND, NWARPS, G, 0>(member_args(a, m));
}

}  // namespace ace
