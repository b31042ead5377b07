// gp_kernels.cuh -- the O(n^2) kernels of the empirical-Bayes GP step (sm_100a):
//   prep_tables_kernel   theta -> exp(-L) tables, e^sigma                       (O(P))
//   logabs_kernel        log|Z| once per upload
//   (pair_kernels.cuh)   kernmat_kernel: fused additive kernel build; grad_kernel: fused trace-gradient pass
//   gemv2_kernel         u = K^-1 y, s = K^-1 1 in one pass over K^-1
//   alpha_kernel         mu closed form, alpha = u - mu s
//   finalize_kernel      assembles gradients/stats, clip, Nadam/Adam/Nesterov, mu refresh
//
// Reference semantics (paths relative to /root/reference), including its quirks (SURVEY.md 8a-Q):
//   build      src/kernel_SE_cpp.cpp:9-134, src/kernel_Matern_cpp.cpp:52-93,190-240
//              length-scale of (d, b) read at theta[1 + b + B*(d+1)]            (Q1)
//   gradient   src/kernel_SE_cpp.cpp:161-243, src/kernel_Matern_cpp.cpp:340-377,420-467,
//              src/include/ace_kernel_utils.hpp:23-36; length-scale at theta[2 + B + b + B*d];
//              Matern constant -0.25*9 and 1+sqrt(3*D_grad) denominator        (Q2)
//              evidence uses y'alpha                                           (Q3)
//   mu         src/utilities_cpp.cpp:6-10 (0.5 * sum(K^-1 y) / sum(K^-1))       (Q4)
//   clip/opt   src/utilities_cpp.cpp:121-129, src/optimizer_cpp.cpp:8-63       (Q5)
// The reference materialises the n x n x B cube; nothing here does (only the API-compat cube
// output of kernmat_kernel, on request).
#pragma once
#include "pair_common.cuh"

namespace ace {

// scalar-slot layout (doubles) in the device buffer `sc`
enum {
  SC_SUM_U = 0, SC_SUM_S, SC_MU_USED, SC_RMSE, SC_EVID, SC_GNORM, SC_FINITE, SC_ITER, SC_LOGDET,
  SC_YTALPHA, SC_SUM_ALPHA, SC_TRW, SC_RESID2, SC_COUNT
};

__device__ __forceinline__ void prep_tables_body(const double* __restrict__ theta, int p, int B, double* __restrict__ tab) {
  const int t = threadIdx.x;
  if (t == 0) tab[TAB_ESIG] = exp(theta[0]);
  for (int b = t; b < BMAXT; b += blockDim.x) tab[TAB_LAM + b] = (b < B) ? theta[2 + b] : 0.0;
  for (int idx = t; idx < PMAX * WSTRIDE; idx += blockDim.x) {
    const int d = idx / WSTRIDE, c = idx % WSTRIDE;
    double w = 0.0;
    // c = B at the last d would index one past the parameter vector only for the build (c <= B-1 there);
    // the gradient's c = b+1 <= B stays inside: 1 + B + B*d + B <= 1 + B + B*p = P - 1
    if (d < p && c <= B) w = exp(-theta[1 + B + B * d + c]);
    tab[TAB_WE + idx] = w;
  }
  for (int idx = t; idx < G3_SIZE; idx += blockDim.x) {  // compact block for the constant-memory gradient kernels
    double w = 0.0;
    if (idx < G3_LAM) {
      if (idx < B) w = theta[2 + idx];
    } else {
      const int d = (idx - G3_LAM) / G3_WS, c = (idx - G3_LAM) % G3_WS;
      if (d < p && c <= B) w = exp(-theta[1 + B + B * d + c]);
    }
    tab[TAB_G3 + idx] = w;
  }
  if (p > PMAX)
    for (int idx = t; idx < p * WSTRIDE; idx += blockDim.x) {
      const int d = idx / WSTRIDE, c = idx % WSTRIDE;
      tab[TAB_WIDE + idx] = (c <= B) ? exp(-theta[1 + B + B * d + c]) : 0.0;
    }
}

__global__ void prep_tables_kernel(const double* __restrict__ theta, int p, int B, double* __restrict__ tab) {
  prep_tables_body(theta, p, B, tab);
}

__global__ void logabs_kernel(const double* __restrict__ z, double* __restrict__ lz, size_t count) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) lz[i] = log(fabs(z[i]));
}

// ---------------------------------------------------------------------------------------------
// u = Kinv y, s = Kinv 1 (columns j < n only): partial sums per column chunk, deterministic.
// ---------------------------------------------------------------------------------------------
namespace gv {
constexpr int ROWS = 256, CHUNK = 512;
}

__device__ __forceinline__ void gemv2_body(const double* __restrict__ Kinv, long ld, int n, const double* __restrict__ y,
                                           double* __restrict__ pu, double* __restrict__ ps, int n_pad) {
  using namespace gv;
  __shared__ double ys[CHUNK];
  const int i = blockIdx.x * ROWS + threadIdx.x;
  const int c0 = blockIdx.y * CHUNK;
  for (int t = threadIdx.x; t < CHUNK; t += ROWS) {
    const int j = c0 + t;
    ys[t] = (j < n) ? y[j] : 0.0;
  }
  __syncthreads();
  const int cend = min(CHUNK, n - c0);  // columns of this chunk that are real data
  double u = 0.0, s = 0.0;
  if (i < n_pad) {
    const double* col = Kinv + i + (size_t)c0 * ld;
    int t = 0;
    for (; t + 8 <= cend; t += 8) {
      double k[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) k[e] = col[(size_t)(t + e) * ld];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        u = fma(k[e], ys[t + e], u);
        s += k[e];
      }
    }
    for (; t < cend; ++t) {
      const double k = col[(size_t)t * ld];
      u = fma(k, ys[t], u);
      s += k;
    }
    pu[(size_t)blockIdx.y * n_pad + i] = u;
    ps[(size_t)blockIdx.y * n_pad + i] = s;
  }
}

__global__ void __launch_bounds__(gv::ROWS) gemv2_kernel(const double* __restrict__ Kinv, long ld, int n,
                                                         const double* __restrict__ y, double* __restrict__ pu,
                                                         double* __restrict__ ps, int n_pad) {
  gemv2_body(Kinv, ld, n, y, pu, ps, n_pad);
}

__device__ __forceinline__ double block_sum_1024(double v, double* red) {
  // deterministic block reduction, blockDim.x <= 1024; red has 32 doubles; result broadcast to all
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  double r = (threadIdx.x < (blockDim.x + 31) / 32) ? red[threadIdx.x] : 0.0;
  if (w == 0) {
    r = warp_sum(r);
    if (l == 0) red[0] = r;
  }
  __syncthreads();
  return red[0];
}

// one CTA: gathers the gemv partials, mu closed form (first iteration only), alpha = u - mu*s
__device__ __forceinline__ void alpha_body(const double* __restrict__ pu, const double* __restrict__ ps, int nchunks,
                                           int n, int n_pad, double* __restrict__ theta, double* __restrict__ uvec,
                                           double* __restrict__ svec, double* __restrict__ alpha,
                                           double* __restrict__ Ka, double* __restrict__ sc, int set_mu_first_iter,
                                           const double* __restrict__ pd, double* __restrict__ kdiag) {
  __shared__ double red[32];
  double su = 0.0, ss = 0.0;
  for (int i = threadIdx.x; i < n_pad; i += blockDim.x) {
    double u = 0.0, s = 0.0, d = 0.0;
    if (i < n) {
      for (int c = 0; c < nchunks; ++c) {
        u += pu[(size_t)c * n_pad + i];
        s += ps[(size_t)c * n_pad + i];
      }
      if (pd != nullptr)
        for (int c = 0; c < nchunks; ++c) d += pd[(size_t)c * n_pad + i];
    }
    if (kdiag != nullptr) kdiag[i] = d;
    uvec[i] = u;
    svec[i] = s;
    su += u;
    ss += s;
  }
  su = block_sum_1024(su, red);
  ss = block_sum_1024(ss, red);
  // R/kernel_SE_R6.R:45 -- on the first iteration mu is replaced by its closed form BEFORE the gradient
  double mu = theta[1];
  if (set_mu_first_iter && sc[SC_ITER] == 1.0) mu = 0.5 * su / ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    theta[1] = mu;
    sc[SC_SUM_U] = su;
    sc[SC_SUM_S] = ss;
    sc[SC_MU_USED] = mu;
  }
  for (int i = threadIdx.x; i < n_pad; i += blockDim.x) {
    alpha[i] = (i < n) ? (uvec[i] - mu * svec[i]) : 0.0;
    Ka[i] = 0.0;
  }
}

__global__ void __launch_bounds__(1024) alpha_kernel(const double* __restrict__ pu, const double* __restrict__ ps,
                                                     int nchunks, int n, int n_pad, double* __restrict__ theta,
                                                     double* __restrict__ uvec, double* __restrict__ svec,
                                                     double* __restrict__ alpha, double* __restrict__ Ka,
                                                     double* __restrict__ sc, int set_mu_first_iter,
                                                     const double* __restrict__ pd = nullptr,
                                                     double* __restrict__ kdiag = nullptr) {
  alpha_body(pu, ps, nchunks, n, n_pad, theta, uvec, svec, alpha, Ka, sc, set_mu_first_iter, pd, kdiag);
}

// ---------------------------------------------------------------------------------------------
// One CTA: reduce partials, assemble gradient + statistics, clip, optimiser step, mu refresh.
// ---------------------------------------------------------------------------------------------
struct FinalizeArgs {
  const double* partials;
  int nparts;
  const double *y, *alpha, *Ka, *dvec, *Kinv;
  const double* kdiag;  // optional: diag(K^-1) as a vector (sharded inverse: no rank holds all diagonal tiles)
  long ld;
  const double* tab;
  double *theta, *m, *v, *grad, *sc;
  int n, p, B, P, kind;
  int optimizer;  // 0 Nadam, 1 Adam, 2 Nesterov
  double lr, beta1, beta2, eps, momentum, std_y, clip_at;
  int norm_clip;
  int do_update;  // 0: gradients + stats only (per-function API)
};

__device__ __forceinline__ void finalize_body(const FinalizeArgs& a) {
  __shared__ double red[32];
  const int n = a.n, B = a.B, P = a.P;
  const double mu = a.sc[SC_MU_USED];
  double s_alpha = 0, s_ya = 0, s_res = 0, s_logd = 0, s_trw = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double al = a.alpha[i];
    s_alpha += al;
    s_ya = fma(a.y[i], al, s_ya);
    const double r = (a.y[i] - mu) - a.Ka[i];
    s_res = fma(r, r, s_res);
    s_logd += log(a.dvec[i]);
    s_trw += ((a.kdiag != nullptr) ? a.kdiag[i] : a.Kinv[i + (size_t)i * a.ld]) - al * al;
  }
  s_alpha = block_sum_1024(s_alpha, red);
  s_ya = block_sum_1024(s_ya, red);
  s_res = block_sum_1024(s_res, red);
  s_logd = block_sum_1024(s_logd, red);
  s_trw = block_sum_1024(s_trw, red);

  // gradient assembly
  double gn2 = 0.0;
  int bad = 0;
  for (int k = threadIdx.x; k < P; k += blockDim.x) {
    double g;
    if (k == 0) {
      g = -0.5 * s_trw * a.tab[TAB_ESIG];  // sigma_gradient
    } else if (k == 1) {
      g = (a.kind == 0) ? s_alpha : 0.0;   // SE: sum(K^-1 ybar); Matern: forced 0
    } else {
      double s = 0.0;
      for (int c = 0; c < a.nparts; ++c) s += a.partials[(size_t)c * P + k];
      if (k < 2 + B) {
        g = -0.5 * s;
      } else {
        const int r = k - 2 - B, b = r % B, d = r / B;
        const double e = a.tab[tab_we(a.p) + d * WSTRIDE + b + 1];
        g = (a.kind == 0) ? (-0.5 * s) * e : -0.25 * 9 * s * e;
      }
    }
    a.grad[k] = g;
    gn2 = fma(g, g, gn2);
    if (!isfinite(g)) bad = 1;
  }
  gn2 = block_sum_1024(gn2, red);
  const double nbad = block_sum_1024((double)bad, red);
  double L2 = sqrt(gn2);
  // norm_clip_cpp: rescale to unit norm (Q5)
  const bool clip = a.norm_clip && (L2 > a.clip_at) && isfinite(L2) && (L2 != 0.0);
  const double iter = a.sc[SC_ITER];
  const double c1 = 1.0 - pow(a.beta1, iter), c2 = 1.0 - pow(a.beta2, iter);
  double gn2c = 0.0;
  for (int k = threadIdx.x; k < P; k += blockDim.x) {
    double g = a.grad[k];
    if (clip) g = g / L2;
    if (a.do_update) {
      a.grad[k] = g;
      double th = a.theta[k];
      if (a.optimizer == 2) {
        const double nu = a.momentum * a.m[k] + a.lr * g;
        a.m[k] = nu;
        th = th + nu;
      } else {
        const double mk = a.beta1 * a.m[k] + (1 - a.beta1) * g;
        const double vk = a.beta2 * a.v[k] + (1 - a.beta2) * (g * g);
        a.m[k] = mk;
        a.v[k] = vk;
        if (a.optimizer == 0)
          th = th + a.lr * ((a.beta1 * mk + (1 - a.beta1) * g) / c1) / (sqrt(vk / c2) + a.eps);
        else
          th = th + a.lr * (mk / c1) / (sqrt(vk / c2) + a.eps);
      }
      a.theta[k] = th;
    }
    gn2c = fma(g, g, gn2c);
  }
  gn2c = block_sum_1024(gn2c, red);
  __syncthreads();
  if (threadIdx.x == 0) {
    a.sc[SC_RMSE] = a.std_y * sqrt(s_res) / sqrt((double)n);
    a.sc[SC_LOGDET] = 2.0 * s_logd;
    a.sc[SC_YTALPHA] = s_ya;
    a.sc[SC_EVID] = -0.5 * ((double)n * log(2.0 * 3.14159265358979323846) + 2.0 * s_logd + s_ya);
    a.sc[SC_SUM_ALPHA] = s_alpha;
    a.sc[SC_TRW] = s_trw;
    a.sc[SC_RESID2] = s_res;
    a.sc[SC_GNORM] = a.do_update ? sqrt(gn2c) : L2;
    a.sc[SC_FINITE] = (nbad == 0.0) ? 1.0 : 0.0;
    if (a.do_update) {
      // mean_solution with the pre-update inverse (R/kernel_SE_R6.R:54, Q4/Q6)
      a.theta[1] = 0.5 * a.sc[SC_SUM_U] / a.sc[SC_SUM_S];
      a.sc[SC_ITER] = iter + 1.0;
    }
  }
}

__global__ void __launch_bounds__(1024) finalize_kernel(const FinalizeArgs a) { finalize_body(a); }

// multi-GPU: sum this rank's per-CTA partial rows into red[0..P) ahead of the all-reduce
__global__ void __launch_bounds__(1024) partials_reduce_kernel(const double* __restrict__ partials, int nparts, int P,
                                                               double* __restrict__ red, int accumulate = 0) {
  for (int k = threadIdx.x; k < P; k += blockDim.x) {
    double s = accumulate ? red[k] : 0.0;
    for (int c = 0; c < nparts; ++c) s += partials[(size_t)c * P + k];
    red[k] = s;
  }
}

// ---------------------------------------------------------------------------------------------
// Sharded inverse: K^-1 = U U^T exists only tile-wise across the ranks, but every rank holds U (upper(A),
// diagonal 128-blocks in the DU tiles).  u = K^-1 y and s = K^-1 1 are two triangular matrix-vector products
// with U, diag(K^-1)_i = sum_k U(i,k)^2 comes with the second one.  HBM bound: the upper triangle is read twice.
// ---------------------------------------------------------------------------------------------
// t_y[k] = sum_{i<=k} U(i,k) y_i, t_1[k] = sum_{i<=k, i<n} U(i,k): one warp per column
__global__ void __launch_bounds__(256) utv2_kernel(const double* __restrict__ A, long ld, const double* __restrict__ DU,
                                                   int n, int n_pad, const double* __restrict__ y,
                                                   double* __restrict__ ty, double* __restrict__ t1) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int k = blockIdx.x * 8 + warp;
  if (k >= n_pad) return;
  const int kb = k >> 7, kl = k & 127;
  double sy = 0.0, s1 = 0.0;
  const double* col = A + (size_t)k * ld;
  const int top = min(kb * 128, n);
  for (int i = lane; i < top; i += 32) {
    const double u = col[i];
    sy = fma(u, y[i], sy);
    s1 += u;
  }
  const double* dcol = DU + (size_t)kb * 16384 + (size_t)kl * 128;
  for (int il = lane; il <= kl; il += 32) {
    const int i = kb * 128 + il;
    if (i < n) {
      const double u = dcol[il];
      sy = fma(u, y[i], sy);
      s1 += u;
    }
  }
  sy = warp_sum(sy);
  s1 = warp_sum(s1);
  if (lane == 0) {
    ty[k] = sy;
    t1[k] = s1;
  }
}

// partial sums over the column chunk blockIdx.y of u_i = sum_{k>=i} U(i,k) t_y[k], s_i (with t_1), d_i = sum U(i,k)^2
__global__ void __launch_bounds__(gv::ROWS) uv2_kernel(const double* __restrict__ A, long ld,
                                                       const double* __restrict__ DU, int n_pad,
                                                       const double* __restrict__ ty, const double* __restrict__ t1,
                                                       double* __restrict__ pu, double* __restrict__ ps,
                                                       double* __restrict__ pd) {
  using namespace gv;
  __shared__ double tys[CHUNK], t1s[CHUNK];
  const int i = blockIdx.x * ROWS + threadIdx.x;
  const int c0 = blockIdx.y * CHUNK;
  const int cend = min(CHUNK, n_pad - c0);
  for (int t = threadIdx.x; t < CHUNK; t += ROWS) {
    tys[t] = (t < cend) ? ty[c0 + t] : 0.0;
    t1s[t] = (t < cend) ? t1[c0 + t] : 0.0;
  }
  __syncthreads();
  if (i >= n_pad) return;
  double u = 0.0, s = 0.0, d = 0.0;
  const int rb = i >> 7, il = i & 127;
  for (int t0 = 0; t0 < cend; t0 += 128) {
    const int cb = (c0 + t0) >> 7;
    if (cb < rb) continue;  // below the diagonal: zero
    const double* src;
    size_t stride;
    if (cb == rb) {
      src = DU + (size_t)rb * 16384 + il;
      stride = 128;
    } else {
      src = A + i + (size_t)(c0 + t0) * ld;
      stride = (size_t)ld;
    }
    for (int t = 0; t < 128; t += 8) {
      double k[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) k[e] = src[(size_t)(t + e) * stride];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        u = fma(k[e], tys[t0 + t + e], u);
        s = fma(k[e], t1s[t0 + t + e], s);
        d = fma(k[e], k[e], d);
      }
    }
  }
  pu[(size_t)blockIdx.y * n_pad + i] = u;
  ps[(size_t)blockIdx.y * n_pad + i] = s;
  pd[(size_t)blockIdx.y * n_pad + i] = d;
}

// statistics only (stats_cpp, src/stats_cpp.cpp:9-32): needs alpha = Kinv (y - mu) and K alpha
__global__ void __launch_bounds__(1024) stats_kernel(const double* __restrict__ y, const double* __restrict__ alpha,
                                                     const double* __restrict__ Ka, const double* __restrict__ dvec,
                                                     int n, double mu, double std_y, double* __restrict__ sc) {
  __shared__ double red[32];
  double s_ya = 0, s_res = 0, s_logd = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    s_ya = fma(y[i], alpha[i], s_ya);
    const double r = (y[i] - mu) - Ka[i];
    s_res = fma(r, r, s_res);
    s_logd += log(dvec[i]);
  }
  s_ya = block_sum_1024(s_ya, red);
  s_res = block_sum_1024(s_res, red);
  s_logd = block_sum_1024(s_logd, red);
  if (threadIdx.x == 0) {
    sc[SC_RMSE] = std_y * sqrt(s_res) / sqrt((double)n);
    sc[SC_EVID] = -0.5 * ((double)n * log(2.0 * 3.14159265358979323846) + 2.0 * s_logd + s_ya);
    sc[SC_LOGDET] = 2.0 * s_logd;
  }
}

}  // namespace ace
