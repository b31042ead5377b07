// pred_kernels.cuh -- small kernels around the posterior (src/pred_cpp.cpp) and the per-function API.
// The O(nx * n^2) product K_xX * K^-1 itself runs in dgemm_nt_kernel; these are the O(nx * n) rows
// and the O(nx^2) averages of pred_marginal_cpp.
#pragma once
#include "pair_kernels.cuh"

namespace ace {

namespace pk {
constexpr int ROWS = 256, CHUNK = 512;
}

// p1[c][i] = sum_{j in chunk c} T(i,j) (y_j - mu);  p2[c][i] = sum_j T(i,j) Kx(i,j)   (j < n)
__global__ void __launch_bounds__(pk::ROWS) rowdot2_kernel(const double* __restrict__ T, const double* __restrict__ Kx,
                                                           long ld, int nx_pad, int n, const double* __restrict__ y,
                                                           double mu, double* __restrict__ p1,
                                                           double* __restrict__ p2) {
  using namespace pk;
  __shared__ double yb[CHUNK];
  const int i = blockIdx.x * ROWS + threadIdx.x;
  const int c0 = blockIdx.y * CHUNK;
  const int cend = min(CHUNK, n - c0);
  for (int t = threadIdx.x; t < CHUNK; t += ROWS) yb[t] = (t < cend) ? (y[c0 + t] - mu) : 0.0;
  __syncthreads();
  if (i >= nx_pad) return;
  const double* tp = T + i + (size_t)c0 * ld;
  const double* kp = Kx + i + (size_t)c0 * ld;
  double s1 = 0.0, s2 = 0.0;
  int t = 0;
  for (; t + 4 <= cend; t += 4) {
    double a[4], b[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      a[e] = tp[(size_t)(t + e) * ld];
      b[e] = kp[(size_t)(t + e) * ld];
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      s1 = fma(a[e], yb[t + e], s1);
      s2 = fma(a[e], b[e], s2);
    }
  }
  for (; t < cend; ++t) {
    const double a = tp[(size_t)t * ld];
    s1 = fma(a, yb[t], s1);
    s2 = fma(a, kp[(size_t)t * ld], s2);
  }
  p1[(size_t)blockIdx.y * nx_pad + i] = s1;
  p2[(size_t)blockIdx.y * nx_pad + i] = s2;
}

// Factor form of the same rows, W = K_xX U with K^-1 = U U^T:  p1[c][i] = sum_j W(i,j) t_j with t = U^T (y - mu) given
// as ty - mu * t1;  p2[c][i] = sum_j W(i,j)^2  (= the row of T K_xX^T)
__global__ void __launch_bounds__(pk::ROWS) rowdot_tri_kernel(const double* __restrict__ W, long ld, int nx_pad, int n,
                                                              const double* __restrict__ ty,
                                                              const double* __restrict__ t1, double mu,
                                                              double* __restrict__ p1, double* __restrict__ p2) {
  using namespace pk;
  __shared__ double tb[CHUNK];
  const int i = blockIdx.x * ROWS + threadIdx.x;
  const int c0 = blockIdx.y * CHUNK;
  const int cend = min(CHUNK, n - c0);
  for (int t = threadIdx.x; t < CHUNK; t += ROWS) tb[t] = (t < cend) ? (ty[c0 + t] - mu * t1[c0 + t]) : 0.0;
  __syncthreads();
  if (i >= nx_pad) return;
  const double* wp = W + i + (size_t)c0 * ld;
  double s1 = 0.0, s2 = 0.0;
  int t = 0;
  for (; t + 8 <= cend; t += 8) {
    double a[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) a[e] = wp[(size_t)(t + e) * ld];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      s1 = fma(a[e], tb[t + e], s1);
      s2 = fma(a[e], a[e], s2);
    }
  }
  for (; t < cend; ++t) {
    const double a = wp[(size_t)t * ld];
    s1 = fma(a, tb[t], s1);
    s2 = fma(a, a, s2);
  }
  p1[(size_t)blockIdx.y * nx_pad + i] = s1;
  p2[(size_t)blockIdx.y * nx_pad + i] = s2;
}

// map_raw[i] = T (y - mu);  var_raw[i] = k(x_i,x_i) - T K_xX^T + noise
__global__ void post_finish_kernel(const double* __restrict__ p1, const double* __restrict__ p2, int chunks, int nx,
                                   int nx_pad, const double* __restrict__ kdiag, double noise,
                                   double* __restrict__ map, double* __restrict__ var) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nx_pad) return;
  double s1 = 0.0, s2 = 0.0;
  if (i < nx) {
    for (int c = 0; c < chunks; ++c) {
      s1 += p1[(size_t)c * nx_pad + i];
      s2 += p2[(size_t)c * nx_pad + i];
    }
    map[i] = s1;
    var[i] = kdiag[i] - s2 + noise;
  } else {
    map[i] = 0.0;
    var[i] = 0.0;
  }
}

// diagonal of the symmetric kernel of the new points: k(x,x) = sum_b term(b, D = 0)
__global__ void kdiag_kernel(const double* __restrict__ Z, const double* __restrict__ LZ, long ld, int nx, int B,
                             int kind, const double* __restrict__ tab, int skip0, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nx) return;
  double s = 0.0;
  for (int b = skip0 ? 1 : 0; b < B; ++b) {
    double z = 1.0, lz = 0.0;
    if (b > 0) {
      z = Z[i + (size_t)(b - 1) * ld];
      lz = LZ[i + (size_t)(b - 1) * ld];
    }
    const double lam = tab[TAB_LAM + b];
    s += (kind == 0) ? term_value<0>(b, lam, 0.0, z, z, lz, lz) : term_value<1>(b, lam, 0.0, z, z, lz, lz);  // D = r = 0
  }
  out[i] = s;
}

__global__ void diag_extract_kernel(const double* __restrict__ A, long ld, int n, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = A[i + (size_t)i * ld];
}

// out[i] = sum_c parts[c][i]
__global__ void reduce_partials_kernel(const double* __restrict__ parts, int chunks, int n, int n_pad,
                                       double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pad) return;
  double s = 0.0;
  if (i < n)
    for (int c = 0; c < chunks; ++c) s += parts[(size_t)c * n_pad + i];
  out[i] = s;
}

// sums the slices first..B-1 of a cube (ld x cols per slice) into out
__global__ void cube_sum_kernel(const double* __restrict__ cube, size_t slice, int first, int B, size_t count,
                                double* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  double s = cube[(size_t)first * slice + i];
  for (int b = first + 1; b < B; ++b) s += cube[(size_t)b * slice + i];
  out[i] = s;
}

// one CTA: q[0] = sum C, q[1] = z' C z, q[2] = u' C u with u = 1[z == 0]   (src/pred_cpp.cpp:89,98,107)
__global__ void __launch_bounds__(1024) quadforms_kernel(const double* __restrict__ C, long ld, int nx,
                                                         const double* __restrict__ z, double* __restrict__ q) {
  __shared__ double red[32];
  double s0 = 0.0, s1 = 0.0, s2 = 0.0;
  const size_t total = (size_t)nx * nx;
  for (size_t idx = threadIdx.x; idx < total; idx += blockDim.x) {
    const int i = (int)(idx % nx), j = (int)(idx / nx);
    const double c = C[i + (size_t)j * ld];
    const double zi = z[i], zj = z[j];
    s0 += c;
    s1 = fma(zi * zj, c, s1);
    s2 += (zi == 0.0 && zj == 0.0) ? c : 0.0;
  }
  s0 = block_sum_1024(s0, red);
  s1 = block_sum_1024(s1, red);
  s2 = block_sum_1024(s2, red);
  if (threadIdx.x == 0) {
    q[0] = s0;
    q[1] = s1;
    q[2] = s2;
  }
}

// one CTA per subset s (0/1 flags m = subsets + s * nx): q[3 s + 0] = m' C m, q[3 s + 1] = (m o z)' C (m o z),
// q[3 s + 2] = (m o 1[z == 0])' C (m o 1[z == 0]): the quadratic forms of src/pred_cpp.cpp:89,98,107 on the
// sub-block C[m, m] that a separate prediction on the subset would form
__global__ void __launch_bounds__(1024) quadforms_subset_kernel(const double* __restrict__ C, long ld, int nx,
                                                                const double* __restrict__ z,
                                                                const unsigned char* __restrict__ subsets,
                                                                double* __restrict__ q) {
  __shared__ double red[32];
  const unsigned char* m = subsets + (size_t)blockIdx.x * nx;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0;
  for (int j = 0; j < nx; ++j) {
    if (!m[j]) continue;  // uniform over the CTA
    const double zj = z[j];
    const double* col = C + (size_t)j * ld;
    for (int i = threadIdx.x; i < nx; i += blockDim.x) {
      if (!m[i]) continue;
      const double c = col[i], zi = z[i];
      s0 += c;
      s1 = fma(zi * zj, c, s1);
      s2 += (zi == 0.0 && zj == 0.0) ? c : 0.0;
    }
  }
  s0 = block_sum_1024(s0, red);
  s1 = block_sum_1024(s1, red);
  s2 = block_sum_1024(s2, red);
  if (threadIdx.x == 0) {
    q[3 * blockIdx.x + 0] = s0;
    q[3 * blockIdx.x + 1] = s1;
    q[3 * blockIdx.x + 2] = s2;
  }
}

namespace qf {
constexpr int THREADS = 256, COLS = 32;  // CTA size and columns of C per CTA
}

// The same quadratic forms on one rank's row block of C (a sharded posterior): C holds the rows lo .. lo + cnt - 1
// of the nx x nx covariance, all columns (column-major, ld).  Set q = 0 is every point, q = 1 + s is subset s of the
// nx x S flags.  CTA (q, slab) writes the partial sums over the set's rows in the block and its columns j in
// [slab * COLS, slab * COLS + COLS) ∩ [0, nx) to part[(slab * sets + q) * 3 + k], k = (1'C1, z'Cz, u'Cu), u = 1[z == 0].
// Set is the fast grid index, so the CTAs that read one slab run side by side and share its reads in L2.
__global__ void __launch_bounds__(qf::THREADS) quadforms_rows_kernel(const double* __restrict__ C, long ld, int lo,
                                                                     int cnt, int nx, const double* __restrict__ z,
                                                                     const unsigned char* __restrict__ subsets,
                                                                     double* __restrict__ part) {
  __shared__ double red[32];
  const int q = blockIdx.x, sets = gridDim.x;
  const unsigned char* m = (q > 0) ? subsets + (size_t)(q - 1) * nx : nullptr;
  const int j0 = blockIdx.y * qf::COLS, j1 = min(nx, j0 + qf::COLS);
  double s0 = 0.0, s1 = 0.0, s2 = 0.0;
  for (int j = j0; j < j1; ++j) {
    if (m && !m[j]) continue;  // uniform over the CTA
    const double zj = z[j];
    const double* col = C + (size_t)j * ld;
    for (int i = threadIdx.x; i < cnt; i += qf::THREADS) {
      if (m && !m[lo + i]) continue;
      const double c = col[i], zi = z[lo + i];
      s0 += c;
      s1 = fma(zi * zj, c, s1);
      s2 += (zi == 0.0 && zj == 0.0) ? c : 0.0;
    }
  }
  s0 = block_sum_1024(s0, red);
  s1 = block_sum_1024(s1, red);
  s2 = block_sum_1024(s2, red);
  if (threadIdx.x == 0) {
    double* out = part + ((size_t)blockIdx.y * sets + q) * 3;
    out[0] = s0;
    out[1] = s1;
    out[2] = s2;
  }
}

// second stage: out[t] = sum over the slabs, in slab order, of part[slab * n3 + t]  (n3 = 3 * sets)
__global__ void quadforms_rows_finish_kernel(const double* __restrict__ part, int slabs, int n3,
                                             double* __restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n3) return;
  double s = 0.0;
  for (int b = 0; b < slabs; ++b) s += part[(size_t)b * n3 + t];
  out[t] = s;
}

}  // namespace ace
