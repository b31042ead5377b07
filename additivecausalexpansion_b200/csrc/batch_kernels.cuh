// batch_kernels.cuh -- the O(P) and O(n) steps of a batched fit (ace_fit_batch): the bodies of prep_tables_kernel,
// gemv2_kernel, alpha_kernel and finalize_kernel (gp_kernels.cuh) for S independent members in one launch.  Member q
// is blockIdx.z (gemv) or blockIdx.x (one CTA per member) and finds its arrays at the pointers of member 0 advanced
// by q times the strides of BatchLayout; a member with active[q] == 0 is frozen and left untouched.
#pragma once
#include "gp_kernels.cuh"

namespace ace {

// strides between members (elements); y: 0 when all members share one training set
struct BatchLayout {
  const int* active;  // nullptr: every member
  long y;             // y
  long vec;           // alpha, u, s, K alpha, diag(L) (n_pad)
  long chunks;        // gemv column-chunk partials (nchunks * n_pad)
  long mat;           // K^-1 (n_pad^2)
  long tab;           // derived tables
  long par;           // theta, m, v, grad (P)
  long sc;            // scalar slots (SC_COUNT)
  long part;          // gradient partials
  const double* std_y;  // per-member RMSE scale (moments of each member's own outcome)
};

__device__ __forceinline__ bool batch_active(const BatchLayout& L, long q) {
  return L.active == nullptr || L.active[q] != 0;
}

__global__ void batch_prep_tables_kernel(const double* __restrict__ theta, int p, int B, double* __restrict__ tab,
                                         const BatchLayout L) {
  const long q = blockIdx.x;
  if (!batch_active(L, q)) return;
  prep_tables_body(theta + q * L.par, p, B, tab + q * L.tab);
}

__global__ void __launch_bounds__(gv::ROWS) batch_gemv2_kernel(const double* __restrict__ Kinv, long ld, int n,
                                                               const double* __restrict__ y, double* __restrict__ pu,
                                                               double* __restrict__ ps, int n_pad, const BatchLayout L) {
  const long q = blockIdx.z;
  if (!batch_active(L, q)) return;
  gemv2_body(Kinv + q * L.mat, ld, n, y + q * L.y, pu + q * L.chunks, ps + q * L.chunks, n_pad);
}

__global__ void __launch_bounds__(1024) batch_alpha_kernel(const double* __restrict__ pu, const double* __restrict__ ps,
                                                           int nchunks, int n, int n_pad, double* __restrict__ theta,
                                                           double* __restrict__ uvec, double* __restrict__ svec,
                                                           double* __restrict__ alpha, double* __restrict__ Ka,
                                                           double* __restrict__ sc, int set_mu_first_iter,
                                                           const BatchLayout L) {
  const long q = blockIdx.x;
  if (!batch_active(L, q)) return;
  const long v = q * L.vec;
  alpha_body(pu + q * L.chunks, ps + q * L.chunks, nchunks, n, n_pad, theta + q * L.par, uvec + v, svec + v, alpha + v,
             Ka + v, sc + q * L.sc, set_mu_first_iter, nullptr, nullptr);
}

__global__ void __launch_bounds__(1024) batch_finalize_kernel(const FinalizeArgs a, const BatchLayout L) {
  const long q = blockIdx.x;
  if (!batch_active(L, q)) return;
  FinalizeArgs f = a;
  f.partials += q * L.part;
  f.y += q * L.y;
  f.alpha += q * L.vec;
  f.Ka += q * L.vec;
  f.dvec += q * L.vec;
  f.Kinv += q * L.mat;
  f.tab += q * L.tab;
  f.theta += q * L.par;
  f.m += q * L.par;
  f.v += q * L.par;
  f.grad += q * L.par;
  f.sc += q * L.sc;
  f.std_y = L.std_y[q];
  finalize_body(f);
}

// sc[SC_ITER] of every member (the iteration number para_update was called with)
__global__ void batch_set_iter_kernel(double* __restrict__ sc, long stride, int S, double iter) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q < S) sc[q * stride + SC_ITER] = iter;
}

}  // namespace ace
