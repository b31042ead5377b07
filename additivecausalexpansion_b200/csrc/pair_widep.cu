// pair_widep.cu -- launchers of the p > PMAX kernel build and gradient pass (widep_kernels.cuh).  Own object so that
// it builds in parallel with the library proper.
#include "../../include/ace_b200.h"
#include "widep_kernels.cuh"

namespace ace {

int launch_kernmat_wide(const KernArgs& a, int kind, unsigned grid, cudaStream_t st) {
  const size_t smem = wp::kb_smem_bytes(a.B - 1);
  auto kern = kind == 0 ? kernmat_wide_kernel<0> : kernmat_wide_kernel<1>;
  ACE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, wp::NTHREADS, smem, st>>>(a);
  ACE_CUDA(cudaGetLastError());
  return 0;
}

// slab width: the widest of 16, 8, 4 columns whose stage fits one CTA's shared memory (0: none)
int grad_wide_slab(int B, int kind) {
  for (int sw : {16, 8, 4})
    if (wp::g_smem_bytes(sw, B, kind) <= 227 * 1024) return sw;
  return 0;
}

int launch_grad_wide(const GradArgs& a, int kind, int sw, int gx, cudaStream_t st) {
  const size_t smem = wp::g_smem_bytes(sw, a.B, kind);
  void (*kern)(const GradArgs);
  switch (kind * 100 + sw) {
    case 16: kern = grad_wide_kernel<0, 16>; break;
    case 8: kern = grad_wide_kernel<0, 8>; break;
    case 4: kern = grad_wide_kernel<0, 4>; break;
    case 116: kern = grad_wide_kernel<1, 16>; break;
    case 108: kern = grad_wide_kernel<1, 8>; break;
    case 104: kern = grad_wide_kernel<1, 4>; break;
    default: set_error("gradient pass (p > 64): no slab width fits shared memory"); return ACE_ERR_UNSUPPORTED;
  }
  ACE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<gx, wp::NTHREADS, smem, st>>>(a);
  ACE_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace ace
