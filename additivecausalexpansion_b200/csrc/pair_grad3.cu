// pair_grad3.cu -- instantiations of grad3_kernel (grad3_kernel.cuh) for one (kernel kind, p tile count) pair.
// Compiled once per -DG3_KIND={0,1} -DG3_NT={1,2,3,4} (see the Makefile) so that the 128 exact shapes
// (B = 1..16 additive terms each) build in parallel; each object exports one launcher.
#include "grad3_kernel.cuh"

#if !defined(G3_KIND) || !defined(G3_NT)
#error "compile with -DG3_KIND=<0|1> -DG3_NT=<1..4>"
#endif

namespace ace {

namespace g3 {
// terms per lock-step group: covers BX without (much) padding, 3..5 independent chains
constexpr int group(int BX) {
#if defined(G3_GRP)  // tuning experiments (Makefile EXTRA)
  if (BX >= G3_GRP) return G3_GRP;
#endif
  if (BX <= 5) return BX;
  int best = 4, waste = (BX + 3) / 4 * 4 - BX;
  const int cand[3] = {5, 3, 6};
  for (int i = 0; i < 3; ++i) {
    const int gg = cand[i], w = (BX + gg - 1) / gg * gg - BX;
    if (w < waste) { best = gg; waste = w; }
  }
  return best;
}
}  // namespace g3

template <int BX, int CW>
static int g3_launch(const GradArgs& a, int gx, size_t smem, cudaStream_t st) {
  constexpr int G = g3::group(BX);
  auto kern = grad3_kernel<BX, G3_NT, G3_KIND, 16, G, CW>;
  ACE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<gx, 512, smem, st>>>(a);
  ACE_CUDA(cudaGetLastError());
  return 0;
}

// cw = 1: the caller holds the per-device serialisation of the constant table (ace_b200.cu: G3Chain)
template <int BX>
static int g3_go(const GradArgs& a, int gx, size_t smem, int cw, cudaStream_t st) {
  if (!cw) return g3_launch<BX, 0>(a, gx, smem, st);
  ACE_CUDA(cudaMemcpyToSymbolAsync(cG3, a.tab + TAB_G3, sizeof(double) * G3_SIZE, 0, cudaMemcpyDeviceToDevice, st));
  return g3_launch<BX, 1>(a, gx, smem, st);
}

// batched fit: gx CTAs per member, members on gridDim.z
template <int BX>
static int g3_batch_go(const GradArgs& a, const MemberStrides& m, int gx, int S, size_t smem, cudaStream_t st) {
  constexpr int G = g3::group(BX);
  auto kern = grad3_batch_kernel<BX, G3_NT, G3_KIND, 16, G>;
  ACE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<dim3(gx, 1, S), 512, smem, st>>>(a, m);
  ACE_CUDA(cudaGetLastError());
  return 0;
}

#define G3_CAT2(a, b, c, d) a##b##c##d
#define G3_CAT(a, b, c, d) G3_CAT2(a, b, c, d)
int G3_CAT(launch_grad3_k, G3_KIND, _nt, G3_NT)(const GradArgs& a, int gx, size_t smem, int cw, cudaStream_t st) {
  switch (a.B) {
    case 1: return g3_go<1>(a, gx, smem, cw, st);
    case 2: return g3_go<2>(a, gx, smem, cw, st);
    case 3: return g3_go<3>(a, gx, smem, cw, st);
    case 4: return g3_go<4>(a, gx, smem, cw, st);
    case 5: return g3_go<5>(a, gx, smem, cw, st);
    case 6: return g3_go<6>(a, gx, smem, cw, st);
    case 7: return g3_go<7>(a, gx, smem, cw, st);
    case 8: return g3_go<8>(a, gx, smem, cw, st);
    case 9: return g3_go<9>(a, gx, smem, cw, st);
    case 10: return g3_go<10>(a, gx, smem, cw, st);
    case 11: return g3_go<11>(a, gx, smem, cw, st);
    case 12: return g3_go<12>(a, gx, smem, cw, st);
    case 13: return g3_go<13>(a, gx, smem, cw, st);
    case 14: return g3_go<14>(a, gx, smem, cw, st);
    case 15: return g3_go<15>(a, gx, smem, cw, st);
    case 16: return g3_go<16>(a, gx, smem, cw, st);
    default: set_error("grad3: B out of range"); return -1;
  }
}

int G3_CAT(launch_grad3_batch_k, G3_KIND, _nt, G3_NT)(const GradArgs& a, const MemberStrides& m, int gx, int S, size_t smem,
                                                   cudaStream_t st) {
  switch (a.B) {
    case 1: return g3_batch_go<1>(a, m, gx, S, smem, st);
    case 2: return g3_batch_go<2>(a, m, gx, S, smem, st);
    case 3: return g3_batch_go<3>(a, m, gx, S, smem, st);
    case 4: return g3_batch_go<4>(a, m, gx, S, smem, st);
    case 5: return g3_batch_go<5>(a, m, gx, S, smem, st);
    case 6: return g3_batch_go<6>(a, m, gx, S, smem, st);
    case 7: return g3_batch_go<7>(a, m, gx, S, smem, st);
    case 8: return g3_batch_go<8>(a, m, gx, S, smem, st);
    case 9: return g3_batch_go<9>(a, m, gx, S, smem, st);
    case 10: return g3_batch_go<10>(a, m, gx, S, smem, st);
    case 11: return g3_batch_go<11>(a, m, gx, S, smem, st);
    case 12: return g3_batch_go<12>(a, m, gx, S, smem, st);
    case 13: return g3_batch_go<13>(a, m, gx, S, smem, st);
    case 14: return g3_batch_go<14>(a, m, gx, S, smem, st);
    case 15: return g3_batch_go<15>(a, m, gx, S, smem, st);
    case 16: return g3_batch_go<16>(a, m, gx, S, smem, st);
    default: set_error("grad3: B out of range"); return -1;
  }
}

}  // namespace ace
