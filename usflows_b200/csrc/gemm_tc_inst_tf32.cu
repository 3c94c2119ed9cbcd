// Instantiations of the CTA-pair tcgen05 contraction for the tf32 engine (own translation unit: parallel build).
#include "gemm_tc2.cuh"

namespace usf {
int launch_gemm_tc2_tf32(const usf_linear_args* a, const Epilogue& ep, cudaStream_t st, int bn) {
  return launch_gemm_tc2_terms<1, tc2::KIND_TF32>(a, ep, st, bn);
}
}  // namespace usf
