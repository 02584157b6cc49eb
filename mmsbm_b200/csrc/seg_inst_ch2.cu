// segment_pass_kernel instantiations with two 32-byte chunks per lane (rows of 33..64 doubles)
#include "segment_pass.cuh"
namespace mmsbm {
int launch_segment_pass_ch2(const SegArgs& a, int G, int UN, int MINB, dim3 grid, size_t smem, cudaStream_t st) {
  MMSBM_SEG_LAUNCH(5, 2, 1, 3) MMSBM_SEG_LAUNCH(6, 2, 1, 3) MMSBM_SEG_LAUNCH(7, 2, 1, 3) MMSBM_SEG_LAUNCH(8, 2, 1, 3)
  return MMSBM_ERANGE;
}
}  // namespace mmsbm
