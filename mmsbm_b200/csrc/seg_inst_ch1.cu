// segment_pass_kernel instantiations with one 32-byte chunk per lane (rows of up to 32 doubles)
#include "segment_pass.cuh"
namespace mmsbm {
int launch_segment_pass_ch1(const SegArgs& a, int G, int UN, int MINB, dim3 grid, size_t smem, cudaStream_t st) {
  MMSBM_SEG_LAUNCH(1, 1, 1, 3) MMSBM_SEG_LAUNCH(2, 1, 2, 3)
  MMSBM_SEG_LAUNCH(3, 1, 3, 3) MMSBM_SEG_LAUNCH(4, 1, 3, 3) MMSBM_SEG_LAUNCH(5, 1, 3, 3) MMSBM_SEG_LAUNCH(6, 1, 3, 3)
  MMSBM_SEG_LAUNCH(7, 1, 3, 3) MMSBM_SEG_LAUNCH(8, 1, 3, 3)
  return MMSBM_ERANGE;
}
}  // namespace mmsbm
