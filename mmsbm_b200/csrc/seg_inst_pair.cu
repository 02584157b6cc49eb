// segment_pass_kernel instantiations serving a PAIR of runs per warp (rows of up to 32 doubles)
#include "segment_pass.cuh"
namespace mmsbm {
int launch_segment_pass_pair(const SegArgs& a, int G, int UN, int MINB, dim3 grid, size_t smem, cudaStream_t st) {
  MMSBM_SEG_LAUNCH_R(1, 1, 2, 3, 2) MMSBM_SEG_LAUNCH_R(2, 1, 3, 3, 2) MMSBM_SEG_LAUNCH_R(3, 1, 3, 3, 2)
  MMSBM_SEG_LAUNCH_R(4, 1, 3, 3, 2) MMSBM_SEG_LAUNCH_R(5, 1, 3, 3, 2) MMSBM_SEG_LAUNCH_R(6, 1, 3, 3, 2)
  MMSBM_SEG_LAUNCH_R(7, 1, 3, 3, 2) MMSBM_SEG_LAUNCH_R(8, 1, 3, 3, 2)
  return MMSBM_ERANGE;
}
}  // namespace mmsbm
