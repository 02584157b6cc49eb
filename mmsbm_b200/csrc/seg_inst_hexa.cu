// segment_pass_kernel instantiations serving SIX runs per warp (5-lane groups: rows of 20 doubles)
#include "segment_pass.cuh"
namespace mmsbm {
int launch_segment_pass_hexa(const SegArgs& a, int G, int UN, int MINB, dim3 grid, size_t smem, cudaStream_t st) {
  MMSBM_SEG_LAUNCH_R(5, 1, 3, 3, 6)
  return MMSBM_ERANGE;
}
}  // namespace mmsbm
