// Host entry points of the K1 instantiations (one translation unit per (G, R)
// shape, see b2a_fill_inst.cu) so nvcc can build them in parallel.
#pragma once
#include <cuda_runtime.h>

#include "b2a_fill.cuh"

namespace b2a {

struct FillLaunch {
  int G, R;
  // launches the variant for `flags`; smem/grid are computed inside. Returns the grid used.
  // dry != 0: nothing is launched, *grid_out = the warps of this variant resident on the whole GPU.
  cudaError_t (*launch)(int flags, const FillParams& prm, uint32_t ntasks, int num_sms,
                        cudaStream_t stream, int* grid_out, int dry);
};

#define B2A_DECLARE_FILL(G, R)                                                                  \
  cudaError_t launch_fill_##G##_##R(int flags, const FillParams& prm, uint32_t ntasks,          \
                                    int num_sms, cudaStream_t stream, int* grid_out, int dry);

B2A_DECLARE_FILL(1, 16)
B2A_DECLARE_FILL(1, 8)
B2A_DECLARE_FILL(1, 20)
B2A_DECLARE_FILL(2, 16)
B2A_DECLARE_FILL(2, 20)
B2A_DECLARE_FILL(4, 16)
B2A_DECLARE_FILL(8, 16)
B2A_DECLARE_FILL(8, 20)
B2A_DECLARE_FILL(32, 8)
B2A_DECLARE_FILL(32, 16)

// the pair-packed 1x16 local fill (b2a_fill_pair16.cuh): two blocks per warp-task, int16x2 cells; notb: score-only
cudaError_t launch_fill_pair16(const FillParams& prm, int32_t bias, bool notb, int num_sms, cudaStream_t stream,
                               int* grid_out, int dry);

}  // namespace b2a
