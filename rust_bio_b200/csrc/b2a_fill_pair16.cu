// Host entry point of the pair-packed K1 fill (b2a_fill_pair16.cuh), shape 1x16.
#include "b2a_fill_launch.h"
#include "b2a_fill_pair16.cuh"

namespace b2a {

namespace {

template <bool NOTB>
cudaError_t go(const FillParams& prm, int32_t bias, int num_sms, cudaStream_t stream, int* grid_out, int dry) {
  auto kern = fill_pair16_kernel<16, NOTB>;
  constexpr int WARPS = 4;
  const size_t smem = 64 + p16_lut_smem_bytes(prm.sc.alpha) + (size_t)WARPS * prm.smem_seq_bytes;
  cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return err;
  int per_sm = 0;
  err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WARPS * 32, smem);
  if (err != cudaSuccess) return err;
  if (per_sm < 1) return cudaErrorLaunchOutOfResources;
  if (dry) {
    if (grid_out) *grid_out = num_sms * per_sm * WARPS;
    return cudaSuccess;
  }
  const uint32_t ntasks = (prm.nblocks + 1) / 2;  // a task is a pair of blocks
  const uint32_t want = (ntasks + WARPS - 1) / WARPS;
  uint32_t grid = (uint32_t)(num_sms * per_sm);
  if (grid > want) grid = want;
  if (prm.task_limit) grid = (want + prm.task_limit - 1) / prm.task_limit;  // every warp retires after task_limit tasks
  if (grid < 1) grid = 1;
  if (grid_out) *grid_out = (int)grid;
  kern<<<grid, WARPS * 32, smem, stream>>>(prm, bias);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_fill_pair16(const FillParams& prm, int32_t bias, bool notb, int num_sms, cudaStream_t stream,
                               int* grid_out, int dry) {
  return notb ? go<true>(prm, bias, num_sms, stream, grid_out, dry) : go<false>(prm, bias, num_sms, stream, grid_out, dry);
}

}  // namespace b2a
