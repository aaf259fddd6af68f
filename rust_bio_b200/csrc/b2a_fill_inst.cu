// One (G, R) shape of the K1 fill kernel: compile with -DB2A_G=<G> -DB2A_R=<R>.
#include "b2a_fill_launch.h"

#ifndef B2A_G
#error "compile with -DB2A_G=... -DB2A_R=..."
#endif

namespace b2a {

namespace {

template <int FLAGS>
cudaError_t go(const FillParams& prm, uint32_t ntasks, int num_sms, cudaStream_t stream,
               int* grid_out, int dry) {
  auto kern = fill_kernel<B2A_G, B2A_R, FLAGS>;
  constexpr int FILL_WARPS = fill_warps_of(B2A_G, B2A_R);
  const uint32_t lut_bytes = (FLAGS & F_LUT) ? lut_smem_bytes(prm.sc.alpha) : 0u;
  const size_t smem = 64 + lut_bytes + (size_t)FILL_WARPS * prm.smem_seq_bytes;
  cudaError_t err =
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return err;
  int per_sm = 0;
  err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, FILL_WARPS * 32, smem);
  if (err != cudaSuccess) return err;
  if (per_sm < 1) return cudaErrorLaunchOutOfResources;
  if (dry) {  // no launch: how many warps of this kernel are resident on the whole GPU
    if (grid_out) *grid_out = num_sms * per_sm * FILL_WARPS;
    return cudaSuccess;
  }
  const uint32_t want = (ntasks + FILL_WARPS - 1) / FILL_WARPS;
  uint32_t grid = (uint32_t)(num_sms * per_sm);
  if (grid > want) grid = want;
  if (prm.task_limit) grid = (want + prm.task_limit - 1) / prm.task_limit;  // every warp retires after task_limit tasks
  if (grid < 1) grid = 1;
  if (grid_out) *grid_out = (int)grid;
  kern<<<grid, FILL_WARPS * 32, smem, stream>>>(prm);
  return cudaGetLastError();
}

}  // namespace

#define B2A_CAT2(a, b, c) a##b##_##c
#define B2A_CAT(a, b, c) B2A_CAT2(a, b, c)

cudaError_t B2A_CAT(launch_fill_, B2A_G, B2A_R)(int flags, const FillParams& prm, uint32_t ntasks,
                                                int num_sms, cudaStream_t stream, int* grid_out, int dry) {
  constexpr int ALL = F_TRACK_ROWS | F_TRACK_COLS | F_CLIPX;
  // every variant twice: with the traceback, and score-only (F_NOTB, b2a_score_batch)
#define B2A_CASE(F)                                                         \
  case (F): return go<(F)>(prm, ntasks, num_sms, stream, grid_out, dry);   \
  case (F) | F_NOTB: return go<(F) | F_NOTB>(prm, ntasks, num_sms, stream, grid_out, dry);
  switch (flags) {
    B2A_CASE(0)
    B2A_CASE(F_TRACK_ROWS)
    B2A_CASE(F_TRACK_ROWS | F_PACKTRK)
    B2A_CASE(ALL)
    B2A_CASE(ALL | F_PACKTRK)
    B2A_CASE(ALL | F_RELU)
    B2A_CASE(ALL | F_PACKTRK | F_RELU)
    B2A_CASE(F_LUT)
    B2A_CASE(F_LUT | F_TRACK_ROWS)
    B2A_CASE(F_LUT | F_TRACK_ROWS | F_PACKTRK)
    B2A_CASE(F_LUT | ALL)
    B2A_CASE(F_LUT | ALL | F_PACKTRK)
    B2A_CASE(F_LUT | ALL | F_RELU)
    B2A_CASE(F_LUT | ALL | F_PACKTRK | F_RELU)
    B2A_CASE(F_TRACK_ROWS | F_PACKREL)
    B2A_CASE(ALL | F_PACKREL)
    B2A_CASE(ALL | F_PACKREL | F_RELU)
    B2A_CASE(F_LUT | F_TRACK_ROWS | F_PACKREL)
    B2A_CASE(F_LUT | ALL | F_PACKREL)
    B2A_CASE(F_LUT | ALL | F_PACKREL | F_RELU)
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace b2a
