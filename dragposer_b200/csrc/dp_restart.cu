// dp_restart.cu -- per-clip restarts of a running batch (dp_engine_restart_clips) and the subset predictor of clips whose
// temporal phase differs from the rest of the batch.  None of this touches the frame kernels: a restarted clip's target rows
// are stored rotated by its phase offset, so the frame kernels keep reading slot `target_index` of every clip.
#include <cuda_runtime.h>

#include "dp_internal.h"

namespace {

constexpr int kRingCols = DP_L + DP_NH + 3;  // one ring row of every buffer: latent | heights | displacement

// One block per restarted clip: what dp_engine_init_clips writes for it -- latent, root position and rotation, and all DP_PAST ring
// rows (latent and heights tiled, displacement 0).  state rows: latent (24) | global_pos (3) | global_rot (4) | heights (6).
__global__ void dp_reset_clips_kernel(const int32_t* __restrict__ ids, const float* __restrict__ state, float* __restrict__ latent,
                                      float* __restrict__ gpos, float* __restrict__ grot, float* __restrict__ latent_buf,
                                      float* __restrict__ disp_buf, float* __restrict__ height_buf) {
  const int i = blockIdx.x;
  const size_t c = (size_t)ids[i];
  const float* s = state + (size_t)i * DP_RESTART_STATE;
  const int t = threadIdx.x;
  if (t < DP_L) latent[c * DP_L + t] = s[t];
  else if (t < DP_L + 3) gpos[c * 3 + t - DP_L] = s[t];
  else if (t < DP_L + 7) grot[c * 4 + t - DP_L - 3] = s[t];
  for (int k = t; k < DP_PAST * kRingCols; k += blockDim.x) {
    const int r = k / kRingCols, col = k % kRingCols;
    if (col < DP_L) latent_buf[(c * DP_PAST + r) * DP_L + col] = s[col];
    else if (col < DP_L + DP_NH) height_buf[(c * DP_PAST + r) * DP_NH + col - DP_L] = s[DP_L + 7 + col - DP_L];
    else disp_buf[(c * DP_PAST + r) * 3 + col - DP_L - DP_NH] = 0.0f;
  }
}

// One block per listed clip: its three ring buffers, slot for slot (the ring head stays the engine's), into compact (n, 60, .) rows.
__global__ void dp_gather_rings_kernel(const int32_t* __restrict__ ids, const float* __restrict__ latent_buf,
                                       const float* __restrict__ disp_buf, const float* __restrict__ height_buf,
                                       float* __restrict__ s_latent, float* __restrict__ s_disp, float* __restrict__ s_height) {
  const size_t i = blockIdx.x, c = (size_t)ids[blockIdx.x];
  for (int k = threadIdx.x; k < DP_PAST * kRingCols; k += blockDim.x) {
    const int r = k / kRingCols, col = k % kRingCols;
    if (col < DP_L) s_latent[(i * DP_PAST + r) * DP_L + col] = latent_buf[(c * DP_PAST + r) * DP_L + col];
    else if (col < DP_L + DP_NH) s_height[(i * DP_PAST + r) * DP_NH + col - DP_L] = height_buf[(c * DP_PAST + r) * DP_NH + col - DP_L];
    else s_disp[(i * DP_PAST + r) * 3 + col - DP_L - DP_NH] = disp_buf[(c * DP_PAST + r) * 3 + col - DP_L - DP_NH];
  }
}

// One block per listed clip: compact predictor rows (n, src_rows, 24) -> rows [r0, dst_rows) of the clip's target rows.
// src_rows == 1: the one row is broadcast.  Otherwise own row k < window lands in slot (k + shift) % window, own row `window` in
// slot `window`.
__global__ void dp_scatter_targets_kernel(const float* __restrict__ src, int src_rows, const int32_t* __restrict__ ids,
                                          float* __restrict__ dst, int dst_rows, int r0, int window, int shift) {
  const size_t i = blockIdx.x, c = (size_t)ids[blockIdx.x];
  for (int k = threadIdx.x; k < (dst_rows - r0) * DP_L; k += blockDim.x) {
    const int r = r0 + k / DP_L, f = k % DP_L;
    const int own = src_rows == 1 ? 0 : (r < window ? (r - shift + window) % window : r);
    dst[(c * dst_rows + r) * DP_L + f] = src[(i * src_rows + own) * DP_L + f];
  }
}

}  // namespace

cudaError_t dp_reset_clips_launch(const int32_t* ids, const float* state, int n, float* latent, float* gpos, float* grot,
                                  float* latent_buf, float* disp_buf, float* height_buf, cudaStream_t st) {
  dp_reset_clips_kernel<<<n, 128, 0, st>>>(ids, state, latent, gpos, grot, latent_buf, disp_buf, height_buf);
  return cudaGetLastError();
}

cudaError_t dp_gather_rings_launch(const int32_t* ids, int n, const float* latent_buf, const float* disp_buf, const float* height_buf,
                                   float* s_latent, float* s_disp, float* s_height, cudaStream_t st) {
  dp_gather_rings_kernel<<<n, 256, 0, st>>>(ids, latent_buf, disp_buf, height_buf, s_latent, s_disp, s_height);
  return cudaGetLastError();
}

cudaError_t dp_scatter_targets_launch(const float* src, int src_rows, const int32_t* ids, int n, float* dst, int dst_rows, int r0,
                                      int window, int shift, cudaStream_t st) {
  dp_scatter_targets_kernel<<<n, 128, 0, st>>>(src, src_rows, ids, dst, dst_rows, r0, window, shift);
  return cudaGetLastError();
}
