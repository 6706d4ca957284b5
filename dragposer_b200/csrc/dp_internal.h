// dp_internal.h -- declarations shared by the engine translation units.
#pragma once
#include <cstdlib>
#include <atomic>

#include "dp_common.cuh"
#include "dp_temporal.cuh"

// Opt-in to more than 48 KB of dynamic shared memory.  Function attributes are per device (context): an engine on a second GPU of
// the same process needs its own call, so the "already done" bit is kept per device; racing threads at worst repeat the call.
template <class Kernel>
inline cudaError_t dp_ensure_smem(Kernel kernel, size_t smem, std::atomic<unsigned long long>& done) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const unsigned long long bit = 1ull << (dev & 63);
  if (done.load(std::memory_order_acquire) & bit) return cudaSuccess;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) done.fetch_or(bit, std::memory_order_release);
  return e;
}

struct TpWork {
  float* enc;
  float* enc2;
  float* dec;
  float* dec2;
  float* dec_lat;
  float* ffpart; // hidden-split partial sums of the feed-forward kernel (DP_FF_PART_FLOATS)
  int num_sms;
  cudaStream_t st_extra;  // second stream + fork/join events: the predictor of a large batch runs in two parts
  cudaEvent_t ev_fork, ev_join;
  struct TpGraphCache* graphs;  // replayable launch chains of small predictor calls (dp_temporal.cu); null = always launch kernel by kernel
};
// A small predictor call (B = 1 streaming: ~70 kernels of a few microseconds each at window 16) is bound by launch gaps, not by work.
// Everything after the ring-buffer embedding depends only on pointers and sizes that stay the same from call to call, so the chain is
// captured once per (clips, window, look-ahead, path, buffers) and replayed as ONE cudaGraphLaunch; the embedding kernel, which takes
// the moving ring head by value, is launched in front of it.  Same kernels, same arguments, same order: bitwise the same targets.
struct TpGraphCache* dp_temporal_graphs_create();
void dp_temporal_graphs_clear(struct TpGraphCache* c);    // drop every captured chain (model / path changes)
void dp_temporal_graphs_destroy(struct TpGraphCache* c);
#define DP_FF_PART_FLOATS ((size_t)8 * 296 * 128 * TP_D / 2)

cudaError_t dp_frame_simt_launch(const DpFrameArgs& args, int num_sms, cudaStream_t stream);
cudaError_t dp_frame_tc16_launch(const DpFrameArgs& args, int num_sms, cudaStream_t stream);  // fp16x2, weights in tensor memory
// fftiles: (TP_NENC + TP_NDEC) x FFT_LAYER_BYTES pre-tiled fp16x2 FF weights (encoder layers first) followed by
// the attention images (ATT_LAYER_BYTES each): TP_NENC encoder self-attention blocks, TP_NDEC decoder self-attention blocks,
// TP_NDEC decoder cross-attention blocks; or null to run the fp32 CUDA-core kernels.
#define DP_TC_ATT_OFFSET ((size_t)(TP_NENC + TP_NDEC) * FFT_LAYER_BYTES)
#define DP_TC_TILES_BYTES (DP_TC_ATT_OFFSET + (size_t)(TP_NENC + 2 * TP_NDEC) * ATT_LAYER_BYTES)
// ... followed by the key projections of the TP_NDEC decoder cross-attention blocks as fp32 [d = key feature][c = input] (the torch
// layout; the blob stores every Linear as [in][out]): the folded single-token cross-attention reads them coalesced over c
#define DP_TC_XA_OFFSET DP_TC_TILES_BYTES
#define DP_TC_IMAGE_TOTAL_BYTES (DP_TC_XA_OFFSET + (size_t)TP_NDEC * TP_D * TP_D * 4)
cudaError_t dp_temporal_run(const float* blob, const TpLayout& L, const float* mu, const float* sigma,
                            const float* latent_buf, const float* disp_buf, const float* height_buf, int head, int B,
                            int window, float* target_buf, const TpWork& w, const unsigned char* fftiles, cudaStream_t st,
                            long long* launches, int lookahead = 1);
// lookahead J > 1 (window 0 only): J virtual clips per real clip, virtual clip c * J + j = clip c as the predictor will see it j
// frames from now; target_buf is then (B, J, 24).  Exact, because the predictor never reads the three newest ring rows:
// train_temporal.param["past_frames"] ends at row 56 of 60 (drag_pose.py:249-266), so what it reads j <= 3 frames from now is
// already in the ring today.
#define DP_LOOKAHEAD 4
// single-token decoder pass with four clips per warp (default) or one (DP_DEC_ROWS=0, the cross-check); read on every call
inline int dp_dec_rows() {
  const char* s = getenv("DP_DEC_ROWS");
  return !(s && s[0] == '0');
}
void dp_attn_tc_pack(const float* w_in_t, const float* b_in, const float* w_out_t, const float* b_out, unsigned char* dst);
cudaError_t dp_attn_tc_launch(const unsigned char* wimg, const float* blob, const TpNorm& N1, const float* xq, int T, int q_stride,
                              const float* xkv, int S, int kv_stride, int n_clips, float* out, cudaStream_t st);
void dp_ff_tc_pack(const float* w1t, const float* b1, const float* w2t, unsigned char* dst);
// part: workspace of part_floats floats for the hidden-split mode used when the row count cannot fill the device (or null)
cudaError_t dp_ff_tc_launch(const unsigned char* wimg, const float* blob, const TpFF& F, const TpNorm& N1, const TpNorm& N2, int has_n2,
                            const float* x, int n_rows, int T, int row_stride, float* out, float* part, size_t part_floats, int num_sms,
                            cudaStream_t st, long long* launches, const TpFfTail* tail = nullptr);
// blob: [A0t (176x112) | b0 | A1t (112x72) | b1 | A2t (72x48) | b2 | head_t (48x48: mu | logvar columns) | head_b (48)], DP_ENC_BLOB_FLOATS
cudaError_t dp_encode_launch(const float* blob, const float* dqs, const float* eps, float* latent, int n, cudaStream_t st);
// per row: mean joint distance, mean end-effector distance of two poses in the engine's output format (root at the origin)
cudaError_t dp_pose_error_launch(const DpModelImage* model, const float* pose_a, const float* pose_b, int n, float* err, cudaStream_t st);
// Per-clip restarts (dp_restart.cu).  state: n rows of latent (24) | global_pos (3) | global_rot (4) | heights (6)
#define DP_RESTART_STATE (DP_L + 3 + 4 + DP_NH)
cudaError_t dp_reset_clips_launch(const int32_t* ids, const float* state, int n, float* latent, float* gpos, float* grot,
                                  float* latent_buf, float* disp_buf, float* height_buf, cudaStream_t st);
// ring rows of the listed clips -> compact (n, DP_PAST, .) buffers, slot for slot
cudaError_t dp_gather_rings_launch(const int32_t* ids, int n, const float* latent_buf, const float* disp_buf, const float* height_buf,
                                   float* s_latent, float* s_disp, float* s_height, cudaStream_t st);
// compact predictor rows (n, src_rows, 24) -> rows [r0, dst_rows) of the listed clips' target rows; src_rows == 1 broadcasts,
// otherwise own row k < window goes to slot (k + shift) % window and own row `window` to slot `window`
cudaError_t dp_scatter_targets_launch(const float* src, int src_rows, const int32_t* ids, int n, float* dst, int dst_rows, int r0,
                                      int window, int shift, cudaStream_t st);
