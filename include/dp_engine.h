/*
 * dp_engine.h -- C ABI of the B200-native DragPoser optimisation engine.
 *
 * One engine owns the HBM-resident state of B independent clips (latent, root
 * pose, the three 60-row ring buffers, the predicted target latents) and runs
 * the reference's per-frame optimisation for all of them in one launch.
 * Plain pointers and sizes only; no torch / C++ types.  Every entry point returns
 * 0 on success or a negative dp_status; dp_engine_last_error() gives the text.
 *
 * Reference interface each entry point replaces (paths under /root/reference):
 *   dp_engine_set_pose_model      python/src/train.py:257-269 (load_model) +
 *                                 python/src/drag_pose.py:13-34 (DragPose.__init__)
 *   dp_engine_set_temporal_model  python/src/train_temporal.py:474-482
 *   dp_engine_init_clips          python/src/drag_pose.py:47-64 (set_initial_pose)
 *   dp_engine_set_global_pos      python/src/run_drag.py:120-124
 *   dp_engine_run_frame_*         python/src/drag_pose.py:196-414 (DragPose.run)
 *   dp_engine_eval_gradient       python/src/drag_pose.py:310-343 (one decode +
 *                                 loss + backward, no optimiser step; test hook)
 *   dp_engine_get_state           attribute reads of DragPose (latent, buffers)
 * The Unity-facing DragPoserDLL ABI (DragPoserDLL/exportFunc.h:61-70) is
 * re-exported on top of this one by include/exportFunc.h.
 */
#ifndef DP_ENGINE_H
#define DP_ENGINE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden: only this header's entry points are exported */
#endif

#define DP_JOINTS 22
#define DP_LATENT 24
#define DP_POSE 88          /* 22 quaternions, standardised root-space */
#define DP_ROW 92           /* packed result row: pose (88) | global_pos (3) | pad -- the wire format of the multi-GPU gather */
#define DP_PAST_ROWS 60     /* train_temporal.param["future_frames"][0] */
#define DP_HEIGHTS 6
#define DP_MAX_WINDOW 116
#define DP_MAX_ITER 4096

typedef enum {
  DP_OK = 0,
  DP_ERR_ARG = -1,
  DP_ERR_CUDA = -2,
  DP_ERR_STATE = -3,
  DP_ERR_UNSUPPORTED = -4
} dp_status;

typedef struct dp_engine dp_engine;

/* Optimiser settings of one DragPose.run call (drag_pose.py:196-215). */
typedef struct {
  double stop_eps_pos;        /* thresholds compared in double like the Python floats */
  double stop_eps_rot;
  double min_loss_incr;       /* -inf disables */
  int32_t max_iter;           /* 1..DP_MAX_ITER */
  float learning_rate;
  float lambda_rot;
  float lambda_temporal;
  int32_t temporal_future_window;   /* multiple of 4, 0..DP_MAX_WINDOW */
  int32_t joint_adjust_joint;       /* -1 = joint adjustment off */
  int32_t joint_adjust_slot;        /* end-effector slot the joint is snapped towards */
  float joint_adjust_weight;
  int32_t decoder_path;             /* 0 = auto, 1 = fp32 CUDA-core decoder, 3 = tcgen05 fp16x2 (2, the bf16x3 kernel of round 1, was removed) */
  int32_t targets_world;            /* 0: tgt_pos is relative to the clip's current global position (what DragPose.run takes);
                                       1: tgt_pos is world-absolute and the kernel subtracts the current global position itself
                                       (eval_drag.py:164-202 -- lets whole BVH clips stream without a per-frame host step) */
  int32_t extension_losses;         /* bit mask of the reference's "Additional Losses" (drag_pose.py:129-183, commented out as shipped;
                                       added to the total loss with weight 1, y axis = 1): DP_EXT_FEET_FLOOR | DP_EXT_FORWARD |
                                       DP_EXT_HEAD_HIPS | DP_EXT_HIPS_FEET; 0 = none (the shipped behaviour).  Runs on the fp32
                                       CUDA-core frame kernel (decoder_path 3 is refused with a non-zero mask). */
  float floor_level;                /* floor height of DP_EXT_FEET_FLOOR (drag_pose.py:134) */
} dp_run_params;
#define DP_EXT_FEET_FLOOR 1   /* mean over the toes (joints 4, 8) of (global y + p_y - floor)^2          drag_pose.py:133-135 */
#define DP_EXT_FORWARD 2      /* (1 - min(1, fwd_head . fwd_hips + 0.2))^2, axes flattened to the ground  drag_pose.py:137-157 */
#define DP_EXT_HEAD_HIPS 4    /* |head - hips|^2 on the ground plane                                      drag_pose.py:159-164 */
#define DP_EXT_HIPS_FEET 8    /* sum over the ankles (3, 7) of max(|hips - ankle|^2 - 0.2^2, 0)           drag_pose.py:166-176 */

/* Pose-VAE decoder folded to three dense layers + statistics + skeleton.
 * All pointers are HOST memory, row-major, float32 unless stated. */
typedef struct {
  const float* A0; const float* b0;     /* (40,24), (40) */
  const float* A1; const float* b1;     /* (60,40), (60) */
  const float* A2; const float* b2;     /* (92,60), (92) */
  const float* mean_q; const float* std_q;   /* (88) quaternion half of the dual-quat stats */
  const float* mean_d; const float* std_d;   /* (3) displacement stats */
  const int32_t* parents;                    /* (22), parents[0] = 0, topologically ordered */
  const float* offsets;                      /* (22,3) */
} dp_pose_model;

int dp_engine_create(dp_engine** out, int device, int max_clips);
int dp_engine_destroy(dp_engine* e);
const char* dp_engine_last_error(void);
int dp_engine_version(void);

int dp_engine_set_pose_model(dp_engine* e, const dp_pose_model* m);

/* Temporal predictor: `blob` is the float32 concatenation, in the order
 * documented in dragposer_b200/engine.py:pack_temporal(), of the reference
 * Temporal.state_dict(); n_floats must be dp_engine_temporal_blob_floats(). */
size_t dp_engine_temporal_blob_floats(void);
int dp_engine_set_temporal_model(dp_engine* e, const float* blob, size_t n_floats,
                                 const float* means_latent, const float* stds_latent);

/* (Re)start n_clips clips: latent (n,24), global_pos (n,3), global_rot (n,4 wxyz),
 * heights (n,6); ring buffers are filled like DragPose.set_initial_pose. HOST pointers. */
int dp_engine_init_clips(dp_engine* e, int n_clips, const float* latent0, const float* global_pos,
                         const float* global_rot, const float* heights);
int dp_engine_set_global_pos(dp_engine* e, int first_clip, int n, const float* global_pos);
int dp_engine_n_clips(const dp_engine* e);

/* One frame for every clip.  Per clip c: n_ee[c] active trackers in slots
 * [0, n_ee[c]); slot arrays have `ee_stride` slots per clip:
 *   joints (B,ee_stride) int32, weights (B,ee_stride,2) (pos,rot),
 *   tgt_pos (B,ee_stride,3), tgt_rot (B,ee_stride,3,3) row-major.
 * n_ee may be NULL (all clips use ee_stride trackers).  joints/weights may be
 * shared by all clips (shared_trackers != 0: arrays have a single row).
 * Outputs: pose (B,88) standardised root-space quats with the root slot holding
 * the standardised world rotation, global_pos (B,3).
 * _device: every pointer is DEVICE memory, work is enqueued on `stream`
 * (a cudaStream_t, may be NULL) and not synchronised.
 * _host: every pointer is HOST memory; copies in, runs, copies out, synchronises. */
int dp_engine_run_frame_device(dp_engine* e, const dp_run_params* p, const int32_t* n_ee,
                               const int32_t* joints, const float* weights, int shared_trackers,
                               const float* tgt_pos, const float* tgt_rot, int ee_stride,
                               float* out_pose, float* out_global_pos, void* stream);
int dp_engine_run_frame_host(dp_engine* e, const dp_run_params* p, const int32_t* n_ee,
                             const int32_t* joints, const float* weights, int shared_trackers,
                             const float* tgt_pos, const float* tgt_rot, int ee_stride,
                             float* out_pose, float* out_global_pos);

/* n_frames consecutive frames from HOST arrays laid out frame-major (tgt_pos (T,B,ee_stride,3), tgt_rot (T,B,ee_stride,3,3),
 * n_ee (T,B) or NULL; joints/weights either one shared row used by every clip and frame (shared_trackers != 0) or
 * (T,B,ee_stride[,2])), results (T,B,88) / (T,B,3).  Same arithmetic as n_frames calls of dp_engine_run_frame_host, but
 * the pageable<->pinned staging and the host<->device copies of frame t+1 / t-1 overlap the kernels of frame t
 * (double-buffered blocks, copy-in and copy-out on their own streams).  Synchronises before returning. */
int dp_engine_run_frames_host(dp_engine* e, const dp_run_params* p, int n_frames, const int32_t* n_ee,
                              const int32_t* joints, const float* weights, int shared_trackers,
                              const float* tgt_pos, const float* tgt_rot, int ee_stride,
                              float* out_pose, float* out_global_pos);

/* n_frames consecutive frames with device-resident inputs laid out frame-major
 * (frame stride = B*ee_stride*{1,2,3,9} elements; n_ee stride = B; joints/weights
 * follow the frame stride unless shared_trackers).  Outputs (n_frames,B,88)/(n_frames,B,3); with out_global_pos == NULL the
 * kernels write packed rows instead: out_pose is (n_frames,B,DP_ROW) = [pose | global_pos | pad], the layout
 * dragposer_b200/dist.py gathers across GPUs without a repacking copy. */
int dp_engine_run_frames_device(dp_engine* e, const dp_run_params* p, int n_frames, const int32_t* n_ee,
                                const int32_t* joints, const float* weights, int shared_trackers,
                                const float* tgt_pos, const float* tgt_rot, int ee_stride,
                                float* out_pose, float* out_global_pos, void* stream);

/* Diagnostics of the last frame (HOST pointers, any may be NULL):
 * iters (B) int32, losses (B,3) = weighted pos, lambda-scaled rot, lambda-scaled temporal. */
int dp_engine_get_frame_stats(dp_engine* e, int32_t* iters, float* losses);
/* Per-iteration trace of the NEXT frames: rows (B,max_iter,52) =
 * [latent(24) | grad(24) | loss_pos | loss_rot | loss_temporal | active]. 0 disables. */
int dp_engine_enable_trace(dp_engine* e, int enable);
int dp_engine_get_trace(dp_engine* e, float* rows, int max_iter);

/* Teacher-forced single evaluation (no state change): latents (n,24), global_rot (n,4),
 * tgt_latent (n,24) + trackers as above; grad (n,24), losses (n,3), positions (n,22,3)
 * (any output may be NULL).  extension_losses / floor_level as in dp_run_params, global_pos (n,3) = the clips' current global
 * positions (only the feet-floor term reads it; NULL = zeros).  HOST pointers. */
int dp_engine_eval_gradient(dp_engine* e, int n, const float* latents, const float* global_rot,
                            const float* tgt_latent, const int32_t* n_ee, const int32_t* joints,
                            const float* weights, int shared_trackers, const float* tgt_pos,
                            const float* tgt_rot, int ee_stride, float lambda_rot, float lambda_temporal,
                            int decoder_path, float* grad, float* losses, float* positions,
                            int extension_losses, float floor_level, const float* global_pos);

/* Copies of the carried state in chronological ring order (HOST pointers, any may be
 * NULL): latent (B,24), global_pos (B,3), global_rot (B,4), latent_buf (B,60,24),
 * disp_buf (B,60,3), height_buf (B,60,6), target_buf (B,window+1,24). */
int dp_engine_get_state(dp_engine* e, float* latent, float* global_pos, float* global_rot,
                        float* latent_buf, float* disp_buf, float* height_buf, float* target_buf,
                        int* current_index);
int dp_engine_set_ring_buffers(dp_engine* e, const float* latent_buf, const float* disp_buf,
                               const float* height_buf);

/* Predictor only (test hook / warm start): fills target_buf for `window` from the
 * current ring buffers, as drag_pose.py:246-290 does when current_index == 0. */
int dp_engine_predict_targets(dp_engine* e, int window, void* stream);

/* Decoder path the last frame actually ran: 1 = fp32 CUDA-core kernel, 3 = tcgen05 kernel (fp16x2), 0 = none yet.
 * dp_run_params.decoder_path = 0 picks tcgen05 (fp16x2) for batches >= 512 clips (the measured crossover) and fp32 below. */
int dp_engine_last_decoder_path(const dp_engine* e);

/* Feed-forward GEMMs of the predictor: 0 = tcgen05 tensor cores, fp16x2 split products (default);
 * 1 = fp32 CUDA-core kernel (kept as an on-device cross-check, same results to ~1e-6). */
int dp_engine_set_predictor_path(dp_engine* e, int path);

/* Device-side timing of the two kernel groups, measured with CUDA events on the
 * launching stream: accumulated milliseconds of the temporal predictor and of the
 * persistent frame kernel over the frames run since profiling was (re)enabled.
 * enable = 2 additionally runs the phase clock read by dp_engine_get_phase_cycles. */
int dp_engine_set_profiling(dp_engine* e, int enable);
int dp_engine_get_profile(dp_engine* e, double* ms_predictor, double* ms_frame_kernel, long long* n_frames);
/* Phase clock of CTA 0 of the tcgen05 frame kernel (device clock64, accumulated since profiling level 2 was enabled),
 * 8 counters: [0] decoder forward, [1] dL/dy scaling + block barrier after the kinematics, [2] decoder backward,
 * [3] Adam + bookkeeping + loop barrier, [4] kinematics + loss + adjoint pass, [5..7] reserved (0). */
int dp_engine_get_phase_cycles(dp_engine* e, unsigned long long* cycles8);
/* Timeline of the two clip groups of CTA 0 over iterations 40..43 of the last frame run at profiling level 2 (device clock64):
 * stamps48[(group * 4 + iteration - 40) * 6 + k], k = loop top, forward done, kinematics done, barrier after the kinematics,
 * first two backward layers done, last backward layer + Adam done.  scripts/timeline.py prints it. */
int dp_engine_get_timeline(dp_engine* e, unsigned long long* stamps48);

/* Clip start-up on the device (SURVEY 8(f) rank 3).  Folded pose-VAE encoder: three dense layers + the mu / logvar heads
 * (autoencoder.py:136-143 folded; python: model.PoseModel.enc_*), HOST pointers, row-major (out,in) like the decoder. */
typedef struct {
  const float* A0; const float* b0;         /* (112,176), (112) */
  const float* A1; const float* b1;         /* (72,112), (72) */
  const float* A2; const float* b2;         /* (48,72), (48) */
  const float* mu_w; const float* mu_b;     /* (24,48), (24) */
  const float* logvar_w; const float* logvar_b;
} dp_encoder_model;
int dp_engine_set_encoder_model(dp_engine* e, const dp_encoder_model* m);
/* latent (n,24) = mu + eps * exp(0.5 logvar) of the standardised dual-quaternion poses dqs (n,176); eps (n,24) are the
 * caller's standard-normal draws (torch's RNG stream cannot be reproduced on the device), NULL gives the mean.  HOST
 * pointers; n <= max_clips.  Feed the result to dp_engine_init_clips. */
int dp_engine_encode_host(dp_engine* e, int n, const float* dqs, const float* eps, float* latent);

/* Accuracy metrics on the device (SURVEY 8(f) rank 2; eval_metrics.py:6-32).  pose_a, pose_b: (n,88) poses in the engine's
 * output format (standardised root-space quaternions, root slot = standardised world root rotation); err (n,2) receives per
 * row the mean joint distance (MPJPE) and the mean distance of the sparse end effectors 4, 8, 13, 17, 21 (MPEEPE), both
 * skeletons with the root at the origin.  HOST pointers. */
int dp_engine_pose_error_host(dp_engine* e, int n, const float* pose_a, const float* pose_b, float* err);

/* Per-clip restarts of a running batch.
 * Restart n clips (ids unique, < n_clips) like DragPose.set_initial_pose, leaving every other clip untouched; each restarted clip's
 * next frame is its own frame 0 (predictor call, look-ahead, ring).  latent0 (n,24), global_pos (n,3), global_rot (n,4 wxyz),
 * heights (n,6).  HOST pointers; enqueued on `stream` (NULL = engine stream), which must be the stream the frames run on.
 * A restart at a boundary (dp_engine_frames_to_boundary == 0) keeps every clip at one predictor phase and adds one kernel.
 * Anywhere else the restarted clips run at their own phase: their predictor calls then run separately, on the frame's stream
 * (no early call in the small-batch mode), and until every clip shares one phase again (dp_engine_init_clips, or restarts) a
 * window change or dp_engine_predict_targets fails with DP_ERR_STATE.  dp_engine_get_state keeps reporting the global
 * current_index and returns target_buf in each clip's own row order. */
int dp_engine_restart_clips(dp_engine* e, int n, const int32_t* clips, const float* latent0, const float* global_pos,
                            const float* global_rot, const float* heights, void* stream);
/* Own temporal index of every clip for the next frame run with `window` (B) -- what DragPose.current_index would be. */
int dp_engine_get_clip_index(dp_engine* e, int window, int32_t* index);
/* Frames until the next frame at which a restart costs no extra predictor call (0 = the next frame), or a negative dp_status. */
int dp_engine_frames_to_boundary(const dp_engine* e, int window);

/* Number of kernels launched by this engine since creation (bench "gpu_launches"). */
long long dp_engine_launch_count(const dp_engine* e);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* DP_ENGINE_H */
