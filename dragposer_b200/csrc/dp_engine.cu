// dp_engine.cu -- host side of the C ABI declared in include/dp_engine.h.
//
// Owns the HBM-resident per-clip state (laid out clip-major so one warp streams one
// clip's rows with coalesced, vectorised accesses), the model images, pinned staging
// buffers for the host-pointer entry points, and launches the persistent frame kernel
// (and, when the reference would, the temporal predictor first).
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <chrono>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

#include "../../include/dp_engine.h"
#include "dp_internal.h"

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t _e = (call);                                                                       \
    if (_e != cudaSuccess) return fail(DP_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e)); \
  } while (0)

static int check_window(int w) {  // drag_pose.py:236
  return (w < 0 || w > DP_MAX_WINDOW || w % 4) ? fail(DP_ERR_ARG, "the temporal window must be a multiple of 4 in [0,116]") : DP_OK;
}

// Which target row every clip reads at the next frame and when the predictor runs (drag_pose.py:237-244,399-402); host state only.
// Look-ahead at temporal_future_window == 0 (the predictor runs every frame): its inputs end three frames in the past
// (train_temporal.param["past_frames"] stops at ring row 56 of 60), so the targets of this frame AND the next three are computed
// in ONE batched predictor call (4 x n_clips virtual clips: fuller tiles, a quarter of the launches) -- the same numbers the
// reference computes frame by frame.
// Per-clip restarts (dp_engine_restart_clips).  Clip c runs at its own predictor phase phase[c]: its own temporal index is
// (current_index - phase[c]) mod window, and its own target row k < window lives in slot (k + phase[c]) % window of d_target_buf
// (row window in slot window), so the frame kernels read slot current_index of every clip as before.  While every clip shares one
// phase it is folded into current_index (all phases 0, n_phases 1) and nothing differs from a batch that was never restarted.
struct TargetSchedule {
  int target_rows = 0;           // window + 1 of d_target_buf, 0 = none yet
  int current_index = 0;
  int look_left = 0;             // window 0: rows of d_target_pre not read yet; the next frame reads row DP_LOOKAHEAD - look_left
  int look_last_row = -1;        // window 0: the row of d_target_pre the last frame read; -1 = it read d_target_buf
  std::vector<int> phase;        // (n_clips)
  int n_phases = 1;              // distinct phases among the clips; >= 2 = mixed
  std::vector<int> class_start;  // mixed phases: the clips of phase s are d_class[class_start[s] .. class_start[s + 1])
  // The index a frame at window W runs at.  The reference keeps current_index when the window changes: rows of the fresh zero buffer
  // are used until it wraps to 0.  An index beyond the new buffer, an IndexError there on every later frame, restarts the cycle here.
  int index_at(int W) const { return current_index > W ? 0 : current_index; }
  int check_window_change(int W) const {
    if (target_rows != W + 1 && n_phases > 1)
      return fail(DP_ERR_STATE, "the temporal window cannot change while restarted clips run at their own predictor phase: "
                                "re-initialise the clips (dp_engine_init_clips) to change it");
    return DP_OK;
  }
  int clip_index(int c, int W) const { return W == 0 ? 0 : (index_at(W) - phase[c] + W) % W; }
  int slot(int c, int k, int W) const { return (k + phase[c]) % W; }  // of clip c's own row k < W
  // The next frame whose index is some clip's phase: a predictor call runs there anyway, a clip restarted just before joins it.
  int frames_to_boundary(int W) const {
    if (W == 0) return target_rows == 1 ? look_left : 0;  // the next look-ahead call covers every clip
    for (int d = 0, g = index_at(W); d <= W; ++d, g = (g + 1) % W)
      if (n_phases > 1 ? class_start[g + 1] > class_start[g] : g == 0) return d;
    return fail(DP_ERR_STATE, "dp_engine_frames_to_boundary: no predictor frame ahead");
  }
  void reset(int n_clips) { *this = TargetSchedule(); phase.assign(n_clips, 0); }
  void advance(int W) { current_index = W == 0 ? 0 : (current_index + 1) % W; }  // drag_pose.py:399-402
};

struct dp_engine {
  int device = 0, max_clips = 0, n_clips = 0, num_sms = 148;
  bool has_pose = false, has_temporal = false;
  DpModelImage* d_model = nullptr;
  DpModelImageTC* d_model_tc = nullptr;
  uint32_t* d_model_tmem = nullptr;
  float* d_encoder = nullptr;  // folded encoder blob (DP_ENC_BLOB_FLOATS), set by dp_engine_set_encoder_model
  float* d_tblob = nullptr;
  unsigned char* d_fftiles = nullptr;  // pre-tiled fp16x2 tensor-core weight images of the predictor (DP_TC_TILES_BYTES)
  int predictor_path = 0;              // 0 = tcgen05 FF (default), 1 = fp32 CUDA-core FF
  int last_path = 0;                   // decoder path of the last frame: 1 = fp32, 3 = tcgen05 fp16x2
  float *d_mu = nullptr, *d_sigma = nullptr;
  TpLayout tl;
  // state
  float *d_latent = nullptr, *d_gpos = nullptr, *d_grot = nullptr;
  float *d_latent_buf = nullptr, *d_disp_buf = nullptr, *d_height_buf = nullptr;
  float* d_target_buf = nullptr;  // (B, DP_MAX_WINDOW+1, 24) capacity; logical rows = window+1
  int ring_head = 0;
  float* d_target_pre = nullptr;  // (B, DP_LOOKAHEAD, 24): the window-0 look-ahead rows (TargetSchedule)
  TargetSchedule sched;
  // Predictor ahead of time in the small-batch streaming mode (window >= 4, <= DP_PREFETCH_MAX_CLIPS clips; DP_PRED_PREFETCH=0 turns it
  // off).  The same three-frame slack as above: what the predictor reads at the window's first frame t (chronological ring rows
  // 0..56) is complete once frame t-4 is, so the call for frame t is issued three frames early, on its own stream, with the ring head
  // advanced by three and a second target buffer as destination; frame t only waits for its event and swaps the two buffers.  Same
  // kernels on the same rows: bitwise the targets of the call at frame t.  A real-time caller (one frame every few milliseconds) never
  // sees the ~0.45 ms predictor chain on its frame path; back-to-back callers overlap it with three frames.
  float* d_target_alt = nullptr;
  cudaStream_t pre_stream = nullptr;
  cudaEvent_t ev_pre_fork = nullptr, ev_pre_done = nullptr;
  bool pre_valid = false;  // an early call into d_target_alt was issued at the current window and not used yet
  int prefetch = 1;
  // outputs / diagnostics
  int32_t* d_iters = nullptr;
  float* d_losses = nullptr;
  float* d_trace = nullptr;
  int trace_iters = 0, trace_enabled = 0;
  float* d_adam = nullptr;
  int adam_iters = 0;
  float adam_lr = -1.0f;
  TpWork tw{};
  // staging for the host-pointer path
  // double-buffered staging of dp_engine_run_frames_host: one contiguous block per slot and direction
  struct FramePipe {
    int stride = 0;
    unsigned char *h_in[2] = {nullptr, nullptr}, *d_in[2] = {nullptr, nullptr};
    float *h_out[2] = {nullptr, nullptr}, *d_out[2] = {nullptr, nullptr};
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_run[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
    cudaStream_t cs_in = nullptr, cs_out = nullptr;
  } pipe;
  cudaStream_t stream = nullptr;
  long long launches = 0;
  // optional device-side timing of the two kernel groups (bench roofline)
  int profiling = 0;
  unsigned long long* d_phase = nullptr;  // 8 phase-cycle counters + 48 timeline stamps of the tcgen05 frame kernel (profiling level 2 only)
  std::vector<cudaEvent_t> prof_events;  // triples: before predictor, before frame kernel, after frame kernel
  int32_t* d_class = nullptr;  // restarts: clip ids grouped by phase (TargetSchedule::class_start), ascending within a phase
  // pinned staging of a restart: restarted ids (max_clips) | ids grouped by phase (max_clips) | state rows (max_clips, DP_RESTART_STATE);
  // ev_restart follows its copies, so the next restart does not overwrite a block still in flight
  unsigned char *h_restart = nullptr, *d_restart = nullptr;
  cudaEvent_t ev_restart = nullptr;
  bool restart_pending = false;
  // compact inputs and outputs of the subset predictor (allocated on first use, max_clips rows)
  float *d_sub_latent = nullptr, *d_sub_disp = nullptr, *d_sub_height = nullptr, *d_sub_target = nullptr;
};

extern "C" const char* dp_engine_last_error(void) { return g_err.c_str(); }
#define DP_PREFETCH_MAX_CLIPS 256
// let the early call finish and forget it: its targets are void (window or clips changed) or its work buffers are needed elsewhere
static void drop_prefetch(dp_engine* e) {
  if (e->pre_valid) cudaStreamSynchronize(e->pre_stream);
  e->pre_valid = false;
}

static void void_targets_ahead(dp_engine* e) {  // the early call and the look-ahead rows: ring rows, clips, model or path changed
  drop_prefetch(e);
  e->sched.look_left = 0;
}

extern "C" int dp_engine_version(void) { return 100; }
extern "C" size_t dp_engine_temporal_blob_floats(void) { return tp_layout().total; }
extern "C" int dp_engine_n_clips(const dp_engine* e) { return e ? e->n_clips : 0; }
extern "C" long long dp_engine_launch_count(const dp_engine* e) { return e ? e->launches : 0; }

extern "C" int dp_engine_create(dp_engine** out, int device, int max_clips) {
  if (!out || max_clips <= 0) return fail(DP_ERR_ARG, "dp_engine_create: bad arguments");
  int count = 0;
  CK(cudaGetDeviceCount(&count));
  if (device < 0 || device >= count) return fail(DP_ERR_ARG, "dp_engine_create: no such CUDA device");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail(DP_ERR_UNSUPPORTED, "dp_engine_create: needs an sm_100 (B200) device");
  dp_engine* e = new dp_engine();
  e->device = device;
  e->max_clips = max_clips;
  e->num_sms = prop.multiProcessorCount;
  e->tl = tp_layout();
  const size_t B = (size_t)max_clips;
  CK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
  CK(cudaMalloc(&e->d_model, sizeof(DpModelImage)));
  CK(cudaMalloc(&e->d_model_tc, sizeof(DpModelImageTC)));
  CK(cudaMalloc(&e->d_model_tmem, (size_t)DP_TC_TMEM_WORDS * 128 * 4));
  CK(cudaMalloc(&e->d_latent, B * DP_L * 4));
  CK(cudaMalloc(&e->d_gpos, B * 3 * 4));
  CK(cudaMalloc(&e->d_grot, B * 4 * 4));
  CK(cudaMalloc(&e->d_latent_buf, B * DP_PAST * DP_L * 4));
  CK(cudaMalloc(&e->d_disp_buf, B * DP_PAST * 3 * 4));
  CK(cudaMalloc(&e->d_height_buf, B * DP_PAST * DP_NH * 4));
  CK(cudaMalloc(&e->d_target_buf, B * (DP_MAX_WINDOW + 1) * DP_L * 4));
  CK(cudaMemset(e->d_target_buf, 0, B * (DP_MAX_WINDOW + 1) * DP_L * 4));
  CK(cudaMalloc(&e->d_iters, B * 4));
  CK(cudaMalloc(&e->d_losses, B * 3 * 4));
  CK(cudaMalloc(&e->d_mu, DP_L * 4));
  CK(cudaMalloc(&e->d_sigma, DP_L * 4));
  const size_t V = B * DP_LOOKAHEAD;  // virtual clips of a look-ahead predictor call
  CK(cudaMalloc(&e->d_target_pre, V * DP_L * 4));
  CK(cudaMemset(e->d_target_pre, 0, V * DP_L * 4));
  CK(cudaMalloc(&e->tw.enc, V * TP_S * TP_D * 4));
  CK(cudaMalloc(&e->tw.enc2, V * TP_S * TP_D * 4));
  CK(cudaMalloc(&e->tw.dec, V * TP_MAXT * TP_D * 4));
  CK(cudaMalloc(&e->tw.dec2, V * TP_MAXT * TP_D * 4));
  CK(cudaMalloc(&e->tw.dec_lat, V * TP_MAXT * TP_LAT * 4));
  CK(cudaMalloc(&e->tw.ffpart, DP_FF_PART_FLOATS * 4));
  e->tw.num_sms = e->num_sms;
  e->tw.graphs = dp_temporal_graphs_create();
  if (const char* s = getenv("DP_PRED_PREFETCH")) e->prefetch = atoi(s) != 0;
  CK(cudaMalloc(&e->d_target_alt, B * (DP_MAX_WINDOW + 1) * DP_L * 4));
  CK(cudaStreamCreateWithFlags(&e->pre_stream, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&e->ev_pre_fork, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&e->ev_pre_done, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&e->tw.ev_fork, cudaEventDisableTiming));
  CK(cudaStreamCreateWithFlags(&e->tw.st_extra, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&e->tw.ev_join, cudaEventDisableTiming));
  *out = e;
  return DP_OK;
}

static void free_pipe(dp_engine* e) {
  for (int i = 0; i < 2; ++i) {
    cudaFreeHost(e->pipe.h_in[i]); cudaFree(e->pipe.d_in[i]); cudaFreeHost(e->pipe.h_out[i]); cudaFree(e->pipe.d_out[i]);
    if (e->pipe.ev_h2d[i]) cudaEventDestroy(e->pipe.ev_h2d[i]);
    if (e->pipe.ev_run[i]) cudaEventDestroy(e->pipe.ev_run[i]);
    if (e->pipe.ev_d2h[i]) cudaEventDestroy(e->pipe.ev_d2h[i]);
  }
  if (e->pipe.cs_in) cudaStreamDestroy(e->pipe.cs_in);
  if (e->pipe.cs_out) cudaStreamDestroy(e->pipe.cs_out);
  e->pipe = dp_engine::FramePipe();
}

extern "C" int dp_engine_destroy(dp_engine* e) {
  if (!e) return DP_OK;
  cudaSetDevice(e->device);
  cudaStreamSynchronize(e->stream);
  free_pipe(e);
  cudaFree(e->d_model); cudaFree(e->d_model_tc); cudaFree(e->d_model_tmem); cudaFree(e->d_encoder); cudaFree(e->d_tblob); cudaFree(e->d_fftiles); cudaFree(e->d_mu); cudaFree(e->d_sigma);
  cudaFree(e->d_latent); cudaFree(e->d_gpos); cudaFree(e->d_grot); cudaFree(e->d_latent_buf);
  cudaFree(e->d_disp_buf); cudaFree(e->d_height_buf); cudaFree(e->d_target_buf); cudaFree(e->d_target_pre); cudaFree(e->d_iters);
  cudaFree(e->d_losses); cudaFree(e->d_trace); cudaFree(e->d_adam); cudaFree(e->d_phase);
  cudaFree(e->tw.enc); cudaFree(e->tw.enc2); cudaFree(e->tw.dec); cudaFree(e->tw.dec2); cudaFree(e->tw.dec_lat); cudaFree(e->tw.ffpart);
  if (e->tw.st_extra) { cudaStreamSynchronize(e->tw.st_extra); cudaStreamDestroy(e->tw.st_extra); }
  if (e->tw.ev_join) cudaEventDestroy(e->tw.ev_join);
  if (e->tw.ev_fork) cudaEventDestroy(e->tw.ev_fork);
  if (e->pre_stream) { cudaStreamSynchronize(e->pre_stream); cudaStreamDestroy(e->pre_stream); }
  if (e->ev_pre_fork) cudaEventDestroy(e->ev_pre_fork);
  if (e->ev_pre_done) cudaEventDestroy(e->ev_pre_done);
  cudaFree(e->d_target_alt);
  cudaFreeHost(e->h_restart); cudaFree(e->d_restart);
  if (e->ev_restart) cudaEventDestroy(e->ev_restart);
  cudaFree(e->d_sub_latent); cudaFree(e->d_sub_disp); cudaFree(e->d_sub_height); cudaFree(e->d_sub_target);
  dp_temporal_graphs_destroy(e->tw.graphs);
  cudaStreamDestroy(e->stream);
  delete e;
  return DP_OK;
}

extern "C" int dp_engine_set_pose_model(dp_engine* e, const dp_pose_model* m) {
  if (!e || !m || !m->A0 || !m->A1 || !m->A2 || !m->parents || !m->offsets)
    return fail(DP_ERR_ARG, "dp_engine_set_pose_model: null argument");
  CK(cudaSetDevice(e->device));
  std::vector<unsigned char> raw(sizeof(DpModelImage), 0);
  DpModelImage& I = *reinterpret_cast<DpModelImage*>(raw.data());
  const float* A[3] = {m->A0, m->A1, m->A2};
  float* Wt[3] = {I.W0t, I.W1t, I.W2t};
  float* Wr[3] = {I.W0, I.W1, I.W2};
  const int dims[4] = {DP_L, DP_H0, DP_H1, DP_Y};
  for (int l = 0; l < 3; ++l) {
    const int K = dims[l], N = dims[l + 1];
    for (int o = 0; o < N; ++o)
      for (int k = 0; k < K; ++k) {
        Wt[l][k * N + o] = A[l][o * K + k];
        Wr[l][o * K + k] = A[l][o * K + k];
      }
  }
  memcpy(I.b0, m->b0, sizeof(I.b0));
  memcpy(I.b1, m->b1, sizeof(I.b1));
  memcpy(I.b2, m->b2, sizeof(I.b2));
  memcpy(I.mean_q, m->mean_q, sizeof(I.mean_q));
  memcpy(I.std_q, m->std_q, sizeof(I.std_q));
  for (int i = 0; i < 3; ++i) { I.mean_d[i] = m->mean_d[i]; I.std_d[i] = m->std_d[i]; }
  // skeleton tables
  const int32_t* par = m->parents;
  if (par[0] != 0) return fail(DP_ERR_ARG, "skeleton: parents[0] must be 0");
  int depth[DP_J] = {0}, nchild[DP_J] = {0}, last[DP_J];
  for (int j = 1; j < DP_J; ++j) {
    if (par[j] < 0 || par[j] >= j) return fail(DP_ERR_ARG, "skeleton: parents must be topologically ordered");
    depth[j] = depth[par[j]] + 1;
    if (depth[j] >= (1 << DP_JUMP_ROUNDS)) return fail(DP_ERR_UNSUPPORTED, "skeleton: chain deeper than 15");
  }
  for (int j = 0; j < DP_J; ++j) last[j] = j;
  for (int j = DP_J - 1; j >= 1; --j) last[par[j]] = last[par[j]] > last[j] ? last[par[j]] : last[j];
  for (int j = 1; j < DP_J; ++j)  // pre-order check: subtree(par) must be the contiguous range [par, last[par]]
    if (j > last[par[j]]) return fail(DP_ERR_UNSUPPORTED, "skeleton: joints must be numbered in DFS pre-order");
  {
    std::vector<int> cnt(DP_J, 1);
    for (int j = DP_J - 1; j >= 1; --j) cnt[par[j]] += cnt[j];
    for (int j = 0; j < DP_J; ++j)
      if (last[j] - j + 1 != cnt[j]) return fail(DP_ERR_UNSUPPORTED, "skeleton: joints must be numbered in DFS pre-order");
  }
  for (int k = 0; k < DP_MAX_CHILD; ++k)
    for (int j = 0; j < 32; ++j) I.child[k][j] = -1;
  for (int r = 0; r < DP_JUMP_ROUNDS; ++r)
    for (int j = 0; j < 32; ++j) I.jump[r][j] = -1;
  const int height_joints[DP_NH] = {0, 4, 8, 13, 17, 21};  // train_temporal.param["height_indices"]
  for (int j = 0; j < 32; ++j) {
    I.parent[j] = 0;
    I.last[j] = j;
    I.height_slot[j] = -1;
  }
  for (int s = 0; s < DP_NH; ++s) I.height_slot[height_joints[s]] = s;
  int max_depth = 0, max_children = 0;
  for (int j = 0; j < DP_J; ++j) {
    I.parent[j] = par[j];
    I.last[j] = last[j];
    for (int i = 0; i < 3; ++i) I.off[j][i] = (j == 0) ? 0.0f : m->offsets[3 * j + i];  // train.py:340
    if (j > 0) {
      const int p = par[j];
      if (nchild[p] >= DP_MAX_CHILD) return fail(DP_ERR_UNSUPPORTED, "skeleton: more than 4 children on one joint");
      I.child[nchild[p]][p] = j;
      for (int i = 0; i < 3; ++i) I.coff[nchild[p]][p][i] = m->offsets[3 * j + i];
      ++nchild[p];
      if (nchild[p] > max_children) max_children = nchild[p];
      if (depth[j] > max_depth) max_depth = depth[j];
      int a = j;
      for (int r = 0, dist = 1; r < DP_JUMP_ROUNDS; ++r, dist <<= 1) {
        // ancestor at distance 2^r, if the chain is that long
        if (depth[j] >= dist) {
          a = j;
          for (int s = 0; s < dist; ++s) a = par[a];
          I.jump[r][j] = a;
        }
      }
      (void)a;
    }
  }
  I.pad[0] = 0;
  while ((1 << I.pad[0]) <= max_depth) ++I.pad[0];  // pointer-jumping rounds: smallest r with 2^r > max depth
  I.pad[1] = max_children;
  CK(cudaMemcpy(e->d_model, raw.data(), raw.size(), cudaMemcpyHostToDevice));
  {  // tcgen05 kernel: the same biases / statistics / skeleton tables, and the weights as a tensor-memory image
    std::vector<unsigned char> raw_tc(sizeof(DpModelImageTC), 0);
    DpModelImageTC& T = *reinterpret_cast<DpModelImageTC*>(raw_tc.data());
    memcpy(T.b0, I.b0, sizeof(I.b0)); memcpy(T.b1, I.b1, sizeof(I.b1)); memcpy(T.b2, I.b2, sizeof(I.b2));
    memcpy(T.mean_q, I.mean_q, sizeof(I.mean_q)); memcpy(T.std_q, I.std_q, sizeof(I.std_q));
    memcpy(T.mean_d, I.mean_d, sizeof(I.mean_d)); memcpy(T.std_d, I.std_d, sizeof(I.std_d));
    memcpy(T.off, I.off, sizeof(I.off)); memcpy(T.coff, I.coff, sizeof(I.coff)); memcpy(T.child, I.child, sizeof(I.child));
    memcpy(T.jump, I.jump, sizeof(I.jump)); memcpy(T.parent, I.parent, sizeof(I.parent)); memcpy(T.last, I.last, sizeof(I.last));
    memcpy(T.height_slot, I.height_slot, sizeof(I.height_slot));
    memcpy(T.pad, I.pad, sizeof(I.pad));
    CK(cudaMemcpy(e->d_model_tc, raw_tc.data(), raw_tc.size(), cudaMemcpyHostToDevice));
    // tensor-memory image (fp16x2 pieces of 16 W): lane m, word c holds K elements (2c', 2c'+1) of row m of the A operand --
    // forward layer l: A = 16 W_l (rows = outputs), backward: A = 16 W_l^T (rows = inputs); order and widths as WT<> in
    // dp_frame_tc16.cu: fwd0 (K 32) fwd1 (48) fwd2 (64) bwd2 (96) bwd1 (64) bwd0 (48), two pieces each
    std::vector<uint32_t> tm((size_t)DP_TC_TMEM_WORDS * 128, 0u);
    const int kpad[3] = {32, 48, 64}, opad[3] = {48, 64, 96};
    uint32_t col = 0;
    // `replicate` = 32: the rows repeat in every 32-lane quarter (the last backward layer: each warp reads dL/dz in its own quarter);
    // 64: they repeat in the upper 64 lanes (layers of <= 64 rows: all eight epilogue warps of a group share the clips); 0: plain
    auto put = [&](int l, bool fwd, int replicate) {
      const int K = dims[l], N = dims[l + 1];          // W_l is [N][K]
      const int kk = fwd ? kpad[l] : opad[l];          // padded reduction length of this operand
      for (int p = 0; p < 2; ++p) {
        for (int lane = 0; lane < 128; ++lane)
          for (int k = 0; k < kk; ++k) {
            const int m = replicate ? (lane % replicate) : lane;
            const bool in = fwd ? (m < N && k < K) : (m < K && k < N);
            float r = in ? 16.0f * (fwd ? A[l][m * K + k] : A[l][k * K + m]) : 0.0f;
            __half h = __float2half_rn(r);
            if (p == 1) { r -= __half2float(h); h = __float2half_rn(r); }
            uint16_t bits;
            memcpy(&bits, &h, 2);
            tm[(size_t)(col + k / 2) * 128 + lane] |= (uint32_t)bits << (16 * (k & 1));
          }
        col += kk / 2;
      }
    };
    static_assert(DP_L <= 32, "the replicated rows of the last backward layer must fit a lane quarter");
    static_assert(DP_H0 <= 64 && DP_H1 <= 64, "the replicated rows of the two hidden layers must fit 64 lanes");
    put(0, true, 64); put(1, true, 64); put(2, true, 0); put(2, false, 64); put(1, false, 64); put(0, false, 32);
    if (col != DP_TC_TMEM_WORDS) return fail(DP_ERR_STATE, "tensor-memory weight image layout");
    CK(cudaMemcpy(e->d_model_tmem, tm.data(), tm.size() * 4, cudaMemcpyHostToDevice));
  }
  e->has_pose = true;
  return DP_OK;
}

extern "C" int dp_engine_set_temporal_model(dp_engine* e, const float* blob, size_t n_floats, const float* means_latent,
                                            const float* stds_latent) {
  if (!e || !blob || !means_latent || !stds_latent) return fail(DP_ERR_ARG, "dp_engine_set_temporal_model: null argument");
  if (n_floats != e->tl.total) return fail(DP_ERR_ARG, "dp_engine_set_temporal_model: blob size mismatch");
  CK(cudaSetDevice(e->device));
  void_targets_ahead(e);
  if (!e->d_tblob) CK(cudaMalloc(&e->d_tblob, n_floats * 4));
  CK(cudaMemcpy(e->d_tblob, blob, n_floats * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(e->d_mu, means_latent, DP_L * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(e->d_sigma, stds_latent, DP_L * 4, cudaMemcpyHostToDevice));
  {
    std::vector<unsigned char> tiles(DP_TC_IMAGE_TOTAL_BYTES);
    for (int l = 0; l < TP_NENC + TP_NDEC; ++l) {
      const TpFF& f = l < TP_NENC ? e->tl.enc[l].ff : e->tl.dec[l - TP_NENC].ff;
      dp_ff_tc_pack(blob + f.w1, blob + f.b1, blob + f.w2, tiles.data() + (size_t)l * FFT_LAYER_BYTES);
    }
    for (int i = 0; i < TP_NENC + 2 * TP_NDEC; ++i) {  // encoder self, decoder self, decoder cross
      const TpAttn& a = i < TP_NENC ? e->tl.enc[i].sa : (i < TP_NENC + TP_NDEC ? e->tl.dec[i - TP_NENC].sa : e->tl.dec[i - TP_NENC - TP_NDEC].ca);
      dp_attn_tc_pack(blob + a.w_in, blob + a.b_in, blob + a.w_out, blob + a.b_out, tiles.data() + DP_TC_ATT_OFFSET + (size_t)i * ATT_LAYER_BYTES);
    }
    float* wk_t = reinterpret_cast<float*>(tiles.data() + DP_TC_XA_OFFSET);
    for (int l = 0; l < TP_NDEC; ++l)
      for (int d = 0; d < TP_D; ++d)
        for (int c = 0; c < TP_D; ++c) wk_t[((size_t)l * TP_D + d) * TP_D + c] = blob[e->tl.dec[l].ca.w_in + (size_t)c * 3 * TP_D + TP_D + d];
    if (!e->d_fftiles) CK(cudaMalloc(&e->d_fftiles, tiles.size()));
    CK(cudaMemcpy(e->d_fftiles, tiles.data(), tiles.size(), cudaMemcpyHostToDevice));
  }
  e->has_temporal = true;
  dp_temporal_graphs_clear(e->tw.graphs);
  return DP_OK;
}

extern "C" int dp_engine_init_clips(dp_engine* e, int n, const float* latent0, const float* gpos, const float* grot,
                                    const float* heights) {
  if (!e || !latent0 || !gpos || !grot || !heights) return fail(DP_ERR_ARG, "dp_engine_init_clips: null argument");
  if (n <= 0 || n > e->max_clips) return fail(DP_ERR_ARG, "dp_engine_init_clips: n_clips out of range");
  CK(cudaSetDevice(e->device));
  CK(cudaStreamSynchronize(e->stream));
  void_targets_ahead(e);
  std::vector<float> lb((size_t)n * DP_PAST * DP_L), hb((size_t)n * DP_PAST * DP_NH);
  for (int c = 0; c < n; ++c)
    for (int r = 0; r < DP_PAST; ++r) {
      memcpy(&lb[((size_t)c * DP_PAST + r) * DP_L], latent0 + (size_t)c * DP_L, DP_L * 4);
      memcpy(&hb[((size_t)c * DP_PAST + r) * DP_NH], heights + (size_t)c * DP_NH, DP_NH * 4);
    }
  CK(cudaMemcpy(e->d_latent, latent0, (size_t)n * DP_L * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(e->d_gpos, gpos, (size_t)n * 3 * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(e->d_grot, grot, (size_t)n * 4 * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(e->d_latent_buf, lb.data(), lb.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(e->d_height_buf, hb.data(), hb.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(e->d_disp_buf, 0, (size_t)n * DP_PAST * 3 * 4));
  e->n_clips = n;
  e->ring_head = 0;
  e->sched.reset(n);
  return DP_OK;
}

extern "C" int dp_engine_set_global_pos(dp_engine* e, int first, int n, const float* gpos) {
  if (!e || !gpos || first < 0 || n <= 0 || first + n > e->n_clips) return fail(DP_ERR_ARG, "dp_engine_set_global_pos: bad range");
  CK(cudaSetDevice(e->device));
  CK(cudaMemcpyAsync(e->d_gpos + (size_t)first * 3, gpos, (size_t)n * 3 * 4, cudaMemcpyHostToDevice, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return DP_OK;
}

static int ensure_adam(dp_engine* e, int max_iter, float lr) {
  if (e->d_adam && e->adam_iters == max_iter && e->adam_lr == lr) return DP_OK;
  // torch/optim/adam.py:414-547: step_size = lr / (1 - beta1^k), sqrt(1 - beta2^k) -- Python doubles
  std::vector<float> tab(2 * (size_t)max_iter);
  const double lrd = (double)lr;
  for (int k = 1; k <= max_iter; ++k) {
    tab[k - 1] = (float)(lrd / (1.0 - std::pow(0.9, (double)k)));
    tab[max_iter + k - 1] = (float)(1.0 / std::pow(1.0 - std::pow(0.999, (double)k), 0.5));  // kernels multiply by the reciprocal
  }
  // earlier frames may still be reading the table on a caller-supplied stream (run_frames_device): settle the whole device first
  CK(cudaDeviceSynchronize());
  if (e->adam_iters != max_iter) {
    cudaFree(e->d_adam);
    e->d_adam = nullptr;
    CK(cudaMalloc(&e->d_adam, tab.size() * 4));
  }
  // ordered after earlier frames on the engine stream
  CK(cudaMemcpyAsync(e->d_adam, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  e->adam_iters = max_iter;
  e->adam_lr = lr;
  return DP_OK;
}

static int check_params(const dp_engine* e, const dp_run_params* p, int ee_stride) {
  if (!e->has_pose) return fail(DP_ERR_STATE, "pose model not set");
  if (e->n_clips <= 0) return fail(DP_ERR_STATE, "no clips initialised");
  if (p->max_iter < 1 || p->max_iter > DP_MAX_ITER) return fail(DP_ERR_ARG, "max_iter out of range");
  if (int rc = check_window(p->temporal_future_window)) return rc;
  if (ee_stride < 1 || ee_stride > DP_JOINTS) return fail(DP_ERR_ARG, "ee_stride out of range");
  if (p->joint_adjust_joint >= DP_JOINTS || (p->joint_adjust_joint >= 0 && (p->joint_adjust_slot < 0 || p->joint_adjust_slot >= ee_stride)))
    return fail(DP_ERR_ARG, "joint adjustment indices out of range");
  if (p->extension_losses < 0 || p->extension_losses > 15) return fail(DP_ERR_ARG, "extension_losses must be a mask of DP_EXT_* bits");
  if (p->extension_losses && p->decoder_path == 3)
    return fail(DP_ERR_UNSUPPORTED, "the extension losses run on the fp32 CUDA-core frame kernel: use decoder_path 0 or 1");
  if (p->decoder_path != 0 && p->decoder_path != 1 && p->decoder_path != 3)
    return fail(DP_ERR_ARG, "decoder_path must be 0 (auto), 1 (fp32 CUDA cores) or 3 (tcgen05 fp16x2); 2 (bf16x3) was removed");
  return DP_OK;
}

// host-side tracker counts: 1 <= n_ee[c] <= ee_stride, and the joint-adjustment slot must be an active tracker of every clip
static int check_n_ee(const int32_t* n_ee, size_t count, int ee_stride, const dp_run_params* p) {
  if (!n_ee) return DP_OK;
  const int need = (p && p->joint_adjust_joint >= 0) ? p->joint_adjust_slot + 1 : 1;
  for (size_t i = 0; i < count; ++i)
    if (n_ee[i] < need || n_ee[i] > ee_stride)
      return fail(DP_ERR_ARG, "n_ee entries must lie in [1, ee_stride] and cover the joint-adjustment slot");
  return DP_OK;
}

// The one caller of the temporal predictor: n clips' rings read from `head` -> (n, J or window + 1, 24) targets at dst, on st.
static int run_predictor(dp_engine* e, const float* latent, const float* disp, const float* height, int head, int n, int window,
                         float* dst, cudaStream_t st, int J = 1) {
  if (!e->has_temporal) return fail(DP_ERR_STATE, "temporal model not set");
  drop_prefetch(e);  // an early call still in flight uses the same work buffers
  CK(dp_temporal_run(e->d_tblob, e->tl, e->d_mu, e->d_sigma, latent, disp, height, head, n, window, dst, e->tw,
                     e->predictor_path == 1 ? nullptr : e->d_fftiles, st, &e->launches, J));
  return DP_OK;
}

// The predictor for the n clips listed at d_ids (device) alone: their ring rows are gathered into compact buffers (same ring head),
// the unmodified predictor runs on those, and its (n, window + 1, 24) rows are scattered into rows [r0, dst_rows) of dst -- rotated
// by `shift` (see TargetSchedule::phase), or broadcast when window is 0.
static int predict_subset(dp_engine* e, const int32_t* d_ids, int n, int window, float* dst, int dst_rows, int r0, int shift,
                          cudaStream_t st) {
  if (!e->d_sub_target) {
    const size_t B = (size_t)e->max_clips;
    CK(cudaMalloc(&e->d_sub_latent, B * DP_PAST * DP_L * 4));
    CK(cudaMalloc(&e->d_sub_disp, B * DP_PAST * 3 * 4));
    CK(cudaMalloc(&e->d_sub_height, B * DP_PAST * DP_NH * 4));
    CK(cudaMalloc(&e->d_sub_target, B * (DP_MAX_WINDOW + 1) * DP_L * 4));
  }
  CK(dp_gather_rings_launch(d_ids, n, e->d_latent_buf, e->d_disp_buf, e->d_height_buf, e->d_sub_latent, e->d_sub_disp, e->d_sub_height, st));
  ++e->launches;
  if (int rc = run_predictor(e, e->d_sub_latent, e->d_sub_disp, e->d_sub_height, e->ring_head, n, window, e->d_sub_target, st)) return rc;
  CK(dp_scatter_targets_launch(e->d_sub_target, window + 1, d_ids, n, dst, dst_rows, r0, window, shift, st));
  ++e->launches;
  return DP_OK;
}

// drag_pose.py:237-244: a fresh zero buffer when the window changes, at the index TargetSchedule::index_at gives
static int set_window(dp_engine* e, int W, cudaStream_t st) {
  if (e->sched.target_rows == W + 1) return DP_OK;
  if (int rc = e->sched.check_window_change(W)) return rc;
  drop_prefetch(e);
  CK(cudaMemsetAsync(e->d_target_buf, 0, (size_t)e->n_clips * (W + 1) * DP_L * 4, st));
  e->sched.current_index = e->sched.index_at(W);
  e->sched.target_rows = W + 1;
  return DP_OK;
}

static int run_one(dp_engine* e, const dp_run_params* p, const int32_t* n_ee, const int32_t* joints, const float* weights,
                   int shared, const float* tgt_pos, const float* tgt_rot, int ee_stride, float* out_pose, float* out_gpos,
                   cudaStream_t st) {
  const int W = p->temporal_future_window;
  int rc = set_window(e, W, st);
  if (rc) return rc;
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  if (e->profiling) {
    for (int i = 0; i < 3; ++i) CK(cudaEventCreate(&ev[i]));
    CK(cudaEventRecord(ev[0], st));
  }
  // the predictor call this frame needs first, if any, and the target rows it reads
  TargetSchedule& s = e->sched;
  const int g = s.current_index;
  DpFrameArgs a{};
  if (W == 0) {
    if (s.look_left == 0) {  // targets of this frame and of the next DP_LOOKAHEAD - 1 frames in one call
      rc = run_predictor(e, e->d_latent_buf, e->d_disp_buf, e->d_height_buf, e->ring_head, e->n_clips, 0, e->d_target_pre, st, DP_LOOKAHEAD);
      if (rc) return rc;
      s.look_left = DP_LOOKAHEAD;
    }
    s.look_last_row = DP_LOOKAHEAD - s.look_left--;
    a.target_buf = e->d_target_pre; a.target_rows = DP_LOOKAHEAD; a.target_index = s.look_last_row;
  } else {
    s.look_left = 0;
    s.look_last_row = -1;
    if (s.n_phases > 1) {  // mixed phases: the clips whose own frame 0 this is get their targets, the others keep theirs
      const int n = s.class_start[g + 1] - s.class_start[g];
      if (n > 0 && (rc = predict_subset(e, e->d_class + s.class_start[g], n, W, e->d_target_buf, W + 1, 0, g, st))) return rc;
    } else if (g == 0) {
      if (e->pre_valid) {  // issued three frames ago into the other buffer
        CK(cudaStreamWaitEvent(st, e->ev_pre_done, 0));
        std::swap(e->d_target_buf, e->d_target_alt);
        e->pre_valid = false;
      } else {
        rc = run_predictor(e, e->d_latent_buf, e->d_disp_buf, e->d_height_buf, e->ring_head, e->n_clips, W, e->d_target_buf, st);
        if (rc) return rc;
      }
    } else if (e->prefetch && g == W - 3 && e->n_clips <= DP_PREFETCH_MAX_CLIPS && e->has_temporal && !e->pre_valid) {
      // three frames before the window's first frame: every ring row that frame's predictor call will read is final (frame t-4 is
      // the newest one in the ring, enqueued on st before this point), and it will see the head three slots further on
      CK(cudaEventRecord(e->ev_pre_fork, st));
      CK(cudaStreamWaitEvent(e->pre_stream, e->ev_pre_fork, 0));
      rc = run_predictor(e, e->d_latent_buf, e->d_disp_buf, e->d_height_buf, (e->ring_head + 3) % DP_PAST, e->n_clips, W, e->d_target_alt,
                         e->pre_stream);
      if (rc) return rc;
      CK(cudaEventRecord(e->ev_pre_done, e->pre_stream));
      e->pre_valid = true;
    }
    a.target_buf = e->d_target_buf; a.target_rows = W + 1; a.target_index = g;
  }
  if (e->trace_enabled && (!e->d_trace || e->trace_iters < p->max_iter)) {
    cudaFree(e->d_trace);
    e->d_trace = nullptr;
    CK(cudaMalloc(&e->d_trace, (size_t)e->max_clips * p->max_iter * 52 * 4));
    e->trace_iters = p->max_iter;
  }
  if (e->trace_enabled) CK(cudaMemsetAsync(e->d_trace, 0, (size_t)e->max_clips * e->trace_iters * 52 * 4, st));
  a.model = e->d_model;
  a.model_tc = e->d_model_tc;
  a.model_tmem = e->d_model_tmem;
  a.n_clips = e->n_clips;
  a.latent = e->d_latent; a.gpos = e->d_gpos; a.grot = e->d_grot;
  a.latent_buf = e->d_latent_buf; a.disp_buf = e->d_disp_buf; a.height_buf = e->d_height_buf;
  a.ring_head = e->ring_head;
  a.n_ee = n_ee; a.joints = joints; a.weights = weights; a.shared_trackers = shared;
  a.tgt_pos = tgt_pos; a.tgt_rot = tgt_rot; a.ee_stride = ee_stride;
  a.targets_world = p->targets_world ? 1 : 0;
  a.eps_pos = p->stop_eps_pos; a.eps_rot = p->stop_eps_rot; a.min_incr = p->min_loss_incr;
  a.max_iter = p->max_iter;
  a.lambda_rot = p->lambda_rot; a.lambda_t = p->lambda_temporal;
  a.adj_joint = p->joint_adjust_joint; a.adj_slot = p->joint_adjust_slot; a.adj_w = p->joint_adjust_weight;
  a.adam_tab = e->d_adam;
  a.out_pose = out_pose; a.out_iters = e->d_iters; a.out_losses = e->d_losses;
  if (out_gpos) { a.out_gpos = out_gpos; a.out_pose_stride = DP_POSE; a.out_gpos_stride = 3; }
  else { a.out_gpos = out_pose + DP_POSE; a.out_pose_stride = a.out_gpos_stride = DP_ROW; }  // packed wire rows
  a.trace = e->trace_enabled ? e->d_trace : nullptr;
  a.trace_iters = e->trace_iters;
  a.phase_cycles = e->profiling >= 2 ? e->d_phase : nullptr;
  if (e->profiling) CK(cudaEventRecord(ev[1], st));
  // auto: tensor-core decoder from 512 clips (measured crossover: 0.63 vs 0.66 ms per frame at 512, 0.63 vs 0.39 at 256); the fp32 warp-per-clip
  // kernel is the low-latency path for small batches (B = 1 streaming)
  a.ext_mask = p->extension_losses;
  a.floor_level = p->floor_level;
  const int path = p->extension_losses ? 1 : (p->decoder_path ? p->decoder_path : (e->n_clips >= 512 ? 3 : 1));
  if (path == 3) CK(dp_frame_tc16_launch(a, e->num_sms, st));
  else CK(dp_frame_simt_launch(a, e->num_sms, st));
  e->last_path = path;
  ++e->launches;
  if (e->profiling) {
    CK(cudaEventRecord(ev[2], st));
    for (int i = 0; i < 3; ++i) e->prof_events.push_back(ev[i]);
  }
  e->ring_head = (e->ring_head + 1) % DP_PAST;
  e->sched.advance(W);
  return DP_OK;
}

extern "C" int dp_engine_run_frames_device(dp_engine* e, const dp_run_params* p, int n_frames, const int32_t* n_ee,
                                           const int32_t* joints, const float* weights, int shared, const float* tgt_pos,
                                           const float* tgt_rot, int ee_stride, float* out_pose, float* out_gpos, void* stream) {
  if (!e || !p || !joints || !weights || !tgt_pos || !tgt_rot || !out_pose || n_frames < 1)
    return fail(DP_ERR_ARG, "dp_engine_run_frames_device: null argument");
  int rc = check_params(e, p, ee_stride);
  if (rc) return rc;
  CK(cudaSetDevice(e->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
  rc = ensure_adam(e, p->max_iter, p->learning_rate);
  if (rc) return rc;
  const size_t B = (size_t)e->n_clips, S = (size_t)ee_stride;
  for (int f = 0; f < n_frames; ++f) {
    rc = run_one(e, p, n_ee ? n_ee + f * B : nullptr, shared ? joints : joints + f * B * S,
                 shared ? weights : weights + f * B * S * 2, shared, tgt_pos + f * B * S * 3, tgt_rot + f * B * S * 9,
                 ee_stride, out_pose + f * B * (out_gpos ? DP_POSE : DP_ROW), out_gpos ? out_gpos + f * B * 3 : nullptr, st);
    if (rc) return rc;
  }
  return DP_OK;
}

extern "C" int dp_engine_run_frame_device(dp_engine* e, const dp_run_params* p, const int32_t* n_ee, const int32_t* joints,
                                          const float* weights, int shared, const float* tgt_pos, const float* tgt_rot,
                                          int ee_stride, float* out_pose, float* out_gpos, void* stream) {
  return dp_engine_run_frames_device(e, p, 1, n_ee, joints, weights, shared, tgt_pos, tgt_rot, ee_stride, out_pose,
                                     out_gpos, stream);
}

// Offsets of the per-frame inputs inside one staging block (all 16-byte aligned): n_ee | joints | weights | tgt_pos | tgt_rot
struct PipeLayout {
  size_t nee, joints, w, tp, tr, total;
  PipeLayout(size_t B, size_t S) {
    auto up = [](size_t x) { return (x + 15) & ~size_t(15); };
    nee = 0;
    joints = up(B * 4);
    w = joints + up(B * S * 4);
    tp = w + up(B * S * 8);
    tr = tp + up(B * S * 12);
    total = tr + up(B * S * 36);
  }
};

static int ensure_pipe(dp_engine* e, int ee_stride) {
  if (e->pipe.stride >= ee_stride) return DP_OK;
  free_pipe(e);
  const PipeLayout L((size_t)e->max_clips, (size_t)ee_stride);
  const size_t out_bytes = (size_t)e->max_clips * (DP_POSE + 3) * 4;
  for (int i = 0; i < 2; ++i) {
    CK(cudaMallocHost(&e->pipe.h_in[i], L.total)); CK(cudaMalloc(&e->pipe.d_in[i], L.total));
    CK(cudaMallocHost(&e->pipe.h_out[i], out_bytes)); CK(cudaMalloc(&e->pipe.d_out[i], out_bytes));
    CK(cudaEventCreateWithFlags(&e->pipe.ev_h2d[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&e->pipe.ev_run[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&e->pipe.ev_d2h[i], cudaEventDisableTiming));
  }
  CK(cudaStreamCreateWithFlags(&e->pipe.cs_in, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&e->pipe.cs_out, cudaStreamNonBlocking));
  e->pipe.stride = ee_stride;
  return DP_OK;
}

extern "C" int dp_engine_run_frame_host(dp_engine* e, const dp_run_params* p, const int32_t* n_ee, const int32_t* joints,
                                        const float* weights, int shared, const float* tgt_pos, const float* tgt_rot,
                                        int ee_stride, float* out_pose, float* out_gpos) {
  if (!e || !p || !joints || !weights || !tgt_pos || !tgt_rot || !out_pose || !out_gpos)
    return fail(DP_ERR_ARG, "dp_engine_run_frame_host: null argument");
  int rc = check_params(e, p, ee_stride);
  if (rc) return rc;
  CK(cudaSetDevice(e->device));
  rc = ensure_pipe(e, ee_stride);
  if (rc) return rc;
  rc = ensure_adam(e, p->max_iter, p->learning_rate);
  if (rc) return rc;
  // one contiguous pinned block in, one out: a single copy each way (this is the B = 1 latency path of the DLL)
  dp_engine::FramePipe& P = e->pipe;
  cudaStream_t st = e->stream;
  const size_t B = (size_t)e->n_clips, S = (size_t)ee_stride;
  const size_t nj = shared ? S : B * S;
  const PipeLayout L((size_t)e->max_clips, (size_t)P.stride);
  unsigned char* h = P.h_in[0];
  if ((rc = check_n_ee(n_ee, B, ee_stride, p)) != DP_OK) return rc;
  if (n_ee) memcpy(h + L.nee, n_ee, B * 4);
  memcpy(h + L.joints, joints, nj * 4);
  memcpy(h + L.w, weights, nj * 8);
  memcpy(h + L.tp, tgt_pos, B * S * 12);
  memcpy(h + L.tr, tgt_rot, B * S * 36);
  // only the used prefix of every section travels when the batch is small: copy up to the end of the last section in use
  const size_t in_bytes = B == (size_t)e->max_clips ? L.total : L.tr + B * S * 36;
  CK(cudaMemcpyAsync(P.d_in[0], h, in_bytes, cudaMemcpyHostToDevice, st));
  unsigned char* d = P.d_in[0];
  float* d_pose = P.d_out[0];
  rc = run_one(e, p, n_ee ? reinterpret_cast<const int32_t*>(d + L.nee) : nullptr, reinterpret_cast<const int32_t*>(d + L.joints),
               reinterpret_cast<const float*>(d + L.w), shared, reinterpret_cast<const float*>(d + L.tp),
               reinterpret_cast<const float*>(d + L.tr), ee_stride, d_pose, d_pose + B * DP_POSE, st);
  if (rc) return rc;
  CK(cudaMemcpyAsync(P.h_out[0], d_pose, B * (DP_POSE + 3) * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  memcpy(out_pose, P.h_out[0], B * DP_POSE * 4);
  memcpy(out_gpos, P.h_out[0] + B * DP_POSE, B * 3 * 4);
  return DP_OK;
}

extern "C" int dp_engine_run_frames_host(dp_engine* e, const dp_run_params* p, int n_frames, const int32_t* n_ee, const int32_t* joints,
                                         const float* weights, int shared, const float* tgt_pos, const float* tgt_rot, int ee_stride,
                                         float* out_pose, float* out_gpos) {
  if (!e || !p || !joints || !weights || !tgt_pos || !tgt_rot || !out_pose || !out_gpos || n_frames < 0)
    return fail(DP_ERR_ARG, "dp_engine_run_frames_host: null argument");
  int rc = check_params(e, p, ee_stride);
  if (rc) return rc;
  CK(cudaSetDevice(e->device));
  rc = ensure_pipe(e, ee_stride);
  if (rc) return rc;
  if ((rc = check_n_ee(n_ee, (size_t)n_frames * (size_t)e->n_clips, ee_stride, p)) != DP_OK) return rc;
  rc = ensure_adam(e, p->max_iter, p->learning_rate);
  if (rc) return rc;
  dp_engine::FramePipe& P = e->pipe;
  cudaStream_t st = e->stream;
  const size_t B = (size_t)e->n_clips, S = (size_t)ee_stride;
  const size_t nj = shared ? S : B * S;
  const PipeLayout L((size_t)e->max_clips, (size_t)P.stride);
  const size_t out_bytes = B * (DP_POSE + 3) * 4;
  static const bool pipe_trace = getenv("DP_PIPE_TRACE") != nullptr;  // debug: host-side time per pipeline stage
  double t_stage = 0, t_enq = 0, t_wait = 0, t_unstage = 0;
  auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  auto unstage = [&](int t) -> int {  // frame t's results: pinned slot -> caller's arrays
    const int slot = t & 1;
    const double w0 = now();
    CK(cudaEventSynchronize(P.ev_d2h[slot]));
    const double w1 = now();
    t_wait += w1 - w0;
    memcpy(out_pose + (size_t)t * B * DP_POSE, P.h_out[slot], B * DP_POSE * 4);
    memcpy(out_gpos + (size_t)t * B * 3, P.h_out[slot] + B * DP_POSE, B * 3 * 4);
    t_unstage += now() - w1;
    return DP_OK;
  };
  for (int t = 0; t < n_frames; ++t) {
    const int slot = t & 1;
    // (1) stage frame t's inputs while the device works on frame t-1
    const double s0 = now();
    if (t >= 2) CK(cudaEventSynchronize(P.ev_h2d[slot]));  // the pinned block was last read by the copy of frame t-2
    unsigned char* h = P.h_in[slot];
    if (n_ee) memcpy(h + L.nee, n_ee + (size_t)t * B, B * 4);
    memcpy(h + L.joints, joints + (shared ? 0 : (size_t)t * nj), nj * 4);
    memcpy(h + L.w, weights + (shared ? 0 : (size_t)t * nj * 2), nj * 8);
    memcpy(h + L.tp, tgt_pos + (size_t)t * B * S * 3, B * S * 12);
    memcpy(h + L.tr, tgt_rot + (size_t)t * B * S * 9, B * S * 36);
    const double s1 = now();
    t_stage += s1 - s0;
    // (2) copy in on its own stream (after frame t-2 has finished reading this device block), run, copy out on a third stream
    if (t >= 2) CK(cudaStreamWaitEvent(P.cs_in, P.ev_run[slot], 0));
    CK(cudaMemcpyAsync(P.d_in[slot], h, L.total, cudaMemcpyHostToDevice, P.cs_in));
    CK(cudaEventRecord(P.ev_h2d[slot], P.cs_in));
    CK(cudaStreamWaitEvent(st, P.ev_h2d[slot], 0));
    if (t >= 2) CK(cudaStreamWaitEvent(st, P.ev_d2h[slot], 0));  // frame t-2's results have left this device block
    unsigned char* d = P.d_in[slot];
    float* d_pose = P.d_out[slot];
    rc = run_one(e, p, n_ee ? reinterpret_cast<const int32_t*>(d + L.nee) : nullptr, reinterpret_cast<const int32_t*>(d + L.joints),
                 reinterpret_cast<const float*>(d + L.w), shared, reinterpret_cast<const float*>(d + L.tp),
                 reinterpret_cast<const float*>(d + L.tr), ee_stride, d_pose, d_pose + B * DP_POSE, st);
    if (rc) { cudaDeviceSynchronize(); return rc; }
    CK(cudaEventRecord(P.ev_run[slot], st));
    CK(cudaStreamWaitEvent(P.cs_out, P.ev_run[slot], 0));
    CK(cudaMemcpyAsync(P.h_out[slot], d_pose, out_bytes, cudaMemcpyDeviceToHost, P.cs_out));
    CK(cudaEventRecord(P.ev_d2h[slot], P.cs_out));
    t_enq += now() - s1;
    // (3) hand frame t-1's results to the caller
    if (t >= 1) { rc = unstage(t - 1); if (rc) return rc; }
  }
  if (n_frames >= 1) { rc = unstage(n_frames - 1); if (rc) return rc; }
  CK(cudaStreamSynchronize(st));
  if (pipe_trace && n_frames > 0)
    fprintf(stderr, "run_frames_host: %d frames, host ms per frame: stage %.3f, enqueue %.3f, wait for device %.3f, unstage %.3f\n", n_frames,
            t_stage / n_frames, t_enq / n_frames, t_wait / n_frames, t_unstage / n_frames);
  return DP_OK;
}

extern "C" int dp_engine_set_encoder_model(dp_engine* e, const dp_encoder_model* m) {
  if (!e || !m || !m->A0 || !m->b0 || !m->A1 || !m->b1 || !m->A2 || !m->b2 || !m->mu_w || !m->mu_b || !m->logvar_w || !m->logvar_b)
    return fail(DP_ERR_ARG, "dp_engine_set_encoder_model: null argument");
  CK(cudaSetDevice(e->device));
  std::vector<float> blob;
  blob.reserve(DP_ENC_BLOB_FLOATS);
  auto layer = [&](const float* W, const float* b, int out, int in) {  // transposed to [in][out]
    for (int i = 0; i < in; ++i)
      for (int o = 0; o < out; ++o) blob.push_back(W[(size_t)o * in + i]);
    blob.insert(blob.end(), b, b + out);
  };
  layer(m->A0, m->b0, DP_ENC_H0, DP_ENC_IN);
  layer(m->A1, m->b1, DP_ENC_H1, DP_ENC_H0);
  layer(m->A2, m->b2, DP_ENC_H2, DP_ENC_H1);
  for (int i = 0; i < DP_ENC_H2; ++i) {  // heads side by side: columns 0..23 mu, 24..47 logvar
    for (int o = 0; o < DP_L; ++o) blob.push_back(m->mu_w[(size_t)o * DP_ENC_H2 + i]);
    for (int o = 0; o < DP_L; ++o) blob.push_back(m->logvar_w[(size_t)o * DP_ENC_H2 + i]);
  }
  blob.insert(blob.end(), m->mu_b, m->mu_b + DP_L);
  blob.insert(blob.end(), m->logvar_b, m->logvar_b + DP_L);
  if (blob.size() != DP_ENC_BLOB_FLOATS) return fail(DP_ERR_STATE, "encoder blob layout");
  if (!e->d_encoder) CK(cudaMalloc(&e->d_encoder, blob.size() * 4));
  CK(cudaMemcpy(e->d_encoder, blob.data(), blob.size() * 4, cudaMemcpyHostToDevice));
  return DP_OK;
}

extern "C" int dp_engine_encode_host(dp_engine* e, int n, const float* dqs, const float* eps, float* latent) {
  if (!e || !dqs || !latent || n < 1) return fail(DP_ERR_ARG, "dp_engine_encode_host: null argument");
  if (!e->d_encoder) return fail(DP_ERR_STATE, "encoder model not set");
  if (n > e->max_clips) return fail(DP_ERR_ARG, "dp_engine_encode_host: more poses than max_clips");
  CK(cudaSetDevice(e->device));
  float *d_dqs = nullptr, *d_eps = nullptr, *d_lat = nullptr;
  CK(cudaMalloc(&d_dqs, (size_t)n * DP_ENC_IN * 4));
  CK(cudaMalloc(&d_lat, (size_t)n * DP_L * 4));
  CK(cudaMemcpyAsync(d_dqs, dqs, (size_t)n * DP_ENC_IN * 4, cudaMemcpyHostToDevice, e->stream));
  if (eps) {
    CK(cudaMalloc(&d_eps, (size_t)n * DP_L * 4));
    CK(cudaMemcpyAsync(d_eps, eps, (size_t)n * DP_L * 4, cudaMemcpyHostToDevice, e->stream));
  }
  CK(dp_encode_launch(e->d_encoder, d_dqs, d_eps, d_lat, n, e->stream));
  ++e->launches;
  CK(cudaMemcpyAsync(latent, d_lat, (size_t)n * DP_L * 4, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  cudaFree(d_dqs); cudaFree(d_eps); cudaFree(d_lat);
  return DP_OK;
}

extern "C" int dp_engine_pose_error_host(dp_engine* e, int n, const float* pose_a, const float* pose_b, float* err) {
  if (!e || !pose_a || !pose_b || !err || n < 1) return fail(DP_ERR_ARG, "dp_engine_pose_error_host: null argument");
  if (!e->has_pose) return fail(DP_ERR_STATE, "pose model not set");
  CK(cudaSetDevice(e->device));
  float *d_a = nullptr, *d_b = nullptr, *d_e = nullptr;
  const size_t bytes = (size_t)n * DP_POSE * 4;
  CK(cudaMalloc(&d_a, bytes)); CK(cudaMalloc(&d_b, bytes)); CK(cudaMalloc(&d_e, (size_t)n * 8));
  CK(cudaMemcpyAsync(d_a, pose_a, bytes, cudaMemcpyHostToDevice, e->stream));
  CK(cudaMemcpyAsync(d_b, pose_b, bytes, cudaMemcpyHostToDevice, e->stream));
  CK(dp_pose_error_launch(e->d_model, d_a, d_b, n, d_e, e->stream));
  ++e->launches;
  CK(cudaMemcpyAsync(err, d_e, (size_t)n * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  cudaFree(d_a); cudaFree(d_b); cudaFree(d_e);
  return DP_OK;
}

extern "C" int dp_engine_get_frame_stats(dp_engine* e, int32_t* iters, float* losses) {
  if (!e) return fail(DP_ERR_ARG, "null engine");
  CK(cudaSetDevice(e->device));
  CK(cudaStreamSynchronize(e->stream));
  CK(cudaDeviceSynchronize());
  if (iters) CK(cudaMemcpy(iters, e->d_iters, (size_t)e->n_clips * 4, cudaMemcpyDeviceToHost));
  if (losses) CK(cudaMemcpy(losses, e->d_losses, (size_t)e->n_clips * 3 * 4, cudaMemcpyDeviceToHost));
  return DP_OK;
}

extern "C" int dp_engine_enable_trace(dp_engine* e, int enable) {
  if (!e) return fail(DP_ERR_ARG, "null engine");
  e->trace_enabled = enable ? 1 : 0;
  return DP_OK;
}

extern "C" int dp_engine_get_trace(dp_engine* e, float* rows, int max_iter) {
  if (!e || !rows) return fail(DP_ERR_ARG, "null argument");
  if (!e->d_trace || max_iter > e->trace_iters) return fail(DP_ERR_STATE, "no trace recorded for that many iterations");
  CK(cudaSetDevice(e->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy2D(rows, (size_t)max_iter * 52 * 4, e->d_trace, (size_t)e->trace_iters * 52 * 4, (size_t)max_iter * 52 * 4,
                  e->n_clips, cudaMemcpyDeviceToHost));
  return DP_OK;
}

extern "C" int dp_engine_eval_gradient(dp_engine* e, int n, const float* latents, const float* grot, const float* tgt_latent,
                                       const int32_t* n_ee, const int32_t* joints, const float* weights, int shared,
                                       const float* tgt_pos, const float* tgt_rot, int ee_stride, float lambda_rot,
                                       float lambda_temporal, int decoder_path, float* grad, float* losses, float* positions,
                                       int extension_losses, float floor_level, const float* global_pos) {
  if (!e || !latents || !grot || !tgt_latent || !joints || !weights || !tgt_pos || !tgt_rot || n < 1)
    return fail(DP_ERR_ARG, "dp_engine_eval_gradient: null argument");
  if (!e->has_pose) return fail(DP_ERR_STATE, "pose model not set");
  if (ee_stride < 1 || ee_stride > DP_JOINTS) return fail(DP_ERR_ARG, "ee_stride out of range");
  if (int rcn = check_n_ee(n_ee, (size_t)n, ee_stride, nullptr)) return rcn;
  if (extension_losses < 0 || extension_losses > 15) return fail(DP_ERR_ARG, "extension_losses must be a mask of DP_EXT_* bits");
  if (extension_losses && decoder_path == 3) return fail(DP_ERR_UNSUPPORTED, "the extension losses run on the fp32 CUDA-core frame kernel");
  CK(cudaSetDevice(e->device));
  CK(cudaDeviceSynchronize());
  const size_t N = (size_t)n, S = (size_t)ee_stride, nj = shared ? S : N * S;
  float *d_lat, *d_g, *d_t, *d_w, *d_tp, *d_tr, *d_grad, *d_loss, *d_pos, *d_adam;
  int32_t *d_ne = nullptr, *d_j;
  CK(cudaMalloc(&d_lat, N * DP_L * 4)); CK(cudaMalloc(&d_g, N * 16)); CK(cudaMalloc(&d_t, N * DP_L * 4));
  CK(cudaMalloc(&d_j, nj * 4)); CK(cudaMalloc(&d_w, nj * 8)); CK(cudaMalloc(&d_tp, N * S * 12)); CK(cudaMalloc(&d_tr, N * S * 36));
  CK(cudaMalloc(&d_grad, N * DP_L * 4)); CK(cudaMalloc(&d_loss, N * 12)); CK(cudaMalloc(&d_pos, N * DP_J * 12));
  CK(cudaMalloc(&d_adam, 8));
  if (n_ee) { CK(cudaMalloc(&d_ne, N * 4)); CK(cudaMemcpy(d_ne, n_ee, N * 4, cudaMemcpyHostToDevice)); }
  float* d_gp = nullptr;
  if (extension_losses) {
    CK(cudaMalloc(&d_gp, N * 12));
    if (global_pos) CK(cudaMemcpy(d_gp, global_pos, N * 12, cudaMemcpyHostToDevice));
    else CK(cudaMemset(d_gp, 0, N * 12));
  }
  CK(cudaMemcpy(d_lat, latents, N * DP_L * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_g, grot, N * 16, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_t, tgt_latent, N * DP_L * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_j, joints, nj * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_w, weights, nj * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_tp, tgt_pos, N * S * 12, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_tr, tgt_rot, N * S * 36, cudaMemcpyHostToDevice));
  CK(cudaMemset(d_adam, 0, 8));
  DpFrameArgs a{};
  a.model = e->d_model; a.model_tc = e->d_model_tc; a.model_tmem = e->d_model_tmem; a.n_clips = n; a.latent = d_lat; a.grot = d_g;
  a.target_buf = d_t; a.target_rows = 1; a.target_index = 0;
  a.n_ee = d_ne; a.joints = d_j; a.weights = d_w; a.shared_trackers = shared; a.tgt_pos = d_tp; a.tgt_rot = d_tr;
  a.ee_stride = ee_stride;
  a.eps_pos = -1.0; a.eps_rot = -1.0; a.min_incr = -std::numeric_limits<double>::infinity();
  a.max_iter = 1; a.lambda_rot = lambda_rot; a.lambda_t = lambda_temporal; a.adj_joint = -1;
  a.adam_tab = d_adam; a.out_losses = d_loss; a.eval_only = 1; a.eval_grad = d_grad; a.eval_pos = d_pos;
  a.gpos = d_gp; a.ext_mask = extension_losses; a.floor_level = floor_level;
  if (decoder_path == 3) CK(dp_frame_tc16_launch(a, e->num_sms, e->stream));
  else CK(dp_frame_simt_launch(a, e->num_sms, e->stream));
  ++e->launches;
  CK(cudaStreamSynchronize(e->stream));
  if (grad) CK(cudaMemcpy(grad, d_grad, N * DP_L * 4, cudaMemcpyDeviceToHost));
  if (losses) CK(cudaMemcpy(losses, d_loss, N * 12, cudaMemcpyDeviceToHost));
  if (positions) CK(cudaMemcpy(positions, d_pos, N * DP_J * 12, cudaMemcpyDeviceToHost));
  cudaFree(d_lat); cudaFree(d_g); cudaFree(d_t); cudaFree(d_j); cudaFree(d_w); cudaFree(d_tp); cudaFree(d_tr);
  cudaFree(d_grad); cudaFree(d_loss); cudaFree(d_pos); cudaFree(d_adam); cudaFree(d_ne); cudaFree(d_gp);
  return DP_OK;
}

static int copy_ring(dp_engine* e, const float* d_src, float* h_dst, int width) {
  // device ring (slot order) -> host chronological order
  const size_t B = (size_t)e->n_clips;
  std::vector<float> tmp(B * DP_PAST * width);
  CK(cudaMemcpy(tmp.data(), d_src, tmp.size() * 4, cudaMemcpyDeviceToHost));
  for (size_t c = 0; c < B; ++c)
    for (int r = 0; r < DP_PAST; ++r)
      memcpy(h_dst + (c * DP_PAST + r) * width, &tmp[(c * DP_PAST + (e->ring_head + r) % DP_PAST) * width], (size_t)width * 4);
  return DP_OK;
}

extern "C" int dp_engine_get_state(dp_engine* e, float* latent, float* gpos, float* grot, float* latent_buf, float* disp_buf,
                                   float* height_buf, float* target_buf, int* current_index) {
  if (!e) return fail(DP_ERR_ARG, "null engine");
  if (e->n_clips <= 0) return fail(DP_ERR_STATE, "no clips initialised");
  CK(cudaSetDevice(e->device));
  CK(cudaDeviceSynchronize());
  const size_t B = (size_t)e->n_clips;
  if (latent) CK(cudaMemcpy(latent, e->d_latent, B * DP_L * 4, cudaMemcpyDeviceToHost));
  if (gpos) CK(cudaMemcpy(gpos, e->d_gpos, B * 12, cudaMemcpyDeviceToHost));
  if (grot) CK(cudaMemcpy(grot, e->d_grot, B * 16, cudaMemcpyDeviceToHost));
  int rc;
  if (latent_buf && (rc = copy_ring(e, e->d_latent_buf, latent_buf, DP_L))) return rc;
  if (disp_buf && (rc = copy_ring(e, e->d_disp_buf, disp_buf, 3))) return rc;
  if (height_buf && (rc = copy_ring(e, e->d_height_buf, height_buf, DP_NH))) return rc;
  const TargetSchedule& s = e->sched;
  if (target_buf) {
    if (s.target_rows <= 0) return fail(DP_ERR_STATE, "no target buffer yet");
    if (s.look_last_row >= 0)  // window 0 with look-ahead: the row the last frame used, as (B,1,24)
      CK(cudaMemcpy2D(target_buf, DP_L * 4, e->d_target_pre + (size_t)s.look_last_row * DP_L, (size_t)DP_LOOKAHEAD * DP_L * 4, DP_L * 4, B,
                      cudaMemcpyDeviceToHost));
    else
      CK(cudaMemcpy(target_buf, e->d_target_buf, B * s.target_rows * DP_L * 4, cudaMemcpyDeviceToHost));
    if (s.n_phases > 1 && s.look_last_row < 0) {  // rotated rows (TargetSchedule::phase) -> each clip's own row order
      const int W = s.target_rows - 1;
      for (size_t c = 0; c < B; ++c) {  // own row k moves from slot(c, k) to k: rows [0, W) rotate left by slot(c, 0)
        float* rows = target_buf + c * s.target_rows * DP_L;
        std::rotate(rows, rows + (size_t)s.slot((int)c, 0, W) * DP_L, rows + (size_t)W * DP_L);
      }
    }
  }
  if (current_index) *current_index = s.current_index;
  return DP_OK;
}

extern "C" int dp_engine_set_ring_buffers(dp_engine* e, const float* latent_buf, const float* disp_buf, const float* height_buf) {
  if (!e || !latent_buf || !disp_buf || !height_buf) return fail(DP_ERR_ARG, "null argument");
  if (e->n_clips <= 0) return fail(DP_ERR_STATE, "no clips initialised");
  CK(cudaSetDevice(e->device));
  CK(cudaDeviceSynchronize());
  const size_t B = (size_t)e->n_clips;
  CK(cudaMemcpy(e->d_latent_buf, latent_buf, B * DP_PAST * DP_L * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(e->d_disp_buf, disp_buf, B * DP_PAST * 3 * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(e->d_height_buf, height_buf, B * DP_PAST * DP_NH * 4, cudaMemcpyHostToDevice));
  e->ring_head = 0;  // rows were given in chronological order
  void_targets_ahead(e);
  return DP_OK;
}

extern "C" int dp_engine_predict_targets(dp_engine* e, int window, void* stream) {
  if (!e) return fail(DP_ERR_ARG, "null engine");
  if (!e->has_temporal) return fail(DP_ERR_STATE, "temporal model not set");
  if (e->n_clips <= 0) return fail(DP_ERR_STATE, "no clips initialised");
  if (int rc = check_window(window)) return rc;
  if (e->sched.n_phases > 1)
    return fail(DP_ERR_STATE, "dp_engine_predict_targets: restarted clips run at their own predictor phase (it predicts every clip at once)");
  CK(cudaSetDevice(e->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
  if (int rc = set_window(e, window, st)) return rc;
  e->sched.look_last_row = -1;  // dp_engine_get_state reports what this call writes
  return run_predictor(e, e->d_latent_buf, e->d_disp_buf, e->d_height_buf, e->ring_head, e->n_clips, window, e->d_target_buf, st);
}

extern "C" int dp_engine_set_profiling(dp_engine* e, int enable) {
  if (!e) return fail(DP_ERR_ARG, "null engine");
  CK(cudaSetDevice(e->device));
  CK(cudaDeviceSynchronize());
  for (cudaEvent_t ev : e->prof_events) cudaEventDestroy(ev);
  e->prof_events.clear();
  e->profiling = enable < 0 ? 0 : (enable > 2 ? 2 : enable);
  if (enable >= 2) {
    if (!e->d_phase) CK(cudaMalloc(&e->d_phase, 64 * sizeof(unsigned long long)));
    CK(cudaMemset(e->d_phase, 0, 64 * sizeof(unsigned long long)));
  }
  return DP_OK;
}

extern "C" int dp_engine_get_phase_cycles(dp_engine* e, unsigned long long* cycles8) {
  if (!e || !cycles8) return fail(DP_ERR_ARG, "null argument");
  if (!e->d_phase) return fail(DP_ERR_STATE, "profiling was never enabled");
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(cycles8, e->d_phase, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return DP_OK;
}

extern "C" int dp_engine_get_timeline(dp_engine* e, unsigned long long* stamps48) {
  if (!e || !stamps48) return fail(DP_ERR_ARG, "null argument");
  if (!e->d_phase) return fail(DP_ERR_STATE, "profiling was never enabled");
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(stamps48, e->d_phase + 16, 48 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return DP_OK;
}

extern "C" int dp_engine_get_profile(dp_engine* e, double* ms_predictor, double* ms_frame_kernel, long long* n_frames) {
  if (!e) return fail(DP_ERR_ARG, "null engine");
  CK(cudaSetDevice(e->device));
  CK(cudaDeviceSynchronize());
  double tp = 0.0, tf = 0.0;
  for (size_t i = 0; i + 2 < e->prof_events.size(); i += 3) {
    float a = 0.f, b = 0.f;
    CK(cudaEventElapsedTime(&a, e->prof_events[i], e->prof_events[i + 1]));
    CK(cudaEventElapsedTime(&b, e->prof_events[i + 1], e->prof_events[i + 2]));
    tp += a;
    tf += b;
  }
  if (ms_predictor) *ms_predictor = tp;
  if (ms_frame_kernel) *ms_frame_kernel = tf;
  if (n_frames) *n_frames = (long long)(e->prof_events.size() / 3);
  return DP_OK;
}

extern "C" int dp_engine_set_predictor_path(dp_engine* e, int path) {
  if (!e || path < 0 || path > 1) return fail(DP_ERR_ARG, "predictor path must be 0 (tcgen05 fp16x2 attention + FF) or 1 (fp32 CUDA-core kernels)");
  e->predictor_path = path;
  void_targets_ahead(e);
  return DP_OK;
}

extern "C" int dp_engine_last_decoder_path(const dp_engine* e) { return e ? e->last_path : 0; }

extern "C" int dp_engine_restart_clips(dp_engine* e, int n, const int32_t* clips, const float* latent0, const float* gpos,
                                       const float* grot, const float* heights, void* stream) {
  if (!e || !clips || !latent0 || !gpos || !grot || !heights) return fail(DP_ERR_ARG, "dp_engine_restart_clips: null argument");
  if (e->n_clips <= 0) return fail(DP_ERR_STATE, "dp_engine_restart_clips: no clips initialised (dp_engine_init_clips)");
  if (n < 1 || n > e->n_clips) return fail(DP_ERR_ARG, "dp_engine_restart_clips: n out of range");
  const int B = e->n_clips;
  std::vector<char> seen(B, 0);
  for (int i = 0; i < n; ++i) {
    if (clips[i] < 0 || clips[i] >= B) return fail(DP_ERR_ARG, "dp_engine_restart_clips: clip id out of range");
    if (seen[clips[i]]) return fail(DP_ERR_ARG, "dp_engine_restart_clips: duplicate clip id");
    seen[clips[i]] = 1;
  }
  CK(cudaSetDevice(e->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
  const size_t cap = (size_t)e->max_clips;
  if (!e->h_restart) {
    const size_t bytes = cap * (8 + DP_RESTART_STATE * 4);
    CK(cudaMallocHost(&e->h_restart, bytes));
    CK(cudaMalloc(&e->d_restart, bytes));
    CK(cudaEventCreateWithFlags(&e->ev_restart, cudaEventDisableTiming));
    e->d_class = reinterpret_cast<int32_t*>(e->d_restart + cap * 4);
  }
  if (e->restart_pending) CK(cudaEventSynchronize(e->ev_restart));  // the previous restart's copies have left the pinned block
  e->restart_pending = false;
  drop_prefetch(e);  // targets computed ahead from the restarted clips' old rows are void
  // Each restarted clip's next frame is its own frame 0, i.e. its phase is the index the next frame runs at.
  TargetSchedule& sc = e->sched;
  const int g = sc.current_index;
  std::vector<int> phase = sc.phase;
  for (int i = 0; i < n; ++i) phase[clips[i]] = g;
  std::vector<int> count(DP_MAX_WINDOW + 1, 0);
  int distinct = 0;
  for (int c = 0; c < B; ++c) distinct += count[phase[c]]++ == 0;
  int32_t* h_ids = reinterpret_cast<int32_t*>(e->h_restart);
  int32_t* h_class = h_ids + cap;
  float* h_state = reinterpret_cast<float*>(e->h_restart + cap * 8);
  memcpy(h_ids, clips, (size_t)n * 4);
  for (int i = 0; i < n; ++i) {
    float* s = h_state + (size_t)i * DP_RESTART_STATE;
    memcpy(s, latent0 + (size_t)i * DP_L, DP_L * 4);
    memcpy(s + DP_L, gpos + (size_t)i * 3, 12);
    memcpy(s + DP_L + 3, grot + (size_t)i * 4, 16);
    memcpy(s + DP_L + 7, heights + (size_t)i * DP_NH, DP_NH * 4);
  }
  std::vector<int> start(DP_MAX_WINDOW + 2, 0);
  if (distinct > 1) {  // clip ids grouped by phase, ascending within a phase (a counting sort)
    for (int s = 0; s <= DP_MAX_WINDOW; ++s) start[s + 1] = start[s] + count[s];
    std::vector<int> at(start.begin(), start.end() - 1);
    for (int c = 0; c < B; ++c) h_class[at[phase[c]]++] = c;
  }
  CK(cudaMemcpyAsync(e->d_restart, h_ids, (size_t)n * 4, cudaMemcpyHostToDevice, st));
  if (distinct > 1) CK(cudaMemcpyAsync(e->d_class, h_class, (size_t)B * 4, cudaMemcpyHostToDevice, st));
  float* d_state = reinterpret_cast<float*>(e->d_restart + cap * 8);
  CK(cudaMemcpyAsync(d_state, h_state, (size_t)n * DP_RESTART_STATE * 4, cudaMemcpyHostToDevice, st));
  CK(cudaEventRecord(e->ev_restart, st));
  e->restart_pending = true;
  const int32_t* d_ids = reinterpret_cast<const int32_t*>(e->d_restart);
  CK(dp_reset_clips_launch(d_ids, d_state, n, e->d_latent, e->d_gpos, e->d_grot, e->d_latent_buf, e->d_disp_buf, e->d_height_buf, st));
  ++e->launches;
  if (sc.target_rows == 1 && sc.look_left > 0) {
    // Window 0 between look-ahead boundaries: the restarted clips need targets for the rest of the current four-frame cycle.  What
    // the predictor reads at their own frames 0..3 (chronological ring rows <= 56) is all initial rows, so one single-view call on
    // them, broadcast into the rows from DP_LOOKAHEAD - look_left to 3, is what the reference computes frame by frame.
    const int rc = predict_subset(e, d_ids, n, 0, e->d_target_pre, DP_LOOKAHEAD, DP_LOOKAHEAD - sc.look_left, 0, st);
    if (rc) return rc;
  }
  if (distinct == 1) {  // one phase for every clip: fold it into current_index (lockstep path, prefetch and graph replay stay on)
    std::fill(sc.phase.begin(), sc.phase.end(), 0);
    sc.current_index = 0;  // that phase is g: every clip starts its own window at the next frame
  } else {
    sc.phase = phase;
    sc.class_start = start;
  }
  sc.n_phases = distinct;
  return DP_OK;
}

extern "C" int dp_engine_get_clip_index(dp_engine* e, int window, int32_t* index) {
  if (!e || !index) return fail(DP_ERR_ARG, "dp_engine_get_clip_index: null argument");
  if (int rc = check_window(window)) return rc;
  if (e->n_clips <= 0) return fail(DP_ERR_STATE, "no clips initialised");
  if (int rc = e->sched.check_window_change(window)) return rc;
  for (int c = 0; c < e->n_clips; ++c) index[c] = e->sched.clip_index(c, window);
  return DP_OK;
}

extern "C" int dp_engine_frames_to_boundary(const dp_engine* e, int window) {
  if (!e) return fail(DP_ERR_ARG, "null engine");
  if (int rc = check_window(window)) return rc;
  if (e->n_clips <= 0) return fail(DP_ERR_STATE, "no clips initialised");
  if (int rc = e->sched.check_window_change(window)) return rc;
  return e->sched.frames_to_boundary(window);
}
