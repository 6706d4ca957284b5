// dp_common.cuh -- shared definitions of the B200 DragPoser engine kernels.
//
// Model image: one contiguous, 16-byte aligned block in HBM that every CTA pulls into
// shared memory with a single bulk-TMA copy (cp.async.bulk, UBLKCP in SASS) and keeps
// resident for the whole frame.  Layout of the folded decoder (reference:
// python/src/autoencoder.py:224-256 folded to 24->40->60->92, see dragposer_b200/model.py):
//   W?t  forward operand,  [k][o]  (lanes own consecutive outputs -> conflict-free LDS.64)
//   W?   backward operand, [o][k]  (same access pattern with the roles swapped)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define DP_J 22
#define DP_L 24
// folded encoder widths (autoencoder.py:136-143 folded): 176 -> 112 -> 72 -> 48 -> (mu 24 | logvar 24)
#define DP_ENC_IN 176
#define DP_ENC_H0 112
#define DP_ENC_H1 72
#define DP_ENC_H2 48
#define DP_ENC_BLOB_FLOATS (DP_ENC_IN * DP_ENC_H0 + DP_ENC_H0 + DP_ENC_H0 * DP_ENC_H1 + DP_ENC_H1 + DP_ENC_H1 * DP_ENC_H2 + DP_ENC_H2 + DP_ENC_H2 * 48 + 48)
#define DP_H0 40
#define DP_H1 60
#define DP_Y 92
#define DP_PAST 60
#define DP_NH 6
#define DP_MAX_CHILD 4
#define DP_JUMP_ROUNDS 4
#define DP_SCRATCH 96  // floats per ping/pong activation buffer

struct __align__(16) DpModelImage {
  float W0t[DP_L * DP_H0];
  float W1t[DP_H0 * DP_H1];
  float W2t[DP_H1 * DP_Y];
  float W0[DP_H0 * DP_L];
  float W1[DP_H1 * DP_H0];
  float W2[DP_Y * DP_H1];
  float b0[DP_H0];
  float b1[DP_H1];
  float b2[DP_Y];
  float mean_q[DP_J * 4];
  float std_q[DP_J * 4];
  float mean_d[4];
  float std_d[4];
  float off[32][4];                    // offset of joint j
  float coff[DP_MAX_CHILD][32][4];     // offsets of the children of joint j
  int32_t child[DP_MAX_CHILD][32];     // child joints of j or -1
  int32_t jump[DP_JUMP_ROUNDS][32];    // ancestor of j at distance 1,2,4,8 or -1
  int32_t parent[32];
  int32_t last[32];                    // last joint of j's (preorder-contiguous) subtree
  int32_t height_slot[32];             // slot in the heights vector or -1
  int32_t pad[32];
};
static_assert(sizeof(DpModelImage) % 16 == 0, "bulk copy needs a multiple of 16 bytes");

// Table image of the tcgen05 frame kernel (biases, statistics, skeleton tables; one bulk-TMA copy per CTA).  Its weights do not
// live here: they are fp16x2 pieces in TENSOR memory, loaded from the [word][lane] image described below.
struct __align__(16) DpModelImageTC {
  float b0[DP_H0];
  float b1[DP_H1];
  float b2[DP_Y];
  float mean_q[DP_J * 4];
  float std_q[DP_J * 4];
  float mean_d[4];
  float std_d[4];
  float off[32][4];
  float coff[DP_MAX_CHILD][32][4];
  int32_t child[DP_MAX_CHILD][32];
  int32_t jump[DP_JUMP_ROUNDS][32];
  int32_t parent[32];
  int32_t last[32];
  int32_t height_slot[32];
  int32_t pad[32];
};
// fp16x2 weights for the tensor-memory-resident kernel (dp_frame_tc16.cu): 352 32-bit words per TMEM lane, image [word][128 lanes]
#define DP_TC_TMEM_WORDS 352
static_assert(sizeof(DpModelImageTC) % 16 == 0, "bulk copy needs a multiple of 16 bytes");

// A clip's optimiser settings (dp_clip_settings, include/dp_engine.h) with the Adam step table of its learning rate.  With a
// per-clip table the tcgen05 kernel copies each clip's entry to shared memory once per frame and reads it from there: the kernel has
// no registers to spare for three doubles per clip.
struct DpClipSetting {
  double eps_pos, eps_rot, min_incr;
  const float* adam_tab;  // [2][max_iter]: lr/(1-b1^k), 1/sqrt(1-b2^k), k = 1..max_iter; readable up to index max_iter + the
                          // launch's max_iter (per-clip tables are padded: a stopped clip's warp still reads them, unused)
  int max_iter;
  float lambda_rot, lambda_t;
  int adj_joint, adj_slot;
  float adj_w;
};
static_assert(sizeof(DpClipSetting) == 56, "copied as seven 8-byte words");
// lanes 0..6 of a warp copy the entry; the caller synchronises the warp before another lane reads it
__device__ __forceinline__ void copy_clip_setting(DpClipSetting* dst, const DpClipSetting* src, int lane) {
  if (lane < (int)(sizeof(DpClipSetting) / 8)) reinterpret_cast<uint2*>(dst)[lane] = reinterpret_cast<const uint2*>(src)[lane];
}

struct DpFrameArgs {
  const DpModelImage* model;
  const DpModelImageTC* model_tc;    // tables of the tcgen05 kernel
  const uint32_t* model_tmem;        // fp16x2 pieces of 16 W and 16 W^T as tensor-memory words [DP_TC_TMEM_WORDS][128]
  int n_clips;
  // carried state (HBM)
  float* latent;        // (B,24) latent after the last Adam step (seeds the next frame)
  float* gpos;          // (B,3)
  float* grot;          // (B,4) wxyz
  float* latent_buf;    // (B,60,24) ring, slot = (head + chronological row) % 60
  float* disp_buf;      // (B,60,3)
  float* height_buf;    // (B,60,6)
  int ring_head;        // slot holding the oldest row == slot written this frame
  const float* target_buf;  // (B,target_rows,24) predicted target latents
  int target_rows;
  int target_index;
  // per-frame inputs
  const int32_t* n_ee;
  const int32_t* joints;
  const float* weights;
  int shared_trackers;
  const float* tgt_pos;
  const float* tgt_rot;
  int ee_stride;
  int targets_world;  // tgt_pos is world-absolute: subtract the clip's current global position when loading it
  // optimiser: every clip runs with `uniform` (settings null), or, tcgen05 kernel only, clip c with settings[clip_setting[c]]
  // (settings[0] when clip_setting is null).  The two cases are separate instantiations of the tcgen05 kernel: reading a per-clip
  // entry from shared memory puts a load in front of the Adam step's table reads and its stop test, which measured 0.956 against
  // 0.920 ms per frame at 4 096 clips (DESIGN.md section 3.4); the uniform instantiation reads `uniform` from the kernel parameters.
  // The fp32 kernel runs a table as one launch per setting, each with that setting as `uniform` over compact copies of its clips.
  DpClipSetting uniform;
  const DpClipSetting* settings;
  const int32_t* clip_setting;
  int max_iter;      // loop bound: the largest max_iter of the settings in use
  int fixed_iters;   // every setting in use runs a fixed number of iterations (negative thresholds, min_incr = -inf)
  // outputs
  float* out_pose;    // (B,88), or the packed rows (B,92) = [pose 88 | global_pos 3 | pad] with out_gpos = out_pose + 88
  float* out_gpos;    // (B,3)
  int out_pose_stride, out_gpos_stride;  // floats per clip: 88 / 3, or 92 / 92 for packed rows
  int32_t* out_iters; // (B)
  float* out_losses;  // (B,3)
  float* trace;       // (B,trace_iters,52) or null
  int trace_iters;
  int clips_per_cta;  // tcgen05 kernel: real clips per 32-column tile (<= 32), chosen so that the grid covers every SM
  // teacher-forced evaluation (dp_engine_eval_gradient)
  int eval_only;
  float* eval_grad;   // (B,24)
  float* eval_pos;    // (B,22,3)
  // optional phase clock of CTA 0 (tcgen05 kernel), 8 counters, see dp_engine_get_phase_cycles
  unsigned long long* phase_cycles;
  // extension losses (drag_pose.py:129-183), fp32 CUDA-core kernel only: bit mask (0 = none) and floor height
  int ext_mask;
  float floor_level;
};

// ---------------------------------------------------------------- small math helpers
__device__ __forceinline__ void quat_mul(const float a[4], const float b[4], float r[4]) {
  r[0] = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3];
  r[1] = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
  r[2] = a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1];
  r[3] = a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0];
}

// python/src/utils.py:34-76 (no normalisation, 1 - 2(yy+zz) form), row-major 3x3
__device__ __forceinline__ void quat_to_mat(const float q[4], float m[9]) {
  const float w = q[0], x = q[1], y = q[2], z = q[3];
  const float x2 = x + x, y2 = y + y, z2 = z + z;
  const float xx = x * x2, yy = y * y2, wx = w * x2;
  const float xy = x * y2, yz = y * z2, wy = w * y2;
  const float xz = x * z2, zz = z * z2, wz = w * z2;
  m[0] = 1.0f - (yy + zz); m[1] = xy - wz;          m[2] = xz + wy;
  m[3] = xy + wz;          m[4] = 1.0f - (xx + zz); m[5] = yz - wx;
  m[6] = xz - wy;          m[7] = yz + wx;          m[8] = 1.0f - (xx + yy);
}

// adjoint of quat_to_mat: G = dL/dM  ->  dL/dq   (SURVEY.md appendix B, Mbar2q)
__device__ __forceinline__ void mat_bar_to_quat(const float q[4], const float G[9], float qb[4]) {
  const float w = q[0], x = q[1], y = q[2], z = q[3];
  qb[0] = 2.0f * (-z * G[1] + y * G[2] + z * G[3] - x * G[5] - y * G[6] + x * G[7]);
  qb[1] = 2.0f * (y * G[1] + z * G[2] + y * G[3] - 2.0f * x * G[4] - w * G[5] + z * G[6] + w * G[7] - 2.0f * x * G[8]);
  qb[2] = 2.0f * (-2.0f * y * G[0] + x * G[1] + w * G[2] + x * G[3] + z * G[5] - w * G[6] + z * G[7] - 2.0f * y * G[8]);
  qb[3] = 2.0f * (-2.0f * z * G[0] - w * G[1] + x * G[2] + w * G[3] - 2.0f * z * G[4] + y * G[5] + x * G[6] + y * G[7]);
}

__device__ __forceinline__ void mat_mul(const float a[9], const float b[9], float c[9]) {  // c = a b
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) c[3 * i + j] = a[3 * i] * b[j] + a[3 * i + 1] * b[3 + j] + a[3 * i + 2] * b[6 + j];
}
__device__ __forceinline__ void mat_mul_bt(const float a[9], const float b[9], float c[9]) {  // c = a b^T
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) c[3 * i + j] = a[3 * i] * b[3 * j] + a[3 * i + 1] * b[3 * j + 1] + a[3 * i + 2] * b[3 * j + 2];
}
__device__ __forceinline__ void mat_mul_at(const float a[9], const float b[9], float c[9]) {  // c = a^T b
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) c[3 * i + j] = a[i] * b[j] + a[3 + i] * b[3 + j] + a[6 + i] * b[6 + j];
}
__device__ __forceinline__ void mat_vec(const float a[9], const float v[3], float r[3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) r[i] = a[3 * i] * v[0] + a[3 * i + 1] * v[1] + a[3 * i + 2] * v[2];
}
__device__ __forceinline__ void mat_t_vec(const float a[9], const float v[3], float r[3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) r[i] = a[i] * v[0] + a[3 + i] * v[1] + a[6 + i] * v[2];
}

// fast reciprocal / square root (MUFU, <= 2 ulp): used where the reference's own fp32 noise is orders of magnitude larger
__device__ __forceinline__ float fast_rcp(float x) { return __fdividef(1.0f, x); }
__device__ __forceinline__ float fast_sqrt(float x) {
  float r;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// sum of 4 per-lane values over the warp with 6 shuffles instead of 20: halve the value set while halving the lane set.
// Afterwards lane (8*c) holds the total of component c (c = 0..3); other lanes hold totals of their own component.
__device__ __forceinline__ float warp_sum4_scatter(const float (&a)[4], int lane) {
  const bool b4 = lane & 16, b3 = lane & 8;
  float k0 = b4 ? a[2] : a[0], k1 = b4 ? a[3] : a[1];
  k0 += __shfl_xor_sync(0xffffffffu, b4 ? a[0] : a[2], 16);
  k1 += __shfl_xor_sync(0xffffffffu, b4 ? a[1] : a[3], 16);
  float k = b3 ? k1 : k0;
  k += __shfl_xor_sync(0xffffffffu, b3 ? k0 : k1, 8);
  k += __shfl_xor_sync(0xffffffffu, k, 4);
  k += __shfl_xor_sync(0xffffffffu, k, 2);
  k += __shfl_xor_sync(0xffffffffu, k, 1);
  return k;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// one lane of a fully converged warp (elect.sync): the pattern the compiler needs to emit a single
// predicated UTCHMMA / UBLKCP instead of a per-lane serialisation loop
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .b32 %%rx;\n"
      ".reg .pred %%px;\n"
      "elect.sync %%rx|%%px, %1;\n"
      "@%%px mov.s32 %0, 1;\n"
      "}\n"
      : "+r"(pred)
      : "r"(0xFFFFFFFFu));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier / bulk TMA
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_inval(uint64_t* bar) {  // required before the same shared-memory word is initialised again
  asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!done);
}
// 1-D bulk tensor-memory-accelerator copy global -> shared, completion on an mbarrier
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
