#pragma once
// dp_temporal_tc4.cuh -- feed-forward block of the temporal predictor on tcgen05 tensor cores, four CTAs per SM.
//
//   out = LayerNorm(x + W2 relu(W1 x + b1) + b2)   [+ optional second LayerNorm]
// (torch nn.TransformerEncoderLayer / DecoderLayer FF sub-block, post-norm, d_model 48, dim_feedforward 2048;
// python/src/temporal_transformer.py:26-33): 95% of the predictor's FLOPs.  One CTA owns a tile of 128 tokens (the UMMA M
// dimension) and walks the 2048 hidden units in chunks of 32.  Precision: fp16x2 split products on kind::f16 -- every fp32 value
// is two fp16 pieces, three products (2,1)(1,2)(1,1) accumulate in fp32; the weight image stores 64 W (an exact power of two,
// undone in the epilogues) so that the second piece of the small FF weights stays a normal fp16.  A operands live in tensor memory
// (TS mode): X is split once into TMEM and the epilogue warps write the packed pieces of relu(H) over the accumulator they came
// from, so activations never touch shared memory.  Weights are pre-split and pre-tiled on the host (dp_ff_tc_pack) into the exact
// shared-memory operand image: one pipeline step is ONE bulk-TMA copy, fed by a producer warp to an issuer warp through a
// mbarrier ring.
// A CTA is small in every resource -- 128 tensor-memory columns (ONE 32-unit H buffer that the pieces overwrite in place), a
// 3 x 12 KB weight ring, four epilogue warps -- so four of them share an SM and its tensor pipe: a tile saturates the pipe inside
// its chunks and loses time around them (the L2 fill burst of a wave at its start, the row epilogue at its end,
// profiles/r2_ff_pipeline_clock.md), and while one CTA is starting or finishing, three are multiplying.
//   MMA1  H[128x32]  = X[128x48] . W1c^T     (K = 48, 9 MMAs)
//   epi   H -> +b1, relu, split -> the same 32 columns (two packed pieces of 16 words)
//   MMA2  O[128x48] += H[128x32] . W2c^T     (K = 32, 6 MMAs)
// One H buffer: the issuer sends MMA2(c) and MMA1(c+1) back to back (the pipe executes in order, so MMA1(c+1) may overwrite what
// MMA2(c) has read), the epilogue of chunk c+1 follows their commit.  Weight step t = [W2(t-1) pieces | W1(t) pieces].
#include "dp_common.cuh"
#include "dp_internal.h"
#include "dp_umma.cuh"

namespace tpf {

constexpr int kTM = 128;
constexpr int kHC = FFT_HC;                    // 32 hidden units per chunk
constexpr int kChunks = TP_FF / kHC;           // 64
constexpr int kLag = 1;                        // step t carries W2 of chunk t - kLag
constexpr float kFfWScale = 64.0f;             // weight image holds 64 W
constexpr uint32_t kW1Bytes = kHC * TP_D * 2;  // 3072: one fp16 image of W1c [32][48]
constexpr uint32_t kW2Bytes = TP_D * kHC * 2;  // 3072: one fp16 image of W2c [48][32]
constexpr uint32_t kStepBytes = 2 * kW2Bytes + 2 * kW1Bytes;
static_assert(kHC == 32 && kStepBytes == FFT_STEP_BYTES && TP_FF * 4 + (kChunks + kLag) * kStepBytes == FFT_LAYER_BYTES, "image size");
// shared-memory B-operand geometry (bytes), K-major no-swizzle fp16: element (n,k) at (n/8)*128 + (k/8)*LBO + (n%8)*16 + (k%8)*2
constexpr uint32_t kW1_LBO = 128 * (kHC / 8), kW2_LBO = 128 * (TP_D / 8), kB_SBO = 128;

constexpr int kStages = 3;
struct Smem {
  unsigned char w[kStages][kStepBytes];
  float b1[TP_FF];
  uint64_t wfull[kStages], wfree[kStages], hfull, hready, b1full;
  uint32_t tmem_base;
};
// tensor-memory columns: X pieces | H (accumulator, then its two pieces in place) | output accumulator
constexpr uint32_t kT_X1 = 0, kT_X2 = 24, kT_H = 48, kT_OUT = 80, kT_COLS = 128;
constexpr uint32_t kIdescF16 = (1u << 4);  // fp32 accumulate, fp16 A/B, both K-major; N and M added below
constexpr int kCtasPerSm = 4;

__device__ __forceinline__ void issue_mma1(const Smem& S, int stage, uint32_t tmem) {
  constexpr uint32_t idesc = kIdescF16 | ((uint32_t)(kHC >> 3) << 17) | ((uint32_t)(kTM >> 4) << 24);
  const uint32_t base = smem_u32(S.w[stage]) + 2 * kW2Bytes;
  const UmmaDescBase w1 = umma_desc_base(base, kW1_LBO, kB_SBO);
  const UmmaDescBase w2 = umma_desc_base(base + kW1Bytes, kW1_LBO, kB_SBO);
  const uint32_t d = tmem + kT_H, x1 = tmem + kT_X1, x2 = tmem + kT_X2;
#pragma unroll
  for (int k = 0; k < TP_D / 16; ++k) {
    const uint32_t bo = k * 2 * kW1_LBO;
    if (k == 0) umma_f16_ts_c<false>(d, x2 + 8 * k, umma_desc_at(w1, bo), idesc);
    else umma_f16_ts_c<true>(d, x2 + 8 * k, umma_desc_at(w1, bo), idesc);
    umma_f16_ts_c<true>(d, x1 + 8 * k, umma_desc_at(w2, bo), idesc);
    umma_f16_ts_c<true>(d, x1 + 8 * k, umma_desc_at(w1, bo), idesc);
  }
}
__device__ __forceinline__ void issue_mma2(const Smem& S, int stage, uint32_t tmem, bool first) {
  constexpr uint32_t idesc = kIdescF16 | ((uint32_t)(TP_D >> 3) << 17) | ((uint32_t)(kTM >> 4) << 24);
  const UmmaDescBase w1 = umma_desc_base(smem_u32(S.w[stage]), kW2_LBO, kB_SBO);
  const UmmaDescBase w2 = umma_desc_base(smem_u32(S.w[stage]) + kW2Bytes, kW2_LBO, kB_SBO);
  const uint32_t d = tmem + kT_OUT;
#pragma unroll
  for (int k = 0; k < kHC / 16; ++k) {
    const uint32_t bo = k * 2 * kW2_LBO;
    const uint32_t h1 = tmem + kT_H + k * 8, h2 = h1 + 16;  // piece 1: words 0..15, piece 2: words 16..31
    if (k == 0) {
      if (first) umma_f16_ts_c<false>(d, h2, umma_desc_at(w1, bo), idesc);
      else umma_f16_ts_c<true>(d, h2, umma_desc_at(w1, bo), idesc);
    } else {
      umma_f16_ts_c<true>(d, h2, umma_desc_at(w1, bo), idesc);
    }
    umma_f16_ts_c<true>(d, h1, umma_desc_at(w2, bo), idesc);
    umma_f16_ts_c<true>(d, h1, umma_desc_at(w1, bo), idesc);
  }
}

constexpr int kEpiThreads = 128, kThreads = kEpiThreads + 64;  // 4 epilogue warps + MMA issuer warp (4) + TMA producer warp (5)

// local step j of the CTA's chunk range into ring stage st; step 0 is only read for its W1 half, step n_loc only for its W2 half
__device__ __forceinline__ void load_step(Smem& S, const unsigned char* steps, int c0, int j, int n_loc, int st) {
  const unsigned char* src = steps + (size_t)(c0 + j) * kStepBytes;
  uint32_t off = 0, bytes = kStepBytes;
  if (j < kLag) { off = 2 * kW2Bytes; bytes = 2 * kW1Bytes; }
  else if (j >= n_loc) bytes = 2 * kW2Bytes;
  mbar_expect_tx(&S.wfull[st], bytes);
  tma_bulk_g2s(S.w[st] + off, src + off, bytes, &S.wfull[st]);
}
__device__ __forceinline__ void ff_init_barriers(Smem& S) {
  for (int i = 0; i < kStages; ++i) { mbar_init(&S.wfull[i], 1); mbar_init(&S.wfree[i], 1); }
  mbar_init(&S.hfull, 1);
  mbar_init(&S.hready, kEpiThreads);
  mbar_init(&S.b1full, 1);
}
// One feed-forward block for the 128-row tile starting at row0 (rows >= m_limit of the tile are padding).  (split, n_split): this
// call takes the hidden chunks [split, split + 1) * kChunks / n_split; with n_split > 1 the raw partial sums go to `part`
// ([n_split][n_rows][48]) and tp_ff_finish_kernel adds bias, residual and the LayerNorms.  Called by all kThreads threads with
// kT_COLS columns of tensor memory at `tmem` and the mbarriers of S freshly initialised and published by a block barrier; returns
// after a block barrier.
__device__ __forceinline__ void ff_tile(Smem& S, const uint32_t tmem, const unsigned char* wimg, const float* blob, TpFF F, TpNorm N1, TpNorm N2, int has_n2,
                                        const float* x_g, int n_rows, int T, int row_stride, int row0, int m_limit, int split, int n_split,
                                        float* out_g, float* part, long long* trace) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_loc = kChunks / n_split, c0 = split * n_loc;  // this call's chunks: c0 .. c0 + n_loc - 1
  const unsigned char* steps = wimg + TP_FF * 4;
  const bool trace0 = trace && blockIdx.x == (unsigned)trace[3] && blockIdx.y == 0;
  if (warp == 5 && elect_one()) {  // TMA producer, part 1 (no waits before the block barrier below): bias slice + first stages
    mbar_expect_tx(&S.b1full, (uint32_t)(n_loc * kHC * 4));
    tma_bulk_g2s(S.b1 + c0 * kHC, wimg + (size_t)c0 * kHC * 4, (uint32_t)(n_loc * kHC * 4), &S.b1full);
    for (int j = 0; j < kStages && j < n_loc + kLag; ++j) load_step(S, steps, c0, j, n_loc, j);
  }
  const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
  const int m = (warp & 3) * 32 + lane;          // token row == TMEM lane owned by this thread
  const int row = row0 + m;
  const bool row_ok = row < n_rows && m < m_limit;
  const size_t g = row_ok ? ((size_t)(row / T) * row_stride + row % T) * TP_D : 0;
  if (warp < 4) {  // X tile -> tensor memory as the A operand (two fp16 pieces, two K elements per word)
    float p1[24], p2[24];
#pragma unroll
    for (int j = 0; j < TP_D; j += 4) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row_ok) v = __ldcg(reinterpret_cast<const float4*>(x_g + g + j));
      split_h2(v.x, v.y, p1[j / 2], p2[j / 2]);
      split_h2(v.z, v.w, p1[j / 2 + 1], p2[j / 2 + 1]);
    }
    tmem_st8(tmem + lane_base + kT_X1, &p1[0]);
    tmem_st8(tmem + lane_base + kT_X1 + 8, &p1[8]);
    tmem_st8(tmem + lane_base + kT_X1 + 16, &p1[16]);
    tmem_st8(tmem + lane_base + kT_X2, &p2[0]);
    tmem_st8(tmem + lane_base + kT_X2 + 8, &p2[8]);
    tmem_st8(tmem + lane_base + kT_X2 + 16, &p2[16]);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    // ===== MMA issuer warp: iteration i: MMA2(i), MMA1(i+1), one commit
    tc_fence_after();
    mbar_wait(&S.wfull[0], 0);
    if (elect_one()) {
      issue_mma1(S, 0, tmem);
      umma_commit(&S.hfull);
      umma_commit(&S.wfree[0]);
    }
    __syncwarp();
    for (int i = 0; i < n_loc; ++i) {
      const int step = i + 1, st = step % kStages;
      mbar_wait(&S.wfull[st], (step / kStages) & 1);
      const bool traced = trace0 && lane == 0;
      if (traced && i < 32) trace[i * 8 + 0] = clock64();
      mbar_wait(&S.hready, i & 1);  // all epilogue threads converted H(i) into its pieces
      tc_fence_after();
      if (traced && i < 32) trace[i * 8 + 1] = clock64();
      if (elect_one()) {
        issue_mma2(S, st, tmem, i == 0);
        if (i + 1 < n_loc) issue_mma1(S, st, tmem);
        umma_commit(&S.hfull);
        umma_commit(&S.wfree[st]);
      }
      __syncwarp();
      if (traced && i < 32) trace[i * 8 + 2] = clock64();
    }
  } else if (warp == 5) {
    // ===== TMA producer warp, part 2
    if (elect_one()) {
      for (int j = kStages; j < n_loc + kLag; ++j) {
        const int st = j % kStages;
        mbar_wait(&S.wfree[st], ((j / kStages) - 1) & 1);
        load_step(S, steps, c0, j, n_loc, st);
      }
    }
    __syncwarp();
  } else {
    // ===== epilogue warps: H(i) accumulator -> relu(H / 64 + b1) -> two packed fp16 pieces, in place
    mbar_wait(&S.b1full, 0);
    for (int i = 0; i < n_loc; ++i) {
      const float* b1 = S.b1 + (c0 + i) * kHC;
      mbar_wait(&S.hfull, i & 1);  // H(i) accumulated (and MMA2(i-1) retired)
      tc_fence_after();
      const bool traced = trace0 && tid == 0;
      if (traced && i < 32) trace[i * 8 + 4] = clock64();
      float v[32], p1[16], p2[16];
      tmem_ld32(tmem + lane_base + kT_H, v);
      tmem_ld_wait();
      if (traced && i < 32) trace[i * 8 + 5] = clock64();
      // three CUDA-core instructions per hidden unit: packed FFMA2 for scale + bias and FADD2 for the residual, the ReLU folded into
      // the conversions.  Piece 1 is relu(h) rounded TOWARDS ZERO (cvt.rz.relu), so the residual h - p1 of a positive h is never
      // negative, while a negative h (p1 = 0) leaves a negative residual that piece 2's cvt.rn.relu clamps: p1 + p2 = relu(h) to 2^-21
#pragma unroll
      for (int j = 0; j < 32; j += 2) {
        const float2 h = __ffma2_rn(make_float2(v[j], v[j + 1]), make_float2(1.0f / kFfWScale, 1.0f / kFfWScale), make_float2(b1[j], b1[j + 1]));
        uint32_t w, w2;
        asm("cvt.rz.relu.f16x2.f32 %0, %1, %2;" : "=r"(w) : "f"(h.y), "f"(h.x));
        float2 f;
        asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;\n\t}\n" : "=f"(f.x), "=f"(f.y) : "r"(w));
        const float2 d = __fadd2_rn(h, make_float2(-f.x, -f.y));
        asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(w2) : "f"(d.y), "f"(d.x));
        p1[j / 2] = __uint_as_float(w);
        p2[j / 2] = __uint_as_float(w2);
      }
      tmem_st16(tmem + lane_base + kT_H, p1);
      tmem_st16(tmem + lane_base + kT_H + 16u, p2);
      tmem_st_wait();
      if (traced && i < 32) trace[i * 8 + 6] = clock64();
      tc_fence_before();
      mbar_arrive(&S.hready);
    }
    // the commit of the last iteration (completion n_loc of hfull) covers MMA2(n_loc - 1): the output accumulator is final
    mbar_wait(&S.hfull, n_loc & 1);
    tc_fence_after();
    float o[TP_D];
#pragma unroll
    for (int j0 = 0; j0 < TP_D; j0 += 16) {
      float v[16];
      tmem_ld16(tmem + lane_base + kT_OUT + (uint32_t)j0, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; ++j) o[j0 + j] = v[j] * (1.0f / kFfWScale);
    }
    if (row_ok) {
      if (n_split > 1) {
        float* dst = part + ((size_t)split * n_rows + row) * TP_D;
#pragma unroll
        for (int j = 0; j < TP_D; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]);
      } else {
        const float* b2 = blob + F.b2;
#pragma unroll
        for (int j = 0; j < TP_D; j += 4) {
          const float4 xv = __ldcg(reinterpret_cast<const float4*>(x_g + g + j));
          o[j] += b2[j] + xv.x; o[j + 1] += b2[j + 1] + xv.y; o[j + 2] += b2[j + 2] + xv.z; o[j + 3] += b2[j + 3] + xv.w;
        }
        ln48(o, blob + N1.w, blob + N1.b);
        if (has_n2) ln48(o, blob + N2.w, blob + N2.b);
#pragma unroll
        for (int j = 0; j < TP_D; j += 4) *reinterpret_cast<float4*>(out_g + g + j) = make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (trace0 && tid == 0) trace[15] = clock64();
}

}  // namespace tpf
