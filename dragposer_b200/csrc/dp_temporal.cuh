// dp_temporal.cuh -- weight blob layout of the temporal predictor (host + device).
//
// Reference: python/src/temporal_transformer.py:6-78 (Temporal), torch nn.Transformer
// (d_model 48, 4 heads, 3+3 post-norm layers, FF 2048, ReLU, final LayerNorms),
// python/src/positional_encoding.py:15-32, python/src/train_temporal.py:17-37.
// Every Linear weight is stored TRANSPOSED ([in][out]) so that consecutive threads
// (consecutive output features) read consecutive floats.
#pragma once
#include <stddef.h>

#define TP_D 48
#define TP_H 4
#define TP_HD 12
#define TP_FF 2048
#define TP_ENC_IN 33
#define TP_LAT 24
#define TP_S 14        // encoder tokens
#define TP_MAXT 32     // decoder tokens <= 1 + DP_MAX_WINDOW/4 = 30
#define TP_PE 30
#define TP_NENC 3
#define TP_NDEC 3
// weight image of the tensor-core feed-forward block (dp_temporal_tc4.cuh)
#define FFT_HC 32                 // hidden units per tensor-core FF chunk
#define FFT_STEP_BYTES 12288      // one pipeline step: W2c pieces of chunk t-1 (2 x 3072 fp16) + W1c pieces of chunk t (2 x 3072 fp16)
#define FFT_LAYER_BYTES (TP_FF * 4 + (TP_FF / FFT_HC + 1) * FFT_STEP_BYTES)   // b1 (fp32) + 65 steps
#define ATT_LAYER_BYTES 37632      // W_in pieces (2 x 13824 fp16) + W_o pieces (2 x 4608 fp16) + b_in (576) + b_o (192)

struct TpAttn {   // offsets (floats) into the blob
  size_t w_in;    // [48][144]  (q | k | v columns)
  size_t b_in;    // [144]
  size_t w_out;   // [48][48]
  size_t b_out;   // [48]
};
struct TpFF {
  size_t w1;      // [48][2048]
  size_t b1;      // [2048]
  size_t w2;      // [2048][48]
  size_t b2;      // [48]
};
struct TpNorm { size_t w, b; };

struct TpLayout {
  size_t enc_in_w, enc_in_b;   // [33][48], [48]
  size_t dec_in_w, dec_in_b;   // [24][48], [48]
  size_t pe;                   // [30][48]
  struct { TpAttn sa; TpFF ff; TpNorm n1, n2; } enc[TP_NENC];
  TpNorm enc_norm;
  struct { TpAttn sa, ca; TpFF ff; TpNorm n1, n2, n3; } dec[TP_NDEC];
  TpNorm dec_norm;
  size_t out_w, out_b;         // [48][24], [24]
  size_t total;
};

inline TpLayout tp_layout() {
  TpLayout L;
  size_t o = 0;
  auto take = [&](size_t n) { size_t r = o; o += (n + 3) & ~size_t(3); return r; };  // keep 16-byte alignment
  auto attn = [&](TpAttn& a) { a.w_in = take(TP_D * 3 * TP_D); a.b_in = take(3 * TP_D); a.w_out = take(TP_D * TP_D); a.b_out = take(TP_D); };
  auto ff = [&](TpFF& f) { f.w1 = take(TP_D * TP_FF); f.b1 = take(TP_FF); f.w2 = take(TP_FF * TP_D); f.b2 = take(TP_D); };
  auto norm = [&](TpNorm& n) { n.w = take(TP_D); n.b = take(TP_D); };
  L.enc_in_w = take(TP_ENC_IN * TP_D); L.enc_in_b = take(TP_D);
  L.dec_in_w = take(TP_LAT * TP_D); L.dec_in_b = take(TP_D);
  L.pe = take(TP_PE * TP_D);
  for (int l = 0; l < TP_NENC; ++l) { attn(L.enc[l].sa); ff(L.enc[l].ff); norm(L.enc[l].n1); norm(L.enc[l].n2); }
  norm(L.enc_norm);
  for (int l = 0; l < TP_NDEC; ++l) { attn(L.dec[l].sa); attn(L.dec[l].ca); ff(L.dec[l].ff); norm(L.dec[l].n1); norm(L.dec[l].n2); norm(L.dec[l].n3); }
  norm(L.dec_norm);
  L.out_w = take(TP_D * TP_LAT); L.out_b = take(TP_LAT);
  L.total = o;
  return L;
}

// Optional work fused behind the feed-forward block of a SINGLE-TOKEN decoder pass (T == 1: the first autoregressive step, the only
// one when temporal_future_window == 0): the finished row goes straight through the next decoder layer's self-attention block
// (one key: softmax == 1, so the block is LN(x + W_o (W_v x + b_v) + b_o), a row-local map) and / or through the prediction head
// of drag_pose.py:275-289.  Saves the 32-CTA attention launch and the head launch of every layer of the pass.  The cross-attention
// block of a single query is row-local too once W_k is folded into the query and W_v behind the weighted sum of the memory tokens
// (tp_cross_attn_single): it rides in the same kernels, so the pass needs no attention launch at all.
struct TpFfTail {
  int next_self_attn;
  TpAttn sa;
  TpNorm n1;
  int next_cross_attn;     // ... followed by that layer's cross-attention block against the clip's encoder memory (tp_cross_attn_single)
  TpAttn ca;
  TpNorm n2;
  const float* wk_t;       // that block's key projection as [key feature][input] (DP_TC_XA_OFFSET)
  const float* mem;        // encoder memory (n_clips, TP_S, TP_D)
  int out_head;
  size_t out_w, out_b;
  const float* mu;
  const float* sigma;
  float* dec_lat;
  float* target_buf;
  int step_i, window;
};

#ifdef __CUDACC__
// ---- one warp owns one 48-wide row: lane holds features lane and lane + 32 (< 48)
__device__ __forceinline__ float tp_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ void tp_ln_row_warp(float& v0, float& v1, const float* __restrict__ w, const float* __restrict__ b, int lane) {
  const bool has1 = lane + 32 < TP_D;
  const float mean = tp_warp_sum(v0 + (has1 ? v1 : 0.0f)) * (1.0f / TP_D);
  const float d0 = v0 - mean, d1 = has1 ? v1 - mean : 0.0f;
  const float rstd = rsqrtf(tp_warp_sum(d0 * d0 + d1 * d1) * (1.0f / TP_D) + 1e-5f);
  v0 = d0 * rstd * w[lane] + b[lane];
  v1 = has1 ? d1 * rstd * w[lane + 32] + b[lane + 32] : 0.0f;
}
// y = bias + x W for a [K][ldw] weight block starting at column col0 (blob layout: [in][out]); K <= 48 inputs held like a row
template <int K>
__device__ __forceinline__ void tp_warp_matvec(float x0, float x1, const float* __restrict__ W, int ldw, int col0, const float* __restrict__ bias,
                                               int n_out, int lane, float& y0, float& y1) {
  const bool has0 = lane < n_out, has1 = lane + 32 < n_out;
  y0 = has0 ? bias[lane] : 0.0f;
  y1 = has1 ? bias[lane + 32] : 0.0f;
#pragma unroll 8
  for (int i = 0; i < K; ++i) {
    const float xi = __shfl_sync(0xffffffffu, i < 32 ? x0 : x1, i & 31);
    const float* w = W + (size_t)i * ldw + col0;
    if (has0) y0 = fmaf(xi, w[lane], y0);
    if (has1) y1 = fmaf(xi, w[lane + 32], y1);
  }
}
// the same with the input row staged in shared memory (xs: K floats, 16-byte aligned, visible to the whole warp): the inputs arrive as
// broadcast LDS.128 (K / 4 loads) instead of K shuffles -- a shuffle costs four issue cycles of a sub-partition, and the single-token
// decoder blocks below are chains of these products
template <int K>
__device__ __forceinline__ void tp_warp_matvec_s(const float* __restrict__ xs, const float* __restrict__ W, int ldw, int col0,
                                                 const float* __restrict__ bias, int n_out, int lane, float& y0, float& y1) {
  static_assert(K % 4 == 0, "vectorised input row");
  const bool has0 = lane < n_out, has1 = lane + 32 < n_out;
  y0 = has0 ? bias[lane] : 0.0f;
  y1 = has1 ? bias[lane + 32] : 0.0f;
  const float* w = W + col0 + (has0 ? lane : 0);
  const float* w1 = W + col0 + (has1 ? lane + 32 : 0);
#pragma unroll 4
  for (int i = 0; i < K; i += 4) {
    const float4 xv = *reinterpret_cast<const float4*>(xs + i);
    y0 = fmaf(xv.x, w[(size_t)i * ldw], fmaf(xv.y, w[(size_t)(i + 1) * ldw], fmaf(xv.z, w[(size_t)(i + 2) * ldw], fmaf(xv.w, w[(size_t)(i + 3) * ldw], y0))));
    y1 = fmaf(xv.x, w1[(size_t)i * ldw], fmaf(xv.y, w1[(size_t)(i + 1) * ldw], fmaf(xv.z, w1[(size_t)(i + 2) * ldw], fmaf(xv.w, w1[(size_t)(i + 3) * ldw], y1))));
  }
  if (!has0) y0 = 0.0f;
  if (!has1) y1 = 0.0f;
}
// publish a row held as (lane, lane + 32) to the warp's staging row
__device__ __forceinline__ void tp_stage_row(float* __restrict__ xs, int lane, float v0, float v1) {
  __syncwarp();  // earlier readers of the staging row are done
  xs[lane] = v0;
  if (lane + 32 < TP_D) xs[lane + 32] = v1;
  __syncwarp();
}
// self-attention block of a single token (its only key is itself): x <- LN(x + W_o (W_v x + b_v) + b_o); xs: TP_D floats of
// shared memory owned by this warp (staging row)
__device__ __forceinline__ void tp_self_attn_single_s(const float* __restrict__ blob, const TpAttn& A, const TpNorm& N, float* __restrict__ xs, int lane,
                                                      float& x0, float& x1) {
  float v0, v1, o0, o1;
  tp_stage_row(xs, lane, x0, x1);
  tp_warp_matvec_s<TP_D>(xs, blob + A.w_in, 3 * TP_D, 2 * TP_D, blob + A.b_in + 2 * TP_D, TP_D, lane, v0, v1);
  tp_stage_row(xs, lane, v0, v1);
  tp_warp_matvec_s<TP_D>(xs, blob + A.w_out, TP_D, 0, blob + A.b_out, TP_D, lane, o0, o1);
  x0 += o0;
  x1 += o1;
  tp_ln_row_warp(x0, x1, blob + N.w, blob + N.b, lane);
}
// Cross-attention block of a SINGLE decoder token against the S = 14 encoder-memory rows m_s of its clip, one warp per token:
//   x <- LN(x + W_o concat_h(W_v,h mbar_h + b_v,h) + b_o),  mbar_h = sum_s a_hs m_s,  a_h = softmax_s((W_k,h^T q_h) . m_s / sqrt(12))
// -- nn.MultiheadAttention (temporal_transformer.py:53-78) with the key projection folded into the query (the bias term q_h . b_k,h is
// the same for every key and cancels in the softmax) and the value projection applied once to the weighted sum of the memory tokens
// (the probabilities sum to one, so b_v passes through): 4 x 48 x 12 + 4 x 48 x 12 multiply-adds instead of two 14 x 48 x 48
// projections, all in fp32, nothing but the 14 memory rows read.  `scr`: TP_XA_SCR floats of shared memory owned by this warp.
#define TP_XA_STRIDE 52   // row stride of the scratch (floats): 16-byte aligned rows that start in different banks
#define TP_XA_SCR ((TP_H + TP_S) * TP_XA_STRIDE + TP_D + TP_S * TP_H)   // four per-head rows + the clip's 14 memory rows + a staging row + the probabilities
// wk_t: the key projection as [key feature d][input c] (so that a warp reads one d-row coalesced over c).
__device__ __forceinline__ void tp_cross_attn_single(const float* __restrict__ blob, const TpAttn& A, const TpNorm& N, const float* __restrict__ wk_t,
                                                     const float* __restrict__ mem, float* __restrict__ scr, int lane, float& x0, float& x1) {
  static_assert(TP_H * TP_HD == TP_D && TP_S <= 16 && TP_D % 4 == 0, "layout of the folded cross-attention");
  const bool has1 = lane + 32 < TP_D;
  const float* Win = blob + A.w_in;   // [in 48][q 48 | k 48 | v 48]
  float* ms = scr + TP_H * TP_XA_STRIDE;  // the clip's memory rows, staged once (coalesced) and read three times
  float* xs = scr + (TP_H + TP_S) * TP_XA_STRIDE;      // staging row of the matrix-vector products
  float* as = xs + TP_D;                               // probabilities a[s][h] (14 x 4 floats)
  static_assert(((TP_H + TP_S) * TP_XA_STRIDE) % 4 == 0 && TP_D % 4 == 0 && TP_XA_SCR % 4 == 0, "16-byte aligned scratch rows");
  for (int i = lane; i < TP_S * (TP_D / 4); i += 32) {
    const int s = i / (TP_D / 4), c4 = i % (TP_D / 4);
    reinterpret_cast<float4*>(ms + s * TP_XA_STRIDE)[c4] = reinterpret_cast<const float4*>(mem)[i];
  }
  float q0, q1;
  tp_stage_row(xs, lane, x0, x1);
  tp_warp_matvec_s<TP_D>(xs, Win, 3 * TP_D, 0, blob + A.b_in, TP_D, lane, q0, q1);
  tp_stage_row(xs, lane, q0, q1);
  // qt_h[c] = (1 / sqrt(12)) sum_{d in head h} W_k[d][c] q[d]; this lane owns c = lane and c = lane + 32
  {
    const float scale = rsqrtf((float)TP_HD);
#pragma unroll
    for (int h = 0; h < TP_H; ++h) {
      float a0 = 0.0f, a1 = 0.0f;
#pragma unroll
      for (int j4 = 0; j4 < TP_HD; j4 += 4) {
        const int d = h * TP_HD + j4;
        const float4 qv = *reinterpret_cast<const float4*>(xs + d);  // broadcast
        a0 = fmaf(wk_t[d * TP_D + lane], qv.x, fmaf(wk_t[(d + 1) * TP_D + lane], qv.y, fmaf(wk_t[(d + 2) * TP_D + lane], qv.z, fmaf(wk_t[(d + 3) * TP_D + lane], qv.w, a0))));
        if (has1)
          a1 = fmaf(wk_t[d * TP_D + lane + 32], qv.x,
                    fmaf(wk_t[(d + 1) * TP_D + lane + 32], qv.y, fmaf(wk_t[(d + 2) * TP_D + lane + 32], qv.z, fmaf(wk_t[(d + 3) * TP_D + lane + 32], qv.w, a1))));
      }
      scr[h * TP_XA_STRIDE + lane] = a0 * scale;
      if (has1) scr[h * TP_XA_STRIDE + lane + 32] = a1 * scale;
    }
  }
  __syncwarp();
  // scores of key s on lane s (all heads), softmax across the lanes
  {
    float a[TP_H];
    const bool key = lane < TP_S;
    float sc[TP_H] = {0.0f, 0.0f, 0.0f, 0.0f};
    const float4* mrow = reinterpret_cast<const float4*>(ms + (key ? lane : 0) * TP_XA_STRIDE);
#pragma unroll
    for (int c4 = 0; c4 < TP_D / 4; ++c4) {
      const float4 mv = mrow[c4];
#pragma unroll
      for (int h = 0; h < TP_H; ++h) {
        const float4 qv = reinterpret_cast<const float4*>(scr + h * TP_XA_STRIDE)[c4];
        sc[h] = fmaf(mv.x, qv.x, fmaf(mv.y, qv.y, fmaf(mv.z, qv.z, fmaf(mv.w, qv.w, sc[h]))));
      }
    }
#pragma unroll
    for (int h = 0; h < TP_H; ++h) {
      const float v = key ? sc[h] : -3.0e38f;
      float mx = v;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));  // the keys live on lanes 0..13 of the lower half
      const float p = key ? expf(v - mx) : 0.0f;
      float sum = p;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      a[h] = key ? p / sum : 0.0f;  // (the upper half-warp sums to zero; its lanes publish nothing)
    }
    if (key) *reinterpret_cast<float4*>(as + 4 * lane) = make_float4(a[0], a[1], a[2], a[3]);
  }
  __syncwarp();  // probabilities published; every lane has read the folded queries: the per-head rows are free again
  // mbar_h[c] = sum_s a_hs m_s[c]
  {
    float b0[TP_H] = {0.0f, 0.0f, 0.0f, 0.0f}, b1[TP_H] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
    for (int s = 0; s < TP_S; ++s) {
      const float m0 = ms[s * TP_XA_STRIDE + lane], m1 = has1 ? ms[s * TP_XA_STRIDE + lane + 32] : 0.0f;
      const float4 av = *reinterpret_cast<const float4*>(as + 4 * s);  // broadcast
      b0[0] = fmaf(av.x, m0, b0[0]); b0[1] = fmaf(av.y, m0, b0[1]); b0[2] = fmaf(av.z, m0, b0[2]); b0[3] = fmaf(av.w, m0, b0[3]);
      b1[0] = fmaf(av.x, m1, b1[0]); b1[1] = fmaf(av.y, m1, b1[1]); b1[2] = fmaf(av.z, m1, b1[2]); b1[3] = fmaf(av.w, m1, b1[3]);
    }
#pragma unroll
    for (int h = 0; h < TP_H; ++h) {
      scr[h * TP_XA_STRIDE + lane] = b0[h];
      if (has1) scr[h * TP_XA_STRIDE + lane + 32] = b1[h];
    }
  }
  __syncwarp();
  // o[d] = b_v[d] + sum_c W_v[c][d] mbar_{head(d)}[c]; this lane owns d = lane and d = lane + 32
  float o0 = blob[A.b_in + 2 * TP_D + lane], o1 = has1 ? blob[A.b_in + 2 * TP_D + lane + 32] : 0.0f;
  {
    const float* mb0 = scr + (lane / TP_HD) * TP_XA_STRIDE;
    const float* mb1 = scr + ((has1 ? lane + 32 : lane) / TP_HD) * TP_XA_STRIDE;
    const float* wv = Win + 2 * TP_D;
#pragma unroll 8
    for (int c = 0; c < TP_D; ++c) {
      o0 = fmaf(mb0[c], wv[(size_t)c * 3 * TP_D + lane], o0);
      if (has1) o1 = fmaf(mb1[c], wv[(size_t)c * 3 * TP_D + lane + 32], o1);
    }
  }
  float y0, y1;
  tp_stage_row(xs, lane, o0, o1);
  tp_warp_matvec_s<TP_D>(xs, blob + A.w_out, TP_D, 0, blob + A.b_out, TP_D, lane, y0, y1);
  x0 += y0;
  x1 += y1;
  tp_ln_row_warp(x0, x1, blob + N.w, blob + N.b, lane);
}
// ---- the same single-token blocks for TP_R rows per warp.  The blocks above are chains of 48 x 48 matrix-vector products whose
// cost is the weight loads (two per multiply-add pair and row); here a warp carries TP_R rows through every product, so a weight is
// loaded once per TP_R rows and the inputs of all rows at one k arrive as ONE broadcast LDS.128 (staging layout [k][row]): 12 memory
// instructions per 32 multiply-adds instead of 9 per 8.  Every row's arithmetic -- the order of every fused multiply-add, the softmax,
// the LayerNorm reductions -- is exactly that of the one-row functions, so the results are bitwise the same.
#define TP_R 4
// per-warp scratch (floats): staging [48][TP_R] | per-row per-head rows [TP_R][4][52] (folded queries, then weighted memory sums) |
// ONE clip's 14 memory rows [14][52] | its probabilities [14][4]
#define TP_XR_SCR (TP_D * TP_R + TP_R * TP_H * TP_XA_STRIDE + TP_S * TP_XA_STRIDE + TP_S * TP_H)
__device__ __forceinline__ void tp_stage_rows(float* __restrict__ xs, int lane, const float (&v0)[TP_R], const float (&v1)[TP_R]) {
  static_assert(TP_R == 4, "one float4 per k");
  __syncwarp();  // earlier readers of the staging rows are done
  *reinterpret_cast<float4*>(xs + 4 * lane) = make_float4(v0[0], v0[1], v0[2], v0[3]);
  if (lane + 32 < TP_D) *reinterpret_cast<float4*>(xs + 4 * (lane + 32)) = make_float4(v1[0], v1[1], v1[2], v1[3]);
  __syncwarp();
}
// tp_warp_matvec_s for TP_R rows (inputs staged as [k][row])
template <int K>
__device__ __forceinline__ void tp_warp_matvec_r(const float* __restrict__ xs, const float* __restrict__ W, int ldw, int col0,
                                                 const float* __restrict__ bias, int n_out, int lane, float (&y0)[TP_R], float (&y1)[TP_R]) {
  static_assert(K % 4 == 0, "vectorised input rows");
  const bool has0 = lane < n_out, has1 = lane + 32 < n_out;
  const float b0 = has0 ? bias[lane] : 0.0f, b1 = has1 ? bias[lane + 32] : 0.0f;
#pragma unroll
  for (int r = 0; r < TP_R; ++r) { y0[r] = b0; y1[r] = b1; }
  const float* w = W + col0 + (has0 ? lane : 0);
  const float* w1 = W + col0 + (has1 ? lane + 32 : 0);
#pragma unroll 4
  for (int i = 0; i < K; i += 4) {
    float xk[4][TP_R];
#pragma unroll
    for (int j = 0; j < 4; ++j) *reinterpret_cast<float4*>(xk[j]) = *reinterpret_cast<const float4*>(xs + 4 * (i + j));
    const float wa0 = w[(size_t)i * ldw], wa1 = w[(size_t)(i + 1) * ldw], wa2 = w[(size_t)(i + 2) * ldw], wa3 = w[(size_t)(i + 3) * ldw];
    const float wb0 = w1[(size_t)i * ldw], wb1 = w1[(size_t)(i + 1) * ldw], wb2 = w1[(size_t)(i + 2) * ldw], wb3 = w1[(size_t)(i + 3) * ldw];
#pragma unroll
    for (int r = 0; r < TP_R; ++r) {
      y0[r] = fmaf(xk[0][r], wa0, fmaf(xk[1][r], wa1, fmaf(xk[2][r], wa2, fmaf(xk[3][r], wa3, y0[r]))));
      y1[r] = fmaf(xk[0][r], wb0, fmaf(xk[1][r], wb1, fmaf(xk[2][r], wb2, fmaf(xk[3][r], wb3, y1[r]))));
    }
  }
#pragma unroll
  for (int r = 0; r < TP_R; ++r) {
    if (!has0) y0[r] = 0.0f;
    if (!has1) y1[r] = 0.0f;
  }
}
// tp_warp_matvec (ascending one-by-one accumulation: the embedding and the prediction head) for TP_R rows, inputs staged as [k][row]
template <int K>
__device__ __forceinline__ void tp_warp_matvec_asc_r(const float* __restrict__ xs, const float* __restrict__ W, int ldw, const float* __restrict__ bias,
                                                     int n_out, int lane, float (&y0)[TP_R], float (&y1)[TP_R]) {
  const bool has0 = lane < n_out, has1 = lane + 32 < n_out;
  const float b0 = has0 ? bias[lane] : 0.0f, b1 = has1 ? bias[lane + 32] : 0.0f;
#pragma unroll
  for (int r = 0; r < TP_R; ++r) { y0[r] = b0; y1[r] = b1; }
#pragma unroll 8
  for (int i = 0; i < K; ++i) {
    float xi[TP_R];
    *reinterpret_cast<float4*>(xi) = *reinterpret_cast<const float4*>(xs + 4 * i);
    const float* w = W + (size_t)i * ldw;
    const float wa = has0 ? w[lane] : 0.0f, wb = has1 ? w[lane + 32] : 0.0f;
#pragma unroll
    for (int r = 0; r < TP_R; ++r) {
      if (has0) y0[r] = fmaf(xi[r], wa, y0[r]);
      if (has1) y1[r] = fmaf(xi[r], wb, y1[r]);
    }
  }
}
__device__ __forceinline__ void tp_self_attn_rows(const float* __restrict__ blob, const TpAttn& A, const TpNorm& N, float* __restrict__ xs, int lane,
                                                  float (&x0)[TP_R], float (&x1)[TP_R]) {
  float v0[TP_R], v1[TP_R], o0[TP_R], o1[TP_R];
  tp_stage_rows(xs, lane, x0, x1);
  tp_warp_matvec_r<TP_D>(xs, blob + A.w_in, 3 * TP_D, 2 * TP_D, blob + A.b_in + 2 * TP_D, TP_D, lane, v0, v1);
  tp_stage_rows(xs, lane, v0, v1);
  tp_warp_matvec_r<TP_D>(xs, blob + A.w_out, TP_D, 0, blob + A.b_out, TP_D, lane, o0, o1);
#pragma unroll
  for (int r = 0; r < TP_R; ++r) {
    x0[r] += o0[r];
    x1[r] += o1[r];
    tp_ln_row_warp(x0[r], x1[r], blob + N.w, blob + N.b, lane);
  }
}
// mem: encoder memory of the FIRST of the warp's rows (consecutive clips: row r at mem + r * TP_S * TP_D); rows >= n_here are padding
// (they read the last valid clip's memory and their results are discarded by the caller).  scr: TP_XR_SCR floats owned by this warp.
__device__ __forceinline__ void tp_cross_attn_rows(const float* __restrict__ blob, const TpAttn& A, const TpNorm& N, const float* __restrict__ wk_t,
                                                   const float* __restrict__ mem, int n_here, float* __restrict__ scr, int lane,
                                                   float (&x0)[TP_R], float (&x1)[TP_R]) {
  const bool has1 = lane + 32 < TP_D;
  const float* Win = blob + A.w_in;   // [in 48][q 48 | k 48 | v 48]
  float* xs = scr;                                      // staging [48][TP_R]
  float* hr = xs + TP_D * TP_R;                         // [TP_R][TP_H][TP_XA_STRIDE]
  float* ms = hr + TP_R * TP_H * TP_XA_STRIDE;          // one clip's memory rows
  float* as = ms + TP_S * TP_XA_STRIDE;                 // its probabilities a[s][h]
  static_assert((TP_D * TP_R) % 4 == 0 && (TP_R * TP_H * TP_XA_STRIDE) % 4 == 0 && (TP_S * TP_XA_STRIDE) % 4 == 0, "16-byte aligned scratch parts");
  float q0[TP_R], q1[TP_R];
  tp_stage_rows(xs, lane, x0, x1);
  tp_warp_matvec_r<TP_D>(xs, Win, 3 * TP_D, 0, blob + A.b_in, TP_D, lane, q0, q1);
  tp_stage_rows(xs, lane, q0, q1);
  // qt_{r,h}[c] = (1 / sqrt(12)) sum_{d in head h} W_k[d][c] q_r[d]; this lane owns c = lane and c = lane + 32
  {
    const float scale = rsqrtf((float)TP_HD);
#pragma unroll
    for (int h = 0; h < TP_H; ++h) {
      float a0[TP_R], a1[TP_R];
#pragma unroll
      for (int r = 0; r < TP_R; ++r) a0[r] = a1[r] = 0.0f;
#pragma unroll
      for (int j4 = 0; j4 < TP_HD; j4 += 4) {
        const int d = h * TP_HD + j4;
        float qk[4][TP_R];
#pragma unroll
        for (int j = 0; j < 4; ++j) *reinterpret_cast<float4*>(qk[j]) = *reinterpret_cast<const float4*>(xs + 4 * (d + j));
        const float wa0 = wk_t[d * TP_D + lane], wa1 = wk_t[(d + 1) * TP_D + lane], wa2 = wk_t[(d + 2) * TP_D + lane], wa3 = wk_t[(d + 3) * TP_D + lane];
        float wb0 = 0.f, wb1 = 0.f, wb2 = 0.f, wb3 = 0.f;
        if (has1) { wb0 = wk_t[d * TP_D + lane + 32]; wb1 = wk_t[(d + 1) * TP_D + lane + 32]; wb2 = wk_t[(d + 2) * TP_D + lane + 32]; wb3 = wk_t[(d + 3) * TP_D + lane + 32]; }
#pragma unroll
        for (int r = 0; r < TP_R; ++r) {
          a0[r] = fmaf(wa0, qk[0][r], fmaf(wa1, qk[1][r], fmaf(wa2, qk[2][r], fmaf(wa3, qk[3][r], a0[r]))));
          if (has1) a1[r] = fmaf(wb0, qk[0][r], fmaf(wb1, qk[1][r], fmaf(wb2, qk[2][r], fmaf(wb3, qk[3][r], a1[r]))));
        }
      }
#pragma unroll
      for (int r = 0; r < TP_R; ++r) {
        hr[(r * TP_H + h) * TP_XA_STRIDE + lane] = a0[r] * scale;
        if (has1) hr[(r * TP_H + h) * TP_XA_STRIDE + lane + 32] = a1[r] * scale;
      }
    }
  }
  // per clip: scores of key s on lane s (all heads), softmax across the lanes, weighted memory sums over its own folded queries
  // (the next clip's memory rows travel while this clip's scores are computed: a warp has few others to hide that latency behind)
  constexpr int kMemV = TP_S * (TP_D / 4), kMemPer = (kMemV + 31) / 32;
  float4 pre[kMemPer];
  auto fetch = [&](int r) {
    const float4* mr = reinterpret_cast<const float4*>(mem + (size_t)(r < n_here ? r : n_here - 1) * TP_S * TP_D);
#pragma unroll
    for (int j = 0; j < kMemPer; ++j) {
      const int i = lane + 32 * j;
      pre[j] = i < kMemV ? __ldcs(mr + i) : make_float4(0.f, 0.f, 0.f, 0.f);  // streamed once: keep the weights in L1
    }
  };
  fetch(0);
  for (int r = 0; r < TP_R; ++r) {
    float* hq = hr + r * TP_H * TP_XA_STRIDE;
    __syncwarp();  // folded queries published (first clip); the previous clip's readers of ms / as are done
#pragma unroll
    for (int j = 0; j < kMemPer; ++j) {
      const int i = lane + 32 * j;
      if (i < kMemV) reinterpret_cast<float4*>(ms + (i / (TP_D / 4)) * TP_XA_STRIDE)[i % (TP_D / 4)] = pre[j];
    }
    if (r + 1 < TP_R) fetch(r + 1);
    __syncwarp();
    {
      float a[TP_H];
      const bool key = lane < TP_S;
      float sc[TP_H] = {0.0f, 0.0f, 0.0f, 0.0f};
      const float4* mrow = reinterpret_cast<const float4*>(ms + (key ? lane : 0) * TP_XA_STRIDE);
#pragma unroll
      for (int c4 = 0; c4 < TP_D / 4; ++c4) {
        const float4 mv = mrow[c4];
#pragma unroll
        for (int h = 0; h < TP_H; ++h) {
          const float4 qv = reinterpret_cast<const float4*>(hq + h * TP_XA_STRIDE)[c4];
          sc[h] = fmaf(mv.x, qv.x, fmaf(mv.y, qv.y, fmaf(mv.z, qv.z, fmaf(mv.w, qv.w, sc[h]))));
        }
      }
#pragma unroll
      for (int h = 0; h < TP_H; ++h) {
        const float v = key ? sc[h] : -3.0e38f;
        float mx = v;
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        const float p = key ? expf(v - mx) : 0.0f;
        float sum = p;
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        a[h] = key ? p / sum : 0.0f;
      }
      if (key) *reinterpret_cast<float4*>(as + 4 * lane) = make_float4(a[0], a[1], a[2], a[3]);
    }
    __syncwarp();  // probabilities published; every lane has read this clip's folded queries: its per-head rows are free again
    {
      float b0[TP_H] = {0.0f, 0.0f, 0.0f, 0.0f}, b1[TP_H] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
      for (int s = 0; s < TP_S; ++s) {
        const float m0 = ms[s * TP_XA_STRIDE + lane], m1 = has1 ? ms[s * TP_XA_STRIDE + lane + 32] : 0.0f;
        const float4 av = *reinterpret_cast<const float4*>(as + 4 * s);  // broadcast
        b0[0] = fmaf(av.x, m0, b0[0]); b0[1] = fmaf(av.y, m0, b0[1]); b0[2] = fmaf(av.z, m0, b0[2]); b0[3] = fmaf(av.w, m0, b0[3]);
        b1[0] = fmaf(av.x, m1, b1[0]); b1[1] = fmaf(av.y, m1, b1[1]); b1[2] = fmaf(av.z, m1, b1[2]); b1[3] = fmaf(av.w, m1, b1[3]);
      }
#pragma unroll
      for (int h = 0; h < TP_H; ++h) {
        hq[h * TP_XA_STRIDE + lane] = b0[h];
        if (has1) hq[h * TP_XA_STRIDE + lane + 32] = b1[h];
      }
    }
  }
  __syncwarp();
  // o_r[d] = b_v[d] + sum_c W_v[c][d] mbar_{r,head(d)}[c]; this lane owns d = lane and d = lane + 32
  float o0[TP_R], o1[TP_R];
  {
    const float bv0 = blob[A.b_in + 2 * TP_D + lane], bv1 = has1 ? blob[A.b_in + 2 * TP_D + lane + 32] : 0.0f;
#pragma unroll
    for (int r = 0; r < TP_R; ++r) { o0[r] = bv0; o1[r] = bv1; }
    const float* mb0 = hr + (lane / TP_HD) * TP_XA_STRIDE;
    const float* mb1 = hr + ((has1 ? lane + 32 : lane) / TP_HD) * TP_XA_STRIDE;
    const float* wv = Win + 2 * TP_D;
#pragma unroll 2
    for (int c = 0; c < TP_D; c += 4) {
      float wa[4], wb[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        wa[j] = wv[(size_t)(c + j) * 3 * TP_D + lane];
        wb[j] = has1 ? wv[(size_t)(c + j) * 3 * TP_D + lane + 32] : 0.0f;
      }
#pragma unroll
      for (int r = 0; r < TP_R; ++r) {
        const float4 ma = *reinterpret_cast<const float4*>(mb0 + r * TP_H * TP_XA_STRIDE + c);
        o0[r] = fmaf(ma.w, wa[3], fmaf(ma.z, wa[2], fmaf(ma.y, wa[1], fmaf(ma.x, wa[0], o0[r]))));
        if (has1) {
          const float4 mb = *reinterpret_cast<const float4*>(mb1 + r * TP_H * TP_XA_STRIDE + c);
          o1[r] = fmaf(mb.w, wb[3], fmaf(mb.z, wb[2], fmaf(mb.y, wb[1], fmaf(mb.x, wb[0], o1[r]))));
        }
      }
    }
  }
  float y0[TP_R], y1[TP_R];
  tp_stage_rows(xs, lane, o0, o1);
  tp_warp_matvec_r<TP_D>(xs, blob + A.w_out, TP_D, 0, blob + A.b_out, TP_D, lane, y0, y1);
#pragma unroll
  for (int r = 0; r < TP_R; ++r) {
    x0[r] += y0[r];
    x1[r] += y1[r];
    tp_ln_row_warp(x0[r], x1[r], blob + N.w, blob + N.b, lane);
  }
}
// prediction head on a finished last-token row (drag_pose.py:275-289): appends the standardised prediction to the decoder inputs
// and writes the de-standardised one into target_buf with the step-function up-sampling
__device__ __forceinline__ void tp_out_head_row(const float* __restrict__ blob, const TpFfTail& t, int b, int T, int lane, float x0, float x1) {
  float a, unused;
  tp_warp_matvec<TP_D>(x0, x1, blob + t.out_w, TP_LAT, 0, blob + t.out_b, TP_LAT, lane, a, unused);
  if (lane >= TP_LAT) return;
  if (T < TP_MAXT) t.dec_lat[((size_t)b * TP_MAXT + T) * TP_LAT + lane] = a;
  const float val = a * t.sigma[lane] + t.mu[lane];
  float* tb = t.target_buf + (size_t)b * (t.window + 1) * TP_LAT;
  if (t.window == 0) {
    tb[lane] = val;
  } else if (t.step_i >= 4) {
    for (int r = t.step_i - 4; r < t.step_i; ++r) tb[r * TP_LAT + lane] = val;
    if (t.step_i == t.window) tb[t.window * TP_LAT + lane] = val;
  }
}

// LayerNorm of one 48-wide row held by one thread (eps 1e-5, torch nn.LayerNorm)
__device__ __forceinline__ void ln48(float (&v)[TP_D], const float* __restrict__ w, const float* __restrict__ b) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < TP_D; ++i) s += v[i];
  const float mean = s * (1.0f / TP_D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < TP_D; ++i) { v[i] -= mean; q = fmaf(v[i], v[i], q); }
  const float rstd = rsqrtf(q * (1.0f / TP_D) + 1e-5f);
#pragma unroll
  for (int i = 0; i < TP_D; ++i) v[i] = v[i] * rstd * w[i] + b[i];
}
#endif
