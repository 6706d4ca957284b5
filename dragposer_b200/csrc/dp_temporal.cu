// dp_temporal.cu -- temporal predictor (target-latent warm start) on the GPU, fp32.
//
// Restates drag_pose.py:246-290 + temporal_transformer.py:53-78 for B clips at once:
//   encoder tokens  = 14 x [ standardised latent(24) | sum of 4 displacements(3) | heights(6) ]
//   decoder tokens  = standardised latent of ring row 56, then the predictions so far
//   for i = 0,4,..,W: full decoder pass (NO causal mask), last token -> prediction@i
// The encoder memory is computed once per call (the reference recomputes the identical
// value on every autoregressive step).  The step-function "lerp" of drag_pose.py:282-289
// is applied while writing target_buf: prediction@i lands in rows i-4..i-1 (and row W).
#include <cstdlib>
#include <cstring>

#include "dp_common.cuh"
#include "dp_temporal.cuh"
#include "dp_internal.h"

namespace {

__device__ __forceinline__ void layer_norm_row(float v0, float v1, bool has1, const float* __restrict__ w,
                                               const float* __restrict__ b, int lane, float& o0, float& o1) {
  // one warp normalises one 48-wide row: lane holds features lane and lane+32 (<48)
  const float s = warp_sum(v0 + (has1 ? v1 : 0.0f));
  const float mean = s * (1.0f / TP_D);
  const float d0 = v0 - mean, d1 = has1 ? v1 - mean : 0.0f;
  const float var = warp_sum(d0 * d0 + d1 * d1) * (1.0f / TP_D);
  const float rstd = rsqrtf(var + 1e-5f);
  o0 = d0 * rstd * w[lane] + b[lane];
  o1 = has1 ? d1 * rstd * w[lane + 32] + b[lane + 32] : 0.0f;
}

// ---- encoder token embedding + first decoder token (drag_pose.py:249-266, temporal_transformer.py:62-66): ring buffers -> 14 x 33
// inputs per clip -> Linear(33, 48) + positional encoding.  A CTA takes nine clips (126 tokens): the inputs are staged in shared
// memory, a thread owns one output feature and keeps its 33 weights in registers for 21 tokens.  (Round 1 launched one 192-thread CTA
// per clip: 31 us at 4 096 clips, most of it CTA turnover.)
#define EMB_CLIPS 9
#define EMB_THREADS 288
#define EMB_XS (TP_ENC_IN + 3)
__global__ void __launch_bounds__(EMB_THREADS) tp_embed_kernel(const float* __restrict__ blob, TpLayout L, const float* __restrict__ mu,
                                                               const float* __restrict__ sigma, const float* __restrict__ latent_buf,
                                                               const float* __restrict__ disp_buf, const float* __restrict__ height_buf, int head,
                                                               int n_clips, int v0, int J, float* __restrict__ enc, float* __restrict__ dec_lat) {
  // n_clips VIRTUAL clips starting at virtual index v0: virtual clip v is real clip v / J seen j = v % J frames ahead (its ring
  // buffers read j rows later) -- the look-ahead batching of dp_engine.cu; J = 1 is the plain case.  enc / dec_lat are indexed by
  // the local virtual clip, the ring buffers by the real clip.
  __shared__ float xs[EMB_CLIPS * TP_S * EMB_XS];
  const int tid = threadIdx.x, clip0 = blockIdx.x * EMB_CLIPS;
  const int g_here = min(EMB_CLIPS, n_clips - clip0), rows = g_here * TP_S;
#pragma unroll 4  // the loads of four elements in flight (the gather is latency-bound: index arithmetic, then a dependent load)
  for (int idx = tid; idx < rows * TP_ENC_IN; idx += EMB_THREADS) {
    const int r = idx / TP_ENC_IN, i = idx % TP_ENC_IN, k = r % TP_S;
    const int v = v0 + clip0 + r / TP_S, ahead = v % J;
    const size_t b = (size_t)(v / J);
    const int slot = (head + 4 * k + ahead) % DP_PAST;
    float x;
    if (i < TP_LAT) {
      x = (latent_buf[(b * DP_PAST + slot) * DP_L + i] - mu[i]) / sigma[i];
    } else if (i < TP_LAT + 3) {
      x = 0.0f;
      for (int q = 0; q < 4; ++q) x += disp_buf[(b * DP_PAST + (head + 4 * k + q + ahead) % DP_PAST) * 3 + (i - TP_LAT)];
    } else {
      x = height_buf[(b * DP_PAST + slot) * DP_NH + (i - TP_LAT - 3)];
    }
    xs[r * EMB_XS + i] = x;
  }
  for (int idx = tid; idx < g_here * TP_LAT; idx += EMB_THREADS) {
    const int lv = clip0 + idx / TP_LAT, v = v0 + lv;
    const size_t b = (size_t)(v / J);
    const int i = idx % TP_LAT, slot = (head + 56 + v % J) % DP_PAST;
    dec_lat[(size_t)lv * TP_MAXT * TP_LAT + i] = (latent_buf[(b * DP_PAST + slot) * DP_L + i] - mu[i]) / sigma[i];
  }
  __syncthreads();
  const int f = tid % TP_D, rg = tid / TP_D;  // 6 row groups
  float w[TP_ENC_IN];
#pragma unroll
  for (int i = 0; i < TP_ENC_IN; ++i) w[i] = blob[L.enc_in_w + i * TP_D + f];
  const float bias = blob[L.enc_in_b + f];
  for (int r = rg; r < rows; r += EMB_THREADS / TP_D) {
    float a = bias;
#pragma unroll
    for (int i = 0; i < TP_ENC_IN; ++i) a = fmaf(xs[r * EMB_XS + i], w[i], a);
    enc[((size_t)clip0 * TP_S + r) * TP_D + f] = a + blob[L.pe + (r % TP_S) * TP_D + f];
  }
}

__global__ void tp_dec_embed_kernel(const float* __restrict__ blob, TpLayout L, const float* __restrict__ dec_lat, int T,
                                    float* __restrict__ dec) {
  __shared__ float x[TP_MAXT][TP_LAT];
  const int b = blockIdx.x, tid = threadIdx.x;
  for (int idx = tid; idx < T * TP_LAT; idx += blockDim.x) x[idx / TP_LAT][idx % TP_LAT] = dec_lat[(size_t)b * TP_MAXT * TP_LAT + idx];
  __syncthreads();
  const float* W = blob + L.dec_in_w;
  for (int idx = tid; idx < T * TP_D; idx += blockDim.x) {
    const int t = idx / TP_D, f = idx % TP_D;
    float a = blob[L.dec_in_b + f];
    for (int i = 0; i < TP_LAT; ++i) a = fmaf(x[t][i], W[i * TP_D + f], a);
    dec[((size_t)b * TP_MAXT + t) * TP_D + f] = a + blob[L.pe + t * TP_D + f];
  }
}

// ---- the same embedding for the look-ahead batching (J > 1 virtual clips per real clip): the J views of a clip, J consecutive shifts of
// its ring buffers, touch every ring row of the clip exactly once between them (token k of shift j is row 4k + j), so instead of
// gathering 33 inputs per token from global memory -- index arithmetic, then a dependent load, per element -- a CTA copies the WHOLE
// ring of its (at most three) real clips into shared memory with coalesced 16-byte loads, standardising the latents on the way, and
// every token reads its inputs from there.  Eight virtual clips (112 tokens) per CTA.  Each value is computed by the same operations
// in the same order as in tp_embed_kernel (which stays for J = 1 and as the cross-check, DP_EMBED_RING=0): bitwise the same tokens.
#define EMBR_CLIPS 8
#define EMBR_REAL 3
#define EMBR_THREADS 288
__global__ void __launch_bounds__(EMBR_THREADS) tp_embed_ring_kernel(const float* __restrict__ blob, TpLayout L, const float* __restrict__ mu,
                                                                     const float* __restrict__ sigma, const float* __restrict__ latent_buf,
                                                                     const float* __restrict__ disp_buf, const float* __restrict__ height_buf, int head,
                                                                     int n_clips, int v0, int J, float* __restrict__ enc, float* __restrict__ dec_lat) {
  __shared__ __align__(16) float lat[EMBR_REAL][DP_PAST * DP_L];   // standardised latents, physical slot order
  __shared__ __align__(16) float dsp[EMBR_REAL][DP_PAST * 3];
  __shared__ __align__(16) float hgt[EMBR_REAL][DP_PAST * DP_NH];
  const int tid = threadIdx.x, clip0 = blockIdx.x * EMBR_CLIPS;
  const int g_here = min(EMBR_CLIPS, n_clips - clip0), rows = g_here * TP_S;
  const int real0 = (v0 + clip0) / J, n_real = (v0 + clip0 + g_here - 1) / J - real0 + 1;  // <= EMBR_REAL for J >= 4
  for (int idx = tid; idx < n_real * (DP_PAST * DP_L / 4); idx += EMBR_THREADS) {
    const int c = idx / (DP_PAST * DP_L / 4), q = idx % (DP_PAST * DP_L / 4), i = (4 * q) % DP_L;  // DP_L is a multiple of 4
    const float4 v = reinterpret_cast<const float4*>(latent_buf + (size_t)(real0 + c) * DP_PAST * DP_L)[q];
    reinterpret_cast<float4*>(lat[c])[q] = make_float4((v.x - mu[i]) / sigma[i], (v.y - mu[i + 1]) / sigma[i + 1], (v.z - mu[i + 2]) / sigma[i + 2],
                                                       (v.w - mu[i + 3]) / sigma[i + 3]);
  }
  for (int idx = tid; idx < n_real * (DP_PAST * 3 / 4); idx += EMBR_THREADS) {
    const int c = idx / (DP_PAST * 3 / 4), q = idx % (DP_PAST * 3 / 4);
    reinterpret_cast<float4*>(dsp[c])[q] = reinterpret_cast<const float4*>(disp_buf + (size_t)(real0 + c) * DP_PAST * 3)[q];
  }
  for (int idx = tid; idx < n_real * (DP_PAST * DP_NH / 4); idx += EMBR_THREADS) {
    const int c = idx / (DP_PAST * DP_NH / 4), q = idx % (DP_PAST * DP_NH / 4);
    reinterpret_cast<float4*>(hgt[c])[q] = reinterpret_cast<const float4*>(height_buf + (size_t)(real0 + c) * DP_PAST * DP_NH)[q];
  }
  __syncthreads();
  for (int idx = tid; idx < g_here * TP_LAT; idx += EMBR_THREADS) {
    const int lv = clip0 + idx / TP_LAT, v = v0 + lv, i = idx % TP_LAT;
    dec_lat[(size_t)lv * TP_MAXT * TP_LAT + i] = lat[v / J - real0][((head + 56 + v % J) % DP_PAST) * DP_L + i];
  }
  const int f = tid % TP_D, rg = tid / TP_D;  // 6 row groups
  float w[TP_ENC_IN];
#pragma unroll
  for (int i = 0; i < TP_ENC_IN; ++i) w[i] = blob[L.enc_in_w + i * TP_D + f];
  const float bias = blob[L.enc_in_b + f];
  for (int r = rg; r < rows; r += EMBR_THREADS / TP_D) {
    const int v = v0 + clip0 + r / TP_S, k = r % TP_S, ahead = v % J, c = v / J - real0;
    const int slot = (head + 4 * k + ahead) % DP_PAST;
    float a = bias;
    const float4* lr = reinterpret_cast<const float4*>(lat[c] + slot * DP_L);
#pragma unroll
    for (int i4 = 0; i4 < DP_L / 4; ++i4) {
      const float4 x = lr[i4];
      a = fmaf(x.x, w[4 * i4], a); a = fmaf(x.y, w[4 * i4 + 1], a); a = fmaf(x.z, w[4 * i4 + 2], a); a = fmaf(x.w, w[4 * i4 + 3], a);
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      float x = 0.0f;
#pragma unroll
      for (int q = 0; q < 4; ++q) x += dsp[c][((head + 4 * k + q + ahead) % DP_PAST) * 3 + i];
      a = fmaf(x, w[TP_LAT + i], a);
    }
#pragma unroll
    for (int i = 0; i < DP_NH; ++i) a = fmaf(hgt[c][slot * DP_NH + i], w[TP_LAT + 3 + i], a);
    enc[((size_t)clip0 * TP_S + r) * TP_D + f] = a + blob[L.pe + k * TP_D + f];
  }
}

// ---- single-token decoder pass, first kernel: embedding of the one decoder token + the first layer's self-attention block
// (one key: row-local, see TpFfTail) + its cross-attention block against the clip's encoder memory (tp_cross_attn_single); one warp
// per clip.
__global__ void __launch_bounds__(256) tp_dec_start_kernel(const float* __restrict__ blob, TpLayout L, const float* __restrict__ dec_lat,
                                                           const float* __restrict__ wk_t, const float* __restrict__ mem, int n_clips,
                                                           float* __restrict__ dec) {
  __shared__ __align__(16) float scr[8][TP_XA_SCR];
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= n_clips) return;
  const float lat = lane < TP_LAT ? dec_lat[(size_t)b * TP_MAXT * TP_LAT + lane] : 0.0f;
  float x0, x1;
  tp_warp_matvec<TP_LAT>(lat, 0.0f, blob + L.dec_in_w, TP_D, 0, blob + L.dec_in_b, TP_D, lane, x0, x1);
  x0 += blob[L.pe + lane];
  if (lane + 32 < TP_D) x1 += blob[L.pe + lane + 32];
  tp_self_attn_single_s(blob, L.dec[0].sa, L.dec[0].n1, scr[threadIdx.x >> 5] + (TP_H + TP_S) * TP_XA_STRIDE, lane, x0, x1);
  tp_cross_attn_single(blob, L.dec[0].ca, L.dec[0].n2, wk_t, mem + (size_t)b * TP_S * TP_D, scr[threadIdx.x >> 5], lane, x0, x1);
  float* dst = dec + (size_t)b * TP_MAXT * TP_D;
  dst[lane] = x0;
  if (lane + 32 < TP_D) dst[lane + 32] = x1;
}

// The same for TP_R clips per warp (tp_self_attn_rows / tp_cross_attn_rows: every weight is loaded once per four clips); bitwise the
// results of tp_dec_start_kernel, which stays as the cross-check (DP_DEC_ROWS=0).
__global__ void __launch_bounds__(128) tp_dec_start_rows_kernel(const float* __restrict__ blob, TpLayout L, const float* __restrict__ dec_lat,
                                                                const float* __restrict__ wk_t, const float* __restrict__ mem, int n_clips,
                                                                float* __restrict__ dec) {
  __shared__ __align__(16) float scr[4][TP_XR_SCR];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b0 = (blockIdx.x * 4 + warp) * TP_R;
  if (b0 >= n_clips) return;
  const int n_here = min(TP_R, n_clips - b0);
  float* xs = scr[warp];
  if (lane < TP_LAT) {
    float v[TP_R];
#pragma unroll
    for (int r = 0; r < TP_R; ++r) v[r] = dec_lat[(size_t)(b0 + min(r, n_here - 1)) * TP_MAXT * TP_LAT + lane];
    *reinterpret_cast<float4*>(xs + 4 * lane) = make_float4(v[0], v[1], v[2], v[3]);
  }
  __syncwarp();
  float x0[TP_R], x1[TP_R];
  tp_warp_matvec_asc_r<TP_LAT>(xs, blob + L.dec_in_w, TP_D, blob + L.dec_in_b, TP_D, lane, x0, x1);
  const bool has1 = lane + 32 < TP_D;
  const float pe0 = blob[L.pe + lane], pe1 = has1 ? blob[L.pe + lane + 32] : 0.0f;
#pragma unroll
  for (int r = 0; r < TP_R; ++r) {
    x0[r] += pe0;
    if (has1) x1[r] += pe1;
  }
  tp_self_attn_rows(blob, L.dec[0].sa, L.dec[0].n1, xs, lane, x0, x1);
  tp_cross_attn_rows(blob, L.dec[0].ca, L.dec[0].n2, wk_t, mem + (size_t)b0 * TP_S * TP_D, n_here, scr[warp], lane, x0, x1);
#pragma unroll
  for (int r = 0; r < TP_R; ++r) {
    if (r < n_here) {
      float* dst = dec + (size_t)(b0 + r) * TP_MAXT * TP_D;
      dst[lane] = x0[r];
      if (has1) dst[lane + 32] = x1[r];
    }
  }
}

// ---- out = LayerNorm(xq + MHA(xq, xkv, xkv)); one CTA (160 threads) per clip.
// Projections are register tiled: a thread owns ONE output feature and keeps the accumulators of up to 16
// tokens in registers, so every weight is fetched once per CTA (coalesced, L1/L2 resident) and every
// activation is a broadcast LDS.128.
#define MHA_THREADS 160
#define MHA_TT 16
template <int NT>
__device__ __forceinline__ void project_feature(const float (*x)[TP_D], int t0, int nt, const float* __restrict__ W, int ldw, int col,
                                                float bias, float (&acc)[NT]) {
#pragma unroll
  for (int t = 0; t < NT; ++t) acc[t] = bias;
#pragma unroll 2
  for (int i = 0; i < TP_D; i += 4) {
    const float w0 = W[(i + 0) * ldw + col], w1 = W[(i + 1) * ldw + col], w2 = W[(i + 2) * ldw + col], w3 = W[(i + 3) * ldw + col];
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      if (t < nt) {
        const float4 xv = *reinterpret_cast<const float4*>(&x[t0 + t][i]);
        acc[t] = fmaf(xv.x, w0, acc[t]);
        acc[t] = fmaf(xv.y, w1, acc[t]);
        acc[t] = fmaf(xv.z, w2, acc[t]);
        acc[t] = fmaf(xv.w, w3, acc[t]);
      }
    }
  }
}

template <int MQ, int MKV>
struct MhaSmem {
  float xq[MQ][TP_D], q[MQ][TP_D], o[MQ][TP_D];
  float xkv[MKV][TP_D], k[MKV][TP_D + 1], v[MKV][TP_D];
  float sc[MQ][TP_H][TP_MAXT + 1];  // attention scores / probabilities of a query row against its own clip's keys
};

// One CTA handles G clips: their G*T query rows and G*S key/value rows are projected together (register tiled per output
// feature), attention stays per clip.  Short sequences (decoder steps with T = 1..5) would otherwise launch 4096 CTAs that
// each have almost nothing to do; G packs them.  Every phase uses all 160 threads.
template <int MQ, int MKV>
__global__ void __launch_bounds__(MHA_THREADS) tp_mha_ln_kernel(const float* __restrict__ blob, TpAttn A, TpNorm N,
                                                                const float* __restrict__ xq_g, int T, int q_stride,
                                                                const float* __restrict__ xkv_g, int S, int kv_stride,
                                                                float* __restrict__ out_g, int n_clips, int G) {
  extern __shared__ __align__(16) unsigned char mha_raw[];
  MhaSmem<MQ, MKV>& M = *reinterpret_cast<MhaSmem<MQ, MKV>*>(mha_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b0 = blockIdx.x * G;
  const int g_here = min(G, n_clips - b0);
  const int RQ = g_here * T, RK = g_here * S;  // rows in this CTA
  float (*xq)[TP_D] = M.xq;
  float (*xkv)[TP_D] = M.xkv;
  float (*q)[TP_D] = M.q;
  float (*k)[TP_D + 1] = M.k;
  float (*v)[TP_D] = M.v;
  float (*o)[TP_D] = M.o;
  for (int idx = tid; idx < RQ * (TP_D / 4); idx += MHA_THREADS) {
    const int r = idx / (TP_D / 4), c4 = idx % (TP_D / 4);
    reinterpret_cast<float4*>(&xq[r][0])[c4] = reinterpret_cast<const float4*>(xq_g + ((size_t)(b0 + r / T) * q_stride + r % T) * TP_D)[c4];
  }
  for (int idx = tid; idx < RK * (TP_D / 4); idx += MHA_THREADS) {
    const int r = idx / (TP_D / 4), c4 = idx % (TP_D / 4);
    reinterpret_cast<float4*>(&xkv[r][0])[c4] = reinterpret_cast<const float4*>(xkv_g + ((size_t)(b0 + r / S) * kv_stride + r % S) * TP_D)[c4];
  }
  __syncthreads();
  const float* Win = blob + A.w_in;
  if (tid < 3 * TP_D) {  // feature tid of [q | k | v]
    const bool is_q = tid < TP_D;
    const int n_tok = is_q ? RQ : RK;
    const float (*src)[TP_D] = is_q ? xq : xkv;
    const float bias = blob[A.b_in + tid];
    const float scale = is_q ? rsqrtf((float)TP_HD) : 1.0f;
    for (int t0 = 0; t0 < n_tok; t0 += MHA_TT) {
      float acc[MHA_TT];
      const int nt = min(MHA_TT, n_tok - t0);
      project_feature<MHA_TT>(src, t0, nt, Win, 3 * TP_D, tid, bias, acc);
#pragma unroll
      for (int t = 0; t < MHA_TT; ++t)
        if (t < nt) {
          if (is_q) q[t0 + t][tid] = acc[t] * scale;
          else if (tid < 2 * TP_D) k[t0 + t][tid - TP_D] = acc[t];
          else v[t0 + t][tid - 2 * TP_D] = acc[t];
        }
    }
  }
  __syncthreads();
  for (int idx = tid; idx < RQ * TP_H * S; idx += MHA_THREADS) {  // scores of query row r against the S keys of its clip
    const int s = idx % S, h = (idx / S) % TP_H, r = idx / (S * TP_H);
    const float* kr = k[(r / T) * S + s];
    float a = 0.0f;
#pragma unroll
    for (int d = 0; d < TP_HD; ++d) a = fmaf(q[r][h * TP_HD + d], kr[h * TP_HD + d], a);
    M.sc[r][h][s] = a;
  }
  __syncthreads();
  for (int idx = tid; idx < RQ * TP_H; idx += MHA_THREADS) {  // softmax rows (max-subtracted, like torch)
    float* row = M.sc[idx / TP_H][idx % TP_H];
    float mx = -3.0e38f;
    for (int s = 0; s < S; ++s) mx = fmaxf(mx, row[s]);
    float den = 0.0f;
    for (int s = 0; s < S; ++s) {
      const float e = expf(row[s] - mx);
      row[s] = e;
      den += e;
    }
    const float inv = 1.0f / den;
    for (int s = 0; s < S; ++s) row[s] *= inv;
  }
  __syncthreads();
  for (int idx = tid; idx < RQ * TP_D; idx += MHA_THREADS) {  // weighted values
    const int f = idx % TP_D, r = idx / TP_D;
    const float* row = M.sc[r][f / TP_HD];
    const int kv0 = (r / T) * S;
    float a = 0.0f;
    for (int s = 0; s < S; ++s) a = fmaf(row[s], v[kv0 + s][f], a);
    o[r][f] = a;
  }
  __syncthreads();
  {  // output projection + residual, register tiled (48 features x 3 row groups); q is dead: reuse it for the sums
    const int f = tid % TP_D, grp = tid / TP_D;
    if (grp < 3) {
      const int per = (RQ + 2) / 3;
      const int t0 = grp * per, nt = max(0, min(per, RQ - t0));
      if (nt > 0) {
        float acc[11];  // ceil(32 / 3)
        project_feature<11>(o, t0, nt, blob + A.w_out, TP_D, f, blob[A.b_out + f], acc);
#pragma unroll
        for (int t = 0; t < 11; ++t)
          if (t < nt) q[t0 + t][f] = acc[t] + xq[t0 + t][f];
      }
    }
  }
  __syncthreads();
  for (int r = warp; r < RQ; r += MHA_THREADS / 32) {
    const bool has1 = lane + 32 < TP_D;
    float r0, r1;
    layer_norm_row(q[r][lane], has1 ? q[r][lane + 32] : 0.0f, has1, blob + N.w, blob + N.b, lane, r0, r1);
    float* dst = out_g + ((size_t)(b0 + r / T) * q_stride + r % T) * TP_D;
    dst[lane] = r0;
    if (has1) dst[lane + 32] = r1;
  }
}

template <int MQ, int MKV>
static cudaError_t launch_mha_t(const float* blob, const TpAttn& A, const TpNorm& N, const float* xq, int T, int q_stride, const float* xkv,
                                int S, int kv_stride, float* out, int B, cudaStream_t st) {
  static std::atomic<unsigned long long> configured{0};
  if (cudaError_t e = dp_ensure_smem(tp_mha_ln_kernel<MQ, MKV>, sizeof(MhaSmem<MQ, MKV>), configured); e != cudaSuccess) return e;
  int G = MQ / T < MKV / S ? MQ / T : MKV / S;
  G = G < 1 ? 1 : G;
  tp_mha_ln_kernel<MQ, MKV><<<(B + G - 1) / G, MHA_THREADS, sizeof(MhaSmem<MQ, MKV>), st>>>(blob, A, N, xq, T, q_stride, xkv, S, kv_stride, out, B, G);
  return cudaGetLastError();
}

static cudaError_t launch_mha(const float* blob, const TpAttn& A, const TpNorm& N, const float* xq, int T, int q_stride, const float* xkv,
                              int S, int kv_stride, float* out, int B, cudaStream_t st) {
  // (query rows, key rows) per CTA: short decoder self-attention packs 16/T clips, cross-attention min(16/T, 4) clips,
  // the 14-token encoder 2 clips; long decoder sequences fall back to one clip per CTA
  const bool cross = xq != xkv;
  if (cross && T <= 16) return launch_mha_t<16, 64>(blob, A, N, xq, T, q_stride, xkv, S, kv_stride, out, B, st);
  if (!cross && T <= 8) return launch_mha_t<16, 16>(blob, A, N, xq, T, q_stride, xkv, S, kv_stride, out, B, st);
  return launch_mha_t<32, 32>(blob, A, N, xq, T, q_stride, xkv, S, kv_stride, out, B, st);
}

// ---- out = LN(x + W2 relu(W1 x + b1) + b2) [then an optional second LayerNorm]; 64 tokens per CTA.
// Rows are addressed as (clip, token): row r -> clip r / T, token r % T, stride `row_stride` tokens per clip.
#define FF_TM 64
#define FF_HC 64
__global__ void __launch_bounds__(256) tp_ff_ln_kernel(const float* __restrict__ blob, TpFF F, TpNorm N, TpNorm N2, int has_n2,
                                                       const float* __restrict__ x_g, int n_rows, int T, int row_stride,
                                                       float* __restrict__ out_g) {
  extern __shared__ __align__(16) unsigned char ff_smem[];
  float (*w1s)[FF_HC] = reinterpret_cast<float (*)[FF_HC]>(ff_smem);
  float (*w2s)[TP_D] = reinterpret_cast<float (*)[TP_D]>(ff_smem + sizeof(float) * TP_D * FF_HC);
  float (*xs)[TP_D + 1] = reinterpret_cast<float (*)[TP_D + 1]>(ff_smem + sizeof(float) * 2 * TP_D * FF_HC);
  float (*hs)[FF_HC + 1] = reinterpret_cast<float (*)[FF_HC + 1]>(ff_smem + sizeof(float) * (2 * TP_D * FF_HC + FF_TM * (TP_D + 1)));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int row0 = blockIdx.x * FF_TM;
  for (int idx = tid; idx < FF_TM * TP_D; idx += 256) {
    const int r = idx / TP_D, f = idx % TP_D, row = row0 + r;
    float v = 0.0f;
    if (row < n_rows) v = x_g[((size_t)(row / T) * row_stride + row % T) * TP_D + f];
    xs[r][f] = v;
  }
  const int ty = tid >> 4, tx = tid & 15;       // phase A: 4 tokens x 4 hidden per thread
  const bool outer = tx < 12;                   // phase B: 4 tokens x 4 features, 12 x 16 threads
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
  const float* W1 = blob + F.w1;
  const float* W2 = blob + F.w2;
  for (int hc = 0; hc < TP_FF; hc += FF_HC) {
    __syncthreads();
    for (int idx = tid; idx < TP_D * FF_HC / 4; idx += 256) {
      const int kx = idx / (FF_HC / 4), c4 = idx % (FF_HC / 4);
      reinterpret_cast<float4*>(&w1s[kx][0])[c4] = *reinterpret_cast<const float4*>(W1 + (size_t)kx * TP_FF + hc + 4 * c4);
    }
    for (int idx = tid; idx < FF_HC * TP_D / 4; idx += 256)
      reinterpret_cast<float4*>(&w2s[0][0])[idx] = *reinterpret_cast<const float4*>(W2 + (size_t)hc * TP_D + 4 * idx);
    __syncthreads();
    float h[4][4];
    {
      const float4 bb = *reinterpret_cast<const float4*>(blob + F.b1 + hc + 4 * tx);
#pragma unroll
      for (int i = 0; i < 4; ++i) { h[i][0] = bb.x; h[i][1] = bb.y; h[i][2] = bb.z; h[i][3] = bb.w; }
    }
#pragma unroll 4
    for (int kx = 0; kx < TP_D; ++kx) {
      const float4 w = *reinterpret_cast<const float4*>(&w1s[kx][4 * tx]);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float xv = xs[4 * ty + i][kx];
        h[i][0] = fmaf(xv, w.x, h[i][0]); h[i][1] = fmaf(xv, w.y, h[i][1]);
        h[i][2] = fmaf(xv, w.z, h[i][2]); h[i][3] = fmaf(xv, w.w, h[i][3]);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) hs[4 * ty + i][4 * tx + j] = fmaxf(h[i][j], 0.0f);
    __syncthreads();
    if (outer) {
#pragma unroll 4
      for (int hx = 0; hx < FF_HC; ++hx) {
        const float4 w = *reinterpret_cast<const float4*>(&w2s[hx][4 * tx]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float hv = hs[4 * ty + i][hx];
          acc[i][0] = fmaf(hv, w.x, acc[i][0]); acc[i][1] = fmaf(hv, w.y, acc[i][1]);
          acc[i][2] = fmaf(hv, w.z, acc[i][2]); acc[i][3] = fmaf(hv, w.w, acc[i][3]);
        }
      }
    }
  }
  __syncthreads();
  if (outer) {
    const float4 bb = *reinterpret_cast<const float4*>(blob + F.b2 + 4 * tx);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float* d = &hs[4 * ty + i][4 * tx];  // reuse hs as the residual-sum tile
      d[0] = acc[i][0] + bb.x + xs[4 * ty + i][4 * tx];
      d[1] = acc[i][1] + bb.y + xs[4 * ty + i][4 * tx + 1];
      d[2] = acc[i][2] + bb.z + xs[4 * ty + i][4 * tx + 2];
      d[3] = acc[i][3] + bb.w + xs[4 * ty + i][4 * tx + 3];
    }
  }
  __syncthreads();
  for (int r = warp; r < FF_TM; r += 8) {
    const int row = row0 + r;
    if (row >= n_rows) continue;
    const bool has1 = lane + 32 < TP_D;
    float r0, r1;
    layer_norm_row(hs[r][lane], has1 ? hs[r][lane + 32] : 0.0f, has1, blob + N.w, blob + N.b, lane, r0, r1);
    if (has_n2) layer_norm_row(r0, r1, has1, blob + N2.w, blob + N2.b, lane, r0, r1);
    float* dst = out_g + ((size_t)(row / T) * row_stride + row % T) * TP_D;
    dst[lane] = r0;
    if (has1) dst[lane + 32] = r1;
  }
}

// ---- prediction head on the last decoder token; appends to the decoder inputs and
// writes the de-standardised prediction into target_buf with the step-function upsampling.
__global__ void tp_out_kernel(const float* __restrict__ blob, TpLayout L, const float* __restrict__ mu,
                              const float* __restrict__ sigma, const float* __restrict__ dec, int T, int step_i, int window,
                              float* __restrict__ dec_lat, float* __restrict__ target_buf) {
  const int b = blockIdx.x, f = threadIdx.x;
  if (f >= TP_LAT) return;
  const float* x = dec + ((size_t)b * TP_MAXT + (T - 1)) * TP_D;
  float a = blob[L.out_b + f];
  for (int i = 0; i < TP_D; ++i) a = fmaf(x[i], blob[L.out_w + i * TP_LAT + f], a);
  if (T < TP_MAXT) dec_lat[((size_t)b * TP_MAXT + T) * TP_LAT + f] = a;
  const float val = a * sigma[f] + mu[f];
  float* tb = target_buf + (size_t)b * (window + 1) * TP_LAT;
  if (window == 0) {
    tb[f] = val;
  } else if (step_i >= 4) {
    for (int r = step_i - 4; r < step_i; ++r) tb[r * TP_LAT + f] = val;
    if (step_i == window) tb[window * TP_LAT + f] = val;
  }
}

}  // namespace

static const size_t kFfSmem = sizeof(float) * (2 * TP_D * FF_HC + FF_TM * (TP_D + 1) + FF_TM * (FF_HC + 1));

// B virtual clips starting at virtual clip v0 (J virtual clips per real clip, see tp_embed_kernel); latent_buf / disp_buf /
// height_buf are the UNSHIFTED ring buffers, target_buf and the work buffers of `w` start at the part's first virtual clip.
static cudaError_t run_part(const float* blob, const TpLayout& L, const float* mu, const float* sigma, const float* latent_buf,
                            const float* disp_buf, const float* height_buf, int head, int B, int v0, int J, int window, float* target_buf,
                            const TpWork& w, size_t part_floats, const unsigned char* fftiles, cudaStream_t st, long long* launches,
                            int stage = 0) {  // stage 0: everything; 1: only the embedding (the one kernel that sees `head`); 2: the rest
  cudaError_t err = cudaSuccess;

  float* e = w.enc;
  float* e2 = w.enc2;
  const int enc_rows = B * TP_S;
  if (stage != 2) {
    const char* ring_env = getenv("DP_EMBED_RING");  // read on every call (test switch)
    if (J >= 4 && !(ring_env && ring_env[0] == '0'))
      tp_embed_ring_kernel<<<(B + EMBR_CLIPS - 1) / EMBR_CLIPS, EMBR_THREADS, 0, st>>>(blob, L, mu, sigma, latent_buf, disp_buf, height_buf, head, B, v0, J, w.enc, w.dec_lat);
    else
      tp_embed_kernel<<<(B + EMB_CLIPS - 1) / EMB_CLIPS, EMB_THREADS, 0, st>>>(blob, L, mu, sigma, latent_buf, disp_buf, height_buf, head, B, v0, J, w.enc, w.dec_lat);
    ++*launches;
    if (stage == 1) return cudaGetLastError();
  }
  for (int l = 0; l < TP_NENC; ++l) {
    if (fftiles)
      err = dp_attn_tc_launch(fftiles + DP_TC_ATT_OFFSET + (size_t)l * ATT_LAYER_BYTES, blob, L.enc[l].n1, e, TP_S, TP_S, e, TP_S, TP_S, B, e2, st);
    else
      err = launch_mha(blob, L.enc[l].sa, L.enc[l].n1, e, TP_S, TP_S, e, TP_S, TP_S, e2, B, st);
    if (err != cudaSuccess) return err;
    if (fftiles) {
      err = dp_ff_tc_launch(fftiles + (size_t)l * FFT_LAYER_BYTES, blob, L.enc[l].ff, L.enc[l].n2, L.enc_norm, l == TP_NENC - 1, e2,
                            enc_rows, TP_S, TP_S, e, w.ffpart, part_floats, w.num_sms, st, launches);
      if (err != cudaSuccess) return err;
      --*launches;  // counted again below
    } else {
      tp_ff_ln_kernel<<<(enc_rows + FF_TM - 1) / FF_TM, 256, kFfSmem, st>>>(blob, L.enc[l].ff, L.enc[l].n2, L.enc_norm,
                                                                      l == TP_NENC - 1, e2, enc_rows, TP_S, TP_S, e);
    }
    *launches += 2;
  }
  int T = 1;
  for (int i = 0; i <= window; i += 4, ++T) {
    if (fftiles && T == 1 && (size_t)4 * B * TP_D <= part_floats) {
      // single-token pass: embedding + self- and cross-attention of layer 0 in one small kernel, then per layer the feed-forward block
      // with the next layer's two attention blocks (or the prediction head) fused into its finishing kernel: 7 launches, none of them
      // an attention kernel (round 2 started at 17, then 10 with tcgen05 cross-attention launches)
      float* cur = w.dec;
      float* nxt = w.dec2;
      const float* wk_t = reinterpret_cast<const float*>(fftiles + DP_TC_XA_OFFSET);  // [layer][key feature][input]
      if (dp_dec_rows())
        tp_dec_start_rows_kernel<<<(B + 4 * TP_R - 1) / (4 * TP_R), 128, 0, st>>>(blob, L, w.dec_lat, wk_t, e, B, cur);
      else
        tp_dec_start_kernel<<<(B + 7) / 8, 256, 0, st>>>(blob, L, w.dec_lat, wk_t, e, B, cur);
      ++*launches;
      for (int l = 0; l < TP_NDEC; ++l) {
        TpFfTail tail;
        memset(&tail, 0, sizeof(tail));
        if (l + 1 < TP_NDEC) {
          tail.next_self_attn = 1;
          tail.sa = L.dec[l + 1].sa;
          tail.n1 = L.dec[l + 1].n1;
          tail.next_cross_attn = 1;
          tail.ca = L.dec[l + 1].ca;
          tail.n2 = L.dec[l + 1].n2;
          tail.wk_t = wk_t + (size_t)(l + 1) * TP_D * TP_D;
          tail.mem = e;
        } else {
          tail.out_head = 1;
          tail.out_w = L.out_w; tail.out_b = L.out_b;
          tail.mu = mu; tail.sigma = sigma;
          tail.dec_lat = w.dec_lat; tail.target_buf = target_buf;
          tail.step_i = i; tail.window = window;
        }
        err = dp_ff_tc_launch(fftiles + (size_t)(TP_NENC + l) * FFT_LAYER_BYTES, blob, L.dec[l].ff, L.dec[l].n3, L.dec_norm, l == TP_NDEC - 1, cur, B, 1,
                              TP_MAXT, nxt, w.ffpart, part_floats, w.num_sms, st, launches, &tail);
        if (err != cudaSuccess) return err;
        float* t = cur; cur = nxt; nxt = t;
      }
      continue;
    }
    tp_dec_embed_kernel<<<B, 128, 0, st>>>(blob, L, w.dec_lat, T, w.dec);
    ++*launches;
    float* d = w.dec;
    float* d2 = w.dec2;
    const int rows = B * T;
    for (int l = 0; l < TP_NDEC; ++l) {
      if (fftiles) {
        const unsigned char* att = fftiles + DP_TC_ATT_OFFSET;
        err = dp_attn_tc_launch(att + (size_t)(TP_NENC + l) * ATT_LAYER_BYTES, blob, L.dec[l].n1, d, T, TP_MAXT, d, T, TP_MAXT, B, d2, st);
        if (err != cudaSuccess) return err;
        err = dp_attn_tc_launch(att + (size_t)(TP_NENC + TP_NDEC + l) * ATT_LAYER_BYTES, blob, L.dec[l].n2, d2, T, TP_MAXT, e, TP_S, TP_S, B, d, st);
      } else {
        err = launch_mha(blob, L.dec[l].sa, L.dec[l].n1, d, T, TP_MAXT, d, T, TP_MAXT, d2, B, st);
        if (err != cudaSuccess) return err;
        err = launch_mha(blob, L.dec[l].ca, L.dec[l].n2, d2, T, TP_MAXT, e, TP_S, TP_S, d, B, st);
      }
      if (err != cudaSuccess) return err;
      if (fftiles) {
        err = dp_ff_tc_launch(fftiles + (size_t)(TP_NENC + l) * FFT_LAYER_BYTES, blob, L.dec[l].ff, L.dec[l].n3, L.dec_norm,
                              l == TP_NDEC - 1, d, rows, T, TP_MAXT, d2, w.ffpart, part_floats, w.num_sms, st, launches);
        if (err != cudaSuccess) return err;
        --*launches;  // counted again below
      } else {
        tp_ff_ln_kernel<<<(rows + FF_TM - 1) / FF_TM, 256, kFfSmem, st>>>(blob, L.dec[l].ff, L.dec[l].n3, L.dec_norm,
                                                                    l == TP_NDEC - 1, d, rows, T, TP_MAXT, d2);
      }
      float* t = d; d = d2; d2 = t;
      *launches += 3;
    }
    tp_out_kernel<<<B, 32, 0, st>>>(blob, L, mu, sigma, d, T, i, window, w.dec_lat, target_buf);
    ++*launches;
  }
  return cudaGetLastError();
}

struct TpGraphCache {
  struct Entry {
    int B, window, J, state;  // state: 0 seen once, -1 not capturable
    const void *blob, *fftiles, *mu, *sigma, *target;
    cudaGraphExec_t exec;
    long long launches;
  };
  static constexpr int kMax = 8;
  Entry e[kMax];
  int n = 0, next = 0;
  Entry* find(int B, int window, int J, const void* blob, const void* fftiles, const void* mu, const void* sigma, const void* target) {
    for (int i = 0; i < n; ++i)
      if (e[i].B == B && e[i].window == window && e[i].J == J && e[i].blob == blob && e[i].fftiles == fftiles && e[i].mu == mu &&
          e[i].sigma == sigma && e[i].target == target)
        return &e[i];
    return nullptr;
  }
  void add(int B, int window, int J, const void* blob, const void* fftiles, const void* mu, const void* sigma, const void* target) {
    Entry* s = n < kMax ? &e[n++] : &e[next++ % kMax];  // full: recycle round robin
    if (s->exec) cudaGraphExecDestroy(s->exec);
    *s = Entry{B, window, J, 0, blob, fftiles, mu, sigma, target, nullptr, 0};
  }
  void clear() {
    for (int i = 0; i < n; ++i)
      if (e[i].exec) cudaGraphExecDestroy(e[i].exec);
    n = next = 0;
  }
};
TpGraphCache* dp_temporal_graphs_create() {
  TpGraphCache* c = new TpGraphCache();
  memset(c->e, 0, sizeof(c->e));
  return c;
}
void dp_temporal_graphs_clear(TpGraphCache* c) { if (c) c->clear(); }
void dp_temporal_graphs_destroy(TpGraphCache* c) {
  if (!c) return;
  c->clear();
  delete c;
}

// The predictor of a batch of kPredSplitMin or more virtual clips runs as two parts on two streams: each kernel of a part has fewer
// tiles than the device has CTA slots, so the block scheduler interleaves the parts and fills the tail of one kernel with the head of
// the other (448 tiles on 296 slots otherwise leave a third, half-empty round in every encoder kernel).  Two parts measured faster
// than one or four (DESIGN.md section 3.2).
constexpr int kPredSplitMin = 2048;
// Hidden-split workspace of one part: a quarter of DP_FF_PART_FLOATS, not a half.  dp_ff_tc_launch picks the split from it, and with
// a half the decoder feed-forward of an 8 192-virtual-clip part would be split 8-fold instead of 4-fold: another summation order.
constexpr size_t kPredPartFloats = DP_FF_PART_FLOATS / 4;
cudaError_t dp_temporal_run(const float* blob, const TpLayout& L, const float* mu, const float* sigma,
                            const float* latent_buf, const float* disp_buf, const float* height_buf, int head, int n_real,
                            int window, float* target_buf, const TpWork& w, const unsigned char* fftiles, cudaStream_t st,
                            long long* launches, int J) {
  const int B = n_real * J;  // virtual clips
  cudaError_t err = cudaFuncSetAttribute(tp_ff_ln_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFfSmem);
  if (err != cudaSuccess) return err;
  if (!fftiles || B < kPredSplitMin) {
    // no replay while a pipeline clock is on: DP_FF_TRACE / DP_ATTN_TRACE synchronise inside a launch function, which a capture forbids
    static const bool use_graphs = !getenv("DP_FF_TRACE") && !getenv("DP_ATTN_TRACE");
    auto eager = [&](int stage) {
      return run_part(blob, L, mu, sigma, latent_buf, disp_buf, height_buf, head, B, 0, J, window, target_buf, w, DP_FF_PART_FLOATS, fftiles, st, launches, stage);
    };
    if (!use_graphs || !w.graphs) return eager(0);
    // replayable chain (see dp_internal.h): first call of a shape runs kernel by kernel (it also does the one-off function-attribute
    // set-up, which cannot be captured), the second one is captured, later ones replay
    const int variant = J | (dp_dec_rows() << 8);  // everything that changes which kernels the chain holds
    TpGraphCache::Entry* g = w.graphs->find(B, window, variant, blob, fftiles, mu, sigma, target_buf);
    if (!g) {
      w.graphs->add(B, window, variant, blob, fftiles, mu, sigma, target_buf);
      return eager(0);
    }
    if (g->state < 0) return eager(0);  // capture failed once (e.g. a caller's stream that cannot be captured): stay with plain launches
    if ((err = eager(1)) != cudaSuccess) return err;
    if (!g->exec) {
      long long n = 0;
      cudaGraph_t graph = nullptr;
      cudaError_t cerr = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
      if (cerr == cudaSuccess) {
        cerr = run_part(blob, L, mu, sigma, latent_buf, disp_buf, height_buf, head, B, 0, J, window, target_buf, w, DP_FF_PART_FLOATS, fftiles, st, &n, 2);
        const cudaError_t eerr = cudaStreamEndCapture(st, &graph);
        if (cerr == cudaSuccess) cerr = eerr;
      }
      if (cerr == cudaSuccess) cerr = cudaGraphInstantiate(&g->exec, graph, 0);
      if (graph) cudaGraphDestroy(graph);
      if (cerr != cudaSuccess) {
        cudaGetLastError();  // clear the sticky-free error of the failed capture
        g->exec = nullptr;
        g->state = -1;
        return eager(2);
      }
      g->launches = n;
    }
    if ((err = cudaGraphLaunch(g->exec, st)) != cudaSuccess) return err;
    *launches += g->launches;
    return cudaSuccess;
  }
  if ((err = cudaEventRecord(w.ev_fork, st)) != cudaSuccess) return err;
  const int per = (B + 1) / 2;
  for (int p = 0; p < 2; ++p) {
    const int b0 = p * per, nb = p == 0 ? per : B - per;
    cudaStream_t sp = p == 0 ? st : w.st_extra;
    if (p > 0 && (err = cudaStreamWaitEvent(sp, w.ev_fork, 0)) != cudaSuccess) return err;
    TpWork wp = w;
    wp.enc += (size_t)b0 * TP_S * TP_D; wp.enc2 += (size_t)b0 * TP_S * TP_D;
    wp.dec += (size_t)b0 * TP_MAXT * TP_D; wp.dec2 += (size_t)b0 * TP_MAXT * TP_D;
    wp.dec_lat += (size_t)b0 * TP_MAXT * TP_LAT;
    wp.ffpart += kPredPartFloats * p;
    err = run_part(blob, L, mu, sigma, latent_buf, disp_buf, height_buf, head, nb, b0, J, window, target_buf + (size_t)b0 * (window + 1) * TP_LAT, wp,
                   kPredPartFloats, fftiles, sp, launches);
    if (err != cudaSuccess) return err;
    if (p > 0) {
      if ((err = cudaEventRecord(w.ev_join, sp)) != cudaSuccess) return err;
      if ((err = cudaStreamWaitEvent(st, w.ev_join, 0)) != cudaSuccess) return err;
    }
  }
  return cudaSuccess;
}
