// dp_temporal_tc.cu -- launches of the tensor-core feed-forward block (dp_temporal_tc4.cuh) for every encoder and decoder layer,
// the finishing kernels of its hidden-split mode, and the host-side packing of its weight image.
#include <cuda_fp16.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "dp_temporal.cuh"
#include "dp_temporal_tc4.cuh"

using namespace tpf;

namespace {

// Grid: (row tiles, n_split).
__global__ void __launch_bounds__(kThreads, kCtasPerSm)
tp_ff_tc_kernel(const unsigned char* __restrict__ wimg, const float* __restrict__ blob, TpFF F, TpNorm N1, TpNorm N2, int has_n2,
                const float* x_g, int n_rows, int T, int row_stride, float* out_g, float* __restrict__ part, long long* __restrict__ trace) {
  extern __shared__ __align__(1024) unsigned char raw[];
  Smem& S = *reinterpret_cast<Smem*>(raw);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (trace && blockIdx.x == (unsigned)trace[3] && blockIdx.y == 0 && tid == 0) trace[7] = clock64();
  if (tid == 0) {
    ff_init_barriers(S);
    fence_barrier_init();
  }
  if (warp == kEpiThreads / 32) tmem_alloc(&S.tmem_base, kT_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = S.tmem_base;
  ff_tile(S, tmem, wimg, blob, F, N1, N2, has_n2, x_g, n_rows, T, row_stride, blockIdx.x * kTM, kTM, blockIdx.y, gridDim.y, out_g, part, trace);
  if (warp == kEpiThreads / 32) tmem_dealloc(tmem, kT_COLS);
}

// second half of the hidden-split mode: out = LN(x + sum of partials + b2) [+ second LayerNorm] [+ the TpFfTail work of a
// single-token decoder pass]; one warp per row, lane holds features lane and lane + 32 (< 48), so every load is a coalesced row segment
__global__ void __launch_bounds__(256)
tp_ff_finish_kernel(const float* __restrict__ blob, TpFF F, TpNorm N1, TpNorm N2, int has_n2, const float* __restrict__ x_g, int n_rows, int T,
                    int row_stride, const float* __restrict__ part, int n_split, float* __restrict__ out_g, const __grid_constant__ TpFfTail tail) {
  __shared__ __align__(16) float scr[8][TP_XA_SCR];
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const bool has1 = lane + 32 < TP_D;
  const size_t g = ((size_t)(row / T) * row_stride + row % T) * TP_D;
  float v0 = blob[F.b2 + lane] + x_g[g + lane], v1 = has1 ? blob[F.b2 + lane + 32] + x_g[g + lane + 32] : 0.0f;
  float a0 = 0.0f, a1 = 0.0f;
  for (int s = 0; s < n_split; ++s) {  // fixed order: the result does not depend on scheduling
    const float* p = part + ((size_t)s * n_rows + row) * TP_D;
    a0 += p[lane];
    if (has1) a1 += p[lane + 32];
  }
  v0 += a0;
  v1 += a1;
  tp_ln_row_warp(v0, v1, blob + N1.w, blob + N1.b, lane);
  if (has_n2) tp_ln_row_warp(v0, v1, blob + N2.w, blob + N2.b, lane);
  if (tail.next_self_attn) tp_self_attn_single_s(blob, tail.sa, tail.n1, scr[threadIdx.x >> 5] + (TP_H + TP_S) * TP_XA_STRIDE, lane, v0, v1);
  if (tail.next_cross_attn)  // T == 1: row == clip
    tp_cross_attn_single(blob, tail.ca, tail.n2, tail.wk_t, tail.mem + (size_t)row * TP_S * TP_D, scr[threadIdx.x >> 5], lane, v0, v1);
  out_g[g + lane] = v0;
  if (has1) out_g[g + lane + 32] = v1;
  if (tail.out_head) tp_out_head_row(blob, tail, row / T, T, lane, v0, v1);
}

// The finishing kernel of a single-token decoder pass (T == 1: row == clip) with TP_R rows per warp: the partial sums and LayerNorms
// row by row as above, then the next layer's two attention blocks (or the prediction head) with every weight loaded once per four
// rows (tp_self_attn_rows / tp_cross_attn_rows).  Bitwise the results of tp_ff_finish_kernel (DP_DEC_ROWS=0).
__global__ void __launch_bounds__(128)
tp_ff_finish_rows_kernel(const float* __restrict__ blob, TpFF F, TpNorm N1, TpNorm N2, int has_n2, const float* __restrict__ x_g, int n_rows,
                         int row_stride, const float* __restrict__ part, int n_split, float* __restrict__ out_g, const __grid_constant__ TpFfTail tail) {
  __shared__ __align__(16) float scr[4][TP_XR_SCR];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b0 = (blockIdx.x * 4 + warp) * TP_R;
  if (b0 >= n_rows) return;
  const int n_here = min(TP_R, n_rows - b0);
  const bool has1 = lane + 32 < TP_D;
  float v0[TP_R], v1[TP_R];
#pragma unroll
  for (int r = 0; r < TP_R; ++r) {
    const int row = b0 + min(r, n_here - 1);
    const size_t g = (size_t)row * row_stride * TP_D;
    v0[r] = blob[F.b2 + lane] + __ldcs(x_g + g + lane);  // rows and partial sums are streamed once: keep the weights in L1
    v1[r] = has1 ? blob[F.b2 + lane + 32] + __ldcs(x_g + g + lane + 32) : 0.0f;
    float a0 = 0.0f, a1 = 0.0f;
    for (int s = 0; s < n_split; ++s) {  // fixed order: the result does not depend on scheduling
      const float* p = part + ((size_t)s * n_rows + row) * TP_D;
      a0 += __ldcs(p + lane);
      if (has1) a1 += __ldcs(p + lane + 32);
    }
    v0[r] += a0;
    v1[r] += a1;
    tp_ln_row_warp(v0[r], v1[r], blob + N1.w, blob + N1.b, lane);
    if (has_n2) tp_ln_row_warp(v0[r], v1[r], blob + N2.w, blob + N2.b, lane);
  }
  if (tail.next_self_attn) tp_self_attn_rows(blob, tail.sa, tail.n1, scr[warp], lane, v0, v1);
  if (tail.next_cross_attn) tp_cross_attn_rows(blob, tail.ca, tail.n2, tail.wk_t, tail.mem + (size_t)b0 * TP_S * TP_D, n_here, scr[warp], lane, v0, v1);
#pragma unroll
  for (int r = 0; r < TP_R; ++r) {
    if (r < n_here) {
      const size_t g = (size_t)(b0 + r) * row_stride * TP_D;
      out_g[g + lane] = v0[r];
      if (has1) out_g[g + lane + 32] = v1[r];
    }
  }
  if (tail.out_head) {  // tp_out_head_row for the warp's rows
    float a[TP_R], unused[TP_R];
    tp_stage_rows(scr[warp], lane, v0, v1);
    tp_warp_matvec_asc_r<TP_D>(scr[warp], blob + tail.out_w, TP_LAT, blob + tail.out_b, TP_LAT, lane, a, unused);
    if (lane < TP_LAT) {
#pragma unroll
      for (int r = 0; r < TP_R; ++r) {
        if (r >= n_here) continue;
        const int b = b0 + r;
        if (1 < TP_MAXT) tail.dec_lat[((size_t)b * TP_MAXT + 1) * TP_LAT + lane] = a[r];
        const float val = a[r] * tail.sigma[lane] + tail.mu[lane];
        float* tb = tail.target_buf + (size_t)b * (tail.window + 1) * TP_LAT;
        if (tail.window == 0) {
          tb[lane] = val;
        } else if (tail.step_i >= 4) {
          for (int q = tail.step_i - 4; q < tail.step_i; ++q) tb[q * TP_LAT + lane] = val;
          if (tail.step_i == tail.window) tb[tail.window * TP_LAT + lane] = val;
        }
      }
    }
  }
}

}  // namespace

// Host: build the pre-split, pre-tiled weight image of one FF block (FFT_LAYER_BYTES).
// w1t is [48][2048] (in, out), w2t is [2048][48] (in, out) -- the transposed layout of the blob.
void dp_ff_tc_pack(const float* w1t, const float* b1, const float* w2t, unsigned char* dst) {
  memset(dst, 0, FFT_LAYER_BYTES);
  memcpy(dst, b1, TP_FF * sizeof(float));
  unsigned char* steps = dst + TP_FF * 4;
  for (int c = 0; c < kChunks; ++c) {
    // W1c as B operand [N = hidden][K = 48] -> second half of step c
    __half* w1p[2] = {reinterpret_cast<__half*>(steps + (size_t)c * kStepBytes + 2 * kW2Bytes),
                      reinterpret_cast<__half*>(steps + (size_t)c * kStepBytes + 2 * kW2Bytes + kW1Bytes)};
    for (int n = 0; n < kHC; ++n)
      for (int k = 0; k < TP_D; ++k) {
        float r = kFfWScale * w1t[(size_t)k * TP_FF + c * kHC + n];
        const uint32_t off = ((n >> 3) * kB_SBO + (k >> 3) * kW1_LBO + (n & 7) * 16 + (k & 7) * 2) / 2;
        for (int p = 0; p < 2; ++p) {
          w1p[p][off] = __float2half_rn(r);
          r -= __half2float(w1p[p][off]);
        }
      }
    // W2c as B operand [N = out 48][K = hidden chunk] -> first half of step c + kLag
    __half* w2p[2] = {reinterpret_cast<__half*>(steps + (size_t)(c + kLag) * kStepBytes),
                      reinterpret_cast<__half*>(steps + (size_t)(c + kLag) * kStepBytes + kW2Bytes)};
    for (int n = 0; n < TP_D; ++n)
      for (int k = 0; k < kHC; ++k) {
        float r = kFfWScale * w2t[(size_t)(c * kHC + k) * TP_D + n];
        const uint32_t off = ((n >> 3) * kB_SBO + (k >> 3) * kW2_LBO + (n & 7) * 16 + (k & 7) * 2) / 2;
        for (int p = 0; p < 2; ++p) {
          w2p[p][off] = __float2half_rn(r);
          r -= __half2float(w2p[p][off]);
        }
      }
  }
}

cudaError_t dp_ff_tc_launch(const unsigned char* wimg, const float* blob, const TpFF& F, const TpNorm& N1, const TpNorm& N2, int has_n2,
                            const float* x, int n_rows, int T, int row_stride, float* out, float* part, size_t part_floats, int num_sms,
                            cudaStream_t st, long long* launches, const TpFfTail* tail) {
  static std::atomic<unsigned long long> configured{0};
  const size_t smem = sizeof(Smem) + 1024;
  if (cudaError_t e = dp_ensure_smem(tp_ff_tc_kernel, smem, configured); e != cudaSuccess) return e;
  const int tiles = (n_rows + kTM - 1) / kTM;
  // hidden split: largest power of two that still leaves every CTA resident at once (kCtasPerSm per SM) and >= 4 chunks each
  int n_split = 1;
  constexpr int kMaxSplit = kChunks / 4;  // at least four chunks per CTA: 16
  while (n_split < kMaxSplit && tiles * n_split * 2 <= kCtasPerSm * num_sms && (size_t)(n_split * 2) * n_rows * TP_D <= part_floats) n_split *= 2;
  if (!part) n_split = 1;
  if (tail) {  // the tail runs in the finish kernel: keep the split path even for a batch that would fill the device unsplit
    if (!part || T != 1 || (size_t)4 * n_rows * TP_D > part_floats) return cudaErrorInvalidValue;
    if (n_split < 2) n_split = 2;
  }
  // debug: DP_FF_TRACE=n prints the pipeline clock of CTA (0,0) of the n-th launch (cycles since its first H accumulator)
  static const int want_trace = getenv("DP_FF_TRACE") ? atoi(getenv("DP_FF_TRACE")) : 0;
  static int n_launch = 0;
  long long* trace = nullptr;
  if (want_trace && ++n_launch == want_trace && cudaMallocManaged(&trace, kChunks * 8 * sizeof(long long)) == cudaSuccess) {
    memset(trace, 0, kChunks * 8 * sizeof(long long));
    trace[3] = getenv("DP_FF_TRACE_CTA") ? atoll(getenv("DP_FF_TRACE_CTA")) : 0;  // which tile's CTA is clocked (a later wave: > 2 x SMs)
    cudaMemPrefetchAsync(trace, kChunks * 8 * sizeof(long long), 0, st);
  }
  tp_ff_tc_kernel<<<dim3(tiles, n_split), kThreads, smem, st>>>(wimg, blob, F, N1, N2, has_n2, x, n_rows, T, row_stride, out, part, trace);
  ++*launches;
  if (trace) {
    cudaStreamSynchronize(st);
    const long long t0 = trace[4];
    printf("FF trace: kernel start %lld, end %lld, chunk 0 pieces computed %lld (cycles relative to the first H accumulator)\n", trace[7] - t0, trace[15] - t0,
           trace[11] - t0);
    printf("FF trace (%d rows, split %d): chunk | issuer: weights ready, pieces ready, issued | epilogue: H ready, loaded, stored\n", n_rows, n_split);
    for (int c = 0; c < kChunks / n_split; ++c)
      printf("  %2d | %7lld %7lld %7lld | %7lld %7lld %7lld\n", c, trace[c * 8] - t0, trace[c * 8 + 1] - t0, trace[c * 8 + 2] - t0, trace[c * 8 + 4] - t0,
             trace[c * 8 + 5] - t0, trace[c * 8 + 6] - t0);
    cudaFree(trace);
  }
  if (n_split > 1) {
    TpFfTail t;
    memset(&t, 0, sizeof(t));
    if (tail) t = *tail;
    if (tail && T == 1 && dp_dec_rows())
      tp_ff_finish_rows_kernel<<<(n_rows + 4 * TP_R - 1) / (4 * TP_R), 128, 0, st>>>(blob, F, N1, N2, has_n2, x, n_rows, row_stride, part, n_split, out, t);
    else
      tp_ff_finish_kernel<<<(n_rows + 7) / 8, 256, 0, st>>>(blob, F, N1, N2, has_n2, x, n_rows, T, row_stride, part, n_split, out, t);
    ++*launches;
  }
  return cudaGetLastError();
}
