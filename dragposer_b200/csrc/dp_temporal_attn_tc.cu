// dp_temporal_attn_tc.cu -- launches of the tensor-core attention block (dp_temporal_attn_tc.cuh): encoder self-attention and
// decoder self- and cross-attention.
#include <cuda_fp16.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "dp_temporal_attn_tc.cuh"

using namespace tpa;

namespace {

template <int SMAX>
__global__ void __launch_bounds__(kThreads, 2)
tp_attn_tc_kernel(const unsigned char* __restrict__ wimg, const float* __restrict__ blob, TpNorm N1, const float* xq_g, int T, int q_stride,
                  const float* xkv_g, int S, int kv_stride, int n_clips, int G, float* out_g, long long* __restrict__ trace) {
  extern __shared__ __align__(1024) unsigned char raw[];
  Smem& S_ = *reinterpret_cast<Smem*>(raw);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (trace && blockIdx.x == 0 && tid == 0) trace[0] = clock64();
  if (tid == 0) {
    attn_init_barriers(S_);
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc(&S_.tmem_base, kT_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = S_.tmem_base;
  attn_tile<SMAX>(S_, tmem, wimg, blob, N1, xq_g, T, q_stride, xkv_g, S, kv_stride, n_clips, G, blockIdx.x * G, out_g, trace);
  if (warp == 8) tmem_dealloc(tmem, kT_COLS);
}

}  // namespace

// Host: build the pre-split, pre-tiled weight image of one self-attention block (ATT_LAYER_BYTES).
// w_in_t is [48][144] (in, out = q|k|v), w_out_t is [48][48] (in, out) -- the transposed layout of the blob.
void dp_attn_tc_pack(const float* w_in_t, const float* b_in, const float* w_out_t, const float* b_out, unsigned char* dst) {
  auto put = [&](unsigned char* base, uint32_t piece_bytes, uint32_t lbo, int N, const float* wt) {
    __half* pc[2] = {reinterpret_cast<__half*>(base), reinterpret_cast<__half*>(base + piece_bytes)};
    for (int n = 0; n < N; ++n)
      for (int k = 0; k < TP_D; ++k) {
        float r = kWScale * wt[(size_t)k * N + n];
        const uint32_t off = ((n >> 3) * kSBO + (k >> 3) * lbo + (n & 7) * 16 + (k & 7) * 2) / 2;
        for (int p = 0; p < 2; ++p) {
          pc[p][off] = __float2half_rn(r);
          r -= __half2float(pc[p][off]);
        }
      }
  };
  put(dst + kOffWin, kWinBytes, kWin_LBO, 3 * TP_D, w_in_t);
  put(dst + kOffWo, kWoBytes, kWo_LBO, TP_D, w_out_t);
  memcpy(dst + kOffBin, b_in, 3 * TP_D * sizeof(float));
  memcpy(dst + kOffBo, b_out, TP_D * sizeof(float));
}

template <int SMAX>
static cudaError_t launch_attn_t(const unsigned char* wimg, const float* blob, const TpNorm& N1, const float* xq, int T, int q_stride,
                                 const float* xkv, int S, int kv_stride, int n_clips, float* out, cudaStream_t st) {
  static std::atomic<unsigned long long> configured{0};
  const size_t smem = sizeof(Smem) + 1024;
  if (cudaError_t e = dp_ensure_smem(tp_attn_tc_kernel<SMAX>, smem, configured); e != cudaSuccess) return e;
  const int G = kTM / (T > S ? T : S);
  // debug: DP_ATTN_TRACE=n prints the phase clock of CTA 0 of the n-th launch
  static const int want_trace = getenv("DP_ATTN_TRACE") ? atoi(getenv("DP_ATTN_TRACE")) : 0;
  static int n_launch = 0;
  long long* trace = nullptr;
  if (want_trace && ++n_launch == want_trace && cudaMallocManaged(&trace, 16 * sizeof(long long)) == cudaSuccess) {
    memset(trace, 0, 16 * sizeof(long long));
    cudaMemPrefetchAsync(trace, 16 * sizeof(long long), 0, st);
  }
  tp_attn_tc_kernel<SMAX><<<(n_clips + G - 1) / G, kThreads, smem, st>>>(wimg, blob, N1, xq, T, q_stride, xkv, S, kv_stride, n_clips, G, out, trace);
  if (trace) {
    cudaStreamSynchronize(st);
    printf("attention trace (T %d, S %d, %d clips, G %d; cycles): setup+alloc %lld | tokens -> TMEM %lld | projections + K|V,Q epilogue %lld | attention %lld | "
           "output projection + LayerNorm %lld\n", T, S, n_clips, G, trace[1] - trace[0], trace[2] - trace[1], trace[3] - trace[2], trace[4] - trace[3],
           trace[5] - trace[4]);
    cudaFree(trace);
  }
  return cudaGetLastError();
}

// xq == xkv (T == S) selects self-attention; rows are addressed as (clip, token) with `stride` tokens per clip.
cudaError_t dp_attn_tc_launch(const unsigned char* wimg, const float* blob, const TpNorm& N1, const float* xq, int T, int q_stride,
                              const float* xkv, int S, int kv_stride, int n_clips, float* out, cudaStream_t st) {
  if (S <= 16) return launch_attn_t<16>(wimg, blob, N1, xq, T, q_stride, xkv, S, kv_stride, n_clips, out, st);
  return launch_attn_t<32>(wimg, blob, N1, xq, T, q_stride, xkv, S, kv_stride, n_clips, out, st);
}
