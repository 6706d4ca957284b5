// dp_frame_simt.cu -- persistent per-frame optimisation kernel, fp32 CUDA-core decoder.
//
// One launch runs a whole frame of DragPose.run (python/src/drag_pose.py:196-414) for
// every clip: up to max_iter x { decoder forward, forward kinematics, masked tracker
// loss, reverse-mode adjoint, decoder backward, latent Adam step } with per-clip early
// stopping, then the frame epilogue (root update, joint adjustment, ring-buffer push,
// output pose).  No host round trips inside the frame.
//
// Mapping: one warp owns CPW clips.  Decoder phases process the CPW clips together
// (each weight fetched from shared memory feeds CPW FMAs); kinematics phases run one
// clip at a time with lane == joint: the joint hierarchy lives in shared memory
// (DpModelImage), positions accumulate along the parent chain with log-step warp
// shuffles (ancestor pointer jumping), subtree sums of the adjoint use a warp scan over
// the pre-order joint numbering.  Arithmetic follows SURVEY.md appendix B (closed form of
// python/src/utils.py:80-149 + python/src/drag_pose.py:66-194).
#include "dp_common.cuh"
#include "dp_fk.cuh"
#include "dp_internal.h"

namespace {

template <int CPW, int K, int N>
__device__ __forceinline__ void dense_pairs(const float* __restrict__ W, const float* __restrict__ bias,
                                            const float* __restrict__ in, float (&acc)[CPW][3], int lane) {
  // out[o] = bias[o] + sum_k W[k][o] in[k];  lane owns o = 2*lane, 2*lane+1 (< min(N,64)) and 64+lane (< N)
  constexpr bool THIRD = (N > 64);
  const bool pa = (2 * lane < N) && (lane < 32);
  const int o = pa ? 2 * lane : 0;
  const bool pt = THIRD && (64 + lane < N);
  const int o3 = pt ? 64 + lane : 0;
#pragma unroll
  for (int c = 0; c < CPW; ++c) {
    acc[c][0] = bias ? bias[o] : 0.0f;
    acc[c][1] = bias ? bias[o + 1] : 0.0f;
    acc[c][2] = (THIRD && bias) ? bias[o3] : 0.0f;
  }
#pragma unroll 2
  for (int k = 0; k < K; k += 4) {
    float4 a[CPW];
#pragma unroll
    for (int c = 0; c < CPW; ++c) a[c] = *reinterpret_cast<const float4*>(in + c * 2 * DP_SCRATCH + k);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const float2 w = *reinterpret_cast<const float2*>(W + (k + kk) * N + o);
      float w3 = 0.0f;
      if (THIRD) w3 = W[(k + kk) * N + o3];
#pragma unroll
      for (int c = 0; c < CPW; ++c) {
        const float av = kk == 0 ? a[c].x : kk == 1 ? a[c].y : kk == 2 ? a[c].z : a[c].w;
        acc[c][0] = fmaf(w.x, av, acc[c][0]);
        acc[c][1] = fmaf(w.y, av, acc[c][1]);
        if (THIRD) acc[c][2] = fmaf(w3, av, acc[c][2]);
      }
    }
  }
}

template <int CPW>
__global__ void __launch_bounds__(512, 1) dp_frame_simt_kernel(const __grid_constant__ DpFrameArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  DpModelImage& M = *reinterpret_cast<DpModelImage*>(smem_raw);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + sizeof(DpModelImage));
  float* scratch_base = reinterpret_cast<float*>(smem_raw + sizeof(DpModelImage) + 16);
  const int warps = blockDim.x >> 5;
  ClipTrackers* trk_base = reinterpret_cast<ClipTrackers*>(scratch_base + warps * CPW * 2 * DP_SCRATCH);

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // ---- model image -> shared memory: one bulk TMA copy per CTA
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    constexpr uint32_t kBytes = (uint32_t)sizeof(DpModelImage);
    constexpr uint32_t kChunk = 32768;
    mbar_expect_tx(bar, kBytes);
    for (uint32_t o = 0; o < kBytes; o += kChunk)
      tma_bulk_g2s(smem_raw + o, reinterpret_cast<const unsigned char*>(A.model) + o, min(kChunk, kBytes - o), bar);
  }

  float* sa = scratch_base + (warp * CPW) * 2 * DP_SCRATCH;  // clip c: ping = sa + c*2*S, pong = +S
  float* sb = sa + DP_SCRATCH;
  ClipTrackers* trk = trk_base + (warp * CPW) * 32;
  const int clip0 = (blockIdx.x * warps + warp) * CPW;

  // ---- per-clip frame inputs
  bool valid[CPW];
  float g[CPW][4], inv3e[CPW], lrot9e[CPW], gpos_y[CPW];
  float2 z[CPW], tl[CPW], am[CPW], av[CPW], zlast[CPW];
#pragma unroll
  for (int c = 0; c < CPW; ++c) {
    const int clip = clip0 + c;
    valid[c] = clip < A.n_clips;
    const int cc = valid[c] ? clip : 0;
    int ne = A.n_ee ? A.n_ee[cc] : A.ee_stride;
    ne = max(1, min(ne, A.ee_stride));
    gpos_y[c] = A.ext_mask ? A.gpos[cc * 3 + 1] : 0.0f;
    inv3e[c] = 1.0f / (3.0f * (float)ne);
    lrot9e[c] = A.uniform.lambda_rot / (9.0f * (float)ne);
#pragma unroll
    for (int i = 0; i < 4; ++i) g[c][i] = A.grot[cc * 4 + i];
    z[c] = tl[c] = make_float2(0.f, 0.f);
    if (lane < DP_L / 2) {
      z[c] = reinterpret_cast<const float2*>(A.latent + (size_t)cc * DP_L)[lane];
      tl[c] = reinterpret_cast<const float2*>(A.target_buf + ((size_t)cc * A.target_rows + A.target_index) * DP_L)[lane];
    }
    am[c] = av[c] = make_float2(0.f, 0.f);
    zlast[c] = z[c];
    // tracker rows: lane j picks the slot that tracks joint j (joints are unique per clip)
    ClipTrackers row;
    row.pw = row.r0 = row.r1 = row.r2 = make_float4(0.f, 0.f, 0.f, 0.f);
    float origin[3] = {0.f, 0.f, 0.f};  // world-absolute targets are taken relative to the clip's current global position
    if (A.targets_world) { origin[0] = A.gpos[cc * 3]; origin[1] = A.gpos[cc * 3 + 1]; origin[2] = A.gpos[cc * 3 + 2]; }
    const int32_t* jn = A.joints + (A.shared_trackers ? 0 : (size_t)cc * A.ee_stride);
    const float* wt = A.weights + (A.shared_trackers ? 0 : (size_t)cc * A.ee_stride * 2);
    for (int e = 0; e < ne; ++e) {
      if (jn[e] == lane) {
        const float* tp = A.tgt_pos + ((size_t)cc * A.ee_stride + e) * 3;
        const float* tr = A.tgt_rot + ((size_t)cc * A.ee_stride + e) * 9;
        row.pw = make_float4(tp[0] - origin[0], tp[1] - origin[1], tp[2] - origin[2], wt[2 * e]);
        row.r0 = make_float4(tr[0], tr[1], tr[2], wt[2 * e + 1]);
        row.r1 = make_float4(tr[3], tr[4], tr[5], 0.f);
        row.r2 = make_float4(tr[6], tr[7], tr[8], 0.f);
      }
    }
    trk[c * 32 + lane] = row;
  }
  mbar_wait(bar, 0);  // model image has landed
  __syncwarp();

  // ---- optimisation loop (drag_pose.py:296-355)
  bool active[CPW];
  double prev[CPW], incr[CPW];
  float lp[CPW], lr[CPW], lt[CPW];
  int iters[CPW];
#pragma unroll
  for (int c = 0; c < CPW; ++c) {
    active[c] = valid[c];
    prev[c] = 10000000.0;
    incr[c] = 1.0;
    lp[c] = lr[c] = lt[c] = __int_as_float(0x7f800000);
    iters[c] = 0;
  }
  const float lt_scale = A.uniform.lambda_t * (1.0f / (float)DP_L);
  for (int it = 0; it < A.max_iter; ++it) {
    bool any = false;
#pragma unroll
    for (int c = 0; c < CPW; ++c) {
      active[c] = active[c] && ((double)lp[c] > A.uniform.eps_pos || (double)lr[c] > A.uniform.eps_rot) && (incr[c] > A.uniform.min_incr);
      any = any || active[c];
    }
    if (!any) break;
    // decoder forward 24 -> 40 -> 60 -> 92
    float acc[CPW][3];
    unsigned neg0[CPW], neg1[CPW];  // LeakyReLU slope bits of the lane's pair
#pragma unroll
    for (int c = 0; c < CPW; ++c) {
      if (active[c]) zlast[c] = z[c];
      if (lane < DP_L / 2) reinterpret_cast<float2*>(sa + c * 2 * DP_SCRATCH)[lane] = z[c];
    }
    __syncwarp();
    dense_pairs<CPW, DP_L, DP_H0>(M.W0t, M.b0, sa, acc, lane);
#pragma unroll
    for (int c = 0; c < CPW; ++c) {
      neg0[c] = (acc[c][0] > 0.f ? 0u : 1u) | (acc[c][1] > 0.f ? 0u : 2u);
      if (2 * lane < DP_H0) reinterpret_cast<float2*>(sb + c * 2 * DP_SCRATCH)[lane] = make_float2(lrelu(acc[c][0]), lrelu(acc[c][1]));
    }
    __syncwarp();
    dense_pairs<CPW, DP_H0, DP_H1>(M.W1t, M.b1, sb, acc, lane);
#pragma unroll
    for (int c = 0; c < CPW; ++c) {
      neg1[c] = (acc[c][0] > 0.f ? 0u : 1u) | (acc[c][1] > 0.f ? 0u : 2u);
      if (2 * lane < DP_H1) reinterpret_cast<float2*>(sa + c * 2 * DP_SCRATCH)[lane] = make_float2(lrelu(acc[c][0]), lrelu(acc[c][1]));
    }
    __syncwarp();
    dense_pairs<CPW, DP_H1, DP_Y>(M.W2t, M.b2, sa, acc, lane);
#pragma unroll
    for (int c = 0; c < CPW; ++c) {
      float* yb = sb + c * 2 * DP_SCRATCH;
      reinterpret_cast<float2*>(yb)[lane] = make_float2(acc[c][0], acc[c][1]);
      if (64 + lane < DP_Y) yb[64 + lane] = acc[c][2];
    }
    __syncwarp();
    // kinematics + loss + adjoint, one clip at a time (lane == joint); ybar overwrites y
    float nlp[CPW], nlr[CPW], nle[CPW];
#pragma unroll
    for (int c = 0; c < CPW; ++c) {
      nlp[c] = lp[c];
      nlr[c] = lr[c];
      nle[c] = 0.0f;
      if (active[c]) {
        const FkOut o = fk_loss<true, false>(M, sb + c * 2 * DP_SCRATCH, trk + c * 32, g[c], inv3e[c], lrot9e[c], lane,
                                             nullptr, nullptr, nullptr, nullptr, FkExtra{A.ext_mask, A.floor_level, gpos_y[c]});
        nlp[c] = o.lp;
        nlr[c] = o.lr;
        nle[c] = o.le;
      }
    }
    __syncwarp();
    // decoder backward 92 -> 60 -> 40 -> 24 (data gradient only; the decoder is frozen)
    dense_pairs<CPW, DP_Y, DP_H1>(M.W2, nullptr, sb, acc, lane);
#pragma unroll
    for (int c = 0; c < CPW; ++c)
      if (2 * lane < DP_H1)
        reinterpret_cast<float2*>(sa + c * 2 * DP_SCRATCH)[lane] =
            make_float2(acc[c][0] * ((neg1[c] & 1u) ? 0.2f : 1.0f), acc[c][1] * ((neg1[c] & 2u) ? 0.2f : 1.0f));
    __syncwarp();
    dense_pairs<CPW, DP_H1, DP_H0>(M.W1, nullptr, sa, acc, lane);
#pragma unroll
    for (int c = 0; c < CPW; ++c)
      if (2 * lane < DP_H0)
        reinterpret_cast<float2*>(sb + c * 2 * DP_SCRATCH)[lane] =
            make_float2(acc[c][0] * ((neg0[c] & 1u) ? 0.2f : 1.0f), acc[c][1] * ((neg0[c] & 2u) ? 0.2f : 1.0f));
    __syncwarp();
    dense_pairs<CPW, DP_H0, DP_L>(M.W0, nullptr, sb, acc, lane);
    // temporal term, loss bookkeeping, Adam (torch/optim/adam.py single-tensor path)
    const float step_size = A.uniform.adam_tab[it], inv_bc2s = A.uniform.adam_tab[A.max_iter + it];  // lr/(1-b1^k), 1/sqrt(1-b2^k)
#pragma unroll
    for (int c = 0; c < CPW; ++c) {
      const float dx = z[c].x - tl[c].x, dy = z[c].y - tl[c].y;
      float s = (lane < DP_L / 2) ? fmaf(dx, dx, dy * dy) : 0.0f;
      s = warp_sum(s);
      const float nlt = s * lt_scale;
      const float gx = fmaf(2.0f * lt_scale, dx, acc[c][0]);
      const float gy = fmaf(2.0f * lt_scale, dy, acc[c][1]);
      if (A.trace && active[c]) {
        float* row = A.trace + ((size_t)(clip0 + c) * A.trace_iters + it) * 52;
        if (lane < DP_L / 2) {
          reinterpret_cast<float2*>(row)[lane] = z[c];
          reinterpret_cast<float2*>(row + DP_L)[lane] = make_float2(gx, gy);
        }
        if (lane == 0) { row[48] = nlp[c]; row[49] = nlr[c]; row[50] = nlt; row[51] = 1.0f; }
      }
      if (A.eval_only) {
        if (active[c] && lane < DP_L / 2) reinterpret_cast<float2*>(A.eval_grad + (size_t)(clip0 + c) * DP_L)[lane] = make_float2(gx, gy);
      } else if (active[c]) {
        am[c].x = fmaf(0.1f, gx - am[c].x, am[c].x);
        am[c].y = fmaf(0.1f, gy - am[c].y, am[c].y);
        av[c].x = av[c].x * 0.999f + (0.001f * gx) * gx;
        av[c].y = av[c].y * 0.999f + (0.001f * gy) * gy;
        z[c].x += __fdividef(-step_size * am[c].x, fmaf(fast_sqrt(av[c].x), inv_bc2s, 1e-8f));
        z[c].y += __fdividef(-step_size * am[c].y, fmaf(fast_sqrt(av[c].y), inv_bc2s, 1e-8f));
      }
      if (active[c]) {
        lp[c] = nlp[c];
        lr[c] = nlr[c];
        lt[c] = nlt;
        const float total = ((nlp[c] + nlr[c]) + nlt) + nle[c];  // drag_pose.py:338
        incr[c] = prev[c] - (double)total;
        prev[c] = (double)total;
        iters[c] += 1;
      }
    }
  }

  // ---- frame epilogue (drag_pose.py:369-414) from the LAST EVALUATED latent (pre-step)
#pragma unroll
  for (int c = 0; c < CPW; ++c)
    if (lane < DP_L / 2) reinterpret_cast<float2*>(sa + c * 2 * DP_SCRATCH)[lane] = zlast[c];
  __syncwarp();
  {
    float acc[CPW][3];
    dense_pairs<CPW, DP_L, DP_H0>(M.W0t, M.b0, sa, acc, lane);
#pragma unroll
    for (int c = 0; c < CPW; ++c)
      if (2 * lane < DP_H0) reinterpret_cast<float2*>(sb + c * 2 * DP_SCRATCH)[lane] = make_float2(lrelu(acc[c][0]), lrelu(acc[c][1]));
    __syncwarp();
    dense_pairs<CPW, DP_H0, DP_H1>(M.W1t, M.b1, sb, acc, lane);
#pragma unroll
    for (int c = 0; c < CPW; ++c)
      if (2 * lane < DP_H1) reinterpret_cast<float2*>(sa + c * 2 * DP_SCRATCH)[lane] = make_float2(lrelu(acc[c][0]), lrelu(acc[c][1]));
    __syncwarp();
    dense_pairs<CPW, DP_H1, DP_Y>(M.W2t, M.b2, sa, acc, lane);
#pragma unroll
    for (int c = 0; c < CPW; ++c) {
      float* yb = sb + c * 2 * DP_SCRATCH;
      reinterpret_cast<float2*>(yb)[lane] = make_float2(acc[c][0], acc[c][1]);
      if (64 + lane < DP_Y) yb[64 + lane] = acc[c][2];
    }
    __syncwarp();
  }
#pragma unroll
  for (int c = 0; c < CPW; ++c) {
    if (!valid[c]) continue;
    const int clip = clip0 + c;
    float q[4], r[4], p[3], d[3];
    fk_loss<false, true>(M, sb + c * 2 * DP_SCRATCH, trk + c * 32, g[c], inv3e[c], lrot9e[c], lane, q, r, p, d);
    if (A.eval_only) {
      if (lane < DP_J && A.eval_pos) {
        float* o = A.eval_pos + ((size_t)clip * DP_J + lane) * 3;
        o[0] = p[0]; o[1] = p[1]; o[2] = p[2];
      }
      if (lane == 0 && A.out_losses) { A.out_losses[clip * 3] = lp[c]; A.out_losses[clip * 3 + 1] = lr[c]; A.out_losses[clip * 3 + 2] = lt[c]; }
      continue;
    }
    // root update: current_global_pos += world_displacement (= p_0), current_global_rot = world_rotation
    float p0[3], gp[3], adj[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      p0[i] = __shfl_sync(0xffffffffu, p[i], 0);
      gp[i] = A.gpos[clip * 3 + i] + p0[i];
    }
    if (A.uniform.adj_joint >= 0) {  // joint adjustment (drag_pose.py:374-381)
      const float* tp = A.tgt_pos + ((size_t)clip * A.ee_stride + A.uniform.adj_slot) * 3;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const float pj = __shfl_sync(0xffffffffu, p[i], A.uniform.adj_joint);
        adj[i] = ((tp[i] - (A.targets_world ? A.gpos[clip * 3 + i] : 0.0f)) - pj) * A.uniform.adj_w;
        gp[i] += adj[i];
      }
    }
    __syncwarp();
    const int hs = M.height_slot[lane];
    if (hs >= 0) A.height_buf[((size_t)clip * DP_PAST + A.ring_head) * DP_NH + hs] = p[1] + gp[1];
    if (lane < DP_L / 2) {
      reinterpret_cast<float2*>(A.latent_buf + ((size_t)clip * DP_PAST + A.ring_head) * DP_L)[lane] = zlast[c];
      reinterpret_cast<float2*>(A.latent + (size_t)clip * DP_L)[lane] = z[c];
    }
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        A.disp_buf[((size_t)clip * DP_PAST + A.ring_head) * 3 + i] = d[i] + adj[i];
        A.gpos[clip * 3 + i] = gp[i];
        A.out_gpos[(size_t)clip * A.out_gpos_stride + i] = gp[i];
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) A.grot[clip * 4 + i] = r[i];
      A.out_iters[clip] = iters[c];
      A.out_losses[clip * 3] = lp[c];
      A.out_losses[clip * 3 + 1] = lr[c];
      A.out_losses[clip * 3 + 2] = lt[c];
    }
    // output pose: standardised root-space quats, root slot := standardised world rotation
    if (lane < DP_J) {
      const float4 mq = reinterpret_cast<const float4*>(M.mean_q)[lane];
      const float4 sq = reinterpret_cast<const float4*>(M.std_q)[lane];
      const float* s = (lane == 0) ? r : q;
      reinterpret_cast<float4*>(A.out_pose + (size_t)clip * A.out_pose_stride)[lane] =
          make_float4((s[0] - mq.x) / sq.x, (s[1] - mq.y) / sq.y, (s[2] - mq.z) / sq.z, (s[3] - mq.w) / sq.w);
    }
  }
}

}  // namespace

size_t dp_frame_simt_smem_bytes(int warps, int cpw) {
  return sizeof(DpModelImage) + 16 + (size_t)warps * cpw * (2 * DP_SCRATCH * sizeof(float) + 32 * sizeof(ClipTrackers));
}

cudaError_t dp_frame_simt_launch(const DpFrameArgs& args, int num_sms, cudaStream_t stream) {
  // 4096 clips on 148 SMs: two clips per warp, ~14 warps per CTA, one CTA per SM (single wave).
  const int cpw = args.n_clips > 2 * num_sms ? 2 : 1;
  const int total_warps = (args.n_clips + cpw - 1) / cpw;
  int wpc = (total_warps + num_sms - 1) / num_sms;
  wpc = wpc < 1 ? 1 : (wpc > 16 ? 16 : wpc);
  const int grid = (total_warps + wpc - 1) / wpc;
  const size_t smem = dp_frame_simt_smem_bytes(wpc, cpw);
  cudaError_t err;
  if (cpw == 2) {
    err = cudaFuncSetAttribute(dp_frame_simt_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    dp_frame_simt_kernel<2><<<grid, wpc * 32, smem, stream>>>(args);
  } else {
    err = cudaFuncSetAttribute(dp_frame_simt_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    dp_frame_simt_kernel<1><<<grid, wpc * 32, smem, stream>>>(args);
  }
  return cudaGetLastError();
}
