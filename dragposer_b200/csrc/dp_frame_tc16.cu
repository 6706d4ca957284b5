// dp_frame_tc16.cu -- persistent per-frame optimisation kernel, fp16x2 split products on tcgen05 with the WEIGHTS
// resident in tensor memory (default path for batches).
//
// One launch == one frame of DragPose.run (python/src/drag_pose.py:196-414) for every clip, the same contract as the fp32 kernel
// (dp_frame_simt.cu); the decoder forward 24->40->60->92 and its data-gradient run as D[features x clips] = W . X tiles, built
// around what the phase clock and the MMA-rate probes measured on B200:
//   * an MMA whose A operand comes from shared memory costs ~41 cycles at N = 16 whatever the math; with A in tensor memory
//     (TS mode) it costs ~12.  The six weight matrices (forward W_l and backward W_l^T, two fp16 pieces each, 16 W) fit in
//     352 of the 512 tensor-memory columns, so they are loaded there once per launch and shared memory only carries the
//     activations (B operand, MN-major).
//   * the CUDA cores idle during the tensor phases and vice versa, so ONE CTA per SM runs FOUR independent groups of
//     4 warps x 8 clips.  Each group has its own accumulator columns, mbarrier, named block barrier and loop exit; they
//     share the tensor-memory weights and drift apart naturally, one group's kinematics overlapping the others' layers.
//   * kinematics / loss / adjoint: two clips per warp in packed fp32x2 registers (dp_fk2.cuh); optimiser state in shared
//     memory.
#include "dp_fk2.cuh"
#include "dp_internal.h"
#include "dp_umma.cuh"

namespace {

constexpr int NC = 32;                     // clip columns per CTA
constexpr int kWarps = 16;
constexpr int kGroups = 4;                 // independent clip groups of a CTA
constexpr int kGW = kWarps / kGroups;      // warps per group: 4 (8 clips)
constexpr int kGC = NC / kGroups;          // clip columns per group
constexpr int kG8 = kGC / 8;               // 8-clip groups per fp16 piece of a group
constexpr int EC = 8;             // clips per epilogue thread: a group's 4 warps are the 4 TMEM lane quarters, each thread takes all 8 clips
// activation image (B operand, MN-major, no swizzle).  The two fp16 pieces of a group's 8 clips lie SIDE BY SIDE along N, so that
// one N = 16 instruction multiplies a weight piece with both of them: element (feature k, group g, piece p, clip n < 8) at
//   (k / 8) * kB_LBO + (k % 8) * 16 + ((2 g + p) kG8 + n / 8) * kB_SBO + (n % 8) * 2 bytes   (kG8 = 8-clip groups per piece: 1).
// The K 8-groups are padded from 1024 to 1040 bytes: unpadded, every 8-group starts in the same bank and the 32 lanes of an
// epilogue warp (consecutive features, one 16-byte store each) collide four ways; the pad moves each group on by four banks.
constexpr uint32_t kB_SBO = 128, kB_PIECE = kG8 * kB_SBO;
constexpr uint32_t kB_LBO = kB_SBO * 2 * (NC / 8) + 16;
constexpr uint32_t kPingBytes = (64 / 8) * kB_LBO, kPongBytes = (96 / 8) * kB_LBO;  // both pieces
// dL/dy image (B operand of the first backward layer only), K-MAJOR: element (group g, piece p, clip n < 8, feature k) at
//   ((2 g + p) kG8 + n / 8) * kD_SBO + (k / 8) * kD_LBO + (n % 8) * 16 + (k % 8) * 2 bytes,
// so that the kinematics lane of joint j stores its four values dL/dy[4j .. 4j+3] of a clip as ONE 8-byte word per piece -- the
// adjoint writes the tensor-core operand itself and the backward layers start after a single group barrier (round 1 wrote fp32
// rows, and the epilogue warps re-read them transposed, split them and stored them behind a second barrier).  kD_LBO is padded
// from 128 to 144 bytes for the same bank reason as kB_LBO.
constexpr uint32_t kD_LBO = 144, kD_SBO = (96 / 8) * kD_LBO, kD_PIECE = kG8 * kD_SBO, kDyBytes = 2 * (NC / 8) * kD_SBO;
// the weight image holds 16 W and dL/dy is scaled per clip into [16, 32) (dp_fk2.cuh, SCALE): exact powers of two for fp16's narrow
// exponent range, undone in the epilogues and when dL/dz is read
constexpr float kWScale = 16.0f;
// Generic-proxy writes of an operand image (st.shared by the epilogue / kinematics / Adam threads) must be ordered before the
// tensor core's async-proxy reads: the ONE issuing thread executes fence.proxy.async after the group barrier that made the writes
// visible to it -- writer's st.shared -> (program order) barrier arrive -> (synchronizes with) issuer's barrier -> (program order)
// fence.proxy.async -> tcgen05.mma: the proxy fence lies on the base-causality path from the write to the read, which is what the
// PTX memory model asks for; the barrier has drained the stores, so the fence is cheap.  Every writer fencing before the barrier
// (the pattern of CUTLASS's TMA-store epilogues; MEMBAR.ALL.CTA with the warp's stores still in flight, 50-110 cycles in each of
// the 7 hand-offs of an iteration) measured 0.641 against 0.629 ms per frame at 4 096 clips (DESIGN.md section 3.1).
enum { ST_Z = 0, ST_TL = 1, ST_M = 2, ST_V = 3, ST_ZLAST = 4 };
// tensor-memory columns: accumulators of group g at 2 kGC g (kGC columns per B piece); then the weight pieces (two K elements per word)
constexpr uint32_t kT_D = 0, kT_W = 64, kT_COLS = 512;
static_assert(kT_W + DP_TC_TMEM_WORDS <= kT_COLS, "weights must fit in tensor memory");

struct SmemT {
  __align__(16) unsigned char model[sizeof(DpModelImageTC)];  // biases, statistics, skeleton tables
  __align__(16) unsigned char ping[kPingBytes];     // z (24) / a1 (60) / dL/dh1 (60)
  __align__(16) unsigned char pong[kPongBytes];     // a0 (40) / dL/dh0 (40)
  __align__(16) unsigned char dyimg[kDyBytes];      // dL/dy (92), K-major
  __align__(16) float4 y2[NC / 2][2][24];           // y (fp32) of a warp's clip pair, interleaved (dp_fk2.cuh)
  float bscale[NC];                                 // 1 / (per-clip power-of-two scale of dL/dy)
  __align__(16) float4 trk2[NC / 2][8][32];         // tracker tables of a clip pair, interleaved structure of arrays (dp_fk2.cuh)
  // optimiser state of a warp's clip pair, one float2 (.x first clip, .y second) per latent feature:
  // [ST_Z latent | ST_TL target latent | ST_M, ST_V Adam moments | ST_ZLAST last evaluated latent]
  __align__(16) float2 st[NC / 2][5][DP_L];
  __align__(16) float2 groot2[NC / 2][4];           // previous world root rotations g (wxyz) of a clip pair
  __align__(16) float2 fkscr[NC / 2][16];           // per clip pair: R_0, r, d parked between the two halves of the kinematics pass
  double prev[NC];                                  // previous total loss (early stopping compares in double)
  float loss[NC][3];                                // last evaluated lp, lr, lt
  int iters[NC];
  uint64_t bar_w, bar_mma[kGroups];
  uint32_t tmem_base;
  __device__ __forceinline__ const DpModelImageTC& M() const { return *reinterpret_cast<const DpModelImageTC*>(model); }
};

// named block barriers of the groups (ids 1 .. kGroups; id 0 is __syncthreads)
__device__ __forceinline__ void group_sync(int gid) { asm volatile("bar.sync %0, %1;" ::"r"(gid + 1), "n"(kGW * 32) : "memory"); }
__device__ __forceinline__ bool group_or(int gid, bool p) {
  uint32_t r;
  asm volatile(
      "{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %1, 0;\n\tbar.red.or.pred q, %2, %3, p;\n\tselp.u32 %0, 1, 0, q;\n\t}\n"
      : "=r"(r)
      : "r"((uint32_t)p), "r"(gid + 1), "n"(kGW * 32)
      : "memory");
  return r != 0;
}

__device__ __forceinline__ uint32_t pack_f16x2(float lo_elem, float hi_elem) {  // lower address <- lo_elem
  uint32_t p;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(p) : "f"(hi_elem), "f"(lo_elem));
  return p;
}
__device__ __forceinline__ void unpack_f16x2(uint32_t p, float& lo_elem, float& hi_elem) {
  asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;\n\t}\n" : "=f"(lo_elem), "=f"(hi_elem) : "r"(p));
}
// 4 fp32 values (feature k; 8-group `slot`, clips 4 sub .. 4 sub + 3 of it) -> the two fp16 pieces, one 8-byte store each
__device__ __forceinline__ void store_pieces4(unsigned char* img, int k, int slot, int sub, const float (&v)[4]) {
  unsigned char* dst = img + (k >> 3) * kB_LBO + (k & 7) * 16 + slot * kB_SBO + sub * 8;
  const uint32_t a = pack_f16x2(v[0], v[1]), b = pack_f16x2(v[2], v[3]);
  float h0, h1, h2, h3;
  unpack_f16x2(a, h0, h1);
  unpack_f16x2(b, h2, h3);
  *reinterpret_cast<uint2*>(dst) = make_uint2(a, b);
  *reinterpret_cast<uint2*>(dst + kB_PIECE) = make_uint2(pack_f16x2(v[0] - h0, v[1] - h1), pack_f16x2(v[2] - h2, v[3] - h3));
}
// one feature of a clip PAIR (columns cl, cl + 1 of group g, cl even) -> its pieces, one 32-bit store each (latent rows of ping)
__device__ __forceinline__ void store_piece_pair(unsigned char* img, int k, int g, int cl, float x0, float x1) {
  unsigned char* dst = img + (k >> 3) * kB_LBO + (k & 7) * 16 + (2 * kG8 * g + (cl >> 3)) * kB_SBO + (cl & 7) * 2;
  const uint32_t p = pack_f16x2(x0, x1);
  float h0, h1;
  unpack_f16x2(p, h0, h1);
  *reinterpret_cast<uint32_t*>(dst) = p;
  *reinterpret_cast<uint32_t*>(dst + kB_PIECE) = pack_f16x2(x0 - h0, x1 - h1);
}

// weight pieces in tensor memory (word offsets inside kT_W): layer l forward = W_l (rows = outputs), backward = W_l^T
template <int L, bool FWD> struct WT;
template <> struct WT<0, true>  { static constexpr uint32_t p1 = 0,   p2 = 16,  ksteps = 2; };   // K = 32 (24 latent + pad)
template <> struct WT<1, true>  { static constexpr uint32_t p1 = 32,  p2 = 56,  ksteps = 3; };   // K = 48
template <> struct WT<2, true>  { static constexpr uint32_t p1 = 80,  p2 = 112, ksteps = 4; };   // K = 64
template <> struct WT<2, false> { static constexpr uint32_t p1 = 144, p2 = 192, ksteps = 6; };   // K = 96
template <> struct WT<1, false> { static constexpr uint32_t p1 = 240, p2 = 272, ksteps = 4; };   // K = 64
template <> struct WT<0, false> { static constexpr uint32_t p1 = 304, p2 = 328, ksteps = 3; };   // K = 48
static_assert(WT<0, false>::p2 + 24 == DP_TC_TMEM_WORDS, "tensor-memory weight map");

// sink of the kinematics adjoint: the (scaled) dL/dy of the warp's two clips as fp16 pieces of the K-major operand image
struct EmitDyPieces {
  unsigned char* img;
  int g, cl, lane;  // group, (even) column of the warp's first clip inside the group
  static __device__ __forceinline__ void put(unsigned char* dst, float x0, float x1, float x2, float x3) {
    const uint32_t a = pack_f16x2(x0, x1), b = pack_f16x2(x2, x3);
    float h0, h1, h2, h3;
    unpack_f16x2(a, h0, h1);
    unpack_f16x2(b, h2, h3);
    *reinterpret_cast<uint2*>(dst) = make_uint2(a, b);
    *reinterpret_cast<uint2*>(dst + kD_PIECE) = make_uint2(pack_f16x2(x0 - h0, x1 - h1), pack_f16x2(x2 - h2, x3 - h3));
  }
  __device__ __forceinline__ void operator()(const P2 (&o)[4], const P2 (&db)[3]) const {
    // the two clips share an 8-group (cl is even): rows (cl % 8) and (cl % 8) + 1 of the same core matrices
    unsigned char* base = img + (2 * kG8 * g + (cl >> 3)) * kD_SBO + (cl & 7) * 16;
    if (lane < DP_J) {
      unsigned char* dst = base + (lane >> 1) * kD_LBO + (lane & 1) * 8;  // k = 4 lane: 8-group lane / 2, first or second half
      put(dst, o[0].v.x, o[1].v.x, o[2].v.x, o[3].v.x);
      put(dst + 16, o[0].v.y, o[1].v.y, o[2].v.y, o[3].v.y);
    }
    if (lane == 0) {  // k = 88 .. 91 (91 is the unused pad output: zero)
      unsigned char* dst = base + 11 * kD_LBO;
      put(dst, db[0].v.x, db[1].v.x, db[2].v.x, 0.0f);
      put(dst + 16, db[0].v.y, db[1].v.y, db[2].v.y, 0.0f);
    }
  }
};

struct Ctx {
  SmemT* S;
  uint32_t tmem;
  int gid, wg, lane;
  uint32_t phase;  // parity of the group's next MMA completion
};

// MMAs of one dense layer of one group; every thread of the group calls this, one elected lane of the group's first warp issues.
// A = weight pieces in tensor memory, B = the group's clip columns of the activation image: per K step of 16
//   D[:, 0..15] (+)= A1 . [B1 | B2]   (N = 16: the (1,1) product lands in columns 0..7, the (1,2) product in columns 8..15)
//   D[:, 0..15]  += A2 . [B1 | B2]    (N = 16: the (2,1) product)
// and the epilogue adds the two column blocks -- two instructions per K step instead of three (an instruction costs ~20 issue
// cycles whatever its N).  The second instruction takes both pieces as well because an M = 128 instruction needs N >= 16: it adds
// the (2,2) product, a term of relative size 2^-22, to the second column block.  B_KMAJOR: the B operand is the K-major dL/dy
// image instead of an MN-major activation image.
template <int L, bool FWD, bool B_KMAJOR = false>
__device__ __forceinline__ void tc_issue(Ctx& c, const unsigned char* src) {
  if (c.wg == 0) {
    tc_fence_after();
    if (elect_one()) {
      fence_proxy_async();  // orders the group's st.shared operand writes before the MMAs (see "Generic-proxy writes" above)
      // fp16 x fp16 -> fp32, M 128, N = 2 kGC; bit 16: B is MN-major
      constexpr uint32_t idesc = (1u << 4) | (B_KMAJOR ? 0u : (1u << 16)) | ((uint32_t)((2 * kGC) >> 3) << 17) | (8u << 24);
      constexpr uint32_t lbo = B_KMAJOR ? kD_LBO : kB_LBO, sbo = B_KMAJOR ? kD_SBO : kB_SBO;
      const UmmaDescBase b = umma_desc_base(smem_u32(src) + (uint32_t)c.gid * 2 * kG8 * sbo, lbo, sbo);  // the group's 8-groups (both pieces)
      const uint32_t d = c.tmem + kT_D + 2 * kGC * c.gid, a1 = c.tmem + kT_W + WT<L, FWD>::p1, a2 = c.tmem + kT_W + WT<L, FWD>::p2;
#pragma unroll
      for (int k = 0; k < (int)WT<L, FWD>::ksteps; ++k) {
        const uint32_t bo = k * 2 * lbo;  // K = 16 per instruction: two 8-groups of K
        if (k == 0) umma_f16_ts_c<false>(d, a1 + 8 * k, umma_desc_at(b, bo), idesc);
        else umma_f16_ts_c<true>(d, a1 + 8 * k, umma_desc_at(b, bo), idesc);
        umma_f16_ts_c<true>(d, a2 + 8 * k, umma_desc_at(b, bo), idesc);
      }
      umma_commit(&c.S->bar_mma[c.gid]);
    }
    __syncwarp();
  }
}
// one dense layer + its epilogue (lane == output feature, 8 clips per thread); ends with the group barrier
template <int L, bool FWD, bool B_KMAJOR = false, class Epi>
__device__ __forceinline__ void tc_layer(Ctx& c, const unsigned char* src, int out_rows, Epi epi) {
  SmemT& S = *c.S;
  tc_issue<L, FWD, B_KMAJOR>(c, src);
  const int quarter = c.wg & 3;
  if (quarter * 32 < out_rows) {
    mbar_wait(&S.bar_mma[c.gid], c.phase);
      tc_fence_after();
    float v[EC], w[EC];
    const uint32_t t = c.tmem + ((uint32_t)(quarter * 32) << 16) + kT_D + (uint32_t)(2 * kGC * c.gid);
    tmem_ld8(t, v);
    tmem_ld8(t + kGC, w);
    tmem_ld_wait();
  #pragma unroll
    for (int i = 0; i < EC; ++i) v[i] += w[i];
    const int k = quarter * 32 + c.lane;
    if (k < out_rows) epi(k, v);
    tc_fence_before();
    }
  c.phase ^= 1u;
  group_sync(c.gid);
}

// the same for a layer with at most 64 output rows whose weight rows are REPLICATED in the upper 64 lanes of the tensor-memory operand:
// all four warps of the group take part, lane quarters 0 / 1 on clips 0..3, quarters 2 / 3 (the replicas) on clips 4..7 -- four
// clips per thread instead of eight halves the dependent chain of the epilogue (the longest part of a layer)
template <int L, bool FWD, bool B_KMAJOR = false, class Epi>
__device__ __forceinline__ void tc_layer4(Ctx& c, const unsigned char* src, int out_rows, Epi epi) {
  SmemT& S = *c.S;
  tc_issue<L, FWD, B_KMAJOR>(c, src);
  const int quarter = c.wg & 3, sub = quarter >> 1;
  if ((quarter & 1) * 32 < out_rows) {
    mbar_wait(&S.bar_mma[c.gid], c.phase);
    tc_fence_after();
    float v[4], w[4];
    const uint32_t t = c.tmem + ((uint32_t)(quarter * 32) << 16) + kT_D + (uint32_t)(2 * kGC * c.gid + 4 * sub);
    tmem_ld4(t, v);
    tmem_ld4(t + kGC, w);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] += w[i];
    const int k = (quarter & 1) * 32 + c.lane;
    if (k < out_rows) epi(k, sub, v);
    tc_fence_before();
  }
  c.phase ^= 1u;
  group_sync(c.gid);
}

// CLOCK: the phase clock / timeline of CTA 0 (profiling level 2) is compiled into a second instantiation only
template <bool CLOCK>
__global__ void __launch_bounds__(kWarps * 32, 1) dp_frame_tc16_kernel(const __grid_constant__ DpFrameArgs A) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  SmemT& S = *reinterpret_cast<SmemT*>(smem_raw);
  const DpModelImageTC& M = S.M();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gid = warp / kGW, wg = warp % kGW;  // group, warp within the group
  if (threadIdx.x == 0) {
    mbar_init(&S.bar_w, 1);
    for (int g = 0; g < kGroups; ++g) mbar_init(&S.bar_mma[g], 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(&S.tmem_base, kT_COLS);
  static_assert(offsetof(SmemT, dyimg) == offsetof(SmemT, ping) + sizeof(S.ping) + sizeof(S.pong), "operand images are contiguous");
  for (int i = threadIdx.x; i < (int)(sizeof(S.ping) + sizeof(S.pong) + sizeof(S.dyimg)) / 16; i += kWarps * 32)
    reinterpret_cast<uint4*>(&S.ping[0])[i] = make_uint4(0u, 0u, 0u, 0u);  // pad rows / columns must stay finite
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (threadIdx.x == 0) {
    mbar_expect_tx(&S.bar_w, (uint32_t)sizeof(S.model));
    tma_bulk_g2s(S.model, A.model_tc, (uint32_t)sizeof(S.model), &S.bar_w);
  }
  const uint32_t tmem = S.tmem_base;
  {  // weight pieces -> tensor memory: warp w fills lanes 32 (w % 4) .. +31, columns 88 (w / 4) .. +87 (coalesced reads)
    const uint32_t* img = A.model_tmem;
    const int row = (warp & 3) * 32 + lane, c0 = (warp >> 2) * (DP_TC_TMEM_WORDS / 4);
#pragma unroll 1
    for (int j = 0; j < DP_TC_TMEM_WORDS / 4; j += 8) {
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(img[(size_t)(c0 + j + i) * 128 + row]);
      tmem_st8(tmem + ((uint32_t)((warp & 3) * 32) << 16) + kT_W + (uint32_t)(c0 + j), v);
    }
    tmem_st_wait();
  }
  Ctx ctx{&S, tmem, gid, wg, lane, 0u};
  constexpr int CPW = 2;            // clips per warp in the per-clip phases
  const int n0 = warp * CPW;        // clip column of this warp's first clip (group g owns columns kGC g .. kGC g + kGC - 1)
  // the CTA's clip PAIRS are dealt to the groups as evenly as possible (28 clips = 14 pairs: 7 + 7, or 4 + 4 + 3 + 3), one pair per warp
  const int n_pairs = (A.clips_per_cta + 1) / 2;
  int first_pair = 0;
  for (int g = 0; g < gid; ++g) first_pair += (n_pairs + kGroups - 1 - g) / kGroups;
  const int my_pairs = (n_pairs + kGroups - 1 - gid) / kGroups;
  const int col0 = 2 * (first_pair + wg);  // this warp's first clip inside the CTA's tile
  const int clip0 = blockIdx.x * A.clips_per_cta + col0;

  // ---- per-clip frame inputs (same as the fp32 kernel)
  static_assert(CPW == 2, "the kinematics pass packs exactly two clips per warp");
  bool valid[CPW];
  float inv3e[CPW], lrot9e[CPW];
#pragma unroll
  for (int c = 0; c < CPW; ++c) {
    const int clip = clip0 + c;
    valid[c] = clip < A.n_clips && wg < my_pairs && col0 + c < A.clips_per_cta;
    const int cc = valid[c] ? clip : 0;
    int ne = A.n_ee ? A.n_ee[cc] : A.ee_stride;
    ne = max(1, min(ne, A.ee_stride));
    inv3e[c] = 1.0f / (3.0f * (float)ne);
    lrot9e[c] = A.lambda_rot / (9.0f * (float)ne);
    if (lane < 4) reinterpret_cast<float*>(&S.groot2[warp][lane])[c] = A.grot[cc * 4 + lane];
    if (lane == 0) {
      S.prev[n0 + c] = 10000000.0;
      S.loss[n0 + c][0] = S.loss[n0 + c][1] = S.loss[n0 + c][2] = __int_as_float(0x7f800000);
      S.iters[n0 + c] = 0;
    }
    // tracker stream of the clip: lane e loads slot e (all slots in flight at once, neighbouring lanes read neighbouring
    // addresses) and scatters its row to the lane of the joint it tracks; untracked joints keep zero weights
    if (c == 0) {
      const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int i = 0; i < 8; ++i) S.trk2[warp][i][lane] = zero4;
    }
    __syncwarp();
    if (lane < ne) {
      float origin[3] = {0.f, 0.f, 0.f};  // world-absolute targets are taken relative to the clip's current global position
      if (A.targets_world) { origin[0] = A.gpos[cc * 3]; origin[1] = A.gpos[cc * 3 + 1]; origin[2] = A.gpos[cc * 3 + 2]; }
      const int j = A.joints[(A.shared_trackers ? 0 : (size_t)cc * A.ee_stride) + lane];
      const float2 wt = reinterpret_cast<const float2*>(A.weights + (A.shared_trackers ? 0 : (size_t)cc * A.ee_stride * 2))[lane];
      const float* tp = A.tgt_pos + ((size_t)cc * A.ee_stride + lane) * 3;
      const float* tr = A.tgt_rot + ((size_t)cc * A.ee_stride + lane) * 9;
      if (j >= 0 && j < DP_J) {
        // row r of the table = (x, y, z, w): packed halves [2r][j] = (x a, x b, y a, y b), [2r+1][j] = (z a, z b, w a, w b); clip c is the .x / .y half
        auto put = [&](int r, float x, float y, float z, float w) {
          float* lo = reinterpret_cast<float*>(&S.trk2[warp][2 * r][j]) + c;
          float* hi = reinterpret_cast<float*>(&S.trk2[warp][2 * r + 1][j]) + c;
          lo[0] = x; lo[2] = y; hi[0] = z; hi[2] = w;
        };
        put(0, tp[0] - origin[0], tp[1] - origin[1], tp[2] - origin[2], wt.x);
        put(1, tr[0], tr[1], tr[2], wt.y);
        put(2, tr[3], tr[4], tr[5], 0.f);
        put(3, tr[6], tr[7], tr[8], 0.f);
      }
    }
  }
  if (lane < DP_L) {  // optimiser state of the pair; latent -> B operand of the first layer
    float2 z = make_float2(0.f, 0.f), tl = z;
    if (valid[0]) {
      z.x = A.latent[(size_t)clip0 * DP_L + lane];
      tl.x = A.target_buf[((size_t)clip0 * A.target_rows + A.target_index) * DP_L + lane];
    }
    if (valid[1]) {
      z.y = A.latent[(size_t)(clip0 + 1) * DP_L + lane];
      tl.y = A.target_buf[((size_t)(clip0 + 1) * A.target_rows + A.target_index) * DP_L + lane];
    }
    S.st[warp][ST_Z][lane] = z;
    S.st[warp][ST_TL][lane] = tl;
    S.st[warp][ST_M][lane] = make_float2(0.f, 0.f);
    S.st[warp][ST_V][lane] = make_float2(0.f, 0.f);
    S.st[warp][ST_ZLAST][lane] = z;
    store_piece_pair(S.ping, lane, gid, 2 * wg, z.x, z.y);
  }
  const P2 inv3e2 = mk2(inv3e[0], inv3e[1]), lrot9e2 = mk2(lrot9e[0], lrot9e[1]);
  __syncwarp();
  fence_proxy_async();
  mbar_wait(&S.bar_w, 0);  // model image (biases, statistics, skeleton tables) has landed
  tc_fence_before();
  __syncthreads();         // tensor-memory weights written by all warps; latent pieces and tracker rows of every group in place
  tc_fence_after();

  const FkLaneIdx lane_idx = fk_lane_idx(M, lane);  // skeleton indices of this lane, in registers for the whole launch
  constexpr float wsc = 1.0f / kWScale;  // undoes the weight-image scaling
  const int slot0 = 2 * kG8 * gid;       // first 8-group (piece 1) of this group in the activation images
  unsigned neg0 = 0, neg1 = 0;           // LeakyReLU slope bits of (feature k, this thread's 4 clips) for the backward pass
  auto forward = [&]() {
    tc_layer4<0, true>(ctx, S.ping, DP_H0, [&](int k, int sub, float (&v)[4]) {
      const float b = M.b0[k];
      neg0 = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) { v[i] = fmaf(v[i], wsc, b); neg0 |= (v[i] > 0.f ? 0u : 1u) << i; v[i] = lrelu(v[i]); }
      store_pieces4(S.pong, k, slot0, sub, v);
    });
    tc_layer4<1, true>(ctx, S.pong, DP_H1, [&](int k, int sub, float (&v)[4]) {
      const float b = M.b1[k];
      neg1 = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) { v[i] = fmaf(v[i], wsc, b); neg1 |= (v[i] > 0.f ? 0u : 1u) << i; v[i] = lrelu(v[i]); }
      store_pieces4(S.ping, k, slot0, sub, v);
    });
    tc_layer<2, true>(ctx, S.ping, DP_Y, [&](int k, float (&v)[EC]) {
      const float b = M.b2[k];
#pragma unroll
      for (int i = 0; i < EC; i += 2)  // clips 2p, 2p + 1 of the group = pair kGW gid + p; feature k = 4 j + c
        *reinterpret_cast<float2*>(reinterpret_cast<float*>(&S.y2[kGW * gid + i / 2][(k >> 1) & 1][k >> 2]) + 2 * (k & 1)) =
            make_float2(fmaf(v[i], wsc, b), fmaf(v[i + 1], wsc, b));
    });
  };

  // ---- optimisation loop (drag_pose.py:296-355)
  // early-stop test of the NEXT iteration, evaluated right after each Adam step (initial losses are +inf, initial increment 1)
  bool active[CPW] = {valid[0] && 1.0 > A.min_incr, valid[1] && 1.0 > A.min_incr};
  const float lt_scale = A.lambda_t * (1.0f / (float)DP_L);
  // A fixed number of iterations (negative stop thresholds, min_loss_incr = -inf: the headline workload) looks at the tracker losses
  // of an iteration only to report the last ones: their warp sums are skipped on the other iterations (dp_fk2.cuh, want_loss)
  const bool fixed_iters = A.eps_pos < 0.0 && A.eps_rot < 0.0 && A.min_incr < -1.7e308 && !A.trace && !A.eval_only;
  const bool clocked = CLOCK && A.phase_cycles != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
  long long tick = clocked ? clock64() : 0;
  auto phase_done = [&](int i) {
    if (CLOCK && clocked) {
      const long long now = clock64();
      A.phase_cycles[i] += (unsigned long long)(now - tick);
      tick = now;
    }
  };
  // optional timeline of both groups over iterations 40..43 (scripts/timeline.py): six stamps per group and iteration
  const bool tl_on = CLOCK && A.phase_cycles != nullptr && blockIdx.x == 0 && wg == 0 && lane == 0 && gid < 2;  // the first two groups
  auto stamp = [&](int it, int k) {
    if (CLOCK && tl_on && it >= 40 && it < 44) A.phase_cycles[16 + gid * 24 + (it - 40) * 6 + k] = (unsigned long long)clock64();
  };
  for (int it = 0; it < A.max_iter; ++it) {
    if (!group_or(gid, active[0] || active[1])) break;  // also publishes the latent pieces written by the Adam epilogue
    if (lane == 0) {  // the Adam epilogue reads two table entries: pull their lines into L1 now instead of stalling there
      asm volatile("prefetch.global.L1 [%0];" ::"l"(A.adam_tab + it));
      asm volatile("prefetch.global.L1 [%0];" ::"l"(A.adam_tab + A.max_iter + it));
    }
    phase_done(3);
    stamp(it, 0);
    forward();
    phase_done(0);
    stamp(it, 1);
    float nlp[CPW] = {0.f, 0.f}, nlr[CPW] = {0.f, 0.f};
    if (active[0] || active[1]) {  // both clips of the warp in one packed pass; results of a stopped clip are discarded
      // one packed pass; dL/dy leaves it scaled per clip into [16, 32) (exact powers of two, undone when dL/dz is read)
      const FkOut2 o = fk_loss2<true, false, true>(M, lane_idx, &S.y2[warp][0][0], &S.trk2[warp][0][0], &S.groot2[warp][0], &S.fkscr[warp][0],
                                                   inv3e2, lrot9e2, lane, nullptr, nullptr, nullptr, nullptr, &S.bscale[n0],
                                                   EmitDyPieces{S.dyimg, gid, 2 * wg, lane}, !fixed_iters || it + 1 == A.max_iter);
      phase_done(4);
      if (active[0]) { nlp[0] = o.lp.v.x; nlr[0] = o.lr.v.x; }
      if (active[1]) { nlp[1] = o.lp.v.y; nlr[1] = o.lr.v.y; }
    }
    stamp(it, 2);
    group_sync(gid);
    phase_done(1);
    stamp(it, 3);
    // backward layers; dL/dy pieces were written by the kinematics warps (EmitDyPieces)
    tc_layer4<2, false, true>(ctx, S.dyimg, DP_H1, [&](int k, int sub, float (&v)[4]) {
#pragma unroll
      for (int i = 0; i < 4; ++i) v[i] *= ((neg1 >> i) & 1u) ? 0.2f * wsc : wsc;
      store_pieces4(S.ping, k, slot0, sub, v);
    });
    tc_layer4<1, false>(ctx, S.ping, DP_H0, [&](int k, int sub, float (&v)[4]) {
#pragma unroll
      for (int i = 0; i < 4; ++i) v[i] *= ((neg0 >> i) & 1u) ? 0.2f * wsc : wsc;
      store_pieces4(S.pong, k, slot0, sub, v);
    });
    phase_done(2);
    stamp(it, 4);
    // last backward layer (dL/dz = W_0^T dL/dh0) with the optimiser step as its epilogue.  The 24 rows of W_0^T are replicated in all
    // four lane quarters of the tensor-memory operand, so EVERY warp of the group reads dL/dz of its own clip pair (lane == latent
    // feature, two accumulator columns) and does the pair's Adam step, latent loss and early-stop bookkeeping -- no fp32 staging
    // of dL/dz, no separate optimiser phase behind another group barrier.  Everything that does not depend on dL/dz (state loads,
    // the latent loss and its warp sum) is done while the MMAs are in flight.
    tc_issue<0, false>(ctx, S.pong);
    {
      const bool lat = lane < DP_L;
      float2 z = make_float2(0.f, 0.f), tl = z, am = z, av = z;
      if (lat) { z = S.st[warp][ST_Z][lane]; tl = S.st[warp][ST_TL][lane]; am = S.st[warp][ST_M][lane]; av = S.st[warp][ST_V][lane]; }
      const float step_size = A.adam_tab[it], inv_bc2s = A.adam_tab[A.max_iter + it];  // lr/(1-b1^k), 1/sqrt(1-b2^k)
      const float us0 = wsc * S.bscale[n0], us1 = wsc * S.bscale[n0 + 1];               // undo the weight and dL/dy scalings
      const double prev0 = S.prev[n0], prev1 = S.prev[n0 + 1];
      const float dx = z.x - tl.x, dy = z.y - tl.y;
      float s0 = dx * dx, s1 = dy * dy;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {  // lanes >= 24 hold zeros; every lane ends with the same two sums
        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      }
      const float nlt0 = s0 * lt_scale, nlt1 = s1 * lt_scale;
      mbar_wait(&S.bar_mma[gid], ctx.phase);
      tc_fence_after();
      float d1[2], d2[2];
      const uint32_t t = tmem + ((uint32_t)((wg & 3) * 32) << 16) + kT_D + (uint32_t)(2 * kGC * gid + 2 * wg);
      tmem_ld2(t, d1);
      tmem_ld2(t + kGC, d2);
      tmem_ld_wait();
      tc_fence_before();
      ctx.phase ^= 1u;
      const float gx = fmaf(2.0f * lt_scale, dx, (d1[0] + d2[0]) * us0), gy = fmaf(2.0f * lt_scale, dy, (d1[1] + d2[1]) * us1);
      if (A.trace && lat) {
        if (active[0]) {
          float* row = A.trace + ((size_t)clip0 * A.trace_iters + it) * 52;
          row[lane] = z.x; row[DP_L + lane] = gx;
          if (lane == 0) { row[48] = nlp[0]; row[49] = nlr[0]; row[50] = nlt0; row[51] = 1.0f; }
        }
        if (active[1]) {
          float* row = A.trace + ((size_t)(clip0 + 1) * A.trace_iters + it) * 52;
          row[lane] = z.y; row[DP_L + lane] = gy;
          if (lane == 0) { row[48] = nlp[1]; row[49] = nlr[1]; row[50] = nlt1; row[51] = 1.0f; }
        }
      }
      if (A.eval_only) {
        if (lat && active[0]) A.eval_grad[(size_t)clip0 * DP_L + lane] = gx;
        if (lat && active[1]) A.eval_grad[(size_t)(clip0 + 1) * DP_L + lane] = gy;
      } else if (lat) {
        // branch-free: both clips are stepped, a stopped (or padding) clip keeps its state through the selects
        const float2 zl = S.st[warp][ST_ZLAST][lane];
        const float mx = fmaf(0.1f, gx - am.x, am.x), my = fmaf(0.1f, gy - am.y, am.y);
        const float vx = av.x * 0.999f + (0.001f * gx) * gx, vy = av.y * 0.999f + (0.001f * gy) * gy;
        // MUFU square root / reciprocal without the denormal range extension: a denormal second moment is far below eps = 1e-8
        const float ux = (-step_size * mx) * rcp_ftz(fmaf(sqrt_ftz(vx), inv_bc2s, 1e-8f));
        const float uy = (-step_size * my) * rcp_ftz(fmaf(sqrt_ftz(vy), inv_bc2s, 1e-8f));
        const bool a0 = active[0], a1 = active[1];
        S.st[warp][ST_M][lane] = make_float2(a0 ? mx : am.x, a1 ? my : am.y);
        S.st[warp][ST_V][lane] = make_float2(a0 ? vx : av.x, a1 ? vy : av.y);
        S.st[warp][ST_ZLAST][lane] = make_float2(a0 ? z.x : zl.x, a1 ? z.y : zl.y);  // the output is decoded from the last EVALUATED latent
        z.x = a0 ? z.x + ux : z.x;
        z.y = a1 ? z.y + uy : z.y;
        S.st[warp][ST_Z][lane] = z;
      }
      // the latent rows of the ping image were overwritten by the a1 / dL/dh1 pieces of this iteration: restore them for
      // EVERY clip (stopped and padding clips included) so that no column ever feeds back on its own garbage -- a
      // non-finite value in a K-padding row would poison the column through 0 x NaN
      if (lat) store_piece_pair(S.ping, lane, gid, 2 * wg, z.x, z.y);
      // early-stop bookkeeping: every lane holds the same (warp-uniform) numbers
      const float total0 = (nlp[0] + nlr[0]) + nlt0, total1 = (nlp[1] + nlr[1]) + nlt1;
      const double incr0 = prev0 - (double)total0, incr1 = prev1 - (double)total1;
      if (lane == 0) {
        if (active[0]) {
          S.prev[n0] = (double)total0;
          S.loss[n0][0] = nlp[0]; S.loss[n0][1] = nlr[0]; S.loss[n0][2] = nlt0;
          S.iters[n0] += 1;
        }
        if (active[1]) {
          S.prev[n0 + 1] = (double)total1;
          S.loss[n0 + 1][0] = nlp[1]; S.loss[n0 + 1][1] = nlr[1]; S.loss[n0 + 1][2] = nlt1;
          S.iters[n0 + 1] += 1;
        }
      }
      active[0] = active[0] && ((double)nlp[0] > A.eps_pos || (double)nlr[0] > A.eps_rot) && (incr0 > A.min_incr);
      active[1] = active[1] && ((double)nlp[1] > A.eps_pos || (double)nlr[1] > A.eps_rot) && (incr1 > A.min_incr);
      __syncwarp();
    }
    stamp(it, 5);
  }

  // ---- frame epilogue (drag_pose.py:369-414) from the LAST EVALUATED latent (pre-step)
  __syncwarp();
  if (lane < DP_L) {
    const float2 zl = S.st[warp][ST_ZLAST][lane];
    store_piece_pair(S.ping, lane, gid, 2 * wg, zl.x, zl.y);
  }
  group_sync(gid);
  forward();
  P2 q2[4], r2[4], p2[3], d2[3];
  if (valid[0] || valid[1])
    fk_loss2<false, true>(M, lane_idx, &S.y2[warp][0][0], &S.trk2[warp][0][0], &S.groot2[warp][0], &S.fkscr[warp][0], inv3e2, lrot9e2, lane, q2, r2, p2, d2);
#pragma unroll
  for (int c = 0; c < CPW; ++c) {
    if (!valid[c]) continue;
    const int clip = clip0 + c;
    float q[4], r[4], p[3], d[3];
#pragma unroll
    for (int i = 0; i < 4; ++i) { q[i] = c ? q2[i].v.y : q2[i].v.x; r[i] = c ? r2[i].v.y : r2[i].v.x; }
#pragma unroll
    for (int i = 0; i < 3; ++i) { p[i] = c ? p2[i].v.y : p2[i].v.x; d[i] = c ? d2[i].v.y : d2[i].v.x; }
    if (A.eval_only) {
      if (lane < DP_J && A.eval_pos) {
        float* o = A.eval_pos + ((size_t)clip * DP_J + lane) * 3;
        o[0] = p[0]; o[1] = p[1]; o[2] = p[2];
      }
      if (lane < 3 && A.out_losses) A.out_losses[clip * 3 + lane] = S.loss[n0 + c][lane];
      continue;
    }
    float p0[3], gp[3], adj[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      p0[i] = __shfl_sync(0xffffffffu, p[i], 0);
      gp[i] = A.gpos[clip * 3 + i] + p0[i];
    }
    if (A.adj_joint >= 0) {
      const float* tp = A.tgt_pos + ((size_t)clip * A.ee_stride + A.adj_slot) * 3;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const float pj = __shfl_sync(0xffffffffu, p[i], A.adj_joint);
        adj[i] = ((tp[i] - (A.targets_world ? A.gpos[clip * 3 + i] : 0.0f)) - pj) * A.adj_w;
        gp[i] += adj[i];
      }
    }
    __syncwarp();
    const int hs = M.height_slot[lane];
    if (hs >= 0) A.height_buf[((size_t)clip * DP_PAST + A.ring_head) * DP_NH + hs] = p[1] + gp[1];
    if (lane < DP_L) {
      const float2 zl = S.st[warp][ST_ZLAST][lane], zn = S.st[warp][ST_Z][lane];
      A.latent_buf[((size_t)clip * DP_PAST + A.ring_head) * DP_L + lane] = c ? zl.y : zl.x;
      A.latent[(size_t)clip * DP_L + lane] = c ? zn.y : zn.x;
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
      A.out_iters[clip] = S.iters[n0 + c];
      A.out_losses[clip * 3] = S.loss[n0 + c][0];
      A.out_losses[clip * 3 + 1] = S.loss[n0 + c][1];
      A.out_losses[clip * 3 + 2] = S.loss[n0 + c][2];
    }
    if (lane < DP_J) {
      const float4 mq = reinterpret_cast<const float4*>(M.mean_q)[lane];
      const float4 sq = reinterpret_cast<const float4*>(M.std_q)[lane];
      const float* s = (lane == 0) ? r : q;
      reinterpret_cast<float4*>(A.out_pose + (size_t)clip * A.out_pose_stride)[lane] =
          make_float4((s[0] - mq.x) / sq.x, (s[1] - mq.y) / sq.y, (s[2] - mq.z) / sq.z, (s[3] - mq.w) / sq.w);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(ctx.tmem, kT_COLS);
}

}  // namespace

cudaError_t dp_frame_tc16_launch(const DpFrameArgs& args, int num_sms, cudaStream_t stream) {
  static std::atomic<unsigned long long> configured{0}, configured_clk{0};
  const size_t smem = sizeof(SmemT) + 1024;
  const bool clk = args.phase_cycles != nullptr;
  if (cudaError_t e = clk ? dp_ensure_smem(dp_frame_tc16_kernel<true>, smem, configured_clk) : dp_ensure_smem(dp_frame_tc16_kernel<false>, smem, configured);
      e != cudaSuccess)
    return e;
  // spread the clips over every SM: 4096 clips -> 28 per CTA (14 pairs dealt 4 + 4 + 3 + 3 to the groups) on 147 SMs
  DpFrameArgs a = args;
  int cpc = (args.n_clips + num_sms - 1) / num_sms;
  cpc = cpc < 1 ? 1 : (cpc > NC ? NC : cpc);
  if (args.n_clips > num_sms * NC) cpc = NC;  // several waves anyway: use full tiles
  a.clips_per_cta = cpc;
  const int grid = (args.n_clips + cpc - 1) / cpc;
  if (clk) dp_frame_tc16_kernel<true><<<grid, kWarps * 32, smem, stream>>>(a);
  else dp_frame_tc16_kernel<false><<<grid, kWarps * 32, smem, stream>>>(a);
  return cudaGetLastError();
}
