// Stage 4, fused: open-loop rollouts through a learned MLP-ensemble System (BASELINE config 4).
//
// vmap(vmap(rollout_actions)) (mbpo/utils/optimizer_utils.py:11-59) + the particle summary of
// iCemTO.objective (icem_optimizer.py:155-160) for a System whose step is
//     x_next = x + MLP_e([x, u])           (template: mbpo/utils/network_utils.py:5-17, swish)
//     reward = pendulum reward on (x, u)   (rewards/pendulum_reward.py:27-42)
// with particle p rolled through ensemble member p (num_particles == num_members).
//
// A CTA PAIR (thread-block cluster of 2, tcgen05 cta_group::2) owns 256 candidate rows; each CTA
// owns 128 rows = its 128 TMEM lanes.  ALL FOUR layers run on the tensor cores, and the MMAs of
// layer l+1 are issued K-chunk by K-chunk while the CUDA cores are still producing layer l's
// activations (software pipeline through mbarriers; no __syncthreads inside the horizon loop):
//
//   warps 0-15  "epilogue" warps.  Warp w owns TMEM lanes 32*(w%4).. (rows) and, in every
//               64-column round, the 16 accumulator columns 64*r + 16*(w/4)..: tcgen05.ld -> bias +
//               swish -> bf16 -> the canonical K-major A chunk in shared memory -> mbarrier arrive.
//   warp 16     one elected thread of the leader CTA issues every tcgen05.mma (M256, 2-SM) as soon
//               as the chunk it consumes has been published by both CTAs, and tcgen05.commit
//               (multicast to both CTAs) when a layer's accumulator is complete.
//
//   layer 0  (K = 4 inputs)  one UMMA with K = 16: the fp32 inputs are split into bf16 hi + lo parts
//            and the fp32 weights / bias into hi + lo (+ lo2) parts, slots carry the cross products
//            hi*wh + hi*wl + lo*wh (+ bias against a column of ones): ~2^-16 relative, far inside
//            the bf16 rounding the activations receive next.  Weights are pre-scaled by 0.5.
//   layer 1,2 (256 x 256)    16 UMMAs (M256 N256 K16) each, weights resident in shared memory for the
//            whole horizon, split along N across the pair (64 KB per layer per CTA, by TMA).
//   layer 3  (N = 3 outputs) 16 UMMAs with N = 16: columns 0-2 hold the hi parts of w_out, 3-5 the
//            lo parts; delta = (c_j + c_{3+j}) + b_out.
//   swish(v) = h + h * tanh(h) with h = v / 2: one FFMA (0.5 * acc + 0.5 * bias, exact scaling), one
//            MUFU.TANH, one FFMA per activation.
// Two 256-column accumulators alternate (layer l writes D[l & 1]), so layer l+1's MMAs never touch
// the accumulator the epilogue of layer l is still reading.  The state never leaves registers;
// returns are averaged (or maxed) over members in registers in member order: deterministic, no
// workspace.
#pragma once
#include "mathx.cuh"
#include "mlp_tc_kernels.cuh"
#include "pendulum.cuh"

namespace mbpo {
namespace ens {

using namespace tc;

constexpr int EPI_WARPS = 16;
constexpr int MMA_WARP = EPI_WARPS;                 // warp index of the MMA issuer
constexpr int ENS_THREADS = (EPI_WARPS + 1) * 32;   // 544
constexpr uint32_t WH_BYTES = 128 * HID * 2;        // one hidden layer's N-half: 65536
constexpr uint32_t WH_LBO = 128 * 16;               // 2048: next K-chunk of a weight half
constexpr uint32_t W3_LBO = 8 * 16;                 // 128: next K-chunk of the 8-row output-layer tile
constexpr int ENS_TMEM_COLS = 512;                  // two 256-column accumulators
// A layer's 256 activation columns are published to the MMA issuer in rounds of 64, 64, 64, 32, 16, 16
// columns (4, 4, 4, 2, 1, 1 UMMA K-steps): the rounds shrink towards the end so that the MMA work that is
// still outstanding when the last round is published -- the only part the next epilogue has to wait for --
// is a single K-step.
constexpr int ROUNDS = 6;
__host__ __device__ constexpr int round_cols(int r) { return r < 3 ? 64 : (r == 3 ? 32 : 16); }
__host__ __device__ constexpr int round_first_col(int r) { return r < 3 ? 64 * r : (r == 3 ? 192 : (r == 4 ? 224 : 240)); }

struct Smem {
  static constexpr uint32_t A = 0;                        // 128 x 256 bf16 activations (4 chunks of 16 KB)
  static constexpr uint32_t W1 = A + A_BYTES;             // W[e,0] rows [128*rank, +128)
  static constexpr uint32_t W2 = W1 + WH_BYTES;           // W[e,1] rows [128*rank, +128)
  static constexpr uint32_t A0 = W2 + WH_BYTES;           // 128 x 16 bf16: split inputs (layer 0 A operand)
  static constexpr uint32_t W0 = A0 + TILE_M * 32;        // 128 x 16 bf16: split layer-0 weights (N-half)
  static constexpr uint32_t W3 = W0 + 128 * 32;           // 8 x 256 bf16: output layer hi/lo rows
  static constexpr uint32_t HB = W3 + 8 * HID * 2;        // float [2][256]: 0.5 * b_h
  static constexpr uint32_t B_OUT = HB + 2 * HID * 4;     // float [4]
  static constexpr uint32_t BARS = B_OUT + 16;            // full[ROUNDS], full_a0, bar_mma, bar_out, bar_w
  static constexpr uint32_t TMEM_PTR = BARS + (ROUNDS + 4) * 8;
  static constexpr uint32_t TOTAL = TMEM_PTR + 16;
};
static_assert(Smem::TOTAL <= 227 * 1024, "ensemble rollout shared memory plan exceeds 227 KB");

struct EnsArgs {
  int num_members, R, H, M, summarize;  // R = B * M rows; row r belongs to problem r / M
  const float* w_in;    // [E, 4, 256]
  const float* b_in;    // [E, 256]
  const float* b_h;     // [E, 2, 256]
  const float* w_out;   // [E, 256, 3]
  const float* b_out;   // [E, 3]
  const float* x0;      // [B, 3]
  const float* actions; // [R, H]
  float* returns_out;   // [R]
  MbpoPendulumParams reward;
};

__device__ __forceinline__ float tanh_approx(float z) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(z));
  return t;
}
// swish(2h) = 2h * sigmoid(2h) = h + h * tanh(h)
__device__ __forceinline__ float swish_half(float h) { return fmaf(h, tanh_approx(h), h); }

__device__ __forceinline__ float bf16_hi(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // default semantics (.release.cta): the data this arrive publishes stays in the arriving CTA's own shared
  // memory (each SM's tensor core reads its own half of A), made visible to the async proxy by the
  // fence.proxy.async before it; a cluster-scope release would cost a full memory barrier per round.
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_ss_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(static_cast<uint16_t>(3))
      : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}
// tcgen05.ld without the wait, so that the next round's load overlaps this round's arithmetic
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8_nowait(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld4_nowait(uint32_t taddr, uint32_t (&v)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld4(uint32_t (&v)[4]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]) : : "memory");
}
// The wait names the destination registers so that no use of them can be scheduled above it.
__device__ __forceinline__ void tmem_wait_ld16(uint32_t (&v)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                 "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_wait_ld8(uint32_t (&v)[8]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7])
               :
               : "memory");
}

// One epilogue round: NC accumulator values of this thread's row -> NC bf16 activations in the A tile
// (a_dst points at the first of them).  NC = 16: two 16-byte K-chunks; 8: one; 4: half of one.
template <int NC, bool HAS_BIAS>
__device__ __forceinline__ void epilogue_round(const uint32_t (&v)[NC], const float* hb, uint8_t* a_dst) {
  float s[NC];
#pragma unroll
  for (int j4 = 0; j4 < NC / 4; ++j4) {
    float4 b = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (HAS_BIAS) b = *reinterpret_cast<const float4*>(hb + j4 * 4);
    const float bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float acc = __uint_as_float(v[j4 * 4 + j]);
      const float h = HAS_BIAS ? fmaf(acc, 0.5f, bb[j]) : acc;
      s[j4 * 4 + j] = swish_half(h);
    }
  }
  if (NC == 4) {
    uint2 pk;
    pk.x = pack_bf16(s[0], s[1]); pk.y = pack_bf16(s[2], s[3]);
    *reinterpret_cast<uint2*>(a_dst) = pk;
  } else {
#pragma unroll
    for (int q = 0; q < NC / 8; ++q) {
      uint4 pk;
      pk.x = pack_bf16(s[q * 8 + 0], s[q * 8 + 1]); pk.y = pack_bf16(s[q * 8 + 2], s[q * 8 + 3]);
      pk.z = pack_bf16(s[q * 8 + 4], s[q * 8 + 5]); pk.w = pack_bf16(s[q * 8 + 6], s[q * 8 + 7]);
      *reinterpret_cast<uint4*>(a_dst + q * A_LBO) = pk;
    }
  }
}

// Publish a finished round: generic-proxy writes of A -> async proxy (tensor core); this thread's tcgen05.ld
// ordered before the MMAs that follow the arrive; one arrive per warp on the leader's barrier.
__device__ __forceinline__ void publish_round(uint32_t bar_cluster_addr, int lane) {
  fence_proxy_async();
  tc_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive_cluster(bar_cluster_addr);
}

// The split-input row of the layer-0 A operand: per input [hi, hi, lo], then [1, 1, 1, 0].
__device__ __forceinline__ void build_a0_row(uint8_t* a0_row, float x0, float x1, float x2, float u) {
  const float v[4] = {x0, x1, x2, u};
  float hi[4], lo[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    hi[i] = bf16_hi(v[i]);
    lo[i] = v[i] - hi[i];
  }
  uint4 p0, p1;
  p0.x = pack_bf16(hi[0], hi[0]); p0.y = pack_bf16(lo[0], hi[1]);
  p0.z = pack_bf16(hi[1], lo[1]); p0.w = pack_bf16(hi[2], hi[2]);
  p1.x = pack_bf16(lo[2], hi[3]); p1.y = pack_bf16(hi[3], lo[3]);
  p1.z = pack_bf16(1.0f, 1.0f);   p1.w = pack_bf16(1.0f, 0.0f);
  *reinterpret_cast<uint4*>(a0_row) = p0;
  *reinterpret_cast<uint4*>(a0_row + A_LBO) = p1;
}

#ifdef MBPO_ENS_TRACE
__device__ long long g_ens_trace[256];
#define ENS_TRACE(cond, slot) do { if ((cond) && blockIdx.x == 0 && e == 0 && t == 10) g_ens_trace[slot] = clock64(); } while (0)
#else
#define ENS_TRACE(cond, slot) do { } while (0)
#endif

// The kernel body.  TR: the row owners also store member e's Transition fields of each valid row,
// obs_out [R, E, H, 3] (the state before step t) and reward_out [R, E, H] (the reward term of step t), and leave
// returns_out alone; the MMA / epilogue / mbarrier schedule is the same either way.
template <bool TR>
__device__ __forceinline__ void ensemble_rollout_body(const EnsArgs& a, const CUtensorMap& w_map, float* obs_out,
                                                      float* reward_out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int quarter = warp >> 2;                       // which 16 of a round's 64 columns (epilogue warps)
  const int lrow = ((warp & 3) << 5) | lane;           // row within the CTA's tile = TMEM lane
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const bool row_owner = quarter == 3;   // warps 12-15 carry the rows' state: the warp scheduler favours the
                                          // highest warp ids, and the state update is the serial link between steps
  float* s_hb = reinterpret_cast<float*>(smem + Smem::HB);
  float* s_b_out = reinterpret_cast<float*>(smem + Smem::B_OUT);
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem + Smem::BARS);  // [ROUNDS] leader: round r of A published by both CTAs
  uint64_t* bar_a0 = bar_full + ROUNDS;                                 // leader: A0 rows published by both CTAs
  uint64_t* bar_mma = bar_full + ROUNDS + 1;                            // accumulator of layer 0/1/2 complete (multicast)
  uint64_t* bar_out = bar_full + ROUNDS + 2;                            // output-layer accumulator complete (multicast)
  uint64_t* bar_w = bar_full + ROUNDS + 3;                              // this CTA's weight halves landed
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + Smem::TMEM_PTR);

  // ---- one-time setup --------------------------------------------------------------------------
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                 "r"(ENS_TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  if (tid == 0) {
    for (int r = 0; r < ROUNDS; ++r) mbar_init(bar_full + r, 2 * EPI_WARPS);
    mbar_init(bar_a0, 2 * 4);
    mbar_init(bar_mma, 1);
    mbar_init(bar_out, 1);
    mbar_init(bar_w, 1);
    fence_barrier_init();
  }
  // the output-layer tile of the non-leader CTA stays all zero (its 8 rows are columns 8-15 of D3)
  for (int i = tid; i < 8 * HID * 2 / 16; i += ENS_THREADS)
    reinterpret_cast<uint4*>(smem + Smem::W3)[i] = make_uint4(0u, 0u, 0u, 0u);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  cluster_sync();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;
  const uint32_t tmem_lane = tmem_base + (static_cast<uint32_t>((warp & 3) * 32) << 16);
  const uint32_t a_addr = smem_u32(smem + Smem::A);
  const uint32_t bar_full_leader = map_to_cta(smem_u32(bar_full), 0);
  const uint32_t bar_a0_leader = map_to_cta(smem_u32(bar_a0), 0);
  constexpr uint32_t IDESC = umma_idesc_bf16(2 * TILE_M, HID);
  constexpr uint32_t IDESC_OUT = umma_idesc_bf16(2 * TILE_M, 16);
  uint32_t phase_w = 0;
  uint32_t ph_mma = 0, ph_out = 0;       // epilogue warps
  uint32_t ph_full = 0, ph_a0 = 0;       // MMA thread
  const PendulumConsts pc(a.reward);

  const int num_groups = (a.R + 2 * TILE_M - 1) / (2 * TILE_M);
  for (int group = blockIdx.x >> 1; group < num_groups; group += gridDim.x >> 1) {
    const int row = group * 2 * TILE_M + static_cast<int>(rank) * TILE_M + lrow;
    const bool valid = row < a.R;
    const int rr = valid ? row : a.R - 1;
    const int b = rr / a.M;
    const float x_init[3] = {a.x0[3 * b], a.x0[3 * b + 1], a.x0[3 * b + 2]};
    const float* act = a.actions + static_cast<size_t>(rr) * a.H;
    float summary = 0.0f;

    for (int e = 0; e < a.num_members; ++e) {
      // ---- member e: hidden weight halves by TMA; the small layers are split into bf16 parts here ----
      __syncthreads();  // every MMA of the previous member has completed (row owners waited bar_out)
      if (tid == 0) {
        mbar_expect_tx(bar_w, 2 * WH_BYTES);
        for (int l = 0; l < 2; ++l)
          for (int kc = 0; kc < KCHUNKS; ++kc)
            tma_load_2d(smem + (l ? Smem::W2 : Smem::W1) + kc * WH_LBO, &w_map, kc * 8,
                        (e * 2 + l) * HID + static_cast<int>(rank) * 128, bar_w);
      }
      if (tid < 128) {
        // layer 0, this CTA's 128 output units: per input [wh, wl, wh], then the bias [bh, bm, bl, 0]; all * 0.5
        const int n = static_cast<int>(rank) * 128 + tid;
        float wh[4], wl[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float w = 0.5f * a.w_in[(static_cast<size_t>(e) * 4 + i) * HID + n];
          wh[i] = bf16_hi(w);
          wl[i] = w - wh[i];
        }
        const float bias = 0.5f * a.b_in[e * HID + n];
        const float bh = bf16_hi(bias), bm = bf16_hi(bias - bh), bl = (bias - bh) - bm;
        uint4 p0, p1;
        p0.x = pack_bf16(wh[0], wl[0]); p0.y = pack_bf16(wh[0], wh[1]);
        p0.z = pack_bf16(wl[1], wh[1]); p0.w = pack_bf16(wh[2], wl[2]);
        p1.x = pack_bf16(wh[2], wh[3]); p1.y = pack_bf16(wl[3], wh[3]);
        p1.z = pack_bf16(bh, bm);       p1.w = pack_bf16(bl, 0.0f);
        *reinterpret_cast<uint4*>(smem + Smem::W0 + tid * 16) = p0;
        *reinterpret_cast<uint4*>(smem + Smem::W0 + WH_LBO + tid * 16) = p1;
      } else if (tid < 128 + HID && leader) {
        // output layer: row j (j < 3) = hi part of w_out[:, j], row 3 + j = lo part; rows 6, 7 stay zero
        const int k = tid - 128;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          const float w = a.w_out[(static_cast<size_t>(e) * HID + k) * 3 + j];
          const __nv_bfloat16 h = __float2bfloat16_rn(w);
          const __nv_bfloat16 l = __float2bfloat16_rn(w - __bfloat162float(h));
          uint8_t* base = smem + Smem::W3 + (k >> 3) * W3_LBO + (k & 7) * 2;
          *reinterpret_cast<__nv_bfloat16*>(base + j * 16) = h;
          *reinterpret_cast<__nv_bfloat16*>(base + (3 + j) * 16) = l;
        }
      }
      for (int i = tid; i < 2 * HID; i += ENS_THREADS) s_hb[i] = 0.5f * a.b_h[e * 2 * HID + i];
      if (tid < 3) s_b_out[tid] = a.b_out[e * 3 + tid];
      fence_proxy_async();        // generic-proxy writes of W0 / W3 -> visible to the tensor core
      mbar_wait(bar_w, phase_w);  // every thread observes the TMA completion
      phase_w ^= 1;
      __syncthreads();

      if (warp == MMA_WARP) {
        // ================= MMA issuer: warp 16 of the leader CTA =====================================
        // The whole warp runs the (warp-uniform) waits; one elected lane issues.  Every operand below is
        // derived from warp-uniform values and compile-time offsets, so the descriptors live in uniform
        // registers and each tcgen05.mma costs a handful of instructions.
        if (leader) {
          const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
          const bool elected = elect_one();
          const uint64_t desc_a = umma_desc(a_addr, A_LBO, SBO);
          const uint64_t desc_a0 = umma_desc(smem_u32(smem + Smem::A0), A_LBO, SBO);
          const uint64_t desc_w0 = umma_desc(smem_u32(smem + Smem::W0), WH_LBO, SBO);
          const uint64_t desc_w1 = umma_desc(smem_u32(smem + Smem::W1), WH_LBO, SBO);
          const uint64_t desc_w2 = umma_desc(smem_u32(smem + Smem::W2), WH_LBO, SBO);
          const uint64_t desc_w3 = umma_desc(smem_u32(smem + Smem::W3), W3_LBO, SBO);
#pragma unroll 1
          for (int t = 0; t < a.H; ++t) {
            mbar_wait(bar_a0, ph_a0);
            ph_a0 ^= 1;
            tc_fence_after();
            ENS_TRACE(lane == 0, 0);
            if (elected) {
              umma_bf16_ss_2sm(tmem_u, desc_a0, desc_w0, IDESC, 0u);
              umma_commit_2sm(bar_mma);
            }
            ENS_TRACE(lane == 0, 1);
#pragma unroll
            for (int layer = 1; layer <= 3; ++layer) {
              const uint32_t d = tmem_u + (layer & 1) * HID;
              const uint64_t desc_w = layer == 1 ? desc_w1 : (layer == 2 ? desc_w2 : desc_w3);
              constexpr uint32_t A_STEP = (2 * A_LBO) >> 4;      // one K = 16 step, in descriptor units
              const uint32_t w_step = (layer < 3 ? 2 * WH_LBO : 2 * W3_LBO) >> 4;
#pragma unroll
              for (int r = 0; r < ROUNDS; ++r) {
                mbar_wait(bar_full + r, ph_full);
                tc_fence_after();
                ENS_TRACE(lane == 0, 2 + (layer - 1) * 12 + r * 2);
                if (elected) {
#pragma unroll
                  for (int s = round_first_col(r) / 16; s < (round_first_col(r) + round_cols(r)) / 16; ++s)
                    umma_bf16_ss_2sm(d, desc_a + static_cast<uint64_t>(s * A_STEP),
                                     desc_w + static_cast<uint64_t>(s * w_step), layer < 3 ? IDESC : IDESC_OUT,
                                     s > 0 ? 1u : 0u);
                  if (r == ROUNDS - 1) umma_commit_2sm(layer < 3 ? bar_mma : bar_out);
                }
                ENS_TRACE(lane == 0, 3 + (layer - 1) * 12 + r * 2);
              }
              ph_full ^= 1;
            }
          }
        }
      } else {
        // ================= epilogue warps ============================================================
        float x[3] = {x_init[0], x_init[1], x_init[2]};
        float acc = 0.0f;
        float u = 0.0f;
        if (row_owner) {
          u = __ldg(act);
          build_a0_row(smem + Smem::A0 + lrow * 16, x[0], x[1], x[2], u);
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(bar_a0_leader);
        }
#pragma unroll 1
        for (int t = 0; t < a.H; ++t) {
          float u_next = 0.0f;
          if (row_owner) {
            // reward on the current state and the raw action (pendulum_reward.py:32-40); runs under MMA 0
            const float rw = reward_from(pc, atan2_bounded(x[1], x[0]), x[2], u);
            if (TR && valid) {
              const size_t o = (static_cast<size_t>(row) * a.num_members + e) * a.H + t;
              obs_out[3 * o] = x[0]; obs_out[3 * o + 1] = x[1]; obs_out[3 * o + 2] = x[2];
              reward_out[o] = rw;
            }
            acc = __fadd_rn(acc, rw);
            if (t + 1 < a.H) u_next = __ldg(act + t + 1);
          }
#pragma unroll
          for (int layer = 0; layer < 3; ++layer) {
            mbar_wait(bar_mma, ph_mma);   // accumulator of this layer complete; the A tile is free again
            ph_mma ^= 1;
            tc_fence_after();
            ENS_TRACE(tid == 0, 39 + layer * 8);
            ENS_TRACE(tid == 480, 71 + layer * 8);
            const uint32_t d_src = tmem_lane + (layer & 1) * HID;
            const float* hb = s_hb + (layer > 0 ? layer - 1 : 0) * HID;   // layers 1, 2 (layer 0's bias is in the MMA)
            uint8_t* a_row = smem + Smem::A + lrow * 16;
            // rounds 0-2: 16 columns per thread (K-step 4r + quarter); the loads run one round ahead
            uint32_t v[2][16];
            tmem_ld16_nowait(d_src + quarter * 16, v[0]);
#pragma unroll
            for (int r = 0; r < 3; ++r) {
              tmem_wait_ld16(v[r & 1]);
              if (r + 1 < 3) tmem_ld16_nowait(d_src + (r + 1) * 64 + quarter * 16, v[(r + 1) & 1]);
              uint8_t* dst = a_row + (8 * r + 2 * quarter) * A_LBO;
              if (layer == 0) epilogue_round<16, false>(v[r & 1], nullptr, dst);
              else epilogue_round<16, true>(v[r & 1], hb + r * 64 + quarter * 16, dst);
              publish_round(bar_full_leader + r * 8, lane);
              ENS_TRACE(tid == 0, 40 + layer * 8 + r);
              ENS_TRACE(tid == 480, 72 + layer * 8 + r);
            }
            {  // round 3: 8 columns per thread (K-chunk 24 + quarter)
              uint32_t w8[8];
              tmem_ld8_nowait(d_src + 192 + quarter * 8, w8);
              tmem_wait_ld8(w8);
              uint8_t* dst = a_row + (24 + quarter) * A_LBO;
              if (layer == 0) epilogue_round<8, false>(w8, nullptr, dst);
              else epilogue_round<8, true>(w8, hb + 192 + quarter * 8, dst);
              publish_round(bar_full_leader + 3 * 8, lane);
              ENS_TRACE(tid == 0, 40 + layer * 8 + 3);
            }
#pragma unroll
            for (int r = 4; r < 6; ++r) {  // rounds 4, 5: 4 columns per thread (half of K-chunk 28 / 30 + quarter / 2)
              uint32_t w4[4];
              const int col = round_first_col(r) + quarter * 4;
              tmem_ld4_nowait(d_src + col, w4);
              tmem_wait_ld4(w4);
              uint8_t* dst = a_row + (col >> 3) * A_LBO + (col & 7) * 2;
              if (layer == 0) epilogue_round<4, false>(w4, nullptr, dst);
              else epilogue_round<4, true>(w4, hb + col, dst);
              publish_round(bar_full_leader + r * 8, lane);
              ENS_TRACE(tid == 0, 40 + layer * 8 + r);
              ENS_TRACE(tid == 480, 72 + layer * 8 + r);
            }
          }
          if (row_owner) {
            mbar_wait(bar_out, ph_out);
            ph_out ^= 1;
            tc_fence_after();
            ENS_TRACE(tid == 384, 100);
            uint32_t o[8];
            tmem_ld8_nowait(tmem_lane + HID, o);
            tmem_wait_ld8(o);
            tc_fence_before();
            x[0] = __fadd_rn(x[0], (__uint_as_float(o[0]) + __uint_as_float(o[3])) + s_b_out[0]);
            x[1] = __fadd_rn(x[1], (__uint_as_float(o[1]) + __uint_as_float(o[4])) + s_b_out[1]);
            x[2] = __fadd_rn(x[2], (__uint_as_float(o[2]) + __uint_as_float(o[5])) + s_b_out[2]);
            if (t + 1 < a.H) {
              u = u_next;
              build_a0_row(smem + Smem::A0 + lrow * 16, x[0], x[1], x[2], u);
              fence_proxy_async();
              __syncwarp();
              if (lane == 0) mbar_arrive_cluster(bar_a0_leader);
              ENS_TRACE(tid == 384, 101);
            }
          }
        }
        if (row_owner) {
          const float ret = __fdiv_rn(acc, static_cast<float>(a.H));
          if (a.summarize == MBPO_SUMMARIZE_MAX) summary = (e == 0) ? ret : fmaxf(summary, ret);
          else summary = __fadd_rn(summary, ret);
        }
      }
    }
    if (row_owner && warp != MMA_WARP) {
      if (a.summarize != MBPO_SUMMARIZE_MAX) summary = __fdiv_rn(summary, static_cast<float>(a.num_members));
      if (!TR && valid) a.returns_out[row] = summary;   // TR: the caller summarises reward_out
    }
  }

  // ---- teardown --------------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  cluster_sync();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ENS_TMEM_COLS));
  }
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(ENS_THREADS, 1)
    ensemble_rollout_kernel(const __grid_constant__ EnsArgs a, const __grid_constant__ CUtensorMap w_map) {
  ensemble_rollout_body<false>(a, w_map, nullptr, nullptr);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(ENS_THREADS, 1)
    ensemble_transitions_kernel(const __grid_constant__ EnsArgs a, const __grid_constant__ CUtensorMap w_map,
                                float* __restrict__ obs_out, float* __restrict__ reward_out) {
  ensemble_rollout_body<true>(a, w_map, obs_out, reward_out);
}

// obs_out / reward_out null: the summary-only kernel; both set: ensemble_transitions_kernel, which also writes them.
inline int launch_ensemble_rollout(const MbpoMlpEnsembleParams& p, int horizon, const float* x0, const float* actions,
                                   int B, int M, int summarize, float* returns_out, float* obs_out, float* reward_out,
                                   cudaStream_t st, char* err, size_t errlen) {
  if (p.hidden != HID || p.x_dim != 3 || p.u_dim != 1 || p.num_members < 1) {
    snprintf(err, errlen,
             "ensemble rollout: the tcgen05 kernel needs hidden == 256, x_dim == 3, u_dim == 1 (got %d, %d, %d)",
             p.hidden, p.x_dim, p.u_dim);
    return MBPO_EUNSUPPORTED;
  }
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) {
    snprintf(err, errlen, "ensemble rollout: cuTensorMapEncodeTiled is not available from the driver");
    return MBPO_ECUDA;
  }
  CUtensorMap map;
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(HID), static_cast<cuuint64_t>(p.num_members) * 2 * HID};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(HID) * 2};
  const cuuint32_t box[2] = {8, 128};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult cr = enc(&map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<uint16_t*>(p.w_h), dims, strides, box,
                          estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) {
    snprintf(err, errlen, "ensemble rollout: cuTensorMapEncodeTiled failed (CUresult %d)", static_cast<int>(cr));
    return MBPO_ECUDA;
  }
  EnsArgs a;
  a.num_members = p.num_members; a.R = B * M; a.H = horizon; a.M = M; a.summarize = summarize;
  a.w_in = p.w_in; a.b_in = p.b_in; a.b_h = p.b_h; a.w_out = p.w_out; a.b_out = p.b_out;
  a.x0 = x0; a.actions = actions; a.returns_out = returns_out; a.reward = p.reward;
  const bool tr = obs_out != nullptr;
  cudaError_t ce = cudaFuncSetAttribute(tr ? reinterpret_cast<const void*>(ensemble_transitions_kernel)
                                           : reinterpret_cast<const void*>(ensemble_rollout_kernel),
                                        cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(Smem::TOTAL));
  if (ce != cudaSuccess) {
    snprintf(err, errlen, "ensemble rollout: smem attribute: %s", cudaGetErrorString(ce));
    return MBPO_ECUDA;
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int groups = (a.R + 2 * TILE_M - 1) / (2 * TILE_M);
  const int pairs = groups < sms / 2 ? groups : sms / 2;
  if (tr) ensemble_transitions_kernel<<<2 * pairs, ENS_THREADS, Smem::TOTAL, st>>>(a, map, obs_out, reward_out);
  else ensemble_rollout_kernel<<<2 * pairs, ENS_THREADS, Smem::TOTAL, st>>>(a, map);
  return MBPO_OK;
}

}  // namespace ens
}  // namespace mbpo
