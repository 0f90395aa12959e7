// Policy-in-the-loop data collection with the policy network on the 5th-generation tensor cores.
//
// Same computation, arguments and outputs as actor_rollout_pendulum_kernel (actor_kernels.cuh: T steps of
// actor_step, sac/acting.py:35-55, for E envs in one launch).  The hidden -> hidden layers of the policy MLP
// (64 x 64, the GEMM-shaped part: M = envs) run as tcgen05.mma kind::tf32 with the accumulator in TMEM; the
// reference network is float32, so every operand is split into a TF32 head and a TF32 tail
//     a = a_hi + a_lo,  w = w_hi + w_lo,   a.w ~= a_hi.w_hi + a_lo.w_hi + a_hi.w_lo      (fp32 accumulate)
// with both parts rounded to nearest (|a_lo| <= 2^-12 |a|): the dropped a_lo.w_lo term is 2^-24 relative, i.e.
// the products are fp32-accurate and the actions agree with the float32 oracle to the same tolerance as the
// CUDA-core kernel.
//
//   CTA           four independent tiles of 128 envs (512 producer threads: thread = env = TMEM lane) plus one
//                 MMA-issuing warp per tile.  A tile's step is a chain of short phases separated by tensor-core
//                 latencies; four tiles per SM (four producer warps per scheduler) keep the issue slots busy, and
//                 the warps of a tile meet only through mbarriers (no block or named barrier in the step loop)
//   A operand     a tile never holds a whole [128 x 64] activation matrix: the producer (layer 0 on the CUDA
//                 cores, or the epilogue of the previous accumulator) emits 16 columns at a time into a ring of
//                 two 16 KB slots (hi and lo planes, canonical K-major no-swizzle UMMA layout: 16-byte chunk kc of
//                 row r at kc * 2048 + r * 16); each producer warp arrives on the slot's `full` mbarrier, the tile's
//                 issuer waits for the four arrivals and issues the six MMAs that consume the slot, and a
//                 tcgen05.commit per slot tells the producers when it may be overwritten -- the MMAs of one quarter
//                 run under the production of the next
//   B operand     each hidden -> hidden weight matrix as two planes (hi, lo), element (n, k) at
//                 (k / 4) * 1024 + n * 16 + (k % 4) * 4, resident in shared memory for the whole launch
//   D             two 64-column TMEM accumulators per tile, alternating between layers (512 columns per CTA)
//   layer 0       (K = 3) and the output layer (N = 2) stay on the CUDA cores, fused into the producers
//   head, PRNG, wrapped env step, Transition stores: the shared device functions of actor_kernels.cuh
#pragma once
#include "actor_kernels.cuh"
#include "mlp_tc_kernels.cuh"

namespace mbpo {
namespace atc {

using namespace tc;   // PTX wrappers: mbarrier, fences, umma_desc, umma_commit

constexpr int TILE = 128;                 // envs per tile = TMEM lanes
constexpr int TILES_PER_CTA = 4;
constexpr int ENV_THREADS_ = TILE * TILES_PER_CTA;      // 512 producer threads: thread = env
constexpr int THREADS = ENV_THREADS_ + 32 * TILES_PER_CTA;   // + one MMA-issuing warp per tile (one lane active)
constexpr int W = ACT_W;                  // 64
#ifndef MBPO_ATC_QC
#define MBPO_ATC_QC 16
#endif
#ifndef MBPO_ATC_SLOTS
#define MBPO_ATC_SLOTS 2
#endif
constexpr int QC = MBPO_ATC_QC;           // columns a producer emits per ring slot (QC / 8 MMA K-steps)
constexpr int QUARTERS = W / QC;
constexpr uint32_t A_LBO_ = TILE * 16;    // 2048: next 16-byte K-chunk of A
constexpr uint32_t W_LBO_ = W * 16;       // 1024: next 16-byte K-chunk of W
constexpr uint32_t SLOT_PLANE = (QC / 4) * A_LBO_;   // 8192: one plane (hi or lo) of a slot
constexpr uint32_t SLOT_BYTES = 2 * SLOT_PLANE;      // 16384
constexpr int SLOTS = MBPO_ATC_SLOTS;
constexpr uint32_t W_PLANE = W * W * 4;   // 16384
constexpr int MAX_HH = 2;                 // hidden -> hidden layers held in shared memory (num_hidden <= 3)
constexpr int TMEM_COLS_ = 512;           // 4 tiles x 2 accumulators x 64 fp32 columns

constexpr int BARS_PER_TILE = 2 * SLOTS + 2;
constexpr uint32_t BAR_FULL = SLOTS * 8u, BAR_LAYER = 2u * SLOTS * 8u;   // byte offsets inside a tile's barrier block
struct Smem {
  static constexpr uint32_t A = 0;                                         // [tile][slot][hi, lo]
  static constexpr uint32_t WH = A + TILES_PER_CTA * SLOTS * SLOT_BYTES;   // [layer][hi, lo] planes
  static constexpr uint32_t W0 = WH + MAX_HH * 2 * W_PLANE;                // float [3][64]
  static constexpr uint32_t B0 = W0 + 3 * W * 4;                           // float [64]
  static constexpr uint32_t BH = B0 + W * 4;                               // float [MAX_HH][64]
  static constexpr uint32_t WO = BH + MAX_HH * W * 4;                      // float [64][2]
  static constexpr uint32_t BO = WO + W * 2 * 4;                           // float [2] (+ pad)
  static constexpr uint32_t TILES = BO + 16;                               // float [16 warps][96]: row transposition
  static constexpr uint32_t BARS = TILES + (ENV_THREADS_ / 32) * 96 * 4;   // per tile: slot_free[SLOTS], full[SLOTS], layer_done
  static constexpr uint32_t TMEM_PTR = BARS + TILES_PER_CTA * BARS_PER_TILE * 8;
  static constexpr uint32_t TOTAL = TMEM_PTR + 16;
};
static_assert(Smem::TOTAL <= 227 * 1024, "tensor-core actor kernel shared memory plan exceeds 227 KB");

// Instruction descriptor for kind::tf32: D = F32 (1 @ [4,6)), A = B = TF32 (2 @ [7,10), [10,13)), K-major,
// N >> 3 @ [17,23), M >> 4 @ [24,29).
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ldq(uint32_t taddr, uint32_t (&v)[16]) { tmem_ld16(taddr, v); }
__device__ __forceinline__ void tmem_ldq(uint32_t taddr, uint32_t (&v)[8]) { tmem_ld8(taddr, v); }
__device__ __forceinline__ void tmem_ldq(uint32_t taddr, uint32_t (&v)[32]) { tmem_ld32(taddr, v); }
// mbarrier helpers on precomputed 32-bit shared addresses (the generic -> shared conversion stays out of the loops)
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void umma_commit_a(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// round to nearest TF32 (low 13 mantissa bits clear, ties away from zero like cvt.rna.tf32.f32 -- which ptxas
// expands to a five-instruction sequence on sm_100a; the integer form is two)
__device__ __forceinline__ float to_tf32(float v) {
  return __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u);
}
// v ~= hi + lo, both exactly representable in TF32: hi = v rounded to nearest, so |lo| <= 2^-12 |v| and rounding
// lo loses <= 2^-24 |v| -- the three-product sum is fp32-accurate.
__device__ __forceinline__ void split_tf32(float v, float& hi, float& lo) {
  hi = to_tf32(v);
  lo = to_tf32(v - hi);
}
__device__ __forceinline__ float ex2_approx(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// swish on a pair: x * sigmoid(x), sigmoid = 1 / (1 + ex2(-x * log2(e))).  The MUFU pipe (4 results per clock per
// scheduler) is what bounds this kernel, so the two reciprocals share one MUFU.RCP: r = rcp(a0 * a1), 1 / a0 = r * a1,
// 1 / a1 = r * a0 (three MUFU per pair instead of four; ~2^-22 relative instead of 2^-23).  The exponent is clamped
// to 2^64 so that a0 * a1 overflows to +inf at worst -- rcp(inf) = 0 and 0 * finite = 0, which is what x * sigmoid(x)
// rounds to there (|x| > 44) -- and never meets an infinite factor.
__device__ __forceinline__ void swish2(float x0, float x1, float& y0, float& y1) {
  const f32x2_t x = pack2(x0, x1);
  float t0, t1;
  unpack2(mul2(x, pack2(-1.44269504f, -1.44269504f)), t0, t1);
  float a0, a1;
  unpack2(add2(pack2(ex2_approx(fminf(t0, 64.0f)), ex2_approx(fminf(t1, 64.0f))), pack2(1.0f, 1.0f)), a0, a1);
  const float r = rcp_approx(a0 * a1);
  unpack2(mul2(x, mul2(pack2(r, r), pack2(a1, a0))), y0, y1);
}
// v ~= hi + lo for a pair.  The tensor core reads TF32 operands from 32-bit containers and ignores the low 13
// mantissa bits, so lo needs no mask: adding half a TF32 ulp to its bit pattern makes that truncation a
// round-to-nearest (|lo| <= 2^-12 |v|: the rounding loses at most 2^-24 |v|).
__device__ __forceinline__ void split_tf32_2(float v0, float v1, float& h0, float& h1, float& l0, float& l1) {
  h0 = to_tf32(v0); h1 = to_tf32(v1);
  float d0, d1;
  unpack2(add2(pack2(v0, v1), pack2(-h0, -h1)), d0, d1);
  l0 = __uint_as_float(__float_as_uint(d0) + 0x1000u);
  l1 = __uint_as_float(__float_as_uint(d1) + 0x1000u);
}

template <int PRNG, int MATH>
__global__ void __launch_bounds__(THREADS, 1) actor_rollout_tc_kernel(const __grid_constant__ ActorArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ float norm_sm[8];     // normaliser mean [0..2], std [4..6]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < 3) {
    norm_sm[tid] = a.obs_mean_dev ? a.obs_mean_dev[tid] : a.obs_mean[tid];
    norm_sm[4 + tid] = a.obs_std_dev ? a.obs_std_dev[tid] : a.obs_std[tid];
  }
  const bool issuer_warp = tid >= ENV_THREADS_;
  const int g = issuer_warp ? (tid - ENV_THREADS_) / 32 : tid / TILE;   // tile of the CTA
  const int r = tid % TILE;                                             // row of the tile (producer threads)
  float* s_w0 = reinterpret_cast<float*>(smem + Smem::W0);
  float* s_b0 = reinterpret_cast<float*>(smem + Smem::B0);
  float* s_bh = reinterpret_cast<float*>(smem + Smem::BH);
  float* s_wo = reinterpret_cast<float*>(smem + Smem::WO);
  float* s_bo = reinterpret_cast<float*>(smem + Smem::BO);
  float* tile = reinterpret_cast<float*>(smem + Smem::TILES) + (warp & 15) * 96;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Smem::BARS) + g * BARS_PER_TILE;
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + Smem::TMEM_PTR);
  const int L = a.num_hidden, HH = L - 1;

  // ---- one-time setup: TMEM, mbarriers, policy parameters -> shared memory ---------------------------------
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                 "r"(TMEM_COLS_));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (!issuer_warp && r == 0) {
    for (int i = 0; i < SLOTS; ++i) {
      mbar_init(&bars[i], 1);                    // slot_free: one tcgen05.commit
      mbar_init(&bars[SLOTS + i], TILE / 32);    // full: one arrival per producer warp
    }
    mbar_init(&bars[2 * SLOTS], 1);              // layer_done
    fence_barrier_init();
  }
  for (int l = 0; l < HH; ++l) {
    const float* wl = a.w[l + 1];                        // flax Dense kernel [in = k][out = n]
    uint8_t* hi = smem + Smem::WH + (l * 2 + 0) * W_PLANE;
    uint8_t* lo = smem + Smem::WH + (l * 2 + 1) * W_PLANE;
    for (int i = tid; i < W * W; i += THREADS) {
      const int k = i / W, n = i % W;
      float h, t;
      split_tf32(wl[i], h, t);
      const uint32_t off = (k / 4) * W_LBO_ + n * 16 + (k % 4) * 4;
      *reinterpret_cast<float*>(hi + off) = h;
      *reinterpret_cast<float*>(lo + off) = t;
    }
    for (int i = tid; i < W; i += THREADS) s_bh[l * W + i] = a.b[l + 1][i];
  }
  for (int i = tid; i < 3 * W; i += THREADS) s_w0[i] = a.w[0][i];
  for (int i = tid; i < W; i += THREADS) s_b0[i] = a.b[0][i];
  for (int i = tid; i < W * 2; i += THREADS) s_wo[i] = a.w[L][i];
  if (tid < 2) s_bo[tid] = a.b[L][tid];
  fence_proxy_async();          // the weight planes are read by the tensor core (async proxy)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  // Few envs: spread the tiles over more SMs (a.tiles_per_cta < 4) -- a tile alone on an SM steps faster than
  // four sharing it, and the launch is T sequential steps whatever the grid.
  const int tile_idx = blockIdx.x * a.tiles_per_cta + g;
  const int tile_e0 = g < a.tiles_per_cta ? tile_idx * TILE : a.E;
  const uint32_t tmem_tile = tmem_base + g * 2 * W;                                          // two accumulators
  uint8_t* ring = smem + Smem::A + g * SLOTS * SLOT_BYTES;
  if (issuer_warp) {
    // ---- MMA issuer of tile g: one lane follows the producers' schedule (T steps x HH stages x 4 quarters) -----
    if (tile_e0 < a.E && lane == 0) {
      // descriptors: only the start-address field (16-byte units, bits [0,14)) varies
      const uint64_t da0 = umma_desc(smem_u32(ring), A_LBO_, SBO);
      const uint64_t db0 = umma_desc(smem_u32(smem + Smem::WH), W_LBO_, SBO);
      constexpr uint32_t IDESC = umma_idesc_tf32(TILE, W);
      uint32_t uses = 0;
      const uint32_t bar0 = smem_u32(bars);
#pragma unroll 1
      for (int t = 0; t < a.T; ++t) {
#pragma unroll 1
        for (int s = 0; s < HH; ++s) {
          const uint32_t d = tmem_tile + (s & 1) * W;
#pragma unroll 1
          for (int qd = 0; qd < QUARTERS; ++qd) {
            const uint32_t slot = uses % SLOTS;
            mbar_wait_a(bar0 + BAR_FULL + slot * 8u, (uses / SLOTS) & 1u);   // the four producer warps have written the slot
            tc_fence_after();
            // ---- 6 x tcgen05.mma (M128 N64 K8): lo.hi + hi.lo + hi.hi for the two K-steps of this slot ----------------
            const uint64_t a_hi = da0 + ((slot * SLOT_BYTES) >> 4), a_lo = a_hi + (SLOT_PLANE >> 4);
            const uint64_t b_hi = db0 + ((static_cast<uint32_t>(s) * 2u * W_PLANE + qd * (QC / 4) * W_LBO_) >> 4);
            const uint64_t b_lo = b_hi + (W_PLANE >> 4);
#pragma unroll
            for (int j = 0; j < QC / 8; ++j) {
              const uint64_t ao = static_cast<uint64_t>((j * 2 * A_LBO_) >> 4), bo = static_cast<uint64_t>((j * 2 * W_LBO_) >> 4);
              umma_tf32_ss(d, a_lo + ao, b_hi + bo, IDESC, (qd | j) ? 1u : 0u);     // small terms first
              umma_tf32_ss(d, a_hi + ao, b_lo + bo, IDESC, 1u);
              umma_tf32_ss(d, a_hi + ao, b_hi + bo, IDESC, 1u);
            }
            umma_commit_a(bar0 + slot * 8u);                        // slot free when these MMAs have read it
            if (qd == QUARTERS - 1) umma_commit_a(bar0 + BAR_LAYER);   // accumulator s & 1 complete
            ++uses;
          }
        }
      }
    }
  } else if (tile_e0 < a.E) {   // tile-uniform: an idle tile skips the loop (tiles share no barrier in it)
    const uint32_t tmem_rd = tmem_tile + (static_cast<uint32_t>((warp & 3) * 32) << 16);    // this warp's 32 lanes
    uint32_t uses = 0;          // ring slots written so far (slot = uses & 1)
    uint32_t layer_phase = 0;
    const uint32_t bar0 = smem_u32(bars);

    const PendulumConsts pc(a.sys);
    const float ep_len = static_cast<float>(a.episode_length);
    const float rep = static_cast<float>(a.action_repeat);
    const size_t E = static_cast<size_t>(a.E);
    const int e = tile_e0 + r;
    const bool live = e < a.E;
    const int ee = live ? e : a.E - 1;                 // dead rows shadow the last env, their stores are masked
    const int warp_e0 = e - lane;
    const int rem = a.E - warp_e0;
    const int n_valid = (rem < 32 ? (rem > 0 ? rem : 0) : 32) * 3;
    ActorEnv v;
    v.c = a.obs[3 * ee]; v.s = a.obs[3 * ee + 1]; v.w = a.obs[3 * ee + 2];
    v.f_c = a.first_obs[3 * ee]; v.f_s = a.first_obs[3 * ee + 1]; v.f_w = a.first_obs[3 * ee + 2];
    v.steps = a.steps[ee]; v.done = a.done[ee];
    v.th = (MATH == MBPO_MATH_REFERENCE) ? 0.0f : atan2_bounded(v.s, v.c);
    v.f_th = (MATH == MBPO_MATH_REFERENCE) ? 0.0f : atan2_bounded(v.f_s, v.f_c);
    Key2 key{a.key_in[0], a.key_in[1]};
    // (every thread carries the same keys) per step: k, k_t = split(k) in the caller's convention
    auto advance_keys = [&](Key2 k, Key2& k_act, Key2& k_carry) {
      k_act = k; k_carry = k;
      if (a.key_convention != 2) {
        Key2 first, second;
        split2<PRNG>(k, first, second);
        if (a.key_convention == 0) { k_carry = first; k_act = second; }   // sac.py:290
        else { k_act = first; k_carry = second; }                          // acting.py:70
      }
    };
    Key2 k_actor_next, key_next;
    advance_keys(key, k_actor_next, key_next);

#pragma unroll 1
    for (int t = 0; t < a.T; ++t) {
      // ---- key plumbing: this step's keys were derived during the previous step's last MMA wait ------------------
      const Key2 k_actor = k_actor_next;
      key = key_next;
      float xin[3] = {v.c, v.s, v.w};
      if (a.normalize) {
#pragma unroll
        for (int i = 0; i < 3; ++i) xin[i] = __fdiv_rn(__fsub_rn(xin[i], norm_sm[i]), norm_sm[4 + i]);
      }
      float loc = 0.0f, raw_sc = 0.0f, eps = 0.0f;
      const f32x2_t x0p = pack2(xin[0], xin[0]), x1p = pack2(xin[1], xin[1]), x2p = pack2(xin[2], xin[2]);

      // stage s produces the A operand of hidden -> hidden layer s: from layer 0 on the CUDA cores (s = 0) or from
      // accumulator (s - 1) & 1; its MMAs accumulate into accumulator s & 1.  Stage HH is the output layer.
#pragma unroll 1
      for (int s = 0; s <= HH; ++s) {
        const bool to_mma = s < HH;
        const float* bias = s_bh + (s - 1) * W;
        const uint32_t acc_src = tmem_rd + ((s - 1) & 1) * W;
#pragma unroll 1
        for (int qd = 0; qd < QUARTERS; ++qd) {
          float h[QC];
          if (s == 0) {
            // ---- layer 0: the same float operations as the CUDA-core kernel's first layer -------------------------
#pragma unroll
            for (int j4 = 0; j4 < QC / 4; ++j4) {
              const int c0 = qd * QC + j4 * 4;
              const float4 r0 = *reinterpret_cast<const float4*>(s_w0 + c0);
              const float4 r1 = *reinterpret_cast<const float4*>(s_w0 + W + c0);
              const float4 r2 = *reinterpret_cast<const float4*>(s_w0 + 2 * W + c0);
              const float4 bb = *reinterpret_cast<const float4*>(s_b0 + c0);
              const float w0r[4] = {r0.x, r0.y, r0.z, r0.w}, w1r[4] = {r1.x, r1.y, r1.z, r1.w};
              const float w2r[4] = {r2.x, r2.y, r2.z, r2.w}, b0r[4] = {bb.x, bb.y, bb.z, bb.w};
              // the same float operations per element as the CUDA-core kernel's first layer, two units per instruction
              float pre[4];
#pragma unroll
              for (int i = 0; i < 4; i += 2) {
                const f32x2_t acc2 = fma2(x2p, pack2(w2r[i], w2r[i + 1]),
                                          fma2(x1p, pack2(w1r[i], w1r[i + 1]), mul2(x0p, pack2(w0r[i], w0r[i + 1]))));
                unpack2(add2(acc2, pack2(b0r[i], b0r[i + 1])), pre[i], pre[i + 1]);
              }
              swish2(pre[0], pre[1], h[j4 * 4], h[j4 * 4 + 1]);
              swish2(pre[2], pre[3], h[j4 * 4 + 2], h[j4 * 4 + 3]);
            }
          } else {
            // ---- epilogue of the previous layer: 16 accumulator columns, bias + swish ---------------------------
            uint32_t acc[QC];
            tmem_ldq(acc_src + qd * QC, acc);
#pragma unroll
            for (int j4 = 0; j4 < QC / 4; ++j4) {
              const float4 bb = *reinterpret_cast<const float4*>(bias + qd * QC + j4 * 4);
              float x0, x1, x2, x3;
              unpack2(add2(pack2(__uint_as_float(acc[j4 * 4]), __uint_as_float(acc[j4 * 4 + 1])), pack2(bb.x, bb.y)), x0, x1);
              unpack2(add2(pack2(__uint_as_float(acc[j4 * 4 + 2]), __uint_as_float(acc[j4 * 4 + 3])), pack2(bb.z, bb.w)), x2, x3);
              swish2(x0, x1, h[j4 * 4], h[j4 * 4 + 1]);
              swish2(x2, x3, h[j4 * 4 + 2], h[j4 * 4 + 3]);
            }
          }
          if (!to_mma) {        // output layer on the CUDA cores, float32
            // one partial per 16-column quarter, the quarters added in order: the order of the wide kernel
            // (actor_tc_wide_kernels.cuh), whose quarters live in different threads -- both kernels agree bit for bit
            static_assert(QC <= 16 && 16 % QC == 0, "output-layer partials are per 16 columns");
            float pl = 0.0f, ps = 0.0f;
#pragma unroll
            for (int i = 0; i < QC; i += 2) {
              const float4 wo = *reinterpret_cast<const float4*>(s_wo + (qd * QC + i) * 2);
              pl = fmaf(h[i], wo.x, pl);
              ps = fmaf(h[i], wo.y, ps);
              pl = fmaf(h[i + 1], wo.z, pl);
              ps = fmaf(h[i + 1], wo.w, ps);
            }
#ifdef MBPO_ATC_SERIAL_OUT     // A/B switch: the single 64-term chain of the first version (not bit-equal to the wide kernel)
            if (false) {
#else
            if (QC == 16) {
#endif
              loc = qd == 0 ? pl : __fadd_rn(loc, pl);
              raw_sc = qd == 0 ? ps : __fadd_rn(raw_sc, ps);
            } else {            // ring experiments with narrower slots: plain running sum
              loc += pl;
              raw_sc += ps;
            }
            continue;
          }
          // ---- hi / lo planes of the 16 columns into the ring slot ----------------------------------------------------
          const uint32_t slot = uses % SLOTS;
          if (uses >= SLOTS) mbar_wait_a(bar0 + slot * 8u, ((uses / SLOTS) - 1u) & 1u);   // the MMAs that read it have retired
          uint8_t* dst = ring + slot * SLOT_BYTES + r * 16;
#pragma unroll
          for (int j4 = 0; j4 < QC / 4; ++j4) {
            float hi[4], lo[4];
            split_tf32_2(h[j4 * 4], h[j4 * 4 + 1], hi[0], hi[1], lo[0], lo[1]);
            split_tf32_2(h[j4 * 4 + 2], h[j4 * 4 + 3], hi[2], hi[3], lo[2], lo[3]);
            *reinterpret_cast<float4*>(dst + j4 * A_LBO_) = make_float4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<float4*>(dst + SLOT_PLANE + j4 * A_LBO_) = make_float4(lo[0], lo[1], lo[2], lo[3]);
          }
          fence_proxy_async();      // generic-proxy writes of A -> visible to the tensor core
          tc_fence_before();        // and this thread's accumulator reads are ordered before the MMAs they feed
          __syncwarp();
          if (lane == 0) mbar_arrive_a(bar0 + BAR_FULL + slot * 8u);
          ++uses;
        }
        // network-independent work fills the MMA waits: this step's draw, the next step's keys
        if (s == 0) eps = actor_draw<PRNG>(a, k_actor, ee);
        if (s == HH - 1) advance_keys(key, k_actor_next, key_next);
        if (to_mma) {
          mbar_wait_a(bar0 + BAR_LAYER, layer_phase);
          layer_phase ^= 1u;
          tc_fence_after();
        }
      }
      // ---- head, wrapped env step, Transition ------------------------------------------------------------------
      const float u = actor_head(a, eps, loc + s_bo[0], raw_sc + s_bo[1], ee, live, t);
      float trunc;
      const float rew = actor_env_step<MATH>(a, pc, v, u, ep_len, rep, trunc);
      const size_t row = static_cast<size_t>(t) * E;
      if (warp_e0 < a.E)        // warp-uniform
        warp_store3(tile, a.next_observation_out + (row + warp_e0) * 3 + lane, lane, n_valid, v.c, v.s, v.w);
      if (live) {
        a.action_out[row + e] = u;
        a.reward_out[row + e] = rew;
        a.discount_out[row + e] = 1.0f - v.done;
        a.truncation_out[row + e] = trunc;
      }
    }
    if (live) {
      a.obs[3 * e] = v.c; a.obs[3 * e + 1] = v.s; a.obs[3 * e + 2] = v.w;
      a.steps[e] = v.steps;
      a.done[e] = v.done;
    }
    if (tile_idx == 0 && r == 0 && a.key_out) { a.key_out[0] = key.k0; a.key_out[1] = key.k1; }
  }

  // ---- teardown ----------------------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS_));
  }
}

}  // namespace atc
}  // namespace mbpo
