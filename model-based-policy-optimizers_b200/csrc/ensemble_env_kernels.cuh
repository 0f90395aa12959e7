// Env rollouts and the policy in the loop for the learned MLP ensemble (MLPEnsembleSystem as a SAC / PPO env).
//
// The wrapper stack is general_wrapped_step's (general_env_kernels.cuh) around MLPEnsembleSystem.step:
//     x_next = x + MLP_m([x, u]),   reward = pendulum reward on (x, u)
// with env e rolled through member m[e] for its whole lifetime.  The model runs as in ensemble_rollout_kernel
// (ensemble_kernels.cuh): a CTA pair (tcgen05 cta_group::2) owns a tile of 256 rows, all four layers on the tensor
// cores with the same operand splits and roundings, the hidden weights resident by TMA, 16 epilogue warps and one
// issuer warp.  What changes:
//   tiles     a tile is 256 envs of ONE member.  The host hands over a stable env order sorted by member and the
//             per-member offsets (member_offsets[k] .. member_offsets[k + 1] are member k's envs in that order);
//             tile i maps to (member, rows) on the device, member after member, ceil(count / 256) tiles each.  The
//             pair grid-strides over tiles and reloads the weights only when the member changes; tiles past the
//             last member's exit.  Every row is read and written at its env's original index, so an env's outputs
//             do not depend on how the other envs are grouped.
//   per step  the row-owner warps (12-15, one thread per row) carry the env state and run the wrapper bookkeeping:
//             action_repeat model steps with the reward summed from 0, the step counter, truncation and done, obs =
//             first_obs where the episode ended, and the stores of the time-major Transition fields.
//   policy    with a policy (mode 1) the row owners run the NormalTanh policy of actor_rollout_general_kernel on the
//             env's observation between the output-layer commit (bar_out) and the next layer-0 MMA.  Its weights sit
//             past the model's shared memory; its hidden activations pass through the 64 KB activation tile A, free
//             in that window: every MMA that reads A has retired and the next layer-0 epilogue has not written it.
//             Without a policy (mode 0) the actions are read from [T, E, 1].
#pragma once
#include "ensemble_kernels.cuh"
#include "general_env_kernels.cuh"

namespace mbpo {
namespace ens {

// The policy fields fill_policy / load_general_policy / ens_policy_logits read (as GeneralActorArgs).
struct EnsPolicyArgs {
  int num_hidden, normalize, draw_offset, draw_total;
  float min_std;
  float obs_mean[4], obs_std[4];
  const float* obs_mean_dev;
  const float* obs_std_dev;
  const float* w[ACT_MAX_HIDDEN + 1];
  const float* b[ACT_MAX_HIDDEN + 1];
};

struct EnsEnvArgs {
  int num_members, E, T, episode_length, action_repeat, num_tiles;
  int policy, deterministic, key_convention;   // policy: 1 = policy in the loop, 0 = actions given
  const float* w_in;    // [M, 4, 256]
  const float* b_in;    // [M, 256]
  const float* b_h;     // [M, 2, 256]
  const float* w_out;   // [M, 256, 3]
  const float* b_out;   // [M, 3]
  MbpoPendulumParams reward;
  const int32_t* env_order;        // [E] env indices, stable-sorted by member
  const int32_t* member_offsets;   // [M + 1]
  float* obs;                      // [E,3] in/out
  float* steps;                    // [E]   in/out
  float* done;                     // [E]   in/out
  const float* first_obs;          // [E,3]
  const float* actions;            // [T,E] (mode 0)
  const uint32_t* key_in;          // [2] the policy's carry key (mode 1)
  uint32_t* key_out;               // [2] or NULL
  float* action_out;               // [T,E] (mode 1)
  float* reward_out;               // [T,E]
  float* discount_out;             // [T,E]
  float* next_observation_out;     // [T,E,3]
  float* truncation_out;           // [T,E]
  float* raw_action_out;           // [T,E] or NULL
  float* log_prob_out;             // [T,E] or NULL
  EnsPolicyArgs pol;
  GeneralActorSmem lay;            // the policy's float offsets past Smem::TOTAL (lay.h unused: A holds the columns)
};

constexpr uint32_t ENV_POLICY_NORM = Smem::TOTAL;             // float [8]: the normaliser's mean, std
constexpr uint32_t ENV_POLICY_W = ENV_POLICY_NORM + 8 * 4;    // the policy's weights and biases (lay offsets)
static_assert(ENV_POLICY_W % 16 == 0, "the policy's weights are read as float4");

// Tile -> (member, first slot in env_order, rows); member = -1 past the last member's tiles.
__device__ __forceinline__ void env_tile(const EnsEnvArgs& a, int tile, int& member, int& slot0, int& rows) {
  member = -1;
  int first = 0;
  for (int k = 0; k < a.num_members; ++k) {
    const int lo = __ldg(a.member_offsets + k), hi = __ldg(a.member_offsets + k + 1);
    const int nt = (hi - lo + 2 * TILE_M - 1) / (2 * TILE_M);
    if (tile < first + nt) {
      member = k;
      slot0 = lo + (tile - first) * 2 * TILE_M;
      rows = min(hi - slot0, 2 * TILE_M);
      return;
    }
    first += nt;
  }
}

// general_policy_logits (general_env_kernels.cuh) with the hidden activations in shared memory: the row's two
// 64-float columns h / h + 64 * TILE_M (stride TILE_M) in the free A tile hold layer l's input and output, so that
// no layer keeps 64 activations in registers (this kernel has 96 registers a thread).  Every output is the same
// operations in the same order as there.
__device__ __forceinline__ void ens_policy_logits(const EnsPolicyArgs& a, const float (&x)[3], const float* gsm,
                                                  const GeneralActorSmem& lay, const float* norm_sm, float* h,
                                                  float (&logits)[2]) {
  float xin[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) xin[i] = a.normalize ? __fdiv_rn(__fsub_rn(x[i], norm_sm[i]), norm_sm[4 + i]) : x[i];
  float* hc = h;
  float* hn = h + ACT_W * TILE_M;
  {
    const float* w0 = gsm + lay.w[0];   // [3][64]
    const float* b0 = gsm + lay.b[0];
#pragma unroll 8
    for (int j = 0; j < ACT_W; ++j) {
      float acc = xin[0] * w0[j];
      acc = fmaf(xin[1], w0[ACT_W + j], acc);
      acc = fmaf(xin[2], w0[2 * ACT_W + j], acc);
      hc[j * TILE_M] = swish_exact(acc + b0[j]);
    }
  }
  constexpr int JC = 16;   // outputs per pass
#pragma unroll 1
  for (int l = 1; l < a.num_hidden; ++l) {
    const float* wl = gsm + lay.w[l];
    const float* bl = gsm + lay.b[l];
#pragma unroll 1
    for (int jc = 0; jc < ACT_W / JC; ++jc) {
      float acc[JC];
#pragma unroll
      for (int i = 0; i < JC; ++i) acc[i] = 0.0f;
      const float4* wrow = reinterpret_cast<const float4*>(wl + jc * JC);
#pragma unroll 4
      for (int k = 0; k < ACT_W; ++k) {
        const float hk = hc[k * TILE_M];
#pragma unroll
        for (int q = 0; q < JC / 4; ++q) {
          const float4 w = wrow[k * (ACT_W / 4) + q];
          acc[4 * q + 0] = fmaf(hk, w.x, acc[4 * q + 0]); acc[4 * q + 1] = fmaf(hk, w.y, acc[4 * q + 1]);
          acc[4 * q + 2] = fmaf(hk, w.z, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(hk, w.w, acc[4 * q + 3]);
        }
      }
#pragma unroll
      for (int i = 0; i < JC; ++i) hn[(jc * JC + i) * TILE_M] = swish_exact(acc[i] + bl[jc * JC + i]);
    }
    float* tmp = hc; hc = hn; hn = tmp;
  }
  const float* wo = gsm + lay.w[a.num_hidden];   // [64][2]
  const float* bo = gsm + lay.b[a.num_hidden];
  logits[0] = 0.0f;
  logits[1] = 0.0f;
#pragma unroll 8
  for (int k = 0; k < ACT_W; ++k) {
    const float hk = hc[k * TILE_M];
    logits[0] = fmaf(hk, wo[2 * k], logits[0]);
    logits[1] = fmaf(hk, wo[2 * k + 1], logits[1]);
  }
  logits[0] += bo[0];
  logits[1] += bo[1];
}

// The action of env `env` at its observation x: mode 0 reads it, mode 1 runs the policy (the key plumbing of
// actor_rollout_general_kernel, then the network and the NormalTanh head) and stores action / raw_action / log_prob.
template <int PRNG>
__device__ __forceinline__ float env_action(const EnsEnvArgs& a, const float (&x)[3], int t, int env, bool valid,
                                            Key2& key, const float* gsm, const float* norm_sm, float* h_col) {
  const size_t i = static_cast<size_t>(t) * a.E + env;
  if (!a.policy) return valid ? __ldg(a.actions + i) : 0.0f;
  Key2 k_actor = key;
  if (a.key_convention != MBPO_KEYS_AS_IS) {
    Key2 first_k, second_k;
    split2<PRNG>(key, first_k, second_k);
    if (a.key_convention == MBPO_KEYS_SAC) { key = first_k; k_actor = second_k; }
    else { k_actor = first_k; key = second_k; }
  }
  float logits[2];
  ens_policy_logits(a.pol, x, gsm, a.lay, norm_sm, h_col, logits);
  const float mu = logits[0];
  float u;
  if (a.deterministic) {               // mode(): tanh(loc)
    u = tanhf(mu);
  } else {
    const uint32_t i_draw = static_cast<uint32_t>(a.pol.draw_offset + env);
    const float eps = bits_to_normal(random_bits_at<PRNG>(k_actor, static_cast<uint32_t>(a.pol.draw_total), i_draw));
    const float scale = softplus_exact(logits[1]) + a.pol.min_std;
    const float raw = __fadd_rn(__fmul_rn(scale, eps), mu);
    u = tanhf(raw);
    if (a.raw_action_out && valid) {
      const float z = __fdiv_rn(__fsub_rn(raw, mu), scale);
      const float lp = __fsub_rn(__fmul_rn(-0.5f, __fmul_rn(z, z)), __fadd_rn(0.918938533f, logf(scale)));
      const float ldj = __fmul_rn(2.0f, __fsub_rn(__fsub_rn(0.693147181f, raw), softplus_exact(__fmul_rn(-2.0f, raw))));
      a.raw_action_out[i] = raw;
      a.log_prob_out[i] = __fsub_rn(lp, ldj);
    }
  }
  if (valid) a.action_out[i] = u;
  return u;
}

template <int PRNG>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(ENS_THREADS, 1)
    ensemble_env_kernel(const __grid_constant__ EnsEnvArgs a, const __grid_constant__ CUtensorMap w_map) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int quarter = warp >> 2;
  const int lrow = ((warp & 3) << 5) | lane;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const bool row_owner = quarter == 3;   // warps 12-15 carry the envs' state (ensemble_rollout_kernel)
  float* s_hb = reinterpret_cast<float*>(smem + Smem::HB);
  float* s_b_out = reinterpret_cast<float*>(smem + Smem::B_OUT);
  float* norm_sm = reinterpret_cast<float*>(smem + ENV_POLICY_NORM);
  float* gsm = reinterpret_cast<float*>(smem + ENV_POLICY_W);
  float* h_col = reinterpret_cast<float*>(smem + Smem::A) + lrow;   // the policy's columns in the free A tile
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(smem + Smem::BARS);
  uint64_t* bar_a0 = bar_full + ROUNDS;
  uint64_t* bar_mma = bar_full + ROUNDS + 1;
  uint64_t* bar_out = bar_full + ROUNDS + 2;
  uint64_t* bar_w = bar_full + ROUNDS + 3;
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + Smem::TMEM_PTR);

  // ---- one-time setup (ensemble_rollout_kernel), plus the policy's weights ---------------------------------
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
  for (int i = tid; i < 8 * HID * 2 / 16; i += ENS_THREADS)
    reinterpret_cast<uint4*>(smem + Smem::W3)[i] = make_uint4(0u, 0u, 0u, 0u);
  if (a.policy) load_general_policy<3, 1>(a.pol, a.lay, gsm, norm_sm, tid, ENS_THREADS);
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
  uint32_t ph_mma = 0, ph_out = 0;
  uint32_t ph_full = 0, ph_a0 = 0;       // MMA thread; the phases carry over from tile to tile
  const PendulumConsts pc(a.reward);
  const int S = a.T * a.action_repeat;   // model steps per tile
  const float ep_len = static_cast<float>(a.episode_length);
  const float rep = static_cast<float>(a.action_repeat);
  int loaded = -1;

  for (int tile = blockIdx.x >> 1; tile < a.num_tiles; tile += gridDim.x >> 1) {
    int e = -1, slot0 = 0, rows = 0;
    env_tile(a, tile, e, slot0, rows);
    if (e < 0) break;   // the same tile index in both CTAs: the pair leaves together
    if (e != loaded) {
      // ---- member e: as ensemble_rollout_kernel ----------------------------------------------------------------
      loaded = e;
      __syncthreads();  // every MMA of the previous tile has completed (row owners waited bar_out)
      if (tid == 0) {
        mbar_expect_tx(bar_w, 2 * WH_BYTES);
        for (int l = 0; l < 2; ++l)
          for (int kc = 0; kc < KCHUNKS; ++kc)
            tma_load_2d(smem + (l ? Smem::W2 : Smem::W1) + kc * WH_LBO, &w_map, kc * 8,
                        (e * 2 + l) * HID + static_cast<int>(rank) * 128, bar_w);
      }
      if (tid < 128) {
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
      fence_proxy_async();
      mbar_wait(bar_w, phase_w);
      phase_w ^= 1;
      __syncthreads();
    }

    if (warp == MMA_WARP) {
      // ================= MMA issuer: S model steps, as ensemble_rollout_kernel's H ===========================
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
        for (int s = 0; s < S; ++s) {
          mbar_wait(bar_a0, ph_a0);
          ph_a0 ^= 1;
          tc_fence_after();
          if (elected) {
            umma_bf16_ss_2sm(tmem_u, desc_a0, desc_w0, IDESC, 0u);
            umma_commit_2sm(bar_mma);
          }
#pragma unroll
          for (int layer = 1; layer <= 3; ++layer) {
            const uint32_t d = tmem_u + (layer & 1) * HID;
            const uint64_t desc_w = layer == 1 ? desc_w1 : (layer == 2 ? desc_w2 : desc_w3);
            constexpr uint32_t A_STEP = (2 * A_LBO) >> 4;
            const uint32_t w_step = (layer < 3 ? 2 * WH_LBO : 2 * W3_LBO) >> 4;
#pragma unroll
            for (int r = 0; r < ROUNDS; ++r) {
              mbar_wait(bar_full + r, ph_full);
              tc_fence_after();
              if (elected) {
#pragma unroll
                for (int s2 = round_first_col(r) / 16; s2 < (round_first_col(r) + round_cols(r)) / 16; ++s2)
                  umma_bf16_ss_2sm(d, desc_a + static_cast<uint64_t>(s2 * A_STEP),
                                   desc_w + static_cast<uint64_t>(s2 * w_step), layer < 3 ? IDESC : IDESC_OUT,
                                   s2 > 0 ? 1u : 0u);
                if (r == ROUNDS - 1) umma_commit_2sm(layer < 3 ? bar_mma : bar_out);
              }
            }
            ph_full ^= 1;
          }
        }
      }
    } else {
      // ================= epilogue warps =====================================================================
      const int slot = static_cast<int>(rank) * TILE_M + lrow;
      const bool valid = slot < rows;
      const int env = valid ? __ldg(a.env_order + slot0 + slot) : 0;
      float x[3] = {0.0f, 0.0f, 0.0f};
      float steps = 0.0f, done = 0.0f, rew = 0.0f, u = 0.0f;
      Key2 key{0u, 0u};
      const float* first = a.first_obs + static_cast<size_t>(env) * 3;
      if (row_owner) {
        if (valid) {
#pragma unroll
          for (int k = 0; k < 3; ++k) x[k] = a.obs[static_cast<size_t>(env) * 3 + k];
          steps = a.steps[env];
          done = a.done[env];
        }
        if (a.policy) key = Key2{a.key_in[0], a.key_in[1]};
        // env step 0: AutoReset pre-step, the action
        steps = (done != 0.0f) ? 0.0f : steps;
        done = 0.0f;
        u = env_action<PRNG>(a, x, 0, env, valid, key, gsm, norm_sm, h_col);
        build_a0_row(smem + Smem::A0 + lrow * 16, x[0], x[1], x[2], u);
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(bar_a0_leader);
      }
      int t = 0, r_sub = 0;   // env step and model step within it (row owners)
#pragma unroll 1
      for (int s = 0; s < S; ++s) {
        if (row_owner) rew = __fadd_rn(rew, reward_from(pc, atan2_bounded(x[1], x[0]), x[2], u));   // under MMA 0
#pragma unroll
        for (int layer = 0; layer < 3; ++layer) {
          mbar_wait(bar_mma, ph_mma);
          ph_mma ^= 1;
          tc_fence_after();
          const uint32_t d_src = tmem_lane + (layer & 1) * HID;
          const float* hb = s_hb + (layer > 0 ? layer - 1 : 0) * HID;
          uint8_t* a_row = smem + Smem::A + lrow * 16;
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
          }
          {
            uint32_t w8[8];
            tmem_ld8_nowait(d_src + 192 + quarter * 8, w8);
            tmem_wait_ld8(w8);
            uint8_t* dst = a_row + (24 + quarter) * A_LBO;
            if (layer == 0) epilogue_round<8, false>(w8, nullptr, dst);
            else epilogue_round<8, true>(w8, hb + 192 + quarter * 8, dst);
            publish_round(bar_full_leader + 3 * 8, lane);
          }
#pragma unroll
          for (int r = 4; r < 6; ++r) {
            uint32_t w4[4];
            const int col = round_first_col(r) + quarter * 4;
            tmem_ld4_nowait(d_src + col, w4);
            tmem_wait_ld4(w4);
            uint8_t* dst = a_row + (col >> 3) * A_LBO + (col & 7) * 2;
            if (layer == 0) epilogue_round<4, false>(w4, nullptr, dst);
            else epilogue_round<4, true>(w4, hb + col, dst);
            publish_round(bar_full_leader + r * 8, lane);
          }
        }
        if (row_owner) {
          mbar_wait(bar_out, ph_out);
          ph_out ^= 1;
          tc_fence_after();
          uint32_t o[8];
          tmem_ld8_nowait(tmem_lane + HID, o);
          tmem_wait_ld8(o);
          tc_fence_before();
          x[0] = __fadd_rn(x[0], (__uint_as_float(o[0]) + __uint_as_float(o[3])) + s_b_out[0]);
          x[1] = __fadd_rn(x[1], (__uint_as_float(o[1]) + __uint_as_float(o[4])) + s_b_out[1]);
          x[2] = __fadd_rn(x[2], (__uint_as_float(o[2]) + __uint_as_float(o[5])) + s_b_out[2]);
          if (++r_sub == a.action_repeat) {
            // ---- end of env step t: Episode / AutoReset bookkeeping (general_wrapped_step), Transition out ----
            r_sub = 0;
            steps = __fadd_rn(steps, rep);
            const bool over = steps >= ep_len;
            const float trunc = over ? (1.0f - done) : 0.0f;
            done = over ? 1.0f : done;
            if (over) {
#pragma unroll
              for (int k = 0; k < 3; ++k) x[k] = __ldg(first + k);
            }
            if (valid) {
              const size_t i = static_cast<size_t>(t) * a.E + env;
              float* no = a.next_observation_out + i * 3;
              no[0] = x[0]; no[1] = x[1]; no[2] = x[2];
              a.reward_out[i] = rew;
              a.discount_out[i] = 1.0f - done;
              a.truncation_out[i] = trunc;
            }
            rew = 0.0f;
            if (++t < a.T) {
              steps = (done != 0.0f) ? 0.0f : steps;
              done = 0.0f;
              u = env_action<PRNG>(a, x, t, env, valid, key, gsm, norm_sm, h_col);
            }
          }
          if (s + 1 < S) {
            build_a0_row(smem + Smem::A0 + lrow * 16, x[0], x[1], x[2], u);
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(bar_a0_leader);
          }
        }
      }
      if (row_owner && valid) {
#pragma unroll
        for (int k = 0; k < 3; ++k) a.obs[static_cast<size_t>(env) * 3 + k] = x[k];
        a.steps[env] = steps;
        a.done[env] = done;
      }
    }
  }

  // the carry key after T steps: the same for every env, so one thread replays its splits
  if (a.policy && a.key_out && blockIdx.x == 0 && tid == 0) {
    Key2 key{a.key_in[0], a.key_in[1]};
    if (a.key_convention != MBPO_KEYS_AS_IS) {
      for (int t = 0; t < a.T; ++t) {
        Key2 first_k, second_k;
        split2<PRNG>(key, first_k, second_k);
        key = a.key_convention == MBPO_KEYS_SAC ? first_k : second_k;
      }
    }
    a.key_out[0] = key.k0;
    a.key_out[1] = key.k1;
  }

  // ---- teardown --------------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  cluster_sync();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ENS_TMEM_COLS));
  }
}

}  // namespace ens
}  // namespace mbpo
