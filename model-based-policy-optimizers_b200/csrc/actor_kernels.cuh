// Policy-in-the-loop data collection: actor_step / generate_unroll / SAC get_experience.
//
// Reference (per env and step):
//   policy            sac/sac_networks.py:58-73     logits = MLP(obs)  (swish, Dense = x @ W + b,
//                                                   utils/network_utils.py:5-17 style stack)
//   NormalTanh        sac/parametric_distribution.py:97-125   loc, scale = split(logits, 2);
//                                                   scale = softplus(scale) + min_std;
//                                                   raw = scale * normal(key, [E, A]) + loc; action = tanh(raw)
//                                                   (deterministic: action = tanh(loc))
//   actor_step        sac/acting.py:35-55           nstate = env.step(state, action); Transition(obs, action,
//                                                   reward, 1 - done, next_obs, truncation)
//   key per step      sac/sac.py:288-292            k, k_t = split(k); actor key = k_t          (convention 0)
//                     sac/acting.py:68-73           current, next = split(current); actor key = current,
//                                                   carry = next                                  (convention 1)
//   env.step          the wrapper stack of env_kernels.cuh (AutoReset / Episode / BraxWrapper / System.step)
//
// One thread per PAIR of environments, T steps per launch.  The network runs in float32 on the CUDA cores (the
// reference network is float32; operand rounding to bf16 would change the collected actions): the
// thread's current activations live in registers as packed (env 0, env 1) pairs, the weights are read from
// shared memory with warp-broadcast 128-bit loads, and each weight feeds one packed FFMA2 (scalar weight x
// activation pair): 2 loads per 16 FMAs -- the kernel is bound by shared-memory load issue, so sharing every
// weight fetch between two envs is what sets its speed.  The next layer's activations pass through a column of
// shared memory private to the thread (no block barrier).
// The random draw is JAX's: normal(key, (E * A,))[e] costs one threefry block per env and step.
// CTAs are sized so that the envs spread evenly over the SMs in a single wave (one CTA per SM).
#pragma once
#include "env_kernels.cuh"
#include "host_util.h"
#include "mathx.cuh"
#include "threefry.cuh"

namespace mbpo {

constexpr int ACT_W = 64;             // hidden width
constexpr int ACT_MAX_HIDDEN = 4;     // hidden layers
constexpr int ACT_MAX_THREADS = 256;  // 8 warps x 64 envs; 128 activation + ~100 other registers per thread

struct ActorArgs {
  MbpoPendulumParams sys;
  int E, T, episode_length, action_repeat;
  int num_hidden, deterministic, key_convention;  // 0: SAC get_experience, 1: generate_unroll, 2: use key as is
  float min_std;
  // policy head (MBPO_HEAD_*): NormalTanh of SAC/PPO, or the BPTT actor (bptt_optimizer.py:123-142,306-326)
  int head, shared_noise, normalize;
  int draw_offset, draw_total;   // env sharding of the draw normal(key, (draw_total, A))[draw_offset + e]
  int tiles_per_cta;             // tcgen05 kernel: live 128-env tiles per CTA (1..4), fewer when E is small
  int rows_per_cta;              // wide tcgen05 kernel: live rows of a CTA's 128-row tile (32, 64 or 128)
  float sig_bias, sig_min, sig_max, action_clip;
  float obs_mean[3], obs_std[3];
  const float* obs_mean_dev;    // device-resident statistics (override obs_mean / obs_std when non-null)
  const float* obs_std_dev;
  const float* w[ACT_MAX_HIDDEN + 1];  // [3,64], [64,64] x (num_hidden-1), [64,2]   (flax Dense kernels, [in, out])
  const float* b[ACT_MAX_HIDDEN + 1];
  const uint32_t* key_in;       // [2] device
  float* obs;            // [E,3] in/out
  float* steps;          // [E]   in/out
  float* done;           // [E]   in/out
  const float* first_obs;       // [E,3]
  float* action_out;            // [T,E]
  float* reward_out;            // [T,E]
  float* discount_out;          // [T,E]
  float* next_observation_out;  // [T,E,3]
  float* truncation_out;        // [T,E]
  uint32_t* key_out;            // [2] carry key after T steps
  float* raw_action_out;        // [T,E] or NULL: PPO's policy_extras['raw_action'] (pre-tanh sample)
  float* log_prob_out;          // [T,E] or NULL: PPO's policy_extras['log_prob']
};

// Host side of both actor entry points (mbpo_actor_rollout_extras, mbpo_actor_rollout_general): checks the policy
// against E envs of a System with X state and A action dims, and fills the fields ActorArgs and GeneralActorArgs
// share.  `what` prefixes the messages.
template <class Args>
int fill_policy(const char* what, const MbpoPolicyParams* p, int E, int X, int A, Args& a) {
  if (p->hidden != ACT_W || p->obs_dim != X || p->action_dim != A || p->num_hidden < 1 || p->num_hidden > ACT_MAX_HIDDEN)
    return fail(MBPO_EUNSUPPORTED,
                "%s: the policy kernel needs obs_dim == %d, action_dim == %d, 1..%d hidden layers of width %d "
                "(got obs %d, act %d, %d x %d)",
                what, X, A, ACT_MAX_HIDDEN, ACT_W, p->obs_dim, p->action_dim, p->num_hidden, p->hidden);
  for (int l = 0; l <= p->num_hidden; ++l)
    MBPO_REQUIRE(p->w[l] && p->b[l], "%s: null policy weights (layer %d)", what, l);
  MBPO_REQUIRE((p->obs_mean_dev == nullptr) == (p->obs_std_dev == nullptr),
               "%s: obs_mean_dev and obs_std_dev come together", what);
  MBPO_REQUIRE(p->draw_total == 0 || (p->draw_offset >= 0 && p->draw_offset + E <= p->draw_total),
               "%s: envs [%d, %d) are not inside draw_total %d", what, p->draw_offset, p->draw_offset + E,
               p->draw_total);
  a.num_hidden = p->num_hidden;
  a.min_std = p->min_std;
  a.normalize = p->normalize;
  a.draw_total = p->draw_total > 0 ? p->draw_total : E;
  a.draw_offset = p->draw_total > 0 ? p->draw_offset : 0;
  for (size_t i = 0; i < sizeof(a.obs_mean) / sizeof(a.obs_mean[0]); ++i) {
    a.obs_mean[i] = p->obs_mean[i];
    a.obs_std[i] = p->obs_std[i];
  }
  a.obs_mean_dev = p->obs_mean_dev; a.obs_std_dev = p->obs_std_dev;
  for (int l = 0; l <= ACT_MAX_HIDDEN; ++l) {
    a.w[l] = l <= a.num_hidden ? p->w[l] : nullptr;
    a.b[l] = l <= a.num_hidden ? p->b[l] : nullptr;
  }
  return MBPO_OK;
}

// jax.nn.swish(x) = x * sigmoid(x), sigmoid = 1 / (1 + exp(-x)).  ex2.approx (2^-22 relative) and rcp.approx
// (1 ulp) keep the activation within ~5e-7 relative of the float32 reference at 5 instructions; the accurate
// expf + IEEE division cost 20, i.e. a quarter of the whole kernel for the 192 hidden units.
__device__ __forceinline__ float swish_exact(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + __expf(-x)));
  return x * r;
}
// jax.nn.softplus(x) = logaddexp(x, 0) = max(x, 0) + log1p(exp(-|x|))
__device__ __forceinline__ float softplus_exact(float x) { return fmaxf(x, 0.0f) + log1pf(expf(-fabsf(x))); }

// acc += s * v  (s scalar, v and acc packed pairs, mathx.cuh).  A 3-register FFMA issues every other cycle per
// scheduler; FFMA2 takes the scalar and a register pair and retires two FMAs per issue slot.
__device__ __forceinline__ void fma2_scalar(f32x2_t& acc, float s, f32x2_t w) { acc = fma2(splat2(s), w, acc); }

struct ActorSmem {
  // float offsets into dynamic shared memory
  int w[ACT_MAX_HIDDEN + 1], b[ACT_MAX_HIDDEN + 1], h;
};

// Per-env state of the wrapper stack, two envs per thread.
struct ActorEnv {
  float c, s, w, th, f_c, f_s, f_w, f_th, steps, done;
};

// The policy's standard-normal draw for env `e`: normal(key, (E, A))[e], or the one draw normal(key, (A,)) every
// env shares (BPTT); 0 for a deterministic policy.  Independent of the network, so a kernel may take it early.
template <int PRNG>
__device__ __forceinline__ float actor_draw(const ActorArgs& a, Key2 k_actor, int e) {
  if (a.deterministic) return 0.0f;
  const uint32_t n_draw = a.shared_noise ? 1u : static_cast<uint32_t>(a.draw_total);
  const uint32_t i_draw = a.shared_noise ? 0u : static_cast<uint32_t>(a.draw_offset + e);
  return bits_to_normal(random_bits_at<PRNG>(k_actor, n_draw, i_draw));
}

// The policy head: turns the network's two outputs (loc, raw scale; biases already added) and the draw eps into
// the action of env `e` at step t, and emits PPO's policy_extras when asked.
__device__ __forceinline__ float actor_head(const ActorArgs& a, float eps, float mu, float raw_sc, int e, bool live,
                                            int t) {
  if (a.head == MBPO_HEAD_BPTT_ACTOR) {
    // Actor.__call__ :137-142: sig = clip(softplus(sig + inv_softplus(init_stddev)), sig_min, sig_max);
    // act :306-326: squash(mu) or squash(mu + normal(sample_key, mu.shape) * sig), squash = clip(tanh, +-0.999)
    float pre = mu;
    if (!a.deterministic) {
      const float sig = fminf(fmaxf(softplus_exact(__fadd_rn(raw_sc, a.sig_bias)), a.sig_min), a.sig_max);
      pre = __fadd_rn(pre, __fmul_rn(eps, sig));
    }
    return fminf(fmaxf(tanhf(pre), -a.action_clip), a.action_clip);
  }
  if (a.deterministic) return tanhf(mu);                               // mode(): tanh(loc)
  const float scale = softplus_exact(raw_sc) + a.min_std;
  const float raw = __fadd_rn(__fmul_rn(scale, eps), mu);              // distrax Normal.sample: scale * rnd + loc
  if (a.raw_action_out && live) {
    // ppo_network.py:72-80: raw_actions = sample_no_postprocessing; log_prob = Normal.log_prob(raw) -
    // Tanh.forward_log_det_jacobian(raw), summed over the action axis (parametric_distribution.py:76-83);
    // distrax: -0.5 * ((x - loc) / scale)^2 - (0.5 * log(2 pi) + log(scale)); 2 * (log 2 - x - softplus(-2 x))
    const float z = __fdiv_rn(__fsub_rn(raw, mu), scale);
    const float lp = __fsub_rn(__fmul_rn(-0.5f, __fmul_rn(z, z)), __fadd_rn(0.918938533f, logf(scale)));
    const float ldj = __fmul_rn(2.0f, __fsub_rn(__fsub_rn(0.693147181f, raw), softplus_exact(__fmul_rn(-2.0f, raw))));
    const size_t i = static_cast<size_t>(t) * a.E + e;
    a.raw_action_out[i] = raw;
    a.log_prob_out[i] = __fsub_rn(lp, ldj);
  }
  return tanhf(raw);
}

// The wrapped env step of env_kernels.cuh on one env's registers; returns the step's reward, sets trunc.
template <int MATH>
__device__ __forceinline__ float actor_env_step(const ActorArgs& a, const PendulumConsts& pc, ActorEnv& v, float u,
                                                float ep_len, float rep, float& trunc) {
  v.steps = (v.done != 0.0f) ? 0.0f : v.steps;
  v.done = 0.0f;
  float rew = 0.0f;
  for (int r = 0; r < a.action_repeat; ++r) {
    float rr;
    if (MATH == MBPO_MATH_REFERENCE) pendulum_step_ref(pc, v.c, v.s, v.w, u, rr);
    else pendulum_step_theta(pc, v.th, v.w, u, rr);
    rew = __fadd_rn(rew, rr);
  }
  if (MATH != MBPO_MATH_REFERENCE) sincos_bounded(v.th, v.s, v.c);
  v.steps = __fadd_rn(v.steps, rep);
  const bool over = v.steps >= ep_len;
  trunc = over ? (1.0f - v.done) : 0.0f;
  v.done = over ? 1.0f : v.done;
  if (over) { v.c = v.f_c; v.s = v.f_s; v.w = v.f_w; v.th = v.f_th; }
  return rew;
}

template <int PRNG, int MATH>
__global__ void __launch_bounds__(ACT_MAX_THREADS, 1) actor_rollout_pendulum_kernel(const __grid_constant__ ActorArgs a,
                                                                                    const ActorSmem lay) {
  extern __shared__ __align__(16) float act_sm[];
  __shared__ float tiles[ACT_MAX_THREADS / 32][96];
  __shared__ float norm_sm[8];     // normaliser mean [0..2], std [4..6]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = blockDim.x;
  if (tid < 3) {
    norm_sm[tid] = a.obs_mean_dev ? a.obs_mean_dev[tid] : a.obs_mean[tid];
    norm_sm[4 + tid] = a.obs_std_dev ? a.obs_std_dev[tid] : a.obs_std[tid];
  }
  // ---- policy parameters -> shared memory (once per launch) ----------------------------------------
  {
    const int L = a.num_hidden;
    for (int i = tid; i < 3 * ACT_W; i += nthr) act_sm[lay.w[0] + i] = a.w[0][i];
    for (int l = 1; l < L; ++l)
      for (int i = tid; i < ACT_W * ACT_W; i += nthr) act_sm[lay.w[l] + i] = a.w[l][i];
    for (int i = tid; i < ACT_W * 2; i += nthr) act_sm[lay.w[L] + i] = a.w[L][i];
    for (int l = 0; l < L; ++l)
      for (int i = tid; i < ACT_W; i += nthr) act_sm[lay.b[l] + i] = a.b[l][i];
    if (tid < 2) act_sm[lay.b[L] + tid] = a.b[L][tid];
  }
  __syncthreads();
  // A warp owns 64 consecutive envs: lane i carries env warp_e0 + i (slot 0) and warp_e0 + 32 + i (slot 1), so
  // every weight fetched from shared memory feeds both and every store stays a full 128-byte line.
  const int warp_e0 = (blockIdx.x * (nthr >> 5) + warp) * 64;
  if (warp_e0 >= a.E) return;
  const PendulumConsts pc(a.sys);
  float* tile = tiles[warp];
  f32x2_t* h_col = reinterpret_cast<f32x2_t*>(act_sm + lay.h) + tid;   // this thread's activation column (env pair)
  const float ep_len = static_cast<float>(a.episode_length);
  const float rep = static_cast<float>(a.action_repeat);
  const size_t E = static_cast<size_t>(a.E);

  ActorEnv env[2];
  int e_idx[2], ee[2], half_e0[2], n_valid[2];
  bool live[2], half_live[2];
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    half_e0[q] = warp_e0 + 32 * q;
    e_idx[q] = half_e0[q] + lane;
    live[q] = e_idx[q] < a.E;
    half_live[q] = half_e0[q] < a.E;
    ee[q] = live[q] ? e_idx[q] : a.E - 1;   // dead lanes shadow the last env, their stores are masked
    const int rem = a.E - half_e0[q];
    n_valid[q] = (rem < 32 ? (rem > 0 ? rem : 0) : 32) * 3;
    env[q].c = a.obs[3 * ee[q]]; env[q].s = a.obs[3 * ee[q] + 1]; env[q].w = a.obs[3 * ee[q] + 2];
    env[q].f_c = a.first_obs[3 * ee[q]]; env[q].f_s = a.first_obs[3 * ee[q] + 1]; env[q].f_w = a.first_obs[3 * ee[q] + 2];
    env[q].steps = a.steps[ee[q]]; env[q].done = a.done[ee[q]];
    env[q].th = (MATH == MBPO_MATH_REFERENCE) ? 0.0f : atan2_bounded(env[q].s, env[q].c);
    env[q].f_th = (MATH == MBPO_MATH_REFERENCE) ? 0.0f : atan2_bounded(env[q].f_s, env[q].f_c);
  }
  Key2 key{a.key_in[0], a.key_in[1]};

#pragma unroll 1
  for (int t = 0; t < a.T; ++t) {
    // ---- key plumbing ---------------------------------------------------------------------------------
    Key2 k_actor = key;
    if (a.key_convention != 2) {
      Key2 first, second;
      split2<PRNG>(key, first, second);
      if (a.key_convention == 0) { key = first; k_actor = second; }   // sac.py:290
      else { k_actor = first; key = second; }                          // acting.py:70
    }
    // ---- policy network, float32; every activation is a pair (env slot 0, env slot 1) -------------------
    f32x2_t h[ACT_W];
    float xin[2][3];   // the network input: obs, or (obs - mean) / std (bptt_optimizer.py:70-72,310)
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      xin[q][0] = env[q].c; xin[q][1] = env[q].s; xin[q][2] = env[q].w;
      if (a.normalize) {
#pragma unroll
        for (int i = 0; i < 3; ++i) xin[q][i] = __fdiv_rn(__fsub_rn(xin[q][i], norm_sm[i]), norm_sm[4 + i]);
      }
    }
    {
      const float4* w0 = reinterpret_cast<const float4*>(act_sm + lay.w[0]);   // [3][64]
      const float4* b0 = reinterpret_cast<const float4*>(act_sm + lay.b[0]);
#pragma unroll
      for (int j4 = 0; j4 < ACT_W / 4; ++j4) {
        const float4 r0 = w0[j4], r1 = w0[ACT_W / 4 + j4], r2 = w0[2 * (ACT_W / 4) + j4], bb = b0[j4];
        const float wr0[4] = {r0.x, r0.y, r0.z, r0.w}, wr1[4] = {r1.x, r1.y, r1.z, r1.w};
        const float wr2[4] = {r2.x, r2.y, r2.z, r2.w}, wb[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float v[2];
#pragma unroll
          for (int q = 0; q < 2; ++q)
            v[q] = swish_exact(fmaf(xin[q][2], wr2[i], fmaf(xin[q][1], wr1[i], xin[q][0] * wr0[i])) + wb[i]);
          h[4 * j4 + i] = pack2(v[0], v[1]);
        }
      }
    }
#pragma unroll 1
    for (int l = 1; l < a.num_hidden; ++l) {
      const float* wl = act_sm + lay.w[l];
      const float* bl = act_sm + lay.b[l];
#pragma unroll 1
      for (int jc = 0; jc < ACT_W / 8; ++jc) {
        f32x2_t acc2[8] = {0ull, 0ull, 0ull, 0ull, 0ull, 0ull, 0ull, 0ull};   // 8 output units x the env pair
        const float4* wrow = reinterpret_cast<const float4*>(wl + jc * 8);
#pragma unroll
        for (int k = 0; k < ACT_W; ++k) {
          const float4 wa = wrow[k * (ACT_W / 4)], wb = wrow[k * (ACT_W / 4) + 1];
          fma2_scalar(acc2[0], wa.x, h[k]); fma2_scalar(acc2[1], wa.y, h[k]);
          fma2_scalar(acc2[2], wa.z, h[k]); fma2_scalar(acc2[3], wa.w, h[k]);
          fma2_scalar(acc2[4], wb.x, h[k]); fma2_scalar(acc2[5], wb.y, h[k]);
          fma2_scalar(acc2[6], wb.z, h[k]); fma2_scalar(acc2[7], wb.w, h[k]);
        }
        const float4 ba = *reinterpret_cast<const float4*>(bl + jc * 8);
        const float4 bb = *reinterpret_cast<const float4*>(bl + jc * 8 + 4);
        const float bias[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float v0, v1;
          unpack2(acc2[i], v0, v1);
          h_col[(jc * 8 + i) * nthr] = pack2(swish_exact(v0 + bias[i]), swish_exact(v1 + bias[i]));
        }
      }
#pragma unroll
      for (int k = 0; k < ACT_W; ++k) h[k] = h_col[k * nthr];
    }
    float loc[2], raw_scale[2];
    {
      const float2* wo = reinterpret_cast<const float2*>(act_sm + lay.w[a.num_hidden]);   // [64][2]
      f32x2_t l2 = 0ull, s2 = 0ull;
#pragma unroll
      for (int k = 0; k < ACT_W; ++k) {
        const float2 v = wo[k];
        fma2_scalar(l2, v.x, h[k]);
        fma2_scalar(s2, v.y, h[k]);
      }
      unpack2(l2, loc[0], loc[1]);
      unpack2(s2, raw_scale[0], raw_scale[1]);
    }
    const float b_loc = act_sm[lay.b[a.num_hidden]], b_scale = act_sm[lay.b[a.num_hidden] + 1];
    const size_t row = static_cast<size_t>(t) * E;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      if (!half_live[q]) continue;   // warp-uniform
      ActorEnv& v = env[q];
      const float u = actor_head(a, actor_draw<PRNG>(a, k_actor, ee[q]), loc[q] + b_loc, raw_scale[q] + b_scale, ee[q],
                                 live[q], t);
      float trunc;
      const float rew = actor_env_step<MATH>(a, pc, v, u, ep_len, rep, trunc);
      warp_store3(tile, a.next_observation_out + (row + half_e0[q]) * 3 + lane, lane, n_valid[q], v.c, v.s, v.w);
      if (live[q]) {
        a.action_out[row + e_idx[q]] = u;
        a.reward_out[row + e_idx[q]] = rew;
        a.discount_out[row + e_idx[q]] = 1.0f - v.done;
        a.truncation_out[row + e_idx[q]] = trunc;
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    if (live[q]) {
      const int e = e_idx[q];
      a.obs[3 * e] = env[q].c; a.obs[3 * e + 1] = env[q].s; a.obs[3 * e + 2] = env[q].w;
      a.steps[e] = env[q].steps;
      a.done[e] = env[q].done;
    }
  }
  if (blockIdx.x == 0 && tid == 0 && a.key_out) { a.key_out[0] = key.k0; a.key_out[1] = key.k1; }
}

}  // namespace mbpo
