// Env rollouts and the policy in the loop for the general Systems (systems.cuh: NoisyPendulumSys, PointMassSys).
//
// The wrapper stack is the one env_kernels.cuh restates for the pendulum (AutoReset / Episode / BraxWrapper /
// System.step, brax_utils/training.py:91-137, brax_wrapper.py:40-50); what is new here is what a general System adds:
//   key       every System.step does key, sub = split(key) (NoisyPendulum), so with action_repeat = r the env's
//             system_params.key advances r times per env step.  AutoReset resets obs to first_obs but NOT
//             system_params (training.py:119-137): the key keeps advancing across episode boundaries.  It lives in
//             registers for the T steps and the final key is written out.
//   A > 1     actions are [T,E,A]; the policy's draw is normal(key, (draw_total, A)) flattened: env e, dim a reads
//             element (draw_offset + e) * A + a (the legacy layout pads draw_total * A to even inside random_bits_at).
//   extras    PPO's log_prob sums over the A action dims; raw_action is [T,E,A].
// One thread per env, state and keys in registers.  The observation rows leave through the warp transposes of
// env_kernels.cuh (X = 3) or as one 16-byte store per env (X = 4).  env_unroll_general_kernel also serves the
// pendulum's env rollouts whose Transition buffers are not all present (collection.cu launch_env).
// rollout_policy_general_kernel is BPTT's forward on the same policy network: the plain scan of rollout_policy
// (no wrapper), with BPTT's actor head.
#pragma once
#include "actor_kernels.cuh"
#include "systems.cuh"

namespace mbpo {

constexpr int GEN_ENV_THREADS = 64;
constexpr int GEN_ACT_THREADS = 128;

struct GeneralEnvArgs {
  MbpoGeneralSystemParams sys;
  int E, T, episode_length, action_repeat;
  const float* obs_in;          // [E,X]
  const float* steps_in;        // [E]
  const float* done_in;         // [E]
  const uint32_t* keys_in;      // [E,2] (keyed Systems)
  float* obs_out;               // [E,X]
  float* steps_out;             // [E]
  float* done_out;              // [E]
  uint32_t* keys_out;           // [E,2] (keyed Systems)
  const float* first_obs;       // [E,X]
  const float* actions;         // [T,E,A]
  float* observation_out;       // [T,E,X] or NULL
  float* reward_out;            // [T,E]   or NULL
  float* discount_out;          // [T,E]   or NULL
  float* next_observation_out;  // [T,E,X] or NULL
  float* truncation_out;        // [T,E]   or NULL
};

// One wrapped env step on one env's registers: AutoReset pre-step (training.py:120-124), action_repeat x
// System.step with the same action and the reward summed from 0 (:92-97), the step counter and the episode end
// (:98-107; a general System's own done is 0), obs = first_obs where the episode ended (:136).  The env's first_obs
// row is read from memory at the reset: it is needed once per episode, and registers are scarce in the actor kernel.
template <class Sys, int PRNG>
__device__ __forceinline__ float general_wrapped_step(const Sys& sys, float (&x)[Sys::X], const float* first,
                                                      const float* u, Key2& key, float& steps, float& done,
                                                      int action_repeat, float ep_len, float rep, float& trunc) {
  steps = (done != 0.0f) ? 0.0f : steps;
  done = 0.0f;
  float rew = 0.0f;
  for (int r = 0; r < action_repeat; ++r) rew = __fadd_rn(rew, sys.template step<PRNG>(x, u, 1, key));
  steps = __fadd_rn(steps, rep);
  const bool over = steps >= ep_len;
  trunc = over ? (1.0f - done) : 0.0f;
  done = over ? 1.0f : done;
  if (over) {
#pragma unroll
    for (int k = 0; k < Sys::X; ++k) x[k] = __ldg(first + k);
  }
  return rew;
}

// Row t of an [T,E,X] field for the warp whose first env is warp_e0; every lane of the warp calls it.
template <int X>
__device__ __forceinline__ void store_obs_row(float* tile, float* field, size_t row_e0, int lane, bool live,
                                              int n_valid_envs, const float (&x)[X]) {
  if constexpr (X == 3) {
    warp_store3(tile, field + row_e0 * 3 + lane, lane, n_valid_envs * 3, x[0], x[1], x[2]);
  } else {
    static_assert(X == 4, "observation rows of 3 or 4 floats");
    if (live) *reinterpret_cast<float4*>(field + (row_e0 + lane) * 4) = make_float4(x[0], x[1], x[2], x[3]);
  }
}

// T wrapped env steps of E envs; the env state is read from *_in and the state after step T written to *_out.
// Actions are prefetched ENV_CHUNK steps ahead.  X = 4 needs 16-byte aligned observation buffers (host-checked).
template <class Sys, int PRNG>
__global__ void __launch_bounds__(GEN_ENV_THREADS) env_unroll_general_kernel(const __grid_constant__ GeneralEnvArgs a) {
  constexpr int X = Sys::X, A = Sys::A;
  __shared__ float tiles[GEN_ENV_THREADS / 32][96];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int e = blockIdx.x * GEN_ENV_THREADS + threadIdx.x;
  const int warp_e0 = e - lane;
  if (warp_e0 >= a.E) return;
  const bool live = e < a.E;
  const int ee = live ? e : a.E - 1;   // dead lanes shadow the last env, their stores are masked
  const int n_valid = min(a.E - warp_e0, 32);
  float* tile = tiles[warp];
  const Sys sys(a.sys);
  float x[X];
#pragma unroll
  for (int k = 0; k < X; ++k) x[k] = a.obs_in[static_cast<size_t>(ee) * X + k];
  const float* first = a.first_obs + static_cast<size_t>(ee) * X;
  float steps = a.steps_in[ee], done = a.done_in[ee];
  Key2 key{0u, 0u};
  if (Sys::KEYED) key = Key2{a.keys_in[2 * ee], a.keys_in[2 * ee + 1]};
  const float ep_len = static_cast<float>(a.episode_length);
  const float rep = static_cast<float>(a.action_repeat);
  const size_t E = static_cast<size_t>(a.E);

  float u_buf[ENV_CHUNK][A];
#pragma unroll
  for (int k = 0; k < ENV_CHUNK; ++k)
#pragma unroll
    for (int j = 0; j < A; ++j) u_buf[k][j] = (k < a.T) ? __ldg(a.actions + (k * E + ee) * A + j) : 0.0f;
  for (int t0 = 0; t0 < a.T; t0 += ENV_CHUNK) {
    float u_cur[ENV_CHUNK][A];
#pragma unroll
    for (int k = 0; k < ENV_CHUNK; ++k)
#pragma unroll
      for (int j = 0; j < A; ++j) {
        u_cur[k][j] = u_buf[k][j];
        const int tn = t0 + ENV_CHUNK + k;
        u_buf[k][j] = (tn < a.T) ? __ldg(a.actions + (static_cast<size_t>(tn) * E + ee) * A + j) : 0.0f;
      }
    const int kmax = min(a.T - t0, ENV_CHUNK);
#pragma unroll
    for (int k = 0; k < ENV_CHUNK; ++k) {
      if (k < kmax) {
        const size_t row = static_cast<size_t>(t0 + k) * E;
        if (a.observation_out) store_obs_row<X>(tile, a.observation_out, row + warp_e0, lane, live, n_valid, x);
        float trunc;
        const float rew = general_wrapped_step<Sys, PRNG>(sys, x, first, u_cur[k], key, steps, done, a.action_repeat,
                                                          ep_len, rep, trunc);
        if (a.next_observation_out)
          store_obs_row<X>(tile, a.next_observation_out, row + warp_e0, lane, live, n_valid, x);
        if (live) {
          if (a.reward_out) a.reward_out[row + e] = rew;
          if (a.discount_out) a.discount_out[row + e] = 1.0f - done;
          if (a.truncation_out) a.truncation_out[row + e] = trunc;
        }
      }
    }
  }
  if (live) {
#pragma unroll
    for (int k = 0; k < X; ++k) a.obs_out[static_cast<size_t>(e) * X + k] = x[k];
    a.steps_out[e] = steps;
    a.done_out[e] = done;
    if (Sys::KEYED) { a.keys_out[2 * e] = key.k0; a.keys_out[2 * e + 1] = key.k1; }
  }
}

struct GeneralActorArgs {
  MbpoGeneralSystemParams sys;
  int E, T, episode_length, action_repeat;
  int num_hidden, deterministic, key_convention;   // MBPO_KEYS_*
  float min_std;
  int normalize;
  int draw_offset, draw_total;   // env sharding of the draw normal(key, (draw_total, A))
  float obs_mean[4], obs_std[4];
  const float* obs_mean_dev;     // device-resident statistics (override obs_mean / obs_std when non-null)
  const float* obs_std_dev;
  const float* w[ACT_MAX_HIDDEN + 1];   // [X,64], [64,64] x (num_hidden-1), [64,2A]   (flax Dense kernels, [in, out])
  const float* b[ACT_MAX_HIDDEN + 1];
  const uint32_t* key_in;        // [2] the policy's carry key
  uint32_t* key_out;             // [2]
  float* obs;                    // [E,X] in/out
  float* steps;                  // [E]   in/out
  float* done;                   // [E]   in/out
  const uint32_t* sys_keys_in;   // [E,2] (keyed Systems)
  uint32_t* sys_keys_out;        // [E,2] (keyed Systems)
  const float* first_obs;        // [E,X]
  float* action_out;             // [T,E,A]
  float* reward_out;             // [T,E]
  float* discount_out;           // [T,E]
  float* next_observation_out;   // [T,E,X]
  float* truncation_out;         // [T,E]
  float* raw_action_out;         // [T,E,A] or NULL
  float* log_prob_out;           // [T,E]   or NULL
};

// Dynamic shared memory of the general actor kernel, in floats: the weights and biases at their flax shapes, then
// one 64-float activation column per thread ([64][threads]).
struct GeneralActorSmem {
  int w[ACT_MAX_HIDDEN + 1], b[ACT_MAX_HIDDEN + 1], h, total;
};

// The policy's weights and biases into shared memory at `lay`, the normaliser's statistics into norm_sm (mean
// [0..3], std [4..7]); every thread of the block takes part, and a barrier must follow.  Args is GeneralActorArgs or
// GeneralPolicyArgs.
template <int X, int A, class Args>
__device__ __forceinline__ void load_general_policy(const Args& a, const GeneralActorSmem& lay, float* gsm,
                                                    float* norm_sm, int tid, int nthr) {
  if (tid < X) {
    norm_sm[tid] = a.obs_mean_dev ? a.obs_mean_dev[tid] : a.obs_mean[tid];
    norm_sm[4 + tid] = a.obs_std_dev ? a.obs_std_dev[tid] : a.obs_std[tid];
  }
  const int L = a.num_hidden;
  for (int i = tid; i < X * ACT_W; i += nthr) gsm[lay.w[0] + i] = a.w[0][i];
  for (int l = 1; l < L; ++l)
    for (int i = tid; i < ACT_W * ACT_W; i += nthr) gsm[lay.w[l] + i] = a.w[l][i];
  for (int i = tid; i < ACT_W * 2 * A; i += nthr) gsm[lay.w[L] + i] = a.w[L][i];
  for (int l = 0; l < L; ++l)
    for (int i = tid; i < ACT_W; i += nthr) gsm[lay.b[l] + i] = a.b[l][i];
  if (tid < 2 * A) gsm[lay.b[L] + tid] = a.b[L][tid];
}

// The policy network on one thread's state x: the normaliser (x - mean) / std when a.normalize, then the MLP in
// float32 on the CUDA cores (swish), whose hidden layers pass through the thread's shared-memory column h_col, and
// the 2A logits (loc / mu first, then the raw scale) with their biases added.  gsm holds the weights at `lay`,
// norm_sm the normaliser's mean [0..3] and std [4..7].
template <int X, int A, class Args>
__device__ __forceinline__ void general_policy_logits(const Args& a, const float (&x)[X], const float* gsm,
                                                      const GeneralActorSmem& lay, const float* norm_sm,
                                                      float* h_col, int nthr, float (&logits)[2 * A]) {
  float xin[X];
#pragma unroll
  for (int i = 0; i < X; ++i)
    xin[i] = a.normalize ? __fdiv_rn(__fsub_rn(x[i], norm_sm[i]), norm_sm[4 + i]) : x[i];
  float h[ACT_W];
  {
    const float* w0 = gsm + lay.w[0];   // [X][64]
    const float* b0 = gsm + lay.b[0];
#pragma unroll
    for (int j = 0; j < ACT_W; ++j) {
      float acc = xin[0] * w0[j];
#pragma unroll
      for (int i = 1; i < X; ++i) acc = fmaf(xin[i], w0[i * ACT_W + j], acc);
      h[j] = swish_exact(acc + b0[j]);
    }
  }
#pragma unroll 1
  for (int l = 1; l < a.num_hidden; ++l) {
    const float* wl = gsm + lay.w[l];
    const float* bl = gsm + lay.b[l];
#pragma unroll 1
    for (int jc = 0; jc < ACT_W / 8; ++jc) {
      float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      const float4* wrow = reinterpret_cast<const float4*>(wl + jc * 8);
#pragma unroll
      for (int k = 0; k < ACT_W; ++k) {
        const float4 wa = wrow[k * (ACT_W / 4)], wb = wrow[k * (ACT_W / 4) + 1];
        acc[0] = fmaf(h[k], wa.x, acc[0]); acc[1] = fmaf(h[k], wa.y, acc[1]);
        acc[2] = fmaf(h[k], wa.z, acc[2]); acc[3] = fmaf(h[k], wa.w, acc[3]);
        acc[4] = fmaf(h[k], wb.x, acc[4]); acc[5] = fmaf(h[k], wb.y, acc[5]);
        acc[6] = fmaf(h[k], wb.z, acc[6]); acc[7] = fmaf(h[k], wb.w, acc[7]);
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) h_col[(jc * 8 + i) * nthr] = swish_exact(acc[i] + bl[jc * 8 + i]);
    }
#pragma unroll
    for (int k = 0; k < ACT_W; ++k) h[k] = h_col[k * nthr];
  }
  const float* wo = gsm + lay.w[a.num_hidden];   // [64][2A]
  const float* bo = gsm + lay.b[a.num_hidden];
#pragma unroll
  for (int j = 0; j < 2 * A; ++j) logits[j] = 0.0f;
#pragma unroll
  for (int k = 0; k < ACT_W; ++k)
#pragma unroll
    for (int j = 0; j < 2 * A; ++j) logits[j] = fmaf(h[k], wo[k * 2 * A + j], logits[j]);
#pragma unroll
  for (int j = 0; j < 2 * A; ++j) logits[j] += bo[j];
}

// T steps of actor_step for E envs: policy MLP (float32 on the CUDA cores), NormalTanh sample, the wrapped env step
// with the System's key, Transition out.  One thread per env; the activations of the current layer live in
// registers, the next layer's pass through the thread's own shared-memory column.
template <class Sys, int PRNG>
__global__ void __launch_bounds__(GEN_ACT_THREADS) actor_rollout_general_kernel(const __grid_constant__ GeneralActorArgs a,
                                                                               const GeneralActorSmem lay) {
  constexpr int X = Sys::X, A = Sys::A;
  extern __shared__ __align__(16) float gsm[];
  __shared__ float tiles[GEN_ACT_THREADS / 32][96];
  __shared__ float norm_sm[8];     // normaliser mean [0..3], std [4..7]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = blockDim.x;
  load_general_policy<X, A>(a, lay, gsm, norm_sm, tid, nthr);
  __syncthreads();
  const int e = blockIdx.x * nthr + tid;
  const int warp_e0 = e - lane;
  if (warp_e0 >= a.E) return;
  const bool live = e < a.E;
  const int ee = live ? e : a.E - 1;
  const int n_valid = min(a.E - warp_e0, 32);
  float* tile = tiles[warp];
  float* h_col = gsm + lay.h + tid;
  const Sys sys(a.sys);
  float x[X];
#pragma unroll
  for (int k = 0; k < X; ++k) x[k] = a.obs[static_cast<size_t>(ee) * X + k];
  const float* first = a.first_obs + static_cast<size_t>(ee) * X;
  float steps = a.steps[ee], done = a.done[ee];
  Key2 skey{0u, 0u};
  if (Sys::KEYED) skey = Key2{a.sys_keys_in[2 * ee], a.sys_keys_in[2 * ee + 1]};
  Key2 key{a.key_in[0], a.key_in[1]};
  const float ep_len = static_cast<float>(a.episode_length);
  const float rep = static_cast<float>(a.action_repeat);
  const size_t E = static_cast<size_t>(a.E);
  const uint32_t n_draw = static_cast<uint32_t>(a.draw_total) * A;

#pragma unroll 1
  for (int t = 0; t < a.T; ++t) {
    // ---- key plumbing (actor_kernels.cuh) -----------------------------------------------------------------
    Key2 k_actor = key;
    if (a.key_convention != MBPO_KEYS_AS_IS) {
      Key2 first_k, second_k;
      split2<PRNG>(key, first_k, second_k);
      if (a.key_convention == MBPO_KEYS_SAC) { key = first_k; k_actor = second_k; }
      else { k_actor = first_k; key = second_k; }
    }
    // ---- policy network --------------------------------------------------------------------------------------
    float logits[2 * A];
    general_policy_logits<X, A>(a, x, gsm, lay, norm_sm, h_col, nthr, logits);
    // ---- NormalTanh head (actor_kernels.cuh actor_head), A dims ----------------------------------------------
    const size_t row = static_cast<size_t>(t) * E;
    float u[A], log_prob = 0.0f;
#pragma unroll
    for (int j = 0; j < A; ++j) {
      const float mu = logits[j];
      if (a.deterministic) {               // mode(): tanh(loc)
        u[j] = tanhf(mu);
      } else {
      const uint32_t i_draw = static_cast<uint32_t>(a.draw_offset + ee) * A + j;
      const float eps = bits_to_normal(random_bits_at<PRNG>(k_actor, n_draw, i_draw));
      const float scale = softplus_exact(logits[A + j]) + a.min_std;
      const float raw = __fadd_rn(__fmul_rn(scale, eps), mu);
      u[j] = tanhf(raw);
      if (a.raw_action_out) {
        const float z = __fdiv_rn(__fsub_rn(raw, mu), scale);
        const float lp = __fsub_rn(__fmul_rn(-0.5f, __fmul_rn(z, z)), __fadd_rn(0.918938533f, logf(scale)));
        const float ldj = __fmul_rn(2.0f, __fsub_rn(__fsub_rn(0.693147181f, raw), softplus_exact(__fmul_rn(-2.0f, raw))));
        const float v = __fsub_rn(lp, ldj);
        log_prob = (j == 0) ? v : __fadd_rn(log_prob, v);   // summed over the action axis, left to right
        if (live) a.raw_action_out[(row + e) * A + j] = raw;
      }
      }
    }
    if (a.raw_action_out && live) a.log_prob_out[row + e] = log_prob;
    // ---- the wrapped env step with the System's key ----------------------------------------------------------
    float trunc;
    const float rew = general_wrapped_step<Sys, PRNG>(sys, x, first, u, skey, steps, done, a.action_repeat, ep_len,
                                                      rep, trunc);
    store_obs_row<X>(tile, a.next_observation_out, row + warp_e0, lane, live, n_valid, x);
    if (live) {
#pragma unroll
      for (int j = 0; j < A; ++j) a.action_out[(row + e) * A + j] = u[j];
      a.reward_out[row + e] = rew;
      a.discount_out[row + e] = 1.0f - done;
      a.truncation_out[row + e] = trunc;
    }
  }
  if (live) {
#pragma unroll
    for (int k = 0; k < X; ++k) a.obs[static_cast<size_t>(e) * X + k] = x[k];
    a.steps[e] = steps;
    a.done[e] = done;
    if (Sys::KEYED) { a.sys_keys_out[2 * e] = skey.k0; a.sys_keys_out[2 * e + 1] = skey.k1; }
  }
  if (blockIdx.x == 0 && tid == 0 && a.key_out) { a.key_out[0] = key.k0; a.key_out[1] = key.k1; }
}

struct GeneralPolicyArgs {
  MbpoGeneralSystemParams sys;
  int E, T;
  int num_hidden, deterministic, key_convention;   // MBPO_KEYS_*
  float min_std;
  int head, shared_noise, normalize;               // MBPO_HEAD_*
  int draw_offset, draw_total;   // env sharding of the NormalTanh draw normal(key, (draw_total, A))
  float sig_bias, sig_min, sig_max, action_clip;   // the BPTT head
  float obs_mean[4], obs_std[4];
  const float* obs_mean_dev;     // device-resident statistics (override obs_mean / obs_std when non-null)
  const float* obs_std_dev;
  const float* w[ACT_MAX_HIDDEN + 1];   // as GeneralActorArgs
  const float* b[ACT_MAX_HIDDEN + 1];
  const uint32_t* key_in;        // [2] the policy's carry key
  uint32_t* key_out;             // [2]
  const float* x0;               // [E,X]
  const uint32_t* sys_keys_in;   // keyed Systems: [2] (sys_keys_shared) or [E,2]
  uint32_t* sys_keys_out;        // same shape
  int sys_keys_shared;
  float* action_out;             // [T,E,A]
  float* reward_out;             // [T,E]
  float* next_observation_out;   // [T,E,X]
};

// rollout_policy (optimizer_utils.py:62-116) for E trajectories of T steps: per step the policy network (as
// actor_rollout_general_kernel), its head, then the plain System.step -- no Episode / AutoReset wrapper, so no step
// counter, done or truncation.  The head is BPTT's actor (bptt_optimizer.py:137-142,306-326: sig = clip(softplus(sig
// + sig_bias), sig_min, sig_max), a = clip(tanh(mu + eps * sig), +-action_clip), clip(tanh(mu)) when deterministic)
// or SAC's NormalTanh; with shared_noise the draw is normal(k_actor, (A,)), the same for every trajectory.  A keyed
// System's key is per trajectory or one shared by all; a shared key advances identically in every thread.
template <class Sys, int PRNG>
__global__ void __launch_bounds__(GEN_ACT_THREADS) rollout_policy_general_kernel(const __grid_constant__ GeneralPolicyArgs a,
                                                                                const GeneralActorSmem lay) {
  constexpr int X = Sys::X, A = Sys::A;
  extern __shared__ __align__(16) float gsm[];
  __shared__ float tiles[GEN_ACT_THREADS / 32][96];
  __shared__ float norm_sm[8];     // normaliser mean [0..3], std [4..7]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = blockDim.x;
  load_general_policy<X, A>(a, lay, gsm, norm_sm, tid, nthr);
  __syncthreads();
  const int e = blockIdx.x * nthr + tid;
  const int warp_e0 = e - lane;
  if (warp_e0 >= a.E) return;
  const bool live = e < a.E;
  const int ee = live ? e : a.E - 1;
  const int n_valid = min(a.E - warp_e0, 32);
  float* tile = tiles[warp];
  float* h_col = gsm + lay.h + tid;
  const Sys sys(a.sys);
  float x[X];
#pragma unroll
  for (int k = 0; k < X; ++k) x[k] = a.x0[static_cast<size_t>(ee) * X + k];
  Key2 skey{0u, 0u};
  if (Sys::KEYED) {
    const int ks = a.sys_keys_shared ? 0 : ee;
    skey = Key2{a.sys_keys_in[2 * ks], a.sys_keys_in[2 * ks + 1]};
  }
  Key2 key{a.key_in[0], a.key_in[1]};
  const size_t E = static_cast<size_t>(a.E);
  const bool bptt = a.head == MBPO_HEAD_BPTT_ACTOR;
  const uint32_t n_draw = a.shared_noise ? static_cast<uint32_t>(A) : static_cast<uint32_t>(a.draw_total) * A;
  const uint32_t i_draw0 = a.shared_noise ? 0u : static_cast<uint32_t>(a.draw_offset + ee) * A;

#pragma unroll 1
  for (int t = 0; t < a.T; ++t) {
    // ---- key plumbing (actor_kernels.cuh): BPTT.act splits as MBPO_KEYS_UNROLL, evaluate keeps it as is ----------
    Key2 k_actor = key;
    if (a.key_convention != MBPO_KEYS_AS_IS) {
      Key2 first_k, second_k;
      split2<PRNG>(key, first_k, second_k);
      if (a.key_convention == MBPO_KEYS_SAC) { key = first_k; k_actor = second_k; }
      else { k_actor = first_k; key = second_k; }
    }
    float logits[2 * A];
    general_policy_logits<X, A>(a, x, gsm, lay, norm_sm, h_col, nthr, logits);
    // ---- the head, A dims ----------------------------------------------------------------------------------------
    float u[A];
#pragma unroll
    for (int j = 0; j < A; ++j) {
      const float mu = logits[j];
      const float eps = a.deterministic ? 0.0f : bits_to_normal(random_bits_at<PRNG>(k_actor, n_draw, i_draw0 + j));
      if (bptt) {
        float pre = mu;
        if (!a.deterministic) {
          const float sig = fminf(fmaxf(softplus_exact(__fadd_rn(logits[A + j], a.sig_bias)), a.sig_min), a.sig_max);
          pre = __fadd_rn(pre, __fmul_rn(eps, sig));
        }
        u[j] = fminf(fmaxf(tanhf(pre), -a.action_clip), a.action_clip);
      } else if (a.deterministic) {
        u[j] = tanhf(mu);
      } else {
        const float scale = softplus_exact(logits[A + j]) + a.min_std;
        u[j] = tanhf(__fadd_rn(__fmul_rn(scale, eps), mu));
      }
    }
    // ---- System.step ------------------------------------------------------------------------------------------
    const size_t row = static_cast<size_t>(t) * E;
    const float rew = sys.template step<PRNG>(x, u, 1, skey);
    store_obs_row<X>(tile, a.next_observation_out, row + warp_e0, lane, live, n_valid, x);
    if (live) {
#pragma unroll
      for (int j = 0; j < A; ++j) a.action_out[(row + e) * A + j] = u[j];
      a.reward_out[row + e] = rew;
    }
  }
  if (Sys::KEYED && (a.sys_keys_shared ? e == 0 : live)) {
    a.sys_keys_out[2 * e] = skey.k0;
    a.sys_keys_out[2 * e + 1] = skey.k1;
  }
  if (blockIdx.x == 0 && tid == 0 && a.key_out) { a.key_out[0] = key.k0; a.key_out[1] = key.k1; }
}

}  // namespace mbpo
