// Vmapped env rollouts for SAC/PPO data collection (BASELINE config 3).
//
// One thread per environment runs T wrapped env steps and streams brax Transition fields,
// time-major, to HBM.  Per env and step (reference):
//   AutoResetWrapper.step   brax_utils/training.py:119-137  steps = where(done,0,steps); done = 0;
//                                                           obs = where(done_after, first_obs, obs)
//   VmapWrapper.step        brax_utils/training.py:71-74    (this kernel's thread index)
//   EpisodeWrapper.step     brax_utils/training.py:91-107   action_repeat x system.step, reward sum,
//                                                           steps += repeat, done/truncation at episode_length
//   BraxWrapper.step        systems/brax_wrapper.py:40-50   system.step(obs, action, params)
//   actor_step              sac/acting.py:35-55             Transition(obs_prev, action, reward,
//                                                           1 - done, obs_after_reset, truncation)
// HBM traffic per transition (pendulum): 4 B action read + 24 B written (next_obs 12, reward 4,
// discount 4, truncation 4).  observation[t] is next_observation[t-1] (the post-reset state), so
// the host side passes observation_out = NULL and exposes both fields as overlapping views of
// one [T+1, E, 3] buffer; a separate observation buffer (+12 B) is written only when the caller
// asks for one.  The Transition's `action` field aliases the caller's input.
#pragma once
#include "pendulum.cuh"

namespace mbpo {

struct EnvArgs {
  MbpoPendulumParams sys;
  int E, T, episode_length, action_repeat;
  const float* obs_in;   // [E,3]
  const float* steps_in; // [E]
  const float* done_in;  // [E]
  float* obs;            // [E,3] out (may alias obs_in when segmented == 0)
  float* steps;          // [E]   out
  float* done;           // [E]   out
  const float* first_obs;  // [E,3]
  const float* actions;  // [T,E]
  float* observation_out;       // [T,E,3] or NULL
  float* reward_out;            // [T,E]   or NULL
  float* discount_out;          // [T,E]   or NULL
  float* next_observation_out;  // [T,E,3] or NULL
  float* truncation_out;        // [T,E]   or NULL
  int segmented;                // 1: blockIdx.y = episode segment (in/out state must not alias)
};

constexpr int ENV_CHUNK = 8;     // actions prefetched per thread (registers)
constexpr int ENV_THREADS = 64;   // 1,024 CTAs for 65,536 envs: 6.9 per SM, 1% imbalance (128 threads: 14%)

// Transposes a warp's 32 x 3 floats through shared memory so the [E,3] rows leave as three
// fully coalesced 128-byte stores.  dst already points at this lane's first element; m0/m1/m2 say
// whether the env owning element lane / lane+32 / lane+64 of the tile is written by this warp.
__device__ __forceinline__ void warp_store3(float* tile, float* dst, int lane, bool m0, bool m1, bool m2, float a,
                                            float b, float c) {
  tile[lane * 3] = a;
  tile[lane * 3 + 1] = b;
  tile[lane * 3 + 2] = c;
  __syncwarp();
  const float v0 = tile[lane], v1 = tile[lane + 32], v2 = tile[lane + 64];
  __syncwarp();
  if (m0) dst[0] = v0;
  if (m1) dst[32] = v1;
  if (m2) dst[64] = v2;
}
__device__ __forceinline__ void warp_store3(float* tile, float* dst, int lane, int n_valid, float a, float b, float c) {
  warp_store3(tile, dst, lane, lane < n_valid, lane + 32 < n_valid, lane + 64 < n_valid, a, b, c);
}

// Episode segments.  The pendulum System never terminates an episode itself (done = 0.0,
// pendulum_system.py:36), so the AutoReset points of an env are known from its step counter alone
// (training.py:98-107,120-124): the first after n0 = max(1, ceil((episode_length - steps) / repeat))
// steps, then every L = ceil(episode_length / repeat) steps, and each reset restarts the env from
// first_obs with steps = 0 (training.py:136).  The T-step rollout of one env is therefore 1 +
// ceil((T - 1) / L) independent pieces; thread (env, k) rolls piece k, which multiplies the number
// of independent dependency chains (65,536 envs alone are 3.5 warps per SM sub-partition).  The
// results are those of the sequential scan, bit for bit.  steps must be integer-valued (< 2^24),
// as brax's are.
//
// OBS: also write the separate observation buffer.  All of next_obs / reward / discount /
// truncation are non-NULL (otherwise the C ABI runs env_unroll_general_kernel, general_env_kernels.cuh).
//
// FAST (host-checked: action_repeat == 1, |target_angle| <= 6, E % 4 == 0, 16-byte aligned
// observation buffers, T*E*3 < 2^31): warps whose 32 envs are all live and share their piece
// boundaries take a loop without per-lane masks, with 32-bit offsets and one 16-byte store per
// lane for the [32,3] observation row; other warps (and FAST = false) take the general loop.
template <int MATH, bool OBS, bool FAST>
__global__ void __launch_bounds__(ENV_THREADS, 18) env_rollout_pendulum_kernel(const __grid_constant__ EnvArgs a) {
  __shared__ __align__(16) float tiles[ENV_THREADS / 32][96];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int e = blockIdx.x * ENV_THREADS + threadIdx.x;
  const int warp_e0 = e - lane;
  if (warp_e0 >= a.E) return;
  const bool live = e < a.E;
  const int ee = live ? e : a.E - 1;  // dead lanes shadow the last env, their stores are masked
  const PendulumConsts pc(a.sys);
  float* tile = tiles[warp];
  const int seg = a.segmented ? static_cast<int>(blockIdx.y) : 0;

  float steps = a.steps_in[ee], done = a.done_in[ee];
  // this thread's piece [t_beg, t_end) of the env's T steps
  int t_beg = 0, t_end = a.T;
  if (a.segmented) {
    const int s0 = (done != 0.0f) ? 0 : __float2int_rn(steps);
    const int rep_i = a.action_repeat;
    const int n0 = (a.episode_length > s0) ? max(1, (a.episode_length - s0 + rep_i - 1) / rep_i) : 1;
    const int len = max(1, (a.episode_length + rep_i - 1) / rep_i);
    t_beg = (seg == 0) ? 0 : min(a.T, n0 + (seg - 1) * len);
    t_end = min(a.T, n0 + seg * len);
  }
  const int w_beg = __reduce_min_sync(0xffffffffu, t_beg);
  const int w_end = __reduce_max_sync(0xffffffffu, t_end);
  if (w_beg >= w_end) return;

  const float f_c = a.first_obs[3 * ee], f_s = a.first_obs[3 * ee + 1], f_w = a.first_obs[3 * ee + 2];
  float c, s, w;
  if (seg == 0) {
    c = a.obs_in[3 * ee]; s = a.obs_in[3 * ee + 1]; w = a.obs_in[3 * ee + 2];
  } else {  // the step before this piece ended an episode: obs = first_obs, done = 1 (steps -> 0 below)
    c = f_c; s = f_s; w = f_w;
    done = 1.0f;
  }
  const float ep_len = static_cast<float>(a.episode_length);
  const float rep = static_cast<float>(a.action_repeat);
  const size_t E = static_cast<size_t>(a.E);
  // theta-carry: the angle lives in a register across steps; [cos, sin] are only outputs.  Reference math in the
  // uniform-warp loop carries it too -- theta = atan2(sin, cos) of the CURRENT state, re-derived after every step
  // from the fresh unit [cos, sin] (pendulum_step_ref_thcs: the guard-free atan2; same bits) -- so the guarded atan2
  // runs only here, on the caller's arbitrary states.
  float th = (MATH == MBPO_MATH_REFERENCE && !FAST) ? 0.0f : atan2_bounded(s, c);
  const float f_th = (MATH == MBPO_MATH_REFERENCE && !FAST) ? 0.0f : atan2_bounded(f_s, f_c);
  if (FAST) {
    const bool uniform = __all_sync(0xffffffffu, live && t_beg == w_beg && t_end == w_end);
    if (uniform) {
      const unsigned Eu = static_cast<unsigned>(a.E);
      unsigned off = static_cast<unsigned>(w_beg) * Eu + static_cast<unsigned>(e);            // [T,E] streams
      unsigned off3 = (static_cast<unsigned>(w_beg) * Eu + static_cast<unsigned>(warp_e0)) * 3u + 4u * lane;
      const bool row_lane = lane < 24;             // 24 lanes x 16 B = one [32,3] row
      float* tile3 = tile + 3 * lane;
      const float4* tile4 = reinterpret_cast<const float4*>(tile) + (row_lane ? lane : 0);
      float u_buf[ENV_CHUNK];
#pragma unroll
      for (int k = 0; k < ENV_CHUNK; ++k) u_buf[k] = (w_beg + k < w_end) ? __ldg(a.actions + off + k * Eu) : 0.0f;
      for (int t0 = w_beg; t0 < w_end; t0 += ENV_CHUNK) {
        float u_cur[ENV_CHUNK];
#pragma unroll
        for (int k = 0; k < ENV_CHUNK; ++k) u_cur[k] = u_buf[k];
#pragma unroll
        for (int k = 0; k < ENV_CHUNK; ++k)
          u_buf[k] = (t0 + ENV_CHUNK + k < w_end) ? __ldg(a.actions + off + (ENV_CHUNK + k) * Eu) : 0.0f;
        const int kmax = (w_end - t0) < ENV_CHUNK ? (w_end - t0) : ENV_CHUNK;
#pragma unroll
        for (int k = 0; k < ENV_CHUNK; ++k) {
          if (k < kmax) {
            steps = (done != 0.0f) ? 0.0f : steps;               // training.py:120-124
            if (OBS) {
              tile3[0] = c; tile3[1] = s; tile3[2] = w;
              __syncwarp();
              const float4 v = *tile4;
              __syncwarp();
              if (row_lane) *reinterpret_cast<float4*>(a.observation_out + off3) = v;
            }
            float rew;
            if (MATH == MBPO_MATH_REFERENCE) pendulum_step_ref_thcs<true>(pc, th, c, s, w, u_cur[k], rew);
            else { pendulum_step_theta<true>(pc, th, w, u_cur[k], rew); sincos_bounded(th, s, c); }
            rew = __fadd_rn(0.0f, rew);                          // the wrapper's reward sum starts at 0
            steps = __fadd_rn(steps, 1.0f);
            const bool over = steps >= ep_len;                   // training.py:98-107
            done = over ? 1.0f : 0.0f;
            if (over) { c = f_c; s = f_s; w = f_w; th = f_th; }  // training.py:136
            tile3[0] = c; tile3[1] = s; tile3[2] = w;
            __syncwarp();
            const float4 v = *tile4;
            __syncwarp();
            if (row_lane) *reinterpret_cast<float4*>(a.next_observation_out + off3) = v;
            a.reward_out[off] = rew;
            a.discount_out[off] = 1.0f - done;
            a.truncation_out[off] = done;                        // 1 - done_sys where the episode ends
            off += Eu;
            off3 += 3u * Eu;
          }
        }
      }
      if (t_end == a.T) {
        a.obs[3 * e] = c; a.obs[3 * e + 1] = s; a.obs[3 * e + 2] = w;
        a.steps[e] = steps;
        a.done[e] = done;
      }
      return;
    }
  }
  // tile element j of a row belongs to env warp_e0 + j / 3
  const int own0 = lane / 3, own1 = (lane + 32) / 3, own2 = (lane + 64) / 3;

  // running pointers, advanced by one time step per iteration
  const size_t row0 = static_cast<size_t>(w_beg) * E;
  const float* p_act = a.actions + row0 + ee;
  float* p_rew = a.reward_out + row0 + ee;
  float* p_dis = a.discount_out + row0 + ee;
  float* p_tru = a.truncation_out + row0 + ee;
  float* p_nxt = a.next_observation_out + (row0 + warp_e0) * 3 + lane;
  float* p_obs = OBS ? a.observation_out + (row0 + warp_e0) * 3 + lane : nullptr;

  float u_buf[ENV_CHUNK];
#pragma unroll
  for (int k = 0; k < ENV_CHUNK; ++k) u_buf[k] = (w_beg + k < w_end) ? __ldg(p_act + k * E) : 0.0f;
  p_act += ENV_CHUNK * E;

  for (int t0 = w_beg; t0 < w_end; t0 += ENV_CHUNK) {
    float u_cur[ENV_CHUNK];
#pragma unroll
    for (int k = 0; k < ENV_CHUNK; ++k) u_cur[k] = u_buf[k];
    // prefetch the next chunk while this one computes
#pragma unroll
    for (int k = 0; k < ENV_CHUNK; ++k) u_buf[k] = (t0 + ENV_CHUNK + k < w_end) ? __ldg(p_act + k * E) : 0.0f;
    p_act += ENV_CHUNK * E;
    const int kmax = (w_end - t0) < ENV_CHUNK ? (w_end - t0) : ENV_CHUNK;
#pragma unroll
    for (int k = 0; k < ENV_CHUNK; ++k) {
      if (k < kmax) {
        // envs of one warp share their piece boundaries unless their step counters differ
        const bool act = live && (t0 + k >= t_beg) && (t0 + k < t_end);
        const unsigned am = __ballot_sync(0xffffffffu, act);
        const bool m0 = (am >> own0) & 1u, m1 = (am >> own1) & 1u, m2 = (am >> own2) & 1u;
        // AutoReset pre-step (training.py:120-124)
        if (act) {
          steps = (done != 0.0f) ? 0.0f : steps;
          done = 0.0f;
        }
        if (OBS) {
          warp_store3(tile, p_obs, lane, m0, m1, m2, c, s, w);
          p_obs += 3 * E;
        }
        float rew = 0.0f, trunc = 0.0f;
        if (act) {
          // Episode: action_repeat x system.step with the same action (training.py:92-97)
          for (int r = 0; r < a.action_repeat; ++r) {
            float rr;
            if (MATH == MBPO_MATH_REFERENCE) pendulum_step_ref(pc, c, s, w, u_cur[k], rr);
            else pendulum_step_theta(pc, th, w, u_cur[k], rr);
            rew = __fadd_rn(rew, rr);
          }
          if (MATH != MBPO_MATH_REFERENCE) sincos_bounded(th, s, c);
          steps = __fadd_rn(steps, rep);
          const bool over = steps >= ep_len;                   // training.py:98-107
          trunc = over ? (1.0f - done) : 0.0f;                 // system done is always 0.0
          done = over ? 1.0f : done;
          if (over) { c = f_c; s = f_s; w = f_w; th = f_th; }  // training.py:136
        }
        warp_store3(tile, p_nxt, lane, m0, m1, m2, c, s, w);
        p_nxt += 3 * E;
        if (act) {
          *p_rew = rew;
          *p_dis = 1.0f - done;
          *p_tru = trunc;
        }
        p_rew += E; p_dis += E; p_tru += E;
      }
    }
  }
  if (live && t_beg < t_end && t_end == a.T) {  // the piece holding the last step owns the final state
    a.obs[3 * e] = c; a.obs[3 * e + 1] = s; a.obs[3 * e + 2] = w;
    a.steps[e] = steps;
    a.done[e] = done;
  }
}

}  // namespace mbpo
