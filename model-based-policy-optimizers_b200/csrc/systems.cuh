// Systems behind the general (any action_dim, key-consuming) rollout kernels.
//
// The reference's System interface (mbpo/systems/base_systems.py:28-60) is step(x, u, system_params) ->
// SystemState(x_next, reward, system_params, done); system_params carries a PRNG key that iCemTO sets per particle
// (icem_optimizer.py:146-147,155-156) and rollout_actions threads through its scan (optimizer_utils.py:28-46).
// The reference ships one System, the deterministic pendulum, which drops that key (pendulum_system.py:38); the
// two below are the smallest Systems that exercise the rest of iCemTO's own code -- a transition that is SAMPLED
// with the System's key, and an action space with more than one dimension (icem_optimizer.py:180):
//
//   NoisyPendulum   PendulumDynamics.next_state already returns distrax.Normal(mean, std) (pendulum_dynamics.py:45-46);
//                   here std = noise_std and step draws:  key, sub = split(system_params.key);
//                   x_next = mean + noise_std * normal(sub, (3,));  the returned SystemParams carries `key`.
//   PointMass       planar double integrator, state [px, py, vx, vy], action [ax, ay]:
//                   a = clip(u, +-1) * max_accel; v' = clip(v + a dt, +-max_speed); p' = p + v' dt;
//                   reward = -(|p - target|^2 + speed_cost |v|^2) - control_cost |u|^2 on the current state.
//
// Every float operation is rounded once, in the order the oracle (oracle/mbpo_oracle.py NoisyPendulumOracle,
// PointMassOracle) writes it.
#pragma once
#include "../../include/mbpo_b200.h"
#include "pendulum.cuh"
#include "threefry.cuh"

namespace mbpo {

struct PendulumSys {
  static constexpr int KIND = MBPO_SYSTEM_PENDULUM, X = 3, A = 1;
  static constexpr bool KEYED = false;
  PendulumConsts pc;
  __device__ explicit PendulumSys(const MbpoGeneralSystemParams& p) : pc(p.pendulum) {}
  template <int PRNG>
  __device__ __forceinline__ float step(float (&x)[X], const float* u, int ustride, Key2&) const {
    float r;
    pendulum_step_ref(pc, x[0], x[1], x[2], u[0], r);
    return r;
  }
};

// The pendulum under MBPO_MATH_THETA_CARRY where theta is not carried between steps: each step re-derives it from
// [cos, sin], steps it with pendulum_step_theta and writes [cos, sin] back (system_step_pendulum_kernel<1>).
struct PendulumThetaSys : PendulumSys {
  using PendulumSys::PendulumSys;
  template <int PRNG>
  __device__ __forceinline__ float step(float (&x)[X], const float* u, int ustride, Key2&) const {
    float th = atan2_bounded(x[1], x[0]), r;
    pendulum_step_theta(pc, th, x[2], u[0], r);
    sincos_bounded(th, x[1], x[0]);
    return r;
  }
};

struct NoisyPendulumSys {
  static constexpr int KIND = MBPO_SYSTEM_NOISY_PENDULUM, X = 3, A = 1;
  static constexpr bool KEYED = true;
  PendulumConsts pc;
  float noise_std;
  __device__ explicit NoisyPendulumSys(const MbpoGeneralSystemParams& p) : pc(p.pendulum), noise_std(p.noise_std) {}
  template <int PRNG>
  __device__ __forceinline__ float step(float (&x)[X], const float* u, int ustride, Key2& key) const {
    float r;
    pendulum_step_ref(pc, x[0], x[1], x[2], u[0], r);            // the mean of next_state; reward on the current state
    Key2 next, sub;
    split2<PRNG>(key, next, sub);                                // key, sub = split(system_params.key)
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const float z = bits_to_normal(random_bits_at<PRNG>(sub, 3u, static_cast<uint32_t>(i)));
      x[i] = __fadd_rn(x[i], __fmul_rn(noise_std, z));           // loc + scale * normal
    }
    key = next;
    return r;
  }
  // Cotangents of step: g_next of x_next, g_r of the reward -> g_x, g_u.  The noise is added to the mean and
  // depends on neither x nor u, so the Jacobians are the pendulum's at the stored (noisy) state.
  __device__ __forceinline__ void step_vjp(const float (&x)[X], const float (&u)[A], const float (&g_next)[X],
                                           float g_r, float (&g_x)[X], float (&g_u)[A]) const {
    pendulum_step_vjp(pc, x[0], x[1], x[2], u[0], g_next[0], g_next[1], g_next[2], g_r, g_x[0], g_x[1], g_x[2],
                      g_u[0]);
  }
};

struct PointMassSys {
  static constexpr int KIND = MBPO_SYSTEM_POINT_MASS, X = 4, A = 2;
  static constexpr bool KEYED = false;
  MbpoPointMassParams p;
  __device__ explicit PointMassSys(const MbpoGeneralSystemParams& g) : p(g.point_mass) {}
  template <int PRNG>
  __device__ __forceinline__ float step(float (&x)[X], const float* u, int ustride, Key2&) const {
    const float u0 = u[0], u1 = u[ustride];
    const float dx = __fsub_rn(x[0], p.target_x), dy = __fsub_rn(x[1], p.target_y);
    const float dist2 = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
    const float spd2 = __fadd_rn(__fmul_rn(x[2], x[2]), __fmul_rn(x[3], x[3]));
    const float uu = __fadd_rn(__fmul_rn(u0, u0), __fmul_rn(u1, u1));
    const float reward = __fsub_rn(-__fadd_rn(dist2, __fmul_rn(p.speed_cost, spd2)), __fmul_rn(p.control_cost, uu));
    const float a0 = __fmul_rn(fminf(fmaxf(u0, -1.0f), 1.0f), p.max_accel);
    const float a1 = __fmul_rn(fminf(fmaxf(u1, -1.0f), 1.0f), p.max_accel);
    const float v0 = fminf(fmaxf(__fadd_rn(x[2], __fmul_rn(a0, p.dt)), -p.max_speed), p.max_speed);
    const float v1 = fminf(fmaxf(__fadd_rn(x[3], __fmul_rn(a1, p.dt)), -p.max_speed), p.max_speed);
    x[0] = __fadd_rn(x[0], __fmul_rn(v0, p.dt));
    x[1] = __fadd_rn(x[1], __fmul_rn(v1, p.dt));
    x[2] = v0;
    x[3] = v1;
    return reward;
  }
  // Cotangents of step, per axis k with pre = v + a dt: g_v' = g_next_v + dt g_next_p; g_pre = g_v' clip'(pre);
  // g_v = g_pre - g_r 2 speed_cost v; g_p = g_next_p - g_r 2 (p - target);
  // g_u = g_pre dt max_accel clip'(u) - g_r 2 control_cost u.
  __device__ __forceinline__ void step_vjp(const float (&x)[X], const float (&u)[A], const float (&g_next)[X],
                                           float g_r, float (&g_x)[X], float (&g_u)[A]) const {
    const float target[2] = {p.target_x, p.target_y};
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const float ak = __fmul_rn(fminf(fmaxf(u[k], -1.0f), 1.0f), p.max_accel);
      const float pre = __fadd_rn(x[2 + k], __fmul_rn(ak, p.dt));                // as step rounds it: same clip ties
      const float g_pre = (g_next[2 + k] + p.dt * g_next[k]) * clip_grad(pre, -p.max_speed, p.max_speed);
      g_x[k] = g_next[k] - g_r * 2.0f * (x[k] - target[k]);
      g_x[2 + k] = g_pre - g_r * 2.0f * p.speed_cost * x[2 + k];
      g_u[k] = g_pre * p.dt * p.max_accel * clip_grad(u[k], -1.0f, 1.0f) - g_r * 2.0f * p.control_cost * u[k];
    }
  }
};

template <class T>
struct TypeTag { using type = T; };

// Runtime system_kind -> System struct: f(TypeTag<Sys>{}) for the one of the listed Systems whose KIND is `kind`,
// MBPO_EUNSUPPORTED (no message) when none is.  Each call site lists the Systems it serves, so only their kernels
// are instantiated.
template <class... Sys, class F>
int with_system(int kind, F&& f) {
  int rc = MBPO_EUNSUPPORTED;
  (void)((kind == Sys::KIND && (rc = f(TypeTag<Sys>{}), true)) || ...);
  return rc;
}

// X, A and KEYED of a general System; MBPO_EUNSUPPORTED (no message) for any other kind.
inline int general_system_dims(int kind, int* X, int* A, bool* keyed) {
  return with_system<PendulumSys, NoisyPendulumSys, PointMassSys>(kind, [&](auto t) {
    using Sys = typename decltype(t)::type;
    *X = Sys::X; *A = Sys::A; *keyed = Sys::KEYED;
    return MBPO_OK;
  });
}

// vmap(System.step): one thread per row.
template <class Sys, int PRNG>
__global__ void system_step_general_kernel(const MbpoGeneralSystemParams gp, const float* __restrict__ x,
                                           const float* __restrict__ u, const uint32_t* __restrict__ keys_in, int R,
                                           float* __restrict__ x_next, float* __restrict__ reward,
                                           uint32_t* __restrict__ keys_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R) return;
  const Sys sys(gp);
  float s[Sys::X];
#pragma unroll
  for (int k = 0; k < Sys::X; ++k) s[k] = x[static_cast<size_t>(i) * Sys::X + k];
  Key2 key{0u, 0u};
  if (Sys::KEYED) key = Key2{keys_in[2 * i], keys_in[2 * i + 1]};
  const float r = sys.template step<PRNG>(s, u + static_cast<size_t>(i) * Sys::A, 1, key);
#pragma unroll
  for (int k = 0; k < Sys::X; ++k) x_next[static_cast<size_t>(i) * Sys::X + k] = s[k];
  reward[i] = r;
  if (Sys::KEYED && keys_out) { keys_out[2 * i] = key.k0; keys_out[2 * i + 1] = key.k1; }
}

// One rollout of row `acts` ([H, A] row-major) from state s0 with `key`; returns the horizon-mean reward
// (icem_optimizer.py:160 inner mean) and optionally writes the Transition fields of the row.
template <class Sys, int PRNG>
__device__ __forceinline__ float general_rollout(const Sys& sys, const float (&s0)[Sys::X], const float* acts, int H,
                                                 Key2 key, float* obs_out, float* reward_out, float* next_obs_out,
                                                 Key2* key_final) {
  float s[Sys::X];
#pragma unroll
  for (int k = 0; k < Sys::X; ++k) s[k] = s0[k];
  float acc = 0.0f;
  for (int t = 0; t < H; ++t) {
    if (obs_out) {
#pragma unroll
      for (int k = 0; k < Sys::X; ++k) obs_out[t * Sys::X + k] = s[k];
    }
    const float r = sys.template step<PRNG>(s, acts + static_cast<size_t>(t) * Sys::A, 1, key);
    if (reward_out) reward_out[t] = r;
    if (next_obs_out) {
#pragma unroll
      for (int k = 0; k < Sys::X; ++k) next_obs_out[t * Sys::X + k] = s[k];
    }
    acc = __fadd_rn(acc, r);
  }
  if (key_final) *key_final = key;
  return __fdiv_rn(acc, static_cast<float>(H));
}

// vmap(vmap(objective)) (icem_optimizer.py:144-160,195): one thread per candidate row.  P == 0: a single rollout
// per row with the row's key as it is (vmap(rollout_actions), Transition buffers optional).  P >= 1: the row's key
// is split into P particle keys (:155), one rollout per particle, summarised by the left-to-right mean or the max
// (:112-115,160); a deterministic System rolls out once and summarises P identical values.
template <class Sys, int PRNG>
__global__ void __launch_bounds__(128)
    general_objective_kernel(const MbpoGeneralSystemParams gp, int H, const float* __restrict__ x0,
                             const float* __restrict__ actions, const uint32_t* __restrict__ keys, int B, int M, int P,
                             int summarize, float* __restrict__ values_out, float* __restrict__ obs_out,
                             float* __restrict__ reward_out, float* __restrict__ next_obs_out) {
  const long long r = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (r >= static_cast<long long>(B) * M) return;
  const int b = static_cast<int>(r / M);
  const Sys sys(gp);
  float s0[Sys::X];
#pragma unroll
  for (int k = 0; k < Sys::X; ++k) s0[k] = x0[static_cast<size_t>(b) * Sys::X + k];
  const float* acts = actions + static_cast<size_t>(r) * H * Sys::A;
  Key2 key{0u, 0u};
  if (Sys::KEYED) key = Key2{keys[2 * r], keys[2 * r + 1]};
  if (P == 0) {
    const size_t o = static_cast<size_t>(r) * H;
    const float ret = general_rollout<Sys, PRNG>(sys, s0, acts, H, key, obs_out ? obs_out + o * Sys::X : nullptr,
                                                 reward_out ? reward_out + o : nullptr,
                                                 next_obs_out ? next_obs_out + o * Sys::X : nullptr, nullptr);
    if (values_out) values_out[r] = ret;
    return;
  }
  float out;
  if (!Sys::KEYED) {
    const float ret = general_rollout<Sys, PRNG>(sys, s0, acts, H, key, nullptr, nullptr, nullptr, nullptr);
    if (summarize == MBPO_SUMMARIZE_MAX || P == 1) {
      out = ret;
    } else {
      float acc = 0.0f;
      for (int p = 0; p < P; ++p) acc = __fadd_rn(acc, ret);
      out = __fdiv_rn(acc, static_cast<float>(P));
    }
  } else {
    float acc = 0.0f, mx = 0.0f;
    for (int p = 0; p < P; ++p) {
      const Key2 pk = split_at<PRNG>(key, static_cast<uint32_t>(P), static_cast<uint32_t>(p));   // :155
      const float ret = general_rollout<Sys, PRNG>(sys, s0, acts, H, pk, nullptr, nullptr, nullptr, nullptr);
      acc = __fadd_rn(acc, ret);
      mx = (p == 0) ? ret : fmaxf(mx, ret);
    }
    out = (summarize == MBPO_SUMMARIZE_MAX) ? mx : __fdiv_rn(acc, static_cast<float>(P));
  }
  values_out[r] = out;
}

// general_objective_kernel's P >= 1 path with the Transition buffers of every particle: particle p of row r writes
// obs / next_obs [r, p, H, X] and reward [r, p, H] from the rollout with key split(key, P)[p] (:155); an unkeyed System
// runs its one rollout P times, so the P copies and the summary are those of P identical particles.  values_out
// (optional) gets the summary general_objective_kernel computes.  A kernel of its own, so that the summary-only
// kernel stays as it is.
template <class Sys, int PRNG>
__global__ void __launch_bounds__(128)
    general_particles_kernel(const MbpoGeneralSystemParams gp, int H, const float* __restrict__ x0,
                             const float* __restrict__ actions, const uint32_t* __restrict__ keys, int B, int M, int P,
                             int summarize, float* __restrict__ values_out, float* __restrict__ obs_out,
                             float* __restrict__ reward_out, float* __restrict__ next_obs_out) {
  const long long r = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (r >= static_cast<long long>(B) * M) return;
  const int b = static_cast<int>(r / M);
  const Sys sys(gp);
  float s0[Sys::X];
#pragma unroll
  for (int k = 0; k < Sys::X; ++k) s0[k] = x0[static_cast<size_t>(b) * Sys::X + k];
  const float* acts = actions + static_cast<size_t>(r) * H * Sys::A;
  Key2 key{0u, 0u};
  if (Sys::KEYED) key = Key2{keys[2 * r], keys[2 * r + 1]};
  float acc = 0.0f, mx = 0.0f;
  for (int p = 0; p < P; ++p) {
    const Key2 pk = Sys::KEYED ? split_at<PRNG>(key, static_cast<uint32_t>(P), static_cast<uint32_t>(p)) : key;
    const size_t o = (static_cast<size_t>(r) * P + p) * H;
    const float ret = general_rollout<Sys, PRNG>(sys, s0, acts, H, pk, obs_out ? obs_out + o * Sys::X : nullptr,
                                                 reward_out ? reward_out + o : nullptr,
                                                 next_obs_out ? next_obs_out + o * Sys::X : nullptr, nullptr);
    acc = __fadd_rn(acc, ret);
    mx = (p == 0) ? ret : fmaxf(mx, ret);
  }
  if (values_out) values_out[r] = (summarize == MBPO_SUMMARIZE_MAX) ? mx : __fdiv_rn(acc, static_cast<float>(P));
}

}  // namespace mbpo
