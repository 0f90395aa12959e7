// Reverse-mode pass through System.step rollouts, and the lambda-return scan (SURVEY 8f-4).
//
// BPTT differentiates rollout_policy (mbpo/utils/optimizer_utils.py:62-116) with
// jax.value_and_grad (bptt_optimizer.py:361-376).  With stop_grads=True (:337, the only way the
// reference calls it) the policy sees stop_gradient(obs), so the cotangent reaches the policy
// parameters only through the actions:
//     x_{t+1} = f(x_t, a_t)        r_t = r(x_t, a_t)        a_t = pi_theta(sg(x_t))
//     lam_T   = 0
//     lam_t   = (df/dx)^T (g_next_obs[t] + lam_{t+1}) + g_reward[t] dr/dx          (state adjoint)
//     ga_t    = g_action[t] + (df/da)^T (g_next_obs[t] + lam_{t+1}) + g_reward[t] dr/da
// rollout_adjoint_pendulum_kernel runs that reverse scan for one trajectory per thread (the 3 x 3
// Jacobian-transpose products written out for pendulum_dynamics.py:29-63 and pendulum_reward.py:27-42,
// pendulum.cuh pendulum_step_vjp), re-deriving the step's intermediates from the stored (observation, action)
// instead of saving them; rollout_adjoint_general_kernel does the same for the general Systems through their
// step_vjp (systems.cuh).
// The parameter gradient sum_t (da_t/dtheta)^T ga_t has no sequential dependency left and is one
// batched network backward over all T*E (obs, ga) rows -- the caller's autodiff.
//
// lambda_return_kernel: optimizer_utils.py:119-131 (Dreamer's lambda return): inputs_t = reward_t +
// discount * next_values_t * (1 - lambda); returns_t = inputs_t + discount * lambda * returns_{t+1},
// returns_T = next_values[-1] -- and its transpose (a forward scan), since BPTT differentiates it too.
//
// All arrays are addressed as base[t * stride_t + e * stride_e] (elements), so both the vmapped
// reference layout [B, H, ...] and the time-major [T, E, ...] layout of the rollout kernels work
// without copies; time-major makes every warp access a contiguous line.
#pragma once
#include "pendulum.cuh"
#include "systems.cuh"

namespace mbpo {

struct AdjointArgs {
  MbpoPendulumParams sys;
  int E, T;
  long long st_t, st_e;            // strides of the scalar-per-step arrays (action, reward, g_*), in elements
  long long sx_t, sx_e;            // strides of the [.,.,3] arrays, in elements (innermost stride 1)
  const float* observation;        // x_t
  const float* action;             // a_t
  const float* g_reward;           // cotangent of reward[t]            (NULL = 0)
  const float* g_next_obs;         // cotangent of next_observation[t]  (NULL = 0)
  const float* g_obs;              // cotangent of observation[t]       (NULL = 0; observation[t] = next_observation[t-1], observation[0] = x0)
  const float* g_action_in;        // direct cotangent of action[t]     (NULL = 0)
  float* g_action_out;             // total cotangent reaching a_t
  float* g_x0_out;                 // [E,3] cotangent of the initial state (NULL = not wanted)
};

__global__ void __launch_bounds__(128) rollout_adjoint_pendulum_kernel(const __grid_constant__ AdjointArgs a) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.E) return;
  const PendulumConsts pc(a.sys);
  const long long be = static_cast<long long>(e) * a.st_e, bx = static_cast<long long>(e) * a.sx_e;
  float lc = 0.0f, ls = 0.0f, lw = 0.0f;     // lam_{t+1}
  for (int t = a.T - 1; t >= 0; --t) {
    const long long i1 = be + t * a.st_t, i3 = bx + t * a.sx_t;
    const float c = a.observation[i3], s = a.observation[i3 + 1], w = a.observation[i3 + 2];
    const float u = a.action[i1];
    const float gr = a.g_reward ? a.g_reward[i1] : 0.0f;
    float gc = lc, gs = ls, gw = lw;
    if (a.g_next_obs) { gc += a.g_next_obs[i3]; gs += a.g_next_obs[i3 + 1]; gw += a.g_next_obs[i3 + 2]; }
    if (a.g_obs && t + 1 < a.T) {            // observation[t+1] is the same value as next_observation[t]
      const long long j3 = i3 + a.sx_t;
      gc += a.g_obs[j3]; gs += a.g_obs[j3 + 1]; gw += a.g_obs[j3 + 2];
    }
    float g_u;
    pendulum_step_vjp(pc, c, s, w, u, gc, gs, gw, gr, lc, ls, lw, g_u);
    if (a.g_action_in) g_u += a.g_action_in[i1];
    a.g_action_out[i1] = g_u;
  }
  if (a.g_x0_out) {
    float gc = lc, gs = ls, gw = lw;
    if (a.g_obs && a.T > 0) { gc += a.g_obs[bx]; gs += a.g_obs[bx + 1]; gw += a.g_obs[bx + 2]; }
    a.g_x0_out[3 * e] = gc; a.g_x0_out[3 * e + 1] = gs; a.g_x0_out[3 * e + 2] = gw;
  }
}

struct AdjointGeneralArgs {
  MbpoGeneralSystemParams sys;
  int E, T;
  long long st_t, st_e;            // strides of g_reward, in elements
  long long sx_t, sx_e;            // strides of the [.,.,X] arrays (innermost stride 1)
  long long sa_t, sa_e;            // strides of the [.,.,A] arrays: action, g_action_in, g_action_out (innermost 1)
  const float* observation;        // as AdjointArgs
  const float* action;
  const float* g_reward;
  const float* g_next_obs;
  const float* g_obs;
  const float* g_action_in;
  float* g_action_out;
  float* g_x0_out;                 // [E,X]
};

// The same reverse scan for a general System (systems.cuh), through its step_vjp: X-float state adjoint, A action
// cotangents per step.  A keyed System's noise enters its step additively and depends on neither x nor u, so the
// scan needs no keys.
template <class Sys>
__global__ void __launch_bounds__(128) rollout_adjoint_general_kernel(const __grid_constant__ AdjointGeneralArgs a) {
  constexpr int X = Sys::X, A = Sys::A;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.E) return;
  const Sys sys(a.sys);
  const long long be = static_cast<long long>(e) * a.st_e, bx = static_cast<long long>(e) * a.sx_e;
  const long long ba = static_cast<long long>(e) * a.sa_e;
  float lam[X];                              // lam_{t+1}
#pragma unroll
  for (int k = 0; k < X; ++k) lam[k] = 0.0f;
  for (int t = a.T - 1; t >= 0; --t) {
    const long long i1 = be + t * a.st_t, ix = bx + t * a.sx_t, ia = ba + t * a.sa_t;
    float x[X], u[A], g[X], g_u[A];
#pragma unroll
    for (int k = 0; k < X; ++k) {
      x[k] = a.observation[ix + k];
      g[k] = lam[k];
      if (a.g_next_obs) g[k] += a.g_next_obs[ix + k];
      if (a.g_obs && t + 1 < a.T) g[k] += a.g_obs[ix + a.sx_t + k];   // observation[t+1] = next_observation[t]
    }
#pragma unroll
    for (int j = 0; j < A; ++j) u[j] = a.action[ia + j];
    const float gr = a.g_reward ? a.g_reward[i1] : 0.0f;
    sys.step_vjp(x, u, g, gr, lam, g_u);
#pragma unroll
    for (int j = 0; j < A; ++j) a.g_action_out[ia + j] = a.g_action_in ? g_u[j] + a.g_action_in[ia + j] : g_u[j];
  }
  if (a.g_x0_out) {
#pragma unroll
    for (int k = 0; k < X; ++k)
      a.g_x0_out[static_cast<long long>(e) * X + k] = (a.g_obs && a.T > 0) ? lam[k] + a.g_obs[bx + k] : lam[k];
  }
}

struct LambdaArgs {
  int E, T;
  long long st_t, st_e;
  float discount, lambda_, one_minus_lambda, discount_lambda;
  const float* reward;        // forward: reward;        transpose: g_returns
  const float* next_values;   // forward: next_values;   transpose: unused
  float* out;                 // forward: returns;       transpose: g_reward
  float* out2;                // forward: unused;        transpose: g_next_values
};

// returns[t] = reward[t] + discount * next_values[t] * (1 - lambda) + discount * lambda * returns[t+1]
__global__ void __launch_bounds__(128) lambda_return_kernel(const __grid_constant__ LambdaArgs a) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.E || a.T == 0) return;
  const long long be = static_cast<long long>(e) * a.st_e;
  const float one_minus = a.one_minus_lambda, dl = a.discount_lambda;
  float agg = a.next_values[be + (a.T - 1) * a.st_t];
  for (int t = a.T - 1; t >= 0; --t) {
    const long long i = be + t * a.st_t;
    // inputs = reward + discount * next_values * (1 - lambda_)   (left to right, unfused)
    const float inp = __fadd_rn(a.reward[i], __fmul_rn(__fmul_rn(a.discount, a.next_values[i]), one_minus));
    agg = __fadd_rn(inp, __fmul_rn(dl, agg));        // inp + discount * lambda_ * agg
    a.out[i] = agg;
  }
}

// Transpose of the scan above: g_inputs[t] = g_returns[t] + discount * lambda * g_inputs[t-1];
// g_reward = g_inputs; g_next_values = discount * (1 - lambda) * g_inputs, plus the bootstrap
// start next_values[-1], which receives discount * lambda * g_inputs[T-1].
__global__ void __launch_bounds__(128) lambda_return_transpose_kernel(const __grid_constant__ LambdaArgs a) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.E || a.T == 0) return;
  const long long be = static_cast<long long>(e) * a.st_e;
  const float dl = a.discount_lambda, dn = a.discount * a.one_minus_lambda;
  float g = 0.0f;
  for (int t = 0; t < a.T; ++t) {
    const long long i = be + t * a.st_t;
    g = fmaf(dl, g, a.reward[i]);
    a.out[i] = g;
    a.out2[i] = dn * g + (t == a.T - 1 ? dl * g : 0.0f);
  }
}

}  // namespace mbpo
