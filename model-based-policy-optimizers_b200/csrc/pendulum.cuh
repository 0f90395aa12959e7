// Analytic pendulum System.step, inlined for the rollout kernels.
//
// Follows mbpo/systems/pendulum_system.py:18-39,
//         mbpo/systems/dynamics/pendulum_dynamics.py:29-63 (next_state / ode) and
//         mbpo/systems/rewards/pendulum_reward.py:27-42 (reward on the CURRENT state).
#pragma once
#include "../../include/mbpo_b200.h"
#include "mathx.cuh"

namespace mbpo {

// Loop-invariant constants derived from MbpoPendulumParams exactly as the reference's
// float32 expressions evaluate them: 3*g/(2*l) and 3.0/(m*l**2) (pendulum_dynamics.py:60).
struct PendulumConsts {
  float max_speed, max_torque, dt, c_g, c_u;
  float control_cost, angle_cost, target_angle;
  __host__ __device__ explicit PendulumConsts(const MbpoPendulumParams& p) {
    max_speed = p.max_speed;
    max_torque = p.max_torque;
    dt = p.dt;
#ifdef __CUDA_ARCH__
    c_g = __fdiv_rn(__fmul_rn(3.0f, p.g), __fmul_rn(2.0f, p.l));
    c_u = __fdiv_rn(3.0f, __fmul_rn(p.m, __fmul_rn(p.l, p.l)));
#else
    c_g = (3.0f * p.g) / (2.0f * p.l);
    c_u = 3.0f / (p.m * (p.l * p.l));
#endif
    control_cost = p.control_cost;
    angle_cost = p.angle_cost;
    target_angle = p.target_angle;
  }
};

#define MBPO_PI_F 3.14159274f      /* float32(jnp.pi)   */
#define MBPO_TWO_PI_F 6.28318548f  /* float32(2*jnp.pi) */

// ((d + pi) % (2*pi)) - pi with jnp's floored remainder (pendulum_reward.py:35).
// SMALL: the caller guarantees |d + pi| < 4*pi (|theta| <= pi + max_speed*dt and a target angle
// the host checked), which drops the fmod slow path from the instruction stream.
template <bool SMALL = false>
__device__ __forceinline__ float wrap_diff(float d) {
  const float x = d + MBPO_PI_F;
  float r;
  if (SMALL || fabsf(x) < 2.0f * MBPO_TWO_PI_F) {
    // fmod is exact; for |x| < 4*pi it is x or x -/+ 2*pi (Sterbenz-exact subtraction)
    r = x;
    if (r >= MBPO_TWO_PI_F) r -= MBPO_TWO_PI_F;
    if (r <= -MBPO_TWO_PI_F) r += MBPO_TWO_PI_F;
  } else {
    r = fmodf(x, MBPO_TWO_PI_F);
  }
  if (r < 0.0f) r += MBPO_TWO_PI_F;
  return r - MBPO_PI_F;
}

template <bool SMALL = false>
__device__ __forceinline__ float reward_from(const PendulumConsts& p, float th, float thdot, float u) {
  // Every contraction is spelled out: a*b + c*d leaves the compiler a choice of which product to
  // fuse, and it chooses differently in different loops -- the kernels must agree bit for bit.
  const float diff = wrap_diff<SMALL>(th - p.target_angle);
  const float t = fmaf(0.1f, __fmul_rn(thdot, thdot), __fmul_rn(p.angle_cost, __fmul_rn(diff, diff)));
  return fmaf(-p.control_cost, __fmul_rn(u, u), -t);
}

// thdot + (3g/(2l) sin(th) + 3/(ml^2) u) dt, clipped (pendulum_dynamics.py:59-62)
__device__ __forceinline__ float pendulum_next_thdot(const PendulumConsts& p, float sin_th, float w, float u) {
  const float uu = __fmul_rn(fminf(fmaxf(u, -1.0f), 1.0f), p.max_torque);   // :59
  const float thdd = fmaf(p.c_g, sin_th, __fmul_rn(p.c_u, uu));               // :60
  return fminf(fmaxf(fmaf(thdd, p.dt, w), -p.max_speed), p.max_speed);        // :61-62 (=:41-42)
}

// One reference-literal step on the [cos, sin, thdot] state.
template <bool SMALL = false>
__device__ __forceinline__ void pendulum_step_ref(const PendulumConsts& p, float& c, float& s, float& w,
                                                  float u, float& reward) {
  const float th = atan2_bounded(s, c);                             // dynamics :35 / reward :32
  reward = reward_from<SMALL>(p, th, w, u);                         // reward uses x, raw u
  const float nw = pendulum_next_thdot(p, sin_bounded(th), w, u);
  const float nth = fmaf(nw, p.dt, th);                             // :40
  sincos_bounded(nth, s, c);                                        // :43
  w = nw;
}

// The same reference-literal step for a loop that only needs the rewards: theta = atan2(sin, cos) of the CURRENT
// state comes in, theta of the NEXT state goes out -- atan2 of the freshly computed [cos(newth), sin(newth)] as
// pendulum_dynamics.py:35 evaluates it at the next step, so every value has the bits pendulum_step_ref produces;
// the pair is a unit vector, which lets atan2 skip its zero / denormal guard.  The first theta of a rollout is
// atan2_bounded(s0, c0) (guarded: the caller's initial state is arbitrary).
template <bool SMALL = false>
__device__ __forceinline__ void pendulum_step_ref_th(const PendulumConsts& p, float& th, float& w, float u,
                                                     float& reward) {
  reward = reward_from<SMALL>(p, th, w, u);
  const float nw = pendulum_next_thdot(p, sin_bounded(th), w, u);
  const float nth = fmaf(nw, p.dt, th);
  float s, c;
  sincos_bounded(nth, s, c);
  th = atan2_bounded<true>(s, c);
  w = nw;
}

// The same step for a loop that also needs [cos, sin] of every state (the env kernels stream them out): theta of the
// current state in, the next state's [cos, sin] and its theta out.  Same bits as pendulum_step_ref.
template <bool SMALL = false>
__device__ __forceinline__ void pendulum_step_ref_thcs(const PendulumConsts& p, float& th, float& c, float& s,
                                                       float& w, float u, float& reward) {
  reward = reward_from<SMALL>(p, th, w, u);
  const float nw = pendulum_next_thdot(p, sin_bounded(th), w, u);
  const float nth = fmaf(nw, p.dt, th);
  sincos_bounded(nth, s, c);
  th = atan2_bounded<true>(s, c);
  w = nw;
}

// Theta-carry variant: the state is (theta, thdot) with theta kept in (-pi, pi], which is
// what atan2(sin(newth), cos(newth)) returns up to rounding.
template <bool SMALL = false>
__device__ __forceinline__ void pendulum_step_theta(const PendulumConsts& p, float& th, float& w, float u,
                                                    float& reward) {
  reward = reward_from<SMALL>(p, th, w, u);
  const float nw = pendulum_next_thdot(p, sin_bounded(th), w, u);
  float nth = fmaf(nw, p.dt, th);
  if (nth > MBPO_PI_F) nth -= MBPO_TWO_PI_F;
  if (nth < -MBPO_PI_F) nth += MBPO_TWO_PI_F;
  th = nth;
  w = nw;
}

// ---- pair forms: two independent chains in one thread (rollout_return2), SMALL only ---------------------------
// Each packs the scalar function's float additions, multiplications and FMAs into FADD2 / FMUL2 / FFMA2 on the same
// operands in the same order; clips, compares and the conditional +-2 pi run per element.  Same bits per element.

// wrap_diff<true> of both elements.
__device__ __forceinline__ f32x2_t wrap_diff_small2(f32x2_t d) {
  float r[2];
  unpack2(add2(d, splat2(MBPO_PI_F)), r[0], r[1]);
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    if (r[i] >= MBPO_TWO_PI_F) r[i] -= MBPO_TWO_PI_F;
    if (r[i] <= -MBPO_TWO_PI_F) r[i] += MBPO_TWO_PI_F;
    if (r[i] < 0.0f) r[i] += MBPO_TWO_PI_F;
  }
  return sub2(pack2(r[0], r[1]), splat2(MBPO_PI_F));
}

// MINUS the reward of both elements: reward_from<true> computes fma(-control_cost, u*u, -t); this is
// fma(control_cost, u*u, t), its exact negation under round-to-nearest except that an exact zero comes out +0 where
// the reward is -0.  Subtracted from a sum that starts at +0 it gives the bits adding the reward gives.
__device__ __forceinline__ f32x2_t neg_reward_small2(const PendulumConsts& p, f32x2_t th, f32x2_t thdot, f32x2_t u) {
  const f32x2_t diff = wrap_diff_small2(sub2(th, splat2(p.target_angle)));
  const f32x2_t t = fma2(splat2(0.1f), mul2(thdot, thdot), mul2(splat2(p.angle_cost), mul2(diff, diff)));
  return fma2(splat2(p.control_cost), mul2(u, u), t);
}

// pendulum_next_thdot of both elements.
__device__ __forceinline__ f32x2_t pendulum_next_thdot2(const PendulumConsts& p, f32x2_t sin_th, f32x2_t w,
                                                        f32x2_t u) {
  float u0, u1;
  unpack2(u, u0, u1);
  const f32x2_t uu = mul2(pack2(fminf(fmaxf(u0, -1.0f), 1.0f), fminf(fmaxf(u1, -1.0f), 1.0f)), splat2(p.max_torque));
  const f32x2_t thdd = fma2(splat2(p.c_g), sin_th, mul2(splat2(p.c_u), uu));
  float v0, v1;
  unpack2(fma2(thdd, splat2(p.dt), w), v0, v1);
  return pack2(fminf(fmaxf(v0, -p.max_speed), p.max_speed), fminf(fmaxf(v1, -p.max_speed), p.max_speed));
}

// pendulum_step_ref_th<true> of two chains; neg_reward as neg_reward_small2.
__device__ __forceinline__ void pendulum_step_ref_th2(const PendulumConsts& p, f32x2_t& th, f32x2_t& w, f32x2_t u,
                                                      f32x2_t& neg_reward) {
  neg_reward = neg_reward_small2(p, th, w, u);
  f32x2_t s, c;
  sincos_bounded2(th, s, c);
  const f32x2_t nw = pendulum_next_thdot2(p, s, w, u);
  sincos_bounded2(fma2(nw, splat2(p.dt), th), s, c);
  th = atan2_bounded_unit2(s, c);
  w = nw;
}

// pendulum_step_theta<true> of two chains; neg_reward as neg_reward_small2.
__device__ __forceinline__ void pendulum_step_theta2(const PendulumConsts& p, f32x2_t& th, f32x2_t& w, f32x2_t u,
                                                     f32x2_t& neg_reward) {
  neg_reward = neg_reward_small2(p, th, w, u);
  f32x2_t s, c;
  sincos_bounded2(th, s, c);
  const f32x2_t nw = pendulum_next_thdot2(p, s, w, u);
  float nth[2];
  unpack2(fma2(nw, splat2(p.dt), th), nth[0], nth[1]);
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    if (nth[i] > MBPO_PI_F) nth[i] -= MBPO_TWO_PI_F;
    if (nth[i] < -MBPO_PI_F) nth[i] += MBPO_TWO_PI_F;
  }
  th = pack2(nth[0], nth[1]);
  w = nw;
}

// jnp.clip = minimum(maximum(x, lo), hi): lax.max / lax.min split the cotangent evenly at a tie.
__device__ __forceinline__ float clip_grad(float x, float lo, float hi) {
  const float a = (x > lo) ? 1.0f : (x == lo ? 0.5f : 0.0f);          // d max(x, lo) / dx
  const float m = fmaxf(x, lo);
  const float b = (m < hi) ? 1.0f : (m == hi ? 0.5f : 0.0f);          // d min(m, hi) / dm
  return a * b;
}

// Cotangents of one pendulum System.step at state [c, s, w] and action u (the 3 x 3 Jacobian-transpose products
// written out for pendulum_dynamics.py:29-63 and pendulum_reward.py:27-42), re-deriving the step's intermediates:
// [gc, gs, gw] is the cotangent of x_next, gr that of the reward; out come the cotangent [lc, ls, lw] of the state
// and g_u of the action.  [c, s] need not be a unit vector: the atan2 derivative divides by c^2 + s^2.
__device__ __forceinline__ void pendulum_step_vjp(const PendulumConsts& pc, float c, float s, float w, float u,
                                                  float gc, float gs, float gw, float gr, float& lc, float& ls,
                                                  float& lw, float& g_u) {
  // forward intermediates of this step (pendulum_dynamics.py:35,59-62,40,43)
  const float th = atan2_bounded(s, c);
  float sin_th, cos_th;
  sincos_bounded(th, sin_th, cos_th);
  const float uu = __fmul_rn(fminf(fmaxf(u, -1.0f), 1.0f), pc.max_torque);
  const float thdd = fmaf(pc.c_g, sin_th, __fmul_rn(pc.c_u, uu));
  const float v = fmaf(thdd, pc.dt, w);
  const float nw = fminf(fmaxf(v, -pc.max_speed), pc.max_speed);
  const float nth = fmaf(nw, pc.dt, th);
  float sn, cn;
  sincos_bounded(nth, sn, cn);
  // x_next = [cos(nth), sin(nth), nw]
  const float g_nth = cn * gs - sn * gc;
  const float g_nw = gw + pc.dt * g_nth;
  const float g_v = g_nw * clip_grad(v, -pc.max_speed, pc.max_speed);
  const float g_thdd = pc.dt * g_v;
  // reward on (x_t, a_t) (pendulum_reward.py:32-39); d/dth of the wrapped difference is 1
  const float diff = wrap_diff(th - pc.target_angle);
  float g_th = g_nth + g_thdd * pc.c_g * cos_th - gr * 2.0f * pc.angle_cost * diff;
  const float g_w = g_v - gr * 0.2f * w;
  g_u = g_thdd * pc.c_u * pc.max_torque * clip_grad(u, -1.0f, 1.0f) - gr * 2.0f * pc.control_cost * u;
  // th = atan2(s, c): dth/dc = -s / (c^2 + s^2), dth/ds = c / (c^2 + s^2)
  const float r2 = c * c + s * s;
  const float inv = r2 > 0.0f ? 1.0f / r2 : 0.0f;
  lc = -g_th * s * inv;
  ls = g_th * c * inv;
  lw = g_w;
}

}  // namespace mbpo
