// iCEM kernels: fused plan (sample -> rollout -> select -> refit, all S iterations in one
// launch, one CTA per planning problem) and the staged kernels behind the per-stage C ABI.
//
// Reference: mbpo/optimizers/trajectory_optimizers/icem_optimizer.py:134-252 (optimize),
// mbpo/utils/optimizer_utils.py:11-59 (rollout_actions), pendulum_*.py (System.step).
#pragma once
#include <cuda_runtime.h>

#include "noise.cuh"
#include "pendulum.cuh"
#include "select.cuh"
#include "systems.cuh"

namespace mbpo {

// ------------------------------------------------------------------------------------------
// Rollout of one action row held in shared/global memory; returns the horizon-mean reward
// (icem_optimizer.py:160 inner jnp.mean over rollout_actions(...).reward).
// ------------------------------------------------------------------------------------------
// SMALL: the host checked |target_angle| <= 6, so the reward's floored mod needs no fmod slow path.
// th0 = atan2_bounded(s0, c0) of the initial state.
template <int MATH, bool SMALL = false, typename ActFn>
__device__ __forceinline__ float rollout_return_th(const PendulumConsts& pc, float th0, float w0, int H, ActFn act) {
  float acc = 0.0f;
  float th = th0, w = w0;
#pragma unroll 2
  for (int t = 0; t < H; ++t) {
    float r;
    if (MATH == MBPO_MATH_REFERENCE) pendulum_step_ref_th<SMALL>(pc, th, w, act(t), r);
    else pendulum_step_theta<SMALL>(pc, th, w, act(t), r);
    acc = __fadd_rn(acc, r);
  }
  return __fdiv_rn(acc, static_cast<float>(H));
}

template <int MATH, bool SMALL = false, typename ActFn>
__device__ __forceinline__ float rollout_return(const PendulumConsts& pc, float c0, float s0, float w0, int H,
                                                ActFn act) {
  return rollout_return_th<MATH, SMALL>(pc, atan2_bounded(s0, c0), w0, H, act);
}

// Two independent rollouts from the same initial state (th0 = atan2(s0, c0), computed once per problem by the
// caller), interleaved step by step: the horizon recurrence is a serial dependency chain, so a second chain in
// the same thread doubles the instruction-level parallelism at a cost of ~8 registers.  The two chains run as the
// halves of packed pairs (pendulum.cuh pair forms): one FFMA2 / FMUL2 / FADD2 issue slot serves both, same bits as
// two scalar steps.  SMALL only (|target_angle| <= 6, host-checked).
template <int MATH>
__device__ __forceinline__ void rollout_return2(const PendulumConsts& pc, float th0, float w0, int H,
                                                const float* __restrict__ row_a, const float* __restrict__ row_b,
                                                float& ret_a, float& ret_b) {
  f32x2_t acc = splat2(0.0f), th = splat2(th0), w = splat2(w0);
#pragma unroll 1
  for (int t = 0; t < H; ++t) {
    f32x2_t neg_r;
    if (MATH == MBPO_MATH_REFERENCE) pendulum_step_ref_th2(pc, th, w, pack2(row_a[t], row_b[t]), neg_r);
    else pendulum_step_theta2(pc, th, w, pack2(row_a[t], row_b[t]), neg_r);
    acc = sub2(acc, neg_r);   // acc + reward
  }
  float acc_a, acc_b;
  unpack2(acc, acc_a, acc_b);
  ret_a = __fdiv_rn(acc_a, static_cast<float>(H));
  ret_b = __fdiv_rn(acc_b, static_cast<float>(H));
}

// summarize over P identical particles (deterministic System): jnp.mean / jnp.max  (:160)
__device__ __forceinline__ float summarize_particles(float ret, int P, int summarize) {
  if (summarize == MBPO_SUMMARIZE_MAX || P == 1) return ret;
  float acc = 0.0f;
  for (int p = 0; p < P; ++p) acc = __fadd_rn(acc, ret);
  return __fdiv_rn(acc, static_cast<float>(P));
}

// ------------------------------------------------------------------------------------------
// Fused plan kernel
// ------------------------------------------------------------------------------------------
struct PlanArgs {
  // shapes / hyper-parameters (H: the horizon, read by the any-horizon kernels only; the others have it as a template argument)
  int B, N, Np, K, P, S, H;
  int warm_start, summarize;
  float init_std, alpha, one_minus_alpha, u_min, u_max;
  MbpoPendulumParams sys;
  MbpoGeneralSystemParams gsys;  // the general Systems (systems.cuh): fused general plan only
  float scale[MBPO_MAX_FREQ];  // fill_noise_scale()
  // I/O
  const float* x0;           // [B,3]
  const uint32_t* key_in;    // [B,2]
  const float* best_seq_in;  // [B,H]
  float* best_seq_out;       // [B,H]
  float* best_value_out;     // [B]
  uint32_t* key_out;         // [B,2]
  MbpoIcemTrace trace;       // optional dumps
  // 1: best_value_out[b] holds, on entry, the objective of the all-zero action row of problem b
  // (zero_row_value_kernel) -- the kept-elite rows are then no rollout job inside the plan.
  int zero_value_precomputed;
};

// HT: the horizon as a template argument (unrolled sampling, immediate twiddles) or 0 = any horizon, read from
// PlanArgs::H at run time (rolled sampling; needs a staging row per thread besides the action rows).
constexpr int PLAN_THREADS = 256;

template <int HT>
struct PlanSmem {
  static constexpr int HS = HT | 1;  // odd row stride: conflict-free per-thread rows (HT != 0)
  static size_t bytes(int N, int Np, int K, int H_rt = 0) {
    const int H = HT ? HT : H_rt;
    const int hs = H | 1;
    size_t words = static_cast<size_t>(N + 1) * hs  // action rows + one all-zero row
                   + (N + Np)                   // sort keys
                   + 2 * (N + 1)                // legacy split words
                   + 3 * H                      // mean, std, best_seq
                   + 2 * K                      // elite_idx, sel_idx
                   + select_scratch_words(K, N + Np)  // selection histogram + lists
                   + 8                          // best_value, carry key, state key, pad
                   + (HT ? 0 : static_cast<size_t>(PLAN_THREADS) * hs);  // any horizon: staged normals of the row in flight
    return words * 4;
  }
};

// Shared-memory carve-up of one planning CTA.
template <int HT>
struct PlanCtaSmem {
  float* act;          // [N + 1][HS] action rows of the sampled candidates; row N is all zeros
  uint32_t* skey;      // [M]     total-order keys of the objective values
  uint32_t* flat;      // [2(N+1)] legacy split(sampling_rng, N+1) words
  float* mean;         // [H]
  float* std_;         // [H]
  float* best_seq;     // [H]
  int* elite_idx;      // [K]
  int* sel_idx;        // [K]
  uint32_t* sel_scratch;  // [select_scratch_words(K, M)]
  float* best_value;   // [1]
  uint32_t* carry;     // [2] carry.key
  uint32_t* state_key; // [2] opt_state.key (closed loop)
  float* stage;        // [THREADS][HS] (HT == 0 only)
  __device__ __forceinline__ PlanCtaSmem(uint32_t* base, int N, int Np, int K, int H_rt = 0) {
    const int H = HT ? HT : H_rt;
    const int HS = H | 1;
    act = reinterpret_cast<float*>(base);
    skey = base + static_cast<size_t>(N + 1) * HS;
    flat = skey + (N + Np);
    mean = reinterpret_cast<float*>(flat + 2 * (N + 1));
    std_ = mean + H;
    best_seq = std_ + H;
    elite_idx = reinterpret_cast<int*>(best_seq + H);
    sel_idx = elite_idx + K;
    sel_scratch = reinterpret_cast<uint32_t*>(sel_idx + K);
    best_value = reinterpret_cast<float*>(sel_scratch + select_scratch_words(K, N + Np));
    carry = reinterpret_cast<uint32_t*>(best_value + 1);
    state_key = carry + 2;
    stage = reinterpret_cast<float*>(state_key + 5);
  }
};

// iCemTO.optimize for ONE problem, executed by the whole CTA (icem_optimizer.py:134-252).
// Thread n owns samples n, n+THREADS, ...: it derives the sample's key, generates the
// colored-noise row straight into its shared-memory action row, rolls the row out with the
// state in registers and publishes the total-order key of the objective.  The CTA then selects
// and refits together (select.cuh).  `prev_best` ([H], global or this CTA's own sm.best_seq) is the previous plan's
// best sequence for the warm start; `key_in` is opt_state.key; the new opt_state.key is
// returned through key_new (valid in thread 0 only).  `slot` indexes the optional trace
// dumps ([S, B, ...] with problem slot `slot` of `slots`).
template <int HT, int PRNG, int MATH, int THREADS>
__device__ __forceinline__ void plan_problem(const PlanArgs& a, const PlanCtaSmem<HT>& sm, const PendulumConsts& pc,
                                             const RefitScalars& rs, const float* prev_best, Key2 key_in,
                                             Key2& key_new, float x_th, float x_w, int slot, int slots,
                                             const TwiddleTable* tw = nullptr) {
  const int H = HT ? HT : a.H;
  const int HS = H | 1;
  const int N = a.N, M = a.N + a.Np, K = a.K;
  const int tid = threadIdx.x;
  float* act = sm.act;
  uint32_t* skey = sm.skey;
  uint32_t* flat = sm.flat;
  float* mean = sm.mean;
  float* std_ = sm.std_;
  float* best_seq = sm.best_seq;

  // ---- prologue: warm start, key split (icem_optimizer.py:235-249) ------------------------
  float m0 = 0.0f;
  if (tid < H && a.warm_start) m0 = prev_best[tid + 1 < H ? tid + 1 : H - 1];
  __syncthreads();  // prev_best may alias best_seq
  if (tid < H) {
    mean[tid] = m0;
    std_[tid] = a.init_std;
    best_seq[tid] = m0;
  }
  if (tid < HS) act[static_cast<size_t>(N) * HS + tid] = 0.0f;   // the all-zero row
  if (tid == 0) {
    *sm.best_value = __int_as_float(0xFF800000);  // -inf
    Key2 k_opt;
    split2<PRNG>(key_in, k_opt, key_new);         // optimizer_key, key = split(opt_state.key, 2)
    sm.carry[0] = k_opt.k0;
    sm.carry[1] = k_opt.k1;
  }
  __syncthreads();

  for (int it = 0; it < a.S; ++it) {
    const size_t tslot = static_cast<size_t>(it) * slots + slot;
    // ---- key plumbing (:174-180) -----------------------------------------------------------
    Key2 ck{sm.carry[0], sm.carry[1]}, sampling_rng, particles_rng;
    split2<PRNG>(ck, sampling_rng, particles_rng);  // particles_rng is dead for a deterministic System
    if (PRNG == MBPO_PRNG_LEGACY) {
      // split(sampling_rng, N+1): block j -> flat[j], flat[N+1+j]
      for (int j = tid; j < N + 1; j += THREADS) {
        uint32_t y0 = static_cast<uint32_t>(j), y1 = static_cast<uint32_t>(N + 1 + j);
        threefry2x32(sampling_rng.k0, sampling_rng.k1, y0, y1);
        flat[j] = y0;
        flat[N + 1 + j] = y1;
      }
    }
    __syncthreads();  // flat complete; every thread has read carry
    if (tid == 0) {
      Key2 nk;
      if (PRNG == MBPO_PRNG_LEGACY) { nk.k0 = flat[0]; nk.k1 = flat[1]; }
      else nk = split_at<1>(sampling_rng, static_cast<uint32_t>(N + 1), 0u);
      sm.carry[0] = nk.k0; sm.carry[1] = nk.k1;   // key = sampling_rng[0]  (:176)
    }

    // ---- sample + rollout ----------------------------------------------------------------------
    // Jobs 0..N-1 are the sampled candidates, job N is the closure's all-zero kept-elite row
    // (:192,:245; deterministic System: one rollout serves all Np rows and all iterations, so it
    // is only a job in iteration 0).  A thread takes jobs tid, tid + THREADS, ... two at a time:
    // both rows are sampled first, then rolled out together (rollout_return2).
    const int jobs = (it == 0 && !a.zero_value_precomputed) ? N + 1 : N;
    if (it == 0 && a.zero_value_precomputed && tid == THREADS - 1) {
      const uint32_t zk = total_order_key(a.best_value_out[slot]);
      for (int j = N; j < M; ++j) skey[j] = zk;
    }
    for (int n0 = tid; n0 < jobs; n0 += 2 * THREADS) {
      const int n1 = n0 + THREADS;
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        const int n = h ? n1 : n0;
        if (n >= N) continue;
        Key2 skey_n;
        if (PRNG == MBPO_PRNG_LEGACY) { skey_n.k0 = flat[2 * (n + 1)]; skey_n.k1 = flat[2 * (n + 1) + 1]; }
        else skey_n = split_at<1>(sampling_rng, static_cast<uint32_t>(N + 1), static_cast<uint32_t>(n + 1));
        const Key2 dim_key = split1<PRNG>(skey_n);             // vmap(split(x, action_dim)), A == 1  (:180)
        float* row = act + static_cast<size_t>(n) * HS;
        auto emit = [&](int t, float y) {
          const float v = __fadd_rn(mean[t], __fmul_rn(y, std_[t]));           // :190
          row[t] = fminf(fmaxf(v, a.u_min), a.u_max);                          // :191
        };
        if constexpr (HT != 0) colored_noise_row<HT, PRNG>(dim_key, a.scale, row, nullptr, emit);
        else colored_noise_row_rt<PRNG>(H, dim_key, a.scale, *tw, sm.stage + static_cast<size_t>(tid) * HS, nullptr, emit);
      }
      const int r0 = n0 < N ? n0 : N, r1 = n1 < N ? n1 : N;   // idle slots roll out the zero row
      float ret0, ret1;
      rollout_return2<MATH>(pc, x_th, x_w, H, act + static_cast<size_t>(r0) * HS, act + static_cast<size_t>(r1) * HS,
                            ret0, ret1);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int n = h ? n1 : n0;
        const float val = summarize_particles(h ? ret1 : ret0, a.P, a.summarize);
        if (n < N) {
          skey[n] = total_order_key(val);
          if (a.trace.values) a.trace.values[tslot * M + n] = val;
          if (a.trace.actions) {
            const float* row = act + static_cast<size_t>(n) * HS;
            float* dst = a.trace.actions + (tslot * M + n) * H;
            for (int t = 0; t < H; ++t) dst[t] = row[t];
          }
        } else if (n == N && it == 0) {
          const uint32_t zk = total_order_key(val);
          for (int j = N; j < M; ++j) skey[j] = zk;
        }
      }
    }
    __syncthreads();
    if (a.trace.values || a.trace.actions) {
      const uint32_t zk = skey[N];
      const float zv = __uint_as_float((zk & 0x80000000u) ? (zk & 0x7FFFFFFFu) : ~zk);
      for (int j = N + tid; j < M; j += THREADS) {
        if (a.trace.values) a.trace.values[tslot * M + j] = zv;
        if (a.trace.actions) {
          float* dst = a.trace.actions + (tslot * M + j) * H;
          for (int t = 0; t < H; ++t) dst[t] = 0.0f;
        }
      }
    }

    // ---- select + refit + best tracking (:199-226), whole CTA --------------------------------
    cta_select_refit<THREADS>(rs, skey, sm.elite_idx, sm.sel_idx, sm.sel_scratch,
                              [&](int i, int d) { return i < N ? act[static_cast<size_t>(i) * HS + d] : 0.0f; },
                              mean, std_, best_seq, sm.best_value);
    if (a.trace.elite_idx)
      for (int e = tid; e < K; e += THREADS) a.trace.elite_idx[tslot * K + e] = sm.elite_idx[e];
    for (int d = tid; d < H; d += THREADS) {
      if (a.trace.mean) a.trace.mean[tslot * H + d] = mean[d];
      if (a.trace.std) a.trace.std[tslot * H + d] = std_[d];
    }
    if (a.trace.best_value && tid == 0) a.trace.best_value[tslot] = *sm.best_value;
    __syncthreads();
  }
}

// Objective of the all-zero action row (the closure's kept-elite rows, :192,:245) for every
// problem, one thread per problem: keeps a one-lane rollout out of the plan kernel's CTAs.
template <int MATH>
__global__ void zero_row_value_kernel(const MbpoPendulumParams sys, int H, int P, int summarize,
                                      const float* __restrict__ x0, int B, float* __restrict__ out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const PendulumConsts pc(sys);
  const float ret = rollout_return<MATH, true>(pc, x0[3 * b], x0[3 * b + 1], x0[3 * b + 2], H,
                                               [](int) { return 0.0f; });
  out[b] = summarize_particles(ret, P, summarize);
}

// Fused plan: one CTA plans one problem at a time (grid-stride over problems).
template <int HT, int PRNG, int MATH, int THREADS>
__device__ __forceinline__ void plan_kernel_body(const PlanArgs& a, const TwiddleTable* tw) {
  extern __shared__ __align__(16) uint32_t smem_u32[];
  const int H = HT ? HT : a.H;
  const PlanCtaSmem<HT> sm(smem_u32, a.N, a.Np, a.K, H);
  const int tid = threadIdx.x;
  const PendulumConsts pc(a.sys);
  RefitScalars rs;
  rs.M = a.N + a.Np; rs.K = a.K; rs.D = H; rs.alpha = a.alpha; rs.one_minus_alpha = a.one_minus_alpha;

  for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
    const float x_c = a.x0[3 * b], x_s = a.x0[3 * b + 1], x_w = a.x0[3 * b + 2];
    Key2 k_in{a.key_in[2 * b], a.key_in[2 * b + 1]}, k_new;
    plan_problem<HT, PRNG, MATH, THREADS>(a, sm, pc, rs, a.best_seq_in + static_cast<size_t>(b) * H, k_in, k_new,
                                          atan2_bounded(x_s, x_c), x_w, b, a.B, tw);
    // ---- epilogue (:251) -----------------------------------------------------------------
    if (tid < H) a.best_seq_out[static_cast<size_t>(b) * H + tid] = sm.best_seq[tid];
    if (tid == 0) {
      a.best_value_out[b] = *sm.best_value;
      a.key_out[2 * b] = k_new.k0;
      a.key_out[2 * b + 1] = k_new.k1;
    }
    __syncthreads();
  }
}

template <int H, int PRNG, int MATH, int THREADS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB) icem_plan_pendulum_kernel(const __grid_constant__ PlanArgs a) {
  plan_kernel_body<H, PRNG, MATH, THREADS>(a, nullptr);
}

// The same for ANY horizon in [2, MBPO_MAX_HORIZON] (PlanArgs::H): rolled sampling, twiddle table in the constant bank.
template <int PRNG, int MATH>
__global__ void __launch_bounds__(PLAN_THREADS, 1)
    icem_plan_pendulum_rt_kernel(const __grid_constant__ PlanArgs a, const __grid_constant__ TwiddleTable tw) {
  plan_kernel_body<0, PRNG, MATH, PLAN_THREADS>(a, &tw);
}

// Closed-loop MPC (tests/test_icemopt.py:19-32): T times { act = optimize(x)[0]; x = true
// system.step(x, act); warm start from the previous best sequence }, one CTA per problem,
// the whole loop in one launch (the reference runs it as one lax.scan).
struct MpcArgs {
  int T;
  float* states_out;   // [T,B,3]
  float* rewards_out;  // [T,B]
  float* actions_out;  // [T,B,1]
};

template <int HT, int PRNG, int MATH, int THREADS>
__device__ __forceinline__ void mpc_kernel_body(const PlanArgs& a, const MpcArgs& m, const TwiddleTable* tw) {
  extern __shared__ __align__(16) uint32_t smem_u32[];
  const int H = HT ? HT : a.H;
  const PlanCtaSmem<HT> sm(smem_u32, a.N, a.Np, a.K, H);
  __shared__ float xs[4];
  const int tid = threadIdx.x;
  const PendulumConsts pc(a.sys);
  RefitScalars rs;
  rs.M = a.N + a.Np; rs.K = a.K; rs.D = H; rs.alpha = a.alpha; rs.one_minus_alpha = a.one_minus_alpha;

  for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
    if (tid < H) sm.best_seq[tid] = a.best_seq_in[static_cast<size_t>(b) * H + tid];
    if (tid < 3) xs[tid] = a.x0[3 * b + tid];
    if (tid == 0) { sm.state_key[0] = a.key_in[2 * b]; sm.state_key[1] = a.key_in[2 * b + 1]; }
    __syncthreads();
    for (int t = 0; t < m.T; ++t) {
      const float x_c = xs[0], x_s = xs[1], x_w = xs[2];
      Key2 k_in{sm.state_key[0], sm.state_key[1]}, k_new;
      plan_problem<HT, PRNG, MATH, THREADS>(a, sm, pc, rs, sm.best_seq, k_in, k_new, atan2_bounded(x_s, x_c), x_w, 0,
                                            1, tw);
      if (tid == 0) {
        sm.state_key[0] = k_new.k0; sm.state_key[1] = k_new.k1;
        const float u = sm.best_seq[0];                       // opt_state.action (:67-69)
        float c = x_c, s = x_s, w = x_w, r;
        if (MATH == MBPO_MATH_REFERENCE) {
          pendulum_step_ref(pc, c, s, w, u, r);
        } else {
          float th = atan2_bounded(s, c);
          pendulum_step_theta(pc, th, w, u, r);
          sincos_bounded(th, s, c);
        }
        xs[0] = c; xs[1] = s; xs[2] = w;
        const size_t o = static_cast<size_t>(t) * a.B + b;
        if (m.states_out) { m.states_out[o * 3] = c; m.states_out[o * 3 + 1] = s; m.states_out[o * 3 + 2] = w; }
        if (m.rewards_out) m.rewards_out[o] = r;
        if (m.actions_out) m.actions_out[o] = u;
      }
      __syncthreads();
    }
    if (tid < H) a.best_seq_out[static_cast<size_t>(b) * H + tid] = sm.best_seq[tid];
    if (tid == 0) {
      a.best_value_out ? (void)(a.best_value_out[b] = *sm.best_value) : (void)0;
      a.key_out[2 * b] = sm.state_key[0];
      a.key_out[2 * b + 1] = sm.state_key[1];
    }
    __syncthreads();
  }
}

template <int H, int PRNG, int MATH, int THREADS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB)
    icem_mpc_pendulum_kernel(const __grid_constant__ PlanArgs a, const __grid_constant__ MpcArgs m) {
  mpc_kernel_body<H, PRNG, MATH, THREADS>(a, m, nullptr);
}

template <int PRNG, int MATH>
__global__ void __launch_bounds__(PLAN_THREADS, 1)
    icem_mpc_pendulum_rt_kernel(const __grid_constant__ PlanArgs a, const __grid_constant__ MpcArgs m,
                                const __grid_constant__ TwiddleTable tw) {
  mpc_kernel_body<0, PRNG, MATH, PLAN_THREADS>(a, m, &tw);
}

// ------------------------------------------------------------------------------------------
// Fused plan over the general Systems (systems.cuh): any action_dim, P distinct particles per candidate when the
// System consumes its key (icem_optimizer.py:146-160,180).  One CTA per problem like the pendulum kernel, one
// candidate at a time per thread.  A candidate's actions live in shared memory DIMENSION-MAJOR ([A][H]): the H
// floats of a dimension double as the staging area of its noise row, and System.step reads u[t] with stride H.
// The Np kept-elite rows (the closure's zeros, :192,:245) are candidates N .. N+Np-1 with their own particle keys:
// for a System that draws they are distinct rollouts every iteration.  Same device functions as the staged path
// (sample_actions_kernel, general_objective_kernel, elite_refit_kernel): same bits.
// ------------------------------------------------------------------------------------------
template <int H, int A>
struct GenPlanSmem {
  static constexpr int RS = (H * A) | 1;   // odd row stride
  static size_t bytes(int N, int Np, int K) {
    const size_t words = static_cast<size_t>(N + 1) * RS + (N + Np) + 3 * H * A + 2 * K +
                         select_scratch_words(K, N + Np) + 8;
    return words * 4;
  }
};

template <class Sys, int H, int PRNG>
__global__ void __launch_bounds__(256, 1) icem_plan_general_kernel(const __grid_constant__ PlanArgs a) {
  constexpr int A = Sys::A, X = Sys::X, D = H * A, RS = GenPlanSmem<H, A>::RS, THREADS = 256;
  extern __shared__ __align__(16) uint32_t smem_u32[];
  const int N = a.N, M = a.N + a.Np, K = a.K;
  float* act = reinterpret_cast<float*>(smem_u32);               // [N + 1][RS], row N all zeros
  uint32_t* skey = smem_u32 + static_cast<size_t>(N + 1) * RS;   // [M]
  float* mean = reinterpret_cast<float*>(skey + M);              // [H*A] in the ABI's (t, a) order
  float* std_ = mean + D;
  float* best_seq = std_ + D;
  int* elite_idx = reinterpret_cast<int*>(best_seq + D);
  int* sel_idx = elite_idx + K;
  uint32_t* scratch = reinterpret_cast<uint32_t*>(sel_idx + K);
  float* best_value = reinterpret_cast<float*>(scratch + select_scratch_words(K, M));
  uint32_t* carry = reinterpret_cast<uint32_t*>(best_value + 1);
  const int tid = threadIdx.x;
  const Sys sys(a.gsys);
  RefitScalars rs;
  rs.M = M; rs.K = K; rs.D = D; rs.alpha = a.alpha; rs.one_minus_alpha = a.one_minus_alpha;
  // element d = t * A + ad of candidate i (ABI order) in the dimension-major shared row
  auto elem = [&](int i, int d) { return i < N ? act[static_cast<size_t>(i) * RS + (d % A) * H + d / A] : 0.0f; };

  for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
    float s0[X];
#pragma unroll
    for (int k = 0; k < X; ++k) s0[k] = a.x0[static_cast<size_t>(b) * X + k];
    // ---- prologue (:235-249): warm start shifts by one step = A elements --------------------------------
    const float* prev = a.best_seq_in + static_cast<size_t>(b) * D;
    for (int d = tid; d < D; d += THREADS) {
      float m = 0.0f;
      if (a.warm_start) m = prev[(d + A < D) ? d + A : (D - A + d % A)];
      mean[d] = m;
      std_[d] = a.init_std;
      best_seq[d] = m;
    }
    for (int d = tid; d < RS; d += THREADS) act[static_cast<size_t>(N) * RS + d] = 0.0f;
    Key2 k_new{0u, 0u};
    if (tid == 0) {
      *best_value = __int_as_float(0xFF800000);
      Key2 k_opt;
      split2<PRNG>(Key2{a.key_in[2 * b], a.key_in[2 * b + 1]}, k_opt, k_new);
      carry[0] = k_opt.k0;
      carry[1] = k_opt.k1;
    }
    __syncthreads();
    float zero_value = 0.0f;   // deterministic System: the objective of the all-zero row, computed once (thread 0)

    for (int it = 0; it < a.S; ++it) {
      const size_t tslot = static_cast<size_t>(it) * a.B + b;
      Key2 ck{carry[0], carry[1]}, sampling_rng, particles_rng;
      split2<PRNG>(ck, sampling_rng, particles_rng);                                            // :174
      __syncthreads();  // every thread has read carry
      if (tid == 0) {
        const Key2 nk = split_at<PRNG>(sampling_rng, static_cast<uint32_t>(N + 1), 0u);         // :176
        carry[0] = nk.k0;
        carry[1] = nk.k1;
      }
      // candidates 0 .. N-1 are sampled; N .. M-1 are the zero rows (rolled out only if the System draws, or once)
      const int jobs = Sys::KEYED ? M : ((it == 0) ? N + 1 : N);
      for (int n = tid; n < jobs; n += THREADS) {
        float* row = act + static_cast<size_t>(n < N ? n : N) * RS;
        if (n < N) {
          const Key2 sk = split_at<PRNG>(sampling_rng, static_cast<uint32_t>(N + 1), static_cast<uint32_t>(n + 1));
#pragma unroll 1
          for (int ad = 0; ad < A; ++ad) {
            const Key2 dk = split_at<PRNG>(sk, static_cast<uint32_t>(A), static_cast<uint32_t>(ad));   // :180
            float* dim = row + ad * H;
            colored_noise_row<H, PRNG>(dk, a.scale, dim, nullptr, [&](int t, float y) {
              const float v = __fadd_rn(mean[t * A + ad], __fmul_rn(y, std_[t * A + ad]));              // :190
              dim[t] = fminf(fmaxf(v, a.u_min), a.u_max);                                               // :191
            });
          }
        }
        // ---- objective (:144-160) ----------------------------------------------------------------------
        float val;
        auto roll = [&](Key2 key) {
          float s[X];
#pragma unroll
          for (int k = 0; k < X; ++k) s[k] = s0[k];
          float acc = 0.0f;
          for (int t = 0; t < H; ++t) acc = __fadd_rn(acc, sys.template step<PRNG>(s, row + t, H, key));
          return __fdiv_rn(acc, static_cast<float>(H));
        };
        if (!Sys::KEYED) {
          const float ret = roll(Key2{0u, 0u});
          if (a.summarize == MBPO_SUMMARIZE_MAX || a.P == 1) {
            val = ret;
          } else {
            float acc = 0.0f;
            for (int p = 0; p < a.P; ++p) acc = __fadd_rn(acc, ret);
            val = __fdiv_rn(acc, static_cast<float>(a.P));
          }
        } else {
          const Key2 pkey = split_at<PRNG>(particles_rng, static_cast<uint32_t>(M), static_cast<uint32_t>(n));   // :177
          float acc = 0.0f, mx = 0.0f;
          for (int p = 0; p < a.P; ++p) {
            const float ret = roll(split_at<PRNG>(pkey, static_cast<uint32_t>(a.P), static_cast<uint32_t>(p)));  // :155
            acc = __fadd_rn(acc, ret);
            mx = (p == 0) ? ret : fmaxf(mx, ret);
          }
          val = (a.summarize == MBPO_SUMMARIZE_MAX) ? mx : __fdiv_rn(acc, static_cast<float>(a.P));
        }
        if (n < N || Sys::KEYED) {
          skey[n] = total_order_key(val);
          if (a.trace.values) a.trace.values[tslot * M + n] = val;
        } else {
          zero_value = val;                                   // n == N, deterministic System, iteration 0: thread N % THREADS
          for (int j = N; j < M; ++j) skey[j] = total_order_key(val);
        }
        if (a.trace.actions) {
          float* dst = a.trace.actions + (tslot * M + n) * D;
          for (int d = 0; d < D; ++d) dst[d] = (n < N) ? row[(d % A) * H + d / A] : 0.0f;
        }
      }
      __syncthreads();
      if (!Sys::KEYED && (a.trace.values || a.trace.actions)) {   // the zero rows' dumps (one value serves them all)
        const float zv = value_of_key(skey[N]);
        for (int j = N + tid; j < M; j += THREADS) {
          if (a.trace.values) a.trace.values[tslot * M + j] = zv;
          if (a.trace.actions && !(j == N && it == 0)) {
            float* dst = a.trace.actions + (tslot * M + j) * D;
            for (int d = 0; d < D; ++d) dst[d] = 0.0f;
          }
        }
      }
      (void)zero_value;
      cta_select_refit<THREADS>(rs, skey, elite_idx, sel_idx, scratch, elem, mean, std_, best_seq, best_value);
      if (a.trace.elite_idx)
        for (int e = tid; e < K; e += THREADS) a.trace.elite_idx[tslot * K + e] = elite_idx[e];
      for (int d = tid; d < D; d += THREADS) {
        if (a.trace.mean) a.trace.mean[tslot * D + d] = mean[d];
        if (a.trace.std) a.trace.std[tslot * D + d] = std_[d];
      }
      if (a.trace.best_value && tid == 0) a.trace.best_value[tslot] = *best_value;
      __syncthreads();
    }
    for (int d = tid; d < D; d += THREADS) a.best_seq_out[static_cast<size_t>(b) * D + d] = best_seq[d];
    if (tid == 0) {
      a.best_value_out[b] = *best_value;
      a.key_out[2 * b] = k_new.k0;
      a.key_out[2 * b + 1] = k_new.k1;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// Staged kernels
// ------------------------------------------------------------------------------------------

// Per-bin noise multipliers (fill_noise_scale) passed by value: the staged kernels need no
// device allocation and the table is read straight from the constant bank.
struct ScaleTable {
  float v[MBPO_MAX_FREQ];
};

constexpr int STAGED_THREADS = 128;  // block size of the staged sampling kernels

// vmap(powerlaw_psd_gaussian): one thread per key.
template <int H, int PRNG>
__global__ void __launch_bounds__(STAGED_THREADS) powerlaw_noise_kernel(const __grid_constant__ ScaleTable tbl, const uint32_t* __restrict__ keys, int M,
                                      float* __restrict__ out, uint32_t* __restrict__ bits_out) {
  __shared__ float stage[STAGED_THREADS][H | 1];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  Key2 k{keys[2 * i], keys[2 * i + 1]};
  float* row = out + static_cast<size_t>(i) * H;
  colored_noise_row<H, PRNG>(k, tbl.v, stage[threadIdx.x],
                             bits_out ? bits_out + static_cast<size_t>(i) * 2 * NoiseShape<H>::F : nullptr,
                             [&](int t, float y) { row[t] = y; });
}

// One iCEM iteration of key plumbing + sampling for B problems (icem_optimizer.py:174-192).
// grid = (ceil((N+Np)*A / blockDim), B); thread = (candidate n, action dim a).
template <int H, int PRNG>
__global__ void __launch_bounds__(STAGED_THREADS) sample_actions_kernel(const __grid_constant__ ScaleTable tbl, const uint32_t* __restrict__ carry_key,
                                      const float* __restrict__ mean, const float* __restrict__ std_, int N, int Np,
                                      int A, float u_min, float u_max, float* __restrict__ actions,
                                      uint32_t* __restrict__ next_key, uint32_t* __restrict__ particle_keys) {
  __shared__ float stage[STAGED_THREADS][H | 1];
  const int b = blockIdx.y;
  const int M = N + Np;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * A) return;
  const int n = idx / A, ad = idx % A;
  Key2 ck{carry_key[2 * b], carry_key[2 * b + 1]}, sampling_rng, particles_rng;
  split2<PRNG>(ck, sampling_rng, particles_rng);                                                          // :174
  if (ad == 0 && particle_keys) {
    const Key2 pk = split_at<PRNG>(particles_rng, static_cast<uint32_t>(M), static_cast<uint32_t>(n));   // :177
    particle_keys[(static_cast<size_t>(b) * M + n) * 2] = pk.k0;
    particle_keys[(static_cast<size_t>(b) * M + n) * 2 + 1] = pk.k1;
  }
  if (idx == 0) {
    const Key2 nk = split_at<PRNG>(sampling_rng, static_cast<uint32_t>(N + 1), 0u);                       // :176
    next_key[2 * b] = nk.k0;
    next_key[2 * b + 1] = nk.k1;
  }
  float* row = actions + (static_cast<size_t>(b) * M + n) * H * A + ad;  // element t at row[t*A]
  if (n >= N) {  // kept-elite rows: closure zeros (:192,:245)
    for (int t = 0; t < H; ++t) row[static_cast<size_t>(t) * A] = 0.0f;
    return;
  }
  const Key2 sk = split_at<PRNG>(sampling_rng, static_cast<uint32_t>(N + 1), static_cast<uint32_t>(n + 1));
  const Key2 dk = split_at<PRNG>(sk, static_cast<uint32_t>(A), static_cast<uint32_t>(ad));                // :180
  const float* mrow = mean + static_cast<size_t>(b) * H * A + ad;
  const float* srow = std_ + static_cast<size_t>(b) * H * A + ad;
  colored_noise_row<H, PRNG>(dk, tbl.v, stage[threadIdx.x], nullptr, [&](int t, float y) {
    const float v = __fadd_rn(mrow[static_cast<size_t>(t) * A], __fmul_rn(y, srow[static_cast<size_t>(t) * A]));
    row[static_cast<size_t>(t) * A] = fminf(fmaxf(v, u_min), u_max);
  });
}

// ---- any horizon (runtime H): same key tree and operation order, rolled loops (noise.cuh) --------------
// `stage` is dynamic shared memory: blockDim.x rows of (H | 1) floats.
template <int PRNG>
__global__ void __launch_bounds__(STAGED_THREADS)
    powerlaw_noise_rt_kernel(const __grid_constant__ ScaleTable tbl, const __grid_constant__ TwiddleTable tw, int H,
                             const uint32_t* __restrict__ keys, int M, float* __restrict__ out,
                             uint32_t* __restrict__ bits_out) {
  extern __shared__ __align__(16) float stage_rt[];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  Key2 k{keys[2 * i], keys[2 * i + 1]};
  float* row = out + static_cast<size_t>(i) * H;
  colored_noise_row_rt<PRNG>(H, k, tbl.v, tw, stage_rt + static_cast<size_t>(threadIdx.x) * (H | 1),
                             bits_out ? bits_out + static_cast<size_t>(i) * 2 * (H / 2 + 1) : nullptr,
                             [&](int t, float y) { row[t] = y; });
}

template <int PRNG>
__global__ void __launch_bounds__(STAGED_THREADS)
    sample_actions_rt_kernel(const __grid_constant__ ScaleTable tbl, const __grid_constant__ TwiddleTable tw, int H,
                             const uint32_t* __restrict__ carry_key, const float* __restrict__ mean,
                             const float* __restrict__ std_, int N, int Np, int A, float u_min, float u_max,
                             float* __restrict__ actions, uint32_t* __restrict__ next_key,
                             uint32_t* __restrict__ particle_keys) {
  extern __shared__ __align__(16) float stage_rt[];
  const int b = blockIdx.y;
  const int M = N + Np;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * A) return;
  const int n = idx / A, ad = idx % A;
  Key2 ck{carry_key[2 * b], carry_key[2 * b + 1]}, sampling_rng, particles_rng;
  split2<PRNG>(ck, sampling_rng, particles_rng);                                                          // :174
  if (ad == 0 && particle_keys) {
    const Key2 pk = split_at<PRNG>(particles_rng, static_cast<uint32_t>(M), static_cast<uint32_t>(n));   // :177
    particle_keys[(static_cast<size_t>(b) * M + n) * 2] = pk.k0;
    particle_keys[(static_cast<size_t>(b) * M + n) * 2 + 1] = pk.k1;
  }
  if (idx == 0) {
    const Key2 nk = split_at<PRNG>(sampling_rng, static_cast<uint32_t>(N + 1), 0u);                       // :176
    next_key[2 * b] = nk.k0;
    next_key[2 * b + 1] = nk.k1;
  }
  float* row = actions + (static_cast<size_t>(b) * M + n) * H * A + ad;  // element t at row[t*A]
  if (n >= N) {  // kept-elite rows: closure zeros (:192,:245)
    for (int t = 0; t < H; ++t) row[static_cast<size_t>(t) * A] = 0.0f;
    return;
  }
  const Key2 sk = split_at<PRNG>(sampling_rng, static_cast<uint32_t>(N + 1), static_cast<uint32_t>(n + 1));
  const Key2 dk = split_at<PRNG>(sk, static_cast<uint32_t>(A), static_cast<uint32_t>(ad));                // :180
  const float* mrow = mean + static_cast<size_t>(b) * H * A + ad;
  const float* srow = std_ + static_cast<size_t>(b) * H * A + ad;
  colored_noise_row_rt<PRNG>(H, dk, tbl.v, tw, stage_rt + static_cast<size_t>(threadIdx.x) * (H | 1), nullptr,
                             [&](int t, float y) {
    const float v = __fadd_rn(mrow[static_cast<size_t>(t) * A], __fmul_rn(y, srow[static_cast<size_t>(t) * A]));
    row[static_cast<size_t>(t) * A] = fminf(fmaxf(v, u_min), u_max);
  });
}

}  // namespace mbpo
