// Horizon-independent staged kernels behind the per-stage C ABI: System.step, rollout_actions,
// elite select + refit, the staged-plan prologue.  Included by mbpo_b200.cu only.
//
// Reference: mbpo/systems/pendulum_system.py:18-39, mbpo/utils/optimizer_utils.py:11-59,
// mbpo/optimizers/trajectory_optimizers/icem_optimizer.py:199-226,235-249.
#pragma once
#include "icem_kernels.cuh"

namespace mbpo {

// vmap(System.step): one thread per row.
template <int MATH>
__global__ void system_step_pendulum_kernel(const MbpoPendulumParams sys, const float* __restrict__ x,
                                            const float* __restrict__ u, int R, float* __restrict__ x_next,
                                            float* __restrict__ reward) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R) return;
  const PendulumConsts pc(sys);
  float c = x[3 * i], s = x[3 * i + 1], w = x[3 * i + 2], r;
  if (MATH == MBPO_MATH_REFERENCE) {
    pendulum_step_ref(pc, c, s, w, u[i], r);
  } else {
    float th = atan2_bounded(s, c);
    pendulum_step_theta(pc, th, w, u[i], r);
    sincos_bounded(th, s, c);
  }
  x_next[3 * i] = c; x_next[3 * i + 1] = s; x_next[3 * i + 2] = w;
  reward[i] = r;
}

// vmap(vmap(rollout_actions)) for the pendulum: one thread per action row.  A warp's 32 rows
// are contiguous in HBM (32*H floats); the warp stages them through shared memory with
// coalesced 128-bit loads so the stream runs at full sector efficiency, then each thread
// walks its own row (odd stride: conflict-free).  Optional Transition buffers are written
// from registers.
template <int MATH>
__global__ void __launch_bounds__(128) rollout_actions_pendulum_kernel(
    const MbpoPendulumParams sys, int H, const float* __restrict__ x0, const float* __restrict__ actions, int B,
    int M, float* __restrict__ returns_out, float* __restrict__ obs_out, float* __restrict__ reward_out,
    float* __restrict__ next_obs_out) {
  extern __shared__ __align__(16) float stage[];  // [warps][32*HS]
  const int HS = H | 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long total = static_cast<long long>(B) * M;
  const long long row0 = (static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + warp) * 32;
  if (row0 >= total) return;
  float* tile = stage + static_cast<size_t>(warp) * 32 * HS;
  const long long rows_here = (total - row0) < 32 ? (total - row0) : 32;
  const long long nfl = rows_here * H;
  const float* src = actions + row0 * H;
  // coalesced copy; 128-bit when the tile start is 16-byte aligned
  if (((row0 * H) & 3) == 0) {
    const float4* src4 = reinterpret_cast<const float4*>(src);
    const long long n4 = nfl >> 2;
    for (long long q = lane; q < n4; q += 32) {
      const float4 v = __ldg(src4 + q);
      const long long e = q << 2;
      const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const long long ee = e + k;
        tile[(ee / H) * HS + (ee % H)] = vv[k];
      }
    }
    for (long long e = (n4 << 2) + lane; e < nfl; e += 32) tile[(e / H) * HS + (e % H)] = __ldg(src + e);
  } else {
    for (long long e = lane; e < nfl; e += 32) tile[(e / H) * HS + (e % H)] = __ldg(src + e);
  }
  __syncwarp();
  const long long r = row0 + lane;
  if (r >= total) return;
  const int b = static_cast<int>(r / M);
  const PendulumConsts pc(sys);
  const float* row = tile + lane * HS;
  float c = x0[3 * b], s = x0[3 * b + 1], w = x0[3 * b + 2];
  const bool full = (obs_out != nullptr) || (reward_out != nullptr) || (next_obs_out != nullptr);
  if (!full) {
    const float ret = rollout_return<MATH>(pc, c, s, w, H, [&](int t) { return row[t]; });
    if (returns_out) returns_out[r] = ret;
    return;
  }
  float acc = 0.0f;
  float th = (MATH == MBPO_MATH_REFERENCE) ? 0.0f : atan2_bounded(s, c);
  for (int t = 0; t < H; ++t) {
    const size_t o = (static_cast<size_t>(r) * H + t);
    if (obs_out) { obs_out[o * 3] = c; obs_out[o * 3 + 1] = s; obs_out[o * 3 + 2] = w; }
    float rew;
    if (MATH == MBPO_MATH_REFERENCE) {
      pendulum_step_ref(pc, c, s, w, row[t], rew);
    } else {
      pendulum_step_theta(pc, th, w, row[t], rew);
      sincos_bounded(th, s, c);
    }
    if (reward_out) reward_out[o] = rew;
    if (next_obs_out) { next_obs_out[o * 3] = c; next_obs_out[o * 3 + 1] = s; next_obs_out[o * 3 + 2] = w; }
    acc = __fadd_rn(acc, rew);
  }
  if (returns_out) returns_out[r] = __fdiv_rn(acc, static_cast<float>(H));
}

// Stage 3 standalone: one CTA per problem; keys staged in shared memory, rows read from HBM.
constexpr int REFIT_THREADS = 128;

__global__ void __launch_bounds__(REFIT_THREADS) elite_refit_kernel(
    RefitScalars rs, const float* __restrict__ actions, const float* __restrict__ values,
    const float* __restrict__ mean_in, const float* __restrict__ std_in, const float* __restrict__ best_value_in,
    const float* __restrict__ best_seq_in, float* mean_out, float* std_out, float* best_value_out,
    float* best_seq_out, int* elite_idx_out) {
  extern __shared__ __align__(16) uint32_t refit_sm[];
  const int b = blockIdx.x, tid = threadIdx.x;
  uint32_t* keys = refit_sm;                             // [M]
  int* elite_idx = reinterpret_cast<int*>(keys + rs.M);  // [K]
  int* sel_idx = elite_idx + rs.K;                       // [K]
  uint32_t* scratch = reinterpret_cast<uint32_t*>(sel_idx + rs.K);
  float* mean = reinterpret_cast<float*>(scratch + select_scratch_words(rs.K, rs.M));
  float* std_ = mean + rs.D;
  float* best_seq = std_ + rs.D;
  float* best_value = best_seq + rs.D;
  for (int i = tid; i < rs.M; i += REFIT_THREADS) keys[i] = total_order_key(values[static_cast<size_t>(b) * rs.M + i]);
  for (int d = tid; d < rs.D; d += REFIT_THREADS) {
    mean[d] = mean_in[static_cast<size_t>(b) * rs.D + d];
    std_[d] = std_in[static_cast<size_t>(b) * rs.D + d];
    best_seq[d] = best_seq_in[static_cast<size_t>(b) * rs.D + d];
  }
  if (tid == 0) *best_value = best_value_in[b];
  __syncthreads();
  const float* rows = actions + static_cast<size_t>(b) * rs.M * rs.D;
  cta_select_refit<REFIT_THREADS>(rs, keys, elite_idx, sel_idx, scratch,
                                  [&](int i, int d) { return __ldg(rows + static_cast<size_t>(i) * rs.D + d); }, mean,
                                  std_, best_seq, best_value);
  for (int d = tid; d < rs.D; d += REFIT_THREADS) {
    mean_out[static_cast<size_t>(b) * rs.D + d] = mean[d];
    std_out[static_cast<size_t>(b) * rs.D + d] = std_[d];
    best_seq_out[static_cast<size_t>(b) * rs.D + d] = best_seq[d];
  }
  if (tid == 0) best_value_out[b] = *best_value;
  if (elite_idx_out)
    for (int e = tid; e < rs.K; e += REFIT_THREADS) elite_idx_out[static_cast<size_t>(b) * rs.K + e] = elite_idx[e];
}

// Warm-start prologue of optimize (:235-249) for the staged plan.
template <int PRNG>
__global__ void plan_prologue_kernel(int B, int D, int A, int warm_start, float init_std,
                                     const uint32_t* __restrict__ key_in, const float* __restrict__ best_seq_in,
                                     uint32_t* carry_key, uint32_t* key_out, float* mean, float* std_, float* best_seq,
                                     float* best_value) {
  const int b = blockIdx.x;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float m = 0.0f;
    if (warm_start) {
      const int src = (d + A < D) ? d + A : (D - A + d % A);  // shift one step, repeat the last action
      m = best_seq_in[static_cast<size_t>(b) * D + src];
    }
    mean[static_cast<size_t>(b) * D + d] = m;
    std_[static_cast<size_t>(b) * D + d] = init_std;
    best_seq[static_cast<size_t>(b) * D + d] = m;
  }
  if (threadIdx.x == 0) {
    best_value[b] = __int_as_float(0xFF800000);
    Key2 k{key_in[2 * b], key_in[2 * b + 1]}, k_opt, k_new;
    split2<PRNG>(k, k_opt, k_new);
    carry_key[2 * b] = k_opt.k0; carry_key[2 * b + 1] = k_opt.k1;
    key_out[2 * b] = k_new.k0; key_out[2 * b + 1] = k_new.k1;
  }
}

// jnp.mean / jnp.max over P identical particles applied to a returns buffer.
__global__ void summarize_particles_kernel(float* values, long long n, int P, int summarize) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) values[i] = summarize_particles(values[i], P, summarize);
}

// iCemTO.objective's tail (icem_optimizer.py:158-166) for a deterministic System, whose P particles are
// identical: values[i] = summarize(reward_i) - lambda * relu(summarize_cost(cost_i)).  cost may be null.
__global__ void penalize_kernel(float* values, const float* __restrict__ cost, long long n, int P,
                                int summarize_reward, int summarize_cost, float lambda) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float v = summarize_particles(values[i], P, summarize_reward);
  if (cost) {
    const float c = summarize_particles(cost[i], P, summarize_cost);
    v = __fsub_rn(v, __fmul_rn(lambda, fmaxf(c, 0.0f)));
  }
  values[i] = v;
}

// The same tail over P distinct particles (a keyed System, or the ensemble's members): per particle the horizon mean
// of reward [n, P, H] (a left-to-right sum from 0, divided by H, as general_rollout and the ensemble kernels round
// it), then the left-to-right mean or the max over particles; the same for cost [n, P] (may be null).
__global__ void penalize_particles_kernel(float* __restrict__ values_out, const float* __restrict__ reward, int H,
                                          const float* __restrict__ cost, long long n, int P, int summarize_reward,
                                          int summarize_cost, float lambda) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* rw = reward + static_cast<size_t>(i) * P * H;
  float sum = 0.0f, mx = 0.0f;
  for (int p = 0; p < P; ++p) {
    float acc = 0.0f;
    for (int t = 0; t < H; ++t) acc = __fadd_rn(acc, __ldg(rw + static_cast<size_t>(p) * H + t));
    const float ret = __fdiv_rn(acc, static_cast<float>(H));
    sum = __fadd_rn(sum, ret);
    mx = (p == 0) ? ret : fmaxf(mx, ret);
  }
  float v = (summarize_reward == MBPO_SUMMARIZE_MAX) ? mx : __fdiv_rn(sum, static_cast<float>(P));
  if (cost) {
    float csum = 0.0f, cmx = 0.0f;
    for (int p = 0; p < P; ++p) {
      const float c = __ldg(cost + static_cast<size_t>(i) * P + p);
      csum = __fadd_rn(csum, c);
      cmx = (p == 0) ? c : fmaxf(cmx, c);
    }
    const float c = (summarize_cost == MBPO_SUMMARIZE_MAX) ? cmx : __fdiv_rn(csum, static_cast<float>(P));
    v = __fsub_rn(v, __fmul_rn(lambda, fmaxf(c, 0.0f)));
  }
  values_out[i] = v;
}

// jnp.clip(actions, u_min, u_max) with bounds broadcast to [H, A] (icem_optimizer.py:47-48,191): the N
// sampled rows of every problem; the kept-elite rows (n >= N) are not clipped (:192).
__global__ void clip_actions_kernel(float* actions, const float* __restrict__ u_min, const float* __restrict__ u_max,
                                    long long total, int M, int N, int D) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int d = static_cast<int>(i % D);
  const int m = static_cast<int>((i / D) % M);
  if (m < N) actions[i] = fminf(fmaxf(actions[i], u_min[d]), u_max[d]);
}

}  // namespace mbpo
