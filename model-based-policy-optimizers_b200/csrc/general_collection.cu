// C ABI of the SAC / PPO collection path for the general Systems (declared in include/mbpo_b200.h):
// mbpo_env_unroll_general and mbpo_actor_rollout_general, kernels in general_env_kernels.cuh.
#include <cuda_runtime.h>

#include <cstdint>

#include "../../include/mbpo_b200.h"
#include "general_env_kernels.cuh"
#include "host_util.h"

using namespace mbpo;

namespace {

// The Systems these entry points step.  The pendulum keeps its tuned entry points (mbpo_env_unroll,
// mbpo_actor_rollout(_extras)); the learned ensemble is not an env.
int collection_dims(const char* what, int kind, int* X, int* A, bool* keyed) {
  switch (kind) {
    case MBPO_SYSTEM_NOISY_PENDULUM: *X = 3; *A = 1; *keyed = true; return MBPO_OK;
    case MBPO_SYSTEM_POINT_MASS: *X = 4; *A = 2; *keyed = false; return MBPO_OK;
    case MBPO_SYSTEM_PENDULUM:
      return fail(MBPO_EINVAL, "%s: MBPO_SYSTEM_PENDULUM has its own entry points (mbpo_env_unroll, mbpo_env_rollout, "
                  "mbpo_actor_rollout, mbpo_actor_rollout_extras)", what);
    default:
      return fail(MBPO_EUNSUPPORTED, "%s: system_kind %d is not one of the general Systems (NOISY_PENDULUM, POINT_MASS)",
                  what, kind);
  }
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int copy_async(void* dst, const void* src, size_t bytes, cudaStream_t st, const char* what) {
  if (bytes == 0 || dst == src) return MBPO_OK;
  const cudaError_t ce = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, st);
  return ce == cudaSuccess ? MBPO_OK : fail(MBPO_ECUDA, "%s copy: %s", what, cudaGetErrorString(ce));
}

template <class Sys>
int launch_env_general(const GeneralEnvArgs& a, int prng_mode, cudaStream_t st) {
  const unsigned blocks = static_cast<unsigned>((a.E + GEN_ENV_THREADS - 1) / GEN_ENV_THREADS);
  if (prng_mode == 0) env_unroll_general_kernel<Sys, 0><<<blocks, GEN_ENV_THREADS, 0, st>>>(a);
  else env_unroll_general_kernel<Sys, 1><<<blocks, GEN_ENV_THREADS, 0, st>>>(a);
  return check_launch("env_unroll_general_kernel");
}

template <class Sys>
int launch_actor_general(const GeneralActorArgs& a, int prng_mode, cudaStream_t st) {
  constexpr int X = Sys::X, A = Sys::A;
  GeneralActorSmem lay;
  int off = 0;
  auto take = [&](int n) { const int o = off; off += (n + 3) / 4 * 4; return o; };
  lay.w[0] = take(X * ACT_W);
  for (int l = 1; l < a.num_hidden; ++l) lay.w[l] = take(ACT_W * ACT_W);
  lay.w[a.num_hidden] = take(ACT_W * 2 * A);
  for (int l = 0; l < a.num_hidden; ++l) lay.b[l] = take(ACT_W);
  lay.b[a.num_hidden] = take(2 * A);
  lay.h = take(ACT_W * GEN_ACT_THREADS);
  lay.total = off;
  const size_t smem = static_cast<size_t>(off) * sizeof(float);
  auto kernel = prng_mode == 0 ? actor_rollout_general_kernel<Sys, 0> : actor_rollout_general_kernel<Sys, 1>;
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  if (e != cudaSuccess)
    return fail(MBPO_ECUDA, "actor_rollout_general: smem attribute (%zu B): %s", smem, cudaGetErrorString(e));
  const unsigned blocks = static_cast<unsigned>((a.E + GEN_ACT_THREADS - 1) / GEN_ACT_THREADS);
  kernel<<<blocks, GEN_ACT_THREADS, smem, st>>>(a, lay);
  return check_launch("actor_rollout_general_kernel");
}

}  // namespace

int mbpo_env_unroll_general(int system_kind, const MbpoGeneralSystemParams* params_host, int prng_mode,
                            int episode_length, int action_repeat, const float* obs_in, const float* steps_in,
                            const float* done_in, const uint32_t* sys_keys_in, float* obs_out, float* steps_out,
                            float* done_out, uint32_t* sys_keys_out, const float* first_obs, const float* actions,
                            int E, int T, float* observation_out, float* reward_out, float* discount_out,
                            float* next_observation_out, float* truncation_out, void* stream) {
  int X, A;
  bool keyed;
  const int rc = collection_dims("env_unroll_general", system_kind, &X, &A, &keyed);
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(prng_mode == 0 || prng_mode == 1, "env_unroll_general: bad prng_mode %d", prng_mode);
  MBPO_REQUIRE(episode_length >= 1 && action_repeat >= 1, "env_unroll_general: episode_length/action_repeat < 1");
  MBPO_REQUIRE(E >= 0 && T >= 0, "env_unroll_general: negative size");
  if (E == 0) return MBPO_OK;     // empty arrays have no address
  MBPO_REQUIRE(params_host && obs_in && steps_in && done_in && obs_out && steps_out && done_out,
               "env_unroll_general: null pointer");
  MBPO_REQUIRE(!keyed || (sys_keys_in && sys_keys_out),
               "env_unroll_general: this System draws from system_params.key: sys_keys_in / sys_keys_out are null");
  cudaStream_t st = as_stream(stream);
  if (T == 0) {                   // the state passes through unchanged
    int r = copy_async(obs_out, obs_in, sizeof(float) * E * X, st, "env_unroll_general");
    if (r == MBPO_OK) r = copy_async(steps_out, steps_in, sizeof(float) * E, st, "env_unroll_general");
    if (r == MBPO_OK) r = copy_async(done_out, done_in, sizeof(float) * E, st, "env_unroll_general");
    if (r == MBPO_OK && keyed) r = copy_async(sys_keys_out, sys_keys_in, sizeof(uint32_t) * 2 * E, st, "env_unroll_general");
    return r;
  }
  MBPO_REQUIRE(first_obs && actions, "env_unroll_general: null pointer");
  MBPO_REQUIRE(X != 4 || ((!observation_out || aligned16(observation_out)) &&
                          (!next_observation_out || aligned16(next_observation_out))),
               "env_unroll_general: observation buffers of a 4-float state must be 16-byte aligned");
  GeneralEnvArgs a;
  a.sys = *params_host;
  a.E = E; a.T = T; a.episode_length = episode_length; a.action_repeat = action_repeat;
  a.obs_in = obs_in; a.steps_in = steps_in; a.done_in = done_in; a.keys_in = sys_keys_in;
  a.obs_out = obs_out; a.steps_out = steps_out; a.done_out = done_out; a.keys_out = sys_keys_out;
  a.first_obs = first_obs; a.actions = actions;
  a.observation_out = observation_out; a.reward_out = reward_out; a.discount_out = discount_out;
  a.next_observation_out = next_observation_out; a.truncation_out = truncation_out;
  if (system_kind == MBPO_SYSTEM_NOISY_PENDULUM) return launch_env_general<NoisyPendulumSys>(a, prng_mode, st);
  return launch_env_general<PointMassSys>(a, prng_mode, st);
}

int mbpo_actor_rollout_general(int system_kind, const MbpoGeneralSystemParams* params_host, int prng_mode,
                               const MbpoPolicyParams* policy_host, int deterministic, int key_convention,
                               const uint32_t* key_in, int episode_length, int action_repeat, float* obs, float* steps,
                               float* done, const uint32_t* sys_keys_in, uint32_t* sys_keys_out,
                               const float* first_obs, int E, int T, float* action_out, float* reward_out,
                               float* discount_out, float* next_observation_out, float* truncation_out,
                               uint32_t* key_out, float* raw_action_out, float* log_prob_out, void* stream) {
  int X, A;
  bool keyed;
  const int rc = collection_dims("actor_rollout_general", system_kind, &X, &A, &keyed);
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(params_host && policy_host && key_in, "actor_rollout_general: null pointer");
  MBPO_REQUIRE((raw_action_out == nullptr) == (log_prob_out == nullptr),
               "actor_rollout_general: raw_action_out and log_prob_out come together");
  MBPO_REQUIRE(prng_mode == 0 || prng_mode == 1, "actor_rollout_general: bad prng_mode %d", prng_mode);
  MBPO_REQUIRE(key_convention >= 0 && key_convention <= 2, "actor_rollout_general: bad key_convention %d",
               key_convention);
  MBPO_REQUIRE(E >= 0 && T >= 0 && episode_length >= 1 && action_repeat >= 1, "actor_rollout_general: bad sizes");
  MBPO_REQUIRE(policy_host->head == MBPO_HEAD_NORMAL_TANH || policy_host->head == MBPO_HEAD_BPTT_ACTOR,
               "actor_rollout_general: bad policy head %d", policy_host->head);
  MBPO_REQUIRE(policy_host->kernel >= MBPO_ACTOR_AUTO && policy_host->kernel <= MBPO_ACTOR_TCGEN05_WIDE,
               "actor_rollout_general: bad policy kernel selector %d", policy_host->kernel);
  if (policy_host->head != MBPO_HEAD_NORMAL_TANH || policy_host->shared_noise)
    return fail(MBPO_EUNSUPPORTED, "actor_rollout_general: the BPTT actor head (one shared draw) runs on the pendulum "
                "only; the general Systems take the NormalTanh head");
  if (policy_host->kernel == MBPO_ACTOR_TCGEN05 || policy_host->kernel == MBPO_ACTOR_TCGEN05_WIDE)
    return fail(MBPO_EUNSUPPORTED, "actor_rollout_general: the tcgen05 policy kernels hold the pendulum only; the "
                "general Systems run the CUDA-core kernel (MBPO_ACTOR_AUTO or MBPO_ACTOR_CUDA_CORES)");
  if (policy_host->hidden != ACT_W || policy_host->obs_dim != X || policy_host->action_dim != A ||
      policy_host->num_hidden < 1 || policy_host->num_hidden > ACT_MAX_HIDDEN)
    return fail(MBPO_EUNSUPPORTED,
                "actor_rollout_general: this System's policy kernel needs obs_dim == %d, action_dim == %d, 1..%d hidden "
                "layers of width %d (got obs %d, act %d, %d x %d)",
                X, A, ACT_MAX_HIDDEN, ACT_W, policy_host->obs_dim, policy_host->action_dim, policy_host->num_hidden,
                policy_host->hidden);
  for (int l = 0; l <= policy_host->num_hidden; ++l)
    MBPO_REQUIRE(policy_host->w[l] && policy_host->b[l], "actor_rollout_general: null policy weights (layer %d)", l);
  MBPO_REQUIRE((policy_host->obs_mean_dev == nullptr) == (policy_host->obs_std_dev == nullptr),
               "actor_rollout_general: obs_mean_dev and obs_std_dev come together");
  MBPO_REQUIRE(policy_host->draw_total == 0 ||
                   (policy_host->draw_offset >= 0 && policy_host->draw_offset + E <= policy_host->draw_total),
               "actor_rollout_general: envs [%d, %d) are not inside draw_total %d", policy_host->draw_offset,
               policy_host->draw_offset + E, policy_host->draw_total);
  MBPO_REQUIRE(!keyed || E == 0 || (sys_keys_in && sys_keys_out),
               "actor_rollout_general: this System draws from system_params.key: sys_keys_in / sys_keys_out are null");
  cudaStream_t st = as_stream(stream);
  if (E == 0 || T == 0) {        // empty arrays have no address; keys pass through
    int r = copy_async(key_out, key_in, key_out ? 2 * sizeof(uint32_t) : 0, st, "actor_rollout_general");
    if (r == MBPO_OK && keyed && E > 0)
      r = copy_async(sys_keys_out, sys_keys_in, sizeof(uint32_t) * 2 * E, st, "actor_rollout_general");
    return r;
  }
  MBPO_REQUIRE(obs && steps && done && first_obs, "actor_rollout_general: null pointer");
  MBPO_REQUIRE(action_out && reward_out && discount_out && next_observation_out && truncation_out,
               "actor_rollout_general: every Transition buffer is required");
  MBPO_REQUIRE(X != 4 || aligned16(next_observation_out),
               "actor_rollout_general: next_observation_out of a 4-float state must be 16-byte aligned");
  GeneralActorArgs a;
  a.sys = *params_host;
  a.E = E; a.T = T; a.episode_length = episode_length; a.action_repeat = action_repeat;
  a.num_hidden = policy_host->num_hidden; a.deterministic = deterministic; a.key_convention = key_convention;
  a.min_std = policy_host->min_std;
  a.normalize = policy_host->normalize;
  a.draw_total = policy_host->draw_total > 0 ? policy_host->draw_total : E;
  a.draw_offset = policy_host->draw_total > 0 ? policy_host->draw_offset : 0;
  for (int i = 0; i < 4; ++i) { a.obs_mean[i] = policy_host->obs_mean[i]; a.obs_std[i] = policy_host->obs_std[i]; }
  a.obs_mean_dev = policy_host->obs_mean_dev; a.obs_std_dev = policy_host->obs_std_dev;
  for (int l = 0; l <= ACT_MAX_HIDDEN; ++l) {
    a.w[l] = l <= a.num_hidden ? policy_host->w[l] : nullptr;
    a.b[l] = l <= a.num_hidden ? policy_host->b[l] : nullptr;
  }
  a.key_in = key_in; a.key_out = key_out;
  a.obs = obs; a.steps = steps; a.done = done; a.sys_keys_in = sys_keys_in; a.sys_keys_out = sys_keys_out;
  a.first_obs = first_obs;
  a.action_out = action_out; a.reward_out = reward_out; a.discount_out = discount_out;
  a.next_observation_out = next_observation_out; a.truncation_out = truncation_out;
  a.raw_action_out = deterministic ? nullptr : raw_action_out;
  a.log_prob_out = deterministic ? nullptr : log_prob_out;
  if (system_kind == MBPO_SYSTEM_NOISY_PENDULUM) return launch_actor_general<NoisyPendulumSys>(a, prng_mode, st);
  return launch_actor_general<PointMassSys>(a, prng_mode, st);
}
