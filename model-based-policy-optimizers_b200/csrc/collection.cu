// C ABI of the SAC / PPO env rollouts (declared in include/mbpo_b200.h): mbpo_env_rollout and mbpo_env_unroll for
// the pendulum (env_kernels.cuh), mbpo_env_unroll_general and mbpo_actor_rollout_general for the general Systems
// (general_env_kernels.cuh), and BPTT's forward on them, mbpo_rollout_policy_general.  The pendulum's
// policy-in-the-loop entry points stay in mbpo_b200.cu: its tcgen05 kernels include mlp_tc_kernels.cuh, whose
// stage-4 kernel would otherwise be compiled into both units.  For the same reason (adjoint_kernels.cuh holds
// non-template kernels) the general Systems' adjoint, mbpo_rollout_adjoint_general, sits beside the pendulum's in
// mbpo_b200.cu.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>

#include "../../include/mbpo_b200.h"
#include "general_env_kernels.cuh"
#include "host_util.h"

using namespace mbpo;

namespace {

// The pendulum keeps its tuned entry points (mbpo_env_unroll, mbpo_actor_rollout(_extras)); the learned ensemble is
// not an env.
int collection_system(const char* what, int kind, int* X, int* A, bool* keyed) {
  if (kind == MBPO_SYSTEM_PENDULUM)
    return fail(MBPO_EINVAL, "%s: MBPO_SYSTEM_PENDULUM has its own entry points (mbpo_env_unroll, mbpo_env_rollout, "
                "mbpo_actor_rollout, mbpo_actor_rollout_extras)", what);
  if (general_system_dims(kind, X, A, keyed) != MBPO_OK)
    return fail(MBPO_EUNSUPPORTED, "%s: system_kind %d is not one of the general Systems (NOISY_PENDULUM, POINT_MASS)",
                what, kind);
  return MBPO_OK;
}

template <class Sys>
int launch_env_general(const GeneralEnvArgs& a, int prng_mode, cudaStream_t st) {
  const unsigned blocks = static_cast<unsigned>((a.E + GEN_ENV_THREADS - 1) / GEN_ENV_THREADS);
  return with_prng(prng_mode, [&](auto P) {
    env_unroll_general_kernel<Sys, P><<<blocks, GEN_ENV_THREADS, 0, st>>>(a);
    return check_launch("env_unroll_general_kernel");
  });
}

// Dynamic shared memory of the CUDA-core policy kernels for a network of num_hidden layers on an X -> 2A System.
template <class Sys>
GeneralActorSmem general_policy_smem(int num_hidden) {
  constexpr int X = Sys::X, A = Sys::A;
  GeneralActorSmem lay;
  int off = 0;
  auto take = [&](int n) { const int o = off; off += (n + 3) / 4 * 4; return o; };
  lay.w[0] = take(X * ACT_W);
  for (int l = 1; l < num_hidden; ++l) lay.w[l] = take(ACT_W * ACT_W);
  lay.w[num_hidden] = take(ACT_W * 2 * A);
  for (int l = 0; l < num_hidden; ++l) lay.b[l] = take(ACT_W);
  lay.b[num_hidden] = take(2 * A);
  lay.h = take(ACT_W * GEN_ACT_THREADS);
  lay.total = off;
  return lay;
}

// One launch of a CUDA-core policy kernel (actor_rollout_general_kernel / rollout_policy_general_kernel): E threads
// in blocks of GEN_ACT_THREADS, with the dynamic shared memory `lay` asks for.
template <class Kernel, class Args>
int launch_general_policy_kernel(Kernel kernel, const char* what, const Args& a, const GeneralActorSmem& lay,
                                 cudaStream_t st) {
  const size_t smem = static_cast<size_t>(lay.total) * sizeof(float);
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             static_cast<int>(smem));
  if (e != cudaSuccess) return fail(MBPO_ECUDA, "%s: smem attribute (%zu B): %s", what, smem, cudaGetErrorString(e));
  const unsigned blocks = static_cast<unsigned>((a.E + GEN_ACT_THREADS - 1) / GEN_ACT_THREADS);
  kernel<<<blocks, GEN_ACT_THREADS, smem, st>>>(a, lay);
  return MBPO_OK;
}

template <class Sys>
int launch_actor_general(const GeneralActorArgs& a, int prng_mode, cudaStream_t st) {
  const GeneralActorSmem lay = general_policy_smem<Sys>(a.num_hidden);
  return with_prng(prng_mode, [&](auto P) {
    const int rc = launch_general_policy_kernel(actor_rollout_general_kernel<Sys, P>, "actor_rollout_general", a,
                                                lay, st);
    return rc != MBPO_OK ? rc : check_launch("actor_rollout_general_kernel");
  });
}

template <class Sys>
int launch_rollout_policy_general(const GeneralPolicyArgs& a, int prng_mode, cudaStream_t st) {
  const GeneralActorSmem lay = general_policy_smem<Sys>(a.num_hidden);
  return with_prng(prng_mode, [&](auto P) {
    const int rc = launch_general_policy_kernel(rollout_policy_general_kernel<Sys, P>, "rollout_policy_general", a,
                                                lay, st);
    return rc != MBPO_OK ? rc : check_launch("rollout_policy_general_kernel");
  });
}

// The pendulum's env rollouts.  With every Transition buffer but `observation` present: the segmented / FAST
// kernel; otherwise the general kernel, which takes NULL outputs.
int launch_env(int system_kind, const void* sys_params_host, int math_mode, int x_dim, int action_dim,
               int episode_length, int action_repeat, const float* obs_in, const float* steps_in,
               const float* done_in, float* obs, float* steps, float* done, const float* first_obs,
               const float* actions, int E, int T, float* observation_out, float* reward_out, float* discount_out,
               float* next_observation_out, float* truncation_out, bool segmented, void* stream) {
  if (system_kind != MBPO_SYSTEM_PENDULUM)
    return fail(MBPO_EUNSUPPORTED, "env_rollout: only MBPO_SYSTEM_PENDULUM has an inlined step");
  MBPO_REQUIRE(action_dim == 1 && x_dim == 3, "env_rollout: pendulum needs action_dim == 1, x_dim == 3");
  MBPO_REQUIRE(math_mode == 0 || math_mode == 1, "env_rollout: bad math_mode %d", math_mode);
  MBPO_REQUIRE(episode_length >= 1 && action_repeat >= 1, "env_rollout: episode_length/action_repeat < 1");
  MBPO_REQUIRE(E >= 0 && T >= 0, "env_rollout: negative size");
  if (E == 0 || T == 0) return MBPO_OK;     // empty arrays have no address
  MBPO_REQUIRE(sys_params_host && obs_in && steps_in && done_in && obs && steps && done && first_obs && actions,
               "env_rollout: null pointer");
  const MbpoPendulumParams& sys = *static_cast<const MbpoPendulumParams*>(sys_params_host);
  const unsigned env_blocks = static_cast<unsigned>((E + ENV_THREADS - 1) / ENV_THREADS);
  cudaStream_t st = as_stream(stream);
  const bool all_out = reward_out && discount_out && next_observation_out && truncation_out;
  if (!all_out) {
    static_assert(GEN_ENV_THREADS == ENV_THREADS, "the pendulum's env kernels run 64 envs per block");
    GeneralEnvArgs g = {};
    g.sys.pendulum = sys;
    g.E = E; g.T = T; g.episode_length = episode_length; g.action_repeat = action_repeat;
    g.obs_in = obs_in; g.steps_in = steps_in; g.done_in = done_in;
    g.obs_out = obs; g.steps_out = steps; g.done_out = done; g.first_obs = first_obs; g.actions = actions;
    g.observation_out = observation_out; g.reward_out = reward_out; g.discount_out = discount_out;
    g.next_observation_out = next_observation_out; g.truncation_out = truncation_out;
    if (math_mode == MBPO_MATH_REFERENCE) env_unroll_general_kernel<PendulumSys, 0><<<env_blocks, ENV_THREADS, 0, st>>>(g);
    else env_unroll_general_kernel<PendulumThetaSys, 0><<<env_blocks, ENV_THREADS, 0, st>>>(g);
    return check_launch("env_unroll_general_kernel");
  }
  EnvArgs a;
  a.sys = sys;
  a.E = E; a.T = T; a.episode_length = episode_length; a.action_repeat = action_repeat;
  a.obs_in = obs_in; a.steps_in = steps_in; a.done_in = done_in;
  a.obs = obs; a.steps = steps; a.done = done; a.first_obs = first_obs; a.actions = actions;
  a.observation_out = observation_out; a.reward_out = reward_out; a.discount_out = discount_out;
  a.next_observation_out = next_observation_out; a.truncation_out = truncation_out;
  // pieces between AutoReset points (env_kernels.cuh): the first is at least one step long
  const long long len = (static_cast<long long>(episode_length) + action_repeat - 1) / action_repeat;
  long long pieces = 1 + (static_cast<long long>(T) - 1 + len - 1) / len;
  if (pieces > 65535) pieces = 1;
  a.segmented = (segmented && pieces > 1) ? 1 : 0;
  if (a.segmented)
    MBPO_REQUIRE(obs != obs_in && steps != steps_in && done != done_in,
                 "env_unroll: the outgoing env state must not alias the incoming one");
  const dim3 blocks(env_blocks, a.segmented ? static_cast<unsigned>(pieces) : 1u);
  const bool fast = action_repeat == 1 && std::fabs(a.sys.target_angle) <= 6.0f && E % 4 == 0 &&
                    aligned16(next_observation_out) && aligned16(observation_out) &&
                    static_cast<long long>(T) * E * 3 < (1ll << 31);
  const auto launch = [&](auto math, auto obs_out, auto fast_loop) {
    env_rollout_pendulum_kernel<math, obs_out, fast_loop><<<blocks, ENV_THREADS, 0, st>>>(a);
    return check_launch("env_rollout_pendulum_kernel");
  };
  using Yes = std::true_type;
  using No = std::false_type;
  return with_math(math_mode, [&](auto M) {
    if (observation_out) return fast ? launch(M, Yes{}, Yes{}) : launch(M, Yes{}, No{});
    return fast ? launch(M, No{}, Yes{}) : launch(M, No{}, No{});
  });
}

}  // namespace

int mbpo_env_rollout(int system_kind, const void* sys_params_host, int math_mode, int x_dim, int action_dim,
                     int episode_length, int action_repeat, float* obs, float* steps, float* done,
                     const float* first_obs, const float* actions, int E, int T, float* observation_out,
                     float* reward_out, float* discount_out, float* next_observation_out, float* truncation_out,
                     void* stream) {
  return launch_env(system_kind, sys_params_host, math_mode, x_dim, action_dim, episode_length, action_repeat, obs,
                    steps, done, obs, steps, done, first_obs, actions, E, T, observation_out, reward_out,
                    discount_out, next_observation_out, truncation_out, false, stream);
}

int mbpo_env_unroll(int system_kind, const void* sys_params_host, int math_mode, int x_dim, int action_dim,
                    int episode_length, int action_repeat, const float* obs_in, const float* steps_in,
                    const float* done_in, float* obs_out, float* steps_out, float* done_out,
                    const float* first_obs, const float* actions, int E, int T, float* observation_out,
                    float* reward_out, float* discount_out, float* next_observation_out, float* truncation_out,
                    void* stream) {
  return launch_env(system_kind, sys_params_host, math_mode, x_dim, action_dim, episode_length, action_repeat,
                    obs_in, steps_in, done_in, obs_out, steps_out, done_out, first_obs, actions, E, T,
                    observation_out, reward_out, discount_out, next_observation_out, truncation_out, true, stream);
}

int mbpo_env_unroll_general(int system_kind, const MbpoGeneralSystemParams* params_host, int prng_mode,
                            int episode_length, int action_repeat, const float* obs_in, const float* steps_in,
                            const float* done_in, const uint32_t* sys_keys_in, float* obs_out, float* steps_out,
                            float* done_out, uint32_t* sys_keys_out, const float* first_obs, const float* actions,
                            int E, int T, float* observation_out, float* reward_out, float* discount_out,
                            float* next_observation_out, float* truncation_out, void* stream) {
  int X, A;
  bool keyed;
  const int rc = collection_system("env_unroll_general", system_kind, &X, &A, &keyed);
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
  return with_system<NoisyPendulumSys, PointMassSys>(system_kind, [&](auto t) {
    return launch_env_general<typename decltype(t)::type>(a, prng_mode, st);
  });
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
  int rc = collection_system("actor_rollout_general", system_kind, &X, &A, &keyed);
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
  GeneralActorArgs a;
  rc = fill_policy("actor_rollout_general", policy_host, E, X, A, a);
  if (rc != MBPO_OK) return rc;
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
  a.sys = *params_host;
  a.E = E; a.T = T; a.episode_length = episode_length; a.action_repeat = action_repeat;
  a.deterministic = deterministic; a.key_convention = key_convention;
  a.key_in = key_in; a.key_out = key_out;
  a.obs = obs; a.steps = steps; a.done = done; a.sys_keys_in = sys_keys_in; a.sys_keys_out = sys_keys_out;
  a.first_obs = first_obs;
  a.action_out = action_out; a.reward_out = reward_out; a.discount_out = discount_out;
  a.next_observation_out = next_observation_out; a.truncation_out = truncation_out;
  a.raw_action_out = deterministic ? nullptr : raw_action_out;
  a.log_prob_out = deterministic ? nullptr : log_prob_out;
  return with_system<NoisyPendulumSys, PointMassSys>(system_kind, [&](auto t) {
    return launch_actor_general<typename decltype(t)::type>(a, prng_mode, st);
  });
}

int mbpo_rollout_policy_general(int system_kind, const MbpoGeneralSystemParams* params_host, int prng_mode,
                                const MbpoPolicyParams* policy_host, int deterministic, int key_convention,
                                const uint32_t* key_in, const uint32_t* sys_keys_in, int sys_keys_shared,
                                const float* x0, int E, int T, float* action_out, float* reward_out,
                                float* next_observation_out, uint32_t* key_out, uint32_t* sys_keys_out, void* stream) {
  int X, A;
  bool keyed;
  int rc = collection_system("rollout_policy_general", system_kind, &X, &A, &keyed);
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(params_host && policy_host && key_in, "rollout_policy_general: null pointer");
  MBPO_REQUIRE(prng_mode == 0 || prng_mode == 1, "rollout_policy_general: bad prng_mode %d", prng_mode);
  MBPO_REQUIRE(key_convention >= 0 && key_convention <= 2, "rollout_policy_general: bad key_convention %d",
               key_convention);
  MBPO_REQUIRE(E >= 0 && T >= 0, "rollout_policy_general: negative size");
  MBPO_REQUIRE(policy_host->head == MBPO_HEAD_NORMAL_TANH || policy_host->head == MBPO_HEAD_BPTT_ACTOR,
               "rollout_policy_general: bad policy head %d", policy_host->head);
  MBPO_REQUIRE(policy_host->kernel >= MBPO_ACTOR_AUTO && policy_host->kernel <= MBPO_ACTOR_TCGEN05_WIDE,
               "rollout_policy_general: bad policy kernel selector %d", policy_host->kernel);
  if (policy_host->kernel == MBPO_ACTOR_TCGEN05 || policy_host->kernel == MBPO_ACTOR_TCGEN05_WIDE)
    return fail(MBPO_EUNSUPPORTED, "rollout_policy_general: the tcgen05 policy kernels hold the pendulum only; the "
                "general Systems run the CUDA-core kernel (MBPO_ACTOR_AUTO or MBPO_ACTOR_CUDA_CORES)");
  GeneralPolicyArgs a;
  rc = fill_policy("rollout_policy_general", policy_host, E, X, A, a);
  if (rc != MBPO_OK) return rc;
  const size_t sys_key_words = keyed ? (sys_keys_shared ? 2 : 2 * static_cast<size_t>(E)) : 0;
  MBPO_REQUIRE(sys_key_words == 0 || (sys_keys_in && sys_keys_out),
               "rollout_policy_general: this System draws from system_params.key: sys_keys_in / sys_keys_out are "
               "null");
  cudaStream_t st = as_stream(stream);
  if (E == 0 || T == 0) {        // empty arrays have no address; keys pass through
    int r = copy_async(key_out, key_in, key_out ? 2 * sizeof(uint32_t) : 0, st, "rollout_policy_general");
    if (r == MBPO_OK) r = copy_async(sys_keys_out, sys_keys_in, sizeof(uint32_t) * sys_key_words, st,
                                     "rollout_policy_general");
    return r;
  }
  MBPO_REQUIRE(x0 && action_out && reward_out && next_observation_out, "rollout_policy_general: null pointer");
  MBPO_REQUIRE(X != 4 || aligned16(next_observation_out),
               "rollout_policy_general: next_observation_out of a 4-float state must be 16-byte aligned");
  a.sys = *params_host;
  a.E = E; a.T = T;
  a.deterministic = deterministic; a.key_convention = key_convention;
  a.head = policy_host->head; a.shared_noise = policy_host->shared_noise;
  a.sig_bias = policy_host->sig_bias; a.sig_min = policy_host->sig_min; a.sig_max = policy_host->sig_max;
  a.action_clip = policy_host->action_clip;
  a.key_in = key_in; a.key_out = key_out;
  a.x0 = x0;
  a.sys_keys_in = sys_keys_in; a.sys_keys_out = sys_keys_out; a.sys_keys_shared = sys_keys_shared ? 1 : 0;
  a.action_out = action_out; a.reward_out = reward_out; a.next_observation_out = next_observation_out;
  return with_system<NoisyPendulumSys, PointMassSys>(system_kind, [&](auto t) {
    return launch_rollout_policy_general<typename decltype(t)::type>(a, prng_mode, st);
  });
}
