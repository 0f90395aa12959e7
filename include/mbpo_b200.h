/*
 * mbpo_b200.h -- C ABI of the B200-native iCEM planning hot path.
 *
 * Drop-in boundary for lasgroup/Model-based-policy-optimizers (reference paths below are
 * relative to the reference repository root).  The reference has no FFI of its own (it
 * is pure JAX); every entry point here replaces one jitted Python function, and the
 * Python host package (model-based-policy-optimizers_b200/mbpo_b200) binds them with
 * ctypes behind the reference's unchanged call signatures.  See INTEGRATION.md.
 *
 * Conventions
 *   - All pointers are DEVICE pointers unless the name ends in _host.
 *   - All arrays are dense row-major with the shapes in the comments; float = IEEE
 *     binary32, keys = uint32[2] (JAX threefry key data).
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on that
 *     stream, never synchronises the device, and allocates no device memory.
 *   - Return value: 0 (MBPO_OK) or a negative MBPO_E* code; the message is available
 *     from mbpo_last_error() (thread local).  There is NO CPU fallback.
 */
#ifndef MBPO_B200_H_
#define MBPO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MBPO_ABI_VERSION 1
#define MBPO_MAX_HORIZON 128
#define MBPO_MAX_FREQ (MBPO_MAX_HORIZON / 2 + 1)

enum {
  MBPO_OK = 0,
  MBPO_EINVAL = -1,      /* bad shape / null pointer / inconsistent config */
  MBPO_EUNSUPPORTED = -2,/* unsupported system_kind / horizon / action_dim for this kernel */
  MBPO_ECUDA = -3,       /* CUDA runtime error (launch, attribute)          */
  MBPO_EWORKSPACE = -4   /* caller workspace too small                      */
};

enum { MBPO_PRNG_LEGACY = 0, MBPO_PRNG_PARTITIONABLE = 1 }; /* jax_threefry_partitionable */
enum { MBPO_SUMMARIZE_MEAN = 0, MBPO_SUMMARIZE_MAX = 1 };   /* icem_optimizer.py:112-115 */
/* 2, 3: the general Systems (csrc/systems.cuh) -- a pendulum whose transition is SAMPLED with the System's own key
 * (the per-particle key of icem_optimizer.py:146-156) and a two-action point mass (action_dim > 1, :180). */
enum { MBPO_SYSTEM_PENDULUM = 0, MBPO_SYSTEM_MLP_ENSEMBLE = 1, MBPO_SYSTEM_NOISY_PENDULUM = 2,
       MBPO_SYSTEM_POINT_MASS = 3 };
/* MBPO_MATH_REFERENCE follows pendulum_dynamics.py:35,43 literally (theta re-derived with
 * atan2 from [cos, sin] every step).  MBPO_MATH_THETA_CARRY keeps theta in a register and
 * wraps it to (-pi, pi]; mathematically identical, rounding differs (see DESIGN.md). */
enum { MBPO_MATH_REFERENCE = 0, MBPO_MATH_THETA_CARRY = 1 };

/* PendulumDynamicsParams (mbpo/systems/dynamics/pendulum_dynamics.py:12-19) followed by
 * PendulumRewardParams (mbpo/systems/rewards/pendulum_reward.py:12-16), same order. */
typedef struct MbpoPendulumParams {
  float max_speed, max_torque, dt, g, m, l;
  float control_cost, angle_cost, target_angle;
} MbpoPendulumParams;

/* Parameters of the general Systems: MBPO_SYSTEM_NOISY_PENDULUM reads `pendulum` and `noise_std` (the scale of the
 * Normal that PendulumDynamics.next_state returns, pendulum_dynamics.py:45-46 -- 0 in the reference);
 * MBPO_SYSTEM_POINT_MASS reads `point_mass` (state [px, py, vx, vy], action [ax, ay]). */
typedef struct MbpoPointMassParams {
  float dt, max_accel, max_speed, target_x, target_y, speed_cost, control_cost;
} MbpoPointMassParams;
typedef struct MbpoGeneralSystemParams {
  MbpoPendulumParams pendulum;
  float noise_std;
  MbpoPointMassParams point_mass;
} MbpoGeneralSystemParams;

/* Learned MLP-ensemble System (template: mbpo/utils/network_utils.py:5-17, swish).
 * E members of [x_dim+u_dim -> hidden -> hidden -> hidden -> x_dim], predicting delta-x.
 * w_in  float[E, x_dim+u_dim, hidden]   b_in  float[E, hidden]
 * w_h   bf16 [E, 2, hidden(out), hidden(in)]  (K-major, i.e. transposed Dense kernels)
 * b_h   float[E, 2, hidden]
 * w_out float[E, hidden, x_dim]         b_out float[E, x_dim]
 * The reward is the pendulum reward on the current state. */
typedef struct MbpoMlpEnsembleParams {
  int32_t num_members, hidden, x_dim, u_dim;
  const float* w_in;
  const float* b_in;
  const uint16_t* w_h;
  const float* b_h;
  const float* w_out;
  const float* b_out;
  MbpoPendulumParams reward;
} MbpoMlpEnsembleParams;

/* iCemParams (mbpo/optimizers/trajectory_optimizers/icem_optimizer.py:25-50) plus the
 * static shapes jit closes over.  Fill with mbpo_icem_cfg_init(). */
typedef struct MbpoIcemCfg {
  int32_t horizon;          /* H */
  int32_t action_dim;       /* A */
  int32_t x_dim;            /* X */
  int32_t num_samples;      /* N  :40 */
  int32_t num_elites;       /* K  :41 */
  int32_t num_prev_elites;  /* Np = max(int(elite_set_fraction*K),1)  :170 */
  int32_t num_particles;    /* P  :39 */
  int32_t num_steps;        /* S  :44 */
  int32_t warm_start;       /* :49 */
  int32_t prng_mode;        /* MBPO_PRNG_* */
  int32_t summarize;        /* MBPO_SUMMARIZE_* (use_optimism) */
  int32_t system_kind;      /* MBPO_SYSTEM_* */
  int32_t math_mode;        /* MBPO_MATH_* */
  float init_std;           /* :42 */
  float alpha;              /* :43 */
  float exponent;           /* :45 */
  float u_min, u_max;       /* :47-48 (scalar form) */
  float lambda_constraint;  /* :50 (unused without cost_fn) */
  /* trace-time constants of powerlaw_psd_gaussian (general_utils.py:143-178) */
  float sigma;
  float s_scale[MBPO_MAX_FREQ];
} MbpoIcemCfg;

/* Optional per-iteration dumps of mbpo_icem_plan for parity tests (any pointer may be
 * NULL).  M = N + Np. */
typedef struct MbpoIcemTrace {
  float* actions;      /* [S, B, M, H*A]  clipped samples + zero rows  (:190-192) */
  float* values;       /* [S, B, M]       objective values             (:195)     */
  int32_t* elite_idx;  /* [S, B, K]       argsort(values)[-K:]         (:199)     */
  float* mean;         /* [S, B, H*A]     refit mean after iteration   (:210)     */
  float* std;          /* [S, B, H*A]     refit std after iteration    (:214)     */
  float* best_value;   /* [S, B]          best-so-far value            (:217-226) */
} MbpoIcemTrace;

int mbpo_abi_version(void);
const char* mbpo_last_error(void);
/* sizeof() of the ABI structs, so that a foreign binding can verify its own layout:
 * which = 0 MbpoIcemCfg, 1 MbpoPendulumParams, 2 MbpoMlpEnsembleParams, 3 MbpoIcemTrace,
 * 4 MbpoPolicyParams, 5 MbpoReplayState, 6 MbpoReplayFields, 7 MbpoGeneralSystemParams;
 * anything else returns 0. */
size_t mbpo_struct_size(int which);

/* Host helper: fills every field from iCemParams + shapes and computes s_scale/sigma
 * exactly as general_utils.py:143-178 does at trace time (float32 arithmetic). */
int mbpo_icem_cfg_init(MbpoIcemCfg* cfg_host, int horizon, int action_dim, int x_dim,
                       int num_particles, int num_samples, int num_elites, float init_std,
                       float alpha, int num_steps, float exponent, float elite_set_fraction,
                       float u_min, float u_max, int warm_start, float lambda_constraint);

/* ---- JAX PRNG (jax.random.split / random_bits / uniform / normal), vmapped over M keys --- */
int mbpo_prng_split(const uint32_t* keys /*[M,2]*/, int M, int num, int prng_mode,
                    uint32_t* keys_out /*[M,num,2]*/, void* stream);
int mbpo_prng_random_bits(const uint32_t* keys /*[M,2]*/, int M, int n, int prng_mode,
                          uint32_t* bits_out /*[M,n]*/, void* stream);
int mbpo_prng_uniform(const uint32_t* keys, int M, int n, int prng_mode, float lo, float hi,
                      float* out /*[M,n]*/, void* stream);
int mbpo_prng_normal(const uint32_t* keys, int M, int n, int prng_mode, float* out /*[M,n]*/,
                     void* stream);

/* ---- stage 1: colored-noise action sampling ------------------------------------------- */
/* vmap(powerlaw_psd_gaussian(exponent, H, key)) (general_utils.py:81-208).
 * bits_out (optional) receives the raw uint32 words behind sr and si: [M, 2, H/2+1]. */
int mbpo_powerlaw_noise(const MbpoIcemCfg* cfg_host, const uint32_t* keys /*[M,2]*/, int M,
                        float* noise_out /*[M,H]*/, uint32_t* bits_out, void* stream);
/* The same function through the any-horizon kernel (rolled loops, twiddle table in the constant
 * bank; general_utils.py:134-143 takes any `size`, iCemTO any `horizon`, icem_optimizer.py:94-96).
 * mbpo_powerlaw_noise / mbpo_icem_sample_actions use it for every horizon in [2, MBPO_MAX_HORIZON]
 * without an unrolled instance; for the unrolled horizons both give the same bits. */
int mbpo_powerlaw_noise_rolled(const MbpoIcemCfg* cfg_host, const uint32_t* keys /*[M,2]*/, int M,
                               float* noise_out /*[M,H]*/, uint32_t* bits_out, void* stream);
/* One iCEM iteration of key plumbing + sampling (icem_optimizer.py:174-192) for B problems. */
int mbpo_icem_sample_actions(const MbpoIcemCfg* cfg_host, const uint32_t* carry_key /*[B,2]*/,
                             const float* mean /*[B,H,A]*/, const float* std /*[B,H,A]*/, int B,
                             float* actions_out /*[B,N+Np,H,A]*/, uint32_t* next_key_out /*[B,2]*/,
                             uint32_t* particle_keys_out /*[B,N+Np,2] or NULL*/, void* stream);

/* ---- stage 2: rollouts ------------------------------------------------------------------ */
/* vmap(System.step) (base_systems.py:40-52; pendulum_system.py:18-39). */
int mbpo_system_step(int system_kind, const void* sys_params_host, int math_mode,
                     const float* x /*[R,X]*/, const float* u /*[R,A]*/, int R,
                     float* x_next /*[R,X]*/, float* reward /*[R]*/, void* stream);
/* vmap(vmap(rollout_actions)) (optimizer_utils.py:11-59) + horizon mean (icem :160).
 * x0 [B,X]; actions [B,M,H,A]; returns_out [B,M] (NULL to skip).  The Transition buffers
 * obs_out/next_obs_out [B,M,H,X] and reward_out [B,M,H] are optional (NULL to skip). */
int mbpo_rollout_actions(int system_kind, const void* sys_params_host, int math_mode,
                         int horizon, int action_dim, int x_dim, const float* x0,
                         const float* actions, int B, int M, float* returns_out, float* obs_out,
                         float* reward_out, float* next_obs_out, void* stream);

/* ---- general Systems: any action_dim, key-consuming transitions (SURVEY 8f-3) ------------------------ */
/* vmap(System.step) for MBPO_SYSTEM_PENDULUM / _NOISY_PENDULUM / _POINT_MASS: x [R,X], u [R,A]; keys_in / keys_out
 * uint32 [R,2] are system_params.key before / after the step (NULL for a System that draws nothing). */
int mbpo_system_step_general(int system_kind, const MbpoGeneralSystemParams* params_host, int prng_mode,
                             const float* x, const float* u, const uint32_t* keys_in, int R, float* x_next,
                             float* reward, uint32_t* keys_out, void* stream);
/* vmap(vmap(objective)) (icem_optimizer.py:144-160,195) over B problems x M candidates: actions [B,M,H,A],
 * keys [B,M,2] = split(particles_rng, N+Np) (:177; NULL for a System that draws nothing).
 * num_particles >= 1: split(key, P) (:155), one rollout per particle key, horizon mean, then the left-to-right mean
 * (MBPO_SUMMARIZE_MEAN) or the max over particles -> values_out [B,M].
 * With num_particles = P >= 1 the Transition buffers are optional too and carry the particle axis: obs_out /
 * next_obs_out [B,M,P,H,X] and reward_out [B,M,P,H], particle p being the rollout with key split(keys[b,m], P)[p]
 * (a System that draws nothing writes its single rollout P times); values_out may then be NULL.
 * num_particles == 0: vmap(rollout_actions) (optimizer_utils.py:11-59) -- ONE rollout per row with keys[b,m] as
 * system_params.key; values_out (horizon mean) and the Transition buffers obs_out [B,M,H,X], reward_out [B,M,H],
 * next_obs_out [B,M,H,X] are each optional. */
int mbpo_system_objective(int system_kind, const MbpoGeneralSystemParams* params_host, int prng_mode, int horizon,
                          const float* x0 /*[B,X]*/, const float* actions, const uint32_t* keys, int B, int M,
                          int num_particles, int summarize, float* values_out, float* obs_out, float* reward_out,
                          float* next_obs_out, void* stream);

/* ---- stage 3: elite selection + refit + best tracking (icem_optimizer.py:199-226) ------- */
int mbpo_icem_elite_refit(const MbpoIcemCfg* cfg_host, const float* actions /*[B,M,H*A]*/,
                          const float* values /*[B,M]*/, const float* mean_in /*[B,H*A]*/,
                          const float* std_in, const float* best_value_in /*[B]*/,
                          const float* best_seq_in /*[B,H*A]*/, int B, float* mean_out,
                          float* std_out, float* best_value_out, float* best_seq_out,
                          int32_t* elite_idx_out /*[B,K] or NULL*/, void* stream);

/* ---- fused plan: iCemTO.optimize (icem_optimizer.py:134-252) vmapped over B problems ---- */
int mbpo_icem_plan(const MbpoIcemCfg* cfg_host, const void* sys_params_host,
                   const float* x0 /*[B,X]*/, const uint32_t* key_in /*[B,2]*/,
                   const float* best_seq_in /*[B,H,A]*/, int B, float* best_seq_out /*[B,H,A]*/,
                   float* best_value_out /*[B]*/, uint32_t* key_out /*[B,2]*/,
                   const MbpoIcemTrace* trace_host /*NULL = no dumps*/, void* stream);
/* The same plan with an explicit thread-block-cluster size: few problems leave most of the 148 SMs idle when each
 * gets one CTA, so a problem can be spread over a cluster of 2, 4, 8 or 16 CTAs (16 is a non-portable size: devices
 * that refuse it return MBPO_ECUDA for an explicit 16; the library's own choice falls back to 8, then to one CTA)
 * whose key / elite exchange runs through distributed shared memory and whose spare warps sample the next
 * iteration's noise under the rollouts (csrc/icem_cluster_kernels.cuh).  Results are bit-identical for every
 * cluster size.  cluster_size: -1 = the library's choice for (B, num_samples) -- what mbpo_icem_plan uses; 1 = one
 * CTA per problem; 2, 4, 8, 16 (at most 256 candidates per CTA).  mbpo_icem_plan_cluster_size returns that choice
 * (0 or 1: no cluster).
 * Reference: icem_optimizer.py:134-252 at B = 1 is tests/test_icemopt.py's shape. */
int mbpo_icem_plan_clustered(const MbpoIcemCfg* cfg_host, const void* sys_params_host, const float* x0,
                             const uint32_t* key_in, const float* best_seq_in, int B, float* best_seq_out,
                             float* best_value_out, uint32_t* key_out, const MbpoIcemTrace* trace_host,
                             int cluster_size, void* stream);
int mbpo_icem_plan_cluster_size(const MbpoIcemCfg* cfg_host, int B);
/* How many clusters of that size run at once on the current device (the GPCs decide, not the SM count: 7 of 16, 15 of
 * 8, 33 of 4, 74 of 2 on a B200); the library's choice is the largest size with B <= capacity, since a second round
 * of clusters costs a whole plan.  0: the size is not available for this configuration. */
int mbpo_icem_plan_cluster_capacity(const MbpoIcemCfg* cfg_host, int cluster_size);

/* 1 if mbpo_icem_plan runs this configuration as the single fused kernel, 0 if it composes
 * the staged kernels through `workspace`. */
int mbpo_icem_plan_is_fused(const MbpoIcemCfg* cfg_host);
size_t mbpo_icem_workspace_bytes(const MbpoIcemCfg* cfg_host, int B);
int mbpo_icem_plan_staged(const MbpoIcemCfg* cfg_host, const void* sys_params_host,
                          const float* x0, const uint32_t* key_in, const float* best_seq_in, int B,
                          float* best_seq_out, float* best_value_out, uint32_t* key_out,
                          void* workspace, size_t workspace_bytes, void* stream);

/* ---- objective tail + array-valued bounds: pieces of the general staged plan ---------------- */
/* iCemTO.objective's tail (icem_optimizer.py:158-166) for a deterministic System (P identical
 * particles): values[i] <- summarize_reward(values[i]) - lambda * relu(summarize_cost(cost[i])).
 * values [n] holds the horizon-mean reward of one particle; cost [n] (NULL = no cost_fn) the
 * trajectory cost AbstractCost.__call__ returned (:78-90).  summarize_* are MBPO_SUMMARIZE_*
 * (use_optimism :112-115, use_pessimism :116-119). */
int mbpo_icem_penalize(float* values, const float* cost, long long n, int num_particles,
                       int summarize_reward, int summarize_cost, float lambda_constraint, void* stream);
/* The same tail over P distinct particles (a System that draws from its key, or the ensemble's members):
 * values_out[i] = summarize_reward_p(mean_t reward[i,p,t]) - lambda * relu(summarize_cost_p(cost[i,p])).
 * reward [n,P,H] is the Transition reward of every particle (mbpo_system_objective / mbpo_ensemble_rollout_transitions),
 * cost [n,P] (NULL = no cost_fn).  The horizon mean is a left-to-right sum from 0 divided by H and the particle mean
 * a left-to-right sum divided by P: with cost == NULL the values are bit-equal to mbpo_system_objective's values_out
 * and mbpo_ensemble_rollout's returns_out. */
int mbpo_icem_penalize_particles(float* values_out /*[n]*/, const float* reward /*[n,P,H]*/, int horizon,
                                 const float* cost /*[n,P] or NULL*/, long long n, int num_particles,
                                 int summarize_reward, int summarize_cost, float lambda_constraint, void* stream);
/* jnp.clip(actions, u_min, u_max) with bounds broadcast to [H, A] (icem_optimizer.py:47-48,191):
 * clips the N sampled rows of every problem of actions [B, M, D], D = H*A; u_min/u_max [D]. */
int mbpo_icem_clip_actions(float* actions, const float* u_min, const float* u_max, int B, int M, int N,
                           int D, void* stream);

/* ---- closed-loop MPC (tests/test_icemopt.py:19-32): plan -> system.step -> warm start ---- */
int mbpo_icem_mpc_closed_loop(const MbpoIcemCfg* cfg_host, const void* sys_params_host,
                              const float* x0 /*[B,X]*/, const uint32_t* key_in /*[B,2]*/,
                              const float* best_seq_in /*[B,H,A]*/, int B, int num_mpc_steps,
                              float* states_out /*[T,B,X]*/, float* rewards_out /*[T,B]*/,
                              float* actions_out /*[T,B,A]*/, float* best_seq_out /*[B,H,A]*/,
                              uint32_t* key_out /*[B,2]*/, void* stream);
int mbpo_icem_mpc_closed_loop_clustered(const MbpoIcemCfg* cfg_host, const void* sys_params_host, const float* x0,
                                        const uint32_t* key_in, const float* best_seq_in, int B, int num_mpc_steps,
                                        float* states_out, float* rewards_out, float* actions_out,
                                        float* best_seq_out, uint32_t* key_out, int cluster_size, void* stream);


/* ---- vmapped env rollouts for SAC/PPO collection ---------------------------------------- */
/* brax_wrapper.py:40-50 + brax_utils/training.py:71-74,91-107,119-137 + sac/acting.py:35-55.
 * In/out env state: obs [E,X], steps [E], done [E] (float, as brax), first_obs [E,X].
 * actions [T,E,A].  Transition outputs are time-major: observation/next_observation
 * [T,E,X], reward/discount/truncation [T,E].  Any output pointer may be NULL.
 * observation[t] equals next_observation[t-1] (the post-reset state) and observation[0] is the
 * incoming obs, so a caller that lays both out as overlapping views of one [T+1,E,X] buffer
 * passes observation_out = NULL and next_observation_out = buffer + E*X (12 B/transition less
 * HBM traffic for the pendulum); the kernel never reads its outputs. */
int mbpo_env_rollout(int system_kind, const void* sys_params_host, int math_mode, int x_dim,
                     int action_dim, int episode_length, int action_repeat, float* obs,
                     float* steps, float* done, const float* first_obs, const float* actions,
                     int E, int T, float* observation_out, float* reward_out, float* discount_out,
                     float* next_observation_out, float* truncation_out, void* stream);

/* The same T steps with the env state passed by value: obs_in/steps_in/done_in are read, the state
 * after step T goes to obs_out/steps_out/done_out, which must NOT alias the inputs.  The pendulum
 * System never ends an episode itself, so the AutoReset points follow from the step counters and
 * the pieces between them are rolled concurrently (one thread per env and piece); results are
 * bit-identical to mbpo_env_rollout.  steps must be integer-valued, as brax's are. */
int mbpo_env_unroll(int system_kind, const void* sys_params_host, int math_mode, int x_dim,
                    int action_dim, int episode_length, int action_repeat, const float* obs_in,
                    const float* steps_in, const float* done_in, float* obs_out, float* steps_out,
                    float* done_out, const float* first_obs, const float* actions, int E, int T,
                    float* observation_out, float* reward_out, float* discount_out,
                    float* next_observation_out, float* truncation_out, void* stream);

/* mbpo_env_unroll for the general Systems (csrc/systems.cuh): MBPO_SYSTEM_NOISY_PENDULUM (X = 3, A = 1, keyed) and
 * MBPO_SYSTEM_POINT_MASS (X = 4, A = 2).  MBPO_SYSTEM_PENDULUM is MBPO_EINVAL here (it keeps mbpo_env_unroll /
 * mbpo_env_rollout); any other kind is MBPO_EUNSUPPORTED.  Same wrapper stack, layouts and overlapping-buffer
 * convention as mbpo_env_unroll, with actions [T,E,A].  sys_keys_in / sys_keys_out: uint32 [E,2], every env's
 * system_params.key before / after the T steps -- required for a keyed System, ignored (may be NULL) otherwise.
 * Each System.step advances the key once (key, sub = split(key)), so it advances action_repeat times per env step,
 * and AutoReset does not reset it.  The outgoing state may alias the incoming one.  T == 0 copies the state
 * through.  X = 4 needs 16-byte aligned observation buffers. */
int mbpo_env_unroll_general(int system_kind, const MbpoGeneralSystemParams* params_host, int prng_mode,
                            int episode_length, int action_repeat, const float* obs_in, const float* steps_in,
                            const float* done_in, const uint32_t* sys_keys_in /*[E,2] or NULL*/, float* obs_out,
                            float* steps_out, float* done_out, uint32_t* sys_keys_out, const float* first_obs,
                            const float* actions /*[T,E,A]*/, int E, int T, float* observation_out,
                            float* reward_out, float* discount_out, float* next_observation_out,
                            float* truncation_out, void* stream);

/* ---- policy in the env loop: SAC / PPO data collection ------------------------------------- */
/* The stochastic policy of sac/sac_networks.py:58-73 + sac/parametric_distribution.py:97-125:
 * logits = MLP(obs) (swish; Dense = x @ W + b), loc, scale = split(logits, 2),
 * action = tanh((softplus(scale) + min_std) * normal(key, [E, A]) + loc), or tanh(loc) when
 * deterministic.  w[l] are flax Dense kernels [in, out] (device pointers, float32): w[0] [obs_dim, hidden],
 * w[1..num_hidden-1] [hidden, hidden], w[num_hidden] [hidden, 2 * action_dim]; b[l] the biases. */
#define MBPO_POLICY_MAX_LAYERS 5
typedef struct MbpoPolicyParams {
  int32_t num_hidden, hidden, obs_dim, action_dim;
  const float* w[MBPO_POLICY_MAX_LAYERS];
  const float* b[MBPO_POLICY_MAX_LAYERS];
  float min_std;
  /* head: MBPO_HEAD_NORMAL_TANH (above) or MBPO_HEAD_BPTT_ACTOR, the actor of bptt_optimizer.py:123-142,306-326:
   * mu, sig = split(MLP((obs - obs_mean) / obs_std), 2); sig = clip(softplus(sig + sig_bias), sig_min, sig_max)
   * (sig_bias = inv_softplus(init_stddev)); action = clip(tanh(mu + normal(key, (A,)) * sig), +-action_clip),
   * or clip(tanh(mu)) when deterministic.  shared_noise = 1 draws normal(key, (A,)) once for every env (the key
   * is not vmapped in BPTT's vmap(actor_loss, in_axes=(0, None, None)), bptt_optimizer.py:366-368).
   * normalize = 0 feeds obs to the network as is. */
  int32_t head, shared_noise, normalize;
  float sig_bias, sig_min, sig_max, action_clip;
  float obs_mean[4], obs_std[4];
  /* device-resident normaliser statistics (float[obs_dim] each): when non-NULL the kernels read these instead of
   * obs_mean / obs_std, so a collection loop never reads the running statistics back to the host. */
  const float* obs_mean_dev;
  const float* obs_std_dev;
  /* which kernel runs the network: MBPO_ACTOR_AUTO picks the tcgen05 kernel (hidden -> hidden layers as TF32 x 3
   * split-precision MMAs, fp32 accumulate in TMEM) for 2..3 hidden layers and the CUDA-core kernel otherwise;
   * MBPO_ACTOR_TCGEN05 with an unsupported depth is MBPO_EUNSUPPORTED. */
  int32_t kernel;
  /* env sharding: the policy's draw is normal(key, (num_envs, A))[env], so a rank that owns envs
   * [draw_offset, draw_offset + E) of draw_total reproduces the unsharded stream bit for bit (draw_total = 0: the
   * launch owns every env, i.e. draw_total = E, draw_offset = 0). */
  int32_t draw_offset, draw_total;
} MbpoPolicyParams;
enum { MBPO_HEAD_NORMAL_TANH = 0, MBPO_HEAD_BPTT_ACTOR = 1 };
/* MBPO_ACTOR_TCGEN05 = the throughput kernel (four 128-env tiles per CTA, thread = env); MBPO_ACTOR_TCGEN05_WIDE = the
 * latency kernel (one tile per CTA, sixteen producer warps + PRNG warps: a step takes a third of the time when the
 * envs do not fill the GPU).  Both produce the same bits.  MBPO_ACTOR_AUTO takes the wide kernel when there is at most
 * one tile per SM. */
enum { MBPO_ACTOR_AUTO = 0, MBPO_ACTOR_CUDA_CORES = 1, MBPO_ACTOR_TCGEN05 = 2, MBPO_ACTOR_TCGEN05_WIDE = 3 };
enum {
  MBPO_KEYS_SAC = 0,     /* sac/sac.py:288-292      k, k_t = split(k); policy key = k_t          */
  MBPO_KEYS_UNROLL = 1,  /* sac/acting.py:68-73     current, next = split(current); policy key = current, carry = next */
  MBPO_KEYS_AS_IS = 2    /* sac/acting.py:35-55     actor_step(env, state, policy, key): key used directly */
};
/* T steps of actor_step (sac/acting.py:35-55) for E envs in one launch: policy forward, NormalTanh
 * sample, the wrapped env step of mbpo_env_rollout, Transition out (time-major; action_out [T,E,A];
 * observation[t] = next_observation[t-1], observation[0] = the incoming obs, as in mbpo_env_rollout).
 * key_in / key_out: device uint32[2], the scan's carry key before / after the T steps. */
int mbpo_actor_rollout(int system_kind, const void* sys_params_host, int math_mode, int prng_mode,
                       const MbpoPolicyParams* policy_host, int deterministic, int key_convention,
                       const uint32_t* key_in, int episode_length, int action_repeat, float* obs,
                       float* steps, float* done, const float* first_obs, int E, int T, float* action_out,
                       float* reward_out, float* discount_out, float* next_observation_out,
                       float* truncation_out, uint32_t* key_out, void* stream);

/* The same launch, also emitting what PPO's policy returns beside the action (ppo/ppo_network.py:59-84;
 * sac/parametric_distribution.py:66-83): raw_action_out [T,E,A] = the pre-tanh sample, log_prob_out [T,E] =
 * Normal(loc, scale).log_prob(raw) - Tanh.forward_log_det_jacobian(raw) summed over the action axis.  Both NULL
 * or both given; ignored for deterministic policies (the reference returns {} there). */
int mbpo_actor_rollout_extras(int system_kind, const void* sys_params_host, int math_mode, int prng_mode,
                              const MbpoPolicyParams* policy_host, int deterministic, int key_convention,
                              const uint32_t* key_in, int episode_length, int action_repeat, float* obs,
                              float* steps, float* done, const float* first_obs, int E, int T,
                              float* action_out, float* reward_out, float* discount_out,
                              float* next_observation_out, float* truncation_out, uint32_t* key_out,
                              float* raw_action_out, float* log_prob_out, void* stream);

/* mbpo_actor_rollout_extras for the general Systems (see mbpo_env_unroll_general for the kinds and their refusals):
 * the policy kernel on the CUDA cores with obs_dim = X and action_dim = A (width 64, 1..4 hidden layers), the
 * NormalTanh head, all three key conventions, deterministic mode and PPO's extras (log_prob summed over the A
 * action dims, raw_action_out [T,E,A]).  The policy's draw is normal(key, (draw_total, A)) flattened: env e, dim a
 * reads element (draw_offset + e) * A + a, so a sharded launch reproduces the unsharded one.  obs / steps / done are
 * updated in place; sys_keys_in / sys_keys_out as in mbpo_env_unroll_general.  The general Systems have one math
 * (every operation rounded once), so there is no math_mode.  MBPO_EUNSUPPORTED: MBPO_HEAD_BPTT_ACTOR (or
 * shared_noise), kernel = MBPO_ACTOR_TCGEN05 / MBPO_ACTOR_TCGEN05_WIDE, and policy shapes other than the above;
 * MBPO_ACTOR_AUTO selects the CUDA-core kernel. */
int mbpo_actor_rollout_general(int system_kind, const MbpoGeneralSystemParams* params_host, int prng_mode,
                               const MbpoPolicyParams* policy_host, int deterministic, int key_convention,
                               const uint32_t* key_in, int episode_length, int action_repeat, float* obs,
                               float* steps, float* done, const uint32_t* sys_keys_in /*[E,2] or NULL*/,
                               uint32_t* sys_keys_out, const float* first_obs, int E, int T, float* action_out,
                               float* reward_out, float* discount_out, float* next_observation_out,
                               float* truncation_out, uint32_t* key_out, float* raw_action_out,
                               float* log_prob_out, void* stream);

/* rollout_policy (mbpo/utils/optimizer_utils.py:62-116) for the general Systems: the plain scan of T System.steps
 * from x0 [E,X] with the policy in the loop -- no Episode / AutoReset wrapper, so no step counter, done or
 * truncation (discount is 1).  The policy runs on the CUDA cores as in mbpo_actor_rollout_general; its head is
 * MBPO_HEAD_BPTT_ACTOR (BPTT.act, bptt_optimizer.py:123-142,306-326; with shared_noise the draw normal(key, (A,)) is
 * the same for every trajectory, element a for action dim a) or MBPO_HEAD_NORMAL_TANH (the draw of
 * mbpo_actor_rollout_general).  key_convention as there (BPTT: MBPO_KEYS_UNROLL, or MBPO_KEYS_AS_IS to evaluate).
 * Outputs are time-major: action_out [T,E,A], reward_out [T,E], next_observation_out [T,E,X] (observation[t] =
 * next_observation[t-1], observation[0] = x0).  sys_keys_in / sys_keys_out: a keyed System's system_params.key,
 * uint32 [2] shared by every trajectory (sys_keys_shared = 1) or [E,2] -- required for a keyed System, ignored
 * otherwise; each System.step advances it once.  key_in / key_out: the policy's carry key.  E or T == 0 copies the
 * keys through.  X = 4 needs a 16-byte aligned next_observation_out.  MBPO_SYSTEM_PENDULUM is MBPO_EINVAL (it keeps
 * mbpo_actor_rollout); MBPO_EUNSUPPORTED: any other non-general kind, kernel = MBPO_ACTOR_TCGEN05 /
 * MBPO_ACTOR_TCGEN05_WIDE and policy shapes other than those of mbpo_actor_rollout_general. */
int mbpo_rollout_policy_general(int system_kind, const MbpoGeneralSystemParams* params_host, int prng_mode,
                                const MbpoPolicyParams* policy_host, int deterministic, int key_convention,
                                const uint32_t* key_in, const uint32_t* sys_keys_in /*[2] or [E,2] or NULL*/,
                                int sys_keys_shared, const float* x0 /*[E,X]*/, int E, int T,
                                float* action_out /*[T,E,A]*/, float* reward_out /*[T,E]*/,
                                float* next_observation_out /*[T,E,X]*/, uint32_t* key_out, uint32_t* sys_keys_out,
                                void* stream);

/* ---- reverse pass through System.step rollouts; lambda returns (BPTT) ----------------------- */
/* The cotangent pass of jax.value_and_grad through rollout_policy(..., stop_grads=True)
 * (mbpo/utils/optimizer_utils.py:62-116; bptt_optimizer.py:327-376): the policy sees
 * stop_gradient(obs), so cotangents reach its parameters through the actions only.  For E
 * trajectories of T steps, given the forward trajectory (observation x_t, action a_t) and the
 * cotangents of the Transition fields, writes g_action_out[t] = total cotangent reaching a_t and
 * g_x0_out [E,X] (or NULL).  g_reward / g_next_obs / g_obs / g_action_in may be NULL (zero).
 * observation[t+1] and next_observation[t] are the same value; g_obs[0] flows to g_x0_out.
 * Element (t, e) of a per-step scalar array is base[t*stride_t + e*stride_e]; of an [.,.,X] array
 * base[t*stride_xt + e*stride_xe + i]: the reference's vmapped [B,H,...] layout and the rollout
 * kernels' time-major [T,E,...] layout both work without copies. */
int mbpo_rollout_adjoint(int system_kind, const void* sys_params_host, int x_dim, int action_dim, int E,
                         int T, long long stride_t, long long stride_e, long long stride_xt,
                         long long stride_xe, const float* observation, const float* action,
                         const float* g_reward, const float* g_next_obs, const float* g_obs,
                         const float* g_action_in, float* g_action_out, float* g_x0_out, void* stream);

/* mbpo_rollout_adjoint for the general Systems (the trajectory of mbpo_rollout_policy_general):
 * MBPO_SYSTEM_NOISY_PENDULUM, whose noise does not depend on (x, u), so its Jacobians are the pendulum's at the
 * stored noisy observation and no key is needed; and MBPO_SYSTEM_POINT_MASS (clip ties split the cotangent in half,
 * as jnp.clip does).  stride_t / stride_e address g_reward; stride_xt / stride_xe the [.,.,X] arrays (observation,
 * g_next_obs, g_obs); stride_at / stride_ae the [.,.,A] arrays (action, g_action_in, g_action_out), innermost
 * stride 1 for both.  g_x0_out is [E,X].  MBPO_SYSTEM_PENDULUM is MBPO_EINVAL (it keeps mbpo_rollout_adjoint); any
 * other non-general kind is MBPO_EUNSUPPORTED. */
int mbpo_rollout_adjoint_general(int system_kind, const MbpoGeneralSystemParams* params_host, int E, int T,
                                 long long stride_t, long long stride_e, long long stride_xt, long long stride_xe,
                                 long long stride_at, long long stride_ae, const float* observation,
                                 const float* action, const float* g_reward, const float* g_next_obs,
                                 const float* g_obs, const float* g_action_in, float* g_action_out, float* g_x0_out,
                                 void* stream);

/* lambda_return (mbpo/utils/optimizer_utils.py:119-131): inputs = reward + discount * next_values *
 * (1 - lambda); returns[t] = inputs[t] + discount * lambda * returns[t+1], returns[T] = next_values[-1].
 * E independent sequences of T steps, element (t, e) at base[t*stride_t + e*stride_e]. */
int mbpo_lambda_return(const float* reward, const float* next_values, int E, int T, long long stride_t,
                       long long stride_e, double discount, double lambda_, float* returns_out,
                       void* stream);
/* Its transpose (what jax.grad computes through it): cotangents of reward and next_values. */
int mbpo_lambda_return_vjp(const float* g_returns, int E, int T, long long stride_t, long long stride_e,
                           double discount, double lambda_, float* g_reward_out,
                           float* g_next_values_out, void* stream);

/* ---- stage 4: learned MLP-ensemble dynamics, batched forward on tcgen05 ------------------ */
/* inp [R, x_dim+u_dim], member [R] (int32 ensemble member per row) -> delta [R, x_dim]. */
int mbpo_mlp_dynamics_forward(const MbpoMlpEnsembleParams* params_host, const float* inp,
                              const int32_t* member, int R, float* delta_out, void* stream);

/* vmap(vmap(rollout_actions)) + the particle summary of iCemTO.objective (icem_optimizer.py:155-160)
 * through the learned ensemble System: particle p is rolled through ensemble member p
 * (num_particles == num_members), x_next = x + MLP_p([x, u]), reward = pendulum reward on (x, u).
 * x0 [B,X]; actions [B,M,H,A]; returns_out [B,M] = mean (MBPO_SUMMARIZE_MEAN) or max over members of
 * the horizon-mean reward.  One fused tcgen05 kernel (CTA pairs, weights resident in shared memory). */
int mbpo_ensemble_rollout(const MbpoMlpEnsembleParams* params_host, int horizon, const float* x0,
                          const float* actions, int B, int M, int summarize, float* returns_out, void* stream);
/* The same rollouts with the Transition fields of every member instead of the summary: obs_out[b,m,e,t] is the
 * state member e's rollout is in before step t (obs_out[b,m,e,0] = x0[b]) and reward_out[b,m,e,t] the pendulum
 * reward on (that state, u_t).  Same kernels, roundings and checks as mbpo_ensemble_rollout; mbpo_icem_penalize_particles
 * turns reward_out into its returns_out, bit for bit. */
int mbpo_ensemble_rollout_transitions(const MbpoMlpEnsembleParams* params_host, int horizon, const float* x0 /*[B,X]*/,
                                      const float* actions /*[B,M,H,1]*/, int B, int M,
                                      float* obs_out /*[B,M,E,H,X]*/, float* reward_out /*[B,M,E,H]*/, void* stream);

/* The learned ensemble as a SAC / PPO env: T wrapped env steps of E envs (the Episode / AutoReset stack of
 * mbpo_env_unroll_general around x_next = x + MLP_m([x, u]), the reward the pendulum reward on (x, u); a System's
 * own done is 0), env e rolled through member m[e] for all T steps.  env_order [E] (int32) lists the envs stably
 * sorted by member, and member_offsets [num_members + 1] (int32) bounds each member's run in it; envs whose member
 * is outside [0, num_members) are in no run and are not stepped.  obs [E,3] / steps [E] / done [E] are read and
 * overwritten in place.  policy_host == NULL: the actions are given, actions [T,E,1]; otherwise the policy runs in
 * the loop as in mbpo_actor_rollout_general (NormalTanh head, deterministic, key_convention, key_in / key_out, the
 * draw window, raw_action_out / log_prob_out), writing action_out [T,E,1].  Every env's rows are written at its own
 * index: reward_out, discount_out, truncation_out [T,E], next_observation_out [T,E,3] (observation[t] =
 * next_observation[t-1]).  E or T == 0 copies the carry key through.  MBPO_EUNSUPPORTED: ensembles other than
 * hidden 256, x_dim 3, u_dim 1; the BPTT head; the tcgen05 policy kernels; a policy too large for the shared memory
 * beside the ensemble's (1..2 hidden layers of width 64 fit). */
int mbpo_ensemble_env_rollout(const MbpoMlpEnsembleParams* params_host, int prng_mode,
                              const MbpoPolicyParams* policy_host /* NULL: actions given */, int deterministic,
                              int key_convention, const uint32_t* key_in, int episode_length, int action_repeat,
                              const int32_t* env_order, const int32_t* member_offsets, float* obs, float* steps,
                              float* done, const float* first_obs, int E, int T, const float* actions,
                              float* action_out, float* reward_out, float* discount_out,
                              float* next_observation_out, float* truncation_out, uint32_t* key_out,
                              float* raw_action_out, float* log_prob_out, void* stream);

/* ---- replay buffer (brax UniformSamplingQueue) and BraxWrapper.reset ---------------------------
 * The data format either side of the env rollouts: SAC appends every collected Transition to a
 * brax UniformSamplingQueue (mbpo/optimizers/policy_optimizers/sac/sac.py:202-205,303) and
 * BraxWrapper.reset draws each env's first observation from the true buffer
 * (mbpo/systems/brax_wrapper.py:25-38, tests/test_sac.py:15-28).  brax is a third-party
 * dependency; its published algorithm (brax/training/replay_buffers.py: QueueBase.insert_internal,
 * UniformSamplingQueue.sample_internal) is restated in oracle/brax_replay.py.
 *
 * Storage is a RING: logical row i (brax's data[i]) lives in physical row (head + i) % capacity.
 * brax's jnp.roll(data, roll) of the whole buffer on every insert into a full queue becomes
 * head -= roll; no row moves.  A row is ravel_pytree(Transition): the fields side by side. */
typedef struct MbpoReplayState {
  float* data;               /* device, [capacity, row_width] physical rows            */
  long long capacity;        /* max_replay_size                                         */
  int32_t row_width;         /* D                                                       */
  int32_t reserved;
  long long head;            /* physical row of logical row 0                           */
  long long insert_position; /* brax ReplayBufferState.insert_position (logical)        */
  long long sample_position; /* brax ReplayBufferState.sample_position (logical)        */
} MbpoReplayState;

#define MBPO_REPLAY_MAX_FIELDS 8
typedef struct MbpoReplayFields {
  int32_t num_fields;
  int32_t width[MBPO_REPLAY_MAX_FIELDS];    /* columns of field f                      */
  const float* ptr[MBPO_REPLAY_MAX_FIELDS]; /* device, [n_rows, width[f]] dense        */
} MbpoReplayFields;

/* jax.random.randint(key, (n,), minval, maxval) (int32) for M keys: out int32[M, n]. */
int mbpo_prng_randint(const uint32_t* keys /*[M,2]*/, int M, int n, int prng_mode, int minval, int maxval,
                      int32_t* out /*[M,n]*/, void* stream);

/* QueueBase.insert_internal: appends n_rows rows assembled from the field arrays (time-major
 * rollout buffers [T, E, w] are [T*E, w] dense: the order jnp.concatenate gives at sac.py:296) and
 * updates head / insert_position / sample_position of *state_host exactly like brax's roll.
 * n_rows > capacity is MBPO_EINVAL (brax raises ValueError). */
int mbpo_replay_insert(MbpoReplayState* state_host, const MbpoReplayFields* fields_host, long long n_rows,
                       void* stream);

/* UniformSamplingQueue.sample_internal: key_out = split(key)[0]; idx = randint(split(key)[1],
 * (batch,), sample_position, insert_position); batch_out[i] = data[idx[i] mod capacity].
 * idx_out may be NULL. */
int mbpo_replay_sample(const MbpoReplayState* state_host, const uint32_t* key /*[2]*/, int prng_mode,
                       int sample_batch_size, uint32_t* key_out /*[2]*/, int32_t* idx_out /*[batch]*/,
                       float* batch_out /*[batch, D]*/, void* stream);

/* Logical rows [first, first + n) in brax's order (ReplayBufferState.data[first:first+n]). */
int mbpo_replay_read(const MbpoReplayState* state_host, long long first, long long n, float* rows_out /*[n,D]*/,
                     void* stream);

/* vmap(BraxWrapper.reset)(rngs) (brax_wrapper.py:25-38 under VmapWrapper.reset,
 * brax_utils/training.py:66-69): per env keys = split(rng, 2); the buffer is sampled under keys[0]
 * (a batch of sample_batch_size, element 0 kept, :30); obs = row[0:x_dim], reward = row[reward_col];
 * system_params.key = keys[1].  idx_out (the logical row each env drew) may be NULL. */
int mbpo_env_reset_from_buffer(const MbpoReplayState* state_host, const uint32_t* rngs /*[E,2]*/, int E,
                               int prng_mode, int sample_batch_size, int x_dim, int reward_col,
                               float* obs_out /*[E,X]*/, float* reward_out /*[E]*/,
                               uint32_t* sys_key_out /*[E,2]*/, int32_t* idx_out /*[E]*/, void* stream);

/* EvalWrapper (mbpo/optimizers/policy_optimizers/brax_utils/training.py:156-199) folded over the Transition of an
 * unroll, as acting.Evaluator uses it (sac/acting.py:82-151): per env, in step order and in float32,
 *   episode_steps  = active ? steps_t : episode_steps     (steps_t: EpisodeWrapper's counter after step t)
 *   episode_reward += reward_t * active
 *   active        *= discount_t                            (discount = 1 - done, acting.py:51)
 * steps_t is rebuilt from steps_in / done_in (the env state the unroll started from) and the discount stream:
 * steps = (done ? 0 : steps) + action_repeat (training.py:98,120-124).  reward / discount are [T, E] with the
 * given strides; episode_reward, episode_steps, active are [E], read and written (EvalWrapper.reset gives 0, 0, 1),
 * so an evaluation may be folded chunk by chunk. */
int mbpo_eval_metrics(const float* reward, const float* discount, const float* steps_in /*[E]*/,
                      const float* done_in /*[E]*/, int action_repeat, int E, int T, long long stride_t,
                      long long stride_e, float* episode_reward, float* episode_steps, float* active, void* stream);

/* ---- observation normaliser (brax running_statistics) ------------------------------------------
 * running_statistics.update(normalizer_params, transitions.observation, pmap_axis_name) as SAC / PPO call it after
 * every collection (sac/sac.py:298-301): count += n; mean += sum(batch - mean) / count; summed_variance +=
 * sum((batch - old_mean) * (batch - new_mean)); std = clip(sqrt(max(summed_variance, 0) / count)).
 * Split at the one exchange step of the path: _accumulate reduces this rank's rows to sums[2X + 1] (float64:
 * sum d, sum d*d with d = batch - old_mean in float32, and the row count), the caller all-reduces sums over the ranks
 * (the reference's psum), _finalize applies the update with step_increment = sums[2X].  sum(d * (d - mean_update)) = sum d*d - mean_update * sum d,
 * so one pass over the rows and one all-reduce replace the reference's two of each.  Deterministic: per-CTA partials
 * are combined in a fixed order (no atomics).  workspace: mbpo_running_statistics_workspace_bytes(X) bytes. */
size_t mbpo_running_statistics_workspace_bytes(int X);
int mbpo_running_statistics_accumulate(const float* batch /*[n_rows, X]*/, long long n_rows, int X,
                                       const float* mean /*[X]*/, void* workspace, size_t workspace_bytes,
                                       double* sums_out /*[2X+1]*/, void* stream);
int mbpo_running_statistics_finalize(const double* sums /*[2X+1]*/, int X,
                                     const float* count_in /*[1]*/, const float* mean_in /*[X]*/,
                                     const float* summed_variance_in /*[X]*/, float std_min_value, float std_max_value,
                                     float* count_out /*[1]*/, float* mean_out /*[X]*/, float* summed_variance_out /*[X]*/,
                                     float* std_out /*[X]*/, void* stream);
/* running_statistics.normalize: out = (batch - mean) / std, clipped to +-max_abs_value when it is > 0. */
int mbpo_running_statistics_normalize(const float* batch /*[n_rows, X]*/, long long n_rows, int X, const float* mean,
                                      const float* std, float max_abs_value, float* out, void* stream);

/* BPTT's own Normalizer (mbpo/optimizers/policy_optimizers/bptt_optimizer.py:31-75; update_normalizers :297-303, the
 * state normaliser's mean / std are what the BPTT actor kernel reads): update(x, state) with n = x.shape[0]:
 *   new_mean = (mean * size + sum(x)) / total;  s_n = std^2 * size + sum((x - new_mean)^2) + size * (mean - new_mean)^2;
 *   std = max(sqrt(s_n / total), 1e-8);  size = total.
 * Same split as the running statistics: sums[2X+1] from mbpo_running_statistics_accumulate (d = x - mean), all-reduced
 * by the caller when the batch is sharded, then this call; with delta = sum d / total,
 * sum((x - new_mean)^2) = sum d*d - 2 delta sum d + n delta^2.  size is a float64 scalar on the device. */
int mbpo_normalizer_finalize(const double* sums /*[2X+1]*/, int X, const double* size_in /*[1]*/,
                             const float* mean_in /*[X]*/, const float* std_in /*[X]*/, float eps,
                             double* size_out /*[1]*/, float* mean_out /*[X]*/, float* std_out /*[X]*/, void* stream);

/* Normalizer.inverse (bptt_optimizer.py:73-75): out = x * std + mean. */
int mbpo_normalizer_inverse(const float* batch /*[n_rows, X]*/, long long n_rows, int X, const float* mean,
                            const float* std, float* out, void* stream);

/* jnp.take(buffer_state.data, idx, axis=0, mode='wrap') (bptt_optimizer.py:447-449): rows_out[i] = data[idx[i] mod
 * capacity] in brax's logical row order. */
int mbpo_replay_take(const MbpoReplayState* state_host, const int32_t* idx /*[n]*/, long long n,
                     float* rows_out /*[n, D]*/, void* stream);

/* PPO's generalised advantage estimation over the Transition of an unroll
 * (mbpo/optimizers/policy_optimizers/ppo/losses.py:128-184 compute_gae; call site :87-99): per env, one reverse scan
 *   deltas = (rewards + discount * (1 - termination) * values[t+1] - values) * (1 - truncation)
 *   acc    = deltas + discount * (1 - termination) * (1 - truncation) * lambda * acc
 *   vs     = acc + values;   advantages = (rewards + discount * (1 - termination) * vs[t+1] - values) * (1 - truncation)
 * with values[T] = vs[T] = bootstrap_value, every product and sum rounded once in the order written (python floats are
 * weakly typed: discount and lambda are rounded to float32).  All [T, E] arrays share (stride_t, stride_e); both
 * outputs are stop_gradient in the reference, so there is no transpose. */
int mbpo_compute_gae(const float* truncation, const float* termination, const float* rewards, const float* values,
                     const float* bootstrap_value /*[E]*/, int E, int T, long long stride_t, long long stride_e,
                     double discount, double lambda_, float* vs_out, float* advantages_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MBPO_B200_H_ */
