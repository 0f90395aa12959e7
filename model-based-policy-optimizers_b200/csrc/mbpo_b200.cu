// C ABI of the B200-native iCEM planning hot path (declared in include/mbpo_b200.h).
//
// Host side only validates arguments, fills kernel argument structs and launches on the
// caller's stream.  No allocation, no synchronisation, no CPU fallback: an unsupported
// configuration is an error (MBPO_EUNSUPPORTED), never a slow path.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <tuple>

#include "../../include/mbpo_b200.h"
#include "host_util.h"
#include "mlp_tc_kernels.cuh"
#include "actor_kernels.cuh"
#include "actor_tc_kernels.cuh"
#include "actor_tc_wide_kernels.cuh"
#include "adjoint_kernels.cuh"
#include "ensemble_env_kernels.cuh"
#include "ensemble_pp_kernels.cuh"
#include "plan_dispatch.h"
#include "staged_kernels.cuh"
#include "systems.cuh"

namespace mbpo {
thread_local char g_err[512] = "";
}

using namespace mbpo;

namespace {

bool horizon_supported(int H) {
  switch (H) {
#define X(h) case h:
    MBPO_FOR_EACH_H(X)
#undef X
    return true;
    default:
      return false;
  }
}

// ------------------------------------------------------------------------------------------
// PRNG primitive kernels (runtime mode; one thread per output word / key)
// ------------------------------------------------------------------------------------------
template <int MODE>
__global__ void prng_split_kernel(const uint32_t* __restrict__ keys, long long total, int num,
                                  uint32_t* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long m = i / num;
  const uint32_t j = static_cast<uint32_t>(i % num);
  const Key2 k{keys[2 * m], keys[2 * m + 1]};
  const Key2 o = split_at<MODE>(k, static_cast<uint32_t>(num), j);
  out[2 * i] = o.k0;
  out[2 * i + 1] = o.k1;
}

// what: 0 bits, 1 uniform(lo,hi), 2 normal
template <int MODE>
__global__ void prng_draw_kernel(const uint32_t* __restrict__ keys, long long total, int n, int what, float lo,
                                 float hi, void* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long m = i / n;
  const uint32_t w = static_cast<uint32_t>(i % n);
  const Key2 k{keys[2 * m], keys[2 * m + 1]};
  const uint32_t bits = random_bits_at<MODE>(k, static_cast<uint32_t>(n), w);
  if (what == 0) static_cast<uint32_t*>(out)[i] = bits;
  else if (what == 1) static_cast<float*>(out)[i] = bits_to_uniform(bits, lo, hi);
  else static_cast<float*>(out)[i] = bits_to_normal(bits);
}

int prng_draw(const uint32_t* keys, int M, int n, int prng_mode, int what, float lo, float hi, void* out,
              void* stream) {
  MBPO_REQUIRE(M >= 0 && n >= 0, "prng: negative size");
  MBPO_REQUIRE(prng_mode == 0 || prng_mode == 1, "prng: bad prng_mode %d", prng_mode);
  const long long total = static_cast<long long>(M) * n;
  if (total == 0) return MBPO_OK;
  MBPO_REQUIRE(keys && out, "prng: null pointer");
  const int threads = 256;
  const unsigned blocks = static_cast<unsigned>((total + threads - 1) / threads);
  return with_prng(prng_mode, [&](auto P) {
    prng_draw_kernel<P><<<blocks, threads, 0, as_stream(stream)>>>(keys, total, n, what, lo, hi, out);
    return check_launch("prng_draw_kernel");
  });
}

int validate_cfg(const MbpoIcemCfg* c) {
  MBPO_REQUIRE(c != nullptr, "cfg is null");
  MBPO_REQUIRE(c->horizon >= 2 && c->horizon <= MBPO_MAX_HORIZON, "horizon %d outside [2, %d]", c->horizon,
               MBPO_MAX_HORIZON);
  MBPO_REQUIRE(c->action_dim >= 1, "action_dim %d < 1", c->action_dim);
  MBPO_REQUIRE(c->x_dim >= 1, "x_dim %d < 1", c->x_dim);
  MBPO_REQUIRE(c->num_samples >= 1, "num_samples %d < 1", c->num_samples);
  MBPO_REQUIRE(c->num_prev_elites >= 1, "num_prev_elites %d < 1", c->num_prev_elites);
  MBPO_REQUIRE(c->num_elites >= 1 && c->num_elites <= c->num_samples + c->num_prev_elites,
               "num_elites %d outside [1, num_samples + num_prev_elites = %d]", c->num_elites,
               c->num_samples + c->num_prev_elites);
  MBPO_REQUIRE(c->num_particles >= 1, "num_particles %d < 1", c->num_particles);
  MBPO_REQUIRE(c->num_steps >= 1, "num_steps %d < 1", c->num_steps);
  MBPO_REQUIRE(c->prng_mode == 0 || c->prng_mode == 1, "bad prng_mode %d", c->prng_mode);
  MBPO_REQUIRE(c->summarize == 0 || c->summarize == 1, "bad summarize %d", c->summarize);
  MBPO_REQUIRE(c->math_mode == 0 || c->math_mode == 1, "bad math_mode %d", c->math_mode);
  MBPO_REQUIRE(c->sigma > 0.0f && std::isfinite(c->sigma), "sigma must be positive and finite");
  return MBPO_OK;
}

ScaleTable make_scale_table(const MbpoIcemCfg* c) {
  ScaleTable t;
  std::memset(&t, 0, sizeof(t));
  fill_noise_scale(c->s_scale, c->sigma, c->horizon, t.v);
  return t;
}

int launch_noise_rolled(const MbpoIcemCfg* cfg, const ScaleTable& tbl, const uint32_t* keys, int M, float* noise_out,
                        uint32_t* bits_out, void* stream) {
  TwiddleTable tw;
  fill_twiddles(cfg->horizon, tw);
  const int threads = STAGED_THREADS;
  const size_t smem = static_cast<size_t>(threads) * (cfg->horizon | 1) * sizeof(float);
  const unsigned blocks = static_cast<unsigned>((M + threads - 1) / threads);
  return with_prng(cfg->prng_mode, [&](auto P) {
    auto kernel = powerlaw_noise_rt_kernel<P>;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               static_cast<int>(smem));
    if (e != cudaSuccess) return fail(MBPO_ECUDA, "powerlaw_noise smem attr: %s", cudaGetErrorString(e));
    kernel<<<blocks, threads, smem, as_stream(stream)>>>(tbl, tw, cfg->horizon, keys, M, noise_out, bits_out);
    return check_launch("powerlaw_noise_rt_kernel");
  });
}

// ---- fused plan --------------------------------------------------------------------------
void fill_plan_args(PlanArgs& a, const MbpoIcemCfg* c, const MbpoPendulumParams* sys, const float* x0,
                    const uint32_t* key_in, const float* best_seq_in, int B, float* best_seq_out,
                    float* best_value_out, uint32_t* key_out, const MbpoIcemTrace* trace) {
  std::memset(&a, 0, sizeof(a));
  a.B = B; a.N = c->num_samples; a.Np = c->num_prev_elites; a.K = c->num_elites; a.P = c->num_particles;
  a.H = c->horizon;
  a.S = c->num_steps; a.warm_start = c->warm_start; a.summarize = c->summarize;
  a.init_std = c->init_std; a.alpha = c->alpha; a.one_minus_alpha = static_cast<float>(1.0 - static_cast<double>(c->alpha));
  a.u_min = c->u_min; a.u_max = c->u_max;
  if (sys) a.sys = *sys;
  fill_noise_scale(c->s_scale, c->sigma, c->horizon, a.scale);
  a.x0 = x0; a.key_in = key_in; a.best_seq_in = best_seq_in; a.best_seq_out = best_seq_out;
  a.best_value_out = best_value_out; a.key_out = key_out;
  if (trace) a.trace = *trace;
}

// The general Systems whose plans run the general kernels (icem_plan_general_kernel, general_objective_kernel); the
// pendulum, a general System too, keeps its tuned plan kernels.
bool general_plan_kind(int kind, int* X, int* A) {
  bool keyed;
  return kind != MBPO_SYSTEM_PENDULUM && general_system_dims(kind, X, A, &keyed) == MBPO_OK;
}
bool general_plan_kind(int kind) {
  int X, A;
  return general_plan_kind(kind, &X, &A);
}

int plan_fusable(const MbpoIcemCfg* c, bool set_error) {
  const char* why = nullptr;
  int X, A;
  if (general_plan_kind(c->system_kind, &X, &A)) {
    const size_t RS = static_cast<size_t>(c->horizon * A) | 1;
    const size_t words = static_cast<size_t>(c->num_samples + 1) * RS + (c->num_samples + c->num_prev_elites) +
                         3 * c->horizon * A + 2 * c->num_elites +
                         select_scratch_words(c->num_elites, c->num_samples + c->num_prev_elites) + 8;
    if (c->action_dim != A || c->x_dim != X) why = "fused plan: action_dim / x_dim do not match the System";
    else if (!horizon_supported(c->horizon)) why = "fused plan: horizon has no compiled kernel (" MBPO_H_LIST_STR ")";
    else if (words * 4 > 227 * 1024) why = "fused plan: population does not fit 227 KB of shared memory";
    if (why && set_error) fail(MBPO_EUNSUPPORTED, "%s", why);
    return why == nullptr;
  }
  if (c->system_kind != MBPO_SYSTEM_PENDULUM) why = "fused plan supports the pendulum and the general Systems only";
  else if (c->action_dim != 1 || c->x_dim != 3) why = "fused plan requires action_dim == 1 and x_dim == 3";
  else {
    const int HS = c->horizon | 1;
    size_t words = static_cast<size_t>(c->num_samples + 1) * HS + (c->num_samples + c->num_prev_elites) +
                   2 * (c->num_samples + 1) + 3 * c->horizon + 2 * c->num_elites +
                   select_scratch_words(c->num_elites, c->num_samples + c->num_prev_elites) + 8;
    if (!horizon_supported(c->horizon)) words += static_cast<size_t>(PLAN_THREADS) * HS;   // the any-horizon kernel's staging rows
    if (words * 4 > 227 * 1024) why = "fused plan: population does not fit 227 KB of shared memory";
  }
  if (why && set_error) fail(MBPO_EUNSUPPORTED, "%s", why);
  return why == nullptr;
}

// Capacities of cluster sizes 16, 8, 4, 2 for a configuration on the current device, cached: the occupancy queries
// cost more than a plan at B = 1.
struct ClusterCaps { int cap[4]; };
ClusterCaps cluster_caps(const MbpoIcemCfg* c, bool mpc) {
  static std::mutex mu;
  static std::map<std::tuple<int, int, int, int, int, int, int, int, int, int>, ClusterCaps> cache;
  int dev = 0;
  cudaGetDevice(&dev);
  const bool general = general_plan_kind(c->system_kind);
  // the general cluster kernels' block size depends on the particles as well
  const auto key = std::make_tuple(dev, c->system_kind, c->horizon, c->prng_mode, c->math_mode, mpc ? 1 : 0,
                                   c->num_samples, c->num_prev_elites, c->num_elites, general ? c->num_particles : 0);
  std::lock_guard<std::mutex> lock(mu);
  const auto it = cache.find(key);
  if (it != cache.end()) return it->second;
  ClusterCaps caps = {{0, 0, 0, 0}};
  for (int i = 0, cl = 16; i < 4; ++i, cl >>= 1) {
    const int R = (c->num_samples + cl - 1) / cl;
    if (R < 32 || R > 256) continue;
    switch (c->horizon) {
#define X(h)                                                                                                      \
  case h:                                                                                                         \
    caps.cap[i] = general ? general_plan_cluster_capacity<h>(c->system_kind, c->prng_mode, mpc, c->num_samples,   \
                                                             c->num_prev_elites, c->num_elites, c->num_particles,  \
                                                             cl)                                                   \
                          : plan_cluster_capacity<h>(c->prng_mode, c->math_mode, mpc, c->num_samples,             \
                                                     c->num_prev_elites, c->num_elites, cl);                      \
    break;
      MBPO_FOR_EACH_H(X)
#undef X
      default: break;
    }
  }
  cache[key] = caps;
  return caps;
}

// The cluster size to run: the caller's, or for -1 the library's choice for B problems (0 / 1: one CTA each).
int plan_cluster_size(const MbpoIcemCfg* c, int B, bool mpc, int cluster_size) {
  if (cluster_size >= 0) return cluster_size;
  if (!horizon_supported(c->horizon) || c->num_samples + c->num_prev_elites < 36) return 0;
  const ClusterCaps caps = cluster_caps(c, mpc);
  return plan_cluster_choice(B, c->num_samples, caps.cap);
}

// Runs dispatch(cluster) and, where the library chose the size and the device refuses it, falls back: a refused 16
// runs at 8, a refused cluster at one CTA per problem (the same bits).
template <class F>
int dispatch_with_fallback(int cluster, int cluster_size, F&& dispatch) {
  int rc = dispatch(cluster);
  if (rc == MBPO_ECUDA && cluster_size < 0 && cluster == 16) {
    cudaGetLastError();                 // the device refused the non-portable size the library picked: use 8
    cluster = 8;
    rc = dispatch(8);
  }
  if (rc == MBPO_ECUDA && cluster_size < 0 && cluster > 1) {
    cudaGetLastError();                 // no cluster of the library's own choice can be placed (e.g. a partitioned
    rc = dispatch(1);                   // device): the one-CTA kernel gives the same bits
  }
  return rc;
}

// The cluster sizes a plan takes: 2, 4, 8, 16, with the population limits of the cluster kernels.
int check_cluster_size(const MbpoIcemCfg* c, int cluster) {
  MBPO_REQUIRE(cluster == 2 || cluster == 4 || cluster == 8 || cluster == 16,
               "plan: cluster_size %d (use -1, 1, 2, 4, 8 or 16)", cluster);
  const int N = c->num_samples, Np = c->num_prev_elites;
  // the pendulum's CTAs own candidates of N, the general Systems' candidate rows of N + Np
  const int R = ((general_plan_kind(c->system_kind) ? N + Np : N) + cluster - 1) / cluster;
  if (R > 256) return fail(MBPO_EUNSUPPORTED, "plan: %d candidates per CTA of a %d-cluster (at most 256)", R, cluster);
  if (N + Np < 36)   // the cluster kernel keeps its elite list in the selection scratch (words 299 .. 300 + K)
    return fail(MBPO_EUNSUPPORTED, "plan: population (%d + %d) outside what a %d-cluster handles", N, Np, cluster);
  return MBPO_OK;
}

// Fused plan (gm == nullptr) or closed loop over a general System.
int run_general_plan(const MbpoIcemCfg* c, const MbpoGeneralSystemParams* gp, const float* x0, const uint32_t* key_in,
                     const float* best_seq_in, int B, float* best_seq_out, float* best_value_out, uint32_t* key_out,
                     const MbpoIcemTrace* trace, const GeneralMpcArgs* gm, int cluster_size, void* stream) {
  PlanArgs g;
  fill_plan_args(g, c, nullptr, x0, key_in, best_seq_in, B, best_seq_out, best_value_out, key_out, trace);
  g.gsys = *gp;
  const int cluster = plan_cluster_size(c, B, gm != nullptr, cluster_size);
  if (cluster > 1) {
    const int rc = check_cluster_size(c, cluster);
    if (rc != MBPO_OK) return rc;
  }
  return dispatch_with_fallback(cluster, cluster_size, [&](int cl) -> int {
    switch (c->horizon) {
#define X(h) \
  case h:    \
    return general_plan_entry<h>(c->system_kind, c->prng_mode, g, gm, as_stream(stream), cl);
      MBPO_FOR_EACH_H(X)
#undef X
      default:
        return fail(MBPO_EUNSUPPORTED, "horizon %d has no compiled kernel", c->horizon);
    }
  });
}

int run_plan(const MbpoIcemCfg* c, const void* sys_params_host, const float* x0, const uint32_t* key_in,
             const float* best_seq_in, int B, float* best_seq_out, float* best_value_out, uint32_t* key_out,
             const MbpoIcemTrace* trace, const MpcArgs* mpc, int cluster_size, void* stream) {
  int rc = validate_cfg(c);
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(B >= 0, "plan: B < 0");
  if (!plan_fusable(c, true)) return MBPO_EUNSUPPORTED;
  if (B == 0) return MBPO_OK;
  MBPO_REQUIRE(sys_params_host && x0 && key_in && best_seq_in && best_seq_out && key_out, "plan: null pointer");
  MBPO_REQUIRE(mpc != nullptr || best_value_out != nullptr, "plan: best_value_out is null");
  if (general_plan_kind(c->system_kind)) {
    if (mpc != nullptr)
      return fail(MBPO_EUNSUPPORTED, "closed loop over a general System: use mbpo_icem_mpc_closed_loop_general, "
                  "which carries the System's keys");
    return run_general_plan(c, static_cast<const MbpoGeneralSystemParams*>(sys_params_host), x0, key_in, best_seq_in,
                            B, best_seq_out, best_value_out, key_out, trace, nullptr, cluster_size, stream);
  }
  // the fused kernel's reward wrap has no fmod slow path (pendulum.cuh wrap_diff<true>): |theta - target + pi| < 4 pi
  if (!(std::fabs(static_cast<const MbpoPendulumParams*>(sys_params_host)->target_angle) <= 6.0f))
    return fail(MBPO_EUNSUPPORTED, "fused plan: |target_angle| > 6 rad; use mbpo_icem_plan_staged");
  PlanArgs a;
  fill_plan_args(a, c, static_cast<const MbpoPendulumParams*>(sys_params_host), x0, key_in, best_seq_in, B,
                 best_seq_out, best_value_out, key_out, trace);
  // few problems: spread each over a thread-block cluster (same bits; icem_cluster_kernels.cuh)
  const int cluster = plan_cluster_size(c, B, mpc != nullptr, cluster_size);
  if (!horizon_supported(c->horizon)) {
    if (cluster_size > 1) return fail(MBPO_EUNSUPPORTED, "plan: clusters exist for the unrolled horizons (" MBPO_H_LIST_STR ")");
    return plan_entry_rt(c->prng_mode, c->math_mode, a, mpc, as_stream(stream));
  }
  if (cluster > 1) {
    const int rc2 = check_cluster_size(c, cluster);
    if (rc2 != MBPO_OK) return rc2;
  }
  return dispatch_with_fallback(cluster, cluster_size, [&](int cl) -> int {
    switch (c->horizon) {
#define X(h) \
  case h:    \
    return plan_entry<h>(c->prng_mode, c->math_mode, a, mpc, as_stream(stream), cl);
      MBPO_FOR_EACH_H(X)
#undef X
      default:
        return fail(MBPO_EUNSUPPORTED, "horizon %d has no compiled kernel", c->horizon);
    }
  });
}

}  // namespace

// ============================================================================================
// extern "C"
// ============================================================================================
extern "C" {

int mbpo_abi_version(void) { return MBPO_ABI_VERSION; }

const char* mbpo_last_error(void) { return g_err; }

size_t mbpo_struct_size(int which) {
  switch (which) {
    case 0: return sizeof(MbpoIcemCfg);
    case 1: return sizeof(MbpoPendulumParams);
    case 2: return sizeof(MbpoMlpEnsembleParams);
    case 3: return sizeof(MbpoIcemTrace);
    case 4: return sizeof(MbpoPolicyParams);
    case 5: return sizeof(MbpoReplayState);
    case 6: return sizeof(MbpoReplayFields);
    case 7: return sizeof(MbpoGeneralSystemParams);
    default: return 0;
  }
}

int mbpo_icem_cfg_init(MbpoIcemCfg* cfg, int horizon, int action_dim, int x_dim, int num_particles, int num_samples,
                       int num_elites, float init_std, float alpha, int num_steps, float exponent,
                       float elite_set_fraction, float u_min, float u_max, int warm_start, float lambda_constraint) {
  MBPO_REQUIRE(cfg != nullptr, "cfg is null");
  MBPO_REQUIRE(horizon >= 2 && horizon <= MBPO_MAX_HORIZON, "horizon %d outside [2, %d]", horizon, MBPO_MAX_HORIZON);
  std::memset(cfg, 0, sizeof(*cfg));
  cfg->horizon = horizon;
  cfg->action_dim = action_dim;
  cfg->x_dim = x_dim;
  cfg->num_samples = num_samples;
  cfg->num_elites = num_elites;
  // num_prev_elites_per_iter = max(int(elite_set_fraction * num_elites), 1): python float (double) product
  const int npe = static_cast<int>(static_cast<double>(elite_set_fraction) * num_elites);
  cfg->num_prev_elites = npe > 1 ? npe : 1;
  cfg->num_particles = num_particles;
  cfg->num_steps = num_steps;
  cfg->warm_start = warm_start ? 1 : 0;
  cfg->prng_mode = MBPO_PRNG_LEGACY;
  cfg->summarize = MBPO_SUMMARIZE_MEAN;
  cfg->system_kind = MBPO_SYSTEM_PENDULUM;
  cfg->math_mode = MBPO_MATH_REFERENCE;
  cfg->init_std = init_std;
  cfg->alpha = alpha;
  cfg->exponent = exponent;
  cfg->u_min = u_min;
  cfg->u_max = u_max;
  cfg->lambda_constraint = lambda_constraint;
  // general_utils.py:143-178 in float32: f = rfftfreq(H); s_scale[:ix] = s_scale[ix] with
  // ix = sum(f < 1/H) = 1; s_scale **= -exponent/2; w = s_scale[1:]; w[-1] *= (1 + H%2)/2;
  // sigma = 2*sqrt(sum(w^2))/H.
  const int F = horizon / 2 + 1;
  const float fmin = static_cast<float>(1.0 / horizon);
  float f[MBPO_MAX_FREQ];
  for (int i = 0; i < F; ++i) f[i] = static_cast<float>(i) / static_cast<float>(horizon);
  int ix = 0;
  for (int i = 0; i < F; ++i) ix += (f[i] < fmin) ? 1 : 0;
  if (ix && ix < F)
    for (int i = 0; i < ix; ++i) f[i] = f[ix];
  const float pw = static_cast<float>(-static_cast<double>(exponent) / 2.0);
  float sumsq = 0.0f;
  for (int i = 0; i < F; ++i) {
    cfg->s_scale[i] = powf(f[i], pw);
    if (i >= 1) {
      float w = cfg->s_scale[i];
      if (i == F - 1) w = w * static_cast<float>((1 + (horizon % 2)) / 2.0);
      sumsq += w * w;
    }
  }
  cfg->sigma = 2.0f * sqrtf(sumsq) / static_cast<float>(horizon);
  return MBPO_OK;
}

// ---- PRNG ------------------------------------------------------------------------------------
int mbpo_prng_split(const uint32_t* keys, int M, int num, int prng_mode, uint32_t* keys_out, void* stream) {
  MBPO_REQUIRE(M >= 0 && num >= 0, "prng_split: negative size");
  MBPO_REQUIRE(prng_mode == 0 || prng_mode == 1, "prng_split: bad prng_mode %d", prng_mode);
  const long long total = static_cast<long long>(M) * num;
  if (total == 0) return MBPO_OK;
  MBPO_REQUIRE(keys && keys_out, "prng_split: null pointer");
  const int threads = 256;
  const unsigned blocks = static_cast<unsigned>((total + threads - 1) / threads);
  return with_prng(prng_mode, [&](auto P) {
    prng_split_kernel<P><<<blocks, threads, 0, as_stream(stream)>>>(keys, total, num, keys_out);
    return check_launch("prng_split_kernel");
  });
}

int mbpo_prng_random_bits(const uint32_t* keys, int M, int n, int prng_mode, uint32_t* bits_out, void* stream) {
  return prng_draw(keys, M, n, prng_mode, 0, 0.0f, 0.0f, bits_out, stream);
}

int mbpo_prng_uniform(const uint32_t* keys, int M, int n, int prng_mode, float lo, float hi, float* out,
                      void* stream) {
  return prng_draw(keys, M, n, prng_mode, 1, lo, hi, out, stream);
}

int mbpo_prng_normal(const uint32_t* keys, int M, int n, int prng_mode, float* out, void* stream) {
  return prng_draw(keys, M, n, prng_mode, 2, 0.0f, 0.0f, out, stream);
}

// ---- stage 1 -----------------------------------------------------------------------------------
int mbpo_powerlaw_noise(const MbpoIcemCfg* cfg, const uint32_t* keys, int M, float* noise_out, uint32_t* bits_out,
                        void* stream) {
  const int rc = validate_cfg(cfg);
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(M >= 0, "powerlaw_noise: M < 0");
  if (M == 0) return MBPO_OK;
  MBPO_REQUIRE(keys && noise_out, "powerlaw_noise: null pointer");
  const ScaleTable tbl = make_scale_table(cfg);
  // any other horizon: the rolled-loop kernel (same words, same operation order)
  if (!horizon_supported(cfg->horizon)) return launch_noise_rolled(cfg, tbl, keys, M, noise_out, bits_out, stream);
  switch (cfg->horizon) {
#define X(h) \
  case h:    \
    return noise_entry<h>(cfg->prng_mode, tbl, keys, M, noise_out, bits_out, as_stream(stream));
    MBPO_FOR_EACH_H(X)
#undef X
  }
  return MBPO_EUNSUPPORTED;
}

int mbpo_powerlaw_noise_rolled(const MbpoIcemCfg* cfg, const uint32_t* keys, int M, float* noise_out,
                               uint32_t* bits_out, void* stream) {
  const int rc = validate_cfg(cfg);
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(M >= 0, "powerlaw_noise_rolled: M < 0");
  if (M == 0) return MBPO_OK;
  MBPO_REQUIRE(keys && noise_out, "powerlaw_noise_rolled: null pointer");
  return launch_noise_rolled(cfg, make_scale_table(cfg), keys, M, noise_out, bits_out, stream);
}

int mbpo_icem_sample_actions(const MbpoIcemCfg* cfg, const uint32_t* carry_key, const float* mean, const float* std_,
                             int B, float* actions_out, uint32_t* next_key_out, uint32_t* particle_keys_out,
                             void* stream) {
  const int rc = validate_cfg(cfg);
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(B >= 0 && B <= 65535, "sample_actions: B %d outside [0, 65535]", B);
  if (B == 0) return MBPO_OK;
  MBPO_REQUIRE(carry_key && mean && std_ && actions_out && next_key_out, "sample_actions: null pointer");
  const ScaleTable tbl = make_scale_table(cfg);
  if (!horizon_supported(cfg->horizon)) {   // any other horizon: the rolled-loop kernel (same words, same order)
    TwiddleTable tw;
    fill_twiddles(cfg->horizon, tw);
    const int threads = STAGED_THREADS;
    const size_t smem = static_cast<size_t>(threads) * (cfg->horizon | 1) * sizeof(float);
    const int N = cfg->num_samples, Np = cfg->num_prev_elites, A = cfg->action_dim;
    const dim3 grid(static_cast<unsigned>(((N + Np) * A + threads - 1) / threads), static_cast<unsigned>(B));
    return with_prng(cfg->prng_mode, [&](auto P) {
      auto kernel = sample_actions_rt_kernel<P>;
      const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 static_cast<int>(smem));
      if (e != cudaSuccess) return fail(MBPO_ECUDA, "sample_actions smem attr: %s", cudaGetErrorString(e));
      kernel<<<grid, threads, smem, as_stream(stream)>>>(tbl, tw, cfg->horizon, carry_key, mean, std_, N, Np, A,
                                                         cfg->u_min, cfg->u_max, actions_out, next_key_out,
                                                         particle_keys_out);
      return check_launch("sample_actions_rt_kernel");
    });
  }
  switch (cfg->horizon) {
#define X(h)                                                                                                    \
  case h:                                                                                                       \
    return sample_entry<h>(cfg->prng_mode, tbl, carry_key, mean, std_, cfg->num_samples, cfg->num_prev_elites, \
                           cfg->action_dim, cfg->u_min, cfg->u_max, B, actions_out, next_key_out,               \
                           particle_keys_out, as_stream(stream));
    MBPO_FOR_EACH_H(X)
#undef X
  }
  return MBPO_EUNSUPPORTED;
}

// ---- stage 2 -----------------------------------------------------------------------------------
int mbpo_system_step(int system_kind, const void* sys_params_host, int math_mode, const float* x, const float* u,
                     int R, float* x_next, float* reward, void* stream) {
  MBPO_REQUIRE(system_kind == MBPO_SYSTEM_PENDULUM || system_kind == MBPO_SYSTEM_MLP_ENSEMBLE,
               "system_step: unknown system_kind %d", system_kind);
  if (system_kind != MBPO_SYSTEM_PENDULUM)
    return fail(MBPO_EUNSUPPORTED, "system_step: only MBPO_SYSTEM_PENDULUM has an inlined step");
  MBPO_REQUIRE(math_mode == 0 || math_mode == 1, "system_step: bad math_mode %d", math_mode);
  MBPO_REQUIRE(R >= 0, "system_step: R < 0");
  if (R == 0) return MBPO_OK;
  MBPO_REQUIRE(sys_params_host && x && u && x_next && reward, "system_step: null pointer");
  const MbpoPendulumParams sys = *static_cast<const MbpoPendulumParams*>(sys_params_host);
  const int threads = 128;
  const unsigned blocks = static_cast<unsigned>((R + threads - 1) / threads);
  return with_math(math_mode, [&](auto M) {
    system_step_pendulum_kernel<M><<<blocks, threads, 0, as_stream(stream)>>>(sys, x, u, R, x_next, reward);
    return check_launch("system_step_pendulum_kernel");
  });
}

int mbpo_rollout_actions(int system_kind, const void* sys_params_host, int math_mode, int horizon, int action_dim,
                         int x_dim, const float* x0, const float* actions, int B, int M, float* returns_out,
                         float* obs_out, float* reward_out, float* next_obs_out, void* stream) {
  if (system_kind == MBPO_SYSTEM_MLP_ENSEMBLE) {
    if (obs_out || reward_out || next_obs_out)
      return fail(MBPO_EUNSUPPORTED, "rollout_actions: the ensemble System returns objectives only (no Transition buffers)");
    MBPO_REQUIRE(action_dim == 1 && x_dim == 3, "rollout_actions: ensemble System needs action_dim == 1, x_dim == 3");
    return mbpo_ensemble_rollout(static_cast<const MbpoMlpEnsembleParams*>(sys_params_host), horizon, x0, actions, B, M,
                                 MBPO_SUMMARIZE_MEAN, returns_out, stream);
  }
  if (system_kind != MBPO_SYSTEM_PENDULUM)
    return fail(MBPO_EUNSUPPORTED, "rollout_actions: unknown system_kind %d", system_kind);
  MBPO_REQUIRE(action_dim == 1 && x_dim == 3, "rollout_actions: pendulum needs action_dim == 1, x_dim == 3");
  MBPO_REQUIRE(horizon >= 1 && horizon <= 4096, "rollout_actions: horizon %d outside [1, 4096]", horizon);
  MBPO_REQUIRE(math_mode == 0 || math_mode == 1, "rollout_actions: bad math_mode %d", math_mode);
  MBPO_REQUIRE(B >= 0 && M >= 0, "rollout_actions: negative size");
  const long long total = static_cast<long long>(B) * M;
  if (total == 0) return MBPO_OK;
  MBPO_REQUIRE(sys_params_host && x0 && actions, "rollout_actions: null pointer");
  const MbpoPendulumParams sys = *static_cast<const MbpoPendulumParams*>(sys_params_host);
  const int threads = 128;
  const int HS = horizon | 1;
  const size_t smem = static_cast<size_t>(threads / 32) * 32 * HS * sizeof(float);
  if (smem > 227 * 1024) return fail(MBPO_EUNSUPPORTED, "rollout_actions: horizon %d too long to stage", horizon);
  const long long warps = (total + 31) / 32;
  const unsigned blocks = static_cast<unsigned>((warps + threads / 32 - 1) / (threads / 32));
  return with_math(math_mode, [&](auto MATH) {
    auto kernel = rollout_actions_pendulum_kernel<MATH>;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               static_cast<int>(smem));
    if (e != cudaSuccess) return fail(MBPO_ECUDA, "rollout_actions smem attr: %s", cudaGetErrorString(e));
    kernel<<<blocks, threads, smem, as_stream(stream)>>>(sys, horizon, x0, actions, B, M, returns_out, obs_out,
                                                         reward_out, next_obs_out);
    return check_launch("rollout_actions_pendulum_kernel");
  });
}

// ---- general Systems (any action_dim, key-consuming) ---------------------------------------------
int mbpo_system_step_general(int system_kind, const MbpoGeneralSystemParams* params_host, int prng_mode,
                             const float* x, const float* u, const uint32_t* keys_in, int R, float* x_next,
                             float* reward, uint32_t* keys_out, void* stream) {
  int X, A; bool keyed;
  if (general_system_dims(system_kind, &X, &A, &keyed) != MBPO_OK)
    return fail(MBPO_EUNSUPPORTED, "system_step_general: system_kind %d is not one of the general Systems",
                system_kind);
  MBPO_REQUIRE(prng_mode == 0 || prng_mode == 1, "system_step_general: bad prng_mode %d", prng_mode);
  MBPO_REQUIRE(R >= 0, "system_step_general: R < 0");
  if (R == 0) return MBPO_OK;
  MBPO_REQUIRE(params_host && x && u && x_next && reward, "system_step_general: null pointer");
  MBPO_REQUIRE(!keyed || keys_in, "system_step_general: this System draws from system_params.key: keys_in is null");
  const unsigned blocks = static_cast<unsigned>((R + 127) / 128);
  return with_system<PendulumSys, NoisyPendulumSys, PointMassSys>(system_kind, [&](auto t) {
    using Sys = typename decltype(t)::type;
    return with_prng(prng_mode, [&](auto P) {
      system_step_general_kernel<Sys, P><<<blocks, 128, 0, as_stream(stream)>>>(*params_host, x, u, keys_in, R,
                                                                                 x_next, reward, keys_out);
      return check_launch("system_step_general_kernel");
    });
  });
}

int mbpo_system_objective(int system_kind, const MbpoGeneralSystemParams* params_host, int prng_mode, int horizon,
                          const float* x0, const float* actions, const uint32_t* keys, int B, int M,
                          int num_particles, int summarize, float* values_out, float* obs_out, float* reward_out,
                          float* next_obs_out, void* stream) {
  int X, A; bool keyed;
  if (general_system_dims(system_kind, &X, &A, &keyed) != MBPO_OK)
    return fail(MBPO_EUNSUPPORTED, "system_objective: system_kind %d is not one of the general Systems", system_kind);
  MBPO_REQUIRE(prng_mode == 0 || prng_mode == 1, "system_objective: bad prng_mode %d", prng_mode);
  MBPO_REQUIRE(horizon >= 1 && B >= 0 && M >= 0 && num_particles >= 0, "system_objective: bad sizes");
  MBPO_REQUIRE(summarize == 0 || summarize == 1, "system_objective: bad summarize %d", summarize);
  const long long total = static_cast<long long>(B) * M;
  if (total == 0) return MBPO_OK;
  MBPO_REQUIRE(params_host && x0 && actions, "system_objective: null pointer");
  MBPO_REQUIRE(!keyed || keys, "system_objective: this System draws from system_params.key: keys is null");
  const bool buffers = obs_out || reward_out || next_obs_out;
  MBPO_REQUIRE(num_particles == 0 || values_out || buffers, "system_objective: values_out is null");
  const unsigned blocks = static_cast<unsigned>((total + 127) / 128);
  return with_system<PendulumSys, NoisyPendulumSys, PointMassSys>(system_kind, [&](auto t) {
    using Sys = typename decltype(t)::type;
    return with_prng(prng_mode, [&](auto P) {
      if (num_particles > 0 && buffers) {
        general_particles_kernel<Sys, P><<<blocks, 128, 0, as_stream(stream)>>>(
            *params_host, horizon, x0, actions, keys, B, M, num_particles, summarize, values_out, obs_out, reward_out,
            next_obs_out);
        return check_launch("general_particles_kernel");
      }
      general_objective_kernel<Sys, P><<<blocks, 128, 0, as_stream(stream)>>>(
          *params_host, horizon, x0, actions, keys, B, M, num_particles, summarize, values_out, obs_out, reward_out,
          next_obs_out);
      return check_launch("general_objective_kernel");
    });
  });
}

// ---- stage 3 -----------------------------------------------------------------------------------
int mbpo_icem_elite_refit(const MbpoIcemCfg* cfg, const float* actions, const float* values, const float* mean_in,
                          const float* std_in, const float* best_value_in, const float* best_seq_in, int B,
                          float* mean_out, float* std_out, float* best_value_out, float* best_seq_out,
                          int32_t* elite_idx_out, void* stream) {
  const int rc = validate_cfg(cfg);
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(B >= 0, "elite_refit: B < 0");
  if (B == 0) return MBPO_OK;
  MBPO_REQUIRE(actions && values && mean_in && std_in && best_value_in && best_seq_in && mean_out && std_out &&
                   best_value_out && best_seq_out,
               "elite_refit: null pointer");
  RefitScalars rs;
  rs.M = cfg->num_samples + cfg->num_prev_elites;
  rs.K = cfg->num_elites;
  rs.D = cfg->horizon * cfg->action_dim;
  rs.alpha = cfg->alpha;
  rs.one_minus_alpha = static_cast<float>(1.0 - static_cast<double>(cfg->alpha));
  const size_t smem = (static_cast<size_t>(rs.M) + 2 * rs.K + select_scratch_words(rs.K, rs.M) + 3 * rs.D + 4) * 4;
  if (smem > 227 * 1024) return fail(MBPO_EUNSUPPORTED, "elite_refit: population too large for shared memory");
  const cudaError_t e =
      cudaFuncSetAttribute(elite_refit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  if (e != cudaSuccess) return fail(MBPO_ECUDA, "elite_refit smem attr: %s", cudaGetErrorString(e));
  elite_refit_kernel<<<B, REFIT_THREADS, smem, as_stream(stream)>>>(rs, actions, values, mean_in, std_in, best_value_in,
                                                          best_seq_in, mean_out, std_out, best_value_out, best_seq_out,
                                                          elite_idx_out);
  return check_launch("elite_refit_kernel");
}

// ---- fused plan ----------------------------------------------------------------------------------
int mbpo_icem_plan_is_fused(const MbpoIcemCfg* cfg) {
  if (validate_cfg(cfg) != MBPO_OK) return 0;
  return plan_fusable(cfg, false);
}

int mbpo_icem_plan(const MbpoIcemCfg* cfg, const void* sys_params_host, const float* x0, const uint32_t* key_in,
                   const float* best_seq_in, int B, float* best_seq_out, float* best_value_out, uint32_t* key_out,
                   const MbpoIcemTrace* trace_host, void* stream) {
  return run_plan(cfg, sys_params_host, x0, key_in, best_seq_in, B, best_seq_out, best_value_out, key_out,
                  trace_host, nullptr, -1, stream);
}

int mbpo_icem_plan_clustered(const MbpoIcemCfg* cfg, const void* sys_params_host, const float* x0,
                             const uint32_t* key_in, const float* best_seq_in, int B, float* best_seq_out,
                             float* best_value_out, uint32_t* key_out, const MbpoIcemTrace* trace_host,
                             int cluster_size, void* stream) {
  return run_plan(cfg, sys_params_host, x0, key_in, best_seq_in, B, best_seq_out, best_value_out, key_out,
                  trace_host, nullptr, cluster_size, stream);
}

int mbpo_icem_plan_cluster_size(const MbpoIcemCfg* cfg, int B) {
  if (validate_cfg(cfg) != MBPO_OK || !plan_fusable(cfg, false) || B < 0) return 0;
  return plan_cluster_size(cfg, B, false, -1);
}

int mbpo_icem_plan_cluster_capacity(const MbpoIcemCfg* cfg, int cluster_size) {
  if (validate_cfg(cfg) != MBPO_OK || !plan_fusable(cfg, false) || !horizon_supported(cfg->horizon)) return 0;
  const ClusterCaps caps = cluster_caps(cfg, false);
  switch (cluster_size) {
    case 16: return caps.cap[0];
    case 8: return caps.cap[1];
    case 4: return caps.cap[2];
    case 2: return caps.cap[3];
    default: return 0;
  }
}

// Staged plan workspace layout (floats unless noted), all [B, ...]:
//   actions [B,M,D] | values [B,M] | mean [B,D] | std [B,D] | mean2 [B,D] | std2 [B,D] | best_seq2 [B,D]
//   | best_value [B] | best_value2 [B] | carry_key u32[B,2] | carry_key2 u32[B,2]
size_t mbpo_icem_workspace_bytes(const MbpoIcemCfg* cfg, int B) {
  if (validate_cfg(cfg) != MBPO_OK || B < 0) return 0;
  const size_t M = static_cast<size_t>(cfg->num_samples) + cfg->num_prev_elites;
  const size_t D = static_cast<size_t>(cfg->horizon) * cfg->action_dim;
  const size_t b = static_cast<size_t>(B);
  const size_t words = b * M * D + b * M + 5 * b * D + 2 * b + 4 * b + 2 * b * M /* particle keys */;
  return words * 4 + 256;
}

int mbpo_icem_plan_staged(const MbpoIcemCfg* cfg, const void* sys_params_host, const float* x0,
                          const uint32_t* key_in, const float* best_seq_in, int B, float* best_seq_out,
                          float* best_value_out, uint32_t* key_out, void* workspace, size_t workspace_bytes,
                          void* stream) {
  int rc = validate_cfg(cfg);
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(sys_params_host, "plan_staged: null pointer");
  MBPO_REQUIRE(B >= 0 && B <= 65535, "plan_staged: B %d outside [0, 65535]", B);
  int X, A;
  const bool general = general_plan_kind(cfg->system_kind, &X, &A);
  if (cfg->system_kind != MBPO_SYSTEM_PENDULUM && cfg->system_kind != MBPO_SYSTEM_MLP_ENSEMBLE && !general)
    return fail(MBPO_EUNSUPPORTED, "plan_staged: unknown system_kind %d", cfg->system_kind);
  if (general) {
    MBPO_REQUIRE(cfg->action_dim == A && cfg->x_dim == X, "plan_staged: system_kind %d has x_dim %d, action_dim %d "
                 "(cfg says %d, %d)", cfg->system_kind, X, A, cfg->x_dim, cfg->action_dim);
  }
  if (cfg->system_kind == MBPO_SYSTEM_MLP_ENSEMBLE) {
    const MbpoMlpEnsembleParams* ep = static_cast<const MbpoMlpEnsembleParams*>(sys_params_host);
    if (cfg->num_particles != ep->num_members)
      return fail(MBPO_EUNSUPPORTED, "plan_staged: the ensemble System rolls particle p through member p; "
                  "num_particles (%d) must equal num_members (%d)", cfg->num_particles, ep->num_members);
    MBPO_REQUIRE(cfg->action_dim == 1 && cfg->x_dim == 3, "plan_staged: ensemble System needs action_dim == 1, x_dim == 3");
  }
  if (workspace_bytes < mbpo_icem_workspace_bytes(cfg, B))
    return fail(MBPO_EWORKSPACE, "plan_staged: workspace %zu B < required %zu B", workspace_bytes,
                mbpo_icem_workspace_bytes(cfg, B));
  if (B == 0) return MBPO_OK;
  MBPO_REQUIRE(x0 && key_in && best_seq_in && best_seq_out && best_value_out && key_out && workspace,
               "plan_staged: null pointer");
  const size_t M = static_cast<size_t>(cfg->num_samples) + cfg->num_prev_elites;
  const size_t D = static_cast<size_t>(cfg->horizon) * cfg->action_dim;
  const size_t b = static_cast<size_t>(B);
  uintptr_t p = reinterpret_cast<uintptr_t>(workspace);
  p = (p + 255) & ~static_cast<uintptr_t>(255);
  float* w = reinterpret_cast<float*>(p);
  float* actions = w;            w += b * M * D;
  float* values = w;             w += b * M;
  float* mean[2];  float* std_[2];
  mean[0] = w; w += b * D;  std_[0] = w; w += b * D;
  mean[1] = w; w += b * D;  std_[1] = w; w += b * D;
  float* bseq[2];  bseq[0] = best_seq_out;  bseq[1] = w;  w += b * D;
  float* bval[2];  bval[0] = w; w += b;  bval[1] = w; w += b;
  uint32_t* ckey[2];
  ckey[0] = reinterpret_cast<uint32_t*>(w); w += 2 * b;
  ckey[1] = reinterpret_cast<uint32_t*>(w); w += 2 * b;
  uint32_t* pkeys = reinterpret_cast<uint32_t*>(w); w += 2 * b * M;      // split(particles_rng, N + Np)  (:177)
  cudaStream_t st = as_stream(stream);

  // ping-pong so that after S iterations the results land in slot 0 (= the caller's buffers)
  int cur = (cfg->num_steps % 2 == 0) ? 0 : 1;
  rc = with_prng(cfg->prng_mode, [&](auto P) {
    plan_prologue_kernel<P><<<B, 64, 0, st>>>(B, static_cast<int>(D), cfg->action_dim, cfg->warm_start, cfg->init_std,
                                              key_in, best_seq_in, ckey[cur], key_out, mean[cur], std_[cur], bseq[cur],
                                              bval[cur]);
    return check_launch("plan_prologue_kernel");
  });
  if (rc != MBPO_OK) return rc;
  for (int it = 0; it < cfg->num_steps; ++it) {
    const int nxt = cur ^ 1;
    rc = mbpo_icem_sample_actions(cfg, ckey[cur], mean[cur], std_[cur], B, actions, ckey[nxt],
                                  general ? pkeys : nullptr, stream);
    if (rc != MBPO_OK) return rc;
    if (general) {
      // one rollout per particle key, horizon mean, mean / max over the particles (:144-160)
      rc = mbpo_system_objective(cfg->system_kind, static_cast<const MbpoGeneralSystemParams*>(sys_params_host),
                                 cfg->prng_mode, cfg->horizon, x0, actions, pkeys, B, static_cast<int>(M),
                                 cfg->num_particles, cfg->summarize, values, nullptr, nullptr, nullptr, stream);
      if (rc != MBPO_OK) return rc;
    } else if (cfg->system_kind == MBPO_SYSTEM_MLP_ENSEMBLE) {
      // particles = ensemble members; the kernel summarises over them itself (:160)
      rc = mbpo_ensemble_rollout(static_cast<const MbpoMlpEnsembleParams*>(sys_params_host), cfg->horizon, x0, actions,
                                 B, static_cast<int>(M), cfg->summarize, values, stream);
      if (rc != MBPO_OK) return rc;
    } else {
      rc = mbpo_rollout_actions(cfg->system_kind, sys_params_host, cfg->math_mode, cfg->horizon, cfg->action_dim,
                                cfg->x_dim, x0, actions, B, static_cast<int>(M), values, nullptr, nullptr, nullptr,
                                stream);
      if (rc != MBPO_OK) return rc;
      if (cfg->num_particles > 1 && cfg->summarize == MBPO_SUMMARIZE_MEAN) {
        const long long n = static_cast<long long>(b * M);
        summarize_particles_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(values, n,
                                                                                           cfg->num_particles,
                                                                                           cfg->summarize);
        rc = check_launch("summarize_particles_kernel");
        if (rc != MBPO_OK) return rc;
      }
    }
    rc = mbpo_icem_elite_refit(cfg, actions, values, mean[cur], std_[cur], bval[cur], bseq[cur], B, mean[nxt],
                               std_[nxt], bval[nxt], bseq[nxt], nullptr, stream);
    if (rc != MBPO_OK) return rc;
    cur = nxt;
  }
  // cur == 0 here; best value lives in the workspace, copy it out
  const cudaError_t e = cudaMemcpyAsync(best_value_out, bval[cur], b * sizeof(float), cudaMemcpyDeviceToDevice, st);
  if (e != cudaSuccess) return fail(MBPO_ECUDA, "plan_staged copy: %s", cudaGetErrorString(e));
  return MBPO_OK;
}

// ---- objective tail and array-valued bounds (the general staged plan composes these) -----------------
int mbpo_icem_penalize(float* values, const float* cost, long long n, int num_particles, int summarize_reward,
                       int summarize_cost, float lambda_constraint, void* stream) {
  MBPO_REQUIRE(values, "penalize: null values");
  MBPO_REQUIRE(n >= 0 && num_particles >= 1, "penalize: bad sizes");
  MBPO_REQUIRE((summarize_reward == 0 || summarize_reward == 1) && (summarize_cost == 0 || summarize_cost == 1),
               "penalize: bad summarize");
  if (n == 0) return MBPO_OK;
  penalize_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, as_stream(stream)>>>(
      values, cost, n, num_particles, summarize_reward, summarize_cost, lambda_constraint);
  return check_launch("penalize_kernel");
}

int mbpo_icem_penalize_particles(float* values_out, const float* reward, int horizon, const float* cost, long long n,
                                 int num_particles, int summarize_reward, int summarize_cost, float lambda_constraint,
                                 void* stream) {
  MBPO_REQUIRE(n >= 0 && num_particles >= 1 && horizon >= 1, "penalize_particles: bad sizes");
  MBPO_REQUIRE((summarize_reward == 0 || summarize_reward == 1) && (summarize_cost == 0 || summarize_cost == 1),
               "penalize_particles: bad summarize");
  if (n == 0) return MBPO_OK;
  MBPO_REQUIRE(values_out && reward, "penalize_particles: null pointer");
  penalize_particles_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, as_stream(stream)>>>(
      values_out, reward, horizon, cost, n, num_particles, summarize_reward, summarize_cost, lambda_constraint);
  return check_launch("penalize_particles_kernel");
}

int mbpo_icem_clip_actions(float* actions, const float* u_min, const float* u_max, int B, int M, int N, int D,
                           void* stream) {
  MBPO_REQUIRE(B >= 0 && M >= 0 && N >= 0 && N <= M && D >= 1, "clip_actions: bad sizes");
  const long long total = static_cast<long long>(B) * M * D;
  if (total == 0) return MBPO_OK;
  MBPO_REQUIRE(actions && u_min && u_max, "clip_actions: null pointer");
  clip_actions_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, as_stream(stream)>>>(actions, u_min, u_max,
                                                                                                 total, M, N, D);
  return check_launch("clip_actions_kernel");
}

// ---- closed-loop MPC -------------------------------------------------------------------------------
int mbpo_icem_mpc_closed_loop(const MbpoIcemCfg* cfg, const void* sys_params_host, const float* x0,
                              const uint32_t* key_in, const float* best_seq_in, int B, int num_mpc_steps,
                              float* states_out, float* rewards_out, float* actions_out, float* best_seq_out,
                              uint32_t* key_out, void* stream) {
  return mbpo_icem_mpc_closed_loop_clustered(cfg, sys_params_host, x0, key_in, best_seq_in, B, num_mpc_steps,
                                             states_out, rewards_out, actions_out, best_seq_out, key_out, -1, stream);
}

int mbpo_icem_mpc_closed_loop_clustered(const MbpoIcemCfg* cfg, const void* sys_params_host, const float* x0,
                                        const uint32_t* key_in, const float* best_seq_in, int B, int num_mpc_steps,
                                        float* states_out, float* rewards_out, float* actions_out,
                                        float* best_seq_out, uint32_t* key_out, int cluster_size, void* stream) {
  MBPO_REQUIRE(num_mpc_steps >= 0, "mpc_closed_loop: num_mpc_steps < 0");
  MpcArgs m;
  m.T = num_mpc_steps;
  m.states_out = states_out;
  m.rewards_out = rewards_out;
  m.actions_out = actions_out;
  return run_plan(cfg, sys_params_host, x0, key_in, best_seq_in, B, best_seq_out, nullptr, key_out, nullptr, &m,
                  cluster_size, stream);
}

int mbpo_icem_mpc_closed_loop_general(const MbpoIcemCfg* cfg, const MbpoGeneralSystemParams* sys_params_host,
                                      const float* x0, const uint32_t* key_in, const float* best_seq_in,
                                      const uint32_t* sys_keys_in, int B, int num_mpc_steps, float* states_out,
                                      float* rewards_out, float* actions_out, float* best_seq_out, uint32_t* key_out,
                                      uint32_t* sys_keys_out, int cluster_size, void* stream) {
  int rc = validate_cfg(cfg);
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(B >= 0, "mpc_closed_loop_general: B < 0");
  MBPO_REQUIRE(num_mpc_steps >= 0, "mpc_closed_loop_general: num_mpc_steps < 0");
  int X, A;
  bool keyed = false;
  if (!general_plan_kind(cfg->system_kind, &X, &A))
    return fail(MBPO_EUNSUPPORTED, "mpc_closed_loop_general: system_kind %d is not a general System (the pendulum "
                "has mbpo_icem_mpc_closed_loop)", cfg->system_kind);
  general_system_dims(cfg->system_kind, &X, &A, &keyed);
  if (!plan_fusable(cfg, true)) return MBPO_EUNSUPPORTED;
  if (B == 0) return MBPO_OK;
  MBPO_REQUIRE(sys_params_host && x0 && key_in && best_seq_in && best_seq_out && key_out,
               "mpc_closed_loop_general: null pointer");
  MBPO_REQUIRE(num_mpc_steps == 0 || (states_out && rewards_out && actions_out),
               "mpc_closed_loop_general: null output");
  MBPO_REQUIRE(!keyed || sys_keys_in, "mpc_closed_loop_general: system_kind %d draws from its key: sys_keys_in is null",
               cfg->system_kind);
  MBPO_REQUIRE(sys_keys_out == nullptr || sys_keys_in, "mpc_closed_loop_general: sys_keys_out without sys_keys_in");
  GeneralMpcArgs m;
  m.T = num_mpc_steps;
  m.states_out = states_out;
  m.rewards_out = rewards_out;
  m.actions_out = actions_out;
  m.sys_key_in = sys_keys_in;
  m.sys_key_out = sys_keys_out;
  return run_general_plan(cfg, sys_params_host, x0, key_in, best_seq_in, B, best_seq_out, nullptr, key_out, nullptr,
                          &m, cluster_size, stream);
}

// ---- policy in the env loop: actor_step / generate_unroll / get_experience ------------------------------
extern "C++" {
namespace {
template <int PRNG, int MATH>
int launch_actor(const mbpo::ActorArgs& a, cudaStream_t st) {
  using namespace mbpo;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  // one wave, one CTA per SM: a warp carries 64 envs; warps = ceil(E / 64 / SMs), at most ACT_MAX_THREADS / 32
  const int warps_total = (a.E + 63) / 64;
  int warps = (warps_total + sms - 1) / sms;
  if (warps > ACT_MAX_THREADS / 32) warps = ACT_MAX_THREADS / 32;
  if (warps < 1) warps = 1;
  const int threads = warps * 32;
  ActorSmem lay;
  int off = 0;
  auto take = [&](int n) { const int o = off; off += (n + 3) / 4 * 4; return o; };
  lay.w[0] = take(3 * ACT_W);
  for (int l = 1; l < a.num_hidden; ++l) lay.w[l] = take(ACT_W * ACT_W);
  lay.w[a.num_hidden] = take(ACT_W * 2);
  for (int l = 0; l < a.num_hidden; ++l) lay.b[l] = take(ACT_W);
  lay.b[a.num_hidden] = take(2);
  lay.h = take(2 * ACT_W * threads);   // pairs
  const size_t smem = static_cast<size_t>(off) * sizeof(float);
  auto kernel = actor_rollout_pendulum_kernel<PRNG, MATH>;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  if (e != cudaSuccess) return fail(MBPO_ECUDA, "actor_rollout: smem attribute (%zu B): %s", smem, cudaGetErrorString(e));
  const unsigned blocks = static_cast<unsigned>((warps_total + warps - 1) / warps);
  kernel<<<blocks, threads, smem, st>>>(a, lay);
  return check_launch("actor_rollout_pendulum_kernel");
}

template <int PRNG, int MATH>
int launch_actor_tc(const mbpo::ActorArgs& a, cudaStream_t st) {
  using namespace mbpo;
  auto kernel = atc::actor_rollout_tc_kernel<PRNG, MATH>;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(atc::Smem::TOTAL));
  if (e != cudaSuccess)
    return fail(MBPO_ECUDA, "actor_rollout (tcgen05): smem attribute (%u B): %s", atc::Smem::TOTAL, cudaGetErrorString(e));
  const int tiles = (a.E + atc::TILE - 1) / atc::TILE;
  const int sms = device_sm_count();
  int tpc = (tiles + sms - 1) / sms;
  tpc = tpc < 1 ? 1 : (tpc > atc::TILES_PER_CTA ? atc::TILES_PER_CTA : tpc);
  ActorArgs b = a;
  b.tiles_per_cta = tpc;
  const unsigned blocks = static_cast<unsigned>((tiles + tpc - 1) / tpc);
  kernel<<<blocks, atc::THREADS, atc::Smem::TOTAL, st>>>(b);
  return check_launch("actor_rollout_tc_kernel");
}
template <int PRNG, int MATH>
int launch_actor_tc_wide(const mbpo::ActorArgs& a, cudaStream_t st) {
  using namespace mbpo;
  auto kernel = atcw::actor_rollout_tc_wide_kernel<PRNG, MATH>;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(atcw::WSmem::TOTAL));
  if (e != cudaSuccess)
    return fail(MBPO_ECUDA, "actor_rollout (tcgen05, wide): smem attribute (%u B): %s", atcw::WSmem::TOTAL,
                cudaGetErrorString(e));
  // fewer live rows per CTA while that still leaves an SM for every CTA (the issue slots of an SM bound a step)
  const int sms = device_sm_count();
  ActorArgs b = a;
  b.rows_per_cta = a.E <= 32 * sms ? 32 : (a.E <= 64 * sms ? 64 : atc::TILE);
  const unsigned ctas = static_cast<unsigned>((a.E + b.rows_per_cta - 1) / b.rows_per_cta);
  kernel<<<ctas, atcw::WTHREADS, atcw::WSmem::TOTAL, st>>>(b);
  return check_launch("actor_rollout_tc_wide_kernel");
}
}  // namespace
}  // extern "C++"

int mbpo_actor_rollout(int system_kind, const void* sys_params_host, int math_mode, int prng_mode,
                       const MbpoPolicyParams* policy_host, int deterministic, int key_convention,
                       const uint32_t* key_in, int episode_length, int action_repeat, float* obs, float* steps,
                       float* done, const float* first_obs, int E, int T, float* action_out, float* reward_out,
                       float* discount_out, float* next_observation_out, float* truncation_out, uint32_t* key_out,
                       void* stream) {
  return mbpo_actor_rollout_extras(system_kind, sys_params_host, math_mode, prng_mode, policy_host, deterministic,
                                   key_convention, key_in, episode_length, action_repeat, obs, steps, done, first_obs,
                                   E, T, action_out, reward_out, discount_out, next_observation_out, truncation_out,
                                   key_out, nullptr, nullptr, stream);
}

int mbpo_actor_rollout_extras(int system_kind, const void* sys_params_host, int math_mode, int prng_mode,
                              const MbpoPolicyParams* policy_host, int deterministic, int key_convention,
                              const uint32_t* key_in, int episode_length, int action_repeat, float* obs,
                              float* steps, float* done, const float* first_obs, int E, int T, float* action_out,
                              float* reward_out, float* discount_out, float* next_observation_out,
                              float* truncation_out, uint32_t* key_out, float* raw_action_out, float* log_prob_out,
                              void* stream) {
  MBPO_REQUIRE(system_kind == MBPO_SYSTEM_PENDULUM || system_kind == MBPO_SYSTEM_MLP_ENSEMBLE,
               "actor_rollout: unknown system_kind %d", system_kind);
  if (system_kind != MBPO_SYSTEM_PENDULUM)
    return fail(MBPO_EUNSUPPORTED, "actor_rollout: only MBPO_SYSTEM_PENDULUM has an inlined step");
  MBPO_REQUIRE(sys_params_host && policy_host && key_in, "actor_rollout: null pointer");
  MBPO_REQUIRE((raw_action_out == nullptr) == (log_prob_out == nullptr),
               "actor_rollout: raw_action_out and log_prob_out come together");
  if (E > 0 && T > 0) {                      // empty arrays have no address
    MBPO_REQUIRE(obs && steps && done && first_obs, "actor_rollout: null pointer");
    MBPO_REQUIRE(action_out && reward_out && discount_out && next_observation_out && truncation_out,
                 "actor_rollout: every Transition buffer is required");
  }
  MBPO_REQUIRE(math_mode == 0 || math_mode == 1, "actor_rollout: bad math_mode %d", math_mode);
  MBPO_REQUIRE(prng_mode == 0 || prng_mode == 1, "actor_rollout: bad prng_mode %d", prng_mode);
  MBPO_REQUIRE(key_convention >= 0 && key_convention <= 2, "actor_rollout: bad key_convention %d", key_convention);
  MBPO_REQUIRE(E >= 0 && T >= 0 && episode_length >= 1 && action_repeat >= 1, "actor_rollout: bad sizes");
  mbpo::ActorArgs a;
  int rc = fill_policy("actor_rollout", policy_host, E, PendulumSys::X, PendulumSys::A, a);
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(policy_host->head == MBPO_HEAD_NORMAL_TANH || policy_host->head == MBPO_HEAD_BPTT_ACTOR,
               "actor_rollout: bad policy head %d", policy_host->head);
  MBPO_REQUIRE(policy_host->kernel >= MBPO_ACTOR_AUTO && policy_host->kernel <= MBPO_ACTOR_TCGEN05_WIDE,
               "actor_rollout: bad policy kernel selector %d", policy_host->kernel);
  cudaStream_t st = as_stream(stream);
  if (E == 0 || T == 0) return copy_async(key_out, key_in, key_out ? 2 * sizeof(uint32_t) : 0, st, "actor_rollout");
  a.sys = *static_cast<const MbpoPendulumParams*>(sys_params_host);
  a.E = E; a.T = T; a.episode_length = episode_length; a.action_repeat = action_repeat;
  a.deterministic = deterministic; a.key_convention = key_convention;
  a.head = policy_host->head; a.shared_noise = policy_host->shared_noise;
  a.sig_bias = policy_host->sig_bias; a.sig_min = policy_host->sig_min; a.sig_max = policy_host->sig_max;
  a.action_clip = policy_host->action_clip;
  a.key_in = key_in;
  a.obs = obs; a.steps = steps; a.done = done; a.first_obs = first_obs;
  a.action_out = action_out; a.reward_out = reward_out; a.discount_out = discount_out;
  a.next_observation_out = next_observation_out; a.truncation_out = truncation_out; a.key_out = key_out;
  a.raw_action_out = raw_action_out; a.log_prob_out = log_prob_out;
  const bool tc_ok = a.num_hidden >= 2 && a.num_hidden <= 1 + mbpo::atc::MAX_HH;
  if ((policy_host->kernel == MBPO_ACTOR_TCGEN05 || policy_host->kernel == MBPO_ACTOR_TCGEN05_WIDE) && !tc_ok)
    return fail(MBPO_EUNSUPPORTED, "actor_rollout: the tcgen05 kernel holds 1..%d hidden -> hidden layers (got %d hidden layers)",
                mbpo::atc::MAX_HH, a.num_hidden);
  // few envs (at most one 128-env tile per SM): the latency kernel; otherwise the throughput kernel
  const bool wide = policy_host->kernel == MBPO_ACTOR_TCGEN05_WIDE ||
                    (policy_host->kernel == MBPO_ACTOR_AUTO && (E + mbpo::atc::TILE - 1) / mbpo::atc::TILE <= device_sm_count());
  return with_prng_math(prng_mode, math_mode, [&](auto P, auto M) {
    if (tc_ok && wide) return launch_actor_tc_wide<P, M>(a, st);
    if (tc_ok && policy_host->kernel != MBPO_ACTOR_CUDA_CORES) return launch_actor_tc<P, M>(a, st);
    return launch_actor<P, M>(a, st);
  });
}

// ---- reverse pass through System.step rollouts, lambda returns (SURVEY 8f-4) ---------------------------
int mbpo_rollout_adjoint(int system_kind, const void* sys_params_host, int x_dim, int action_dim, int E, int T,
                         long long stride_t, long long stride_e, long long stride_xt, long long stride_xe,
                         const float* observation, const float* action, const float* g_reward,
                         const float* g_next_obs, const float* g_obs, const float* g_action_in,
                         float* g_action_out, float* g_x0_out, void* stream) {
  if (system_kind != MBPO_SYSTEM_PENDULUM)
    return fail(MBPO_EUNSUPPORTED, "rollout_adjoint: only MBPO_SYSTEM_PENDULUM has a hand-written adjoint");
  MBPO_REQUIRE(action_dim == 1 && x_dim == 3, "rollout_adjoint: pendulum needs action_dim == 1, x_dim == 3");
  MBPO_REQUIRE(E >= 0 && T >= 0, "rollout_adjoint: negative size");
  if (E == 0) return MBPO_OK;
  MBPO_REQUIRE(sys_params_host && observation && action && g_action_out, "rollout_adjoint: null pointer");
  mbpo::AdjointArgs a;
  a.sys = *static_cast<const MbpoPendulumParams*>(sys_params_host);
  a.E = E; a.T = T; a.st_t = stride_t; a.st_e = stride_e; a.sx_t = stride_xt; a.sx_e = stride_xe;
  a.observation = observation; a.action = action; a.g_reward = g_reward; a.g_next_obs = g_next_obs;
  a.g_obs = g_obs; a.g_action_in = g_action_in; a.g_action_out = g_action_out; a.g_x0_out = g_x0_out;
  mbpo::rollout_adjoint_pendulum_kernel<<<(E + 127) / 128, 128, 0, as_stream(stream)>>>(a);
  return check_launch("rollout_adjoint_pendulum_kernel");
}

int mbpo_rollout_adjoint_general(int system_kind, const MbpoGeneralSystemParams* params_host, int E, int T,
                                 long long stride_t, long long stride_e, long long stride_xt, long long stride_xe,
                                 long long stride_at, long long stride_ae, const float* observation,
                                 const float* action, const float* g_reward, const float* g_next_obs,
                                 const float* g_obs, const float* g_action_in, float* g_action_out, float* g_x0_out,
                                 void* stream) {
  if (system_kind == MBPO_SYSTEM_PENDULUM)
    return fail(MBPO_EINVAL, "rollout_adjoint_general: MBPO_SYSTEM_PENDULUM has its own entry point "
                "(mbpo_rollout_adjoint)");
  int X, A;
  bool keyed;
  if (general_system_dims(system_kind, &X, &A, &keyed) != MBPO_OK)
    return fail(MBPO_EUNSUPPORTED, "rollout_adjoint_general: system_kind %d is not one of the general Systems "
                "(NOISY_PENDULUM, POINT_MASS)", system_kind);
  MBPO_REQUIRE(E >= 0 && T >= 0, "rollout_adjoint_general: negative size");
  if (E == 0) return MBPO_OK;
  MBPO_REQUIRE(params_host && (T == 0 || (observation && action && g_action_out)),   // T == 0: only g_x0_out
               "rollout_adjoint_general: null pointer");
  mbpo::AdjointGeneralArgs a;
  a.sys = *params_host;
  a.E = E; a.T = T; a.st_t = stride_t; a.st_e = stride_e; a.sx_t = stride_xt; a.sx_e = stride_xe;
  a.sa_t = stride_at; a.sa_e = stride_ae;
  a.observation = observation; a.action = action; a.g_reward = g_reward; a.g_next_obs = g_next_obs;
  a.g_obs = g_obs; a.g_action_in = g_action_in; a.g_action_out = g_action_out; a.g_x0_out = g_x0_out;
  return with_system<NoisyPendulumSys, PointMassSys>(system_kind, [&](auto t) {
    mbpo::rollout_adjoint_general_kernel<typename decltype(t)::type><<<(E + 127) / 128, 128, 0, as_stream(stream)>>>(a);
    return check_launch("rollout_adjoint_general_kernel");
  });
}

extern "C++" {
namespace {
mbpo::LambdaArgs lambda_args(int E, int T, long long stride_t, long long stride_e, double discount, double lambda_) {
  mbpo::LambdaArgs a;
  a.E = E; a.T = T; a.st_t = stride_t; a.st_e = stride_e;
  // python floats are weakly typed: `discount * lambda_` and `1 - lambda_` are evaluated in double and
  // rounded once when they meet the float32 arrays (optimizer_utils.py:127-130)
  a.discount = static_cast<float>(discount);
  a.lambda_ = static_cast<float>(lambda_);
  a.one_minus_lambda = static_cast<float>(1.0 - lambda_);
  a.discount_lambda = static_cast<float>(discount * lambda_);
  return a;
}
}  // namespace
}  // extern "C++"

int mbpo_lambda_return(const float* reward, const float* next_values, int E, int T, long long stride_t,
                       long long stride_e, double discount, double lambda_, float* returns_out, void* stream) {
  MBPO_REQUIRE(E >= 0 && T >= 0, "lambda_return: negative size");
  if (E == 0 || T == 0) return MBPO_OK;
  MBPO_REQUIRE(reward && next_values && returns_out, "lambda_return: null pointer");
  mbpo::LambdaArgs a = lambda_args(E, T, stride_t, stride_e, discount, lambda_);
  a.reward = reward; a.next_values = next_values; a.out = returns_out; a.out2 = nullptr;
  mbpo::lambda_return_kernel<<<(E + 127) / 128, 128, 0, as_stream(stream)>>>(a);
  return check_launch("lambda_return_kernel");
}

int mbpo_lambda_return_vjp(const float* g_returns, int E, int T, long long stride_t, long long stride_e,
                           double discount, double lambda_, float* g_reward_out, float* g_next_values_out,
                           void* stream) {
  MBPO_REQUIRE(E >= 0 && T >= 0, "lambda_return_vjp: negative size");
  if (E == 0 || T == 0) return MBPO_OK;
  MBPO_REQUIRE(g_returns && g_reward_out && g_next_values_out, "lambda_return_vjp: null pointer");
  mbpo::LambdaArgs a = lambda_args(E, T, stride_t, stride_e, discount, lambda_);
  a.reward = g_returns; a.next_values = nullptr; a.out = g_reward_out; a.out2 = g_next_values_out;
  mbpo::lambda_return_transpose_kernel<<<(E + 127) / 128, 128, 0, as_stream(stream)>>>(a);
  return check_launch("lambda_return_transpose_kernel");
}

// ---- stage 4 ---------------------------------------------------------------------------------------
int mbpo_mlp_dynamics_forward(const MbpoMlpEnsembleParams* p, const float* inp, const int32_t* member, int R,
                              float* delta_out, void* stream) {
  MBPO_REQUIRE(p && inp && member && delta_out, "mlp_dynamics_forward: null pointer");
  MBPO_REQUIRE(R >= 0, "mlp_dynamics_forward: R < 0");
  MBPO_REQUIRE(p->w_in && p->b_in && p->w_h && p->b_h && p->w_out && p->b_out, "mlp_dynamics_forward: null weights");
  if (R == 0) return MBPO_OK;
  const int rc = tc::launch_mlp_forward_tc(*p, inp, member, R, delta_out, as_stream(stream), g_err, sizeof(g_err));
  if (rc != MBPO_OK) return rc;
  return check_launch("mlp_dynamics_forward");
}

int mbpo_ensemble_rollout(const MbpoMlpEnsembleParams* p, int horizon, const float* x0, const float* actions, int B,
                          int M, int summarize, float* returns_out, void* stream) {
  MBPO_REQUIRE(p && x0 && actions && returns_out, "ensemble_rollout: null pointer");
  MBPO_REQUIRE(p->w_in && p->b_in && p->w_h && p->b_h && p->w_out && p->b_out, "ensemble_rollout: null weights");
  MBPO_REQUIRE(horizon >= 1 && B >= 0 && M >= 0, "ensemble_rollout: bad sizes");
  MBPO_REQUIRE(summarize == 0 || summarize == 1, "ensemble_rollout: bad summarize %d", summarize);
  if (static_cast<long long>(B) * M == 0) return MBPO_OK;
  const int rc = ens::launch_ensemble_rollout_auto(*p, horizon, x0, actions, B, M, summarize, returns_out, nullptr,
                                                   nullptr, as_stream(stream), g_err, sizeof(g_err));
  if (rc != MBPO_OK) return rc;
  return check_launch("ensemble_rollout_kernel");
}

int mbpo_ensemble_rollout_transitions(const MbpoMlpEnsembleParams* p, int horizon, const float* x0,
                                      const float* actions, int B, int M, float* obs_out, float* reward_out,
                                      void* stream) {
  MBPO_REQUIRE(p && x0 && actions && obs_out && reward_out, "ensemble_rollout_transitions: null pointer");
  MBPO_REQUIRE(p->w_in && p->b_in && p->w_h && p->b_h && p->w_out && p->b_out,
               "ensemble_rollout_transitions: null weights");
  MBPO_REQUIRE(horizon >= 1 && B >= 0 && M >= 0, "ensemble_rollout_transitions: bad sizes");
  if (static_cast<long long>(B) * M == 0) return MBPO_OK;
  const int rc = ens::launch_ensemble_rollout_auto(*p, horizon, x0, actions, B, M, MBPO_SUMMARIZE_MEAN, nullptr,
                                                   obs_out, reward_out, as_stream(stream), g_err, sizeof(g_err));
  if (rc != MBPO_OK) return rc;
  return check_launch("ensemble_transitions_kernel");
}

// ---- the learned ensemble as a SAC / PPO env (ensemble_env_kernels.cuh) ----------------------------------------
int mbpo_ensemble_env_rollout(const MbpoMlpEnsembleParams* p, int prng_mode, const MbpoPolicyParams* policy_host,
                              int deterministic, int key_convention, const uint32_t* key_in, int episode_length,
                              int action_repeat, const int32_t* env_order, const int32_t* member_offsets, float* obs,
                              float* steps, float* done, const float* first_obs, int E, int T, const float* actions,
                              float* action_out, float* reward_out, float* discount_out, float* next_observation_out,
                              float* truncation_out, uint32_t* key_out, float* raw_action_out, float* log_prob_out,
                              void* stream) {
  using namespace mbpo;
  using namespace mbpo::ens;
  MBPO_REQUIRE(p, "ensemble_env_rollout: null pointer");
  MBPO_REQUIRE(p->w_in && p->b_in && p->w_h && p->b_h && p->w_out && p->b_out, "ensemble_env_rollout: null weights");
  if (p->hidden != HID || p->x_dim != 3 || p->u_dim != 1 || p->num_members < 1)
    return fail(MBPO_EUNSUPPORTED, "ensemble_env_rollout: the tcgen05 kernel needs hidden == 256, x_dim == 3, "
                "u_dim == 1 and at least one member (got %d, %d, %d, %d members)", p->hidden, p->x_dim, p->u_dim,
                p->num_members);
  MBPO_REQUIRE(prng_mode == 0 || prng_mode == 1, "ensemble_env_rollout: bad prng_mode %d", prng_mode);
  MBPO_REQUIRE(E >= 0 && T >= 0 && episode_length >= 1 && action_repeat >= 1, "ensemble_env_rollout: bad sizes");
  MBPO_REQUIRE(static_cast<long long>(T) * action_repeat < (1ll << 31), "ensemble_env_rollout: T * action_repeat "
               "overflows int");
  EnsEnvArgs a = {};
  size_t smem = ens::Smem::TOTAL;
  if (policy_host) {
    MBPO_REQUIRE(key_in, "ensemble_env_rollout: null pointer");
    MBPO_REQUIRE((raw_action_out == nullptr) == (log_prob_out == nullptr),
                 "ensemble_env_rollout: raw_action_out and log_prob_out come together");
    MBPO_REQUIRE(key_convention >= 0 && key_convention <= 2, "ensemble_env_rollout: bad key_convention %d",
                 key_convention);
    MBPO_REQUIRE(policy_host->head == MBPO_HEAD_NORMAL_TANH || policy_host->head == MBPO_HEAD_BPTT_ACTOR,
                 "ensemble_env_rollout: bad policy head %d", policy_host->head);
    MBPO_REQUIRE(policy_host->kernel >= MBPO_ACTOR_AUTO && policy_host->kernel <= MBPO_ACTOR_TCGEN05_WIDE,
                 "ensemble_env_rollout: bad policy kernel selector %d", policy_host->kernel);
    if (policy_host->head != MBPO_HEAD_NORMAL_TANH || policy_host->shared_noise)
      return fail(MBPO_EUNSUPPORTED, "ensemble_env_rollout: the BPTT actor head (one shared draw) runs on the "
                  "pendulum only; the learned ensemble takes the NormalTanh head");
    if (policy_host->kernel == MBPO_ACTOR_TCGEN05 || policy_host->kernel == MBPO_ACTOR_TCGEN05_WIDE)
      return fail(MBPO_EUNSUPPORTED, "ensemble_env_rollout: the tcgen05 policy kernels hold the pendulum only; in "
                  "the ensemble's env kernel the policy runs on the CUDA cores (MBPO_ACTOR_AUTO or "
                  "MBPO_ACTOR_CUDA_CORES)");
    const int rc = fill_policy("ensemble_env_rollout", policy_host, E, 3, 1, a.pol);
    if (rc != MBPO_OK) return rc;
    // the policy's weights and biases at their flax shapes, past the model's shared memory
    GeneralActorSmem lay;
    int off = 0;
    auto take = [&](int n) { const int o = off; off += (n + 3) / 4 * 4; return o; };
    lay.w[0] = take(3 * ACT_W);
    for (int l = 1; l < a.pol.num_hidden; ++l) lay.w[l] = take(ACT_W * ACT_W);
    lay.w[a.pol.num_hidden] = take(ACT_W * 2);
    for (int l = 0; l < a.pol.num_hidden; ++l) lay.b[l] = take(ACT_W);
    lay.b[a.pol.num_hidden] = take(2);
    lay.h = 0;
    lay.total = off;
    a.lay = lay;
    smem = ENV_POLICY_W + static_cast<size_t>(off) * sizeof(float);
    if (smem > 227 * 1024)
      return fail(MBPO_EUNSUPPORTED, "ensemble_env_rollout: a policy of %d hidden layers needs %zu B of shared memory "
                  "beside the ensemble's %u B; a CTA has 232448 B (1..2 hidden layers of width 64 fit)",
                  a.pol.num_hidden, static_cast<size_t>(off) * sizeof(float), ENV_POLICY_W);
  }
  cudaStream_t st = as_stream(stream);
  if (E == 0 || T == 0)          // empty arrays have no address; the carry key passes through
    return policy_host ? copy_async(key_out, key_in, key_out ? 2 * sizeof(uint32_t) : 0, st, "ensemble_env_rollout")
                       : MBPO_OK;
  MBPO_REQUIRE(env_order && member_offsets && obs && steps && done && first_obs, "ensemble_env_rollout: null pointer");
  MBPO_REQUIRE(reward_out && discount_out && next_observation_out && truncation_out && (policy_host ? action_out : actions),
               "ensemble_env_rollout: every Transition buffer is required (actions, or action_out with a policy)");
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return fail(MBPO_ECUDA, "ensemble_env_rollout: cuTensorMapEncodeTiled is not available from the driver");
  CUtensorMap map;
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(HID), static_cast<cuuint64_t>(p->num_members) * 2 * HID};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(HID) * 2};
  const cuuint32_t box[2] = {8, 128};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult cr = enc(&map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<uint16_t*>(p->w_h), dims, strides, box,
                          estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS)
    return fail(MBPO_ECUDA, "ensemble_env_rollout: cuTensorMapEncodeTiled failed (CUresult %d)", static_cast<int>(cr));
  a.num_members = p->num_members; a.E = E; a.T = T; a.episode_length = episode_length; a.action_repeat = action_repeat;
  // each member's envs fill whole tiles but its last: at most one partial tile per member
  const long long tiles = (static_cast<long long>(E) + 2 * TILE_M - 1) / (2 * TILE_M) + p->num_members - 1;
  a.num_tiles = static_cast<int>(tiles);
  a.policy = policy_host ? 1 : 0;
  a.deterministic = deterministic ? 1 : 0;
  a.key_convention = policy_host ? key_convention : 0;
  a.w_in = p->w_in; a.b_in = p->b_in; a.b_h = p->b_h; a.w_out = p->w_out; a.b_out = p->b_out; a.reward = p->reward;
  a.env_order = env_order; a.member_offsets = member_offsets;
  a.obs = obs; a.steps = steps; a.done = done; a.first_obs = first_obs; a.actions = actions;
  a.key_in = policy_host ? key_in : nullptr; a.key_out = policy_host ? key_out : nullptr;
  a.action_out = action_out; a.reward_out = reward_out; a.discount_out = discount_out;
  a.next_observation_out = next_observation_out; a.truncation_out = truncation_out;
  a.raw_action_out = (policy_host && !deterministic) ? raw_action_out : nullptr;
  a.log_prob_out = (policy_host && !deterministic) ? log_prob_out : nullptr;
  const int pairs_max = device_sm_count() / 2;
  const int pairs = static_cast<int>(tiles < pairs_max ? tiles : pairs_max);
  return with_prng(prng_mode, [&](auto P) {
    auto kernel = ensemble_env_kernel<P>;
    const cudaError_t ce = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                static_cast<int>(smem));
    if (ce != cudaSuccess)
      return fail(MBPO_ECUDA, "ensemble_env_rollout: smem attribute (%zu B): %s", smem, cudaGetErrorString(ce));
    kernel<<<2 * pairs, ENS_THREADS, smem, st>>>(a, map);
    return check_launch("ensemble_env_kernel");
  });
}

}  // extern "C"

#ifdef MBPO_ENS_TRACE
extern "C" int mbpo_debug_ens_trace(long long* out_host) {
  return cudaMemcpyFromSymbol(out_host, mbpo::ens::g_ens_trace, sizeof(long long) * 256) == cudaSuccess ? 0 : -3;
}
#endif
