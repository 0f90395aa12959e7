// Instantiates the horizon-specialised kernels for H = MBPO_INST_H (see plan_dispatch.h).
#ifndef MBPO_INST_H
#error "compile with -DMBPO_INST_H=<horizon>"
#endif
#include "plan_dispatch.h"

namespace mbpo {

namespace {

constexpr int kH = MBPO_INST_H;
constexpr int kPlanThreads = 256;
// Resident CTAs per SM the register budget is tuned for (shared memory may allow fewer).
constexpr int kMinBlocks = kH <= 20 ? 4 : (kH <= 30 ? 3 : 1);

template <typename Kernel>
int prepare_plan_kernel(Kernel kernel, size_t smem, int B, int* grid_out) {
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  if (e != cudaSuccess) return fail(MBPO_ECUDA, "cudaFuncSetAttribute(smem=%zu): %s", smem, cudaGetErrorString(e));
  int per_sm = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kPlanThreads, smem);
  if (e != cudaSuccess) return fail(MBPO_ECUDA, "occupancy query: %s", cudaGetErrorString(e));
  if (per_sm < 1) return fail(MBPO_EUNSUPPORTED, "plan kernel does not fit one SM (smem=%zu)", smem);
  const long long resident = static_cast<long long>(per_sm) * device_sm_count();
  *grid_out = static_cast<int>(B < resident ? B : resident);
  return MBPO_OK;
}

// Block size of a cluster CTA that owns R candidates (0: more than the kernel takes).
int cluster_threads(int R) {
  // Per chunk of 32 candidates one rollout warp (a thread per candidate) and up to seven sampling warps, which share
  // the sampling of the chunk's rows for the next iteration under the rollouts (coop_sample_rows); all warps share the
  // selection.  At least one sampling warp per chunk.
  const int chunks = (R + 31) / 32;
  int threads = 32 * COOP_WARPS_PER_CHUNK * chunks;
  if (threads > CLUSTER_MAX_THREADS) threads = CLUSTER_MAX_THREADS;
  return threads < 64 * chunks ? 0 : threads;
}

// A cluster plan is a latency path: two of its CTAs on one SM would share the issue slots of the rollout chain
// (measured at 16 CTAs per cluster: 48 -> 59 us).  Asking for more than half an SM's shared memory keeps every CTA
// on an SM of its own, and makes the occupancy answer (cluster_capacity) count exactly those placements.
size_t cluster_smem_alloc(size_t smem) {
  const size_t half_sm = 117 * 1024;
  return smem > half_sm ? smem : half_sm;
}

template <typename Kernel>
cudaError_t prepare_cluster_kernel(Kernel kernel, int cluster, size_t smem) {
  if (cluster > 8) {
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) return e;
  }
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
}

template <int PRNG, int MATH>
int cluster_capacity(bool mpc, int N, int Np, int K, int cluster) {
  const int R = (N + cluster - 1) / cluster;
  const int threads = cluster_threads(R);
  if (threads == 0) return 0;
  const size_t smem = cluster_smem_alloc(ClusterSmem<kH>::bytes(R, N, Np, K));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(cluster), 1, 1);
  cfg.blockDim = dim3(static_cast<unsigned>(threads), 1, 1);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = static_cast<unsigned>(cluster);
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  cudaError_t e;
  if (mpc) {
    auto kernel = icem_mpc_cluster_kernel<kH, PRNG, MATH>;
    e = prepare_cluster_kernel(kernel, cluster, smem);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveClusters(&n, kernel, &cfg);
  } else {
    auto kernel = icem_plan_cluster_kernel<kH, PRNG, MATH>;
    e = prepare_cluster_kernel(kernel, cluster, smem);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveClusters(&n, kernel, &cfg);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

// One problem per cluster of `cluster` CTAs (icem_cluster_kernels.cuh).
template <int PRNG, int MATH>
int launch_cluster(const PlanArgs& a, const MpcArgs* mpc, cudaStream_t st, int cluster) {
  const int R = (a.N + cluster - 1) / cluster;               // candidates per CTA, one per thread
  const int threads = cluster_threads(R);
  if (threads == 0)
    return fail(MBPO_EUNSUPPORTED, "cluster plan: %d candidates per CTA (max %d)", R, CLUSTER_MAX_THREADS / 2);
  const size_t smem = cluster_smem_alloc(ClusterSmem<kH>::bytes(R, a.N, a.Np, a.K));
  const int sms = device_sm_count();
  long long clusters = sms / cluster;
  if (clusters > a.B) clusters = a.B;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(clusters * cluster), 1, 1);
  cfg.blockDim = dim3(static_cast<unsigned>(threads), 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = static_cast<unsigned>(cluster);
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e;
  if (mpc == nullptr) {
    auto kernel = icem_plan_cluster_kernel<kH, PRNG, MATH>;
    e = prepare_cluster_kernel(kernel, cluster, smem);
    if (e != cudaSuccess)
      return fail(MBPO_ECUDA, "cluster plan attributes (cluster %d, smem %zu): %s", cluster, smem, cudaGetErrorString(e));
    e = cudaLaunchKernelEx(&cfg, kernel, a, R);   // (the all-zero row is rolled out inside, beside iteration 0's sampling)
    if (e != cudaSuccess) return fail(MBPO_ECUDA, "icem_plan_cluster_kernel launch: %s", cudaGetErrorString(e));
    return check_launch("icem_plan_cluster_kernel");
  }
  auto kernel = icem_mpc_cluster_kernel<kH, PRNG, MATH>;
  e = prepare_cluster_kernel(kernel, cluster, smem);
  if (e != cudaSuccess)
    return fail(MBPO_ECUDA, "cluster mpc attributes (cluster %d, smem %zu): %s", cluster, smem, cudaGetErrorString(e));
  e = cudaLaunchKernelEx(&cfg, kernel, a, *mpc, R);
  if (e != cudaSuccess) return fail(MBPO_ECUDA, "icem_mpc_cluster_kernel launch: %s", cudaGetErrorString(e));
  return check_launch("icem_mpc_cluster_kernel");
}

template <int PRNG, int MATH>
int launch(const PlanArgs& a, const MpcArgs* mpc, cudaStream_t st) {
  const size_t smem = PlanSmem<kH>::bytes(a.N, a.Np, a.K);
  int grid = 0;
  if (mpc == nullptr) {
    auto kernel = icem_plan_pendulum_kernel<kH, PRNG, MATH, kPlanThreads, kMinBlocks>;
    const int rc = prepare_plan_kernel(kernel, smem, a.B, &grid);
    if (rc != MBPO_OK) return rc;
    PlanArgs b = a;
    b.zero_value_precomputed = 1;   // best_value_out doubles as the hand-over buffer
    zero_row_value_kernel<MATH><<<(a.B + 127) / 128, 128, 0, st>>>(a.sys, kH, a.P, a.summarize, a.x0, a.B,
                                                                  a.best_value_out);
    const int rc2 = check_launch("zero_row_value_kernel");
    if (rc2 != MBPO_OK) return rc2;
    kernel<<<grid, kPlanThreads, smem, st>>>(b);
    return check_launch("icem_plan_pendulum_kernel");
  }
  auto kernel = icem_mpc_pendulum_kernel<kH, PRNG, MATH, kPlanThreads, kMinBlocks>;
  const int rc = prepare_plan_kernel(kernel, smem, a.B, &grid);
  if (rc != MBPO_OK) return rc;
  kernel<<<grid, kPlanThreads, smem, st>>>(a, *mpc);
  return check_launch("icem_mpc_pendulum_kernel");
}

}  // namespace

template <>
int plan_entry<MBPO_INST_H>(int prng_mode, int math_mode, const PlanArgs& a, const MpcArgs* mpc, cudaStream_t st,
                            int cluster) {
  return with_prng_math(prng_mode, math_mode, [&](auto P, auto M) {
    return cluster > 1 ? launch_cluster<P, M>(a, mpc, st, cluster) : launch<P, M>(a, mpc, st);
  });
}

template <>
int plan_cluster_capacity<MBPO_INST_H>(int prng_mode, int math_mode, bool mpc, int N, int Np, int K, int cluster) {
  return with_prng_math(prng_mode, math_mode,
                        [&](auto P, auto M) { return cluster_capacity<P, M>(mpc, N, Np, K, cluster); });
}

namespace {
template <class Sys, int PRNG>
int launch_general(const PlanArgs& a, const GeneralMpcArgs* mpc, cudaStream_t st) {
  const size_t smem = GenPlanSmem<kH, Sys::A>::bytes(a.N, a.Np, a.K) +
                      (mpc ? 4 * gen_mpc_extra_words<kH, Sys::A>() : 0);
  if (smem > 227 * 1024) return fail(MBPO_EUNSUPPORTED, "general fused plan: %zu B of shared memory", smem);
  auto run = [&](auto kernel, const char* name, auto... extra) {
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return fail(MBPO_ECUDA, "general plan smem attr (%zu): %s", smem, cudaGetErrorString(e));
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    const long long resident = static_cast<long long>(per_sm) * device_sm_count();
    const int grid = static_cast<int>(a.B < resident ? a.B : resident);
    kernel<<<grid, 256, smem, st>>>(a, extra...);
    return check_launch(name);
  };
  if (mpc == nullptr) return run(icem_plan_general_kernel<Sys, kH, PRNG>, "icem_plan_general_kernel");
  return run(icem_mpc_general_kernel<Sys, kH, PRNG>, "icem_mpc_general_kernel", *mpc);
}

// Block size of a general cluster CTA with R rows of Pe rollouts and A action dimensions each: a thread per rollout
// and per sampled noise row, at least 256 threads for the selection and the refit.
int general_cluster_threads(int R, int Pe, int A) {
  const int work = R * Pe > R * A ? R * Pe : R * A;
  const int threads = (work + 31) / 32 * 32;
  return threads < 256 ? 256 : (threads > CLUSTER_MAX_THREADS ? CLUSTER_MAX_THREADS : threads);
}

template <class Sys>
size_t general_cluster_smem(int N, int Np, int K, int P, int cluster, int* R_out) {
  const int R = (N + Np + cluster - 1) / cluster;
  *R_out = R;
  return cluster_smem_alloc(GenClusterSmem<kH, Sys::A>::bytes(R, Sys::KEYED ? P : 1, N, Np, K));
}

cudaLaunchConfig_t cluster_launch_config(int clusters, int cluster, int threads, size_t smem, cudaStream_t st,
                                         cudaLaunchAttribute* attr) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(clusters * cluster), 1, 1);
  cfg.blockDim = dim3(static_cast<unsigned>(threads), 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = static_cast<unsigned>(cluster);
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cfg;
}

template <class Sys, int PRNG>
int general_cluster_capacity(bool mpc, int N, int Np, int K, int P, int cluster) {
  int R = 0;
  const size_t smem = general_cluster_smem<Sys>(N, Np, K, P, cluster, &R);
  if (R > 256 || smem > 227 * 1024) return 0;
  cudaLaunchAttribute attr[1];
  const cudaLaunchConfig_t cfg = cluster_launch_config(1, cluster, general_cluster_threads(R, Sys::KEYED ? P : 1, Sys::A),
                                                       smem, nullptr, attr);
  int n = 0;
  cudaError_t e;
  if (mpc) {
    auto kernel = icem_mpc_general_cluster_kernel<Sys, kH, PRNG>;
    e = prepare_cluster_kernel(kernel, cluster, smem);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveClusters(&n, kernel, &cfg);
  } else {
    auto kernel = icem_plan_general_cluster_kernel<Sys, kH, PRNG>;
    e = prepare_cluster_kernel(kernel, cluster, smem);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveClusters(&n, kernel, &cfg);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

// One problem per cluster of `cluster` CTAs (icem_general_cluster_kernels.cuh).
template <class Sys, int PRNG>
int launch_general_cluster(const PlanArgs& a, const GeneralMpcArgs* mpc, cudaStream_t st, int cluster) {
  int R = 0;
  const size_t smem = general_cluster_smem<Sys>(a.N, a.Np, a.K, a.P, cluster, &R);
  if (R > 256)
    return fail(MBPO_EUNSUPPORTED, "plan: %d candidate rows per CTA of a %d-cluster (at most 256)", R, cluster);
  if (smem > 227 * 1024) return fail(MBPO_EUNSUPPORTED, "general cluster plan: %zu B of shared memory", smem);
  const int threads = general_cluster_threads(R, Sys::KEYED ? a.P : 1, Sys::A);
  long long clusters = device_sm_count() / cluster;
  if (clusters > a.B) clusters = a.B;
  cudaLaunchAttribute attr[1];
  const cudaLaunchConfig_t cfg = cluster_launch_config(static_cast<int>(clusters), cluster, threads, smem, st, attr);
  cudaError_t e;
  if (mpc == nullptr) {
    auto kernel = icem_plan_general_cluster_kernel<Sys, kH, PRNG>;
    e = prepare_cluster_kernel(kernel, cluster, smem);
    if (e != cudaSuccess)
      return fail(MBPO_ECUDA, "general cluster plan attributes (cluster %d, smem %zu): %s", cluster, smem,
                  cudaGetErrorString(e));
    e = cudaLaunchKernelEx(&cfg, kernel, a, R);
    if (e != cudaSuccess) return fail(MBPO_ECUDA, "icem_plan_general_cluster_kernel launch: %s", cudaGetErrorString(e));
    return check_launch("icem_plan_general_cluster_kernel");
  }
  auto kernel = icem_mpc_general_cluster_kernel<Sys, kH, PRNG>;
  e = prepare_cluster_kernel(kernel, cluster, smem);
  if (e != cudaSuccess)
    return fail(MBPO_ECUDA, "general cluster mpc attributes (cluster %d, smem %zu): %s", cluster, smem,
                cudaGetErrorString(e));
  e = cudaLaunchKernelEx(&cfg, kernel, a, *mpc, R);
  if (e != cudaSuccess) return fail(MBPO_ECUDA, "icem_mpc_general_cluster_kernel launch: %s", cudaGetErrorString(e));
  return check_launch("icem_mpc_general_cluster_kernel");
}
}  // namespace

template <>
int general_plan_entry<MBPO_INST_H>(int system_kind, int prng_mode, const PlanArgs& a, const GeneralMpcArgs* mpc,
                                    cudaStream_t st, int cluster) {
  return with_system<NoisyPendulumSys, PointMassSys>(system_kind, [&](auto t) {
    using Sys = typename decltype(t)::type;
    return with_prng(prng_mode, [&](auto P) {
      return cluster > 1 ? launch_general_cluster<Sys, P>(a, mpc, st, cluster) : launch_general<Sys, P>(a, mpc, st);
    });
  });
}

template <>
int general_plan_cluster_capacity<MBPO_INST_H>(int system_kind, int prng_mode, bool mpc, int N, int Np, int K, int P,
                                               int cluster) {
  const int n = with_system<NoisyPendulumSys, PointMassSys>(system_kind, [&](auto t) {
    using Sys = typename decltype(t)::type;
    return with_prng(prng_mode, [&](auto PR) { return general_cluster_capacity<Sys, PR>(mpc, N, Np, K, P, cluster); });
  });
  return n > 0 ? n : 0;
}

template <>
int noise_entry<MBPO_INST_H>(int prng_mode, const ScaleTable& tbl, const uint32_t* keys, int M, float* noise_out,
                             uint32_t* bits_out, cudaStream_t st) {
  const int threads = STAGED_THREADS;
  const unsigned blocks = static_cast<unsigned>((M + threads - 1) / threads);
  return with_prng(prng_mode, [&](auto P) {
    powerlaw_noise_kernel<kH, P><<<blocks, threads, 0, st>>>(tbl, keys, M, noise_out, bits_out);
    return check_launch("powerlaw_noise_kernel");
  });
}

template <>
int sample_entry<MBPO_INST_H>(int prng_mode, const ScaleTable& tbl, const uint32_t* carry_key, const float* mean,
                              const float* std_, int N, int Np, int A, float u_min, float u_max, int B,
                              float* actions, uint32_t* next_key, uint32_t* particle_keys, cudaStream_t st) {
  const int threads = STAGED_THREADS;
  const dim3 grid(static_cast<unsigned>(((N + Np) * A + threads - 1) / threads), static_cast<unsigned>(B));
  return with_prng(prng_mode, [&](auto P) {
    sample_actions_kernel<kH, P><<<grid, threads, 0, st>>>(tbl, carry_key, mean, std_, N, Np, A, u_min, u_max,
                                                           actions, next_key, particle_keys);
    return check_launch("sample_actions_kernel");
  });
}

#ifdef MBPO_CLUSTER_CLOCKS
extern "C" int mbpo_debug_cluster_clocks(long long* out_host) {
  return cudaMemcpyFromSymbol(out_host, g_cluster_clocks, sizeof(long long) * 64) == cudaSuccess ? 0 : -3;
}
extern "C" int mbpo_debug_select_clocks(long long* out_host) {
  return cudaMemcpyFromSymbol(out_host, g_select_clocks, sizeof(long long) * 16) == cudaSuccess ? 0 : -3;
}
#endif

}  // namespace mbpo
