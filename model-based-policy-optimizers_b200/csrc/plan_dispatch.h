// Per-horizon kernel entry points.  Each horizon H in MBPO_FOR_EACH_H is compiled in its own
// translation unit (plan_inst.cu with -DMBPO_INST_H=H) so the build parallelises; this header
// declares what those units define.
#pragma once
#include "host_util.h"
#include "icem_cluster_kernels.cuh"
#include "icem_general_cluster_kernels.cuh"
#include "icem_kernels.cuh"

namespace mbpo {

// Fused plan (mpc == nullptr) or closed-loop MPC (mpc != nullptr); selects PRNG / MATH
// template variants from prng_mode / math_mode.  cluster > 1: every problem is spread over a thread-block cluster
// of that many CTAs (icem_cluster_kernels.cuh; same bits, for few problems); 0 / 1: one CTA per problem.
template <int H>
int plan_entry(int prng_mode, int math_mode, const PlanArgs& a, const MpcArgs* mpc, cudaStream_t st, int cluster);

// The same for a horizon without an unrolled instance (plan_rt.cu; PlanArgs::H).
int plan_entry_rt(int prng_mode, int math_mode, const PlanArgs& a, const MpcArgs* mpc, cudaStream_t st);

// Fused plan (mpc == nullptr) or closed-loop MPC over the general Systems (MBPO_SYSTEM_NOISY_PENDULUM,
// MBPO_SYSTEM_POINT_MASS): one CTA per problem (cluster 0 / 1: icem_plan_general_kernel, icem_mpc_general_kernel) or
// one cluster of that many CTAs per problem (icem_general_cluster_kernels.cuh; same bits).
template <int H>
int general_plan_entry(int system_kind, int prng_mode, const PlanArgs& a, const GeneralMpcArgs* mpc, cudaStream_t st,
                       int cluster);

// plan_cluster_capacity for the general cluster kernels (their block size depends on the particles P as well).
template <int H>
int general_plan_cluster_capacity(int system_kind, int prng_mode, bool mpc, int N, int Np, int K, int P, int cluster);

// How many clusters of `cluster` CTAs of the cluster plan (mpc: of the closed loop) run at once on the current device
// (cudaOccupancyMaxActiveClusters: the GPCs, not the SM count, decide -- 7 of 16, 15 of 8, 33 of 4, 74 of 2 on a
// B200); 0 if the size cannot be launched.
template <int H>
int plan_cluster_capacity(int prng_mode, int math_mode, bool mpc, int N, int Np, int K, int cluster);

// Cluster size for B problems given the capacities of sizes 16, 8, 4, 2 (cap[0..3]): the largest size whose clusters
// all run at once (a second round of clusters costs a whole plan) with 32 .. 256 candidates per CTA; 0: one CTA per
// problem.
inline int plan_cluster_choice(int B, int N, const int cap[4]) {
  if (B <= 0) return 0;
  for (int i = 0, c = 16; i < 4; ++i, c >>= 1) {
    const int R = (N + c - 1) / c;
    if (R >= 32 && R <= 256 && B <= cap[i]) return c;
  }
  return 0;
}

// vmap(powerlaw_psd_gaussian) over M keys.
template <int H>
int noise_entry(int prng_mode, const ScaleTable& tbl, const uint32_t* keys, int M, float* noise_out,
                uint32_t* bits_out, cudaStream_t st);

// One iteration of key plumbing + sampling for B problems.
template <int H>
int sample_entry(int prng_mode, const ScaleTable& tbl, const uint32_t* carry_key, const float* mean,
                 const float* std_, int N, int Np, int A, float u_min, float u_max, int B, float* actions,
                 uint32_t* next_key, uint32_t* particle_keys, cudaStream_t st);

}  // namespace mbpo
