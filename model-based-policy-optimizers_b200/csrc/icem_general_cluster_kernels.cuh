// Few problems, many SMs, for the general Systems (systems.cuh): one planning problem over a thread-block CLUSTER of
// C = 2, 4, 8 or 16 CTAs, like the pendulum's cluster plan (icem_cluster_kernels.cuh).
//
// The one-CTA general plan (icem_plan_general_kernel) gives each of its 256 threads whole candidates: a System that
// draws from its key rolls every candidate out once per particle, so at P = 10 one thread works through ~20
// candidate-particle rollouts one after another, and a problem takes as long at B = 1 as at B = 148.  Here CTA r owns
// the candidate rows [r R, (r + 1) R) of M = N + Np (R = ceil(M / C); rows N .. M-1 are the closure's all-zero
// kept-elite rows, :192,:245), and the unit of work inside a CTA is ONE (candidate, particle) rollout per thread.
// One iteration:
//
//   1. sampling: one thread per (row, action dimension) writes clip(mean + noise * std) into the row  (:174-191)
//   2. rollouts: one thread per (row, particle); the returns go to shared memory
//   3. one thread per row reduces its particles in particle order (__fadd_rn / fmaxf, as the one-CTA loop does) and
//      stores the total-order key into ALL C copies of skey[] (distributed shared memory)
//   4. cluster.sync()
//   5. every CTA selects on its full copy of the keys (cta_select: identical results everywhere); the owner of an
//      elite row pushes its D = H * A floats to every CTA, in rank order (ebuf[K][D])
//   6. cluster.sync()
//   7. every CTA refits for itself (rank-ordered sums on identical inputs: identical mean / std / best everywhere)
//
// A System that draws rolls out its Np kept-elite rows as distinct candidates (their own particle keys), as the
// one-CTA kernel does; for a deterministic System the first zero row is rolled out once per iteration and its value
// serves all Np.  Every number is produced by the device functions of the one-CTA kernel in the same order: the
// results are its bits for every C (tests/test_gpu_general_mpc.py).
//
// Reference: mbpo/optimizers/trajectory_optimizers/icem_optimizer.py:134-252; tests/test_icemopt.py:19-32.
#pragma once
#include "icem_cluster_kernels.cuh"

namespace mbpo {

// Shared memory of one CTA of a general cluster plan (words); R rows of this CTA, Pe rollouts per row.
template <int H, int A>
struct GenClusterSmem {
  static constexpr int D = H * A, RS = D | 1;
  static size_t bytes(int R, int Pe, int N, int Np, int K) {
    const size_t words = static_cast<size_t>(R) * RS          // this CTA's action rows (dimension-major)
                         + static_cast<size_t>(K) * D          // rank-ordered elite rows (filled by their owners)
                         + (N + Np)                            // sort keys of ALL candidates (filled by their owners)
                         + static_cast<size_t>(R) * Pe         // returns of this CTA's rollouts
                         + 4 * D                               // mean, std, best_seq, warm-start sequence
                         + 2 * K                               // elite_idx, sel_idx
                         + select_scratch_words(K, N + Np)
                         + 12;                                 // best_value, true state [4], planner key, System key
    return words * 4;
  }
};

template <int H, int A>
struct GenClusterCtaSmem {
  float* act;        // [R][RS]
  float* ebuf;       // [K][D]
  uint32_t* skey;    // [M]
  float* rets;       // [R][Pe]
  float* mean;       // [D] (t, a) order
  float* std_;
  float* best_seq;
  float* prev;       // [D] warm-start sequence of the next plan (closed loop)
  int* elite_idx;
  int* sel_idx;
  uint32_t* sel_scratch;
  float* best_value;  // [1]
  float* xs;          // [4] true state (closed loop)
  uint32_t* pkey;     // [2] opt_state.key (closed loop)
  uint32_t* syskey;   // [2] system_params.key (closed loop)
  __device__ __forceinline__ GenClusterCtaSmem(uint32_t* base, int R, int Pe, int N, int Np, int K) {
    constexpr int D = H * A, RS = D | 1;
    act = reinterpret_cast<float*>(base);
    ebuf = act + static_cast<size_t>(R) * RS;
    skey = reinterpret_cast<uint32_t*>(ebuf + static_cast<size_t>(K) * D);
    rets = reinterpret_cast<float*>(skey + (N + Np));
    mean = rets + static_cast<size_t>(R) * Pe;
    std_ = mean + D;
    best_seq = std_ + D;
    prev = best_seq + D;
    elite_idx = reinterpret_cast<int*>(prev + D);
    sel_idx = elite_idx + K;
    sel_scratch = reinterpret_cast<uint32_t*>(sel_idx + K);
    best_value = reinterpret_cast<float*>(sel_scratch + select_scratch_words(K, N + Np));
    xs = best_value + 4;
    pkey = reinterpret_cast<uint32_t*>(xs + 4);
    syskey = pkey + 2;
  }
};

// iCemTO.optimize for ONE problem over a general System, executed by the whole cluster.  Same contract as
// plan_problem_general, except that k_new is valid in every thread and sm.prev is the warm-start sequence.  Trace
// dumps are written by the row owners (values, actions) and by CTA 0 (the rest).  Ends with a barrier.
template <class Sys, int H, int PRNG>
__device__ __forceinline__ void plan_problem_general_cluster(const PlanArgs& a, const GenClusterCtaSmem<H, Sys::A>& sm,
                                                             const Sys& sys, const RefitScalars& rs,
                                                             const float (&s0)[Sys::X], Key2 key_in, Key2& k_new,
                                                             int slot, int slots, int R) {
  constexpr int A = Sys::A, X = Sys::X, D = H * A, RS = D | 1;
  cg::cluster_group cluster = cg::this_cluster();
  const int C = static_cast<int>(cluster.num_blocks());
  const int rank = static_cast<int>(cluster.block_rank());
  const int N = a.N, M = a.N + a.Np, K = a.K, P = a.P;
  const int Pe = Sys::KEYED ? P : 1;                 // rollouts per row: a deterministic System's particles are equal
  const int tid = threadIdx.x, NT = blockDim.x;
  const int row0 = rank * R;
  float* mean = sm.mean;
  float* std_ = sm.std_;
  float* best_seq = sm.best_seq;

  // ---- prologue (:235-249), redundantly in every CTA; the rows past N stay all zero ----------------------------
  for (int d = tid; d < D; d += NT) {
    float m = 0.0f;
    if (a.warm_start) m = sm.prev[(d + A < D) ? d + A : (D - A + d % A)];
    mean[d] = m;
    std_[d] = a.init_std;
    best_seq[d] = m;
  }
  for (int w = tid; w < R * RS; w += NT)
    if (row0 + w / RS >= N) sm.act[w] = 0.0f;
  if (tid == 0) *sm.best_value = __int_as_float(0xFF800000);   // -inf
  // The carry key (:174-180) does not depend on data: every thread advances its own copy in registers.
  Key2 chain;
  split2<PRNG>(key_in, chain, k_new);
  __syncthreads();

  for (int it = 0; it < a.S; ++it) {
    const size_t tslot = static_cast<size_t>(it) * slots + slot;
    Key2 sampling_rng, particles_rng;
    split2<PRNG>(chain, sampling_rng, particles_rng);                                           // :174
    chain = split_at<PRNG>(sampling_rng, static_cast<uint32_t>(N + 1), 0u);                     // :176

    // ---- 1. sampling, one thread per (row, action dimension) ------------------------------------------------
    for (int j = tid; j < R * A; j += NT) {
      const int r = j / A, ad = j - r * A, n = row0 + r;
      if (n >= N) continue;
      const Key2 sk = split_at<PRNG>(sampling_rng, static_cast<uint32_t>(N + 1), static_cast<uint32_t>(n + 1));
      const Key2 dk = split_at<PRNG>(sk, static_cast<uint32_t>(A), static_cast<uint32_t>(ad));     // :180
      float* dim = sm.act + static_cast<size_t>(r) * RS + ad * H;
      colored_noise_row<H, PRNG>(dk, a.scale, dim, nullptr, [&](int t, float y) {
        const float v = __fadd_rn(mean[t * A + ad], __fmul_rn(y, std_[t * A + ad]));                // :190
        dim[t] = fminf(fmaxf(v, a.u_min), a.u_max);                                                 // :191
      });
    }
    __syncthreads();

    // ---- 2. rollouts, one thread per (row, particle) (:144-160) -----------------------------------------------
    for (int w = tid; w < R * Pe; w += NT) {
      const int r = w / Pe, p = w - r * Pe, n = row0 + r;
      if (n >= M || (!Sys::KEYED && n > N)) continue;
      Key2 key{0u, 0u};
      if (Sys::KEYED) {
        const Key2 pkey = split_at<PRNG>(particles_rng, static_cast<uint32_t>(M), static_cast<uint32_t>(n));   // :177
        key = split_at<PRNG>(pkey, static_cast<uint32_t>(P), static_cast<uint32_t>(p));                       // :155
      }
      const float* row = sm.act + static_cast<size_t>(r) * RS;
      float s[X];
#pragma unroll
      for (int k = 0; k < X; ++k) s[k] = s0[k];
      float acc = 0.0f;
      for (int t = 0; t < H; ++t) acc = __fadd_rn(acc, sys.template step<PRNG>(s, row + t, H, key));
      sm.rets[w] = __fdiv_rn(acc, static_cast<float>(H));
    }
    __syncthreads();

    // ---- 3. a row's value from its particles, in particle order; its key goes to every CTA -------------------
    for (int r = tid; r < R; r += NT) {
      const int n = row0 + r;
      if (n >= M || (!Sys::KEYED && n > N)) continue;
      const float* ret = sm.rets + static_cast<size_t>(r) * Pe;
      float val;
      if (!Sys::KEYED) {
        if (a.summarize == MBPO_SUMMARIZE_MAX || P == 1) {
          val = ret[0];
        } else {
          float acc = 0.0f;
          for (int p = 0; p < P; ++p) acc = __fadd_rn(acc, ret[0]);
          val = __fdiv_rn(acc, static_cast<float>(P));
        }
      } else {
        float acc = 0.0f, mx = 0.0f;
        for (int p = 0; p < P; ++p) {
          acc = __fadd_rn(acc, ret[p]);
          mx = (p == 0) ? ret[p] : fmaxf(mx, ret[p]);
        }
        val = (a.summarize == MBPO_SUMMARIZE_MAX) ? mx : __fdiv_rn(acc, static_cast<float>(P));
      }
      const uint32_t key = total_order_key(val);
      // a deterministic System's first zero row stands for all Np of them
      const int j1 = (Sys::KEYED || n < N) ? n + 1 : M;
      for (int j = n; j < j1; ++j) {
        for (int c = 0; c < C; ++c) cluster.map_shared_rank(sm.skey, c)[j] = key;
        if (a.trace.values) a.trace.values[tslot * M + j] = val;
        if (a.trace.actions) {
          const float* row = sm.act + static_cast<size_t>(r) * RS;
          float* dst = a.trace.actions + (tslot * M + j) * D;
          for (int d = 0; d < D; ++d) dst[d] = (j < N) ? row[(d % A) * H + d / A] : 0.0f;
        }
      }
    }
    cluster.sync();   // all keys are in every copy

    // ---- 5. selection on every CTA's full copy (:199-203); the owners send their elite rows, rank-ordered ------
    cta_select<0>(rs, sm.skey, sm.elite_idx, sm.sel_idx, sm.sel_scratch);    // ends with a barrier
    const float best_elite = value_of_key(sm.skey[sm.elite_idx[K - 1]]);
    for (int w = tid; w < K * D; w += NT) {
      const int e = w / D, d = w - e * D;
      const int src = sm.elite_idx[e];
      if (src < row0 || src >= row0 + R) continue;
      const float v = src < N ? sm.act[static_cast<size_t>(src - row0) * RS + (d % A) * H + d / A] : 0.0f;
      for (int c = 0; c < C; ++c) cluster.map_shared_rank(sm.ebuf, c)[w] = v;
    }
    cluster.sync();   // the elite rows are complete in every CTA

    // ---- 7. refit + best tracking (:206-226), every CTA for itself.  (A CTA that runs ahead writes skey of the
    // next iteration only after its rollouts and ebuf only after the next first cluster.sync: a slower CTA has read
    // its keys before this iteration's second cluster.sync and reads ebuf before it reaches the next first one.)
    cta_refit<0>(rs, best_elite, [&](int e, int d) { return sm.ebuf[e * D + d]; }, mean, std_, best_seq,
                 sm.best_value);
    if (rank == 0) {
      if (a.trace.elite_idx)
        for (int e = tid; e < K; e += NT) a.trace.elite_idx[tslot * K + e] = sm.elite_idx[e];
      for (int d = tid; d < D; d += NT) {
        if (a.trace.mean) a.trace.mean[tslot * D + d] = mean[d];
        if (a.trace.std) a.trace.std[tslot * D + d] = std_[d];
      }
      if (a.trace.best_value && tid == 0) a.trace.best_value[tslot] = *sm.best_value;
    }
    __syncthreads();
  }
}

// One cluster plans one problem at a time (cluster-stride over problems), cluster dimension C along x.
template <class Sys, int H, int PRNG>
__global__ void __launch_bounds__(CLUSTER_MAX_THREADS, 1)
    icem_plan_general_cluster_kernel(const __grid_constant__ PlanArgs a, int R) {
  constexpr int A = Sys::A, X = Sys::X, D = H * A;
  extern __shared__ __align__(16) uint32_t smem_u32[];
  cg::cluster_group cluster = cg::this_cluster();
  const int C = static_cast<int>(cluster.num_blocks());
  const int rank = static_cast<int>(cluster.block_rank());
  const GenClusterCtaSmem<H, A> sm(smem_u32, R, Sys::KEYED ? a.P : 1, a.N, a.Np, a.K);
  const int tid = threadIdx.x, NT = blockDim.x;
  const Sys sys(a.gsys);
  RefitScalars rs;
  rs.M = a.N + a.Np; rs.K = a.K; rs.D = D; rs.alpha = a.alpha; rs.one_minus_alpha = a.one_minus_alpha;
  const int clusters = static_cast<int>(gridDim.x) / C;
  for (int b = static_cast<int>(blockIdx.x) / C; b < a.B; b += clusters) {
    float s0[X];
#pragma unroll
    for (int k = 0; k < X; ++k) s0[k] = a.x0[static_cast<size_t>(b) * X + k];
    for (int d = tid; d < D; d += NT) sm.prev[d] = a.best_seq_in[static_cast<size_t>(b) * D + d];
    __syncthreads();
    Key2 k_new;
    plan_problem_general_cluster<Sys, H, PRNG>(a, sm, sys, rs, s0, Key2{a.key_in[2 * b], a.key_in[2 * b + 1]}, k_new,
                                               b, a.B, R);
    cluster.sync();   // no CTA runs ahead into the next problem while a lagging CTA still reads this one's buffers
    if (rank == 0) {
      for (int d = tid; d < D; d += NT) a.best_seq_out[static_cast<size_t>(b) * D + d] = sm.best_seq[d];
      if (tid == 0) {
        a.best_value_out[b] = *sm.best_value;
        a.key_out[2 * b] = k_new.k0;
        a.key_out[2 * b + 1] = k_new.k1;
      }
    }
    __syncthreads();
  }
}

// The closed loop on a cluster: every CTA keeps its own copy of the true state, both keys and the warm-start
// sequence (identical by construction) and steps the System itself; CTA 0 writes the outputs.
template <class Sys, int H, int PRNG>
__global__ void __launch_bounds__(CLUSTER_MAX_THREADS, 1)
    icem_mpc_general_cluster_kernel(const __grid_constant__ PlanArgs a, const __grid_constant__ GeneralMpcArgs m,
                                    int R) {
  constexpr int A = Sys::A, X = Sys::X, D = H * A;
  extern __shared__ __align__(16) uint32_t smem_u32[];
  cg::cluster_group cluster = cg::this_cluster();
  const int C = static_cast<int>(cluster.num_blocks());
  const int rank = static_cast<int>(cluster.block_rank());
  const GenClusterCtaSmem<H, A> sm(smem_u32, R, Sys::KEYED ? a.P : 1, a.N, a.Np, a.K);
  const int tid = threadIdx.x, NT = blockDim.x;
  const Sys sys(a.gsys);
  RefitScalars rs;
  rs.M = a.N + a.Np; rs.K = a.K; rs.D = D; rs.alpha = a.alpha; rs.one_minus_alpha = a.one_minus_alpha;
  const int clusters = static_cast<int>(gridDim.x) / C;
  for (int b = static_cast<int>(blockIdx.x) / C; b < a.B; b += clusters) {
    for (int d = tid; d < D; d += NT) sm.prev[d] = a.best_seq_in[static_cast<size_t>(b) * D + d];
    if (tid < X) sm.xs[tid] = a.x0[static_cast<size_t>(b) * X + tid];
    if (tid == 0) {
      sm.pkey[0] = a.key_in[2 * b]; sm.pkey[1] = a.key_in[2 * b + 1];
      sm.syskey[0] = m.sys_key_in ? m.sys_key_in[2 * b] : 0u;
      sm.syskey[1] = m.sys_key_in ? m.sys_key_in[2 * b + 1] : 0u;
    }
    __syncthreads();
    for (int t = 0; t < m.T; ++t) {
      float s0[X];
#pragma unroll
      for (int k = 0; k < X; ++k) s0[k] = sm.xs[k];
      Key2 k_new;
      plan_problem_general_cluster<Sys, H, PRNG>(a, sm, sys, rs, s0, Key2{sm.pkey[0], sm.pkey[1]}, k_new, 0, 1, R);
      if (tid == 0) {
        sm.pkey[0] = k_new.k0; sm.pkey[1] = k_new.k1;
        general_mpc_step<Sys, PRNG>(sys, m, a.B, b, t, sm.best_seq, sm.xs, sm.syskey, rank == 0);
      }
      for (int d = tid; d < D; d += NT) sm.prev[d] = sm.best_seq[d];
      __syncthreads();
    }
    cluster.sync();
    if (rank == 0) {
      for (int d = tid; d < D; d += NT) a.best_seq_out[static_cast<size_t>(b) * D + d] = sm.prev[d];
      if (tid == 0) {
        a.key_out[2 * b] = sm.pkey[0];
        a.key_out[2 * b + 1] = sm.pkey[1];
        if (m.sys_key_out) { m.sys_key_out[2 * b] = sm.syskey[0]; m.sys_key_out[2 * b + 1] = sm.syskey[1]; }
      }
    }
    __syncthreads();
  }
}

}  // namespace mbpo
