// Replay buffer (brax UniformSamplingQueue) and BraxWrapper.reset: C ABI + kernels.
//
// Replaces brax/training/replay_buffers.py QueueBase.insert_internal / UniformSamplingQueue.sample_internal as the
// reference calls them at mbpo/optimizers/policy_optimizers/sac/sac.py:202-205,303 and
// mbpo/systems/brax_wrapper.py:25-38.  The queue is a ring in HBM (logical row i = physical row (head + i) % capacity),
// so inserting into a full queue moves no rows (brax rolls the whole buffer).  HBM-bound byte shuffling: insert reads
// and writes 4*D bytes per row, both coalesced.
#include <cuda_runtime.h>

#include "../../include/mbpo_b200.h"
#include "host_util.h"
#include "threefry.cuh"

using namespace mbpo;

namespace {

struct FieldTable {
  int num_fields;
  int col_end[MBPO_REPLAY_MAX_FIELDS];  // exclusive prefix end of field f
  int width[MBPO_REPLAY_MAX_FIELDS];
  unsigned magic[MBPO_REPLAY_MAX_FIELDS];  // floor(2^32 / width) + 1: j / width = umulhi(j, magic) inside a tile
  const float* ptr[MBPO_REPLAY_MAX_FIELDS];
};

// offset of randint inside [0, span): jax/_src/random.py _randint on 32-bit words
template <int MODE>
__device__ __forceinline__ uint32_t randint_offset_at(Key2 key, uint32_t n, uint32_t w, uint32_t span) {
  Key2 k1, k2;
  split2<MODE>(key, k1, k2);
  const uint32_t hi = random_bits_at<MODE>(k1, n, w);
  const uint32_t lo = random_bits_at<MODE>(k2, n, w);
  uint32_t mult = 65536u % span;
  mult = (mult * mult) % span;
  const uint32_t off = (hi % span) * mult + (lo % span);
  return off % span;
}

__host__ __device__ __forceinline__ uint32_t randint_span(int minval, int maxval) {
  return (maxval <= minval) ? 1u : static_cast<uint32_t>(maxval) - static_cast<uint32_t>(minval);
}

template <int MODE>
__global__ void prng_randint_kernel(const uint32_t* __restrict__ keys, long long total, int n, int minval,
                                    uint32_t span, int32_t* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long m = i / n;
  const uint32_t w = static_cast<uint32_t>(i % n);
  const Key2 k{keys[2 * m], keys[2 * m + 1]};
  out[i] = static_cast<int32_t>(static_cast<uint32_t>(minval) + randint_offset_at<MODE>(k, n, w, span));
}

// One CTA packs `rows_per_cta` consecutive rows through shared memory: every field's block of the tile is one dense
// run in HBM, read with 16-byte loads (one per field issued before the first is used), the tile is assembled row-major
// in shared memory and leaves as one dense run of the ring with 16-byte stores.  The tile sits in shared memory at the
// same offset modulo 16 bytes as its destination, so both sides of the copy are aligned.  (First version: one thread
// per word with the field looked up per word -- ~100 instructions per word, issue-bound at 38% of HBM.)
constexpr int PACK_THREADS = 256;
constexpr int PACK_LOADS = 5;   // 16-byte loads a thread keeps in flight

// scatters the words j .. j+n-1 of field (w, col0) of the tile into its row-major image
__device__ __forceinline__ void pack_scatter(float* tile, int D, unsigned w, unsigned col0, unsigned magic,
                                             unsigned j, const float* x, int n) {
  unsigned r = (w == 1u) ? j : __umulhi(j, magic);   // j / w (exact: j * w < 2^32)
  unsigned c = j - r * w;
  unsigned at = r * static_cast<unsigned>(D) + col0 + c;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (k < n) tile[at] = x[k];
    ++c;
    ++at;
    if (c == w) {
      c = 0;
      at += static_cast<unsigned>(D) - w;
    }
  }
}

template <bool VEC>
__global__ void __launch_bounds__(PACK_THREADS)
replay_pack_kernel(FieldTable ft, int D, int rows_per_cta, long long n_rows, float* __restrict__ data,
                   long long capacity, long long first_physical) {
  extern __shared__ __align__(16) float pack_smem[];
  const unsigned tid = threadIdx.x;
  const long long row0 = static_cast<long long>(blockIdx.x) * rows_per_cta;
  const long long left = n_rows - row0;
  const unsigned rows = static_cast<unsigned>(left < rows_per_cta ? left : rows_per_cta);
  long long p0 = first_physical + row0;                  // physical row of the tile's first row
  if (p0 >= capacity) p0 -= capacity;
  const long long g0 = p0 * D;                           // first word of the tile in the ring
  const unsigned total = rows * static_cast<unsigned>(D);
  const long long until_end = capacity * D - g0;         // words before the ring wraps
  const unsigned shift = VEC ? static_cast<unsigned>(g0 & 3) : 0u;
  float* tile = pack_smem + shift;

  if (VEC && (rows & 3u) == 0u) {
    // The tile's 16-byte words in field-major order: q4 in [rows * col_start(f) / 4, rows * col_end(f) / 4) walks
    // field f's dense block.  PACK_LOADS loads per thread are issued before the first is scattered.
    const unsigned total4 = total >> 2;
    for (unsigned base = tid; base < total4; base += PACK_THREADS * PACK_LOADS) {
      float4 x[PACK_LOADS];
      unsigned fld[PACK_LOADS], j0[PACK_LOADS];
#pragma unroll
      for (int k = 0; k < PACK_LOADS; ++k) {
        const unsigned q4 = base + k * PACK_THREADS;
        fld[k] = 0xFFFFFFFFu;
        if (q4 < total4) {
          unsigned f = 0;
#pragma unroll
          for (int g = 0; g < MBPO_REPLAY_MAX_FIELDS - 1; ++g)
            f += (g < ft.num_fields - 1 && 4u * q4 >= rows * static_cast<unsigned>(ft.col_end[g])) ? 1u : 0u;
          const unsigned w = static_cast<unsigned>(ft.width[f]);
          const unsigned j = 4u * q4 - rows * (static_cast<unsigned>(ft.col_end[f]) - w);
          x[k] = __ldcs(reinterpret_cast<const float4*>(ft.ptr[f] + row0 * w + j));
          fld[k] = f;
          j0[k] = j;
        }
      }
#pragma unroll
      for (int k = 0; k < PACK_LOADS; ++k) {
        if (fld[k] != 0xFFFFFFFFu) {
          const unsigned w = static_cast<unsigned>(ft.width[fld[k]]);
          pack_scatter(tile, D, w, static_cast<unsigned>(ft.col_end[fld[k]]) - w, ft.magic[fld[k]], j0[k], &x[k].x, 4);
        }
      }
    }
  } else {
    for (int f = 0; f < ft.num_fields; ++f) {
      const unsigned w = static_cast<unsigned>(ft.width[f]);
      const unsigned col0 = static_cast<unsigned>(ft.col_end[f]) - w;
      const unsigned words = rows * w;
      const float* __restrict__ src = ft.ptr[f] + row0 * w;
      for (unsigned j = tid; j < words; j += PACK_THREADS) {
        const float y = __ldcs(src + j);
        pack_scatter(tile, D, w, col0, ft.magic[f], j, &y, 1);
      }
    }
  }
  __syncthreads();
  if (VEC && static_cast<long long>(total) <= until_end) {
    float* __restrict__ dst = data + g0;
    const unsigned head = (4u - shift) & 3u;
    const unsigned h = head < total ? head : total;
    if (tid < h) dst[tid] = tile[tid];
    const unsigned nvec = (total - h) >> 2;
    const float4* t4 = reinterpret_cast<const float4*>(tile + h);
    float4* d4 = reinterpret_cast<float4*>(dst + h);
    for (unsigned k = tid; k < nvec; k += PACK_THREADS) d4[k] = t4[k];
    for (unsigned i = h + 4u * nvec + tid; i < total; i += PACK_THREADS) dst[i] = tile[i];
  } else {
    float* __restrict__ dst = data + g0;
    for (unsigned i = tid; i < total; i += PACK_THREADS) {
      if (static_cast<long long>(i) < until_end) dst[i] = tile[i];
      else data[static_cast<long long>(i) - until_end] = tile[i];
    }
  }
}

template <int MODE>
__global__ void replay_sample_kernel(const float* __restrict__ data, long long capacity, int D, long long head,
                                     const uint32_t* __restrict__ key, int batch, int minval, uint32_t span,
                                     uint32_t* __restrict__ key_out, int32_t* __restrict__ idx_out,
                                     float* __restrict__ batch_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= batch) return;
  const Key2 k{key[0], key[1]};
  Key2 next, sample_key;
  split2<MODE>(k, next, sample_key);
  if (i == 0) {
    key_out[0] = next.k0;
    key_out[1] = next.k1;
  }
  const int32_t idx = static_cast<int32_t>(static_cast<uint32_t>(minval) +
                                           randint_offset_at<MODE>(sample_key, static_cast<uint32_t>(batch),
                                                                   static_cast<uint32_t>(i), span));
  if (idx_out) idx_out[i] = idx;
  long long l = static_cast<long long>(idx) % capacity;  // jnp.take(mode='wrap')
  if (l < 0) l += capacity;
  long long p = head + l;
  if (p >= capacity) p -= capacity;
  const float* src = data + p * D;
  float* dst = batch_out + static_cast<long long>(i) * D;
  for (int c = 0; c < D; ++c) dst[c] = src[c];
}

__global__ void replay_read_kernel(const float* __restrict__ data, long long capacity, int D, long long head,
                                   long long first, long long total_words, float* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total_words) return;
  const long long r = i / D;
  const int c = static_cast<int>(i - r * D);
  long long p = head + first + r;
  p %= capacity;
  out[i] = data[p * D + c];
}

template <int MODE>
__global__ void env_reset_kernel(const float* __restrict__ data, long long capacity, int D, long long head,
                                 const uint32_t* __restrict__ rngs, int E, int batch, int minval, uint32_t span,
                                 int x_dim, int reward_col, float* __restrict__ obs_out,
                                 float* __restrict__ reward_out, uint32_t* __restrict__ sys_key_out,
                                 int32_t* __restrict__ idx_out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const Key2 rng{rngs[2 * e], rngs[2 * e + 1]};
  Key2 buffer_key, sys_key, next, sample_key;
  split2<MODE>(rng, buffer_key, sys_key);          // brax_wrapper.py:26
  split2<MODE>(buffer_key, next, sample_key);      // sample_internal: key, sample_key = split(buffer_state.key)
  const int32_t idx = static_cast<int32_t>(static_cast<uint32_t>(minval) +
                                           randint_offset_at<MODE>(sample_key, static_cast<uint32_t>(batch), 0u, span));
  long long l = static_cast<long long>(idx) % capacity;
  if (l < 0) l += capacity;
  long long p = head + l;
  if (p >= capacity) p -= capacity;
  const float* row = data + p * D;
  for (int c = 0; c < x_dim; ++c) obs_out[static_cast<long long>(e) * x_dim + c] = row[c];
  reward_out[e] = row[reward_col];
  sys_key_out[2 * e] = sys_key.k0;
  sys_key_out[2 * e + 1] = sys_key.k1;
  if (idx_out) idx_out[e] = idx;
}

// EvalWrapper folded over an unroll: one thread per env, the [T, E] streams are read a line per warp per step.
__global__ void eval_metrics_kernel(const float* __restrict__ reward, const float* __restrict__ discount,
                                    const float* __restrict__ steps_in, const float* __restrict__ done_in,
                                    float action_repeat, int E, int T, long long stride_t, long long stride_e,
                                    float* __restrict__ episode_reward, float* __restrict__ episode_steps,
                                    float* __restrict__ active) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  float steps = steps_in[e], done = done_in[e];
  float sum = episode_reward[e], ep_steps = episode_steps[e], act = active[e];
  const float* r = reward + e * stride_e;
  const float* d = discount + e * stride_e;
#pragma unroll 4
  for (int t = 0; t < T; ++t) {
    const float rt = __ldcs(r + t * stride_t), dt = __ldcs(d + t * stride_t);
    steps = __fadd_rn(done != 0.0f ? 0.0f : steps, action_repeat);       // training.py:98,120-124
    ep_steps = act != 0.0f ? steps : ep_steps;                           // :181-185
    sum = __fadd_rn(sum, __fmul_rn(rt, act));                            // :186-190 (a + b * active, unfused)
    act = __fmul_rn(act, dt);                                            // :191
    done = __fsub_rn(1.0f, dt);
  }
  episode_reward[e] = sum;
  episode_steps[e] = ep_steps;
  active[e] = act;
}

// ---- running statistics ---------------------------------------------------------------------------------------
constexpr int RS_THREADS = 256;
constexpr int RS_CTAS = 148 * 4;
constexpr int RS_MAX_X = 64;

// Pass 1: every thread walks words i = gid, gid + stride, ... of the flat [n_rows * X] batch with stride a multiple
// of X, so its column x = i % X never changes: two float64 accumulators per thread, coalesced 4-byte reads.
__global__ void __launch_bounds__(RS_THREADS)
running_stats_partial_kernel(const float* __restrict__ batch, long long total_words, int X,
                             const float* __restrict__ mean, long long stride, double* __restrict__ partials) {
  __shared__ double sh[2][RS_THREADS];
  const long long gid = static_cast<long long>(blockIdx.x) * RS_THREADS + threadIdx.x;
  double s1 = 0.0, s2 = 0.0;
  if (gid < stride) {
    const float m = mean[gid % X];
    for (long long i = gid; i < total_words; i += stride) {
      const float d = __fsub_rn(__ldcs(batch + i), m);      // diff_to_old_mean in float32, like the reference
      s1 += static_cast<double>(d);
      s2 += static_cast<double>(d) * static_cast<double>(d);
    }
  }
  sh[0][threadIdx.x] = s1;
  sh[1][threadIdx.x] = s2;
  __syncthreads();
  // fixed-order combine: thread x (< X) adds the lanes of its column in index order
  if (threadIdx.x < X) {
    const int first = static_cast<int>(((threadIdx.x - (static_cast<long long>(blockIdx.x) * RS_THREADS) % X) % X + X) % X);
    double a = 0.0, b = 0.0;
    for (int t = first; t < RS_THREADS; t += X) {
      a += sh[0][t];
      b += sh[1][t];
    }
    partials[(static_cast<long long>(blockIdx.x) * 2) * X + threadIdx.x] = a;
    partials[(static_cast<long long>(blockIdx.x) * 2 + 1) * X + threadIdx.x] = b;
  }
}

__global__ void running_stats_combine_kernel(const double* __restrict__ partials, int ctas, int X, double n_rows,
                                             double* __restrict__ sums) {
  const int j = threadIdx.x;  // 0 .. 2X-1: (which, x)
  if (j == 2 * X) sums[j] = n_rows;
  if (j >= 2 * X) return;
  const int which = j / X, x = j % X;
  double a = 0.0;
  for (int c = 0; c < ctas; ++c) a += partials[(static_cast<long long>(c) * 2 + which) * X + x];
  sums[j] = a;
}

__global__ void running_stats_finalize_kernel(const double* __restrict__ sums, int X,
                                              const float* __restrict__ count_in, const float* __restrict__ mean_in,
                                              const float* __restrict__ sv_in, float std_min, float std_max,
                                              float* __restrict__ count_out, float* __restrict__ mean_out,
                                              float* __restrict__ sv_out, float* __restrict__ std_out) {
  const int x = threadIdx.x;
  if (x >= X) return;
  const float count = __fadd_rn(count_in[0], static_cast<float>(sums[2 * X]));   // step_increment (psum-ed)
  const double mean_update = sums[x] / static_cast<double>(count);
  const float mean = __fadd_rn(mean_in[x], static_cast<float>(mean_update));
  // sum(d_old * d_new) with d_new = d_old - mean_update
  const double variance_update = sums[X + x] - mean_update * sums[x];
  const float sv = __fadd_rn(sv_in[x], static_cast<float>(variance_update));
  float sd = sqrtf(__fdiv_rn(fmaxf(sv, 0.0f), count));
  sd = fminf(fmaxf(sd, std_min), std_max);
  __syncthreads();
  if (x == 0) count_out[0] = count;
  mean_out[x] = mean;
  sv_out[x] = sv;
  std_out[x] = sd;
}

__global__ void running_stats_normalize_kernel(const float* __restrict__ batch, long long total_words, int X,
                                               const float* __restrict__ mean, const float* __restrict__ std,
                                               float max_abs, float* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total_words) return;
  const int x = static_cast<int>(i % X);
  float v = __fdiv_rn(__fsub_rn(batch[i], mean[x]), std[x]);
  if (max_abs > 0.0f) v = fminf(fmaxf(v, -max_abs), max_abs);
  out[i] = v;
}

__global__ void normalizer_finalize_kernel(const double* __restrict__ sums, int X, const double* __restrict__ size_in,
                                          const float* __restrict__ mean_in, const float* __restrict__ std_in, float eps,
                                          double* __restrict__ size_out, float* __restrict__ mean_out,
                                          float* __restrict__ std_out) {
  const int x = threadIdx.x;
  if (x >= X) return;
  const double size = size_in[0], n = sums[2 * X], total = size + n;
  const double delta = sums[x] / total;                                   // new_mean - mean
  const double sq = sums[X + x] - 2.0 * delta * sums[x] + n * delta * delta;   // sum((x - new_mean)^2)
  const double sd = static_cast<double>(std_in[x]);
  const double s_n = sd * sd * size + sq + size * delta * delta;
  const float mean = static_cast<float>(static_cast<double>(mean_in[x]) + delta);
  const float new_std = sqrtf(static_cast<float>(s_n / total));
  __syncthreads();
  if (x == 0) size_out[0] = total;
  mean_out[x] = mean;
  std_out[x] = fmaxf(new_std, eps);
}

__global__ void normalizer_inverse_kernel(const float* __restrict__ batch, long long total_words, int X,
                                         const float* __restrict__ mean, const float* __restrict__ std,
                                         float* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total_words) return;
  const int x = static_cast<int>(i % X);
  out[i] = __fadd_rn(__fmul_rn(batch[i], std[x]), mean[x]);
}

__global__ void replay_take_kernel(const float* __restrict__ data, long long capacity, int D, long long head,
                                   const int32_t* __restrict__ idx, long long total_words, float* __restrict__ out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total_words) return;
  const long long r = i / D;
  const int c = static_cast<int>(i - r * D);
  long long l = static_cast<long long>(idx[r]) % capacity;  // mode='wrap'
  if (l < 0) l += capacity;
  long long p = head + l;
  if (p >= capacity) p -= capacity;
  out[i] = data[p * D + c];
}

// PPO's GAE: one thread per env, one reverse pass, six [T, E] streams (a line per warp per step).
__global__ void compute_gae_kernel(const float* __restrict__ truncation, const float* __restrict__ termination,
                                   const float* __restrict__ rewards, const float* __restrict__ values,
                                   const float* __restrict__ bootstrap, int E, int T, long long st_t, long long st_e,
                                   float discount, float lambda_, float* __restrict__ vs_out,
                                   float* __restrict__ adv_out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const long long base = e * st_e;
  float v_next = bootstrap[e], vs_next = v_next, acc = 0.0f;
#pragma unroll 4
  for (int t = T - 1; t >= 0; --t) {
    const long long i = base + t * st_t;
    const float tm = __fsub_rn(1.0f, __ldcs(truncation + i));
    const float dn = __fmul_rn(discount, __fsub_rn(1.0f, __ldcs(termination + i)));   // discount * (1 - termination)
    const float r = __ldcs(rewards + i), v = __ldcs(values + i);
    const float delta = __fmul_rn(__fsub_rn(__fadd_rn(r, __fmul_rn(dn, v_next)), v), tm);                    // :160-161
    acc = __fadd_rn(delta, __fmul_rn(__fmul_rn(__fmul_rn(dn, tm), lambda_), acc));                           // :169
    const float vs = __fadd_rn(acc, v);                                                                      // :178
    adv_out[i] = __fmul_rn(__fsub_rn(__fadd_rn(r, __fmul_rn(dn, vs_next)), v), tm);                          // :182-183
    vs_out[i] = vs;
    v_next = v;
    vs_next = vs;
  }
}

int check_state(const MbpoReplayState* s, const char* who) {
  MBPO_REQUIRE(s != nullptr, "%s: state is null", who);
  MBPO_REQUIRE(s->data != nullptr, "%s: data is null", who);
  MBPO_REQUIRE(s->capacity >= 1 && s->row_width >= 1, "%s: capacity %lld / row_width %d", who, s->capacity,
               s->row_width);
  MBPO_REQUIRE(s->head >= 0 && s->head < s->capacity, "%s: head %lld outside [0, %lld)", who, s->head, s->capacity);
  MBPO_REQUIRE(s->insert_position >= 0 && s->insert_position <= s->capacity && s->sample_position >= 0 &&
                   s->sample_position <= s->capacity,
               "%s: positions (%lld, %lld) outside [0, %lld]", who, s->insert_position, s->sample_position,
               s->capacity);
  MBPO_REQUIRE(s->capacity < (1LL << 31), "%s: capacity %lld needs int32 indices like brax", who, s->capacity);
  return MBPO_OK;
}

}  // namespace

extern "C" {

int mbpo_prng_randint(const uint32_t* keys, int M, int n, int prng_mode, int minval, int maxval, int32_t* out,
                      void* stream) {
  MBPO_REQUIRE(M >= 0 && n >= 0, "prng_randint: negative size");
  MBPO_REQUIRE(prng_mode == 0 || prng_mode == 1, "prng_randint: bad prng_mode %d", prng_mode);
  const long long total = static_cast<long long>(M) * n;
  if (total == 0) return MBPO_OK;
  MBPO_REQUIRE(keys && out, "prng_randint: null pointer");
  const uint32_t span = randint_span(minval, maxval);
  const int threads = 256;
  const unsigned blocks = static_cast<unsigned>((total + threads - 1) / threads);
  return with_prng(prng_mode, [&](auto P) {
    prng_randint_kernel<P><<<blocks, threads, 0, as_stream(stream)>>>(keys, total, n, minval, span, out);
    return check_launch("prng_randint_kernel");
  });
}

int mbpo_replay_insert(MbpoReplayState* s, const MbpoReplayFields* fields, long long n_rows, void* stream) {
  int rc = check_state(s, "replay_insert");
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(fields != nullptr, "replay_insert: fields is null");
  MBPO_REQUIRE(fields->num_fields >= 1 && fields->num_fields <= MBPO_REPLAY_MAX_FIELDS,
               "replay_insert: num_fields %d outside [1, %d]", fields->num_fields, MBPO_REPLAY_MAX_FIELDS);
  MBPO_REQUIRE(n_rows >= 0, "replay_insert: n_rows < 0");
  MBPO_REQUIRE(n_rows <= s->capacity,
               "replay_insert: trying to insert a batch of %lld samples larger than the maximum replay size %lld",
               n_rows, s->capacity);
  FieldTable ft{};
  ft.num_fields = fields->num_fields;
  int col = 0;
  for (int f = 0; f < fields->num_fields; ++f) {
    MBPO_REQUIRE(fields->width[f] >= 1, "replay_insert: field %d has width %d", f, fields->width[f]);
    MBPO_REQUIRE(n_rows == 0 || fields->ptr[f] != nullptr, "replay_insert: field %d is null", f);
    col += fields->width[f];
    ft.col_end[f] = col;
    ft.width[f] = fields->width[f];
    ft.magic[f] = static_cast<unsigned>((1ULL << 32) / static_cast<unsigned>(fields->width[f]) + 1ULL);
    ft.ptr[f] = fields->ptr[f];
  }
  MBPO_REQUIRE(col == s->row_width, "replay_insert: field widths sum to %d, row_width is %d", col, s->row_width);
  if (n_rows == 0) return MBPO_OK;
  // brax insert_internal: roll = min(0, len(data) - position - len(update)); data = roll(data, roll); position += roll
  long long roll = s->capacity - s->insert_position - n_rows;
  if (roll > 0) roll = 0;
  const long long head = ((s->head - roll) % s->capacity + s->capacity) % s->capacity;  // roll by r: new[i] = old[i - r]
  const long long position = s->insert_position + roll;
  const long long first_physical = (head + position) % s->capacity;
  // tile of rows_per_cta rows in at most 20 KB of shared memory: 5 x 16 bytes per thread in flight
  int rows_per_cta = static_cast<int>((20 * 1024) / (4 * static_cast<long long>(s->row_width)));
  if (rows_per_cta > 512) rows_per_cta = 512;
  if (rows_per_cta >= 32) rows_per_cta &= ~31;
  MBPO_REQUIRE(rows_per_cta >= 1, "replay_insert: a row of %d floats does not fit the staging tile", s->row_width);
  const long long blocks = (n_rows + rows_per_cta - 1) / rows_per_cta;
  MBPO_REQUIRE(blocks < (1LL << 31), "replay_insert: n_rows %lld too large for one launch", n_rows);
  const size_t smem = (static_cast<size_t>(rows_per_cta) * s->row_width + 4) * sizeof(float);
  // 16-byte copies when every block of a tile starts on a 16-byte boundary
  bool vec = (reinterpret_cast<uintptr_t>(s->data) & 15u) == 0 && rows_per_cta % 4 == 0;
  for (int f = 0; f < fields->num_fields; ++f) vec = vec && (reinterpret_cast<uintptr_t>(fields->ptr[f]) & 15u) == 0;
  if (vec)
    replay_pack_kernel<true><<<static_cast<unsigned>(blocks), PACK_THREADS, smem, as_stream(stream)>>>(
        ft, s->row_width, rows_per_cta, n_rows, s->data, s->capacity, first_physical);
  else
    replay_pack_kernel<false><<<static_cast<unsigned>(blocks), PACK_THREADS, smem, as_stream(stream)>>>(
        ft, s->row_width, rows_per_cta, n_rows, s->data, s->capacity, first_physical);
  rc = check_launch("replay_pack_kernel");
  if (rc != MBPO_OK) return rc;
  s->head = head;
  s->insert_position = (position + n_rows) % (s->capacity + 1);
  const long long sp = s->sample_position + roll;
  s->sample_position = sp > 0 ? sp : 0;
  return MBPO_OK;
}

int mbpo_replay_sample(const MbpoReplayState* s, const uint32_t* key, int prng_mode, int sample_batch_size,
                       uint32_t* key_out, int32_t* idx_out, float* batch_out, void* stream) {
  int rc = check_state(s, "replay_sample");
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(prng_mode == 0 || prng_mode == 1, "replay_sample: bad prng_mode %d", prng_mode);
  MBPO_REQUIRE(sample_batch_size >= 1, "replay_sample: sample_batch_size %d < 1", sample_batch_size);
  MBPO_REQUIRE(key && key_out && batch_out, "replay_sample: null pointer");
  const int minval = static_cast<int>(s->sample_position), maxval = static_cast<int>(s->insert_position);
  const uint32_t span = randint_span(minval, maxval);
  const int threads = 128;
  const unsigned blocks = static_cast<unsigned>((sample_batch_size + threads - 1) / threads);
  return with_prng(prng_mode, [&](auto P) {
    replay_sample_kernel<P><<<blocks, threads, 0, as_stream(stream)>>>(
        s->data, s->capacity, s->row_width, s->head, key, sample_batch_size, minval, span, key_out, idx_out, batch_out);
    return check_launch("replay_sample_kernel");
  });
}

int mbpo_replay_read(const MbpoReplayState* s, long long first, long long n, float* rows_out, void* stream) {
  int rc = check_state(s, "replay_read");
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(first >= 0 && n >= 0 && first + n <= s->capacity, "replay_read: rows [%lld, %lld) outside [0, %lld)",
               first, first + n, s->capacity);
  if (n == 0) return MBPO_OK;
  MBPO_REQUIRE(rows_out != nullptr, "replay_read: rows_out is null");
  const long long total = n * s->row_width;
  const int threads = 256;
  const long long blocks = (total + threads - 1) / threads;
  MBPO_REQUIRE(blocks < (1LL << 31), "replay_read: too many rows for one launch");
  replay_read_kernel<<<static_cast<unsigned>(blocks), threads, 0, as_stream(stream)>>>(
      s->data, s->capacity, s->row_width, s->head, first, total, rows_out);
  return check_launch("replay_read_kernel");
}

int mbpo_env_reset_from_buffer(const MbpoReplayState* s, const uint32_t* rngs, int E, int prng_mode,
                               int sample_batch_size, int x_dim, int reward_col, float* obs_out, float* reward_out,
                               uint32_t* sys_key_out, int32_t* idx_out, void* stream) {
  int rc = check_state(s, "env_reset_from_buffer");
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(prng_mode == 0 || prng_mode == 1, "env_reset_from_buffer: bad prng_mode %d", prng_mode);
  MBPO_REQUIRE(E >= 0, "env_reset_from_buffer: E < 0");
  MBPO_REQUIRE(sample_batch_size >= 1, "env_reset_from_buffer: sample_batch_size %d < 1", sample_batch_size);
  MBPO_REQUIRE(x_dim >= 1 && x_dim <= s->row_width && reward_col >= 0 && reward_col < s->row_width,
               "env_reset_from_buffer: x_dim %d / reward_col %d outside a row of %d", x_dim, reward_col, s->row_width);
  if (E == 0) return MBPO_OK;
  MBPO_REQUIRE(rngs && obs_out && reward_out && sys_key_out, "env_reset_from_buffer: null pointer");
  const int minval = static_cast<int>(s->sample_position), maxval = static_cast<int>(s->insert_position);
  const uint32_t span = randint_span(minval, maxval);
  const int threads = 128;
  const unsigned blocks = static_cast<unsigned>((E + threads - 1) / threads);
  return with_prng(prng_mode, [&](auto P) {
    env_reset_kernel<P><<<blocks, threads, 0, as_stream(stream)>>>(s->data, s->capacity, s->row_width, s->head, rngs, E,
                                                                  sample_batch_size, minval, span, x_dim, reward_col,
                                                                  obs_out, reward_out, sys_key_out, idx_out);
    return check_launch("env_reset_kernel");
  });
}

int mbpo_eval_metrics(const float* reward, const float* discount, const float* steps_in, const float* done_in,
                      int action_repeat, int E, int T, long long stride_t, long long stride_e, float* episode_reward,
                      float* episode_steps, float* active, void* stream) {
  MBPO_REQUIRE(E >= 0 && T >= 0, "eval_metrics: negative size");
  MBPO_REQUIRE(action_repeat >= 1, "eval_metrics: action_repeat %d < 1", action_repeat);
  if (E == 0) return MBPO_OK;
  MBPO_REQUIRE(steps_in && done_in && episode_reward && episode_steps && active, "eval_metrics: null pointer");
  MBPO_REQUIRE(T == 0 || (reward && discount), "eval_metrics: null pointer");
  const int threads = 128;
  eval_metrics_kernel<<<(E + threads - 1) / threads, threads, 0, as_stream(stream)>>>(
      reward, discount, steps_in, done_in, static_cast<float>(action_repeat), E, T, stride_t, stride_e, episode_reward,
      episode_steps, active);
  return check_launch("eval_metrics_kernel");
}

size_t mbpo_running_statistics_workspace_bytes(int X) {
  if (X < 1 || X > RS_MAX_X) return 0;
  return static_cast<size_t>(RS_CTAS) * 2 * X * sizeof(double);
}

int mbpo_running_statistics_accumulate(const float* batch, long long n_rows, int X, const float* mean,
                                       void* workspace, size_t workspace_bytes, double* sums_out, void* stream) {
  MBPO_REQUIRE(X >= 1 && X <= RS_MAX_X, "running_statistics: X %d outside [1, %d]", X, RS_MAX_X);
  MBPO_REQUIRE(n_rows >= 0, "running_statistics: n_rows < 0");
  MBPO_REQUIRE(mean && workspace && sums_out, "running_statistics: null pointer");
  MBPO_REQUIRE(n_rows == 0 || batch, "running_statistics: batch is null");
  if (workspace_bytes < mbpo_running_statistics_workspace_bytes(X))
    return fail(MBPO_EWORKSPACE, "running_statistics: workspace %zu < %zu bytes", workspace_bytes,
                mbpo_running_statistics_workspace_bytes(X));
  MBPO_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 7u) == 0, "running_statistics: workspace not 8-byte aligned");
  const long long total = n_rows * X;
  // the largest multiple of X that the grid covers: every thread keeps one column
  const long long stride = (static_cast<long long>(RS_CTAS) * RS_THREADS / X) * X;
  running_stats_partial_kernel<<<RS_CTAS, RS_THREADS, 0, as_stream(stream)>>>(batch, total, X, mean, stride,
                                                                             static_cast<double*>(workspace));
  int rc = check_launch("running_stats_partial_kernel");
  if (rc != MBPO_OK) return rc;
  running_stats_combine_kernel<<<1, 2 * RS_MAX_X + 32, 0, as_stream(stream)>>>(
      static_cast<const double*>(workspace), RS_CTAS, X, static_cast<double>(n_rows), sums_out);
  return check_launch("running_stats_combine_kernel");
}

int mbpo_running_statistics_finalize(const double* sums, int X, const float* count_in,
                                     const float* mean_in, const float* summed_variance_in, float std_min_value,
                                     float std_max_value, float* count_out, float* mean_out,
                                     float* summed_variance_out, float* std_out, void* stream) {
  MBPO_REQUIRE(X >= 1 && X <= RS_MAX_X, "running_statistics: X %d outside [1, %d]", X, RS_MAX_X);
  MBPO_REQUIRE(sums && count_in && mean_in && summed_variance_in && count_out && mean_out && summed_variance_out &&
                   std_out, "running_statistics: null pointer");
  running_stats_finalize_kernel<<<1, RS_MAX_X, 0, as_stream(stream)>>>(sums, X, count_in, mean_in,
                                                                       summed_variance_in, std_min_value,
                                                                       std_max_value, count_out, mean_out,
                                                                       summed_variance_out, std_out);
  return check_launch("running_stats_finalize_kernel");
}

int mbpo_running_statistics_normalize(const float* batch, long long n_rows, int X, const float* mean,
                                      const float* std, float max_abs_value, float* out, void* stream) {
  MBPO_REQUIRE(X >= 1 && X <= RS_MAX_X, "running_statistics: X %d outside [1, %d]", X, RS_MAX_X);
  MBPO_REQUIRE(n_rows >= 0, "running_statistics: n_rows < 0");
  if (n_rows == 0) return MBPO_OK;
  MBPO_REQUIRE(batch && mean && std && out, "running_statistics: null pointer");
  const long long total = n_rows * X;
  const int threads = 256;
  const long long blocks = (total + threads - 1) / threads;
  MBPO_REQUIRE(blocks < (1LL << 31), "running_statistics: too many rows for one launch");
  running_stats_normalize_kernel<<<static_cast<unsigned>(blocks), threads, 0, as_stream(stream)>>>(
      batch, total, X, mean, std, max_abs_value, out);
  return check_launch("running_stats_normalize_kernel");
}

int mbpo_normalizer_finalize(const double* sums, int X, const double* size_in, const float* mean_in,
                             const float* std_in, float eps, double* size_out, float* mean_out, float* std_out,
                             void* stream) {
  MBPO_REQUIRE(X >= 1 && X <= RS_MAX_X, "normalizer: X %d outside [1, %d]", X, RS_MAX_X);
  MBPO_REQUIRE(sums && size_in && mean_in && std_in && size_out && mean_out && std_out, "normalizer: null pointer");
  normalizer_finalize_kernel<<<1, RS_MAX_X, 0, as_stream(stream)>>>(sums, X, size_in, mean_in, std_in, eps, size_out,
                                                                    mean_out, std_out);
  return check_launch("normalizer_finalize_kernel");
}

int mbpo_normalizer_inverse(const float* batch, long long n_rows, int X, const float* mean, const float* std,
                            float* out, void* stream) {
  MBPO_REQUIRE(X >= 1 && X <= RS_MAX_X, "normalizer: X %d outside [1, %d]", X, RS_MAX_X);
  MBPO_REQUIRE(n_rows >= 0, "normalizer: n_rows < 0");
  if (n_rows == 0) return MBPO_OK;
  MBPO_REQUIRE(batch && mean && std && out, "normalizer: null pointer");
  const long long total = n_rows * X;
  const int threads = 256;
  const long long blocks = (total + threads - 1) / threads;
  MBPO_REQUIRE(blocks < (1LL << 31), "normalizer: too many rows for one launch");
  normalizer_inverse_kernel<<<static_cast<unsigned>(blocks), threads, 0, as_stream(stream)>>>(batch, total, X, mean, std,
                                                                                            out);
  return check_launch("normalizer_inverse_kernel");
}

int mbpo_replay_take(const MbpoReplayState* s, const int32_t* idx, long long n, float* rows_out, void* stream) {
  int rc = check_state(s, "replay_take");
  if (rc != MBPO_OK) return rc;
  MBPO_REQUIRE(n >= 0, "replay_take: n < 0");
  if (n == 0) return MBPO_OK;
  MBPO_REQUIRE(idx && rows_out, "replay_take: null pointer");
  const long long total = n * s->row_width;
  const int threads = 256;
  const long long blocks = (total + threads - 1) / threads;
  MBPO_REQUIRE(blocks < (1LL << 31), "replay_take: too many rows for one launch");
  replay_take_kernel<<<static_cast<unsigned>(blocks), threads, 0, as_stream(stream)>>>(
      s->data, s->capacity, s->row_width, s->head, idx, total, rows_out);
  return check_launch("replay_take_kernel");
}

int mbpo_compute_gae(const float* truncation, const float* termination, const float* rewards, const float* values,
                     const float* bootstrap_value, int E, int T, long long stride_t, long long stride_e,
                     double discount, double lambda_, float* vs_out, float* advantages_out, void* stream) {
  MBPO_REQUIRE(E >= 0 && T >= 0, "compute_gae: negative size");
  if (E == 0 || T == 0) return MBPO_OK;
  MBPO_REQUIRE(truncation && termination && rewards && values && bootstrap_value && vs_out && advantages_out,
               "compute_gae: null pointer");
  const int threads = 128;
  compute_gae_kernel<<<(E + threads - 1) / threads, threads, 0, as_stream(stream)>>>(
      truncation, termination, rewards, values, bootstrap_value, E, T, stride_t, stride_e,
      static_cast<float>(discount), static_cast<float>(lambda_), vs_out, advantages_out);
  return check_launch("compute_gae_kernel");
}

}  // extern "C"
