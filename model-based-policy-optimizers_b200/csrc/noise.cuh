// Colored (power-law) Gaussian noise row: powerlaw_psd_gaussian(exponent, H, rng)
// (mbpo/utils/general_utils.py:81-208), one row per thread.
//
//   key_sr, key_si, _ = split(rng, 3)                         :189
//   sr = normal(key_sr, (F,)) * s_scale ; si likewise         :190-191
//   Nyquist (even H) and DC: imaginary part 0, real part * sqrt(2)   :195-201
//   y = irfft(sr + i*si, n=H) / sigma                         :207
//
// The irfft is a direct real DFT with compile-time twiddles (they fold into FFMA immediates)
// that exploits y[t], y[H-t] sharing the cosine sum and having opposite sine sums.
#pragma once
#include "../../include/mbpo_b200.h"
#include "mathx.cuh"
#include "threefry.cuh"

namespace mbpo {

namespace detail {
constexpr double csin(double x) {
  double t = x, s = x;
  for (int n = 1; n < 30; ++n) {
    t *= -x * x / ((2 * n) * (2 * n + 1));
    s += t;
  }
  return s;
}
constexpr double ccos(double x) {
  double t = 1, s = 1;
  for (int n = 1; n < 30; ++n) {
    t *= -x * x / ((2 * n - 1) * (2 * n));
    s += t;
  }
  return s;
}
// cos/sin(2*pi*j/H) * weight/H folded: c[j], s[j] for j in [0, H)
template <int H>
struct Twiddle {
  float c[H];
  float s[H];
  constexpr Twiddle() : c(), s() {
    for (int j = 0; j < H; ++j) {
      double a = 6.283185307179586476925 * j / H;
      if (a > 3.14159265358979323846) a -= 6.283185307179586476925;
      c[j] = static_cast<float>(ccos(a) / H);
      s[j] = static_cast<float>(csin(a) / H);
    }
  }
};
}  // namespace detail

template <int H>
struct NoiseShape {
  static constexpr int F = H / 2 + 1;          // rfft bins
  static constexpr int FPAD = F + (F & 1);     // legacy counter padding
  static constexpr int HALF = FPAD / 2;        // threefry blocks per normal vector (legacy)
  static constexpr bool EVEN = (H % 2) == 0;
};

// Stages the scaled normals of one spectrum half (real or imaginary part) into `stage`:
//   stage[k]         = sr[k]            k in [0, F)
//   stage[F + k - 1] = si[k]            k in [1, LASTK)   (DC and, for even H, Nyquist have no
//                                                           imaginary part: general_utils.py:195-201)
// so the H needed values fill exactly the H floats of the caller's row.  The threefry blocks run
// in a rolled loop (small code: the instruction cache matters more than the last bit of ILP);
// `scale` is indexed dynamically (constant bank / shared memory).
// One unit of that work: in the legacy layout threefry block j, whose two words are normals j and HALF + j; in the
// partitionable layout the block of word j.  NoiseShape<H>::tasks(MODE) units make one half spectrum; they are
// independent, so one thread may run them in a loop (stage_normals) or several threads may share them (the
// cluster plan, icem_cluster_kernels.cuh) with the same results.
template <int H, int MODE, bool IMAG>
__device__ __forceinline__ void stage_normals_task(Key2 key, const float* __restrict__ scale, float* stage,
                                                   uint32_t* bits_out, int j) {
  using S = NoiseShape<H>;
  constexpr int LASTK = S::EVEN ? S::F - 1 : S::F;
  // v = bits_to_normal(word) * scale[k]
  auto put = [&](int k, uint32_t word, float v) {
    if (bits_out) bits_out[k] = word;
    if (!IMAG) {
      stage[k] = v;
    } else if (k >= 1 && k < LASTK) {
      stage[S::F + k - 1] = v;
    }
  };
  if (MODE == 1) {
    uint32_t x0 = 0u, x1 = static_cast<uint32_t>(j);
    threefry2x32(key.k0, key.k1, x0, x1);
    put(j, x0 ^ x1, bits_to_normal(x0 ^ x1) * scale[j]);
  } else {
    uint32_t x0 = static_cast<uint32_t>(j);
    uint32_t x1 = (S::HALF + j < S::F) ? static_cast<uint32_t>(S::HALF + j) : 0u;
    threefry2x32(key.k0, key.k1, x0, x1);
    if (S::HALF + j < S::F) {   // both words are normals: one packed chain
      float v0, v1;
      unpack2(mul2(bits_to_normal2(x0, x1), pack2(scale[j], scale[S::HALF + j])), v0, v1);
      put(j, x0, v0);
      put(S::HALF + j, x1, v1);
    } else {
      put(j, x0, bits_to_normal(x0) * scale[j]);
    }
  }
}

template <int H, int MODE>
__host__ __device__ constexpr int noise_tasks() { return MODE == 1 ? NoiseShape<H>::F : NoiseShape<H>::HALF; }

template <int H, int MODE, bool IMAG>
__device__ __forceinline__ void stage_normals(Key2 key, const float* __restrict__ scale, float* stage,
                                              uint32_t* bits_out) {
#pragma unroll 2
  for (int j = 0; j < noise_tasks<H, MODE>(); ++j) stage_normals_task<H, MODE, IMAG>(key, scale, stage, bits_out, j);
}

// The inverse real DFT as independent GROUPS of outputs (each output is one thread's multiply-add chain in a fixed
// order, so the groups may run in one thread one after the other or in different threads):
//   odd H :  group 0 = {y[0]};  group t = {y[t], y[H - t]}, t = 1 .. (H - 1) / 2   (shared cosine sum, opposite sine sums)
//   even H:  one more split.  With h = H/2, cos(2 pi k (t + h) / H) = (-1)^k cos(2 pi k t / H) (sin likewise), so the
//            even-k and odd-k partial sums ae, ao (cosine) and be, bo (sine) of one t give FOUR outputs:
//              y[t]     = (ae + ao) - (be + bo) + n        y[H - t] = (ae + ao) + (be + bo) + n
//              y[h + t] = (ae - ao) - (be - bo) + nh       y[h - t] = (ae - ao) + (be - bo) + nh
//            (n, nh: the Nyquist bin with the sign of (-1)^t, (-1)^(t + h)) -- half the multiply-adds of the t / H - t
//            pairing alone.  group 0 = {y[0], y[h]};  group t = those four (two when 2 t == h), t = 1 .. h / 2.
// colored_noise_row_rt evaluates the same expressions in the same order.  __fmul_rn / __fadd_rn where a plain
// product feeds a sum: such a pair is a candidate for FMA contraction, which the compiler applies differently in
// differently shaped code (1 ulp apart); these are not.
template <int H>
__host__ __device__ constexpr int dft_groups() { return (H % 2 == 0) ? 1 + (H / 2) / 2 : 1 + (H - 1) / 2; }

template <int H, int G, typename Emit>
__device__ __forceinline__ void dft_group(const float (&sr)[NoiseShape<H>::F], const float (&si)[NoiseShape<H>::F],
                                          Emit emit) {
  using S = NoiseShape<H>;
  constexpr detail::Twiddle<H> tw{};
  constexpr int LASTK = S::EVEN ? S::F - 1 : S::F;  // bins [1, LASTK) have weight 2
  constexpr int t = G;
  if constexpr (!S::EVEN) {
    if constexpr (G == 0) {
      float a = __fmul_rn(sr[0], tw.c[0]);
#pragma unroll
      for (int k = 1; k < LASTK; ++k) a = fmaf(sr[k], 2.0f * tw.c[0], a);
      emit(0, a);
    } else {
      float a = __fmul_rn(sr[0], tw.c[0]);
      float b = 0.0f;
#pragma unroll
      for (int k = 1; k < LASTK; ++k) {
        a = fmaf(sr[k], 2.0f * tw.c[(k * t) % H], a);
        b = fmaf(si[k], 2.0f * tw.s[(k * t) % H], b);
      }
      emit(t, __fsub_rn(a, b));
      emit(H - t, __fadd_rn(a, b));
    }
  } else {
    constexpr int h = H / 2;
    const float d = __fmul_rn(sr[0], tw.c[0]);
    const float nq = __fmul_rn(sr[h], tw.c[0]);
    if constexpr (G == 0) {
      float ae = d, ao = 0.0f;
#pragma unroll
      for (int k = 1; k < h; ++k) {
        if (k & 1) ao = fmaf(sr[k], 2.0f * tw.c[0], ao);
        else ae = fmaf(sr[k], 2.0f * tw.c[0], ae);
      }
      emit(0, __fadd_rn(__fadd_rn(ae, ao), nq));
      emit(h, __fadd_rn(__fsub_rn(ae, ao), (h & 1) ? -nq : nq));
    } else {
      float ae = d, ao = 0.0f, be = 0.0f, bo = 0.0f;
#pragma unroll
      for (int k = 1; k < h; ++k) {
        if (k & 1) {
          ao = fmaf(sr[k], 2.0f * tw.c[(k * t) % H], ao);
          bo = fmaf(si[k], 2.0f * tw.s[(k * t) % H], bo);
        } else {
          ae = fmaf(sr[k], 2.0f * tw.c[(k * t) % H], ae);
          be = fmaf(si[k], 2.0f * tw.s[(k * t) % H], be);
        }
      }
      const float n = (t & 1) ? -nq : nq;
      const float p = __fadd_rn(ae, ao), r = __fadd_rn(be, bo);
      emit(t, __fadd_rn(__fsub_rn(p, r), n));
      emit(H - t, __fadd_rn(__fadd_rn(p, r), n));
      if constexpr (2 * t < h) {
        const float nh = ((t + h) & 1) ? -nq : nq;
        const float q = __fsub_rn(ae, ao), v = __fsub_rn(be, bo);
        emit(h + t, __fadd_rn(__fsub_rn(q, v), nh));
        emit(h - t, __fadd_rn(__fadd_rn(q, v), nh));
      }
    }
  }
}

// Loads the staged half spectra of one row into registers.
template <int H>
__device__ __forceinline__ void load_staged(const float* stage, float (&sr)[NoiseShape<H>::F],
                                            float (&si)[NoiseShape<H>::F]) {
  using S = NoiseShape<H>;
  constexpr int LASTK = S::EVEN ? S::F - 1 : S::F;
#pragma unroll
  for (int k = 0; k < S::F; ++k) sr[k] = stage[k];
  si[0] = 0.0f;
#pragma unroll
  for (int k = 1; k < S::F; ++k) si[k] = (k < LASTK) ? stage[S::F + k - 1] : 0.0f;
}

namespace detail {
template <int H, int G, typename Emit>
__device__ __forceinline__ void dft_all_groups(const float (&sr)[NoiseShape<H>::F],
                                               const float (&si)[NoiseShape<H>::F], Emit emit) {
  if constexpr (G < dft_groups<H>()) {
    dft_group<H, G>(sr, si, emit);
    dft_all_groups<H, G + 1>(sr, si, emit);
  }
}
// group g (runtime, uniform across the caller's warp) of the row
template <int H, int G, typename Emit>
__device__ __forceinline__ void dft_one_group(int g, const float (&sr)[NoiseShape<H>::F],
                                              const float (&si)[NoiseShape<H>::F], Emit emit) {
  if constexpr (G < dft_groups<H>()) {
    if (g == G) dft_group<H, G>(sr, si, emit);
    else dft_one_group<H, G + 1>(g, sr, si, emit);
  }
}
}  // namespace detail

// Emits y[t] for every t in [0, H) through emit(t, value).  `stage` is H floats private to the
// calling thread (its own shared-memory action row: emit may overwrite it, every staged value is
// in a register by then).  `scale` may live in shared or constant memory (F floats).
template <int H, int MODE, typename Emit>
__device__ __forceinline__ void colored_noise_row(Key2 rng, const float* __restrict__ scale, float* stage,
                                                  uint32_t* bits_out, Emit emit) {
  using S = NoiseShape<H>;
  Key2 key_sr, key_si;
  split3_first2<MODE>(rng, key_sr, key_si);
  stage_normals<H, MODE, false>(key_sr, scale, stage, bits_out);
  stage_normals<H, MODE, true>(key_si, scale, stage, bits_out ? bits_out + S::F : nullptr);
  float sr[S::F], si[S::F];
  load_staged<H>(stage, sr, si);
  detail::dft_all_groups<H, 0>(sr, si, emit);
}

// ------------------------------------------------------------------------------------------
// Any horizon (iCemTO(horizon=...) is a free int in the reference, icem_optimizer.py:94-96;
// powerlaw_psd_gaussian takes any size, general_utils.py:134-143).  Same key tree, same words,
// same operation ORDER as the unrolled instances above -- so the six compiled horizons give the
// same bits through either routine -- but rolled loops and a twiddle table in the constant bank
// (every lane of a warp reads the same entry: a broadcast).  The staged normals stay in `stage`
// while the outputs are emitted, so `emit` must not write to `stage`.
// ------------------------------------------------------------------------------------------
struct TwiddleTable {
  float c[MBPO_MAX_HORIZON];  // cos(2 pi j / H) / H
  float s[MBPO_MAX_HORIZON];  // sin(2 pi j / H) / H
};

// Host: the table detail::Twiddle<H> holds at compile time, by the same double arithmetic.
inline void fill_twiddles(int H, TwiddleTable& t) {
  for (int j = 0; j < MBPO_MAX_HORIZON; ++j) t.c[j] = t.s[j] = 0.0f;
  for (int j = 0; j < H; ++j) {
    double a = 6.283185307179586476925 * j / H;
    if (a > 3.14159265358979323846) a -= 6.283185307179586476925;
    t.c[j] = static_cast<float>(detail::ccos(a) / H);
    t.s[j] = static_cast<float>(detail::csin(a) / H);
  }
}

template <int MODE, bool IMAG>
__device__ __forceinline__ void stage_normals_rt(int H, Key2 key, const float* __restrict__ scale, float* stage,
                                                 uint32_t* bits_out) {
  const int F = H / 2 + 1;
  const int HALF = (F + (F & 1)) / 2;
  const int LASTK = (H % 2 == 0) ? F - 1 : F;
  auto put = [&](int k, uint32_t word) {
    if (bits_out) bits_out[k] = word;
    if (!IMAG) {
      stage[k] = bits_to_normal(word) * scale[k];
    } else if (k >= 1 && k < LASTK) {
      stage[F + k - 1] = bits_to_normal(word) * scale[k];
    }
  };
  if (MODE == 1) {
#pragma unroll 2
    for (int f = 0; f < F; ++f) {
      uint32_t x0 = 0u, x1 = static_cast<uint32_t>(f);
      threefry2x32(key.k0, key.k1, x0, x1);
      put(f, x0 ^ x1);
    }
  } else {
#pragma unroll 2
    for (int j = 0; j < HALF; ++j) {
      uint32_t x0 = static_cast<uint32_t>(j);
      uint32_t x1 = (HALF + j < F) ? static_cast<uint32_t>(HALF + j) : 0u;
      threefry2x32(key.k0, key.k1, x0, x1);
      put(j, x0);
      if (HALF + j < F) put(HALF + j, x1);
    }
  }
}

template <int MODE, typename Emit>
__device__ __forceinline__ void colored_noise_row_rt(int H, Key2 rng, const float* __restrict__ scale,
                                                     const TwiddleTable& tw, float* stage, uint32_t* bits_out,
                                                     Emit emit) {
  const int F = H / 2 + 1;
  const bool even = (H % 2) == 0;
  const int LASTK = even ? F - 1 : F;
  Key2 key_sr, key_si;
  split3_first2<MODE>(rng, key_sr, key_si);
  stage_normals_rt<MODE, false>(H, key_sr, scale, stage, bits_out);
  stage_normals_rt<MODE, true>(H, key_si, scale, stage, bits_out ? bits_out + F : nullptr);
  const float* sr = stage;          // sr[k], k in [0, F)
  const float* si = stage + F - 1;  // si[k], k in [1, LASTK)
  const float c0 = tw.c[0];
  if (!even) {
    {
      float a = __fmul_rn(sr[0], c0);
      for (int k = 1; k < LASTK; ++k) a = fmaf(sr[k], 2.0f * c0, a);
      emit(0, a);
    }
    for (int t = 1; 2 * t < H; ++t) {
      float a = __fmul_rn(sr[0], c0);
      float b = 0.0f;
      int j = 0;  // (k * t) % H
#pragma unroll 4
      for (int k = 1; k < LASTK; ++k) {
        j += t;
        if (j >= H) j -= H;
        a = fmaf(sr[k], 2.0f * tw.c[j], a);
        b = fmaf(si[k], 2.0f * tw.s[j], b);
      }
      emit(t, __fsub_rn(a, b));
      emit(H - t, __fadd_rn(a, b));
    }
  } else {
    const int h = H / 2;
    const float d = __fmul_rn(sr[0], c0);
    const float nq = __fmul_rn(sr[h], c0);
    {
      float ae = d, ao = 0.0f;
      for (int k = 1; k + 1 < h; k += 2) {
        ao = fmaf(sr[k], 2.0f * c0, ao);
        ae = fmaf(sr[k + 1], 2.0f * c0, ae);
      }
      if ((h & 1) == 0) ao = fmaf(sr[h - 1], 2.0f * c0, ao);   // k = h - 1 is odd and has no even partner below h
      emit(0, __fadd_rn(__fadd_rn(ae, ao), nq));
      emit(h, __fadd_rn(__fsub_rn(ae, ao), (h & 1) ? -nq : nq));
    }
    for (int t = 1; 2 * t <= h; ++t) {
      float ae = d, ao = 0.0f, be = 0.0f, bo = 0.0f;
      int j = 0;  // (k * t) % H
#pragma unroll 2
      for (int k = 1; k + 1 < h; k += 2) {
        j += t;
        if (j >= H) j -= H;
        ao = fmaf(sr[k], 2.0f * tw.c[j], ao);
        bo = fmaf(si[k], 2.0f * tw.s[j], bo);
        j += t;
        if (j >= H) j -= H;
        ae = fmaf(sr[k + 1], 2.0f * tw.c[j], ae);
        be = fmaf(si[k + 1], 2.0f * tw.s[j], be);
      }
      if ((h & 1) == 0) {
        j += t;
        if (j >= H) j -= H;
        ao = fmaf(sr[h - 1], 2.0f * tw.c[j], ao);
        bo = fmaf(si[h - 1], 2.0f * tw.s[j], bo);
      }
      const float n = (t & 1) ? -nq : nq;
      const float p = __fadd_rn(ae, ao), r = __fadd_rn(be, bo);
      emit(t, __fadd_rn(__fsub_rn(p, r), n));
      emit(H - t, __fadd_rn(__fadd_rn(p, r), n));
      if (2 * t < h) {
        const float nh = ((t + h) & 1) ? -nq : nq;
        const float q = __fsub_rn(ae, ao), v = __fsub_rn(be, bo);
        emit(h + t, __fadd_rn(__fsub_rn(q, v), nh));
        emit(h - t, __fadd_rn(__fadd_rn(q, v), nh));
      }
    }
  }
}

// Host/device helper: the per-bin multiplier table colored_noise_row expects.
//   scale[f] = s_scale[f] / sigma, times sqrt(2) for the DC bin and (even H) the Nyquist bin.
inline void fill_noise_scale(const float* s_scale, float sigma, int horizon, float* scale_out) {
  const int F = horizon / 2 + 1;
  const float inv_sigma = 1.0f / sigma;
  for (int f = 0; f < F; ++f) {
    float s = s_scale[f] * inv_sigma;
    if (f == 0 || (f == F - 1 && horizon % 2 == 0)) s *= 1.41421356f;
    scale_out[f] = s;
  }
}

}  // namespace mbpo
