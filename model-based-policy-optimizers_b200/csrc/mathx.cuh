// bits -> uniform -> normal, as jax.random does it (jax/_src/random.py _uniform,
// _normal_real) with XLA's float32 erf_inv (Giles' polynomials, xla ErfInv32).
// Call sites in the reference: mbpo/utils/general_utils.py:190-191.
#pragma once
#include <stdint.h>

namespace mbpo {

// Packed float32 pairs (sm_100: FADD2 / FMUL2 / FFMA2).  One issue slot retires the operation for both elements,
// each IEEE-rounded exactly like the scalar instruction, so a pair form that applies the scalar code's operations to
// the same operands in the same order gives the same bits.  An operand may be a scalar broadcast to both elements
// (pack2(s, s): a register or a 32-bit immediate in the SASS).  Compares, selects, min / max, integer ops and MUFU
// have no packed form here: they run per element on unpack2's halves.
// Contraction: ptxas (CUDA 12.9) fuses a mul.rn.f32x2 whose result feeds an add / sub.rn.f32x2 into one FFMA2 --
// unlike the scalar mul.rn / add.rn, which it never contracts -- and the fused result rounds once instead of twice.
// So a pair form never adds or subtracts a mul2 result: where the scalar code rounds a product before a sum, that sum
// runs per element (__fadd_rn / __fsub_rn on unpack2's halves).
typedef unsigned long long f32x2_t;
__device__ __forceinline__ f32x2_t pack2(float lo, float hi) {
  f32x2_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ f32x2_t splat2(float v) { return pack2(v, v); }
__device__ __forceinline__ void unpack2(f32x2_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2_t add2(f32x2_t x, f32x2_t y) {
  f32x2_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(x), "l"(y));
  return r;
}
__device__ __forceinline__ f32x2_t sub2(f32x2_t x, f32x2_t y) {
  f32x2_t r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(x), "l"(y));
  return r;
}
__device__ __forceinline__ f32x2_t mul2(f32x2_t x, f32x2_t y) {
  f32x2_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(x), "l"(y));
  return r;
}
__device__ __forceinline__ f32x2_t fma2(f32x2_t x, f32x2_t y, f32x2_t z) {
  f32x2_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(x), "l"(y), "l"(z));
  return r;
}

// uniform in [lo, hi): mantissa trick, then max(lo, f*(hi-lo)+lo)
__device__ __forceinline__ float bits_to_uniform(uint32_t bits, float lo, float hi) {
  const float f = __uint_as_float((bits >> 9) | 0x3F800000u) - 1.0f;
  return fmaxf(lo, __fadd_rn(__fmul_rn(f, hi - lo), lo));  // unfused, as the oracle
}

// XLA ErfInv32: w = -log1p(-x*x); w < 5 ? poly(w-2.5) : poly(sqrt(w)-3); result p*x.
// Like the reference formula, x*x is rounded to float32 first (this rounding dominates the
// tail: for |x| -> 1 it is a several-percent perturbation of 1 - x*x, so a "more accurate"
// (1-x)(1+x) would NOT match JAX).  log1p(-t) is then evaluated as log(1 - t) with the hardware
// log2 (MUFU.LG2): 1 - t is exact for t >= 0.5 (Sterbenz) and otherwise perturbs w by <= 6e-8
// absolute, i.e. the result by <= ~2e-8 relative (|p'(w)| <= 0.25) -- below the 1-2 ulp spread
// between log1p implementations (XLA's own is a polynomial), ~20 instructions cheaper.
// GUARD = false drops the |x| == 1 -> +-inf special case for callers whose argument is provably
// inside (-1, 1).
// log(v) = lg2(v) * ln 2 with the bare MUFU.LG2 (lg2.approx.ftz): what __logf computes for a normal v, without
// the denormal-input guard nvcc wraps around it (three instructions per call).  The callers' arguments are 0
// (-> -inf in both) or >= 2^-24.
__device__ __forceinline__ float log_normal_arg(float v) {
  float l;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(v));
  return l * 0.693147182f;
}

// ErfInv32's polynomial for w >= 5 (the tail: ~0.3% of uniform arguments).
__device__ __forceinline__ float erf_inv_tail(float w) {
  w = sqrtf(w) - 3.0f;
  float p = -0.000200214257f;
  p = fmaf(p, w, 0.000100950558f);
  p = fmaf(p, w, 0.00134934322f);
  p = fmaf(p, w, -0.00367342844f);
  p = fmaf(p, w, 0.00573950773f);
  p = fmaf(p, w, -0.0076224613f);
  p = fmaf(p, w, 0.00943887047f);
  p = fmaf(p, w, 1.00167406f);
  p = fmaf(p, w, 2.83297682f);
  return p;
}

template <bool GUARD = true>
__device__ __forceinline__ float erf_inv_f32(float x) {
  float w = -log_normal_arg(1.0f - __fmul_rn(x, x));
  float p;
  if (w < 5.0f) {
    w = w - 2.5f;
    p = 2.81022636e-08f;
    p = fmaf(p, w, 3.43273939e-07f);
    p = fmaf(p, w, -3.5233877e-06f);
    p = fmaf(p, w, -4.39150654e-06f);
    p = fmaf(p, w, 0.00021858087f);
    p = fmaf(p, w, -0.00125372503f);
    p = fmaf(p, w, -0.00417768164f);
    p = fmaf(p, w, 0.246640727f);
    p = fmaf(p, w, 1.50140941f);
  } else {
    p = erf_inv_tail(w);
  }
  return GUARD ? ((fabsf(x) == 1.0f) ? __int_as_float(0x7F800000) * x : p * x) : p * x;
}

// jax.random.normal for one 32-bit word: sqrt(2) * erf_inv(uniform(nextafter(-1,0), 1)).
// hi - lo = 1 - (-0.99999994) rounds to exactly 2.0f in float32, so f * 2 is exact and
// u = f * 2 + lo lies in [lo, 0.99999982]: jax's max(lo, u) is the identity and |u| < 1.
__device__ __forceinline__ float bits_to_normal(uint32_t bits) {
  const float lo = -0.99999994f;  // nextafter(-1, 0)
  const float f = __uint_as_float((bits >> 9) | 0x3F800000u) - 1.0f;
  const float u = f * 2.0f + lo;
  return 1.41421356f * erf_inv_f32<false>(u);
}

// bits_to_normal of two words, packed.  nvcc contracts f * 2.0f + lo into one FFMA and leaves w - 2.5f (w the
// negated product l * ln 2) a separate FMUL and FADD; the pair form does the same.  The two sums that take a product
// (1 - x*x and w - 2.5f) run per element: see the pair helpers on contraction.  erf_inv_f32 branches per element
// on w < 5: the central polynomial runs packed for both elements, and an element in the tail replaces its result by
// erf_inv_tail (the scalar code's else branch).  Same bits as bits_to_normal on each word.
__device__ __forceinline__ f32x2_t bits_to_normal2(uint32_t b0, uint32_t b1) {
  const f32x2_t f = sub2(pack2(__uint_as_float((b0 >> 9) | 0x3F800000u), __uint_as_float((b1 >> 9) | 0x3F800000u)),
                         splat2(1.0f));
  const f32x2_t u = fma2(f, splat2(2.0f), splat2(-0.99999994f));
  float uu0, uu1;
  unpack2(mul2(u, u), uu0, uu1);
  float l0, l1;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l0) : "f"(__fsub_rn(1.0f, uu0)));
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l1) : "f"(__fsub_rn(1.0f, uu1)));
  const f32x2_t neg_w = mul2(pack2(l0, l1), splat2(0.693147182f));   // log_normal_arg
  float nw0, nw1;
  unpack2(neg_w, nw0, nw1);
  const f32x2_t w = pack2(__fsub_rn(-2.5f, nw0), __fsub_rn(-2.5f, nw1));   // w - 2.5f
  f32x2_t p = fma2(splat2(2.81022636e-08f), w, splat2(3.43273939e-07f));
  p = fma2(p, w, splat2(-3.5233877e-06f));
  p = fma2(p, w, splat2(-4.39150654e-06f));
  p = fma2(p, w, splat2(0.00021858087f));
  p = fma2(p, w, splat2(-0.00125372503f));
  p = fma2(p, w, splat2(-0.00417768164f));
  p = fma2(p, w, splat2(0.246640727f));
  p = fma2(p, w, splat2(1.50140941f));
  float p0, p1;
  unpack2(p, p0, p1);
  if (!(-nw0 < 5.0f)) p0 = erf_inv_tail(-nw0);
  if (!(-nw1 < 5.0f)) p1 = erf_inv_tail(-nw1);
  return mul2(splat2(1.41421356f), mul2(pack2(p0, p1), u));
}

// Sort key of jnp.argsort (stable, ascending; icem_optimizer.py:199): monotone uint32 image
// of the float under JAX's sort order (jax/_src/lax/lax.py _float_to_int_for_sort): the
// IEEE total order with -0.0 == +0.0 and every NaN equal and last.
__device__ __forceinline__ uint32_t total_order_key(float v) {
  uint32_t b = __float_as_uint(v);
  if (v == 0.0f) b = 0u;
  if (v != v) b = 0x7FC00000u;
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// ---- bounded-range trigonometry for the pendulum (|angle| <= ~4 rad) ------------------------
// Branch-free float32 sin/cos/atan2 with 1-2 ulp accuracy (the same accuracy class as libm /
// XLA's own polynomial implementations; the parity bar is rel 1e-5).  No large-argument
// slow path: the callers' angles are bounded by pi + max_speed*dt.

// sin and cos of x from those of the reduced argument r = x - q pi/2 (sr, cr) and the quadrant q.
__device__ __forceinline__ void sincos_quadrant(int q, float sr, float cr, float& s, float& c) {
  const bool odd = q & 1;
  const float s0 = odd ? cr : sr;
  const float c0 = odd ? sr : cr;
  s = __int_as_float(__float_as_int(s0) ^ ((q & 2) << 30));
  c = __int_as_float(__float_as_int(c0) ^ (((q + 1) & 2) << 30));
}

// sin and cos of x, |x| < 2^20.  Cody-Waite reduction by pi/2 in three terms, Cephes minimax
// polynomials on [-pi/4, pi/4].
__device__ __forceinline__ void sincos_bounded(float x, float& s, float& c) {
  const float m = fmaf(x, 0.636619747f, 12582912.0f);  // round(x * 2/pi) in the low mantissa bits
  const int q = __float_as_int(m);
  const float fq = m - 12582912.0f;
  float r = fmaf(fq, -1.57079601e+00f, x);
  r = fmaf(fq, -3.13916473e-07f, r);
  r = fmaf(fq, -5.39030253e-15f, r);
  const float r2 = r * r;
  float sp = fmaf(-1.9515295891e-4f, r2, 8.3321608736e-3f);
  sp = fmaf(sp, r2, -1.6666654611e-1f);
  const float sr = fmaf(sp * r2, r, r);
  float cp = fmaf(2.443315711809948e-5f, r2, -1.388731625493765e-3f);
  cp = fmaf(cp, r2, 4.166664568298827e-2f);
  const float cr = fmaf(cp * r2, r2, fmaf(-0.5f, r2, 1.0f));
  sincos_quadrant(q, sr, cr, s, c);
}

// sincos_bounded of both elements of a pair: the same operations packed, the quadrant fix-up per element.
__device__ __forceinline__ void sincos_bounded2(f32x2_t x, f32x2_t& s, f32x2_t& c) {
  const f32x2_t m = fma2(x, splat2(0.636619747f), splat2(12582912.0f));
  const f32x2_t fq = sub2(m, splat2(12582912.0f));
  f32x2_t r = fma2(fq, splat2(-1.57079601e+00f), x);
  r = fma2(fq, splat2(-3.13916473e-07f), r);
  r = fma2(fq, splat2(-5.39030253e-15f), r);
  const f32x2_t r2 = mul2(r, r);
  f32x2_t sp = fma2(splat2(-1.9515295891e-4f), r2, splat2(8.3321608736e-3f));
  sp = fma2(sp, r2, splat2(-1.6666654611e-1f));
  const f32x2_t sr = fma2(mul2(sp, r2), r, r);
  f32x2_t cp = fma2(splat2(2.443315711809948e-5f), r2, splat2(-1.388731625493765e-3f));
  cp = fma2(cp, r2, splat2(4.166664568298827e-2f));
  const f32x2_t cr = fma2(mul2(cp, r2), r2, fma2(splat2(-0.5f), r2, splat2(1.0f)));
  float m0, m1, sr0, sr1, cr0, cr1, s0, s1, c0, c1;
  unpack2(m, m0, m1);
  unpack2(sr, sr0, sr1);
  unpack2(cr, cr0, cr1);
  sincos_quadrant(__float_as_int(m0), sr0, cr0, s0, c0);
  sincos_quadrant(__float_as_int(m1), sr1, cr1, s1, c1);
  s = pack2(s0, s1);
  c = pack2(c0, c1);
}

__device__ __forceinline__ float sin_bounded(float x) {
  float s, c;
  sincos_bounded(x, s, c);
  return s;
}

// atan2(y, x) from r = atan(min(|x|, |y|) / max(|x|, |y|)) (ax = |x|, ay = |y|): the quadrant fix-ups.
__device__ __forceinline__ float atan2_quadrant(float r, float ax, float ay, float x, float y) {
  if (ay > ax) r = 1.57079637f - r;
  if (x < 0.0f) r = 3.14159274f - r;
  return copysignf(r, y);
}

// atan2(y, x) for finite inputs: atan(min/max) by a degree-17 odd minimax polynomial
// (max abs error 7e-8 on [0, 1]) and quadrant fix-ups; atan2(+-0, +-0) = +-0 like NumPy/XLA
// for (0, +0).
// UNIT = true: the caller guarantees max(|x|, |y|) is a normal float (a [cos, sin] pair out of sincos_bounded has
// max >= 0.707): min * MUFU.RCP(max) without the zero test and the denormal scaling __fdividef carries -- the
// same bits as the guarded form for every such input, eight instructions shorter.
template <bool UNIT = false>
__device__ __forceinline__ float atan2_bounded(float y, float x) {
  const float ax = fabsf(x), ay = fabsf(y);
  const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
  float t;
  if (UNIT) {
    float rcp;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rcp) : "f"(mx));
    t = __fmul_rn(rcp, mn);
  } else {
    t = (mx > 0.0f) ? __fdividef(mn, mx) : 0.0f;
  }
  const float u = t * t;
  float q = 2.974586547e-03f;
  q = fmaf(q, u, -1.658116880e-02f);
  q = fmaf(q, u, 4.355351503e-02f);
  q = fmaf(q, u, -7.580576113e-02f);
  q = fmaf(q, u, 1.067893936e-01f);
  q = fmaf(q, u, -1.421420891e-01f);
  q = fmaf(q, u, 1.999413718e-01f);
  q = fmaf(q, u, -3.333316696e-01f);
  return atan2_quadrant(fmaf(t * u, q, t), ax, ay, x, y);
}

// atan2_bounded<true> of both elements of a pair (y, x): the same operations packed, min / max, MUFU.RCP and the
// quadrant fix-up per element.
__device__ __forceinline__ f32x2_t atan2_bounded_unit2(f32x2_t y, f32x2_t x) {
  float y0, y1, x0, x1;
  unpack2(y, y0, y1);
  unpack2(x, x0, x1);
  const float ax0 = fabsf(x0), ay0 = fabsf(y0), ax1 = fabsf(x1), ay1 = fabsf(y1);
  float rcp0, rcp1;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rcp0) : "f"(fmaxf(ax0, ay0)));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rcp1) : "f"(fmaxf(ax1, ay1)));
  const f32x2_t t = mul2(pack2(rcp0, rcp1), pack2(fminf(ax0, ay0), fminf(ax1, ay1)));
  const f32x2_t u = mul2(t, t);
  f32x2_t q = fma2(splat2(2.974586547e-03f), u, splat2(-1.658116880e-02f));
  q = fma2(q, u, splat2(4.355351503e-02f));
  q = fma2(q, u, splat2(-7.580576113e-02f));
  q = fma2(q, u, splat2(1.067893936e-01f));
  q = fma2(q, u, splat2(-1.421420891e-01f));
  q = fma2(q, u, splat2(1.999413718e-01f));
  q = fma2(q, u, splat2(-3.333316696e-01f));
  float r0, r1;
  unpack2(fma2(mul2(t, u), q, t), r0, r1);
  return pack2(atan2_quadrant(r0, ax0, ay0, x0, y0), atan2_quadrant(r1, ax1, ay1, x1, y1));
}

}  // namespace mbpo
