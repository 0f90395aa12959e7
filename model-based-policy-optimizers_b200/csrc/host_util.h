// Host-side helpers shared by the translation units of libmbpo_b200.so.
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <type_traits>

#include "../../include/mbpo_b200.h"

namespace mbpo {

extern thread_local char g_err[512];  // text behind mbpo_last_error()

inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

inline int check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(MBPO_ECUDA, "%s: %s", what, cudaGetErrorString(e));
  return MBPO_OK;
}

#define MBPO_REQUIRE(cond, ...)                         \
  do {                                                  \
    if (!(cond)) return ::mbpo::fail(MBPO_EINVAL, __VA_ARGS__); \
  } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

inline int copy_async(void* dst, const void* src, size_t bytes, cudaStream_t st, const char* what) {
  if (bytes == 0 || dst == src) return MBPO_OK;
  const cudaError_t ce = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, st);
  return ce == cudaSuccess ? MBPO_OK : fail(MBPO_ECUDA, "%s copy: %s", what, cudaGetErrorString(ce));
}

// Runtime mode -> template argument: f(std::integral_constant<int, MODE>) for a prng_mode (MBPO_PRNG_*) or
// math_mode (MBPO_MATH_*) the caller has already checked to be 0 or 1, so that f can name kernel<MODE>.  Each
// call site instantiates only the modes it dispatches on.
template <class F>
int with_prng(int prng_mode, F&& f) {
  if (prng_mode == 0) return f(std::integral_constant<int, 0>{});
  return f(std::integral_constant<int, 1>{});
}
template <class F>
int with_math(int math_mode, F&& f) {
  if (math_mode == 0) return f(std::integral_constant<int, 0>{});
  return f(std::integral_constant<int, 1>{});
}
template <class F>
int with_prng_math(int prng_mode, int math_mode, F&& f) {
  return with_prng(prng_mode, [&](auto p) { return with_math(math_mode, [&](auto m) { return f(p, m); }); });
}

inline int device_sm_count() {
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms > 0 ? sms : 148;
}

// Horizons with a compiled (fully unrolled, immediate-twiddle) sampling kernel.  One
// translation unit per horizon (plan_inst.cu compiled with -DMBPO_INST_H=<h>).
#define MBPO_FOR_EACH_H(X) X(5) X(8) X(15) X(20) X(30) X(50)
#define MBPO_H_LIST_STR "5, 8, 15, 20, 30, 50"

}  // namespace mbpo
