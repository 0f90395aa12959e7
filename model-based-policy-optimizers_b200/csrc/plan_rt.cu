// The fused plan and the one-launch closed loop for ANY horizon in [2, MBPO_MAX_HORIZON]: iCemTO(horizon=...) is a
// free int in the reference (icem_optimizer.py:94-96).  Horizons with an unrolled instance go through plan_inst.cu;
// every other one lands here (same device functions with rolled sampling loops: same bits as the staged plan).
#include "plan_dispatch.h"

namespace mbpo {

namespace {
template <int PRNG, int MATH>
int launch_rt(const PlanArgs& a, const MpcArgs* mpc, cudaStream_t st) {
  TwiddleTable tw;
  fill_twiddles(a.H, tw);
  const size_t smem = PlanSmem<0>::bytes(a.N, a.Np, a.K, a.H);
  if (smem > 227 * 1024) return fail(MBPO_EUNSUPPORTED, "fused plan (any horizon): %zu B of shared memory", smem);
  const int sms = device_sm_count();
  cudaError_t e;
  if (mpc == nullptr) {
    auto kernel = icem_plan_pendulum_rt_kernel<PRNG, MATH>;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return fail(MBPO_ECUDA, "cudaFuncSetAttribute(smem=%zu): %s", smem, cudaGetErrorString(e));
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, PLAN_THREADS, smem) != cudaSuccess || per_sm < 1)
      per_sm = 1;
    const long long resident = static_cast<long long>(per_sm) * sms;
    PlanArgs b = a;
    b.zero_value_precomputed = 1;   // best_value_out doubles as the hand-over buffer
    zero_row_value_kernel<MATH><<<(a.B + 127) / 128, 128, 0, st>>>(a.sys, a.H, a.P, a.summarize, a.x0, a.B,
                                                                  a.best_value_out);
    const int rc = check_launch("zero_row_value_kernel");
    if (rc != MBPO_OK) return rc;
    kernel<<<static_cast<unsigned>(a.B < resident ? a.B : resident), PLAN_THREADS, smem, st>>>(b, tw);
    return check_launch("icem_plan_pendulum_rt_kernel");
  }
  auto kernel = icem_mpc_pendulum_rt_kernel<PRNG, MATH>;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  if (e != cudaSuccess) return fail(MBPO_ECUDA, "cudaFuncSetAttribute(smem=%zu): %s", smem, cudaGetErrorString(e));
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, PLAN_THREADS, smem) != cudaSuccess || per_sm < 1)
    per_sm = 1;
  const long long resident = static_cast<long long>(per_sm) * sms;
  kernel<<<static_cast<unsigned>(a.B < resident ? a.B : resident), PLAN_THREADS, smem, st>>>(a, *mpc, tw);
  return check_launch("icem_mpc_pendulum_rt_kernel");
}
}  // namespace

int plan_entry_rt(int prng_mode, int math_mode, const PlanArgs& a, const MpcArgs* mpc, cudaStream_t st) {
  return with_prng_math(prng_mode, math_mode, [&](auto P, auto M) { return launch_rt<P, M>(a, mpc, st); });
}

}  // namespace mbpo
