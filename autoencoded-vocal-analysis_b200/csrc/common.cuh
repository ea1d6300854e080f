// Shared helpers for the ava_b200 kernels (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/ava_b200.h"

namespace ava {

constexpr float kBnEps = 1e-5f;
constexpr int kStatsStride = AVA_STATS_STRIDE;  // doubles per BN layer
constexpr int kNumSMs = 148;

void set_error(const char* fmt, ...);
// cuTensorMapEncodeTiled, fetched through the runtime (no libcuda link dependency)
typedef CUresult (*TensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                      const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
TensorMapEncodeFn get_tensor_map_encode_fn();
void count_launch(int n = 1);

inline int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return 1;
  }
  count_launch();
  return 0;
}

#define AVA_REQUIRE(cond, ...)   \
  do {                           \
    if (!(cond)) {               \
      ava::set_error(__VA_ARGS__); \
      return 1;                  \
    }                            \
  } while (0)

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// The Adam update, shared by adam_kernel (adam.cu) and the fused data-parallel kernel (dp.cu) with
// every rounding spelled out, so that the two produce the same bits from the same summed gradient
// whatever the compiler contracts around them: a 1-ulp difference in the first steps is amplified
// by ReLU kinks and Adam's scale invariance into lr-sized differences of ~1 % of the parameters
// within a few steps (seen when the two kernels were written independently).
struct AdamCoef {
  float b1, b2, omb1, omb2, eps, step_size, inv_sqrt_bc2;
};
// Scalars exactly as torch.optim.Adam forms them (Python doubles, rounded to fp32 once); t = the
// step number of THIS update (torch increments `step` before using it)
__device__ __forceinline__ AdamCoef adam_coef(double lr_d, double b1_d, double b2_d, double eps_d, double t) {
  const double bc1 = 1.0 - pow(b1_d, t);
  const double bc2 = 1.0 - pow(b2_d, t);
  AdamCoef k;
  k.step_size = (float)(lr_d / bc1);
  k.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
  k.b1 = (float)b1_d;
  k.b2 = (float)b2_d;
  k.eps = (float)eps_d;
  k.omb1 = (float)(1.0 - b1_d);
  k.omb2 = (float)(1.0 - b2_d);
  return k;
}
__device__ __forceinline__ void adam_update(const AdamCoef& k, float gg, float& p, float& m, float& v) {
  m = __fmaf_rn(k.b1, m, __fmul_rn(k.omb1, gg));
  v = __fmaf_rn(k.b2, v, __fmul_rn(__fmul_rn(k.omb2, gg), gg));
  const float denom = __fmaf_rn(__fsqrt_rn(v), k.inv_sqrt_bc2, k.eps);
  p = __fmaf_rn(-k.step_size, __fdiv_rn(m, denom), p);
}

// Cross-GPU flag handshake of the data-parallel kernels (dp.cu, bnsync.cu): flags hold monotonically
// increasing sequence numbers; a waiter gives up after kDpTimeoutNs and records it in *status.
constexpr unsigned long long kDpTimeoutNs = 20ull * 1000ull * 1000ull * 1000ull;

__device__ __forceinline__ unsigned long long dp_now_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void dp_signal(unsigned int* flag, unsigned int seq) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(seq) : "memory");
}
__device__ __forceinline__ void dp_wait(const unsigned int* flag, unsigned int seq, unsigned int* status) {
  const unsigned long long t0 = dp_now_ns();
  for (;;) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
    if ((int)(v - seq) >= 0) return;
    if (dp_now_ns() - t0 > kDpTimeoutNs) {
      atomicExch(status, 1u);
      return;
    }
    __nanosleep(64);
  }
}

// BatchNorm running-buffer update of channel c from the sums of a stats block over n values (torch's
// momentum form, unbiased variance): bn_update_running_kernel (elbo.cu) and the synchronised-BatchNorm
// exchange (bnsync.cu) share it so that both round alike.
__device__ __forceinline__ void bn_running_update(const double* st, int c, double n, float* rm, float* rv,
                                                  float momentum) {
  double mean = st[c] / n;
  double var = st[32 + c] / n - mean * mean;
  if (var < 0) var = 0;
  double unb = (n > 1) ? var * n / (n - 1) : var;
  rm[c] = (1.f - momentum) * rm[c] + momentum * (float)mean;
  rv[c] = (1.f - momentum) * rv[c] + momentum * (float)unb;
}

// BatchNorm coefficients for one channel from accumulated sums (train) or running
// buffers (eval):  bn(x) = x*scale + shift.
struct BnCoef {
  float mean, invstd, scale, shift;
};
__device__ __forceinline__ BnCoef bn_coef(const double* stats, int c, double count, const float* gamma,
                                          const float* beta, const float* rmean, const float* rvar, bool train) {
  double mean, var;
  if (train) {
    mean = stats[c] / count;
    var = stats[32 + c] / count - mean * mean;
    if (var < 0.0) var = 0.0;
  } else {
    mean = (double)rmean[c];
    var = (double)rvar[c];
  }
  double invstd = rsqrt(var + (double)kBnEps);
  BnCoef k;
  k.mean = (float)mean;
  k.invstd = (float)invstd;
  double g = gamma ? (double)gamma[c] : 1.0;
  double b = beta ? (double)beta[c] : 0.0;
  k.scale = (float)(g * invstd);
  k.shift = (float)(b - mean * g * invstd);
  return k;
}

// Backward of the BatchNorm that consumes y (train mode), SURVEY.md appendix A:
//   dx = gamma*invstd*(dy - dbeta/N - xhat*dgamma/N)
//      = p*(dy - c1) + q*(y - mean),   p = gamma*invstd, c1 = dbeta/N,
//                                      q = -gamma*invstd^3 * S/N, S = sum dy*(y-mean)
// with dstats[c] = sum dy (= dbeta) and dstats[32+c] = S (= dgamma/invstd).
// Evaluated in fp64: the two terms cancel heavily (BN backward projects out the mean and
// the xhat direction), and a coefficient rounded to fp32 would add a *coherent* error to
// every element of the channel, which bias / BN-affine gradients then sum up.
// Eval mode (rvar != NULL): the BatchNorm is the fixed affine map of the running buffers, so
// dx = gamma*invstd_r*dy: p = gamma/sqrt(rvar + eps), q = c1 = 0.
struct DzCoef {
  double p, q, mean, c1;
};
__device__ __forceinline__ DzCoef dz_coef(const float* gamma, const double* stats, const double* dstats, int c,
                                          double count, const float* rvar = nullptr) {
  DzCoef k;
  if (gamma == nullptr) {
    k.p = 1.0;
    k.q = 0.0;
    k.mean = 0.0;
    k.c1 = 0.0;
    return k;
  }
  double mean = 0.0, var, s = 0.0, c1 = 0.0;
  if (rvar != nullptr) {
    var = (double)rvar[c];
  } else {
    mean = stats[c] / count;
    var = stats[32 + c] / count - mean * mean;
    if (var < 0.0) var = 0.0;
    s = dstats[32 + c];
    c1 = dstats[c] / count;
  }
  double invstd = rsqrt(var + (double)kBnEps);
  double g = (double)gamma[c];
  k.p = g * invstd;
  k.q = -g * invstd * invstd * invstd * s / count;
  k.mean = mean;
  k.c1 = c1;
  return k;
}
__device__ __forceinline__ float dz_apply(const DzCoef& k, float g, float y) {
  return (float)(k.p * ((double)g - k.c1) + k.q * ((double)y - k.mean));
}

}  // namespace ava
