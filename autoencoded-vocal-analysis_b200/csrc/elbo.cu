// BatchNorm bookkeeping kernels and the fused ELBO kernels (latent sample + prior +
// entropy with analytic gradients; reconstruction term + its gradient).
//
// Reference: ava/models/vae.py:311-323 and torch.distributions.LowRankMultivariateNormal
// (rank-1 case: capacitance 1 + sum u^2/d is a scalar, so the Cholesky is a sqrt).
#include "common.cuh"

namespace ava {

// ------------------------------------------------------------------ channel statistics
__global__ void __launch_bounds__(256)
channel_stats_kernel(const float* __restrict__ x, int B, int C, int HW, double* stats) {
  __shared__ float s1[8], s2[8];
  const int c = blockIdx.y;
  const int hw4 = HW >> 2;  // HW is a multiple of 4 (256 or 16384)
  const long long total4 = (long long)B * hw4;
  // four independent 16-byte loads in flight per thread (one dependent load per trip left the kernel at
  // 0.32 of HBM); HW/4 is a power of two for every caller (64 or 4096), so the (sample, offset) split is
  // a shift, with a 64-bit division only as the general fallback
  const bool pow2 = (hw4 & (hw4 - 1)) == 0;
  const int sh = 31 - __clz(hw4);
  auto addr = [&](long long i) {
    long long n;
    int p;
    if (pow2) {
      n = i >> sh;
      p = (int)(i & (hw4 - 1));
    } else {
      n = i / hw4;
      p = (int)(i - n * hw4);
    }
    return reinterpret_cast<const float4*>(x + ((size_t)n * C + c) * HW) + p;
  };
  auto acc4 = [](const float4 v, float& a, float& b) {
    a += (v.x + v.y) + (v.z + v.w);
    b = fmaf(v.x, v.x, b);
    b = fmaf(v.y, v.y, b);
    b = fmaf(v.z, v.z, b);
    b = fmaf(v.w, v.w, b);
  };
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, b0 = 0.f, b1 = 0.f, b2 = 0.f, b3 = 0.f;
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < total4; i += 4 * stride) {
    const float4 v0 = __ldg(addr(i)), v1 = __ldg(addr(i + stride));
    const float4 v2 = __ldg(addr(i + 2 * stride)), v3 = __ldg(addr(i + 3 * stride));
    acc4(v0, a0, b0);
    acc4(v1, a1, b1);
    acc4(v2, a2, b2);
    acc4(v3, a3, b3);
  }
  for (; i < total4; i += stride) acc4(__ldg(addr(i)), a0, b0);
  float a = (a0 + a1) + (a2 + a3), b = (b0 + b1) + (b2 + b3);
  a = warp_sum(a);
  b = warp_sum(b);
  if ((threadIdx.x & 31) == 0) {
    s1[threadIdx.x >> 5] = a;
    s2[threadIdx.x >> 5] = b;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ta = 0, tb = 0;
    for (int w = 0; w < 8; ++w) {
      ta += s1[w];
      tb += s2[w];
    }
    atomicAdd(&stats[c], ta);
    atomicAdd(&stats[32 + c], tb);
  }
}

struct BnTable {
  int channels[AVA_NUM_BN_LAYERS];
  long long counts[AVA_NUM_BN_LAYERS];
  int off_a[AVA_NUM_BN_LAYERS];
  int off_b[AVA_NUM_BN_LAYERS];
};

__global__ void bn_update_running_kernel(const double* stats, BnTable T, float* running, long long* nbt,
                                         float momentum) {
  const int l = blockIdx.x, c = threadIdx.x;
  if (T.counts[l] == 0) return;  // layer not run this pass (e.g. encoder-only get_latent)
  if (c == 0) nbt[l] += 1;
  if (c >= T.channels[l]) return;
  bn_running_update(stats + (size_t)l * kStatsStride, c, (double)T.counts[l], running + T.off_a[l],
                    running + T.off_b[l], momentum);
}

// eval-mode BatchNorm (running != NULL): layer l's running variance at running[rv_off[l]]
struct BnRunVar {
  int rv_off[AVA_NUM_BN_LAYERS];
};

__global__ void bn_param_grads_kernel(const double* stats, const double* dstats, BnTable T, float* grads,
                                      const float* running, BnRunVar R) {
  const int l = blockIdx.x, c = threadIdx.x;
  if (c >= T.channels[l] || T.counts[l] == 0) return;
  const double* ds = dstats + (size_t)l * kStatsStride;
  double var;
  if (running == nullptr) {
    const double n = (double)T.counts[l];
    const double* st = stats + (size_t)l * kStatsStride;
    double mean = st[c] / n;
    var = st[32 + c] / n - mean * mean;
    if (var < 0) var = 0;
  } else {
    var = (double)running[R.rv_off[l] + c];
  }
  double invstd = rsqrt(var + (double)kBnEps);
  grads[T.off_a[l] + c] = (float)(invstd * ds[32 + c]);  // dgamma
  grads[T.off_b[l] + c] = (float)ds[c];                  // dbeta
}

// The nine per-channel border sums of a dz tensor (mode 0 of ava_b200_dz_border_sums: total, first /
// last row, first / last column, the four corners), accumulated by the kernel that WRITES the dz
// so that no separate pass reads it again.  fp32 per thread (a few hundred values), fp64 from
// the warp reduction on.
struct BorderAcc {
  float a[9];
  __device__ __forceinline__ void clear() {
#pragma unroll
    for (int i = 0; i < 9; ++i) a[i] = 0.f;
  }
  // v = 4 consecutive values of row y starting at column x0 of an H x W plane
  __device__ __forceinline__ void add(const float4& v, int y, int x0, int H, int W) {
    const float s = (v.x + v.y) + (v.z + v.w);
    a[0] += s;
    const bool fr = (y == 0), lr = (y == H - 1);
    if (fr) a[1] += s;
    if (lr) a[2] += s;
    if (x0 == 0) {
      a[3] += v.x;
      if (fr) a[5] += v.x;
      if (lr) a[7] += v.x;
    }
    if (x0 + 4 == W) {
      a[4] += v.w;
      if (fr) a[6] += v.w;
      if (lr) a[8] += v.w;
    }
  }
  // block-wide (256 threads) reduction, one fp64 atomic per slot and CTA into tsums[slot*32 + c]
  __device__ __forceinline__ void flush(double (*s_red)[9], int c, double* tsums) {
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      const double s = warp_sum((double)a[i]);
      if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5][i] = s;
    }
    __syncthreads();
    if (threadIdx.x < 9) {
      double s = 0.0;
      for (int w = 0; w < 8; ++w) s += s_red[w][threadIdx.x];
      atomicAdd(&tsums[threadIdx.x * 32 + c], s);
    }
  }
};

// grid (chunks, C): a CTA stays within one channel (its coefficients are scalars, and the optional
// border sums of the written dz are per channel)
__global__ void __launch_bounds__(256)
bn_relu_bwd_apply_kernel(const float* g, const float* __restrict__ a, const float* gamma,
                         const double* stats, const double* dstats, int B, int C, int HW, int W, double count,
                         int relu, float* out, double* tsums) {
  // HW is a multiple of 4, so a float4 never straddles a channel
  __shared__ double s_red[8][9];
  const int c = blockIdx.y;
  const DzCoef k = dz_coef(gamma, stats, dstats, c, count);
  const int hw4 = HW >> 2, w4 = W >> 2, H = HW / W;
  const long long total4 = (long long)B * hw4;
  BorderAcc acc;
  acc.clear();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total4;
       i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / hw4;
    const int q = (int)(i - n * hw4);
    const size_t idx = ((size_t)n * C + c) * hw4 + q;
    float4 gv = reinterpret_cast<const float4*>(g)[idx];
    float4 av = __ldg(reinterpret_cast<const float4*>(a) + idx);
    float4 o;
    o.x = (relu && !(av.x > 0.f)) ? 0.f : dz_apply(k, gv.x, av.x);
    o.y = (relu && !(av.y > 0.f)) ? 0.f : dz_apply(k, gv.y, av.y);
    o.z = (relu && !(av.z > 0.f)) ? 0.f : dz_apply(k, gv.z, av.z);
    o.w = (relu && !(av.w > 0.f)) ? 0.f : dz_apply(k, gv.w, av.w);
    reinterpret_cast<float4*>(out)[idx] = o;
    if (tsums) {
      const int y = q / w4;
      acc.add(o, y, (q - y * w4) * 4, H, W);
    }
  }
  if (tsums) acc.flush(s_red, c, tsums);
}

// ----------------------------------------------------------------------------- latent
// One warp per sample.  heads = (mu | u | logd), row stride 3Z.
__global__ void __launch_bounds__(256)
latent_fwd_kernel(const float* __restrict__ heads, const float* __restrict__ eps_w,
                  const float* __restrict__ eps_d, int B, int Z, float* __restrict__ z, float* __restrict__ d_out,
                  double* acc) {
  __shared__ double s_z2[8], s_h[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * 8 + warp;
  double z2 = 0.0, hb = 0.0;
  if (b < B) {
    const float* row = heads + (size_t)b * 3 * Z;
    const float ew = eps_w[b];
    float sz2 = 0.f, s = 0.f, slogd = 0.f;
    for (int i = lane; i < Z; i += 32) {
      float mu = row[i], u = row[Z + i], ld = row[2 * Z + i];
      float d = expf(ld);
      float zz = mu + u * ew + sqrtf(d) * eps_d[(size_t)b * Z + i];
      z[(size_t)b * Z + i] = zz;
      if (d_out) d_out[(size_t)b * Z + i] = d;
      sz2 = fmaf(zz, zz, sz2);
      s += u * u / d;
      slogd += ld;
    }
    sz2 = warp_sum(sz2);
    s = warp_sum(s);
    slogd = warp_sum(slogd);
    z2 = sz2;
    // H = 1/2 (Z (1 + ln 2pi) + ln(1 + s) + sum ln d)
    hb = 0.5 * ((double)Z * (1.0 + 1.8378770664093453) + (double)log1pf(s) + (double)slogd);
  }
  if (lane == 0) {
    s_z2[warp] = z2;
    s_h[warp] = hb;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, h = 0;
    for (int w = 0; w < 8; ++w) {
      a += s_z2[w];
      h += s_h[w];
    }
    atomicAdd(&acc[0], a);
    atomicAdd(&acc[2], h);
  }
}

__global__ void __launch_bounds__(256)
latent_bwd_kernel(const float* __restrict__ heads, const float* __restrict__ eps_w,
                  const float* __restrict__ eps_d, const float* __restrict__ z, const float* __restrict__ gz,
                  int B, int Z, float* __restrict__ g_heads) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * 8 + warp;
  if (b >= B) return;
  const float* row = heads + (size_t)b * 3 * Z;
  float* grow = g_heads + (size_t)b * 3 * Z;
  const float ew = eps_w[b];
  float s = 0.f;
  for (int i = lane; i < Z; i += 32) {
    float u = row[Z + i];
    s += u * u * expf(-row[2 * Z + i]);
  }
  s = warp_sum(s);
  const float inv1s = 1.f / (1.f + s);
  for (int i = lane; i < Z; i += 32) {
    float u = row[Z + i], ld = row[2 * Z + i];
    float d = expf(ld);
    float g = gz[(size_t)b * Z + i] + z[(size_t)b * Z + i];  // decoder path + prior term
    float uod = u / d;
    grow[i] = g;                                   // dL/dmu
    grow[Z + i] = g * ew - uod * inv1s;            // dL/du
    // dL/dlogd = d * dL/dd = g*eps_d*sqrt(d)/2 - 1/2 (1 - u^2/(d (1+s)))
    grow[2 * Z + i] = 0.5f * g * eps_d[(size_t)b * Z + i] * sqrtf(d) - 0.5f * (1.f - u * uod * inv1s);
  }
}

// encode()'s backward seed: g_heads = (dmu | du | dd * d), d = exp(logd) as the forward returned it;
// a NULL seed is zero
__global__ void __launch_bounds__(256)
latent_heads_grad_kernel(const float* __restrict__ dmu, const float* __restrict__ du, const float* __restrict__ dd,
                         const float* __restrict__ d, long long n, int Z, float* __restrict__ g_heads) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / Z;
    float* grow = g_heads + b * 3 * Z + (i - b * Z);
    grow[0] = dmu ? dmu[i] : 0.f;
    grow[Z] = du ? du[i] : 0.f;
    grow[2 * Z] = dd ? dd[i] * d[i] : 0.f;
  }
}

// forward()'s input gradient: the encoder's part plus the direct reconstruction term,
// dx = dx_enc - prec * (x_rec - x)
__global__ void __launch_bounds__(256)
recon_input_grad_kernel(const float* dx_enc, const float* __restrict__ x, const float* __restrict__ xr,
                        long long n4, float prec, float* dx) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
       i += (long long)gridDim.x * blockDim.x) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(x) + i);
    const float4 r = __ldg(reinterpret_cast<const float4*>(xr) + i);
    float4 e = dx_enc ? reinterpret_cast<const float4*>(dx_enc)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    e.x -= prec * (r.x - a.x);
    e.y -= prec * (r.y - a.y);
    e.z -= prec * (r.z - a.z);
    e.w -= prec * (r.w - a.w);
    reinterpret_cast<float4*>(dx)[i] = e;
  }
}

// ------------------------------------------------------------------------------ recon
// tsums (optional): the border sums of the written gradient g viewed as [*, 1, H, W] planes
__global__ void __launch_bounds__(256)
recon_kernel(const float* __restrict__ x, const float* __restrict__ xr, long long n4, float prec,
             float* __restrict__ g, double* acc, double* tsums, int H, int W) {
  __shared__ float s_p[8];
  __shared__ double s_red[8][9];
  float sse = 0.f;
  const int w4 = W >> 2, hw4 = (H * W) >> 2;
  BorderAcc bacc;
  bacc.clear();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
       i += (long long)gridDim.x * blockDim.x) {
    float4 a = __ldg(reinterpret_cast<const float4*>(x) + i);
    float4 r = __ldg(reinterpret_cast<const float4*>(xr) + i);
    float4 d = make_float4(r.x - a.x, r.y - a.y, r.z - a.z, r.w - a.w);
    sse = fmaf(d.x, d.x, sse);
    sse = fmaf(d.y, d.y, sse);
    sse = fmaf(d.z, d.z, sse);
    sse = fmaf(d.w, d.w, sse);
    if (g) {
      const float4 gv = make_float4(prec * d.x, prec * d.y, prec * d.z, prec * d.w);
      reinterpret_cast<float4*>(g)[i] = gv;
      if (tsums) {
        const int q = (int)(i % hw4);
        const int y = q / w4;
        bacc.add(gv, y, (q - y * w4) * 4, H, W);
      }
    }
  }
  sse = warp_sum(sse);
  if ((threadIdx.x & 31) == 0) s_p[threadIdx.x >> 5] = sse;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int w = 0; w < 8; ++w) t += s_p[w];
    atomicAdd(&acc[1], t);
  }
  if (g && tsums) bacc.flush(s_red, 0, tsums);
}

__global__ void elbo_finalize_kernel(const double* acc, int Z, int xdim, float prec, float* loss,
                                     double* loss_sum) {
  const double ln2pi = 1.8378770664093453;
  // -elbo, ava/models/vae.py:316-323 (constants once per batch)
  double l = 0.5 * (acc[0] + Z * ln2pi) + 0.5 * xdim * (ln2pi - log((double)prec)) + 0.5 * (double)prec * acc[1] -
             acc[2];
  loss[0] = (float)l;
  if (loss_sum) loss_sum[0] += l;
}

static BnTable make_table(const int* channels, const long long* counts, const int* off_a, const int* off_b) {
  BnTable T;
  for (int l = 0; l < AVA_NUM_BN_LAYERS; ++l) {
    T.channels[l] = channels[l];
    T.counts[l] = counts[l];
    T.off_a[l] = off_a[l];
    T.off_b[l] = off_b[l];
  }
  return T;
}

}  // namespace ava

using namespace ava;

extern "C" int ava_b200_channel_stats(const float* x, int B, int C, int HW, double* stats, void* stream) {
  AVA_REQUIRE(C >= 1 && C <= 32 && HW % 4 == 0, "channel_stats: C=%d HW=%d unsupported", C, HW);
  if (B <= 0) return 0;
  long long total4 = (long long)B * (HW / 4);
  int chunks = (int)((total4 + 256 * 8 - 1) / (256 * 8));
  int maxc = (4 * kNumSMs + C - 1) / C;
  if (chunks > maxc) chunks = maxc;
  if (chunks < 1) chunks = 1;
  channel_stats_kernel<<<dim3(chunks, C), 256, 0, (cudaStream_t)stream>>>(x, B, C, HW, stats);
  return check_launch("channel_stats");
}

extern "C" int ava_b200_bn_update_running(const double* stats, const int* h_channels, const long long* h_counts,
                                          float* running, const int* h_rm_off, const int* h_rv_off,
                                          long long* nbt, float momentum, void* stream) {
  BnTable T = make_table(h_channels, h_counts, h_rm_off, h_rv_off);
  bn_update_running_kernel<<<AVA_NUM_BN_LAYERS, 32, 0, (cudaStream_t)stream>>>(stats, T, running, nbt, momentum);
  return check_launch("bn_update_running");
}

extern "C" int ava_b200_bn_param_grads_ex(const double* stats, const double* dstats, const int* h_channels,
                                          const long long* h_counts, float* grads, const int* h_dgamma_off,
                                          const int* h_dbeta_off, const float* running, const int* h_rv_off,
                                          int train, void* stream) {
  AVA_REQUIRE(train || (running != nullptr && h_rv_off != nullptr),
              "bn_param_grads: eval mode needs the running buffers and their offsets");
  BnTable T = make_table(h_channels, h_counts, h_dgamma_off, h_dbeta_off);
  BnRunVar R = {};
  if (!train)
    for (int l = 0; l < AVA_NUM_BN_LAYERS; ++l) R.rv_off[l] = h_rv_off[l];
  bn_param_grads_kernel<<<AVA_NUM_BN_LAYERS, 32, 0, (cudaStream_t)stream>>>(stats, dstats, T, grads,
                                                                          train ? nullptr : running, R);
  return check_launch("bn_param_grads");
}

extern "C" int ava_b200_bn_param_grads(const double* stats, const double* dstats, const int* h_channels,
                                       const long long* h_counts, float* grads, const int* h_dgamma_off,
                                       const int* h_dbeta_off, void* stream) {
  return ava_b200_bn_param_grads_ex(stats, dstats, h_channels, h_counts, grads, h_dgamma_off, h_dbeta_off, nullptr,
                                    nullptr, 1, stream);
}

extern "C" int ava_b200_bn_relu_bwd_apply(const float* g, const float* a, const float* gamma, const double* stats,
                                          const double* dstats, int B, int C, int HW, int relu, float* out,
                                          double* tsums, int W, void* stream) {
  AVA_REQUIRE(HW % 4 == 0, "bn_relu_bwd_apply: HW=%d must be a multiple of 4", HW);
  AVA_REQUIRE(C >= 1 && C <= 32, "bn_relu_bwd_apply: C=%d", C);
  AVA_REQUIRE(tsums == nullptr || (W >= 4 && W % 4 == 0 && HW % W == 0 && HW / W >= 2),
              "bn_relu_bwd_apply: border sums need a row width W (multiple of 4) dividing HW, got %d", W);
  if (B <= 0) return 0;
  if (tsums == nullptr) W = 4;
  long long total4 = (long long)B * HW / 4;
  long long want = (total4 + 255) / 256;
  int gx = (int)(want < 1 ? 1 : want);
  const int cap = (8 * kNumSMs + C - 1) / C;
  if (gx > cap) gx = cap;
  bn_relu_bwd_apply_kernel<<<dim3(gx, C), 256, 0, (cudaStream_t)stream>>>(g, a, gamma, stats, dstats, B, C, HW, W,
                                                                         (double)B * HW, relu, out, tsums);
  return check_launch("bn_relu_bwd_apply");
}

extern "C" int ava_b200_latent_fwd(const float* heads, const float* eps_w, const float* eps_d, int B, int Z,
                                   float* z, float* d_out, double* acc, void* stream) {
  if (B <= 0) return 0;
  latent_fwd_kernel<<<(B + 7) / 8, 256, 0, (cudaStream_t)stream>>>(heads, eps_w, eps_d, B, Z, z, d_out, acc);
  return check_launch("latent_fwd");
}

extern "C" int ava_b200_latent_bwd(const float* heads, const float* eps_w, const float* eps_d, const float* z,
                                   const float* gz, int B, int Z, float* g_heads, void* stream) {
  if (B <= 0) return 0;
  latent_bwd_kernel<<<(B + 7) / 8, 256, 0, (cudaStream_t)stream>>>(heads, eps_w, eps_d, z, gz, B, Z, g_heads);
  return check_launch("latent_bwd");
}

extern "C" int ava_b200_latent_heads_grad(const float* dmu, const float* du, const float* dd, const float* d, int B,
                                          int Z, float* g_heads, void* stream) {
  AVA_REQUIRE(Z >= 1 && B >= 0, "latent_heads_grad: B=%d Z=%d", B, Z);
  AVA_REQUIRE(dd == nullptr || d != nullptr, "latent_heads_grad: a seed on d needs d");
  if (B == 0) return 0;
  const long long n = (long long)B * Z;
  long long grid = (n + 255) / 256;
  if (grid > 8 * kNumSMs) grid = 8 * kNumSMs;
  latent_heads_grad_kernel<<<(int)grid, 256, 0, (cudaStream_t)stream>>>(dmu, du, dd, d, n, Z, g_heads);
  return check_launch("latent_heads_grad");
}

extern "C" int ava_b200_recon_input_grad(const float* dx_enc, const float* x, const float* x_rec, long long n,
                                         float precision, float* dx, void* stream) {
  AVA_REQUIRE(n % 4 == 0 && n >= 0, "recon_input_grad: n=%lld must be a non-negative multiple of 4", n);
  if (n == 0) return 0;
  const long long n4 = n / 4;
  long long grid = (n4 + 255) / 256;
  if (grid > 8 * kNumSMs) grid = 8 * kNumSMs;
  recon_input_grad_kernel<<<(int)grid, 256, 0, (cudaStream_t)stream>>>(dx_enc, x, x_rec, n4, precision, dx);
  return check_launch("recon_input_grad");
}

extern "C" int ava_b200_recon(const float* x, const float* x_rec, long long n, float precision, float* g,
                              double* acc, double* tsums, int H, int W, void* stream) {
  AVA_REQUIRE(n % 4 == 0, "recon: n must be a multiple of 4");
  AVA_REQUIRE(tsums == nullptr || (H >= 2 && W >= 4 && W % 4 == 0 && n % ((long long)H * W) == 0),
              "recon: border sums need the plane shape (H=%d, W=%d) dividing n", H, W);
  if (n <= 0) return 0;
  if (tsums == nullptr) H = W = 4;
  long long n4 = n / 4;
  int grid = (int)((n4 + 255) / 256);
  if (grid > 8 * kNumSMs) grid = 8 * kNumSMs;
  recon_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, x_rec, n4, precision, g, acc, tsums, H, W);
  return check_launch("recon");
}

extern "C" int ava_b200_elbo_finalize(const double* acc, int Z, int xdim, float precision, float* loss,
                                      double* loss_sum, void* stream) {
  elbo_finalize_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(acc, Z, xdim, precision, loss, loss_sum);
  return check_launch("elbo_finalize");
}
