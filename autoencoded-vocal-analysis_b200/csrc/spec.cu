// Batched GPU `get_spec`: STFT -> log magnitude -> bilinear resampling onto the
// 128x128 (freq x time) grid -> normalise/clip.  One CTA per window, fp64 throughout, so parity
// with the reference's float64 scipy path is ~1e-12.  The kernel is bound by fp64 arithmetic and
// shared-memory latency (FFT butterflies, log / hypot), not by its HBM traffic (14 KB in, 64 KB
// out per finch window): see profiles/ for the measured rate against the HBM roofline.
//
// Reference: ava/preprocessing/utils.py:59-104 and scipy.signal.stft (_spectral_helper):
// zero boundary extension by nperseg/2, zero padding to a hop multiple, no detrend,
// window multiply, one-sided FFT, scale 1/sum(window).
//
#include "common.cuh"

namespace ava {

struct SpecParams {
  const void* audio;
  int is_f32;
  const long long* seg_start;
  const int* seg_len;
  int nperseg, hop, log2n, remove_dc;
  const double* window;
  double scale;
  const int* t_idx;
  const double* t_frac;
  int n_t;
  const int* f_idx;
  const double* f_frac;
  int n_f;
  int max_frames;
  double spec_min, inv_range;
  double fill;   // interp2d's fill value -1e12 after normalise + clip (0 unless spec_max < spec_min)
  float* out;
  double* out64;
};

// audio sample type: 0 int16, 1 float32, 2 float64 (the reference's stft runs in complex128 on
// int16 / float64 audio; everything here is fp64)
__device__ __forceinline__ double load_sample(const SpecParams& P, long long i) {
  if (P.is_f32 == 2) return reinterpret_cast<const double*>(P.audio)[i];
  if (P.is_f32 == 1) return (double)reinterpret_cast<const float*>(P.audio)[i];
  return (double)reinterpret_cast<const short*>(P.audio)[i];
}

// Kernel anatomy (one CTA of 256 threads per window):
//  * only the STFT frames some target time touches are computed ("needed" frames: two per target);
//  * the frames are real, so TWO of them share one complex FFT (frame a in the real part, frame b
//    in the imaginary part; X_a[k] = (Z[k] + conj Z[N-k]) / 2, X_b[k] = (Z[k] - conj Z[N-k]) / 2i),
//    and G such packed transforms run side by side in shared memory, so every radix-2 stage (one
//    __syncthreads) moves G*N/2 butterflies -- G per thread at nperseg 512 -- instead of one;
//  * the log-magnitude spectra of a whole run of needed frames stay in shared memory (CF slots);
//    the output pass then walks the [n_f, n_t] grid row-major, so a warp writes 128 consecutive
//    floats of one frequency row, and every output is written exactly once (no zero-fill pass).
//    Windows with more needed frames than slots are handled in overlapping runs of slots.
struct SpecSmem {
  int G, CF, NBP;   // packed transforms per batch, log-spectrum slots, slot pitch (doubles)
};

// LOG2N = log2(nperseg) is a template parameter: every index split in the hot loops is then a shift
// (the first version of this kernel spent 25 % of its instructions in IMAD / software division).
template <int LOG2N>
__global__ void __launch_bounds__(256) get_spec_kernel(const SpecParams P, const SpecSmem S) {
  extern __shared__ __align__(16) double sm[];
  constexpr int N = 1 << LOG2N, half = N / 2;
  double2* s_x = reinterpret_cast<double2*>(sm);                  // [G][N] packed FFT buffers
  double2* s_tw = s_x + (size_t)S.G * N;                          // [N] per-stage twiddle tables (N-1 used)
  double* s_log = reinterpret_cast<double*>(s_tw + N);            // [CF][NBP] log spectra
  double* s_red = s_log + (size_t)S.CF * S.NBP;                   // [8]
  int* s_list = reinterpret_cast<int*>(s_red + 8);                // [max_frames+1] needed frames, ascending
  int* s_slot = s_list + (P.max_frames + 1);                      // [max_frames+1] frame -> slot in the current run
  int* s_cnt = s_slot + (P.max_frames + 1);                       // [2]
  int* s_fi = s_cnt + 2;                                          // [n_f] frequency bracket index
  double* s_wy = reinterpret_cast<double*>(s_fi + ((P.n_f + 1) & ~1));   // [n_f] and weight

  const int tid = threadIdx.x;
  const int w = blockIdx.x;
  const int len = P.seg_len[w];
  const size_t out_base = (size_t)w * P.n_f * P.n_t;
  const int n_out = P.n_f * P.n_t;
  if (len <= 0) {
    // too-short segment (the reference returns zeros, ava/preprocessing/utils.py:69-71)
    for (int i = tid; i < n_out; i += 256) {
      if (P.out) P.out[out_base + i] = 0.f;
      if (P.out64) P.out64[out_base + i] = 0.0;
    }
    return;
  }
  const long long start = P.seg_start[w];
  const int L = len + 2 * half;
  const int nadd = ((P.hop - (L - N) % P.hop) % P.hop) % N;
  int K = (L + nadd - N) / P.hop + 1;
  if (K > P.max_frames) K = P.max_frames;

  // twiddles, one contiguous table per radix-2 stage (stage st, mh = 2^(st-1) butterflies per group:
  // entries [mh-1, 2mh-1) = exp(-2 pi i pos / (2 mh)) -- lanes then read consecutive entries instead
  // of a strided walk through one table, which put 16 of them on the same banks in the middle
  // stages); frame -> "needed" flags (in s_slot for now)
  for (int e = tid; e < N - 1; e += 256) {
    const int st = 31 - __clz(e + 1);                 // e + 1 in [mh, 2mh)
    const int mh = 1 << st;
    const int pos = e + 1 - mh;
    double sn, cs;
    sincospi(-(double)pos / (double)mh, &sn, &cs);    // -2 pi pos / (2 mh)
    s_tw[e] = make_double2(cs, sn);
  }
  for (int k = tid; k <= K; k += 256) s_slot[k] = 0;
  for (int f = tid; f < P.n_f; f += 256) {
    s_fi[f] = P.f_idx[f];
    s_wy[f] = P.f_frac[f];
  }
  __syncthreads();
  const int* tix = P.t_idx + (size_t)w * P.n_t;
  const double* tfr = P.t_frac + (size_t)w * P.n_t;
  for (int j = tid; j < P.n_t; j += 256) {
    const int i = tix[j];
    if (i >= 0 && i + 1 < K) {
      s_slot[i] = 1;
      s_slot[i + 1] = 1;
    }
  }
  // mean (np.mean: exact for int16 in fp64)
  double mean = 0.0;
  if (P.remove_dc) {
    double acc = 0.0;
    for (int i = tid; i < len; i += 256) acc += load_sample(P, start + i);
    acc = warp_sum(acc);
    if ((tid & 31) == 0) s_red[tid >> 5] = acc;
    __syncthreads();
    for (int i = 0; i < 8; ++i) mean += s_red[i];
    mean /= (double)len;
  }
  __syncthreads();
  if (tid == 0) {
    int n = 0;
    for (int k = 0; k < K; ++k)
      if (s_slot[k]) s_list[n++] = k;
    *s_cnt = n;
  }
  __syncthreads();
  const int nneed = *s_cnt;

  // runs of needed frames: [a, a + CF) of the list; consecutive runs overlap by one entry so that
  // both frames of every target's bracketing pair fall into one run
  bool first_run = true;
  for (int a = 0; first_run || a + 1 < nneed; a += S.CF - 1) {
    const int nrun = min(S.CF, nneed - a);
    __syncthreads();                                    // previous run's output pass is done with s_log / s_slot
    for (int k = tid; k <= K; k += 256) s_slot[k] = -1;
    __syncthreads();
    for (int j = tid; j < nrun; j += 256) s_slot[s_list[a + j]] = j;
    // ---- packed FFTs of this run, G at a time
    for (int p0 = 0; p0 < nrun; p0 += 2 * S.G) {
      const int npair = min(S.G, (nrun - p0 + 1) / 2);
      __syncthreads();
      // windowed frames, bit-reversed order: real part = entry p0+2g, imaginary = entry p0+2g+1
      for (int idx = tid; idx < npair * N; idx += 256) {
        // destination index r runs with the lanes (conflict-free stores); the source sample index
        // j = bitrev(r) scatters over the 2*N bytes of a frame, which sit in L1
        const int g = idx >> LOG2N, r = idx & (N - 1);
        const int j = (int)(__brev((unsigned)r) >> (32 - LOG2N));
        const int fa = s_list[a + p0 + 2 * g];
        const int eb = p0 + 2 * g + 1;
        const double wj = P.window[j];
        double va = 0.0, vb = 0.0;
        int ia = fa * P.hop + j - half;
        if (ia >= 0 && ia < len) va = (load_sample(P, start + ia) - mean) * wj;
        if (eb < nrun) {
          const int ib = s_list[a + eb] * P.hop + j - half;
          if (ib >= 0 && ib < len) vb = (load_sample(P, start + ib) - mean) * wj;
        }
        s_x[(size_t)g * N + r] = make_double2(va, vb);
      }
      __syncthreads();
      // radix-2 DIT over all npair transforms
#pragma unroll 1
      for (int st = 1; st <= LOG2N; ++st) {
        const int mh = 1 << (st - 1);
        const double2* twst = s_tw + (mh - 1);
        for (int b = tid; b < npair * half; b += 256) {
          const int g = b >> (LOG2N - 1), bb = b & (half - 1);
          const int grp = bb >> (st - 1), pos = bb & (mh - 1);
          const int i0 = (grp << st) + pos, i1 = i0 + mh;
          double2* x = s_x + (size_t)g * N;
          const double2 wv = twst[pos];
          const double2 u = x[i0], c = x[i1];
          const double tr = wv.x * c.x - wv.y * c.y, ti = wv.x * c.y + wv.y * c.x;
          x[i0] = make_double2(u.x + tr, u.y + ti);
          x[i1] = make_double2(u.x - tr, u.y - ti);
        }
        __syncthreads();
      }
      // unpack the two real spectra and take log magnitudes (ava/preprocessing/utils.py:79)
      auto logmag = [&](double re, double im) {
        // |X| * scale: audio-scale magnitudes cannot overflow or underflow the squares, so a plain
        // sqrt of the sum of squares stands in for hypot (<= 1 ulp apart)
        return log(sqrt(re * re + im * im) * P.scale + 1e-12);
      };
      for (int idx = tid; idx < npair * half; idx += 256) {
        const int g = idx >> (LOG2N - 1), k = idx & (half - 1);
        const double2* x = s_x + (size_t)g * N;
        const double2 z = x[k], zc = x[(N - k) & (N - 1)];
        // X_a = (Z[k] + conj Z[N-k]) / 2 ; X_b = (Z[k] - conj Z[N-k]) / (2i)
        const double ar = 0.5 * (z.x + zc.x), ai = 0.5 * (z.y - zc.y);
        const double br = 0.5 * (z.y + zc.y), bi = -0.5 * (z.x - zc.x);
        const int ea = p0 + 2 * g;
        s_log[(size_t)ea * S.NBP + k] = logmag(ar, ai);
        if (ea + 1 < nrun) s_log[(size_t)(ea + 1) * S.NBP + k] = logmag(br, bi);
      }
      if (tid < npair) {
        // Nyquist bin k = N/2: Z[N/2] pairs with itself -> X_a = Re Z, X_b = Im Z
        const double2 z = s_x[(size_t)tid * N + half];
        const int ea = p0 + 2 * tid;
        s_log[(size_t)ea * S.NBP + half] = logmag(z.x, 0.0);
        if (ea + 1 < nrun) s_log[(size_t)(ea + 1) * S.NBP + half] = logmag(z.y, 0.0);
      }
    }
    __syncthreads();
    // ---- output pass, row-major over [n_f, n_t]: the targets whose bracketing frames are the
    // entries (j, j+1) of this run with j + 1 < nrun; on the first run also everything that is
    // out of range (the fill value after normalise + clip)
    // (a thread keeps its target times: slot and weight are looked up once per run, then it walks the
    // frequency rows; a warp's lanes are consecutive t of one row -> 128-byte coalesced stores)
    for (int t0 = 0; t0 < P.n_t; t0 += 128) {
      const int t = t0 + (tid & 127);
      const bool t_in = t < P.n_t;
      const int ti = t_in ? tix[t] : -1;
      const bool t_valid = (ti >= 0) && (ti + 1 < K);
      const int j = t_valid ? s_slot[ti] : -1;
      const bool here = (j >= 0) && (j + 1 < nrun);   // (a run's last entry is the next run's first: handled there)
      const double wx = here ? tfr[t] : 0.0;
      const double* lo = s_log + (size_t)(here ? j : 0) * S.NBP;
      const double* hi = lo + S.NBP;
      size_t o = out_base + (size_t)(tid >> 7) * P.n_t + t;
      for (int f = tid >> 7; f < P.n_f; f += 2, o += 2 * (size_t)P.n_t) {
        const int fi = s_fi[f];
        double v = 0.0;
        bool write = false;
        if (!t_valid || fi < 0) {
          v = P.fill;                                   // out of range: fill value after normalise + clip
          write = first_run;
        } else if (here) {
          const double wy = s_wy[f];
          const double s00 = lo[fi], s01 = hi[fi], s10 = lo[fi + 1], s11 = hi[fi + 1];
          v = (1.0 - wy) * ((1.0 - wx) * s00 + wx * s01) + wy * ((1.0 - wx) * s10 + wx * s11);
          v = (v - P.spec_min) * P.inv_range;
          v = fmin(fmax(v, 0.0), 1.0);
          write = true;
        }
        if (write && t_in) {
          if (P.out) P.out[o] = (float)v;
          if (P.out64) P.out64[o] = v;
        }
      }
    }
    first_run = false;
    if (nneed == 0) break;
  }
}

}  // namespace ava

// ------------------------------------------------------------------ within_syll_normalize
// ava/preprocessing/utils.py:106-109, per spectrogram (one CTA each, the m = n_f*n_t values in
// shared memory):   spec -= np.quantile(spec, q); spec[spec < 0] = 0; spec /= spec.max() + 1e-12
// np.quantile (method 'linear'): the two order statistics bracketing q*(m-1), found exactly by a
// radix select over the bit patterns (the values are clipped to [0,1], so the IEEE-754 patterns
// of the doubles are ordered like the values), combined with numpy's own lerp formula.
namespace ava {
__device__ double radix_select(const double* v, int m, int k, unsigned int* hist, unsigned long long* s_state) {
  // returns the k-th smallest (0-based) of v[0..m); all threads of the CTA call this together
  unsigned long long prefix = 0ull;   // high bits decided so far
  int rank = k;
  for (int shift = 56; shift >= 0; shift -= 8) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0u;
    __syncthreads();
    const unsigned long long mask = (shift == 56) ? 0ull : (~0ull << (shift + 8));
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
      const unsigned long long b = (unsigned long long)__double_as_longlong(v[i]);
      if ((b & mask) == prefix) atomicAdd(&hist[(unsigned)((b >> shift) & 0xffull)], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int r = rank, bin = 0;
      for (; bin < 255; ++bin) {
        if (r < (int)hist[bin]) break;
        r -= (int)hist[bin];
      }
      s_state[0] = prefix | ((unsigned long long)bin << shift);
      s_state[1] = (unsigned long long)r;
    }
    __syncthreads();
    prefix = s_state[0];
    rank = (int)s_state[1];
    __syncthreads();
  }
  return __longlong_as_double((long long)prefix);
}

__global__ void __launch_bounds__(1024)
quantile_normalize_kernel(double* __restrict__ spec64, float* __restrict__ spec32, int m, double q) {
  extern __shared__ __align__(16) double qs[];
  double* v = qs;                                                   // [m]
  unsigned long long* s_state = reinterpret_cast<unsigned long long*>(v + m);   // [2]
  double* s_max = reinterpret_cast<double*>(s_state + 2);           // [32]
  unsigned int* hist = reinterpret_cast<unsigned int*>(s_max + 32);  // [256]
  double* g64 = spec64 + (size_t)blockIdx.x * m;
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    double x = g64[i];
    v[i] = (x == 0.0) ? 0.0 : x;      // -0.0 -> +0.0 (bit-pattern order)
  }
  __syncthreads();
  // numpy: virtual index q*(m-1), previous = floor, next = previous + 1 (clipped), gamma = fraction
  const double pos = q * (double)(m - 1);
  int lo = (int)floor(pos);
  lo = lo < 0 ? 0 : (lo > m - 1 ? m - 1 : lo);
  const int hi = (lo + 1 > m - 1) ? m - 1 : lo + 1;
  const double t = pos - (double)lo;
  const double a = radix_select(v, m, lo, hist, s_state);
  const double b = radix_select(v, m, hi, hist, s_state);
  // numpy.lib._function_base_impl._lerp: a + (b-a)*t, and b - (b-a)*(1-t) where t >= 0.5, each
  // product rounded before the add (a contracted FMA rounds once and differs in the last bit)
  const double diff = b - a;
  double qv = (t >= 0.5) ? __dsub_rn(b, __dmul_rn(diff, 1.0 - t)) : __dadd_rn(a, __dmul_rn(diff, t));
  if (t == 0.0) qv = a;
  double mx = 0.0;
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    double x = v[i] - qv;
    if (x < 0.0) x = 0.0;
    v[i] = x;
    mx = fmax(mx, x);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = 0.0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) mx = fmax(mx, s_max[w]);
  const double den = mx + 1e-12;
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    const double x = v[i] / den;
    g64[i] = x;
    if (spec32) spec32[(size_t)blockIdx.x * m + i] = (float)x;
  }
}
}  // namespace ava

extern "C" int ava_b200_quantile_normalize(double* spec64, float* spec32, int n, int m, double q, void* stream) {
  using namespace ava;
  AVA_REQUIRE(spec64 != nullptr && m >= 2 && m <= 24576, "quantile_normalize: m=%d (2..24576 values per spectrogram)", m);
  AVA_REQUIRE(q >= 0.0 && q <= 1.0, "quantile_normalize: quantile %f outside [0,1]", q);
  if (n <= 0) return 0;
  const size_t smem = (size_t)m * 8 + 16 + 32 * 8 + 256 * 4;
  static size_t configured = 0;
  if (smem > configured) {
    if (cudaFuncSetAttribute(quantile_normalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
        cudaSuccess) {
      cudaGetLastError();
      set_error("quantile_normalize: %zu bytes of shared memory unavailable", smem);
      return 1;
    }
    configured = smem;
  }
  quantile_normalize_kernel<<<n, 1024, smem, (cudaStream_t)stream>>>(spec64, spec32, m, q);
  return check_launch("quantile_normalize");
}

// Target-time tables of a batch of fixed-duration windows, on the device.  Bit-for-bit the
// float64 arithmetic of the host path (preprocessing/utils.py::bracket), which follows
// ava/models/window_vae_dataset.py:231-235 (target_times = np.linspace(onset, offset, n_t)) and
// the scipy interp2d bracketing / fill rule behind ava/preprocessing/utils.py:80-81,99:
//   T_j   = fl(fl(j * step) + tstart), step = fl(fl(tstop - tstart) / (n_t-1)), T_{n_t-1} = tstop
//   g_k   = fl(base[k] + grid0)                     (frame times, the reference's t += max(0,t1))
//   i     = the interval [g_i, g_{i+1}] containing T (i <= K-2), w = (T-g_i)/(g_{i+1}-g_i)
//   T < g_0 or T > g_{K-1}: i = -1, w = 0 (fill value)
// No FMA contraction anywhere (numpy multiplies, then adds).
namespace ava {
__global__ void __launch_bounds__(128)
time_tables_kernel(const double* __restrict__ grid0, const int* __restrict__ K, const double* __restrict__ base,
                   const double* __restrict__ tstart, const double* __restrict__ tstop, int n, int n_t,
                   int* __restrict__ t_idx, double* __restrict__ t_frac) {
  const int w = blockIdx.x;
  if (w >= n) return;
  const double g0 = grid0[w];
  const int Kw = K[w];
  const long long km2 = Kw - 2;
  const double start = tstart[w], stop = tstop[w];
  const double step = __ddiv_rn(__dsub_rn(stop, start), (double)(n_t - 1));
  const double dt = __dsub_rn(base[1], base[0]);
  const double first = __dadd_rn(base[0], g0);
  const double last = __dadd_rn(base[Kw - 1], g0);
  for (int j = threadIdx.x; j < n_t; j += blockDim.x) {
    const double T = (j == n_t - 1 && n_t > 1) ? stop : __dadd_rn(__dmul_rn((double)j, step), start);
    double f = floor(__ddiv_rn(__dsub_rn(T, first), dt));
    f = fmin(fmax(f, 0.0), (double)km2);
    long long i = (long long)f;
    for (int it = 0; it < 2; ++it) {
      if (__dadd_rn(base[i], g0) > T) --i;
      i = i < 0 ? 0 : (i > km2 ? km2 : i);
      if (__dadd_rn(base[i + 1], g0) <= T && i < km2) ++i;
    }
    const double lo = __dadd_rn(base[i], g0), hi = __dadd_rn(base[i + 1], g0);
    const double wgt = __ddiv_rn(__dsub_rn(T, lo), __dsub_rn(hi, lo));
    const bool bad = (T < first) || (T > last);
    t_idx[(size_t)w * n_t + j] = bad ? -1 : (int)i;
    t_frac[(size_t)w * n_t + j] = bad ? 0.0 : wgt;
  }
}
}  // namespace ava

extern "C" int ava_b200_window_time_tables(const double* grid0, const int* K, const double* base, int kmax,
                                           const double* tstart, const double* tstop, int n, int n_t, int* t_idx,
                                           double* t_frac, void* stream) {
  using namespace ava;
  AVA_REQUIRE(kmax >= 3 && n_t >= 2, "window_time_tables: kmax=%d n_t=%d", kmax, n_t);
  if (n <= 0) return 0;
  time_tables_kernel<<<n, 128, 0, (cudaStream_t)stream>>>(grid0, K, base, tstart, tstop, n, n_t, t_idx, t_frac);
  return check_launch("window_time_tables");
}

extern "C" int ava_b200_get_spec_batch(const void* audio, int is_f32, const long long* seg_start,
                                       const int* seg_len, int n, int nperseg, int noverlap, int remove_dc,
                                       const double* window, double scale, const int* t_idx,
                                       const double* t_frac, int n_t, const int* f_idx, const double* f_frac,
                                       int n_f, int max_frames, double spec_min, double spec_max, float* out,
                                       double* out64, void* stream) {
  using namespace ava;
  AVA_REQUIRE(nperseg >= 16 && nperseg <= 4096 && (nperseg & (nperseg - 1)) == 0,
              "get_spec: nperseg=%d must be a power of two in [16,4096]", nperseg);
  AVA_REQUIRE(noverlap >= 0 && noverlap < nperseg, "get_spec: bad noverlap %d", noverlap);
  AVA_REQUIRE(spec_max != spec_min, "get_spec: spec_max_val == spec_min_val");
  AVA_REQUIRE(is_f32 >= 0 && is_f32 <= 2, "get_spec: sample type %d (0 int16, 1 float32, 2 float64)", is_f32);
  AVA_REQUIRE(n_f >= 1 && n_t >= 1, "get_spec: n_f=%d n_t=%d", n_f, n_t);
  AVA_REQUIRE(out != nullptr || out64 != nullptr, "get_spec: no output (out and out64 both null)");
  if (n <= 0) return 0;
  SpecParams P;
  P.audio = audio;
  P.is_f32 = is_f32;
  P.seg_start = seg_start;
  P.seg_len = seg_len;
  P.nperseg = nperseg;
  P.hop = nperseg - noverlap;
  P.log2n = 0;
  while ((1 << P.log2n) < nperseg) ++P.log2n;
  P.remove_dc = remove_dc;
  P.window = window;
  P.scale = scale;
  P.t_idx = t_idx;
  P.t_frac = t_frac;
  P.n_t = n_t;
  P.f_idx = f_idx;
  P.f_frac = f_frac;
  P.n_f = n_f;
  P.max_frames = max_frames;
  P.spec_min = spec_min;
  P.inv_range = 1.0 / (spec_max - spec_min);
  // ava/preprocessing/utils.py:99-104: fill value -1/EPSILON, then (x - min) / (max - min), clipped
  P.fill = fmin(fmax((-1.0 / 1e-12 - spec_min) / (spec_max - spec_min), 0.0), 1.0);
  P.out = out;
  P.out64 = out64;
  // shared memory: G packed transforms (G*N ~ 2048 points), twiddles, CF log-spectrum slots within
  // ~96 KB (two CTAs per SM), frame lists
  SpecSmem S;
  S.G = 2048 / nperseg;
  if (S.G < 1) S.G = 1;
  if (S.G > 8) S.G = 8;
  S.NBP = nperseg / 2 + 2;
  const size_t fixed = (size_t)S.G * nperseg * 16 + (size_t)nperseg * 16 + 64 +
                       (size_t)2 * (max_frames + 1) * 4 + 16 + (size_t)(n_f + 2) * 12 + 16;
  const size_t budget = (size_t)96 * 1024;
  long long cf = fixed < budget ? (long long)((budget - fixed) / ((size_t)S.NBP * 8)) : 0;
  if (cf < 4) cf = 4;
  if (cf > max_frames + 1) cf = max_frames + 1;
  if (cf < 2) cf = 2;
  S.CF = (int)cf;
  size_t smem = fixed + (size_t)S.CF * S.NBP * 8;
  smem = (smem + 15) / 16 * 16;
  AVA_REQUIRE(smem <= 227 * 1024, "get_spec: %zu bytes of shared memory needed (nperseg %d)", smem, nperseg);
  // one instantiation per power-of-two nperseg
  using Kern = void (*)(const SpecParams, const SpecSmem);
  static const Kern kerns[13] = {nullptr, nullptr, nullptr, nullptr, get_spec_kernel<4>, get_spec_kernel<5>,
                                 get_spec_kernel<6>, get_spec_kernel<7>, get_spec_kernel<8>, get_spec_kernel<9>,
                                 get_spec_kernel<10>, get_spec_kernel<11>, get_spec_kernel<12>};
  static size_t configured[13] = {0};
  Kern kern = kerns[P.log2n];
  if (smem > configured[P.log2n]) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
      cudaGetLastError();
      set_error("get_spec: %zu bytes of shared memory unavailable", smem);
      return 1;
    }
    configured[P.log2n] = smem;
  }
  kern<<<n, 256, smem, (cudaStream_t)stream>>>(P, S);
  return check_launch("get_spec");
}
