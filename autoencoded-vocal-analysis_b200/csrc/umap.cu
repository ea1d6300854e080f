// UMAP of the latent means: the device stages of umap-learn 0.5's UMAP(metric='euclidean').fit_transform,
// the projection the reference builds in ava/data/data_container.py (_make_latent_mean_umap_projection)
// with umap.UMAP(n_components=2, n_neighbors=20, min_dist=0.1, metric='euclidean', random_state=42).
//
//   1. exact kNN (replaces umap.umap_.nearest_neighbors / NNDescent): brute force over all N^2 pairs.
//      Pass 0: the rows shifted by the mean of the first rows and scaled by a power of two to |y| < 1,
//      rounded to fp32 (so the fp32 pass sees O(1) values whatever the data's offset and scale).
//      Pass 1, fp32: each thread owns one query row (in registers) and a sorted top-KP list (distances
//      in registers, indices in a shared-memory column of its own); candidate rows stream through shared
//      memory in tiles.  Squared distance in the difference form sum (x - y)^2.  KP >= k + 8 keeps a
//      margin for fp32 near-ties; the query itself enters with distance -1, so it is always kept.
//      Pass 2, fp64: a warp per query recomputes the KP candidates' distances from the input rows and
//      ranks them by (distance, not-self, index); the first k are written.  The row is certified when
//      its k-th distance is strictly below a rounding-error bound on the distance of every candidate
//      pass 1 dropped (knn_reject_bound); the rest are rescanned over all rows in fp64 and ranked again.
//      Cost: N^2 * D subtract + FMA pairs on the FP32 pipe (pass 1); pass 2 is O(N * KP * D).
//   2. smooth_knn_dist + compute_membership_strengths (umap.umap_), one thread per row, fp64.
//   3. the fuzzy union P = A + A^T - A.*A^T (umap.umap_.fuzzy_simplicial_set, set_op_mix_ratio = 1):
//      the caller sorts and de-duplicates the directed-edge keys row * N + col (a sort is plumbing);
//      the weights, row pointers and the SGD schedule (umap.umap_.make_epochs_per_sample, the set-up
//      of umap.layouts.optimize_layout_euclidean) are computed here.
//   4. spectral initialisation (umap.spectral.spectral_layout / multi_component_layout): connected
//      components by min-label propagation, the normalised-Laplacian product of LOBPCG as a CSR SpMM
//      (warp per row), fixed-order tall-skinny Gram and combination kernels, the final expansion,
//      noise and per-axis rescale.
//   5. the layout SGD (umap.layouts._optimize_layout_euclidean_single_epoch), one launch per epoch, one
//      thread per edge, Hogwild updates of the shared fp32 embedding.
//
// Random numbers (negative samples, noise, random initialisations) come from a counter-based hash:
// splitmix64 applied along the key (seed, stream, i, j), so every draw is a pure function of its key.
// Every output of stages 1-4 is bitwise reproducible (no atomics in any sum); stage 5 is not, as
// Hogwild updates race by design (umap-learn's parallel mode).
#include <float.h>
#include <limits.h>

#include <algorithm>

#include "common.cuh"

namespace ava {

// ------------------------------------------------------------------------------------------ hash
__host__ __device__ __forceinline__ unsigned long long umap_mix(unsigned long long z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ unsigned long long umap_hash(unsigned long long seed, unsigned long long a,
                                                                 unsigned long long b, unsigned long long c) {
  return umap_mix(umap_mix(umap_mix(umap_mix(seed) ^ a) ^ b) ^ c);
}
// uniform in (0, 1): the top 53 bits, offset by half an ulp
__device__ __forceinline__ double umap_unit(unsigned long long h) {
  return ((double)(h >> 11) + 0.5) * (1.0 / 9007199254740992.0);
}

// ------------------------------------------------------------------------------------------ kNN
constexpr int KNN_THREADS = 128;   // queries per CTA
constexpr int KNN_TILE = 64;       // candidate rows per shared-memory tile
constexpr int KNN_MAX_D = 64;
constexpr int KNN_SHIFT_ROWS = 1024;
// The data rows are split into S slices, one per grid row, when the query CTAs alone would leave SMs idle
// (knn_slices).  Each slice keeps its own top-KP; the refine pass ranks the S * KP candidates of a query.
constexpr int KNN_CTAS_PER_SM = 4;       // knn_select_kernel<float, float, 32, 32, *>: 102 registers x 128 threads
constexpr int KNN_MAX_CAND = 256;        // S * KP: the refine pass ranks them in shared memory, in O(S^2 KP^2)
constexpr int KNN_MIN_SLICE_ROWS = 1024;
constexpr int KNN_REFINE_WARPS = 8;

// Workspace: cand [Nq][S][KP] int | d32 [Nq][S] float (the worst kept fp32 distance of each query in each slice) |
// list [Nq] int (the queries the certificate rejects) | y [N][D] float (the scaled data rows) | yq [Nq][D] float (the
// scaled queries; absent when the data is its own query set) | shift [64] double | range (max |x - shift| over the
// data and the queries, as fp64 bits) | count.
struct KnnWs {
  int* cand;
  float* y;
  float* yq;
  float* d32;
  int* list;
  double* shift;
  unsigned long long* range;
  int* count;
};
static long long knn_ws_layout(int Nq, int N, int D, int KP, int S, bool self, void* base, KnnWs* w) {
  const long long nq = Nq, n = N;
  const long long o_d32 = nq * S * KP * 4, o_list = o_d32 + nq * S * 4, o_y = o_list + nq * 4;
  const long long o_yq = o_y + n * D * 4;
  const long long o_hdr = (o_yq + (self ? 0 : nq * D * 4) + 7) / 8 * 8;
  const long long o_range = o_hdr + KNN_MAX_D * 8, o_count = o_range + 8;
  if (w) {
    char* b = (char*)base;
    w->cand = (int*)b;
    w->d32 = (float*)(b + o_d32);
    w->list = (int*)(b + o_list);
    w->y = (float*)(b + o_y);
    w->yq = self ? w->y : (float*)(b + o_yq);
    w->shift = (double*)(b + o_hdr);
    w->range = (unsigned long long*)(b + o_range);
    w->count = (int*)(b + o_count);
  }
  return o_count + 8;
}

// The number of slices: 1 when the Q = ceil(Nq / 128) query CTAs fill one wave of KNN_CTAS_PER_SM per SM; otherwise
// the S whose Q S CTAs fill their last wave best, among S * KP <= KNN_MAX_CAND and slices of at least
// KNN_MIN_SLICE_ROWS rows; a larger S is taken only if it fills 2% more than the best smaller one.
static int knn_slices(int Nq, int N, int KP) {
  const long long ctas = (Nq + KNN_THREADS - 1) / KNN_THREADS;
  const long long slots = (long long)KNN_CTAS_PER_SM * kNumSMs;
  if (ctas >= slots) return 1;
  int best = 1;
  double best_fill = 0.0;
  for (int S = 1; S * KP <= KNN_MAX_CAND && (S == 1 || N / S >= KNN_MIN_SLICE_ROWS); ++S) {
    const long long c = ctas * S;
    const double fill = (double)c / (double)((c + slots - 1) / slots * slots);
    if (fill > best_fill * 1.02) {
      best = S;
      best_fill = fill;
    }
  }
  return best;
}
// rows per slice: all N for one slice, else a whole number of tiles (the last slices may be short or empty)
static int knn_slice_rows(int N, int S) {
  if (S == 1) return N;
  const int per = (N + S - 1) / S;
  return (per + KNN_TILE - 1) / KNN_TILE * KNN_TILE;
}

// The fp32 pass selects on y = (x - shift) 2^-e, with shift the mean of the first data rows and e the exponent of
// M = max |x - shift| over the data and the queries (M = ms 2^e, ms in [0.5, 1)): the values are O(1) whatever the
// offset and scale.  2^-e is applied as two factors so that neither overflows for any finite M.
struct KnnScale {
  double f1, f2;
};
__device__ __forceinline__ KnnScale knn_scale(const unsigned long long* range) {
  const double M = __longlong_as_double((long long)*range);
  int e = 0;
  if (M > 0.0) frexp(M, &e);
  KnnScale s;
  s.f1 = ldexp(1.0, -(e / 2));
  s.f2 = ldexp(1.0, -(e - e / 2));
  return s;
}

// shift[d] = mean of the first KNN_SHIFT_ROWS rows; zeroes the range and the rejected-row count
template <typename T>
__global__ void knn_shift_kernel(const T* __restrict__ x, int N, int D, double* __restrict__ shift,
                                 unsigned long long* __restrict__ range, int* __restrict__ count) {
  const int d = threadIdx.x;
  if (d == 0) {
    *range = 0ull;
    *count = 0;
  }
  if (d >= D) return;
  const int R = min(N, KNN_SHIFT_ROWS);
  double s = 0.0;
  for (int r = 0; r < R; ++r) s += (double)x[(long long)r * D + d];
  shift[d] = s / (double)R;
}

// range = max(range, max |x - shift| over all n values) (the bits of a non-negative double order like the value)
template <typename T>
__global__ void knn_range_kernel(const T* __restrict__ x, long long n, int D, const double* __restrict__ shift,
                                 unsigned long long* __restrict__ range) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  int d = (int)(i % D);
  const int dstep = (int)(stride % D);
  double m = 0.0;
  for (; i < n; i += stride) {
    m = fmax(m, fabs((double)x[i] - shift[d]));
    d += dstep;
    if (d >= D) d -= D;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (threadIdx.x % 32 == 0 && m > 0.0) atomicMax(range, (unsigned long long)__double_as_longlong(m));
}

// y = (float)((x - shift) 2^-e), the values the fp32 pass selects on
template <typename T>
__global__ void knn_scaled_kernel(const T* __restrict__ x, long long n, int D, const double* __restrict__ shift,
                                  const unsigned long long* __restrict__ range, float* __restrict__ y) {
  const KnnScale sc = knn_scale(range);
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  int d = (int)(i % D);
  const int dstep = (int)(stride % D);
  for (; i < n; i += stride) {
    y[i] = (float)((((double)x[i] - shift[d]) * sc.f1) * sc.f2);
    d += dstep;
    if (d >= D) d -= D;
  }
}

// Top-KP candidates of each query row xq[q] among the data rows of slice blockIdx.y (rows [y L, y L + L) of x), by
// squared Euclidean distance in the difference form, written to cand[q][slice].
// ACC = float: the selection pass on the scaled rows; also records the worst kept distance d32[q][slice], which bounds
//   the distance of every candidate of the slice it did not keep.
// ACC = double: the rescan of the queries list[0 .. *count) on the input rows, with the same formula (and so the same
//   bits) as knn_refine_kernel; ties go to the lower index, as in the refine ranking.
// SELF: the data is its own query set (xq == x), and query q enters its own list with distance -1, so it is kept.
template <typename T, typename ACC, int DP, int KP, bool SELF>
__global__ void __launch_bounds__(KNN_THREADS, 1)
knn_select_kernel(const T* __restrict__ xq, int Nq, const T* __restrict__ x, int N, int D, int L,
                  const int* __restrict__ list, const int* __restrict__ count, int* __restrict__ cand,
                  float* __restrict__ d32) {
  constexpr bool F64 = sizeof(ACC) == 8;
  __shared__ __align__(16) ACC tile[KNN_TILE * DP];
  extern __shared__ int sidx[];   // [KP][KNN_THREADS]
  const int tid = threadIdx.x;
  const int S = gridDim.y, slice = blockIdx.y;
  const int c_lo = slice * L, c_hi = min(N, c_lo + L);
  int q;
  if (F64) {
    const int n_list = *count;
    if (blockIdx.x * KNN_THREADS >= n_list) return;
    const int p = blockIdx.x * KNN_THREADS + tid;
    q = p < n_list ? list[p] : -1;
  } else {
    q = blockIdx.x * KNN_THREADS + tid;
    if (q >= Nq) q = -1;
  }
  ACC xr[DP];
#pragma unroll
  for (int d = 0; d < DP; ++d) xr[d] = (q >= 0 && d < D) ? (ACC)xq[(long long)q * D + d] : (ACC)0;
  ACC dk[KP];
#pragma unroll
  for (int j = 0; j < KP; ++j) {
    dk[j] = F64 ? (ACC)INFINITY : (ACC)FLT_MAX;
    sidx[j * KNN_THREADS + tid] = -1;
  }
  for (int c0 = c_lo; c0 < c_hi; c0 += KNN_TILE) {
    __syncthreads();
    for (int e = tid; e < KNN_TILE * DP; e += KNN_THREADS) {
      const int r = e / DP, d = e - r * DP;
      tile[e] = (c0 + r < c_hi && d < D) ? (ACC)x[(long long)(c0 + r) * D + d] : (ACC)0;
    }
    __syncthreads();
    const int nc = min(KNN_TILE, c_hi - c0);
    for (int r = 0; r < nc; ++r) {
      ACC dist;
      if constexpr (F64) {
        double s = 0.0;
#pragma unroll
        for (int d = 0; d < DP; ++d) {
          const double e = xr[d] - tile[r * DP + d];
          s = __fma_rn(e, e, s);
        }
        dist = fmin(s, DBL_MAX);   // an overflowed distance still fills an empty slot
      } else {
        const float4* t4 = reinterpret_cast<const float4*>(tile + r * DP);
        float s0 = 0.f, s1 = 0.f;
#pragma unroll
        for (int d4 = 0; d4 < DP / 4; ++d4) {
          const float4 v = t4[d4];
          const float e0 = xr[4 * d4] - v.x, e1 = xr[4 * d4 + 1] - v.y;
          const float e2 = xr[4 * d4 + 2] - v.z, e3 = xr[4 * d4 + 3] - v.w;
          s0 = fmaf(e0, e0, s0);
          s1 = fmaf(e1, e1, s1);
          s0 = fmaf(e2, e2, s0);
          s1 = fmaf(e3, e3, s1);
        }
        dist = s0 + s1;
      }
      const int c = c0 + r;
      if (SELF && c == q) dist = (ACC)-1;
      if (dist < dk[KP - 1]) {
#pragma unroll
        for (int j = KP - 1; j > 0; --j) {
          if (dist < dk[j - 1]) {
            dk[j] = dk[j - 1];
            sidx[j * KNN_THREADS + tid] = sidx[(j - 1) * KNN_THREADS + tid];
          } else if (dist < dk[j]) {
            dk[j] = dist;
            sidx[j * KNN_THREADS + tid] = c;
          }
        }
        if (dist < dk[0]) {
          dk[0] = dist;
          sidx[tid] = c;
        }
      }
    }
  }
  if (q >= 0) {
    int* out = cand + ((long long)q * S + slice) * KP;
    for (int j = 0; j < KP; ++j) out[j] = sidx[j * KNN_THREADS + tid];
    if (!F64) d32[(long long)q * S + slice] = (float)dk[KP - 1];
  }
}

// A lower bound, in the input's units, on the distance of every candidate the fp32 pass did not keep for a
// row whose worst kept fp32 squared distance is t32 (each of those has a computed fp32 distance >= t32).
// With u = 2^-24 and ms = M 2^-e <= 1 the largest scaled |value|:
//  - each scaled value is within delta = (u + 2^-52) ms + 2^-149 of the exact (x - shift) 2^-e;
//  - the fp32 sum of DP squared differences (two chains of DP/2 FMAs and one add; subtraction results that
//    are subnormal are exact) is at most (1 + g)(exact sum of the rounded values) + (DP + 1) 2^-149,
//    g = (DP/2 + 3) u (1.001);
// so the true scaled distance is at least sqrt((t32 - (DP + 1) 2^-149) / (1 + g)) - 2 delta sqrt(D).  The
// result is shrunk by 2^-40 to cover the rounding of this evaluation and of the fp64 distances it meets.
__device__ __forceinline__ double knn_reject_bound(float t32, const unsigned long long* range, int D, int DP) {
  const double M = __longlong_as_double((long long)*range);
  int e = 0;
  const double ms = M > 0.0 ? frexp(M, &e) : 0.0;
  const double u = 0x1p-24;
  const double g = (DP / 2 + 3) * u * 1.001;
  const double delta = (u + 0x1p-52) * ms + 0x1p-149;
  const double a = sqrt(fmax((double)t32 - (DP + 1) * 0x1p-149, 0.0) / (1.0 + g));
  const double lb = a - 2.0 * delta * sqrt((double)D);
  return lb > 0.0 ? ldexp(lb * (1.0 - 0x1p-40), e) : 0.0;
}

// One warp per query: fp64 distances of its S * KP candidates (the slices' lists, which share no row), ranked by
// (distance, index), with the query itself first when SELF; the first k are written.  certify: queries 0..Nq-1, and a
// query whose k-th distance is not strictly below knn_reject_bound of the smallest of its slices' worst kept fp32
// distances (a slice's dropped candidates are at least its own bound away) is appended to list for the fp64 rescan;
// all_kept: no slice dropped a candidate.  Otherwise: the queries list[0 .. *count).
template <typename T, bool SELF>
__global__ void knn_refine_kernel(const T* __restrict__ xq, int Nq, const T* __restrict__ x, int D, int DP, int S,
                                  int KP, int k, const int* __restrict__ cand, int certify, int all_kept,
                                  const float* __restrict__ d32, const unsigned long long* __restrict__ range,
                                  int* __restrict__ list, int* __restrict__ count, int* __restrict__ knn_idx,
                                  double* __restrict__ knn_dist) {
  extern __shared__ double sref[];
  const int C = S * KP;
  const int warps = blockDim.x / 32, w = threadIdx.x / 32, lane = threadIdx.x % 32;
  double* sd = sref + w * C;
  int* si = reinterpret_cast<int*>(sref + warps * C) + w * C;
  int q = blockIdx.x * warps + w;
  if (certify) {
    if (q >= Nq) return;
  } else {
    if (q >= *count) return;
    q = list[q];
  }
  for (int j = lane; j < C; j += 32) {
    const int c = cand[(long long)q * C + j];
    double s = INFINITY;
    if (c >= 0) {
      s = 0.0;
      for (int d = 0; d < D; ++d) {
        const double e = (double)xq[(long long)q * D + d] - (double)x[(long long)c * D + d];
        s = __fma_rn(e, e, s);
      }
    }
    sd[j] = s;
    si[j] = c;
  }
  __syncwarp();
  double kth = 0.0;   // the k-th fp64 squared distance
  for (int j = lane; j < C; j += 32) {
    const int c = si[j];
    if (c < 0) continue;
    const double dj = sd[j];
    const int kj = (SELF && c == q) ? -1 : c;
    int rank = 0;
    for (int i = 0; i < C; ++i) {
      const int ci = si[i];
      if (ci < 0) continue;
      const double di = sd[i];
      const int ki = (SELF && ci == q) ? -1 : ci;
      rank += (di < dj) || (di == dj && ki < kj);
    }
    if (rank < k) {
      knn_idx[(long long)q * k + rank] = c;
      knn_dist[(long long)q * k + rank] = sqrt(dj);
    }
    if (rank == k - 1) kth = dj;
  }
  if (!certify || all_kept) return;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) kth = fmax(kth, __shfl_xor_sync(0xffffffffu, kth, o));
  if (lane == 0) {
    float t32 = FLT_MAX;
    for (int sl = 0; sl < S; ++sl) t32 = fminf(t32, d32[(long long)q * S + sl]);
    if (!(sqrt(kth) < knn_reject_bound(t32, range, D, DP))) list[atomicAdd(count, 1)] = q;
  }
}

static int knn_padded(int k) {
  for (int kp : {16, 32, 64, 128})
    if (kp >= k + 8 || kp == 128) return kp;
  return 128;
}
static int knn_dpad(int D) {
  for (int dp : {8, 16, 32, 64})
    if (dp >= D) return dp;
  return -1;
}

struct KnnShape {
  int Nq, N, D, KP, S, L;
};

template <typename T, typename ACC, int DP, int KP, bool SELF>
static int knn_launch(const T* xq, const T* x, const KnnShape& sh, const KnnWs& w, cudaStream_t s) {
  const size_t smem = (size_t)KP * KNN_THREADS * sizeof(int);
  auto kern = knn_select_kernel<T, ACC, DP, KP, SELF>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    set_error("umap knn_select_kernel: cudaFuncSetAttribute failed");
    return 1;
  }
  const dim3 grid((sh.Nq + KNN_THREADS - 1) / KNN_THREADS, sh.S);
  kern<<<grid, KNN_THREADS, smem, s>>>(xq, sh.Nq, x, sh.N, sh.D, sh.L, w.list, w.count, w.cand, w.d32);
  return check_launch(sizeof(ACC) == 4 ? "umap knn_select_kernel" : "umap knn_select_kernel (fp64 rescan)");
}

template <typename T, typename ACC, int DP, bool SELF>
static int knn_launch_k(const T* xq, const T* x, const KnnShape& sh, const KnnWs& w, cudaStream_t s) {
  switch (sh.KP) {
    case 16: return knn_launch<T, ACC, DP, 16, SELF>(xq, x, sh, w, s);
    case 32: return knn_launch<T, ACC, DP, 32, SELF>(xq, x, sh, w, s);
    case 64: return knn_launch<T, ACC, DP, 64, SELF>(xq, x, sh, w, s);
    default: return knn_launch<T, ACC, DP, 128, SELF>(xq, x, sh, w, s);
  }
}

template <typename T, typename ACC, bool SELF>
static int knn_select(const T* xq, const T* x, const KnnShape& sh, const KnnWs& w, cudaStream_t s) {
  switch (knn_dpad(sh.D)) {
    case 8: return knn_launch_k<T, ACC, 8, SELF>(xq, x, sh, w, s);
    case 16: return knn_launch_k<T, ACC, 16, SELF>(xq, x, sh, w, s);
    case 32: return knn_launch_k<T, ACC, 32, SELF>(xq, x, sh, w, s);
    default: return knn_launch_k<T, ACC, 64, SELF>(xq, x, sh, w, s);
  }
}

static KnnShape knn_shape(int Nq, int N, int D, int k) {
  KnnShape sh;
  sh.Nq = Nq;
  sh.N = N;
  sh.D = D;
  sh.KP = knn_padded(k);
  sh.S = knn_slices(Nq, N, sh.KP);
  sh.L = knn_slice_rows(N, sh.S);
  return sh;
}

// range and scaled rows of one row set
template <typename T>
static int knn_scale_rows(const T* x, int rows, int D, const KnnWs& w, float* y, bool range_only, cudaStream_t s) {
  const long long n = (long long)rows * D;
  if (range_only) {
    knn_range_kernel<T><<<(unsigned)std::min<long long>((n + 255) / 256, 4 * kNumSMs), 256, 0, s>>>(x, n, D, w.shift,
                                                                                                    w.range);
    return check_launch("umap knn_range_kernel");
  }
  knn_scaled_kernel<T><<<(unsigned)std::min<long long>((n + 255) / 256, 8 * kNumSMs), 256, 0, s>>>(x, n, D, w.shift,
                                                                                                   w.range, y);
  return check_launch("umap knn_scaled_kernel");
}

// Queries xq [Nq, D] against data x [N, D] (SELF: xq == x).  Shift and range (over both sets); fp32 selection per
// slice; fp64 refine with the certificate; fp64 rescan and refine of the queries it rejects (the last two launches
// find an empty list and return at once in the usual case).
template <typename T, bool SELF>
static int knn_run(const T* xq, int Nq, const T* x, int N, int D, int k, int* knn_idx, double* knn_dist, void* ws,
                   cudaStream_t s) {
  const KnnShape sh = knn_shape(Nq, N, D, k);
  const int DP = knn_dpad(D);
  KnnWs w;
  knn_ws_layout(Nq, N, D, sh.KP, sh.S, SELF, ws, &w);
  knn_shift_kernel<T><<<1, KNN_MAX_D, 0, s>>>(x, N, D, w.shift, w.range, w.count);
  if (check_launch("umap knn_shift_kernel")) return 1;
  if (knn_scale_rows(x, N, D, w, w.y, true, s)) return 1;
  if (!SELF && knn_scale_rows(xq, Nq, D, w, w.yq, true, s)) return 1;
  if (knn_scale_rows(x, N, D, w, w.y, false, s)) return 1;
  if (!SELF && knn_scale_rows(xq, Nq, D, w, w.yq, false, s)) return 1;
  if (knn_select<float, float, SELF>(w.yq, w.y, sh, w, s)) return 1;
  const size_t smem = (size_t)KNN_REFINE_WARPS * sh.S * sh.KP * (sizeof(double) + sizeof(int));
  auto refine = knn_refine_kernel<T, SELF>;
  if (cudaFuncSetAttribute(refine, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    set_error("umap knn_refine_kernel: cudaFuncSetAttribute failed");
    return 1;
  }
  const unsigned grid = (unsigned)((Nq + KNN_REFINE_WARPS - 1) / KNN_REFINE_WARPS);
  const int all_kept = sh.L <= sh.KP;
  refine<<<grid, KNN_REFINE_WARPS * 32, smem, s>>>(xq, Nq, x, D, DP, sh.S, sh.KP, k, w.cand, 1, all_kept, w.d32,
                                                   w.range, w.list, w.count, knn_idx, knn_dist);
  if (check_launch("umap knn_refine_kernel")) return 1;
  if (knn_select<T, double, SELF>(xq, x, sh, w, s)) return 1;
  refine<<<grid, KNN_REFINE_WARPS * 32, smem, s>>>(xq, Nq, x, D, DP, sh.S, sh.KP, k, w.cand, 0, all_kept, w.d32,
                                                   w.range, w.list, w.count, knn_idx, knn_dist);
  return check_launch("umap knn_refine_kernel (rescanned rows)");
}

// --------------------------------------------------------------------- smooth kNN, memberships
constexpr int SMOOTH_N_ITER = 64;
constexpr double SMOOTH_K_TOLERANCE = 1e-5;
constexpr double MIN_K_DIST_SCALE = 1e-3;

// fixed-order mean of all N*k distances (one CTA)
__global__ void mean_kernel(const double* __restrict__ v, long long n, double* __restrict__ out) {
  __shared__ double red[1024];
  double s = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) s += v[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = red[0] / (double)n;
}

// BIPARTITE: the rows are queries against another row set (umap-learn's transform), so no entry is the row itself
template <bool BIPARTITE>
__global__ void smooth_knn_kernel(const int* __restrict__ knn_idx, const double* __restrict__ knn_dist, int N, int k,
                                  double local_connectivity, const double* __restrict__ mean_all,
                                  double* __restrict__ rho_out, double* __restrict__ sigma_out,
                                  double* __restrict__ w) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const double* di = knn_dist + (long long)i * k;
  const double target = log2((double)k);
  // rho: the local_connectivity-th nonzero distance (interpolated), or the largest if there are fewer
  int n_nz = 0;
  double last_nz = 0.0, row_sum = 0.0;
  for (int j = 0; j < k; ++j) {
    row_sum += di[j];
    if (di[j] > 0.0) {
      ++n_nz;
      last_nz = di[j];
    }
  }
  double rho = 0.0;
  if ((double)n_nz >= local_connectivity) {
    const int index = (int)floor(local_connectivity);
    const double interpolation = local_connectivity - index;
    int seen = 0;
    double nz_prev = 0.0, nz_at = 0.0, nz_first = 0.0;
    for (int j = 0; j < k; ++j)
      if (di[j] > 0.0) {
        if (seen == 0) nz_first = di[j];
        if (seen == index - 1) nz_prev = di[j];
        if (seen == index) nz_at = di[j];
        ++seen;
      }
    if (index > 0) {
      rho = nz_prev;
      // umap-learn's rounding (no contraction into an FMA), so that rho repeats its bits
      if (interpolation > SMOOTH_K_TOLERANCE) rho = __dadd_rn(rho, __dmul_rn(interpolation, nz_at - nz_prev));
    } else {
      rho = interpolation * nz_first;
    }
  } else if (n_nz > 0) {
    rho = last_nz;   // distances are sorted: the last nonzero one is the largest
  }
  double lo = 0.0, hi = INFINITY, mid = 1.0;
  for (int it = 0; it < SMOOTH_N_ITER; ++it) {
    double psum = 0.0;
    for (int j = 1; j < k; ++j) {
      const double d = di[j] - rho;
      psum += d > 0.0 ? exp(-(d / mid)) : 1.0;
    }
    if (fabs(psum - target) < SMOOTH_K_TOLERANCE) break;
    if (psum > target) {
      hi = mid;
      mid = (lo + hi) / 2.0;
    } else {
      lo = mid;
      if (hi == INFINITY) mid *= 2.0;
      else mid = (lo + hi) / 2.0;
    }
  }
  double sigma = mid;
  const double floor_ref = rho > 0.0 ? row_sum / (double)k : *mean_all;
  if (sigma < MIN_K_DIST_SCALE * floor_ref) sigma = MIN_K_DIST_SCALE * floor_ref;
  rho_out[i] = rho;
  sigma_out[i] = sigma;
  for (int j = 0; j < k; ++j) {
    const int c = knn_idx[(long long)i * k + j];
    double v;
    if (!BIPARTITE && c == i) v = 0.0;
    else if (di[j] - rho <= 0.0 || sigma == 0.0) v = 1.0;
    else v = exp(-((di[j] - rho) / sigma));
    w[(long long)i * k + j] = v;
  }
}

// ------------------------------------------------------------------------------- fuzzy union
// directed-edge keys: (i, j) and (j, i) for every neighbour j != i of i; -1 for the self entries
__global__ void edge_keys_kernel(const int* __restrict__ knn_idx, int N, int k, long long* __restrict__ keys) {
  const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (e >= (long long)N * k) return;
  const long long i = e / k;
  const long long j = knn_idx[e];
  keys[2 * e] = (j == i) ? -1 : i * N + j;
  keys[2 * e + 1] = (j == i) ? -1 : j * N + i;
}

__device__ __forceinline__ double knn_weight(const int* __restrict__ knn_idx, const double* __restrict__ w, int k,
                                             long long r, int c) {
  const int* row = knn_idx + r * k;
  for (int j = 0; j < k; ++j)
    if (row[j] == c) return w[r * k + j];
  return 0.0;
}

// keys: sorted, unique, non-negative.  P[r, c] = a + b - a*b with a = A[r, c], b = A[c, r]; rowptr[N + 1].
__global__ void graph_weights_kernel(const long long* __restrict__ keys, long long nnz, int N,
                                     const int* __restrict__ knn_idx, const double* __restrict__ w, int k,
                                     int* __restrict__ rows, int* __restrict__ cols, double* __restrict__ vals,
                                     long long* __restrict__ rowptr) {
  const long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (p > nnz) return;
  if (p == nnz) {
    const long long last = nnz > 0 ? keys[nnz - 1] / N : -1;
    for (long long r = last + 1; r <= N; ++r) rowptr[r] = nnz;
    return;
  }
  const long long key = keys[p];
  const long long r = key / N;
  const int c = (int)(key - r * N);
  const long long prev = p > 0 ? keys[p - 1] / N : -1;
  for (long long rr = prev + 1; rr <= r; ++rr) rowptr[rr] = p;
  const double a = knn_weight(knn_idx, w, k, r, c);
  const double b = knn_weight(knn_idx, w, k, c, (int)r);
  rows[p] = (int)r;
  cols[p] = c;
  vals[p] = __dsub_rn(__dadd_rn(a, b), __dmul_rn(a, b));   // (a + b) - ab, as scipy's A + A^T - A.*A^T rounds
}

__global__ void epochs_per_sample_kernel(const double* __restrict__ vals, long long n, const double* __restrict__ vmax,
                                         int n_epochs, double negative_sample_rate, double* __restrict__ eps,
                                         double* __restrict__ eps_neg, double* __restrict__ next,
                                         double* __restrict__ next_neg) {
  const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (e >= n) return;
  const double ns = (double)n_epochs * (vals[e] / *vmax);
  const double r = ns > 0.0 ? (double)n_epochs / ns : -1.0;
  const double rn = r / negative_sample_rate;
  eps[e] = r;
  eps_neg[e] = rn;
  next[e] = r;
  next_neg[e] = rn;
}

// ---------------------------------------------------------------------- connected components
// one round of min-label hooking; labels only decrease and always name a vertex of the same component
__global__ void components_kernel(const long long* __restrict__ rowptr, const int* __restrict__ cols, int N,
                                  int* __restrict__ label, int* __restrict__ changed) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const int l = label[i];
  int m = label[l];
  for (long long p = rowptr[i]; p < rowptr[i + 1]; ++p) m = min(m, label[cols[p]]);
  if (m < l) {
    atomicMin(&label[i], m);
    atomicMin(&label[l], m);
    *changed = 1;
  }
}

// ------------------------------------------------------------------------- spectral kernels
// dis[i] = 1/sqrt(sum_j P[i, j])
__global__ void degree_kernel(const long long* __restrict__ rowptr, const double* __restrict__ vals, int N,
                              double* __restrict__ dis) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  double s = 0.0;
  for (long long p = rowptr[i]; p < rowptr[i + 1]; ++p) s += vals[p];
  dis[i] = 1.0 / sqrt(s);
}

// Y[r, :] = X[r, :] - dis[v] * sum_j P[v, j] * dis[j] * X[pos[j], :] for v = verts[r]: the normalised
// Laplacian I - D^-1/2 P D^-1/2 of the component whose vertices verts lists (pos: vertex -> row).
// A warp per row; lanes stride the row's entries, then a fixed butterfly sums the lanes.
template <int MM>
__global__ void spmm_kernel(const long long* __restrict__ rowptr, const int* __restrict__ cols,
                            const double* __restrict__ vals, const int* __restrict__ verts, int n,
                            const int* __restrict__ pos, const double* __restrict__ dis, const double* __restrict__ X,
                            int m, double* __restrict__ Y) {
  const int r = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x % 32;
  if (r >= n) return;
  const int v = verts[r];
  double acc[MM];
#pragma unroll
  for (int c = 0; c < MM; ++c) acc[c] = 0.0;
  for (long long p = rowptr[v] + lane; p < rowptr[v + 1]; p += 32) {
    const int j = cols[p];
    const double f = vals[p] * dis[j];
    const double* xj = X + (long long)pos[j] * m;
#pragma unroll
    for (int c = 0; c < MM; ++c)
      if (c < m) acc[c] = fma(f, xj[c], acc[c]);
  }
#pragma unroll
  for (int c = 0; c < MM; ++c) {
    const double s = warp_sum(acc[c]);
    if (lane == c && c < m) Y[(long long)r * m + c] = X[(long long)r * m + c] - dis[v] * s;
  }
}

// out[p, q] = A^T B for A [n, p], B [n, q] row-major: CTA g sums the rows of its contiguous chunk into
// partial[g]; gram_finish adds the partials in CTA order.
constexpr int GRAM_THREADS = 256;
constexpr int GRAM_CTAS = 2 * kNumSMs;
constexpr int GRAM_ROWS = 32;
__global__ void __launch_bounds__(GRAM_THREADS)
gram_kernel(const double* __restrict__ A, int p, const double* __restrict__ B, int q, int n,
            double* __restrict__ partial) {
  extern __shared__ double sg[];
  double* sa = sg;
  double* sb = sg + GRAM_ROWS * p;
  const int outs = p * q;
  const int per = (n + gridDim.x - 1) / gridDim.x;
  const int r0 = blockIdx.x * per, r1 = min(n, r0 + per);
  double acc[8];
#pragma unroll
  for (int t = 0; t < 8; ++t) acc[t] = 0.0;
  for (int t0 = r0; t0 < r1; t0 += GRAM_ROWS) {
    const int nr = min(GRAM_ROWS, r1 - t0);
    __syncthreads();
    for (int e = threadIdx.x; e < nr * p; e += blockDim.x) sa[e] = A[(long long)t0 * p + e];
    for (int e = threadIdx.x; e < nr * q; e += blockDim.x) sb[e] = B[(long long)t0 * q + e];
    __syncthreads();
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int o = threadIdx.x + t * GRAM_THREADS;
      if (o < outs) {
        const int i = o / q, j = o - i * q;
        double s = acc[t];
        for (int rr = 0; rr < nr; ++rr) s = fma(sa[rr * p + i], sb[rr * q + j], s);
        acc[t] = s;
      }
    }
  }
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    const int o = threadIdx.x + t * GRAM_THREADS;
    if (o < outs) partial[(long long)blockIdx.x * outs + o] = acc[t];
  }
}
__global__ void gram_finish_kernel(const double* __restrict__ partial, int outs, int ctas, double* __restrict__ out) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= outs) return;
  double s = 0.0;
  for (int g = 0; g < ctas; ++g) s += partial[(long long)g * outs + o];
  out[o] = s;
}

// Y[n, q] = A[n, p] . C[p, q]
__global__ void combine_kernel(const double* __restrict__ A, int p, const double* __restrict__ C, int q, int n,
                               double* __restrict__ Y) {
  const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (e >= (long long)n * q) return;
  const long long r = e / q;
  const int j = (int)(e - r * q);
  double s = 0.0;
  for (int i = 0; i < p; ++i) s = fma(A[r * p + i], C[(long long)i * q + j], s);
  Y[e] = s;
}

// kind 0: uniform(-scale, scale); kind 1: normal(0, scale) (Box-Muller on two hashed uniforms)
__global__ void random_kernel(unsigned long long seed, unsigned long long stream_id, long long n, int kind,
                              double scale, double* __restrict__ out) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double u1 = umap_unit(umap_hash(seed, stream_id, (unsigned long long)i, 0));
  if (kind == 0) {
    out[i] = scale * (2.0 * u1 - 1.0);
  } else {
    const double u2 = umap_unit(umap_hash(seed, stream_id, (unsigned long long)i, 1));
    out[i] = scale * sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
  }
}

// one CTA per axis: v = (float)(init * expansion) + (float)noise, then 10 * (v - min) / (max - min)
__global__ void init_layout_kernel(const double* __restrict__ init, const double* __restrict__ noise,
                                   double expansion, int N, int dim, float* __restrict__ emb) {
  __shared__ float smin[1024], smax[1024];
  const int d = blockIdx.x;
  auto val = [&](long long i) {
    float v = (float)(init[i * dim + d] * expansion);
    if (noise) v = __fadd_rn(v, (float)noise[i * dim + d]);
    return v;
  };
  float lo = FLT_MAX, hi = -FLT_MAX;
  for (long long i = threadIdx.x; i < N; i += blockDim.x) {
    const float v = val(i);
    lo = fminf(lo, v);
    hi = fmaxf(hi, v);
  }
  smin[threadIdx.x] = lo;
  smax[threadIdx.x] = hi;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
      smin[threadIdx.x] = fminf(smin[threadIdx.x], smin[threadIdx.x + o]);
      smax[threadIdx.x] = fmaxf(smax[threadIdx.x], smax[threadIdx.x + o]);
    }
    __syncthreads();
  }
  const float mn = smin[0], range = __fsub_rn(smax[0], smin[0]);
  for (long long i = threadIdx.x; i < N; i += blockDim.x)
    emb[i * dim + d] = range > 0.f ? __fdiv_rn(__fmul_rn(10.f, __fsub_rn(val(i), mn)), range) : 0.f;
}

// --------------------------------------------------------------------------------- layout SGD
constexpr int UMAP_MAX_DIM = 8;

__device__ __forceinline__ double umap_clip(double v) { return v > 4.0 ? 4.0 : (v < -4.0 ? -4.0 : v); }

__global__ void sgd_epoch_kernel(float* __restrict__ emb, int N, int dim, const int* __restrict__ head,
                                 const int* __restrict__ tail, const double* __restrict__ eps,
                                 const double* __restrict__ eps_neg, double* __restrict__ next,
                                 double* __restrict__ next_neg, long long e0, long long e1, int epoch, double a,
                                 double b, double gamma, double alpha, unsigned long long seed) {
  const long long e = e0 + blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (e >= e1) return;
  const double nxt = next[e];
  if (!(nxt <= (double)epoch)) return;
  const int j = head[e], kk = tail[e];
  float cur[UMAP_MAX_DIM], oth[UMAP_MAX_DIM];
  volatile float* ve = emb;   // Hogwild: re-read what other threads wrote
  double d2 = 0.0;
  #pragma unroll
  for (int d = 0; d < UMAP_MAX_DIM; ++d) {
    if (d >= dim) break;
    cur[d] = ve[(long long)j * dim + d];
    oth[d] = ve[(long long)kk * dim + d];
    const double t = (double)cur[d] - (double)oth[d];
    d2 = __dadd_rn(d2, __dmul_rn(t, t));
  }
  double gc = 0.0;
  if (d2 > 0.0) gc = (-2.0 * a * b * pow(d2, b - 1.0)) / (a * pow(d2, b) + 1.0);
  #pragma unroll
  for (int d = 0; d < UMAP_MAX_DIM; ++d) {
    if (d >= dim) break;
    const double g = umap_clip(gc * ((double)cur[d] - (double)oth[d]));
    const float c_new = (float)__dadd_rn((double)cur[d], __dmul_rn(g, alpha));
    const float o_new = (float)__dadd_rn((double)oth[d], __dmul_rn(-g, alpha));
    cur[d] = c_new;
    oth[d] = o_new;
    ve[(long long)j * dim + d] = c_new;
    ve[(long long)kk * dim + d] = o_new;
  }
  next[e] = nxt + eps[e];
  const double en = eps_neg[e];
  const int n_neg = (int)(((double)epoch - next_neg[e]) / en);
  for (int p = 0; p < n_neg; ++p) {
    const int k = (int)(umap_hash(seed, (unsigned long long)epoch, (unsigned long long)e, (unsigned long long)p) %
                        (unsigned long long)N);
    if (k == j) continue;
    double s = 0.0;
    #pragma unroll
  for (int d = 0; d < UMAP_MAX_DIM; ++d) {
    if (d >= dim) break;
      oth[d] = ve[(long long)k * dim + d];
      const double t = (double)cur[d] - (double)oth[d];
      s = __dadd_rn(s, __dmul_rn(t, t));
    }
    double rc = 0.0;
    if (s > 0.0) rc = (2.0 * gamma * b) / ((0.001 + s) * (a * pow(s, b) + 1.0));
    #pragma unroll
  for (int d = 0; d < UMAP_MAX_DIM; ++d) {
    if (d >= dim) break;
      const double g = rc > 0.0 ? umap_clip(rc * ((double)cur[d] - (double)oth[d])) : 4.0;
      cur[d] = (float)__dadd_rn((double)cur[d], __dmul_rn(g, alpha));
      ve[(long long)j * dim + d] = cur[d];
    }
  }
  next_neg[e] = next_neg[e] + (double)n_neg * en;
}


// --------------------------------------------------------------------------------- transform
constexpr unsigned long long UMAP_S_TRANSFORM = 5ull << 32;   // stream tag of the transform's negative samples

// umap.umap_.init_graph_transform: one thread per query row over its k (column, weight) entries in column order.
// A weight of exactly 1 puts the row at that column's embedding; otherwise out += (w / row_sum) emb[col], the
// product in fp64 and each sum rounded to fp32, as numba evaluates the float32 += float64 expression.
__global__ void init_transform_kernel(const int* __restrict__ cols, const double* __restrict__ w, int Nq, int k,
                                      const float* __restrict__ emb, int dim, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Nq) return;
  const int* ci = cols + (long long)i * k;
  const double* wi = w + (long long)i * k;
  double row_sum = 0.0;
  for (int j = 0; j < k; ++j) row_sum = __dadd_rn(row_sum, wi[j]);
  float o[UMAP_MAX_DIM];
#pragma unroll
  for (int d = 0; d < UMAP_MAX_DIM; ++d) o[d] = 0.f;
  for (int j = 0; j < k; ++j) {
    const float* e = emb + (long long)ci[j] * dim;
    if (wi[j] == 1.0) {
#pragma unroll
      for (int d = 0; d < UMAP_MAX_DIM; ++d)
        if (d < dim) o[d] = e[d];
      break;
    }
    const double f = __ddiv_rn(wi[j], row_sum);
#pragma unroll
    for (int d = 0; d < UMAP_MAX_DIM; ++d)
      if (d < dim) o[d] = (float)__dadd_rn((double)o[d], __dmul_rn(f, (double)e[d]));
  }
#pragma unroll
  for (int d = 0; d < UMAP_MAX_DIM; ++d)
    if (d < dim) out[(long long)i * dim + d] = o[d];
}

// umap.layouts.optimize_layout_euclidean(move_other=False) for the transform, all epochs in one launch.  Every edge
// moves only its head, a query row, and reads only the fitted embedding, so one thread owns one query row: it keeps
// the row in registers and walks its own edges [rowptr[i], rowptr[i + 1]) epoch by epoch.  No two threads write the
// same memory, so the result is the sequential algorithm's and repeats bit for bit.  The arithmetic is
// sgd_epoch_kernel's, except that a negative sample is never skipped (it is drawn from the other set).
__global__ void sgd_transform_kernel(float* __restrict__ emb_q, int Nq, const float* __restrict__ emb, int N, int dim,
                                     const long long* __restrict__ rowptr, const int* __restrict__ tail,
                                     const double* __restrict__ eps, const double* __restrict__ eps_neg,
                                     double* __restrict__ next, double* __restrict__ next_neg, int n_epochs, double a,
                                     double b, double gamma, double alpha0, unsigned long long seed) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Nq) return;
  float cur[UMAP_MAX_DIM], oth[UMAP_MAX_DIM];
#pragma unroll
  for (int d = 0; d < UMAP_MAX_DIM; ++d) cur[d] = d < dim ? emb_q[(long long)i * dim + d] : 0.f;
  const long long p0 = rowptr[i], p1 = rowptr[i + 1];
  for (int n = 0; n < n_epochs; ++n) {
    const double alpha = alpha0 * (1.0 - (double)n / (double)n_epochs);
    for (long long e = p0; e < p1; ++e) {
      const double nxt = next[e];
      if (!(nxt <= (double)n)) continue;
      const float* te = emb + (long long)tail[e] * dim;
      double d2 = 0.0;
#pragma unroll
      for (int d = 0; d < UMAP_MAX_DIM; ++d) {
        if (d >= dim) break;
        oth[d] = __ldg(te + d);
        const double t = (double)cur[d] - (double)oth[d];
        d2 = __dadd_rn(d2, __dmul_rn(t, t));
      }
      double gc = 0.0;
      if (d2 > 0.0) gc = (-2.0 * a * b * pow(d2, b - 1.0)) / (a * pow(d2, b) + 1.0);
#pragma unroll
      for (int d = 0; d < UMAP_MAX_DIM; ++d) {
        if (d >= dim) break;
        const double g = umap_clip(gc * ((double)cur[d] - (double)oth[d]));
        cur[d] = (float)__dadd_rn((double)cur[d], __dmul_rn(g, alpha));
      }
      next[e] = nxt + eps[e];
      const double en = eps_neg[e];
      const double nn = next_neg[e];
      const int n_neg = (int)(((double)n - nn) / en);
      for (int p = 0; p < n_neg; ++p) {
        const int kk = (int)(umap_hash(seed, (unsigned long long)n, (unsigned long long)e, (unsigned long long)p) %
                             (unsigned long long)N);
        const float* ke = emb + (long long)kk * dim;
        double s = 0.0;
#pragma unroll
        for (int d = 0; d < UMAP_MAX_DIM; ++d) {
          if (d >= dim) break;
          oth[d] = __ldg(ke + d);
          const double t = (double)cur[d] - (double)oth[d];
          s = __dadd_rn(s, __dmul_rn(t, t));
        }
        double rc = 0.0;
        if (s > 0.0) rc = (2.0 * gamma * b) / ((0.001 + s) * (a * pow(s, b) + 1.0));
#pragma unroll
        for (int d = 0; d < UMAP_MAX_DIM; ++d) {
          if (d >= dim) break;
          const double g = rc > 0.0 ? umap_clip(rc * ((double)cur[d] - (double)oth[d])) : 4.0;
          cur[d] = (float)__dadd_rn((double)cur[d], __dmul_rn(g, alpha));
        }
      }
      next_neg[e] = nn + (double)n_neg * en;
    }
  }
#pragma unroll
  for (int d = 0; d < UMAP_MAX_DIM; ++d)
    if (d < dim) emb_q[(long long)i * dim + d] = cur[d];
}

}  // namespace ava

using namespace ava;

#define UMAP_STREAM cudaStream_t s = (cudaStream_t)stream

extern "C" long long ava_b200_umap_knn_ws_bytes(int N, int D, int k) {
  if (N < 1 || D < 1 || D > KNN_MAX_D || k < 1 || k > 100) return -1;
  const int KP = knn_padded(k);
  return knn_ws_layout(N, N, D, KP, knn_slices(N, N, KP), true, nullptr, nullptr);
}

extern "C" int ava_b200_umap_knn(const void* x, int is_f32, int N, int D, int k, int* knn_idx, double* knn_dist,
                                 void* ws, long long ws_bytes, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(x && knn_idx && knn_dist && ws, "umap_knn: null pointer");
  AVA_REQUIRE(N >= 1 && k >= 1 && k <= 100 && k <= N, "umap_knn: need 1 <= k <= min(N, 100), got N=%d k=%d", N, k);
  AVA_REQUIRE(D >= 1 && D <= 64, "umap_knn: D=%d outside 1..64", D);
  AVA_REQUIRE(is_f32 == 0 || is_f32 == 1, "umap_knn: is_f32 must be 0 or 1");
  AVA_REQUIRE(ws_bytes >= ava_b200_umap_knn_ws_bytes(N, D, k), "umap_knn: workspace too small");
  if (is_f32) return knn_run<float, true>((const float*)x, N, (const float*)x, N, D, k, knn_idx, knn_dist, ws, s);
  return knn_run<double, true>((const double*)x, N, (const double*)x, N, D, k, knn_idx, knn_dist, ws, s);
}

extern "C" int ava_b200_umap_smooth_knn(const int* knn_idx, const double* knn_dist, int N, int k,
                                        double local_connectivity, double* rho, double* sigma, double* weights,
                                        double* ws, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(knn_idx && knn_dist && rho && sigma && weights && ws, "umap_smooth_knn: null pointer");
  AVA_REQUIRE(N >= 1 && k >= 2, "umap_smooth_knn: need N >= 1 and k >= 2");
  AVA_REQUIRE(local_connectivity >= 0.0, "umap_smooth_knn: local_connectivity must be >= 0");
  mean_kernel<<<1, 1024, 0, s>>>(knn_dist, (long long)N * k, ws);
  if (check_launch("umap mean_kernel")) return 1;
  smooth_knn_kernel<false><<<(N + 127) / 128, 128, 0, s>>>(knn_idx, knn_dist, N, k, local_connectivity, ws, rho,
                                                           sigma, weights);
  return check_launch("umap smooth_knn_kernel");
}

extern "C" int ava_b200_umap_edge_keys(const int* knn_idx, int N, int k, long long* keys, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(knn_idx && keys && N >= 1 && k >= 1, "umap_edge_keys: bad arguments");
  const long long n = (long long)N * k;
  edge_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(knn_idx, N, k, keys);
  return check_launch("umap edge_keys_kernel");
}

extern "C" int ava_b200_umap_graph(const long long* keys, long long nnz, int N, const int* knn_idx,
                                   const double* weights, int k, int* rows, int* cols, double* vals,
                                   long long* rowptr, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(keys && knn_idx && weights && rows && cols && vals && rowptr, "umap_graph: null pointer");
  AVA_REQUIRE(N >= 1 && k >= 1 && nnz >= 0, "umap_graph: bad sizes");
  graph_weights_kernel<<<(unsigned)((nnz + 1 + 255) / 256), 256, 0, s>>>(keys, nnz, N, knn_idx, weights, k, rows,
                                                                       cols, vals, rowptr);
  return check_launch("umap graph_weights_kernel");
}

extern "C" int ava_b200_umap_epochs_per_sample(const double* vals, long long n, const double* vmax, int n_epochs,
                                               double negative_sample_rate, double* eps, double* eps_neg,
                                               double* next, double* next_neg, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(vals && vmax && eps && eps_neg && next && next_neg, "umap_epochs_per_sample: null pointer");
  AVA_REQUIRE(n >= 0 && n_epochs >= 1 && negative_sample_rate > 0.0, "umap_epochs_per_sample: bad arguments");
  if (n == 0) return 0;
  epochs_per_sample_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(vals, n, vmax, n_epochs, negative_sample_rate,
                                                                     eps, eps_neg, next, next_neg);
  return check_launch("umap epochs_per_sample_kernel");
}

extern "C" int ava_b200_umap_components_step(const long long* rowptr, const int* cols, int N, int* labels,
                                             int* changed, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(rowptr && cols && labels && changed && N >= 1, "umap_components_step: bad arguments");
  components_kernel<<<(N + 255) / 256, 256, 0, s>>>(rowptr, cols, N, labels, changed);
  return check_launch("umap components_kernel");
}

extern "C" int ava_b200_umap_degree(const long long* rowptr, const double* vals, int N, double* dis, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(rowptr && vals && dis && N >= 1, "umap_degree: bad arguments");
  degree_kernel<<<(N + 255) / 256, 256, 0, s>>>(rowptr, vals, N, dis);
  return check_launch("umap degree_kernel");
}

extern "C" int ava_b200_umap_spmm(const long long* rowptr, const int* cols, const double* vals, const int* verts,
                                  int n, const int* pos, const double* dis, const double* X, int m, double* Y,
                                  void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(rowptr && cols && vals && verts && pos && dis && X && Y, "umap_spmm: null pointer");
  AVA_REQUIRE(n >= 1 && m >= 1 && m <= 32, "umap_spmm: need n >= 1 and 1 <= m <= 32");
  constexpr int WARPS = 8;
  const unsigned grid = (unsigned)((n + WARPS - 1) / WARPS);
  if (m <= 8) spmm_kernel<8><<<grid, WARPS * 32, 0, s>>>(rowptr, cols, vals, verts, n, pos, dis, X, m, Y);
  else if (m <= 16) spmm_kernel<16><<<grid, WARPS * 32, 0, s>>>(rowptr, cols, vals, verts, n, pos, dis, X, m, Y);
  else spmm_kernel<32><<<grid, WARPS * 32, 0, s>>>(rowptr, cols, vals, verts, n, pos, dis, X, m, Y);
  return check_launch("umap spmm_kernel");
}

// p*q outputs over 8 accumulators per thread; GRAM_ROWS (p + q) doubles of staged rows within the 48 KB of
// shared memory a launch gets without opting in
constexpr int GRAM_MAX_PQ = 8 * GRAM_THREADS;
constexpr int GRAM_MAX_P_PLUS_Q = 48 * 1024 / (GRAM_ROWS * (int)sizeof(double));
static bool gram_shape_ok(int p, int q) {
  return p >= 1 && q >= 1 && p <= GRAM_MAX_PQ && q <= GRAM_MAX_PQ && p * q <= GRAM_MAX_PQ && p + q <= GRAM_MAX_P_PLUS_Q;
}

extern "C" long long ava_b200_umap_gram_ws_bytes(int p, int q) {
  if (!gram_shape_ok(p, q)) return -1;
  return (long long)GRAM_CTAS * p * q * (long long)sizeof(double);
}

extern "C" int ava_b200_umap_gram(const double* A, int p, const double* B, int q, int n, double* out, void* ws,
                                  long long ws_bytes, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(A && B && out && ws, "umap_gram: null pointer");
  AVA_REQUIRE(n >= 1 && gram_shape_ok(p, q), "umap_gram: need n >= 1, p, q >= 1, p*q <= %d and p + q <= %d, got "
              "n=%d p=%d q=%d", GRAM_MAX_PQ, GRAM_MAX_P_PLUS_Q, n, p, q);
  AVA_REQUIRE(ws_bytes >= ava_b200_umap_gram_ws_bytes(p, q), "umap_gram: workspace too small");
  const size_t smem = (size_t)GRAM_ROWS * (p + q) * sizeof(double);
  gram_kernel<<<GRAM_CTAS, GRAM_THREADS, smem, s>>>(A, p, B, q, n, (double*)ws);
  if (check_launch("umap gram_kernel")) return 1;
  gram_finish_kernel<<<(p * q + 255) / 256, 256, 0, s>>>((const double*)ws, p * q, GRAM_CTAS, out);
  return check_launch("umap gram_finish_kernel");
}

extern "C" int ava_b200_umap_combine(const double* A, int p, const double* C, int q, int n, double* Y, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(A && C && Y && n >= 1 && p >= 1 && q >= 1, "umap_combine: bad arguments");
  const long long t = (long long)n * q;
  combine_kernel<<<(unsigned)((t + 255) / 256), 256, 0, s>>>(A, p, C, q, n, Y);
  return check_launch("umap combine_kernel");
}

extern "C" int ava_b200_umap_random(unsigned long long seed, unsigned long long stream_id, long long n, int kind,
                                    double scale, double* out, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(out && n >= 0 && (kind == 0 || kind == 1), "umap_random: bad arguments");
  if (n == 0) return 0;
  random_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(seed, stream_id, n, kind, scale, out);
  return check_launch("umap random_kernel");
}

extern "C" int ava_b200_umap_init_layout(const double* init, const double* noise, double expansion, int N, int dim,
                                         float* emb, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(init && emb && N >= 1 && dim >= 1 && dim <= UMAP_MAX_DIM, "umap_init_layout: bad arguments");
  init_layout_kernel<<<dim, 1024, 0, s>>>(init, noise, expansion, N, dim, emb);
  return check_launch("umap init_layout_kernel");
}

extern "C" int ava_b200_umap_sgd_epoch(float* emb, int N, int dim, const int* head, const int* tail,
                                       const double* eps, const double* eps_neg, double* next, double* next_neg,
                                       long long e0, long long e1, int epoch, double a, double b, double gamma,
                                       double alpha, unsigned long long seed, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(emb && head && tail && eps && eps_neg && next && next_neg, "umap_sgd_epoch: null pointer");
  AVA_REQUIRE(N >= 1 && dim >= 1 && dim <= UMAP_MAX_DIM && e0 >= 0 && e1 >= e0 && epoch >= 0,
              "umap_sgd_epoch: bad arguments");
  if (e1 == e0) return 0;
  const long long n = e1 - e0;
  sgd_epoch_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(emb, N, dim, head, tail, eps, eps_neg, next, next_neg,
                                                             e0, e1, epoch, a, b, gamma, alpha, seed);
  return check_launch("umap sgd_epoch_kernel");
}

extern "C" long long ava_b200_umap_knn_query_ws_bytes(int Nq, int N, int D, int k) {
  if (Nq < 0 || N < 1 || D < 1 || D > KNN_MAX_D || k < 1 || k > 100) return -1;
  const KnnShape sh = knn_shape(Nq, N, D, k);
  return knn_ws_layout(Nq, N, D, sh.KP, sh.S, false, nullptr, nullptr);
}

extern "C" int ava_b200_umap_knn_query(const void* q, int Nq, const void* x, int N, int is_f32, int D, int k,
                                       int* knn_idx, double* knn_dist, void* ws, long long ws_bytes, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(x && ws && (Nq == 0 || (q && knn_idx && knn_dist)), "umap_knn_query: null pointer");
  AVA_REQUIRE(Nq >= 0 && N >= 1 && k >= 1 && k <= 100 && k <= N,
              "umap_knn_query: need Nq >= 0 and 1 <= k <= min(N, 100), got Nq=%d N=%d k=%d", Nq, N, k);
  AVA_REQUIRE(D >= 1 && D <= 64, "umap_knn_query: D=%d outside 1..64", D);
  AVA_REQUIRE(is_f32 == 0 || is_f32 == 1, "umap_knn_query: is_f32 must be 0 or 1");
  AVA_REQUIRE(ws_bytes >= ava_b200_umap_knn_query_ws_bytes(Nq, N, D, k), "umap_knn_query: workspace too small");
  if (Nq == 0) return 0;
  if (is_f32) return knn_run<float, false>((const float*)q, Nq, (const float*)x, N, D, k, knn_idx, knn_dist, ws, s);
  return knn_run<double, false>((const double*)q, Nq, (const double*)x, N, D, k, knn_idx, knn_dist, ws, s);
}

extern "C" int ava_b200_umap_smooth_knn_query(const int* knn_idx, const double* knn_dist, int Nq, int k,
                                              double local_connectivity, double* rho, double* sigma, double* weights,
                                              double* ws, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(knn_idx && knn_dist && rho && sigma && weights && ws, "umap_smooth_knn_query: null pointer");
  AVA_REQUIRE(Nq >= 1 && k >= 2, "umap_smooth_knn_query: need Nq >= 1 and k >= 2");
  AVA_REQUIRE(local_connectivity >= 0.0, "umap_smooth_knn_query: local_connectivity must be >= 0");
  mean_kernel<<<1, 1024, 0, s>>>(knn_dist, (long long)Nq * k, ws);
  if (check_launch("umap mean_kernel")) return 1;
  smooth_knn_kernel<true><<<(Nq + 127) / 128, 128, 0, s>>>(knn_idx, knn_dist, Nq, k,
                                                           std::max(0.0, local_connectivity - 1.0), ws, rho, sigma,
                                                           weights);
  return check_launch("umap smooth_knn_kernel (bipartite)");
}

extern "C" int ava_b200_umap_init_transform(const int* cols, const double* weights, int Nq, int k, const float* emb,
                                            int N, int dim, float* out, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(cols && weights && emb && out, "umap_init_transform: null pointer");
  AVA_REQUIRE(Nq >= 1 && k >= 1 && k <= N && dim >= 1 && dim <= UMAP_MAX_DIM, "umap_init_transform: bad arguments");
  init_transform_kernel<<<(Nq + 127) / 128, 128, 0, s>>>(cols, weights, Nq, k, emb, dim, out);
  return check_launch("umap init_transform_kernel");
}

extern "C" int ava_b200_umap_sgd_transform(float* emb_q, int Nq, const float* emb, int N, int dim,
                                           const long long* rowptr, const int* tail, const double* eps,
                                           const double* eps_neg, double* next, double* next_neg, int n_epochs,
                                           double a, double b, double gamma, double initial_alpha,
                                           unsigned long long seed, void* stream) {
  UMAP_STREAM;
  AVA_REQUIRE(emb_q && emb && rowptr && tail && eps && eps_neg && next && next_neg, "umap_sgd_transform: null pointer");
  AVA_REQUIRE(Nq >= 1 && N >= 1 && dim >= 1 && dim <= UMAP_MAX_DIM && n_epochs >= 0,
              "umap_sgd_transform: bad arguments");
  if (n_epochs == 0) return 0;
  sgd_transform_kernel<<<(Nq + 127) / 128, 128, 0, s>>>(emb_q, Nq, emb, N, dim, rowptr, tail, eps, eps_neg, next,
                                                        next_neg, n_epochs, a, b, gamma, initial_alpha,
                                                        umap_hash(seed, UMAP_S_TRANSFORM, 0, 0));
  return check_launch("umap sgd_transform_kernel");
}
