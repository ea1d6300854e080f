// Dense (torch.nn.Linear) layers: forward, backward-data, backward-weight.
//
// precision 0: fp32 SIMT GEMM (exact mode, also used for the small layers): 64x64x16
// tiles, 4x4 register micro-tiles, float4 global loads, deterministic split-K through a
// workspace so that M = batch 64 still fills 148 SMs.
// precision 1: tcgen05/TMEM GEMM (gemm_tc.cu) for the two 8192x1024 layers.
//
// Reference call sites: ava/models/vae.py:225-232 (fc1..fc43), 258-261 (fc5..fc8) and
// autograd's addmm backward for vae.py:352.
#include <stdlib.h>

#include "common.cuh"

namespace ava {

int tc_gemm_supported(int M, int N, int K);
long long tc_ws_bytes(int M, int N, int K);
int tc_gemm(const float* a, int lda, bool a_trans, const float* a_mask, const float* b, int ldb, bool b_trans,
            const float* bias, float* d, int ldd, int M, int N, int K, int act, int precision, void* ws,
            long long ws_bytes, cudaStream_t stream);

constexpr int BM = 64, BN = 64, BK = 16;

// C'(m,n) = sum_k A'(m,k) B'(k,n);  A'(m,k) = A[m*sam + k*sak], B'(k,n) = B[k*sbk + n*sbn]
struct GemmParams {
  const float* A;
  const float* Amask;  // optional, same indexing as A: A' = Amask>0 ? A : 0
  const float* B;
  float* C;            // direct output (splits == 1)
  float* part;         // split-K partials [groups*splits][M][N]
  const float* bias;   // per n (direct epilogue only)
  long long sam, sak, sbk, sbn;
  int ldc;
  int M, N, K;
  int act;
  int splits, kchunk;
  int groups;
  long long a_gs, b_gs, c_gs, bias_gs;
};

__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == 1) return fmaxf(v, 0.f);
  if (act == 2) return expf(v);
  return v;
}

// Load 4 consecutive elements (stride 1) starting at p, `valid` of them in range.
__device__ __forceinline__ float4 load4(const float* p, int valid) {
  if (valid >= 4 && ((uintptr_t)p & 15) == 0) return __ldg(reinterpret_cast<const float4*>(p));
  float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
  if (valid > 0) r.x = __ldg(p);
  if (valid > 1) r.y = __ldg(p + 1);
  if (valid > 2) r.z = __ldg(p + 2);
  if (valid > 3) r.w = __ldg(p + 3);
  return r;
}
__device__ __forceinline__ float4 mask4(float4 v, float4 m) {
  return make_float4(m.x > 0.f ? v.x : 0.f, m.y > 0.f ? v.y : 0.f, m.z > 0.f ? v.z : 0.f, m.w > 0.f ? v.w : 0.f);
}

// Tensor-core inner product for the same tiles (TERMS = 1: single-pass TF32): each 8-deep step
// on a zero accumulator, summed with round-to-nearest FADDs.
__device__ __forceinline__ void gm_mma_zero(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
      : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "f"(0.f));
}

// A_KCONTIG: A' contiguous along k (sak == 1) else along m (sam == 1)
// B_NCONTIG: B' contiguous along n (sbn == 1) else along k (sbk == 1)
// TERMS: 0 = fp32 FMA (4x4 register micro-tiles); 1 = tensor cores (mma.sync m16n8k8 TF32):
//   warp w owns rows 16*(w&3).. and columns 32*(w>>2).. of the 64x64 tile (4 n8 tiles); the
//   row pitch of the staged tiles is 72 floats (8 mod 32) so fragment loads are conflict-free.
template <bool A_KCONTIG, bool B_NCONTIG, bool MASK, int TERMS>
__device__ __forceinline__ void sgemm_body(const GemmParams& P, const int bx, const int by, const int bz) {
  constexpr int PAD = TERMS ? 8 : 4;
  __shared__ __align__(16) float As[2][BK][BM + PAD];
  __shared__ __align__(16) float Bs[2][BK][BN + PAD];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  // tensor-core thread coordinates
  const int lane = tid & 31, warp = tid >> 5;
  const int fg = lane >> 2, ft = lane & 3;
  const int wm0 = (warp & 3) * 16, wn0 = (warp >> 2) * 32;
  const int m0 = by * BM, n0 = bx * BN;
  const int grp = bz / P.splits, split = bz % P.splits;
  const float* A = P.A + (size_t)grp * P.a_gs;
  const float* Am = (MASK && P.Amask != nullptr) ? P.Amask + (size_t)grp * P.a_gs : nullptr;
  const float* B = P.B + (size_t)grp * P.b_gs;
  // split-K by INTERLEAVED 16-deep chunks: split s takes chunks s, s+splits, s+2*splits, ...  The
  // CTAs that share an output tile run concurrently and march through K together, so at any
  // moment they read adjacent 64-byte pieces of the same weight rows (one DRAM page) instead of
  // `splits` streams 1.7 KB apart per row (measured at batch 64: see DESIGN.md 3.3).
  const int k_end = P.K;
  const int total_chunks = (P.K + BK - 1) / BK;
  const int nk = total_chunks > split ? (total_chunks - split + P.splits - 1) / P.splits : 0;
  // (starting each tile's walk at a different chunk, to spread concurrent CTAs over the DRAM
  // channels, was measured too: no effect -- the kernel is issue bound, see pick_splits)
  auto chunk_k = [&](int j) { return (split + j * P.splits) * BK; };

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  // two register sets: chunk c+1 and c+2 are in flight while chunk c is being multiplied
  float4 ra0, rb0, ra1, rb1;
  auto gload = [&](int k0, float4& ra, float4& rb) {
    if (A_KCONTIG) {
      int m = m0 + (tid >> 2), k = k0 + (tid & 3) * 4;
      int valid = (m < P.M) ? (k_end - k) : 0;
      const float* p = A + (size_t)m * P.sam + k;
      ra = load4(p, valid);
      if (MASK && Am != nullptr) ra = mask4(ra, load4(Am + (size_t)m * P.sam + k, valid));
    } else {
      int k = k0 + (tid >> 4), m = m0 + (tid & 15) * 4;
      int valid = (k < k_end) ? (P.M - m) : 0;
      const float* p = A + (size_t)k * P.sak + m;
      ra = load4(p, valid);
      if (MASK && Am != nullptr) ra = mask4(ra, load4(Am + (size_t)k * P.sak + m, valid));
    }
    if (B_NCONTIG) {
      int k = k0 + (tid >> 4), n = n0 + (tid & 15) * 4;
      int valid = (k < k_end) ? (P.N - n) : 0;
      rb = load4(B + (size_t)k * P.sbk + n, valid);
    } else {
      int n = n0 + (tid >> 2), k = k0 + (tid & 3) * 4;
      int valid = (n < P.N) ? (k_end - k) : 0;
      rb = load4(B + (size_t)n * P.sbn + k, valid);
    }
  };
  auto sstore = [&](int buf, const float4& ra, const float4& rb) {
    if (A_KCONTIG) {
      int m = tid >> 2, k = (tid & 3) * 4;
      As[buf][k + 0][m] = ra.x;
      As[buf][k + 1][m] = ra.y;
      As[buf][k + 2][m] = ra.z;
      As[buf][k + 3][m] = ra.w;
    } else {
      int k = tid >> 4, m = (tid & 15) * 4;
      *reinterpret_cast<float4*>(&As[buf][k][m]) = ra;
    }
    if (B_NCONTIG) {
      int k = tid >> 4, n = (tid & 15) * 4;
      *reinterpret_cast<float4*>(&Bs[buf][k][n]) = rb;
    } else {
      int n = tid >> 2, k = (tid & 3) * 4;
      Bs[buf][k + 0][n] = rb.x;
      Bs[buf][k + 1][n] = rb.y;
      Bs[buf][k + 2][n] = rb.z;
      Bs[buf][k + 3][n] = rb.w;
    }
  };

  auto compute = [&](int buf) {
    if constexpr (TERMS == 0) {
#pragma unroll
      for (int k = 0; k < BK; ++k) {
        float4 a = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
        float4 b = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
        const float av[4] = {a.x, a.y, a.z, a.w};
        const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
      }
    } else {
      // acc[nt][0..3] = C fragment of n8-tile nt: rows fg / fg+8, columns 2*ft / 2*ft+1.
      // The tensor core adds into a non-zero accumulator with truncation, so every product
      // block starts from a zero accumulator and is added to the running sum with a
      // round-to-nearest FADD.
#pragma unroll
      for (int ks = 0; ks < BK / 8; ++ks) {
        const int k0 = ks * 8;
        const float av[4] = {As[buf][k0 + ft][wm0 + fg], As[buf][k0 + ft][wm0 + fg + 8],
                             As[buf][k0 + ft + 4][wm0 + fg], As[buf][k0 + ft + 4][wm0 + fg + 8]};
        uint32_t ah[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) ah[j] = __float_as_uint(av[j]);
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const float b0 = Bs[buf][k0 + ft][wn0 + nt * 8 + fg], b1 = Bs[buf][k0 + ft + 4][wn0 + nt * 8 + fg];
          float cf[4];
          gm_mma_zero(cf, ah, __float_as_uint(b0), __float_as_uint(b1));
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[nt][j] += cf[j];
        }
      }
    }
  };
  if (nk > 0) {
    gload(chunk_k(0), ra0, rb0);
    sstore(0, ra0, rb0);
  }
  if (nk > 1) gload(chunk_k(1), ra0, rb0);
  if (nk > 2) gload(chunk_k(2), ra1, rb1);
  __syncthreads();
  for (int it = 0; it < nk; it += 2) {
    // chunk `it` (buffer 0); chunk it+1 waits in register set 0
    compute(0);
    if (it + 1 < nk) sstore(1, ra0, rb0);
    if (it + 3 < nk) gload(chunk_k(it + 3), ra0, rb0);
    __syncthreads();
    if (it + 1 >= nk) break;
    // chunk it+1 (buffer 1); chunk it+2 waits in register set 1
    compute(1);
    if (it + 2 < nk) sstore(0, ra1, rb1);
    if (it + 4 < nk) gload(chunk_k(it + 4), ra1, rb1);
    __syncthreads();
  }

  // element (i, j) of this thread's 16 accumulators -> (row, column) of the tile
  auto row_of = [&](int i, int j) { return TERMS ? wm0 + fg + 8 * (j >> 1) : ty * 4 + i; };
  auto col_of = [&](int i, int j) { return TERMS ? wn0 + i * 8 + 2 * ft + (j & 1) : tx * 4 + j; };
  if (P.splits == 1) {
    float* C = P.C + (size_t)grp * P.c_gs;
    const float* bias = P.bias ? P.bias + (size_t)grp * P.bias_gs : nullptr;
    if constexpr (TERMS == 0) {
      // a thread's 4 consecutive columns go out as one 16-byte store when the row allows it
      const int n = n0 + tx * 4;
      const bool vec = (n + 3 < P.N) && ((P.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= P.M) continue;
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
          v[j] = apply_act(acc[i][j] + ((bias && n + j < P.N) ? bias[n + j] : 0.f), P.act);
        if (vec) {
          *reinterpret_cast<float4*>(&C[(size_t)m * P.ldc + n]) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (n + j < P.N) C[(size_t)m * P.ldc + n + j] = v[j];
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int m = m0 + row_of(i, j), n = n0 + col_of(i, j);
          if (m >= P.M || n >= P.N) continue;
          float v = acc[i][j] + (bias ? bias[n] : 0.f);
          C[(size_t)m * P.ldc + n] = apply_act(v, P.act);
        }
      }
    }
  } else {
    float* part = P.part + (size_t)bz * P.M * P.N;
    if constexpr (TERMS == 0) {
      const int n = n0 + tx * 4;
      const bool vec = (n + 3 < P.N) && ((P.N & 3) == 0) && ((reinterpret_cast<uintptr_t>(part) & 15) == 0);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= P.M) continue;
        if (vec) {
          *reinterpret_cast<float4*>(&part[(size_t)m * P.N + n]) =
              make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (n + j < P.N) part[(size_t)m * P.N + n + j] = acc[i][j];
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int m = m0 + row_of(i, j), n = n0 + col_of(i, j);
          if (m < P.M && n < P.N) part[(size_t)m * P.N + n] = acc[i][j];
        }
      }
    }
  }
}

template <bool A_KCONTIG, bool B_NCONTIG, bool MASK, int TERMS>
__global__ void __launch_bounds__(256, 4) sgemm_kernel(const GemmParams P) {
  sgemm_body<A_KCONTIG, B_NCONTIG, MASK, TERMS>(P, blockIdx.x, blockIdx.y, blockIdx.z);
}

__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const float* part, int splits, int groups, int M, int N, const float* bias, long long bias_gs,
                     float* C, int ldc, long long c_gs, int act) {
  const long long total = (long long)groups * M * N;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int n = (int)(i % N);
    long long r = i / N;
    int m = (int)(r % M);
    int g = (int)(r / M);
    float s = 0.f;
    for (int sp = 0; sp < splits; ++sp) s += part[((size_t)(g * splits + sp) * M + m) * N + n];
    if (bias) s += bias[(size_t)g * bias_gs + n];
    C[(size_t)g * c_gs + (size_t)m * ldc + n] = apply_act(s, act);
  }
}

// db[n] = sum_m (mask>0 ? dy : 0)[m, n].  grid (ceil(N/32), row splits): each block sums its
// slice of rows for 32 columns; with more than one split the per-split sums go to `part`
// [splits][N] and colsum_finish_kernel adds them in a fixed order (deterministic).
__global__ void __launch_bounds__(256)
colsum_kernel(const float* __restrict__ dy, const float* __restrict__ mask, int ld, int M, int N, int rows_per_split,
              float* __restrict__ out) {
  __shared__ float s[8][33];
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int r = threadIdx.x >> 5;
  const int m0 = blockIdx.y * rows_per_split;
  const int m1 = min(M, m0 + rows_per_split);
  float acc = 0.f;
  if (n < N) {
    for (int m = m0 + r; m < m1; m += 8) {
      float v = dy[(size_t)m * ld + n];
      if (mask && !(mask[(size_t)m * ld + n] > 0.f)) v = 0.f;
      acc += v;
    }
  }
  s[r][threadIdx.x & 31] = acc;
  __syncthreads();
  if (r == 0 && n < N) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += s[i][threadIdx.x];
    out[(size_t)blockIdx.y * N + n] = t;
  }
}
__global__ void colsum_finish_kernel(const float* __restrict__ part, int splits, int N, float* __restrict__ db) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float t = 0.f;
  for (int sp = 0; sp < splits; ++sp) t += part[(size_t)sp * N + n];
  db[n] = t;
}

static int launch_colsum(const float* dy, const float* mask, int ld, int M, int N, float* db, void* ws,
                         long long ws_bytes, cudaStream_t stream) {
  int splits = 1;
  const int col_blocks = (N + 31) / 32;
  while (col_blocks * splits < 2 * kNumSMs && M / (splits * 2) >= 64) splits *= 2;
  if (ws == nullptr || ws_bytes < (long long)splits * N * 4) splits = 1;
  const int rows = (M + splits - 1) / splits;
  float* out = splits > 1 ? reinterpret_cast<float*>(ws) : db;
  colsum_kernel<<<dim3(col_blocks, splits), 256, 0, stream>>>(dy, mask, ld, M, N, rows, out);
  if (check_launch("colsum")) return 1;
  if (splits > 1) {
    colsum_finish_kernel<<<(N + 255) / 256, 256, 0, stream>>>(out, splits, N, db);
    return check_launch("colsum_finish");
  }
  return 0;
}

// Bias gradients of several Linear layers in two launches (instead of two per layer): job j is
// db_j[n] = sum_m (mask_j > 0 ? dy_j : 0)[m, n].  The grid is the concatenation of the jobs' (column
// block, row split) tiles; per-split sums go to the workspace, the finish kernel adds them in a
// fixed order (deterministic).
struct BiasJobs {
  const float* dy[AVA_MAX_BIAS_JOBS];
  const float* mask[AVA_MAX_BIAS_JOBS];
  float* db[AVA_MAX_BIAS_JOBS];
  int ld[AVA_MAX_BIAS_JOBS], M[AVA_MAX_BIAS_JOBS], N[AVA_MAX_BIAS_JOBS];
  int splits[AVA_MAX_BIAS_JOBS], rows[AVA_MAX_BIAS_JOBS];
  int blk0[AVA_MAX_BIAS_JOBS + 1];    // first CTA of job j (kernel 1)
  int col0[AVA_MAX_BIAS_JOBS + 1];    // first column of job j in the concatenated partial rows
  int n;
};

__global__ void __launch_bounds__(256) bias_partial_kernel(const BiasJobs J, float* __restrict__ part) {
  __shared__ float s[8][33];
  int j = 0;
  while (j + 1 < J.n && (int)blockIdx.x >= J.blk0[j + 1]) ++j;
  const int local = blockIdx.x - J.blk0[j];
  const int col_blocks = (J.N[j] + 31) / 32;
  const int cb = local % col_blocks, sp = local / col_blocks;
  const int n = cb * 32 + (threadIdx.x & 31);
  const int r = threadIdx.x >> 5;
  const int m0 = sp * J.rows[j];
  const int m1 = min(J.M[j], m0 + J.rows[j]);
  const float* dy = J.dy[j];
  const float* mask = J.mask[j];
  const int ld = J.ld[j];
  float acc = 0.f;
  if (n < J.N[j]) {
    // 4 rows in flight per thread (the loop is otherwise one dependent load after another)
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int m = m0 + r;
    for (; m + 24 < m1; m += 32) {
      float v0 = dy[(size_t)m * ld + n], v1 = dy[(size_t)(m + 8) * ld + n];
      float v2 = dy[(size_t)(m + 16) * ld + n], v3 = dy[(size_t)(m + 24) * ld + n];
      if (mask) {
        const float k0 = mask[(size_t)m * ld + n], k1 = mask[(size_t)(m + 8) * ld + n];
        const float k2 = mask[(size_t)(m + 16) * ld + n], k3 = mask[(size_t)(m + 24) * ld + n];
        if (!(k0 > 0.f)) v0 = 0.f;
        if (!(k1 > 0.f)) v1 = 0.f;
        if (!(k2 > 0.f)) v2 = 0.f;
        if (!(k3 > 0.f)) v3 = 0.f;
      }
      a0 += v0;
      a1 += v1;
      a2 += v2;
      a3 += v3;
    }
    for (; m < m1; m += 8) {
      float v = dy[(size_t)m * ld + n];
      if (mask && !(mask[(size_t)m * ld + n] > 0.f)) v = 0.f;
      a0 += v;
    }
    acc = (a0 + a1) + (a2 + a3);
  }
  s[r][threadIdx.x & 31] = acc;
  __syncthreads();
  if (r == 0 && n < J.N[j]) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += s[i][threadIdx.x];
    // partial layout: job j owns columns [col0[j], col0[j+1]) of up to 64 rows (splits)
    part[(size_t)sp * J.col0[J.n] + J.col0[j] + n] = t;
  }
}
__global__ void __launch_bounds__(256) bias_finish_kernel(const BiasJobs J, const float* __restrict__ part) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= J.col0[J.n]) return;
  int j = 0;
  while (j + 1 < J.n && c >= J.col0[j + 1]) ++j;
  float t = 0.f;
  for (int sp = 0; sp < J.splits[j]; ++sp) t += part[(size_t)sp * J.col0[J.n] + c];
  J.db[j][c - J.col0[j]] = t;
}

void launch_splitk_reduce(const float* part, int splits, int M, int N, const float* bias, float* C, int ldc, int act,
                          cudaStream_t stream) {
  long long total = (long long)M * N;
  int g = (int)((total + 255) / 256);
  if (g > 8 * kNumSMs) g = 8 * kNumSMs;
  splitk_reduce_kernel<<<g, 256, 0, stream>>>(part, splits, 1, M, N, bias, 0, C, ldc, 0, act);
  check_launch("splitk_reduce");
}

// Split-K factor.  ncu of the fc1 forward at batch 64 (profiles/r01_ncu_sgemm_b64.txt): with 16 x 19 =
// 304 CTAs the kernel is FMA-issue bound at 64 % issue activity with only 4 warps per scheduler,
// and 304 CTAs over 148 SMs leave some SMs with 3 CTAs and most with 2 (the slowest SM sets the
// time).  So: as many CTAs as are resident at once (4 per SM at <= 64 registers), never more.
static int pick_splits(int M, int N, int K, int groups) {
  long long tiles = (long long)((M + BM - 1) / BM) * ((N + BN - 1) / BN) * groups;
  int splits = 1;
  if (tiles < 2 * kNumSMs) {
    splits = (int)((4 * kNumSMs) / tiles);
    if (splits < 1) splits = 1;
    int maxs = K / 128;  // at least 128 of K per split
    if (maxs < 1) maxs = 1;
    if (splits > maxs) splits = maxs;
    if (splits > 64) splits = 64;
  }
  return splits;
}

static long long ws_need(int M, int N, int K, int groups) {
  int s = pick_splits(M, N, K, groups);
  return s > 1 ? (long long)s * groups * M * N * (long long)sizeof(float) : 0;
}

static int run_gemm(GemmParams P, int a_kcontig, int b_ncontig, void* ws, long long ws_bytes,
                    cudaStream_t stream, int terms = 0) {
  if (P.M <= 0 || P.N <= 0) return 0;
  P.splits = pick_splits(P.M, P.N, P.K, P.groups);
  if (P.splits > 1 && (ws == nullptr || ws_bytes < ws_need(P.M, P.N, P.K, P.groups))) P.splits = 1;
  int kc = (P.K + P.splits - 1) / P.splits;
  kc = (kc + BK - 1) / BK * BK;
  P.kchunk = kc;
  P.splits = (P.K + kc - 1) / kc;
  P.part = reinterpret_cast<float*>(ws);
  dim3 grid((P.N + BN - 1) / BN, (P.M + BM - 1) / BM, P.groups * P.splits);
  const bool mask = P.Amask != nullptr;
#define AVA_GEMM_LAUNCH(AK, BNC, MK)                                                  \
  do {                                                                                \
    if (terms == 1)                                                                   \
      sgemm_kernel<AK, BNC, MK, 1><<<grid, 256, 0, stream>>>(P);                      \
    else                                                                              \
      sgemm_kernel<AK, BNC, MK, 0><<<grid, 256, 0, stream>>>(P);                      \
  } while (0)
#define AVA_GEMM_CASE(AK, BNC)                                                        \
  if (a_kcontig == AK && b_ncontig == BNC) {                                          \
    if (mask)                                                                         \
      AVA_GEMM_LAUNCH(AK, BNC, true);                                                 \
    else                                                                              \
      AVA_GEMM_LAUNCH(AK, BNC, false);                                                \
  }
  AVA_GEMM_CASE(true, true)
  AVA_GEMM_CASE(true, false)
  AVA_GEMM_CASE(false, true)
  AVA_GEMM_CASE(false, false)
#undef AVA_GEMM_CASE
#undef AVA_GEMM_LAUNCH
  if (check_launch("sgemm")) return 1;
  if (P.splits > 1) {
    long long total = (long long)P.groups * P.M * P.N;
    int g = (int)((total + 255) / 256);
    if (g > 8 * kNumSMs) g = 8 * kNumSMs;
    splitk_reduce_kernel<<<g, 256, 0, stream>>>(P.part, P.splits, P.groups, P.M, P.N, P.bias, P.bias_gs, P.C,
                                                P.ldc, P.c_gs, P.act);
    return check_launch("splitk_reduce");
  }
  return 0;
}

// Shapes the tcgen05 kernel does not tile (batch not a multiple of 128), layers large enough
// for it to matter (>= 256 K weights): the same 64x64x16 kernel with its inner product on the
// tensor cores (mma.sync) --
//   precision 1 ('tf32'): single TF32 term;
//   precision 2 ('tf32x3'/'auto'): stays on the fp32 FMA inner product.  A 3-term (3xTF32)
//   mma.sync inner product was measured as accurate (fc1 shape, batch 64: 4.6e-8 rms / no bias
//   vs 6.3e-8 for FMA) but no faster: at batch 64 these GEMMs are bound by the weight stream,
//   not by the inner product.
static int mma_terms(int precision, int groups, int M, int N, int K) {
  (void)M;
  if (precision != 1 || groups != 1 || (long long)N * K < (1 << 18)) return 0;
  return 1;
}

}  // namespace ava

using namespace ava;

extern "C" long long ava_b200_linear_ws_bytes(int M, int N, int K) {
  long long a = ws_need(M, N, K, 1), b = ws_need(M, K, N, 1), c = ws_need(N, K, M, 1);
  long long m = a > b ? a : b;
  m = m > c ? m : c;
  // tensor-core path: TF32 hi/lo copies of both operands + split-K partials
  if (tc_gemm_supported(M, N, K)) m = m > tc_ws_bytes(M, N, K) ? m : tc_ws_bytes(M, N, K);
  if (tc_gemm_supported(M, K, N)) m = m > tc_ws_bytes(M, K, N) ? m : tc_ws_bytes(M, K, N);
  if (tc_gemm_supported(N, K, M)) m = m > tc_ws_bytes(N, K, M) ? m : tc_ws_bytes(N, K, M);
  return m + 256;
}

extern "C" int ava_b200_linear_fwd(const float* x, int ldx, const float* w, const float* b, float* y, int ldy,
                                   int M, int N, int K, int act, int groups, long long x_gs, long long w_gs,
                                   long long b_gs, long long y_gs, int precision, void* ws, long long ws_bytes,
                                   void* stream) {
  AVA_REQUIRE(groups >= 1 && act >= 0 && act <= 2, "linear_fwd: bad groups/act");
  // tensor cores when asked for and the shape tiles (else the exact SIMT kernel below)
  if (precision >= 1 && groups == 1 && tc_gemm_supported(M, N, K))
    return tc_gemm(x, ldx, false, nullptr, w, K, false, b, y, ldy, M, N, K, act, precision, ws, ws_bytes,
                   (cudaStream_t)stream);
  GemmParams P = {};
  P.A = x; P.sam = ldx; P.sak = 1;
  P.B = w; P.sbk = 1; P.sbn = K;  // B'(k,n) = W[n*K + k]
  P.C = y; P.ldc = ldy; P.bias = b;
  P.M = M; P.N = N; P.K = K; P.act = act;
  P.groups = groups; P.a_gs = x_gs; P.b_gs = w_gs; P.c_gs = y_gs; P.bias_gs = b_gs;
  return run_gemm(P, 1, 0, ws, ws_bytes, (cudaStream_t)stream, mma_terms(precision, groups, M, N, K));
}

extern "C" int ava_b200_linear_bwd_data(const float* dy, int lddy, const float* ymask, const float* w, float* dx,
                                        int lddx, int M, int N, int K, int groups, long long dy_gs,
                                        long long w_gs, long long dx_gs, int accumulate, int precision, void* ws,
                                        long long ws_bytes, void* stream) {
  AVA_REQUIRE(accumulate == 0, "linear_bwd_data: accumulate not supported");
  // dX[M,K] = dY[M,N] . W[N,K]  -> gemm (M, K, N); W is stored [N,K] = [contraction, out]
  if (precision >= 1 && groups == 1 && tc_gemm_supported(M, K, N))
    return tc_gemm(dy, lddy, false, ymask, w, K, true, nullptr, dx, lddx, M, K, N, 0, precision, ws, ws_bytes,
                   (cudaStream_t)stream);
  GemmParams P = {};
  P.A = dy; P.Amask = ymask; P.sam = lddy; P.sak = 1;
  P.B = w; P.sbk = K; P.sbn = 1;
  P.C = dx; P.ldc = lddx;
  P.M = M; P.N = K; P.K = N; P.act = 0;
  P.groups = groups; P.a_gs = dy_gs; P.b_gs = w_gs; P.c_gs = dx_gs;
  return run_gemm(P, 1, 1, ws, ws_bytes, (cudaStream_t)stream, mma_terms(precision, groups, M, N, K));
}

extern "C" int ava_b200_linear_bwd_weight(const float* dy, int lddy, const float* ymask, const float* x, int ldx,
                                          float* dw, float* db, int M, int N, int K, int groups, long long dy_gs,
                                          long long x_gs, long long dw_gs, long long db_gs, int precision,
                                          void* ws, long long ws_bytes, void* stream) {
  // dW[N,K] = dY^T[N,M] . X[M,K] -> gemm (N, K, M); A'(n,m) = dY[m*lddy + n]
  if (precision >= 1 && groups == 1 && tc_gemm_supported(N, K, M)) {
    if (tc_gemm(dy, lddy, true, ymask, x, ldx, true, nullptr, dw, K, N, K, M, 0, precision, ws, ws_bytes,
                (cudaStream_t)stream))
      return 1;
  } else {
    GemmParams P = {};
    P.A = dy; P.Amask = ymask; P.sam = 1; P.sak = lddy;
    P.B = x; P.sbk = ldx; P.sbn = 1;
    P.C = dw; P.ldc = K;
    P.M = N; P.N = K; P.K = M; P.act = 0;
    P.groups = groups; P.a_gs = dy_gs; P.b_gs = x_gs; P.c_gs = dw_gs;
    if (run_gemm(P, 0, 1, ws, ws_bytes, (cudaStream_t)stream, mma_terms(precision, groups, M, N, K))) return 1;
  }
  if (db) {
    for (int g = 0; g < groups; ++g) {
      if (launch_colsum(dy + (size_t)g * dy_gs, ymask ? ymask + (size_t)g * dy_gs : nullptr, lddy, M, N,
                        db + (size_t)g * db_gs, ws, ws_bytes, (cudaStream_t)stream))
        return 1;
    }
  }
  return 0;
}

extern "C" long long ava_b200_bias_grads_ws_bytes(const ava_b200_bias_job* h_jobs, int njobs) {
  long long cols = 0;
  for (int j = 0; j < njobs; ++j) cols += h_jobs[j].N;
  return 64 * cols * (long long)sizeof(float);
}

extern "C" int ava_b200_bias_grads(const ava_b200_bias_job* h_jobs, int njobs, void* ws, long long ws_bytes,
                                   void* stream_) {
  AVA_REQUIRE(h_jobs != nullptr && njobs >= 1 && njobs <= AVA_MAX_BIAS_JOBS, "bias_grads: 1..%d jobs", AVA_MAX_BIAS_JOBS);
  AVA_REQUIRE(ws != nullptr && ws_bytes >= ava_b200_bias_grads_ws_bytes(h_jobs, njobs), "bias_grads: workspace too small");
  BiasJobs J = {};
  J.n = njobs;
  int blk = 0, col = 0;
  for (int j = 0; j < njobs; ++j) {
    const ava_b200_bias_job& h = h_jobs[j];
    AVA_REQUIRE(h.dy && h.db && h.M > 0 && h.N > 0 && h.ld >= h.N, "bias_grads: bad job %d", j);
    J.dy[j] = h.dy;
    J.mask[j] = h.mask;
    J.db[j] = h.db;
    J.ld[j] = h.ld;
    J.M[j] = h.M;
    J.N[j] = h.N;
    const int col_blocks = (h.N + 31) / 32;
    int splits = 1;
    while (col_blocks * splits < 8 * kNumSMs && h.M / (splits * 2) >= 32 && splits < 64) splits *= 2;
    J.splits[j] = splits;
    J.rows[j] = (h.M + splits - 1) / splits;
    J.blk0[j] = blk;
    J.col0[j] = col;
    blk += col_blocks * splits;
    col += h.N;
  }
  J.blk0[njobs] = blk;
  J.col0[njobs] = col;
  cudaStream_t stream = (cudaStream_t)stream_;
  bias_partial_kernel<<<blk, 256, 0, stream>>>(J, reinterpret_cast<float*>(ws));
  if (check_launch("bias_partial")) return 1;
  bias_finish_kernel<<<(col + 255) / 256, 256, 0, stream>>>(J, reinterpret_cast<const float*>(ws));
  return check_launch("bias_finish");
}
