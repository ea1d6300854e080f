// Data-parallel optimizer step fused with its two collectives over NVLink / NVSwitch peer memory.
//
// Replaces, for one-process-per-GPU training (SURVEY section 5), the sequence
//     NCCL all-reduce(SUM) of the flat gradient buffer  ->  Adam on every rank
// (the data-parallel form of optimizer.step(), ava/models/vae.py:353) by ONE kernel per rank:
//
//   phase 0  cross-GPU barrier: "my backward pass is done, my gradient buffer is final"
//   phase 1  rank r owns the r-th 1/world slice of the flat buffers.  For its slice it
//              * reads the gradient of every rank (plain peer loads over NVLink, or ONE
//                multimem.ld_reduce: the NVSwitch adds the world copies in the fabric),
//              * applies the Adam update (the same arithmetic as adam_kernel, adam.cu) to its
//                slice of the parameters and of the two moment buffers -- the moments of the
//                other slices are never touched on this rank (optimizer state is sharded, ZeRO-1),
//              * writes the new parameters into EVERY rank's parameter buffer (peer stores, or one
//                multimem.st broadcast through the switch).
//   phase 2  cross-GPU barrier: "all my parameter stores have landed"; the kernel does not retire
//            before every peer has said so, so the next forward pass reads complete parameters.
//
// Per rank and step this moves 2 x (world-1)/world x 70 MB over NVLink (2 x 70/world MB with
// multimem) instead of the ring all-reduce's 2 x (world-1)/world x 70 MB PLUS a full 488 MB Adam
// pass on every rank, and it takes no SMs away from the backward pass (the NCCL kernels of an
// overlapped all-reduce displace CTAs of the persistent conv kernels).  Every parameter element
// is computed by exactly one rank and broadcast, so the replicas stay bit-identical.
//
// The buffers live in symmetric memory (torch.distributed._symmetric_memory: the same virtual
// layout on every rank, peer-mapped); the caller passes the table of peer pointers.  Flags are
// monotonically increasing step sequence numbers: nothing is ever reset, so a late rank cannot
// confuse two steps.  Every spin is bounded (kDpTimeoutNs); on timeout the kernel records it in
// local[2] and carries on -- a missing peer turns into a reported error, not a hung GPU.
#include "common.cuh"

namespace ava {

struct DpPeers {
  const float* grad[AVA_DP_MAX_WORLD];
  float* param[AVA_DP_MAX_WORLD];
  unsigned int* flags[AVA_DP_MAX_WORLD];
  const float* grad_mc;   // multicast (NVLS) views of the same buffers, or nullptr
  float* param_mc;
};

__device__ __forceinline__ float4 dp_ld_peer(const float* p) {
  float4 v;
  // (strong system-scope accesses throughout: weak ones measured no faster -- 156 vs 155 us at 2
  // GPUs -- and the multimem variant then drifted from the NCCL result beyond summation-order noise)
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
__device__ __forceinline__ void dp_st_peer(float* p, const float4& v) {
  asm volatile("st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}
__device__ __forceinline__ float4 dp_ld_reduce_mc(const float* p) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
__device__ __forceinline__ void dp_st_mc(float* p, const float4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}

// local: [0] sequence number of the last completed step, [1] CTA arrival counter, [2] timeout flag
template <bool MC>
__global__ void __launch_bounds__(256)
adam_dp_kernel(const DpPeers P, const int rank, const int world, float* __restrict__ m, float* __restrict__ v,
               const long long n4, const float* step_count, const double* __restrict__ hyper, const float gscale,
               unsigned int* local) {
  __shared__ int s_last;
  const int tid = threadIdx.x;
  const unsigned int seq = local[0] + 1u;
  unsigned int* my_flags = P.flags[rank];

  // ---- phase 0: every rank's gradient buffer is final (they were written by earlier kernels of
  // each rank's stream; the release / acquire pair on the flag makes them visible here)
  if (blockIdx.x == 0 && tid < world) {
    __threadfence_system();
    dp_signal(P.flags[tid] + rank, seq);
  }
  if (tid < world) dp_wait(my_flags + tid, seq, local + 2);
  __syncthreads();

  const AdamCoef k = adam_coef(hyper[0], hyper[1], hyper[2], hyper[3], (double)step_count[0] + 1.0);

  // ---- phase 1: this rank's slice (float4 units), U float4 per thread and trip with every
  // gradient load of the trip issued before the first is used (an NVLink / NVSwitch round trip is
  // several microseconds: the kernel lives on memory-level parallelism)
  constexpr int U = 4;
  const long long lo = n4 * rank / world, hi = n4 * (rank + 1) / world;
  float* p_own = P.param[rank];
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i0 = lo + (long long)blockIdx.x * blockDim.x + tid; i0 < hi; i0 += U * stride) {
    float4 gv[U], pv[U], mv[U], vv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = i0 + u * stride;
      if (i < hi) {
        if (MC) {
          gv[u] = dp_ld_reduce_mc(P.grad_mc + 4 * i);
        } else {
          gv[u] = dp_ld_peer(P.grad[0] + 4 * i);
        }
      }
    }
    if (!MC) {
      // fixed order 0..world-1: the sum does not depend on which rank owns the slice
      for (int r = 1; r < world; ++r) {
        float4 a[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const long long i = i0 + u * stride;
          if (i < hi) a[u] = dp_ld_peer(P.grad[r] + 4 * i);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const long long i = i0 + u * stride;
          if (i < hi) {
            gv[u].x += a[u].x;
            gv[u].y += a[u].y;
            gv[u].z += a[u].z;
            gv[u].w += a[u].w;
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = i0 + u * stride;
      if (i < hi) {
        pv[u] = reinterpret_cast<const float4*>(p_own)[i];
        mv[u] = reinterpret_cast<float4*>(m)[i];
        vv[u] = reinterpret_cast<float4*>(v)[i];
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = i0 + u * stride;
      if (i >= hi) continue;
      adam_update(k, __fmul_rn(gv[u].x, gscale), pv[u].x, mv[u].x, vv[u].x);
      adam_update(k, __fmul_rn(gv[u].y, gscale), pv[u].y, mv[u].y, vv[u].y);
      adam_update(k, __fmul_rn(gv[u].z, gscale), pv[u].z, mv[u].z, vv[u].z);
      adam_update(k, __fmul_rn(gv[u].w, gscale), pv[u].w, mv[u].w, vv[u].w);
      reinterpret_cast<float4*>(m)[i] = mv[u];
      reinterpret_cast<float4*>(v)[i] = vv[u];
      if (MC) {
        dp_st_mc(P.param_mc + 4 * i, pv[u]);
      } else {
        for (int r = 0; r < world; ++r) dp_st_peer(P.param[r] + 4 * i, pv[u]);
      }
    }
  }

  // ---- phase 2: all parameter stores of this rank are out; tell the peers, and do not retire
  // before every peer's stores have landed here
  __threadfence_system();
  __syncthreads();
  if (tid == 0) {
    const unsigned int prev = atomicAdd(local + 1, 1u);
    s_last = (prev == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (s_last) {
    if (tid == 0) local[1] = 0u;
    __threadfence_system();
    if (tid < world) {
      dp_signal(P.flags[tid] + AVA_DP_MAX_WORLD + rank, seq);
      dp_wait(my_flags + AVA_DP_MAX_WORLD + tid, seq, local + 2);
    }
  }
}

__global__ void adam_dp_bump_kernel(float* step_count, unsigned int* local) {
  step_count[0] += 1.f;
  local[0] += 1u;
}

}  // namespace ava

extern "C" int ava_b200_adam_step_dp(const ava_b200_dp_peers* h_peers, int rank, int world, float* m, float* v,
                                     long long n, float* step_count, const double* hyper, float grad_scale,
                                     unsigned int* local, void* stream_) {
  using namespace ava;
  AVA_REQUIRE(h_peers != nullptr && hyper != nullptr && local != nullptr, "adam_step_dp: null argument");
  AVA_REQUIRE(world >= 1 && world <= AVA_DP_MAX_WORLD && rank >= 0 && rank < world,
              "adam_step_dp: world %d / rank %d out of range (max %d ranks)", world, rank, AVA_DP_MAX_WORLD);
  AVA_REQUIRE(n > 0 && n % 4 == 0, "adam_step_dp: n must be a positive multiple of 4");
  DpPeers P;
  for (int r = 0; r < AVA_DP_MAX_WORLD; ++r) {
    P.grad[r] = r < world ? h_peers->grad[r] : nullptr;
    P.param[r] = r < world ? h_peers->param[r] : nullptr;
    P.flags[r] = r < world ? h_peers->flags[r] : nullptr;
    if (r < world) {
      AVA_REQUIRE(P.grad[r] && P.param[r] && P.flags[r], "adam_step_dp: missing peer pointer for rank %d", r);
      AVA_REQUIRE(((uintptr_t)P.grad[r] % 16 == 0) && ((uintptr_t)P.param[r] % 16 == 0),
                  "adam_step_dp: peer buffers must be 16-byte aligned");
    }
  }
  P.grad_mc = h_peers->grad_mc;
  P.param_mc = h_peers->param_mc;
  const bool mc = P.grad_mc != nullptr && P.param_mc != nullptr;
  AVA_REQUIRE(((uintptr_t)m % 16 == 0) && ((uintptr_t)v % 16 == 0), "adam_step_dp: moment buffers must be 16-byte aligned");
  cudaStream_t stream = (cudaStream_t)stream_;
  const long long n4 = n / 4;
  // (no co-residency requirement: whichever CTA finishes last does the phase-2 handshake)
  long long want = (n4 / world + 4 * 256 - 1) / (4 * 256);
  int grid = (int)(want < 1 ? 1 : (want > 4 * kNumSMs ? 4 * kNumSMs : want));
  if (mc)
    adam_dp_kernel<true><<<grid, 256, 0, stream>>>(P, rank, world, m, v, n4, step_count, hyper, grad_scale, local);
  else
    adam_dp_kernel<false><<<grid, 256, 0, stream>>>(P, rank, world, m, v, n4, step_count, hyper, grad_scale, local);
  if (check_launch("adam_dp")) return 1;
  adam_dp_bump_kernel<<<1, 1, 0, stream>>>(step_count, local);
  return check_launch("adam_dp_bump");
}
