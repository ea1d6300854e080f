// Synchronised BatchNorm for data-parallel training: one layer's BatchNorm sums exchanged over NVLink
// peer memory, so that every rank normalises with the statistics of the global batch.
//
// Every BatchNorm consumer (the fused conv kernels, bn_param_grads, bn_relu_bwd_apply) derives its count
// N = B*H*W from its own B and reads fp64 SUMS.  Rank r holds B_r of the B_g = sum B_r samples of a
// global batch.  If the stats block holds the global sums times B_r / B_g, every division by the local N
// yields the global mean and biased variance; the same holds for the backward block dstats = (sum g,
// sum g*(x - mean)), from which bnconv_bwd_data forms c1 and q.  bn_param_grads then gives B_r / B_g of
// the global dgamma / dbeta on each rank, and the gradient reduction the step already does sums them to
// the global value.  So no layer kernel changes: only the numbers in stats / dstats do.
//
// Protocol (one CTA per call; `local[0]` is this rank's sequence number s of the last exchange):
//   1. write the local sums and count into this rank's slot s & 1 (its own symmetric memory);
//   2. __threadfence_system, then st.release.sys of s on this rank's flag;
//   3. ld.acquire.sys on every peer's flag until it reaches s (bounded: kDpTimeoutNs, then local[1] = 1
//      and carry on -- a missing peer becomes a reported error, not a hung GPU);
//   4. add the world slots s & 1 in rank order 0..world-1 in fp64 (same bits on every rank), scale by
//      local_count / global_count into `sums`; forward exchanges also apply the running-buffer update
//      with the global sums and count (bn_running_update, shared with bn_update_running), so the
//      running buffers are identical on every rank and an empty shard updates them too.
//
// Why two slots and one flag suffice: a rank publishes exchange s+1 only after it has read every peer's
// slot of exchange s, which needs every peer's flag at >= s, which each peer raised only after it had
// finished reading exchange s-1.  So no rank is more than one exchange ahead of any other; the slot a
// rank overwrites at s+1 (parity of s-1) has been read by everyone, and the slot of s it is still read
// in is not touched before every peer has passed s.  A flag that is already at s+1 when read for s is
// fine for the same reason: that peer's slot of s is the other parity.  Flags only grow (wrap-safe
// comparison), so nothing is ever reset, and graph replays advance `local[0]` on the device.
//
// The payload is 65 doubles per rank: peer loads only (a multimem reduction has nothing to win here).
#include "common.cuh"

namespace ava {

constexpr int kBnSyncSlot = AVA_BN_SYNC_SLOT;

struct BnSyncPeers {
  double* slots[AVA_DP_MAX_WORLD];
  unsigned int* flags[AVA_DP_MAX_WORLD];
};

__device__ __forceinline__ double bn_ld_peer(const double* p) {
  double v;
  asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}

// thread t < 64 owns entry t of the stats block (sum of channel t & 31, or of its square when t >= 32)
__global__ void __launch_bounds__(64)
bn_stats_exchange_kernel(const BnSyncPeers P, const int rank, const int world, double* sums, const int channels,
                         const long long local_count, float* running, const int rm_off, const int rv_off,
                         long long* nbt, const float momentum, unsigned int* local) {
  __shared__ double s_tot[64];
  __shared__ double s_count;
  const int t = threadIdx.x;
  const bool mine = (t & 31) < channels;
  const unsigned int seq = local[0] + 1u;
  const int slot = (int)(seq & 1u) * kBnSyncSlot;

  double* own = P.slots[rank] + slot;
  if (mine) own[t] = sums[t];
  if (t == 0) own[64] = (double)local_count;
  __syncthreads();
  if (t == 0) {
    __threadfence_system();
    dp_signal(P.flags[rank], seq);
  }
  if (t < world) dp_wait(P.flags[t], seq, local + 1);
  __syncthreads();

  double tot = 0.0;
  if (mine) {
    tot = bn_ld_peer(P.slots[0] + slot + t);
    for (int r = 1; r < world; ++r) tot += bn_ld_peer(P.slots[r] + slot + t);
  }
  if (t == 0) {
    double n = bn_ld_peer(P.slots[0] + slot + 64);
    for (int r = 1; r < world; ++r) n += bn_ld_peer(P.slots[r] + slot + 64);
    s_count = n;
  }
  s_tot[t] = tot;
  __syncthreads();
  const double n = s_count;
  if (mine) sums[t] = n > 0.0 ? tot * ((double)local_count / n) : 0.0;
  if (running != nullptr && n > 0.0) {
    if (t < channels) bn_running_update(s_tot, t, n, running + rm_off, running + rv_off, momentum);
    if (t == 0) nbt[0] += 1;
  }
  if (t == 0) local[0] = seq;
}

}  // namespace ava

extern "C" int ava_b200_bn_stats_exchange(const ava_b200_bn_sync_peers* h_peers, int rank, int world, double* sums,
                                          int channels, long long local_count, float* running, int rm_off,
                                          int rv_off, long long* nbt, float momentum, unsigned int* local,
                                          void* stream) {
  using namespace ava;
  AVA_REQUIRE(h_peers != nullptr && sums != nullptr && local != nullptr, "bn_stats_exchange: null argument");
  AVA_REQUIRE(world >= 1 && world <= AVA_DP_MAX_WORLD && rank >= 0 && rank < world,
              "bn_stats_exchange: world %d / rank %d out of range (max %d ranks)", world, rank, AVA_DP_MAX_WORLD);
  AVA_REQUIRE(channels >= 1 && channels <= 32, "bn_stats_exchange: channels=%d (1..32)", channels);
  AVA_REQUIRE(local_count >= 0, "bn_stats_exchange: negative count %lld", local_count);
  AVA_REQUIRE(running == nullptr || (nbt != nullptr && rm_off >= 0 && rv_off >= 0),
              "bn_stats_exchange: a running-buffer update needs nbt and non-negative offsets");
  BnSyncPeers P;
  for (int r = 0; r < AVA_DP_MAX_WORLD; ++r) {
    P.slots[r] = r < world ? h_peers->slots[r] : nullptr;
    P.flags[r] = r < world ? h_peers->flags[r] : nullptr;
    if (r < world)
      AVA_REQUIRE(P.slots[r] && P.flags[r], "bn_stats_exchange: missing peer pointer for rank %d", r);
  }
  bn_stats_exchange_kernel<<<1, 64, 0, (cudaStream_t)stream>>>(P, rank, world, sums, channels, local_count, running,
                                                               rm_off, rv_off, nbt, momentum, local);
  return check_launch("bn_stats_exchange");
}
