// Fused BatchNorm -> 3x3 conv / conv-transpose -> ReLU layers, forward and backward,
// as direct fp32 SIMT kernels for sm_100a.
//
// Replaces, per layer, the reference's bn_k(x) -> conv_k / convt_k -> F.relu chain
// (ava/models/vae.py:217-223, 263-269) and autograd's backward of it (vae.py:352).
//
// One "gather" kernel template covers all 28 forward / backward-data passes:
//   K_S1: out[o,y,x] = sum in[i, y+ky-1,  x+kx-1 ] * W(o,i,ky,kx)      (3x3, stride 1)
//   K_S2: out[o,y,x] = sum in[i, 2y+ky-1, 2x+kx-1] * W(o,i,ky,kx)      (stride 2, down)
//   K_UP: out[o,y,x] = sum in[i, (y+1-ky)/2, (x+1-kx)/2] * W(o,i,ky,kx) over taps with
//         even numerators                                               (stride 2, up)
// conv fwd = S1/S2, convT fwd = S1(flipped)/UP, conv bwd-data = S1(flipped)/UP,
// convT bwd-data = S1/S2; the weight tensor is addressed through (stride_o, stride_i, flip).
//
// Prologue (while staging the input tile in shared memory):
//   IN_AFFINE: v = x*scale[c] + shift[c]  (BatchNorm apply; zero padding AFTER bn)
//   IN_PLAIN:  v = g  (a gradient already pushed through the next BN's backward and this layer's
//              ReLU by ava_b200_bn_relu_bwd_apply; its zero padding is TMA's out-of-bounds fill)
// Epilogue:
//   EPI_FWD: + bias, ReLU, store, and per-channel sum / sum-of-squares of the output
//            (the next BatchNorm's batch statistics) via warp shuffles -> smem -> fp64 atomics
//   EPI_BWD: this layer's BatchNorm backward + the producing layer's ReLU backward applied to the
//            accumulators (coefficients from the weight-gradient pass), store the next dz
//
// Thread mapping: a warp's lanes run along x (coalesced loads/stores, conflict-free
// shared-memory reads), each thread owns 4 output rows x COT(<=8) output channels in
// registers; output-channel groups of 8 are warp-uniform so weight reads are broadcasts.
#include <cuda.h>

#include "common.cuh"

namespace ava {

enum { K_S1 = 0, K_S2 = 1, K_UP = 2 };
enum { IN_AFFINE = 0, IN_PLAIN = 1 };
enum { EPI_FWD = 0, EPI_BWD = 1 };

struct GconvParams {
  const float* in;    // AFFINE: x;  PLAIN: dz
  // coefficient sources for the input transform
  const float* gamma;
  const float* beta;
  const double* stats;
  const float* rmean;
  const float* rvar;
  int train;
  double in_count;
  // weights
  const float* w;
  int w_so, w_si, w_flip;
  const float* bias;
  // output
  float* out;
  int relu_out;
  double* stats_out;
  // EPI_BWD: this layer's own BatchNorm (applied to x_self in the forward pass).  Its backward
  // and the ReLU backward of the layer that produced x_self run in the epilogue:
  //   out = [x_self > 0] * (p*(g - c1) + q*(x_self - mean))      (common.cuh: dz_coef / dz_apply)
  // with the two BatchNorm-backward reductions dstats_in = (sum g, sum g*(x-mean)) supplied by
  // the weight-gradient pass of the same layer (see bnconv_finalize_kernel): the gradient g
  // w.r.t. the BatchNorm output never goes to memory.
  const float* x_self;
  const double* stats_self;
  const float* gamma_self;
  const double* dstats_in;
  const float* rvar_self;   // eval-mode BatchNorm: its running variance (NULL: train mode, batch statistics)
  int mask_in;
  // EPI_BWD, optional: the nine per-channel border sums of the dz written here (what
  // ava_b200_dz_border_sums would compute in a separate pass; mode 0 / 1 as there), accumulated
  // in the epilogue -- the consumer layer's weight-gradient finalisation needs them
  double* tsums_out;
  int tsum_mode;
  double out_count;
  int B, H_in, W_in;
};

template <int KIND, int TW, bool MMA = false>
struct TileGeom {
  // sub-tile handled by 64 thread slots: output tile (S1,S2) or input tile (UP); the stride-2
  // tensor-core tile is 128 output pixels (its staging buffers are twice as large per pixel)
  static constexpr int TH = (KIND == K_UP || (MMA && KIND == K_S2)) ? 128 / TW : 256 / TW;
  static constexpr int IN_ROWS = (KIND == K_S1) ? TH + 2 : (KIND == K_S2 ? 2 * TH + 1 : TH + 1);
  // aligned interior of a staged row, loaded as float4 quads; halo columns are scalars
  static constexpr int QUADS = (KIND == K_S2) ? TW / 2 : TW / 4;
  // shared-memory row layout (floats):
  //   S1: [3]=left halo, [4..TW+3]=interior, [TW+4]=right halo
  //   S2: odd input columns at [3..TW+3] (j=0 is the left halo), even columns at [EO..EO+TW-1]
  //   UP: [0..TW-1]=interior, [TW]=right halo
  // pitches: interior 16-byte aligned, and for TW=16 (two row groups per warp) the second
  // group lands 16 banks away from the first; stride-1 planes (IN_ROWS*PITCH) are 24 (mod 32)
  // floats so that the tensor-core fragment loads (4 channels x 8 pixels per warp) hit 32 banks
  static constexpr int EO = TW + 4;
  static constexpr int PITCH = (KIND == K_S1) ? (TW == 32 ? 44 : 28)
                               : (KIND == K_S2) ? (MMA ? (TW == 32 ? 72 : 40) : (TW == 32 ? 68 : 38))
                                                : (TW == 32 ? (MMA ? 40 : 36) : 24);
  static constexpr int PLANE = IN_ROWS * PITCH;
  // raw (untransformed) staging tile = one dense TMA box [CIC][IN_ROWS][RAW_PITCH] whose first
  // column is input column X0-4 (S1,S2) or X0 (UP), so that the interior quads stay 16-byte
  // aligned: S1 [3]=left halo [4..TW+3] interior [TW+4] right halo; S2 [3]=left halo,
  // [4..2TW+3] interleaved interior; UP [0..TW-1] interior, [TW] right halo
  static constexpr int RAW_PITCH = (KIND == K_S1) ? TW + 8 : (KIND == K_S2 ? 2 * TW + 4 : TW + 4);
  static constexpr int RAW_PLANE = IN_ROWS * RAW_PITCH;
  static constexpr int RAW_X_SHIFT = (KIND == K_UP) ? 0 : 4;
};

// TERMS == 0: fp32 SIMT FMA loop.  TERMS == 1 / 3: the inner product runs on the tensor cores as
// mma.sync m16n8k8 TF32 (1 term: operands rounded to TF32; 3 terms: error-compensated
// a_lo*b_hi + a_hi*b_lo + a_hi*b_hi with x = x_hi + x_lo, fp32-level accuracy).  TERMS == 2: the
// same compensated product with BOTH correction terms of a tap in ONE BF16 m16n8k16 instruction
// (cv_mma_bf16 below: k16 = {a_lo | a} x {b | b_lo}), 2 tensor-core instructions per tap instead
// of 3.  Every warp then
// owns 4 output rows x 16 pixels x all output channels, one 8-input-channel chunk per stage;
// a CTA is 4 warps on one 256-pixel sub-tile, 4 (3 for the widest layers) CTAs per SM, so that
// the load / transform / MMA / epilogue phases of independent CTAs overlap.
template <int KIND, int CI, int CO, int TW, int INMODE, int TERMS = 0>
struct GconvCfg {
  using G = TileGeom<KIND, TW, (TERMS > 0)>;
  static constexpr bool MMA = TERMS > 0;
  static constexpr int COT = (CO >= 8) ? 8 : CO;
  static constexpr int NCOG = CO / COT;
  static constexpr int NTL = CO / 8;  // MMA: n-tiles of 8 output channels per warp
  // threads: 64 slots x NCOG channel groups x NSUB sub-tiles (256, or 192 for CO=24);
  // MMA: 4 warps on one sub-tile
  static constexpr int NSUB = MMA ? 1 : (NCOG >= 3) ? 1 : 4 / NCOG;
  // (the stride-2-up tensor-core CTA is 8 warps: one input row x 16 pixels and its 2x2 output
  // parity classes per warp)
  static constexpr int NT = MMA ? (KIND == K_UP ? 256 : 128) : 64 * NCOG * NSUB;
  // IN_PLAIN input (an already materialised gradient) needs no per-element transform and its
  // zero padding is exactly TMA's out-of-bounds fill: for the stride-1 / up kernels the boxes
  // land DIRECTly in the layout the FMA loop reads (double buffered, no staging pass at all).
  // The stride-2 kernels still de-interleave even/odd columns through a staging buffer.
  static constexpr bool DIRECT = (INMODE == IN_PLAIN) && (KIND != K_S2);
  static constexpr int BOX_W = DIRECT ? G::PITCH : G::RAW_PITCH;
  static constexpr int BOX_PLANE = G::IN_ROWS * BOX_W;
  // input channels per pipeline stage: largest divisor of CI keeping a stage <= 37 KB
  static constexpr int LIMIT = 9472;
  static constexpr int stage_floats(int c) { return NSUB * c * BOX_PLANE; }
  static constexpr int CIC = (MMA || (CI % 8 == 0 && stage_floats(8) <= LIMIT)) ? 8
                             : (CI % 4 == 0 && stage_floats(4) <= LIMIT) ? 4
                             : (CI % 2 == 0 && stage_floats(2) <= LIMIT) ? 2
                                                                         : 1;
  static constexpr int NCHUNK = CI / CIC;
  static constexpr int FIN_SUB = (CIC * G::PLANE + 31) / 32 * 32;           // floats, 128-byte aligned
  static constexpr int RAW_SUB = (CIC * G::RAW_PLANE + 31) / 32 * 32;
  static constexpr int STAGE = NSUB * FIN_SUB;                              // transformed tile(s)
  static constexpr int RAW_STAGE = NSUB * RAW_SUB;                          // staging (non-DIRECT)
  static constexpr int BUF_FLOATS = DIRECT ? 2 * STAGE : RAW_STAGE + STAGE;
  static constexpr int BOX_BYTES = CIC * BOX_PLANE * 4;
  // transform work items per sub-tile and per thread (non-DIRECT)
  static constexpr int NQUAD = CIC * G::IN_ROWS * G::QUADS;
  static constexpr int QITERS = (NQUAD + NT - 1) / NT;
  static constexpr int NHALO = CIC * G::IN_ROWS;
  static constexpr int HITERS = (NHALO + NT - 1) / NT;
  // CTAs per SM the register budget is tuned for
  static constexpr int MINB = (MMA && KIND == K_UP) ? 2 : (MMA || COT == 1) ? 4 : 2;
  // staged weights: SIMT [CI][9][CO]; MMA: B fragments in register order
  // [CI/8][9][NTL][32 lanes]: {b0,b1} TF32-rounded (TERMS 1); {b0_hi,b1_hi,b0_lo,b1_lo}
  // (TERMS 3, PRESPLIT) or, for the widest layers, {b0,b1} in full fp32 split where used
  static constexpr bool PRESPLIT = (TERMS >= 2) && (CI * CO <= 384);
  static constexpr int WF = PRESPLIT ? 4 : 2;   // floats per lane per fragment
  // A-resident loop order when the fragments of 6 input rows fit next to the accumulators
  static constexpr bool ARES = (TERMS == 1) ? (NTL <= 3) : (NTL <= 2);
  static constexpr int W_FLOATS = CI * 9 * CO * (PRESPLIT ? 2 : 1);
  static constexpr int RED_FLOATS = MMA ? (NT / 32) * 128 : 128;   // MMA: [warps][64] doubles
  static_assert(!MMA || (CI % 8 == 0 && CO % 8 == 0), "tensor-core path: channels % 8");
  static_assert(!MMA || (G::PLANE % 32 == 8 || G::PLANE % 32 == 24), "tensor-core path: conflict-free channel planes");
  // output rows per warp (16 pixels wide)
  static constexpr int R = (KIND == K_S1) ? 4 : (KIND == K_S2 ? 2 : 4);   // K_UP: the 4 parity classes
};

__device__ __forceinline__ uint32_t cv_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
// x rounded to the nearest TF32 value (ties away from zero, like cvt.rna, in two integer ops):
// exactly representable in TF32, and |x - hi| <= 2^-12 |x|, so the dropped lo*lo term of the
// 3-term product is 2^-24 relative and unbiased
__device__ __forceinline__ uint32_t cv_tf32_hi(float x) { return (__float_as_uint(x) + 0x1000u) & 0xFFFFE000u; }
// The tensor core adds into its fp32 accumulator with truncation (measured: 2000 chained
// accumulations drift by 1.6e-4), a bias that BatchNorm backward amplifies.  The 3-term product
// is therefore evaluated as a short chain on a fresh accumulator, smallest terms first
// (t = a_lo*b_hi; t += a_hi*b_lo; t += a_hi*b_hi), and t is added to the running sum with an
// ordinary round-to-nearest FADD.
__device__ __forceinline__ void cv_mma_tf32_zero(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
      : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "f"(0.f));
}
__device__ __forceinline__ void cv_mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// TERMS == 2: the error-compensated product with its two correction terms at half the tensor-core
// cost.  x = x_hi + x_lo as above; a*b = a_hi*b_hi + a_lo*b + a*b_lo - a_lo*b_lo.  The main term
// stays on mma.m16n8k8 TF32; the corrections are 2^-11 of it, so their factors only need 8
// significant bits: a_lo*b and a*b_lo run as BF16 mma.m16n8k16, which covers TWO k-chunks per
// instruction at the TF32 instruction's issue cost (probe: profiles/probes/hmma_kinds.cu, 8.9
// cycles per SMSP for either shape).  4 tensor-core instructions per pair of k-chunks instead of
// 6; per-product error <= 2^-11 * 2 * 2^-8 = 2^-18 relative, unbiased (round-to-nearest
// everywhere), i.e. ~1e-6 of the result's scale after the random-sign sum.
// A pair of k-chunks (c0, c1) maps onto the k16 fragment as k16 = {2t: c0[t], 2t+1: c1[t],
// 2t+8: c0[t+4], 2t+9: c1[t+4]} for BOTH operands, so every lane packs only its own registers.
__device__ __forceinline__ uint32_t cv_pack_bf16(float lo_half, float hi_half) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi_half), "f"(lo_half));
  return r;
}
__device__ __forceinline__ void cv_mma_bf16_zero(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
      : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "f"(0.f));
}
__device__ __forceinline__ void cv_mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ uint32_t cv_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cv_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(cv_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void cv_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(cv_smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void cv_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "CV_WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra CV_DONE;\n"
      "bra CV_WAIT_LOOP;\n"
      "CV_DONE:\n"
      "}\n" ::"r"(cv_smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// 3-D box [channels][rows][cols] of a [B*C, H, W] activation tensor; out-of-range rows/columns
// (image border, negative coordinates) are zero-filled by the TMA unit
// (gconv_kernel's issue(): also requesting the stage AFTER the one being fetched into L2.  Measured:
// forward family 1970 -> 2009 us per step at batch 1024, backward-data +35 us -- the extra TMA
// requests compete with the loads that are needed now.  Off.)
constexpr bool kPrefetchAhead = false;
// request a box into L2 only (no shared-memory destination, no completion to wait for)
__device__ __forceinline__ void cv_tma_prefetch_3d(const CUtensorMap* map, int x, int y, int z) {
  asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global [%0, {%1, %2, %3}];" ::"l"(map), "r"(x), "r"(y), "r"(z)
               : "memory");
}
__device__ __forceinline__ void cv_tma_load_3d(void* smem_dst, const CUtensorMap* map, int x, int y, int z,
                                               uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(cv_smem_u32(smem_dst)),
      "l"(map), "r"(x), "r"(y), "r"(z), "r"(cv_smem_u32(bar))
      : "memory");
}

// Software-pipelined: while the FMA loop runs on stage i, the boxes of stage i+1 are fetched
// by TMA (one cp.async.bulk.tensor box per sub-tile, issued by a single thread: no register or
// LSU cost, completion on an mbarrier).  IN_AFFINE: a short table-driven shared->shared pass
// applies the BatchNorm scale/shift and writes literal zeros for the padding (padding is
// applied AFTER BatchNorm).  IN_PLAIN: see GconvCfg::DIRECT.  2 (4 for CO=1) CTAs per SM.
template <int KIND, int CI, int CO, int TW, int INMODE, int EPI, int HIN, int TERMS>
__global__ void __launch_bounds__(GconvCfg<KIND, CI, CO, TW, INMODE, TERMS>::NT,
                                  GconvCfg<KIND, CI, CO, TW, INMODE, TERMS>::MINB)
    gconv_kernel(const __grid_constant__ CUtensorMap map_in, const GconvParams P) {
  using C = GconvCfg<KIND, CI, CO, TW, INMODE, TERMS>;
  using G = typename C::G;
  constexpr int COT = C::COT, NCOG = C::NCOG, NSUB = C::NSUB, NT = C::NT;
  constexpr int CIC = C::CIC, NCHUNK = C::NCHUNK;
  constexpr bool DIRECT = C::DIRECT;
  constexpr int NOUT = (KIND == K_UP) ? 8 : 4;

  extern __shared__ __align__(128) float smem[];
  // DIRECT: [2][STAGE] ring of ready-to-use tiles; else [RAW_STAGE] staging + [STAGE] transformed
  float* s_raw = smem;
  float* s_in = DIRECT ? smem : smem + C::RAW_STAGE;
  float* s_w = smem + C::BUF_FLOATS;                // [CI][9][CO] (MMA: B fragments, see GconvCfg)
  float* s_c0 = s_w + C::W_FLOATS;                  // AFFINE scale
  float* s_c1 = s_c0 + 32;                          // AFFINE shift
  float* s_red = s_c1 + 32;                         // per-warp partial sums
  float* s_bias = s_red + C::RED_FLOATS;            // [CO]
  double* s_dz = reinterpret_cast<double*>(s_bias + 32);  // EPI_BWD coefficients of own BN, as
  float* s_dzf = reinterpret_cast<float*>(s_dz);          // floats [3: p | q | k][32]
  double* s_ts = s_dz + 128;                               // [9][32] EPI_BWD: border sums of the output
  double* s_tsw = s_ts + 288;                              // [warps][4][32] EPI_BWD: per-warp totals / classes
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_tsw + (EPI == EPI_BWD ? (NT / 32) * 128 : 0));

  const int tid = threadIdx.x;
  // every instantiation serves exactly one layer, so the image size is a compile-time constant
  // (tile decoding and all address arithmetic fold to shifts / immediates)
  constexpr int H_in = HIN, W_in = HIN;
  constexpr int H_out = (KIND == K_S1) ? H_in : (KIND == K_S2 ? H_in / 2 : H_in * 2);
  constexpr int W_out = (KIND == K_S1) ? W_in : (KIND == K_S2 ? W_in / 2 : W_in * 2);
  // tiles are counted in output space for S1/S2 and in input space for UP
  constexpr int tiles_x = ((KIND == K_UP) ? W_in : W_out) / TW;
  constexpr int tiles_y = ((KIND == K_UP) ? H_in : H_out) / G::TH;
  constexpr int tiles_per_img = tiles_x * tiles_y;
  const int ntiles = P.B * tiles_per_img;
  const int ngroups = (ntiles + NSUB - 1) / NSUB;

  // ---- EPI_BWD: the epilogue reads this layer's forward input x_self for the tile it has just
  // computed (BatchNorm backward + ReLU mask); straight from DRAM those loads are the largest stall of
  // the backward-data kernels (long scoreboard 20-41% of the samples, profiles/r02_ncu_top_kernels.txt).
  // The tile's lines are requested into L2 when the tile STARTS, so that they arrive while the
  // inner product runs (no registers or shared memory held).
  auto prefetch_x = [&](int n, int ty, int tx, int me, int nthr) {
    constexpr int OTH = (KIND == K_UP) ? 2 * G::TH : G::TH;
    constexpr int OTW = (KIND == K_UP) ? 2 * TW : TW;
    constexpr int LPR = (OTW * 4 + 127) / 128;   // 128-byte lines per row segment
    const float* base = P.x_self + ((size_t)n * CO * H_out + (size_t)ty * OTH) * W_out + tx * OTW;
    for (int i = me; i < CO * OTH * LPR; i += nthr) {
      const int l = i % LPR, r = (i / LPR) % OTH, c = i / (LPR * OTH);
      asm volatile("prefetch.global.L2 [%0];" ::"l"(base + ((size_t)c * H_out + r) * W_out + l * 32));
    }
  };

  // ---- TMA: boxes of stage (grp, ch) into ring slot `buf`, issued by thread 0
  auto issue = [&](int grp, int ch, int buf) {
    if (tid != 0) return;
    int nsub = ntiles - grp * NSUB;
    if (nsub > NSUB) nsub = NSUB;
    cv_mbar_expect_tx(s_bar, (uint32_t)(nsub * C::BOX_BYTES));
    float* dst = DIRECT ? s_in + buf * C::STAGE : s_raw;
    constexpr int SUBF = DIRECT ? C::FIN_SUB : C::RAW_SUB;
    for (int sb = 0; sb < nsub; ++sb) {
      const int ltile = grp * NSUB + sb;
      const int ln = ltile / tiles_per_img;
      const int lrem = ltile - ln * tiles_per_img;
      const int lty = lrem / tiles_x, ltx = lrem - lty * tiles_x;
      const int iy0 = (KIND == K_S1) ? lty * G::TH - 1 : (KIND == K_S2 ? 2 * lty * G::TH - 1 : lty * G::TH);
      const int X0 = (KIND == K_S2) ? 2 * ltx * TW : ltx * TW;
      cv_tma_load_3d(dst + sb * SUBF, &map_in, X0 - G::RAW_X_SHIFT, iy0, ln * CI + ch * CIC, s_bar);
    }
    // ... and the stage AFTER this one is requested into L2 (one stage of look-ahead hides the TMA
    // round trip only when the inner product of a stage outlasts a DRAM access)
    int g2 = grp, c2 = ch + 1;
    if (c2 == NCHUNK) {
      g2 = grp + gridDim.x;
      c2 = 0;
    }
    if (kPrefetchAhead && g2 < ngroups) {
      int nsub2 = ntiles - g2 * NSUB;
      if (nsub2 > NSUB) nsub2 = NSUB;
      for (int sb = 0; sb < nsub2; ++sb) {
        const int ltile = g2 * NSUB + sb;
        const int ln = ltile / tiles_per_img;
        const int lrem = ltile - ln * tiles_per_img;
        const int lty = lrem / tiles_x, ltx = lrem - lty * tiles_x;
        const int iy0 = (KIND == K_S1) ? lty * G::TH - 1 : (KIND == K_S2 ? 2 * lty * G::TH - 1 : lty * G::TH);
        const int X0 = (KIND == K_S2) ? 2 * ltx * TW : ltx * TW;
        cv_tma_prefetch_3d(&map_in, X0 - G::RAW_X_SHIFT, iy0, ln * CI + c2 * CIC);
      }
    }
  };

  if (tid == 0) {
    cv_mbar_init(s_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  // ---- per-thread transform work list (identical for every sub-tile and stage)
  int q_raw[C::QITERS], q_fin[C::QITERS], q_meta[C::QITERS];   // meta: row | ci<<8, -1 = none
  int h_raw[C::HITERS], h_fin[C::HITERS], h_meta[C::HITERS];
  if (!DIRECT) {
#pragma unroll
    for (int j = 0; j < C::QITERS; ++j) {
      const int t = tid + j * NT;
      q_meta[j] = -1;
      q_raw[j] = q_fin[j] = 0;
      if (t < C::NQUAD) {
        const int q = t % G::QUADS;
        const int rr = t / G::QUADS;
        const int r = rr % G::IN_ROWS;
        const int ci = rr / G::IN_ROWS;
        q_raw[j] = ci * G::RAW_PLANE + r * G::RAW_PITCH + ((KIND == K_UP) ? 4 * q : 4 + 4 * q);
        const int frow = ci * G::PLANE + r * G::PITCH;
        q_fin[j] = (KIND == K_S1) ? frow + 4 + 4 * q : (KIND == K_S2 ? frow + 2 * q : frow + 4 * q);
        q_meta[j] = r | (ci << 8);
      }
    }
#pragma unroll
    for (int j = 0; j < C::HITERS; ++j) {
      const int t = tid + j * NT;
      h_meta[j] = -1;
      h_raw[j] = h_fin[j] = 0;
      if (t < C::NHALO) {
        const int r = t % G::IN_ROWS;
        const int ci = t / G::IN_ROWS;
        h_raw[j] = ci * G::RAW_PLANE + r * G::RAW_PITCH;
        h_fin[j] = ci * G::PLANE + r * G::PITCH;
        h_meta[j] = r | (ci << 8);
      }
    }
  }

  auto xform1 = [&](float a, int cc) -> float {
    if (INMODE == IN_AFFINE) return fmaf(a, s_c0[cc], s_c1[cc]);
    return a;
  };

  // ---- staging buffer -> tile the FMA loop reads (BN apply; zero padding AFTER; even/odd split)
  auto transform = [&](int grp, int ch) {
    const int tile0 = grp * NSUB;
#pragma unroll
    for (int sb = 0; sb < NSUB; ++sb) {
      const int ltile = tile0 + sb;
      if (ltile >= ntiles) break;
      const int lrem = ltile % tiles_per_img;
      const int lty = lrem / tiles_x, ltx = lrem - lty * tiles_x;
      const int iy0 = (KIND == K_S1) ? lty * G::TH - 1 : (KIND == K_S2 ? 2 * lty * G::TH - 1 : lty * G::TH);
      const int X0 = (KIND == K_S2) ? 2 * ltx * TW : ltx * TW;
      const float* rg = s_raw + sb * C::RAW_SUB;
      float* sdst = s_in + sb * C::FIN_SUB;
#pragma unroll
      for (int j = 0; j < C::QITERS; ++j) {
        const int m = q_meta[j];
        if (m < 0) continue;
        const int gy = iy0 + (m & 0xff);
        const int cc = ch * CIC + (m >> 8);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gy >= 0 && gy < H_in) {
          const float4 a = *reinterpret_cast<const float4*>(rg + q_raw[j]);
          v = make_float4(xform1(a.x, cc), xform1(a.y, cc), xform1(a.z, cc), xform1(a.w, cc));
        }
        float* d = sdst + q_fin[j];
        if (KIND == K_S2) {
          *reinterpret_cast<float2*>(d + G::EO) = make_float2(v.x, v.z);  // even columns
          *reinterpret_cast<float2*>(d + 4) = make_float2(v.y, v.w);      // odd j=2q+1,2q+2
        } else {
          *reinterpret_cast<float4*>(d) = v;
        }
      }
#pragma unroll
      for (int j = 0; j < C::HITERS; ++j) {
        const int m = h_meta[j];
        if (m < 0) continue;
        const int gy = iy0 + (m & 0xff);
        const int cc = ch * CIC + (m >> 8);
        const bool rowok = gy >= 0 && gy < H_in;
        const int gx0 = (KIND == K_UP) ? X0 + TW : X0 - 1;
        const int sc0 = (KIND == K_UP) ? TW : 3;
        float h0 = 0.f;
        if (rowok && gx0 >= 0 && gx0 < W_in) h0 = xform1(rg[h_raw[j] + sc0], cc);
        sdst[h_fin[j] + sc0] = h0;
        if (KIND == K_S1) {
          float h1 = 0.f;
          if (rowok && X0 + TW < W_in) h1 = xform1(rg[h_raw[j] + TW + 4], cc);
          sdst[h_fin[j] + TW + 4] = h1;
        }
      }
    }
  };

  // ---- one-time per CTA: weights, coefficients
  if constexpr (C::MMA) {
    // (Measured and dropped: copying the contiguous weight tensor into shared memory with coalesced
    // loads first and gathering from there.  ncu -- which flushes the caches -- shows this gather as
    // 7-10% of a mid-layer kernel's samples, but in a real step the 27 KB are L2-hot and the two extra
    // barriers cost more than the gather: +2 us per launch.)
    // B fragments of mma.m16n8k8 (col): lane (g = lane>>2, t = lane&3) holds b0 = W[k=t][n=g],
    // b1 = W[k=t+4][n=g], k = input channel within the 8-channel chunk, n = output channel
    for (int idx = tid; idx < (CI / 8) * 9 * C::NTL * 32; idx += NT) {
      const int ln = idx & 31;
      int rest = idx >> 5;
      const int nt = rest % C::NTL;
      rest /= C::NTL;
      const int k = rest % 9, ks = rest / 9;
      const int co = nt * 8 + (ln >> 2), ci0 = ks * 8 + (ln & 3);
      const int kk = P.w_flip ? 8 - k : k;
      const float w0 = P.w[(size_t)co * P.w_so + (size_t)ci0 * P.w_si + kk];
      const float w1 = P.w[(size_t)co * P.w_so + (size_t)(ci0 + 4) * P.w_si + kk];
      if (C::PRESPLIT) {
        const float h0 = __uint_as_float(cv_tf32(w0)), h1 = __uint_as_float(cv_tf32(w1));
        if (TERMS == 2)   // {b_hi | k16 B fragment: (b, paired with a_lo), (b_lo, paired with a)}
          *reinterpret_cast<float4*>(s_w + 4 * idx) =
              make_float4(h0, h1, __uint_as_float(cv_pack_bf16(w0, w1)),
                          __uint_as_float(cv_pack_bf16(w0 - h0, w1 - h1)));
        else
          *reinterpret_cast<float4*>(s_w + 4 * idx) = make_float4(h0, h1, w0 - h0, w1 - h1);
      } else if (TERMS >= 2) {
        *reinterpret_cast<float2*>(s_w + 2 * idx) = make_float2(w0, w1);
      } else {
        *reinterpret_cast<float2*>(s_w + 2 * idx) =
            make_float2(__uint_as_float(cv_tf32(w0)), __uint_as_float(cv_tf32(w1)));
      }
    }
  } else {
    for (int idx = tid; idx < CI * 9 * CO; idx += NT) {
      int co = idx % CO;
      int k = (idx / CO) % 9;
      int ci = idx / (9 * CO);
      int kk = P.w_flip ? 8 - k : k;
      s_w[idx] = P.w[(size_t)co * P.w_so + (size_t)ci * P.w_si + kk];
    }
  }
  if ((int)blockIdx.x < ngroups) issue(blockIdx.x, 0, 0);
  if (INMODE == IN_AFFINE && tid < CI) {
    BnCoef k = bn_coef(P.stats, tid, P.in_count, P.gamma, P.beta, P.rmean, P.rvar, P.train != 0);
    s_c0[tid] = k.scale;
    s_c1[tid] = k.shift;
  }
  if (tid < CO) {
    s_bias[tid] = (EPI == EPI_FWD && P.bias) ? P.bias[tid] : 0.f;
    if (EPI == EPI_BWD) {
      // out = p*(g - c1) + q*(x - mean) = p*g + q*x + k: p, q rounded to fp32 (a relative error of
      // 6e-8 on a whole channel's gradient), k = -(p*c1 + q*mean) formed in fp64 from the ROUNDED
      // p, q, then rounded once (a constant shift of <= 6e-8 |k| for the whole channel)
      const DzCoef k = dz_coef(P.gamma_self, P.stats_self, P.dstats_in, tid, P.out_count, P.rvar_self);
      const float pf = (float)k.p, qf = (float)k.q;
      s_dzf[tid] = pf;
      s_dzf[32 + tid] = qf;
      s_dzf[64 + tid] = (float)(-((double)pf * k.c1 + (double)qf * k.mean));
    }
  }
  __syncthreads();
  // EPI_BWD epilogue: BatchNorm backward + ReLU mask,  out = [x > 0] * (p*(g - c1) + q*(x - mean)),
  // in fp32 against fp64-exact constants.  The expression is well conditioned -- measured over
  // the network (profiles/probes/exp_algebraic_dstats.py): |mean g| <= 0.2 std g and
  // |q (x-mean)| <= 0.5 |p (g-c1)| in every layer, so nothing cancels.  (A float64 evaluation
  // costs three F2F conversions per element on a 16-lane pipe: +0.75 ms per step at batch 1024
  // when it ran in this epilogue.)
  auto dzap = [&](int co, float g, float x) -> float {
    const float d = fmaf(s_dzf[co], g, fmaf(s_dzf[32 + co], x, s_dzf[64 + co]));
    return (P.mask_in && !(x > 0.f)) ? 0.f : d;
  };
  const bool want_ts = (EPI == EPI_BWD) && P.tsums_out != nullptr;
  if (want_ts) {
    for (int i = tid; i < 288; i += NT) s_ts[i] = 0.0;
    for (int i = tid; i < (NT / 32) * 128; i += NT) s_tsw[i] = 0.0;
    __syncthreads();
  }
  auto ts_add = [&](int slot, int co, float v) { atomicAdd(&s_ts[slot * 32 + co], (double)v); };

  if constexpr (C::MMA) {
    // ---------------------------------------------------------------- tensor-core path (K_S1, K_S2)
    // warp -> (sub-tile, 16-pixel half xh, R output rows from r0); lane -> (g, t) of the fragments
    constexpr int NTL = C::NTL, R = C::R;
    const int warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    constexpr int sub = 0;
    const int wq = warp;
    const int xh = (TW == 32) ? (wq & 1) : 0;
    // K_UP: r0 = the warp's input row; its accumulator index is the output parity class 2*oa+ob
    const int r0 = (KIND == K_UP) ? ((TW == 32) ? (wq >> 1) : wq) : (TW == 32) ? R * (wq >> 1) : R * wq;
    // per-channel statistics: fp32 only within one tile (8 values per thread and channel slot);
    // every tile's warp-level partial sums are added to per-warp fp64 slots in shared memory
    // (fixed order: deterministic), so no fp32 rounding accumulates over the CTA's many tiles
    double* s_accd = reinterpret_cast<double*>(s_red) + warp * 64;
    const bool want_stats = (EPI == EPI_FWD) && P.stats_out != nullptr;
    if (lane < 4) {
#pragma unroll
      for (int i = 0; i < NTL; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) s_accd[i * 8 + 2 * t + j] = s_accd[32 + i * 8 + 2 * t + j] = 0.0;
    }

    // EPI_BWD border sums: totals (mode 0) / parity classes (mode 1) of the written dz, summed in
    // fp32 per thread over ALL of this CTA's tiles and reduced once at the end (each partial is a
    // few hundred values; the rounding errors of the ~1e5 independent partials of a layer are
    // random and average out)
    float ts_hot[2][NTL][2];
#pragma unroll
    for (int rp = 0; rp < 2; ++rp)
#pragma unroll
      for (int i = 0; i < NTL; ++i) ts_hot[rp][i][0] = ts_hot[rp][i][1] = 0.f;

    uint32_t phase = 0;
    int it = 0;
    for (int grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
      float st1[NTL][2], st2[NTL][2];
#pragma unroll
      for (int i = 0; i < NTL; ++i) st1[i][0] = st1[i][1] = st2[i][0] = st2[i][1] = 0.f;
      const int tile = grp * NSUB + sub;
      const bool tvalid = tile < ntiles;
      const int n = tile / tiles_per_img;
      const int trem = tile - n * tiles_per_img;
      const int ty = trem / tiles_x, tx = trem - ty * tiles_x;
      if (EPI == EPI_BWD && tvalid) prefetch_x(n, ty, tx, tid, NT);

      float acc[R][NTL][4];
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int i = 0; i < NTL; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[r][i][j] = 0.f;

#pragma unroll 1
      for (int ch = 0; ch < NCHUNK; ++ch, ++it) {
        const int buf = DIRECT ? (it & 1) : 0;
        cv_mbar_wait(s_bar, phase);
        phase ^= 1;
        if (!DIRECT) transform(grp, ch);
        __syncthreads();
        if (ch + 1 < NCHUNK) {
          issue(grp, ch + 1, buf ^ 1);
        } else if (grp + (int)gridDim.x < ngroups) {
          issue(grp + gridDim.x, 0, buf ^ 1);
        }
        if (tvalid) {
          // A fragment (row-major 16 pixels x 8 channels): a0 = (pixel g, channel t),
          // a1 = (g+8, t), a2 = (g, t+4), a3 = (g+8, t+4); tile column 3 is the left halo
          const float* tin = s_in + (DIRECT ? buf * C::STAGE : 0) + sub * C::FIN_SUB + t * G::PLANE +
                             (KIND == K_S2 ? 2 * r0 : r0) * G::PITCH + (KIND == K_S1 ? 3 : 0) + xh * 16 + g;
          const float* wf = s_w + (ch * 9) * NTL * 32 * C::WF + lane * C::WF;
          // TF32 operands: the tensor core reads the top 19 bits of an fp32 register.  3 terms:
          // hi = x rounded to TF32, lo = x - hi (exact; its own low bits fall off at 2^-22 relative)
          auto load_a = [&](const float* p, uint32_t (&ah)[4], uint32_t (&al)[4]) {
            const float av[4] = {p[0], p[8], p[4 * G::PLANE], p[4 * G::PLANE + 8]};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              ah[j] = (TERMS >= 2) ? cv_tf32_hi(av[j]) : __float_as_uint(av[j]);
              al[j] = (TERMS == 3) ? __float_as_uint(av[j] - __uint_as_float(ah[j])) : 0u;
            }
            if (TERMS == 2) {
              // k16 A fragment of the correction instruction: k = {2t, 2t+1} <- a_lo of channels
              // (t, t+4), k = {2t+8, 2t+9} <- a itself; rows g (regs 0, 2) and g+8 (regs 1, 3)
              al[0] = cv_pack_bf16(av[0] - __uint_as_float(ah[0]), av[2] - __uint_as_float(ah[2]));
              al[1] = cv_pack_bf16(av[1] - __uint_as_float(ah[1]), av[3] - __uint_as_float(ah[3]));
              al[2] = cv_pack_bf16(av[0], av[2]);
              al[3] = cv_pack_bf16(av[1], av[3]);
            }
          };
          auto load_b = [&](int k, int i, uint32_t (&bh)[2], uint32_t (&bl)[2]) {
            const float* wp = wf + (k * NTL + i) * 32 * C::WF;
            if (C::PRESPLIT) {
              const float4 b = *reinterpret_cast<const float4*>(wp);
              bh[0] = __float_as_uint(b.x);
              bh[1] = __float_as_uint(b.y);
              bl[0] = __float_as_uint(b.z);
              bl[1] = __float_as_uint(b.w);
            } else {
              const float2 b = *reinterpret_cast<const float2*>(wp);
              bh[0] = (TERMS >= 2) ? cv_tf32_hi(b.x) : __float_as_uint(b.x);
              bh[1] = (TERMS >= 2) ? cv_tf32_hi(b.y) : __float_as_uint(b.y);
              bl[0] = (TERMS == 3) ? __float_as_uint(b.x - __uint_as_float(bh[0])) : 0u;
              bl[1] = (TERMS == 3) ? __float_as_uint(b.y - __uint_as_float(bh[1])) : 0u;
              if (TERMS == 2) {
                bl[0] = cv_pack_bf16(b.x, b.y);
                bl[1] = cv_pack_bf16(b.x - __uint_as_float(bh[0]), b.y - __uint_as_float(bh[1]));
              }
            }
          };
          if constexpr (KIND == K_UP) {
            // stride 2 up (gather form): input pixel (a, x) feeds the outputs (2a+oa, 2x+ob); tap
            // (ky,kx) belongs to class oa = (ky != 1), ob = (kx != 1) and reads the input at
            // (a + (ky == 0), x + (kx == 0)).  The four neighbour fragments stay resident.
            uint32_t ah[2][2][4], al[2][2][4];
#pragma unroll
            for (int dy = 0; dy < 2; ++dy)
#pragma unroll
              for (int dx = 0; dx < 2; ++dx) load_a(tin + dy * G::PITCH + dx, ah[dy][dx], al[dy][dx]);
#pragma unroll
            for (int i = 0; i < NTL; ++i) {
#pragma unroll
              for (int pass = 0; pass < 2; ++pass) {
                // pass 0: classes (0,0) [tap 4] and (1,1) [taps 0,2,6,8]; pass 1: (0,1) [3,5] and (1,0) [1,7]
                constexpr int NTAP = 5;
                const int taps[2][NTAP] = {{4, 0, 2, 6, 8}, {3, 5, 1, 7, -1}};
                uint32_t bh[NTAP][2], bl[NTAP][2];
#pragma unroll
                for (int q = 0; q < NTAP; ++q)
                  if (taps[pass][q] >= 0) load_b(taps[pass][q], i, bh[q], bl[q]);
                if (TERMS >= 2) {
                  // one short chain per tap (a_lo*b_hi, a_hi*b_lo, a_hi*b_hi on a fresh accumulator:
                  // a single truncating add at full magnitude), the taps of the pass interleaved
                  float tq[NTAP][4];
#pragma unroll
                  for (int term = 0; term < 3; ++term)
#pragma unroll
                    for (int q = 0; q < NTAP; ++q) {
                      const int k = taps[pass][q];
                      if (k < 0) continue;
                      const int dy = (k / 3 == 0) ? 1 : 0, dx = (k % 3 == 0) ? 1 : 0;
                      if (TERMS == 2) {
                        if (term == 0) cv_mma_bf16_zero(tq[q], al[dy][dx], bl[q][0], bl[q][1]);
                        else if (term == 2) cv_mma_tf32(tq[q], ah[dy][dx], bh[q][0], bh[q][1]);
                      } else if (term == 0) cv_mma_tf32_zero(tq[q], al[dy][dx], bh[q][0], bh[q][1]);
                      else if (term == 1) cv_mma_tf32(tq[q], ah[dy][dx], bl[q][0], bl[q][1]);
                      else cv_mma_tf32(tq[q], ah[dy][dx], bh[q][0], bh[q][1]);
                    }
#pragma unroll
                  for (int q = 0; q < NTAP; ++q) {
                    const int k = taps[pass][q];
                    if (k < 0) continue;
                    const int cls = 2 * ((k / 3 == 1) ? 0 : 1) + ((k % 3 == 1) ? 0 : 1);
#pragma unroll
                    for (int e = 0; e < 4; ++e) acc[cls][i][e] += tq[q][e];
                  }
                } else {
#pragma unroll
                  for (int q = 0; q < NTAP; ++q) {
                    const int k = taps[pass][q];
                    if (k < 0) continue;
                    const int dy = (k / 3 == 0) ? 1 : 0, dx = (k % 3 == 0) ? 1 : 0;
                    const int cls = 2 * ((k / 3 == 1) ? 0 : 1) + ((k % 3 == 1) ? 0 : 1);
                    cv_mma_tf32(acc[cls][i], ah[dy][dx], bh[q][0], bh[q][1]);
                  }
                }
              }
            }
          } else if constexpr (KIND == K_S2) {
            // stride 2: output row o reads input rows 2o+ky of the tile (5 rows for the warp's 2
            // output rows); the staged rows hold odd columns at [3..], even columns at [EO..], so
            // tap kx reads column offset 3 / EO / 4 with unit stride across the 16 pixels.
            // Per kernel column: the 5 row fragments stay resident, the 3 taps of the column are
            // chained on a fresh accumulator and flushed with one round-to-nearest add.
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
              const int off = (kx == 0) ? 3 : (kx == 1 ? G::EO : 4);
              uint32_t ah[5][4], al[5][4];
#pragma unroll
              for (int ir = 0; ir < 5; ++ir) load_a(tin + ir * G::PITCH + off, ah[ir], al[ir]);
#pragma unroll
              for (int i = 0; i < NTL; ++i) {
                uint32_t bh[3][2], bl[3][2];
#pragma unroll
                for (int ky = 0; ky < 3; ++ky) load_b(ky * 3 + kx, i, bh[ky], bl[ky]);
                if (TERMS == 2) {
                  float tq[2][4];
#pragma unroll
                  for (int o = 0; o < 2; ++o) cv_mma_bf16_zero(tq[o], al[2 * o], bl[0][0], bl[0][1]);
#pragma unroll
                  for (int ky = 1; ky < 3; ++ky)
#pragma unroll
                    for (int o = 0; o < 2; ++o) cv_mma_bf16(tq[o], al[2 * o + ky], bl[ky][0], bl[ky][1]);
#pragma unroll
                  for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int o = 0; o < 2; ++o) cv_mma_tf32(tq[o], ah[2 * o + ky], bh[ky][0], bh[ky][1]);
#pragma unroll
                  for (int o = 0; o < 2; ++o)
#pragma unroll
                    for (int q = 0; q < 4; ++q) acc[o][i][q] += tq[o][q];
                } else if (TERMS == 3) {
                  float tq[2][4];
#pragma unroll
                  for (int o = 0; o < 2; ++o) cv_mma_tf32_zero(tq[o], al[2 * o], bh[0][0], bh[0][1]);
#pragma unroll
                  for (int o = 0; o < 2; ++o) cv_mma_tf32(tq[o], ah[2 * o], bl[0][0], bl[0][1]);
#pragma unroll
                  for (int ky = 1; ky < 3; ++ky) {
#pragma unroll
                    for (int o = 0; o < 2; ++o) cv_mma_tf32(tq[o], al[2 * o + ky], bh[ky][0], bh[ky][1]);
#pragma unroll
                    for (int o = 0; o < 2; ++o) cv_mma_tf32(tq[o], ah[2 * o + ky], bl[ky][0], bl[ky][1]);
                  }
#pragma unroll
                  for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int o = 0; o < 2; ++o) cv_mma_tf32(tq[o], ah[2 * o + ky], bh[ky][0], bh[ky][1]);
#pragma unroll
                  for (int o = 0; o < 2; ++o)
#pragma unroll
                    for (int q = 0; q < 4; ++q) acc[o][i][q] += tq[o][q];
                } else {
#pragma unroll
                  for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int o = 0; o < 2; ++o) cv_mma_tf32(acc[o][i], ah[2 * o + ky], bh[ky][0], bh[ky][1]);
                }
              }
            }
          } else if constexpr (C::ARES) {
            // A-resident order: the 6 input-row fragments of one kx stay in registers, every B
            // fragment is loaded once per tap and feeds the 4 output rows (independent accumulators,
            // issued term by term)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
              uint32_t ah[6][4], al[6][4];
#pragma unroll
              for (int r = 0; r < 6; ++r) load_a(tin + r * G::PITCH + kx, ah[r], al[r]);
              if constexpr (TERMS == 2) {
                // as below with one BF16 k16 instruction per tap for both correction terms
#pragma unroll
                for (int i = 0; i < NTL; ++i) {
                  uint32_t bh[3][2], bl[3][2];
#pragma unroll
                  for (int ky = 0; ky < 3; ++ky) load_b(ky * 3 + kx, i, bh[ky], bl[ky]);
                  float tq[4][4];
#pragma unroll
                  for (int o = 0; o < 4; ++o) cv_mma_bf16_zero(tq[o], al[o], bl[0][0], bl[0][1]);
#pragma unroll
                  for (int ky = 1; ky < 3; ++ky)
#pragma unroll
                    for (int o = 0; o < 4; ++o) cv_mma_bf16(tq[o], al[o + ky], bl[ky][0], bl[ky][1]);
#pragma unroll
                  for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int o = 0; o < 4; ++o) cv_mma_tf32(tq[o], ah[o + ky], bh[ky][0], bh[ky][1]);
#pragma unroll
                  for (int o = 0; o < 4; ++o)
#pragma unroll
                    for (int q = 0; q < 4; ++q) acc[o][i][q] += tq[o][q];
                }
              } else if constexpr (TERMS == 3) {
                // chain over the 3 taps of this kernel column on a fresh accumulator (6 small-term
                // MMAs, then the 3 main terms), then one round-to-nearest add into the running sum
#pragma unroll
                for (int i = 0; i < NTL; ++i) {
                  uint32_t bh[3][2], bl[3][2];
#pragma unroll
                  for (int ky = 0; ky < 3; ++ky) load_b(ky * 3 + kx, i, bh[ky], bl[ky]);
                  float tq[4][4];
#pragma unroll
                  for (int o = 0; o < 4; ++o) cv_mma_tf32_zero(tq[o], al[o], bh[0][0], bh[0][1]);
#pragma unroll
                  for (int o = 0; o < 4; ++o) cv_mma_tf32(tq[o], ah[o], bl[0][0], bl[0][1]);
#pragma unroll
                  for (int ky = 1; ky < 3; ++ky) {
#pragma unroll
                    for (int o = 0; o < 4; ++o) cv_mma_tf32(tq[o], al[o + ky], bh[ky][0], bh[ky][1]);
#pragma unroll
                    for (int o = 0; o < 4; ++o) cv_mma_tf32(tq[o], ah[o + ky], bl[ky][0], bl[ky][1]);
                  }
#pragma unroll
                  for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int o = 0; o < 4; ++o) cv_mma_tf32(tq[o], ah[o + ky], bh[ky][0], bh[ky][1]);
#pragma unroll
                  for (int o = 0; o < 4; ++o)
#pragma unroll
                    for (int q = 0; q < 4; ++q) acc[o][i][q] += tq[o][q];
                }
              } else {
#pragma unroll
                for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                  for (int i = 0; i < NTL; ++i) {
                    uint32_t bh[2], bl[2];
                    load_b(ky * 3 + kx, i, bh, bl);
#pragma unroll
                    for (int o = 0; o < 4; ++o) cv_mma_tf32(acc[o][i], ah[o + ky], bh[0], bh[1]);
                  }
              }
            }
          } else {
            // rolling order (register-light): one input-row fragment at a time; the taps (ky) that
            // use it feed different output rows
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
#pragma unroll
              for (int r = 0; r < 6; ++r) {   // input rows r0 + r (tile row 0 is the top halo)
                uint32_t ah[4], al[4];
                load_a(tin + r * G::PITCH + kx, ah, al);
#pragma unroll
                for (int i = 0; i < NTL; ++i) {
                  uint32_t bh[3][2], bl[3][2];
#pragma unroll
                  for (int ky = 0; ky < 3; ++ky)
                    if (r - ky >= 0 && r - ky <= 3) load_b(ky * 3 + kx, i, bh[ky], bl[ky]);
                  if (TERMS == 2) {
                    float tq[3][4];
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky)
                      if (r - ky >= 0 && r - ky <= 3) cv_mma_bf16_zero(tq[ky], al, bl[ky][0], bl[ky][1]);
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky)
                      if (r - ky >= 0 && r - ky <= 3) cv_mma_tf32(tq[ky], ah, bh[ky][0], bh[ky][1]);
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky)
                      if (r - ky >= 0 && r - ky <= 3) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) acc[r - ky][i][q] += tq[ky][q];
                      }
                  } else if (TERMS == 3) {
                    float tq[3][4];
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky)
                      if (r - ky >= 0 && r - ky <= 3) cv_mma_tf32_zero(tq[ky], al, bh[ky][0], bh[ky][1]);
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky)
                      if (r - ky >= 0 && r - ky <= 3) cv_mma_tf32(tq[ky], ah, bl[ky][0], bl[ky][1]);
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky)
                      if (r - ky >= 0 && r - ky <= 3) cv_mma_tf32(tq[ky], ah, bh[ky][0], bh[ky][1]);
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky)
                      if (r - ky >= 0 && r - ky <= 3) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) acc[r - ky][i][q] += tq[ky][q];
                      }
                  } else {
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky)
                      if (r - ky >= 0 && r - ky <= 3) cv_mma_tf32(acc[r - ky][i], ah, bh[ky][0], bh[ky][1]);
                  }
                }
              }
            }
          }
        }
        __syncthreads();
      }
      if (!tvalid) continue;

      if constexpr (KIND == K_UP) {
        // ---- epilogue, stride-2 up: acc[2*oa+ob][i][j] -> output (2a+oa, 2x+ob), pixel x = ox_in
        // (+8 for j >= 2), channel i*8 + 2t + (j&1); the two column parities form one float2
        const int a_in = ty * G::TH + r0, x_in = tx * TW + xh * 16 + g;
#pragma unroll
        for (int oa = 0; oa < 2; ++oa) {
          // EPI_BWD: all loads of x for this output row are issued before the first one is used
          float2 xv[NTL][4];
          if (EPI == EPI_BWD) {
#pragma unroll
            for (int i = 0; i < NTL; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const int co = i * 8 + 2 * t + (j & 1);
                const float* px = P.x_self + (((size_t)n * CO + co) * H_out + 2 * a_in + oa) * W_out + 2 * (x_in + 8 * (j >> 1));
                asm volatile("ld.global.nc.v2.f32 {%0, %1}, [%2];" : "=f"(xv[i][j].x), "=f"(xv[i][j].y) : "l"(px));
              }
          }
#pragma unroll
          for (int i = 0; i < NTL; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int co = i * 8 + 2 * t + (j & 1);
              const size_t o = (((size_t)n * CO + co) * H_out + 2 * a_in + oa) * W_out + 2 * (x_in + 8 * (j >> 1));
              float v0 = acc[2 * oa][i][j], v1 = acc[2 * oa + 1][i][j];
              if (EPI == EPI_BWD) {
                v0 = dzap(co, v0, xv[i][j].x);
                v1 = dzap(co, v1, xv[i][j].y);
              } else {
                v0 += s_bias[co];
                v1 += s_bias[co];
                if (P.relu_out) {
                  v0 = fmaxf(v0, 0.f);
                  v1 = fmaxf(v1, 0.f);
                }
                st1[i][j & 1] += v0 + v1;
                st2[i][j & 1] = fmaf(v0, v0, fmaf(v1, v1, st2[i][j & 1]));
              }
              if (P.out) *reinterpret_cast<float2*>(P.out + o) = make_float2(v0, v1);
              acc[2 * oa][i][j] = v0;
              acc[2 * oa + 1][i][j] = v1;
            }
        }
        if (want_ts) {
          // border sums of the written dz (mode 0; the stride-2-up kernels never feed a stride-2
          // conv-transpose layer): output (2a+oa, 2x+ob), x = x_in (+8 for j >= 2), channel
          // i*8 + 2t + (j&1).  Totals go to ts_hot (reduced after the tile loop).  Border rows /
          // columns / corners are rare: the per-channel values are moved so that lane L holds
          // channel L and ONE shared atomic per lane follows.
          auto spread = [&](float (&v)[NTL][2], int src_base, int slot) {
            float mine = 0.f;
#pragma unroll
            for (int i = 0; i < NTL; ++i)
#pragma unroll
              for (int c = 0; c < 2; ++c) {
                const float tmp = __shfl_sync(0xffffffffu, v[i][c], src_base + ((lane & 7) >> 1));
                if ((lane >> 3) == i && (lane & 1) == c) mine = tmp;
              }
            if (lane < CO) ts_add(slot, lane, mine);
          };
          const bool tile_c0 = (tx == 0) && (xh == 0);
          const bool tile_cl = (tx == tiles_x - 1) && (TW == 16 || xh == 1);
          float cf[NTL][2], cl[NTL][2];
#pragma unroll
          for (int i = 0; i < NTL; ++i) cf[i][0] = cf[i][1] = cl[i][0] = cl[i][1] = 0.f;
#pragma unroll
          for (int oa = 0; oa < 2; ++oa) {
            const int oy = 2 * a_in + oa;
            const bool rb = (oy == 0) || (oy == H_out - 1);      // warp-uniform
            float rw[NTL][2], c0v[NTL][2], clv[NTL][2];
#pragma unroll
            for (int i = 0; i < NTL; ++i)
#pragma unroll
              for (int c = 0; c < 2; ++c) {
                rw[i][c] = (acc[2 * oa][i][c] + acc[2 * oa + 1][i][c]) + (acc[2 * oa][i][2 + c] + acc[2 * oa + 1][i][2 + c]);
                ts_hot[0][i][c] += rw[i][c];
                c0v[i][c] = acc[2 * oa][i][c];            // output column 0: x = 0 (j < 2), ob = 0, lanes g == 0
                clv[i][c] = acc[2 * oa + 1][i][2 + c];    // last output column: x = W_in-1 (j >= 2), ob = 1, lanes g == 7
                cf[i][c] += c0v[i][c];
                cl[i][c] += clv[i][c];
              }
            if (rb) {
#pragma unroll
              for (int i = 0; i < NTL; ++i)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                  float a = rw[i][c];
                  a += __shfl_xor_sync(0xffffffffu, a, 4);
                  a += __shfl_xor_sync(0xffffffffu, a, 8);
                  a += __shfl_xor_sync(0xffffffffu, a, 16);
                  rw[i][c] = a;
                }
              spread(rw, 0, (oy == 0) ? 1 : 2);
              if (tile_c0) spread(c0v, 0, (oy == 0) ? 5 : 7);
              if (tile_cl) spread(clv, 28, (oy == 0) ? 6 : 8);
            }
          }
          if (tile_c0) spread(cf, 0, 3);
          if (tile_cl) spread(cl, 28, 4);
        }
      } else {
        // ---- epilogue on the accumulator fragments: c0 = (pixel g, channel 2t), c1 = (g, 2t+1),
        // c2 = (g+8, 2t), c3 = (g+8, 2t+1)
        const int oy0 = ty * G::TH + r0, ox0 = tx * TW + xh * 16 + g;
        if (EPI == EPI_BWD) {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            float xs[NTL][4];
#pragma unroll
            for (int i = 0; i < NTL; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const int co = i * 8 + 2 * t + (j & 1);
                const float* px = P.x_self + (((size_t)n * CO + co) * H_out + oy0 + r) * W_out + ox0 + 8 * (j >> 1);
                asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(xs[i][j]) : "l"(px));
              }
#pragma unroll
            for (int i = 0; i < NTL; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) acc[r][i][j] = dzap(i * 8 + 2 * t + (j & 1), acc[r][i][j], xs[i][j]);
          }
        } else {
#pragma unroll
          for (int r = 0; r < R; ++r)
#pragma unroll
            for (int i = 0; i < NTL; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                float v = acc[r][i][j] + s_bias[i * 8 + 2 * t + (j & 1)];
                if (P.relu_out) v = fmaxf(v, 0.f);
                st1[i][j & 1] += v;
                st2[i][j & 1] = fmaf(v, v, st2[i][j & 1]);
                acc[r][i][j] = v;
              }
        }
        if (P.out) {
#pragma unroll
          for (int r = 0; r < R; ++r)
#pragma unroll
            for (int i = 0; i < NTL; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const int co = i * 8 + 2 * t + (j & 1);
                P.out[(((size_t)n * CO + co) * H_out + oy0 + r) * W_out + ox0 + 8 * (j >> 1)] = acc[r][i][j];
              }
        }
        if (want_ts) {
          // border sums of the written dz: element (row oy0+r, column ox0 + 8*(j>>1), channel
          // i*8 + 2t + (j&1)).  Totals / parity classes go to ts_hot (reduced after the tile loop).
          // Border rows / columns / corners are rare: values are moved so that lane L holds
          // channel L, then one shared atomic per lane.
          auto spread = [&](float (&v)[NTL][2], int src_base, int slot) {
            float mine = 0.f;
#pragma unroll
            for (int i = 0; i < NTL; ++i)
#pragma unroll
              for (int c = 0; c < 2; ++c) {
                const float tmp = __shfl_sync(0xffffffffu, v[i][c], src_base + ((lane & 7) >> 1));
                if ((lane >> 3) == i && (lane & 1) == c) mine = tmp;
              }
            if (lane < CO) ts_add(slot, lane, mine);
          };
          const bool tile_c0 = (tx == 0) && (xh == 0);
          const bool tile_cl = (tx == tiles_x - 1) && (TW == 16 || xh == 1);
          if (P.tsum_mode == 0) {
            float cf[NTL][2], cl[NTL][2];
#pragma unroll
            for (int i = 0; i < NTL; ++i) cf[i][0] = cf[i][1] = cl[i][0] = cl[i][1] = 0.f;
#pragma unroll
            for (int r = 0; r < R; ++r) {
              const int oy = oy0 + r;
              const bool rb = (oy == 0) || (oy == H_out - 1);    // warp-uniform
              float rw[NTL][2], c0v[NTL][2], clv[NTL][2];
#pragma unroll
              for (int i = 0; i < NTL; ++i)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                  rw[i][c] = acc[r][i][c] + acc[r][i][2 + c];
                  ts_hot[0][i][c] += rw[i][c];
                  c0v[i][c] = acc[r][i][c];         // column 0 lives in lanes g == 0 (j < 2)
                  clv[i][c] = acc[r][i][2 + c];     // the last column in lanes g == 7 (j >= 2)
                  cf[i][c] += c0v[i][c];
                  cl[i][c] += clv[i][c];
                }
              if (rb) {
#pragma unroll
                for (int i = 0; i < NTL; ++i)
#pragma unroll
                  for (int c = 0; c < 2; ++c) {
                    float a = rw[i][c];
                    a += __shfl_xor_sync(0xffffffffu, a, 4);
                    a += __shfl_xor_sync(0xffffffffu, a, 8);
                    a += __shfl_xor_sync(0xffffffffu, a, 16);
                    rw[i][c] = a;
                  }
                spread(rw, 0, (oy == 0) ? 1 : 2);
                if (tile_c0) spread(c0v, 0, (oy == 0) ? 5 : 7);
                if (tile_cl) spread(clv, 28, (oy == 0) ? 6 : 8);
              }
            }
            if (tile_c0) spread(cf, 0, 3);
            if (tile_cl) spread(cl, 28, 4);
          } else {
            // mode 1: row-parity x column-parity classes (the column parity of this lane's pixels
            // is g & 1: tile origins and the +8 step are even; oy0 is even, so row parity = r & 1),
            // last row by column parity, last column by row parity, last corner
            float lc[2][NTL][2];
#pragma unroll
            for (int rp = 0; rp < 2; ++rp)
#pragma unroll
              for (int i = 0; i < NTL; ++i) lc[rp][i][0] = lc[rp][i][1] = 0.f;
#pragma unroll
            for (int r = 0; r < R; ++r) {
              float rw[NTL][2], clv[NTL][2];
#pragma unroll
              for (int i = 0; i < NTL; ++i)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                  rw[i][c] = acc[r][i][c] + acc[r][i][2 + c];
                  clv[i][c] = acc[r][i][2 + c];
                  ts_hot[r & 1][i][c] += rw[i][c];
                  lc[r & 1][i][c] += clv[i][c];
                }
              if (oy0 + r == H_out - 1) {                       // warp-uniform
#pragma unroll
                for (int i = 0; i < NTL; ++i)
#pragma unroll
                  for (int c = 0; c < 2; ++c) {
                    float a = rw[i][c];
                    a += __shfl_xor_sync(0xffffffffu, a, 8);
                    a += __shfl_xor_sync(0xffffffffu, a, 16);
                    rw[i][c] = a;                               // lanes g = 0 / 1: even / odd columns
                  }
                spread(rw, 0, 4);
                spread(rw, 4, 5);
                if (tile_cl) spread(clv, 28, 8);
              }
            }
            if (tile_cl) {
              spread(lc[0], 28, 6);
              spread(lc[1], 28, 7);
            }
          }
        }
      }
      // this tile's statistics: lanes sharing t hold the same channels -> xor-shuffle over g, then
      // lanes 0..3 add to the warp's fp64 slots
      if (want_stats) {
#pragma unroll
        for (int i = 0; i < NTL; ++i)
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            float a = st1[i][j], b = st2[i][j];
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {
              a += __shfl_xor_sync(0xffffffffu, a, o);
              b += __shfl_xor_sync(0xffffffffu, b, o);
            }
            if (g == 0) {
              s_accd[i * 8 + 2 * t + j] += (double)a;
              s_accd[32 + i * 8 + 2 * t + j] += (double)b;
            }
          }
      }
    }

    // ---- fixed-order sum over the warps, one fp64 atomic per channel per CTA
    double* dst = (EPI == EPI_FWD) ? P.stats_out : nullptr;
    if (dst != nullptr) {
      __syncthreads();
      if (tid < CO) {
        const double* sd = reinterpret_cast<const double*>(s_red);
        double a = 0.0, b = 0.0;
#pragma unroll
        for (int w = 0; w < NT / 32; ++w) {
          a += sd[w * 64 + tid];
          b += sd[w * 64 + 32 + tid];
        }
        atomicAdd(&dst[tid], a);
        atomicAdd(&dst[32 + tid], b);
      }
    }
    if (want_ts) {
      // this warp's totals / classes: shuffle over g (mode 1: over the lanes of equal column
      // parity g & 1), one add per lane into the warp's own fp64 slots; then the warps are summed
      // in a fixed order and every value goes out as one fp64 atomic per CTA
      double* tw = s_tsw + warp * 128;
#pragma unroll
      for (int rp = 0; rp < 2; ++rp)
#pragma unroll
        for (int i = 0; i < NTL; ++i)
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            float a = ts_hot[rp][i][c];
            if (P.tsum_mode == 0) a += __shfl_xor_sync(0xffffffffu, a, 4);
            a += __shfl_xor_sync(0xffffffffu, a, 8);
            a += __shfl_xor_sync(0xffffffffu, a, 16);
            if (P.tsum_mode == 0) {
              if (rp == 0 && g == 0) tw[i * 8 + 2 * t + c] = (double)a;
            } else if (g < 2) {
              tw[(rp * 2 + g) * 32 + i * 8 + 2 * t + c] = (double)a;
            }
          }
      __syncthreads();
      const int nhot = (P.tsum_mode == 0) ? 32 : 128;
      for (int i = tid; i < nhot; i += NT) {
        double a = 0.0;
#pragma unroll
        for (int w = 0; w < NT / 32; ++w) a += s_tsw[w * 128 + i];
        s_ts[i] = a;
      }
      __syncthreads();
      for (int i = tid; i < 288; i += NT)
        if ((i & 31) < CO && s_ts[i] != 0.0) atomicAdd(&P.tsums_out[i], s_ts[i]);
    }
  } else {
    // ---------------------------------------------------------------- fp32 SIMT path
  const int sub = tid / (64 * NCOG);
  const int t2 = tid - sub * (64 * NCOG);
  const int slot = t2 & 63;
  const int cog = t2 >> 6;
  const int lx = slot % TW;
  const int rg = slot / TW;

  float st1[COT], st2[COT];
#pragma unroll
  for (int c = 0; c < COT; ++c) st1[c] = st2[c] = 0.f;
  // EPI_BWD border sums: totals / parity classes of the written dz (see the tensor-core path)
  float ts_hot[2][COT];
#pragma unroll
  for (int c = 0; c < COT; ++c) ts_hot[0][c] = ts_hot[1][c] = 0.f;

  uint32_t phase = 0;
  int it = 0;
  for (int grp = blockIdx.x; grp < ngroups; grp += gridDim.x) {
    const int tile = grp * NSUB + sub;
    const bool tvalid = tile < ntiles;
    const int n = tile / tiles_per_img;
    const int trem = tile - n * tiles_per_img;
    const int ty = trem / tiles_x, tx = trem - ty * tiles_x;
    if (EPI == EPI_BWD && tvalid) prefetch_x(n, ty, tx, t2, 64 * NCOG);

    float acc[NOUT][COT];
#pragma unroll
    for (int o = 0; o < NOUT; ++o)
#pragma unroll
      for (int c = 0; c < COT; ++c) acc[o][c] = 0.f;

#pragma unroll 1
    for (int ch = 0; ch < NCHUNK; ++ch, ++it) {
      const int buf = DIRECT ? (it & 1) : 0;
      cv_mbar_wait(s_bar, phase);  // this stage's boxes have landed
      phase ^= 1;
      if (!DIRECT) transform(grp, ch);
      __syncthreads();  // everyone has seen this phase (and, if staged, the tile is ready)
      // prefetch the next stage while computing this one
      if (ch + 1 < NCHUNK) {
        issue(grp, ch + 1, buf ^ 1);
      } else if (grp + (int)gridDim.x < ngroups) {
        issue(grp + gridDim.x, 0, buf ^ 1);
      }
      if (tvalid) {
        const float* s_mine = s_in + (DIRECT ? buf * C::STAGE : 0) + sub * C::FIN_SUB;
#pragma unroll 2
        for (int ci = 0; ci < CIC; ++ci) {
          const float* tw = s_w + ((ch * CIC + ci) * 9) * CO + cog * COT;
          if (KIND == K_S1) {
            const float* tin = s_mine + ci * G::PLANE + (4 * rg) * G::PITCH + lx + 3;
            float v[6][3];
#pragma unroll
            for (int r = 0; r < 6; ++r)
#pragma unroll
              for (int c = 0; c < 3; ++c) v[r][c] = tin[r * G::PITCH + c];
#pragma unroll
            for (int k = 0; k < 9; ++k) {
              float wv[COT];
#pragma unroll
              for (int c = 0; c < COT; ++c) wv[c] = tw[k * CO + c];
#pragma unroll
              for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < COT; ++c) acc[r][c] = fmaf(v[r + k / 3][k % 3], wv[c], acc[r][c]);
            }
          } else if (KIND == K_S2) {
            const float* tin = s_mine + ci * G::PLANE + (8 * rg) * G::PITCH;
            float v[9][3];
#pragma unroll
            for (int r = 0; r < 9; ++r) {
              v[r][0] = tin[r * G::PITCH + 3 + lx];       // input col 2x-1
              v[r][1] = tin[r * G::PITCH + G::EO + lx];   // input col 2x
              v[r][2] = tin[r * G::PITCH + 4 + lx];       // input col 2x+1
            }
#pragma unroll
            for (int k = 0; k < 9; ++k) {
              float wv[COT];
#pragma unroll
              for (int c = 0; c < COT; ++c) wv[c] = tw[k * CO + c];
#pragma unroll
              for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < COT; ++c) acc[r][c] = fmaf(v[2 * r + k / 3][k % 3], wv[c], acc[r][c]);
            }
          } else {
            const float* tin = s_mine + ci * G::PLANE + (2 * rg) * G::PITCH + lx;
            float v[3][2];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
              v[r][0] = tin[r * G::PITCH];
              v[r][1] = tin[r * G::PITCH + 1];
            }
            // out index o = a*4 + oa*2 + ob  (a: input row of the pair, oa/ob: output parity)
#pragma unroll
            for (int k = 0; k < 9; ++k) {
              const int ky = k / 3, kx = k % 3;
              float wv[COT];
#pragma unroll
              for (int c = 0; c < COT; ++c) wv[c] = tw[k * CO + c];
              // output parity this tap feeds, and which neighbour it reads
              const int oa = (ky == 1) ? 0 : 1, dy = (ky == 0) ? 1 : 0;
              const int ob = (kx == 1) ? 0 : 1, dx = (kx == 0) ? 1 : 0;
#pragma unroll
              for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int c = 0; c < COT; ++c)
                  acc[a * 4 + oa * 2 + ob][c] = fmaf(v[a + dy][dx], wv[c], acc[a * 4 + oa * 2 + ob][c]);
            }
          }
        }
      }
      __syncthreads();  // FMA loop done with this tile before it is overwritten
    }
    if (!tvalid) continue;

    // ---- epilogue (the next tile group's loads are already in flight)
    if (EPI == EPI_BWD) {
      // all NOUT*COT loads of x are issued before the first one is used
      float xs[NOUT][COT];
#pragma unroll
      for (int o = 0; o < NOUT; ++o) {
        int oy, ox;
        if (KIND == K_UP) {
          oy = 2 * (ty * G::TH + 2 * rg + (o >> 2)) + ((o >> 1) & 1);
          ox = 2 * (tx * TW + lx) + (o & 1);
        } else {
          oy = ty * G::TH + 4 * rg + o;
          ox = tx * TW + lx;
        }
#pragma unroll
        for (int c = 0; c < COT; ++c) {
          const int co = cog * COT + c;
          const float* px = P.x_self + (((size_t)n * CO + co) * H_out + oy) * W_out + ox;
          asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(xs[o][c]) : "l"(px));
        }
      }
#pragma unroll
      for (int o = 0; o < NOUT; ++o)
#pragma unroll
        for (int c = 0; c < COT; ++c) acc[o][c] = dzap(cog * COT + c, acc[o][c], xs[o][c]);
    } else {
#pragma unroll
      for (int o = 0; o < NOUT; ++o)
#pragma unroll
        for (int c = 0; c < COT; ++c) {
          float v = acc[o][c] + s_bias[cog * COT + c];
          if (P.relu_out) v = fmaxf(v, 0.f);
          st1[c] += v;
          st2[c] = fmaf(v, v, st2[c]);
          acc[o][c] = v;
        }
    }
    if (P.out) {
      if (KIND == K_UP) {
#pragma unroll
        for (int o = 0; o < NOUT; o += 2) {
          int oy = 2 * (ty * G::TH + 2 * rg + (o >> 2)) + ((o >> 1) & 1);
          int ox = 2 * (tx * TW + lx);
#pragma unroll
          for (int c = 0; c < COT; ++c) {
            const int co = cog * COT + c;
            float2* dst = reinterpret_cast<float2*>(P.out + (((size_t)n * CO + co) * H_out + oy) * W_out + ox);
            *dst = make_float2(acc[o][c], acc[o + 1][c]);
          }
        }
      } else {
#pragma unroll
        for (int o = 0; o < NOUT; ++o) {
          int oy = ty * G::TH + 4 * rg + o;
          int ox = tx * TW + lx;
#pragma unroll
          for (int c = 0; c < COT; ++c) {
            const int co = cog * COT + c;
            P.out[(((size_t)n * CO + co) * H_out + oy) * W_out + ox] = acc[o][c];
          }
        }
      }
    }
    if (want_ts) {
      // border sums of the written dz.  Lanes of a row group run along x (lx); a row group is a
      // whole warp (TW == 32) or a half warp (TW == 16).  Totals / parity classes: xor-shuffle
      // reduction over the WARP (the butterfly leaves the sum in every lane), then lane k adds
      // value k to this warp's own fp64 slot k (no atomics, one add per lane).  Border rows /
      // columns / corners are rare: one shared atomic per lane after the same kind of spreading.
      const int lane = tid & 31;
      // v[c] valid in lane `src` of every row group -> channel c to lane c of that group -> atomic
      auto spread_from = [&](float (&v)[COT], int src, int slot, bool on) {
        float mine = 0.f;
#pragma unroll
        for (int c = 0; c < COT; ++c) {
          const float tmp = __shfl_sync(0xffffffffu, v[c], (lane & ~(TW - 1) & 31) + src);
          if (lx == c) mine = tmp;
        }
        if (on && lx < COT) ts_add(slot, cog * COT + lx, mine);
      };
      const bool tile_c0 = (tx == 0), tile_cl = (tx == tiles_x - 1);
      if (P.tsum_mode == 0) {
        float cfv[COT], clv[COT];
#pragma unroll
        for (int c = 0; c < COT; ++c) cfv[c] = clv[c] = 0.f;
#pragma unroll
        for (int o = 0; o < NOUT; ++o) {
          int oy;
          bool is_c0, is_cl;     // does this element sit in the first / last output column (owner lanes only)
          if (KIND == K_UP) {
            oy = 2 * (ty * G::TH + 2 * rg + (o >> 2)) + ((o >> 1) & 1);
            is_c0 = (o & 1) == 0;      // column 2*lx + ob: first for lx == 0, ob == 0
            is_cl = (o & 1) == 1;      // last for lx == TW-1, ob == 1
          } else {
            oy = ty * G::TH + 4 * rg + o;
            is_c0 = is_cl = true;
          }
          const bool rb = (oy == 0) || (oy == H_out - 1);      // uniform over the row group
          float rv[COT];
#pragma unroll
          for (int c = 0; c < COT; ++c) {
            rv[c] = acc[o][c];
            ts_hot[0][c] += rv[c];
          }
          if (tile_c0 && is_c0) {
#pragma unroll
            for (int c = 0; c < COT; ++c) cfv[c] += rv[c];
          }
          if (tile_cl && is_cl) {
#pragma unroll
            for (int c = 0; c < COT; ++c) clv[c] += rv[c];
          }
          // (TW == 16: the two half warps may differ in rb; shuffles run warp-wide, the atomic is predicated)
          const bool any_rb = __any_sync(0xffffffffu, rb);
          if (any_rb) {
            if (tile_c0 && is_c0) spread_from(rv, 0, (oy == 0) ? 5 : 7, rb);
            if (tile_cl && is_cl) spread_from(rv, TW - 1, (oy == 0) ? 6 : 8, rb);
#pragma unroll
            for (int c = 0; c < COT; ++c) {
#pragma unroll
              for (int sh = 1; sh < TW; sh <<= 1) rv[c] += __shfl_xor_sync(0xffffffffu, rv[c], sh);
            }
            spread_from(rv, 0, (oy == 0) ? 1 : 2, rb);
          }
        }
        if (tile_c0) spread_from(cfv, 0, 3, true);
        if (tile_cl) spread_from(clv, TW - 1, 4, true);
      } else if (KIND != K_UP) {
        // mode 1: parity classes (row parity = o & 1, column parity = lx & 1: tile origins are even)
        float lcv[2][COT];
#pragma unroll
        for (int c = 0; c < COT; ++c) lcv[0][c] = lcv[1][c] = 0.f;
#pragma unroll
        for (int o = 0; o < NOUT; ++o) {
          const int oy = ty * G::TH + 4 * rg + o;
          const bool last_row = (oy == H_out - 1);              // uniform over the row group
          float rv[COT];
#pragma unroll
          for (int c = 0; c < COT; ++c) {
            rv[c] = acc[o][c];
            ts_hot[o & 1][c] += rv[c];
          }
          if (tile_cl) {
#pragma unroll
            for (int c = 0; c < COT; ++c) lcv[o & 1][c] += rv[c];
          }
          if (__any_sync(0xffffffffu, last_row)) {
            if (tile_cl) spread_from(rv, TW - 1, 8, last_row);
#pragma unroll
            for (int c = 0; c < COT; ++c) {
#pragma unroll
              for (int sh = 2; sh < TW; sh <<= 1) rv[c] += __shfl_xor_sync(0xffffffffu, rv[c], sh);
            }
            spread_from(rv, 0, 4, last_row);      // lane 0 of the group: even columns
            spread_from(rv, 1, 5, last_row);      // lane 1: odd columns
          }
        }
        if (tile_cl) {
          spread_from(lcv[0], TW - 1, 6, true);
          spread_from(lcv[1], TW - 1, 7, true);
        }
      }
    }
  }
  if (want_ts) {
    // this warp's totals / classes: butterfly over the warp (mode 1: over the lanes of equal
    // column parity), lane k writes value k to the warp's own fp64 slots; then as above
    const int lane = tid & 31;
    double* tw = s_tsw + (tid >> 5) * 128;
    float mine = 0.f;
#pragma unroll
    for (int rp = 0; rp < 2; ++rp)
#pragma unroll
      for (int c = 0; c < COT; ++c) {
        float a = ts_hot[rp][c];
        if (P.tsum_mode == 0) a += __shfl_xor_sync(0xffffffffu, a, 1);
#pragma unroll
        for (int sh = 2; sh < 32; sh <<= 1) a += __shfl_xor_sync(0xffffffffu, a, sh);
        if (P.tsum_mode == 0 ? (rp == 0 && lane == c) : ((lane >> 1) == rp * COT + c)) mine = a;
      }
    if (P.tsum_mode == 0) {
      if (lane < COT) tw[cog * COT + lane] = (double)mine;
    } else if ((lane >> 1) < 2 * COT) {
      const int rp = (lane >> 1) / COT, c = (lane >> 1) % COT;
      tw[(rp * 2 + (lane & 1)) * 32 + cog * COT + c] = (double)mine;
    }
    __syncthreads();
    const int nhot = (P.tsum_mode == 0) ? 32 : 128;
    for (int i = tid; i < nhot; i += NT) {
      double a = 0.0;
#pragma unroll
      for (int w = 0; w < NT / 32; ++w) a += s_tsw[w * 128 + i];
      s_ts[i] = a;
    }
    __syncthreads();
    for (int i = tid; i < 288; i += NT)
      if ((i & 31) < CO && s_ts[i] != 0.0) atomicAdd(&P.tsums_out[i], s_ts[i]);
  }

  // ---- per-channel statistics: warp shuffle -> per-warp smem slots -> fixed-order sum ->
  // one fp64 atomic per channel per CTA (the in-CTA part is deterministic)
  double* dst = (EPI == EPI_FWD) ? P.stats_out : nullptr;
  if (dst != nullptr) {
    const int warp = tid >> 5;
#pragma unroll
    for (int c = 0; c < COT; ++c) {
      float a = warp_sum(st1[c]);
      float b = warp_sum(st2[c]);
      if ((tid & 31) == 0) {
        s_red[warp * 16 + c] = a;
        s_red[warp * 16 + 8 + c] = b;
      }
    }
    __syncthreads();
    if (tid < CO) {
      const int mycog = tid / COT, c = tid % COT;
      float a = 0.f, b = 0.f;
      for (int w = 0; w < NT / 32; ++w) {
        const int wcog = ((w * 32) % (64 * NCOG)) >> 6;
        if (wcog == mycog) {
          a += s_red[w * 16 + c];
          b += s_red[w * 16 + 8 + c];
        }
      }
      atomicAdd(&dst[tid], (double)a);
      atomicAdd(&dst[32 + tid], (double)b);
    }
  }
  }
}

// [B*C, H, W] fp32 activation tensor -> boxes [CIC][IN_ROWS][RAW_PITCH], no swizzle, zero fill
static int make_act_map(CUtensorMap* map, const float* base, long long nc, int H, int W, int box_w, int box_h,
                        int box_c) {
  TensorMapEncodeFn fn = get_tensor_map_encode_fn();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled unavailable");
    return 1;
  }
  cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)nc};
  cuuint64_t strides[2] = {(cuuint64_t)W * 4, (cuuint64_t)H * W * 4};
  cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)box_c};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(activation) failed (%d)", (int)r);
    return 1;
  }
  return 0;
}

// 0: fp32 SIMT; 1: TF32 tensor cores; 3: error-compensated 3xTF32 (layers the tensor-core path covers)
static int g_conv_terms = 0;
// 3-term layers: correction terms as half-rate BF16 k16 instructions (cv_pack_bf16), a bit mask:
// 1 = the weight-gradient kernels, 2 = the backward-data kernels, 4 = the forward kernels, 8 = the
// forward kernels of the decoder (layers 7..13) only
// (ava_b200_set_conv_precision: mode 3 = 1, mode 5 = 1|2, mode 6 = 1|2|8, mode 4 = 1|2|4; mode 2 keeps
// all three terms in TF32)
static int g_conv_bf16corr = 0;

template <int KIND, int CI, int CO, int TW, int INMODE, int EPI, int HIN, int TERMS = 0>
static int launch_gconv(const GconvParams& P, cudaStream_t stream) {
  using C = GconvCfg<KIND, CI, CO, TW, INMODE, TERMS>;
  using G = typename C::G;
  const size_t smem = (size_t)(C::BUF_FLOATS + C::W_FLOATS + 64 + C::RED_FLOATS + 32) * sizeof(float) +
                      (128 + 288 + (EPI == EPI_BWD ? (C::NT / 32) * 128 : 0)) * sizeof(double) + 16 + 128;
  if (P.H_in != HIN || P.W_in != HIN) {
    set_error("gconv: layer geometry mismatch");
    return 1;
  }
  auto kern = gconv_kernel<KIND, CI, CO, TW, INMODE, EPI, HIN, TERMS>;
  static int max_ctas = 0;
  if (max_ctas == 0) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
      cudaGetLastError();
      set_error("gconv: cannot reserve %zu bytes of shared memory", smem);
      return 1;
    }
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, C::NT, smem);
    if (per_sm < 1) per_sm = 1;
    max_ctas = per_sm * kNumSMs;
  }
  const int H_out = (KIND == K_S1) ? P.H_in : (KIND == K_S2 ? P.H_in / 2 : P.H_in * 2);
  const int W_out = (KIND == K_S1) ? P.W_in : (KIND == K_S2 ? P.W_in / 2 : P.W_in * 2);
  const int tiles_x = ((KIND == K_UP) ? P.W_in : W_out) / TW;
  const int tiles_y = ((KIND == K_UP) ? P.H_in : H_out) / G::TH;
  const long long ntiles = (long long)P.B * tiles_x * tiles_y;
  if (ntiles == 0) return 0;
  CUtensorMap map_in;
  if (make_act_map(&map_in, P.in, (long long)P.B * CI, P.H_in, P.W_in, C::BOX_W, G::IN_ROWS, C::CIC)) return 1;
  const long long ngroups = (ntiles + C::NSUB - 1) / C::NSUB;
  int grid = (int)(ngroups < max_ctas ? ngroups : max_ctas);
  kern<<<grid, C::NT, smem, stream>>>(map_in, P);
  return check_launch("gconv");
}

// ------------------------------------------------------------------------------------
// Weight gradient.  D[g][i][k] = sum_{n,y,x} Gt[n,g,y,x] * It[n,i,S*y+ky-1,S*x+kx-1]
//   conv layers : Gt = dz (DZ loader),    It = x - mean (zero padded), D ~ dW[co][ci][3][3]
//   convT layers: Gt = x - mean,          It = dz (DZ),                D ~ dW[ci][co][3][3]
// The kernels accumulate the CENTRED RAW product Rc = sum dz * (x - mean)_pad; the finalize pass
// (bnconv_finalize_kernel) turns it into the weight gradient
//   dW = gamma*invstd * Rc + beta * T_k        T_k[co] = sum of dz over the pixels whose tap-k
//                                              partner lies inside the image
// AND into this layer's two BatchNorm-backward reductions, which are linear in the same sums:
//   sum_q g[ci,q]              = sum_{co,k} W[co,ci,k] * T_k[co]
//   sum_q g[ci,q]*(x-mean)[q]  = sum_{co,k} W[co,ci,k] * Rc[co,ci,k]       (g = conv-transpose(dz, W))
// so the backward-data kernel of the same layer can apply the BatchNorm backward in its
// epilogue without a separate pass over g (measured equivalence: profiles/probes/
// exp_algebraic_dstats.py -- the algebraic values agree with epilogue-accumulated ones to 1e-8
// of the gradient's scale, and the whole-model gradients are unchanged at the 1e-6 level).
// Each thread owns GT g-channels x one i-channel x 9 taps in registers and walks 4-pixel
// strips of the tile; thread groups split the strips; partial sums live in registers
// across the CTA's whole persistent loop and are reduced once at the end
// (smem -> per-CTA partial in the workspace -> deterministic second-stage sum).
struct WgradParams {
  const float* g_a;  // "G" tensor (low resolution when S == 2): conv layers dz, convT layers x
  const float* i_a;  // "I" tensor: conv layers x, convT layers dz
  // BatchNorm of this layer (applied to x on load)
  const float* gamma;
  const float* beta;
  const double* stats;
  double bn_count;
  // eval mode (train == 0): x is centred at the running mean instead of the batch mean
  const float* rmean;
  int train;
  float* partial;  // [grid][CG*CI*9 + 32]
  int B, Hg, Wg;   // dims of the G tensor
};

template <int S, int TWG>
struct WTile {
  static constexpr int THG = (S == 1) ? 256 / TWG : 8;  // S1: 32x8 or 16x16 ; S2: TWGx8
  static constexpr int I_ROWS = S * THG + (S == 1 ? 2 : 1);
  // I rows (one TMA box row, first column = input column X0-4 because the TMA start coordinate
  // must be 16-byte aligned): [3] = left halo (X0-1), [4 .. 4+S*TWG-1] interior, then the right
  // halo (S1).  Stride-1 pitches are padded so that the channel-plane stride is 8/24 (mod 32).
  static constexpr int I_PITCH = (S == 1) ? (TWG == 32 ? 44 : 28) : 2 * TWG + 4;
  static constexpr int I_PLANE_RAW = I_ROWS * I_PITCH;
  // dense planes: the whole I tile is one TMA box (plane stride is 4 (mod 32) floats for the
  // stride-2 tiles, i.e. conflict-free across channel planes; 8 (mod 32) for stride 1)
  static constexpr int I_PLANE = I_PLANE_RAW;
  static constexpr int G_PLANE = THG * TWG;  // dense: the whole G tile is one TMA box
  static constexpr int NSTRIPS = THG * TWG / 4;
};

// CONVT == 0: G uses the DZ loader, I the AFFINE loader; CONVT == 1: the other way round.
// Staging: TMA boxes land directly in the layout the FMA loop reads (G: one [CG][THG][TWG] box;
// I: one [CI][I_ROWS][I_PITCH] box, halo columns and image borders zero-filled by the TMA unit), then a table-driven pass transforms them IN PLACE (BN apply on one side,
// next-BN backward + ReLU backward on the other, literal zeros for padding).
template <int S, int CG, int CI, int TWG, int CONVT>
__global__ void __launch_bounds__(256, 2)
    wgrad_kernel(const __grid_constant__ CUtensorMap map_g, const __grid_constant__ CUtensorMap map_i,
                 const WgradParams P) {
  using T = WTile<S, TWG>;
  constexpr int GT = (CI == 1) ? 1 : 8;   // g-channels per thread
  constexpr int NGQ = CG / GT;
  constexpr int NSLOT = NGQ * CI;         // (gq, i) pairs
  constexpr int NPG = 256 / NSLOT;        // pixel groups
  constexpr int NACT = NPG * NSLOT;       // active threads
  // one g-channel per thread (CI == 1): lanes differ in the g-channel, so the G planes are padded
  // to 4 (mod 32) floats (box with 4 spare columns and one spare row) against bank conflicts
  constexpr int GW = (CI == 1) ? TWG + 4 : TWG, GROWS = (CI == 1) ? T::THG + 1 : T::THG;
  constexpr int GPL = GW * GROWS;
  constexpr int G_FLOATS = CG * GPL;
  constexpr int I_FLOATS = CI * T::I_PLANE;
  constexpr int G_PAD = (G_FLOATS + 31) / 32 * 32;
  constexpr int I_PAD = (I_FLOATS + 31) / 32 * 32;
  constexpr int NQG = CG * T::THG * (TWG / 4);                 // G quads
  constexpr int NQI = CI * T::I_ROWS * (T::I_PITCH / 4);       // I quads
  constexpr int GITERS = (NQG + 255) / 256;
  constexpr int IITERS = (NQI + 255) / 256;

  // double buffering (the next tile's boxes fly while this one is transformed and consumed) when
  // two stages leave room for >= 2 CTAs per SM
  // (measured: pays for the small tiles and for the convT layers, whose in-place transform only
  // touches the small G tile)
  constexpr bool DB = (G_PAD + I_PAD) * 4 <= (CONVT ? 48 : 40) * 1024;
  constexpr int NSTG = DB ? 2 : 1;
  extern __shared__ __align__(128) float smem[];
  float* s_aff = smem + NSTG * (G_PAD + I_PAD);        // BN coefs: scale[32] | shift[32]
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_aff + 64);   // [NSTG]

  const int tid = threadIdx.x;
  const bool active = tid < NACT;
  const int slot = tid % NSLOT;
  const int pg = tid / NSLOT;
  const int ti = slot % CI;
  const int gq = slot / CI;

  const int Hg = P.Hg, Wg = P.Wg, Hi = S * Hg, Wi = S * Wg;
  const int tiles_x = Wg / TWG, tiles_y = Hg / T::THG;
  const int tiles_per_img = tiles_x * tiles_y;
  const int ntiles = P.B * tiles_per_img;

  if (tid == 0) {
    cv_mbar_init(&s_bar[0], 1);
    if (DB) cv_mbar_init(&s_bar[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // TMA: boxes of `tile` into stage `st` (thread 0)
  auto issue = [&](int tile, int st) {
    const int n = tile / tiles_per_img;
    const int trem = tile - n * tiles_per_img;
    const int ty = trem / tiles_x, tx = trem - ty * tiles_x;
    constexpr uint32_t BYTES = (uint32_t)(G_FLOATS * 4 + CI * T::I_PLANE_RAW * 4);
    float* sg = smem + st * (G_PAD + I_PAD);
    cv_mbar_expect_tx(&s_bar[st], BYTES);
    cv_tma_load_3d(sg, &map_g, tx * TWG, ty * T::THG, n * CG, &s_bar[st]);
    cv_tma_load_3d(sg + G_PAD, &map_i, S * tx * TWG - 4, S * ty * T::THG - 1, n * CI, &s_bar[st]);
  };
  // coefficients
  if (tid < 32) {
    const int c = tid;
    constexpr int CA = CONVT ? CG : CI;  // channels of x
    if (c < CA) {
      // centred raw input: x - mean (mean rounded to fp32; the finalize pass corrects for the
      // rounding and applies gamma*invstd / beta, see bnconv_finalize_kernel); eval mode: x - running mean
      const float mean =
          P.train ? bn_coef(P.stats, c, P.bn_count, nullptr, nullptr, nullptr, nullptr, true).mean : P.rmean[c];
      s_aff[c] = 1.f;
      s_aff[32 + c] = -mean;
    }
  }
  // per-thread transform work lists (identical for every tile)
  int g_off[GITERS], g_ch[GITERS];
#pragma unroll
  for (int j = 0; j < (CONVT ? GITERS : 0); ++j) {
    const int t = tid + j * 256;
    g_ch[j] = -1;
    g_off[j] = 0;
    if (t < NQG) {
      const int q = t % (TWG / 4);
      const int y = (t / (TWG / 4)) % T::THG;
      const int c = t / ((TWG / 4) * T::THG);
      g_off[j] = c * GPL + y * GW + 4 * q;
      g_ch[j] = c;
    }
  }
  int i_off[IITERS], i_meta[IITERS];   // meta: channel | row<<8 | quad<<16, -1 = none
#pragma unroll
  for (int j = 0; j < (CONVT ? 0 : IITERS); ++j) {
    const int t = tid + j * 256;
    i_meta[j] = -1;
    i_off[j] = 0;
    if (t < NQI) {
      const int q = t % (T::I_PITCH / 4);
      const int y = (t / (T::I_PITCH / 4)) % T::I_ROWS;
      const int c = t / ((T::I_PITCH / 4) * T::I_ROWS);
      i_off[j] = c * T::I_PLANE + y * T::I_PITCH + 4 * q;
      i_meta[j] = c | (y << 8) | (q << 16);
    }
  }

  float acc[GT][9];
#pragma unroll
  for (int g = 0; g < GT; ++g)
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[g][k] = 0.f;
  // bias gradient: conv layers sum dz == G (threads with ti == 0, one value per owned g);
  // convT layers sum dz == I over the pixels a strip covers (threads with gq == 0, bs[0]).
  float bs[GT];
#pragma unroll
  for (int g = 0; g < GT; ++g) bs[g] = 0.f;

  __syncthreads();   // barriers initialised
  if (DB && tid == 0 && (int)blockIdx.x < ntiles) issue(blockIdx.x, 0);
  int it = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
    const int st = DB ? (it & 1) : 0;
    const int n = tile / tiles_per_img;
    const int trem = tile - n * tiles_per_img;
    const int ty = trem / tiles_x, tx = trem - ty * tiles_x;
    const int gy0 = ty * T::THG, gx0 = tx * TWG;
    const int iy0 = S * gy0 - 1;
    const int X0 = S * gx0;
    (void)gy0;
    float* s_g = smem + st * (G_PAD + I_PAD);           // [CG][G_PLANE]
    float* s_i = s_g + G_PAD;                            // [CI][I_PLANE]
    __syncthreads();  // previous tile's FMA loop is done with the buffers
    if (tid == 0) {
      if (!DB) issue(tile, 0);
      else if (tile + (int)gridDim.x < ntiles) issue(tile + gridDim.x, st ^ 1);
    }
    cv_mbar_wait(&s_bar[st], DB ? ((it >> 1) & 1) : (it & 1));
    if (CONVT) {
      // ---- G = x: BatchNorm in place (no halo, always in range)
#pragma unroll
      for (int j = 0; j < GITERS; ++j) {
        const int c = g_ch[j];
        if (c < 0) continue;
        float4* p = reinterpret_cast<float4*>(s_g + g_off[j]);
        const float4 a = *p;
        const float sc = s_aff[c], sh = s_aff[32 + c];
        *p = make_float4(fmaf(a.x, sc, sh), fmaf(a.y, sc, sh), fmaf(a.z, sc, sh), fmaf(a.w, sc, sh));
      }
    } else {
      // ---- I = x: BatchNorm in place; rows/cols outside the image are zero AFTER the transform
#pragma unroll
      for (int j = 0; j < IITERS; ++j) {
        const int m = i_meta[j];
        if (m < 0) continue;
        const int c = m & 0xff;
        const int gy = iy0 + ((m >> 8) & 0xff);
        const int gx = X0 - 4 + 4 * (m >> 16);   // quads are entirely inside or outside the image
        float4* p = reinterpret_cast<float4*>(s_i + i_off[j]);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gy >= 0 && gy < Hi && gx >= 0 && gx < Wi) {
          const float4 a = *p;
          const float sc = s_aff[c], sh = s_aff[32 + c];
          v = make_float4(fmaf(a.x, sc, sh), fmaf(a.y, sc, sh), fmaf(a.z, sc, sh), fmaf(a.w, sc, sh));
        }
        *p = v;
      }
    }
    __syncthreads();
    if (!active) continue;

    for (int s = pg; s < T::NSTRIPS; s += NPG) {
      const int sy = s / (TWG / 4);
      const int sx = (s % (TWG / 4)) * 4;
      // I window
      constexpr int WR = 3;
      constexpr int WC = (S == 1) ? 6 : 9;
      float iv[WR][WC];
      // window of the strip: tile columns 3 + S*sx .. (left halo sits in column 3)
      const float* ip = s_i + ti * T::I_PLANE + (S * sy) * T::I_PITCH + S * sx;
#pragma unroll
      for (int r = 0; r < WR; ++r) {
        const float* rp = ip + r * T::I_PITCH;
        if (S == 1) {
          float4 a = *reinterpret_cast<const float4*>(rp + 4);
          iv[r][0] = rp[3];
          iv[r][1] = a.x; iv[r][2] = a.y; iv[r][3] = a.z; iv[r][4] = a.w;
          iv[r][5] = rp[8];
        } else {
          float4 a = *reinterpret_cast<const float4*>(rp + 4);
          float4 b = *reinterpret_cast<const float4*>(rp + 8);
          iv[r][0] = rp[3];
          iv[r][1] = a.x; iv[r][2] = a.y; iv[r][3] = a.z; iv[r][4] = a.w;
          iv[r][5] = b.x; iv[r][6] = b.y; iv[r][7] = b.z; iv[r][8] = b.w;
        }
      }
      if (CONVT && gq == 0) {
        // bias gradient of a convT layer = sum of dz over the pixels this strip covers
        if (S == 1) {
          bs[0] += iv[1][1] + iv[1][2] + iv[1][3] + iv[1][4];
        } else {
#pragma unroll
          for (int j = 1; j < 9; ++j) bs[0] += iv[1][j] + iv[2][j];
        }
      }
#pragma unroll
      for (int g = 0; g < GT; ++g) {
        float4 gv = *reinterpret_cast<const float4*>(s_g + (gq * GT + g) * GPL + sy * GW + sx);
        const float gg[4] = {gv.x, gv.y, gv.z, gv.w};
        if (!CONVT && ti == 0) bs[g] += (gg[0] + gg[1]) + (gg[2] + gg[3]);
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int k = 0; k < 9; ++k) acc[g][k] = fmaf(gg[j], iv[k / 3][S * j + k % 3], acc[g][k]);
      }
    }
  }

  // ---- cross-group reduction in shared memory (pixel groups add in a fixed order, so the
  // result is deterministic), then one partial per CTA
  __syncthreads();
  float* s_red = smem;  // reuse: [CG*CI*9 + 32]
  for (int idx = tid; idx < CG * CI * 9 + 32; idx += 256) s_red[idx] = 0.f;
  __syncthreads();
  for (int turn = 0; turn < NPG; ++turn) {
    if (active && pg == turn) {
#pragma unroll
      for (int g = 0; g < GT; ++g)
#pragma unroll
        for (int k = 0; k < 9; ++k) s_red[((gq * GT + g) * CI + ti) * 9 + k] += acc[g][k];
      if (CONVT && gq == 0) s_red[CG * CI * 9 + ti] += bs[0];
      if (!CONVT && ti == 0) {
#pragma unroll
        for (int g = 0; g < GT; ++g) s_red[CG * CI * 9 + gq * GT + g] += bs[g];
      }
    }
    __syncthreads();
  }
  float* dst = P.partial + (size_t)blockIdx.x * (CG * CI * 9 + 32);
  for (int idx = tid; idx < CG * CI * 9 + 32; idx += 256) dst[idx] = s_red[idx];

}

// ------------------------------------------------------------------------------------
// Weight gradient on the tensor cores (mma.sync m16n8k8 TF32, 1 or 3 terms as in gconv_kernel).
// Per tap (ky,kx):  D_tap[g][i] += sum_p G[g][p] * I[i][p + tap]   ->  M = 16 g-channels,
// N = 8 i-channels, K = 8 consecutive pixels of one tile row.  A warp owns one (M-tile, N-tile)
// pair and all 9 taps (36 accumulator registers) for its share of a tile's 32 k-steps;
// accumulators persist over the CTA's whole persistent loop.  Fragments are read straight from
// the channel-planar TMA tiles; the planes are 4 (mod 8) floats apart (spare box rows / columns)
// so that the fragment loads (8 channels x 4 pixels per warp) are bank-conflict free.
constexpr int kWgradMmaDbBytes = 47 * 1024;   // stage size up to which the tensor-core kernel double-buffers
template <int S, int TWG>
struct WTileM : WTile<S, TWG> {
  using B = WTile<S, TWG>;
  static constexpr int I_ROWS_BOX = B::I_ROWS + (S == 1 ? 1 : 0);
  static constexpr int I_PLANE = I_ROWS_BOX * B::I_PITCH;
  // G box: 4 spare columns and one spare row, for the same reason (A-fragment loads)
  static constexpr int G_W = TWG + 4, G_ROWS_BOX = B::THG + 1;
  static constexpr int G_PLANE = G_ROWS_BOX * G_W;
  static_assert(I_PLANE % 8 == 4 && G_PLANE % 8 == 4, "plane strides must be 4 (mod 8) floats");
};

template <int S, int CG, int CI, int TWG, int CONVT, int TERMS>
__global__ void __launch_bounds__((((CG + 15) / 16) * (CI / 8) == 6) ? 192 : 256, 2)
    wgrad_mma_kernel(const __grid_constant__ CUtensorMap map_g, const __grid_constant__ CUtensorMap map_i,
                     const WgradParams P) {
  using T = WTileM<S, TWG>;
  constexpr int MT = (CG + 15) / 16, NTI = CI / 8, NPAIR = MT * NTI;
  constexpr int KS = (NPAIR == 6) ? 1 : 8 / NPAIR;     // k-splits (warps per pair)
  constexpr int NTHR = NPAIR * KS * 32;
  constexpr int G_FLOATS = CG * T::G_PLANE;
  constexpr int I_FLOATS = CI * T::I_PLANE;
  constexpr int G_PAD = (G_FLOATS + 31) / 32 * 32;
  constexpr int I_PAD = (I_FLOATS + 31) / 32 * 32;
  constexpr int NQG = CG * T::THG * (T::G_W / 4);
  constexpr int NQI = CI * T::I_ROWS * (T::I_PITCH / 4);
  constexpr int GITERS = (NQG + NTHR - 1) / NTHR;
  constexpr int IITERS = (NQI + NTHR - 1) / NTHR;
  constexpr int KSTEPS = T::THG * TWG / 8;

  // (two stages while two CTAs still fit an SM: 2 x 2 x 47 KB + reductions < 228 KB)
  constexpr bool DB = (G_PAD + I_PAD) * 4 <= kWgradMmaDbBytes;
  constexpr int NSTG = DB ? 2 : 1;
  extern __shared__ __align__(128) float smem[];
  float* s_aff = smem + NSTG * (G_PAD + I_PAD);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_aff + 64);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int pair = warp % NPAIR, ks = warp / NPAIR;
  const int mt = pair / NTI, nt = pair % NTI;

  const int Hg = P.Hg, Wg = P.Wg, Hi = S * Hg, Wi = S * Wg;
  const int tiles_x = Wg / TWG, tiles_y = Hg / T::THG;
  const int tiles_per_img = tiles_x * tiles_y;
  const int ntiles = P.B * tiles_per_img;

  if (tid == 0) {
    cv_mbar_init(&s_bar[0], 1);
    if (DB) cv_mbar_init(&s_bar[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  auto issue = [&](int tile, int st) {
    const int n = tile / tiles_per_img;
    const int trem = tile - n * tiles_per_img;
    const int ty = trem / tiles_x, tx = trem - ty * tiles_x;
    constexpr uint32_t BYTES = (uint32_t)(G_FLOATS * 4 + I_FLOATS * 4);
    float* sg = smem + st * (G_PAD + I_PAD);
    cv_mbar_expect_tx(&s_bar[st], BYTES);
    cv_tma_load_3d(sg, &map_g, tx * TWG, ty * T::THG, n * CG, &s_bar[st]);
    cv_tma_load_3d(sg + G_PAD, &map_i, S * tx * TWG - 4, S * ty * T::THG - 1, n * CI, &s_bar[st]);
  };
  auto prefetch = [&](int tile) {
    const int n = tile / tiles_per_img;
    const int trem = tile - n * tiles_per_img;
    const int ty = trem / tiles_x, tx = trem - ty * tiles_x;
    cv_tma_prefetch_3d(&map_g, tx * TWG, ty * T::THG, n * CG);
    cv_tma_prefetch_3d(&map_i, S * tx * TWG - 4, S * ty * T::THG - 1, n * CI);
  };
  if (tid < 32) {
    constexpr int CA = CONVT ? CG : CI;
    if (tid < CA) {
      const float mean =
          P.train ? bn_coef(P.stats, tid, P.bn_count, nullptr, nullptr, nullptr, nullptr, true).mean : P.rmean[tid];
      s_aff[tid] = 1.f;        // centred raw input, see wgrad_kernel
      s_aff[32 + tid] = -mean;
    }
  }

  float acc[9][4];
#pragma unroll
  for (int k = 0; k < 9; ++k)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[k][j] = 0.f;
  float bs0 = 0.f, bs1 = 0.f;   // bias-gradient partial sums (see below)
  // rows g+8 of the last M-tile do not exist when CG is not a multiple of 16
  const bool hi_rows = (CG % 16 == 0) || (mt + 1 < MT);

  __syncthreads();   // barriers initialised
  if (DB && tid == 0 && (int)blockIdx.x < ntiles) issue(blockIdx.x, 0);
  int it = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
    const int st = DB ? (it & 1) : 0;
    const int n = tile / tiles_per_img;
    const int trem = tile - n * tiles_per_img;
    const int ty = trem / tiles_x, tx = trem - ty * tiles_x;
    const int gy0 = ty * T::THG, gx0 = tx * TWG;
    const int iy0 = S * gy0 - 1;
    const int X0 = S * gx0;
    (void)n;
    float* s_g = smem + st * (G_PAD + I_PAD);
    float* s_i = s_g + G_PAD;
    __syncthreads();   // previous tile's MMA loop is done with the buffers
    if (tid == 0) {
      if (!DB) {
        issue(tile, 0);
        // single stage (two would cost the second CTA of the SM): at least bring the NEXT tile's
        // boxes into L2 while this one is consumed (ncu: 12% of the samples sat on the barrier)
        if (tile + (int)gridDim.x < ntiles) prefetch(tile + gridDim.x);
      } else if (tile + (int)gridDim.x < ntiles) issue(tile + gridDim.x, st ^ 1);
    }
    cv_mbar_wait(&s_bar[st], DB ? ((it >> 1) & 1) : (it & 1));
    if (CONVT) {
      // G = x: BatchNorm in place
#pragma unroll
      for (int j = 0; j < GITERS; ++j) {
        const int q = tid + j * NTHR;
        if (q < NQG) {
          const int c = q / ((T::G_W / 4) * T::THG);
          const int rq = q - c * ((T::G_W / 4) * T::THG);
          float4* p = reinterpret_cast<float4*>(s_g + c * T::G_PLANE + 4 * rq);
          const float4 a = *p;
          const float sc = s_aff[c], sh = s_aff[32 + c];
          *p = make_float4(fmaf(a.x, sc, sh), fmaf(a.y, sc, sh), fmaf(a.z, sc, sh), fmaf(a.w, sc, sh));
        }
      }
    } else {
      // I = x: BatchNorm in place; rows / columns outside the image are zero AFTER the transform
#pragma unroll
      for (int j = 0; j < IITERS; ++j) {
        const int q = tid + j * NTHR;
        if (q < NQI) {
          const int qx = q % (T::I_PITCH / 4);
          const int y = (q / (T::I_PITCH / 4)) % T::I_ROWS;
          const int c = q / ((T::I_PITCH / 4) * T::I_ROWS);
          const int gy = iy0 + y, gx = X0 - 4 + 4 * qx;
          float4* p = reinterpret_cast<float4*>(s_i + c * T::I_PLANE + y * T::I_PITCH + 4 * qx);
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (gy >= 0 && gy < Hi && gx >= 0 && gx < Wi) {
            const float4 a = *p;
            const float sc = s_aff[c], sh = s_aff[32 + c];
            v = make_float4(fmaf(a.x, sc, sh), fmaf(a.y, sc, sh), fmaf(a.z, sc, sh), fmaf(a.w, sc, sh));
          }
          *p = v;
        }
      }
    }
    __syncthreads();

    const float* gbase = s_g + (mt * 16 + g) * T::G_PLANE + t;
    const float* ibase = s_i + (nt * 8 + g) * T::I_PLANE + 3 + S * t;
    float tq[9][4];
    if (TERMS >= 2) {
#pragma unroll
      for (int k = 0; k < 9; ++k)
#pragma unroll
        for (int q = 0; q < 4; ++q) tq[k][q] = 0.f;
    }
    if constexpr (TERMS == 2) {
      // two k-steps (8 pixels each) per iteration: TF32 main terms separately, the two correction
      // terms of both steps as one BF16 k16 instruction each (see cv_pack_bf16)
      static_assert((KSTEPS / KS) % 2 == 0, "k-steps per warp must pair up");
#pragma unroll 1
      for (int j = ks; j < KSTEPS; j += 2 * KS) {
        const int j1 = j + KS;
        const int y0 = j / (TWG / 8), x00 = (j % (TWG / 8)) * 8;
        const int y1 = j1 / (TWG / 8), x01 = (j1 % (TWG / 8)) * 8;
        const float* gp0 = gbase + y0 * T::G_W + x00;
        const float* gp1 = gbase + y1 * T::G_W + x01;
        float av0[4], av1[4];
        av0[0] = gp0[0];
        av0[2] = gp0[4];
        av0[1] = hi_rows ? gp0[8 * T::G_PLANE] : 0.f;
        av0[3] = hi_rows ? gp0[8 * T::G_PLANE + 4] : 0.f;
        av1[0] = gp1[0];
        av1[2] = gp1[4];
        av1[1] = hi_rows ? gp1[8 * T::G_PLANE] : 0.f;
        av1[3] = hi_rows ? gp1[8 * T::G_PLANE + 4] : 0.f;
        if (!CONVT && nt == 0) {
          bs0 += (av0[0] + av0[2]) + (av1[0] + av1[2]);
          bs1 += (av0[1] + av0[3]) + (av1[1] + av1[3]);
        }
        uint32_t ah0[4], ah1[4], alp[4], ap[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          ah0[q] = cv_tf32_hi(av0[q]);
          ah1[q] = cv_tf32_hi(av1[q]);
          alp[q] = cv_pack_bf16(av0[q] - __uint_as_float(ah0[q]), av1[q] - __uint_as_float(ah1[q]));
          ap[q] = cv_pack_bf16(av0[q], av1[q]);
        }
        const float* ip0 = ibase + (S * y0) * T::I_PITCH + S * x00;
        const float* ip1 = ibase + (S * y1) * T::I_PITCH + S * x01;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
          uint32_t bh0[3][2], bh1[3][2], bp[3][2], blp[3][2];
#pragma unroll
          for (int kx = 0; kx < 3; ++kx)
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const float b0 = ip0[ky * T::I_PITCH + kx + 4 * S * q];
              const float b1 = ip1[ky * T::I_PITCH + kx + 4 * S * q];
              if (CONVT && mt == 0) {
                if (S == 1 ? (ky == 1 && kx == 1) : (ky >= 1 && kx >= 1)) bs0 += b0 + b1;
              }
              bh0[kx][q] = cv_tf32_hi(b0);
              bh1[kx][q] = cv_tf32_hi(b1);
              blp[kx][q] = cv_pack_bf16(b0 - __uint_as_float(bh0[kx][q]), b1 - __uint_as_float(bh1[kx][q]));
              bp[kx][q] = cv_pack_bf16(b0, b1);
            }
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) cv_mma_bf16(tq[ky * 3 + kx], alp, bp[kx][0], bp[kx][1]);
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) cv_mma_bf16(tq[ky * 3 + kx], ap, blp[kx][0], blp[kx][1]);
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) cv_mma_tf32(tq[ky * 3 + kx], ah0, bh0[kx][0], bh0[kx][1]);
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) cv_mma_tf32(tq[ky * 3 + kx], ah1, bh1[kx][0], bh1[kx][1]);
        }
      }
    } else {
#pragma unroll 2
    for (int j = ks; j < KSTEPS; j += KS) {
      const int y = j / (TWG / 8), x0 = (j % (TWG / 8)) * 8;
      // A fragment: a0 = G[g][p+t], a1 = G[g+8][p+t], a2 = G[g][p+t+4], a3 = G[g+8][p+t+4]
      const float* gp = gbase + y * T::G_W + x0;
      float av[4];
      av[0] = gp[0];
      av[2] = gp[4];
      av[1] = hi_rows ? gp[8 * T::G_PLANE] : 0.f;
      av[3] = hi_rows ? gp[8 * T::G_PLANE + 4] : 0.f;
      if (!CONVT && nt == 0) {   // conv layers: db = sum of dz = G
        bs0 += av[0] + av[2];
        bs1 += av[1] + av[3];
      }
      uint32_t ah[4], al[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        ah[q] = (TERMS == 3) ? cv_tf32_hi(av[q]) : __float_as_uint(av[q]);
        al[q] = (TERMS == 3) ? __float_as_uint(av[q] - __uint_as_float(ah[q])) : 0u;
      }
      const float* ip = ibase + (S * y) * T::I_PITCH + S * x0;
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        // B fragments of the three taps of this kernel row: b0 = I[g][pixel t + tap],
        // b1 = I[g][pixel t+4 + tap]
        float bv[3][2];
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          bv[kx][0] = ip[ky * T::I_PITCH + kx];
          bv[kx][1] = ip[ky * T::I_PITCH + kx + 4 * S];
          if (CONVT && mt == 0) {   // convT layers: db = sum of dz = I over the pixels of this strip
            if (S == 1 ? (ky == 1 && kx == 1) : (ky >= 1 && kx >= 1)) bs0 += bv[kx][0] + bv[kx][1];
          }
        }
        if (TERMS == 3) {
          // the tile's k-steps are chained in the tensor-core accumulators tq (a weight gradient is
          // not amplified downstream, unlike an activation: a few dozen truncating adds per tile
          // are harmless) and flushed into the running sums once per tile
          uint32_t bh[3][2], bl[3][2];
#pragma unroll
          for (int kx = 0; kx < 3; ++kx)
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              bh[kx][q] = cv_tf32_hi(bv[kx][q]);
              bl[kx][q] = __float_as_uint(bv[kx][q] - __uint_as_float(bh[kx][q]));
            }
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) cv_mma_tf32(tq[ky * 3 + kx], al, bh[kx][0], bh[kx][1]);
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) cv_mma_tf32(tq[ky * 3 + kx], ah, bl[kx][0], bl[kx][1]);
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) cv_mma_tf32(tq[ky * 3 + kx], ah, bh[kx][0], bh[kx][1]);
        } else {
#pragma unroll
          for (int kx = 0; kx < 3; ++kx)
            cv_mma_tf32(acc[ky * 3 + kx], ah, __float_as_uint(bv[kx][0]), __float_as_uint(bv[kx][1]));
        }
      }
    }
    }
    if (TERMS >= 2) {
#pragma unroll
      for (int k = 0; k < 9; ++k)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[k][q] += tq[k][q];
    }
  }

  // ---- k-split warps add in a fixed order (deterministic), then one partial per CTA
  // D fragment: c0 = (g, 2t), c1 = (g, 2t+1), c2 = (g+8, 2t), c3 = (g+8, 2t+1)
  bs0 += __shfl_xor_sync(0xffffffffu, bs0, 1);
  bs0 += __shfl_xor_sync(0xffffffffu, bs0, 2);
  bs1 += __shfl_xor_sync(0xffffffffu, bs1, 1);
  bs1 += __shfl_xor_sync(0xffffffffu, bs1, 2);
  __syncthreads();
  float* s_red = smem;  // reuse: [CG*CI*9 + 32]
  for (int idx = tid; idx < CG * CI * 9 + 32; idx += NTHR) s_red[idx] = 0.f;
  __syncthreads();
  for (int turn = 0; turn < KS; ++turn) {
    if (ks == turn) {
#pragma unroll
      for (int k = 0; k < 9; ++k)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int gc = mt * 16 + g + 8 * (q >> 1), ic = nt * 8 + 2 * t + (q & 1);
          if (gc < CG) s_red[(gc * CI + ic) * 9 + k] += acc[k][q];
        }
      if (t == 0) {
        if (!CONVT && nt == 0) {
          s_red[CG * CI * 9 + mt * 16 + g] += bs0;
          if (hi_rows) s_red[CG * CI * 9 + mt * 16 + g + 8] += bs1;
        }
        if (CONVT && mt == 0) s_red[CG * CI * 9 + nt * 8 + g] += bs0;
      }
    }
    __syncthreads();
  }
  float* dst = P.partial + (size_t)blockIdx.x * (CG * CI * 9 + 32);
  for (int idx = tid; idx < CG * CI * 9 + 32; idx += NTHR) dst[idx] = s_red[idx];
}

constexpr int kWgradMaxCtas = 8 * kNumSMs;  // per-CTA partial slots in the workspace

// Border-trimmed sums of dz: T_k[c] = sum of dz[c] over the pixels whose tap-k partner lies inside
// the image, from the 9 per-channel sums `ts` ([slot][32] doubles) that the kernel producing dz
// accumulated in its epilogue (as ava_b200_dz_border_sums defines them):
//   mode 0 (conv layers, stride-1 conv-transpose): 0 total, 1 first row, 2 last row, 3 first column,
//          4 last column, 5..8 corners (first/last row x first/last column)
//   mode 1 (stride-2 conv-transpose; dz at 2x resolution, tap (ky,kx) reads dz[2p+k-1]):
//          0..3 parity classes (row parity*2 + column parity), 4,5 last row by column parity,
//          6,7 last column by row parity, 8 last corner
__device__ __forceinline__ double trimmed_dz_sum(const double* ts, int c, int ky, int kx, int convt, int s2) {
  if (convt && s2) {
    const int ry = (ky != 1), rx = (kx != 1);
    double v = ts[(ry * 2 + rx) * 32 + c];
    if (ky == 0) v -= ts[(4 + rx) * 32 + c];
    if (kx == 0) v -= ts[(6 + ry) * 32 + c];
    if (ky == 0 && kx == 0) v += ts[8 * 32 + c];
    return v;
  }
  int rex = -1, cex = -1;   // excluded row / column: 0 = first, 1 = last
  if (!convt) {             // partner S*p + k - 1: tap 0 misses p = 0; tap 2 misses the last p (stride 1 only)
    if (ky == 0) rex = 0; else if (ky == 2 && !s2) rex = 1;
    if (kx == 0) cex = 0; else if (kx == 2 && !s2) cex = 1;
  } else {                  // dz pixel p + k - 1: tap 0 never reaches the last row, tap 2 never the first
    if (ky == 0) rex = 1; else if (ky == 2) rex = 0;
    if (kx == 0) cex = 1; else if (kx == 2) cex = 0;
  }
  double v = ts[c];
  if (rex >= 0) v -= ts[(1 + rex) * 32 + c];
  if (cex >= 0) v -= ts[(3 + cex) * 32 + c];
  if (rex >= 0 && cex >= 0) v += ts[(5 + rex * 2 + cex) * 32 + c];
  return v;
}

struct FinalizeParams {
  const float* partial;   // [nparts][stride] per-CTA partial sums of Rc (+ 32 unused slots)
  int nparts, stride;
  int Cx, Cz;             // channels of x (this layer's BatchNorm) and of dz
  int convt, s2;
  const float* w;         // same flat layout as dw
  const float* gamma;
  const float* beta;
  const double* stats;    // sum x | sum x^2 of this layer's input
  double count;
  const float* rmean;     // eval mode (train == 0): the running buffers replace the batch statistics
  const float* rvar;
  int train;
  const double* tsums;    // [9][32], see trimmed_dz_sum
  float* dw;
  float* db;
  double* dstats;         // out: sum g | sum g*(x-mean), accumulated (zeroed by the caller)
};

// Second stage of the weight gradient: a CTA finishes 32 consecutive weight elements.  Lane = element
// (every load is one coalesced 128-byte row of a per-CTA partial), the 32 warps split the partials
// (4 loads in flight each: 296 partials are 3 rounds of latency; with 8 warps it was 10 rounds, 11 us
// per layer ON THE CRITICAL PATH between a layer's weight-gradient and backward-data kernels at any
// batch size), fp64 sums combined through shared memory in a fixed order (deterministic); then dW and
// the element's contribution to this layer's BatchNorm-backward reductions.  (A first version had one
// warp per element with the lanes striding over the partials: 32 scattered 4-byte loads per request.)
constexpr int kFinWarps = 32;
__global__ void __launch_bounds__(kFinWarps * 32) bnconv_finalize_kernel(const FinalizeParams P) {
  __shared__ double s_part[kFinWarps][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + lane;
  const int NW = P.Cx * P.Cz * 9;
  double r = 0.0;
  if (j < NW) {
    const float* src = P.partial + j;
    double r0 = 0.0, r1 = 0.0, r2 = 0.0, r3 = 0.0;
    int p = warp;
    for (; p + 3 * kFinWarps < P.nparts; p += 4 * kFinWarps) {
      const float a0 = src[(size_t)p * P.stride], a1 = src[(size_t)(p + kFinWarps) * P.stride];
      const float a2 = src[(size_t)(p + 2 * kFinWarps) * P.stride], a3 = src[(size_t)(p + 3 * kFinWarps) * P.stride];
      r0 += (double)a0;
      r1 += (double)a1;
      r2 += (double)a2;
      r3 += (double)a3;
    }
    for (; p < P.nparts; p += kFinWarps) r0 += (double)src[(size_t)p * P.stride];
    r = (r0 + r1) + (r2 + r3);
  }
  s_part[warp][lane] = r;
  __syncthreads();
  if (warp != 0) return;
  if (j >= NW + P.Cz) return;
  if (j >= NW) {
    // bias gradient = sum of dz over all pixels
    const int cz = j - NW;
    double v;
    if (P.convt && P.s2)
      v = P.tsums[cz] + P.tsums[32 + cz] + P.tsums[64 + cz] + P.tsums[96 + cz];
    else
      v = P.tsums[cz];
    P.db[cz] = (float)v;
    return;
  }
  r = 0.0;
#pragma unroll
  for (int w = 0; w < kFinWarps; ++w) r += s_part[w][lane];
  const int k = j % 9;
  int cx, cz;
  if (!P.convt) {
    cx = (j / 9) % P.Cx;
    cz = j / (9 * P.Cx);
  } else {
    cz = (j / 9) % P.Cz;
    cx = j / (9 * P.Cz);
  }
  const double T = trimmed_dz_sum(P.tsums, cz, k / 3, k % 3, P.convt, P.s2);
  double mean, var;
  if (P.train) {
    mean = P.stats[cx] / P.count;
    var = P.stats[32 + cx] / P.count - mean * mean;
    if (var < 0.0) var = 0.0;
  } else {
    mean = (double)P.rmean[cx];
    var = (double)P.rvar[cx];
  }
  const double invstd = rsqrt(var + (double)kBnEps);
  // the kernels centred with the fp32-rounded mean: sum dz*(x-mean) = sum dz*(x-mean32) + (mean32-mean)*T
  // (zero in eval mode, where the running mean is fp32 already)
  const double rc = r + ((double)(float)mean - mean) * T;
  const double wv = (double)P.w[j];
  P.dw[j] = (float)((double)P.gamma[cx] * invstd * rc + (double)P.beta[cx] * T);
  atomicAdd(&P.dstats[cx], wv * T);
  atomicAdd(&P.dstats[32 + cx], wv * rc);
}

// The nine per-channel sums of a dz tensor [B, C, H, W] that trimmed_dz_sum consumes.
__global__ void __launch_bounds__(256)
dz_border_sums_kernel(const float* __restrict__ dz, int B, int C, int H, int W, int mode, double* tsums) {
  __shared__ double s_red[8][9];
  const int c = blockIdx.y;
  const int w4 = W >> 2, hw4 = (H * W) >> 2;
  const long long total4 = (long long)B * hw4;
  double a[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) a[i] = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total4;
       i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / hw4;
    const int q = (int)(i - n * hw4);
    const int y = q / w4, x0 = (q - y * w4) * 4;
    const float4 v = __ldg(reinterpret_cast<const float4*>(dz + ((size_t)n * C + c) * H * W) + q);
    const bool first_row = (y == 0), last_row = (y == H - 1), first_col = (x0 == 0), last_col = (x0 + 4 == W);
    if (mode == 0) {
      const float s = (v.x + v.y) + (v.z + v.w);
      a[0] += (double)s;
      if (first_row) a[1] += (double)s;
      if (last_row) a[2] += (double)s;
      if (first_col) {
        a[3] += (double)v.x;
        if (first_row) a[5] += (double)v.x;
        if (last_row) a[7] += (double)v.x;
      }
      if (last_col) {
        a[4] += (double)v.w;
        if (first_row) a[6] += (double)v.w;
        if (last_row) a[8] += (double)v.w;
      }
    } else {
      const int ry = y & 1;
      const float e = v.x + v.z, o = v.y + v.w;
      a[ry * 2] += (double)e;
      a[ry * 2 + 1] += (double)o;
      if (last_row) {
        a[4] += (double)e;
        a[5] += (double)o;
      }
      if (last_col) {
        a[6 + ry] += (double)v.w;
        if (last_row) a[8] += (double)v.w;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    const double s = warp_sum(a[i]);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5][i] = s;
  }
  __syncthreads();
  if (threadIdx.x < 9) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += s_red[w][threadIdx.x];
    atomicAdd(&tsums[threadIdx.x * 32 + c], s);
  }
}

// second stage, shared by both weight-gradient kernels
template <int S, int CG, int CI, int CONVT>
static int launch_finalize(const WgradParams& P, FinalizeParams F, int nparts, cudaStream_t stream) {
  F.partial = P.partial;
  F.nparts = nparts;
  F.stride = CG * CI * 9 + 32;
  F.Cx = CONVT ? CG : CI;
  F.Cz = CONVT ? CI : CG;
  F.convt = CONVT;
  F.s2 = (S == 2);
  F.stats = P.stats;
  F.count = P.bn_count;
  F.rmean = P.rmean;
  F.train = P.train;
  const int n = CG * CI * 9 + F.Cz;
  bnconv_finalize_kernel<<<(n + 31) / 32, kFinWarps * 32, 0, stream>>>(F);
  return check_launch("bnconv_finalize");
}

template <int S, int CG, int CI, int TWG, int CONVT>
static int launch_wgrad(WgradParams P, const FinalizeParams& F, void* ws, cudaStream_t stream) {
  using T = WTile<S, TWG>;
  constexpr int GW = (CI == 1) ? TWG + 4 : TWG, GROWS = (CI == 1) ? T::THG + 1 : T::THG;   // as in the kernel
  constexpr int G_PAD = (CG * GW * GROWS + 31) / 32 * 32;
  constexpr int I_PAD = (CI * T::I_PLANE + 31) / 32 * 32;
  constexpr int NSTG = ((G_PAD + I_PAD) * 4 <= (CONVT ? 48 : 40) * 1024) ? 2 : 1;   // as in the kernel
  size_t smem_f = (size_t)NSTG * (G_PAD + I_PAD) + 64 + 8;
  if (smem_f < (size_t)CG * CI * 9 + 32) smem_f = (size_t)CG * CI * 9 + 32;
  const size_t smem = smem_f * sizeof(float) + 128;
  auto kern = wgrad_kernel<S, CG, CI, TWG, CONVT>;
  static int max_ctas = 0;
  if (max_ctas == 0) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
      cudaGetLastError();
      set_error("wgrad: cannot reserve %zu bytes of shared memory", smem);
      return 1;
    }
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, smem);
    if (per_sm < 1) per_sm = 1;
    max_ctas = per_sm * kNumSMs;
  }
  const long long ntiles = (long long)P.B * (P.Wg / TWG) * (P.Hg / T::THG);
  int grid = (int)(ntiles < max_ctas ? ntiles : max_ctas);
  if (grid > kWgradMaxCtas) grid = kWgradMaxCtas;  // workspace bound, see ava_b200_bnconv_bwd_weight_ws
  CUtensorMap map_g, map_i;
  if (make_act_map(&map_g, P.g_a, (long long)P.B * CG, P.Hg, P.Wg, GW, GROWS, CG)) return 1;
  if (make_act_map(&map_i, P.i_a, (long long)P.B * CI, S * P.Hg, S * P.Wg, T::I_PITCH, T::I_ROWS, CI)) return 1;
  P.partial = reinterpret_cast<float*>(ws);
  kern<<<grid, 256, smem, stream>>>(map_g, map_i, P);
  if (check_launch("wgrad")) return 1;
  return launch_finalize<S, CG, CI, CONVT>(P, F, grid, stream);
}

template <int S, int CG, int CI, int TWG, int CONVT, int TERMS>
static int launch_wgrad_mma(WgradParams P, const FinalizeParams& F, void* ws, cudaStream_t stream) {
  using T = WTileM<S, TWG>;
  constexpr int NPAIR = ((CG + 15) / 16) * (CI / 8);
  constexpr int NTHR = (NPAIR == 6) ? 192 : 256;
  constexpr int G_PAD = (CG * T::G_PLANE + 31) / 32 * 32;
  constexpr int I_PAD = (CI * T::I_PLANE + 31) / 32 * 32;
  constexpr int NSTG = ((G_PAD + I_PAD) * 4 <= kWgradMmaDbBytes) ? 2 : 1;   // as in the kernel
  size_t smem_f = (size_t)NSTG * (G_PAD + I_PAD) + 64 + 8;
  if (smem_f < (size_t)CG * CI * 9 + 32) smem_f = (size_t)CG * CI * 9 + 32;
  const size_t smem = smem_f * sizeof(float) + 128;
  auto kern = wgrad_mma_kernel<S, CG, CI, TWG, CONVT, TERMS>;
  static int max_ctas = 0;
  if (max_ctas == 0) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
      cudaGetLastError();
      set_error("wgrad_mma: cannot reserve %zu bytes of shared memory", smem);
      return 1;
    }
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, NTHR, smem);
    if (per_sm < 1) per_sm = 1;
    max_ctas = per_sm * kNumSMs;
  }
  const long long ntiles = (long long)P.B * (P.Wg / TWG) * (P.Hg / T::THG);
  int grid = (int)(ntiles < max_ctas ? ntiles : max_ctas);
  if (grid > kWgradMaxCtas) grid = kWgradMaxCtas;
  CUtensorMap map_g, map_i;
  if (make_act_map(&map_g, P.g_a, (long long)P.B * CG, P.Hg, P.Wg, T::G_W, T::G_ROWS_BOX, CG)) return 1;
  if (make_act_map(&map_i, P.i_a, (long long)P.B * CI, S * P.Hg, S * P.Wg, T::I_PITCH, T::I_ROWS_BOX, CI)) return 1;
  P.partial = reinterpret_cast<float*>(ws);
  kern<<<grid, NTHR, smem, stream>>>(map_g, map_i, P);
  if (check_launch("wgrad_mma")) return 1;
  return launch_finalize<S, CG, CI, CONVT>(P, F, grid, stream);
}

// tensor-core weight gradient (all layers with >= 8 channels on both sides), else the fp32 FMA kernel
#define WGRAD_TC(S, CG, CI, TWG, CONVT)                                                              \
  (g_conv_terms == 3   ? (g_conv_bf16corr ? launch_wgrad_mma<S, CG, CI, TWG, CONVT, 2>(P, F, ws, stream)  \
                                          : launch_wgrad_mma<S, CG, CI, TWG, CONVT, 3>(P, F, ws, stream)) \
   : g_conv_terms == 1 ? launch_wgrad_mma<S, CG, CI, TWG, CONVT, 1>(P, F, ws, stream)               \
                       : launch_wgrad<S, CG, CI, TWG, CONVT>(P, F, ws, stream))

// ------------------------------------------------------------------------------------
struct LayerGeom {
  int transposed;  // 0: Conv2d, 1: ConvTranspose2d
  int stride;
  int cin, cout;
  int h_in;        // input height == width
  int relu;
};
static const LayerGeom kLayers[14] = {
    {0, 1, 1, 8, 128, 1},  {0, 2, 8, 8, 128, 1},  {0, 1, 8, 16, 64, 1},  {0, 2, 16, 16, 64, 1},
    {0, 1, 16, 24, 32, 1}, {0, 2, 24, 24, 32, 1}, {0, 1, 24, 32, 16, 1}, {1, 1, 32, 24, 16, 1},
    {1, 2, 24, 24, 16, 1}, {1, 1, 24, 16, 32, 1}, {1, 2, 16, 16, 32, 1}, {1, 1, 16, 8, 64, 1},
    {1, 2, 8, 8, 64, 1},   {1, 1, 8, 1, 128, 0}};

static inline int h_out_of(const LayerGeom& L) {
  if (L.stride == 1) return L.h_in;
  return L.transposed ? L.h_in * 2 : L.h_in / 2;
}

}  // namespace ava

using namespace ava;

// layers with channel counts that are multiples of 8 on both sides can run on the tensor cores
#define GCONV_TC(KIND, CI, CO, TW, INMODE, EPI, HIN)                                               \
  (g_conv_terms == 3   ? ((EPI == EPI_FWD ? (g_conv_bf16corr & (layer >= 7 ? 12 : 4))                  \
                                              : (g_conv_bf16corr & 2))                                  \
                              ? launch_gconv<KIND, CI, CO, TW, INMODE, EPI, HIN, 2>(P, stream)         \
                              : launch_gconv<KIND, CI, CO, TW, INMODE, EPI, HIN, 3>(P, stream))        \
   : g_conv_terms == 1 ? launch_gconv<KIND, CI, CO, TW, INMODE, EPI, HIN, 1>(P, stream)            \
                       : launch_gconv<KIND, CI, CO, TW, INMODE, EPI, HIN, 0>(P, stream))

// (HBM-bound layer where the 3-term tensor-core kernel loses to the FMA kernel: tensor cores only
// in plain TF32 mode)
#define GCONV_TC1(KIND, CI, CO, TW, INMODE, EPI, HIN)                                              \
  (g_conv_terms == 1 ? launch_gconv<KIND, CI, CO, TW, INMODE, EPI, HIN, 1>(P, stream)              \
                     : launch_gconv<KIND, CI, CO, TW, INMODE, EPI, HIN, 0>(P, stream))
// (measured again with the 2-instruction-per-tap variant, TERMS == 2: 304.8 vs 307.7 us -- that
// layer is bound by its epilogue's reads of x, not by the inner product)

extern "C" int ava_b200_set_conv_precision(int mode) {
  AVA_REQUIRE(mode >= 0 && mode <= 6,
              "set_conv_precision: mode %d (0 fp32, 1 tf32, 2 tf32x3, 3 .. 6 tf32 + bf16 corrections)", mode);
  g_conv_terms = (mode >= 2) ? 3 : mode;
  g_conv_bf16corr = (mode == 3) ? 1 : (mode == 4) ? 7 : (mode == 5) ? 3 : (mode == 6) ? 11 : 0;
  return 0;
}
extern "C" int ava_b200_get_conv_precision(void) {
  if (g_conv_terms != 3) return g_conv_terms;
  return g_conv_bf16corr == 1 ? 3 : g_conv_bf16corr == 7 ? 4 : g_conv_bf16corr == 3 ? 5 : g_conv_bf16corr == 11 ? 6 : 2;
}

extern "C" int ava_b200_bnconv_fwd(int layer, int B, const float* x, float* y, const float* w, const float* b,
                                   const float* gamma, const float* beta, const double* stats_in,
                                   const float* running_mean, const float* running_var, int train,
                                   double* stats_out, void* stream_) {
  AVA_REQUIRE(layer >= 0 && layer < 14, "bnconv_fwd: bad layer %d", layer);
  AVA_REQUIRE(B >= 0, "bnconv_fwd: bad batch %d", B);
  if (B == 0) return 0;
  cudaStream_t stream = (cudaStream_t)stream_;
  const LayerGeom& L = kLayers[layer];
  GconvParams P = {};
  P.in = x;
  P.gamma = gamma;
  P.beta = beta;
  P.stats = stats_in;
  P.rmean = running_mean;
  P.rvar = running_var;
  P.train = train;
  P.in_count = (double)B * L.h_in * L.h_in;
  P.w = w;
  P.bias = b;
  P.out = y;
  P.relu_out = L.relu;
  P.stats_out = stats_out;
  P.B = B;
  P.H_in = P.W_in = L.h_in;
  if (!L.transposed) {
    P.w_so = L.cin * 9;
    P.w_si = 9;
    P.w_flip = 0;
  } else {
    P.w_so = 9;
    P.w_si = L.cout * 9;
    P.w_flip = (L.stride == 1) ? 1 : 0;
  }
  switch (layer) {
    case 0: return launch_gconv<K_S1, 1, 8, 32, IN_AFFINE, EPI_FWD, 128>(P, stream);
    case 1: return GCONV_TC(K_S2, 8, 8, 32, IN_AFFINE, EPI_FWD, 128);
    case 2: return GCONV_TC(K_S1, 8, 16, 32, IN_AFFINE, EPI_FWD, 64);
    case 3: return GCONV_TC(K_S2, 16, 16, 32, IN_AFFINE, EPI_FWD, 64);
    case 4: return GCONV_TC(K_S1, 16, 24, 32, IN_AFFINE, EPI_FWD, 32);
    case 5: return GCONV_TC(K_S2, 24, 24, 16, IN_AFFINE, EPI_FWD, 32);
    case 6: return GCONV_TC(K_S1, 24, 32, 16, IN_AFFINE, EPI_FWD, 16);
    case 7: return GCONV_TC(K_S1, 32, 24, 16, IN_AFFINE, EPI_FWD, 16);
    case 8: return GCONV_TC(K_UP, 24, 24, 16, IN_AFFINE, EPI_FWD, 16);
    case 9: return GCONV_TC(K_S1, 24, 16, 32, IN_AFFINE, EPI_FWD, 32);
    case 10: return GCONV_TC(K_UP, 16, 16, 32, IN_AFFINE, EPI_FWD, 32);
    case 11: return GCONV_TC(K_S1, 16, 8, 32, IN_AFFINE, EPI_FWD, 64);
    case 12: return GCONV_TC(K_UP, 8, 8, 32, IN_AFFINE, EPI_FWD, 64);
    case 13: return launch_gconv<K_S1, 8, 1, 32, IN_AFFINE, EPI_FWD, 128>(P, stream);
  }
  return 1;
}

extern "C" int ava_b200_bnconv_bwd_data_ex(int layer, int B, const float* dz, const float* w, const float* x,
                                           const float* gamma, const double* stats_in, const float* running_var,
                                           int train, const double* dstats, int relu_mask, float* dz_prev,
                                           double* tsums_prev, void* stream_) {
  AVA_REQUIRE(layer >= 0 && layer < 14, "bnconv_bwd_data: bad layer %d", layer);
  AVA_REQUIRE(dz_prev != nullptr && x != nullptr, "bnconv_bwd_data: output and layer input required");
  AVA_REQUIRE(train || gamma == nullptr || running_var != nullptr,
              "bnconv_bwd_data: eval mode needs the running variance");
  if (B <= 0) return 0;
  cudaStream_t stream = (cudaStream_t)stream_;
  const LayerGeom& L = kLayers[layer];
  const int ho = h_out_of(L);
  GconvParams P = {};
  P.in = dz;
  P.w = w;
  P.out = dz_prev;
  P.x_self = x;
  P.stats_self = stats_in;
  P.gamma_self = gamma;
  P.dstats_in = dstats;
  P.rvar_self = train ? nullptr : running_var;
  P.mask_in = relu_mask;
  P.tsums_out = tsums_prev;
  // the dz written here belongs to layer-1: parity classes if that is a stride-2 conv-transpose
  P.tsum_mode = (layer >= 1 && kLayers[layer - 1].transposed && kLayers[layer - 1].stride == 2) ? 1 : 0;
  P.out_count = (double)B * L.h_in * L.h_in;
  P.B = B;
  P.H_in = P.W_in = ho;  // the gather reads the layer's OUTPUT-shaped gradient
  if (!L.transposed) {
    P.w_so = 9;
    P.w_si = L.cin * 9;
    P.w_flip = (L.stride == 1) ? 1 : 0;
  } else {
    P.w_so = L.cout * 9;
    P.w_si = 9;
    P.w_flip = 0;
  }
  switch (layer) {
    case 0: return launch_gconv<K_S1, 8, 1, 32, IN_PLAIN, EPI_BWD, 128>(P, stream);
    case 1: return GCONV_TC1(K_UP, 8, 8, 32, IN_PLAIN, EPI_BWD, 64);
    case 2: return GCONV_TC(K_S1, 16, 8, 32, IN_PLAIN, EPI_BWD, 64);
    case 3: return GCONV_TC(K_UP, 16, 16, 32, IN_PLAIN, EPI_BWD, 32);
    case 4: return GCONV_TC(K_S1, 24, 16, 32, IN_PLAIN, EPI_BWD, 32);
    case 5: return GCONV_TC(K_UP, 24, 24, 16, IN_PLAIN, EPI_BWD, 16);
    case 6: return GCONV_TC(K_S1, 32, 24, 16, IN_PLAIN, EPI_BWD, 16);
    case 7: return GCONV_TC(K_S1, 24, 32, 16, IN_PLAIN, EPI_BWD, 16);
    case 8: return GCONV_TC(K_S2, 24, 24, 16, IN_PLAIN, EPI_BWD, 32);
    case 9: return GCONV_TC(K_S1, 16, 24, 32, IN_PLAIN, EPI_BWD, 32);
    case 10: return GCONV_TC(K_S2, 16, 16, 32, IN_PLAIN, EPI_BWD, 64);
    case 11: return GCONV_TC(K_S1, 8, 16, 32, IN_PLAIN, EPI_BWD, 64);
    case 12: return GCONV_TC(K_S2, 8, 8, 32, IN_PLAIN, EPI_BWD, 128);
    case 13: return launch_gconv<K_S1, 1, 8, 32, IN_PLAIN, EPI_BWD, 128>(P, stream);
  }
  return 1;
}

extern "C" int ava_b200_bnconv_bwd_data(int layer, int B, const float* dz, const float* w, const float* x,
                                        const float* gamma, const double* stats_in, const double* dstats,
                                        int relu_mask, float* dz_prev, double* tsums_prev, void* stream) {
  return ava_b200_bnconv_bwd_data_ex(layer, B, dz, w, x, gamma, stats_in, nullptr, 1, dstats, relu_mask, dz_prev,
                                     tsums_prev, stream);
}

extern "C" long long ava_b200_bnconv_bwd_weight_ws(int layer, int B) {
  (void)B;
  if (layer < 0 || layer >= 14) return 0;
  const LayerGeom& L = kLayers[layer];
  // one partial of (weights + 32 bias slots) floats per resident CTA (up to 8 per SM)
  return (long long)kWgradMaxCtas * (L.cin * L.cout * 9 + 32) * (long long)sizeof(float);
}

extern "C" int ava_b200_bnconv_bwd_weight_ex(int layer, int B, const float* dz, const float* x, const float* w,
                                             const float* gamma, const float* beta, const double* stats_in,
                                             const float* running_mean, const float* running_var, int train,
                                             const double* tsums, float* dw, float* db, double* dstats, void* ws,
                                             void* stream_) {
  AVA_REQUIRE(layer >= 0 && layer < 14, "bnconv_bwd_weight: bad layer %d", layer);
  AVA_REQUIRE(ws != nullptr, "bnconv_bwd_weight: workspace required");
  AVA_REQUIRE(w != nullptr && tsums != nullptr && dstats != nullptr, "bnconv_bwd_weight: w, tsums, dstats required");
  AVA_REQUIRE(train ? stats_in != nullptr : (running_mean != nullptr && running_var != nullptr),
              "bnconv_bwd_weight: %s required", train ? "stats_in" : "running_mean and running_var");
  if (B <= 0) return 0;
  cudaStream_t stream = (cudaStream_t)stream_;
  const LayerGeom& L = kLayers[layer];
  const int ho = h_out_of(L);
  WgradParams P = {};
  P.stats = stats_in;
  P.bn_count = (double)B * L.h_in * L.h_in;
  P.rmean = running_mean;
  P.train = train ? 1 : 0;
  P.B = B;
  FinalizeParams F = {};
  F.rvar = running_var;
  F.w = w;
  F.gamma = gamma;
  F.beta = beta;
  F.tsums = tsums;
  F.dw = dw;
  F.db = db;
  F.dstats = dstats;
  int rc = 1;
  if (!L.transposed) {
    // G = dz (output resolution), I = x - mean (input resolution)
    P.g_a = dz;
    P.i_a = x;
    P.Hg = P.Wg = ho;
    switch (layer) {
      case 0: rc = launch_wgrad<1, 8, 1, 32, 0>(P, F, ws, stream); break;
      case 1: rc = WGRAD_TC(2, 8, 8, 32, 0); break;
      case 2: rc = WGRAD_TC(1, 16, 8, 32, 0); break;
      case 3: rc = WGRAD_TC(2, 16, 16, 32, 0); break;
      case 4: rc = WGRAD_TC(1, 24, 16, 32, 0); break;
      case 5: rc = WGRAD_TC(2, 24, 24, 16, 0); break;
      case 6: rc = WGRAD_TC(1, 32, 24, 16, 0); break;
    }
    return rc;
  } else {
    // G = x - mean (input resolution), I = dz (output resolution)
    P.g_a = x;
    P.i_a = dz;
    P.Hg = P.Wg = L.h_in;
    switch (layer) {
      case 7: rc = WGRAD_TC(1, 32, 24, 16, 1); break;
      case 8: rc = WGRAD_TC(2, 24, 24, 16, 1); break;
      case 9: rc = WGRAD_TC(1, 24, 16, 32, 1); break;
      case 10: rc = WGRAD_TC(2, 16, 16, 32, 1); break;
      case 11: rc = WGRAD_TC(1, 16, 8, 32, 1); break;
      case 12: rc = launch_wgrad<2, 8, 8, 32, 1>(P, F, ws, stream); break;  // HBM-bound: FMA kernel wins
      case 13: rc = launch_wgrad<1, 8, 1, 32, 1>(P, F, ws, stream); break;
    }
    return rc;
  }
}

extern "C" int ava_b200_bnconv_bwd_weight(int layer, int B, const float* dz, const float* x, const float* w,
                                          const float* gamma, const float* beta, const double* stats_in,
                                          const double* tsums, float* dw, float* db, double* dstats, void* ws,
                                          void* stream) {
  return ava_b200_bnconv_bwd_weight_ex(layer, B, dz, x, w, gamma, beta, stats_in, nullptr, nullptr, 1, tsums, dw, db,
                                       dstats, ws, stream);
}

extern "C" int ava_b200_dz_border_sums(const float* dz, int B, int C, int H, int W, int mode, double* tsums,
                                       void* stream) {
  AVA_REQUIRE(C >= 1 && C <= 32 && W % 4 == 0 && H >= 2 && (mode == 0 || mode == 1),
              "dz_border_sums: C=%d H=%d W=%d mode=%d", C, H, W, mode);
  if (B <= 0) return 0;
  const long long total4 = (long long)B * H * W / 4;
  long long want = (total4 + 255) / 256;
  int gx = (int)(want < 1 ? 1 : want);
  const int cap = (8 * kNumSMs + C - 1) / C;
  if (gx > cap) gx = cap;
  dz_border_sums_kernel<<<dim3(gx, C), 256, 0, (cudaStream_t)stream>>>(dz, B, C, H, W, mode, tsums);
  return check_launch("dz_border_sums");
}
