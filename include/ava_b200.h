/*
 * ava_b200 -- C ABI of the B200-native AVA hot path (VAE train/infer + get_spec).
 *
 * The reference (pearsonlab/autoencoded-vocal-analysis) is pure Python and has no
 * FFI of its own; the drop-in boundary for a maintainer is the Python module
 * surface (ava.models.vae.VAE, ava.models.vae_dataset, ava.models.window_vae_dataset,
 * p['get_spec']).  This header is the native boundary underneath that surface:
 * every entry point replaces one group of library calls the reference makes from
 * Python, cited per function as <reference file>:<lines>.
 *
 * Conventions
 *   - plain C types only; all pointers are DEVICE pointers on the current CUDA
 *     device unless the name starts with h_ (host).  The library never allocates
 *     persistent memory, never frees caller memory and never copies host<->device.
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*) and
 *     is CUDA-graph capturable; no implicit synchronisation.
 *   - every call returns 0 on success, nonzero on error; ava_b200_last_error()
 *     gives the message (thread-local).  No C++ exceptions cross the boundary.
 *   - tensors are contiguous fp32 NCHW / row-major exactly as the reference's
 *     torch tensors are; statistics accumulators are fp64.
 *
 * Layer ids (hard-coded network, ava/models/vae.py:128-168):
 *   0..6   = bn1+conv1 .. bn7+conv7      (encoder, ava/models/vae.py:217-223)
 *   7..13  = bn8+convt1 .. bn14+convt7   (decoder, ava/models/vae.py:263-269)
 */
#ifndef AVA_B200_H
#define AVA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AVA_B200_ABI_VERSION 9
#define AVA_NUM_BN_LAYERS 14
#define AVA_STATS_STRIDE 64 /* doubles per layer in a stats block: [0..31]=sum, [32..63]=sum of squares */

const char* ava_b200_last_error(void);
int ava_b200_abi_version(void);
/* Number of kernels launched by this library since load (bench.py's gpu_launches). */
long long ava_b200_launch_count(void);

/* ------------------------------------------------------------------ BatchNorm
 * Per-channel sums of x[B,C,HW]: stats[c] += sum x, stats[32+c] += sum x^2.
 * Replaces the statistics half of torch.nn.BatchNorm2d for bn1 (input spectrogram)
 * and bn8 (fc8 output viewed as [B,32,16,16]); ava/models/vae.py:217,262-263.
 * All other BN layers get their statistics from the producing layer's epilogue. */
int ava_b200_channel_stats(const float* x, int B, int C, int HW, double* stats, void* stream);

/* Running-buffer update for all 14 BN layers in one launch (momentum 0.1, unbiased
 * variance, num_batches_tracked += 1): torch.nn.BatchNorm2d train-mode side effect,
 * ava/models/vae.py:135-141,162-168.  stats: [14][64] doubles as above; counts[l] =
 * B*H*W of layer l's input; running: flat fp32 buffer, layer l's running_mean at
 * rm_off[l] and running_var at rv_off[l] (element offsets); nbt: int64[14]. */
int ava_b200_bn_update_running(const double* stats, const int* h_channels, const long long* h_counts,
                               float* running, const int* h_rm_off, const int* h_rv_off,
                               long long* nbt, float momentum, void* stream);

/* ------------------------------------------------- fused BN -> conv -> ReLU layers
 * Forward of layer `layer` (0..13): y = act(conv(bn(x)) + b) with
 *   bn: train!=0 -> batch statistics from stats_in (sums over x, N=B*H*W), else
 *       running_mean/running_var; eps 1e-5; zero padding applied AFTER bn.
 *   conv: Conv2d 3x3 pad 1 stride 1|2 (layers 0-6), ConvTranspose2d 3x3 pad 1
 *       stride 1 | stride 2 output_padding 1 (layers 7-13).
 *   act: ReLU except layer 13.
 * If stats_out != NULL, sums of y (the next BN's batch statistics) are accumulated
 * into it in the epilogue.  Replaces bn_k + conv_k + F.relu, ava/models/vae.py:217-223,
 * 263-269. */
int ava_b200_bnconv_fwd(int layer, int B, const float* x, float* y, const float* w, const float* b,
                        const float* gamma, const float* beta, const double* stats_in,
                        const float* running_mean, const float* running_var, int train,
                        double* stats_out, void* stream);

/* Arithmetic of the conv inner products (process-wide, like the reference side's
 * torch.backends.cudnn.allow_tf32 switch that governs the same layers on a GPU):
 *   0  fp32 FMA (default)
 *   1  TF32 tensor cores (mma.sync m16n8k8), operands rounded to TF32: rtol ~2e-3
 *   2  error-compensated 3xTF32 on the tensor cores (x = x_hi + x_lo; a_lo*b_hi + a_hi*b_lo +
 *      a_hi*b_hi, fp32 accumulate): fp32-level accuracy (rtol 1e-4 parity holds)
 *   3  as 2, but where a kernel has the variant (the weight-gradient kernels) the two correction
 *      terms a_lo*b + a*b_lo run as BF16 mma.m16n8k16 -- two k-chunks per instruction, 4 instead
 *      of 6 tensor-core instructions per pair of chunks; per-product error <= 2^-18, unbiased:
 *      rtol 1e-4 parity holds (tests/test_gpu_kernels.py, tests/test_gpu_model.py mode tf32x3b)
 *   4  as 3, and the forward / backward-data kernels form both correction terms of a tap in ONE
 *      BF16 mma.m16n8k16 (k16 = {a_lo | a} x {b | b_lo}): 2 instead of 3 tensor-core instructions
 *      per tap; per-product error <= 2^-19 (3xTF32: 2^-22): rtol 1e-4 parity holds (same tests,
 *      mode tf32x3c) with less margin -- batch-1024 gradients within 7.2e-5 of float64 (mode 3:
 *      4.2e-5), twice as many ReLU units on the other side of zero
 *   5  as 4 for the weight-gradient and backward-data kernels only; the forward kernels (whose
 *      rounding decides ReLU states and feeds every later layer) keep three TF32 terms
 *   6  as 5, plus the forward kernels of the DECODER (layers 7..13): their roundings reach only the
 *      reconstruction, not the latent path -- batch-1024 gradients 4.0e-5 (as mode 5), 260 ReLU units
 *      on the other side of zero (mode 5: 191, mode 4: 403, the float32 reference itself: 129)
 * Layers whose channel counts are not multiples of 8 always use fp32 FMA. */
int ava_b200_set_conv_precision(int mode);
int ava_b200_get_conv_precision(void);

/* Backward of layer `layer`.  `dz` is the gradient w.r.t. this layer's PRE-activation conv output
 * (for layer 13 -- no ReLU, nothing after it -- the loss gradient itself).  Order per layer:
 *
 *   1. tsums: nine per-channel sums of dz (total / first and last row and column / corners; for the
 *      stride-2 conv-transpose layers 8, 10, 12 the four row-parity x column-parity classes and the
 *      last row / column), from which the sum of dz over the pixels whose tap-k partner lies inside
 *      the image follows for each of the 9 taps.  The kernel that writes dz accumulates them in its
 *      epilogue (ava_b200_recon for layer 13, ava_b200_bn_relu_bwd_apply for layer 6,
 *      ava_b200_bnconv_bwd_data of layer+1 for the others).  ava_b200_dz_border_sums is the
 *      stand-alone pass: it defines the nine sums and is the reference the tests compare the
 *      epilogue-accumulated sums against.
 *   2. ava_b200_bnconv_bwd_weight   -> dw, db (OVERWRITTEN) and this layer's two BatchNorm-backward
 *      reductions dstats = (sum g, sum g*(x-mean)), ACCUMULATED (zero them first).  g is the gradient
 *      w.r.t. the BatchNorm output; it is never materialised: both reductions are linear in the
 *      centred raw product Rc = sum dz*(x-mean)_pad the kernel accumulates anyway,
 *         dw = gamma*invstd*Rc + beta*T_k,  sum g = <w, T_k>,  sum g*(x-mean) = <w, Rc>.
 *   3. ava_b200_bnconv_bwd_data     -> dz_prev = [x > 0] * BN-backward(g) with g formed tile by tile
 *      on chip: the gradient w.r.t. the PREVIOUS layer's pre-activation output (same shape as x;
 *      relu_mask = 0 skips the [x > 0] factor).  Not needed for layer 0.
 *
 * Replaces autograd's cudnn_convolution_backward (input + weight), native_batch_norm_backward and
 * threshold_backward for ava/models/vae.py:217-223,263-269 (called from vae.py:352).
 * mode: 1 for the stride-2 conv-transpose layers (8, 10, 12), else 0.  tsums: [9][32] doubles,
 * ACCUMULATED (zero them first). */
#define AVA_TSUM_STRIDE 288 /* doubles per layer in a tsums block: [slot 0..8][channel 0..31] */
int ava_b200_dz_border_sums(const float* dz, int B, int C, int H, int W, int mode, double* tsums, void* stream);

/* x/stats_in: this layer's input and its batch statistics; w/gamma/beta: this layer's parameters.
 * ws: scratch of ava_b200_bnconv_bwd_weight_ws(layer,B) bytes. */
int ava_b200_bnconv_bwd_weight(int layer, int B, const float* dz, const float* x, const float* w,
                               const float* gamma, const float* beta, const double* stats_in,
                               const double* tsums, float* dw, float* db, double* dstats, void* ws,
                               void* stream);
long long ava_b200_bnconv_bwd_weight_ws(int layer, int B);
/* The same with the BatchNorm mode of the forward, as in ava_b200_bnconv_fwd: train != 0 is exactly
 * ava_b200_bnconv_bwd_weight (running_mean / running_var unused).  train == 0: eval-mode BatchNorm,
 * the fixed affine map of the running buffers (invstd_r = 1/sqrt(running_var + eps)); the kernels centre x
 * at running_mean, so Rc = sum dz*(x - running_mean)_pad and
 *    dw = gamma*invstd_r*Rc + beta*T_k,  dstats = (<w, T_k>, <w, Rc>) = (sum g, sum g*(x - running_mean)).
 * stats_in is not read in eval mode (may be NULL). */
int ava_b200_bnconv_bwd_weight_ex(int layer, int B, const float* dz, const float* x, const float* w,
                                  const float* gamma, const float* beta, const double* stats_in,
                                  const float* running_mean, const float* running_var, int train,
                                  const double* tsums, float* dw, float* db, double* dstats, void* ws,
                                  void* stream);

/* gamma == NULL: no BatchNorm backward (dz_prev = [x > 0] * g).
 * tsums_prev (optional): the nine border sums of dz_prev -- layer-1's tsums block -- are accumulated
 * in the epilogue (step 1 for layer-1, without a second read of dz_prev). */
int ava_b200_bnconv_bwd_data(int layer, int B, const float* dz, const float* w, const float* x,
                             const float* gamma, const double* stats_in, const double* dstats, int relu_mask,
                             float* dz_prev, double* tsums_prev, void* stream);
/* The same with the BatchNorm mode of the forward: train != 0 is exactly ava_b200_bnconv_bwd_data
 * (running_var unused).  train == 0 (eval-mode BatchNorm): dz_prev = [x > 0] * gamma*invstd_r * g with
 * invstd_r = 1/sqrt(running_var + eps); stats_in and dstats are not read (may be NULL). */
int ava_b200_bnconv_bwd_data_ex(int layer, int B, const float* dz, const float* w, const float* x,
                                const float* gamma, const double* stats_in, const float* running_var, int train,
                                const double* dstats, int relu_mask, float* dz_prev, double* tsums_prev,
                                void* stream);

/* BN backward finalisation: dgamma[c] = invstd*dstats[32+c], dbeta[c] = dstats[c]
 * for all 14 layers (dstats[32+c] holds sum g*(x-mean)). */
int ava_b200_bn_param_grads(const double* stats, const double* dstats, const int* h_channels,
                            const long long* h_counts, float* grads, const int* h_dgamma_off,
                            const int* h_dbeta_off, void* stream);
/* The same with the BatchNorm mode of the forward: train != 0 is exactly ava_b200_bn_param_grads
 * (running, h_rv_off unused).  train == 0: invstd from layer l's running variance at running[h_rv_off[l]]
 * (element offsets, as in ava_b200_bn_update_running); dstats[32+c] then holds sum g*(x - running_mean).
 * A layer with count 0 is skipped in both modes. */
int ava_b200_bn_param_grads_ex(const double* stats, const double* dstats, const int* h_channels,
                               const long long* h_counts, float* grads, const int* h_dgamma_off,
                               const int* h_dbeta_off, const float* running, const int* h_rv_off, int train,
                               void* stream);

/* out = [a>0] * (p*(g - c1) + q*(a - mean)), per channel c = (i / HW) % C: the backward of
 * the BatchNorm that consumes `a` (train mode; fp64 coefficient math) followed by the ReLU
 * backward of the layer that produced `a`, as one elementwise pass; out may alias g.
 * gamma == NULL: no BatchNorm, only the ReLU mask.  relu == 0: no mask.  The conv layers apply
 * this inside ava_b200_bnconv_bwd_data; the stand-alone pass serves the fc1 -> conv7 seam (ReLU
 * mask of conv7's output on the gradient arriving from fc1).  tsums != NULL: the nine border sums
 * of `out` (rows of width W; mode 0 of ava_b200_dz_border_sums) are accumulated on the way. */
int ava_b200_bn_relu_bwd_apply(const float* g, const float* a, const float* gamma, const double* stats,
                               const double* dstats, int B, int C, int HW, int relu, float* out,
                               double* tsums, int W, void* stream);

/* ------------------------------------------------------------- dense (Linear) layers
 * Y[M,N] = act(X[M,K] . W[N,K]^T + b): torch.nn.Linear (+F.relu / torch.exp),
 * ava/models/vae.py:225-232,258-261.  act: 0 none, 1 relu, 2 exp.
 * `groups` > 1 runs a strided batch: group g uses X + g*x_gs, W + g*w_gs, b + g*b_gs,
 * Y + g*y_gs (the three posterior heads).  precision: 0 = fp32 SIMT,
 * 1 = tcgen05 TF32 tensor cores (rtol 3e-3), 2 = tcgen05 3xTF32 error-compensated
 * (fp32-level, rtol 2e-5).  The tensor-core paths need groups == 1 and M,N multiples of
 * 128, K of 32 (for all three of fwd / bwd_data / bwd_weight); other shapes run on the SIMT
 * kernel regardless of `precision`. */
int ava_b200_linear_fwd(const float* x, int ldx, const float* w, const float* b, float* y, int ldy, int M, int N,
                        int K, int act, int groups, long long x_gs, long long w_gs, long long b_gs,
                        long long y_gs, int precision, void* ws, long long ws_bytes, void* stream);
/* dX[M,K] = (dY (.) mask) . W ; mask = [Ymask>0] if Ymask != NULL (ReLU backward).  Overwrites:
 * `accumulate` must be 0 -- any other value returns an error and leaves dx unchanged. */
int ava_b200_linear_bwd_data(const float* dy, int lddy, const float* ymask, const float* w, float* dx, int lddx,
                             int M, int N, int K, int groups, long long dy_gs, long long w_gs, long long dx_gs,
                             int accumulate, int precision, void* ws, long long ws_bytes, void* stream);
/* dW[N,K] = (dY (.) mask)^T . X ; db[N] = column sums of dY (.) mask.  Overwrites. */
int ava_b200_linear_bwd_weight(const float* dy, int lddy, const float* ymask, const float* x, int ldx, float* dw,
                               float* db, int M, int N, int K, int groups, long long dy_gs, long long x_gs,
                               long long dw_gs, long long db_gs, int precision, void* ws, long long ws_bytes,
                               void* stream);

/* Bias gradients of up to AVA_MAX_BIAS_JOBS Linear layers in two launches: job j computes
 * db[n] = sum_m (mask > 0 ? dy : 0)[m, n] over dy [M, N] (row stride ld; mask may be NULL) --
 * what ava_b200_linear_bwd_weight does per layer when given db; the step passes db = NULL there
 * and collects the layers of a backward segment into one call.  h_jobs is a HOST array.
 * Workspace: ava_b200_bias_grads_ws_bytes.  Replaces the bias half of autograd's Linear backward
 * (ava/models/vae.py:226-232,258-260). */
#define AVA_MAX_BIAS_JOBS 8
typedef struct {
  const float* dy;
  const float* mask;
  float* db;
  int ld, M, N;
} ava_b200_bias_job;
long long ava_b200_bias_grads_ws_bytes(const ava_b200_bias_job* h_jobs, int njobs);
int ava_b200_bias_grads(const ava_b200_bias_job* h_jobs, int njobs, void* ws, long long ws_bytes, void* stream);
long long ava_b200_linear_ws_bytes(int M, int N, int K);

/* ----------------------------------------------------------------------- ELBO
 * Latent part (torch.distributions.LowRankMultivariateNormal(mu,u,d).rsample() /
 * .entropy() + the prior term; ava/models/vae.py:312-316,323):
 *   d = exp(logd); z = mu + u*eps_w + sqrt(d)*eps_d;
 *   acc[0] += sum z^2 ; acc[2] += sum_b H_b,  H_b = 1/2(Z(1+ln 2pi) + ln(1+sum u^2/d) + sum ln d)
 * heads: [B, 3*Z] row-major = (mu | u | logd) as produced by the grouped fc4x layer. */
int ava_b200_latent_fwd(const float* heads, const float* eps_w, const float* eps_d, int B, int Z, float* z,
                        float* d_out, double* acc, void* stream);
/* Gradient of the loss w.r.t. the heads (mu | u | logd) given gz = dL/dz from the
 * decoder (prior term z added here): analytic, SURVEY.md 8(a) "Analytic gradients". */
int ava_b200_latent_bwd(const float* heads, const float* eps_w, const float* eps_d, const float* z,
                        const float* gz, int B, int Z, float* g_heads, void* stream);
/* Backward seed of encode() (VAE.encode returns mu, u, d = exp(logd)): the gradient w.r.t. the heads
 * g_heads [B, 3*Z] = (dmu | du | dd * d) from the seeds dmu, du, dd [B, Z] on encode's three outputs;
 * a NULL seed counts as zero.  d: [B, Z] as the forward returned it (needed when dd != NULL). */
int ava_b200_latent_heads_grad(const float* dmu, const float* du, const float* dd, const float* d, int B, int Z,
                               float* g_heads, void* stream);
/* Input gradient of the loss (VAE.forward with x.requires_grad): dx = dx_enc - precision * (x_rec - x),
 * the encoder's part (layer 0's backward-data output; NULL counts as zero) plus the direct term of the
 * reconstruction loss (ava/models/vae.py:319-320).  n % 4 == 0; dx may alias dx_enc. */
int ava_b200_recon_input_grad(const float* dx_enc, const float* x, const float* x_rec, long long n, float precision,
                              float* dx, void* stream);
/* Reconstruction term (ava/models/vae.py:319-320): acc[1] += sum (x - x_rec)^2 and,
 * if g != NULL, g = precision * (x_rec - x) = dL/dx_rec.  tsums != NULL (with g): also the nine
 * border sums of g viewed as [n/(H*W)] single-channel H x W planes (mode 0 of
 * ava_b200_dz_border_sums, channel 0), accumulated while g is written -- g is the decoder's last
 * layer's dz, whose weight-gradient finalisation needs them. */
int ava_b200_recon(const float* x, const float* x_rec, long long n, float precision, float* g, double* acc,
                   double* tsums, int H, int W, void* stream);
/* loss = 1/2(acc0 + Z ln 2pi) + 1/2 XDIM ln(2pi/prec) + 1/2 prec acc1 - acc2, written as
 * fp32 to loss[0] and accumulated (fp64) into loss_sum[0] if non-NULL (device-side epoch
 * accumulator replacing loss.item() per step, ava/models/vae.py:351). */
int ava_b200_elbo_finalize(const double* acc, int Z, int xdim, float precision, float* loss, double* loss_sum,
                           void* stream);

/* ----------------------------------------------------------------------- Adam
 * torch.optim.Adam (defaults: no weight decay, no amsgrad), one launch over the flat
 * parameter buffer; ava/models/vae.py:119,353.  step_count: device fp32 scalar holding
 * the step number BEFORE this update (incremented by the kernel; mirrors torch's
 * per-tensor `step` state).  lr/betas/eps are doubles, as torch holds them. grad_scale multiplies g on load (1.0 normally). */
int ava_b200_adam_step(float* p, const float* g, float* m, float* v, long long n, float* step_count, double lr,
                       double beta1, double beta2, double eps, float grad_scale, void* stream);

/* Same update with the hyper-parameters read from DEVICE memory: hyper = {lr, beta1, beta2, eps}
 * (doubles), so that a captured CUDA graph of the step follows optimizer.param_groups (learning-
 * rate schedules, the lr a checkpoint restores: ava/models/vae.py:470) without re-capture. */
int ava_b200_adam_step_dev(float* p, const float* g, float* m, float* v, long long n, float* step_count,
                           const double* hyper, float grad_scale, void* stream);

/* Data-parallel optimizer step fused with its collectives over NVLink / NVSwitch peer memory
 * (csrc/dp.cu): the data-parallel form of optimizer.step(), ava/models/vae.py:353 -- replaces
 * "NCCL all-reduce(SUM) of the flat gradient, then Adam on every rank".  Rank r sums the
 * world gradient copies of ITS 1/world slice (peer loads, or one multimem.ld_reduce through the
 * switch when multicast pointers are given), applies Adam to that slice only (moments are sharded)
 * and stores the new parameters into every rank's parameter buffer; two flag barriers order it
 * against the ranks' backward / next forward passes.
 *   h_peers: HOST struct of DEVICE pointers: every rank's flat gradient buffer, flat parameter
 *            buffer and flag block (2*AVA_DP_MAX_WORLD uint32, zero-initialised once), all in
 *            symmetric (peer-mapped) memory; index = rank; grad_mc/param_mc = multicast views or NULL
 *   m, v:    this rank's LOCAL moment buffers (only its slice is read and written)
 *   local:   LOCAL device uint32[4], zero-initialised once: [0] step sequence number,
 *            [1] CTA counter, [2] set to 1 if a peer did not arrive within 20 s (the kernel
 *            then carries on instead of hanging; the caller checks it)
 * Every rank must make the same sequence of calls.  n % 4 == 0; world <= AVA_DP_MAX_WORLD. */
#define AVA_DP_MAX_WORLD 8
typedef struct {
  const float* grad[AVA_DP_MAX_WORLD];
  float* param[AVA_DP_MAX_WORLD];
  unsigned int* flags[AVA_DP_MAX_WORLD];
  const float* grad_mc;
  float* param_mc;
} ava_b200_dp_peers;
int ava_b200_adam_step_dp(const ava_b200_dp_peers* h_peers, int rank, int world, float* m, float* v,
                          long long n, float* step_count, const double* hyper, float grad_scale,
                          unsigned int* local, void* stream);

/* Synchronised BatchNorm for data-parallel training (csrc/bnsync.cu): one layer's BatchNorm sums
 * exchanged over NVLink peer memory so that every rank normalises with the statistics of the GLOBAL
 * batch, as torch.nn.BatchNorm2d does in the reference's single process on the concatenated batch
 * (ava/models/vae.py:135-141,162-168).  One single-CTA launch per layer and pass: rank r publishes its
 * sums and element count, every rank adds the world copies in rank order 0..world-1 in fp64 (so all
 * ranks get the same bits) and writes back
 *     sums[c] = (sum over ranks of sums[c]) * (local_count / global_count),   c < channels, 32 + c,
 * i.e. the global sums scaled to this rank's share: every kernel that divides `sums` by its own local
 * count then sees the global mean and biased variance (forward stats), or the global c1 and q of the
 * BatchNorm backward (dstats).  Entries of channels >= `channels` are left untouched.
 *   h_peers:     HOST struct of DEVICE pointers into symmetric (peer-mapped) memory, index = rank:
 *                slots[r] = rank r's 2 * AVA_BN_SYNC_SLOT doubles, flags[r] = rank r's uint32 flag;
 *                both zero-initialised once, before any rank's first call
 *   local_count: B * H * W of this rank's shard (0 for an empty shard: it contributes zeros)
 *   running:     NULL for the backward (dstats) exchanges; otherwise the forward exchange also applies
 *                the running-buffer update of ava_b200_bn_update_running with the global sums and count
 *                to running[rm_off + c] / running[rv_off + c] and adds 1 to nbt[0] (skipped when the
 *                global count is 0) -- identical on every rank
 *   local:       LOCAL device uint32[2], zero-initialised once: [0] exchange sequence number (advanced by
 *                the kernel, so graph replays need no host involvement), [1] set to 1 if a peer did not
 *                arrive within 20 s (the kernel then carries on; the caller checks it)
 * Every rank must make the same sequence of calls.  world <= AVA_DP_MAX_WORLD, 1 <= channels <= 32. */
#define AVA_BN_SYNC_SLOT 65 /* doubles per slot: [0..63] a stats block, [64] the element count */
typedef struct {
  double* slots[AVA_DP_MAX_WORLD];
  unsigned int* flags[AVA_DP_MAX_WORLD];
} ava_b200_bn_sync_peers;
int ava_b200_bn_stats_exchange(const ava_b200_bn_sync_peers* h_peers, int rank, int world, double* sums,
                               int channels, long long local_count, float* running, int rm_off, int rv_off,
                               long long* nbt, float momentum, unsigned int* local, void* stream);

/* ------------------------------------------------------------------- get_spec
 * Batched spectrogram front end: ava/preprocessing/utils.py:18-110 (get_spec) with
 * scipy.signal.stft semantics (periodic Hann, zero boundary extension, zero padding to a
 * hop multiple, scale 1/sum(win)).  One CTA per window; computed in fp64.
 *   audio:      concatenated audio of all files on device: int16 (is_f32 = 0), fp32 (1) or fp64 (2)
 *   seg_start:  [n] first sample of each segment in `audio`
 *   seg_len:    [n] number of samples (0 => output zeros, the reference's
 *               "too short" branch, ava/preprocessing/utils.py:69-71)
 *   window/scale: the analysis window [nperseg] (fp64) and 1/sum(window), computed by
 *               the host with the same scipy call the reference makes
 *   t_idx/t_frac [n,n_t]: lower frame index and weight of each target time;
 *               t_idx < 0 marks an out-of-range target (the fill value -1e12 normalised and
 *               clipped: 0, or 1 when spec_max < spec_min)
 *   f_idx/f_frac [n_f]: same for the target frequencies (shared by all windows)
 *   max_frames: upper bound on the number of STFT frames of any segment
 *   out: [n, n_f, n_t] fp32 (numpy_to_tensor's float32, ava/models/utils.py:444-446)
 *   out64: optional [n, n_f, n_t] fp64 (the array get_spec itself returns) */
int ava_b200_get_spec_batch(const void* audio, int is_f32, const long long* seg_start, const int* seg_len, int n,
                            int nperseg, int noverlap, int remove_dc, const double* window, double scale,
                            const int* t_idx, const double* t_frac, int n_t, const int* f_idx,
                            const double* f_frac, int n_f, int max_frames, double spec_min, double spec_max,
                            float* out, double* out64, void* stream);

/* within_syll_normalize (ava/preprocessing/utils.py:106-109), per spectrogram of m = n_f*n_t values:
 *   spec -= np.quantile(spec, q); spec[spec < 0] = 0; spec /= spec.max() + 1e-12
 * in float64 on spec64 [n, m] in place (the quantile by an exact radix select + numpy's linear
 * interpolation); spec32 (optional) receives the float32 copy.  The values must be >= 0 (the
 * select orders them by bit pattern; -0.0 is read as +0.0), as get_spec's clipped output is.
 * Bit-identical to numpy except for the sign of zero: every zero written is +0.0, where numpy
 * keeps an input's -0.0 when the quantile is 0. */
int ava_b200_quantile_normalize(double* spec64, float* spec32, int n, int m, double q, void* stream);

/* Target-time tables of a batch of fixed-duration windows computed on the device (the
 * shotgun path, ava/models/window_vae_dataset.py:231-235: target_times = linspace(onset,
 * offset, n_t); bracketing and fill rule of scipy interp2d, ava/preprocessing/utils.py:80-81,99).
 * Same float64 operations as the host tables, bit for bit.
 *   grid0 [n]: max(0, t1) of each window; K [n]: STFT frames of each window (>= 3);
 *   base [kmax]: frame times of a segment starting at 0; tstart/tstop [n]: first / last target
 *   t_idx/t_frac [n,n_t]: outputs in the layout ava_b200_get_spec_batch consumes. */
int ava_b200_window_time_tables(const double* grid0, const int* K, const double* base, int kmax,
                                const double* tstart, const double* tstop, int n, int n_t, int* t_idx,
                                double* t_frac, void* stream);

/* ------------------------------------------------- MMD^2 between sets of latent means
 * Downstream statistic on get_latent's output, ava/plotting/mmd_plots.py:255-312, 450-476.
 * x: [N,D] float64 latent means; seg[i] in [0,n_seg) = condition of row i.
 * S[a*n_seg+b] = sum_{i in a, j in b} exp(A*||x_i-x_j||^2), A = -0.5/sigma^2 (S is zeroed by
 * the call).  MMD^2(a,b) = (S_aa-n_a)/(n_a(n_a-1)) + (S_bb-n_b)/(n_b(n_b-1)) - 2 S_ab/(n_a n_b). */
int ava_b200_mmd_block_sums(const double* x, int N, int D, const int* seg, int n_seg, double A, double* S,
                            void* stream);
/* out[k] = ||x[ia[k]]-x[ib[k]]||^2 (mode 0) or exp(A * that) (mode 1); numpy summation order. */
int ava_b200_pair_kernel(const double* x, int D, const long long* ia, const long long* ib, long long n,
                         double A, int mode, double* out, void* stream);

/* ------------------------------------------------- PCA of the latent means
 * sklearn.decomposition.PCA(n_components=K).fit_transform on get_latent's output,
 * ava/data/data_container.py:538-551 (_make_latent_mean_pca_projection).
 * x: [N,D] rows, float64 (is_f32 = 0) or the encoder's float32 latents (is_f32 = 1), D <= 64.
 * fit: mean[D]; cov[D*D] = sample covariance (divisor N-1); evals[D] descending, clipped at 0;
 * comps[D*D]: row k = unit eigenvector k, its largest-magnitude entry positive (scikit-learn's
 * svd_flip with u_based_decision=False).  ws: ava_b200_pca_ws_bytes(D) bytes of scratch.
 * transform: out[N,K] = (x - mean) . comps[:K]^T. */
long long ava_b200_pca_ws_bytes(int D);
int ava_b200_pca_fit(const void* x, int is_f32, long long N, int D, double* mean, double* cov, double* evals,
                     double* comps, void* ws, long long ws_bytes, void* stream);
int ava_b200_pca_transform(const void* x, int is_f32, long long N, int D, const double* mean, const double* comps,
                           int K, double* out, void* stream);

/* ------------------------------------------------- UMAP of the latent means (csrc/umap.cu)
 * The device stages of umap-learn 0.5's UMAP(metric='euclidean').fit_transform, the projection the
 * reference builds in ava/data/data_container.py (_make_latent_mean_umap_projection).  The Python class
 * LatentUMAP (data/latent_umap.py) strings them together; the sorts, prefix sums and compactions
 * between the stages are its plumbing (torch), every number is computed here.
 *
 * Exact k nearest neighbours (replaces umap.umap_.nearest_neighbors, NNDescent): x [N, D] rows, float64
 * (is_f32 = 0) or float32 (1), finite, D <= 64, 1 <= k <= min(N, 100).  Writes the first k rows by
 * (distance, not-self, index) of fp64 difference-form distances: knn_idx [N, k] int32 (the row itself
 * first), knn_dist [N, k] Euclidean, float64; exact at any scale and offset of the data (up to fp64
 * overflow of the squared distances).  An fp32 brute-force pass on y = (x - shift) 2^-e (shift: the mean
 * of the first 1024 rows; e: the exponent of M = max |x - shift|, so |y| < 1) keeps the best KP >= k + 8
 * candidates per row (KP in {16, 32, 64, 128}) and an fp64 pass ranks them.  A row is certified when its
 * k-th fp64 distance is strictly below a lower bound on the distance of every candidate it dropped:
 *   2^e ((sqrt(t32 - (DP + 1) 2^-149) / (1 + g)) - 2 delta sqrt(D)) (1 - 2^-40),
 * t32 the worst kept fp32 squared distance, DP the padded D, g = (DP/2 + 3) 2^-24 (1.001),
 * delta = (2^-24 + 2^-52) M 2^-e + 2^-149; or when N <= KP.  Other rows are rescanned in fp64.
 * When the ceil(N / 128) query CTAs do not fill one wave, the rows are split into S slices (see
 * ava_b200_umap_knn_query); the lists are exact and unique under the ranking order, so S changes no output.
 * ws: ava_b200_umap_knn_ws_bytes(N, D, k) bytes. */
long long ava_b200_umap_knn_ws_bytes(int N, int D, int k);
int ava_b200_umap_knn(const void* x, int is_f32, int N, int D, int k, int* knn_idx, double* knn_dist, void* ws,
                      long long ws_bytes, void* stream);
/* Exact k nearest rows of x [N, D] for each query row of q [Nq, D] (umap-learn's transform searches its fitted
 * index): the same dtype for both (is_f32), finite, D <= 64, 1 <= k <= min(N, 100), Nq >= 0.  Writes the first k
 * rows by (distance, index) of fp64 difference-form distances, with no preference for any row: knn_idx [Nq, k]
 * int32 (a query equal to a data row has it first, at distance 0; equal data rows come lowest index first),
 * knn_dist [Nq, k] Euclidean, float64.  The same passes as ava_b200_umap_knn, with the shift taken from the data
 * and the range M over the data and the queries together, so queries far outside the data stay exact.  When the
 * Q = ceil(Nq / 128) query CTAs do not fill one wave of 4 CTAs per SM, the data rows are split into S slices
 * (S * KP <= 256, slices of >= 1024 rows, the S whose Q S CTAs fill their last wave best; a larger S only if it
 * fills 2% more), each keeping its own top KP; the fp64 pass ranks all S * KP candidates, and the certificate uses the
 * smallest of the slices' worst kept fp32 distances.  ws: ava_b200_umap_knn_query_ws_bytes(Nq, N, D, k) bytes. */
long long ava_b200_umap_knn_query_ws_bytes(int Nq, int N, int D, int k);
int ava_b200_umap_knn_query(const void* q, int Nq, const void* x, int N, int is_f32, int D, int k, int* knn_idx,
                            double* knn_dist, void* ws, long long ws_bytes, void* stream);
/* umap.umap_.smooth_knn_dist (n_iter 64, tolerance 1e-5, MIN_K_DIST_SCALE 1e-3 against the row's mean
 * distance, or the mean of all N*k distances -- a fixed-order sum -- where rho = 0) followed by
 * umap.umap_.compute_membership_strengths, in fp64: rho [N], sigma [N], weights [N, k] (0 for the row
 * itself).  ws: 1 double of scratch. */
int ava_b200_umap_smooth_knn(const int* knn_idx, const double* knn_dist, int N, int k, double local_connectivity,
                             double* rho, double* sigma, double* weights, double* ws, void* stream);
/* The memberships of umap-learn's transform: smooth_knn_dist of the query lists of ava_b200_umap_knn_query with
 * local_connectivity max(0, local_connectivity - 1) (pass the fitted model's value; the MIN_K_DIST_SCALE floor is
 * against the mean of the Nq*k query distances), then compute_membership_strengths(bipartite=True): no entry is
 * zeroed, as no query is a data row.  rho [Nq], sigma [Nq], weights [Nq, k] in the lists' order; ws: 1 double. */
int ava_b200_umap_smooth_knn_query(const int* knn_idx, const double* knn_dist, int Nq, int k,
                                   double local_connectivity, double* rho, double* sigma, double* weights, double* ws,
                                   void* stream);
/* The fuzzy union of umap.umap_.fuzzy_simplicial_set (set_op_mix_ratio 1): P = A + A^T - A.*A^T.
 * edge_keys writes 2*N*k keys: row*N + col for (i, j) and (j, i) of every neighbour j != i, -1 for the
 * self entries.  The caller sorts them and drops duplicates and -1 (nnz keys remain); graph then writes
 * the CSR of P: rows/cols/vals [nnz] in row-major, column-sorted order and rowptr [N + 1] (int64). */
int ava_b200_umap_edge_keys(const int* knn_idx, int N, int k, long long* keys, void* stream);
int ava_b200_umap_graph(const long long* keys, long long nnz, int N, const int* knn_idx, const double* weights,
                        int k, int* rows, int* cols, double* vals, long long* rowptr, void* stream);
/* umap.umap_.make_epochs_per_sample on the pruned edge weights (vmax: device pointer to their maximum)
 * and the set-up of umap.layouts.optimize_layout_euclidean: eps = n_epochs / (n_epochs * w / vmax) (-1 where
 * that is 0), eps_neg = eps / negative_sample_rate, next = eps, next_neg = eps_neg; all [n]. */
int ava_b200_umap_epochs_per_sample(const double* vals, long long n, const double* vmax, int n_epochs,
                                    double negative_sample_rate, double* eps, double* eps_neg, double* next,
                                    double* next_neg, void* stream);
/* Connected components of the symmetric CSR graph (scipy.sparse.csgraph.connected_components as
 * umap.spectral calls it): one round of min-label hooking.  Start from labels[i] = i and repeat with
 * *changed zeroed until a round leaves it 0; then labels[i] = the smallest vertex of i's component. */
int ava_b200_umap_components_step(const long long* rowptr, const int* cols, int N, int* labels, int* changed,
                                  void* stream);
/* dis[i] = 1 / sqrt(row sum i of P): the D^-1/2 of umap.spectral.spectral_layout. */
int ava_b200_umap_degree(const long long* rowptr, const double* vals, int N, double* dis, void* stream);
/* The normalised Laplacian of one component applied to a block (the product of the eigensolver that replaces
 * scipy.sparse.linalg.eigsh in umap.spectral): for r < n, v = verts[r],
 *   Y[r, :] = X[r, :] - dis[v] * sum_j P[v, j] dis[j] X[pos[j], :],   X, Y [n, m] row-major, m <= 32,
 * pos: vertex -> row of its component.  A warp per row; bitwise reproducible. */
int ava_b200_umap_spmm(const long long* rowptr, const int* cols, const double* vals, const int* verts, int n,
                       const int* pos, const double* dis, const double* X, int m, double* Y, void* stream);
/* out [p, q] = A^T B for A [n, p], B [n, q] row-major (p*q <= 2048 and p + q <= 192), summed in a fixed order; ws:
 * ava_b200_umap_gram_ws_bytes(p, q) bytes.  combine: Y [n, q] = A [n, p] . C [p, q]. */
long long ava_b200_umap_gram_ws_bytes(int p, int q);
int ava_b200_umap_gram(const double* A, int p, const double* B, int q, int n, double* out, void* ws,
                       long long ws_bytes, void* stream);
int ava_b200_umap_combine(const double* A, int p, const double* C, int q, int n, double* Y, void* stream);
/* out[i] = draw i of stream `stream_id` under `seed` (counter-based: the splitmix64 finaliser applied
 * along (seed, stream_id, i, 0|1)): kind 0 uniform(-scale, scale), kind 1 normal(0, scale). */
int ava_b200_umap_random(unsigned long long seed, unsigned long long stream_id, long long n, int kind, double scale,
                         double* out, void* stream);
/* The end of umap.umap_.simplicial_set_embedding's initialisation: per axis d,
 * v = (float)(init * expansion) + (float)noise (noise may be NULL), then emb = 10 (v - min) / (max - min)
 * in fp32 (0 where max == min).  init [N, dim] float64, emb [N, dim] float32, dim <= 8. */
int ava_b200_umap_init_layout(const double* init, const double* noise, double expansion, int N, int dim,
                              float* emb, void* stream);
/* One epoch n of umap.layouts._optimize_layout_euclidean_single_epoch over the edges [e0, e1) (head ->
 * tail, both moved by the attraction; negatives move the head), Hogwild on the fp32 embedding [N, dim].
 * Negative vertex p of edge e in epoch n: umap_hash(seed, n, e, p) mod N (the hash of
 * ava_b200_umap_random).  alpha is the epoch's learning rate. */
int ava_b200_umap_sgd_epoch(float* emb, int N, int dim, const int* head, const int* tail, const double* eps,
                            const double* eps_neg, double* next, double* next_neg, long long e0, long long e1,
                            int epoch, double a, double b, double gamma, double alpha, unsigned long long seed,
                            void* stream);
/* umap.umap_.init_graph_transform: for each query row i, over its k entries in increasing column order
 * (cols/weights [Nq, k], the unpruned bipartite graph with each row sorted by column): a weight of exactly 1 sets
 * out[i] = emb[col] and ends the row; otherwise out[i] += (w / row_sum) emb[col], row_sum the sequential fp64 sum
 * of the row's weights in column order, each product in fp64 and each sum rounded to fp32 (no FMA).  emb [N, dim]
 * is the fitted float32 embedding, out [Nq, dim] float32, dim <= 8. */
int ava_b200_umap_init_transform(const int* cols, const double* weights, int Nq, int k, const float* emb, int N,
                                 int dim, float* out, void* stream);
/* umap.layouts.optimize_layout_euclidean(move_other=False) over all n_epochs of the transform in one launch: the
 * pruned edges of query row i are [rowptr[i], rowptr[i + 1]) (tail: the fitted row; eps, eps_neg, next, next_neg
 * from ava_b200_umap_epochs_per_sample), emb_q [Nq, dim] starts at the initialisation and is updated in place; the
 * fitted embedding emb [N, dim] is only read.  Epoch n uses alpha = initial_alpha (1 - n / n_epochs).  The
 * attraction moves the head only; negative sample p of edge e in epoch n is row
 * umap_hash(umap_hash(seed, 5 << 32, 0, 0), n, e, p) mod N of emb, never skipped (at distance 0 the step is +4 per
 * axis).  One thread per query row: race-free, so bitwise reproducible and equal to the sequential algorithm. */
int ava_b200_umap_sgd_transform(float* emb_q, int Nq, const float* emb, int N, int dim, const long long* rowptr,
                                const int* tail, const double* eps, const double* eps_neg, double* next,
                                double* next_neg, int n_epochs, double a, double b, double gamma,
                                double initial_alpha, unsigned long long seed, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AVA_B200_H */
