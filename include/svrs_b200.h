/*
 * svrs_b200.h - C ABI of the B200-native (sm_100a) kernels behind the Simple-VAE-RS training step.
 *
 * The reference (Etienne-bdt/Simple-VAE-RS) has no FFI layer: its hot path is Python calling
 * torch.nn / torch.nn.functional.  Each entry point below therefore cites the reference CALL SITE
 * whose arithmetic it replaces (file:line into the reference tree).  The Python host code in
 * simple-vae-rs_b200/ binds these with ctypes (see INTEGRATION.md) and keeps the reference's
 * Python API (models.VAE / models.Cond_SRVAE / loss.base_loss / loss.cond_loss / fit()).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless named host_*; the library never allocates, frees,
 *     or synchronises; work is enqueued on `stream` (a cudaStream_t passed as void*).
 *   - activations are NHWC ("pixel-major"): [N][H][W][C], dtype SVRS_F32 or SVRS_BF16.
 *   - weights are consumed in packed per-tap form produced by svrs_pack_weights():
 *         KN pack: [tap][K][N]   (tap = ky*ksize + kx, K = reduction channels, N = output channels)
 *   - return value: 0 = enqueued, <0 = error (SVRS_E_*); svrs_last_error() gives the message.
 *   - thread-safety: calls are re-entrant; the error string is thread-local.
 */
#ifndef SVRS_B200_H
#define SVRS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVRS_F32 0
#define SVRS_BF16 1

#define SVRS_ACT_NONE 0
#define SVRS_ACT_SIGMOID 1  /* nn.Sigmoid   - cond_vae.py:80,143 ; vae.py:84 */
#define SVRS_ACT_HARDTANH7 2 /* nn.Hardtanh(-7,7) - cond_vae.py:230 */

#define SVRS_E_ARG (-1)
#define SVRS_E_CUDA (-2)
#define SVRS_E_UNSUPPORTED (-3)

const char* svrs_last_error(void);
int svrs_abi_version(void);
/* Number of CUDA kernels this library has launched in the process so far (every launch site counts itself); the
 * difference across a step is bench.py's `gpu_launches`. */
int64_t svrs_launch_count(void);
/* Kernel-name trace for profile attribution: svrs_trace_reset(1) starts recording the names of the kernels launched by
 * the calling thread, svrs_trace() returns them comma-separated, svrs_trace_reset(0) switches recording off. */
void svrs_trace_reset(int enable);
const char* svrs_trace(void);
/* compute capability major*10+minor of device `dev`, or <0 */
int svrs_device_cc(int dev);

/* ---- layout glue: nn.Flatten / nn.Unflatten / torch.chunk / torch.cat views
 *      (cond_vae.py:47,52,106,111,163,168,188,192,209,212,229,240-244,254,259,272).
 *      NCHW is the reference's (API-facing) order, NHWC the internal one.  `src_ld`/`dst_ld` are the
 *      per-sample strides (elements) of the NCHW side so that a [B, C*H*W] slice of a wider flat
 *      latent row (torch.cat / torch.chunk) can be addressed in place. */
int svrs_nchw_to_nhwc(const void* src, int src_dtype, int64_t src_ld, void* dst, int dst_dtype,
                      int N, int C, int H, int W, void* stream);
int svrs_nhwc_to_nchw(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t dst_ld,
                      int N, int C, int H, int W, int accumulate, void* stream);

/* ---- weight packing: torch layout w[d0][d1][kk] (fp32 master) -> p01[kk][d0][d1], p10[kk][d1][d0]
 *      in `dtype`.  nn.Conv2d weight is [Cout][Cin][k][k] (layers.py:231-236), nn.ConvTranspose2d
 *      weight is [Cin][Cout][k][k] (layers.py:275-277).  Either output may be NULL. */
int svrs_pack_weights(const float* w, int d0, int d1, int kk, void* p01, void* p10, int dtype,
                      void* stream);

/* All layers in one launch: `jobs` is a DEVICE array of njobs records
 *   { const float* w; void* p01; void* p10; int d0, d1, kk; int tile0; int tiles_b; int pad; }   (svrs_pack_job_bytes() each)
 * where a layer is cut into 32 x 16 tiles of its (d0, d1) plane, tiles_b = ceil(d1/16), and tile0 is the running sum of
 * the tile counts of the preceding jobs; total_tiles = sum of all tile counts; max_kk = largest kk (<= 16); njobs <= 128. */
int svrs_pack_job_bytes(void);
int svrs_pack_weights_multi(const void* jobs, int njobs, int total_tiles, int max_kk, int dtype, void* stream);
/* inverse direction for gradients: same job records with w = torch-layout fp32 gradient (+=) and p01 = the packed
 * fp32 scratch [kk][d1][d0] the tensor-core wgrad kernels accumulated into (see svrs_conv2d_wgrad) */
int svrs_unpack_grads_multi(const void* jobs, int njobs, int total_tiles, int max_kk, void* stream);

/* Two kernels sit behind each fprop/dgrad entry point:
 *   - conv_tc   (csrc/conv_tc.cu): tcgen05.mma + TMEM accumulators + TMA-fed swizzled operands; taken when
 *     dtype == BF16, the reduction channels K are a multiple of 8 and at least 16 (16-byte NHWC rows; when K % 16 != 0
 *     the last 64-channel chunk is TMA zero fill past K), the written channels a multiple of 4 and the output map tiles
 *     into 128-pixel boxes; it consumes the NK pack `w_nk` = [tap][N][K] (K contiguous).
 *   - conv_simt (csrc/conv_simt.cu): fp32-FMA multi-tap GEMM for everything else (fp32 parity mode, 4/16-channel
 *     layers, odd channel counts); it consumes the KN pack `w_kn` = [tap][K][N].
 * The two packs of a layer are each other's transposes, i.e. the (p01, p10) pair of svrs_pack_weights: the KN pack
 * of fprop is the NK pack of dgrad and vice versa.  w_nk may be NULL (forces the SIMT kernel). */
void svrs_set_tc_enabled(int enabled);   /* default 1; 0 forces the SIMT kernels everywhere (A/B tests) */
/* conv3_halo (csrc/conv_halo.cu): 3x3 stride-1 fprop/dgrad on maps tiling into 8x16 blocks load each tile's activation
 * halo ONCE and address the nine taps as shared-memory descriptors.  mode 0 = off (per-tap TMA kernel), 1 = on (default). */
void svrs_set_halo_mode(int mode);
/* 1 if conv_tc takes a GEMM of these dims.  Channel rule of the tcgen05 kernels (conv_tc and the wgrad kernels below):
 * C % 8 == 0 and C >= 16 for the channels a kernel reads through TMA; channel counts with rows that are not 16-byte
 * multiples (42, 84, 53, 106, 212, ...) and 8-channel operands go to the CUDA-core kernels. */
int svrs_tc_would_run(int dtype, int K, int Nc, int OH, int OW);

/* ---- nn.Conv2d k3 s1 p1 / k4 s2 p1 (layers.py:231-236; every bare nn.Conv2d of cond_vae.py / vae.py)
 *      x [N,H,W,Cin] -> y [N,H/s,W/s,Cout];  w_kn = p10 pack [tap][Cin][Cout]; bias fp32 [Cout] or NULL.
 *      ksize 3 => stride 1, ksize 4 => stride 2 (pad 1 both). */
int svrs_conv2d_fprop(const void* x, const void* w_kn, const void* w_nk, const float* bias, void* y, int dtype,
                      int N, int H, int W, int Cin, int Cout, int ksize, int act, void* stream);
/* Extended fprop (same call sites).  Extras, each optional:
 *   out_dtype - storage type of y when it differs from `dtype`: SVRS_F32 output of a bf16 conv is available on the
 *               narrow per-pixel kernel (the 16->4 + Sigmoid tail of both decoders, cond_vae.py:79-80,142-143: x_hat reaches
 *               the NLL without a bf16 rounding);
 *   y_nchw    - second output, fp32, in the reference's NCHW-flat order: y_nchw[n*y_nchw_ld + c*OH*OW + oy*OW + ox], written
 *               by the tcgen05 epilogue straight from the fp32 accumulators (after bias / activation).  This is how the
 *               posterior and prior heads (nn.Flatten + torch.chunk, cond_vae.py:47,106,163,209,229,254,259) leave the
 *               conv stacks: no bf16 rounding of mu / logvar and no separate layout kernel.  y may then be NULL;
 *   bn_sums   - SVRS_BN_REPLICAS x double[2*Cout]: per-channel sum and sum of squares of the conv output (before the
 *               activation), accumulated in the epilogue from the fp32 accumulators - the batch statistics of the
 *               nn.BatchNorm2d that follows (layers.py:237,252-253) without re-reading the tensor (replaces svrs_bn_stats).
 * Returns SVRS_E_UNSUPPORTED when the kernel that takes this shape cannot provide a requested extra (callers then use the
 * separate kernels: svrs_nhwc_to_nchw / svrs_bn_stats). */
int svrs_conv2d_fprop_ex(const void* x, const void* w_kn, const void* w_nk, const float* bias, void* y, int dtype,
                         int out_dtype, float* y_nchw, int64_t y_nchw_ld, double* bn_sums,
                         int N, int H, int W, int Cin, int Cout, int ksize, int act, void* stream);
/* dgrad: dy [N,H/s,W/s,Cout] -> dx [N,H,W,Cin]; w_kn = p01 pack [tap][Cout][Cin].
 * (autograd of the same call sites, reached through loss.backward() models/base.py:105) */
int svrs_conv2d_dgrad(const void* dy, const void* w_kn, const void* w_nk, void* dx, int dtype,
                      int N, int H, int W, int Cin, int Cout, int ksize, void* stream);
/* dw_packed (may be NULL): a zeroed fp32 scratch of the weight's size.  When given, the tcgen05 kernels accumulate
 * there in the per-tap layout [tap][d1][d0] (d0, d1 = the weight's first two torch dims; d0 fastest): each CTA stages
 * its TMEM accumulators in shared memory and adds them with a handful of TMA tensor reductions
 * (cp.reduce.async.bulk.tensor .add.f32) instead of thousands of per-thread atomics - measured: a warp sustains only
 * ~1 global store/atomic per ~100 cycles, which made the epilogue 4-8x longer than the MMA phase on small maps.
 * svrs_unpack_grads_multi() later adds every layer's scratch into the torch-layout gradient in one launch.  The SIMT
 * kernels always accumulate into dw directly.
 * wgrad: dw[Cout][Cin][k][k] += sum x (*) dy  (fp32, torch layout, ATOMIC accumulate - zero it first);
 * db[Cout] += column sums of dy when db != NULL.  `ksplit` <= 0 picks a split automatically. */
int svrs_conv2d_wgrad(const void* x, const void* dy, float* dw, float* dw_packed, float* db, int dtype,
                      int N, int H, int W, int Cin, int Cout, int ksize, int ksplit, void* stream);


/* ---- nn.ConvTranspose2d k4 s2 p1 (layers.py:275-277): x [N,H,W,Cin] -> y [N,2H,2W,Cout].
 *      four output-parity sub-convolutions of 2x2 taps.  w_kn = p01 pack [tap][Cin][Cout]. */
int svrs_convT2d_fprop(const void* x, const void* w_kn, const void* w_nk, const float* bias, void* y, int dtype,
                       int N, int H, int W, int Cin, int Cout, int act, void* stream);
/* with the fused BatchNorm statistics of svrs_conv2d_fprop_ex (up_block: ConvTranspose2d -> BatchNorm2d, layers.py:275-278) */
int svrs_convT2d_fprop_ex(const void* x, const void* w_kn, const void* w_nk, const float* bias, void* y, int dtype,
                          double* bn_sums, int N, int H, int W, int Cin, int Cout, int act, void* stream);
/* dgrad: dy [N,2H,2W,Cout] -> dx [N,H,W,Cin]; w_kn = p10 pack [tap][Cout][Cin]. */
int svrs_convT2d_dgrad(const void* dy, const void* w_kn, const void* w_nk, void* dx, int dtype,
                       int N, int H, int W, int Cin, int Cout, void* stream);
/* wgrad: dw[Cin][Cout][4][4] += ... ; db[Cout] += column sums of dy. */
int svrs_convT2d_wgrad(const void* x, const void* dy, float* dw, float* dw_packed, float* db, int dtype,
                       int N, int H, int W, int Cin, int Cout, int ksplit, void* stream);

/* Layout the wgrad entry points leave in dw_packed for a problem: 1 = per-tap packed [tap][d1][d0] (tcgen05 kernels:
 * bf16 with both channel counts multiples of 8 and at least 16, the channel rule of svrs_tc_would_run, and a map that
 * tiles into 128-pixel boxes; ragged boxes are zero-filled and clipped, nothing outside [kk][d1][d0] is written),
 * 0 = nothing (a SIMT kernel accumulates torch layout into dw).  The fused optimiser (svrs_adam_multi) passes the SAME
 * buffer as dw and dw_packed and reads the gradient in whichever layout this reports, so no unpack pass is needed. */
int svrs_conv2d_wgrad_layout(int dtype, int N, int H, int W, int Cin, int Cout, int ksize);
int svrs_convT2d_wgrad_layout(int dtype, int N, int H, int W, int Cin, int Cout);

/* ---- nn.BatchNorm2d (+ nn.ReLU) of down_block / up_block (layers.py:237-238,252-255,278-279,293-296)
 *      x viewed as [M = N*H*W][C].  `sums` is a zeroed scratch of SVRS_BN_REPLICAS x double[2*C] (sum, sum of squares):
 *      the reduce kernels spread their atomics over the replicas (same-line double atomics serialise), every consumer
 *      (finalize, apply_train, bwd_apply) adds the replicas up. */
#define SVRS_BN_REPLICAS 8
int svrs_bn_stats(const void* x, int dtype, int64_t M, int C, double* sums, void* stream);
/* train: batch stats -> scale/shift (+ saved mean/invstd), running stats updated `n_updates` times
 * (SURVEY Q1: y_to_z runs twice per forward) and *num_batches_tracked += n_updates (may be NULL). */
int svrs_bn_finalize_train(const double* sums, int64_t M, int C, const float* gamma, const float* beta,
                           float eps, float momentum, float* running_mean, float* running_var,
                           int64_t* num_batches_tracked, int n_updates,
                           float* scale, float* shift, float* mean, float* invstd, void* stream);
/* train, fused: svrs_bn_finalize_train + svrs_bn_apply in one launch (same coefficients bit for bit; every block derives
 * them from `sums`, block 0 publishes scale/shift/mean/invstd and advances the running statistics).  C <= 1024.
 * M_stat (0 = M): number of rows the statistics in `sums` were taken over when it differs from the rows of THIS tensor -
 * sync_bn data parallelism all-reduces `sums` across ranks, so M_stat is then the global row count. */
int svrs_bn_apply_train(const void* x, void* y, int dtype, int64_t M, int64_t M_stat, int C, const double* sums,
                        const float* gamma, const float* beta, float eps, float momentum,
                        float* running_mean, float* running_var, int64_t* num_batches_tracked, int n_updates,
                        int relu, float* scale, float* shift, float* mean, float* invstd, void* stream);
/* eval: scale/shift from the running statistics */
int svrs_bn_finalize_eval(int C, const float* gamma, const float* beta, float eps,
                          const float* running_mean, const float* running_var,
                          float* scale, float* shift, void* stream);
/* y = relu?(x*scale[c] + shift[c]) ; in-place (y == x) allowed */
int svrs_bn_apply(const void* x, void* y, int dtype, int64_t M, int C, const float* scale,
                  const float* shift, int relu, void* stream);
/* backward of BN(train)+ReLU.  x = pre-BN conv output, dy = grad wrt the block output.
 * pass 1: sums[0:C] = sum dy*mask, sums[C:2C] = sum dy*mask*xhat (double, zeroed by caller) */
int svrs_bn_bwd_reduce(const void* x, const void* dy, int dtype, int64_t M, int C, const float* scale,
                       const float* shift, const float* mean, const float* invstd, int relu,
                       double* sums, void* stream);
/* pass 2: dx = gamma*invstd*(dym - mean(dym) - xhat*mean(dym*xhat)); dgamma += sums[C:], dbeta += sums[:C] */
int svrs_bn_bwd_apply(const void* x, const void* dy, void* dx, int dtype, int64_t M, int64_t M_stat, int C,
                      const float* scale, const float* shift, const float* mean, const float* invstd,
                      const float* gamma, int relu, const double* sums, float* dgamma, float* dbeta,
                      void* stream);

/* ---- reparameterize (cond_vae.py:261-265, vae.py:94-98) on the NCHW-flat encoder output
 *      enc [B][2*Wd] fp32 (mu = enc[:, :Wd], logvar = enc[:, Wd:], torch.chunk cond_vae.py:254,259).
 *      z[b][j] = mu + eps*exp(0.5*logvar).  eps: injected tensor [B][Wd] (eps != NULL) or on-device
 *      Philox4x32-10 keyed by (seed, stream_id, sample_offset+b, j).  eps_out (may be NULL) receives the
 *      draws.  Backward: denc[:, :Wd] += dz ; denc[:, Wd:] += dz*eps*0.5*std  (eps regenerated). */
int svrs_reparam_fwd(const float* enc, const float* eps, float* z, int64_t z_ld, float* eps_out, int B, int Wd,
                     uint64_t seed, uint32_t stream_id, uint64_t sample_offset, const int64_t* step_ptr,
                     void* stream);
int svrs_reparam_bwd(const float* enc, const float* eps, const float* dz, int64_t dz_ld, float* denc, int B, int Wd,
                     uint64_t seed, uint32_t stream_id, uint64_t sample_offset, const int64_t* step_ptr,
                     void* stream);
/* test hook: n standard normals from the same generator convention (row b = i / Wd, col = i % Wd).
 * step_ptr (device, may be NULL => 0) supplies Philox counter word 3 so a captured CUDA graph draws fresh
 * noise every replay; z_ld / dz_ld are row strides (elements) so z can live inside a torch.cat buffer. */
int svrs_philox_normal(float* out, int B, int Wd, uint64_t seed, uint32_t stream_id,
                       uint64_t sample_offset, const int64_t* step_ptr, void* stream);

/* ---- Gaussian ELBO terms: loss/cond_vae_loss.py:39-58 and loss/vae_loss.py:8-13.
 * A term set is described by up to two NLL pairs, one KL-to-N(0,I) and one KL(q2||p3):
 *   nll k:  ssq_k = sum (recon_k - target_k)^2 over n_k elements (any common layout, dtype given)
 *   kl1  :  sum_b sum_j (mu1^2 + exp(lv1) - 1 - lv1)              rows of width W1, row stride ld1
 *   kl23 :  sum (lv3 - lv2 - 1) + exp(lv2 - lv3) + (mu2-mu3)^2 exp(-lv3)   width W2, strides ld2/ld3
 * fwd accumulates the four raw sums in double acc[4] = {ssq_x, ssq_y, kl1, kl23} (zeroed by caller);
 * finalize turns them into the reference's terms out[5] = {mse_x, kld_u, mse_y, kld_z, their sum} (fp32):
 *   mse = ssq/(2 g^2) + n log g ;  kld = 0.5 * sum / B.   Unused pieces: pass NULL / n = 0.
 * dt_x / dt_y are the dtypes of the reconstructions, dt_tx / dt_ty those of the targets (the fused step keeps the
 * targets in fp32 NHWC next to the bf16 conv operands; any layout works as long as recon and target share it).
 * Requirements (else SVRS_E_ARG, nothing enqueued): every pointer 16-byte aligned; with mu1 given, lv1 too, W1 > 0 and
 * ld1 >= W1; with mu2 given, lv2 / mu3 / lv3 too, W2 > 0 and ld2, ld3 >= W2; all widths and strides multiples of 4. */
int svrs_elbo_fwd(const void* recon_x, const void* x, int dt_x, int dt_tx, int64_t n_x,
                  const void* recon_y, const void* y, int dt_y, int dt_ty, int64_t n_y,
                  const float* mu1, const float* lv1, int64_t ld1, int W1,
                  const float* mu2, const float* lv2, int64_t ld2,
                  const float* mu3, const float* lv3, int64_t ld3, int W2,
                  int B, double* acc, void* stream);
int svrs_elbo_finalize(const double* acc, int64_t n_x, int64_t n_y, int B, const float* gammas /*[2] x,y*/,
                       float* out5, void* stream);
/* backward.  gout[4] = upstream grads of {mse_x, kld_u, mse_y, kld_z} (device).  Any output may be NULL.
 * d_recon = g*(r - t)/gamma^2 ; d_gamma[k] = g*(-ssq/gamma^3 + n/gamma)
 * d_mu1 = g*mu1/B ; d_lv1 = g*0.5*(exp(lv1)-1)/B
 * d_mu2 = g*(mu2-mu3)exp(-lv3)/B = -d_mu3 ; d_lv2 = g*0.5*(exp(lv2-lv3)-1)/B
 * d_lv3 = g*0.5*(1 - exp(lv2-lv3) - (mu2-mu3)^2 exp(-lv3))/B
 * latent grads are written with their own row strides dld1/dld2/dld3: multiples of 4, and >= W1 / W2 / W2 whenever an
 * output of that pair is given; the input requirements of svrs_elbo_fwd apply.
 * dt_dx / dt_dy: dtype of d_recon_x / d_recon_y.  act = SVRS_ACT_SIGMOID: the reconstructions are sigmoid outputs and
 * d_recon_* receives the gradient wrt the PRE-activation, d * r * (1 - r) (nn.Sigmoid backward folded in); else SVRS_ACT_NONE. */
int svrs_elbo_bwd(const void* recon_x, const void* x, int dt_x, int dt_tx, int64_t n_x, void* d_recon_x, int dt_dx,
                  const void* recon_y, const void* y, int dt_y, int dt_ty, int64_t n_y, void* d_recon_y, int dt_dy,
                  const float* mu1, const float* lv1, int64_t ld1, int W1, float* d_mu1, float* d_lv1, int64_t dld1,
                  const float* mu2, const float* lv2, int64_t ld2, float* d_mu2, float* d_lv2, int64_t dld2,
                  const float* mu3, const float* lv3, int64_t ld3, int W2, float* d_mu3, float* d_lv3, int64_t dld3,
                  int B, const double* acc, const float* gammas, const float* gout, float* d_gammas,
                  int act, void* stream);

/* ---- clip_grad_norm_(params, 1.0) + torch.optim.Adam (models/base.py:106-107, train.py:65) on flat buffers */
int svrs_sumsq(const float* g, int64_t n, double* acc /* += */, void* stream);
/* step_ptr: device int64 holding the 1-based step number t (bias corrections 1-b^t computed on device).
 * sumsq == NULL => no clipping (the gamma param group, SURVEY Q3).
 * coef = min(1, max_norm/(sqrt(*sumsq)+1e-6)); g is NOT modified; p,m,v updated in place.
 * grad_scale multiplies g first (1/world_size after a SUM all-reduce). */
int svrs_clip_adam(float* p, const float* g, float* m, float* v, int64_t n, const double* sumsq,
                   float max_norm, float grad_scale, float lr, float beta1, float beta2, float eps,
                   const int64_t* step_ptr, void* stream);
int svrs_step_increment(int64_t* step_ptr, void* stream);
/* first launch of a fused step: ++*step_ptr and *norm_acc = 0 (the svrs_sumsq accumulator) in one kernel - a memset node
 * between kernel nodes of a captured graph costs a ~15 us bubble (CUPTI timeline, profiles/timeline_r02.txt) */
int svrs_step_begin(int64_t* step_ptr, double* norm_acc, void* stream);
/* The optimiser tail of the fused step in ONE launch (csrc/optim.cu adam_multi_kernel): for every conv / convT weight the
 * gradient is read in the layout the wgrad kernel left it in (see svrs_conv2d_wgrad_layout), clip + Adam run on the
 * torch-layout fp32 master weight and moments, and the updated weight is written into both compute-dtype packs
 * ([kk][d0][d1] and [kk][d1][d0], see svrs_pack_weights) - replacing svrs_unpack_grads_multi + svrs_clip_adam +
 * svrs_pack_weights_multi.  `jobs`: DEVICE array of njobs records (svrs_adam_job_bytes() each)
 *   { int64 off; void* p01; void* p10; int d0, d1, kk; int layout; int tile0; int tiles_b; }
 * off = element offset of the parameter in the flat buffers p / g / m / v.  Conv jobs (d1 > 0) are cut into tiles of
 * svrs_adam_tile_rows() x svrs_adam_tile_cols(kk) (16 x 16; 16 x 8 for kk > 9) of the (d0, d1) plane: tiles_b =
 * ceil(d1 / cols), a job has ceil(d0 / rows) * tiles_b tiles; plain jobs (d1 == 0: biases, BatchNorm affine) are cut into
 * runs of 2048 of their d0 elements.  tile0 = running sum of tile counts, total_tiles their total, max_kk <= 16, njobs <= 512.
 * sumsq / max_norm / grad_scale / step_ptr as in svrs_clip_adam.  Persistent CTAs walk the tile list; full tiles of kk = 9 / 16
 * layers with d0, d1 % 8 == 0 and 16-byte aligned buffers run through a bulk-copy pipeline (cp.async.bulk rows through shared
 * memory, SVRS_ADAM_BULK=0 disables it), everything else through a register-file path. */
int svrs_adam_job_bytes(void);
int svrs_adam_tile_rows(void);
int svrs_adam_tile_cols(int kk);
int svrs_adam_multi(const void* jobs, int njobs, int total_tiles, int max_kk, float* p, const float* g, float* m, float* v,
                    int pack_dtype, const double* sumsq, float max_norm, float grad_scale, float lr, float beta1,
                    float beta2, float eps, const int64_t* step_ptr, void* stream);

/* ---- grid patching + per-patch per-channel min-max normalisation
 *      (dataset.py:220-247,265-274 ; utils.py:4-23).  tiles [T][C][S][S] (fp32, or int16 when
 *      src_is_i16) -> patches [(T*(S/P)^2)][...], patch index = tile*(S/P)^2 + row*(S/P) + col.
 *      dst layout NCHW (nhwc=0) or NHWC (nhwc=1), dtype dst_dtype.  fp32 output is bit-exact with
 *      the reference: (x - min) / ((max - min) + 1e-5f). */
int svrs_grid_patch_normalize(const void* tiles, int src_is_i16, void* dst, int dst_dtype, int nhwc,
                              int T, int C, int S, int P, void* stream);

/* General form (TMA gather, csrc/patch.cu): one CTA per patch fetches the patch's C channel planes with ONE 3-D TMA box
 * into shared memory (tiles are read from HBM once), takes min/max there and emits up to three layouts from the staged
 * data: out_nchw_f32 [npatch][C][P][P] (the reference's layout), out_nhwc_f32 [npatch][P][P][C] (NLL target of the fused
 * step) and out_nhwc_bf16 (operand of the first conv layer); any may be NULL.  origins == NULL: grid mode as above;
 * otherwise a DEVICE array int32[npatch][3] = (tile, top, left): the reference's random crop (dataset.py:205-216:
 * LR at (top, left), HR at (2*top, 2*left)) with the draws made by the caller.  Needs S*elem and P*elem multiples of 16
 * bytes and 8 <= P <= 256. */
int svrs_patch_gather_normalize(const void* tiles, int src_is_i16, int T, int C, int S, int P,
                                const int32_t* origins, int npatch, float* out_nchw_f32, float* out_nhwc_f32,
                                void* out_nhwc_bf16, void* stream);

/* ---- inference: Cond_SRVAE.sample (cond_vae.py:299-318) + the uncertainty statistics of BaseVAE.task
 *      (models/base.py:305-313, 341) - BASELINE config 5, SURVEY 8.4 rows a14 / f4 (csrc/sample_stats.cu).
 * svrs_sample_latents: the S posterior-predictive draws of each of B patches,
 *      z(b, s) = mu3[b] + eps(b, s) * exp(0.5 * lv3[b])            (cond_vae.py:305-310)
 *   written together with y_to_z(y) as the decoder_x input rows (torch.cat((y_enc, z), dim=1), cond_vae.py:272):
 *      stack[(b*S + s)][0:Wz] = yflat[b][0:Wz] ; stack[(b*S + s)][Wz:2Wz] = z(b, s)        (fp32, NCHW-flat order)
 *   mu3 / lv3 rows have stride ld3, yflat rows stride ldy.  eps [B*S][Wz] fp32 or NULL = on-device Philox4x32-10 with the
 *   counter layout of svrs_reparam_fwd (row = sample_offset + b*S + s).  Requires Wz, ld3, ldy multiples of 4,
 *   ld3 >= Wz, ldy >= Wz and 16-byte aligned mu3 / lv3 / yflat / eps / stack (else SVRS_E_ARG, nothing enqueued). */
int svrs_sample_latents(const float* mu3, const float* lv3, int64_t ld3, const float* yflat, int64_t ldy,
                        const float* eps, float* stack, int B, int S, int Wz, uint64_t seed, int stream_id,
                        uint64_t sample_offset, const int64_t* step_ptr, void* stream);
/* svrs_sample_tail_stats: the LAST decoder_x layer (nn.Conv2d(16, 4, 3, padding=1) + nn.Sigmoid, cond_vae.py:79-80) over
 * the S draws of every patch, x [B*S][H][W][16] (dtype) -> x_hat(b, s) [4][H][W], with the per-pixel statistics of task()
 * accumulated while the draws are produced (streaming Welford over s; partial ranges of s merged with Chan's formula), so
 * the [S, 4, P, P] sample stack of models/base.py:303 never reaches HBM:
 *      mean_nchw [B][4][H][W] = samples.mean(dim=0)                                   (base.py:307)
 *      std_map   [B][H][W]    = samples.std(dim=0).mean(axis=0)   (unbiased)          (base.py:308)
 *      mae_map   [B][H][W]    = (samples - target).abs().mean(dim=(0, 1))             (base.py:309)
 *      mse_map   [B][H][W]    = (samples - target).pow(2).mean(dim=(0, 1))            (base.py:310)
 *      bias_map  [B][H][W]    = (target - samples.mean(dim=0)).mean(dim=0)            (base.py:341)
 *      sample0_nchw [B][4][H][W] = samples[0]                                          (base.py:318)
 * w_kn = p10 pack [9][16][4] of the layer (dtype), bias fp32[4] or NULL, target_nhwc fp32 [B][H][W][4] or NULL (then only
 * mean / std / sample0 are produced).  Every output pointer may be NULL.  splits in [1, S] (svrs_sample_tail_splits gives
 * the default); scratch = svrs_sample_tail_scratch_floats(B, H, W, splits) floats.  x and target_nhwc must be 16-byte
 * aligned (else SVRS_E_ARG).  Returns SVRS_E_UNSUPPORTED unless (Cin, Cout) == (16, 4). */
int svrs_sample_tail_splits(int B, int S, int H, int W);
int64_t svrs_sample_tail_scratch_floats(int B, int H, int W, int splits);
int svrs_sample_tail_stats(const void* x, int dtype, const void* w_kn, const float* bias, const float* target_nhwc,
                           int B, int S, int H, int W, int Cin, int Cout, int splits, float* scratch,
                           float* mean_nchw, float* std_map, float* mae_map, float* mse_map, float* bias_map,
                           float* sample0_nchw, void* stream);

/* ---- SSIM metrics of evaluate(): Metrics/SSIM_LR, SSIM_HR, SSIM_SR of Cond_SRVAE (cond_vae.py:387-525) and Metrics/SSIM of
 *      VAE (vae.py:142-216), which the reference computes with
 *      skimage.metrics.structural_similarity(a, b, win_size=11, data_range=1.0, channel_axis=0)   (csrc/ssim.cu).
 * svrs_ssim: a, b fp32 NCHW contiguous [N][C][H][W]; out[n] (double) = that value for the pair (a[n], b[n]) with scikit-image's
 *      defaults (uniform win x win window, sample covariance win^2/(win^2-1), C1 = (0.01 R)^2, C2 = (0.03 R)^2, R = data_range):
 *      the mean of the SSIM map over the (H-win+1) x (W-win+1) interior positions of each plane, averaged over the C planes.
 *      win odd, 3 <= win <= min(H, W).  Shared-memory staging of full-width bands limits the width:
 *      4 * W * (2 * (15 + win) + 90) <= 227 KB, i.e. W <= 409 at win = 11.  N == 0 enqueues nothing.
 *      workspace: svrs_ssim_workspace_doubles(N, C, H, W, win) doubles (one partial per band of 16 output rows of a plane),
 *      no initialisation needed.  Two launches, no atomics: repeated calls give bitwise-identical results.
 * svrs_ssim_workspace_doubles returns -1 (with svrs_last_error) for arguments svrs_ssim rejects. */
int64_t svrs_ssim_workspace_doubles(int N, int C, int H, int W, int win);
int svrs_ssim(const float* a, const float* b, int N, int C, int H, int W, int win, float data_range, double* workspace,
              double* out, void* stream);

/* ---- backward of the fused epilogue activations from their OUTPUT y:
 *      sigmoid: dx = dy*y*(1-y) ; hardtanh(-7,7): dx = dy if -7 < y < 7 else 0.  In-place (dx == dy) allowed. */
int svrs_act_bwd(const void* y, const void* dy, void* dx, int dtype, int act, int64_t n, void* stream);

/* ---- strided row copy (torch.cat / torch.chunk along channels, cond_vae.py:244,272):
 *      dst[r*dst_ld + c] (+)= src[r*src_ld + c], r < rows, c < cols, with dtype conversion */
int svrs_copy2d(const void* src, int src_dtype, int64_t src_ld, void* dst, int dst_dtype, int64_t dst_ld,
                int64_t rows, int cols, int accumulate, void* stream);

/* ---- misc elementwise helpers used by the host runtime */
int svrs_fill_zero(void* p, int64_t bytes, void* stream);
int svrs_axpy_f32(float* y, const float* x, float a, int64_t n, void* stream); /* y += a*x */
int svrs_cast(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n, void* stream);

/* ---- host-only test hook: dump the multi-tap GEMM geometry of a conv form (no device work).
 *      form 0 conv3 fprop, 1 conv3 dgrad, 2 conv4s2 fprop (= convT dgrad), 3 convT4s2 fprop (= conv4s2 dgrad);
 *      H, W, Cr describe the tensor being READ, Cw the channels written.  See csrc/conv_simt.cu for the layout
 *      of `out`; returns the number of int64 written (<0 on error). */
int svrs_debug_tap_geometry(int form, int N, int H, int W, int Cr, int Cw, int64_t* out, int cap);

#ifdef __cplusplus
}
#endif
#endif /* SVRS_B200_H */
