/*
 * b200dm.h -- C ABI of libb200dm.so: the sm_100a kernels behind the reference's sampling path.
 *
 * The reference (aayush9400/3D-Condtional-Stable-Diffusion) has no FFI/plugin boundary of its own: the
 * path sits behind Keras layer calls that TensorFlow lowers to cuDNN/cuBLAS/Eigen ops.  Each entry
 * point below replaces the TF op call site(s) it cites (file:line in the reference tree) and is what
 * a binding for this path would bind (see INTEGRATION.md for the ctypes stub).
 *
 * Conventions
 *   - return 0 on success, negative B200DM_ERR_* otherwise; b200dm_last_error() gives the text
 *     (thread-local).
 *   - every data pointer is a DEVICE pointer owned by the caller (16-byte aligned, contiguous,
 *     channels-last N,D,H,W,C).  The library never allocates or frees caller-visible device memory,
 *     never synchronises, and enqueues on the caller's cudaStream_t (passed as void*).
 *   - dtype enums: B200DM_F32 / B200DM_BF16.
 *   - there is NO CPU fallback: on a machine without a B200-class GPU the compute calls fail.
 */
#ifndef B200DM_H
#define B200DM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200DM_VERSION 101

#define B200DM_OK 0
#define B200DM_ERR_INVALID (-1)
#define B200DM_ERR_CUDA (-2)
#define B200DM_ERR_UNSUPPORTED (-3)
#define B200DM_ERR_KERNEL_TIMEOUT (-4)

#define B200DM_F32 0
#define B200DM_BF16 1   /* "the library's 16-bit storage type": bf16 in libb200dm.so, IEEE fp16 in libb200dm_f16.so */

#define B200DM_ACT_NONE 0
#define B200DM_ACT_SILU 1
#define B200DM_ACT_RELU 2

int b200dm_version(void);
const char* b200dm_last_error(void);
/* "bf16" or "fp16": the 16-bit type this build stores activations and packed weights in (every B200DM_BF16 buffer).
 * The same sources are compiled twice; the reference computes in fp32 (conditional_dm3d.py has no mixed-precision
 * policy), so the fp16 build is the closer one (8x smaller storage rounding) and the bf16 build the range-safe one. */
const char* b200dm_storage_dtype(void);
/* number of SMs / compute capability of the current device (major*10+minor); <0 on error */
int b200dm_device_info(int* sm_count, int* cc);

/* ---------------------------------------------------------------------------------------------
 * K10  fused reverse-diffusion update.  Replaces DiffusionModel.sample + the loop body of
 * DiffusionModel.generate (networks/dm3d.py:477-508, 516-530; conditional_dm3d.py:517-548, 559-573):
 * seven table gathers, x0, posterior mean, variance, clip(mean,-1,1), mean + sqrt(max(var,1e-20))*noise,
 * and the tf.random.normal op, as ONE elementwise pass.  Noise is read from `noise` when given,
 * else generated in-register from Philox4x32-10 (key=seed, counter=(elem/4, t, sample_id0+b, 0)).
 * sampler 1 = deterministic DDIM (extension; SURVEY F6).
 * --------------------------------------------------------------------------------------------- */
typedef struct {
  int64_t n_per_sample;            /* S^3 * C */
  int32_t batch;
  int32_t sampler;                 /* 0 = DDPM ancestral (reference), 1 = DDIM eta=0 (extension) */
  const float* beta;               /* device fp32[T] tables == reference Betas (dm3d.py:194-214) */
  const float* sqrt_alpha;
  const float* alpha_bar;
  const float* alpha_bar_prev;
  const float* sqrt_alpha_bar;
  const float* sqrt_alpha_bar_prev;
  const float* sqrt_one_minus_alpha_bar;
  const int32_t* t_dev;            /* device int32[2] = {t, t_prev}; if NULL use t / t_prev below.  With reserved bit 0 set it is
                                    * int32[8] = {t, t_prev, idx, -, seed lo, seed hi, sample base lo, sample base hi} */
  int32_t t;
  int32_t t_prev;                  /* DDIM only: next (smaller) timestep, -1 for the last step */
  uint64_t seed;
  int64_t sample_id0;              /* global index of sample 0 of this batch (multi-GPU sharding) */
  int32_t eps_dtype;               /* dtype of eps */
  int32_t reserved;                /* bit 0: Philox key = t_dev[4..5], sample index = t_dev[6..7] + sample_id0 + b (device-resident:
                                    * one captured step graph serves every seed and every shard) */
} b200dm_update_desc;

int b200dm_ddpm_update(const b200dm_update_desc* d, const float* x_t, const void* eps,
                       const float* noise_or_null, float* x_prev, void* x_prev_bf16_or_null,
                       void* stream);
/* x ~ N(0,1) from the same Philox stream family (stream id 1): replaces tf.random.normal(shape)
 * for x_T (dm3d.py:513). */
int b200dm_philox_normal(float* x, void* x_bf16_or_null, int64_t n_per_sample, int32_t batch,
                         uint64_t seed, int64_t sample_id0, int32_t step, int32_t stream_id,
                         void* stream);
/* t_dev[0] += delta (and t_dev[1] += delta): lets a captured CUDA graph walk the schedule. */
int b200dm_step_advance(int32_t* t_dev, int32_t delta, void* stream);
/* t_dev = {t, t_prev, idx, -}: idx += 1; t = seq[idx]; t_prev = seq[idx + 1] (seq is a device array terminated by two -1
 * entries).  One captured step graph then replays any timestep sequence: range(T-1, last_step-1, -1) of generate()
 * (dm3d.py:516), a strided / non-uniform DDIM schedule, ... with no host work between steps. */
int b200dm_step_advance_seq(int32_t* t_dev, const int32_t* seq, void* stream);
/* out[r][:] = table[idx[r]][:], fp32: the per-sample rows of the hoisted time-embedding tables when network([x, t]) is called
 * with distinct t per sample (train_step, conditional_dm3d.py:474,493) */
int b200dm_gather_rows_f32(const float* table, int32_t table_rows, const int32_t* idx, float* out, int32_t rows, int32_t cols,
                           void* stream);
/* Forward diffusion of train_step (conditional_dm3d.py:481-490): x_t = sqrt_alpha_bar[t[b]] * z + sqrt_one_minus_alpha_bar[t[b]]
 * * noise in the reference's fp32 op order, t device int32[batch].  noise_or_null NULL: Philox4x32-10 stream 2, counter
 * (element/4, 0, sample_id0 + b, 2) (streams 0 / 1 are the sampler's).  Writes x_t as the 16-bit network input and, when
 * x_t32_or_null is given, as fp32. */
int b200dm_q_sample(const float* z, const float* sqrt_alpha_bar, const float* sqrt_one_minus_alpha_bar, const int32_t* t,
                    const float* noise_or_null, int64_t n_per_sample, int32_t batch, uint64_t seed, int64_t sample_id0,
                    void* x_t16, float* x_t32_or_null, void* stream);
/* train_step's loss (conditional_dm3d.py:496-499): MSE(reduction=SUM)(noise, eps_hat) / divisor = sum over (B,D,H,W) of the
 * mean over `channels` of (noise - eps_hat)^2, / divisor -> loss fp32[1] (device).  The noise is regenerated from
 * b200dm_q_sample's stream with the same seed / sample_id0, or read from noise_or_null.  Fixed reduction order: bit-reproducible. */
size_t b200dm_noise_loss_workspace(int32_t batch);
int b200dm_noise_loss(const float* eps_hat, const float* noise_or_null, int64_t n_per_sample, int32_t batch, int32_t channels,
                      double divisor, uint64_t seed, int64_t sample_id0, float* loss, void* workspace, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K6/K7  fused normalisation + activation (+ channel concat, + per-voxel PReLU) in one HBM pass.
 * Replaces BatchNormalization(inference)+swish (dm3d.py:235-236, 243-244, 371-372), the BN of the
 * attention blocks (dm3d.py:46; conditional_dm3d.py:188), GroupNormalization+SiLU
 * (vqgan_attn_cp.py:258,262,269-274,382-383; vqgan_gnorm.py:268-271) and layers.Concatenate
 * (dm3d.py:359) when two sources are given.
 *   kind 0: y = act(x * scale[c] + shift[c])             scale/shift fp32[C]   (BN folded by caller
 *           from gamma,beta,moving_mean,moving_var, eps=1e-3 -- b200dm_bn_fold)
 *   kind 1: y = act((x - mean[n,g]) * rstd[n,g] * gamma[c] + beta[c])   stats from b200dm_gn_stats
 * --------------------------------------------------------------------------------------------- */
typedef struct {
  int64_t voxels;                  /* D*H*W per sample */
  int32_t batch;
  int32_t c0, c1;                  /* channels of source 0 and (optional) source 1; C = c0+c1 */
  int32_t kind;                    /* 0 affine (BN inference), 1 group norm */
  int32_t groups;                  /* kind 1 */
  int32_t act;                     /* B200DM_ACT_* */
  int32_t x_dtype, y_dtype;
} b200dm_norm_desc;

int b200dm_bn_fold(const float* gamma, const float* beta, const float* mean, const float* var,
                   float eps, int32_t c, float* scale, float* shift, void* stream);
int b200dm_gn_stats(const b200dm_norm_desc* d, const void* x, float eps, float* mean_rstd /* [B][G][2] */,
                    float* workspace, size_t ws_bytes, void* stream);
size_t b200dm_gn_stats_workspace(const b200dm_norm_desc* d);
/* BatchNormalization with the statistics of the batch (training=True): x (rows = B*D*H*W, c) 16-bit, per-channel mean and
 * biased variance (tf.nn.moments) -> scale[c] = gamma[c] * rsqrt(var + eps), shift[c] = beta[c] - mean * scale: the
 * coefficients of b200dm_norm_act_fwd kind 0 and of b200dm_conv_plan_set_out_affine.  Deterministic two-pass reduction
 * (fixed-order fp64 combine of per-CTA partials; the second pass sums x - mean).  c in 8..512 with c/8 dividing 256. */
size_t b200dm_bn_stats_workspace(int32_t c);
int b200dm_bn_stats(const void* x, int64_t rows, int32_t c, const float* gamma, const float* beta, float eps, float* scale,
                    float* shift, float* workspace, size_t ws_bytes, void* stream);
int b200dm_norm_act_fwd(const b200dm_norm_desc* d, const void* x0, const void* x1_or_null,
                        const float* scale_or_gamma, const float* shift_or_beta,
                        const float* mean_rstd_or_null, void* y, void* stream);
/* Extended pass for the VQ-GAN decoder variants (vqgan.py:256-284,378-475; vqgan_gnorm.py:256-286,382-484;
 * vqgan_stride.py:256-286,376-480):
 *   y = post_act( residual + act( PReLU_alpha( norm(x) ) ) ),  x optionally read through a nearest x2 up-sampling
 * (layers.UpSampling3D(2)); norm = per-channel affine (kind 0) or GroupNorm with given (mean, rstd) (kind 1).
 * Replaces GroupNormalization -> PReLU -> Add -> ReLU and UpSampling3D -> GroupNormalization -> PReLU.
 * alpha (out voxels, C) bf16 (Keras PReLU: one alpha per (d,h,w,c)); residual / y (B, out voxels, C). */
typedef struct {
  int32_t batch, out_d, out_h, out_w, c;
  int32_t kind, groups;            /* 0 affine, 1 group norm */
  int32_t act, post_act;           /* B200DM_ACT_* */
  int32_t upsample;                /* 1: x has spatial size out/2 */
  int32_t x_dtype, y_dtype;
} b200dm_norm_ex_desc;
int b200dm_norm_act_ex(const b200dm_norm_ex_desc* d, const void* x, const float* scale_or_gamma, const float* shift_or_beta,
                       const float* mean_rstd_or_null, const void* prelu_alpha_or_null, const void* residual_or_null,
                       void* y, void* stream);
/* whole-sample mean / rstd of an fp32 tensor (GroupNormalization with one group over the 1-2 channel network output,
 * vqgan_gnorm.py:460-461): mean_rstd fp32[B][2]; deterministic two-stage reduction, fp64 combine */
size_t b200dm_stats_f32_workspace(int32_t batch);
int b200dm_stats_f32(const float* x, int32_t batch, int64_t per_sample, float eps, float* mean_rstd, void* workspace,
                     size_t ws_bytes, void* stream);

/* LayerNormalization(axis=-1, eps) with up to 3 (gamma,beta) sets applied to ONE read of x:
 * CrossAttentionBlock.norm1/2/3 (conditional_dm3d.py:125-127,191-193).  x,y bf16 (rows, C). */
int b200dm_layernorm_fwd(const void* x, int64_t rows, int32_t c, float eps, int32_t n_out,
                         const float* const* gammas, const float* const* betas, void* const* ys,
                         void* stream);
/* dtype conversion fp32 <-> bf16 (n elements) */
int b200dm_cast(const void* x, int32_t x_dtype, void* y, int32_t y_dtype, int64_t n, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K11  VQ nearest-code search + gather.  Replaces VectorQuantizer.get_code_indices + the lookup
 * in VectorQuantizer.call (networks/vqvae3d_monai.py:165-177,139-144; vqgan_attn_cp.py:189-201,215).
 * d = ||x||^2 + ||e||^2 - 2 x.e, argmin with lowest index on ties; codebook (K,D) row-major
 * ("KD" layout; the caller transposes a (D,K) reference codebook once at load).
 * idx int64[N]; q (N,D) fp32 or bf16 (optional); hist int32[K] += bincount (optional;
 * == codebooks_used.assign_add, vqvae3d_monai.py:161).
 * --------------------------------------------------------------------------------------------- */
typedef struct {
  int64_t n;                       /* rows */
  int32_t d;                       /* embedding dim (multiple of 4, <= 1024) */
  int32_t k;                       /* codes */
  int32_t x_dtype;                 /* B200DM_F32 or B200DM_BF16 */
  int32_t q_dtype;
} b200dm_vq_desc;
int b200dm_vq_argmin_gather(const b200dm_vq_desc* d, const void* x, const float* codebook_kd,
                            const float* code_sqnorm /* fp32[K] from b200dm_vq_prepare */,
                            int64_t* idx, void* q_or_null, int32_t* hist_or_null, void* stream);
int b200dm_vq_prepare(const float* codebook_kd, int32_t k, int32_t d, float* code_sqnorm, void* stream);
/* The same search with the N x K products on the tensor cores (tcgen05, fp16 hi/lo splits of x and E: candidate codes inside a
 * proven error margin of the minimum) and the reference's exact fp32 chain re-evaluated for the candidates only: indices, q and
 * hist are bit-identical to b200dm_vq_argmin_gather.  Shapes: k % 128 == 0, d in {64,128,192,256} (workspace_bytes == 0
 * otherwise: use the call above).  tc_ws: caller-owned, 128-byte aligned, filled once per codebook by b200dm_vq_prepare_tc.
 * stats (optional, uint64[3] += rows rechecked, candidates rechecked, rows scanned in full). */
size_t b200dm_vq_tc_workspace_bytes(int32_t k, int32_t d);
int b200dm_vq_prepare_tc(const float* codebook_kd, const float* code_sqnorm, int32_t k, int32_t d, void* tc_ws, void* stream);
int b200dm_vq_argmin_gather_tc(const b200dm_vq_desc* d, const void* x, const float* codebook_kd, const float* code_sqnorm,
                               const void* tc_ws, int64_t* idx, void* q_or_null, int32_t* hist_or_null, uint64_t* stats_or_null,
                               void* stream);
/* get_code_indices(flat, distribution=True) (vqvae3d_monai.py:165-177): the (N,K) fp32 matrix of squared distances, same
 * arithmetic as the argmin kernel (row-wise argmin of it == idx). */
int b200dm_vq_distances(const b200dm_vq_desc* d, const void* x, const float* codebook_kd, const float* code_sqnorm,
                        float* dist, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K12  small fp32 dense: Y = act(X W + b), X (M,K), W (K,N) Keras layout.  Replaces the Dense layers on the
 * time / context embeddings (dm3d.py:229-232, 280-288; conditional_dm3d.py:310-318): step-invariant,
 * evaluated once per schedule (all T rows) or per generate() call, never per step.
 * --------------------------------------------------------------------------------------------- */
int b200dm_dense_f32(const float* x, const float* w, const float* b_or_null, float* y,
                     int32_t m, int32_t k, int64_t n, int32_t act_in, int32_t act_out, void* stream);

/* row softmax over fp32 scores -> bf16 probabilities (tf.nn.softmax(attn_score,-1), dm3d.py:56;
 * conditional_dm3d.py:178).  scores (rows, cols) fp32, scale applied before the softmax. */
int b200dm_softmax_rows(const float* s, void* p_bf16, int64_t rows, int32_t cols, float scale,
                        void* stream);

/* ---------------------------------------------------------------------------------------------
 * K1-K5, K8/K9 GEMMs  Conv3D as an implicit GEMM on tcgen05/TMEM with TMA-staged NDHWC bf16 tiles.
 * Replaces layers.Conv3D k=3 'same' (dm3d.py:237-239,246-248,318-323,373-375), stride-2 DownSample
 * (dm3d.py:257-263; TF 'same' pad (0,1)), UpSampling3D(2)+Conv3D (dm3d.py:271-274; folded into 8
 * parity sub-convolutions of 2^3 taps), Conv3D k=1 / Dense-on-voxels (dm3d.py:225-227,47-49,62;
 * conditional_dm3d.py:129-138), Conv3DTranspose k=4 s=2 'same' (vqvae3d_monai.py:372-377;
 * vqgan_attn_cp.py:398-403; the same 8-parity form) and, with a per-sample B operand, the two
 * attention matmuls (tf.einsum dm3d.py:51,61).
 *
 *   y[n, o, co] = epilogue( sum_{seg, tap, ci} x_seg[n, in(o,tap), ci] * W[parity(o)][co][seg,tap,ci] )
 *   epilogue: + bias[co] + chan_bias[t][n][co]; * PReLU/act; + residual[n,o,co]
 *
 * A plan owns the TMA descriptors for one fixed set of buffers; create once, run every step.
 * --------------------------------------------------------------------------------------------- */
#define B200DM_CONV_DIRECT 0   /* k^3 taps, stride 1 or 2, TF 'same' padding */
#define B200DM_CONV_PARITY 1   /* out = 2*in: 8 output parities x 2^3 taps (upsample+conv3 / convT k4 s2) */
#define B200DM_CONV_BATCHED_GEMM 2 /* per-sample B operand: y[n] = x[n] (rows,K) . w[n] (N,K)^T */

typedef struct {
  int32_t mode;
  int32_t batch, in_d, in_h, in_w;  /* input spatial size (GEMM mode: in_w = rows per sample, d=h=1) */
  int32_t c0, c1;                   /* channels of the two K-segments (c1 = 0: one source) */
  int32_t c_out;
  int32_t ksize;                    /* DIRECT: 1, 3 or 4 */
  int32_t stride;                   /* DIRECT: 1 or 2 */
  int32_t act;                      /* B200DM_ACT_* applied after bias adds, before the residual add */
  int32_t y_dtype;                  /* B200DM_BF16 or B200DM_F32 */
  int32_t chan_bias_rows;           /* rows in chan_bias per timestep (= batch) */
  int32_t use_halo;                 /* -1: per-tap GEMM kernel only; any other value: the kernel is chosen from the shape */
  int32_t reserved[4];
} b200dm_conv_desc;

typedef struct b200dm_conv_plan b200dm_conv_plan;

/* packed weight size (bytes) for a desc: bf16 [parities][n_pad][chunks*taps*64] */
size_t b200dm_conv_packed_weight_bytes(const b200dm_conv_desc* d);
/* host-side packer: Keras kernel fp32 (k,k,k,Cin,Cout) [or (k,k,k,Cout,Cin) when transposed!=0] ->
 * packed bf16 image (host pointers).  For PARITY mode with ksize 3 the 27 taps are pre-summed into
 * 8x8 (nearest-upsample fold); with ksize 4 (transposed conv) they are re-indexed. */
int b200dm_conv_pack_weights(const b200dm_conv_desc* d, const float* keras_kernel_host,
                             int32_t transposed, void* packed_host);
int b200dm_conv_plan_create(const b200dm_conv_desc* d, const void* x0, const void* x1_or_null,
                            const void* w_packed, const float* bias_or_null,
                            const float* chan_bias_or_null, const int32_t* t_dev_or_null,
                            const void* residual_or_null, const void* prelu_alpha_or_null,
                            void* y, b200dm_conv_plan** out);
int b200dm_conv_plan_run(b200dm_conv_plan* p, void* stream);
void b200dm_conv_plan_destroy(b200dm_conv_plan* p);
double b200dm_conv_plan_flops(const b200dm_conv_plan* p);
/* Fuse the CONSUMER's BatchNormalization (inference, folded by b200dm_bn_fold) into this conv's epilogue:
 * y = act(scale[co] * (acc + bias + chan_bias) + shift[co]), scale/shift device fp32[c_out].  Used for
 * ResidualBlock conv1 -> BN -> swish (dm3d.py:237-244) when the un-normalised tensor has no other reader.
 * NULL, NULL switches it off. */
int b200dm_conv_plan_set_out_affine(b200dm_conv_plan* p, const float* scale, const float* shift);
/* Fuse the reverse-diffusion update (b200dm_ddpm_update: DiffusionModel.sample + the loop body of generate, networks/dm3d.py:
 * 477-508, 516-530) into the epilogue of the U-Net's output conv (dm3d.py:373-374, the fp32 eps_hat): the conv then stores
 * x_{t-1} = step(x_t, eps_hat, Philox noise) to x_prev (fp32; must alias x_t: updated in place) and a copy in the 16-bit storage type to x_prev_16
 * (the next step's network input) INSTEAD of eps_hat -- same arithmetic, same noise stream, no fp32 eps round trip through
 * HBM and no separate update launch.  `u` is read as by b200dm_ddpm_update (tables, t_dev, seed, sample_id0, sampler; no injected
 * noise).  Returns B200DM_ERR_UNSUPPORTED unless the plan is the CTA-pair 3^3 conv with fp32 output and C_out % 128 == 0. */
int b200dm_conv_plan_set_fused_update(b200dm_conv_plan* p, const b200dm_update_desc* u, const float* x_t, float* x_prev, void* x_prev_16);
/* Fold a 1^3 conv of [x0 | x1] (c0 + c1 channels, the plan's input geometry: a ResidualBlock's shortcut) into
 * this 3^3 conv's K loop: y = epilogue(conv(x) + W_sc [x0 | x1] + bias), so the shortcut is never stored and read back.
 * w_packed: each of the plan's packed weight rows (b200dm_conv_pack_weights) followed by the same row of the 1^3 conv's packed
 * weights, zero-padded to a multiple of 3 k-blocks of 64 channels; bias: the combined bias (the two convs' biases summed).
 * Replaces the plan's weights and bias.  Returns B200DM_ERR_UNSUPPORTED unless the plan runs the halo-reuse 3^3 kernel
 * without the fused update. */
int b200dm_conv_plan_set_shortcut(b200dm_conv_plan* p, int32_t c0, int32_t c1, const void* x0, const void* x1, const void* w_packed,
                                  const float* bias);
/* which kernel / tile configuration the plan launches (profiling): halo 1 = persistent halo-reuse kernel */
int b200dm_conv_plan_info(const b200dm_conv_plan* p, int32_t* halo, int32_t* block_n, int32_t* ksplit);
/* GroupNorm statistics as a by-product of the producing conv (replaces a second read of the conv output by
 * tfa GroupNormalization's moments, vqgan_attn_cp.py:258-275): plans that support it (the d-sweeping C_in = C_out = 32 kernel)
 * accumulate per-(work item, channel) partial sums of the STORED values into `workspace` = double[batch * rows_per_sample][C][2]
 * (fp32 sums about a per-item pivot, rebuilt in fp64: exact enough when |mean| >> std);
 * b200dm_gn_finalize reduces them in a fixed order (bit-reproducible) to (mean, rstd) per (sample, group).
 * _bytes returns 0 when the plan cannot produce partials. */
size_t b200dm_conv_plan_gn_partials_bytes(const b200dm_conv_plan* plan, int32_t* rows_per_sample);
int b200dm_conv_plan_set_gn_partials(b200dm_conv_plan* plan, double* workspace, size_t ws_bytes);
int b200dm_gn_finalize(const double* partials, int32_t batch, int32_t rows_per_sample, int32_t c, int32_t groups,
                       int64_t voxels_per_sample, float eps, float* mean_rstd, void* stream);
/* tuning aid: device int64[4*2048] receiving CTA 0's per-role timeline ((clock64 << 8) | tag); NULL switches it off */
int b200dm_conv_plan_set_trace(b200dm_conv_plan* p, void* trace);
/* device-side watchdog flag: non-zero if any tcgen05/TMA pipeline wait timed out since last reset */
int b200dm_debug_flag_read_reset(int32_t* flag_out);

/* ---------------------------------------------------------------------------------------------
 * K8/K9  flattened-voxel attention as one flash-style tcgen05 kernel:  O = softmax(scale * Q K^T) V (+ residual).
 * Replaces the materialised (B,L,L) score path of AttentionBlock.call (networks/dm3d.py:51-61) and of
 * CrossAttentionBlock.attention (conditional_dm3d.py:162-184): einsum -> * units^-0.5 -> tf.nn.softmax -> einsum.
 * Single head (the reference's num_heads is always 1).  bf16 tensors, fp32 softmax statistics and accumulation:
 *   q (B, Lq, D)   k (B, Lk, D)   vt (B, D, Lk) = V transposed per sample (conv transposed-store epilogue)
 *   residual (B, Lq, D) or NULL   o (B, Lq, D);   D in {64, 128, 256};  Lk % 8 == 0.
 * --------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t batch, lq, lk, d;
  float scale;
  int32_t reserved[3];   /* [0], [1]: row strides (elements) of q / k when they are column blocks of one wider projection output
                          * (e.g. a fused [q | k] Dense); 0 = D (contiguous rows).  [2]: 0 */
} b200dm_attn_desc;
typedef struct b200dm_attn_plan b200dm_attn_plan;
int b200dm_attention_plan_create(const b200dm_attn_desc* d, const void* q, const void* k, const void* vt,
                                 const void* residual_or_null, void* o, b200dm_attn_plan** out);
int b200dm_attention_plan_run(b200dm_attn_plan* p, void* stream);
void b200dm_attention_plan_destroy(b200dm_attn_plan* p);
double b200dm_attention_plan_flops(const b200dm_attn_plan* p);

/* ---------------------------------------------------------------------------------------------
 * Step program: an ordered list of the above ops with fixed buffers, launched natively in one
 * call (one ctypes crossing per U-Net forward instead of ~250), CUDA-graph capturable.
 * Every op is checked and sized when it is recorded: add_X returns the code and b200dm_last_error() text that the
 * direct entry point X returns for the same arguments, and records nothing on error (add_conv / add_attention take
 * the plan only on success).  run / run_timed replay the recorded launches and fail only on a CUDA error.
 * --------------------------------------------------------------------------------------------- */
typedef struct b200dm_program b200dm_program;
int b200dm_program_create(b200dm_program** out);
void b200dm_program_destroy(b200dm_program* p);
int b200dm_program_add_conv(b200dm_program* p, b200dm_conv_plan* plan /* ownership moves */);
int b200dm_program_add_norm_act(b200dm_program* p, const b200dm_norm_desc* d, const void* x0,
                                const void* x1_or_null, const float* a, const float* b,
                                const float* mean_rstd_or_null, void* y);
int b200dm_program_add_bn_stats(b200dm_program* p, const void* x, int64_t rows, int32_t c, const float* gamma, const float* beta,
                                float eps, float* scale, float* shift, float* workspace, size_t ws_bytes);
int b200dm_program_add_gn_stats(b200dm_program* p, const b200dm_norm_desc* d, const void* x, float eps,
                                float* mean_rstd, float* workspace, size_t ws_bytes);
int b200dm_program_add_gn_finalize(b200dm_program* p, const double* partials, int32_t batch, int32_t rows_per_sample, int32_t c,
                                   int32_t groups, int64_t voxels_per_sample, float eps, float* mean_rstd);
int b200dm_program_add_layernorm(b200dm_program* p, const void* x, int64_t rows, int32_t c, float eps,
                                 int32_t n_out, const float* const* gammas, const float* const* betas,
                                 void* const* ys);
int b200dm_program_add_norm_act_ex(b200dm_program* p, const b200dm_norm_ex_desc* d, const void* x, const float* a, const float* b,
                                   const float* mean_rstd_or_null, const void* prelu_alpha_or_null,
                                   const void* residual_or_null, void* y);
int b200dm_program_add_stats_f32(b200dm_program* p, const float* x, int32_t batch, int64_t per_sample, float eps,
                                 float* mean_rstd, void* workspace, size_t ws_bytes);
int b200dm_program_add_attention(b200dm_program* p, b200dm_attn_plan* plan /* ownership moves */);
int b200dm_program_add_softmax(b200dm_program* p, const float* s, void* p_bf16, int64_t rows,
                               int32_t cols, float scale);
int b200dm_program_add_update(b200dm_program* p, const b200dm_update_desc* d, const float* x_t,
                              const void* eps, const float* noise_or_null, float* x_prev,
                              void* x_prev_bf16_or_null);
int b200dm_program_add_step_advance(b200dm_program* p, int32_t* t_dev, int32_t delta);
/* Lanes: ops added after set_lane(l) run on lane l (0 = the caller's stream, 1..9 = streams owned by the program);
 * add_sync(a, b) makes everything recorded so far on lane a a prerequisite of what follows on lane b (event record /
 * wait: a fork when a = 0, a join when b = 0).  Every side lane must be joined back to lane 0 before the program ends.
 * Used for the three independent branches of CrossAttentionBlock.call (conditional_dm3d.py:190-192). */
int b200dm_program_set_lane(b200dm_program* p, int32_t lane);
int b200dm_program_add_sync(b200dm_program* p, int32_t from_lane, int32_t to_lane);
int b200dm_program_run(b200dm_program* p, void* stream);
int b200dm_program_num_launches(const b200dm_program* p);
int b200dm_program_num_ops(const b200dm_program* p);
/* profiling aid: same launches with a CUDA-event pair around every op; synchronises the stream */
int b200dm_program_run_timed(b200dm_program* p, void* stream, float* ms_per_op, int32_t n_ops);

#ifdef __cplusplus
}
#endif
#endif /* B200DM_H */
