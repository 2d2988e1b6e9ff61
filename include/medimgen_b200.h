/*
 * medimgen_b200.h -- C ABI of the B200-native medimgen hot path (libmedimgen_b200.so).
 *
 * The reference (VKostoulas/Medical_Image_Generation, `medimgen`) has no FFI of its own: it is pure
 * Python that dispatches to cuDNN/cuBLAS/ATen (SURVEY.md section 2.3). Each entry point below replaces
 * one of those library dispatch sites; the site is cited as `unet:N` =
 * medimgen/diffusion_model_unet_with_strides.py:N, `ae:N` = medimgen/autoencoderkl_with_strides.py:N,
 * `ldm:N` = medimgen/train_ldm.py:N, `aetrain:N` = medimgen/train_autoencoder.py:N.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; no torch types cross the ABI
 *   - activations are channels-last: [N][D][H][W][C] (2-D problems use D = 1)
 *   - conv filters are [Cout][kd][kh][kw][Cin] (== torch channels_last_3d of (Cout,Cin,kd,kh,kw))
 *   - dtype codes: MIG_F32 = 0, MIG_BF16 = 1
 *   - `stream` is a cudaStream_t passed as void*
 *   - return value 0 = ok; otherwise mig_last_error() describes the failure (thread-local)
 *   - no allocation, no hidden global state except a per-device attribute cache
 */
#ifndef MEDIMGEN_B200_H
#define MEDIMGEN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MIG_F32 0
#define MIG_BF16 1

#define MIG_ABI_VERSION 4

/* Geometry of one N-d convolution (1 <= nd <= 3 handled by setting leading dims to 1). */
typedef struct {
  int32_t N;          /* batch */
  int32_t in_dims[3]; /* D,H,W of the conv input  */
  int32_t out_dims[3];/* D,H,W of the conv output */
  int32_t Cin, Cout;
  int32_t ksize[3], stride[3], pad[3];
} mig_conv_geom;

const char* mig_last_error(void);
int mig_abi_version(void);
/* 1 when the running device is sm_100 and the tcgen05 kernels are usable */
int mig_has_tcgen05(void);

/* mig_conv_fwd that ALSO delivers the GroupNorm statistics of its output (north_star: "GroupNorm statistics ... fused
 * into the ... epilogue"): gn_sums[n][g][2] (fp64) = (sum y, sum y^2) per (sample, group) of the bf16-rounded result,
 * consumed by mig_groupnorm_apply for the GroupNorm that follows the convolution (unet:648 after conv1, unet:628 of the
 * next block after conv2, ae:167). Accumulated by the tcgen05 kernel's epilogue (warp-shuffle reduction of the fp32
 * tile, fp64 red.global per (CTA, group)); plans whose epilogue only sees partial sums (split-K) and the other engines
 * run one statistics pass over y instead. Needs mig_groupnorm_can_split(dtype, N, out voxels, Cout, gn_groups). */
int mig_conv_fwd_stats(const mig_conv_geom* g, int dtype, const void* x, const void* w, const float* bias,
                       const float* chan_bias, const void* residual, void* y, double* gn_sums, int32_t gn_groups,
                       int engine, void* workspace, int64_t workspace_bytes, void* stream);
/* 1 when mig_conv_fwd_stats takes the statistics from the tcgen05 epilogue for this geometry and workspace size
 * (0: it runs the statistics pass over y) */
int mig_conv_fwd_stats_in_epilogue(const mig_conv_geom* g, int dtype, int32_t gn_groups, int engine,
                                   int64_t workspace_bytes);

/* ---- K1/K2/K3: Conv{2,3}d as implicit GEMM -------------------------------------------------------
 * replaces nn.Conv{2,3}d inside monai Convolution: unet:510-518,557-565,630-659,664,1820,1935;
 * ae:66-129,158-179,372-381,454-463,523-532,606-615,723-749.
 * y[n,o,co] = sum_{tap,ci} x[n, o*stride - pad + tap, ci] * w[co,tap,ci] + bias[co]
 *             (+ chan_bias[n,co]  -- the time-embedding add, unet:691-695; N x Cout fp32 -- a single embedding shared by
 *                the whole batch, as the inferers' one-timestep calls produce, must be replicated to N rows by the caller)
 *             (+ residual[n,o,co] -- the skip add, unet:701 / ae:204)
 * `engine`: 0 = auto, 1 = SIMT fp32-accumulate CUDA-core path, 2 = tcgen05 tensor-core path (bf16 only). */
int mig_conv_fwd(const mig_conv_geom* g, int dtype, const void* x, const void* w, const float* bias,
                 const float* chan_bias, const void* residual, void* y, int engine,
                 void* workspace, int64_t workspace_bytes, void* stream);
/* dx[n,i,ci] = sum_{tap,co} dy[n,(i+pad-tap)/stride,co] * w[co,tap,ci]   (conv backward-data) */
int mig_conv_dgrad(const mig_conv_geom* g, int dtype, const void* dy, const void* w, void* dx, int engine,
                   void* workspace, int64_t workspace_bytes, void* stream);
/* dw[co,tap,ci] += sum_{n,o} dy[n,o,co] * x[n,o*stride-pad+tap,ci]  (fp32, accumulates into dw);
 * dbias[co] += sum dy[.,co] when dbias != NULL */
int mig_conv_wgrad(const mig_conv_geom* g, int dtype, const void* x, const void* dy, float* dw, float* dbias,
                   int engine, void* workspace, int64_t workspace_bytes, void* stream);
int64_t mig_conv_workspace_bytes(const mig_conv_geom* g, int dtype, int which /*0 fwd,1 dgrad,2 wgrad*/, int engine);

/* ---- generic strided batched GEMM (attention products unet:406-416, ae:271-281) -------------------
 * C[b][m][n] = alpha * sum_k A[b][m][k] * B[b][k][n], element strides given; batch index b = bo*inner+bi
 * with offsets bo*s?_outer + bi*s?_inner (heads live inside the channel dim). */
typedef struct {
  int32_t M, N, K, batch_outer, batch_inner;
  int64_t a_m, a_k, a_outer, a_inner;
  int64_t b_k, b_n, b_outer, b_inner;
  int64_t c_m, c_n, c_outer, c_inner;
  float alpha;
  int32_t accumulate; /* C += ... (fp32 output only) */
} mig_gemm_desc;
int mig_gemm_strided(const mig_gemm_desc* d, int dtype_ab, int dtype_c, const void* A, const void* B, void* C,
                     int engine, void* stream);

/* Fused flash-style attention forward on tcgen05 (replaces xformers.ops.memory_efficient_attention unet:128-135,403
 * and the baddbmm/softmax/bmm chain unet:406-416 when no gradient is needed): out = softmax(scale * q k^T) v per
 * (batch, head). q (B,Lq,H*dh), k/v (B,Lk,H*dh), out (B,Lq,H*dh): contiguous bf16. lse: workspace of B*H*Lq floats
 * (receives the log2-domain log-sum-exp). dh must be a multiple of 64 (above 256: a multiple of 256). */
int mig_flash_attention_fwd(const void* q, const void* k, const void* v, void* out, float* lse, int32_t B, int32_t H,
                            int32_t Lq, int32_t Lk, int32_t dh, float scale, void* stream);
/* The same with q / k / v given as row-strided matrices: row pitch ldq / ldk / ldv in ELEMENTS (>= H*dh, a multiple of 8),
 * batch stride L * ld. This is how attention reads the three column blocks of ONE fused q/k/v projection output
 * (B, L, 3*H*dh) in place (unet:436-438 as one Linear). `out` stays contiguous (B, Lq, H*dh). */
int mig_flash_attention_fwd_ld(const void* q, const void* k, const void* v, void* out, float* lse, int32_t B, int32_t H,
                               int32_t Lq, int32_t Lk, int32_t dh, int64_t ldq, int64_t ldk, int64_t ldv, float scale,
                               void* stream);
/* Backward of the above without any L x L tensor (training path of unet:396-416): P is recomputed per tile from q, k and
 * the forward's `lse`; o / d_o are the forward output and its gradient; `delta` is a workspace of B*H*Lq floats
 * (receives rowsum(d_o * o)). dq (B,Lq,H*dh), dk / dv (B,Lk,H*dh): bf16, fully written. dh: a multiple of 64. Heads wider
 * than the tensor-memory accumulators (the LDM's 512 / 768-channel single heads) are processed in column slices. */
int mig_flash_attention_bwd(const void* q, const void* k, const void* v, const void* o, const void* d_o,
                            const float* lse, float* delta, void* dq, void* dk, void* dv, int32_t B, int32_t H,
                            int32_t Lq, int32_t Lk, int32_t dh, float scale, void* stream);

/* ---- K4/K5: GroupNorm (+SiLU), nn.GroupNorm at unet:628,648,275,377,1932; ae:157,167,238,451,604 ----
 * x,y: [N][S][C] channels-last, S = D*H*W. mean/rstd: [N][G] fp32 (saved for backward). */
int mig_groupnorm_fwd(int dtype, const void* x, const float* gamma, const float* beta, void* y,
                      float* mean, float* rstd, int32_t N, int64_t S, int32_t C, int32_t G, float eps,
                      int fuse_silu, void* workspace, int64_t workspace_bytes, void* stream);
/* dx_colsum (optional, [N][C] fp32): receives sum_s dx[n,s,c] -- the bias / time-embedding gradient of the convolution
 * that produced x (unet:691-695), so that convolution's backward needs no column-sum pass over dy.
 * dx_addend (optional, same shape/dtype as dx): dx = GroupNorm gradient + dx_addend -- the gradient that reaches x through
 * the block's skip path (unet:701: x also feeds the residual add), fused instead of a separate accumulation pass.
 * accumulate_dparams != 0: dgamma / dbeta are ADDED to (they point into the optimiser's flat gradient buffer). */
int mig_groupnorm_bwd(int dtype, const void* x, const void* dy, const float* gamma, const float* beta,
                      const float* mean, const float* rstd, void* dx, float* dgamma, float* dbeta, float* dx_colsum,
                      const void* dx_addend, int accumulate_dparams, int32_t N, int64_t S, int32_t C, int32_t G,
                      int fuse_silu, void* workspace, int64_t workspace_bytes, void* stream);
int64_t mig_groupnorm_workspace_bytes(int32_t N, int64_t S, int32_t C, int32_t G);
/* The two halves of the forward as separate entry points (bf16, C a multiple of 32: mig_groupnorm_can_split() == 1).
 * sums: double [N][G][2] = (sum x, sum x^2) per (sample, group) -- written by mig_groupnorm_stats, or accumulated by
 * the epilogue of the convolution that produced x (mig_conv_fwd_stats), which removes the statistics pass over x.
 * mig_groupnorm_apply derives mean / rstd from the sums itself and stores them ([N][G] fp32) for the backward pass. */
int mig_groupnorm_can_split(int dtype, int32_t N, int64_t S, int32_t C, int32_t G);
int mig_groupnorm_stats(int dtype, const void* x, double* sums, int32_t N, int64_t S, int32_t C, int32_t G,
                        void* stream);
int mig_groupnorm_apply(int dtype, const void* x, const float* gamma, const float* beta, const double* sums, void* y,
                        float* mean, float* rstd, int32_t N, int64_t S, int32_t C, int32_t G, float eps,
                        int fuse_silu, void* stream);

/* LayerNorm over the last dim (BasicTransformerBlock norm1-3, unet:225-227) */
int mig_layernorm_fwd(int dtype, const void* x, const float* gamma, const float* beta, void* y, float* mean,
                      float* rstd, int64_t rows, int32_t C, float eps, void* stream);
int mig_layernorm_bwd(int dtype, const void* x, const void* dy, const float* gamma, const float* mean,
                      const float* rstd, void* dx, float* dgamma, float* dbeta, int64_t rows, int32_t C,
                      void* stream);

/* ---- elementwise family ------------------------------------------------------------------------- */
int mig_silu_fwd(int dtype, const void* x, void* y, int64_t n, void* stream);            /* unet:677,1833 */
int mig_silu_bwd(int dtype, const void* x, const void* dy, void* dx, int64_t n, void* stream);
int mig_add(int dtype, const void* a, const void* b, void* y, int64_t n, void* stream);   /* residual adds */
int mig_scale(int dtype, const void* x, void* y, float s, int64_t n, void* stream);       /* ldm:157 */
int mig_mul(int dtype, const void* a, const void* b, void* y, int64_t n, void* stream);
/* y = a + b*c : the reparameterisation z = mu + eps*sigma (ae:786-787) */
int mig_addcmul(int dtype, const void* a, const void* b, const void* c, void* y, int64_t n, void* stream);
int mig_cast(int src_dtype, int dst_dtype, const void* x, void* y, int64_t n, void* stream);
/* GEGLU: y[r][j] = x[r][j] * gelu(x[r][H+j]) (monai MLPBlock, unet:213) */
int mig_geglu_fwd(int dtype, const void* x, void* y, int64_t rows, int32_t H, void* stream);
int mig_geglu_bwd(int dtype, const void* x, const void* dy, void* dx, int64_t rows, int32_t H, void* stream);
/* torch.cat along channels (unet:1263,1377,1504) and its split backward */
int mig_concat_channels(int dtype, const void* a, const void* b, void* y, int64_t rows, int32_t Ca, int32_t Cb,
                        void* stream);
int mig_split_channels(int dtype, const void* y, void* a, void* b, int64_t rows, int32_t Ca, int32_t Cb,
                       void* stream);
/* F.interpolate(mode="nearest", integer per-axis factors) unet:580, ae:99 and its sum-pool backward */
int mig_upsample_nearest_fwd(int dtype, const void* x, void* y, int32_t N, const int32_t in_dims[3],
                             const int32_t factors[3], int32_t C, void* stream);
int mig_upsample_nearest_bwd(int dtype, const void* dy, void* dx, int32_t N, const int32_t in_dims[3],
                             const int32_t factors[3], int32_t C, void* stream);
/* nn.AvgPool{2,3}d(kernel, stride) without padding: Downsample(use_conv=False) of ResnetBlock(down=True), unet:513-518,
 * 641-644 (resblock_updown=True). in_dims = pooled tensor's INPUT extent; out = (in - k) / s + 1 per axis. */
int mig_avgpool_fwd(int dtype, const void* x, void* y, int32_t N, const int32_t in_dims[3], const int32_t ksize[3],
                    const int32_t stride[3], int32_t C, void* stream);
int mig_avgpool_bwd(int dtype, const void* dy, void* dx, int32_t N, const int32_t in_dims[3], const int32_t ksize[3],
                    const int32_t stride[3], int32_t C, void* stream);
/* NCDHW <-> NDHWC with optional dtype change (module boundary) */
int mig_nchw_to_nhwc(int src_dtype, int dst_dtype, const void* x, void* y, int32_t N, int32_t C, int64_t S,
                     void* stream);
int mig_nhwc_to_nchw(int src_dtype, int dst_dtype, const void* x, void* y, int32_t N, int32_t C, int64_t S,
                     void* stream);
/* column sums of a [rows][C] matrix into fp32 out[C] (bias gradients); out += when accumulate */
int mig_colsum(int dtype, const void* x, float* out, int64_t rows, int32_t C, int accumulate, void* stream);
/* y[r][c] = x[r][c] + bias[c] (channels-last rows; in place allowed). Bias of nn.ConvTranspose{2,3}d inside monai
 * Convolution(is_transposed=True), ae:66-76: the transposed convolution itself runs as mig_conv_dgrad. */
int mig_add_channel_bias(int dtype, const void* x, const float* bias, void* y, int64_t rows, int32_t C, void* stream);
/* per-(n,c) broadcast add over S positions: y[n,s,c] = x[n,s,c] + b[n,c] and its reduction backward */
int mig_chan_bias_bwd(int dtype, const void* dy, float* db, int32_t N, int64_t S, int32_t C, void* stream);

/* row softmax over the last dim (fp32 math), attention_scores.softmax(dim=-1) unet:414 */
int mig_softmax_fwd(int dtype_in, int dtype_out, const void* x, void* y, int64_t rows, int32_t cols, float scale,
                    void* stream);
int mig_softmax_bwd(int dtype_p, int dtype_d, const void* p, const void* dp, void* ds, int64_t rows, int32_t cols,
                    float scale, void* stream);
/* the same with bf16 probabilities, fp32 dP and a bf16 dS written directly (no fp32 dS round trip + cast pass) */
int mig_softmax_bwd_narrow(const void* p, const void* dp, void* ds, int64_t rows, int32_t cols, float scale,
                           void* stream);

/* K6: time_emb_proj(silu(emb)) of ALL ResnetBlocks of a U-Net in one launch per pass (unet:691-695; SURVEY K6 "tiny
 * GEMM batched over all ResnetBlocks once per forward"). x: fp32 [rows][K] (= silu(emb)); layer i has weight w[i]
 * [channels[i]][K], bias b[i] (or NULL) and output y[i] [rows][channels[i]]; n <= MIG_TEMB_MAX layers. The pointer
 * arrays are HOST arrays (copied into the kernel parameters). Backward (rows <= 8): dw[i] / db[i] are ACCUMULATED into
 * (dy[i] == NULL: layer without gradient), dx (optional) receives sum_i dy[i] w[i]. */
#define MIG_TEMB_MAX 32
int mig_temb_proj_all_fwd(const float* x, const float* const* w, const float* const* b, float* const* y,
                          const int32_t* channels, int32_t n, int32_t rows, int32_t K, void* stream);
int mig_temb_proj_all_bwd(const float* x, const float* const* w, const float* const* dy, float* const* dw,
                          float* const* db, float* dx, const int32_t* channels, int32_t n, int32_t rows, int32_t K,
                          void* stream);

/* K7: sinusoidal timestep embedding, cos first (unet:461-485). t: fp32 [B] */
int mig_timestep_embedding(const float* t, void* out, int out_dtype, int32_t B, int32_t dim, float max_period,
                           void* stream);

/* ---- K14/K15: DDPMScheduler (monai-generative, call sites ldm:160,165,362) ------------------------
 * coefficient tables are fp32 [T] device arrays; timesteps int64 [B]; one sample = `per_sample` elements */
int mig_ddpm_add_noise(int dtype, const void* x0, const void* noise, const int64_t* timesteps,
                       const float* alphas_cumprod, void* out, int32_t B, int64_t per_sample, int32_t T,
                       int velocity /*0: add_noise, 1: get_velocity*/, void* stream);
/* one reverse step: prev = c0*clamp(x0_hat) + ct*x + sigma*z ; writes x0_hat when non-NULL.
 * prediction: 0 epsilon, 1 sample, 2 v_prediction. `z` may be NULL when sigma == 0 (t == 0). */
int mig_ddpm_step(int dtype, const void* model_out, const void* x, const void* z, void* prev, void* x0_hat,
                  int64_t n, float sqrt_acp_t, float sqrt_one_minus_acp_t, float c0, float ct, float sigma,
                  int prediction, int clip, void* stream);
/* one DDIM step (DDIMScheduler.step / reversed_step): prev = sqrt_acp_prev*clamp(x0_hat) + dir_coef*eps + sigma*z,
 * eps derived from the UNCLIPPED x0_hat; writes the (clipped) x0_hat when non-NULL. prediction: 0 epsilon, 1 sample,
 * 2 v_prediction. `z` may be NULL when sigma == 0 (eta == 0, and every inversion step). */
int mig_ddim_step(int dtype, const void* model_out, const void* x, const void* z, void* prev, void* x0_hat,
                  int64_t n, float sqrt_acp_t, float sqrt_one_minus_acp_t, float sqrt_acp_prev, float dir_coef,
                  float sigma, int prediction, int clip, void* stream);
/* one timestep of the DDPM variational bound (monai-generative DiffusionInferer.get_likelihood): per element, from the
 * model output, the noisy sample x_t and the clean input x0, the KL between the posterior q(x_{t-1} | x_t, x0) and the
 * model's p(x_{t-1} | x_t) when t > 0, and at t == 0 the negative log-likelihood of x0 under the discretised Gaussian
 * decoder (bins of 2 * half_bin, tanh approximation of the normal CDF). t = timesteps[b] (device int64 [B]); every
 * scalar comes from `table`, a device fp32 [T][7] array (table_len == 7 * T): sqrt(acp_t), sqrt(1 - acp_t), c0, ct,
 * -1 + lv - lv + exp(lv - lv), exp(-lv), exp(-0.5 lv) with lv the log of the scheduler's variance. Writes the fp32 map
 * in x's element order when kl_map is non-NULL, and ADDS each sample's mean into total (DEVICE fp64 [B]).
 * prediction: 0 epsilon, 1 sample, 2 v_prediction. Deterministic (fixed-order fp64 reduction, no atomics);
 * workspace = mig_ddpm_vlb_workspace_bytes(B, per_sample) (-1: invalid shape). */
int64_t mig_ddpm_vlb_workspace_bytes(int32_t B, int64_t per_sample);
int mig_ddpm_vlb_term(int dtype, const void* model_out, const void* x_t, const void* x0, const int64_t* timesteps,
                      const float* table, int64_t table_len, int32_t T, int32_t B, int64_t per_sample, int prediction,
                      int clip, float half_bin, float* kl_map, double* total, void* workspace, int64_t workspace_bytes,
                      void* stream);

/* ---- K16/K17: losses --------------------------------------------------------------------------- */
/* out[0] = mean((a-b)^2) (ldm:169) or mean(|a-b|) (aetrain:414); `partials` needs 2048 floats */
int mig_mse_fwd(int dtype, const void* a, const void* b, float* out, float* partials, int64_t n, int l1,
                void* stream);
/* da = gscale[0] * d/da loss ; gscale is a device scalar (upstream grad) */
int mig_mse_bwd(int dtype, const void* a, const void* b, const float* gscale, void* da, int64_t n, int l1,
                void* stream);
/* KL(N(mu,sigma)||N(0,1)) summed over non-batch dims, averaged over batch (aetrain:67-72) */
int mig_kl_fwd(int dtype, const void* mu, const void* sigma, float* out, float* partials, int64_t n, int32_t B,
               void* stream);
int mig_kl_bwd(int dtype, const void* mu, const void* sigma, const float* gscale, void* dmu, void* dsigma,
               int64_t n, int32_t B, void* stream);
/* encode tail (ae:766-769): sigma = exp(clamp(logvar,-30,20)/2); z = mu + eps*sigma (ae:786-787) */
int mig_vae_sample_fwd(int dtype, const void* mu, const void* logvar, const void* eps, void* sigma, void* z,
                       int64_t n, void* stream);
int mig_vae_sample_bwd(int dtype, const void* logvar, const void* eps, const void* sigma, const void* dz,
                       const void* dsigma_ext, void* dmu, void* dlogvar, int64_t n, void* stream);

/* ---- K18: optimizer on flat fp32 buffers (ldm:121,171-180) ---------------------------------------- */
/* out[0] = sum(g^2) over n elements, deterministic two-stage reduction (`partials` needs 2048 floats): data-
 * parallel replicas must derive bit-identical clip coefficients. torch.nn.utils.clip_grad_norm_ (ldm:177) */
int mig_sumsq(const float* g, float* out, float* partials, int64_t n, void* stream);
/* AdamW (decoupled weight decay, torch.optim.AdamW semantics); grad pre-scale = min(1, max_norm/(norm+1e-6))
 * read from device scalar sumsq when max_norm > 0. bf16_shadow (optional) receives the updated params in bf16.
 * step_device (optional): device int32 holding the 1-based step count; overrides `step` so that a captured CUDA
 * graph of the training step stays correct on replay. */
int mig_adamw_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                   float eps, float weight_decay, int32_t step, const float* sumsq, float max_norm,
                   void* bf16_shadow, const int32_t* step_device, void* stream);
/* Sharded optimiser (data parallel, SURVEY 8e; ZeRO-1 style): the same two kernels over `count` pieces of `piece`
 * elements lying `stride` elements apart -- the slice ONE rank owns of every reduce-scattered gradient bucket. All
 * pointers are passed at the rank's first owned element; piece and stride are multiples of 4. */
int mig_sumsq_strided(const float* g, float* out, float* partials, int64_t piece, int64_t stride, int64_t count,
                      void* stream);
int mig_adamw_step_strided(float* p, const float* g, float* m, float* v, int64_t piece, int64_t stride, int64_t count,
                           float lr, float beta1, float beta2, float eps, float weight_decay, int32_t step,
                           const float* sumsq, float max_norm, void* bf16_shadow, const int32_t* step_device,
                           void* stream);

/* ---- D1-D3: data path (SURVEY 8f-4) -- MedicalDataset.__getitem__, medimgen/data_processing.py:540-598 ------------
 * The preprocessed cases ((C,Z,Y,X) fp32, data_processing.py:536-556) live in ONE device buffer `volumes` (the whole
 * dataset fits 180 GB of HBM3e); a training batch is cut out of it on the device instead of by DataLoader workers.
 * One mig_patch_desc per output patch, as a DEVICE array of B entries. */
#define MIG_PATCH_MAX_CH 8
typedef struct {
  int64_t src_offset;                /* element offset of the case's (C,Z,Y,X) block inside `volumes` */
  int32_t src_dims[4];               /* C, Z, Y, X of the case */
  int32_t lb[3];                     /* bbox lower bound per axis (get_bbox, data_processing.py:463-527); may lie outside
                                        the case: those voxels are `pad_value` (crop_and_pad_nd, :150-225) */
  int32_t flip[3];                   /* MirrorTransform per axis (data_processing.py:841-846) */
  int32_t affine;                    /* 0: plain crop; 1: trilinear resample (SpatialTransform rotation / scaling,
                                        :766-774): source offset from the patch centre = mat * output offset (z,y,x);
                                        corners outside the cropped box or the case contribute 0 (zeros padding) */
  float mat[9];
  float mult[MIG_PATCH_MAX_CH];      /* MultiplicativeBrightnessTransform per output channel (:793-800), 1 = off */
  int32_t channel[MIG_PATCH_MAX_CH]; /* source channel per output channel (channel_ids, :565-566) */
} mig_patch_desc;
/* out[b][c][z][y][x] (channels_last = 0, what the reference's DataLoader delivers) or out[b][z][y][x][c], fp32 or bf16:
 * crop + pad + channel selection + resample + mirror + brightness + clamp(lo, hi) in one pass (pass lo > hi for no clamp).
 * 2-D datasets use patch[0] = 1. */
int mig_patch_gather(const float* volumes, const mig_patch_desc* descs, void* out, int out_dtype, int32_t B, int32_t C,
                     const int32_t patch[3], int channels_last, int any_affine /* 0: no desc has affine set */,
                     float pad_value, float lo, float hi, void* stream);
/* per (patch, channel) row of S contiguous fp32 voxels: stats[row] = {mean, unbiased std, min, max}; rows with
 * active[row] == 0 are skipped (active may be NULL = all). Deterministic two-stage reduction, fp64 sums;
 * workspace = mig_patch_stats_workspace_bytes(rows). ContrastTransform / GammaTransform statistics (:801-839). */
int mig_patch_stats(const float* x, float* stats, const int32_t* active, int32_t rows, int64_t S, void* workspace,
                    int64_t workspace_bytes, void* stream);
int64_t mig_patch_stats_workspace_bytes(int32_t rows);
/* per-row intensity transform, x (fp32 rows of S voxels) -> y (fp32 / bf16; channels_last as above, C channels per
 * patch), then clamp(lo, hi) (data_processing.py:595; lo > hi = none). op[row] = {mode, param, invert, 0} as floats:
 *   0 copy (skipped when y == x and no clamp)
 *   1 contrast, preserve_range: clamp((x - mean) * param + mean, min, max)               with stats0[row]
 *   2 gamma: pow((x' - min') / max(range, 1e-7), param) * range + min', x' = -x if invert  with stats0[row]
 *   3 retain_stats: (x - mean1) * std0 / max(std1, 1e-7) + mean0                          with stats0 / stats1 */
int mig_patch_intensity(const float* x, void* y, int out_dtype, const float* op, const float* stats0,
                        const float* stats1, int32_t B, int32_t C, int64_t S, int channels_last, float lo, float hi,
                        void* stream);

/* ---- K8: nearest upsample folded into the convolution that follows it (unet:576-584, ae:97-106) -----------------
 * "nearest x f, then Conv k^n (stride 1, padding p)" only ever reads low-resolution voxels j + floor((r + t - p)/f) for
 * an output voxel f*j + r: per output residue class r it IS a dense convolution of the low-resolution tensor with the
 * taps that land on the same voxel summed (f = 2, k = 3, p = 1: 2 folded taps per axis instead of 3 -> 64/216 of the
 * multiply-adds of a 2x isotropic upsample, and the f^n-times larger tensor never exists). The convolutions themselves
 * are ordinary mig_conv_fwd / mig_conv_wgrad geometries on the low-resolution tensor (ksize = folded taps, pad = -base,
 * out_dims = in_dims); these entry points are the glue. Filters bf16, k <= 4, f in {1, 2} per axis.
 *   which = 0: folded[class r][Cout][u][Cin], classes concatenated in (r0, r1, r2) order -- forward / wgrad filters
 *   which = 1: folded[Cin][s][Cout], s over (f + k - 1)^n -- the filter of the stride-f convolution over dy (kernel
 *              f + k - 1, padding k - 1 - p) whose result is dx */
int64_t mig_upconv_folded_elems(int32_t Cout, int32_t Cin, const int32_t ksize[3], const int32_t factor[3],
                                const int32_t pad[3], int which);
int mig_upconv_fold_filter(const void* w, void* folded, int32_t Cout, int32_t Cin, const int32_t ksize[3],
                           const int32_t factor[3], const int32_t pad[3], int which, void* stream);
/* The folded forward in one call, every class written straight into its positions of the full-resolution output
 * y[N][f*low...][Cout] (no class buffers, no interleave pass): x bf16 [N][low...][Cin], folded = which-0 filters above.
 * Needs mig_upconv_fwd_direct_ok (tcgen05 box kernel: Cin >= 48, channel counts multiples of 8, a TMA box for `low`). */
int mig_upconv_fwd_direct_ok(int32_t N, const int32_t low[3], int32_t Cin, int32_t Cout);
int mig_upconv_fwd(const void* x, const void* folded, const float* bias, void* y, int32_t N, const int32_t low[3],
                   int32_t Cin, int32_t Cout, const int32_t ksize[3], const int32_t factor[3], const int32_t pad[3],
                   void* stream);
/* dw[Cout][t][Cin] += sum over classes of dwc_r[Cout][u_r(t)][Cin]  (fp32; dwc laid out like which = 0 above) */
int mig_upconv_unfold_wgrad(const float* dwc, float* dw, int32_t Cout, int32_t Cin, const int32_t ksize[3],
                            const int32_t factor[3], const int32_t pad[3], void* stream);
/* classes[r][N][low...][C] <-> full[N][f*low...][C] (to_classes = 1: full -> classes, the split of dy for the wgrads) */
int mig_class_interleave(int dtype, const void* src, void* dst, int32_t N, const int32_t low[3], const int32_t factor[3],
                         int32_t C, int to_classes, void* stream);

/* ---- SSIM / MS-SSIM validation metrics (ldm:241-330: generative.metrics.SSIMMetric / MultiScaleSSIMMetric) --------
 * Replaces monai-generative's compute_ssim_and_cs (five depthwise conv{2,3}d with the dense window, then the SSIM and
 * contrast-structure maps) for a list of image pairs, with the window applied separably and nothing but the inputs in
 * HBM. a: [na][D][H][W][C], b: [nb][D][H][W][C] (channels-last, same dtype; 2-D images use D = 1, ksize[0] = 1).
 * pairs: DEVICE int32 [P][2] of (index into a, index into b); a pair with an index out of range gets NaN.
 * taps_host: the three 1-D windows, D taps then H taps then W taps (ksize[0] + ksize[1] + ksize[2] floats), 1 <= k <= 16
 * and k <= the extent per axis. "Valid" correlation (extent - k + 1 per axis), c1 = (k1 L)^2, c2 = (k2 L)^2 as given.
 * out: DEVICE fp64 [P][2] = (mean ssim, mean cs) over channels and valid voxels. Deterministic (fixed-order fp64
 * reduction, no atomics); workspace = mig_ssim_workspace_bytes(P, C, dims, ksize) (-1: invalid shape). */
int64_t mig_ssim_workspace_bytes(int32_t P, int32_t C, const int32_t dims[3], const int32_t ksize[3]);
int mig_ssim_pairs(int dtype, const void* a, const void* b, int32_t na, int32_t nb, const int32_t* pairs, int32_t P,
                   const int32_t dims[3], int32_t C, const int32_t ksize[3], const float* taps_host, float c1, float c2,
                   double* out, void* workspace, int64_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MEDIMGEN_B200_H */
