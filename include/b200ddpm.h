/*
 * b200ddpm — C ABI of the B200-native DDPM reverse-diffusion sampling path.
 *
 * The reference (TheaQG/DiffusionModelsCustom) is pure Python and has no FFI; its "boundary" for this path is two
 * duck-typed Python contracts (SURVEY.md §8(b)):
 *   sampler -> model : model(x, t, y, cond_img, lsm_cond, topo_cond)
 *                      DDPM_DANRA_conditional/diffusion_DANRA_conditional.py:146, modules_DANRA_conditional.py:597-616
 *                      (Family D: model(x, t, y_lowres), DDPM_clean_application/src/unet_ms.py:148)
 *   script  -> sampler: DiffusionUtils(...).sample(x, model, y, cond_img, lsm_cond, topo_cond)
 *                      DDPM_DANRA_conditional/diffusion_DANRA_conditional.py:105-159
 * The entry points below are what a ctypes/cffi binding of those two calls needs; diffusionmodelscustom_b200/_native.py is
 * that binding and INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a negative error code and never
 * throws; b2d_last_error() returns the message of the calling thread's last failure.  Device pointers are caller-owned
 * and must stay valid until the work queued on `stream` has completed.  A handle owns its packed weights, workspaces,
 * TMA descriptors and CUDA graphs; it is bound to the CUDA device current at b2d_create() and is not thread-safe.
 * `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream).
 * There is no CPU fallback anywhere behind this ABI.
 */
#ifndef B200DDPM_H
#define B200DDPM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2D_ABI_VERSION 1

typedef struct b2d_handle b2d_handle;

enum { B2D_FAMILY_R = 0, /* DiffusionNet(Encoder, Decoder): modules_DANRA_conditional.py / modules_DANRA_flexible.py */
       B2D_FAMILY_D = 1  /* UNet_downscale: DDPM_clean_application/src/unet_ms.py */ };

typedef struct b2d_config {
    int32_t family;        /* B2D_FAMILY_R / B2D_FAMILY_D */
    int32_t img_size;      /* H == W of the high-resolution field (power of two, 32..128) */
    int32_t max_batch;     /* workspaces are sized for this many samples */
    int32_t c_hr;          /* channels of x (Encoder(input_channels=...)), normally 1 */
    int32_t c_out;         /* Decoder(output_channels=...), normally 1 */
    int32_t has_lsm;       /* Encoder built with lsm_tensor (modules_DANRA_conditional.py:157-159) */
    int32_t has_topo;      /* Encoder built with topo_tensor (:160-162) */
    int32_t cond_channels; /* cond_img_dim[0] if cond_on_img else 0 (:163-164); Family D: channels of the low-res field */
    int32_t num_classes;   /* label_emb rows, 0 = none (:194-196) */
    int32_t n_heads;       /* attention heads (default 4) */
    int32_t attn_ff;       /* 1: attention block has the LN-Linear-GELU-Linear tail (src/unet.py:91-96, unet_ms.py:13-18) */
    int32_t debug_simt_conv; /* 1: run GEMM-shaped ops on the CUDA-core cross-check kernel (bring-up only) */
    int32_t interp_mode;   /* Family D: F.interpolate mode of the low-resolution field (unet_ms.py:105,156): B2D_INTERP_* */
    int32_t stem_embedding; /* Family R: 0 = Encoder.pos_encoding (base 1000, [sin | cos] halves, modules_DANRA_conditional.py:203-211);
                              1 = the interleaved base-10000 SinusoidalEmbedding the Downscaling generation uses in its encoder
                              (DDPM_DANRA_Downscaling/modules_DANRA_downscaling.py:190-197) */
} b2d_config;
enum { B2D_INTERP_BICUBIC = 0, B2D_INTERP_BILINEAR = 1, B2D_INTERP_NEAREST = 2 };

/* One named FP32 tensor of a reference state_dict (host memory, contiguous, torch layout). */
typedef struct b2d_tensor {
    const char* name;     /* reference key, e.g. "encoder.layer1.0.conv1.weight" */
    const float* data;    /* host pointer, fp32 */
    int32_t ndim;
    int64_t shape[4];
} b2d_tensor;

const char* b2d_last_error(void);
int b2d_abi_version(void);

/* ---- handle life cycle ------------------------------------------------------------------------------------- */
int b2d_create(const b2d_config* cfg, b2d_handle** out);
void b2d_destroy(b2d_handle* h);

/* Replaces `model.load_state_dict(torch.load(p)['network_params'])` (generation_DANRA_conditional.py:354-360):
 * takes the reference's keys, folds eval-mode BatchNorm into the convolutions, re-packs to K-major f16. */
int b2d_load_weights(b2d_handle* h, const b2d_tensor* tensors, int32_t n);

/* Schedule tables owned by DiffusionUtils (diffusion_DANRA_conditional.py:47-51): T floats each, host memory. */
int b2d_set_schedule(b2d_handle* h, const float* betas, const float* alphas, const float* alpha_hat, int32_t T);

/* Step-invariant conditioning of the current batch (device fp32, NCHW [B,1|C,H,W]; NULL = absent), y = int64 [B] season
 * class (device) or NULL.  Family D: `cond` is the low-resolution field [B,C,h,w] with cond_h x cond_w pixels, which is
 * bicubic-interpolated once (unet_ms.py:156).  Pre-computes everything that does not depend on x or t. */
int b2d_set_conditioning(b2d_handle* h, const float* lsm, const float* topo, const float* cond, int32_t cond_h,
                         int32_t cond_w, const int64_t* y, int32_t B, void* stream);

/* One eps_hat = model(x, t, ...) evaluation.  x, eps_out: device fp32 [B,c_hr,H,W]; t: HOST int64 [B]. */
int b2d_forward(b2d_handle* h, const float* x, const int64_t* t_host, float* eps_out, int32_t B, void* stream);

/* Stand-alone halves of DiffusionNet.forward (Family R), for callers that use Encoder / Decoder on their own
 * (Encoder.forward modules_DANRA_conditional.py:213-312 returns fmap1..fmap5; Decoder.forward :512-536 takes them and t).
 * Feature maps cross this boundary as the reference passes them: device fp32 NCHW, [B,64,H/2,H/2] [B,64,H/4,H/4] [B,128,H/8,H/8]
 * [B,256,H/16,H/16] [B,512,H/32,H/32].  Conditioning for the encoder is whatever b2d_set_conditioning installed. */
int b2d_encoder_forward(b2d_handle* h, const float* x, const int64_t* t_host, float* const* fmaps_out, int32_t B, void* stream);
int b2d_decoder_forward(b2d_handle* h, const float* const* fmaps_in, const int64_t* t_host, float* eps_out, int32_t B, void* stream);

/* Whole reverse loop i = T-1 .. 1 on device memory (DiffusionUtils.sample, diffusion_DANRA_conditional.py:127-157).
 * x_inout: device fp32 [B,c_hr,H,W], x_T in / x_0 out.  noise: device fp32 [T][B*c_hr*H*W] host-generated z_i indexed by
 * i (parity runs) or NULL for in-kernel Philox keyed by (seed, sample_offset + sample index, i).
 * noise_scale multiplies z — drawn or injected — (1.0; 0.005 for data_scaled, src/diffusion_modules.py:173-174).
 * The handle captures its step graphs once per (batch, schedule length): seed, offset, scale, the noise pointer and the state
 * live in device memory, so repeated jobs replay the same graphs (x_inout is copied into / out of the handle's state buffer). */
int b2d_sample(b2d_handle* h, float* x_inout, const float* noise, uint64_t seed, uint64_t sample_offset,
               float noise_scale, int32_t B, void* stream);

/* ---- fewer-step sampling: DDIM (Song, Meng & Ermon 2021, eq. 12) ------------------------------------------------------
 * Over a strictly decreasing timestep sequence tau_0 > ... > tau_{S-1} (each in [1, T-1]) and eta in [0, 1], step k goes from
 * t = tau_k to t' = tau_{k+1} with a = alpha_hat[t], a' = alpha_hat[t'] (a' = 1 after the last step, whose result is x0_hat):
 *   x0_hat = (x - sqrt(1-a) eps_hat) / sqrt(a)
 *   sigma  = eta * sqrt((1-a')/(1-a)) * sqrt(1 - a/a')
 *   x'     = sqrt(a') x0_hat + sqrt(max(0, 1-a'-sigma^2)) eps_hat + sigma * noise_scale * z
 * No x0_hat clipping; the last step draws no noise.  z is Philox keyed by (seed; sample_offset + sample, element) with the step
 * slot set to tau_k, or injected noise [S][B*c_hr*H*W] indexed by k.
 * b2d_set_timesteps switches the handle's sampler: b2d_sample, b2d_sample_host and b2d_ensemble_run then run S evaluations of
 * the DDIM loop instead of the T-1 of the DDPM loop.  The two loops keep separate step graphs. */
/* n == 0 (timesteps NULL) restores the reference DDPM loop.  Validated: strictly decreasing, 1 <= t <= T-1, 0 <= eta <= 1;
 * re-validated at sampling time against the current schedule length. */
int b2d_set_timesteps(b2d_handle* h, const int32_t* timesteps_host, int32_t n, float eta);
/* One DDIM step on device memory (foreign-model loop, op tests).  t_prev = -1: final step to x0 (alpha_hat' = 1).
 * alpha_hat: device fp32 [T]; z_or_null: this step's z [B*per_sample] or NULL for Philox.  Synchronises `stream` once (reads
 * alpha_hat[t] and alpha_hat[t_prev] back for the coefficients). */
int b2d_op_ddim_update(float* x, const float* eps, const float* z_or_null, const float* alpha_hat, int32_t T, int32_t t,
                       int32_t t_prev, float eta, int32_t B, int64_t per_sample, uint64_t seed, uint64_t sample_offset,
                       float noise_scale, void* stream);

/* End-to-end entry with HOST buffers: uploads x_T and the conditioning, runs b2d_sample, downloads x_0, synchronises. */
int b2d_sample_host(b2d_handle* h, float* x_inout_host, const float* lsm_host, const float* topo_host,
                    const float* cond_host, int32_t cond_h, int32_t cond_w, const int64_t* y_host,
                    const float* noise_host, uint64_t seed, uint64_t sample_offset, float noise_scale, int32_t B);

/* ---- ensemble generation (SURVEY.md §8(f1)) ------------------------------------------------------------------
 * "dates x members" through the sampler: replaces the host loop around DiffusionUtils.sample in the reference's generation
 * scripts (generation_DANRA_conditional.py:369-441, DDPM_clean_application/test/generation_ddpm.py:371-439).  The
 * conditioning fields are given once PER DATE (host memory); the flattened date-major member list [first, first+count) is
 * sampled in sub-batches with x_T drawn on the device (Philox keyed by the global member index, so the result does not
 * depend on sub_batch or on how ranks slice the list), uploads / downloads double-buffered on a copy stream. */
typedef struct b2d_ensemble_job {
    int32_t n_dates, members, sub_batch;
    int32_t first, count;      /* slice of the flattened member list this call (this rank) produces */
    const float* lsm;          /* host [n_dates][H][W] or NULL */
    const float* topo;         /* host [n_dates][H][W] or NULL */
    const float* cond;         /* host [n_dates][C][H][W] (Family D: [n_dates][C][cond_h][cond_w]) or NULL */
    int32_t cond_h, cond_w;    /* Family D low-resolution extent, else 0 */
    const int64_t* y;          /* host [n_dates] season classes or NULL */
    float* out;                /* host [count][c_hr][H][W]; page-locked for the call when possible */
    uint64_t seed;
    float noise_scale;         /* multiplies z_i (1.0; 0.005 for data_scaled) */
    float xT_scale;            /* multiplies x_T (1.0; 0.005 for data_scaled, src/diffusion_modules.py:134-137) */
} b2d_ensemble_job;
typedef struct b2d_ensemble_stats {
    int32_t sub_batches;
    int32_t out_pinned;        /* 1: fields were copied straight into `out`; 0: through the driver's pinned bounce buffers */
    int64_t launches;
    double gather_ms;          /* host time spent gathering conditioning rows into the pinned staging */
    double wall_ms;
} b2d_ensemble_stats;
int b2d_ensemble_run(b2d_handle* h, const b2d_ensemble_job* job, b2d_ensemble_stats* stats);

/* fp32 -> fp16 conversions that had to be clamped to +-65504 since the last reset (all handles of this process/device).
 * Activations are stored in fp16; a non-zero count means the loaded checkpoint leaves that range somewhere and the
 * result is clipped there.  Returns 0xFFFFFFFF on a CUDA error. */
unsigned int b2d_saturation_count(int32_t reset);

/* Kernel launches issued by the last b2d_forward / b2d_sample on this handle (graph nodes x replays). */
int64_t b2d_last_launch_count(const b2d_handle* h);
/* Per-launch device time of one eps evaluation: runs the step program `reps` times (after one warm-up) with a CUDA event
 * between launches on the handle's stream and reports, per launch, its layer name, kernel class, algorithmic FLOPs/bytes
 * and mean duration.  x: device fp32 [B,c_hr,H,W]; t_host: host int64 [B].  Used by bench.py for the live roofline. */
typedef struct b2d_op_profile {
    char name[48];
    char klass[24];
    double flops;
    double bytes;
    double ms;
} b2d_op_profile;
int b2d_profile_step(b2d_handle* h, const float* x, const int64_t* t_host, int32_t B, int32_t reps, b2d_op_profile* out,
                     int32_t max_ops, int32_t* n_ops);

/* Bring-up aid: copies a named NHWC f16 activation of the last evaluation ("fmap1".."fmap5", "dec0".."dec3", ...) to
 * host fp32 [B,hw,hw,C]; synchronises the device. */
int b2d_debug_read(b2d_handle* h, const char* name, float* out_host, int64_t max_elems, int32_t* C_out, int32_t* hw_out);

/* ---- forward process, loss and evaluation statistics (SURVEY.md §8(f3), (f4)); all pointers device memory ------------ */
/* DiffusionUtils.noiseImage (diffusion_DANRA_conditional.py:85-103): x_t = sqrt(alpha_hat[t]) x_0 + sqrt(1 - alpha_hat[t]) eps, with
 * eps given (noise_or_null) or drawn in-kernel (Philox keyed by sample_offset + b); eps * noise_scale is written to noise_out
 * (x0.005 for data_scaled).  t_dev: int64 [B]; alpha_hat: float [T]. */
int b2d_op_noise_image(const float* x0, const int64_t* t_dev, const float* alpha_hat, const float* noise_or_null, float* x_t,
                       float* noise_out, int32_t B, int64_t per_sample, uint64_t seed, uint64_t sample_offset, float noise_scale,
                       void* stream);
/* SDFWeightedMSELoss.forward (training_DANRA_conditional.py:33-56): mean(w (input - target)^2), w = sigmoid(sdf) (max_land -
 * min_sea) + min_sea; sdf_or_null == NULL gives nn.MSELoss.  One fused pass, deterministic; scalar written to device memory. */
int b2d_op_weighted_mse(const float* input, const float* target, const float* sdf_or_null, float max_land_weight,
                        float min_sea_weight, float* out_scalar_dev, int64_t n, void* stream);
/* evaluation_DANRA_conditional.py:121-122: per-sample nan-aware MAE and RMSE over the hw pixels of gen/eval [n_samples][hw]. */
int b2d_op_eval_daily(const float* gen, const float* eval, float* mae_out, float* rmse_out, int32_t n_samples, int64_t hw,
                      void* stream);
/* per-pixel nan-aware MAE / RMSE / bias (mean of gen - eval) over the samples; outputs [hw]. */
int b2d_op_eval_pixel(const float* gen, const float* eval, float* mae_out, float* rmse_out, float* bias_out, int32_t n_samples,
                      int64_t hw, void* stream);
/* numpy-style fixed-range histogram (NaN and out-of-range values dropped, right edge closed); counts: uint64 [bins], bins <= 4096. */
int b2d_op_histogram(const float* x, int64_t n, float lo, float hi, int32_t bins, unsigned long long* counts_dev, void* stream);

/* Bring-up aid: per-key-block clock64 stamps of the persistent attention kernel (only filled by a -DAT2_TRACE build):
 * [256][12] int64.  Returns the number of rows. */
int b2d_debug_attn_trace(long long* out_host, int32_t max_elems);

/* ---- single operators (unit-test / profiling entry points; all pointers are device memory) ------------------ */
/* NHWC f16 convolution / projection through the same kernels the model uses.
 * w_packed: f16 [Cout][R*S*Cin] (convt: [(a*2+b)*CoutT+co][Cin]); impl 0 = tcgen05 (kernel chosen as in the model program),
 * 1 = CUDA-core cross-check, 2 = force the streaming GEMM, 3 = force the persistent two-accumulator convolution,
 * 4 = force the one-tile-per-CTA convolution. */
int b2d_op_conv2d(const void* in_f16, const void* w_packed_f16, const float* bias, const void* residual_f16,
                  const float* post_add, int32_t post_stride, void* out_f16, int32_t B, int32_t Hi, int32_t Wi,
                  int32_t Cin, int32_t Cout, int32_t R, int32_t S, int32_t stride, int32_t pad, int32_t convt,
                  int32_t act, int32_t impl, void* stream);
int b2d_op_layernorm(const void* x_f16, const float* gamma, const float* beta, void* y_f16, int32_t rows, int32_t C,
                     void* stream);
int b2d_op_attention(const void* qkv_f16, void* o_f16, int32_t B, int32_t L, int32_t C, int32_t heads, void* stream);
/* Fused low-resolution attention (L <= 64 tokens, 128 % L == 0, head_dim 32/64/128): LayerNorm + QKV projection + softmax(QK^T)V.
 * w_folded: f16 [3C][C] = in_proj_weight * ln_gamma; c1[n] = sum_k w_folded[n][k]; bias[n] = in_proj_bias[n] + sum_k W[n][k]*ln_beta[k].
 * Replaces nn.LayerNorm + the in-projection and scaled-dot-product part of nn.MultiheadAttention
 * (modules_DANRA_conditional.py:100-107); the out-projection is a b2d_op_conv2d. */
int b2d_op_attn_block(const void* x_f16, const void* w_folded_f16, const float* c1, const float* bias, void* o_f16,
                      int32_t B, int32_t L, int32_t C, int32_t heads, void* stream);
/* The whole ImageSelfAttention block in one launch: y = act( out_proj( MHA_core( LN(x) ) ) + x ) (modules_DANRA_conditional.py:91-110).
 * wo: out_proj.weight f16 [C][C]; final_act 0 none / 1 ReLU (DecoderBlock, :459). heads <= 8. */
int b2d_op_attn_block_out(const void* x_f16, const void* w_folded_f16, const float* c1, const float* bias, const void* wo_f16,
                          const float* out_bias, void* y_f16, int32_t B, int32_t L, int32_t C, int32_t heads,
                          int32_t final_act, void* stream);
int b2d_op_instnorm(const void* x_f16, const void* skip_f16, const float* vec, int32_t vec_stride, void* y_f16,
                    float* stats_ws, int32_t B, int32_t HW, int32_t C, void* stream);
/* Decoder.final_layer without its ConvTranspose (modules_DANRA_conditional.py:503-509): InstanceNorm2d(64) -> Conv2d(64 -> 1, 3x3,
 * pad 1) + bias on x [B,H,W,64] f16 -> out [B,1,H,W] fp32.  w: conv weight fp32, K-major [tap * 64 + c] (tap = 3*ky + kx).
 * use_mma_sync != 0 selects the legacy tail_mma_kernel instead of the tcgen05 tail (A/B and the c_out > 1 path). */
int b2d_op_final_layer(const void* x_f16, const float* w_kmajor, const float* bias, float* out, int32_t B, int32_t H, int32_t W,
                       int32_t use_mma_sync, void* stream);
int b2d_op_posterior_update(float* x, const float* eps, const float* z_or_null, const float* betas, const float* alphas,
                            const float* alpha_hat, int32_t i, int32_t B, int64_t per_sample, uint64_t seed,
                            uint64_t sample_offset, float noise_scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200DDPM_H */
