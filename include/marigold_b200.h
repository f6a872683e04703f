/* libmarigold_b200 — C ABI of the B200-native Marigold denoising hot path.
 *
 * The reference (prs-eth/Marigold) has no FFI: its hot path is the Python object protocol
 *   vae.encoder / vae.quant_conv            marigold/marigold_depth_pipeline.py:491-492
 *   scheduler.set_timesteps / .timesteps    marigold/marigold_depth_pipeline.py:423-424
 *   unet(x, t, encoder_hidden_states)       marigold/marigold_depth_pipeline.py:461-463
 *   scheduler.step(...).prev_sample         marigold/marigold_depth_pipeline.py:466-468
 *   vae.post_quant_conv / vae.decoder       marigold/marigold_depth_pipeline.py:512-513
 *   ensemble_depth / ensemble_normals       marigold/util/ensemble.py:39,199
 * Each entry point below names the call(s) it replaces. INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - Every pointer named *_dev is a CUDA device pointer owned by the caller; image-like tensors
 *     are contiguous NCHW fp32 (the reference's layout). NHWC/bf16 is an internal detail.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and the call returns
 *     without synchronising unless stated otherwise.
 *   - Every function returns 0 (MGB_OK) or a negative mgb_status; mgb_last_error() has the text.
 *   - A handle is not thread-safe: one handle per process per GPU.
 *   - There is no CPU fallback anywhere behind this ABI.
 */
#ifndef MARIGOLD_B200_H_
#define MARIGOLD_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  MGB_OK = 0,
  MGB_ERR_INVALID = -1,      /* bad argument (shape, null pointer, unknown key ...) */
  MGB_ERR_CUDA = -2,         /* a CUDA runtime/driver call failed */
  MGB_ERR_STATE = -3,        /* call order violated (e.g. denoise before finalize_weights) */
  MGB_ERR_NOMEM = -4,
  MGB_ERR_UNSUPPORTED = -5   /* valid request this build does not implement */
} mgb_status;

typedef enum { MGB_F32 = 0, MGB_BF16 = 1, MGB_F16 = 2 } mgb_dtype;
typedef enum { MGB_DECODE_DEPTH = 0, MGB_DECODE_NORMALS = 1, MGB_DECODE_RAW3 = 2, MGB_DECODE_UNIT3 = 3 } mgb_decode_mode;

typedef struct mgb_handle mgb_handle;

/* Architecture description (diffusers config.json fields; SURVEY.md App. A).
 * Channel counts must be multiples of 64; attention head_dim is 64 (SD-2: "attention_head_dim"
 * there is a head COUNT, C/64). */
typedef struct {
  int32_t unet_in_channels;        /* 8 = rgb latent (4) | target latent (4); IID with n targets: 4 (n + 1) */
  int32_t unet_out_channels;       /* 4; IID: 4 n (n <= 4)                                          */
  int32_t unet_block_channels[4];  /* 320, 640, 1280, 1280                                          */
  int32_t unet_layers_per_block;   /* 2                                                             */
  int32_t unet_cross_dim;          /* 1024                                                          */
  int32_t vae_block_channels[4];   /* 128, 256, 512, 512                                            */
  int32_t vae_layers_per_block;    /* 2                                                             */
  int32_t vae_latent_channels;     /* 4                                                             */
  int32_t norm_groups;             /* 32                                                            */
  float latent_scale;              /* 0.18215 (marigold_depth_pipeline.py:118)                      */
} mgb_config;

/* ---- lifecycle ------------------------------------------------------------------------------ */
int mgb_create(const mgb_config* cfg, mgb_handle** out);
void mgb_destroy(mgb_handle* h);
const char* mgb_last_error(void);
/* library build info: "sm_100a;tcgen05;..." */
const char* mgb_build_info(void);

/* ---- weights (replaces DiffusionPipeline.from_pretrained state-dict loading) ---------------- */
/* `key` is the diffusers state-dict name prefixed by the sub-model: "unet.conv_in.weight",
 * "vae.decoder.mid_block.attentions.0.to_q.bias", ... `data` is a HOST pointer, contiguous,
 * in the PyTorch layout ([out,in,kh,kw] conv, [out,in] linear). */
int mgb_load_tensor(mgb_handle* h, const char* key, const void* data, const int64_t* shape, int32_t ndim,
                    int32_t dtype);
/* Repack to kernel layouts (bf16, tap-major conv weights, fused QKV, GEGLU-interleaved FF) and
 * verify that every tensor the architecture needs was loaded. */
int mgb_finalize_weights(mgb_handle* h);

/* ---- conditioning --------------------------------------------------------------------------- */
/* Empty-prompt embedding [n_tokens, cross_dim] fp32 HOST (marigold_depth_pipeline.py:381-394,
 * 438-442; n_tokens == 2). Cross-attention K/V of every block are folded here, once. */
int mgb_set_text_embedding(mgb_handle* h, const float* embed_host, int32_t n_tokens);

/* scheduler.set_timesteps + the per-step coefficients of scheduler.step, computed by the host in
 * float64 (marigold_b200/schedulers.py) so scheduler-config handling stays in Python:
 *     x_prev = kx[i] * x + kv[i] * model_output + kz[i] * noise_i
 * (DDIM eta=0: kz = 0; LCM: kz != 0 on every step but the last). All arrays have n entries. */
int mgb_set_schedule(mgb_handle* h, int32_t n, const int32_t* timesteps, const float* kx, const float* kv,
                     const float* kz);

/* ---- the hot path --------------------------------------------------------------------------- */
/* encode_rgb: vae.encoder + quant_conv, mean half, * latent_scale  (…pipeline.py:479-496).
 * rgb_dev [B,3,H,W] in [-1,1]; latent_dev [B,4,H/8,W/8] (floor). Any H, W >= 8: like the reference, sizes that are not
 * multiples of 8 lose the remainder rows / columns in the VAE's stride-2 convs. */
int mgb_encode(mgb_handle* h, const float* rgb_dev, int32_t B, int32_t H, int32_t W, float* latent_dev,
               void* stream);
/* One denoising iteration i: cat -> unet -> scheduler.step (…pipeline.py:456-468).
 * target_dev [B,Ct,h,w] (Ct = unet_out_channels: 4, or 4 n for an n-target IID model, marigold_iid_pipeline.py:538-551)
 * is updated in place; noise_dev (or NULL) is this step's z; if model_out_dev != NULL it also receives the raw UNet
 * output [B,Ct,h,w]. Any h, w >= 1 (odd sizes follow diffusers' `upsample_size` path). */
int mgb_unet_step(mgb_handle* h, const float* rgb_latent_dev, float* target_dev, const float* noise_dev,
                  float* model_out_dev, int32_t step_index, int32_t B, int32_t lh, int32_t lw, void* stream);
/* The whole loop (…pipeline.py:455-468): steps 0..n-1 of the current schedule.
 * step_noise_dev: [n-1, B, Ct, h, w] or NULL (required when any kz != 0). */
int mgb_denoise(mgb_handle* h, const float* rgb_latent_dev, float* target_dev, const float* step_noise_dev,
                int32_t B, int32_t lh, int32_t lw, void* stream);
/* Steps [first_step, first_step + num_steps) of the current schedule only (bench.py times K steps of a
 * longer schedule with it). step_noise_dev is indexed by absolute step: [n-1, B, 4, h, w]. */
int mgb_denoise_range(mgb_handle* h, const float* rgb_latent_dev, float* target_dev, const float* step_noise_dev,
                      int32_t first_step, int32_t num_steps, int32_t B, int32_t lh, int32_t lw, void* stream);
/* decode_depth / decode_normals + the clip / shift / normalise that follow
 * (…depth_pipeline.py:498-516,473-475; …normals_pipeline.py:463-479,438-440).
 * out_dev: DEPTH [B,1,H,W] in [0,1]; NORMALS [B,3,H,W] unit vectors; RAW3 [B,3,H,W]; UNIT3 [B,3,H,W] = (clip(x,-1,1)+1)/2
 * (one IID target, marigold_iid_pipeline.py:562-565,578-585: the caller loops over the targets' 4-channel slices). */
int mgb_decode(mgb_handle* h, const float* latent_dev, int32_t B, int32_t lh, int32_t lw, int32_t mode,
               float* out_dev, void* stream);

/* ---- ensembling (marigold/util/ensemble.py) ------------------------------------------------- */
/* cost_fn of ensemble_depth (ensemble.py:138-152) in ONE pass and ONE host sync:
 * depth_dev [E,HW] fp32; param_host = [s_0..s_{E-1}, t_0..t_{E-1}] (or only s when !shift);
 * returns sum_{i<j} RMSE(a_i - a_j) + reg * (|min(med)| + |1 - max(med)|). Synchronises. */
int mgb_ens_depth_cost(mgb_handle* h, const float* depth_dev, const double* param_host, int32_t E, int64_t HW,
                       int32_t scale_invariant, int32_t shift_invariant, int32_t reduction_median,
                       double regularizer, double* cost_out, void* stream);
/* The same objective for P parameter vectors (params_host [P][2E], or [P][E] when !shift) in ONE launch and ONE
 * synchronisation: the 2E forward-difference points of one scipy BFGS gradient (ensemble.py:165-171; scipy's
 * approx_derivative) are one call. costs_out_host [P]. cost(x) is bit-identical to mgb_ens_depth_cost(x). */
int mgb_ens_depth_cost_batch(mgb_handle* h, const float* depth_dev, const double* params_host, int32_t P, int32_t E,
                             int64_t HW, int32_t scale_invariant, int32_t shift_invariant, int32_t reduction_median,
                             double regularizer, double* costs_out_host, void* stream);
/* One forward-difference gradient of that objective in a single pass (scipy approx_derivative as BFGS calls it,
 * ensemble.py:165-171): base_host [n] is the current point, pert_host [n] the same vector with EVERY coordinate moved to
 * its perturbed value x_i + h_i; costs_out_host [1 + n]: [0] = cost(base), [1 + i] = cost(base with coordinate i
 * perturbed), each bit-identical to mgb_ens_depth_cost of that vector. n = 2E (or E when !shift); E <= 16. */
int mgb_ens_depth_cost_fd(mgb_handle* h, const float* depth_dev, const double* base_host, const double* pert_host,
                          int32_t E, int64_t HW, int32_t scale_invariant, int32_t shift_invariant,
                          int32_t reduction_median, double regularizer, double* costs_out_host, void* stream);
/* Largest ensemble size the ensembling entry points accept (sizes <= 16 run register-resident kernels). */
int mgb_ens_max_members(void);
/* init_param statistics (ensemble.py:91-105): per-member min and max. Synchronises. */
int mgb_ens_minmax(mgb_handle* h, const float* depth_dev, int32_t E, int64_t HW, float* min_host, float* max_host,
                   void* stream);
/* align + ensemble + min-max renormalise (ensemble.py:178-196). pred_dev [HW]; uncert_dev [HW] or NULL.
 * member_idx_dev (int32 [HW] or NULL) receives the index of the member picked by the (lower) median. */
int mgb_ens_depth_reduce(mgb_handle* h, const float* depth_dev, const double* param_host, int32_t E, int64_t HW,
                         int32_t scale_invariant, int32_t shift_invariant, int32_t reduction_median,
                         float* pred_dev, float* uncert_dev, int32_t* member_idx_dev, void* stream);
/* ensemble_normals (ensemble.py:199-249): normals_dev [E,3,HW]; out_dev [3,HW]; uncert_dev [HW] or NULL;
 * member_idx_dev int32 [HW] or NULL = argmax index. reduction_closest: 1 = "closest", 0 = "mean". */
int mgb_ens_normals(mgb_handle* h, const float* normals_dev, int32_t E, int64_t HW, int32_t reduction_closest,
                    float* out_dev, float* uncert_dev, int32_t* member_idx_dev, void* stream);

/* ensemble_iid (ensemble.py:252-270): targets_dev [E, N] (N = 3 n H W) -> pred_dev [N] = lower median (or mean) over the
 * members; uncert_dev [N] or NULL = median absolute deviation (or unbiased std). No alignment, no renormalisation. */
int mgb_ens_iid(mgb_handle* h, const float* targets_dev, int32_t E, int64_t N, int32_t reduction_median, float* pred_dev,
                float* uncert_dev, void* stream);

/* ---- pre / post-processing bookends and the evaluation step ------------------------------------ */
/* torchvision resize(antialias=True) as resize_max_res calls it (marigold/util/image_util.py:90-120) and for the final
 * prediction (marigold_depth_pipeline.py:306-312). src_dev [NC,H,W] uint8 (src_is_u8) or fp32 -> dst_dev fp32 [NC,h,w].
 * mode 0 bilinear, 1 bicubic (both antialiased), 2 nearest-exact. post 0: none; 1: round + clamp to [0,255] (a uint8
 * image stays uint8-valued); 2: that, then x / 255 * 2 - 1 (marigold_depth_pipeline.py:252). tmp_dev: NC*H*w floats. */
int mgb_resize(const void* src_dev, int32_t src_is_u8, int32_t NC, int32_t H, int32_t W, float* dst_dev, int32_t h, int32_t w,
               int32_t mode, int32_t post, float* tmp_dev, void* stream);
/* colorize_depth_maps + chw2hwc + uint8 (image_util.py:38-76, marigold_depth_pipeline.py:326-331): depth_dev fp32 [HW] ->
 * out_hwc_dev uint8 [HW,3]; lut_dev uint8 [256,3] = the colour map's 256-entry table * 255, truncated. */
int mgb_colorize(const float* depth_dev, int64_t HW, float dmin, float dmax, const uint8_t* lut_dev, uint8_t* out_hwc_dev,
                 void* stream);
/* Scratch of every mgb_eval_* call: a fixed size, independent of the image. */
size_t mgb_eval_ws_bytes(void);
/* Least-squares scale / shift alignment to the ground truth over the valid pixels (src/util/alignment.py:35-82), the
 * clips of script/depth/eval.py:201-207 and the masked depth metrics of src/util/metric.py:64-191 in two passes and ONE
 * synchronisation. alignment: 0 none, 1 least squares in depth ("least_square"), 2 least squares in disparity
 * ("least_square_disparity", eval.py:179-199 with depth2disparity, alignment.py:85-95: fit pred to 1 / gt over
 * mask & gt > 0 & pred > 0, depth = 1 / clip(pred * scale + shift, 1e-3)). mask_dev uint8 [HW] or NULL; aligned_out_dev
 * fp32 [HW] or NULL (the final clipped depth); ws_dev: mgb_eval_ws_bytes() bytes.
 * out_host[13] = {scale, shift, n_valid, abs_rel, sq_rel, rmse, rmse_log, log10, delta1, delta2, delta3, i_rmse, silog}
 * (scale, shift in disparity space for alignment 2). */
int mgb_eval_depth(const float* pred_dev, const float* gt_dev, const uint8_t* mask_dev, int64_t HW, int32_t alignment,
                   float dmin, float dmax, float* aligned_out_dev, void* ws_dev, double* out_host, void* stream);
/* compute_cosine_error(masked=True) and the normals metrics mean / median / rmse / sub5 .. sub30_error
 * (src/util/metric.py:194-257 as script/normals/eval.py:145-157 calls them) with ONE synchronisation; the median is an
 * exact order statistic on the device (the reference copies the error map to the host for np.median).
 * pred_dev, gt_dev fp32 [3,HW]; angles_out_dev fp32 [HW] or NULL: degrees, NaN where ||gt|| == 0.
 * out_host[9] = {n_valid, mean, median, rmse, %<5, %<7.5, %<11.25, %<22.5, %<30} (NaN metrics when n_valid == 0). */
int mgb_eval_normals(const float* pred_dev, const float* gt_dev, int64_t HW, float* angles_out_dev, void* ws_dev,
                     double* out_host, void* stream);
/* compute_iid_metric(metric_name="psnr") (src/util/metric.py:263-338 as script/iid/eval.py:182-213 calls it) with ONE
 * synchronisation. pred_dev, gt_dev fp32 [3,HW]; mask_dev uint8 [3,HW] or NULL. transform: 0 none, 1 srgb2linear
 * (x ** 2.2), 2 linear2srgb (x ** (1 / 2.2)), applied to both first. align = 1 (shading, residual): least-squares scale
 * (compute_alignment_scale) and quantile_map, whose 0.9 quantile is an exact order statistic on the device.
 * out_host[5] = {psnr, lstsq_scale, quantile, quantile_scale, n} (the three alignment values NaN when align = 0). */
int mgb_eval_iid(const float* pred_dev, const float* gt_dev, const uint8_t* mask_dev, int64_t HW, int32_t align,
                 int32_t transform, void* ws_dev, double* out_host, void* stream);

/* ---- capacity ------------------------------------------------------------------------------- */
/* Bytes of the activation arena the handle holds for images of H x W with B members per batch. */
size_t mgb_workspace_bytes(mgb_handle* h, int32_t B, int32_t H, int32_t W);
/* Number of kernel launches enqueued by this library since creation (for bench.py gpu_launches). */
int64_t mgb_launch_count(void);

/* ---- operator-level entry points (layer parity tests; tests/test_ops_gpu.py) ---------------- */
/* D[M,N] = A[M,K] W[N,K]^T with the fused epilogue. A, W bf16 row-major (device). */
int mgb_op_linear(const void* a_bf16_dev, const void* w_bf16_dev, const float* bias_dev, const float* residual_dev,
                  float* out_f32_dev, void* out_bf16_dev, int32_t M, int32_t N, int32_t K, int32_t flags,
                  int32_t block_n, int32_t splits, int32_t stages, float* splitk_ws_dev, void* stream);
/* 3x3 / 1x1 convolution on NHWC bf16. kind: 0 = 3x3 stride 1 pad 1, 1 = 1x1, 2 = 3x3 stride 2 pad 1
 * (x is the 4-plane space-to-depth tensor), 3 = 3x3 stride 2 with pad (0,1,0,1) (VAE; same planes).
 * Hout, Wout: OUTPUT size. w_dev: bf16 [Cout, taps*Cin] tap-major. */
int mgb_op_conv2d(const void* x_bf16_dev, const void* w_bf16_dev, const float* bias_dev, const float* residual_dev,
                  float* out_f32_dev, void* out_bf16_dev, int32_t NB, int32_t Hout, int32_t Wout, int32_t Cin,
                  int32_t Cout, int32_t kind, int32_t flags, int32_t block_n, int32_t splits, int32_t stages,
                  float* splitk_ws_dev, void* stream);
/* Flash self-attention, head size 64 (replaces F.scaled_dot_product_attention under diffusers' Attention, reached
 * from marigold_depth_pipeline.py:461-463). qkv: [NB*T, 3C] (Q | K | V column blocks), out: [NB*T, C]. Long
 * sequences are split over KV ranges and merged by a second kernel; the operator-level entry point keeps the
 * split workspace in a process-wide buffer that it grows on demand (a synchronising cudaMalloc on first use or
 * growth) and is therefore not re-entrant across threads. The network path carves the workspace out of its arena. */
int mgb_op_flash_attn64(const void* qkv_bf16_dev, void* out_bf16_dev, int32_t NB, int32_t T, int32_t C, float scale,
                        void* stream);
/* GroupNorm (+SiLU) -> bf16, one launch with a grid-wide barrier, run-to-run deterministic (replaces torch.nn.GroupNorm
 * + F.silu under diffusers' ResnetBlock2D / Transformer2DModel, reached from marigold_depth_pipeline.py:461-463).
 * ws_dev: mgb_op_groupnorm_ws_bytes(NB, HW, C, G) bytes of scratch (0 = unsupported shape). */
size_t mgb_op_groupnorm_ws_bytes(int32_t NB, int32_t HW, int32_t C, int32_t G);
int mgb_op_groupnorm(const float* x_dev, void* y_bf16_dev, const float* gamma_dev, const float* beta_dev,
                     float* ws_dev, int32_t NB, int32_t HW, int32_t C, int32_t G, float eps, int32_t silu,
                     void* stream);
int mgb_op_layernorm(const float* x_dev, void* y_bf16_dev, const float* gamma_dev, const float* beta_dev, int32_t M,
                     int32_t C, float eps, void* stream);
/* attn2 of diffusers' BasicTransformerBlock against the FIXED two-token context CLIP(""), collapsed (marigold_depth_pipeline.py
 * :381-394,438-442,461-463), with the LayerNorm before it (norm2) and after it (norm3):
 *   z = LN2(x);  y = x + c1 + sum_h sigmoid(scale * z . G_h) U_h;  a = LN3(y)        (y, a stored as bf16)
 * GU_bf16_dev: [2][H][C] (G rows, then U rows) and c1_dev [C] are what mgb_set_text_embedding folds from to_q / to_k / to_v /
 * to_out and the text embedding. One launch; one warp per token, or four for C = 1280 with few tokens. */
int mgb_op_xattn2(const float* x_dev, void* y_bf16_dev, void* a_bf16_dev, const float* ln2_g_dev, const float* ln2_b_dev,
                  const float* ln3_g_dev, const float* ln3_b_dev, const void* GU_bf16_dev, const float* c1_dev, int32_t M,
                  int32_t C, int32_t H, float scale, float eps, void* stream);
int mgb_op_space_to_depth(const float* x_dev, void* y_bf16_dev, int32_t NB, int32_t H, int32_t W, int32_t C,
                          void* stream);
int mgb_op_upsample2x(const float* x_dev, void* y_bf16_dev, int32_t NB, int32_t H, int32_t W, int32_t C,
                      void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MARIGOLD_B200_H_ */
