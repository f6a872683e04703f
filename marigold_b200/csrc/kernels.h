// Host-visible declarations of every kernel launcher in libmarigold_b200. Plain C++ (no torch).
// Tensors are NHWC ("tokens x channels") inside the library; NCHW only exists at the C ABI.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/marigold_b200.h"

namespace mgb {

typedef __nv_bfloat16 bf16;

// error plumbing (api.cu)
void set_error(const char* fmt, ...);
const char* get_error();

// ---------------------------------------------------------------------------------------------
// tcgen05 GEMM / implicit-GEMM convolution
//   D[M, N] = A[M, K] * B[N, K]^T   (A, B bf16 K-major; fp32 accumulation in TMEM)
// ---------------------------------------------------------------------------------------------
enum : int {
  EPI_GEGLU = 1,        // acc tile = [value | gate] halves; out = (v + bv) * gelu_erf(g + bg)
  EPI_SCHED = 2,        // out_f32 = kx * sched_x + kv * (acc + bias) + kz * sched_z   (conv_out + DDIM/LCM step)
  EPI_DEPTH = 4,        // N == 3: out_f32[img, h, w] = (clip(mean_c, -1, 1) + 1) / 2              (NCHW, 1 plane)
  EPI_NORMALS = 8,      // N == 3: clip to [-1, 1], divide by max(||.||, 1e-6); out_f32 NCHW, 3 planes
  EPI_NCHW = 16,        // out_f32 written as NCHW planes [img, c, h*w] (needs hw)
  EPI_SILU = 32,        // out = silu(acc + bias)
  EPI_SCALE = 64,       // acc *= scale before bias (used for attention-score GEMMs)
  EPI_UNIT = 128,       // with EPI_NCHW: out = (clip(v, -1, 1) + 1) / 2                     (IID decode head)
};

struct GemmEpilogue {
  const float* bias;      // [N] in accumulator-column order, or nullptr
  const float* residual;  // fp32 [M, ldo] added after activation, or nullptr
  float* out_f32;         // fp32 [M, ldo] or nullptr
  bf16* out_bf16;         // bf16 [M, ldo] or nullptr
  int ldo;                // row stride of residual / outputs (elements)
  int flags;
  int hw;                 // pixels per image (EPI_NCHW / EPI_DEPTH / EPI_NORMALS)
  float scale;            // EPI_SCALE
  const float* sched_x;   // EPI_SCHED: current latent  [M, ldo]
  const float* sched_z;   // EPI_SCHED: fresh noise     [M, ldo] or nullptr
  const float* sched_k;   // EPI_SCHED: device pointer to {kx, kv, kz}
  float* aux_out;         // EPI_SCHED: optional raw model output (acc + bias) [M, ldo], or nullptr
};

struct GemmParams {
  CUtensorMap tmap_a;  // mode 0: 2D {K, M}; mode 1: 5D {C, W, H, P, NB}
  CUtensorMap tmap_b;  // 2D {K, N}
  CUtensorMap tmap_a2; // mode 0, optional: 2D {K2, M}, A = [A1 | A2] along K. Mode 1, optional second A operand: 5D {C2, W, H, 1, NB} of a 1x1 convolution over the same output
                       // pixels whose K blocks follow the 3x3 taps (K concatenation: a ResnetBlock's conv2 + conv_shortcut
                       // as ONE implicit GEMM with weights [W2 | Wsc])
  int mode;            // 0 = row-major activations, 1 = implicit conv (one A tile per tap), 2 = implicit 3x3 conv
                       // whose 9 taps read ONE shared-memory halo per channel block (see gemm_tc.cu)
  int M, N;            // logical GEMM rows / accumulator columns
  int num_kb;          // total K blocks of 64
  int num_kb1;         // K blocks of the first A operand (== num_kb without tmap_a2)
  int kb_per_split;    // K blocks per blockIdx.z
  int stages;          // smem pipeline depth
  // conv geometry (mode 1)
  int H, W;            // OUTPUT image size
  int tile_w, tile_h;  // tile_w * tile_h == 128, tile_w a power of two
  int tile_w_shift;    // log2(tile_w)
  int tiles_x, tiles_y;
  int cblocks;         // Cin / 64
  int ntaps;
  int8_t tap_p[12], tap_dy[12], tap_dx[12];
  // mode 2: halo geometry. halo_copies == 1: one (tile_h+2) x (tile_w+2) pixel box, taps address it at a
  // 128 B-granular offset; halo_copies == 3: three (tile_h+2) x tile_w boxes (dx = -1, 0, +1), taps only shift
  // by whole rows (1024 B-aligned operand starts).
  int halo_w, halo_copies, halo_copy_bytes, halo_slot_bytes, halo_slots, halo_base_off;
  float* partial;      // split-K: fp32 [splits, M, N] raw accumulators (epilogue deferred)
  long long* dbg;      // optional per-CTA phase timestamps [ctas][8] (tools/gemm_phases.py), else nullptr
  GemmEpilogue epi;
};

// Launch. block_n in {16, 32, 64, 128, 160, 256}; ctas_per_sm 1 or 2 (2: p.stages must keep gemm_smem_bytes <= 113 KB,
// block_n >= 64). Returns cudaError_t as int.
int launch_gemm_tc(const GemmParams& p, int block_n, int splits, int ctas_per_sm, cudaStream_t stream);
void set_gemm_debug_buffer(long long* dev_ptr);  // debug hook: phase timestamps of subsequent launches
// Deferred epilogue for split-K: sums `splits` partials and applies p.epi.
int launch_splitk_epilogue(const GemmParams& p, int block_n, int splits, cudaStream_t stream);
size_t gemm_smem_bytes(int block_n, int stages, int a_ring_bytes = -1 /* -1: stages x 16 KB A tiles */);

// Tensor-map helpers (driver entry point fetched through the runtime; no -lcuda needed).
int make_tmap_2d(CUtensorMap* out, const void* base, uint64_t inner, uint64_t outer, uint64_t row_stride_bytes,
                 uint32_t box_inner, uint32_t box_outer);
int make_tmap_3d(CUtensorMap* out, const void* base, const uint64_t dims[3], const uint64_t strides_bytes[2],
                 const uint32_t box[3]);
int make_tmap_5d(CUtensorMap* out, const void* base, const uint64_t dims[5], const uint64_t strides_bytes[4],
                 const uint32_t box[5]);

// ---------------------------------------------------------------------------------------------
// Flash self-attention, head_dim 64 (attn_tc.cu)
//   qkv: bf16 [NB * T, 3 * C] (Q | K | V blocks, head h at columns h*64..), out: bf16 [NB * T, C]
// ---------------------------------------------------------------------------------------------
// ws (optional): split-KV workspace of flash_attn64_ws_bytes(); without it the kernel runs unsplit.
int launch_flash_attn64(const bf16* qkv, bf16* out, int NB, int T, int C, float scale, float* ws, size_t ws_bytes,
                        cudaStream_t stream);
int flash_attn64_splits(int NB, int T, int C);
size_t flash_attn64_ws_bytes(int NB, int T, int C);

// ---------------------------------------------------------------------------------------------
// Memory-bound kernels (norm.cu, elementwise.cu)
// ---------------------------------------------------------------------------------------------
// GroupNorm over NHWC: stats over (pixels x C/G channels) per image and group; ONE launch with a grid barrier,
// run-to-run deterministic (norm.cu).
//   x_f32 [NB, HW, C] -> y_bf16 = act((x - mean) * rstd * gamma + beta); optional raw bf16 copy.
// ws: groupnorm_ws_bytes() of scratch.
int launch_groupnorm(const float* x, bf16* y, bf16* raw_copy, const float* gamma, const float* beta, float* ws,
                     int NB, int HW, int C, int G, float eps, int silu, cudaStream_t stream);
size_t groupnorm_ws_bytes(int NB, int HW, int C, int G);
size_t groupnorm_part_bytes(int NB, int HW, int C, int G);
// GroupNorm(+SiLU) over the channel concat [a | b] (b optional): y bf16 [NB, HW, Ca + Cb]; optional raw bf16 copy of
// the concat. part: groupnorm_part_bytes(NB, HW, Ca + Cb, G) of scratch; counters: NB unsigned, zero on entry.
int launch_gn_fused(const float* xa, int Ca, const float* xb, int Cb, bf16* y, bf16* raw_copy, const float* gamma,
                    const float* beta, int NB, int HW, int G, float eps, int silu, void* part, unsigned* counters,
                    cudaStream_t stream);
// LayerNorm over the channel dim: x_f32 [M, C] -> y_bf16 [M, C]
int launch_layernorm(const float* x, bf16* y, const float* gamma, const float* beta, int M, int C, float eps,
                     cudaStream_t stream);
// Collapsed cross attention against the fixed 2-token context, fused with norm2 and norm3 (norm.cu):
//   y = bf16(x + c1 + sum_h sigmoid(scale * LN2(x) . G_h) U_h) ;  a_out = bf16(LN3(y in fp32))
int launch_xattn2_fused(const float* x, bf16* y, bf16* a_out, const float* g2, const float* b2, const float* g3,
                        const float* b3, const bf16* GU, const float* c1, int M, int C, int H, float scale, float eps,
                        cudaStream_t stream);
int launch_xattn2_fold(const float* wq, const float* wo, const float* bo, const float* kv, bf16* GU, float* c1, int C,
                       cudaStream_t stream);
// y[NB, 4, ceil(H/2), ceil(W/2), C] (parity planes p = (h&1)*2 + (w&1), zero where the source pixel does not exist) from
// x fp32 [NB, H, W, C]
int launch_space_to_depth(const float* x, bf16* y, int NB, int H, int W, int C, cudaStream_t stream);
// nearest upsampling: x fp32 [NB, H, W, C] -> y bf16 [NB, Ho, Wo, C], Ho in {2H - 1, 2H}, Wo in {2W - 1, 2W}
int launch_upsample2x(const float* x, bf16* y, int NB, int H, int W, int C, int Ho, int Wo, cudaStream_t stream);
// channel concat (fp32): out[M, Ca + Cb] = [a | b]
int launch_concat(const float* a, const float* b, float* out, int M, int Ca, int Cb, cudaStream_t stream);
// fp32 -> bf16 cast
int launch_cast_bf16(const float* x, bf16* y, size_t n, cudaStream_t stream);
// UNet conv_in operand: [rgb(4) | target(Ct) | zeros] bf16 NHWC-64 from the fp32 NHWC latents (Ct = 4, or 4 n for IID)
int launch_pack_latents(const float* rgb, const float* tgt, bf16* out, int M, int Ct, cudaStream_t stream);
// NCHW fp32 <-> NHWC fp32 (small tensors at the ABI)
int launch_nchw_to_nhwc(const float* x, float* y, int NB, int C, int HW, float scale, cudaStream_t stream);
int launch_nhwc_to_nchw(const float* x, float* y, int NB, int C, int HW, float scale, cudaStream_t stream);
// rgb [NB,3,H,W] (fp32, already in [-1,1]) -> bf16 NHWC with 64 channels (3 real + zero padding)
int launch_pack_rgb(const float* rgb_nchw, bf16* out, int NB, int HW, cudaStream_t stream);
// decoder input: post_quant_conv(latent / scale) -> bf16 NHWC-64; latent fp32 NCHW [NB,4,HW]; w fp32 [4,4]
int launch_pack_decoder_latent(const float* latent_nchw, const float* w, const float* b, float inv_scale, bf16* out,
                               int NB, int HW, cudaStream_t stream);
// Per-step table selection: cur_bias <- bias_table[i], cur_k <- sched_k[i], with i = step (>= 0) or *counter (< 0).
int launch_select_step(const float* bias_table, int bias_total, const float* sched_k, float* cur_bias, float* cur_k,
                       const int* counter, int step, cudaStream_t stream);
int launch_advance_counter(int* counter, cudaStream_t stream);
// One-time fp32 product P = A[M,K] B[K,N], stored as bf16 at out[m * ldo + col0 + n] (weight folding at finalize)
int launch_fold_matmul(const float* A, const float* B, bf16* out, int M, int N, int K, int ldo, int col0, cudaStream_t stream);
// Tiny dense layer for M <= 16 rows (time MLP, text K/V): y[M,N] = act(x[M,K]) W[N,K]^T + b ; fp32
int launch_linear_small(const float* x, const float* w, const float* b, float* y, int M, int N, int K,
                        int silu_in, int silu_out, cudaStream_t stream);
// sinusoidal timestep embedding (flip_sin_to_cos, shift 0): t[M] -> emb[M, dim] = [cos | sin]
int launch_timestep_embedding(const float* t, float* emb, int M, int dim, cudaStream_t stream);
// row softmax: fp32 scores s[M, ld] (first n valid) -> bf16 p[M, ld] with columns [n, ld) zeroed
int launch_softmax_rows(const float* s, bf16* p, int M, int n, int ld, cudaStream_t stream);
// x bf16 [M, N] -> y bf16 [N, ld] (columns [M, ld) zeroed)
int launch_transpose_bf16(const bf16* x, bf16* y, int M, int N, int ld, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// Pre / post-processing bookends (image.cu) and the evaluation step (eval.cu)
// ---------------------------------------------------------------------------------------------
// src [NC, H, W] (u8 or f32) -> dst f32 [NC, h, w]; tmp: NC * H * w floats. mode 0 bilinear-aa, 1 bicubic-aa, 2 nearest-exact;
// post 0 none, 1 round + clamp to [0, 255], 2 that and then x / 255 * 2 - 1
int launch_resize(const void* src, int src_is_u8, int NC, int H, int W, float* dst, int h, int w, int mode, int post, float* tmp,
                  cudaStream_t stream);
int launch_colorize(const float* depth, long long HW, float dmin, float dmax, const uint8_t* lut, uint8_t* out,
                    cudaStream_t stream);
size_t eval_ws_bytes();
// alignment 0 none, 1 least squares in depth, 2 least squares in disparity; out_dev: 13 doubles
int launch_eval_depth(const float* pred, const float* gt, const uint8_t* mask, long long HW, int alignment, float dmin, float dmax,
                      float* aligned_out, void* ws, double* out_dev, cudaStream_t stream);
// pred, gt [3, HW]; angles_out [HW] or null; out_dev: 9 doubles {n_valid, mean, median, rmse, sub5 .. sub30}
int launch_eval_normals(const float* pred, const float* gt, long long HW, float* angles_out, void* ws, double* out_dev,
                        cudaStream_t stream);
// pred, gt, mask (or null) [3, HW]; transform 0 / 1 / 2 (none, ** 2.2, ** (1 / 2.2)); out_dev: 5 doubles
// {psnr, lstsq_scale, quantile, quantile_scale, n}
int launch_eval_iid(const float* pred, const float* gt, const uint8_t* mask, long long HW, int align, int transform, void* ws,
                    double* out_dev, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// Ensemble kernels (ensemble.cu)
// ---------------------------------------------------------------------------------------------
size_t ens_ws_bytes();
int ens_max_batch();     // parameter sets per launch_ens_depth_cost call
int ens_max_members();   // largest supported ensemble size
// st_host (pinned): float [P][2E] = {s_0..s_{E-1}, t_0..t_{E-1}} per parameter set; out_host_pinned: double [P][3] =
// {cost, min(pred), max(pred)}; one synchronisation per call. *launches = kernels launched.
int launch_ens_depth_cost(const float* depth, const float* st_host, int P, int E, long long HW, int shift, int median,
                          double reg, void* ws, double* out_host_pinned, int* launches, cudaStream_t stream);
// One forward-difference gradient: st_host (pinned) float [4E] = base {s | t}, perturbed {s' | t'}; out double [1 + n][3]
int launch_ens_depth_cost_fd(const float* depth, const float* st_host, int E, long long HW, int shift, int median,
                             double reg, void* ws, float* v3, double* out_host_pinned, int* launches, cudaStream_t stream);
int launch_ens_minmax(const float* depth, int E, long long HW, float* ws, float* host_pinned, int* blocks_out,
                      cudaStream_t stream);
int launch_ens_depth_reduce(const float* depth, const float* st_host, int E, long long HW, int shift, int median,
                            int use_min, float* pred, float* unc, int* idx, void* ws, cudaStream_t stream);
// ensemble_iid: x [E, N] -> pred [N] (median | mean), unc [N] or null (MAD | unbiased std)
int launch_ens_iid(const float* x, int E, long long N, int median, float* pred, float* unc, cudaStream_t stream);
int launch_ens_normals(const float* nrm, int E, long long HW, int closest, float* out, float* unc, int* idx,
                       cudaStream_t stream);

}  // namespace mgb
