// C ABI: error plumbing + operator-level entry points (layer parity tests call these).
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "kernels.h"
#include "ops.h"

namespace mgb {
static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }
}  // namespace mgb

using namespace mgb;

extern "C" {

const char* mgb_last_error(void) { return get_error(); }
const char* mgb_build_info(void) {
  return "libmarigold_b200 sm_100a: tcgen05.mma kind::f16 (bf16->fp32 TMEM), cp.async.bulk.tensor (TMA) SWIZZLE_128B, "
         "mbarrier pipelines; no CPU fallback";
}
int64_t mgb_launch_count(void) { return launch_count(); }
/* debug hook (not in the public header): per-CTA clock64 phase stamps of subsequent GEMM launches */
void mgb_debug_gemm_timing(void* dev_buffer) { set_gemm_debug_buffer(reinterpret_cast<long long*>(dev_buffer)); }

static void fill_epi(GemmEpilogue* e, const float* bias, const float* residual, float* out_f32, void* out_bf16,
                     int ldo, int flags) {
  memset(e, 0, sizeof(*e));
  e->bias = bias; e->residual = residual; e->out_f32 = out_f32;
  e->out_bf16 = reinterpret_cast<bf16*>(out_bf16);
  e->ldo = ldo; e->flags = flags; e->scale = 1.0f;
}

int mgb_op_linear(const void* a, const void* w, const float* bias, const float* residual, float* out_f32,
                  void* out_bf16, int32_t M, int32_t N, int32_t K, int32_t flags, int32_t block_n, int32_t splits,
                  int32_t stages, float* splitk_ws, void* stream) {
  if (!a || !w || (!out_f32 && !out_bf16)) { set_error("op_linear: null pointer"); return MGB_ERR_INVALID; }
  if (block_n <= 0) {
    int bn, sp, st;
    choose_tile((M + 127) / 128, N, K / 64, (flags & EPI_GEGLU) != 0, splitk_ws != nullptr && !(flags & EPI_GEGLU), &bn, &sp,
                &st);
    block_n = bn; if (splits <= 0) splits = sp; if (stages <= 0) stages = st;
  }
  if (splits <= 0) splits = 1;
  if (stages <= 0) stages = 4;
  GemmParams p;
  int rc = fill_linear_params(&p, reinterpret_cast<const bf16*>(a), reinterpret_cast<const bf16*>(w), M, N, K, block_n,
                              splits, stages);
  if (rc) return rc;
  fill_epi(&p.epi, bias, residual, out_f32, out_bf16, (flags & EPI_GEGLU) ? N / 2 : N, flags);
  return run_gemm(p, block_n, splitk_ws, reinterpret_cast<cudaStream_t>(stream));
}

int mgb_op_conv2d(const void* x, const void* w, const float* bias, const float* residual, float* out_f32,
                  void* out_bf16, int32_t NB, int32_t Hout, int32_t Wout, int32_t Cin, int32_t Cout, int32_t kind,
                  int32_t flags, int32_t block_n, int32_t splits, int32_t stages, float* splitk_ws, void* stream) {
  if (!x || !w || (!out_f32 && !out_bf16)) { set_error("op_conv2d: null pointer"); return MGB_ERR_INVALID; }
  const int taps = kind == 1 ? 1 : 9;
  if (block_n <= 0) {
    int tw, th;
    conv_tile_shape(Hout, Wout, &tw, &th, kind);
    const int m_tiles = NB * ((Wout + tw - 1) / tw) * ((Hout + th - 1) / th);
    int bn, sp, st;
    choose_tile(m_tiles, Cout, taps * Cin / 64, false, splitk_ws != nullptr, &bn, &sp, &st, conv_halo_ring_bytes(kind));
    block_n = bn; if (splits <= 0) splits = sp; if (stages <= 0) stages = st;
  }
  if (splits <= 0) splits = 1;
  if (stages <= 0) stages = 4;
  GemmParams p;
  int rc = fill_conv_params(&p, reinterpret_cast<const bf16*>(x), reinterpret_cast<const bf16*>(w), NB, Hout, Wout,
                            Cin, Cout, kind, block_n, splits, stages);
  if (rc) return rc;
  fill_epi(&p.epi, bias, residual, out_f32, out_bf16, Cout, flags);
  p.epi.hw = Hout * Wout;
  return run_gemm(p, block_n, splitk_ws, reinterpret_cast<cudaStream_t>(stream));
}

int mgb_op_flash_attn64(const void* qkv, void* out, int32_t NB, int32_t T, int32_t C, float scale, void* stream) {
  // split-KV workspace of the operator-level entry point: a process-wide buffer grown on demand (the network
  // path carves it out of its arena instead)
  static float* ws = nullptr;
  static size_t ws_bytes = 0;
  const size_t need = flash_attn64_ws_bytes(NB, T, C);
  if (need > ws_bytes) {
    cudaDeviceSynchronize();
    if (ws) cudaFree(ws);
    ws = nullptr; ws_bytes = 0;
    if (cudaMalloc(&ws, need) != cudaSuccess) { set_error("op_flash_attn64: workspace cudaMalloc(%zu) failed", need); return MGB_ERR_NOMEM; }
    ws_bytes = need;
  }
  int rc = launch_flash_attn64(reinterpret_cast<const bf16*>(qkv), reinterpret_cast<bf16*>(out), NB, T, C, scale,
                               need ? ws : nullptr, need ? ws_bytes : 0, reinterpret_cast<cudaStream_t>(stream));
  if (!rc) count_launch(need ? 2 : 1);
  return rc;
}

size_t mgb_op_groupnorm_ws_bytes(int32_t NB, int32_t HW, int32_t C, int32_t G) { return groupnorm_ws_bytes(NB, HW, C, G); }

int mgb_op_groupnorm(const float* x, void* y, const float* gamma, const float* beta, float* ws, int32_t NB, int32_t HW,
                     int32_t C, int32_t G, float eps, int32_t silu, void* stream) {
  int rc = launch_groupnorm(x, reinterpret_cast<bf16*>(y), nullptr, gamma, beta, ws, NB, HW, C, G, eps, silu,
                            reinterpret_cast<cudaStream_t>(stream));
  if (!rc) count_launch(2);
  return rc;
}

int mgb_op_layernorm(const float* x, void* y, const float* gamma, const float* beta, int32_t M, int32_t C, float eps,
                     void* stream) {
  int rc = launch_layernorm(x, reinterpret_cast<bf16*>(y), gamma, beta, M, C, eps,
                            reinterpret_cast<cudaStream_t>(stream));
  if (!rc) count_launch(1);
  return rc;
}

int mgb_op_xattn2(const float* x, void* y, void* a_out, const float* ln2_g, const float* ln2_b, const float* ln3_g,
                  const float* ln3_b, const void* GU, const float* c1, int32_t M, int32_t C, int32_t H, float scale, float eps,
                  void* stream) {
  if (!x || !y || !a_out || !GU || !c1) { set_error("op_xattn2: null pointer"); return MGB_ERR_INVALID; }
  int rc = launch_xattn2_fused(x, reinterpret_cast<bf16*>(y), reinterpret_cast<bf16*>(a_out), ln2_g, ln2_b, ln3_g, ln3_b,
                               reinterpret_cast<const bf16*>(GU), c1, M, C, H, scale, eps,
                               reinterpret_cast<cudaStream_t>(stream));
  if (!rc) count_launch(1);
  return rc;
}

/* ---- pre / post-processing and evaluation (image.cu, eval.cu) ---- */
int mgb_resize(const void* src, int32_t src_is_u8, int32_t NC, int32_t H, int32_t W, float* dst, int32_t h, int32_t w,
               int32_t mode, int32_t post, float* tmp, void* stream) {
  if (!src || !dst || !tmp) { set_error("mgb_resize: null pointer"); return MGB_ERR_INVALID; }
  int rc = launch_resize(src, src_is_u8, NC, H, W, dst, h, w, mode, post, tmp, reinterpret_cast<cudaStream_t>(stream));
  if (!rc) count_launch(2);
  return rc;
}

int mgb_colorize(const float* depth, int64_t HW, float dmin, float dmax, const uint8_t* lut, uint8_t* out_hwc, void* stream) {
  int rc = launch_colorize(depth, HW, dmin, dmax, lut, out_hwc, reinterpret_cast<cudaStream_t>(stream));
  if (!rc) count_launch(1);
  return rc;
}

size_t mgb_eval_ws_bytes(void) { return eval_ws_bytes() + 16 * sizeof(double); }

// copies n result doubles to the host and synchronises (the one synchronisation of each mgb_eval_* call)
static int eval_fetch(const char* what, double* out_host, const double* out_dev, int n, cudaStream_t s) {
  cudaError_t e = cudaMemcpyAsync(out_host, out_dev, n * sizeof(double), cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) { set_error("%s: %s", what, cudaGetErrorString(e)); return MGB_ERR_CUDA; }
  return MGB_OK;
}

int mgb_eval_depth(const float* pred, const float* gt, const uint8_t* mask, int64_t HW, int32_t alignment, float dmin,
                   float dmax, float* aligned_out, void* ws, double* out_host, void* stream) {
  if (!pred || !gt || !ws || !out_host || HW <= 0 || alignment < 0 || alignment > 2) {
    set_error("mgb_eval_depth: bad argument"); return MGB_ERR_INVALID;
  }
  double* out_dev = reinterpret_cast<double*>(static_cast<char*>(ws) + eval_ws_bytes());
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  int rc = launch_eval_depth(pred, gt, mask, HW, alignment, dmin, dmax, aligned_out, ws, out_dev, s);
  if (rc) return rc;
  count_launch(4);
  return eval_fetch("mgb_eval_depth", out_host, out_dev, 13, s);
}

int mgb_eval_normals(const float* pred, const float* gt, int64_t HW, float* angles_out, void* ws, double* out_host,
                     void* stream) {
  if (!pred || !gt || !ws || !out_host || HW <= 0) { set_error("mgb_eval_normals: bad argument"); return MGB_ERR_INVALID; }
  double* out_dev = reinterpret_cast<double*>(static_cast<char*>(ws) + eval_ws_bytes());
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  int rc = launch_eval_normals(pred, gt, HW, angles_out, ws, out_dev, s);
  if (rc) return rc;
  count_launch(11);                                  // memset, sums, count, 3 x (histogram + pick), above, final
  return eval_fetch("mgb_eval_normals", out_host, out_dev, 9, s);
}

int mgb_eval_iid(const float* pred, const float* gt, const uint8_t* mask, int64_t HW, int32_t align, int32_t transform,
                 void* ws, double* out_host, void* stream) {
  if (!pred || !gt || !ws || !out_host || HW <= 0 || transform < 0 || transform > 2) {
    set_error("mgb_eval_iid: bad argument"); return MGB_ERR_INVALID;
  }
  double* out_dev = reinterpret_cast<double*>(static_cast<char*>(ws) + eval_ws_bytes());
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  int rc = launch_eval_iid(pred, gt, mask, HW, align != 0, transform, ws, out_dev, s);
  if (rc) return rc;
  count_launch(align ? 12 : 2);                      // [memset, sums, solve, 7 selection, quantile], psnr sums, final
  return eval_fetch("mgb_eval_iid", out_host, out_dev, 5, s);
}

int mgb_op_space_to_depth(const float* x, void* y, int32_t NB, int32_t H, int32_t W, int32_t C, void* stream) {
  int rc = launch_space_to_depth(x, reinterpret_cast<bf16*>(y), NB, H, W, C, reinterpret_cast<cudaStream_t>(stream));
  if (!rc) count_launch(1);
  return rc;
}

int mgb_op_upsample2x(const float* x, void* y, int32_t NB, int32_t H, int32_t W, int32_t C, void* stream) {
  int rc = launch_upsample2x(x, reinterpret_cast<bf16*>(y), NB, H, W, C, 2 * H, 2 * W, reinterpret_cast<cudaStream_t>(stream));
  if (!rc) count_launch(1);
  return rc;
}

}  // extern "C"
