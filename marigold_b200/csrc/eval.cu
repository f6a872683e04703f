// Device-side evaluation step that follows the hot path in dataset evaluation (SURVEY.md 8f-4), for the three tasks.
//
// Depth: least-squares scale / shift alignment of a prediction to the ground truth over the valid pixels (reference
// src/util/alignment.py:35-82), in depth or in disparity (script/depth/eval.py:179-199), and the masked depth metrics
// (src/util/metric.py:64-191) in two streaming passes and ONE host synchronisation per sample (the reference does a
// numpy lstsq on the host and one `.item()` per metric).
//   pass 1  sums n, sum p, sum p^2, sum g, sum p g over the fit mask (double) -> scale, shift from the 2 x 2 normal
//           equations; in disparity mode g = 1 / gt and the fit mask also needs gt > 0 and p > 0
//   pass 2  aligned = clip(clip(p * scale + shift, dmin, dmax), 1e-6) (script/depth/eval.py:201-207), in disparity mode
//           after 1 / clip(p * scale + shift, 1e-3), and the sums of every metric; a last block turns them into values.
//   HBM-bound: 9 bytes / pixel / pass (pred f32, gt f32, mask u8).
//
// Normals: compute_cosine_error(masked=True) and the angular metrics (src/util/metric.py:194-257). One pass writes the
// angle map and sums mean / rmse / threshold counts; the median is an exact order statistic (below). 24 B / pixel / pass.
//
// IID: compute_iid_metric's PSNR (src/util/metric.py:263-338): colour transform, least-squares scale, the 0.9 quantile of
// the ground truth's brightness (an exact order statistic again), quantile map, masked PSNR. 27 B / pixel / pass.
//
// Exact order statistic: the values of ranks k and k + 1 of a float array that a functor computes on the fly (angles,
// brightness) without storing it. The values are finite and >= 0, so their bit patterns sort as unsigned integers: a
// radix select over 11 / 11 / 10 bits, one histogram pass per digit (per-block shared-memory histograms merged with
// integer atomics, so the counts are order-independent) and a one-warp kernel that picks the bin and keeps the prefix in
// device memory. Rank k + 1 is the same value when the last bin holds it, else the smallest value above the prefix (one
// more pass, skipped on the device when not needed). The workspace does not grow with the image.
#include <cfloat>

#include "common.cuh"
#include "kernels.h"

namespace mgb {

constexpr int kEvThreads = 256;
constexpr int kEvBlocks = 148 * 2;
constexpr int kEvSums = 12;

__device__ __forceinline__ void block_reduce_store(double (&v)[kEvSums], int n, double* __restrict__ out) {
  __shared__ double sh[kEvThreads / 32][kEvSums];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int k = 0; k < n; ++k) {
    double d = v[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
    if (lane == 0) sh[warp][k] = d;
  }
  __syncthreads();
  if (threadIdx.x < n) {
    double t = 0.0;
    for (int w = 0; w < kEvThreads / 32; ++w) t += sh[w][threadIdx.x];
    out[(size_t)blockIdx.x * kEvSums + threadIdx.x] = t;
  }
}

__global__ void __launch_bounds__(kEvThreads)
    eval_align_sums_kernel(const float* __restrict__ pred, const float* __restrict__ gt, const uint8_t* __restrict__ mask,
                           long long HW, int disparity, double* __restrict__ part) {
  double v[kEvSums] = {0};
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < HW; p += (long long)gridDim.x * blockDim.x) {
    if (mask && !mask[p]) continue;
    const double a = pred[p];
    double g = gt[p];
    if (disparity) {                  // depth2disparity (alignment.py:85-95): fit over mask & gt > 0 & pred > 0
      if (!(gt[p] > 0.f) || !(pred[p] > 0.f)) continue;
      g = double(__fdiv_rn(1.f, gt[p]));
    }
    v[0] += 1.0; v[1] += a; v[2] += a * a; v[3] += g; v[4] += a * g;
  }
  block_reduce_store(v, 5, part);
}

// scale, shift of min || [p 1] [s t]^T - g ||^2 over the valid pixels (np.linalg.lstsq in alignment.py:66-69)
// Sum of quantity k over the blocks' partials by one warp: lane l takes blocks l, l + 32, ... (independent loads), xor tree.
// (A single thread walking 296 x 12 dependent loads took 100 us.)
__device__ __forceinline__ double warp_sum_partials(const double* __restrict__ part, int nblocks, int k) {
  double t = 0.0;
  for (int b = threadIdx.x & 31; b < nblocks; b += 32) t += part[(size_t)b * kEvSums + k];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  return t;
}

// alignment: 0 none, 1 least squares in depth, 2 least squares in disparity
__global__ void eval_align_solve_kernel(const double* __restrict__ part, int nblocks, int alignment, double* __restrict__ st) {
  double s[5];
  for (int k = 0; k < 5; ++k) s[k] = warp_sum_partials(part, nblocks, k);
  if (threadIdx.x != 0) return;
  double scale = 1.0, shift = 0.0;
  if (alignment == 2 && s[0] == 0) {
    scale = 0.0;                      // lstsq of an empty system: the minimum-norm solution 0
  } else if (alignment) {
    const double n = s[0], sp = s[1], spp = s[2], sg = s[3], spg = s[4];
    const double det = n * spp - sp * sp;
    if (n > 0 && fabs(det) > 1e-300) {
      scale = (n * spg - sp * sg) / det;
      shift = (spp * sg - sp * spg) / det;
    } else if (n > 0) {               // constant prediction: lstsq's minimum-norm solution of the rank-1 system
      const double m = sp / n, gm = sg / n;
      scale = gm * m / (m * m + 1.0);
      shift = gm / (m * m + 1.0);
    }
  }
  st[0] = scale; st[1] = shift; st[2] = s[0];
}

__global__ void __launch_bounds__(kEvThreads)
    eval_metric_sums_kernel(const float* __restrict__ pred, const float* __restrict__ gt, const uint8_t* __restrict__ mask,
                            long long HW, const double* __restrict__ st, int disparity, float dmin, float dmax,
                            float* __restrict__ aligned_out, double* __restrict__ part) {
  // numpy: float32 pred * float64 scale + float64 shift is float64, and torch promotes the float64 prediction against the
  // float32 ground truth (script/depth/eval.py:177-213), so the reference's metric arithmetic is double: so is this
  const double scale = st[0], shift = st[1];
  double v[kEvSums] = {0};
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < HW; p += (long long)gridDim.x * blockDim.x) {
    double a = double(pred[p]) * scale + shift;
    if (disparity) a = 1.0 / fmax(a, 1e-3);           // eval.py:196-199: clip the disparity to >= 1e-3, back to depth
    a = fmin(fmax(a, double(dmin)), double(dmax));
    a = fmax(a, 1e-6);
    if (aligned_out) aligned_out[p] = float(a);
    if (mask && !mask[p]) continue;
    const double g = double(gt[p]);
    const double diff = a - g;
    const double dl = log(a) - log(g);
    const double r = fmax(a / g, g / a);
    const double di = 1.0 / a - 1.0 / g;
    v[0] += 1.0;
    v[1] += fabs(diff) / g;                               // abs_relative_difference
    v[2] += diff * diff / g;                              // squared_relative_difference
    v[3] += diff * diff;                                  // rmse_linear
    v[4] += dl * dl;                                      // rmse_log / silog first term
    v[5] += dl;                                           // silog second term
    v[6] += fabs(log10(a) - log10(g));                    // log10
    v[7] += r < 1.25 ? 1.0 : 0.0;                         // delta1
    v[8] += r < 1.25 * 1.25 ? 1.0 : 0.0;                  // delta2
    v[9] += r < 1.25 * 1.25 * 1.25 ? 1.0 : 0.0;           // delta3
    v[10] += di * di;                                     // i_rmse
  }
  block_reduce_store(v, 11, part);
}

__global__ void eval_metric_final_kernel(const double* __restrict__ part, int nblocks, const double* __restrict__ st,
                                         double* __restrict__ out) {
  double s[kEvSums] = {0};
  for (int k = 0; k < 11; ++k) s[k] = warp_sum_partials(part, nblocks, k);
  if (threadIdx.x != 0) return;
  const double n = s[0] > 0 ? s[0] : 1.0;
  out[0] = st[0]; out[1] = st[1]; out[2] = s[0];
  out[3] = s[1] / n;                                     // abs_relative_difference
  out[4] = s[2] / n;                                     // squared_relative_difference
  out[5] = sqrt(s[3] / n);                               // rmse_linear
  out[6] = sqrt(s[4] / n);                               // rmse_log
  out[7] = s[6] / n;                                     // log10
  out[8] = s[7] / n; out[9] = s[8] / n; out[10] = s[9] / n;   // delta1..3
  out[11] = sqrt(s[10] / n);                             // i_rmse
  const double t = s[4] / n - (s[5] * s[5]) / (n * n);
  out[12] = sqrt(t > 0 ? t : 0.0) * 100.0;               // silog_rmse
}


// alignment 0 / 1 / 2 (none, depth, disparity); out_dev: 13 doubles {scale, shift, n_valid, abs_rel, sq_rel, rmse, rmse_log, log10, delta1, delta2, delta3, i_rmse, silog}
int launch_eval_depth(const float* pred, const float* gt, const uint8_t* mask, long long HW, int alignment, float dmin, float dmax,
                      float* aligned_out, void* ws, double* out_dev, cudaStream_t stream) {
  double* part = static_cast<double*>(ws);
  double* st = part + size_t(kEvBlocks) * kEvSums;
  const int blocks = int(std::min<long long>((HW + kEvThreads - 1) / kEvThreads, kEvBlocks));
  const int disp = alignment == 2;
  eval_align_sums_kernel<<<blocks, kEvThreads, 0, stream>>>(pred, gt, mask, HW, disp, part);
  eval_align_solve_kernel<<<1, 32, 0, stream>>>(part, blocks, alignment, st);
  eval_metric_sums_kernel<<<blocks, kEvThreads, 0, stream>>>(pred, gt, mask, HW, st, disp, dmin, dmax, aligned_out, part);
  eval_metric_final_kernel<<<1, 32, 0, stream>>>(part, blocks, st, out_dev);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("eval_depth launch: %s", cudaGetErrorString(e)); return MGB_ERR_CUDA; }
  return MGB_OK;
}


// ---------------------------------------------------------------------------------------------
// Exact order statistic (radix select over the bits of non-negative finite floats)
// ---------------------------------------------------------------------------------------------
constexpr int kSelBins = 2048;                                   // 11-bit digits; the last pass uses 1024 of them
__host__ __device__ constexpr int sel_shift(int pass) { return pass == 0 ? 21 : pass == 1 ? 10 : 0; }
__host__ __device__ constexpr int sel_bins(int pass) { return pass < 2 ? 2048 : 1024; }

struct SelState {                        // zeroed before every selection; lives in the eval workspace
  unsigned long long hist[3][kSelBins];  // global histogram of each digit pass
  unsigned long long n;                  // size of the set (written by the kernel that counts it)
  unsigned long long k;                  // wanted rank (0-based); ranks k and k + 1 are returned
  unsigned long long krem;               // rank of the wanted value among the values that share the prefix so far
  unsigned prefix;                       // bits of the rank-k value fixed so far
  unsigned above_inv;                    // ~(smallest value > rank-k value), by atomicMax (0: none seen)
  int need_above;                        // rank k + 1 lies past the run of values equal to rank k
  int pad;
};

size_t eval_ws_bytes() {
  return size_t(kEvBlocks) * kEvSums * sizeof(double) + 16 * sizeof(double) + 64 + sizeof(SelState);
}
__host__ __device__ inline SelState* sel_state(void* ws) {
  return reinterpret_cast<SelState*>(static_cast<char*>(ws) + size_t(kEvBlocks) * kEvSums * sizeof(double) +
                                     16 * sizeof(double) + 64);
}

// -0 sorts with +0
__device__ __forceinline__ unsigned sel_key(float v) { return v == 0.f ? 0u : __float_as_uint(v); }

// One digit pass: the values whose higher digits equal the prefix are counted by their digit at `pass`.
template <class F>
__global__ void __launch_bounds__(kEvThreads) sel_hist_kernel(F f, long long n_items, SelState* __restrict__ st, int pass) {
  __shared__ unsigned h[kSelBins];
  if (st->n == 0) return;
  const int nb = sel_bins(pass), sh = sel_shift(pass);
  for (int i = threadIdx.x; i < nb; i += blockDim.x) h[i] = 0;
  __syncthreads();
  const unsigned hi_shift = sel_shift(pass - 1 < 0 ? 0 : pass - 1);
  const unsigned want = st->prefix;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_items; i += (long long)gridDim.x * blockDim.x) {
    float v;
    if (!f(i, v)) continue;
    const unsigned u = sel_key(v);
    if (pass > 0 && (u >> hi_shift) != (want >> hi_shift)) continue;
    atomicAdd(&h[(u >> sh) & unsigned(nb - 1)], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nb; i += blockDim.x)
    if (h[i]) atomicAdd(&st->hist[pass][i], (unsigned long long)h[i]);
}

// One warp: the bin of this pass that holds rank krem; the prefix and the remaining rank move to it.
__global__ void sel_pick_kernel(SelState* __restrict__ st, int pass) {
  if (st->n == 0) return;
  const int lane = threadIdx.x & 31, nb = sel_bins(pass), per = nb / 32;
  const unsigned long long* h = st->hist[pass];
  unsigned long long mine = 0;
  for (int b = 0; b < per; ++b) mine += h[lane * per + b];
  unsigned long long incl = mine;                                  // inclusive scan over the lanes' bin groups
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const unsigned long long krem = st->krem, excl = incl - mine;
  const unsigned owner = __ballot_sync(0xffffffffu, excl <= krem && krem < incl);
  if (owner == 0 || lane != __ffs(owner) - 1) return;              // owner == 0 only if the counts are inconsistent
  unsigned long long c = excl;
  int b = lane * per;
  for (; b < lane * per + per - 1 && c + h[b] <= krem; ++b) c += h[b];
  st->prefix |= unsigned(b) << sel_shift(pass);
  st->krem = krem - c;
  if (pass == 2) st->need_above = st->krem + 1 >= h[b];           // rank k + 1 is not in the equal run
}

// Smallest value above the rank-k value (only when rank k + 1 is not equal to it).
template <class F>
__global__ void __launch_bounds__(kEvThreads) sel_above_kernel(F f, long long n_items, SelState* __restrict__ st) {
  if (st->n == 0 || !st->need_above) return;
  const unsigned vk = st->prefix;
  unsigned best = 0;                                               // max of ~u == ~min of u
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_items; i += (long long)gridDim.x * blockDim.x) {
    float v;
    if (!f(i, v)) continue;
    const unsigned u = sel_key(v);
    if (u > vk) best = max(best, ~u);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
  if ((threadIdx.x & 31) == 0 && best) atomicMax(&st->above_inv, best);
}

// Ranks k and k + 1 after the passes (k + 1 past the end of the set returns rank k twice).
__device__ __forceinline__ void sel_result(const SelState* st, float* vk, float* vk1) {
  *vk = __uint_as_float(st->prefix);
  *vk1 = (st->need_above && st->above_inv) ? __uint_as_float(~st->above_inv) : *vk;
}

// The passes of one selection. st->n and st->k must be set on the device before the first pass (by a kernel on the same
// stream); st->krem starts equal to k. 7 launches.
template <class F>
void launch_select(F f, long long n_items, SelState* st, int blocks, cudaStream_t stream) {
  for (int pass = 0; pass < 3; ++pass) {
    sel_hist_kernel<F><<<blocks, kEvThreads, 0, stream>>>(f, n_items, st, pass);
    sel_pick_kernel<<<1, 32, 0, stream>>>(st, pass);
  }
  sel_above_kernel<F><<<blocks, kEvThreads, 0, stream>>>(f, n_items, st);
}

// ---------------------------------------------------------------------------------------------
// Normals: compute_cosine_error(masked=True) + mean / median / rmse / sub-threshold angular errors
// ---------------------------------------------------------------------------------------------
// Angle in degrees between pred and gt at pixel i, as torch.cosine_similarity and metric.py:211-213 compute it in float32:
// each vector divided by max(||.||, 1e-8), the dot product, clamp to [-1, 1], acos * 180 / pi. False where ||gt|| == 0.
struct NormalsAngle {
  const float* __restrict__ pred;
  const float* __restrict__ gt;
  long long HW;
  __device__ __forceinline__ bool operator()(long long i, float& ang) const {
    const float g0 = gt[i], g1 = gt[HW + i], g2 = gt[2 * HW + i];
    const float gg = __fadd_rn(__fadd_rn(__fmul_rn(g0, g0), __fmul_rn(g1, g1)), __fmul_rn(g2, g2));
    if (!(gg > 0.f)) return false;
    const float p0 = pred[i], p1 = pred[HW + i], p2 = pred[2 * HW + i];
    const float pp = __fadd_rn(__fadd_rn(__fmul_rn(p0, p0), __fmul_rn(p1, p1)), __fmul_rn(p2, p2));
    const float gn = fmaxf(__fsqrt_rn(gg), 1e-8f), pn = fmaxf(__fsqrt_rn(pp), 1e-8f);
    float c = __fadd_rn(__fadd_rn(__fmul_rn(__fdiv_rn(p0, pn), __fdiv_rn(g0, gn)), __fmul_rn(__fdiv_rn(p1, pn), __fdiv_rn(g1, gn))),
                        __fmul_rn(__fdiv_rn(p2, pn), __fdiv_rn(g2, gn)));
    c = fminf(fmaxf(c, -1.f), 1.f);
    ang = __fdiv_rn(__fmul_rn(acosf(c), 180.f), 3.14159265358979323846f);
    return true;
  }
};

__global__ void __launch_bounds__(kEvThreads)
    eval_normals_sums_kernel(NormalsAngle f, float* __restrict__ angles_out, double* __restrict__ part) {
  const float thr[5] = {5.f, 7.5f, 11.25f, 22.5f, 30.f};       // sub5_error .. sub30_error
  double v[kEvSums] = {0};
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < f.HW; p += (long long)gridDim.x * blockDim.x) {
    float a;
    const bool ok = f(p, a);
    if (angles_out) angles_out[p] = ok ? a : __int_as_float(0x7fc00000);
    if (!ok) continue;
    v[0] += 1.0; v[1] += a; v[2] += double(a) * a;
#pragma unroll
    for (int t = 0; t < 5; ++t) v[3 + t] += a < thr[t] ? 1.0 : 0.0;
  }
  block_reduce_store(v, 8, part);
}

// n_valid -> the two middle ranks (n - 1) / 2 and n / 2 of np.median
__global__ void eval_normals_count_kernel(const double* __restrict__ part, int nblocks, SelState* __restrict__ st) {
  const double n = warp_sum_partials(part, nblocks, 0);
  if (threadIdx.x != 0) return;
  const unsigned long long nv = (unsigned long long)n;
  st->n = nv; st->k = nv ? (nv - 1) / 2 : 0; st->krem = st->k;
}

// out: {n_valid, mean, median, rmse, sub5, sub7.5, sub11.25, sub22.5, sub30}; NaN metrics when n_valid == 0 (numpy on an
// empty array)
__global__ void eval_normals_final_kernel(const double* __restrict__ part, int nblocks, const SelState* __restrict__ st,
                                          double* __restrict__ out) {
  double s[8];
  for (int k = 0; k < 8; ++k) s[k] = warp_sum_partials(part, nblocks, k);
  if (threadIdx.x != 0) return;
  const double n = s[0];
  out[0] = n;
  if (n == 0) {
    for (int k = 1; k < 9; ++k) out[k] = __longlong_as_double(0x7ff8000000000000ll);
    return;
  }
  float a, b;
  sel_result(st, &a, &b);
  const unsigned long long nv = st->n;
  out[1] = s[1] / n;
  out[2] = (nv & 1) ? a : __fadd_rn(a, b) / 2.f;                  // np.median: float32 mean of the two middle values
  out[3] = sqrt(s[2] / n);
  for (int t = 0; t < 5; ++t) out[4 + t] = 100.0 * (s[3 + t] / n);
}

int launch_eval_normals(const float* pred, const float* gt, long long HW, float* angles_out, void* ws, double* out_dev,
                        cudaStream_t stream) {
  double* part = static_cast<double*>(ws);
  SelState* st = sel_state(ws);
  const int blocks = int(std::min<long long>((HW + kEvThreads - 1) / kEvThreads, kEvBlocks));
  const NormalsAngle f{pred, gt, HW};
  cudaMemsetAsync(st, 0, sizeof(SelState), stream);
  eval_normals_sums_kernel<<<blocks, kEvThreads, 0, stream>>>(f, angles_out, part);
  eval_normals_count_kernel<<<1, 32, 0, stream>>>(part, blocks, st);
  launch_select(f, HW, st, blocks, stream);
  eval_normals_final_kernel<<<1, 32, 0, stream>>>(part, blocks, st, out_dev);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("eval_normals launch: %s", cudaGetErrorString(e)); return MGB_ERR_CUDA; }
  return MGB_OK;
}

// ---------------------------------------------------------------------------------------------
// IID: compute_iid_metric(metric_name="psnr") with its optional colour transform (script/iid/eval.py:183-196)
// ---------------------------------------------------------------------------------------------
// srgb2linear / linear2srgb (marigold/util/image_util.py:144-149): img ** 2.2, img ** (1 / 2.2) in float32
__device__ __forceinline__ float iid_transform(float x, int transform) {
  return transform == 1 ? powf(x, 2.2f) : transform == 2 ? powf(x, float(1.0 / 2.2)) : x;
}

// quantile_map's brightness 0.3 R + 0.59 G + 0.11 B of the (transformed) ground truth, in torch's float32 order, over the
// pixels of mask channel 0 (or all pixels)
struct IidBrightness {
  const float* __restrict__ gt;
  const uint8_t* __restrict__ mask;
  long long HW;
  int transform;
  __device__ __forceinline__ bool operator()(long long i, float& b) const {
    if (mask && !mask[i]) return false;
    const float r = iid_transform(gt[i], transform), g = iid_transform(gt[HW + i], transform);
    const float bl = iid_transform(gt[2 * HW + i], transform);
    b = __fadd_rn(__fadd_rn(__fmul_rn(0.3f, r), __fmul_rn(0.59f, g)), __fmul_rn(0.11f, bl));
    return true;
  }
};

// compute_alignment_scale's sums over the masked elements (all three channels), and the quantile's pixel count
__global__ void __launch_bounds__(kEvThreads)
    eval_iid_align_sums_kernel(const float* __restrict__ pred, const float* __restrict__ gt, const uint8_t* __restrict__ mask,
                               long long HW, int transform, double* __restrict__ part) {
  double v[kEvSums] = {0};
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < HW; p += (long long)gridDim.x * blockDim.x) {
#pragma unroll 1
    for (int c = 0; c < 3; ++c) {
      const long long i = c * HW + p;
      if (mask && !mask[i]) continue;
      const double a = iid_transform(pred[i], transform), g = iid_transform(gt[i], transform);
      v[0] += a * a; v[1] += a * g;
    }
    v[2] += (!mask || mask[p]) ? 1.0 : 0.0;
  }
  block_reduce_store(v, 3, part);
}

// through-origin least-squares scale (torch.linalg.lstsq of one column, float32 result) and the quantile's ranks:
// torch.quantile forms rank = float32(0.9) * float32(n - 1), takes floor and ceil and interpolates by the float32 fraction
__global__ void eval_iid_solve_kernel(const double* __restrict__ part, int nblocks, SelState* __restrict__ st,
                                      double* __restrict__ sc) {
  const double spp = warp_sum_partials(part, nblocks, 0), spg = warp_sum_partials(part, nblocks, 1);
  const double nq = warp_sum_partials(part, nblocks, 2);
  if (threadIdx.x != 0) return;
  sc[0] = spp > 0 ? float(spg / spp) : 0.f;
  const unsigned long long n = (unsigned long long)nq;
  const float rank = n ? __fmul_rn(0.9f, float(n - 1)) : 0.f;
  const unsigned long long k = (unsigned long long)rank;
  sc[1] = __fsub_rn(rank, float(k));
  st->n = n; st->k = k; st->krem = k;
}

// q = lerp(v_k, v_k+1, w) as torch computes it (one fma on either side of w = 0.5); s = q < 1e-4 ? 0 : 0.8 / q with
// torch's 0.8 / tensor == reciprocal(tensor) * 0.8
__global__ void eval_iid_quantile_kernel(const SelState* __restrict__ st, double* __restrict__ sc) {
  float a, b;
  sel_result(st, &a, &b);
  const float w = float(sc[1]);
  float q = w < 0.5f ? fmaf(w, b - a, a) : fmaf(-(b - a), 1.f - w, b);
  if (st->n == 0) q = __int_as_float(0x7fc00000);
  sc[2] = q;
  sc[3] = q < 1e-4f ? 0.f : __fmul_rn(__frcp_rn(q), 0.8f);
}

__global__ void __launch_bounds__(kEvThreads)
    eval_iid_psnr_sums_kernel(const float* __restrict__ pred, const float* __restrict__ gt, const uint8_t* __restrict__ mask,
                              long long HW, int transform, int align, const double* __restrict__ sc, double* __restrict__ part) {
  const float ls = align ? float(sc[0]) : 1.f, qs = align ? float(sc[3]) : 1.f;
  double v[kEvSums] = {0};
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < 3 * HW; i += (long long)gridDim.x * blockDim.x) {
    if (mask && !mask[i]) continue;
    float a = iid_transform(pred[i], transform), g = iid_transform(gt[i], transform);
    if (align) {                                           // quantile_map: clamp(s * (lstsq_scale * pred)), clamp(s * gt)
      a = fminf(fmaxf(__fmul_rn(qs, __fmul_rn(ls, a)), 0.f), 1.f);
      g = fminf(fmaxf(__fmul_rn(qs, g), 0.f), 1.f);
    }
    const double d = __fsub_rn(a, g);
    v[0] += d * d; v[1] += 1.0;
  }
  block_reduce_store(v, 2, part);
}

// out: {psnr, lstsq_scale, quantile, quantile_scale, n}; PSNR(data_range=1) = 10 log10(1 / mse)
__global__ void eval_iid_final_kernel(const double* __restrict__ part, int nblocks, int align, const double* __restrict__ sc,
                                      double* __restrict__ out) {
  const double sse = warp_sum_partials(part, nblocks, 0), n = warp_sum_partials(part, nblocks, 1);
  if (threadIdx.x != 0) return;
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  out[0] = n > 0 ? 10.0 * log10(n / sse) : nan;
  out[1] = align ? sc[0] : nan; out[2] = align ? sc[2] : nan; out[3] = align ? sc[3] : nan;
  out[4] = n;
}

int launch_eval_iid(const float* pred, const float* gt, const uint8_t* mask, long long HW, int align, int transform, void* ws,
                    double* out_dev, cudaStream_t stream) {
  double* part = static_cast<double*>(ws);
  double* sc = part + size_t(kEvBlocks) * kEvSums;
  SelState* st = sel_state(ws);
  const int blocks = int(std::min<long long>((HW + kEvThreads - 1) / kEvThreads, kEvBlocks));
  if (align) {
    cudaMemsetAsync(st, 0, sizeof(SelState), stream);
    eval_iid_align_sums_kernel<<<blocks, kEvThreads, 0, stream>>>(pred, gt, mask, HW, transform, part);
    eval_iid_solve_kernel<<<1, 32, 0, stream>>>(part, blocks, st, sc);
    launch_select(IidBrightness{gt, mask, HW, transform}, HW, st, blocks, stream);
    eval_iid_quantile_kernel<<<1, 1, 0, stream>>>(st, sc);
  }
  const int pblocks = int(std::min<long long>((3 * HW + kEvThreads - 1) / kEvThreads, kEvBlocks));
  eval_iid_psnr_sums_kernel<<<pblocks, kEvThreads, 0, stream>>>(pred, gt, mask, HW, transform, align, sc, part);
  eval_iid_final_kernel<<<1, 32, 0, stream>>>(part, pblocks, align, sc, out_dev);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("eval_iid launch: %s", cudaGetErrorString(e)); return MGB_ERR_CUDA; }
  return MGB_OK;
}

}  // namespace mgb
