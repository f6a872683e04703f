// Flash self-attention for head_dim 64 on sm_100a (tcgen05 + TMEM + TMA).
//
// Replaces F.scaled_dot_product_attention under diffusers' Attention (attn1 of every
// BasicTransformerBlock) reached from reference marigold/marigold_depth_pipeline.py:461-463.
//
//   qkv : bf16 [NB * T, 3C]   (Q | K | V column blocks; head h owns columns h*64 .. h*64+63)
//   out : bf16 [NB * T, C]
//
// One CTA (one per SM) = TWO 128-query tiles A and B of the same (image, head, KV split), keys in blocks of 128;
// 320 threads:
//   warp 0     TMA producer: Q_A and Q_B (128 x 64 each) once, K / V blocks (128 x 64) through 3-stage rings
//   warp 1     TMEM allocator + MMA issuer, per tile t in {A, B}:
//                S_t = Q_t K_j^T        M128 N128 K64, both operands K-major
//                O_t += P_t V_j         M128 N64 K128, A = P_t (bf16) in TMEM (`tcgen05.mma` TS form), B = V in its
//                                       natural [token, d] layout = MN-major operand (no transpose pass)
//   warps 2-5  softmax of tile A, warps 6-9 softmax of tile B: one thread per query row (TMEM lane = row), 128
//              scores per block read with four .x32 loads, row max in registers.
// TMEM (all 512 columns, nothing aliased): S_A [0,128) S_B [128,256) P_A [256,320) P_B [320,384) O_A [384,448)
// O_B [448,512). The issuer starts S_t(j+1) as soon as softmax t has copied S_t(j) to registers ("S drained"), so
// while one softmax group computes exponentials the tensor core runs the other tile's QK^T or PV (ping-pong): the
// softmax of one tile never waits for its own next S.
// Lazy rescaling: a row keeps a reference max m_ref and P = exp2(S*c - m_ref); only when a block's max exceeds m_ref
// by more than 8 (P could exceed 2^8) is O rescaled in TMEM, which after the first blocks of a row is rare.
// Exponentials: kAttnPolyPairs of every 16 pairs of scores go through a degree-3 polynomial on the FMA pipe
// (exp2_poly_f2), the rest through MUFU.EX2; the two pipes run side by side.
#include "common.cuh"
#include "kernels.h"
#include "launch.h"

namespace mgb {

constexpr int kAttnThreads = 320;
constexpr int kTileBytes = 128 * 128;     // 128 rows x 64 bf16: a Q tile, a K block or a V block
constexpr int kKvStages = 3;
constexpr float kRescaleThreshold = 8.0f;  // log2 units
constexpr size_t kAttnSmemBytes = 1024 + 2 * kTileBytes + 2 * kKvStages * kTileBytes + 256;
// Pairs of scores (out of every 16) whose exp2 is evaluated on the FMA pipe; the other pairs use MUFU.EX2. Swept on
// B200 at T = 9216 (profiles/r03_attn_sweep.jsonl): 0 / 2 / 4 / 6 / 8 -> 162.6 / 162.6 / 158.6 / 189.0 / 183.1 us.
constexpr int kAttnPolyPairs = 4;

struct AttnParams {
  CUtensorMap tmap;   // 3D {3C, T, NB}, box {64, 128, 1}: Q tiles and K / V blocks
  bf16* out;
  int T, C, NB;
  float scale_log2;
  // split-KV: blockIdx.z = img * splits + split; split s covers KV blocks [s * nkv / splits, (s+1) * ...). With
  // splits > 1 the CTA writes un-normalised fp32 O plus (m, l) per row; attn_combine_kernel merges them.
  int splits;
  float* part_o;    // [splits][NB][C/64][T][64]
  float* part_ml;   // [splits][NB][C/64][T][2]   (m in log2 units incl. the softmax scale, l)
};

// exp2 of two values on the FMA pipe (no MUFU). Cody-Waite: x = j + f, j = floor(x), f in [0, 1);
// 2^f = 1 + f (c1 + f (c2 + f c3)) (relative minimax, |rel error| <= 8.6e-5 = 2^-13.5, far below bf16's half ulp
// 2^-9; tests/test_host.py restates it); 2^j enters as an integer add to the exponent field. floor(x) comes from
// one round-down add of 1.5 * 2^23, whose low mantissa bits then hold j as a two's complement integer: shifted by 23
// they are the exponent increment. x is clamped at -127 (masked keys are -inf): the result there is below 2^-126.
constexpr float kExp2C1 = 0.6951163411140442f;
constexpr float kExp2C2 = 0.22764700651168823f;
constexpr float kExp2C3 = 0.07706519961357117f;
__device__ __forceinline__ f2 f2_add_rm(f2 a, f2 b) {
  f2 r;
  asm("add.rm.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ void exp2_poly_f2(float x0, float x1, float& y0, float& y1) {
  const f2 x = f2_make(fmaxf(x0, -127.f), fmaxf(x1, -127.f));
  const f2 t = f2_add_rm(x, f2_splat(12582912.f));             // 1.5 * 2^23 + floor(x)
  const f2 f = f2_sub(x, f2_sub(t, f2_splat(12582912.f)));
  f2 q = f2_fma(f2_splat(kExp2C3), f, f2_splat(kExp2C2));
  q = f2_fma(q, f, f2_splat(kExp2C1));
  q = f2_fma(q, f, f2_splat(1.f));
  float q0, q1, t0, t1;
  f2_split(q, q0, q1);
  f2_split(t, t0, t1);
  y0 = __uint_as_float(__float_as_uint(q0) + (__float_as_uint(t0) << 23));
  y1 = __uint_as_float(__float_as_uint(q1) + (__float_as_uint(t1) << 23));
}

// base + off, computed where it is used: keeps ptxas from hoisting every TMEM column address of the softmax loop into
// its own register for the whole loop (the 128 scores of a row already take most of the 168 available)
__device__ __forceinline__ uint32_t addr_at_use(uint32_t base, uint32_t off) {
  uint32_t r;
  asm volatile("add.u32 %0, %1, %2;" : "=r"(r) : "r"(base), "r"(off));
  return r;
}

__global__ void __launch_bounds__(kAttnThreads, 1) flash_attn64_kernel(const __grid_constant__ AttnParams p) {
  pdl_launch_dependents();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                        // [2] A, B
  uint8_t* sK = sQ + 2 * kTileBytes;         // [kKvStages]
  uint8_t* sV = sK + kKvStages * kTileBytes; // [kKvStages]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + kKvStages * kTileBytes);
  uint64_t* q_full = bars;                   // 1
  uint64_t* k_full = bars + 1;               // [3]
  uint64_t* k_empty = bars + 4;              // [3]
  uint64_t* v_full = bars + 7;               // [3]
  uint64_t* v_empty = bars + 10;             // [3]
  uint64_t* s_full = bars + 13;              // [2 tiles]  S_t(j) computed
  uint64_t* s_drained = bars + 15;           // [2]  (128 arrivals) S_t(j) copied to registers: S_t may be rewritten
  uint64_t* p_full = bars + 17;              // [2]  (128 arrivals) P_t(j) stored (and O_t rescaled)
  uint64_t* pv_done = bars + 19;             // [2]  PV_t(j) complete: P_t free, O_t updated
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 21);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * 256, head = blockIdx.y, img = blockIdx.z / p.splits, split = blockIdx.z % p.splits;
  const bool has_b = q0 + 128 < p.T;         // the B tile of the last pair may be empty
  const int nkv_all = (p.T + 127) / 128;
  const int jb0 = split * nkv_all / p.splits;                 // first KV block of this CTA
  const int nkv = (split + 1) * nkv_all / p.splits - jb0;     // its number of KV blocks (>= 1: host keeps splits <= nkv_all)

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmap);
    mbar_init(q_full, 1);
    for (int s = 0; s < kKvStages; ++s) {
      mbar_init(&k_full[s], 1); mbar_init(&k_empty[s], 1);
      mbar_init(&v_full[s], 1); mbar_init(&v_empty[s], 1);
    }
    for (int t = 0; t < 2; ++t) {
      mbar_init(&s_full[t], 1);
      mbar_init(&s_drained[t], 128);
      mbar_init(&p_full[t], 128);
      mbar_init(&pv_done[t], 1);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_ptr_smem, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_wait();

  // Producer and MMA issuer are single-thread latency chains (see gemm_tc.cu): whole loop inside one elected
  // thread, shared-window addresses and descriptor words precomputed, counters instead of % and /.
  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      const uint32_t kfull = smem_u32(k_full), kempty = smem_u32(k_empty), vfull = smem_u32(v_full),
                     vempty = smem_u32(v_empty);
      const uint32_t sK_a = smem_u32(sK), sV_a = smem_u32(sV);
      mbar_arrive_expect_tx(q_full, has_b ? 2 * kTileBytes : kTileBytes);
      tma_load_3d(sQ, &p.tmap, q_full, head * 64, q0, img);
      if (has_b) tma_load_3d(sQ + kTileBytes, &p.tmap, q_full, head * 64, q0 + 128, img);
      const int ck = p.C + head * 64, cv = 2 * p.C + head * 64;
      uint32_t s = 0, ph = 0;
      for (int j = 0; j < nkv; ++j) {
        mbar_wait_a(kempty + s * 8, ph ^ 1);
        mbar_expect_tx_a(kfull + s * 8, kTileBytes);
        tma_load_3d_a(sK_a + s * kTileBytes, &p.tmap, kfull + s * 8, ck, (jb0 + j) * 128, img);
        mbar_wait_a(vempty + s * 8, ph ^ 1);
        mbar_expect_tx_a(vfull + s * 8, kTileBytes);
        tma_load_3d_a(sV_a + s * kTileBytes, &p.tmap, vfull + s * 8, cv, (jb0 + j) * 128, img);
        if (++s == kKvStages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      constexpr uint32_t idesc_s = umma_idesc_bf16(128, 128, false);
      constexpr uint32_t idesc_pv = umma_idesc_bf16(128, 64, true);
      constexpr uint32_t kHi = uint32_t(kDescSw128Hi >> 32), kLbo = 1u << 16;
      const uint32_t kfull = smem_u32(k_full), kempty = smem_u32(k_empty), vfull = smem_u32(v_full),
                     vempty = smem_u32(v_empty), sfull = smem_u32(s_full), sdrained = smem_u32(s_drained),
                     pfull = smem_u32(p_full), pvdone = smem_u32(pv_done);
      const uint32_t dq_lo0 = (smem_u32(sQ) >> 4) | kLbo, dk_lo0 = (smem_u32(sK) >> 4) | kLbo,
                     dv_lo0 = (smem_u32(sV) >> 4) | kLbo;
      const int ntiles = has_b ? 2 : 1;
      // S_t = Q_t K^T into TMEM columns [128 t, 128 t + 128): 4 x K=16 (32 B steps inside the 128 B swizzled rows)
      auto issue_s = [&](int t, uint32_t ks) {
        const uint32_t dq_lo = dq_lo0 + uint32_t(t) * uint32_t(kTileBytes >> 4);
        const uint32_t dk_lo = dk_lo0 + ks * uint32_t(kTileBytes >> 4);
        const uint32_t ts = tmem_base + uint32_t(t) * 128;
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(ts, make_u64(dq_lo + 2 * k, kHi), make_u64(dk_lo + 2 * k, kHi), idesc_s, k > 0 ? 1u : 0u);
        umma_commit_a(sfull + uint32_t(t) * 8);
      };
      // O_t += P_t V: A = P_t (bf16) in TMEM, 16 keys = 8 columns per K=16 step; B = V [kv, d] d-contiguous
      // (MN-major): 16 kv rows = 2048 B per step
      auto issue_pv = [&](int t, uint32_t vs, bool acc) {
        const uint32_t tp = tmem_base + 256 + uint32_t(t) * 64, to = tmem_base + 384 + uint32_t(t) * 64;
        const uint32_t dv_lo = dv_lo0 + vs * uint32_t(kTileBytes >> 4);
#pragma unroll
        for (int k = 0; k < 8; ++k)
          umma_bf16_ts(to, tp + 8 * k, make_u64(dv_lo + 128 * k, kHi), idesc_pv, (acc || k > 0) ? 1u : 0u);
        umma_commit_a(pvdone + uint32_t(t) * 8);
      };
      uint32_t ks = 0, kph = 0, vs = 0, vph = 0;
      mbar_wait_a(smem_u32(q_full), 0);
      mbar_wait_a(kfull, 0);
      tc_fence_after();
      for (int t = 0; t < ntiles; ++t) issue_s(t, 0);
      umma_commit_a(kempty);
      ks = 1;
      for (int j = 0; j < nkv; ++j) {
        const uint32_t ph = uint32_t(j) & 1u;
        const bool next = j + 1 < nkv;
        if (next) mbar_wait_a(kfull + ks * 8, kph);
        mbar_wait_a(vfull + vs * 8, vph);
        for (int t = 0; t < ntiles; ++t) {
          if (next) {   // S_t(j+1) as soon as softmax t holds S_t(j) in registers
            mbar_wait_a(sdrained + uint32_t(t) * 8, ph);
            tc_fence_after();
            issue_s(t, ks);
          }
          mbar_wait_a(pfull + uint32_t(t) * 8, ph);
          tc_fence_after();
          issue_pv(t, vs, j > 0);
        }
        if (next) {
          umma_commit_a(kempty + ks * 8);
          if (++ks == kKvStages) { ks = 0; kph ^= 1; }
        }
        umma_commit_a(vempty + vs * 8);
        if (++vs == kKvStages) { vs = 0; vph ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp < 6 || has_b) {
    // ===================== softmax (tile t) =====================
    const int t = warp >= 6 ? 1 : 0;
    const int qw = warp & 3;                 // TMEM lane quarter
    const int row = qw * 32 + lane;
    const uint32_t lane_off = uint32_t(qw * 32) << 16;
    const uint32_t tS = tmem_base + lane_off + uint32_t(t) * 128, tP = tmem_base + lane_off + 256 + uint32_t(t) * 64,
                   tO = tmem_base + lane_off + 384 + uint32_t(t) * 64;
    float m_ref = 0.f, l_run = 0.f;
    for (int j = 0; j < nkv; ++j) {
      const uint32_t ph = uint32_t(j) & 1u;
      mbar_wait(&s_full[t], ph);
      tc_fence_after();
      uint32_t r[128];
      tmem_ld32(tS, *reinterpret_cast<uint32_t(*)[32]>(r));
      tmem_ld32(addr_at_use(tS, 32), *reinterpret_cast<uint32_t(*)[32]>(r + 32));
      tmem_ld32(addr_at_use(tS, 64), *reinterpret_cast<uint32_t(*)[32]>(r + 64));
      tmem_ld32(addr_at_use(tS, 96), *reinterpret_cast<uint32_t(*)[32]>(r + 96));
      tmem_wait_ld();
      tc_fence_before();
      mbar_arrive(&s_drained[t]);
      const int kv_valid = p.T - (jb0 + j) * 128;   // >= 128 except possibly in the last block
      if (kv_valid < 128) {                         // ragged tail: mask once, then share the fast path
#pragma unroll
        for (int i = 0; i < 128; ++i)
          if (i >= kv_valid) r[i] = 0xff800000u;    // -inf
      }
      // row max with 4 independent chains
      float mx[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) mx[c] = __uint_as_float(r[c]);
#pragma unroll
      for (int i = 4; i < 128; i += 4)
#pragma unroll
        for (int c = 0; c < 4; ++c) mx[c] = fmaxf(mx[c], __uint_as_float(r[i + c]));
      const float m_blk = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])) * p.scale_log2;
      // Lazy rescaling: the O rescale itself runs after the P stores, when the scores no longer hold registers
      bool rescale = false;
      float alpha = 1.f;
      if (j == 0) {
        m_ref = m_blk;
      } else {
        // P_t and O_t are free once PV_t(j-1) has completed
        mbar_wait(&pv_done[t], ph ^ 1);
        tc_fence_after();
        const bool need = m_blk > m_ref + kRescaleThreshold;
        rescale = __any_sync(0xffffffffu, need);    // the TMEM loads of O are warp-collective
        if (need) {                                 // other rows of the warp multiply O by 1
          alpha = ex2_approx(m_ref - m_blk);
          m_ref = m_blk;
          l_run *= alpha;
        }
      }
      // P = exp2(S * c - m_ref) (exp2(-inf) = 0 masks the tail); bf16 pairs; packed partial row sums.
      // Per 32 scores: the scale-and-shift (FFMA2), exponentials (kAttnPolyPairs of 16 pairs on the FMA pipe), F2FP packs,
      // row sums (FADD2), one 16-column store of P.
      const f2 sc2 = f2_splat(p.scale_log2), nm2 = f2_splat(-m_ref);
      f2 ls0 = f2_splat(0.f), ls1 = ls0;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          float t0, t1, a0, a1;
          f2_split(f2_fma(f2_make(__uint_as_float(r[32 * c + 2 * i]), __uint_as_float(r[32 * c + 2 * i + 1])), sc2, nm2),
                   t0, t1);
          if (((i + 1) * kAttnPolyPairs) / 16 != (i * kAttnPolyPairs) / 16) {   // spread evenly over the 16 pairs
            exp2_poly_f2(t0, t1, a0, a1);
          } else {
            a0 = ex2_approx(t0);
            a1 = ex2_approx(t1);
          }
          if (i & 1) ls1 = f2_add(ls1, f2_make(a0, a1));
          else ls0 = f2_add(ls0, f2_make(a0, a1));
          pk[i] = pack_bf16x2(a0, a1);
        }
        tmem_st16(addr_at_use(tP, c * 16), pk);
      }
      {
        float s0, s1, s2, s3;
        f2_split(ls0, s0, s1);
        f2_split(ls1, s2, s3);
        l_run += (s0 + s1) + (s2 + s3);
      }
      if (rescale) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint32_t o[32];
          tmem_ld32(addr_at_use(tO, h * 32), o);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
          tmem_st32(addr_at_use(tO, h * 32), o);
        }
      }
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(&p_full[t]);
    }
    // epilogue: O / l, or the un-normalised split partial
    mbar_wait(&pv_done[t], uint32_t(nkv - 1) & 1u);
    tc_fence_after();
    const int qrow = q0 + t * 128 + row;
    uint32_t o[64];
    tmem_ld32(tO, *reinterpret_cast<uint32_t(*)[32]>(o));
    tmem_ld32(tO + 32, *reinterpret_cast<uint32_t(*)[32]>(o + 32));
    tmem_wait_ld();
    if (qrow < p.T) {
      if (p.splits == 1) {
        const float inv = 1.f / l_run;
        uint4* dst = reinterpret_cast<uint4*>(p.out + ((size_t)img * p.T + qrow) * p.C + head * 64);
#pragma unroll
        for (int i = 0; i < 8; ++i)
          dst[i] = make_uint4(pack_bf16x2(__uint_as_float(o[8 * i]) * inv, __uint_as_float(o[8 * i + 1]) * inv),
                              pack_bf16x2(__uint_as_float(o[8 * i + 2]) * inv, __uint_as_float(o[8 * i + 3]) * inv),
                              pack_bf16x2(__uint_as_float(o[8 * i + 4]) * inv, __uint_as_float(o[8 * i + 5]) * inv),
                              pack_bf16x2(__uint_as_float(o[8 * i + 6]) * inv, __uint_as_float(o[8 * i + 7]) * inv));
      } else {
        const size_t prow = ((size_t(split) * p.NB + img) * gridDim.y + head) * p.T + qrow;
        uint4* dst = reinterpret_cast<uint4*>(p.part_o + prow * 64);
#pragma unroll
        for (int i = 0; i < 16; ++i) dst[i] = make_uint4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
        *reinterpret_cast<float2*>(p.part_ml + prow * 2) = make_float2(m_ref, l_run);
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// Merge the split-KV partials: out[row, :] = sum_s w_s O_s / sum_s w_s l_s, w_s = 2^(m_s - max m). One thread per
// (row, 8 columns).
__global__ void __launch_bounds__(256) attn_combine_kernel(const float* __restrict__ part_o, const float* __restrict__ part_ml,
                                                           bf16* __restrict__ out, int splits, int NB, int heads, int T, int C) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t rows = size_t(NB) * heads * T;
  const size_t gid = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t r = gid >> 3;
  const int c8 = int(gid & 7) * 8;
  if (r >= rows) return;
  float m = -INFINITY;
  for (int s = 0; s < splits; ++s) m = fmaxf(m, __ldg(part_ml + (size_t(s) * rows + r) * 2));
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, l = 0.f;
  for (int s = 0; s < splits; ++s) {
    const float2 ml = __ldg(reinterpret_cast<const float2*>(part_ml + (size_t(s) * rows + r) * 2));
    const float w = ex2_approx(ml.x - m);
    l = fmaf(ml.y, w, l);
    const float4* po = reinterpret_cast<const float4*>(part_o + (size_t(s) * rows + r) * 64 + c8);
    const float4 a = __ldg(po), b = __ldg(po + 1);
    acc[0] = fmaf(a.x, w, acc[0]); acc[1] = fmaf(a.y, w, acc[1]); acc[2] = fmaf(a.z, w, acc[2]); acc[3] = fmaf(a.w, w, acc[3]);
    acc[4] = fmaf(b.x, w, acc[4]); acc[5] = fmaf(b.y, w, acc[5]); acc[6] = fmaf(b.z, w, acc[6]); acc[7] = fmaf(b.w, w, acc[7]);
  }
  const float inv = 1.f / l;
  const size_t t = r % T, ih = r / T;
  const size_t img = ih / heads, head = ih % heads;
  uint4* dst = reinterpret_cast<uint4*>(out + (img * T + t) * C + head * 64 + c8);
  *dst = make_uint4(pack_bf16x2(acc[0] * inv, acc[1] * inv), pack_bf16x2(acc[2] * inv, acc[3] * inv),
                    pack_bf16x2(acc[4] * inv, acc[5] * inv), pack_bf16x2(acc[6] * inv, acc[7] * inv));
}

// KV splits that minimise the number of CTA rounds (one CTA per SM, one CTA = a pair of 128-query tiles) weighted by
// the split's length in 128-key blocks plus a per-CTA fixed cost (prologue, Q load, first S, epilogue) and the
// combine pass. Both costs fitted to forced split counts 1..6 at T = 9216, NB = 1 on B200 (182-242 us,
// profiles/r03_attn_sweep.jsonl): 1.5 us per block and round, fixed cost 4 blocks, combine 11 blocks. The same model
// keeps NB = 8 unsplit (measured: 1216 us unsplit, 1345-1579 us with 2-6 splits).
constexpr double kAttnCtaFixedBlocks = 4.0;
constexpr double kAttnCombineBlocks = 11.0;
int flash_attn64_splits(int NB, int T, int C) {
  const int units = ((T + 255) / 256) * (C / 64) * NB, nkv = (T + 127) / 128, slots = 148;
  int best = 1;
  double best_t = 1e30;
  for (int s = 1; s <= 8; ++s) {
    if (s > 1 && nkv / s < 3) break;
    const double rounds = double((units * s + slots - 1) / slots);
    const double t = rounds * (double(nkv) / s + kAttnCtaFixedBlocks) + (s > 1 ? kAttnCombineBlocks : 0.0);
    if (t < best_t - 1e-9) { best_t = t; best = s; }
  }
  return best;
}
size_t flash_attn64_ws_bytes(int NB, int T, int C) {
  const int s = flash_attn64_splits(NB, T, C);
  if (s == 1) return 0;
  return size_t(s) * NB * (C / 64) * T * (64 + 2) * sizeof(float);
}

int launch_flash_attn64(const bf16* qkv, bf16* out, int NB, int T, int C, float scale, float* ws, size_t ws_bytes,
                        cudaStream_t stream) {
  if (C % 64 != 0 || T <= 0) {
    set_error("flash_attn64: C %% 64 != 0 or bad T");
    return MGB_ERR_INVALID;
  }
  AttnParams p;
  const uint64_t dims[3] = {uint64_t(3 * C), uint64_t(T), uint64_t(NB)};
  const uint64_t strides[2] = {uint64_t(3 * C) * 2, uint64_t(T) * 3 * C * 2};
  const uint32_t box[3] = {64, 128, 1};
  int rc = make_tmap_3d(&p.tmap, qkv, dims, strides, box);
  if (rc) return rc;
  p.out = out; p.T = T; p.C = C; p.NB = NB;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.splits = 1; p.part_o = nullptr; p.part_ml = nullptr;
  {
    const int sp = flash_attn64_splits(NB, T, C);
    if (sp > 1 && ws != nullptr && ws_bytes >= flash_attn64_ws_bytes(NB, T, C)) {
      p.splits = sp;
      p.part_o = ws;
      p.part_ml = ws + size_t(sp) * NB * (C / 64) * T * 64;
    }
  }
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(flash_attn64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         int(kAttnSmemBytes));
    if (e != cudaSuccess) { set_error("flash_attn64 attr: %s", cudaGetErrorString(e)); return MGB_ERR_CUDA; }
    attr_set = true;
  }
  const dim3 grid((T + 255) / 256, C / 64, NB * p.splits);
  cudaError_t e = launch_k(flash_attn64_kernel, grid, kAttnThreads, kAttnSmemBytes, stream, p);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("flash_attn64 launch: %s", cudaGetErrorString(e)); return MGB_ERR_CUDA; }
  if (p.splits > 1) {
    const size_t threads = size_t(NB) * (C / 64) * T * 8;
    e = launch_k(attn_combine_kernel, dim3(unsigned((threads + 255) / 256)), 256, 0, stream, (const float*)p.part_o,
                 (const float*)p.part_ml, out, p.splits, NB, C / 64, T, C);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("attn_combine launch: %s", cudaGetErrorString(e)); return MGB_ERR_CUDA; }
  }
  return MGB_OK;
}

}  // namespace mgb
