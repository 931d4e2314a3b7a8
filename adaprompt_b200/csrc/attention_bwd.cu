// Flash-attention BACKWARD for the long self-attention layers of the Stage-1 training step (SURVEY.md section 8 row T1;
// autograd of CrossAttention.forward, ldm/modules/attention.py:198-242, on the student UNet, ddpm.py:2483-2532).
//
//   P = exp2(S - lse)         S = Q K^T (log2 domain, Q pre-scaled), lse saved by the forward kernel
//   dP = dO V^T               delta_i = sum_c dO_ic O_ic
//   dS = ln2 * P o (dP - delta)
//   dQ = dS K      dK = dS^T Q      dV = P^T dO
//
// Round 1 ran this as seven batched mma.sync GEMMs with P, P^T, dS and dS^T materialised in HBM (4 x B*8*N*N bf16:
// 4.3 GB per micro-batch at N = 4096; 44 ms of the 130 ms optimizer step).  Here nothing of size N x N leaves the SM:
// ONE kernel template, two instantiations, both on tcgen05 with accumulators and the bf16 P / dS operands in TMEM:
//
//   DKV = false (dQ):      CTA = 128 QUERY rows; streams 64-key blocks.   S = Q_i K_c^T, T = dO_i V_c^T,
//                          G = dS (rows = queries: lse / delta are per-thread scalars),   dQ_i += G K_c.
//   DKV = true  (dK, dV):  CTA = 128 KEY rows;   streams 64-query blocks. S = K_j Q_c^T (= S^T), T = V_j dO_c^T (= dP^T),
//                          P^T and G = dS^T (lse / delta are per-COLUMN vectors, broadcast from shared memory),
//                          dV_j += P^T dO_c,   dK_j += G Q_c.
//
// TMEM columns: S [0,64) | T [64,128) | acc0 [128,128+DP) | acc1 [..,+DP).  After a thread has copied its S / T rows to
// registers it writes P over the head of S and G over the head of T; the in-order MMA issuer runs the gradient MMAs of
// block c and only then the score MMAs of block c+1 into the same columns, so "S_{c+1} ready" implies "gradient MMAs of
// block c complete": one wait (s_full) and one arrive (p_full) per block, no other hand-shake.  Two CTAs per SM (d = 40)
// hide each other's MMA round trips, as in attention_tile.cu.
//
// Operands (all bf16, K-major 128B-swizzled TMA tiles; head h at columns h*DP of the row-major matrices, DP = 48 zero-padded
// for d = 40; the *T matrices are the [h*DP, tokens] transposes): rows-side X, Y [tokens, >= h*DP]; column-side U, W likewise;
// the B operands of the gradient MMAs come from the transposed copies (tokens contiguous).
#include <math.h>

#include "../../include/adaface_b200.h"
#include "attn_tile_common.cuh"
#include "common.cuh"

namespace af {

struct AttnBwdParams {
  CUtensorMap tmX, tmY;      // row-tile operands: 3-D {h*DP, N, B}, box {64, 128, 1}
  CUtensorMap tmU, tmW;      // column-block operands: 3-D {h*DP, N, B}, box {64, 64, 1}
  CUtensorMap tmT0, tmT1;    // transposed column-block operands: 2-D {ld, h*DP}, box {64, DP}
  const float* lse;          // [B][heads][N]
  const float* delta;        // [B][heads][N]
  __nv_bfloat16* out0;       // dQ [B*N, ld0] (cols h*DP..) | dV [B*N, ld0] (cols h*d.., d columns)
  __nv_bfloat16* out1;       // dK [B*N, ld1] (DKV only)
  long long ld0, ld1;
  int B, heads, N, d;
  const uint8_t* kmask;      // [B][N] key mask, 1 = attend (masked instantiations only)
};

template <int D>
struct BwdCfg;
template <>
struct BwdCfg<40> {
  static constexpr int DP = 48, STAGES = 2, CTAS = 2;     // TMEM 224 columns, 2 CTAs per SM
};
template <>
struct BwdCfg<80> {
  static constexpr int DP = 80, STAGES = 2, CTAS = 1;     // TMEM 288 (dK, dV) / 208 (dQ) columns; 150-170 KB of tiles
};

template <int D, bool DKV>
struct BwdSmem {
  using C = BwdCfg<D>;
  static constexpr int KA = (C::DP + 63) / 64;
  static constexpr int kRowBytes = KA * 128 * 128;         // X or Y: 128 rows
  static constexpr int kColBytes = KA * 64 * 128;          // U or W: 64 rows
  static constexpr int kTBytes = C::DP * 128;              // transposed tile: DP rows x 64 tokens
  static constexpr int kVecBytes = DKV ? 2 * 64 * 4 : 0;   // lse / delta of the 64-query block
  static constexpr int kStageBytes = 2 * kColBytes + (DKV ? 2 : 1) * kTBytes + 1024;   // vectors live in the last KB
  static constexpr int kStageTx = 2 * kColBytes + (DKV ? 2 : 1) * kTBytes + kVecBytes;
  static constexpr int kXOff = 0, kYOff = kRowBytes, kStageOff = 2 * kRowBytes;
  static constexpr int kBarOff = kStageOff + C::STAGES * kStageBytes;
  static constexpr int kTotal = kBarOff + 256 + 1024;
  static_assert(kTBytes % 1024 == 0 && kColBytes % 1024 == 0, "swizzle atoms are 1024-byte aligned");
};

__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// MASKED: the key mask of attention.py:223-232 (scores of masked keys filled with -finfo.max before the softmax), as the
// exact derivative of af_attention_bf16_lse with a key mask:
//   a sample with a kept key:  P_ij = m_j ? exp2(S_ij - lse_i) : 0,   dS_ij = m_j ? ln2 P_ij (dP_ij - delta_i) : 0;
//   a sample that keeps no key (lse = +inf in every row, the forward output is the mean of V):  P_ij = 1 / N, dS = 0.
// The mask enters through selects only, so whatever masked K / V rows hold never reaches a gradient, and the kept
// keys take the operation order of the unmasked instantiation (an all-ones mask gives bit-identical results).
//   dQ kernel:     the 64 mask bytes of key block c ride in the stage, next to where the DKV kernel keeps lse / delta.
//   dK/dV kernel:  the mask is a per-row scalar; the row's own lse (queries and keys are the same tokens) tells whether
//                  the sample keeps no key.  Then P^T is 1 in every entry and the dV accumulator is scaled by 1/N.
template <int D, bool DKV, bool MASKED>
__device__ __forceinline__ void attention_bwd_body(const AttnBwdParams& p) {
  using C = BwdCfg<D>;
  using S = BwdSmem<D, DKV>;
  constexpr int DP = C::DP, KA = S::KA, NST = C::STAGES;
  constexpr int kStageTx = S::kStageTx + (MASKED && !DKV ? 64 : 0);
  constexpr uint32_t kTmS = 0, kTmT = 64, kTmA0 = 128, kTmA1 = 128 + DP;
  constexpr uint32_t kTmemCols = (128 + (DKV ? 2 : 1) * DP) <= 256 ? 256 : 512;
  constexpr float kLn2 = 0.69314718055994530942f;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t smem_base = smem_u32(smem);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::kBarOff);
  uint64_t* x_full = bars;                   // 1: X and Y landed
  uint64_t* st_full = x_full + 1;            // NST
  uint64_t* st_empty = st_full + NST;        // NST
  uint64_t* s_full = st_empty + NST;         // 1: S_c, T_c in TMEM (and every earlier MMA complete)
  uint64_t* p_full = s_full + 1;             // 1 (4 warps): P / G of block c written
  uint64_t* done = p_full + 1;               // 1: last gradient MMAs complete
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int row0 = blockIdx.x * 128;
  const int h = blockIdx.y;
  const int b = blockIdx.z;
  const int n_blocks = p.N / 64;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&p.tmX);
    tma_prefetch_desc(&p.tmY);
    tma_prefetch_desc(&p.tmU);
    tma_prefetch_desc(&p.tmW);
    tma_prefetch_desc(&p.tmT0);
    if (DKV) tma_prefetch_desc(&p.tmT1);
    mbar_init(x_full, 1);
    for (int s = 0; s < NST; ++s) {
      mbar_init(&st_full[s], 1);
      mbar_init(&st_empty[s], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(p_full, 4);
    mbar_init(done, 1);
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
    if (warp == 0) {
      // ------------------------------------------------------------------ TMA producer
      if (lane == 0) {
        mbar_arrive_expect_tx(x_full, 2 * S::kRowBytes);
#pragma unroll
        for (int a = 0; a < KA; ++a) {
          tma_load_3d(smem + S::kXOff + a * 128 * 128, &p.tmX, x_full, h * DP + a * 64, row0, b);
          tma_load_3d(smem + S::kYOff + a * 128 * 128, &p.tmY, x_full, h * DP + a * 64, row0, b);
        }
        int st = 0;
        uint32_t ph = 0;
        for (int c = 0; c < n_blocks; ++c) {
          mbar_wait_lean(&st_empty[st], ph ^ 1);
          uint8_t* base = smem + S::kStageOff + st * S::kStageBytes;
          mbar_arrive_expect_tx(&st_full[st], kStageTx);
#pragma unroll
          for (int a = 0; a < KA; ++a) {
            tma_load_3d(base + a * 64 * 128, &p.tmU, &st_full[st], h * DP + a * 64, c * 64, b);
            tma_load_3d(base + S::kColBytes + a * 64 * 128, &p.tmW, &st_full[st], h * DP + a * 64, c * 64, b);
          }
          tma_load_2d(base + 2 * S::kColBytes, &p.tmT0, &st_full[st], b * p.N + c * 64, h * DP);
          if (DKV) {
            tma_load_2d(base + 2 * S::kColBytes + S::kTBytes, &p.tmT1, &st_full[st], b * p.N + c * 64, h * DP);
            const size_t voff = (static_cast<size_t>(b) * p.heads + h) * p.N + c * 64;
            uint8_t* vec = base + S::kStageBytes - 1024;
            bulk_load_1d(vec, p.lse + voff, 256, &st_full[st]);
            bulk_load_1d(vec + 256, p.delta + voff, 256, &st_full[st]);
          } else if (MASKED) {
            bulk_load_1d(base + S::kStageBytes - 1024, p.kmask + static_cast<size_t>(b) * p.N + c * 64, 64, &st_full[st]);
          }
          if (++st == NST) { st = 0; ph ^= 1; }
        }
      }
    } else if (warp == 1) {
      // ------------------------------------------------------------------ MMA issuer
      constexpr uint32_t idesc_s = umma_idesc_bf16(128, 64);
      constexpr uint32_t idesc_g = umma_idesc_bf16(128, DP);
      const uint32_t x_addr = smem_base + S::kXOff, y_addr = smem_base + S::kYOff;
      const uint32_t tm_s = tmem_base + kTmS, tm_t = tmem_base + kTmT;
      auto issue_scores = [&](int st) {
        const uint32_t u_addr = smem_base + S::kStageOff + st * S::kStageBytes;
        const uint32_t w_addr = u_addr + S::kColBytes;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < DP / 16; ++k) {
            tc_mma_ss(tm_s, umma_desc_sw128(x_addr + (k >> 2) * 128 * 128) + 2 * (k & 3),
                      umma_desc_sw128(u_addr + (k >> 2) * 64 * 128) + 2 * (k & 3), idesc_s, k != 0 ? 1u : 0u);
          }
#pragma unroll
          for (int k = 0; k < DP / 16; ++k) {
            tc_mma_ss(tm_t, umma_desc_sw128(y_addr + (k >> 2) * 128 * 128) + 2 * (k & 3),
                      umma_desc_sw128(w_addr + (k >> 2) * 64 * 128) + 2 * (k & 3), idesc_s, k != 0 ? 1u : 0u);
          }
          tc_commit(s_full);
        }
        __syncwarp();
      };
      mbar_wait_lean(x_full, 0);
      mbar_wait_lean(&st_full[0], 0);
      tc_fence_after();
      issue_scores(0);
      int st = 0;
      uint32_t ph = 0;
      for (int c = 0; c < n_blocks; ++c) {
        mbar_wait_lean(p_full, c & 1);
        tc_fence_after();
        const uint32_t t0_addr = smem_base + S::kStageOff + st * S::kStageBytes + 2 * S::kColBytes;
        if (elect_one()) {
          if (DKV) {
#pragma unroll
            for (int k = 0; k < 4; ++k)      // dV += P^T dO_c  (64 queries = 4 k-steps)
              tc_mma_ts(tmem_base + kTmA0, tm_s + k * 8, umma_desc_sw128(t0_addr) + 2 * k, idesc_g, (c | k) != 0 ? 1u : 0u);
#pragma unroll
            for (int k = 0; k < 4; ++k)      // dK += dS^T Q_c
              tc_mma_ts(tmem_base + kTmA1, tm_t + k * 8, umma_desc_sw128(t0_addr + S::kTBytes) + 2 * k, idesc_g,
                        (c | k) != 0 ? 1u : 0u);
          } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)      // dQ += dS K_c  (64 keys = 4 k-steps)
              tc_mma_ts(tmem_base + kTmA0, tm_t + k * 8, umma_desc_sw128(t0_addr) + 2 * k, idesc_g, (c | k) != 0 ? 1u : 0u);
          }
          tc_commit(&st_empty[st]);
          if (c == n_blocks - 1) tc_commit(done);
        }
        __syncwarp();
        if (++st == NST) { st = 0; ph ^= 1; }
        if (c + 1 < n_blocks) {
          mbar_wait_lean(&st_full[st], ph);
          tc_fence_after();
          issue_scores(st);
        }
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
    // ------------------------------------------------------------------ elementwise warps: one thread per tile row
    const int qd = warp & 3;
    const int r = qd * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(qd * 32) << 16;
    const uint32_t s_addr = tmem_base + kTmS + lane_off, t_addr = tmem_base + kTmT + lane_off;
    const uint32_t a_s_full = smem_u32(s_full), a_p_full = smem_u32(p_full);
    float lse_r = 0.f, dl_r = 0.f;      // DKV = false: per-row scalars (delta pre-multiplied by ln 2)
    if (!DKV) {
      const size_t voff = (static_cast<size_t>(b) * p.heads + h) * p.N + row0 + r;
      lse_r = __ldg(p.lse + voff);
      dl_r = __ldg(p.delta + voff) * kLn2;
    }
    bool keep = true, empty = false;      // MASKED && DKV: this key row is attended / its sample keeps no key
    if (MASKED && DKV) {
      keep = __ldg(p.kmask + static_cast<size_t>(b) * p.N + row0 + r) != 0;
      empty = isinf(__ldg(p.lse + (static_cast<size_t>(b) * p.heads + h) * p.N + row0 + r));
    }
    const uint32_t p_drop = empty ? pack_bf16x2(1.f, 1.f) : 0u;
    int st = 0;
    for (int c = 0; c < n_blocks; ++c) {
      mbar_wait_lean(a_s_full, c & 1);
      tc_fence_after();
      float sv[64], tv[64];
      tile_ld32(s_addr, reinterpret_cast<uint32_t*>(sv));
      tile_ld32(s_addr + 32, reinterpret_cast<uint32_t*>(sv) + 32);
      tile_ld32(t_addr, reinterpret_cast<uint32_t*>(tv));
      tile_ld32(t_addr + 32, reinterpret_cast<uint32_t*>(tv) + 32);
      tmem_ld_wait();
      uint32_t pkp[32], pkg[32];
      if (DKV) {
        const uint32_t vec = smem_base + S::kStageOff + st * S::kStageBytes + S::kStageBytes - 1024;
#pragma unroll
        for (int e = 0; e < 64; e += 4) {
          const float4 l4 = lds128f(vec + e * 4);          // lse of queries e .. e+3 (same address in every lane)
          const float4 d4 = lds128f(vec + 256 + e * 4);    // delta
          const float p0 = fast_exp2(sv[e] - l4.x), p1 = fast_exp2(sv[e + 1] - l4.y);
          const float p2 = fast_exp2(sv[e + 2] - l4.z), p3 = fast_exp2(sv[e + 3] - l4.w);
          pkp[e >> 1] = pack_bf16x2(p0, p1);
          pkp[(e >> 1) + 1] = pack_bf16x2(p2, p3);
          pkg[e >> 1] = pack_bf16x2(p0 * ((tv[e] - d4.x) * kLn2), p1 * ((tv[e + 1] - d4.y) * kLn2));
          pkg[(e >> 1) + 1] = pack_bf16x2(p2 * ((tv[e + 2] - d4.z) * kLn2), p3 * ((tv[e + 3] - d4.w) * kLn2));
          if (MASKED) {
            pkp[e >> 1] = keep ? pkp[e >> 1] : p_drop;
            pkp[(e >> 1) + 1] = keep ? pkp[(e >> 1) + 1] : p_drop;
            pkg[e >> 1] = keep ? pkg[e >> 1] : 0u;
            pkg[(e >> 1) + 1] = keep ? pkg[(e >> 1) + 1] : 0u;
          }
        }
        tile_st32(s_addr, pkp);          // P^T over the head of S
        tile_st32(t_addr, pkg);          // dS^T over the head of T
      } else if (MASKED) {
        const uint32_t mvec = smem_base + S::kStageOff + st * S::kStageBytes + S::kStageBytes - 1024;
#pragma unroll
        for (int e = 0; e < 64; e += 4) {
          const uint32_t m4 = __float_as_uint(lds32f(mvec + e));     // mask bytes of keys e .. e+3 (broadcast)
#pragma unroll
          for (int u = 0; u < 4; u += 2) {
            const float p0 = fast_exp2(sv[e + u] - lse_r), p1 = fast_exp2(sv[e + u + 1] - lse_r);
            const float g0 = p0 * fmaf(tv[e + u], kLn2, -dl_r), g1 = p1 * fmaf(tv[e + u + 1], kLn2, -dl_r);
            pkg[(e + u) >> 1] = pack_bf16x2((m4 >> (8 * u)) & 0xffu ? g0 : 0.f, (m4 >> (8 * u + 8)) & 0xffu ? g1 : 0.f);
          }
        }
        tile_st32(t_addr, pkg);          // dS over the head of T
      } else {
#pragma unroll
        for (int e = 0; e < 64; e += 2) {
          const float p0 = fast_exp2(sv[e] - lse_r), p1 = fast_exp2(sv[e + 1] - lse_r);
          pkg[e >> 1] = pack_bf16x2(p0 * fmaf(tv[e], kLn2, -dl_r), p1 * fmaf(tv[e + 1], kLn2, -dl_r));
        }
        tile_st32(t_addr, pkg);          // dS over the head of T
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a_p_full) : "memory");
      if (++st == NST) st = 0;
    }
    // epilogue: accumulators -> bf16 rows
    mbar_wait_lean(done, 0);
    tc_fence_after();
    const size_t grow = static_cast<size_t>(b) * p.N + row0 + r;
    auto store_acc = [&](uint32_t tm_col, __nv_bfloat16* out, long long ld, int col0, int ncols, bool mean) {
      __nv_bfloat16* orow = out + grow * ld + col0;
      const float inv_n = 1.f / static_cast<float>(p.N);
#pragma unroll 1
      for (int cc = 0; cc < DP; cc += 16) {
        uint32_t o[16];
        tmem_ld16(tmem_base + tm_col + lane_off + cc, o);
        tmem_ld_wait();
        if (MASKED && mean) {            // dV of a sample that keeps no key: (sum_i dO_i) / N
#pragma unroll
          for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * inv_n);
        }
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          if (cc + g * 8 < ncols) {
            uint4 pk;
            pk.x = pack_bf16x2(__uint_as_float(o[g * 8 + 0]), __uint_as_float(o[g * 8 + 1]));
            pk.y = pack_bf16x2(__uint_as_float(o[g * 8 + 2]), __uint_as_float(o[g * 8 + 3]));
            pk.z = pack_bf16x2(__uint_as_float(o[g * 8 + 4]), __uint_as_float(o[g * 8 + 5]));
            pk.w = pack_bf16x2(__uint_as_float(o[g * 8 + 6]), __uint_as_float(o[g * 8 + 7]));
            *reinterpret_cast<uint4*>(orow + cc + g * 8) = pk;
          }
        }
      }
    };
    if (DKV) {
      store_acc(kTmA0, p.out0, p.ld0, h * p.d, p.d, empty);     // dV: d columns
      store_acc(kTmA1, p.out1, p.ld1, h * DP, DP, false);       // dK: DP columns (pads are exact zeros)
    } else {
      store_acc(kTmA0, p.out0, p.ld0, h * DP, DP, false);       // dQ
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

template <int D, bool DKV>
__global__ void __launch_bounds__(256, BwdCfg<D>::CTAS) attention_bwd_kernel(const __grid_constant__ AttnBwdParams p) {
  attention_bwd_body<D, DKV, false>(p);
}
template <int D, bool DKV>
__global__ void __launch_bounds__(256, BwdCfg<D>::CTAS) attention_bwd_masked_kernel(const __grid_constant__ AttnBwdParams p) {
  attention_bwd_body<D, DKV, true>(p);
}

template <int D, bool DKV, bool MASKED>
static int launch_bwd(const AttnBwdParams& p, cudaStream_t stream) {
  using S = BwdSmem<D, DKV>;
  const auto kernel = MASKED ? attention_bwd_masked_kernel<D, DKV> : attention_bwd_kernel<D, DKV>;
  static bool configured = false;
  if (!configured) {
    AF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal));
    AF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    configured = true;
  }
  dim3 grid(p.N / 128, p.heads, p.B);
  kernel<<<grid, 256, S::kTotal, stream>>>(p);
  AF_LAUNCH_CHECK(MASKED ? "attention_bwd_masked_kernel" : "attention_bwd_kernel");
  return 0;
}

static int make_rows_map(CUtensorMap* m, const void* base, long long ld, int heads, int dp, int N, int B, int box_rows) {
  uint64_t dims[3] = {static_cast<uint64_t>(heads) * dp, static_cast<uint64_t>(N), static_cast<uint64_t>(B)};
  uint64_t str[2] = {static_cast<uint64_t>(ld) * 2, static_cast<uint64_t>(N) * ld * 2};
  uint32_t box[3] = {64, static_cast<uint32_t>(box_rows), 1};
  return make_tmap_bf16(m, base, 3, dims, str, box);
}
static int make_t_map(CUtensorMap* m, const void* base, long long ld, int heads, int dp) {
  uint64_t dims[2] = {static_cast<uint64_t>(ld), static_cast<uint64_t>(heads) * dp};
  uint64_t str[1] = {static_cast<uint64_t>(ld) * 2};
  uint32_t box[2] = {64, static_cast<uint32_t>(dp)};
  return make_tmap_bf16(m, base, 2, dims, str, box);
}

}  // namespace af

using namespace af;

namespace af {

static int attention_bwd(const void* Q, long long ldq, const void* K, long long ldk, const void* Vp, long long ldv,
                         const void* dOp, long long lddo, const void* QT, long long ldqt, const void* KT, long long ldkt,
                         const void* dOT, long long lddot, const float* lse, const float* delta, const unsigned char* key_mask,
                         void* dQ, long long lddq, void* dK, long long lddk, void* dV, long long lddv, int B, int heads,
                         int N, int d, cudaStream_t stream) {
  const int dp = d == 40 ? 48 : 80;
  const bool masked = key_mask != nullptr;
  int rc;
  {   // dQ: rows = queries (X = Q, Y = dO), columns = keys (U = K, W = V), B operand of the gradient MMA = K^T
    AttnBwdParams p;
    memset(&p, 0, sizeof(p));
    if ((rc = make_rows_map(&p.tmX, Q, ldq, heads, dp, N, B, 128))) return rc;
    if ((rc = make_rows_map(&p.tmY, dOp, lddo, heads, dp, N, B, 128))) return rc;
    if ((rc = make_rows_map(&p.tmU, K, ldk, heads, dp, N, B, 64))) return rc;
    if ((rc = make_rows_map(&p.tmW, Vp, ldv, heads, dp, N, B, 64))) return rc;
    if ((rc = make_t_map(&p.tmT0, KT, ldkt, heads, dp))) return rc;
    p.tmT1 = p.tmT0;
    p.lse = lse; p.delta = delta; p.kmask = key_mask;
    p.out0 = static_cast<__nv_bfloat16*>(dQ); p.ld0 = lddq;
    p.B = B; p.heads = heads; p.N = N; p.d = d;
    rc = d == 40 ? (masked ? launch_bwd<40, false, true>(p, stream) : launch_bwd<40, false, false>(p, stream))
                 : (masked ? launch_bwd<80, false, true>(p, stream) : launch_bwd<80, false, false>(p, stream));
    if (rc) return rc;
  }
  {   // dK, dV: rows = keys (X = K, Y = V), columns = queries (U = Q, W = dO), B operands = dO^T (dV) and Q^T (dK)
    AttnBwdParams p;
    memset(&p, 0, sizeof(p));
    if ((rc = make_rows_map(&p.tmX, K, ldk, heads, dp, N, B, 128))) return rc;
    if ((rc = make_rows_map(&p.tmY, Vp, ldv, heads, dp, N, B, 128))) return rc;
    if ((rc = make_rows_map(&p.tmU, Q, ldq, heads, dp, N, B, 64))) return rc;
    if ((rc = make_rows_map(&p.tmW, dOp, lddo, heads, dp, N, B, 64))) return rc;
    if ((rc = make_t_map(&p.tmT0, dOT, lddot, heads, dp))) return rc;
    if ((rc = make_t_map(&p.tmT1, QT, ldqt, heads, dp))) return rc;
    p.lse = lse; p.delta = delta; p.kmask = key_mask;
    p.out0 = static_cast<__nv_bfloat16*>(dV); p.ld0 = lddv;
    p.out1 = static_cast<__nv_bfloat16*>(dK); p.ld1 = lddk;
    p.B = B; p.heads = heads; p.N = N; p.d = d;
    rc = d == 40 ? (masked ? launch_bwd<40, true, true>(p, stream) : launch_bwd<40, true, false>(p, stream))
                 : (masked ? launch_bwd<80, true, true>(p, stream) : launch_bwd<80, true, false>(p, stream));
    if (rc) return rc;
  }
  return 0;
}

}  // namespace af

#define AF_BWD_CHECK_ARGS(fn)                                                                                          \
  AF_CHECK_ARG(Q && K && Vp && dOp && QT && KT && dOT && lse && delta && dQ && dK && dV, fn ": null pointer");          \
  AF_CHECK_ARG(d == 40 || d == 80, fn ": head dim %d unsupported (40 / 80)", d);                                         \
  AF_CHECK_ARG(B > 0 && heads > 0 && N >= 128 && N % 128 == 0, fn ": N=%d must be a positive multiple of 128", N);       \
  AF_CHECK_ARG(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && lddo % 8 == 0 && ldqt % 8 == 0 && ldkt % 8 == 0 &&       \
                   lddot % 8 == 0 && lddq % 8 == 0 && lddk % 8 == 0 && lddv % 8 == 0,                                  \
               fn ": leading dims must be multiples of 8");                                                             \
  AF_CHECK_ARG(ldqt >= static_cast<long long>(B) * N && ldkt >= static_cast<long long>(B) * N &&                        \
                   lddot >= static_cast<long long>(B) * N,                                                              \
               fn ": transposed operands need B*N columns")

extern "C" int af_attention_bwd_bf16(const void* Q, long long ldq, const void* K, long long ldk, const void* Vp,
                                     long long ldv, const void* dOp, long long lddo, const void* QT, long long ldqt,
                                     const void* KT, long long ldkt, const void* dOT, long long lddot, const float* lse,
                                     const float* delta, void* dQ, long long lddq, void* dK, long long lddk, void* dV,
                                     long long lddv, int B, int heads, int N, int d, cudaStream_t stream) {
  AF_BWD_CHECK_ARGS("af_attention_bwd_bf16");
  return af::attention_bwd(Q, ldq, K, ldk, Vp, ldv, dOp, lddo, QT, ldqt, KT, ldkt, dOT, lddot, lse, delta, nullptr, dQ,
                           lddq, dK, lddk, dV, lddv, B, heads, N, d, stream);
}

extern "C" int af_attention_bwd_masked_bf16(const void* Q, long long ldq, const void* K, long long ldk, const void* Vp,
                                            long long ldv, const void* dOp, long long lddo, const void* QT, long long ldqt,
                                            const void* KT, long long ldkt, const void* dOT, long long lddot,
                                            const float* lse, const float* delta, const unsigned char* key_mask, void* dQ,
                                            long long lddq, void* dK, long long lddk, void* dV, long long lddv, int B,
                                            int heads, int N, int d, cudaStream_t stream) {
  AF_BWD_CHECK_ARGS("af_attention_bwd_masked_bf16");
  AF_CHECK_ARG(key_mask && (reinterpret_cast<uintptr_t>(key_mask) & 15) == 0,
               "af_attention_bwd_masked_bf16: key_mask must be a 16-byte aligned [B, N] byte array");
  return af::attention_bwd(Q, ldq, K, ldk, Vp, ldv, dOp, lddo, QT, ldqt, KT, ldkt, dOT, lddot, lse, delta, key_mask, dQ,
                           lddq, dK, lddk, dV, lddv, B, heads, N, d, stream);
}
