// Fused flash-style attention on tcgen05 / TMEM for the SD-1.5 head dims (40 / 80 / 160), 8 heads.
//
//   O[b, i, h*d : (h+1)*d] = softmax_j( Q[b,i,h] . K[b,j,h] [masked] ) V[b,j,h]
//
// Reference: CrossAttention.forward (ldm/modules/attention.py:172-243): sim = q k^T * d^-1/2 (:199),
// optional key mask -> -finfo.max (:223-232), softmax over keys (:238), out = attn v (:240).  The dense
// [B*8, N, N] score tensor the reference materialises never leaves the SM here: S lives in TMEM, P in
// shared memory, O accumulates in TMEM.
//
// Operand conventions (produced by the projection GEMMs, see adaprompt_b200/attention.py):
//   Q  bf16 [B, Nq, ldq]: head h at columns h*DP.., already multiplied by d^-1/2 * log2(e) (folded into
//      to_q at weight-pack time), so the kernel works in the exp2 domain.
//   K  bf16 [B, Nk, ldk]: head h at columns h*DP...   DP = 48 for d = 40 (pad columns are zeros), else d.
//   Vt bf16 [8*d, ldvt]: V transposed (row = channel, column = key); sample b starts at column b*vt_stride.
//   O  bf16 [B, Nq, 8*d].
// Every tile is loaded by TMA into the canonical 128B-swizzled K-major layout; head dims that are not a
// multiple of 64 simply issue fewer 16-wide MMA k-steps on the last swizzle atom (no HBM padding for
// d = 80 / 160).
//
// Roles (192 threads): warp 0 TMA, warp 1 MMA issue + TMEM alloc, warps 2..5 softmax / correction /
// epilogue with one query row per thread (TMEM lane == row, no shuffles).
#include <math.h>

#include "../../include/adaface_b200.h"
#include "common.cuh"

namespace af {

struct AttnParams {
  float* lse;        // optional [B][heads][Nq]: log2-sum-exp of every query row (training: recomputation of P)
  CUtensorMap tmQ;   // 3-D {ldq, Nq, B}, box {64, 128, 1}
  CUtensorMap tmK;   // 3-D {ldk, Nk, B}, box {64, BLOCK_N, 1}
  CUtensorMap tmV;   // 2-D {total keys, 8*d}, box {64, DV}
  int B, heads, Nq, Nk;
  int d;             // true head dim
  int dp;            // head stride in Q / K columns
  int vt_stride;     // keys per sample in Vt
  const uint8_t* key_mask;  // [B, Nk] (1 = keep) or null
  __nv_bfloat16* out;
  long long ldo;
};

template <int D>
struct AttnCfg;
template <>
struct AttnCfg<40> {
  static constexpr int DK = 48, DV = 48, BLOCK_N = 128, KSTAGES = 3, VSTAGES = 3;
};
template <>
struct AttnCfg<80> {
  static constexpr int DK = 80, DV = 80, BLOCK_N = 128, KSTAGES = 2, VSTAGES = 2;
};
template <>
struct AttnCfg<160> {
  static constexpr int DK = 160, DV = 160, BLOCK_N = 64, KSTAGES = 2, VSTAGES = 2;
};

template <int D>
struct AttnSmem {
  using C = AttnCfg<D>;
  static constexpr int KA = (C::DK + 63) / 64;          // swizzle atoms along the head dim
  static constexpr int PA = C::BLOCK_N / 64;            // swizzle atoms along the key dim
  static constexpr int kQBytes = KA * 128 * 128;
  static constexpr int kKBytes = KA * C::BLOCK_N * 128;
  static constexpr int kVAtomBytes = C::DV * 128;
  static constexpr int kVBytes = PA * kVAtomBytes;
  static constexpr int kPBytes = PA * 128 * 128;
  static constexpr int kQOff = 0;
  static constexpr int kKOff = kQOff + kQBytes;
  static constexpr int kVOff = kKOff + C::KSTAGES * kKBytes;
  static constexpr int kPOff = kVOff + ((C::VSTAGES * kVBytes + 1023) / 1024) * 1024;
  static constexpr int kBarOff = kPOff + kPBytes;
  static constexpr int kTotal = kBarOff + 256 + 1024;
};

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
      "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// 32 lanes x 32 columns into 32 consecutive registers of a larger per-thread array
__device__ __forceinline__ void tmem_ld32p(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}

template <int D>
__global__ void __launch_bounds__(192, 1) attention_kernel(const __grid_constant__ AttnParams p) {
  using C = AttnCfg<D>;
  using S = AttnSmem<D>;
  constexpr int DK = C::DK, DV = C::DV, BN = C::BLOCK_N;
  constexpr int KA = S::KA, PA = S::PA;
  constexpr uint32_t kTmemS0 = 0, kTmemS1 = 128, kTmemO = 256;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::kBarOff);
  uint64_t* q_full = bars;                    // 1
  uint64_t* k_full = q_full + 1;              // KSTAGES
  uint64_t* k_empty = k_full + C::KSTAGES;
  uint64_t* v_full = k_empty + C::KSTAGES;    // VSTAGES
  uint64_t* v_empty = v_full + C::VSTAGES;
  uint64_t* s_full = v_empty + C::VSTAGES;    // 2
  uint64_t* p_full = s_full + 2;              // 1
  uint64_t* pv_done = p_full + 1;             // 1
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(pv_done + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * 128;
  const int h = blockIdx.y;
  const int b = blockIdx.z;
  const int n_blocks = (p.Nk + BN - 1) / BN;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&p.tmQ);
    tma_prefetch_desc(&p.tmK);
    tma_prefetch_desc(&p.tmV);
    mbar_init(q_full, 1);
    for (int s = 0; s < C::KSTAGES; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&k_empty[s], 1);
    }
    for (int s = 0; s < C::VSTAGES; ++s) {
      mbar_init(&v_full[s], 1);
      mbar_init(&v_empty[s], 1);
    }
    mbar_init(&s_full[0], 1);
    mbar_init(&s_full[1], 1);
    mbar_init(p_full, 4);
    mbar_init(pv_done, 1);
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // warp-uniform for the tcgen05 issuer

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      mbar_arrive_expect_tx(q_full, S::kQBytes);
#pragma unroll
      for (int a = 0; a < KA; ++a)
        tma_load_3d(smem + S::kQOff + a * 128 * 128, &p.tmQ, q_full, h * p.dp + a * 64, q0, b);
      int ks = 0, vs = 0;
      uint32_t kph = 0, vph = 0;
      for (int j = 0; j < n_blocks; ++j) {
        mbar_wait(&k_empty[ks], kph ^ 1);
        mbar_arrive_expect_tx(&k_full[ks], S::kKBytes);
#pragma unroll
        for (int a = 0; a < KA; ++a)
          tma_load_3d(smem + S::kKOff + ks * S::kKBytes + a * BN * 128, &p.tmK, &k_full[ks], h * p.dp + a * 64,
                      j * BN, b);
        if (++ks == C::KSTAGES) { ks = 0; kph ^= 1; }
        mbar_wait(&v_empty[vs], vph ^ 1);
        mbar_arrive_expect_tx(&v_full[vs], S::kVBytes);
#pragma unroll
        for (int a = 0; a < PA; ++a)
          tma_load_2d(smem + S::kVOff + vs * S::kVBytes + a * S::kVAtomBytes, &p.tmV, &v_full[vs],
                      b * p.vt_stride + j * BN + a * 64, h * p.d);
        if (++vs == C::VSTAGES) { vs = 0; vph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (whole warp, convergent; the tcgen05
    // instructions are issued by one elected lane instead of under `lane == 0`: no per-instruction waterfall loops)
    {
      constexpr uint32_t idesc_s = umma_idesc_bf16(128, BN);
      constexpr uint32_t idesc_o = umma_idesc_bf16(128, DV);
      const uint32_t q_addr = smem_u32(smem + S::kQOff);
      const uint32_t p_addr = smem_u32(smem + S::kPOff);
      int ks = 0, vs = 0;
      uint32_t kph = 0, vph = 0, pph = 0;
      auto issue_s = [&](int j) {
        mbar_wait(&k_full[ks], kph);
        tc_fence_after();
        const uint32_t k_addr = smem_u32(smem + S::kKOff + ks * S::kKBytes);
        const uint32_t d_tmem = tmem_base + ((j & 1) ? kTmemS1 : kTmemS0);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < DK / 16; ++k) {
            const uint64_t ad = umma_desc_sw128(q_addr + (k >> 2) * 128 * 128) + 2 * (k & 3);
            const uint64_t bd = umma_desc_sw128(k_addr + (k >> 2) * BN * 128) + 2 * (k & 3);
            tc_mma_ss(d_tmem, ad, bd, idesc_s, k != 0 ? 1u : 0u);
          }
          tc_commit(&k_empty[ks]);
          tc_commit(&s_full[j & 1]);
        }
        __syncwarp();
        if (++ks == C::KSTAGES) { ks = 0; kph ^= 1; }
      };
      mbar_wait(q_full, 0);
      issue_s(0);
      for (int j = 0; j < n_blocks; ++j) {
        if (j + 1 < n_blocks) issue_s(j + 1);
        mbar_wait(&v_full[vs], vph);
        mbar_wait(p_full, pph);
        pph ^= 1;
        tc_fence_after();
        const uint32_t v_addr = smem_u32(smem + S::kVOff + vs * S::kVBytes);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BN / 16; ++k) {
            const uint64_t ad = umma_desc_sw128(p_addr + (k >> 2) * 128 * 128) + 2 * (k & 3);
            const uint64_t bd = umma_desc_sw128(v_addr + (k >> 2) * S::kVAtomBytes) + 2 * (k & 3);
            tc_mma_ss(tmem_base + kTmemO, ad, bd, idesc_o, (j | k) != 0 ? 1u : 0u);
          }
          tc_commit(&v_empty[vs]);
          tc_commit(pv_done);
        }
        __syncwarp();
        if (++vs == C::VSTAGES) { vs = 0; vph ^= 1; }
      }
    }
  } else {
    // ------------------------------------------------------------------ softmax / correction / epilogue
    const int qd = warp & 3;
    const int r = qd * 32 + lane;                 // row in tile == TMEM lane
    const uint32_t lane_off = static_cast<uint32_t>(qd * 32) << 16;
    const int q_row = q0 + r;
    const uint8_t* mrow = p.key_mask ? p.key_mask + static_cast<size_t>(b) * p.Nk : nullptr;
    uint8_t* p_smem = smem + S::kPOff;
    const uint32_t sw = static_cast<uint32_t>(r & 7);
    uint8_t* p_row = p_smem + (r >> 3) * 1024 + (r & 7) * 128;

    float m_run = -INFINITY, l_run = 0.f;
    uint32_t pvph = 0;
    for (int j = 0; j < n_blocks; ++j) {
      const uint32_t s_addr = tmem_base + ((j & 1) ? kTmemS1 : kTmemS0) + lane_off;
      const int key0 = j * BN;
      mbar_wait(&s_full[j & 1], (j >> 1) & 1);
      tc_fence_after();
      // whole score row -> registers (one TMEM read), then everything below is branch-free straight-line code
      float sc[BN];
#pragma unroll
      for (int c = 0; c < BN; c += 32) tmem_ld32p(s_addr + c, reinterpret_cast<uint32_t*>(sc) + c);
      tmem_ld_wait();
      if (key0 + BN > p.Nk || mrow != nullptr) {  // warp-uniform: only the tail block / an explicit key mask
#pragma unroll
        for (int e = 0; e < BN; ++e) {
          const int key = key0 + e;
          bool ok = key < p.Nk;
          if (mrow != nullptr) ok = ok && (__ldg(mrow + min(key, p.Nk - 1)) != 0);
          sc[e] = ok ? sc[e] : -INFINITY;
        }
      }
      float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
      for (int e = 0; e < BN; e += 4) {
        mx4[0] = fmaxf(mx4[0], sc[e]);
        mx4[1] = fmaxf(mx4[1], sc[e + 1]);
        mx4[2] = fmaxf(mx4[2], sc[e + 2]);
        mx4[3] = fmaxf(mx4[3], sc[e + 3]);
      }
      const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      const float m_new = fmaxf(m_run, mx);
      const float m_use = (m_new == -INFINITY) ? 0.f : m_new;
      const float alpha = fast_exp2(m_run - m_use);  // 0 on the first block
      // P buffer free and O stable once the previous PV finished
      if (j > 0) {
        mbar_wait(pv_done, pvph);
        pvph ^= 1;
        tc_fence_after();
        if (__any_sync(0xffffffffu, alpha != 1.0f)) {
#pragma unroll 1
          for (int c = 0; c < DV; c += 16) {
            uint32_t o[16];
            tmem_ld16(tmem_base + kTmemO + lane_off + c, o);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 16; ++e) o[e] = __float_as_uint(__uint_as_float(o[e]) * alpha);
            tmem_st16(tmem_base + kTmemO + lane_off + c, o);
          }
          tmem_st_wait();
        }
      }
      // P = exp2(S - m) -> bf16 -> swizzled smem; four independent partial sums keep the FADD chain short
      float l4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int c8 = 0; c8 < BN; c8 += 8) {
        float pe[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          pe[e] = fast_exp2(sc[c8 + e] - m_use);
          l4[e & 3] += pe[e];
        }
        uint4 pk;
        pk.x = pack_bf16x2(pe[0], pe[1]);
        pk.y = pack_bf16x2(pe[2], pe[3]);
        pk.z = pack_bf16x2(pe[4], pe[5]);
        pk.w = pack_bf16x2(pe[6], pe[7]);
        uint8_t* atom = p_row + (c8 >> 6) * (128 * 128);
        const uint32_t chunk = static_cast<uint32_t>((c8 & 63) >> 3);  // 16-byte chunk inside the 128-byte row
        sts128(smem_u32(atom) + ((chunk ^ sw) << 4), pk.x, pk.y, pk.z, pk.w);   // STS, not a generic ST.E
      }
      l_run = l_run * alpha + ((l4[0] + l4[1]) + (l4[2] + l4[3]));
      m_run = m_new;
      fence_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
    }
    // epilogue: O / l -> bf16
    mbar_wait(pv_done, pvph);
    tc_fence_after();
    const float inv_l = l_run > 0.f ? 1.0f / l_run : 0.f;
    if (p.lse != nullptr && q_row < p.Nq)
      p.lse[(static_cast<size_t>(b) * p.heads + h) * p.Nq + q_row] = l_run > 0.f ? m_run + __log2f(l_run) : INFINITY;
    __nv_bfloat16* orow = p.out + (static_cast<size_t>(b) * p.Nq + q_row) * p.ldo + h * p.d;
#pragma unroll 1
    for (int c = 0; c < DV; c += 16) {
      uint32_t o[16];
      tmem_ld16(tmem_base + kTmemO + lane_off + c, o);
      tmem_ld_wait();
      if (q_row < p.Nq) {
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          if (c + g * 8 < p.d) {
            uint4 pk;
            pk.x = pack_bf16x2(__uint_as_float(o[g * 8 + 0]) * inv_l, __uint_as_float(o[g * 8 + 1]) * inv_l);
            pk.y = pack_bf16x2(__uint_as_float(o[g * 8 + 2]) * inv_l, __uint_as_float(o[g * 8 + 3]) * inv_l);
            pk.z = pack_bf16x2(__uint_as_float(o[g * 8 + 4]) * inv_l, __uint_as_float(o[g * 8 + 5]) * inv_l);
            pk.w = pack_bf16x2(__uint_as_float(o[g * 8 + 6]) * inv_l, __uint_as_float(o[g * 8 + 7]) * inv_l);
            *reinterpret_cast<uint4*>(orow + c + g * 8) = pk;
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int D>
static int launch_attention(const AttnParams& p, cudaStream_t stream) {
  using S = AttnSmem<D>;
  static bool configured = false;
  if (!configured) {
    AF_CUDA(cudaFuncSetAttribute(attention_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal));
    configured = true;
  }
  dim3 grid((p.Nq + 127) / 128, p.heads, p.B);
  attention_kernel<D><<<grid, 192, S::kTotal, stream>>>(p);
  AF_LAUNCH_CHECK("attention_kernel");
  return 0;
}

// A sample whose key mask keeps no key.  The reference fills masked scores with -finfo.max (attention.py:223-232), so
// such a row's softmax is uniform over the sample's Nk keys and its output is the mean of V over them.  The attention
// kernels end these rows with a zero row sum instead; this pass, run after whichever kernel ran, overwrites them with
// that mean (fp32 sum, rounded to bf16) and their lse with +inf.  grid (ceil(heads*d / 32), B), 256 threads: a block
// owns 32 channels of one sample and returns at once when the sample attends to any key.
__global__ void __launch_bounds__(256) attention_empty_mask_kernel(const uint8_t* __restrict__ key_mask,
                                                                   const __nv_bfloat16* __restrict__ Vt, long long ldvt,
                                                                   int kv_stride, int heads, int Nq, int Nk, int d,
                                                                   __nv_bfloat16* __restrict__ out, float* __restrict__ lse) {
  const int b = blockIdx.y;
  const int C = heads * d;
  const int c0 = blockIdx.x * 32;
  const uint8_t* m = key_mask + static_cast<size_t>(b) * Nk;
  int any = 0;
  for (int j = threadIdx.x; j < Nk; j += blockDim.x) any |= m[j];
  if (__syncthreads_or(any)) return;
  __shared__ float mean[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int c = warp; c < 32 && c0 + c < C; c += 8) {
    const __nv_bfloat16* row = Vt + static_cast<size_t>(c0 + c) * ldvt + static_cast<size_t>(b) * kv_stride;
    float s = 0.f;
    for (int j = lane; j < Nk; j += 32) s += __bfloat162float(row[j]);
    s = warp_sum(s);
    if (lane == 0) mean[c] = s / static_cast<float>(Nk);
  }
  __syncthreads();
  if (c0 + lane < C) {
    const __nv_bfloat16 v = __float2bfloat16(mean[lane]);
    for (int i = warp; i < Nq; i += 8) out[(static_cast<size_t>(b) * Nq + i) * C + c0 + lane] = v;
  }
  if (lse != nullptr && blockIdx.x == 0)
    for (int i = threadIdx.x; i < heads * Nq; i += blockDim.x) lse[static_cast<size_t>(b) * heads * Nq + i] = INFINITY;
}

}  // namespace af

namespace af {
int xattn_dispatch(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt, long long ldvt,
                   int kv_stride, const unsigned char* key_mask, void* O, int B, int heads, int Nq, int Nk, int d,
                   float* lse, cudaStream_t stream);  // xattn.cu
int attention_tile_dispatch(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt, long long ldvt,
                            int kv_stride, const unsigned char* key_mask, void* O, int B, int heads, int Nq, int Nk,
                            int d, float* lse, long long* trace, cudaStream_t stream);  // attention_tile.cu
}

using namespace af;

static int attention_impl(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt, long long ldvt,
                          int kv_stride, const unsigned char* key_mask, void* O, float* lse, long long* trace, int B,
                          int heads, int Nq, int Nk, int d, cudaStream_t stream);

extern "C" int af_attention_bf16(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt,
                                 long long ldvt, int kv_stride, const unsigned char* key_mask, void* O, int B,
                                 int heads, int Nq, int Nk, int d, cudaStream_t stream) {
  return attention_impl(Q, ldq, K, ldk, Vt, ldvt, kv_stride, key_mask, O, nullptr, nullptr, B, heads, Nq, Nk, d, stream);
}

extern "C" int af_attention_bf16_lse(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt,
                                     long long ldvt, int kv_stride, const unsigned char* key_mask, void* O, float* lse,
                                     int B, int heads, int Nq, int Nk, int d, cudaStream_t stream) {
  return attention_impl(Q, ldq, K, ldk, Vt, ldvt, kv_stride, key_mask, O, lse, nullptr, B, heads, Nq, Nk, d, stream);
}

extern "C" int af_attention_bf16_trace(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt,
                                       long long ldvt, int kv_stride, void* O, long long* trace, int B, int heads, int Nq,
                                       int Nk, int d, cudaStream_t stream) {
  AF_CHECK_ARG(trace != nullptr, "af_attention_bf16_trace: null trace buffer");
  AF_CHECK_ARG((d == 40 || d == 80) && Nk > 128 && Nk % (d == 40 ? 128 : 64) == 0,
               "af_attention_bf16_trace: only the long-sequence d = 40 / 80 kernel with whole key blocks has a timeline");
  return attention_impl(Q, ldq, K, ldk, Vt, ldvt, kv_stride, nullptr, O, nullptr, trace, B, heads, Nq, Nk, d, stream);
}

// picks and launches one of the three kernel families from the shape
static int attention_launch(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt, long long ldvt,
                            int kv_stride, const unsigned char* key_mask, void* O, float* lse, long long* trace, int B,
                            int heads, int Nq, int Nk, int d, cudaStream_t stream);

static int attention_impl(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt, long long ldvt,
                          int kv_stride, const unsigned char* key_mask, void* O, float* lse, long long* trace, int B,
                          int heads, int Nq, int Nk, int d, cudaStream_t stream) {
  const int rc = attention_launch(Q, ldq, K, ldk, Vt, ldvt, kv_stride, key_mask, O, lse, trace, B, heads, Nq, Nk, d,
                                  stream);
  if (rc != 0 || key_mask == nullptr) return rc;
  dim3 grid((heads * d + 31) / 32, B);
  attention_empty_mask_kernel<<<grid, 256, 0, stream>>>(key_mask, static_cast<const __nv_bfloat16*>(Vt), ldvt, kv_stride,
                                                        heads, Nq, Nk, d, static_cast<__nv_bfloat16*>(O), lse);
  AF_LAUNCH_CHECK("attention_empty_mask_kernel");
  return 0;
}

static int attention_launch(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt, long long ldvt,
                            int kv_stride, const unsigned char* key_mask, void* O, float* lse, long long* trace, int B,
                            int heads, int Nq, int Nk, int d, cudaStream_t stream) {
  AF_CHECK_ARG(Q && K && Vt && O, "af_attention_bf16: null pointer");
  AF_CHECK_ARG(d == 40 || d == 80 || d == 160, "af_attention_bf16: head dim %d unsupported (40/80/160)", d);
  AF_CHECK_ARG(B > 0 && heads > 0 && Nq > 0 && Nk > 0 && kv_stride >= Nk, "af_attention_bf16: bad sizes");
  AF_CHECK_ARG(ldq % 8 == 0 && ldk % 8 == 0 && ldvt % 8 == 0, "af_attention_bf16: leading dims must be multiples of 8");
  AF_CHECK_ARG(ldvt >= 64, "af_attention_bf16: ldvt=%lld must be >= 64 (one 128-byte swizzle row)", ldvt);
  // TMA needs every box to start on a 16-byte boundary: sample b's keys start at column b*kv_stride of V^T
  AF_CHECK_ARG(B == 1 || kv_stride % 8 == 0, "af_attention_bf16: kv_stride=%d must be a multiple of 8 when B > 1", kv_stride);
  if (Nq >= 256 && Nk <= 128 && (d == 40 || d == 80))    // short context, K / V resident per (sample, head) (xattn.cu)
    return xattn_dispatch(Q, ldq, K, ldk, Vt, ldvt, kv_stride, key_mask, O, B, heads, Nq, Nk, d, lse, stream);
  if (Nk > 128 && (d == 40 || d == 80))                  // one query tile per CTA, two CTAs per SM (attention_tile.cu)
    return attention_tile_dispatch(Q, ldq, K, ldk, Vt, ldvt, kv_stride, key_mask, O, B, heads, Nq, Nk, d, lse, trace,
                                   stream);
  AttnParams p;
  memset(&p, 0, sizeof(p));
  const int dp = d == 40 ? 48 : d;
  const int bn = d == 160 ? 64 : 128;
  const int dv = dp;
  AF_CHECK_ARG(ldq >= static_cast<long long>(heads) * dp && ldk >= static_cast<long long>(heads) * dp,
               "af_attention_bf16: ldq/ldk smaller than heads*%d", dp);
  {
    // dim 0 is the valid width (heads*dp), not the row pitch: boxes of the last head that stick out are
    // zero-filled instead of reading whatever follows (e.g. the K half of a fused [Q|K] buffer)
    uint64_t dims[3] = {static_cast<uint64_t>(heads) * dp, static_cast<uint64_t>(Nq), static_cast<uint64_t>(B)};
    uint64_t str[2] = {static_cast<uint64_t>(ldq) * 2, static_cast<uint64_t>(Nq) * ldq * 2};
    uint32_t box[3] = {64, 128, 1};
    int rc = make_tmap_bf16(&p.tmQ, Q, 3, dims, str, box);
    if (rc) return rc;
  }
  {
    uint64_t dims[3] = {static_cast<uint64_t>(heads) * dp, static_cast<uint64_t>(Nk), static_cast<uint64_t>(B)};
    uint64_t str[2] = {static_cast<uint64_t>(ldk) * 2, static_cast<uint64_t>(kv_stride) * ldk * 2};
    uint32_t box[3] = {64, static_cast<uint32_t>(bn), 1};
    int rc = make_tmap_bf16(&p.tmK, K, 3, dims, str, box);
    if (rc) return rc;
  }
  {
    uint64_t dims[2] = {static_cast<uint64_t>(ldvt), static_cast<uint64_t>(heads) * d};
    uint64_t str[1] = {static_cast<uint64_t>(ldvt) * 2};
    uint32_t box[2] = {64, static_cast<uint32_t>(dv)};
    int rc = make_tmap_bf16(&p.tmV, Vt, 2, dims, str, box);
    if (rc) return rc;
  }
  p.B = B; p.heads = heads; p.Nq = Nq; p.Nk = Nk; p.d = d; p.dp = dp; p.vt_stride = kv_stride;
  p.key_mask = key_mask;
  p.lse = lse;
  p.out = static_cast<__nv_bfloat16*>(O);
  p.ldo = static_cast<long long>(heads) * d;
  switch (d) {
    case 40: return launch_attention<40>(p, stream);
    case 80: return launch_attention<80>(p, stream);
    default: return launch_attention<160>(p, stream);
  }
}
