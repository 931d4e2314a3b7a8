// Self-attention for the long-sequence layers (more than 128 keys, head dims 40 / 80): one 128-query tile per CTA, TWO
// CTAs per SM.
//
// Reference semantics: CrossAttention.forward (ldm/modules/attention.py:172-243), same operand conventions as
// attention.cu (Q pre-scaled into the exp2 domain, K-major bf16 tiles, V transposed).
//
// Why this shape (profiles/r02_attention.md).  At d = 40 one exponential buys only 160 FLOP, so the layer lives between
// the ex2 unit (16 results / clk / SM: 0.48 ms at N = 4096, B = 16) and the latency of the hand-over chains between the
// softmax warps and the MMA issuer (0.52 ms with the exponentials removed).  The round-1 kernels (256 queries per CTA,
// one CTA per SM, two threads per row) ran every warp of the SM through that chain in phase and spent 580 instructions
// per warp and key block on ~320 useful ones.  Here
//   * two independent CTAs share an SM, so one CTA's chain runs under the other CTA's exponentials;
//   * the row sum l is not accumulated by the softmax threads: row D of the V^T tile in shared memory is a constant
//     row of ones (the TMA box covers rows 0..D-1 only and never overwrites it), so column D of the O accumulator IS
//     sum_j P_ij - computed by the tensor core from exactly the bf16 probabilities the numerator uses;
//   * the lazy softmax reference has a 2^64 window and starts at 0 whenever the first block's maximum lies inside it
//     (bf16 P and the fp32 accumulators have the exponent range to spare), so for the UNet's score range the
//     subtraction disappears from the loop: per score one MUFU (or, every POLY-th, an FMA-pipe polynomial), half an
//     F2FP and half an FMNMX3;
//   * no run-time options, probes or generic-address shared-memory accesses in the loop.
//
//   warp 0      TMA producer (Q once; K / V ring)          warp 1   S issuer (S_{j+1} early)    warp 2   PV issuer
//   warp 3      idle (setmaxnreg works per warpgroup)      warps 4-7 softmax, one thread per query row (TMEM lane = row)
// P goes to the PV MMA through tensor memory (tcgen05.st, A operand in TMEM).
#include <type_traits>
#include <math.h>

#include "../../include/adaface_b200.h"
#include "common.cuh"
#include "attn_tile_common.cuh"

namespace af {

struct AttnTileParams {
  long long* trace;  // TRACE instantiation only (af_attention_bf16_trace): softmax warp 4 of the first 512 CTAs (linear
                     // id) [cta][64 key blocks][8 events] clock64 stamps; then 512 SM ids; then MMA issuer and producer
                     // of CTA 0, [64][8] each
  float* lse;        // optional [B][heads][Nq] log2-sum-exp per query row
  CUtensorMap tmQ;   // 3-D {heads*dp, Nq, B}, box {64, 128, 1}
  CUtensorMap tmK;   // 3-D {heads*dp, Nk, B}, box {64, BLOCK_N, 1}
  CUtensorMap tmV;   // 2-D {ldvt, heads*d}, box {64, D}   (D rows: rows D.. of the shared-memory tile are constants)
  int B, heads, Nq, Nk;
  int d, dp, kv_stride;
  const uint8_t* key_mask;
  __nv_bfloat16* out;
  long long ldo;
};

template <int D>
struct TileCfg;
template <>
struct TileCfg<40> {
  // TMEM: S [0,128) | O [128,176) | P [192,256)
  static constexpr int DK = 48, DV = 48, BLOCK_N = 128, KSTAGES = 3, VSTAGES = 3;
  static constexpr uint32_t kTmemS = 0, kTmemO = 128, kTmemP = 192, kTmemCols = 256;
};
template <>
struct TileCfg<80> {
  // TMEM: S [0,64) | O [64,160) | P [160,192)
  static constexpr int DK = 80, DV = 96, BLOCK_N = 64, KSTAGES = 3, VSTAGES = 2;
  static constexpr uint32_t kTmemS = 0, kTmemO = 64, kTmemP = 160, kTmemCols = 256;
};

template <int D>
struct TileSmem {
  using C = TileCfg<D>;
  static constexpr int KA = (C::DK + 63) / 64;            // 64-column swizzle atoms along the head dim
  static constexpr int PA = C::BLOCK_N / 64;              // 64-key swizzle atoms along the key dim
  static constexpr int kQBytes = KA * 128 * 128;
  static constexpr int kKBytes = KA * C::BLOCK_N * 128;
  static constexpr int kVAtomBytes = C::DV * 128;         // DV rows of 64 keys
  static constexpr int kVBytes = PA * kVAtomBytes;
  static constexpr int kVTxBytes = PA * D * 128;          // what the TMA box {64, D} delivers per stage
  static constexpr int kQOff = 0;
  static constexpr int kKOff = kQOff + kQBytes;
  static constexpr int kVOff = kKOff + C::KSTAGES * kKBytes;
  static constexpr int kBarOff = kVOff + C::VSTAGES * kVBytes;
  static constexpr int kTotal = kBarOff + 256 + 1024;
  static_assert(kVAtomBytes % 1024 == 0 && kKBytes % 1024 == 0 && kQBytes % 1024 == 0, "swizzle atoms are 1024-byte aligned");
};

template <int POLY>
__device__ __forceinline__ float tile_exp2(int i, float x) {   // i is a compile-time constant after unrolling
  if constexpr (POLY > 0) {
    if (i % POLY == POLY - 1) return tile_exp2_poly(x);
  }
  return fast_exp2(x);
}

// POLY: every POLY-th exponential on the FMA pipe (0 = none).  MASKED: instantiation for an explicit key mask or a
// ragged last key block (the UNet's own shapes need neither).  TRACE: clock64 timeline (af_attention_bf16_trace).
template <int D, int POLY, bool MASKED, bool TRACE>
__global__ void __launch_bounds__(256, 2) attention_tile_kernel(const __grid_constant__ AttnTileParams p) {
  using C = TileCfg<D>;
  using S = TileSmem<D>;
  constexpr int DK = C::DK, DV = C::DV, BN = C::BLOCK_N;
  constexpr int KA = S::KA, PA = S::PA;
  static_assert(BN % 32 == 0, "a softmax thread owns whole 32-column TMEM loads");
  static_assert(D % 8 == 0 && DV % 16 == 0 && DV >= D + 8, "V^T tile: D data rows, then the ones row, then zero rows");
  static_assert(C::kTmemO + DV <= C::kTmemP && C::kTmemP + BN / 2 <= C::kTmemCols, "TMEM column map");
  // Lazy reference (log2 domain): it only moves when a block maximum exceeds it by more than the window, and the first
  // reference is 0 whenever the first block's maximum lies inside the window.  P <= 2^64 in bf16, O <= 2^64 * Nk * |v|
  // in fp32; scores more than 2^-62 below the row maximum are irrelevant.
  constexpr float kWindow = 64.0f;
  // GUARDLESS (d = 40, no mask): the fast path carries no per-block overflow guard at all - 87 of the ~555 instructions a
  // softmax warp issues per key block, and that warp's issue rate is what bounds the kernel (profiles/r02_attention.md).
  // Instead the row sums and the O accumulators are checked for inf / NaN once, at the end of the tile (any overflow of
  // P, l or O propagates there), and a tile that trips is run a second time on the general path.
  constexpr bool GUARDLESS = D == 40 && !MASKED;
  constexpr int kPasses = GUARDLESS ? 2 : 1;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t smem_base = smem_u32(smem);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::kBarOff);
  uint64_t* q_full = bars;                     // 1
  uint64_t* k_full = q_full + 1;               // KSTAGES
  uint64_t* k_empty = k_full + C::KSTAGES;
  uint64_t* v_full = k_empty + C::KSTAGES;     // VSTAGES
  uint64_t* v_empty = v_full + C::VSTAGES;
  uint64_t* s_full = v_empty + C::VSTAGES;     // S_j in TMEM
  uint64_t* s_free = s_full + 1;               // S_j copied to registers by every softmax warp
  uint64_t* p_full = s_free + 1;               // P_j in TMEM
  uint64_t* pv_done = p_full + 1;              // the MMAs of PV_j are complete (P buffer and O reusable)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(pv_done + 1);
  volatile int* redo = reinterpret_cast<volatile int*>(tmem_slot + 1);   // GUARDLESS: the tile overflowed, run it again

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * 128;
  const int h = blockIdx.y;
  const int b = blockIdx.z;
  const int n_blocks = (p.Nk + BN - 1) / BN;
  const int cta_lin = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
  auto stamp = [&](int actor, int j, int ev) {   // actor 0: softmax warp 4, 2: MMA issuer, 3: producer
    if constexpr (TRACE) {
      if (lane == 0 && j < 64) {
        if (actor < 2) {
          if (cta_lin < 512) p.trace[(cta_lin * 64 + j) * 8 + ev] = clock64();
        } else if (cta_lin == 0) {
          p.trace[512 * 64 * 8 + 512 + ((actor - 2) * 64 + j) * 8 + ev] = clock64();
        }
      }
    }
  };
  if constexpr (TRACE) {
    if (threadIdx.x == 0 && cta_lin < 512) {
      uint32_t smid;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      p.trace[512 * 64 * 8 + cta_lin] = smid;
    }
  }

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
    mbar_init(s_full, 1);
    mbar_init(s_free, 4);
    mbar_init(p_full, 4);
    mbar_init(pv_done, 1);
    mbar_fence_init();
    *redo = 0;
  }
  // constant rows of every V^T stage: row D = 1.0 (column D of O becomes the row sum), rows D+1 .. DV-1 = 0.
  // A row of equal values is invariant under the 128-byte swizzle; the TMA box never touches these rows.
  {
    constexpr int kConstChunks = (DV - D) * 8;       // 16-byte chunks per atom
    for (int i = threadIdx.x; i < C::VSTAGES * PA * kConstChunks; i += 256) {
      const int atom = i / kConstChunks, chunk = i % kConstChunks;
      const uint32_t addr = smem_base + S::kVOff + (atom / PA) * S::kVBytes + (atom % PA) * S::kVAtomBytes + D * 128 + chunk * 16;
      const uint32_t v = chunk < 8 ? 0x3F803F80u : 0u;
      sts128(addr, v, v, v, v);
    }
    fence_async_smem();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, C::kTmemCols);
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
        mbar_arrive_expect_tx(q_full, S::kQBytes);
#pragma unroll
        for (int a = 0; a < KA; ++a)
          tma_load_3d(smem + S::kQOff + a * 128 * 128, &p.tmQ, q_full, h * p.dp + a * 64, q0, b);
      }
    }
    // K / V ring positions, accumulator parities and the running block index survive a second pass over the tile
    int ks = 0, vs = 0, kslot = 0, vslot = 0, gj = 0;
    uint32_t kph = 0, vph = 0, kph_i = 0, vph_i = 0;
    for (int pass = 0; pass < kPasses; ++pass) {
    if (warp == 0) {
      if (lane == 0) {
        for (int j = 0; j < n_blocks; ++j) {
          stamp(3, j, 0);
          mbar_wait_lean(&k_empty[ks], kph ^ 1);
          stamp(3, j, 1);
          mbar_arrive_expect_tx(&k_full[ks], S::kKBytes);
#pragma unroll
          for (int a = 0; a < KA; ++a)
            tma_load_3d(smem + S::kKOff + ks * S::kKBytes + a * BN * 128, &p.tmK, &k_full[ks], h * p.dp + a * 64,
                        j * BN, b);
          if (++ks == C::KSTAGES) { ks = 0; kph ^= 1; }
          stamp(3, j, 2);
          mbar_wait_lean(&v_empty[vs], vph ^ 1);
          stamp(3, j, 3);
          mbar_arrive_expect_tx(&v_full[vs], S::kVTxBytes);
#pragma unroll
          for (int a = 0; a < PA; ++a)
            tma_load_2d(smem + S::kVOff + vs * S::kVBytes + a * S::kVAtomBytes, &p.tmV, &v_full[vs],
                        b * p.kv_stride + j * BN + a * 64, h * p.d);
          if (++vs == C::VSTAGES) { vs = 0; vph ^= 1; }
        }
      }
    } else if (warp == 1) {
      // ------------------------------------------------------------------ S issuer (whole warp walks the chain, one
      // elected lane issues): S_0, then S_{j+1} as soon as S_j has been copied out.  The PV MMAs have their own issuer
      // warp: the two chains touch different TMEM columns and are ordered by the barriers alone, and each walks half as
      // many waits per key block as one combined issuer did (its ~1400 serial cycles per block were the non-ex2 floor
      // of the kernel, profiles/r02_attention.md).
      constexpr uint32_t idesc_s = umma_idesc_bf16(128, BN);
      const uint32_t q_addr = smem_base + S::kQOff;
      const uint32_t tm_s = tmem_base + C::kTmemS;
      if (pass == 0) mbar_wait_lean(q_full, 0);
      for (int j = 0; j < n_blocks; ++j, ++gj) {
        stamp(2, j, 0);
        mbar_wait_lean(&k_full[kslot], kph_i);
        stamp(2, j, 1);
        if (gj > 0) mbar_wait_lean(s_free, (gj - 1) & 1);
        tc_fence_after();
        stamp(2, j, 2);
        const uint32_t k_addr = smem_base + S::kKOff + kslot * S::kKBytes;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < DK / 16; ++k) {
            const uint64_t ad = umma_desc_sw128(q_addr + (k >> 2) * 128 * 128) + 2 * (k & 3);
            const uint64_t bd = umma_desc_sw128(k_addr + (k >> 2) * BN * 128) + 2 * (k & 3);
            tc_mma_ss(tm_s, ad, bd, idesc_s, k != 0 ? 1u : 0u);
          }
          tc_commit(s_full);
          tc_commit(&k_empty[kslot]);
        }
        __syncwarp();
        stamp(2, j, 3);
        if (++kslot == C::KSTAGES) { kslot = 0; kph_i ^= 1; }
      }
    } else if (warp == 2) {
      // ------------------------------------------------------------------ PV issuer: O += P_j V_j once P_j is in TMEM
      constexpr uint32_t idesc_o = umma_idesc_bf16(128, DV);
      const uint32_t tm_o = tmem_base + C::kTmemO, tm_p = tmem_base + C::kTmemP;
      for (int j = 0; j < n_blocks; ++j, ++gj) {
        mbar_wait_lean(&v_full[vslot], vph_i);
        stamp(2, j, 4);
        const uint32_t v_addr = smem_base + S::kVOff + vslot * S::kVBytes;
        mbar_wait_lean(p_full, gj & 1);
        tc_fence_after();
        stamp(2, j, 5);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BN / 16; ++k) {      // 16-key steps of the block
            const uint64_t bd = umma_desc_sw128(v_addr + (k >> 2) * S::kVAtomBytes) + 2 * (k & 3);
            tc_mma_ts(tm_o, tm_p + k * 8, bd, idesc_o, (j | k) != 0 ? 1u : 0u);
          }
          tc_commit(pv_done);
          tc_commit(&v_empty[vslot]);
        }
        __syncwarp();
        stamp(2, j, 6);
        if (++vslot == C::VSTAGES) { vslot = 0; vph_i ^= 1; }
      }
    }
    if constexpr (GUARDLESS) {
      if (pass == 0) {
        tc_fence_before();
        __syncthreads();                 // the softmax warps have judged the tile (and read O)
        tc_fence_after();
        if (*redo == 0) break;
      }
    }
    }  // pass
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
    // ------------------------------------------------------------------ softmax: one thread per query row
    const int qd = warp & 3;                      // TMEM lane quarter (hardware: warp id % 4)
    const int r = qd * 32 + lane;                 // row in tile == TMEM lane
    const uint32_t lane_off = static_cast<uint32_t>(qd * 32) << 16;
    const int q_row = q0 + r;
    const uint8_t* mrow = p.key_mask ? p.key_mask + static_cast<size_t>(b) * p.Nk : nullptr;
    const uint32_t s_addr = tmem_base + C::kTmemS + lane_off;
    const uint32_t o_addr = tmem_base + C::kTmemO + lane_off;
    const uint32_t pt_addr = tmem_base + C::kTmemP + lane_off;
    const uint32_t a_s_full = smem_u32(s_full), a_s_free = smem_u32(s_free);
    const uint32_t a_p_full = smem_u32(p_full), a_pv_done = smem_u32(pv_done);
    const bool tw = TRACE && warp == 4;
    uint32_t par = 0;                             // running block index & 1 (survives a second pass)
    for (int pass = 0; pass < kPasses; ++pass) {
    const bool safe = pass != 0;                  // second pass of a tile that overflowed: general path only
    float m_ref = -INFINITY;
    for (int j = 0; j < n_blocks; ++j, par ^= 1) {
      if (tw) stamp(0, j, 0);
      mbar_wait_lean(a_s_full, par);
      tc_fence_after();
      if (tw) stamp(0, j, 1);
      float sc[BN];
      // first 32 columns now, the rest in flight under the exponentials of the first chunk (fast path below)
      tile_ld32(s_addr, reinterpret_cast<uint32_t*>(sc));
      tmem_ld_wait();
#pragma unroll
      for (int c = 32; c < BN; c += 32) tile_ld32(s_addr + c, reinterpret_cast<uint32_t*>(sc) + c);
      bool s_released = false;
      auto release_s = [&]() {                    // every column of S_j is in registers: the S issuer may overwrite it
        if (!s_released) {
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a_s_free) : "memory");
          s_released = true;
        }
      };
      if constexpr (MASKED) {
        release_s();
        if (tw) stamp(0, j, 2);
        // keep-bits of the block's keys, 32 per ballot (lane l probes key key0 + c + l), then compile-time bit tests
        const int key0 = j * BN;
#pragma unroll
        for (int c = 0; c < BN; c += 32) {
          const int key = key0 + c + lane;
          bool ok = key < p.Nk;
          if (ok && mrow != nullptr) ok = __ldg(mrow + key) != 0;
          const uint32_t keep = __ballot_sync(0xffffffffu, ok);
#pragma unroll
          for (int e = 0; e < 32; ++e) sc[c + e] = ((keep >> e) & 1u) ? sc[c + e] : -INFINITY;
        }
      }
      auto block_max = [&]() {
        float mx8[8];   // eight independent 3-input max chains
#pragma unroll
        for (int c = 0; c < 8; ++c) mx8[c] = fmaxf(sc[2 * c], sc[2 * c + 1]);
#pragma unroll
        for (int e = 16; e < BN; e += 16)
#pragma unroll
          for (int c = 0; c < 8; ++c) mx8[c] = fmaxf(mx8[c], fmaxf(sc[e + 2 * c], sc[e + 2 * c + 1]));
        return fmaxf(fmaxf(fmaxf(mx8[0], mx8[1]), fmaxf(mx8[2], mx8[3])),
                     fmaxf(fmaxf(mx8[4], mx8[5]), fmaxf(mx8[6], mx8[7])));
      };
      auto wait_p_free = [&]() {                  // the P buffer has been consumed by the previous PV
        if (j > 0 || pass > 0) {
          mbar_wait_lean(a_pv_done, par ^ 1);
          tc_fence_after();
        }
      };
      auto exp_block = [&](auto sub, float m_use) {   // sub: subtract the reference (general) or not (reference 0)
#pragma unroll
        for (int c = 0; c < BN; c += 32) {
          if (c == 32) {                              // chunk 0 is queued on the ex2 unit: now collect the other loads
            release_s();
            if (tw) stamp(0, j, 2);
          }
          uint32_t pk[16];
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            const float p0 = tile_exp2<POLY>(e, decltype(sub)::value ? sc[c + e] - m_use : sc[c + e]);
            const float p1 = tile_exp2<POLY>(e + 1, decltype(sub)::value ? sc[c + e + 1] - m_use : sc[c + e + 1]);
            pk[e >> 1] = pack_bf16x2(p0, p1);
          }
          tile_st16(pt_addr + c / 2, pk);
        }
      };
      // Fast path (the reference is 0 in every row of the warp - always, after the first block, for UNet scores): the
      // exponentials do not depend on the block maximum, so they are issued straight away and the maximum is only the
      // overflow guard, computed next to them (ALU pipe under the MUFU queue) instead of in front of them.  A guard trip
      // re-does the block on the general path (P is rewritten before it is handed over).
      bool fast = !safe && __all_sync(0xffffffffu, m_ref == 0.f);
      if (fast) {
        if (tw) stamp(0, j, 3);
        // The first kLate x 32 exponentials go to REGISTERS before the wait for the P buffer (PV_{j-1} may still be reading
        // it): the wait - 360 cycles at the head of the chain before - hides behind them; every later chunk is stored as soon
        // as it is computed (storing everything late was slower: the stores then drain at the tail of the block).
#ifndef AF_TILE_LATE_CHUNKS
#define AF_TILE_LATE_CHUNKS 2
#endif
        constexpr int kLate = AF_TILE_LATE_CHUNKS * 32 < BN ? AF_TILE_LATE_CHUNKS * 32 : BN / 2;
        uint32_t pk0[kLate / 2];
#pragma unroll
        for (int c = 0; c < kLate; c += 32) {
          if (c == 32) release_s();
#pragma unroll
          for (int e = 0; e < 32; e += 2)
            pk0[(c + e) >> 1] = pack_bf16x2(tile_exp2<POLY>(e, sc[c + e]), tile_exp2<POLY>(e + 1, sc[c + e + 1]));
        }
        release_s();
        if (tw) stamp(0, j, 2);
        wait_p_free();
        if (tw) stamp(0, j, 4);
#pragma unroll
        for (int c = 0; c < kLate; c += 32) tile_st16(pt_addr + c / 2, *reinterpret_cast<uint32_t (*)[16]>(&pk0[c >> 1]));
#pragma unroll
        for (int c = kLate; c < BN; c += 32) {
          uint32_t pk[16];
#pragma unroll
          for (int e = 0; e < 32; e += 2)
            pk[e >> 1] = pack_bf16x2(tile_exp2<POLY>(e, sc[c + e]), tile_exp2<POLY>(e + 1, sc[c + e + 1]));
          tile_st16(pt_addr + c / 2, pk);
        }
        if constexpr (!GUARDLESS) fast = !__any_sync(0xffffffffu, block_max() > kWindow);
      }
      if (!fast) {
        release_s();
        const float mx = block_max();
        float alpha = 1.0f;
        if (mx > m_ref + kWindow) {               // also the first finite maximum (m_ref == -inf)
          const float m_new = (m_ref == -INFINITY && fabsf(mx) <= kWindow) ? 0.f : mx;
          alpha = fast_exp2(m_ref - m_new);       // 0 when m_ref == -inf
          m_ref = m_new;
        }
        const float m_use = (m_ref == -INFINITY) ? 0.f : m_ref;
        // O (and its row-sum column) is corrected once every MMA of PV_{j-1} has landed - before P_j is handed over, so no
        // PV MMA of this block can have been issued yet
        if (j > 0 && __any_sync(0xffffffffu, alpha != 1.0f)) {
          mbar_wait_lean(a_pv_done, par ^ 1);
          tc_fence_after();
#pragma unroll 1
          for (int c = 0; c < DV; c += 16) {
            uint32_t o[16];
            tmem_ld16(o_addr + c, o);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 16; ++e) o[e] = __float_as_uint(__uint_as_float(o[e]) * alpha);
            tile_st16(o_addr + c, o);
          }
          tmem_st_wait();
        }
        if (tw) stamp(0, j, 3);
        wait_p_free();
        if (tw) stamp(0, j, 4);
        exp_block(std::true_type{}, m_use);
      }
      if (tw) stamp(0, j, 5);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a_p_full) : "memory");
      if (tw) stamp(0, j, 6);
    }
    // epilogue: l = column D of O; O / l -> bf16
    mbar_wait_lean(a_pv_done, par ^ 1);           // the last block's PV
    tc_fence_after();
    float l_tot;
    {
      uint32_t lv[8];
      tmem_ld8(o_addr + D, lv);
      tmem_ld_wait();
      l_tot = __uint_as_float(lv[0]);
    }
    if constexpr (GUARDLESS) {
      // whole O row in registers: judged first (pass 0), written after the CTA-wide decision
      uint32_t o[DV];
#pragma unroll
      for (int c = 0; c < DV; c += 16) tmem_ld16(o_addr + c, *reinterpret_cast<uint32_t (*)[16]>(o + c));
      tmem_ld_wait();
      if (pass == 0) {
        uint32_t worst = __float_as_uint(l_tot) & 0x7f800000u;       // exponent 255 <=> inf / NaN
#pragma unroll
        for (int c = 0; c < D; ++c) worst = max(worst, o[c] & 0x7f800000u);
        if (__any_sync(0xffffffffu, worst == 0x7f800000u) && lane == 0) *redo = 1;
        tc_fence_before();
        __syncthreads();                          // with the service warps: everybody reads the same verdict
        tc_fence_after();
        if (*redo != 0) continue;                 // run the tile again on the general path
      }
      const float inv_l = l_tot > 0.f ? 1.0f / l_tot : 0.f;
      if (p.lse != nullptr && q_row < p.Nq)
        p.lse[(static_cast<size_t>(b) * p.heads + h) * p.Nq + q_row] = l_tot > 0.f ? m_ref + __log2f(l_tot) : INFINITY;
      if (q_row < p.Nq) {
        __nv_bfloat16* orow = p.out + (static_cast<size_t>(b) * p.Nq + q_row) * p.ldo + h * p.d;
#pragma unroll
        for (int c = 0; c < D; c += 8) {
          uint4 pk;
          pk.x = pack_bf16x2(__uint_as_float(o[c + 0]) * inv_l, __uint_as_float(o[c + 1]) * inv_l);
          pk.y = pack_bf16x2(__uint_as_float(o[c + 2]) * inv_l, __uint_as_float(o[c + 3]) * inv_l);
          pk.z = pack_bf16x2(__uint_as_float(o[c + 4]) * inv_l, __uint_as_float(o[c + 5]) * inv_l);
          pk.w = pack_bf16x2(__uint_as_float(o[c + 6]) * inv_l, __uint_as_float(o[c + 7]) * inv_l);
          *reinterpret_cast<uint4*>(orow + c) = pk;
        }
      }
      break;
    } else {
    const float inv_l = l_tot > 0.f ? 1.0f / l_tot : 0.f;
    if (p.lse != nullptr && q_row < p.Nq)
      p.lse[(static_cast<size_t>(b) * p.heads + h) * p.Nq + q_row] = l_tot > 0.f ? m_ref + __log2f(l_tot) : INFINITY;
    __nv_bfloat16* orow = p.out + (static_cast<size_t>(b) * p.Nq + q_row) * p.ldo + h * p.d;
#pragma unroll 1
    for (int c = 0; c < D; c += 16) {
      uint32_t o[16];
      tmem_ld16(o_addr + c, o);
      tmem_ld_wait();
      if (q_row < p.Nq) {
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          if (c + g * 8 < D) {
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
    }  // pass
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::kTmemCols);
  }
}

template <int D, int POLY, bool MASKED, bool TRACE>
static int launch_tile_m(const AttnTileParams& p, cudaStream_t stream) {
  using S = TileSmem<D>;
  static bool configured = false;
  if (!configured) {
    AF_CUDA(cudaFuncSetAttribute(attention_tile_kernel<D, POLY, MASKED, TRACE>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal));
    AF_CUDA(cudaFuncSetAttribute(attention_tile_kernel<D, POLY, MASKED, TRACE>,
                                 cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    configured = true;
  }
  dim3 grid((p.Nq + 127) / 128, p.heads, p.B);
  attention_tile_kernel<D, POLY, MASKED, TRACE><<<grid, 256, S::kTotal, stream>>>(p);
  AF_LAUNCH_CHECK("attention_tile_kernel");
  return 0;
}
template <int D, int POLY>
static int launch_tile(const AttnTileParams& p, cudaStream_t stream) {
  // the masked kernel takes every exponential from fast_exp2: tile_exp2_poly clamps its argument to -126, so a masked
  // key (score -inf) would get weight 2^-126 instead of 0 and enter P.V and the row sum
  if (p.key_mask != nullptr || p.Nk % TileCfg<D>::BLOCK_N != 0) return launch_tile_m<D, 0, true, false>(p, stream);
  if (p.trace != nullptr) return launch_tile_m<D, POLY, false, true>(p, stream);
  return launch_tile_m<D, POLY, false, false>(p, stream);
}

// Called by af_attention_bf16* (attention.cu) for d in {40, 80} and more than 128 keys.  `trace`: null, or the timeline
// buffer of af_attention_bf16_trace.
int attention_tile_dispatch(const void* Q, long long ldq, const void* K, long long ldk, const void* Vt, long long ldvt,
                            int kv_stride, const unsigned char* key_mask, void* O, int B, int heads, int Nq, int Nk,
                            int d, float* lse, long long* trace, cudaStream_t stream) {
  if (!(d == 40 || d == 80)) return -100;
  AttnTileParams p;
  memset(&p, 0, sizeof(p));
  const int dp = d == 40 ? 48 : d;
  const int bn = d == 40 ? TileCfg<40>::BLOCK_N : TileCfg<80>::BLOCK_N;
  {
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
    uint32_t box[2] = {64, static_cast<uint32_t>(d)};
    int rc = make_tmap_bf16(&p.tmV, Vt, 2, dims, str, box);
    if (rc) return rc;
  }
  p.B = B; p.heads = heads; p.Nq = Nq; p.Nk = Nk; p.d = d; p.dp = dp; p.kv_stride = kv_stride;
  p.key_mask = key_mask;
  p.lse = lse;
  p.trace = trace;
  p.out = static_cast<__nv_bfloat16*>(O);
  p.ldo = static_cast<long long>(heads) * d;
  // d = 40: every third exponential on the FMA pipe (0.764 -> 0.688 ms at N = 4096, profiles/r02_attention.md)
#ifndef AF_TILE_POLY40
#define AF_TILE_POLY40 3
#endif
#ifndef AF_TILE_POLY80
#define AF_TILE_POLY80 0
#endif
  return d == 40 ? launch_tile<40, AF_TILE_POLY40>(p, stream) : launch_tile<80, AF_TILE_POLY80>(p, stream);
}

}  // namespace af
