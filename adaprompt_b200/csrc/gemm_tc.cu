// Persistent, warp-specialised tcgen05 GEMM / implicit-GEMM convolution for sm_100a.
//
//   D[M, N] = A[M, K] * Wt[N, K]^T   (bf16 operands, fp32 accumulation in TMEM)
//
// One kernel template serves every contraction of the SD-1.5 UNet hot path:
//   * Linear / conv1x1 (reference: nn.Linear in ldm/modules/attention.py:35,55,157-165 and the 1x1
//     nn.Conv2d at attention.py:302,313 / openaimodel.py:245): A is a 2-D [M, K] token matrix.
//   * conv3x3 stride 1, pad 1 (openaimodel.py:208,234,530,696 and Upsample :120-122): A is the NHWC
//     activation read through a 4-D TMA map; each of the 9 taps is a shifted box and the zero padding
//     is TMA out-of-bounds fill - no im2col buffer exists anywhere.
//   * conv3x3 stride 2 (Downsample, openaimodel.py:155): the input is viewed as
//     [B, H/2, 2, W/2, 2*C] so every tap is a unit-stride 5-D box.
//   * conv3x3 stride 2 after F.pad(x, (0,1,0,1)) (the VAE encoder's Downsample, model.py:61-79): the same 5-D view with
//     input row 2*oh + ky; its own instantiations (DOWN01) so the other modes' producer loops stay as they are.
//   * the skip-connection concat (openaimodel.py:1019) is never materialised: the K loop walks two
//     tensor maps (A0 then A1).
//
// Roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + single-thread MMA issuer,
// warps 2..9 = epilogue.  An epilogue warp owns 32 rows (its TMEM lane quarter) x 32 columns per work item:
//   TMEM -> registers (row per lane) -> + bias / per-sample time-embedding row / activation
//        -> + fp32 residual that a TMA load prefetched into the warp's shared-memory slot (2-3 items ahead)
//        -> result written back INTO the slot in the TMA 128B/64B-swizzled layout
//        -> GroupNorm partial statistics read column-wise from the slot
//        -> one TMA store (cp.async.bulk.tensor, shared -> global) per item.
// No per-lane global address arithmetic, no transposition pass, edge tiles clipped by TMA; the memory-level
// parallelism of the residual stream lives in the TMA queue instead of registers.
// smem ring of kStages {A 128x64, B BNx64} 128B-swizzled tiles; 2 TMEM accumulator stages so the
// epilogue of tile i overlaps the mainloop of tile i+1.
#include "../../include/adaface_b200.h"
#include <type_traits>

#include "common.cuh"

namespace af {

struct GemmParams {
  CUtensorMap tmA0;
  CUtensorMap tmA1;
  CUtensorMap tmB;
  CUtensorMap tmOut;   // 4-D {cols, w, h, n} (linear: {N, M, 1, 1}), box = 32 columns x one warp's 32 rows
  CUtensorMap tmRes;   // same geometry over the fp32 residual (== tmOut when there is none)
  int sbx, sby;        // conv: the 32-row sub-box of a warp is sbx x sby x (32 / sbx / sby) pixels
  int M, N;            // output rows / packed output columns
  int num_kb;          // K blocks (64 wide) in total
  int cpb;             // K blocks per tap (== num_kb for linear)
  int kb_split;        // K blocks per tap served by A0 (rest by A1)
  int amode;           // 0 linear, 1 conv3x3 s1, 2 conv3x3 s2, 3 conv3x3 s2 after F.pad(0,1,0,1)
  int B, H, W;         // conv: output pixel grid
  int C0;              // conv s2: channels of the (single) source
  int bw, bh, nb;      // conv: tile box (bw*bh*nb == 128)
  int tiles_w, tiles_h;
  int m_tiles, n_tiles;
  const float* bias;       // [N] or null
  const float* rowbias;    // [groups, N] or null; group = out_row / rows_per_group
  int rows_per_group;
  long long ld_rowbias;
  const float* residual;   // [M, ldr] fp32 or null
  long long ldr;
  void* out;
  long long ldo;
  int out_bf16;
  int wide;                // bf16 output without residual, BN % 128 == 0: 64-column epilogue items (128-byte rows)
  long long* trace;        // optional timeline of CTA 0: [3 actors][32 tiles][8 events] clock64 (af_epilogue.trace)
  int geglu;               // tile cols [0,BN/2) = value, [BN/2,BN) = gate; writes BN/2 cols
  int act;                 // 0 none, 1 quick_gelu x*sigmoid(1.702x) on (acc + bias), before the residual add
  float* gn_stats;         // [slots_total][N][2] per-channel (sum, sumsq) over 32-row quarters of the output, or null
  int gn_slots;            // conv: stat slots per sample (= tiles_w * tiles_h * bw * bh / 32)
  // Split-K of the LAST, partial wave of tiles (see "work units" below); split == 1: every unit is a whole tile
  int dp_tiles;            // tiles [0, dp_tiles) are whole-K units; each tile in [dp_tiles, tiles) is `split` units
  int split;               // K ranges per remainder tile
  int kb_per;              // K blocks per range (the last range takes what is left)
  int num_units;           // dp_tiles + (tiles - dp_tiles) * split
  float* ws;               // fp32 partial accumulators [(tile - dp_tiles) * (split - 1) + s][chunk][j][128 rows][4]
  int* ws_flags;           // [(tile - dp_tiles)][2]: partial warps arrived, finisher warps done (zero between launches)
};

constexpr int kEpiWarps = 8;                    // 2 warps per TMEM lane quarter, each takes every other 32-col chunk
constexpr int kGemmThreads = 64 + kEpiWarps * 32 + 32;   // + the B-operand producer warp (last warp)
constexpr int kBProducerWarp = 2 + kEpiWarps;
constexpr int kSmemBudget = 227 * 1024 - 1024 /*align*/ - 512 /*barriers*/;

// SLOTS = per-warp ring of epilogue slots (32 rows x 128 B; 64 B rows for the bf16-only GEGLU output).  3 slots keep
// two residual chunks in flight per warp (64 KB per SM) for the memory-bound small-K GEMMs; everything else uses 2.
template <int BN, bool GEGLU, int SLOTS, bool CTA2>
struct GemmCfg {
  static constexpr int kABytes = 128 * 128;
  static constexpr int kBRows = CTA2 ? BN / 2 : BN;      // CTA pair: each CTA stages half of the B tile
  static constexpr int kBBytes = kBRows * 128;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kSlotBytes = GEGLU ? 2048 : 4096;
  static constexpr int kSlotRegion = kEpiWarps * SLOTS * kSlotBytes;
  static constexpr int kMaxStages = (kSmemBudget - kSlotRegion) / kStageBytes;
  static constexpr int kStages = kMaxStages > 8 ? 8 : kMaxStages;
  static constexpr int kAccStride = BN <= 128 ? 128 : 256;
  static constexpr int kTmemCols = 2 * kAccStride;
  static constexpr int kSmemBytes = kStages * kStageBytes + kSlotRegion + 1024 /*align*/ + 512 /*barriers*/;
  static constexpr int kTxBytes = CTA2 ? 2 * kStageBytes : kStageBytes;   // bytes landing per stage (both CTAs)
  static_assert(kStages >= 3, "not enough shared memory for the operand ring");
};

// ---- TMA store / bulk-group helpers -----------------------------------------------------------------
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// GELU for the GEGLU epilogue: x * Phi(x) in its tanh form, 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3))), one MUFU
// op per element.  |tanh form - erf form| <= 4.8e-4 absolute (rel-L2 2e-4 for unit-variance gates), an order of
// magnitude below the bf16 rounding of the product this epilogue writes (rel-L2 1.7e-3); the erf form cost 3x the
// instructions and left the tensor pipe idle 85 % of the time (ncu --set full of the erf-form epilogue, round 1; the capture was not kept).
__device__ __forceinline__ float gelu_tanh(float x) {
  const float x2 = x * x;
  const float u = x * fmaf(0.0356774081f, x2, 0.7978845608f);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
}

// QuickGELU of the CLIP text MLP (transformers QuickGELUActivation): x * sigmoid(1.702 x)
__device__ __forceinline__ float quick_gelu(float x) { return __fdividef(x, 1.0f + __expf(-1.702f * x)); }

// DOWN01: the producer runs the amode-3 tap walk only (af_conv3x3_down01_bf16; convolution layout, one epilogue slot
// per warp); otherwise it selects mode 0 / 1 / 2 from p.amode.
template <int BN, bool GEGLU, int SLOTS, bool CTA2, bool DOWN01>
__global__ void __launch_bounds__(kGemmThreads, 1) gemm_tc_kernel(const __grid_constant__ GemmParams p) {
  using Cfg = GemmCfg<BN, GEGLU, SLOTS, CTA2>;
  constexpr int kStages = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* slots = smem + kStages * Cfg::kStageBytes;                 // [kEpiWarps][SLOTS][kSlotBytes], 1 KB aligned
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(slots + Cfg::kSlotRegion);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tfull_bar = empty_bar + kStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* res_bar = tempty_bar + 2;                                  // [kEpiWarps][SLOTS] residual slot filled
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_bar + kEpiWarps * SLOTS);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // CTA pair: both CTAs walk the same sequence of 256-row pair tiles; rank r owns m_tile = 2 * pair_m + r
  const uint32_t cta_rank = CTA2 ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;
  const int tile_first = CTA2 ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
  const int tile_step = CTA2 ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);
  const int num_tiles = (CTA2 ? (p.m_tiles + 1) / 2 : p.m_tiles) * p.n_tiles;
  auto tile_mn = [&](int t, int& n_tile, int& m_tile) {
    n_tile = t % p.n_tiles;
    const int pm = t / p.n_tiles;
    m_tile = CTA2 ? 2 * pm + static_cast<int>(cta_rank) : pm;
  };

  // Work units.  A persistent block walks units u = blockIdx.x, + gridDim.x, ...  Units [0, dp_tiles) are whole tiles
  // (the full waves).  The tiles of the last, partial wave would leave most SMs idle for a whole tile time (64 tiles on
  // 148 SMs for the 8x8 convolutions), so each of them is cut into `split` K ranges = `split` units on different
  // blocks: ranges 0 .. split-2 ("partial" units) dump their fp32 accumulator tile to a workspace and signal; the
  // unit with the LAST range (the "finisher") waits for them, adds the partials in range order (fixed order:
  // bit-reproducible) and runs the normal fused epilogue.  A unit only ever waits for units with a smaller index and
  // every block walks its units in increasing order, so with all blocks resident (grid <= SM count, one block per SM)
  // the smallest unfinished unit can always proceed: no deadlock.
  const int num_units = CTA2 ? num_tiles : p.num_units;
  struct Unit {
    int tile, kb0, kb1, kind, rt, s;   // kind: 0 whole tile, 1 partial, 2 finisher; rt = tile - dp_tiles
  };
  auto unit_at = [&](int u) -> Unit {
    Unit w;
    if (CTA2 || u < p.dp_tiles) {
      w.tile = u; w.kb0 = 0; w.kb1 = p.num_kb; w.kind = 0; w.rt = 0; w.s = 0;
    } else {
      const int r = u - p.dp_tiles;
      w.rt = r / p.split;
      w.s = r - w.rt * p.split;
      w.tile = p.dp_tiles + w.rt;
      w.kb0 = w.s * p.kb_per;
      w.kb1 = w.s == p.split - 1 ? p.num_kb : w.kb0 + p.kb_per;
      w.kind = w.s == p.split - 1 ? 2 : 1;
    }
    return w;
  };

  // timeline probe: actor 0 = TMA producer, 1 = MMA issuer, 2 = epilogue warp 0 (lane 0 each), CTA 0, first 32 tiles
  const bool tracing = p.trace != nullptr && blockIdx.x == 0 && lane == 0;
  auto stamp = [&](int actor, int tile_no, int ev) {
    if (tracing && tile_no < 32) p.trace[(actor * 32 + tile_no) * 8 + ev] = clock64();
  };

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&p.tmA0);
    tma_prefetch_desc(&p.tmA1);
    tma_prefetch_desc(&p.tmB);
    tma_prefetch_desc(&p.tmOut);
    tma_prefetch_desc(&p.tmRes);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 2);     // A producer + B producer, each with its own expect_tx
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], CTA2 ? 2 * kEpiWarps : kEpiWarps);   // pair: the leader's barrier collects both CTAs
    }
    for (int s = 0; s < kEpiWarps * SLOTS; ++s) mbar_init(&res_bar[s], 1);
    mbar_fence_init();
  }
  if (warp == 1) {
    if constexpr (CTA2) {
      tmem_alloc2(tmem_slot, Cfg::kTmemCols);
      tmem_relinquish2();
    } else {
      tmem_alloc(tmem_slot, Cfg::kTmemCols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if constexpr (CTA2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  // broadcast from lane 0: marks the address warp-uniform, so tcgen05 instructions take it from a uniform register
  // instead of a per-instruction elect / R2UR.BROADCAST waterfall loop
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp == 0 || warp == kBProducerWarp) {
    // ------------------------------------------------------------------ TMA producers: warp 0 loads the A operand
    // (activations / im2col taps), the last warp the B operand (weights).  One thread issuing both was a serial
    // chain of ~520-780 cycles per ring stage (wait - expect_tx - two tensor-map loads) against 320 cycles of MMA
    // work: the K-deep GEMMs / convolutions were producer bound (profiles/r01_gemm_epilogue_timeline.md).
    const bool loads_a = warp == 0;
    {   // whole warp, convergent: waits are warp-uniform, the TMA instructions are issued by one elected lane
      int stage = 0;
      uint32_t phase = 0;
      constexpr uint32_t kATx = (CTA2 ? 2u : 1u) * Cfg::kABytes, kBTx = (CTA2 ? 2u : 1u) * Cfg::kBBytes;
      for (int unit = tile_first, tno = 0; unit < num_units; unit += tile_step, ++tno) {
        const Unit wu = unit_at(unit);
        const int tile = wu.tile;
        int n_tile, m_tile;
        tile_mn(tile, n_tile, m_tile);
        if (loads_a) stamp(0, tno, 0);
        const int n0 = n_tile * BN + (CTA2 ? static_cast<int>(cta_rank) * (BN / 2) : 0);
        int cw = 0, ch = 0, cn = 0;
        if (loads_a && p.amode != 0) {
          cw = (m_tile % p.tiles_w) * p.bw;
          ch = ((m_tile / p.tiles_w) % p.tiles_h) * p.bh;
          cn = (m_tile / (p.tiles_w * p.tiles_h)) * p.nb;
        }
        // (tap, channel block) of the K chunk are walked incrementally: no run-time integer division per stage.  The
        // operand mode is a compile-time constant inside each loop instance (generic lambda + integral_constant): the
        // per-stage chain of the producer has no option branches left.
        auto a_loop = [&](auto amode_c) {
          constexpr int AM = decltype(amode_c)::value;
          int cblk = wu.kb0, ky = 0, kx = 0;
          if (AM != 0 && wu.kb0 != 0) {               // a K range of a split tile starts inside the (tap, channel) walk
            const int tap = wu.kb0 / p.cpb;
            cblk = wu.kb0 - tap * p.cpb;
            ky = tap / 3;
            kx = tap - 3 * ky;
          }
          for (int kb = wu.kb0; kb < wu.kb1; ++kb) {
            uint8_t* sa = smem + stage * Cfg::kStageBytes;
            const bool second = AM == 0 && cblk >= p.kb_split;     // dual-source K only exists for linear GEMMs ...
            const bool second_c = AM == 1 && cblk >= p.kb_split;   // ... and stride-1 convolutions (concat input)
            const CUtensorMap* tmA = (second || second_c) ? &p.tmA1 : &p.tmA0;
            const int kc = ((second || second_c) ? cblk - p.kb_split : cblk) * 64;
            mbar_wait(&empty_bar[stage], phase ^ 1);
            if (elect_one()) {
              if (leader) mbar_arrive_expect_tx(&full_bar[stage], kATx);
              if constexpr (AM == 0) {
                if constexpr (CTA2) tma_load_2d_pair(sa, tmA, &full_bar[stage], kc, m_tile * 128);
                else tma_load_2d(sa, tmA, &full_bar[stage], kc, m_tile * 128);
              } else if constexpr (AM == 1) {
                if constexpr (CTA2) tma_load_4d_pair(sa, tmA, &full_bar[stage], kc, cw + kx - 1, ch + ky - 1, cn);
                else tma_load_4d(sa, tmA, &full_bar[stage], kc, cw + kx - 1, ch + ky - 1, cn);
              } else if constexpr (AM == 2) {
                // stride 2: input row 2*oh + ky - 1  ->  (coarse row oh + dh, parity ph)
                const int ph = (ky == 1) ? 0 : 1, dh = (ky == 0) ? -1 : 0;
                const int pw = (kx == 1) ? 0 : 1, dw = (kx == 0) ? -1 : 0;
                if constexpr (CTA2) tma_load_5d_pair(sa, tmA, &full_bar[stage], pw * p.C0 + kc, cw + dw, ph, ch + dh, cn);
                else tma_load_5d(sa, tmA, &full_bar[stage], pw * p.C0 + kc, cw + dw, ph, ch + dh, cn);
              } else {
                // stride 2 after F.pad(0,1,0,1): input row 2*oh + ky  ->  (coarse row oh + (ky >> 1), parity ky & 1).
                // ky == 2 on the last output row reads coarse row H/2: out of bounds, TMA fills zeros = the bottom pad
                // (columns likewise: the right pad).
                const int ph = ky & 1, dh = ky >> 1;
                const int pw = kx & 1, dw = kx >> 1;
                if constexpr (CTA2) tma_load_5d_pair(sa, tmA, &full_bar[stage], pw * p.C0 + kc, cw + dw, ph, ch + dh, cn);
                else tma_load_5d(sa, tmA, &full_bar[stage], pw * p.C0 + kc, cw + dw, ph, ch + dh, cn);
              }
            }
            if (AM != 0 && ++cblk == p.cpb) {
              cblk = 0;
              if (++kx == 3) {
                kx = 0;
                ++ky;
              }
            }
            if (AM == 0) ++cblk;
            if (++stage == kStages) {
              stage = 0;
              phase ^= 1;
            }
            if (kb == wu.kb0) stamp(0, tno, 1);
          }
        };
        if (loads_a) {
          if constexpr (DOWN01) a_loop(std::integral_constant<int, 3>{});
          else if (p.amode == 0) a_loop(std::integral_constant<int, 0>{});
          else if (p.amode == 1) a_loop(std::integral_constant<int, 1>{});
          else a_loop(std::integral_constant<int, 2>{});
        } else {
          for (int kb = wu.kb0; kb < wu.kb1; ++kb) {
            uint8_t* sb = smem + stage * Cfg::kStageBytes + Cfg::kABytes;
            mbar_wait(&empty_bar[stage], phase ^ 1);
            if (elect_one()) {
              if (leader) mbar_arrive_expect_tx(&full_bar[stage], kBTx);
              if constexpr (CTA2) tma_load_2d_pair(sb, &p.tmB, &full_bar[stage], kb * 64, n0);
              else tma_load_2d(sb, &p.tmB, &full_bar[stage], kb * 64, n0);
            }
            if (++stage == kStages) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
        if (loads_a) stamp(0, tno, 2);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (pair: leader CTA only)
    // (No __syncwarp after the elected sections: the next elect.sync / warp-uniform wait reconverges the warp.)
    // The whole warp walks the loop (convergent control flow, warp-uniform barrier waits); the tcgen05 instructions are
    // issued by one elected lane.  Under an `if (lane == 0)` branch the compiler wraps EVERY tcgen05.mma / commit in an
    // elect - issue - branch waterfall loop, which cost ~50 cycles per instruction on this serial issue chain.
    if (leader) {
      constexpr uint32_t idesc = umma_idesc_bf16(CTA2 ? 256 : 128, BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int unit = tile_first, tno = 0; unit < num_units; unit += tile_step, ++tno) {
        const Unit wu = unit_at(unit);
        stamp(1, tno, 0);
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        stamp(1, tno, 1);
        const uint32_t d_tmem = tmem_base + acc * Cfg::kAccStride;
        long long waited = 0;       // timeline probe only: cycles this tile's K loop spent waiting for operands
        for (int kb = wu.kb0; kb < wu.kb1; ++kb) {
          const long long w0 = tracing ? clock64() : 0;
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          if (tracing) waited += clock64() - w0;
          if (kb == wu.kb0) stamp(1, tno, 2);
          const uint32_t sa = smem_u32(smem + stage * Cfg::kStageBytes);
          const uint64_t adesc = umma_desc_sw128(sa);
          const uint64_t bdesc = umma_desc_sw128(sa + Cfg::kABytes);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              // +32 bytes (16 bf16) along K inside the 128B swizzle atom == +2 in the >>4 address field
              if constexpr (CTA2) tc_mma_ss2(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
              else tc_mma_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, ((kb - wu.kb0) | k) != 0 ? 1u : 0u);
            }
            if constexpr (CTA2) tc_commit2(&empty_bar[stage]); else tc_commit(&empty_bar[stage]);
          }
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (elect_one()) {
          if constexpr (CTA2) tc_commit2(&tfull_bar[acc]); else tc_commit(&tfull_bar[acc]);
        }
        stamp(1, tno, 3);
        if (tracing && tno < 32) p.trace[(1 * 32 + tno) * 8 + 4] = waited;
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps
    const int ew = warp - 2;
    const int q = warp & 3;          // TMEM lane quarter this warp may access (hardware: warp id % 4)
    const int half = ew >> 2;        // which 32-column chunks of the tile this warp takes: c = half*32 + 64*i
    uint8_t* my_slots = slots + ew * SLOTS * Cfg::kSlotBytes;
    uint64_t* my_res_bar = res_bar + ew * SLOTS;
    constexpr int kOutCols = GEGLU ? BN / 2 : BN;                       // output columns per tile
    const int nch = (kOutCols - half * 32 + 63) / 64;                   // work items of this warp per tile
    const bool has_res = !GEGLU && p.residual != nullptr;

    // TMA row coordinates {c1, c2, c3} of this warp's 32-row box inside tile t (integer divisions by run-time values:
    // done once per TILE, never per 32x32 work item - they used to cost ~1500 of the ~3000 cycles an item took,
    // profiles/r01_gemm_epilogue_timeline.md)
    auto tile_rows = [&](int t, int& n_tile, int& c1, int& c2, int& c3) {
      int m_tile;
      tile_mn(t, n_tile, m_tile);
      if (p.amode == 0) {
        c1 = m_tile * 128 + q * 32; c2 = 0; c3 = 0;
      } else {
        const int tw = m_tile % p.tiles_w;
        const int th = (m_tile / p.tiles_w) % p.tiles_h;
        const int tn = m_tile / (p.tiles_w * p.tiles_h);
        const int r0 = q * 32;
        c1 = tw * p.bw + r0 % p.bw;
        c2 = th * p.bh + (r0 / p.bw) % p.bh;
        c3 = tn * p.nb + r0 / (p.bw * p.bh);
      }
    };
    // residual prefetch cursor: walks this warp's work items (output unit, chunk) in order, kAhead items in front.
    // Partial units of split tiles write no output and read no residual: the cursor skips them.
    auto is_partial = [&](int u) { return !CTA2 && u >= p.dp_tiles && (u - p.dp_tiles) % p.split != p.split - 1; };
    int pf_unit = tile_first, pf_i = 0, pf_n = 0, pf_c1 = 0, pf_c2 = 0, pf_c3 = 0, pf_item = 0;
    auto pf_settle = [&]() {          // first output unit at or after pf_unit, and its row coordinates
      while (pf_unit < num_units && is_partial(pf_unit)) pf_unit += tile_step;
      if (pf_unit < num_units) tile_rows(unit_at(pf_unit).tile, pf_n, pf_c1, pf_c2, pf_c3);
    };
    pf_settle();
    auto issue_res_load = [&]() {   // lane 0 only
      if (pf_unit >= num_units) return;
      const int sl = pf_item % SLOTS;
      mbar_arrive_expect_tx(&my_res_bar[sl], 4096);
      tma_load_4d(my_slots + sl * Cfg::kSlotBytes, &p.tmRes, &my_res_bar[sl], pf_n * kOutCols + half * 32 + 64 * pf_i,
                  pf_c1, pf_c2, pf_c3);
      ++pf_item;
      if (++pf_i == nch) {
        pf_i = 0;
        pf_unit += tile_step;
        pf_settle();
      }
    };
    // All bulk-tensor instructions of this warp (residual loads, stores, group commits / waits) are issued by the lane
    // `elect.sync` picks - the same lane every time for the full member mask, which the per-thread bulk async-groups
    // need - instead of under `lane == 0`, where each of them was wrapped in an elect / branch waterfall loop.
    // residual prefetch distance: SLOTS - 1 items (SLOTS == 1: the next load waits for this item's store to drain)
    constexpr int kAhead = SLOTS > 1 ? SLOTS - 1 : 1;
    if (has_res && elect_one()) {
#pragma unroll
      for (int j = 0; j < kAhead; ++j) issue_res_load();
    }

    int item = 0;                      // running work-item index of this warp (slot = item % SLOTS)
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int unit = tile_first, tno = 0; unit < num_units; unit += tile_step, ++tno) {
      const Unit wu = unit_at(unit);
      const int tile = wu.tile;
      int n_tile, m_tile;
      tile_mn(tile, n_tile, m_tile);
      if (ew == 0) stamp(2, tno, 0);
      int c1, c2, c3;
      {
        int nt;
        tile_rows(tile, nt, c1, c2, c3);
      }
      // this lane's output row (for the per-sample rowbias and the statistics mask)
      bool row_ok;
      uint32_t grow;
      long long stat_slot = -1;
      if (p.amode == 0) {
        grow = m_tile * 128 + q * 32 + lane;
        row_ok = grow < static_cast<uint32_t>(p.M);
        if (m_tile < p.m_tiles) stat_slot = static_cast<long long>(m_tile) * 4 + q;   // (pair: odd tile count)
      } else {
        const int tw = m_tile % p.tiles_w;
        const int th = (m_tile / p.tiles_w) % p.tiles_h;
        const int tn = m_tile / (p.tiles_w * p.tiles_h);
        const int r = q * 32 + lane;
        const int n = tn * p.nb + r / (p.bw * p.bh), h = th * p.bh + (r / p.bw) % p.bh, w = tw * p.bw + r % p.bw;
        row_ok = n < p.B && h < p.H && w < p.W;
        grow = (n * p.H + h) * p.W + w;
        const int per = p.bw * p.bh;                       // pixels of one sample inside the tile (>= 32 if stats)
        const int n0s = tn * p.nb + (q * 32) / per;
        if (n0s < p.B)
          stat_slot = static_cast<long long>(n0s) * p.gn_slots + (th * p.tiles_w + tw) * (per >> 5) + (((q * 32) % per) >> 5);
      }
      const float* rb_row = nullptr;
      if (!GEGLU && p.rowbias && row_ok) rb_row = p.rowbias + static_cast<long long>(grow / static_cast<uint32_t>(p.rows_per_group)) * p.ld_rowbias;
      const uint32_t row_mask = __ballot_sync(0xffffffffu, row_ok);

      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      if (ew == 0) stamp(2, tno, 1);
      const uint32_t t_acc = tmem_base + acc * Cfg::kAccStride + (static_cast<uint32_t>(q * 32) << 16);

      // split tiles: this thread's float4 group j of 32-column chunk ch lives at ws_row[(ch * 8 + j) * 128] (one
      // 512-byte run per warp and group: coalesced both ways)
      float4* ws_row = nullptr;
      if constexpr (!GEGLU && !CTA2) {
        if (wu.kind != 0) {
          constexpr int kTileF4 = 128 * (BN / 4);                              // float4 per partial tile
          ws_row = reinterpret_cast<float4*>(p.ws) + static_cast<size_t>(wu.rt) * (p.split - 1) * kTileF4 + q * 32 + lane;
          if (wu.kind == 1) {
            // ---------------------------------------------------------- partial unit: accumulator -> workspace
            float4* dst = ws_row + static_cast<size_t>(wu.s) * kTileF4;
            for (int i = 0; i < nch; ++i) {
              const int c = half * 32 + 64 * i;
              uint32_t v[32];
              tmem_ld32(t_acc + c, v);
              tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < 8; ++j)
                __stcg(dst + ((c >> 5) * 8 + j) * 128, make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                                                   __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3])));
            }
            __threadfence();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              atomicAdd(p.ws_flags + 2 * wu.rt, 1);
              mbar_arrive(&tempty_bar[acc]);
            }
            if (++acc == 2) {
              acc = 0;
              acc_phase ^= 1;
            }
            continue;
          }
          // ------------------------------------------------------------ finisher: all partial warps have written
          if (lane == 0) {
            const int want = (p.split - 1) * kEpiWarps;
            const volatile int* flag = p.ws_flags + 2 * wu.rt;
            unsigned long long t0 = 0;
            while (*flag < want) {
              if (t0 == 0) t0 = globaltimer_ns();
              else if (globaltimer_ns() - t0 > AF_WATCHDOG_NS) { printf("gemm_tc: split-K finisher timed out (tile %d)\n", tile); __trap(); }
            }
            __threadfence();
          }
          __syncwarp();
        }
      }

      if (!GEGLU && p.wide) {
        // 64-column items for bf16 outputs: the two 32-column halves go through registers one after the other, but the
        // slot hand-over, proxy fence, warp sync and TMA store are paid once per 128-byte row instead of once per 64 bytes.
        // The short-K projections (QK, V^T: 5 K blocks per tile) are bound by exactly those per-item costs.
        const int nchw = (kOutCols - half * 64 + 127) / 128;
        for (int i = 0; i < nchw; ++i) {
          const int c = half * 64 + 128 * i;
          const int col0 = n_tile * kOutCols + c;
          uint8_t* slot = my_slots + (item % SLOTS) * Cfg::kSlotBytes;
          const uint32_t slot_a = smem_u32(slot);
          if (elect_one()) bulk_wait_read<SLOTS - 1>();        // the store that last used this slot has read it
          __syncwarp();
#pragma unroll
          for (int sub = 0; sub < 2; ++sub) {
            uint32_t v[32];
            tmem_ld32(t_acc + c + 32 * sub, v);
            const int cs = col0 + 32 * sub;
            float4 b4[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) b4[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.bias) {
#pragma unroll
              for (int j = 0; j < 8; ++j)
                if (cs + 4 * j < p.N) b4[j] = __ldg(reinterpret_cast<const float4*>(p.bias + cs) + j);
            }
            if (rb_row) {
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                if (cs + 4 * j < p.N) {
                  const float4 rb = __ldg(reinterpret_cast<const float4*>(rb_row + cs) + j);
                  b4[j].x += rb.x; b4[j].y += rb.y; b4[j].z += rb.z; b4[j].w += rb.w;
                }
              }
            }
            tmem_ld_wait();
            if (ws_row != nullptr) {   // finisher of a split tile: + the partial accumulators, in K-range order
              constexpr int kTileF4 = 128 * (BN / 4);
              for (int sp = 0; sp < p.split - 1; ++sp) {
                const float4* src = ws_row + static_cast<size_t>(sp) * kTileF4 + ((c + 32 * sub) >> 5) * 8 * 128;
                float4 part[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) part[j] = __ldcg(src + j * 128);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  v[4 * j] = __float_as_uint(__uint_as_float(v[4 * j]) + part[j].x);
                  v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) + part[j].y);
                  v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) + part[j].z);
                  v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) + part[j].w);
                }
              }
            }
            float4 o[8];
#pragma unroll
            for (int j = 0; j < 8; ++j)
              o[j] = make_float4(__uint_as_float(v[4 * j]) + b4[j].x, __uint_as_float(v[4 * j + 1]) + b4[j].y,
                                 __uint_as_float(v[4 * j + 2]) + b4[j].z, __uint_as_float(v[4 * j + 3]) + b4[j].w);
            if (p.act == 1) {
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                o[j].x = quick_gelu(o[j].x); o[j].y = quick_gelu(o[j].y);
                o[j].z = quick_gelu(o[j].z); o[j].w = quick_gelu(o[j].w);
              }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)     // 16-byte chunk (sub * 4 + j) of the lane's 128-byte row, SWIZZLE_128B
              sts128(slot_a + lane * 128 + (((sub * 4 + j) ^ (lane & 7)) << 4), pack_bf16x2(o[2 * j].x, o[2 * j].y),
                     pack_bf16x2(o[2 * j].z, o[2 * j].w), pack_bf16x2(o[2 * j + 1].x, o[2 * j + 1].y),
                     pack_bf16x2(o[2 * j + 1].z, o[2 * j + 1].w));
          }
          fence_async_smem();
          __syncwarp();
          if (elect_one()) {
            if (col0 < p.N) tma_store_4d(&p.tmOut, slot, col0, c1, c2, c3);
            bulk_commit();
          }
          ++item;
        }
      } else
      // (Fetching chunk i+1 from TMEM into a second register set while chunk i is staged was measured SLOWER: 48.7 ->
      // 59.4 us on M65536 N320 K320 +res, the conversion phase doubles - profiles/r01_gemm_epilogue_timeline.md.)
      for (int i = 0; i < nch; ++i) {
        const int c = half * 32 + 64 * i;                    // first accumulator column of the chunk
        const int col0 = n_tile * kOutCols + c;              // first output column
        const int sl = item % SLOTS;
        uint8_t* slot = my_slots + sl * Cfg::kSlotBytes;
        const uint32_t slot_a = smem_u32(slot);           // shared-space address: LDS / STS, not generic LD.E / ST.E
        const int c0 = col0;

        if constexpr (GEGLU) {
          // out[:, j] = (acc[:, j] + bv[j]) * gelu(acc[:, BN/2 + j] + bg[j]) -> bf16, 64-byte rows, SWIZZLE_64B
          uint32_t v[32], g[32];
          tmem_ld32(t_acc + c, v);
          tmem_ld32(t_acc + BN / 2 + c, g);
          const int pc = n_tile * BN + c;                    // packed column of the value half (bias index)
          const bool col_ok = col0 < p.N / 2;                // N/2 is a multiple of 128: chunks are all-or-nothing
          if (elect_one()) bulk_wait_read<SLOTS - 1>();        // the store that last used this slot has read it
          __syncwarp();
          tmem_ld_wait();
          uint32_t pk[16];
          float4 bvs[8], bgs[8];                             // bias rows of the value / gate halves: ONE option test
#pragma unroll
          for (int j = 0; j < 8; ++j) bvs[j] = bgs[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (p.bias && col_ok) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              bvs[j] = __ldg(reinterpret_cast<const float4*>(p.bias + pc) + j);
              bgs[j] = __ldg(reinterpret_cast<const float4*>(p.bias + pc + BN / 2) + j);
            }
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 bv = bvs[j], bg = bgs[j];
            const float o0 = (__uint_as_float(v[4 * j + 0]) + bv.x) * gelu_tanh(__uint_as_float(g[4 * j + 0]) + bg.x);
            const float o1 = (__uint_as_float(v[4 * j + 1]) + bv.y) * gelu_tanh(__uint_as_float(g[4 * j + 1]) + bg.y);
            const float o2 = (__uint_as_float(v[4 * j + 2]) + bv.z) * gelu_tanh(__uint_as_float(g[4 * j + 2]) + bg.z);
            const float o3 = (__uint_as_float(v[4 * j + 3]) + bv.w) * gelu_tanh(__uint_as_float(g[4 * j + 3]) + bg.w);
            pk[2 * j] = pack_bf16x2(o0, o1);
            pk[2 * j + 1] = pack_bf16x2(o2, o3);
          }
#pragma unroll
          for (int j = 0; j < 4; ++j)
            sts128(slot_a + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4), pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
          fence_async_smem();
          __syncwarp();
          if (elect_one()) {
            tma_store_4d(&p.tmOut, slot, c0, c1, c2, c3);
            bulk_commit();
          }
        } else {
          uint32_t v[32];
          if (ew == 0 && i == 0) stamp(3, tno, 0);
          tmem_ld32(t_acc + c, v);
          if (ew == 0 && i == 0) stamp(3, tno, 1);
          const bool col_ok = col0 < p.N;
          float4 b4[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) b4[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          const bool full_chunk = col0 + 32 <= p.N;     // uniform; partial chunks only at the right edge of N
          if (p.bias) {
            if (full_chunk) {
#pragma unroll
              for (int j = 0; j < 8; ++j) b4[j] = __ldg(reinterpret_cast<const float4*>(p.bias + col0) + j);
            } else {
#pragma unroll
              for (int j = 0; j < 8; ++j)
                if (col0 + 4 * j < p.N) b4[j] = __ldg(reinterpret_cast<const float4*>(p.bias + col0) + j);
            }
          }
          if (rb_row) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              if (full_chunk || col0 + 4 * j < p.N) {
                const float4 rb = __ldg(reinterpret_cast<const float4*>(rb_row + col0) + j);
                b4[j].x += rb.x; b4[j].y += rb.y; b4[j].z += rb.z; b4[j].w += rb.w;
              }
            }
          }
          if (ew == 0 && i == 0) stamp(2, tno, 6);
          if (has_res) {
            mbar_wait(&my_res_bar[sl], (item / SLOTS) & 1);   // residual chunk landed in the slot
            if (ew == 0 && i == 0) stamp(2, tno, 7);
          } else {
            if (elect_one()) bulk_wait_read<SLOTS - 1>();      // the store that last used this slot has read it
            __syncwarp();
          }
          tmem_ld_wait();
          if (ws_row != nullptr) {   // finisher of a split tile: + the partial accumulators, in K-range order
            constexpr int kTileF4 = 128 * (BN / 4);
            for (int sp = 0; sp < p.split - 1; ++sp) {
              const float4* src = ws_row + static_cast<size_t>(sp) * kTileF4 + (c >> 5) * 8 * 128;
              float4 part[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) part[j] = __ldcg(src + j * 128);
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                v[4 * j] = __float_as_uint(__uint_as_float(v[4 * j]) + part[j].x);
                v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) + part[j].y);
                v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) + part[j].z);
                v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) + part[j].w);
              }
            }
          }
          if (ew == 0 && i == 0) stamp(2, tno, 2);
          // one uniform branch per OPTION, not per element group: with the activation / residual tests inside the
          // unrolled loop the compiler kept 16 taken branches per item (~70 cycles each on this serial chain)
          float4 o[8];
#pragma unroll
          for (int j = 0; j < 8; ++j)
            o[j] = make_float4(__uint_as_float(v[4 * j]) + b4[j].x, __uint_as_float(v[4 * j + 1]) + b4[j].y,
                               __uint_as_float(v[4 * j + 2]) + b4[j].z, __uint_as_float(v[4 * j + 3]) + b4[j].w);
          if (p.act == 1) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              o[j].x = quick_gelu(o[j].x); o[j].y = quick_gelu(o[j].y);
              o[j].z = quick_gelu(o[j].z); o[j].w = quick_gelu(o[j].w);
            }
          }
          if (has_res) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 r4 = lds128f(slot_a + lane * 128 + ((j ^ (lane & 7)) << 4));
              o[j].x += r4.x; o[j].y += r4.y; o[j].z += r4.z; o[j].w += r4.w;
            }
          }
          if (ew == 0 && i == 0) stamp(3, tno, 2);
          if (p.out_bf16) {
            if (has_res) __syncwarp();                       // every lane has read its residual row
#pragma unroll
            for (int j = 0; j < 4; ++j)
              sts128(slot_a + lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4), pack_bf16x2(o[2 * j].x, o[2 * j].y),
                     pack_bf16x2(o[2 * j].z, o[2 * j].w), pack_bf16x2(o[2 * j + 1].x, o[2 * j + 1].y),
                     pack_bf16x2(o[2 * j + 1].z, o[2 * j + 1].w));
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              sts128f(slot_a + lane * 128 + ((j ^ (lane & 7)) << 4), o[j]);
          }
          if (ew == 0 && i == 0) stamp(3, tno, 3);
          fence_async_smem();
          if (ew == 0 && i == 0) stamp(3, tno, 4);
          __syncwarp();
          if (p.gn_stats && !p.out_bf16) {
            // per-channel (sum, sum of squares) over this warp's valid rows: lane = column, fixed row order
            float s = 0.f, ss = 0.f;
#pragma unroll 8
            for (int r = 0; r < 32; ++r) {
              if ((row_mask >> r) & 1u) {
                const float x = lds32f(slot_a + r * 128 + ((((lane >> 2) ^ (r & 7))) << 4) + (lane & 3) * 4);
                s += x;
                ss = fmaf(x, x, ss);
              }
            }
            if (stat_slot >= 0 && col0 + lane < p.N)
              *reinterpret_cast<float2*>(p.gn_stats + (stat_slot * p.N + col0 + lane) * 2) = make_float2(s, ss);
          }
          if (ew == 0 && i == 0) stamp(2, tno, 3);
          if (elect_one()) {
            if (col_ok) tma_store_4d(&p.tmOut, slot, c0, c1, c2, c3);
            bulk_commit();
            if (has_res) {
              bulk_wait_read<(SLOTS > 1 ? 1 : 0)>();         // the previous item's store has drained its slot ...
              issue_res_load();                              // ... which is the slot of item + kAhead
            }
          }
          if (ew == 0 && i == 0) stamp(2, tno, 4);
        }
        ++item;
      }
      if (ew == 0) stamp(2, tno, 5);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (ws_row != nullptr) {   // the last finisher warp re-arms the tile's flags for the next launch
          if (atomicAdd(p.ws_flags + 2 * wu.rt + 1, 1) == kEpiWarps - 1) {
            p.ws_flags[2 * wu.rt] = 0;
            p.ws_flags[2 * wu.rt + 1] = 0;
            __threadfence();
          }
        }
        if (CTA2 && !leader) mbar_arrive_cta(&tempty_bar[acc], 0);   // the leader's MMA warp owns both accumulators
        else mbar_arrive(&tempty_bar[acc]);
      }
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (elect_one()) bulk_wait_all();      // shared memory must outlive the bulk stores
  }

  tc_fence_before();
  if constexpr (CTA2) cluster_sync_all(); else __syncthreads();   // pair: no CTA may leave while its peer can still signal it
  if (warp == 1) {
    tc_fence_after();
    if constexpr (CTA2) tmem_dealloc2(tmem_base, Cfg::kTmemCols); else tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// No process-global switches: the tile schedule (af_epilogue.pair_mode) and the timeline probe (af_epilogue.trace) are
// per-call options.

template <int BN, bool GEGLU, int SLOTS, bool CTA2, bool DOWN01 = false>
static int launch_gemm(const GemmParams& p, cudaStream_t stream) {
  using Cfg = GemmCfg<BN, GEGLU, SLOTS, CTA2>;
  void (*kernel)(GemmParams) = gemm_tc_kernel<BN, GEGLU, SLOTS, CTA2, DOWN01>;
  static bool configured = false;
  if (!configured) {
    AF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    configured = true;
  }
  if constexpr (CTA2) {
    const int pair_tiles = ((p.m_tiles + 1) / 2) * p.n_tiles;
    const int max_pairs = num_sms() / 2;
    const int pairs = pair_tiles < max_pairs ? pair_tiles : max_pairs;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * pairs);
    cfg.blockDim = dim3(kGemmThreads);
    cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    AF_CUDA(cudaLaunchKernelEx(&cfg, kernel, p));
  } else {
    const int grid = p.num_units < num_sms() ? p.num_units : num_sms();
    kernel<<<grid, kGemmThreads, Cfg::kSmemBytes, stream>>>(p);
  }
  AF_LAUNCH_CHECK("gemm_tc_kernel");
  return 0;
}

// CTA pairs (cta_group::2: two SMs share one 256-row tile, each stages half of the weight tile).  Re-measured per shape
// with the round-2 kernel (scripts/bench_pair.py, profiles/r02_splitk.md): the pair schedule wins for linear GEMMs from
// 16 row tiles up (M >= 2048: -2 .. -12 %; at 8 row tiles split-K is worth more) and - unlike in round 1, before the producer split - for the stride-1
// convolutions with 160-wide tiles and >= 128 row tiles (64x64: -9 .. -12 %, 32x32 to 640 channels: -3 .. -5 %) or with
// any tile width >= 128 from 512 row tiles (the VAE decoder's 128^2 .. 512^2 layers: -5 .. -10 %); it
// loses where the tile count is small (16x16 / 8x8: those go to split-K, which the pair schedule does not do).
// Mode 1 ("auto") applies that; mode 2 forces pairs wherever they are legal (tests).
static bool want_pair(int pair_mode, int m_tiles, int n_tiles, int bn, int amode) {
  (void)n_tiles;
  if (pair_mode == AF_PAIR_NEVER || m_tiles < 2) return false;
  if (pair_mode == AF_PAIR_ALWAYS) return true;
#ifdef AF_PAIR_R1_RULE
  return amode == 0 && bn >= 160 && ((m_tiles + 1) / 2) * n_tiles >= num_sms();
#endif
  if (amode == 0) return bn >= 160 && m_tiles >= 16;
  if (amode == 1) return (bn == 160 && m_tiles >= 128) || (bn >= 128 && m_tiles >= 512);   // the second clause: VAE decoder layers
  return false;
}

template <int BN, bool GEGLU, int SLOTS, bool DOWN01 = false>
static int launch_gemm_mode(const GemmParams& p, bool pair, cudaStream_t stream) {
  return pair ? launch_gemm<BN, GEGLU, SLOTS, true, DOWN01>(p, stream) : launch_gemm<BN, GEGLU, SLOTS, false, DOWN01>(p, stream);
}

// Split-K of the last partial wave (kernel comment "work units").  Cost model in units of one K block of main-loop
// time, fitted to scripts/bench_splitk.py on B200 (profiles/r02_splitk.md): a unit costs its K blocks + a fixed part
// (pipeline fill, accumulator hand-over, epilogue), the finisher additionally a serial L2 round trip per partial tile
// it adds.  A K block of an implicit-GEMM convolution takes about twice as long as one of a linear GEMM, so the fixed
// parts weigh half as much there.  Picks the split that minimises the critical path; 1 = whole tiles only.
constexpr int kSplitFlagInts = 4096;          // flag region at the head of the workspace: 2 ints per remainder tile
constexpr int kMaxSplit = 16;
static void plan_split(GemmParams& p, int bn, bool pair, const af_epilogue* ep) {
  const int tiles = p.m_tiles * p.n_tiles;
  p.dp_tiles = tiles;
  p.split = 1;
  p.kb_per = p.num_kb;
  p.num_units = tiles;
  p.ws = nullptr;
  p.ws_flags = nullptr;
  if (pair || p.geglu || ep->split_k == 1 || ep->splitk_ws == nullptr) return;
  const int G = num_sms();
  const int dp = (tiles / G) * G, R = tiles - dp;
  if (R == 0 || 2 * R > kSplitFlagInts) return;
  const long long avail = (ep->splitk_ws_bytes - static_cast<long long>(kSplitFlagInts) * 4) / (128ll * bn * 4);   // partial tiles
  const int kUnitFixed = p.amode != 0 ? 15 : 30, kPartialCost = p.amode != 0 ? 10 : 20;
  int best = 1;
  long long best_cost = p.num_kb + kUnitFixed;                 // the remainder wave as whole tiles
  const int lo = ep->split_k > 1 ? ep->split_k : 2, hi = ep->split_k > 1 ? ep->split_k : kMaxSplit;
  for (int S = lo; S <= hi; ++S) {
    const int per = (p.num_kb + S - 1) / S;
    if (per * (S - 1) >= p.num_kb || per < 2) continue;        // every range needs work; tiny ranges are all overhead
    if (static_cast<long long>(R) * (S - 1) > avail) continue;
    const long long rounds = (static_cast<long long>(R) * S + G - 1) / G;
    const long long cost = rounds * (per + kUnitFixed) + static_cast<long long>(kPartialCost) * (S - 1);
    if (ep->split_k > 1 || cost < best_cost) {
      best = S;
      best_cost = cost;
    }
  }
  if (best == 1) return;
  p.dp_tiles = dp;
  p.split = best;
  p.kb_per = (p.num_kb + best - 1) / best;
  p.num_units = dp + R * best;
  p.ws_flags = static_cast<int*>(ep->splitk_ws);
  p.ws = reinterpret_cast<float*>(static_cast<char*>(ep->splitk_ws) + static_cast<size_t>(kSplitFlagInts) * 4);
}

static int dispatch_gemm(int bn, const GemmParams& p, bool pair, cudaStream_t stream) {
  if (p.geglu) return launch_gemm_mode<256, true, 2>(p, pair, stream);
  if (p.amode == 3) {
    switch (bn) {
      case 64: return launch_gemm_mode<64, false, 1, true>(p, pair, stream);
      case 128: return launch_gemm_mode<128, false, 1, true>(p, pair, stream);
      case 160: return launch_gemm_mode<160, false, 1, true>(p, pair, stream);
      case 256: return launch_gemm_mode<256, false, 1, true>(p, pair, stream);
      default: set_error("unsupported BN %d (64/128/160/256)", bn); return -1;
    }
  }
  // epilogue slots per warp: 3 (two residual chunks in flight) for the memory-bound linear GEMMs with a residual,
  // 1 for the K-deep convolutions (their epilogue has slack; the shared memory goes to the operand ring), else 2
  const int slots = p.amode != 0 ? 1 : (p.residual != nullptr ? 3 : 2);
  switch (bn) {
    case 64: return slots == 1 ? launch_gemm_mode<64, false, 1>(p, pair, stream) : slots == 3 ? launch_gemm_mode<64, false, 3>(p, pair, stream) : launch_gemm_mode<64, false, 2>(p, pair, stream);
    case 128: return slots == 1 ? launch_gemm_mode<128, false, 1>(p, pair, stream) : slots == 3 ? launch_gemm_mode<128, false, 3>(p, pair, stream) : launch_gemm_mode<128, false, 2>(p, pair, stream);
    case 160: return slots == 1 ? launch_gemm_mode<160, false, 1>(p, pair, stream) : slots == 3 ? launch_gemm_mode<160, false, 3>(p, pair, stream) : launch_gemm_mode<160, false, 2>(p, pair, stream);
    case 256: return launch_gemm_mode<256, false, 1>(p, pair, stream);
    default: set_error("unsupported BN %d (64/128/160/256)", bn); return -1;
  }
}

// Output / residual tensor maps: 4-D {cols, w, h, n} with one warp's 32 rows x 32 columns as the box.
static int make_epilogue_maps(GemmParams& p, int out_cols, bool conv) {
  const int oes = p.out_bf16 ? 2 : 4;
  uint64_t dims[4], ostr[3], rstr[3];
  uint32_t box[4];
  dims[0] = static_cast<uint64_t>(out_cols);
  if (!conv) {
    dims[1] = static_cast<uint64_t>(p.M); dims[2] = 1; dims[3] = 1;
    box[0] = p.wide ? 64 : 32; box[1] = 32; box[2] = 1; box[3] = 1;
    p.sbx = 32; p.sby = 1;
    ostr[0] = p.ldo * oes; ostr[1] = ostr[0] * dims[1]; ostr[2] = ostr[1];
    rstr[0] = p.ldr * 4; rstr[1] = rstr[0] * dims[1]; rstr[2] = rstr[1];
  } else {
    dims[1] = p.W; dims[2] = p.H; dims[3] = p.B;
    int sbx = p.bw < 32 ? p.bw : 32;
    int sby = p.bh < 32 / sbx ? p.bh : 32 / sbx;
    int sbz = 32 / (sbx * sby);
    p.sbx = sbx; p.sby = sby;
    box[0] = p.wide ? 64 : 32; box[1] = sbx; box[2] = sby; box[3] = sbz;
    ostr[0] = p.ldo * oes; ostr[1] = ostr[0] * p.W; ostr[2] = ostr[1] * p.H;
    rstr[0] = p.ldr * 4; rstr[1] = rstr[0] * p.W; rstr[2] = rstr[1] * p.H;
  }
  int rc = make_tmap(&p.tmOut, p.out, oes, (p.out_bf16 && !p.wide) ? 64 : 128, 4, dims, ostr, box);
  if (rc) return rc;
  p.tmRes = p.tmOut;
  if (p.residual) {
    AF_CHECK_ARG((reinterpret_cast<uintptr_t>(p.residual) & 15) == 0, "epilogue: residual not 16B aligned");
    rc = make_tmap(&p.tmRes, p.residual, 4, 128, 4, dims, rstr, box);
  }
  return rc;
}

// N-tile width.  160 divides every channel count of the UNet (320 .. 2560) without padding and is the default for
// those; the 256-wide tile (the most efficient tcgen05 shape: one A tile feeds 256 output columns) wins once the K loop
// dominates the tile - measured with scripts/bench_bn.py on B200 (profiles/r02_splitk.md): linear GEMMs without a
// residual and N >= 1280 from K = 640, everything from K = 2560 (with an fp32 residual the 160-wide tile has three
// epilogue slots against one at 256, so short-K GEMMs with a residual stay at 160), convolutions
// to 1280 channels from 32 row tiles (16x16 x 16 samples); the 160 remainder tiles of those are what split-K is for.
static int pick_bn(int N, int geglu, int bn_hint, int K, bool residual, bool conv, int m_tiles) {
  if (geglu) return 256;
  if (bn_hint == 64 || bn_hint == 128 || bn_hint == 160 || bn_hint == 256) return bn_hint;
  if (N % 160 == 0) {
#ifdef AF_BN160_ONLY   // A/B builds (scripts/build_alt.sh): the round-1 rule
    return 160;
#endif
    if (conv) return (N % 256 == 0 && N >= 1024 && m_tiles >= 32) ? 256 : 160;
    if (K >= 2560) return 256;
    if (!residual && N >= 1280 && K >= 640) return 256;
    return 160;
  }
  if (N % 256 == 0) return 256;
  if (N % 128 == 0) return 128;
  if (N <= 64) return 64;
  if (N <= 128) return 128;
  return 160;
}

static int fill_epilogue(GemmParams& p, const af_epilogue* ep, long long default_ldo) {
  p.bias = ep->bias;
  p.rowbias = ep->rowbias;
  p.rows_per_group = ep->rows_per_group > 0 ? ep->rows_per_group : 1;
  p.ld_rowbias = ep->ld_rowbias > 0 ? ep->ld_rowbias : p.N;
  p.residual = ep->residual;
  p.ldr = ep->ldr > 0 ? ep->ldr : default_ldo;
  p.out = ep->out;
  p.ldo = ep->ldo > 0 ? ep->ldo : default_ldo;
  p.out_bf16 = ep->out_dtype == AF_DTYPE_BF16;
  p.geglu = ep->geglu;
  p.gn_stats = ep->gn_stats;
  p.act = ep->act;
  AF_CHECK_ARG(ep->act == 0 || (ep->act == 1 && !ep->geglu), "epilogue: act %d unsupported", ep->act);
  AF_CHECK_ARG(!ep->gn_stats || (!ep->geglu && (reinterpret_cast<uintptr_t>(ep->gn_stats) & 15) == 0),
               "epilogue: gn_stats needs the generic epilogue and a 16-byte aligned buffer");
  AF_CHECK_ARG(ep->out != nullptr, "epilogue: out is null");
  AF_CHECK_ARG(ep->out_dtype == AF_DTYPE_BF16 || ep->out_dtype == AF_DTYPE_F32, "epilogue: bad out dtype %d",
               ep->out_dtype);
  AF_CHECK_ARG(!ep->geglu || ep->out_dtype == AF_DTYPE_BF16, "geglu epilogue writes bf16 only");
  AF_CHECK_ARG(!ep->geglu || (!ep->residual && !ep->rowbias), "geglu epilogue: residual / rowbias unsupported");
  AF_CHECK_ARG((reinterpret_cast<uintptr_t>(ep->out) & 15) == 0, "epilogue: out not 16B aligned");
  {
    const long long lim = 1ll << 31, rows = p.M;
    const long long groups = ep->rows_per_group > 0 ? rows / p.rows_per_group + 1 : 4096;  // conv: one group per image
    AF_CHECK_ARG(rows * p.ldo < lim && rows * p.ldr < lim && (!p.rowbias || groups * p.ld_rowbias < lim),
                 "epilogue: output / residual / rowbias larger than 2^31 elements");
  }
  AF_CHECK_ARG(p.ldo % 8 == 0 && p.ldr % 4 == 0 && p.ld_rowbias % 4 == 0, "epilogue: ldo %lld / ldr %lld / ld_rowbias %lld misaligned", p.ldo, p.ldr, p.ld_rowbias);
  return 0;
}

}  // namespace af

using namespace af;

extern "C" int af_gemm_bf16(const void* A0, long long lda0, int K0, const void* A1, long long lda1, int K1,
                            const void* Wt, int M, int N, const af_epilogue* ep, int bn_hint, cudaStream_t stream) {
  AF_CHECK_ARG(A0 && Wt && ep, "af_gemm_bf16: null pointer");
  AF_CHECK_ARG(M > 0 && N > 0 && K0 > 0 && K1 >= 0, "af_gemm_bf16: bad sizes M=%d N=%d K0=%d K1=%d", M, N, K0, K1);
  AF_CHECK_ARG(N % 8 == 0, "af_gemm_bf16: N=%d must be a multiple of 8", N);
  AF_CHECK_ARG(K1 == 0 || K0 % 64 == 0, "af_gemm_bf16: K0=%d must be a multiple of 64 for a dual-source A", K0);
  AF_CHECK_ARG((K0 + K1) % 8 == 0 && lda0 % 8 == 0 && (K1 == 0 || lda1 % 8 == 0),
               "af_gemm_bf16: K / lda must be multiples of 8 (16-byte TMA strides)");
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.trace = ep->trace;
  const int K = K0 + K1;
  const int bn = pick_bn(N, ep->geglu, bn_hint, K, ep->residual != nullptr, false, (M + 127) / 128);
  const bool pair = want_pair(ep->pair_mode, (M + 127) / 128, (N + bn - 1) / bn, bn, 0);
  AF_CHECK_ARG(!ep->geglu || N % 256 == 0, "geglu: packed N=%d must be a multiple of 256", N);
  {
    uint64_t dims[2] = {static_cast<uint64_t>(K0), static_cast<uint64_t>(M)};
    uint64_t str[1] = {static_cast<uint64_t>(lda0) * 2};
    uint32_t box[2] = {64, 128};
    int rc = make_tmap_bf16(&p.tmA0, A0, 2, dims, str, box);
    if (rc) return rc;
    p.tmA1 = p.tmA0;
  }
  if (K1 > 0) {
    AF_CHECK_ARG(A1 != nullptr, "af_gemm_bf16: A1 null with K1=%d", K1);
    uint64_t dims[2] = {static_cast<uint64_t>(K1), static_cast<uint64_t>(M)};
    uint64_t str[1] = {static_cast<uint64_t>(lda1) * 2};
    uint32_t box[2] = {64, 128};
    int rc = make_tmap_bf16(&p.tmA1, A1, 2, dims, str, box);
    if (rc) return rc;
  }
  {
    uint64_t dims[2] = {static_cast<uint64_t>(K), static_cast<uint64_t>(N)};
    uint64_t str[1] = {static_cast<uint64_t>(K) * 2};
    uint32_t box[2] = {64, static_cast<uint32_t>(pair ? bn / 2 : bn)};
    int rc = make_tmap_bf16(&p.tmB, Wt, 2, dims, str, box);
    if (rc) return rc;
  }
  p.M = M;
  p.N = N;
  p.num_kb = (K0 + 63) / 64 + (K1 + 63) / 64;
  p.cpb = p.num_kb;
  p.kb_split = (K0 + 63) / 64;
  p.amode = 0;
  p.m_tiles = (M + 127) / 128;
  p.n_tiles = (N + bn - 1) / bn;
  int rc = fill_epilogue(p, ep, ep->geglu ? N / 2 : N);
  if (rc) return rc;
#ifndef AF_GEMM_NO_WIDE
  p.wide = p.out_bf16 && !p.geglu && p.residual == nullptr && (bn == 128 || bn == 256);
#endif
  rc = make_epilogue_maps(p, ep->geglu ? N / 2 : N, false);
  if (rc) return rc;
  plan_split(p, bn, pair, ep);
  return dispatch_gemm(bn, p, pair, stream);
}

// output-pixel box of one 128-row conv tile: bw = largest power of two <= min(64, next_pow2(Wo)); rows / images
// fill up to 128 pixels
static void conv_tile_box(int Ho, int Wo, int* bw_, int* bh_, int* nb_) {
  int bw = 1;
  while (bw < Wo && bw < 64) bw <<= 1;
  int bh = 1;
  while (bh < Ho && bw * bh < 128) bh <<= 1;
  *bw_ = bw; *bh_ = bh; *nb_ = 128 / (bw * bh);
}

extern "C" int af_conv3x3_gn_slots(int Ho, int Wo) {
  int bw, bh, nb;
  conv_tile_box(Ho, Wo, &bw, &bh, &nb);
  if (bw * bh < 32) return 0;  // a 32-row quarter would straddle samples: use af_groupnorm_stats instead
  return ((Wo + bw - 1) / bw) * ((Ho + bh - 1) / bh) * (bw * bh / 32);
}

// amode 1: stride 1, pad 1 (two sources); 2: stride 2, pad 1; 3: stride 2 after F.pad(0,1,0,1).  The entry points have
// checked the arguments their mode needs.
static int conv3x3_launch(const char* who, const void* X0, int C0, const void* X1, int C1, const void* Wt, int B, int H,
                          int W, int Cout, int amode, const af_epilogue* ep, int bn_hint, cudaStream_t stream) {
  const int stride = amode == 1 ? 1 : 2;
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.trace = ep->trace;
  const int Cin = C0 + C1;
  const int Ho = stride == 1 ? H : H / 2, Wo = stride == 1 ? W : W / 2;
  int bw, bh, nb;
  conv_tile_box(Ho, Wo, &bw, &bh, &nb);
  const int bn = pick_bn(Cout, 0, bn_hint, 9 * Cin, ep->residual != nullptr, true,
                         ((Wo + bw - 1) / bw) * ((Ho + bh - 1) / bh) * ((B + nb - 1) / nb));
  const bool pair = want_pair(ep->pair_mode, ((Wo + bw - 1) / bw) * ((Ho + bh - 1) / bh) * ((B + nb - 1) / nb), (Cout + bn - 1) / bn, bn, 1);
  p.bw = bw; p.bh = bh; p.nb = nb;
  p.tiles_w = (Wo + bw - 1) / bw;
  p.tiles_h = (Ho + bh - 1) / bh;
  p.B = B; p.H = Ho; p.W = Wo; p.C0 = C0;
  const uint64_t es = 2;
  if (stride == 1) {
    uint32_t box[4] = {64, static_cast<uint32_t>(bw), static_cast<uint32_t>(bh), static_cast<uint32_t>(nb)};
    {
      uint64_t dims[4] = {static_cast<uint64_t>(C0), static_cast<uint64_t>(W), static_cast<uint64_t>(H), static_cast<uint64_t>(B)};
      uint64_t str[3] = {C0 * es, static_cast<uint64_t>(W) * C0 * es, static_cast<uint64_t>(H) * W * C0 * es};
      int rc = make_tmap_bf16(&p.tmA0, X0, 4, dims, str, box);
      if (rc) return rc;
      p.tmA1 = p.tmA0;
    }
    if (C1 > 0) {
      AF_CHECK_ARG(X1 != nullptr, "af_conv3x3_bf16: X1 null with C1=%d", C1);
      uint64_t dims[4] = {static_cast<uint64_t>(C1), static_cast<uint64_t>(W), static_cast<uint64_t>(H), static_cast<uint64_t>(B)};
      uint64_t str[3] = {C1 * es, static_cast<uint64_t>(W) * C1 * es, static_cast<uint64_t>(H) * W * C1 * es};
      int rc = make_tmap_bf16(&p.tmA1, X1, 4, dims, str, box);
      if (rc) return rc;
    }
    p.amode = 1;
  } else {
    uint32_t box[5] = {64, static_cast<uint32_t>(bw), 1, static_cast<uint32_t>(bh), static_cast<uint32_t>(nb)};
    uint64_t dims[5] = {static_cast<uint64_t>(2 * C0), static_cast<uint64_t>(W / 2), 2, static_cast<uint64_t>(H / 2),
                        static_cast<uint64_t>(B)};
    uint64_t str[4] = {2 * C0 * es, static_cast<uint64_t>(W) * C0 * es, 2 * static_cast<uint64_t>(W) * C0 * es,
                       static_cast<uint64_t>(H) * W * C0 * es};
    int rc = make_tmap_bf16(&p.tmA0, X0, 5, dims, str, box);
    if (rc) return rc;
    p.tmA1 = p.tmA0;
    p.amode = amode;
  }
  {
    const uint64_t K = 9ull * Cin;
    uint64_t dims[2] = {K, static_cast<uint64_t>(Cout)};
    uint64_t str[1] = {K * 2};
    uint32_t box[2] = {64, static_cast<uint32_t>(pair ? bn / 2 : bn)};
    int rc = make_tmap_bf16(&p.tmB, Wt, 2, dims, str, box);
    if (rc) return rc;
  }
  p.M = B * Ho * Wo;
  p.N = Cout;
  p.cpb = Cin / 64;
  p.kb_split = C0 / 64;
  p.num_kb = 9 * p.cpb;
  p.m_tiles = p.tiles_w * p.tiles_h * ((B + nb - 1) / nb);
  p.n_tiles = (Cout + bn - 1) / bn;
  int rc = fill_epilogue(p, ep, Cout);
  if (rc) return rc;
  if (p.rowbias && ep->rows_per_group <= 0) p.rows_per_group = Ho * Wo;
  if (p.gn_stats) {
    p.gn_slots = af_conv3x3_gn_slots(Ho, Wo);
    AF_CHECK_ARG(p.gn_slots > 0, "%s: gn_stats unsupported for %dx%d outputs (fewer than 32 pixels per tile row group)", who, Ho, Wo);
  }
#ifndef AF_GEMM_NO_WIDE
  p.wide = p.out_bf16 && p.residual == nullptr && (bn == 128 || bn == 256);
#endif
  rc = make_epilogue_maps(p, Cout, true);
  if (rc) return rc;
  plan_split(p, bn, pair, ep);
  return dispatch_gemm(bn, p, pair, stream);
}

extern "C" int af_conv3x3_bf16(const void* X0, int C0, const void* X1, int C1, const void* Wt, int B, int H, int W,
                               int Cout, int stride, const af_epilogue* ep, int bn_hint, cudaStream_t stream) {
  AF_CHECK_ARG(X0 && Wt && ep, "af_conv3x3_bf16: null pointer");
  AF_CHECK_ARG(stride == 1 || stride == 2, "af_conv3x3_bf16: stride %d", stride);
  AF_CHECK_ARG(C0 > 0 && C0 % 64 == 0 && C1 >= 0 && C1 % 64 == 0, "af_conv3x3_bf16: C0=%d C1=%d must be multiples of 64",
               C0, C1);
  AF_CHECK_ARG(Cout % 8 == 0, "af_conv3x3_bf16: Cout=%d must be a multiple of 8", Cout);
  AF_CHECK_ARG(stride == 1 || (C1 == 0 && H % 2 == 0 && W % 2 == 0), "af_conv3x3_bf16: stride 2 needs single source, even H/W");
  AF_CHECK_ARG(!ep->geglu, "af_conv3x3_bf16: geglu epilogue unsupported");
  return conv3x3_launch("af_conv3x3_bf16", X0, C0, X1, C1, Wt, B, H, W, Cout, stride, ep, bn_hint, stream);
}

extern "C" int af_conv3x3_down01_bf16(const void* X, int C, const void* Wt, int B, int H, int W, int Cout,
                                      const af_epilogue* ep, int bn_hint, cudaStream_t stream) {
  AF_CHECK_ARG(X && Wt && ep, "af_conv3x3_down01_bf16: null pointer");
  AF_CHECK_ARG(B > 0 && H > 0 && W > 0, "af_conv3x3_down01_bf16: bad sizes B=%d H=%d W=%d", B, H, W);
  AF_CHECK_ARG(C > 0 && C % 64 == 0, "af_conv3x3_down01_bf16: C=%d must be a multiple of 64", C);
  AF_CHECK_ARG(Cout > 0 && Cout % 8 == 0, "af_conv3x3_down01_bf16: Cout=%d must be a multiple of 8", Cout);
  AF_CHECK_ARG(H % 2 == 0 && W % 2 == 0, "af_conv3x3_down01_bf16: H=%d W=%d must be even", H, W);
  AF_CHECK_ARG(!ep->geglu, "af_conv3x3_down01_bf16: geglu epilogue unsupported");
  return conv3x3_launch("af_conv3x3_down01_bf16", X, C, nullptr, 0, Wt, B, H, W, Cout, 3, ep, bn_hint, stream);
}

// ---------------------------------------------------------------------------------------------
// Schedule introspection (no launch, no device needed: 148 SMs are assumed without one): the tile width, tile schedule
// and split-K plan af_gemm_bf16 / af_conv3x3_bf16 would use - the same pick_bn / want_pair / plan_split calls.
// out[0] = N-tile width, out[1] = 1 if CTA pairs, out[2] = K ranges per remainder tile (1 = whole tiles),
// out[3] = work units, out[4] = whole-K tiles before the split ones, out[5] = 1 if 64-column bf16 epilogue items.
// ---------------------------------------------------------------------------------------------
static void fill_plan(const GemmParams& p, int bn, bool pair, int* out) {
  out[0] = bn;
  out[1] = pair ? 1 : 0;
  out[2] = p.split;
  out[3] = p.num_units;
  out[4] = p.dp_tiles;
  out[5] = p.wide;
}

extern "C" int af_gemm_plan(int M, int N, int K, const af_epilogue* ep, int bn_hint, int* out) {
  AF_CHECK_ARG(ep && out && M > 0 && N > 0 && K > 0, "af_gemm_plan: bad arguments");
  GemmParams p;
  memset(&p, 0, sizeof(p));
  const int bn = pick_bn(N, ep->geglu, bn_hint, K, ep->residual != nullptr, false, (M + 127) / 128);
  const bool pair = want_pair(ep->pair_mode, (M + 127) / 128, (N + bn - 1) / bn, bn, 0);
  p.num_kb = (K + 63) / 64;
  p.m_tiles = (M + 127) / 128;
  p.n_tiles = (N + bn - 1) / bn;
  p.geglu = ep->geglu;
  p.residual = ep->residual;
  p.out_bf16 = ep->out_dtype == AF_DTYPE_BF16;
#ifndef AF_GEMM_NO_WIDE
  p.wide = p.out_bf16 && !p.geglu && p.residual == nullptr && (bn == 128 || bn == 256);
#endif
  plan_split(p, bn, pair, ep);
  fill_plan(p, bn, pair, out);
  return 0;
}

extern "C" int af_conv3x3_plan(int C0, int C1, int B, int H, int W, int Cout, int stride, const af_epilogue* ep,
                               int bn_hint, int* out) {
  AF_CHECK_ARG(ep && out && B > 0 && H > 0 && W > 0 && Cout > 0 && C0 > 0 && (stride == 1 || stride == 2),
               "af_conv3x3_plan: bad arguments");
  GemmParams p;
  memset(&p, 0, sizeof(p));
  const int Cin = C0 + C1;
  const int Ho = stride == 1 ? H : H / 2, Wo = stride == 1 ? W : W / 2;
  int bw, bh, nb;
  conv_tile_box(Ho, Wo, &bw, &bh, &nb);
  const int m_tiles = ((Wo + bw - 1) / bw) * ((Ho + bh - 1) / bh) * ((B + nb - 1) / nb);
  const int bn = pick_bn(Cout, 0, bn_hint, 9 * Cin, ep->residual != nullptr, true, m_tiles);
  const bool pair = want_pair(ep->pair_mode, m_tiles, (Cout + bn - 1) / bn, bn, 1);
  p.amode = stride == 1 ? 1 : 2;
  p.num_kb = 9 * (Cin / 64);
  p.m_tiles = m_tiles;
  p.n_tiles = (Cout + bn - 1) / bn;
  p.residual = ep->residual;
  p.out_bf16 = ep->out_dtype == AF_DTYPE_BF16;
#ifndef AF_GEMM_NO_WIDE
  p.wide = p.out_bf16 && p.residual == nullptr && (bn == 128 || bn == 256);
#endif
  plan_split(p, bn, pair, ep);
  fill_plan(p, bn, pair, out);
  return 0;
}

