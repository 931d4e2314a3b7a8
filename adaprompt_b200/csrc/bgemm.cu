// Batched, strided "NT" GEMM with attention-backward epilogues (Stage-1 training step, SURVEY.md section 8 row T1).
//
//   C[z] = epi( A[z] [M,K] . B[z] [N,K]^T ),   z = (b0, b1) over two batch strides (sample, head)
//
// The backward pass of CrossAttention.forward (ldm/modules/attention.py:198-242; autograd of the einsum / softmax /
// einsum chain) is five small-K or small-N contractions per (sample, head) whose operands are strided column slices
// of the projection buffers.  They are launch- and bandwidth-bound rather than tensor-peak-bound (K or N is the head
// dim 40/80/160), so this kernel uses plain mma.sync.m16n8k16 bf16 tiles fed by cp.async - no TMA descriptors per
// slice - and fuses the softmax recomputation into its epilogue:
//   mode 0   C = alpha * acc
//   mode 1   C = exp2(acc - vec[row])                      P   from S   (vec = log2-sum-exp of the query rows)
//   mode 2   C = exp2(acc - vec[col])                      P^T from S^T
//   mode 3   C = alpha * P[row,col] * (acc - vec[row])     dS   = P   o (dP   - delta)
//   mode 4   C = alpha * P[row,col] * (acc - vec[col])     dS^T = P^T o (dP^T - delta)
// Entries with row >= valid_rows or col >= valid_cols are written as 0 (padded keys / queries).
// With a key mask (bgemm_masked_kernel, modes 1-4: attention.py:223-232) masked keys - columns of modes 1 / 3, rows of
// modes 2 / 4 - get P = 0 and dS = 0, or P = 1 / (number of valid keys) in modes 1 / 2 where vec = +inf (a sample that
// keeps no key: the forward gave its rows the mean of V).  Kept keys take the unmasked arithmetic unchanged.
#include "../../include/adaface_b200.h"
#include "common.cuh"

namespace af {

struct BgemmParams {
  const __nv_bfloat16* A; long long lda, sA0, sA1;
  const __nv_bfloat16* B; long long ldb, sB0, sB1;
  void* C; long long ldc, sC0, sC1; int c_f32;
  const float* vec; long long sV0, sV1;
  const __nv_bfloat16* P; long long ldp, sP0, sP1;
  int M, N, K, nb1, mode, valid_rows, valid_cols, staged;
  float alpha;
  const uint8_t* kmask; long long sM0, sM1;      // masked kernel only
};

__device__ __forceinline__ void cp_async16(void* dst, const void* src, bool valid) {
  const int n = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(p)));
}
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

constexpr int kBM = 128, kBK = 32, kPitch = kBK + 8, kStages = 3;

// MODE is a template parameter: as a run-time field the epilogue carried a five-way option chain inside its 32-iteration
// element loop (the same pattern that cost the tcgen05 GEMM epilogue 70 cycles per iteration).
template <int BN, int MODE, bool MASK>
__device__ __forceinline__ void bgemm_body(const BgemmParams& p) {
  constexpr int WARPS_N = BN / 32, WARPS_M = 8 / WARPS_N, WM = kBM / WARPS_M, MT = WM / 16;
  extern __shared__ __align__(16) uint8_t smem_b[];
  __nv_bfloat16* sA = reinterpret_cast<__nv_bfloat16*>(smem_b);                 // [stages][128][pitch]
  __nv_bfloat16* sB = sA + kStages * kBM * kPitch;                              // [stages][BN][pitch]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = warp / WARPS_N, wn = warp % WARPS_N;
  const int z = blockIdx.z, b0 = z / p.nb1, b1 = z % p.nb1;
  const int m0 = blockIdx.y * kBM, n0 = blockIdx.x * BN;
  const __nv_bfloat16* A = p.A + b0 * p.sA0 + b1 * p.sA1;
  const __nv_bfloat16* B = p.B + b0 * p.sB0 + b1 * p.sB1;
  // Staged epilogue (bf16 outputs with 16-byte aligned rows): the tile is converted into shared memory and leaves in
  // 16-byte row chunks; for modes 3 / 4 the P tile is fetched the same way by cp.async BEFORE the main loop.  (With one
  // 4-byte store / load per accumulator pair the 4096 x 4096 softmax-recompute GEMMs ran at 1.1 TB/s.)
  constexpr int kCP = BN + 8;                                                  // staging pitch (bf16 elements)
  __nv_bfloat16* sC = reinterpret_cast<__nv_bfloat16*>(smem_b);                // reuses the operand ring after the loop
  __nv_bfloat16* sP = sB + kStages * BN * kPitch;                              // [128][kCP], modes 3 / 4 only
  const bool staged = p.staged != 0;
  const __nv_bfloat16* Pt = p.P ? p.P + b0 * p.sP0 + b1 * p.sP1 : nullptr;
  if (MODE >= 3 && staged) {
    for (int i = tid; i < kBM * (BN / 8); i += 256) {
      const int r = i / (BN / 8), c = (i % (BN / 8)) * 8;
      const bool ok = (m0 + r) < p.M && (n0 + c) < p.N;                       // N % 8 == 0 when staged
      cp_async16(sP + r * kCP + c, ok ? Pt + static_cast<long long>(m0 + r) * p.ldp + n0 + c : Pt, ok);
    }
    cp_async_commit();
  }

  auto load_stage = [&](int stage, int k0) {
    __nv_bfloat16* a = sA + stage * kBM * kPitch;
    __nv_bfloat16* b = sB + stage * BN * kPitch;
    for (int i = tid; i < kBM * 4; i += 256) {
      const int r = i >> 2, c = (i & 3) * 8;
      const bool ok = (m0 + r) < p.M && (k0 + c) < p.K;
      cp_async16(a + r * kPitch + c, ok ? A + static_cast<long long>(m0 + r) * p.lda + k0 + c : A, ok);
    }
    for (int i = tid; i < BN * 4; i += 256) {
      const int r = i >> 2, c = (i & 3) * 8;
      const bool ok = (n0 + r) < p.N && (k0 + c) < p.K;
      cp_async16(b + r * kPitch + c, ok ? B + static_cast<long long>(n0 + r) * p.ldb + k0 + c : B, ok);
    }
  };

  float acc[MT][4][4];
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.f;

  const int nk = (p.K + kBK - 1) / kBK;
#pragma unroll
  for (int s = 0; s < kStages - 1; ++s) {
    if (s < nk) load_stage(s, s * kBK);
    cp_async_commit();
  }
  for (int kt = 0; kt < nk; ++kt) {
    cp_async_wait<kStages - 2>();
    __syncthreads();
    if (kt + kStages - 1 < nk) load_stage((kt + kStages - 1) % kStages, (kt + kStages - 1) * kBK);
    cp_async_commit();
    const __nv_bfloat16* a = sA + (kt % kStages) * kBM * kPitch;
    const __nv_bfloat16* b = sB + (kt % kStages) * BN * kPitch;
#pragma unroll
    for (int kk = 0; kk < kBK; kk += 16) {
      uint32_t af[MT][4], bf[2][4];
#pragma unroll
      for (int i = 0; i < MT; ++i)
        ldsm_x4(af[i], a + (wm * WM + i * 16 + (lane & 15)) * kPitch + kk + (lane >> 4) * 8);
#pragma unroll
      for (int j = 0; j < 2; ++j)
        ldsm_x4(bf[j], b + (wn * 32 + j * 16 + (lane & 7) + (lane >> 4) * 8) * kPitch + kk + ((lane >> 3) & 1) * 8);
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) mma_bf16_16816(acc[i][j], af[i], bf[j >> 1][(j & 1) * 2], bf[j >> 1][(j & 1) * 2 + 1]);
    }
  }
  cp_async_wait<0>();

  // ---- epilogue
  const float* vec = p.vec ? p.vec + b0 * p.sV0 + b1 * p.sV1 : nullptr;
  const uint8_t* km = MASK ? p.kmask + b0 * p.sM0 + b1 * p.sM1 : nullptr;
  const __nv_bfloat16* P = Pt;
  uint8_t* Cb = static_cast<uint8_t*>(p.C) + (b0 * p.sC0 + b1 * p.sC1) * (p.c_f32 ? 4 : 2);
  if (staged) __syncthreads();          // every warp is done with the operand ring (sC aliases it); sP has landed
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int hrow = 0; hrow < 2; ++hrow) {
      const int lrow = wm * WM + i * 16 + (lane >> 2) + hrow * 8;
      const int row = m0 + lrow;
      if (row >= p.M) continue;
      const float rv = (vec && (MODE == 1 || MODE == 3) && row < p.valid_rows) ? vec[row] : 0.f;
      const bool keep_row = !MASK || MODE == 1 || MODE == 3 || (row < p.valid_rows && km[row] != 0);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int lcol = wn * 32 + j * 8 + (lane & 3) * 2;
        const int col = n0 + lcol;
        if (col >= p.N) continue;
        float v0 = acc[i][j][hrow * 2], v1 = acc[i][j][hrow * 2 + 1];
        const bool ok0 = row < p.valid_rows && col < p.valid_cols, ok1 = row < p.valid_rows && col + 1 < p.valid_cols;
        if constexpr (MODE == 0) {
          v0 *= p.alpha; v1 *= p.alpha;
        } else if constexpr (MODE == 1) {
          v0 = fast_exp2(v0 - rv); v1 = fast_exp2(v1 - rv);
        } else if constexpr (MODE == 2) {
          v0 = fast_exp2(v0 - (ok0 ? vec[col] : 0.f)); v1 = fast_exp2(v1 - (ok1 ? vec[col + 1] : 0.f));
        } else {
          const __nv_bfloat162 pp = staged ? *reinterpret_cast<const __nv_bfloat162*>(sP + lrow * kCP + lcol)
                                           : *reinterpret_cast<const __nv_bfloat162*>(P + static_cast<long long>(row) * p.ldp + col);
          const float c0 = MODE == 3 ? rv : (ok0 ? vec[col] : 0.f), c1 = MODE == 3 ? rv : (ok1 ? vec[col + 1] : 0.f);
          v0 = p.alpha * __bfloat162float(pp.x) * (v0 - c0);
          v1 = p.alpha * __bfloat162float(pp.y) * (v1 - c1);
        }
        if constexpr (MASK) {
          const bool k0 = MODE == 1 || MODE == 3 ? ok0 && km[col] != 0 : keep_row;
          const bool k1 = MODE == 1 || MODE == 3 ? ok1 && km[col + 1] != 0 : keep_row;
          float e0 = 0.f, e1 = 0.f;       // P of a masked key: 1 / valid keys in a sample that keeps none
          if constexpr (MODE == 1) {
            e0 = e1 = rv == INFINITY ? 1.f / static_cast<float>(p.valid_cols) : 0.f;
          } else if constexpr (MODE == 2) {
            e0 = ok0 && vec[col] == INFINITY ? 1.f / static_cast<float>(p.valid_rows) : 0.f;
            e1 = ok1 && vec[col + 1] == INFINITY ? 1.f / static_cast<float>(p.valid_rows) : 0.f;
          }
          v0 = k0 ? v0 : e0;
          v1 = k1 ? v1 : e1;
        }
        v0 = ok0 ? v0 : 0.f;
        v1 = ok1 ? v1 : 0.f;
        if (staged) {
          *reinterpret_cast<uint32_t*>(sC + lrow * kCP + lcol) = pack_bf16x2(v0, v1);
        } else if (p.c_f32) {
          *reinterpret_cast<float2*>(reinterpret_cast<float*>(Cb) + static_cast<long long>(row) * p.ldc + col) = make_float2(v0, v1);
        } else {
          *reinterpret_cast<uint32_t*>(reinterpret_cast<__nv_bfloat16*>(Cb) + static_cast<long long>(row) * p.ldc + col) = pack_bf16x2(v0, v1);
        }
      }
    }
  if (staged) {
    __syncthreads();
    __nv_bfloat16* Cg = reinterpret_cast<__nv_bfloat16*>(Cb);
    for (int i = tid; i < kBM * (BN / 8); i += 256) {
      const int r = i / (BN / 8), c = (i % (BN / 8)) * 8;
      if (m0 + r < p.M && n0 + c < p.N)
        *reinterpret_cast<uint4*>(Cg + static_cast<long long>(m0 + r) * p.ldc + n0 + c) =
            *reinterpret_cast<const uint4*>(sC + r * kCP + c);
    }
  }
}

template <int BN, int MODE>
__global__ void __launch_bounds__(256) bgemm_kernel(const BgemmParams p) {
  bgemm_body<BN, MODE, false>(p);
}
template <int BN, int MODE>
__global__ void __launch_bounds__(256) bgemm_masked_kernel(const BgemmParams p) {
  bgemm_body<BN, MODE, true>(p);
}

template <int BN, int MODE, bool MASK>
static int launch_bgemm_m(const BgemmParams& p, int batch, cudaStream_t stream) {
  // operand ring (also the output staging tile: 128 x (BN + 8) bf16 fits) + the P tile of modes 3 / 4
  static_assert(kStages * (kBM + BN) * kPitch >= kBM * (BN + 8), "staging tile must fit in the operand ring");
  constexpr int smem = kStages * (kBM + BN) * kPitch * 2 + (MODE >= 3 ? kBM * (BN + 8) * 2 : 0);
  const auto kernel = MASK ? bgemm_masked_kernel<BN, MODE> : bgemm_kernel<BN, MODE>;
  static bool configured = false;
  if (!configured) {
    AF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  dim3 grid((p.N + BN - 1) / BN, (p.M + kBM - 1) / kBM, batch);
  kernel<<<grid, 256, smem, stream>>>(p);
  AF_LAUNCH_CHECK(MASK ? "bgemm_masked_kernel" : "bgemm_kernel");
  return 0;
}
template <int BN>
static int launch_bgemm(const BgemmParams& p, int batch, cudaStream_t stream) {
  if (p.kmask) {
    switch (p.mode) {
      case 1: return launch_bgemm_m<BN, 1, true>(p, batch, stream);
      case 2: return launch_bgemm_m<BN, 2, true>(p, batch, stream);
      case 3: return launch_bgemm_m<BN, 3, true>(p, batch, stream);
      default: return launch_bgemm_m<BN, 4, true>(p, batch, stream);
    }
  }
  switch (p.mode) {
    case 0: return launch_bgemm_m<BN, 0, false>(p, batch, stream);
    case 1: return launch_bgemm_m<BN, 1, false>(p, batch, stream);
    case 2: return launch_bgemm_m<BN, 2, false>(p, batch, stream);
    case 3: return launch_bgemm_m<BN, 3, false>(p, batch, stream);
    default: return launch_bgemm_m<BN, 4, false>(p, batch, stream);
  }
}

static int fill_params(const af_bgemm* g, BgemmParams* out, const char* fn) {
  AF_CHECK_ARG(g && g->A && g->B && g->C, "%s: null pointer", fn);
  AF_CHECK_ARG(g->M > 0 && g->N > 0 && g->K > 0 && g->nb0 > 0 && g->nb1 > 0, "%s: bad sizes", fn);
  AF_CHECK_ARG(g->K % 8 == 0 && g->N % 2 == 0, "%s: K=%d must be a multiple of 8, N=%d even", fn, g->K, g->N);
  AF_CHECK_ARG(g->lda % 8 == 0 && g->ldb % 8 == 0 && g->sA0 % 8 == 0 && g->sA1 % 8 == 0 && g->sB0 % 8 == 0 && g->sB1 % 8 == 0,
               "%s: operand pitches / batch strides must be multiples of 8 elements (16-byte cp.async)", fn);
  AF_CHECK_ARG((reinterpret_cast<uintptr_t>(g->A) & 15) == 0 && (reinterpret_cast<uintptr_t>(g->B) & 15) == 0,
               "%s: operands must be 16-byte aligned", fn);
  AF_CHECK_ARG(g->ldc % 2 == 0 && g->sC0 % 2 == 0 && g->sC1 % 2 == 0, "%s: C pitch / strides must be even", fn);
  AF_CHECK_ARG(g->mode >= 0 && g->mode <= 4, "%s: mode %d", fn, g->mode);
  AF_CHECK_ARG(g->mode == 0 || g->vec, "%s: mode %d needs vec", fn, g->mode);
  AF_CHECK_ARG(g->mode < 3 || (g->P && g->ldp % 2 == 0 && g->sP0 % 2 == 0 && g->sP1 % 2 == 0), "%s: mode %d needs P (even pitch)", fn, g->mode);
  AF_CHECK_ARG(static_cast<long long>(g->nb0) * g->nb1 <= 65535, "%s: batch too large", fn);
  BgemmParams& p = *out;
  memset(&p, 0, sizeof(p));
  p.A = static_cast<const __nv_bfloat16*>(g->A); p.lda = g->lda; p.sA0 = g->sA0; p.sA1 = g->sA1;
  p.B = static_cast<const __nv_bfloat16*>(g->B); p.ldb = g->ldb; p.sB0 = g->sB0; p.sB1 = g->sB1;
  p.C = g->C; p.ldc = g->ldc; p.sC0 = g->sC0; p.sC1 = g->sC1; p.c_f32 = g->c_dtype == AF_DTYPE_F32;
  p.vec = g->vec; p.sV0 = g->sV0; p.sV1 = g->sV1;
  p.P = static_cast<const __nv_bfloat16*>(g->P); p.ldp = g->ldp; p.sP0 = g->sP0; p.sP1 = g->sP1;
  p.M = g->M; p.N = g->N; p.K = g->K; p.nb1 = g->nb1; p.mode = g->mode;
  p.valid_rows = g->valid_rows > 0 ? g->valid_rows : g->M;
  p.valid_cols = g->valid_cols > 0 ? g->valid_cols : g->N;
  p.alpha = g->alpha;
  // staged (coalesced) epilogue: bf16 output whose rows and batch slices start on 16-byte boundaries
  p.staged = (!p.c_f32 && g->mode != 0 && g->N % 8 == 0 && g->ldc % 8 == 0 && g->sC0 % 8 == 0 && g->sC1 % 8 == 0 &&
              (reinterpret_cast<uintptr_t>(g->C) & 15) == 0 &&
              (g->mode < 3 || (g->ldp % 8 == 0 && g->sP0 % 8 == 0 && g->sP1 % 8 == 0 &&
                               (reinterpret_cast<uintptr_t>(g->P) & 15) == 0))) ? 1 : 0;
  return 0;
}

}  // namespace af

using namespace af;

extern "C" int af_bgemm_bf16(const af_bgemm* g, cudaStream_t stream) {
  BgemmParams p;
  if (int rc = fill_params(g, &p, "af_bgemm_bf16")) return rc;
  const int batch = g->nb0 * g->nb1;
  return g->N <= 64 ? launch_bgemm<64>(p, batch, stream) : launch_bgemm<128>(p, batch, stream);
}

extern "C" int af_bgemm_masked_bf16(const af_bgemm* g, const unsigned char* key_mask, long long sM0, long long sM1,
                                    cudaStream_t stream) {
  BgemmParams p;
  if (int rc = fill_params(g, &p, "af_bgemm_masked_bf16")) return rc;
  AF_CHECK_ARG(key_mask, "af_bgemm_masked_bf16: null key_mask");
  AF_CHECK_ARG(g->mode >= 1, "af_bgemm_masked_bf16: mode %d takes no key mask (modes 1-4)", g->mode);
  AF_CHECK_ARG(sM0 >= 0 && sM1 >= 0, "af_bgemm_masked_bf16: negative mask strides");
  p.kmask = key_mask; p.sM0 = sM0; p.sM1 = sM1;
  const int batch = g->nb0 * g->nb1;
  return g->N <= 64 ? launch_bgemm<64>(p, batch, stream) : launch_bgemm<128>(p, batch, stream);
}
