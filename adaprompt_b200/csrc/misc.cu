// Small CUDA-core kernels around the tensor-core path: first/last convolutions (4 channels), time
// embedding, small-M fp32 linears, casts / nearest upsample, CFG + DDIM update.
#include "../../include/adaface_b200.h"
#include "common.cuh"

namespace af {

// ---------------------------------------------------------------------------------------------
// conv_in: NCHW fp32 [B,Cin,H,W] (Cin = 4 or 3) -> NHWC fp32 [B,H,W,Cout], 3x3 pad 1, fp32 math.
// Reference: UNetModel.input_blocks[0] = conv_nd(2, 4, 320, 3, padding=1) (openaimodel.py:527-533), the VAE's
// Decoder.conv_in (4 -> 512) and Encoder.conv_in (3 -> 128, model.py:436-440).
// Block = 32 consecutive pixels of one image row; the weights live in shared memory as [tap*Cin + ci][Cout] so a
// thread reads the four output channels it owns with one 16-byte load per tap, and the input value of a (pixel,
// tap) is one broadcast load shared by all channel quads.  Stores are 512 B contiguous per warp (NHWC).
// ---------------------------------------------------------------------------------------------
template <int CIN>
__global__ void __launch_bounds__(320, 2) conv_in_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                      const float* __restrict__ bias, float* __restrict__ y, int B,
                                                      int H, int W, int Cout, int rows) {
  constexpr int TP = 32, TAPS = CIN * 9;
  extern __shared__ float smem_ci[];
  float* sw = smem_ci;                          // [TAPS][Cout]
  float* patch = smem_ci + TAPS * Cout;         // [CIN][3][TP + 2]
  const int wt = blockIdx.x * TP;
  const int b = blockIdx.z;
  // The 36 x Cout weights are staged ONCE per block and reused for `rows` image rows (a block per row re-read 46 KB of
  // weights for 32 pixels of work: 119 us for the 64x64, batch-16 layer).  Consecutive threads take consecutive output
  // channels: strided global reads of an L2-resident 46 KB array, conflict-free shared-memory writes.
  for (int i = threadIdx.x; i < TAPS * Cout; i += blockDim.x) {
    const int t = i / Cout, co = i - t * Cout;           // global layout [co][ci][ky][kx]
    sw[i] = w[co * TAPS + t];
  }
  const int cq = Cout >> 2;                      // channel quads
  const int groups = blockDim.x / cq;            // pixel groups served concurrently
  const int pg = threadIdx.x / cq, q = threadIdx.x - pg * cq;
  const int ppg = TP / groups;                   // pixels per group (host guarantees divisibility)
  const float4 bv = bias ? *reinterpret_cast<const float4*>(bias + (pg < groups ? q : 0) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
  const int h_end = min(H, static_cast<int>(blockIdx.y + 1) * rows);
  for (int h = blockIdx.y * rows; h < h_end; ++h) {
    __syncthreads();                               // the previous row's patch has been consumed (first pass: weights staged)
    for (int i = threadIdx.x; i < CIN * 3 * (TP + 2); i += blockDim.x) {
      const int c = i / (3 * (TP + 2));
      const int rr = (i / (TP + 2)) % 3;
      const int cc = i % (TP + 2);
      const int hh = h + rr - 1, ww = wt + cc - 1;
      float v = 0.f;
      if (hh >= 0 && hh < H && ww >= 0 && ww < W) v = x[((static_cast<size_t>(b) * CIN + c) * H + hh) * W + ww];
      patch[i] = v;
    }
    __syncthreads();
    if (pg >= groups) continue;
    for (int p0 = 0; p0 < ppg; p0 += 8) {
      float4 acc[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[i] = bv;
#pragma unroll 1
      for (int c = 0; c < CIN; ++c)
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) {
            const float4 wv = *reinterpret_cast<const float4*>(sw + ((c * 3 + ky) * 3 + kx) * Cout + q * 4);
            const float* pr = patch + (c * 3 + ky) * (TP + 2) + pg * ppg + p0 + kx;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float xv = pr[i];
              acc[i].x = fmaf(wv.x, xv, acc[i].x); acc[i].y = fmaf(wv.y, xv, acc[i].y);
              acc[i].z = fmaf(wv.z, xv, acc[i].z); acc[i].w = fmaf(wv.w, xv, acc[i].w);
            }
          }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int px = wt + pg * ppg + p0 + i;
        if (px < W)
          *reinterpret_cast<float4*>(y + ((static_cast<size_t>(b) * H + h) * W + px) * Cout + q * 4) = acc[i];
      }
    }
  }
}

// NHWC fp32 [B, HW, CP] -> NCHW fp32 [B, COUT, HW] (first COUT of the CP padded channels): the UNet's last
// convolution runs on the tensor cores with Cout padded 4 -> 8; this restores the public layout.
__global__ void __launch_bounds__(256) nhwc_to_nchw_kernel(const float* __restrict__ x, float* __restrict__ y, int B,
                                                           int HW, int CP, int COUT) {
  const size_t total = static_cast<size_t>(B) * HW;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t b = i / HW, p = i - b * HW;
    const float4 v = __ldg(reinterpret_cast<const float4*>(x + i * CP));
    float* o = y + b * COUT * HW + p;
    o[0] = v.x;
    if (COUT > 1) o[HW] = v.y;
    if (COUT > 2) o[2 * static_cast<size_t>(HW)] = v.z;
    if (COUT > 3) o[3 * static_cast<size_t>(HW)] = v.w;
  }
}

// ---------------------------------------------------------------------------------------------
// conv_out: NHWC bf16 [B,H,W,C] -> NCHW fp32 [B,COUT,H,W], 3x3 pad 1; warp per output pixel.
// Reference: UNetModel.out[-1] = conv_nd(2, 320, 4, 3, padding=1) (openaimodel.py:693-697).
// Weights pre-packed fp32 [COUT][3][3][C] and staged in shared memory.
// ---------------------------------------------------------------------------------------------
template <int COUT>
__global__ void __launch_bounds__(256) conv_out_kernel(const __nv_bfloat16* __restrict__ x,
                                                       const float* __restrict__ w, const float* __restrict__ bias,
                                                       float* __restrict__ y, int B, int H, int W, int C) {
  extern __shared__ float sw[];  // [COUT*9*C]
  for (int i = threadIdx.x; i < COUT * 9 * C; i += blockDim.x) sw[i] = w[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  const long long total = static_cast<long long>(B) * H * W;
  const int nvec = C >> 3;
  for (long long pix = static_cast<long long>(blockIdx.x) * warps_per_block + (threadIdx.x >> 5); pix < total;
       pix += static_cast<long long>(gridDim.x) * warps_per_block) {
    const int wq = static_cast<int>(pix % W);
    const int hq = static_cast<int>((pix / W) % H);
    const int b = static_cast<int>(pix / (static_cast<long long>(W) * H));
    float acc[COUT];
#pragma unroll
    for (int o = 0; o < COUT; ++o) acc[o] = 0.f;
    for (int tap = 0; tap < 9; ++tap) {
      const int hh = hq + tap / 3 - 1, ww = wq + tap % 3 - 1;
      if (hh < 0 || hh >= H || ww < 0 || ww >= W) continue;
      const uint4* xp = reinterpret_cast<const uint4*>(x + ((static_cast<size_t>(b) * H + hh) * W + ww) * C);
      for (int k = lane; k < nvec; k += 32) {
        const uint4 raw = __ldg(xp + k);
        const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&raw);
        float xv[8];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 f = __bfloat1622float2(h2[e]);
          xv[2 * e] = f.x;
          xv[2 * e + 1] = f.y;
        }
#pragma unroll
        for (int o = 0; o < COUT; ++o) {
          const float* wp = sw + (o * 9 + tap) * C + k * 8;
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[o] += xv[e] * wp[e];
        }
      }
    }
#pragma unroll
    for (int o = 0; o < COUT; ++o) acc[o] = warp_sum(acc[o]);
    if (lane < COUT) {
      float v = 0.f;
#pragma unroll
      for (int o = 0; o < COUT; ++o)
        if (lane == o) v = acc[o];
      y[((static_cast<size_t>(b) * COUT + lane) * H + hq) * W + wq] = v + (bias ? bias[lane] : 0.f);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// sinusoidal timestep embedding (ldm/modules/diffusionmodules/util.py:154-174): [cos | sin], fp32
// ---------------------------------------------------------------------------------------------
__global__ void timestep_embedding_kernel(const float* __restrict__ t, float* __restrict__ out, int B, int dim) {
  const int half = dim >> 1;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * half) return;
  const int b = i / half, j = i - b * half;
  const float freq = expf(-9.210340371976184f * static_cast<float>(j) / static_cast<float>(half));  // ln(10000)
  const float arg = t[b] * freq;
  out[static_cast<size_t>(b) * dim + j] = cosf(arg);
  out[static_cast<size_t>(b) * dim + half + j] = sinf(arg);
  if ((dim & 1) && j == 0) out[static_cast<size_t>(b) * dim + dim - 1] = 0.f;
}

// ---------------------------------------------------------------------------------------------
// small-M fp32 linear: y[M,N] = act_out(act_in(x)[M,K] @ W[N,K]^T + b).
// Used for time_embed (openaimodel.py:518-522,847) and the 22 ResBlock emb_layers (:222-228,268), whose
// weights are concatenated into one [sum Cout, 1280] matrix at load time.  Weight-read bound (113 MB fp32 per
// UNet step): x (<= 16 rows per pass) is staged in shared memory with the input activation applied once, a warp
// produces FOUR output features per pass so every shared-memory read of x is reused four times, and the weights
// stream through 16-byte coalesced loads.
// ---------------------------------------------------------------------------------------------
constexpr int kLsRows = 16, kLsFeat = 4;
__global__ void __launch_bounds__(256) linear_small_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                           const float* __restrict__ bias, float* __restrict__ y,
                                                           int M, int N, int K, int silu_in, int silu_out) {
  extern __shared__ float sx[];  // [kLsRows][K]
  const int lane = threadIdx.x & 31;
  const int n0 = (blockIdx.x * 8 + (threadIdx.x >> 5)) * kLsFeat;
  const int nvec = K >> 2;
  for (int m0 = 0; m0 < M; m0 += kLsRows) {
    const int mr = min(kLsRows, M - m0);
    __syncthreads();
    for (int i = threadIdx.x; i < kLsRows * nvec; i += blockDim.x) {
      const int r = i / nvec;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < mr) {
        v = __ldg(reinterpret_cast<const float4*>(x + static_cast<size_t>(m0 + r) * K) + (i - r * nvec));
        if (silu_in) {
          v.x = silu_f(v.x); v.y = silu_f(v.y); v.z = silu_f(v.z); v.w = silu_f(v.w);
        }
      }
      reinterpret_cast<float4*>(sx)[i] = v;
    }
    __syncthreads();
    if (n0 < N) {
      float acc[kLsFeat][kLsRows];
#pragma unroll
      for (int f = 0; f < kLsFeat; ++f)
#pragma unroll
        for (int r = 0; r < kLsRows; ++r) acc[f][r] = 0.f;
      const float4* wr[kLsFeat];
#pragma unroll
      for (int f = 0; f < kLsFeat; ++f) wr[f] = reinterpret_cast<const float4*>(w + static_cast<size_t>(min(n0 + f, N - 1)) * K);
      for (int k = lane; k < nvec; k += 32) {
        float4 wv[kLsFeat];
#pragma unroll
        for (int f = 0; f < kLsFeat; ++f) wv[f] = __ldg(wr[f] + k);
#pragma unroll
        for (int r = 0; r < kLsRows; ++r) {
          const float4 xv = reinterpret_cast<const float4*>(sx)[r * nvec + k];
#pragma unroll
          for (int f = 0; f < kLsFeat; ++f)
            acc[f][r] = fmaf(wv[f].x, xv.x, fmaf(wv[f].y, xv.y, fmaf(wv[f].z, xv.z, fmaf(wv[f].w, xv.w, acc[f][r]))));
        }
      }
#pragma unroll
      for (int f = 0; f < kLsFeat; ++f)
#pragma unroll
        for (int r = 0; r < kLsRows; ++r) {
          const float sacc = warp_sum(acc[f][r]);
          if (lane == ((f * kLsRows + r) & 31)) acc[f][r] = sacc;   // lane (f*16+r)%32 keeps output (f, r)
        }
      // each lane now owns two outputs: (f, r) and (f + 2, r) with f*16 + r == lane
#pragma unroll
      for (int f = 0; f < kLsFeat; ++f)
#pragma unroll
        for (int r = 0; r < kLsRows; ++r)
          if (lane == ((f * kLsRows + r) & 31) && r < mr && n0 + f < N) {
            float v = acc[f][r] + (bias ? bias[n0 + f] : 0.f);
            if (silu_out) v = silu_f(v);
            y[static_cast<size_t>(m0 + r) * N + n0 + f] = v;
          }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// fp32 -> bf16 cast, optional nearest 2x upsample (Upsample, openaimodel.py:120 F.interpolate nearest)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cast_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y,
                                                        size_t n4) {
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(x) + i);
    uint2 pk;
    pk.x = pack_bf16x2(v.x, v.y);
    pk.y = pack_bf16x2(v.z, v.w);
    reinterpret_cast<uint2*>(y)[i] = pk;
  }
}

__global__ void __launch_bounds__(256) upsample2x_cast_kernel(const float* __restrict__ x,
                                                              __nv_bfloat16* __restrict__ y, int B, int H, int W,
                                                              int C) {
  const int cq = C >> 2;
  const size_t total = static_cast<size_t>(B) * H * W * cq;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int c4 = static_cast<int>(i % cq);
    const size_t pix = i / cq;
    const int w = static_cast<int>(pix % W);
    const int h = static_cast<int>((pix / W) % H);
    const int b = static_cast<int>(pix / (static_cast<size_t>(W) * H));
    const float4 v = __ldg(reinterpret_cast<const float4*>(x) + i);
    uint2 pk;
    pk.x = pack_bf16x2(v.x, v.y);
    pk.y = pack_bf16x2(v.z, v.w);
    const size_t W2 = 2 * static_cast<size_t>(W);
    const size_t base = ((static_cast<size_t>(b) * 2 * H + 2 * h) * W2 + 2 * w) * cq + c4;
    uint2* yo = reinterpret_cast<uint2*>(y);
    yo[base] = pk;
    yo[base + cq] = pk;
    yo[base + W2 * cq] = pk;
    yo[base + W2 * cq + cq] = pk;
  }
}

// ---------------------------------------------------------------------------------------------
// CFG combine + DDIM update (ldm/models/diffusion/ddim.py:260,279,283,295), same fp32 operation order as
// the reference so that given identical eps the update is bit-exact:
//   e      = e_u + g * (e_c - e_u)
//   pred   = (x - sqrt(1-a_t) * e) / sqrt(a_t)
//   dir    = sqrt(1 - a_prev - sigma^2) * e
//   x_prev = sqrt(a_prev) * pred + dir + sigma * noise * temperature
// coef row: [g, sqrt_one_minus_at, sqrt_at, sqrt_a_prev, dir_coef, sigma*temperature, 0, 0]
// eps holds the conditional half first, then the unconditional half (ddim.py:238-243); n = elements per half.
// ---------------------------------------------------------------------------------------------
// x and x_prev may alias (the graph path updates the latent in place): no __restrict__ on them
__global__ void __launch_bounds__(256) cfg_ddim_kernel(const float* x, const float* __restrict__ eps,
                                                       int has_uncond, const float* __restrict__ noise,
                                                       const float* __restrict__ coef_table,
                                                       const int* __restrict__ step_idx, float* x_prev,
                                                       float* __restrict__ pred_x0, size_t n) {
  const float* cf = coef_table + (step_idx ? static_cast<size_t>(*step_idx) * 8 : 0);
  const float g = cf[0], s1m = cf[1], sat = cf[2], sap = cf[3], dcoef = cf[4], sig = cf[5], temp = cf[6];
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    float e = eps[i];
    if (has_uncond) {
      const float eu = eps[n + i];
      e = __fadd_rn(eu, __fmul_rn(g, __fsub_rn(e, eu)));
    }
    const float pred = __fdiv_rn(__fsub_rn(x[i], __fmul_rn(s1m, e)), sat);
    const float dir = __fmul_rn(dcoef, e);
    float xp = __fadd_rn(__fmul_rn(sap, pred), dir);
    const float nz = noise ? __fmul_rn(__fmul_rn(sig, noise[i]), temp) : 0.f;   // (sigma * noise) * temperature, ddim.py:286
    xp = __fadd_rn(xp, nz);
    x_prev[i] = xp;
    if (pred_x0) pred_x0[i] = pred;
  }
}

// bump the device-side step counter and publish the next timestep to t_buf[0..B)
__global__ void advance_step_kernel(int* step_idx, const float* __restrict__ t_table, float* __restrict__ t_buf, int B,
                                    int num_steps) {
  __shared__ int s_next;
  if (threadIdx.x == 0) {
    int nx = *step_idx + 1;
    s_next = nx;
  }
  __syncthreads();
  const int nx = s_next;
  if (nx < num_steps)
    for (int i = threadIdx.x; i < B; i += blockDim.x) t_buf[i] = t_table[nx];
  __syncthreads();
  if (threadIdx.x == 0) *step_idx = nx;
}

}  // namespace af

using namespace af;

static inline int grid_for(size_t work_items, int threads) {
  size_t g = (work_items + threads - 1) / threads;
  const size_t cap = static_cast<size_t>(num_sms()) * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

template <int CIN>
static int launch_conv_in(const float* x_nchw, const float* w, const float* bias, float* y_nhwc, int B, int H, int W,
                          int Cout, cudaStream_t stream) {
  const int cq = Cout / 4;
  int groups = 320 / cq;                       // pixel groups per block; must divide 32 with >= 8 pixels each
  if (groups > 4) groups = 4;
  if (groups == 3) groups = 2;
  if (groups < 1) groups = 1;
  const int threads = ((groups * cq + 31) / 32) * 32;
  const size_t smem = (static_cast<size_t>(9 * CIN) * Cout + CIN * 3 * 34) * sizeof(float);
  static size_t configured = 0;
  if (smem > configured) {
    AF_CUDA(cudaFuncSetAttribute(conv_in_kernel<CIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    configured = smem;
  }
  // rows per block: as many as keep >= 2 blocks per SM in flight
  const int col_blocks = (W + 31) / 32;
  int rows = static_cast<int>((static_cast<long long>(col_blocks) * H * B) / (2ll * num_sms()));
  if (rows < 1) rows = 1;
  if (rows > 16) rows = 16;
  dim3 grid(col_blocks, (H + rows - 1) / rows, B);
  conv_in_kernel<CIN><<<grid, threads, smem, stream>>>(x_nchw, w, bias, y_nhwc, B, H, W, Cout, rows);
  AF_LAUNCH_CHECK("conv_in_kernel");
  return 0;
}

// Cin 4: the UNet's and the VAE decoder's conv_in on latents; Cin 3: the VAE encoder's conv_in on RGB images
// (model.py:436-440).
extern "C" int af_conv_in(const float* x_nchw, const float* w, const float* bias, float* y_nhwc, int B, int Cin, int H,
                          int W, int Cout, cudaStream_t stream) {
  AF_CHECK_ARG(x_nchw && w && y_nhwc, "af_conv_in: null pointer");
  AF_CHECK_ARG(Cin == 3 || Cin == 4, "af_conv_in: Cin=%d unsupported (3 or 4)", Cin);
  AF_CHECK_ARG(Cout % 4 == 0 && Cout >= 32 && Cout <= 1280, "af_conv_in: Cout=%d unsupported", Cout);
  if (Cin == 3) return launch_conv_in<3>(x_nchw, w, bias, y_nhwc, B, H, W, Cout, stream);
  return launch_conv_in<4>(x_nchw, w, bias, y_nhwc, B, H, W, Cout, stream);
}

extern "C" int af_conv_out(const void* x_nhwc_bf16, const float* w_packed, const float* bias, float* y_nchw, int B,
                           int H, int W, int C, int Cout, cudaStream_t stream) {
  AF_CHECK_ARG(x_nhwc_bf16 && w_packed && y_nchw, "af_conv_out: null pointer");
  AF_CHECK_ARG(Cout == 4 && C % 8 == 0, "af_conv_out: Cout=%d C=%d unsupported", Cout, C);
  const size_t smem = static_cast<size_t>(Cout) * 9 * C * sizeof(float);
  AF_CHECK_ARG(smem <= 200 * 1024, "af_conv_out: C=%d too large", C);
  static size_t configured = 0;
  if (smem > configured) {
    AF_CUDA(cudaFuncSetAttribute(conv_out_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    configured = smem;
  }
  const long long total = static_cast<long long>(B) * H * W;
  long long blocks = (total + 7) / 8;
  const long long cap = static_cast<long long>(num_sms()) * 4;
  if (blocks > cap) blocks = cap;
  conv_out_kernel<4><<<static_cast<unsigned>(blocks), 256, smem, stream>>>(
      static_cast<const __nv_bfloat16*>(x_nhwc_bf16), w_packed, bias, y_nchw, B, H, W, C);
  AF_LAUNCH_CHECK("conv_out_kernel");
  return 0;
}

extern "C" int af_nhwc_to_nchw(const float* x_nhwc, float* y_nchw, int B, int HW, int Cp, int Cout, cudaStream_t stream) {
  AF_CHECK_ARG(x_nhwc && y_nchw && B > 0 && HW > 0, "af_nhwc_to_nchw: bad args");
  AF_CHECK_ARG(Cp % 4 == 0 && Cout >= 1 && Cout <= 4 && Cout <= Cp, "af_nhwc_to_nchw: Cp=%d Cout=%d unsupported", Cp, Cout);
  nhwc_to_nchw_kernel<<<grid_for(static_cast<size_t>(B) * HW, 256), 256, 0, stream>>>(x_nhwc, y_nchw, B, HW, Cp, Cout);
  AF_LAUNCH_CHECK("nhwc_to_nchw_kernel");
  return 0;
}

extern "C" int af_timestep_embedding(const float* t, float* out, int B, int dim, cudaStream_t stream) {
  AF_CHECK_ARG(t && out && B > 0 && dim >= 2, "af_timestep_embedding: bad args");
  const int n = B * (dim / 2);
  timestep_embedding_kernel<<<(n + 255) / 256, 256, 0, stream>>>(t, out, B, dim);
  AF_LAUNCH_CHECK("timestep_embedding_kernel");
  return 0;
}

extern "C" int af_linear_small(const float* x, const float* w, const float* bias, float* y, int M, int N, int K,
                               int silu_in, int silu_out, cudaStream_t stream) {
  AF_CHECK_ARG(x && w && y, "af_linear_small: null pointer");
  AF_CHECK_ARG(M > 0 && N > 0 && K > 0 && K % 4 == 0, "af_linear_small: M=%d N=%d K=%d (K%%4)", M, N, K);
  const size_t smem = static_cast<size_t>(kLsRows) * K * sizeof(float);
  AF_CHECK_ARG(smem <= 200 * 1024, "af_linear_small: K=%d too large", K);
  static size_t configured = 0;
  if (smem > configured) {
    AF_CUDA(cudaFuncSetAttribute(linear_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    configured = smem;
  }
  linear_small_kernel<<<(N + 8 * kLsFeat - 1) / (8 * kLsFeat), 256, smem, stream>>>(x, w, bias, y, M, N, K, silu_in, silu_out);
  AF_LAUNCH_CHECK("linear_small_kernel");
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Row softmax of materialised attention scores (VAE AttnBlock, ldm/modules/diffusionmodules/model.py:188-193:
// w_ = softmax(q.k * c^-1/2, dim=2)): fp32 scores [rows][n] -> bf16 probabilities [rows][ldo], one CTA per row,
// the row lives in registers (n <= 256 threads x 16 x 4 = 16384), exp2 domain.
// ---------------------------------------------------------------------------------------------
namespace af {
template <int ITER>
__global__ void __launch_bounds__(256) softmax_rows_kernel(const float* __restrict__ x, long long ldx, int n,
                                                           float scale_log2e, __nv_bfloat16* __restrict__ y,
                                                           long long ldo) {
  __shared__ float red[8];
  __shared__ float bc;
  const float4* xr = reinterpret_cast<const float4*>(x + static_cast<size_t>(blockIdx.x) * ldx);
  const int nv = n >> 2;
  float4 v[ITER];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < ITER; ++i) {
    const int k = threadIdx.x + i * 256;
    if (k < nv) {
      v[i] = __ldg(xr + k);
      mx = fmaxf(mx, fmaxf(fmaxf(v[i].x, v[i].y), fmaxf(v[i].z, v[i].w)));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = red[0];
    for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
    bc = m;
  }
  __syncthreads();
  const float m = bc * scale_log2e;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < ITER; ++i) {
    const int k = threadIdx.x + i * 256;
    if (k < nv) {
      v[i].x = fast_exp2(fmaf(v[i].x, scale_log2e, -m));
      v[i].y = fast_exp2(fmaf(v[i].y, scale_log2e, -m));
      v[i].z = fast_exp2(fmaf(v[i].z, scale_log2e, -m));
      v[i].w = fast_exp2(fmaf(v[i].w, scale_log2e, -m));
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  }
  s = warp_sum(s);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    bc = 1.0f / t;
  }
  __syncthreads();
  const float inv = bc;
  uint2* yr = reinterpret_cast<uint2*>(y + static_cast<size_t>(blockIdx.x) * ldo);
#pragma unroll
  for (int i = 0; i < ITER; ++i) {
    const int k = threadIdx.x + i * 256;
    if (k < nv) {
      uint2 pk;
      pk.x = pack_bf16x2(v[i].x * inv, v[i].y * inv);
      pk.y = pack_bf16x2(v[i].z * inv, v[i].w * inv);
      yr[k] = pk;
    }
  }
}
}  // namespace af

extern "C" int af_softmax_rows(const float* x, long long ldx, long long rows, int n, float scale, void* y_bf16,
                               long long ldo, cudaStream_t stream) {
  AF_CHECK_ARG(x && y_bf16 && rows > 0 && rows < (1ll << 31), "af_softmax_rows: bad args");
  AF_CHECK_ARG(n > 0 && n % 4 == 0 && n <= 16384 && ldx % 4 == 0 && ldo % 4 == 0 && ldx >= n && ldo >= n,
               "af_softmax_rows: n=%d ldx=%lld ldo=%lld (n%%4, n<=16384)", n, ldx, ldo);
  if (n <= 4096)
    softmax_rows_kernel<4><<<static_cast<unsigned>(rows), 256, 0, stream>>>(x, ldx, n, scale * 1.4426950408889634f,
                                                                           static_cast<__nv_bfloat16*>(y_bf16), ldo);
  else
    softmax_rows_kernel<16><<<static_cast<unsigned>(rows), 256, 0, stream>>>(x, ldx, n, scale * 1.4426950408889634f,
                                                                            static_cast<__nv_bfloat16*>(y_bf16), ldo);
  AF_LAUNCH_CHECK("softmax_rows_kernel");
  return 0;
}

// 1x1 convolution over at most 4 channels of an NCHW fp32 tensor, with an input scale: the VAE's post_quant_conv applied
// to z / scale_factor (ldm/models/autoencoder.py:331, ldm/models/diffusion/ddpm.py:1267).
namespace af {
__global__ void __launch_bounds__(256) channel_mix4_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                           const float* __restrict__ bias, float in_scale, int Cin,
                                                           int Cout, long long HW, long long total,
                                                           float* __restrict__ y) {
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * 256) {
    const long long b = i / HW, pix = i - b * HW;
    float v[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) v[c] = c < Cin ? x[(b * Cin + c) * HW + pix] * in_scale : 0.f;
    for (int o = 0; o < Cout; ++o) {
      float acc = bias ? bias[o] : 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c < Cin) acc = fmaf(w[o * Cin + c], v[c], acc);
      y[(b * Cout + o) * HW + pix] = acc;
    }
  }
}
}  // namespace af

extern "C" int af_channel_mix4(const float* x_nchw, const float* w, const float* bias, float in_scale, int B, int Cin,
                               int Cout, long long HW, float* y_nchw, cudaStream_t stream) {
  AF_CHECK_ARG(x_nchw && w && y_nchw && B > 0 && HW > 0, "af_channel_mix4: bad args");
  AF_CHECK_ARG(Cin >= 1 && Cin <= 4 && Cout >= 1 && Cout <= 4, "af_channel_mix4: Cin=%d Cout=%d (1..4)", Cin, Cout);
  const long long total = static_cast<long long>(B) * HW;
  channel_mix4_kernel<<<grid_for(static_cast<size_t>(total), 256), 256, 0, stream>>>(x_nchw, w, bias, in_scale, Cin, Cout,
                                                                                     HW, total, y_nchw);
  AF_LAUNCH_CHECK("channel_mix4_kernel");
  return 0;
}

// DiagonalGaussianDistribution (ldm/modules/distributions/distributions.py:24-44) over the encoder's moments, fused with
// get_first_stage_encoding's scale_factor * z (ddpm.py).  Same fp32 operations in the same order as the reference's torch
// ops: clamp, 0.5 * lv, exp (expf, not the MUFU approximation), std * noise, mean + that, scale * that; no contraction.
namespace af {
__global__ void __launch_bounds__(256) vae_posterior_kernel(const float* __restrict__ moments, long long HW, int zc,
                                                            long long total, const float* __restrict__ noise,
                                                            float out_scale, float* __restrict__ z,
                                                            float* __restrict__ mean_out, float* __restrict__ logvar_out) {
  for (long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * 256) {
    const long long pix = i % HW, bc = i / HW;                 // output index i = (b * zc + c) * HW + pix
    const int c = static_cast<int>(bc % zc);
    const long long b = bc / zc;
    const float* m = moments + (b * HW + pix) * (2 * zc);
    const float mean = m[c];
    float lv = m[zc + c];
    if (!isnan(lv)) lv = fminf(fmaxf(lv, -30.0f), 20.0f);    // torch.clamp(logvar, -30.0, 20.0)
    float v = mean;
    if (noise) {
      const float stdv = expf(__fmul_rn(0.5f, lv));           // torch.exp(0.5 * self.logvar)
      v = __fadd_rn(mean, __fmul_rn(stdv, noise[i]));         // self.mean + self.std * noise
    }
    z[i] = __fmul_rn(out_scale, v);
    if (mean_out) mean_out[i] = mean;
    if (logvar_out) logvar_out[i] = lv;
  }
}
}  // namespace af

extern "C" int af_vae_posterior(const float* moments_nhwc, int B, long long HW, int zc, const float* noise_nchw,
                                float out_scale, float* z_nchw, float* mean_nchw, float* logvar_nchw, cudaStream_t stream) {
  AF_CHECK_ARG(moments_nhwc && z_nchw, "af_vae_posterior: null pointer");
  AF_CHECK_ARG(B > 0 && HW > 0 && zc > 0, "af_vae_posterior: bad sizes B=%d HW=%lld zc=%d", B, HW, zc);
  const long long total = static_cast<long long>(B) * zc * HW;
  vae_posterior_kernel<<<grid_for(static_cast<size_t>(total), 256), 256, 0, stream>>>(
      moments_nhwc, HW, zc, total, noise_nchw, out_scale, z_nchw, mean_nchw, logvar_nchw);
  AF_LAUNCH_CHECK("vae_posterior_kernel");
  return 0;
}

extern "C" int af_cast_bf16(const float* x, void* y_bf16, long long n, cudaStream_t stream) {
  AF_CHECK_ARG(x && y_bf16 && n > 0 && n % 4 == 0, "af_cast_bf16: bad args (n%%4)");
  const size_t n4 = static_cast<size_t>(n) / 4;
  cast_bf16_kernel<<<grid_for(n4, 256), 256, 0, stream>>>(x, static_cast<__nv_bfloat16*>(y_bf16), n4);
  AF_LAUNCH_CHECK("cast_bf16_kernel");
  return 0;
}

extern "C" int af_upsample2x_cast(const float* x_nhwc, void* y_bf16, int B, int H, int W, int C, cudaStream_t stream) {
  AF_CHECK_ARG(x_nhwc && y_bf16 && C % 4 == 0, "af_upsample2x_cast: bad args");
  const size_t total = static_cast<size_t>(B) * H * W * (C / 4);
  upsample2x_cast_kernel<<<grid_for(total, 256), 256, 0, stream>>>(x_nhwc, static_cast<__nv_bfloat16*>(y_bf16), B, H, W, C);
  AF_LAUNCH_CHECK("upsample2x_cast_kernel");
  return 0;
}

extern "C" int af_cfg_ddim_update(const float* x, const float* eps, int has_uncond, const float* noise,
                                  const float* coef_table, const int* step_idx, float* x_prev, float* pred_x0,
                                  long long n, cudaStream_t stream) {
  AF_CHECK_ARG(x && eps && coef_table && x_prev && n > 0, "af_cfg_ddim_update: bad args");
  cfg_ddim_kernel<<<grid_for(static_cast<size_t>(n), 256), 256, 0, stream>>>(x, eps, has_uncond, noise, coef_table,
                                                                              step_idx, x_prev, pred_x0,
                                                                              static_cast<size_t>(n));
  AF_LAUNCH_CHECK("cfg_ddim_kernel");
  return 0;
}

extern "C" int af_advance_step(int* step_idx, const float* t_table, float* t_buf, int B, int num_steps,
                               cudaStream_t stream) {
  AF_CHECK_ARG(step_idx && t_table && t_buf && B > 0, "af_advance_step: bad args");
  advance_step_kernel<<<1, 128, 0, stream>>>(step_idx, t_table, t_buf, B, num_steps);
  AF_LAUNCH_CHECK("advance_step_kernel");
  return 0;
}
