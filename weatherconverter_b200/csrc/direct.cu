// Small CUDA-core kernels around the tensor-core path: boundary layout conversion fused with the 3-channel
// convolutions (conv_in 3->64 reads the reference's NCHW fp32 image; conv_out 64->3 writes NCHW fp32), the
// time-embedding MLP, weight packing, and NCHW<->NHWC converters.
// Reference ops: unet_base.py:7-30 (get_time_embedding), :395-397 (t_proj), :96-98 (t_emb_layers), :399 (conv_in),
// :449 (conv_out); resnet.py:142-145 (conv1+bn1+relu).
#include <algorithm>

#include "wc_host.h"
#include "wc_ptx.cuh"

namespace wc {

namespace {

// ---------------------------------------------------------------------------------------------------------
// conv (Cin small, e.g. 3) from NCHW fp32 to NHWC bf16, KxK, stride s, pad p, optional per-channel affine
// (folded BatchNorm) and ReLU.  Block = 32 pixels x (Cout/8) channel octets.
template <int CIN>
__global__ void conv_small_cin_kernel(const float* __restrict__ x, const float* __restrict__ w /*[Cout][CIN][K][K]*/,
                                      const float* __restrict__ bias, const float* __restrict__ scale,
                                      const float* __restrict__ shift, __nv_bfloat16* __restrict__ y, int B, int H,
                                      int W, int Ho, int Wo, int Cout, int K, int stride, int pad, int ldy, int relu,
                                      const float* __restrict__ prelu) {
  pdl_prologue();
  extern __shared__ float sw[];  // [CIN*K*K][Cout]
  const int taps = CIN * K * K;
  for (int i = threadIdx.x; i < taps * Cout; i += blockDim.x) {
    const int n = i % Cout, t = i / Cout;
    sw[i] = w[static_cast<size_t>(n) * taps + t];
  }
  __syncthreads();
  const int octs = Cout / 8;
  const int oct = threadIdx.x % octs, pl = threadIdx.x / octs;
  const int ppb = blockDim.x / octs;
  const size_t npix = static_cast<size_t>(B) * Ho * Wo;
  for (size_t pix = static_cast<size_t>(blockIdx.x) * ppb + pl; pix < npix; pix += static_cast<size_t>(gridDim.x) * ppb) {
    const int ox = static_cast<int>(pix % Wo), oy = static_cast<int>((pix / Wo) % Ho), b = static_cast<int>(pix / (static_cast<size_t>(Wo) * Ho));
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = bias ? bias[oct * 8 + j] : 0.f;
    for (int c = 0; c < CIN; ++c) {
      const float* xp = x + (static_cast<size_t>(b) * CIN + c) * H * W;
      for (int ky = 0; ky < K; ++ky) {
        const int iy = oy * stride - pad + ky;
        if (iy < 0 || iy >= H) continue;
        for (int kx = 0; kx < K; ++kx) {
          const int ix = ox * stride - pad + kx;
          if (ix < 0 || ix >= W) continue;
          const float v = __ldg(xp + static_cast<size_t>(iy) * W + ix);
          const float* wp = sw + ((c * K + ky) * K + kx) * Cout + oct * 8;
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] = fmaf(v, wp[j], acc[j]);
        }
      }
    }
    if (scale) {
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaf(acc[j], scale[oct * 8 + j], shift[oct * 8 + j]);
    }
    if (relu) {
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaxf(acc[j], 0.f);
    }
    if (prelu) {
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = acc[j] > 0.f ? acc[j] : acc[j] * prelu[oct * 8 + j];
    }
    uint4 u;
    u.x = pack_bf16(acc[0], acc[1]); u.y = pack_bf16(acc[2], acc[3]);
    u.z = pack_bf16(acc[4], acc[5]); u.w = pack_bf16(acc[6], acc[7]);
    *reinterpret_cast<uint4*>(y + pix * ldy + oct * 8) = u;
  }
}

// ---------------------------------------------------------------------------------------------------------
// Same convolution specialised for Cout = 64: one thread per output pixel computes all 64 channels; weights live
// in shared memory as [tap][64] and are read as broadcast 16-byte vectors; the MACs are packed FFMA2.
template <int CIN>
__global__ void __launch_bounds__(128)
conv_stem64_kernel(const float* __restrict__ x, const float* __restrict__ w /*[64][CIN][K][K]*/,
                   const float* __restrict__ bias, const float* __restrict__ scale, const float* __restrict__ shift,
                   __nv_bfloat16* __restrict__ y, int B, int H, int W, int Ho, int Wo, int K, int stride, int pad, int ldy,
                   int relu, const float* __restrict__ prelu) {
  pdl_prologue();
  extern __shared__ float sw[];  // [CIN*K*K][64]
  const int taps = CIN * K * K;
  for (int i = threadIdx.x; i < taps * 64; i += blockDim.x) {
    const int n = i & 63, t = i >> 6;
    sw[i] = w[static_cast<size_t>(n) * taps + t];
  }
  __syncthreads();
  const size_t npix = static_cast<size_t>(B) * Ho * Wo;
  for (size_t pix = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; pix < npix;
       pix += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int ox = static_cast<int>(pix % Wo), oy = static_cast<int>((pix / Wo) % Ho), b = static_cast<int>(pix / (static_cast<size_t>(Wo) * Ho));
    float2 acc[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) acc[j] = bias ? make_float2(bias[2 * j], bias[2 * j + 1]) : make_float2(0.f, 0.f);
    for (int c = 0; c < CIN; ++c) {
      const float* xp = x + (static_cast<size_t>(b) * CIN + c) * H * W;
      for (int ky = 0; ky < K; ++ky) {
        const int iy = oy * stride - pad + ky;
        const bool rowok = iy >= 0 && iy < H;
        for (int kx = 0; kx < K; ++kx) {
          const int ix = ox * stride - pad + kx;
          float v = 0.f;
          if (rowok && ix >= 0 && ix < W) v = __ldg(xp + static_cast<size_t>(iy) * W + ix);
          const float2 vv = make_float2(v, v);
          const float4* wp = reinterpret_cast<const float4*>(sw + ((c * K + ky) * K + kx) * 64);
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float4 w4 = wp[j];
            acc[2 * j] = ffma2(vv, make_float2(w4.x, w4.y), acc[2 * j]);
            acc[2 * j + 1] = ffma2(vv, make_float2(w4.z, w4.w), acc[2 * j + 1]);
          }
        }
      }
    }
    uint4* op = reinterpret_cast<uint4*>(y + pix * ldy);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      float f[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) { f[2 * j] = acc[4 * q + j].x; f[2 * j + 1] = acc[4 * q + j].y; }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int n = 8 * q + j;
        if (scale) f[j] = fmaf(f[j], scale[n], shift[n]);
        if (relu) f[j] = fmaxf(f[j], 0.f);
        if (prelu) f[j] = f[j] > 0.f ? f[j] : f[j] * prelu[n];
      }
      uint4 u;
      u.x = pack_bf16(f[0], f[1]); u.y = pack_bf16(f[2], f[3]); u.z = pack_bf16(f[4], f[5]); u.w = pack_bf16(f[6], f[7]);
      op[q] = u;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// conv KxK (stride 1, pad K/2) from NHWC bf16 (Cin % 8 == 0) to NCHW fp32 with COUT (<=4) outputs; one thread
// per output pixel; optional tanh epilogue y = (tanh(v)+1)/2 (SRGAN, models.py:92).
template <int COUT>
__global__ void conv_small_cout_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w /*[COUT][Cin][K][K]*/,
                                       const float* __restrict__ bias, float* __restrict__ y, int B, int H, int W,
                                       int Cin, int K, int ldx, int tanh_out) {
  pdl_prologue();
  extern __shared__ float sw[];  // [K*K][Cin][COUT]
  const int kk = K * K;
  for (int i = threadIdx.x; i < kk * Cin * COUT; i += blockDim.x) {
    const int n = i % COUT, c = (i / COUT) % Cin, t = i / (COUT * Cin);
    sw[i] = w[(static_cast<size_t>(n) * Cin + c) * kk + t];
  }
  __syncthreads();
  const size_t npix = static_cast<size_t>(B) * H * W;
  const int pad = K / 2;
  for (size_t pix = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; pix < npix;
       pix += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int ox = static_cast<int>(pix % W), oy = static_cast<int>((pix / W) % H), b = static_cast<int>(pix / (static_cast<size_t>(W) * H));
    float acc[COUT];
#pragma unroll
    for (int n = 0; n < COUT; ++n) acc[n] = bias ? bias[n] : 0.f;
    for (int ky = 0; ky < K; ++ky) {
      const int iy = oy - pad + ky;
      if (iy < 0 || iy >= H) continue;
      for (int kx = 0; kx < K; ++kx) {
        const int ix = ox - pad + kx;
        if (ix < 0 || ix >= W) continue;
        const uint4* xp = reinterpret_cast<const uint4*>(x + ((static_cast<size_t>(b) * H + iy) * W + ix) * ldx);
        const float* wp = sw + static_cast<size_t>(ky * K + kx) * Cin * COUT;
        for (int c8 = 0; c8 < Cin / 8; ++c8) {
          const uint4 u = __ldg(xp + c8);
          float f[8];
          float2 t;
          t = unpack_bf16(u.x); f[0] = t.x; f[1] = t.y;
          t = unpack_bf16(u.y); f[2] = t.x; f[3] = t.y;
          t = unpack_bf16(u.z); f[4] = t.x; f[5] = t.y;
          t = unpack_bf16(u.w); f[6] = t.x; f[7] = t.y;
#pragma unroll
          for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int n = 0; n < COUT; ++n) acc[n] = fmaf(f[j], wp[(c8 * 8 + j) * COUT + n], acc[n]);
        }
      }
    }
    const size_t plane = static_cast<size_t>(H) * W;
#pragma unroll
    for (int n = 0; n < COUT; ++n) {
      float v = acc[n];
      if (tanh_out) v = (tanhf(v) + 1.f) * 0.5f;
      y[(static_cast<size_t>(b) * COUT + n) * plane + static_cast<size_t>(oy) * W + ox] = v;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Time embedding: emb = [sin(t/f_j), cos(t/f_j)], f_j = 10000^(j/half); h = W2 silu(W1 emb + b1) + b2;
// writes silu(h) (every consumer applies SiLU first, unet_base.py:97) and h itself.
// `factor` (optional, [dim/2]): the reference's 10000**(arange/half) table as torch evaluates it on the host
// (unet_base.py:22-24), so that t/factor is bit-identical to the reference's argument; NULL -> powf on the device.
__global__ void time_embedding_kernel(const long long* __restrict__ t, int dim, const float* __restrict__ factor,
                                      float* __restrict__ out) {
  pdl_prologue();
  const int b = blockIdx.x, half = dim / 2;
  const float tv = static_cast<float>(t[b]);
  for (int j = threadIdx.x; j < half; j += blockDim.x) {
    const float a = tv / time_factor(factor, j, half);
    out[static_cast<size_t>(b) * dim + j] = sinf(a);
    out[static_cast<size_t>(b) * dim + j + half] = cosf(a);
  }
}

__global__ void temb_mlp_kernel(const long long* __restrict__ t, int dim, const float* __restrict__ factor,
                                const float* __restrict__ w1,
                                const float* __restrict__ b1, const float* __restrict__ w2,
                                const float* __restrict__ b2, float* __restrict__ temb, float* __restrict__ temb_silu) {
  pdl_prologue();
  extern __shared__ float sh[];  // emb[dim], h1[dim]
  float* emb = sh;
  float* h1 = sh + dim;
  const int b = blockIdx.x, half = dim / 2;
  const float tv = static_cast<float>(t[b]);
  for (int j = threadIdx.x; j < half; j += blockDim.x) {
    const float a = tv / time_factor(factor, j, half);
    emb[j] = sinf(a);
    emb[j + half] = cosf(a);
  }
  __syncthreads();
  for (int n = threadIdx.x; n < dim; n += blockDim.x) {
    float acc = b1[n];
    for (int k = 0; k < dim; ++k) acc = fmaf(w1[static_cast<size_t>(n) * dim + k], emb[k], acc);
    h1[n] = acc / (1.f + expf(-acc));
  }
  __syncthreads();
  for (int n = threadIdx.x; n < dim; n += blockDim.x) {
    float acc = b2[n];
    for (int k = 0; k < dim; ++k) acc = fmaf(w2[static_cast<size_t>(n) * dim + k], h1[k], acc);
    temb[static_cast<size_t>(b) * dim + n] = acc;
    temb_silu[static_cast<size_t>(b) * dim + n] = acc / (1.f + expf(-acc));
  }
}

// out[b][n] = bias[n] + sum_k W[n][k] * in[b][k]; one warp per output, all t_emb_layers of the net in one launch.
__global__ void linear_rows_kernel(const float* __restrict__ in, int dim, const float* __restrict__ w,
                                   const float* __restrict__ bias, float* __restrict__ out, int N) {
  pdl_prologue();
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  if (warp >= N) return;
  float acc = 0.f;
  for (int k = lane; k < dim; k += 32) acc = fmaf(w[static_cast<size_t>(warp) * dim + k], in[static_cast<size_t>(b) * dim + k], acc);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) out[static_cast<size_t>(b) * N + warp] = acc + bias[warp];
}

// ---------------------------------------------------------------------------------------------------------
// Weight packing: dst[n][koff + c] (bf16, row pitch ldk) = scale[.] * src[...][ky][kx] for n < Nn, c < Cc,
// zero for c in [Cc, Cpad).  transpose = 0: src is [Nn][Cc][KH][KW] (Conv2d); 1: src is [Cc][Nn][KH][KW]
// (ConvTranspose2d weight, or a dgrad view of a Conv2d weight).  scale (optional) is indexed by the src dim-0.
__global__ void pack_tap_kernel(__nv_bfloat16* __restrict__ dst, int ldk, int koff, const float* __restrict__ src,
                                int Nn, int Cc, int Cpad, int KH, int KW, int ky, int kx, int transpose,
                                const float* __restrict__ scale, int D0, int D1src) {
  pdl_prologue();
  const size_t total = static_cast<size_t>(Nn) * Cpad;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % Cpad), n = static_cast<int>(i / Cpad);
    float v = 0.f;
    if (c < Cc) {
      const size_t d0 = transpose ? c : n, d1 = transpose ? n : c;
      const size_t D1 = D1src;
      v = src[((d0 * D1 + d1) * KH + ky) * KW + kx];
      if (scale) v *= scale[d0];
    }
    dst[static_cast<size_t>(n) * ldk + koff + c] = __float2bfloat16_rn(v);
  }
}

// All taps of one plan in one launch (blockIdx.y = tap): the per-step re-packing of the training plans.
struct PackTapDesc {
  const float* src;
  const float* scale;
  int koff, Nn, Cc, Cpad, KH, KW, ky, kx, transpose, D1;
};
constexpr int kPackMaxTaps = 20;
struct PackTapsArgs {
  __nv_bfloat16* dst;
  int ldk, ntaps;
  PackTapDesc t[kPackMaxTaps];
};
__global__ void pack_taps_kernel(const __grid_constant__ PackTapsArgs a) {
  pdl_prologue();
  const PackTapDesc t = a.t[blockIdx.y];
  const size_t total = static_cast<size_t>(t.Nn) * t.Cpad;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % t.Cpad), n = static_cast<int>(i / t.Cpad);
    float v = 0.f;
    if (c < t.Cc) {
      const size_t d0 = t.transpose ? c : n, d1 = t.transpose ? n : c;
      v = t.src[((d0 * t.D1 + d1) * t.KH + t.ky) * t.KW + t.kx];
      if (t.scale) v *= t.scale[d0];
    }
    a.dst[static_cast<size_t>(n) * a.ldk + t.koff + c] = __float2bfloat16_rn(v);
  }
}

__global__ void nchw_f32_to_nhwc_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int B, int C,
                                             int HW, int ldy) {
  pdl_prologue();
  const size_t total = static_cast<size_t>(B) * HW * C;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    const size_t p = (i / C) % HW, b = i / (static_cast<size_t>(C) * HW);
    y[(b * HW + p) * ldy + c] = __float2bfloat16_rn(x[(b * C + c) * HW + p]);
  }
}
__global__ void nhwc_bf16_to_nchw_f32_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ y, int B, int C,
                                             int HW, int ldx) {
  pdl_prologue();
  const size_t total = static_cast<size_t>(B) * HW * C;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t p = i % HW;
    const int c = static_cast<int>((i / HW) % C);
    const size_t b = i / (static_cast<size_t>(C) * HW);
    y[i] = __bfloat162float(x[(b * HW + p) * ldx + c]);
  }
}

inline int grid_for(size_t n_items, int per_block = 256) {
  const size_t blocks = (n_items + per_block - 1) / per_block;
  const size_t cap = static_cast<size_t>(num_sms()) * 8;
  return static_cast<int>(blocks < cap ? (blocks ? blocks : 1) : cap);
}

}  // namespace

int conv_small_cin(const float* x, const float* w, const float* bias, const float* scale, const float* shift,
                   __nv_bfloat16* y, int B, int Cin, int H, int W, int Cout, int K, int stride, int pad, int ldy,
                   int relu, cudaStream_t st, const float* prelu) {
  WC_REQUIRE(Cin == 3, "conv_small_cin supports Cin == 3");
  WC_REQUIRE(Cout % 8 == 0 && Cout <= 256, "Cout must be a multiple of 8, <= 256");
  const int Ho = (H + 2 * pad - K) / stride + 1, Wo = (W + 2 * pad - K) / stride + 1;
  const int octs = Cout / 8, threads = (256 / octs) * octs;
  const size_t smem = static_cast<size_t>(Cin) * K * K * Cout * sizeof(float);
  if (smem > 48 * 1024)
    WC_CHECK_CUDA(cudaFuncSetAttribute(conv_small_cin_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
  const size_t npix = static_cast<size_t>(B) * Ho * Wo;
  ProfScope prof(kProfBoundaryConv, st, static_cast<double>(B) * (12.0 * H * W + 2.0 * Ho * Wo * Cout));
  if (Cout == 64) {
    static size_t attr_set = 0;
    if (smem > 48 * 1024 && smem > attr_set) {
      WC_CHECK_CUDA(cudaFuncSetAttribute(conv_stem64_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
      attr_set = smem;
    }
    launch_k(conv_stem64_kernel<3>, grid_for(npix, 128), 128, smem, st, x, w, bias, scale, shift, y, B, H, W, Ho, Wo, K, stride, pad,
                                                                 ldy, relu, prelu);
    WC_LAUNCH_CHECK();
    return 0;
  }
  launch_k(conv_small_cin_kernel<3>, grid_for(npix, threads / octs), threads, smem, st, 
      x, w, bias, scale, shift, y, B, H, W, Ho, Wo, Cout, K, stride, pad, ldy, relu, prelu);
  WC_LAUNCH_CHECK();
  return 0;
}

int conv_small_cout(const __nv_bfloat16* x, const float* w, const float* bias, float* y, int B, int H, int W, int Cin,
                    int Cout, int K, int ldx, int tanh_out, cudaStream_t st) {
  WC_REQUIRE(Cout == 3, "conv_small_cout supports Cout == 3");
  WC_REQUIRE(Cin % 8 == 0, "Cin must be a multiple of 8");
  const size_t smem = static_cast<size_t>(K) * K * Cin * Cout * sizeof(float);
  if (smem > 48 * 1024)
    WC_CHECK_CUDA(cudaFuncSetAttribute(conv_small_cout_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem)));
  const size_t npix = static_cast<size_t>(B) * H * W;
  ProfScope prof(kProfBoundaryConv, st, static_cast<double>(npix) * (2.0 * Cin + 4.0 * Cout));
  launch_k(conv_small_cout_kernel<3>, grid_for(npix, 128), 128, smem, st, x, w, bias, y, B, H, W, Cin, K, ldx, tanh_out);
  WC_LAUNCH_CHECK();
  return 0;
}

// ---- ResNet stem on the tensor core (conv.cu: build_conv_stem7s2): input re-layout and weight re-layout
__global__ void stem_prepare_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ xp, int B, int H, int W) {
  pdl_prologue();
  const int Wp = W + 8;
  const size_t total = static_cast<size_t>(B) * H * Wp;
  const size_t plane = static_cast<size_t>(H) * W;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int xq = static_cast<int>(i % Wp) - 4;
    const size_t by = i / Wp;
    const int y = static_cast<int>(by % H);
    const size_t b = by / H;
    uint4 u = make_uint4(0u, 0u, 0u, 0u);
    if (xq >= 0 && xq < W) {
      const float* src = x + (b * 3) * plane + static_cast<size_t>(y) * W + xq;
      u.x = pack_bf16(__ldg(src), __ldg(src + plane));
      u.y = pack_bf16(__ldg(src + 2 * plane), 0.f);
    }
    *reinterpret_cast<uint4*>(xp + i * 8) = u;
  }
}
__global__ void stem_weights_kernel(const float* __restrict__ w, float* __restrict__ wp, int N) {
  pdl_prologue();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;   // over [N][64][7]
  if (i >= N * 64 * 7) return;
  const int ky = i % 7, e = (i / 7) % 64, n = i / (7 * 64);
  const int kx = e / 8, c = e % 8;
  wp[i] = (kx < 7 && c < 3) ? w[((n * 3 + c) * 7 + ky) * 7 + kx] : 0.f;
}
int stem_prepare(const float* x_nchw, __nv_bfloat16* xp, int B, int H, int W, cudaStream_t st) {
  const size_t total = static_cast<size_t>(B) * H * (W + 8);
  ProfScope prof(kProfBoundaryConv, st, static_cast<double>(B) * H * (12.0 * W + 16.0 * (W + 8)));
  launch_k(stem_prepare_kernel, grid_for(total), 256, 0, st, x_nchw, xp, B, H, W);
  WC_LAUNCH_CHECK();
  return 0;
}
int stem_weights(const float* w, float* wprime, int N, cudaStream_t st) {
  launch_k(stem_weights_kernel, (N * 64 * 7 + 255) / 256, 256, 0, st, w, wprime, N);
  WC_LAUNCH_CHECK();
  return 0;
}

int temb_mlp(const long long* t, int Bt, int dim, const float* w1, const float* b1, const float* w2, const float* b2,
             float* temb, float* temb_silu, cudaStream_t st) {
  launch_k(temb_mlp_kernel, Bt, 128, 2 * dim * sizeof(float), st, t, dim, time_factor_table(dim / 2), w1, b1, w2, b2, temb, temb_silu);
  WC_LAUNCH_CHECK();
  return 0;
}

// get_time_embedding (unet_base.py:7-30): out [n, dim] = [sin(t/f), cos(t/f)]
int time_embedding(const long long* t, int n, int dim, float* out, cudaStream_t st) {
  WC_REQUIRE(n >= 1 && dim >= 2 && dim % 2 == 0, "time_embedding: dim must be even");
  launch_k(time_embedding_kernel, n, 64, 0, st, t, dim, time_factor_table(dim / 2), out);
  WC_LAUNCH_CHECK();
  return 0;
}

int linear_rows(const float* in, int Bt, int dim, const float* w, const float* bias, float* out, int N,
                cudaStream_t st) {
  const int warps_per_block = 8;
  launch_k(linear_rows_kernel, dim3((N + warps_per_block - 1) / warps_per_block, Bt), warps_per_block * 32, 0, st, 
      in, dim, w, bias, out, N);
  WC_LAUNCH_CHECK();
  return 0;
}

int pack_tap(__nv_bfloat16* dst, int ldk, int koff, const float* src, int Nn, int Cc, int Cpad, int KH, int KW, int ky,
             int kx, int transpose, const float* scale, cudaStream_t st) {
  // source dim-1 extent: transposed sources are [Cc][Nn], plain sources [rows][Cc]
  launch_k(pack_tap_kernel, grid_for(static_cast<size_t>(Nn) * Cpad), 256, 0, st, dst, ldk, koff, src, Nn, Cc, Cpad, KH, KW,
                                                                           ky, kx, transpose, scale, 0,
                                                                           transpose ? Nn : Cc);
  WC_LAUNCH_CHECK();
  return 0;
}

// One launch for up to 20 taps; taps[i] = {src, scale, koff, Nn, Cc, Cpad, KH, KW, ky, kx, transpose}
int pack_taps(__nv_bfloat16* dst, int ldk, int ntaps, const float* const* src, const float* const* scale, const int* params /*[ntaps][9]*/,
              cudaStream_t st) {
  WC_REQUIRE(ntaps >= 1 && ntaps <= kPackMaxTaps, "pack_taps: tap count out of range");
  PackTapsArgs a;
  a.dst = dst; a.ldk = ldk; a.ntaps = ntaps;
  size_t max_total = 0;
  for (int i = 0; i < ntaps; ++i) {
    const int* p = params + i * 9;
    PackTapDesc& t = a.t[i];
    t.src = src[i]; t.scale = scale[i];
    t.koff = p[0]; t.Nn = p[1]; t.Cc = p[2]; t.Cpad = p[3]; t.KH = p[4]; t.KW = p[5]; t.ky = p[6]; t.kx = p[7];
    t.transpose = p[8];
    t.D1 = t.transpose ? t.Nn : t.Cc;
    max_total = std::max(max_total, static_cast<size_t>(t.Nn) * t.Cpad);
  }
  const int gx = static_cast<int>(std::min<size_t>((max_total + 255) / 256, 256));
  launch_k(pack_taps_kernel, dim3(gx, ntaps), 256, 0, st, a);
  WC_LAUNCH_CHECK();
  return 0;
}

int nchw_f32_to_nhwc_bf16(const float* x, __nv_bfloat16* y, int B, int C, int HW, int ldy, cudaStream_t st) {
  launch_k(nchw_f32_to_nhwc_bf16_kernel, grid_for(static_cast<size_t>(B) * C * HW), 256, 0, st, x, y, B, C, HW, ldy);
  WC_LAUNCH_CHECK();
  return 0;
}
int nhwc_bf16_to_nchw_f32(const __nv_bfloat16* x, float* y, int B, int C, int HW, int ldx, cudaStream_t st) {
  launch_k(nhwc_bf16_to_nchw_f32_kernel, grid_for(static_cast<size_t>(B) * C * HW), 256, 0, st, x, y, B, C, HW, ldx);
  WC_LAUNCH_CHECK();
  return 0;
}

}  // namespace wc
