// Bandwidth-bound kernels of the DeepLabV3+ forward / input-gradient path and of the SRGAN generator
// (NHWC bf16 activations).  Reference ops:
//   resnet.py:145 MaxPool2d(3,2,1) (+ its backward), _deeplab.py:125-131 AdaptiveAvgPool2d(1) + bilinear broadcast,
//   _deeplab.py:50 / network/utils.py:17 F.interpolate(bilinear, align_corners=False) (+ adjoints),
//   seg_model/inference.py:124-141 argmax + CrossEntropyLoss(ignore_index=255) + backward,
//   srgan_model/models.py:5-21 depthwise convolutions.
#include <cuda_fp16.h>
#include <cstdlib>
#include "wc_host.h"
#include "wc_ptx.cuh"

namespace wc {

namespace {

inline int grid_for(size_t n_items, int per_block = 256) {
  const size_t blocks = (n_items + per_block - 1) / per_block;
  const size_t cap = static_cast<size_t>(num_sms()) * 16;
  return static_cast<int>(blocks < cap ? (blocks ? blocks : 1) : cap);
}

// scale = gamma / sqrt(var + eps), shift = beta - mean * scale  (eval-mode BatchNorm folded into the conv)
__global__ void bn_fold_kernel(const float* g, const float* b, const float* mean, const float* var, float eps,
                               float* scale, float* shift, int n, int n_pad) {
  pdl_prologue();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pad) return;
  if (i < n) {
    const float s = g[i] / sqrtf(var[i] + eps);
    scale[i] = s;
    shift[i] = b[i] - mean[i] * s;
  } else {
    scale[i] = 0.f;
    shift[i] = 0.f;
  }
}

// ---- MaxPool 3x3 s2 p1, NHWC bf16, 8 channels per thread; stores the argmax tap (0..8) per element.
__global__ void maxpool_fwd_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y,
                                   uint8_t* __restrict__ idx, int B, int H, int W, int C, int Ho, int Wo) {
  pdl_prologue();
  const int c8n = C / 8;
  const size_t total = static_cast<size_t>(B) * Ho * Wo * c8n;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % c8n);
    size_t p = i / c8n;
    const int ox = static_cast<int>(p % Wo), oy = static_cast<int>((p / Wo) % Ho), b = static_cast<int>(p / (static_cast<size_t>(Wo) * Ho));
    float best[8];
    int bi[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { best[j] = -INFINITY; bi[j] = 0; }
    for (int ky = 0; ky < 3; ++ky) {
      const int iy = oy * 2 - 1 + ky;
      if (iy < 0 || iy >= H) continue;
      for (int kx = 0; kx < 3; ++kx) {
        const int ix = ox * 2 - 1 + kx;
        if (ix < 0 || ix >= W) continue;
        const uint4 u = __ldg(reinterpret_cast<const uint4*>(x + ((static_cast<size_t>(b) * H + iy) * W + ix) * C + c8 * 8));
        float f[8];
        float2 t;
        t = unpack_bf16(u.x); f[0] = t.x; f[1] = t.y;
        t = unpack_bf16(u.y); f[2] = t.x; f[3] = t.y;
        t = unpack_bf16(u.z); f[4] = t.x; f[5] = t.y;
        t = unpack_bf16(u.w); f[6] = t.x; f[7] = t.y;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (f[j] > best[j]) { best[j] = f[j]; bi[j] = ky * 3 + kx; }  // first maximum wins (PyTorch order)
      }
    }
    uint4 o;
    o.x = pack_bf16(best[0], best[1]); o.y = pack_bf16(best[2], best[3]);
    o.z = pack_bf16(best[4], best[5]); o.w = pack_bf16(best[6], best[7]);
    *reinterpret_cast<uint4*>(y + p * C + c8 * 8) = o;
    uint2 ii;
    ii.x = bi[0] | (bi[1] << 8) | (bi[2] << 16) | (bi[3] << 24);
    ii.y = bi[4] | (bi[5] << 8) | (bi[6] << 16) | (bi[7] << 24);
    *reinterpret_cast<uint2*>(idx + p * C + c8 * 8) = ii;
  }
}

// dX[b,iy,ix,c] = sum over the (<= 4) pooling windows containing (iy,ix) whose argmax is this pixel; then the
// ReLU mask of the pre-pool activation (x > 0) is applied (conv1+bn1+relu precede the pool, resnet.py:142-145).
// 8 channels (16 bytes) per thread.
__global__ void maxpool_bwd_kernel(const __nv_bfloat16* __restrict__ dy, const uint8_t* __restrict__ idx,
                                   const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ dx, int B, int H,
                                   int W, int C, int Ho, int Wo) {
  pdl_prologue();
  const int c8n = C / 8;
  const size_t total = static_cast<size_t>(B) * H * W * c8n;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % c8n);
    size_t p = i / c8n;
    const int ix = static_cast<int>(p % W), iy = static_cast<int>((p / W) % H), b = static_cast<int>(p / (static_cast<size_t>(W) * H));
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int oy = iy / 2; oy <= (iy + 1) / 2; ++oy) {   // windows with 2*oy-1 <= iy <= 2*oy+1
      if (oy >= Ho) continue;
      const int ky = iy - (2 * oy - 1);
      for (int ox = ix / 2; ox <= (ix + 1) / 2; ++ox) {
        if (ox >= Wo) continue;
        const int kx = ix - (2 * ox - 1);
        const uint32_t tap = static_cast<uint32_t>(ky * 3 + kx);
        const size_t q = ((static_cast<size_t>(b) * Ho + oy) * Wo + ox) * C + c8 * 8;
        const uint2 ii = __ldg(reinterpret_cast<const uint2*>(idx + q));
        const uint4 g = __ldg(reinterpret_cast<const uint4*>(dy + q));
        const uint32_t* gp = &g.x;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t t = ((j < 4 ? ii.x : ii.y) >> (8 * (j & 3))) & 0xffu;
          const float2 f = unpack_bf16(gp[j >> 1]);
          if (t == tap) acc[j] += (j & 1) ? f.y : f.x;
        }
      }
    }
    const uint4 xv = __ldg(reinterpret_cast<const uint4*>(x + p * C + c8 * 8));
    const uint32_t* xp = &xv.x;
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = unpack_bf16(xp[j]);
      o[j] = pack_bf16(f.x > 0.f ? acc[2 * j] : 0.f, f.y > 0.f ? acc[2 * j + 1] : 0.f);
    }
    *reinterpret_cast<uint4*>(dx + p * C + c8 * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// ---- global average pool: x [B,HW,C] (ld) -> y [B,C]; one block per (b, 64-channel slab)
__global__ void gap_fwd_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, int HW, int C, int ld) {
  pdl_prologue();
  __shared__ float red[4][64];
  const int b = blockIdx.y, c = blockIdx.x * 64 + (threadIdx.x & 63), part = threadIdx.x >> 6;
  float acc = 0.f;
  if (c < C)
    for (int p = part; p < HW; p += 4) acc += __bfloat162float(x[(static_cast<size_t>(b) * HW + p) * ld + c]);
  red[part][threadIdx.x & 63] = acc;
  __syncthreads();
  if (part == 0 && c < C)
    y[static_cast<size_t>(b) * C + c] = __float2bfloat16_rn((red[0][threadIdx.x] + red[1][threadIdx.x] + red[2][threadIdx.x] + red[3][threadIdx.x]) / HW);
}
// y[b,p,c] (ldy) = v[b,c]  (bilinear up-sampling of a 1x1 map = broadcast, _deeplab.py:131)
__global__ void broadcast_kernel(const __nv_bfloat16* __restrict__ v, __nv_bfloat16* __restrict__ y, int B, int HW, int C, int ldy) {
  pdl_prologue();
  const int c8n = C / 8;
  const size_t total = static_cast<size_t>(B) * HW * c8n;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % c8n);
    const size_t p = i / c8n, b = p / HW;
    *reinterpret_cast<uint4*>(y + p * ldy + c8 * 8) = __ldg(reinterpret_cast<const uint4*>(v + b * C + c8 * 8));
  }
}
// adjoint of broadcast: v[b,c] = sum_p y[b,p,c], optionally masked by (m[b,c] > 0) (ReLU of the pooled branch)
__global__ void sum_hw_kernel(const __nv_bfloat16* __restrict__ y, const __nv_bfloat16* __restrict__ m,
                              __nv_bfloat16* __restrict__ v, int HW, int C, int ldy) {
  pdl_prologue();
  __shared__ float red[4][64];
  const int b = blockIdx.y, c = blockIdx.x * 64 + (threadIdx.x & 63), part = threadIdx.x >> 6;
  float acc = 0.f;
  if (c < C)
    for (int p = part; p < HW; p += 4) acc += __bfloat162float(y[(static_cast<size_t>(b) * HW + p) * ldy + c]);
  red[part][threadIdx.x & 63] = acc;
  __syncthreads();
  if (part == 0 && c < C) {
    float s = red[0][threadIdx.x] + red[1][threadIdx.x] + red[2][threadIdx.x] + red[3][threadIdx.x];
    if (m && !(__bfloat162float(m[static_cast<size_t>(b) * C + c]) > 0.f)) s = 0.f;
    v[static_cast<size_t>(b) * C + c] = __float2bfloat16_rn(s);
  }
}
// adjoint of the global average pool, accumulated into dx: dx[b,p,c] += g[b,c] / HW
__global__ void gap_bwd_add_kernel(const __nv_bfloat16* __restrict__ g, __nv_bfloat16* __restrict__ dx, int B, int HW, int C, int ld) {
  pdl_prologue();
  const size_t total = static_cast<size_t>(B) * HW * C;
  const float inv = 1.f / HW;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    const size_t p = i / C, b = p / HW;
    __nv_bfloat16* d = dx + p * ld + c;
    *d = __float2bfloat16_rn(__bfloat162float(*d) + __bfloat162float(g[b * C + c]) * inv);
  }
}

// ---- bilinear resize, align_corners=False (PyTorch area_pixel_compute_source_index semantics)
__device__ __forceinline__ void bilinear_src(int dst, float scale, int in_size, int& i0, int& i1, float& l1) {
  float src = (dst + 0.5f) * scale - 0.5f;
  if (src < 0.f) src = 0.f;
  i0 = static_cast<int>(src);
  if (i0 > in_size - 1) i0 = in_size - 1;
  i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
  l1 = src - i0;
}

// NHWC bf16 -> NHWC bf16 (channel slice views allowed), 8 channels per thread
__global__ void bilinear_fwd_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, int B, int Hi,
                                    int Wi, int Ho, int Wo, int C, int ldx, int ldy) {
  pdl_prologue();
  const int c8n = C / 8;
  const size_t total = static_cast<size_t>(B) * Ho * Wo * c8n;
  const float sy = static_cast<float>(Hi) / Ho, sx = static_cast<float>(Wi) / Wo;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % c8n);
    size_t p = i / c8n;
    const int ox = static_cast<int>(p % Wo), oy = static_cast<int>((p / Wo) % Ho), b = static_cast<int>(p / (static_cast<size_t>(Wo) * Ho));
    int y0, y1, x0, x1;
    float ly, lx;
    bilinear_src(oy, sy, Hi, y0, y1, ly);
    bilinear_src(ox, sx, Wi, x0, x1, lx);
    const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
    const __nv_bfloat16* xb = x + static_cast<size_t>(b) * Hi * Wi * ldx + c8 * 8;
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(xb + (static_cast<size_t>(y0) * Wi + x0) * ldx));
    const uint4 bq = __ldg(reinterpret_cast<const uint4*>(xb + (static_cast<size_t>(y0) * Wi + x1) * ldx));
    const uint4 c = __ldg(reinterpret_cast<const uint4*>(xb + (static_cast<size_t>(y1) * Wi + x0) * ldx));
    const uint4 d = __ldg(reinterpret_cast<const uint4*>(xb + (static_cast<size_t>(y1) * Wi + x1) * ldx));
    const uint32_t* pa = &a.x; const uint32_t* pb = &bq.x; const uint32_t* pc = &c.x; const uint32_t* pd = &d.x;
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 fa = unpack_bf16(pa[j]), fb = unpack_bf16(pb[j]), fc = unpack_bf16(pc[j]), fd = unpack_bf16(pd[j]);
      o[j] = pack_bf16(w00 * fa.x + w01 * fb.x + w10 * fc.x + w11 * fd.x, w00 * fa.y + w01 * fb.y + w10 * fc.y + w11 * fd.y);
    }
    *reinterpret_cast<uint4*>(y + p * ldy + c8 * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// Adjoint (gather form): dx[b,iy,ix,c] = sum over output pixels whose 2x2 stencil touches (iy,ix).  For an integer
// up-sampling factor f every input pixel is touched by outputs within [f*i - f, f*i + 2f) per axis.
// Optional ReLU mask (m > 0).  Source may be a channel slice (ldy); fp32 accumulation.
__global__ void bilinear_bwd_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ m,
                                    __nv_bfloat16* __restrict__ dx, int B, int Hi, int Wi, int Ho, int Wo, int C,
                                    int ldy, int ldm, int ldx) {
  pdl_prologue();
  const int c8n = C / 8;
  const size_t total = static_cast<size_t>(B) * Hi * Wi * c8n;
  const float sy = static_cast<float>(Hi) / Ho, sx = static_cast<float>(Wi) / Wo;
  const int fy = (Ho + Hi - 1) / Hi, fx = (Wo + Wi - 1) / Wi;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int c8 = static_cast<int>(i % c8n);
    size_t p = i / c8n;
    const int ix = static_cast<int>(p % Wi), iy = static_cast<int>((p / Wi) % Hi), b = static_cast<int>(p / (static_cast<size_t>(Wi) * Hi));
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    const int oy_lo = max(0, fy * iy - fy - 1), oy_hi = min(Ho - 1, fy * iy + 2 * fy);
    const int ox_lo = max(0, fx * ix - fx - 1), ox_hi = min(Wo - 1, fx * ix + 2 * fx);
    for (int oy = oy_lo; oy <= oy_hi; ++oy) {
      int y0, y1; float ly;
      bilinear_src(oy, sy, Hi, y0, y1, ly);
      float wy = 0.f;
      if (y0 == iy) wy += 1.f - ly;
      if (y1 == iy) wy += ly;
      if (wy == 0.f) continue;
      for (int ox = ox_lo; ox <= ox_hi; ++ox) {
        int x0, x1; float lx;
        bilinear_src(ox, sx, Wi, x0, x1, lx);
        float wx = 0.f;
        if (x0 == ix) wx += 1.f - lx;
        if (x1 == ix) wx += lx;
        if (wx == 0.f) continue;
        const float ww = wy * wx;
        const uint4 u = __ldg(reinterpret_cast<const uint4*>(dy + ((static_cast<size_t>(b) * Ho + oy) * Wo + ox) * ldy + c8 * 8));
        const uint32_t* up = &u.x;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = unpack_bf16(up[j]);
          acc[2 * j] = fmaf(ww, f.x, acc[2 * j]);
          acc[2 * j + 1] = fmaf(ww, f.y, acc[2 * j + 1]);
        }
      }
    }
    if (m) {
      const uint4 mv = __ldg(reinterpret_cast<const uint4*>(m + p * ldm + c8 * 8));
      const uint32_t* mp = &mv.x;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = unpack_bf16(mp[j]);
        if (!(f.x > 0.f)) acc[2 * j] = 0.f;
        if (!(f.y > 0.f)) acc[2 * j + 1] = 0.f;
      }
    }
    uint4 o;
    o.x = pack_bf16(acc[0], acc[1]); o.y = pack_bf16(acc[2], acc[3]); o.z = pack_bf16(acc[4], acc[5]); o.w = pack_bf16(acc[6], acc[7]);
    *reinterpret_cast<uint4*>(dx + p * ldx + c8 * 8) = o;
  }
}

// ---- segmentation loss head (seg_model/inference.py:124-141 + network/utils.py:17)
// n_valid[b] = #pixels with label != ignore
__global__ void count_valid_kernel(const long long* __restrict__ labels, int HW, int ignore, int* __restrict__ n_valid) {
  pdl_prologue();
  const int b = blockIdx.y;
  int cnt = 0;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < HW; p += gridDim.x * blockDim.x)
    cnt += labels[static_cast<size_t>(b) * HW + p] != ignore;
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(n_valid + b, cnt);
}

// One thread per full-resolution pixel: bilinear logits (from low-res NCHW fp32 planes), argmax -> pred,
// softmax-CE: dlogit = (softmax - onehot) / n_valid[b] (0 where ignored) written as fp32 class planes [B,NC,H,W];
// per-image loss accumulated with one atomic per warp.  labels == NULL (then pred, dlogit_hi and loss are NULL too): only the
// up-sampled logits are written.
template <int NC>
__global__ void seg_loss_grad_kernel(const float* __restrict__ logits_lo, const long long* __restrict__ labels,
                                     const int* __restrict__ n_valid, long long* __restrict__ pred,
                                     float* __restrict__ dlogit_hi, float* __restrict__ loss, float* __restrict__ logits_hi,
                                     int B, int h, int w, int H, int W, int ignore) {
  pdl_prologue();
  const size_t total = static_cast<size_t>(B) * H * W;
  const float sy = static_cast<float>(h) / H, sx = static_cast<float>(w) / W;
  // warp-uniform trip count (the loss reduction below uses full-warp shuffles)
  const size_t lane = threadIdx.x & 31;
  for (size_t wb = (blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x) - lane; wb < total;
       wb += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t i = wb + lane;
    float lsum = 0.f;
    int b = 0;
    if (i < total) {
      const int ox = static_cast<int>(i % W), oy = static_cast<int>((i / W) % H);
      b = static_cast<int>(i / (static_cast<size_t>(W) * H));
      int y0, y1, x0, x1;
      float ly, lx;
      bilinear_src(oy, sy, h, y0, y1, ly);
      bilinear_src(ox, sx, w, x0, x1, lx);
      const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
      const size_t plane = static_cast<size_t>(h) * w;
      const float* lb = logits_lo + static_cast<size_t>(b) * NC * plane;
      float v[NC];
      float mx = -INFINITY;
      int am = 0;
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        const float* pl = lb + c * plane;
        v[c] = w00 * pl[y0 * w + x0] + w01 * pl[y0 * w + x1] + w10 * pl[y1 * w + x0] + w11 * pl[y1 * w + x1];
        if (v[c] > mx) { mx = v[c]; am = c; }
      }
      if (pred) pred[i] = am;
      if (logits_hi) {
        const size_t pl_hi = static_cast<size_t>(H) * W;
#pragma unroll
        for (int c = 0; c < NC; ++c) logits_hi[(static_cast<size_t>(b) * NC + c) * pl_hi + static_cast<size_t>(oy) * W + ox] = v[c];
      }
      if (!labels) continue;   // uniform across the grid: loss is NULL too, so no warp reduction is skipped
      const long long lab = labels[i];
      const size_t pl_hi2 = static_cast<size_t>(H) * W;
      float* d = dlogit_hi + static_cast<size_t>(b) * NC * pl_hi2 + static_cast<size_t>(oy) * W + ox;   // class planes
      if (lab == ignore) {
#pragma unroll
        for (int c = 0; c < NC; ++c) d[c * pl_hi2] = 0.f;
      } else {
        float s = 0.f;
#pragma unroll
        for (int c = 0; c < NC; ++c) { v[c] = __expf(v[c] - mx); s += v[c]; }
        const float inv = 1.f / s, invn = 1.f / static_cast<float>(n_valid[b]);
#pragma unroll
        for (int c = 0; c < NC; ++c) d[c * pl_hi2] = (v[c] * inv - (c == lab ? 1.f : 0.f)) * invn;
        lsum = -__logf(v[lab < NC && lab >= 0 ? lab : 0] * inv) * invn;
      }
    }
    // warp-level loss reduction (warps never straddle images when H*W % 32 == 0; otherwise per-lane atomics)
    if (loss) {
      const int b0 = __shfl_sync(0xffffffffu, b, 0);
      if (__all_sync(0xffffffffu, b == b0)) {
        float t = lsum;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if ((threadIdx.x & 31) == 0 && t != 0.f) atomicAdd(loss + b0, t);
      } else if (lsum != 0.f) {
        atomicAdd(loss + b, lsum);
      }
    }
  }
}

// Adjoint of the final bilinear up-sampling for the NC logit channels: dlo[b,y,x,c] (NHWC bf16, ld = ldo, channels
// >= NC zero-filled up to CP) = sum_hi w * dhi[b,Y,X,c].
template <int NC>
__global__ void logits_bilinear_bwd_kernel(const float* __restrict__ dhi, __nv_bfloat16* __restrict__ dlo, int B, int h,
                                           int w, int H, int W, int CP, int ldo) {
  pdl_prologue();
  const size_t total = static_cast<size_t>(B) * h * w;
  const float sy = static_cast<float>(h) / H, sx = static_cast<float>(w) / W;
  const int fy = (H + h - 1) / h, fx = (W + w - 1) / w;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int ix = static_cast<int>(i % w), iy = static_cast<int>((i / w) % h), b = static_cast<int>(i / (static_cast<size_t>(w) * h));
    float acc[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) acc[c] = 0.f;
    const int oy_lo = max(0, fy * iy - fy - 1), oy_hi = min(H - 1, fy * iy + 2 * fy);
    const int ox_lo = max(0, fx * ix - fx - 1), ox_hi = min(W - 1, fx * ix + 2 * fx);
    for (int oy = oy_lo; oy <= oy_hi; ++oy) {
      int y0, y1; float ly;
      bilinear_src(oy, sy, h, y0, y1, ly);
      float wy = 0.f;
      if (y0 == iy) wy += 1.f - ly;
      if (y1 == iy) wy += ly;
      if (wy == 0.f) continue;
      for (int ox = ox_lo; ox <= ox_hi; ++ox) {
        int x0, x1; float lx;
        bilinear_src(ox, sx, w, x0, x1, lx);
        float wx = 0.f;
        if (x0 == ix) wx += 1.f - lx;
        if (x1 == ix) wx += lx;
        if (wx == 0.f) continue;
        const float ww = wy * wx;
        const size_t plane = static_cast<size_t>(H) * W;
        const float* d = dhi + static_cast<size_t>(b) * NC * plane + static_cast<size_t>(oy) * W + ox;
#pragma unroll
        for (int c = 0; c < NC; ++c) acc[c] += ww * __ldg(d + c * plane);
      }
    }
    __nv_bfloat16* o = dlo + i * ldo;
    for (int c = 0; c < CP; ++c) o[c] = __float2bfloat16_rn(c < NC ? acc[c] : 0.f);
  }
}

// Fused loss head (round 2): seg_loss_grad_kernel + logits_bilinear_bwd_kernel without the full-resolution fp32 d-logit tensor
// (19 planes x H x W x 4 B = 319 MB per 32 images at 256x512, written once and read once).  One block owns a tile of kLhTY x kLhTX
// LOW-resolution pixels: phase A evaluates softmax-CE for every full-resolution pixel whose bilinear footprint touches the tile
// (the up-sampled logits are recomputed from the low-res planes; pixels in the halo are evaluated by up to four blocks) and keeps
// d loss / d logit_hi in shared memory; the pixels the block OWNS also give pred and the loss.  Phase B applies the adjoint of the
// bilinear up-sampling from shared memory.  Needs integer up-sampling factors (H = fy h, W = fx w); otherwise the two-pass path runs.
constexpr int kLhTY = 4, kLhTX = 8, kLhThreads = 256;
template <int NC>
__global__ void __launch_bounds__(kLhThreads)
seg_loss_head_fused_kernel(const float* __restrict__ logits_lo, const long long* __restrict__ labels, const int* __restrict__ n_valid,
                           long long* __restrict__ pred, float* __restrict__ loss, __nv_bfloat16* __restrict__ dlo, int h, int w,
                           int H, int W, int fy, int fx, int RWmax, int CP, int ldo, int ignore) {
  pdl_prologue();
  extern __shared__ float lh_s[];   // [region pixel][NC]
  __shared__ float lh_loss[kLhThreads / 32];
  const int b = blockIdx.z, ty0 = blockIdx.y * kLhTY, tx0 = blockIdx.x * kLhTX;
  const float sy = static_cast<float>(h) / H, sx = static_cast<float>(w) / W;
  // full-resolution pixel o feeds low-resolution rows floor(src), floor(src) + 1 with src = (o + 0.5) / f - 0.5, i.e. row i is fed by
  // o in [f i - f/2 - 0.5, f i + 3f/2 - 0.5): the bounds below are that range rounded outwards
  const int ry0 = max(0, fy * ty0 - (fy + 1) / 2), ry1 = min(H - 1, fy * (ty0 + kLhTY - 1) + (3 * fy) / 2);
  const int rx0 = max(0, fx * tx0 - (fx + 1) / 2), rx1 = min(W - 1, fx * (tx0 + kLhTX - 1) + (3 * fx) / 2);
  const int RH = ry1 - ry0 + 1, RW = rx1 - rx0 + 1;
  (void)RWmax;
  const size_t plane = static_cast<size_t>(h) * w, plane_hi = static_cast<size_t>(H) * W;
  const float* lb = logits_lo + static_cast<size_t>(b) * NC * plane;
  const float invn = 1.f / static_cast<float>(max(n_valid[b], 1));
  float lsum = 0.f;
  // ---- phase A
  for (int idx = threadIdx.x; idx < RH * RW; idx += kLhThreads) {
    const int oy = ry0 + idx / RW, ox = rx0 + idx % RW;
    int y0, y1, x0, x1;
    float ly, lx;
    bilinear_src(oy, sy, h, y0, y1, ly);
    bilinear_src(ox, sx, w, x0, x1, lx);
    const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
    float v[NC];
    float mx = -INFINITY;
    int am = 0;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const float* pl = lb + c * plane;
      v[c] = w00 * __ldg(pl + y0 * w + x0) + w01 * __ldg(pl + y0 * w + x1) + w10 * __ldg(pl + y1 * w + x0) + w11 * __ldg(pl + y1 * w + x1);
      if (v[c] > mx) { mx = v[c]; am = c; }
    }
    const size_t hi = static_cast<size_t>(b) * plane_hi + static_cast<size_t>(oy) * W + ox;
    const long long lab = labels[hi];
    const bool owned = (oy / fy >= ty0) && (oy / fy < ty0 + kLhTY) && (ox / fx >= tx0) && (ox / fx < tx0 + kLhTX);
    if (owned && pred) pred[hi] = am;
    float* d = lh_s + static_cast<size_t>(idx) * NC;
    if (lab == ignore) {
#pragma unroll
      for (int c = 0; c < NC; ++c) d[c] = 0.f;
    } else {
      float s = 0.f;
#pragma unroll
      for (int c = 0; c < NC; ++c) { v[c] = __expf(v[c] - mx); s += v[c]; }
      const float inv = 1.f / s;
#pragma unroll
      for (int c = 0; c < NC; ++c) d[c] = (v[c] * inv - (c == lab ? 1.f : 0.f)) * invn;
      if (owned) lsum -= __logf(v[lab < NC && lab >= 0 ? lab : 0] * inv) * invn;
    }
  }
  if (loss) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
    if ((threadIdx.x & 31) == 0) lh_loss[threadIdx.x >> 5] = lsum;
  }
  __syncthreads();
  if (loss && threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < kLhThreads / 32; ++i) t += lh_loss[i];
    if (t != 0.f) atomicAdd(loss + b, t);
  }
  // ---- phase B: thread = (low-res pixel of the tile, class residue mod 8)
  const int p = threadIdx.x >> 3, k = threadIdx.x & 7;
  const int iy = ty0 + p / kLhTX, ix = tx0 + p % kLhTX;
  if (iy >= h || ix >= w) return;
  float acc[3] = {0.f, 0.f, 0.f};
  // the (at most 2f) rows / columns that feed this pixel and their weights, once per thread
  constexpr int kMaxTap = 16;
  float wys[kMaxTap], wxs[kMaxTap];
  int nyt = 0, nxt = 0, oy_first = 0, ox_first = 0;
  {
    const int lo = max(ry0, fy * iy - (fy + 1) / 2), hi = min(ry1, fy * iy + (3 * fy) / 2);
    oy_first = lo;
    for (int oy = lo; oy <= hi && nyt < kMaxTap; ++oy) {
      int y0, y1; float ly;
      bilinear_src(oy, sy, h, y0, y1, ly);
      float wy = 0.f;
      if (y0 == iy) wy += 1.f - ly;
      if (y1 == iy) wy += ly;
      wys[nyt++] = wy;
    }
  }
  {
    const int lo = max(rx0, fx * ix - (fx + 1) / 2), hi = min(rx1, fx * ix + (3 * fx) / 2);
    ox_first = lo;
    for (int ox = lo; ox <= hi && nxt < kMaxTap; ++ox) {
      int x0, x1; float lx;
      bilinear_src(ox, sx, w, x0, x1, lx);
      float wx = 0.f;
      if (x0 == ix) wx += 1.f - lx;
      if (x1 == ix) wx += lx;
      wxs[nxt++] = wx;
    }
  }
#pragma unroll 1
  for (int jy = 0; jy < nyt; ++jy) {
    const float wy = wys[jy];
    if (wy == 0.f) continue;
    const float* drow = lh_s + (static_cast<size_t>(oy_first + jy - ry0) * RW + (ox_first - rx0)) * NC + k;
#pragma unroll 4
    for (int jx = 0; jx < nxt; ++jx) {
      const float ww = wy * wxs[jx];
      const float* d = drow + jx * NC;
      acc[0] += ww * d[0];
      acc[1] += ww * d[8];
      if (k + 16 < NC) acc[2] += ww * d[16];
    }
  }
  __nv_bfloat16* o = dlo + ((static_cast<size_t>(b) * h + iy) * w + ix) * ldo;
  for (int c = k, j = 0; c < CP; c += 8, ++j) o[c] = __float2bfloat16_rn(c < NC ? acc[j] : 0.f);
}

// ---- data gradient of conv1 (7x7, stride 2, pad 3, 3 input channels) to the NCHW fp32 image:
// dX[b,c,y,x] = sum_{ky,kx: parity ok} sum_o dZ[b,(y+3-ky)/2,(x+3-kx)/2,o] * W[o,c,ky,kx] * scale[o]
// blockIdx.y = parity class (y&1, x&1): every thread of a block uses the same tap subset, so the weight reads are
// warp-uniform broadcasts ([tap][c][64] floats in shared memory, 16-byte vectors) and the MACs are packed FFMA2.
__global__ void __launch_bounds__(128)
conv1_dgrad_kernel(const __nv_bfloat16* __restrict__ dz, const float* __restrict__ w /*[64][3][7][7]*/,
                   const float* __restrict__ scale, float* __restrict__ dx, int B, int H, int W, int Ho, int Wo) {
  pdl_prologue();
  extern __shared__ float sw[];  // [49][3][64]
  for (int i = threadIdx.x; i < 49 * 3 * 64; i += blockDim.x) {
    const int o = i & 63, c = (i >> 6) % 3, t = i / 192;
    sw[i] = w[(static_cast<size_t>(o) * 3 + c) * 49 + t] * (scale ? scale[o] : 1.f);
  }
  __syncthreads();
  const int py = blockIdx.y >> 1, px = blockIdx.y & 1;
  const int Hh = H / 2, Wh = W / 2;
  const size_t total = static_cast<size_t>(B) * Hh * Wh;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int xh = static_cast<int>(i % Wh), yh = static_cast<int>((i / Wh) % Hh), b = static_cast<int>(i / (static_cast<size_t>(Wh) * Hh));
    const int x = 2 * xh + px, y = 2 * yh + py;
    float2 a0 = make_float2(0.f, 0.f), a1 = a0, a2 = a0;
    for (int ky = (py + 1) & 1; ky < 7; ky += 2) {
      const int ny = y + 3 - ky;
      const int oy = ny >> 1;
      if (ny < 0 || oy >= Ho) continue;
      for (int kx = (px + 1) & 1; kx < 7; kx += 2) {
        const int nx = x + 3 - kx;
        const int ox = nx >> 1;
        if (nx < 0 || ox >= Wo) continue;
        const uint4* zp = reinterpret_cast<const uint4*>(dz + ((static_cast<size_t>(b) * Ho + oy) * Wo + ox) * 64);
        const float4* wp = reinterpret_cast<const float4*>(sw + (ky * 7 + kx) * 192);
#pragma unroll
        for (int o8 = 0; o8 < 8; ++o8) {
          const uint4 u = __ldg(zp + o8);
          const float2 f0 = unpack_bf16(u.x), f1 = unpack_bf16(u.y), f2 = unpack_bf16(u.z), f3 = unpack_bf16(u.w);
          const float4 w0a = wp[o8 * 2], w0b = wp[o8 * 2 + 1];
          const float4 w1a = wp[16 + o8 * 2], w1b = wp[16 + o8 * 2 + 1];
          const float4 w2a = wp[32 + o8 * 2], w2b = wp[32 + o8 * 2 + 1];
          a0 = ffma2(f0, make_float2(w0a.x, w0a.y), a0); a0 = ffma2(f1, make_float2(w0a.z, w0a.w), a0);
          a0 = ffma2(f2, make_float2(w0b.x, w0b.y), a0); a0 = ffma2(f3, make_float2(w0b.z, w0b.w), a0);
          a1 = ffma2(f0, make_float2(w1a.x, w1a.y), a1); a1 = ffma2(f1, make_float2(w1a.z, w1a.w), a1);
          a1 = ffma2(f2, make_float2(w1b.x, w1b.y), a1); a1 = ffma2(f3, make_float2(w1b.z, w1b.w), a1);
          a2 = ffma2(f0, make_float2(w2a.x, w2a.y), a2); a2 = ffma2(f1, make_float2(w2a.z, w2a.w), a2);
          a2 = ffma2(f2, make_float2(w2b.x, w2b.y), a2); a2 = ffma2(f3, make_float2(w2b.z, w2b.w), a2);
        }
      }
    }
    const size_t plane = static_cast<size_t>(H) * W, o = static_cast<size_t>(b) * 3 * plane + static_cast<size_t>(y) * W + x;
    dx[o] = a0.x + a0.y; dx[o + plane] = a1.x + a1.y; dx[o + 2 * plane] = a2.x + a2.y;
  }
}

// ---- avg_pool2d(P) of the conv1 data gradient, fused (both are linear):
//   pooled[b,c,Y,X] = (1/P^2) sum_{j,i<P} dX[b,c,P*Y+j,P*X+i] = sum_{r,s} sum_o dZ[b,(P/2)*Y+r,(P/2)*X+s,o] * Weff[r,s,c,o]
//   Weff[r,s,c,o] = scale[o]/P^2 * sum_{j: 0<=j+3-2r<=6} sum_{i: 0<=i+3-2s<=6} W[o,c,j+3-2r,i+3-2s],  r,s in [-1, P/2+1]
// (position independent; dZ outside the map contributes nothing).  One thread per pooled pixel, weights in smem.
__global__ void conv1_dgrad_weff_kernel(const float* __restrict__ w, const float* __restrict__ scale, float* __restrict__ weff,
                                        int P) {
  pdl_prologue();
  const int R = P / 2 + 3;
  const int total = R * R * 3 * 64;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int o = idx & 63, c = (idx >> 6) % 3, rs = idx / 192, s_ = rs % R - 1, r_ = rs / R - 1;
    float acc = 0.f;
    for (int j = 0; j < P; ++j) {
      const int ky = j + 3 - 2 * r_;
      if (ky < 0 || ky > 6) continue;
      for (int i = 0; i < P; ++i) {
        const int kx = i + 3 - 2 * s_;
        if (kx < 0 || kx > 6) continue;
        acc += w[((static_cast<size_t>(o) * 3 + c) * 7 + ky) * 7 + kx];
      }
    }
    weff[idx] = acc * (scale ? scale[o] : 1.f) / static_cast<float>(P * P);
  }
}

__global__ void __launch_bounds__(128)
conv1_dgrad_pooled_kernel(const __nv_bfloat16* __restrict__ dz, const float* __restrict__ weff, float* __restrict__ out, int B,
                          int Ho, int Wo, int P) {
  pdl_prologue();
  extern __shared__ float sw[];  // [R*R][3][64]
  const int R = P / 2 + 3, half = P / 2;
  for (int i = threadIdx.x; i < R * R * 192; i += blockDim.x) sw[i] = weff[i];
  __syncthreads();
  const int Hp = Ho / half, Wp = Wo / half;
  const size_t total = static_cast<size_t>(B) * Hp * Wp;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int X = static_cast<int>(i % Wp), Y = static_cast<int>((i / Wp) % Hp), b = static_cast<int>(i / (static_cast<size_t>(Wp) * Hp));
    float2 a0 = make_float2(0.f, 0.f), a1 = a0, a2 = a0;
    for (int r = 0; r < R; ++r) {
      const int oy = half * Y + r - 1;
      if (oy < 0 || oy >= Ho) continue;
      for (int s_ = 0; s_ < R; ++s_) {
        const int ox = half * X + s_ - 1;
        if (ox < 0 || ox >= Wo) continue;
        const uint4* zp = reinterpret_cast<const uint4*>(dz + ((static_cast<size_t>(b) * Ho + oy) * Wo + ox) * 64);
        const float4* wp = reinterpret_cast<const float4*>(sw + (r * R + s_) * 192);
#pragma unroll
        for (int o8 = 0; o8 < 8; ++o8) {
          const uint4 u = __ldg(zp + o8);
          const float2 f0 = unpack_bf16(u.x), f1 = unpack_bf16(u.y), f2 = unpack_bf16(u.z), f3 = unpack_bf16(u.w);
          const float4 w0a = wp[o8 * 2], w0b = wp[o8 * 2 + 1];
          const float4 w1a = wp[16 + o8 * 2], w1b = wp[16 + o8 * 2 + 1];
          const float4 w2a = wp[32 + o8 * 2], w2b = wp[32 + o8 * 2 + 1];
          a0 = ffma2(f0, make_float2(w0a.x, w0a.y), a0); a0 = ffma2(f1, make_float2(w0a.z, w0a.w), a0);
          a0 = ffma2(f2, make_float2(w0b.x, w0b.y), a0); a0 = ffma2(f3, make_float2(w0b.z, w0b.w), a0);
          a1 = ffma2(f0, make_float2(w1a.x, w1a.y), a1); a1 = ffma2(f1, make_float2(w1a.z, w1a.w), a1);
          a1 = ffma2(f2, make_float2(w1b.x, w1b.y), a1); a1 = ffma2(f3, make_float2(w1b.z, w1b.w), a1);
          a2 = ffma2(f0, make_float2(w2a.x, w2a.y), a2); a2 = ffma2(f1, make_float2(w2a.z, w2a.w), a2);
          a2 = ffma2(f2, make_float2(w2b.x, w2b.y), a2); a2 = ffma2(f3, make_float2(w2b.z, w2b.w), a2);
        }
      }
    }
    const size_t plane = static_cast<size_t>(Hp) * Wp, o = static_cast<size_t>(b) * 3 * plane + static_cast<size_t>(Y) * Wp + X;
    out[o] = a0.x + a0.y; out[o + plane] = a1.x + a1.y; out[o + 2 * plane] = a2.x + a2.y;
  }
}

// d[p,c] = 0 where m[p,c] <= 0 (ReLU derivative applied to a gradient slice in place)
__global__ void relu_mask_kernel(__nv_bfloat16* __restrict__ d, const __nv_bfloat16* __restrict__ m, size_t npix, int C,
                                 int ldd, int ldm) {
  pdl_prologue();
  const size_t total = npix * C;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t p = i / C;
    const int c = static_cast<int>(i % C);
    if (!(__bfloat162float(m[p * ldm + c]) > 0.f)) d[p * ldd + c] = __float2bfloat16_rn(0.f);
  }
}

// ---- composed separable-conv weights (srgan_model/models.py:5-21): W[o,c,ky,kx] = pw[o,c] * dw[c,0,ky,kx];
// bias[o] = pw_bias[o] + sum_c pw[o,c] * dw_bias[c]
__global__ void compose_sep_kernel(const float* __restrict__ dw, const float* __restrict__ pw, const float* __restrict__ dwb,
                                   const float* __restrict__ pwb, float* __restrict__ w, float* __restrict__ bias, int Co,
                                   int Ci, int KK) {
  pdl_prologue();
  const size_t total = static_cast<size_t>(Co) * Ci * KK;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int t = static_cast<int>(i % KK), c = static_cast<int>((i / KK) % Ci), o = static_cast<int>(i / (static_cast<size_t>(KK) * Ci));
    w[i] = pw[static_cast<size_t>(o) * Ci + c] * dw[static_cast<size_t>(c) * KK + t];
  }
  if (bias) {
    for (int o = blockIdx.x * blockDim.x + threadIdx.x; o < Co; o += gridDim.x * blockDim.x) {
      float s = pwb ? pwb[o] : 0.f;
      if (dwb)
        for (int c = 0; c < Ci; ++c) s += pw[static_cast<size_t>(o) * Ci + c] * dwb[c];
      bias[o] = s;
    }
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------ host launchers
int bn_fold(const float* g, const float* b, const float* mean, const float* var, float eps, float* scale, float* shift,
            int n, int n_pad, cudaStream_t st) {
  launch_k(bn_fold_kernel, (n_pad + 255) / 256, 256, 0, st, g, b, mean, var, eps, scale, shift, n, n_pad);
  WC_LAUNCH_CHECK();
  return 0;
}
int maxpool_fwd(const __nv_bfloat16* x, __nv_bfloat16* y, uint8_t* idx, int B, int H, int W, int C, cudaStream_t st) {
  const int Ho = (H + 2 - 3) / 2 + 1, Wo = (W + 2 - 3) / 2 + 1;
  ProfScope prof(kProfOther, st, 0);
  launch_k(maxpool_fwd_kernel, grid_for(static_cast<size_t>(B) * Ho * Wo * C / 8), 256, 0, st, x, y, idx, B, H, W, C, Ho, Wo);
  WC_LAUNCH_CHECK();
  return 0;
}
int maxpool_bwd(const __nv_bfloat16* dy, const uint8_t* idx, const __nv_bfloat16* x, __nv_bfloat16* dx, int B, int H,
                int W, int C, cudaStream_t st) {
  const int Ho = (H + 2 - 3) / 2 + 1, Wo = (W + 2 - 3) / 2 + 1;
  ProfScope prof(kProfOther, st, 0);
  launch_k(maxpool_bwd_kernel, grid_for(static_cast<size_t>(B) * H * W * C / 8), 256, 0, st, dy, idx, x, dx, B, H, W, C, Ho, Wo);
  WC_LAUNCH_CHECK();
  return 0;
}
int gap_fwd(const __nv_bfloat16* x, __nv_bfloat16* y, int B, int HW, int C, int ld, cudaStream_t st) {
  ProfScope prof(kProfOther, st, 0);
  launch_k(gap_fwd_kernel, dim3((C + 63) / 64, B), 256, 0, st, x, y, HW, C, ld);
  WC_LAUNCH_CHECK();
  return 0;
}
int broadcast_hw(const __nv_bfloat16* v, __nv_bfloat16* y, int B, int HW, int C, int ldy, cudaStream_t st) {
  ProfScope prof(kProfOther, st, 0);
  launch_k(broadcast_kernel, grid_for(static_cast<size_t>(B) * HW * C / 8), 256, 0, st, v, y, B, HW, C, ldy);
  WC_LAUNCH_CHECK();
  return 0;
}
int sum_hw(const __nv_bfloat16* y, const __nv_bfloat16* mask, __nv_bfloat16* v, int B, int HW, int C, int ldy, cudaStream_t st) {
  ProfScope prof(kProfOther, st, 0);
  launch_k(sum_hw_kernel, dim3((C + 63) / 64, B), 256, 0, st, y, mask, v, HW, C, ldy);
  WC_LAUNCH_CHECK();
  return 0;
}
int gap_bwd_add(const __nv_bfloat16* g, __nv_bfloat16* dx, int B, int HW, int C, int ld, cudaStream_t st) {
  ProfScope prof(kProfOther, st, 0);
  launch_k(gap_bwd_add_kernel, grid_for(static_cast<size_t>(B) * HW * C), 256, 0, st, g, dx, B, HW, C, ld);
  WC_LAUNCH_CHECK();
  return 0;
}
int bilinear_fwd(const __nv_bfloat16* x, __nv_bfloat16* y, int B, int Hi, int Wi, int Ho, int Wo, int C, int ldx, int ldy,
                 cudaStream_t st) {
  WC_REQUIRE(C % 8 == 0, "bilinear: C must be a multiple of 8");
  ProfScope prof(kProfOther, st, 0);
  launch_k(bilinear_fwd_kernel, grid_for(static_cast<size_t>(B) * Ho * Wo * C / 8), 256, 0, st, x, y, B, Hi, Wi, Ho, Wo, C, ldx, ldy);
  WC_LAUNCH_CHECK();
  return 0;
}
int bilinear_bwd(const __nv_bfloat16* dy, const __nv_bfloat16* mask, __nv_bfloat16* dx, int B, int Hi, int Wi, int Ho,
                 int Wo, int C, int ldy, int ldm, int ldx, cudaStream_t st) {
  ProfScope prof(kProfOther, st, 0);
  WC_REQUIRE(C % 8 == 0 && ldy % 8 == 0 && ldx % 8 == 0, "bilinear_bwd: channels / strides must be multiples of 8");
  launch_k(bilinear_bwd_kernel, grid_for(static_cast<size_t>(B) * Hi * Wi * C / 8), 256, 0, st, dy, mask, dx, B, Hi, Wi, Ho, Wo, C, ldy, ldm, ldx);
  WC_LAUNCH_CHECK();
  return 0;
}
int seg_loss_grad(const float* logits_lo, const long long* labels, int* n_valid, long long* pred, float* dlogit_hi,
                  float* loss, float* logits_hi, int B, int h, int w, int H, int W, int nc, int ignore, cudaStream_t st) {
  WC_REQUIRE(nc == 19, "loss head is compiled for 19 classes (Cityscapes trainIds)");
  WC_REQUIRE(labels || (!pred && !dlogit_hi && !loss), "seg_loss_grad without labels writes the up-sampled logits only");
  ProfScope prof(kProfOther, st, 0);
  if (labels) {
    WC_CHECK_CUDA(cudaMemsetAsync(n_valid, 0, B * sizeof(int), st));
    if (loss) WC_CHECK_CUDA(cudaMemsetAsync(loss, 0, B * sizeof(float), st));
    launch_k(count_valid_kernel, dim3(std::min(64, (H * W + 255) / 256), B), 256, 0, st, labels, H * W, ignore, n_valid);
    WC_LAUNCH_CHECK();
  }
  launch_k(seg_loss_grad_kernel<19>, grid_for(static_cast<size_t>(B) * H * W, 128), 128, 0, st, logits_lo, labels, n_valid, pred, dlogit_hi, loss, logits_hi, B, h, w, H, W, ignore);
  WC_LAUNCH_CHECK();
  return 0;
}
// Fused loss head: pred, loss and the low-resolution d-logits in one pass (see seg_loss_head_fused_kernel).  Returns -1 (nothing
// launched) when the geometry is outside what the fused kernel covers; the caller then runs the two-pass path.
int seg_loss_head_fused(const float* logits_lo, const long long* labels, int* n_valid, long long* pred, float* loss,
                        __nv_bfloat16* dlo, int B, int h, int w, int H, int W, int nc, int cp, int ldo, int ignore, cudaStream_t st) {
  WC_REQUIRE(nc == 19, "loss head is compiled for 19 classes (Cityscapes trainIds)");
  if (H % h != 0 || W % w != 0 || cp > 32) return -1;
  const int fy = H / h, fx = W / w;
  if (fy > 8 || fx > 8) return -1;   // per-thread tap arrays hold 2f <= 16 rows / columns
  const int RH = fy * (kLhTY - 1) + (3 * fy) / 2 + (fy + 1) / 2 + 1, RW = fx * (kLhTX - 1) + (3 * fx) / 2 + (fx + 1) / 2 + 1;
  const size_t smem = static_cast<size_t>(RH) * RW * 19 * sizeof(float) + 64;
  if (smem > 200 * 1024) return -1;
  static size_t attr = 0;
  if (smem > attr) {
    WC_CHECK_CUDA(cudaFuncSetAttribute(seg_loss_head_fused_kernel<19>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    attr = smem;
  }
  ProfScope prof(kProfOther, st, 0);
  WC_CHECK_CUDA(cudaMemsetAsync(n_valid, 0, B * sizeof(int), st));
  if (loss) WC_CHECK_CUDA(cudaMemsetAsync(loss, 0, B * sizeof(float), st));
  launch_k(count_valid_kernel, dim3(std::min(64, (H * W + 255) / 256), B), 256, 0, st, labels, H * W, ignore, n_valid);
  WC_LAUNCH_CHECK();
  launch_k(seg_loss_head_fused_kernel<19>, dim3((w + kLhTX - 1) / kLhTX, (h + kLhTY - 1) / kLhTY, B), kLhThreads, smem, st, logits_lo, labels,
           n_valid, pred, loss, dlo, h, w, H, W, fy, fx, RW, cp, ldo, ignore);
  WC_LAUNCH_CHECK();
  return 0;
}
int logits_bilinear_bwd(const float* dhi, __nv_bfloat16* dlo, int B, int h, int w, int H, int W, int nc, int cp, int ldo,
                        cudaStream_t st) {
  WC_REQUIRE(nc == 19, "loss head is compiled for 19 classes");
  ProfScope prof(kProfOther, st, 0);
  launch_k(logits_bilinear_bwd_kernel<19>, grid_for(static_cast<size_t>(B) * h * w, 128), 128, 0, st, dhi, dlo, B, h, w, H, W, cp, ldo);
  WC_LAUNCH_CHECK();
  return 0;
}
int conv1_dgrad(const __nv_bfloat16* dz, const float* w, const float* scale, float* dx, int B, int H, int W, int Cout,
                cudaStream_t st) {
  WC_REQUIRE(Cout == 64 && H % 2 == 0 && W % 2 == 0, "conv1 data gradient is built for 64 output channels and even image dims");
  const int Ho = H / 2, Wo = W / 2;
  const size_t smem = static_cast<size_t>(49) * 64 * 3 * sizeof(float);
  ProfScope prof(kProfBoundaryConv, st, static_cast<double>(B) * (12.0 * H * W + 2.0 * Ho * Wo * Cout));
  const int gx = std::max(1, grid_for(static_cast<size_t>(B) * Ho * Wo, 128) / 2);
  launch_k(conv1_dgrad_kernel, dim3(gx, 4), 128, smem, st, dz, w, scale, dx, B, H, W, Ho, Wo);
  WC_LAUNCH_CHECK();
  return 0;
}
int conv1_dgrad_weff(const float* w, const float* scale, float* weff, int P, cudaStream_t st) {
  launch_k(conv1_dgrad_weff_kernel, 8, 256, 0, st, w, scale, weff, P);
  WC_LAUNCH_CHECK();
  return 0;
}
// out: [B,3,H/P,W/P] fp32 = avg_pool2d(conv1 data gradient, P); dz: [B,H/2,W/2,64] bf16
int conv1_dgrad_pooled(const __nv_bfloat16* dz, const float* weff, float* out, int B, int H, int W, int P, cudaStream_t st) {
  WC_REQUIRE(P >= 2 && P % 2 == 0 && P <= 8 && H % P == 0 && W % P == 0, "pooled stem gradient needs an even pool <= 8 dividing H and W");
  const int R = P / 2 + 3;
  const size_t smem = static_cast<size_t>(R) * R * 192 * sizeof(float);
  static size_t attr = 0;
  if (smem > 48 * 1024 && smem > attr) {
    WC_CHECK_CUDA(cudaFuncSetAttribute(conv1_dgrad_pooled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    attr = smem;
  }
  ProfScope prof(kProfBoundaryConv, st, static_cast<double>(B) * (12.0 * (H / P) * (W / P) + 2.0 * (H / 2) * (W / 2) * 64));
  launch_k(conv1_dgrad_pooled_kernel, grid_for(static_cast<size_t>(B) * (H / P) * (W / P), 128), 128, smem, st, dz, weff, out, B, H / 2, W / 2, P);
  WC_LAUNCH_CHECK();
  return 0;
}
int relu_mask_inplace(__nv_bfloat16* d, const __nv_bfloat16* m, size_t npix, int C, int ldd, int ldm, cudaStream_t st) {
  ProfScope prof(kProfOther, st, 0);
  launch_k(relu_mask_kernel, grid_for(npix * C), 256, 0, st, d, m, npix, C, ldd, ldm);
  WC_LAUNCH_CHECK();
  return 0;
}
int compose_sep(const float* dw, const float* pw, const float* dwb, const float* pwb, float* w, float* bias, int Co, int Ci,
                int KK, cudaStream_t st) {
  launch_k(compose_sep_kernel, grid_for(static_cast<size_t>(Co) * Ci * KK), 256, 0, st, dw, pw, dwb, pwb, w, bias, Co, Ci, KK);
  WC_LAUNCH_CHECK();
  return 0;
}

}  // namespace wc

// =====================================================================================================================
// SRGAN final layer (srgan_model/models.py:85,92): depthwise 9x9 (64 ch, bias) -> pointwise 64->3 (bias) -> (tanh+1)/2,
// NHWC bf16 in, NCHW fp32 out.  One CTA = an 8 x 64 output tile; the (8+8) x (64+8) x 64-channel halo tile is staged
// in shared memory as 32 channel-pair planes of half2 (conflict-free row reads); each thread owns 4 adjacent pixels and half
// of the channel pairs, sliding a 12-wide register window over every kernel row.
namespace wc {
namespace {

constexpr int kFT_H = 8, kFT_W = 64, kFHalo = 4, kFPlaneW = kFT_W + 2 * kFHalo /*72*/, kFPlaneH = kFT_H + 2 * kFHalo /*16*/;
constexpr int kFPlane = kFPlaneW * kFPlaneH + 1;  // +1 word: de-phase the planes across banks for the staging writes

__global__ void __launch_bounds__(512, 1)
srgan_final_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ dw /*[64][81]*/,
                   const float* __restrict__ dwb, const float* __restrict__ pw /*[3][64]*/, const float* __restrict__ pwb,
                   float* __restrict__ y, int B, int H, int W, int ldx) {
  pdl_prologue();
  extern __shared__ uint32_t sm[];
  uint32_t* tile = sm;                                            // [32][kFPlane] half2
  float* wsm = reinterpret_cast<float*>(sm + 32 * kFPlane);       // [32][81] half2 in the first half of [32][81][2] words
  float* red = wsm + 32 * 81 * 2;                                 // [3 groups][128 threads][12]
  const int tiles_x = (W + kFT_W - 1) / kFT_W, tiles_y = (H + kFT_H - 1) / kFT_H;
  const int tid = threadIdx.x;
  {
    __half2* wh = reinterpret_cast<__half2*>(wsm);
    for (int i = tid; i < 32 * 81; i += 512) {
      const int tap = i % 81, c2 = i / 81;
      wh[i] = __floats2half2_rn(dw[(c2 * 2) * 81 + tap], dw[(c2 * 2 + 1) * 81 + tap]);
    }
  }
  // thread -> column tx (lanes sweep x: conflict-free shared-memory reads) and 4 vertically adjacent output rows
  const int grp = tid >> 7, t = tid & 127, tx = t & 63, ty = (t >> 6) * 4;
  for (int tl = blockIdx.x; tl < B * tiles_x * tiles_y; tl += gridDim.x) {
    const int b = tl / (tiles_x * tiles_y), r = tl % (tiles_x * tiles_y), y0 = (r / tiles_x) * kFT_H, x0 = (r % tiles_x) * kFT_W;
    __syncthreads();
    // stage the halo tile: one 16-byte (8-channel) chunk per thread-iteration
    for (int i = tid; i < kFPlaneH * kFPlaneW * 8; i += 512) {
      const int c8 = i & 7, px = (i >> 3) % kFPlaneW, py = (i >> 3) / kFPlaneW;
      const int gy = y0 + py - kFHalo, gx = x0 + px - kFHalo;
      uint4 u = make_uint4(0, 0, 0, 0);
      if (gy >= 0 && gy < H && gx >= 0 && gx < W)
        u = __ldg(reinterpret_cast<const uint4*>(x + ((static_cast<size_t>(b) * H + gy) * W + gx) * ldx + c8 * 8));
      uint32_t* dst = tile + (c8 * 4) * kFPlane + py * kFPlaneW + px;
      // channel pairs as half2 (11-bit mantissa: exact for bf16 values inside the fp16 range)
      auto h2 = [](uint32_t w) {
        const __half2 h = __floats2half2_rn(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
        return *reinterpret_cast<const uint32_t*>(&h);
      };
      u.x = h2(u.x); u.y = h2(u.y); u.z = h2(u.z); u.w = h2(u.w);
      dst[0] = u.x; dst[kFPlane] = u.y; dst[2 * kFPlane] = u.z; dst[3 * kFPlane] = u.w;
    }
    __syncthreads();
    float o[3][4];
#pragma unroll
    for (int n = 0; n < 3; ++n)
#pragma unroll
      for (int p = 0; p < 4; ++p) o[n][p] = 0.f;
    for (int c2 = grp * 8; c2 < grp * 8 + 8; ++c2) {
      float2 acc2[4];
      const float b0 = dwb ? dwb[2 * c2] : 0.f, b1 = dwb ? dwb[2 * c2 + 1] : 0.f;
#pragma unroll
      for (int p = 0; p < 4; ++p) acc2[p] = make_float2(b0, b1);
      const uint32_t* pl = tile + c2 * kFPlane + ty * kFPlaneW + tx;
      // packed fp16 FMAs (HFMA2: two channels per instruction, no bf16 unpacking) over the nine rows of one kernel column,
      // folded into the fp32 accumulators after every column: 9 fp16 roundings per partial sum instead of 81
      const __half2* wh = reinterpret_cast<const __half2*>(wsm) + c2 * 81;
#pragma unroll
      for (int kx = 0; kx < 9; ++kx) {
        __half2 v[12];   // 12-row register window of column tx + kx (rows ty .. ty+11 of the halo tile)
#pragma unroll
        for (int i = 0; i < 12; ++i) {
          const uint32_t u = pl[i * kFPlaneW + kx];
          v[i] = *reinterpret_cast<const __half2*>(&u);
        }
        __half2 part[4];
#pragma unroll
        for (int p = 0; p < 4; ++p) part[p] = __hmul2(v[p], wh[kx]);
#pragma unroll
        for (int ky = 1; ky < 9; ++ky) {
          const __half2 wv = wh[ky * 9 + kx];
#pragma unroll
          for (int p = 0; p < 4; ++p) part[p] = __hfma2(v[p + ky], wv, part[p]);
        }
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          const float2 f = __half22float2(part[p]);
          acc2[p].x += f.x; acc2[p].y += f.y;
        }
      }
#pragma unroll
      for (int n = 0; n < 3; ++n) {
        const float w0 = pw[n * 64 + 2 * c2], w1 = pw[n * 64 + 2 * c2 + 1];
#pragma unroll
        for (int p = 0; p < 4; ++p) o[n][p] = fmaf(acc2[p].x, w0, fmaf(acc2[p].y, w1, o[n][p]));
      }
    }
    if (grp > 0) {
#pragma unroll
      for (int n = 0; n < 3; ++n)
#pragma unroll
        for (int p = 0; p < 4; ++p) red[((grp - 1) * 128 + t) * 12 + n * 4 + p] = o[n][p];
    }
    __syncthreads();
    if (grp == 0) {
      const int gx = x0 + tx;
      const size_t plane = static_cast<size_t>(H) * W;
#pragma unroll
      for (int n = 0; n < 3; ++n)
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          const int gy = y0 + ty + p;
          if (gy < H && gx < W) {
            const float v = o[n][p] + red[t * 12 + n * 4 + p] + red[(128 + t) * 12 + n * 4 + p] + red[(256 + t) * 12 + n * 4 + p] +
                            (pwb ? pwb[n] : 0.f);
            y[(static_cast<size_t>(b) * 3 + n) * plane + static_cast<size_t>(gy) * W + gx] = (tanhf(v) + 1.f) * 0.5f;
          }
        }
    }
  }
}

// ---- SRGAN final layer on the tensor core (round 2).  out[y][x][o] = sum_ty sum_tx sum_c in[y+ty-4][x+tx-4][c] pw[o][c] dw[c][ty][tx]
// is split into  T[y'][x][(ty, o)] = sum_tx sum_c in[y'][x+tx-4][c] Wq[(ty, o)][c][tx]  - a 1x9 horizontal convolution with
// N = 27 (padded to 32) output columns, run by the implicit-GEMM kernel into 27 fp32 planes - and the vertical shift-add
// out[y][x][o] = sum_ty T[y+ty-4][x][(ty, o)] + bias, (tanh + 1)/2, done here.  36 tcgen05.mma (128x32x16) per 128 pixels replace
// 5376 FMAs per pixel on the CUDA cores.
__global__ void srgan_final_compose_kernel(const float* __restrict__ dw, const float* __restrict__ dwb, const float* __restrict__ pw,
                                           const float* __restrict__ pwb, float* __restrict__ wq /*[32][64][1][9]*/,
                                           float* __restrict__ bias3) {
  pdl_prologue();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 32 * 64 * 9) {
    const int tx = i % 9, c = (i / 9) % 64, n = i / (9 * 64);
    float v = 0.f;
    if (n < 27) {
      const int ty = n / 3, o = n % 3;
      v = pw[o * 64 + c] * dw[(c * 9 + ty) * 9 + tx];
    }
    wq[i] = v;
  }
  if (i < 3) {
    float b = pwb ? pwb[i] : 0.f;
    if (dwb)
      for (int c = 0; c < 64; ++c) b = fmaf(pw[i * 64 + c], dwb[c], b);
    bias3[i] = b;
  }
}

__global__ void __launch_bounds__(256)
srgan_final_combine_kernel(const float* __restrict__ t /*[B][27][H][W]*/, const float* __restrict__ bias3, float* __restrict__ y /*[B][3][H][W]*/,
                           int H, int W4) {
  pdl_prologue();
  const int x4 = blockIdx.x * blockDim.x + threadIdx.x;   // group of four pixels of one row
  const int yy = blockIdx.y, b = blockIdx.z;
  if (x4 >= W4) return;
  const size_t plane4 = static_cast<size_t>(H) * W4;
  const float4* tp = reinterpret_cast<const float4*>(t) + static_cast<size_t>(b) * 27 * plane4 + x4;
  float4 acc[3];
#pragma unroll
  for (int o = 0; o < 3; ++o) {
    const float bo = bias3[o];
    acc[o] = make_float4(bo, bo, bo, bo);
  }
#pragma unroll
  for (int ty = 0; ty < 9; ++ty) {
    const int r = yy + ty - 4;
    if (r < 0 || r >= H) continue;
#pragma unroll
    for (int o = 0; o < 3; ++o) {
      const float4 v = __ldg(tp + static_cast<size_t>(ty * 3 + o) * plane4 + static_cast<size_t>(r) * W4);
      acc[o].x += v.x; acc[o].y += v.y; acc[o].z += v.z; acc[o].w += v.w;
    }
  }
  float4* yp = reinterpret_cast<float4*>(y) + static_cast<size_t>(b) * 3 * plane4 + static_cast<size_t>(yy) * W4 + x4;
#pragma unroll
  for (int o = 0; o < 3; ++o) {
    float4 v;
    v.x = (tanhf(acc[o].x) + 1.f) * 0.5f; v.y = (tanhf(acc[o].y) + 1.f) * 0.5f;
    v.z = (tanhf(acc[o].z) + 1.f) * 0.5f; v.w = (tanhf(acc[o].w) + 1.f) * 0.5f;
    yp[static_cast<size_t>(o) * plane4] = v;
  }
}

// PixelShuffle(r = 2) as phase-major output rows: dst row q*cb + c = src row c*4 + q (rows of `len` floats); with rep_src = 1 the
// source has only cb rows and is replicated to every phase (per-channel PReLU slopes).
__global__ void phase_major_rows_kernel(const float* __restrict__ src, float* __restrict__ dst, int cb, int len, int rep_src) {
  pdl_prologue();
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i >= static_cast<size_t>(4) * cb * len) return;
  const int e = static_cast<int>(i % len), n = static_cast<int>(i / len), q = n / cb, c = n % cb;
  dst[i] = src[static_cast<size_t>(rep_src ? c : c * 4 + q) * len + e];
}

}  // namespace

int srgan_final(const __nv_bfloat16* x, const float* dw, const float* dwb, const float* pw, const float* pwb, float* y, int B,
                int H, int W, int ldx, cudaStream_t st) {
  const size_t smem = (32 * kFPlane) * 4 + 32 * 81 * 2 * 4 + 3 * 128 * 12 * 4;
  static bool attr = false;
  if (!attr) {
    WC_CHECK_CUDA(cudaFuncSetAttribute(srgan_final_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    attr = true;
  }
  const int tiles = B * ((W + kFT_W - 1) / kFT_W) * ((H + kFT_H - 1) / kFT_H);
  ProfScope prof(kProfBoundaryConv, st, static_cast<double>(B) * H * W * (128.0 + 12.0));
  launch_k(srgan_final_kernel, std::min(tiles, num_sms()), 512, smem, st, x, dw, dwb, pw, pwb, y, B, H, W, ldx);
  WC_LAUNCH_CHECK();
  return 0;
}
int srgan_final_compose(const float* dw, const float* dwb, const float* pw, const float* pwb, float* wq, float* bias3, cudaStream_t st) {
  launch_k(srgan_final_compose_kernel, (32 * 64 * 9 + 255) / 256, 256, 0, st, dw, dwb, pw, pwb, wq, bias3);
  WC_LAUNCH_CHECK();
  return 0;
}
int srgan_final_combine(const float* t, const float* bias3, float* y, int B, int H, int W, cudaStream_t st) {
  WC_REQUIRE(W % 4 == 0, "srgan_final_combine: width must be a multiple of 4");
  const int W4 = W / 4;
  ProfScope prof(kProfBoundaryConv, st, static_cast<double>(B) * H * W * (27.0 * 4 + 12.0));
  launch_k(srgan_final_combine_kernel, dim3((W4 + 255) / 256, H, B), 256, 0, st, t, bias3, y, H, W4);
  WC_LAUNCH_CHECK();
  return 0;
}
// SRGAN `initial` block (srgan_model/models.py:74, ConvBlock(3, 64, k9, use_bn=False)): depthwise 9x9 on the 3 input
// channels (+bias), pointwise 3 -> 64 (+bias), PReLU(64); NCHW fp32 in, NHWC bf16 out.  Run SEPARABLY as the reference
// does (435 MAC per pixel); the composed dense 9x9 3 -> 64 convolution it replaces cost 15552 MAC per pixel (0.39 ms per
// C3 step).  One thread per pixel, 16 x 16 tiles with a 4-pixel halo staged in shared memory.
constexpr int kSI_T = 16;
__global__ void __launch_bounds__(kSI_T * kSI_T)
srgan_initial_kernel(const float* __restrict__ x, const float* __restrict__ dw, const float* __restrict__ dwb,
                     const float* __restrict__ pw, const float* __restrict__ pwb, const float* __restrict__ slope,
                     __nv_bfloat16* __restrict__ y, int H, int W, int ldy) {
  pdl_prologue();
  constexpr int HT = kSI_T + 8;
  __shared__ float tile[3][HT][HT + 1];
  __shared__ float s_dw[3][81], s_pw[64][3], s_b[64], s_sl[64], s_dwb[3];
  const int tid = threadIdx.y * kSI_T + threadIdx.x;
  const int b = blockIdx.z, x0 = blockIdx.x * kSI_T, y0 = blockIdx.y * kSI_T;
  for (int i = tid; i < 243; i += kSI_T * kSI_T) s_dw[i / 81][i % 81] = dw[i];
  for (int i = tid; i < 192; i += kSI_T * kSI_T) s_pw[i / 3][i % 3] = pw[i];
  if (tid < 64) { s_b[tid] = pwb ? pwb[tid] : 0.f; s_sl[tid] = slope[tid]; }
  if (tid < 3) s_dwb[tid] = dwb ? dwb[tid] : 0.f;
  const float* xb = x + static_cast<size_t>(b) * 3 * H * W;
  for (int i = tid; i < 3 * HT * HT; i += kSI_T * kSI_T) {
    const int c = i / (HT * HT), r = (i / HT) % HT, q = i % HT;
    const int yy = y0 + r - 4, xx = x0 + q - 4;
    tile[c][r][q] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? xb[(static_cast<size_t>(c) * H + yy) * W + xx] : 0.f;
  }
  __syncthreads();
  const int px = x0 + threadIdx.x, py = y0 + threadIdx.y;
  if (px >= W || py >= H) return;
  float d[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float a = s_dwb[c];
#pragma unroll
    for (int ky = 0; ky < 9; ++ky)
#pragma unroll
      for (int kx = 0; kx < 9; ++kx) a = fmaf(tile[c][threadIdx.y + ky][threadIdx.x + kx], s_dw[c][ky * 9 + kx], a);
    d[c] = a;
  }
  uint4* dst = reinterpret_cast<uint4*>(y + ((static_cast<size_t>(b) * H + py) * W + px) * ldy);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int n = 8 * j + i;
      float a = fmaf(d[2], s_pw[n][2], fmaf(d[1], s_pw[n][1], fmaf(d[0], s_pw[n][0], s_b[n])));
      v[i] = a > 0.f ? a : a * s_sl[n];
    }
    uint4 u;
    u.x = pack_bf16(v[0], v[1]); u.y = pack_bf16(v[2], v[3]); u.z = pack_bf16(v[4], v[5]); u.w = pack_bf16(v[6], v[7]);
    dst[j] = u;
  }
}

int srgan_initial(const float* x, const float* dw, const float* dwb, const float* pw, const float* pwb, const float* slope,
                  __nv_bfloat16* y, int B, int H, int W, int ldy, cudaStream_t st) {
  WC_REQUIRE(ldy % 8 == 0, "output pixel stride must be a multiple of 8");
  ProfScope prof(kProfBoundaryConv, st, static_cast<double>(B) * H * W * (3 * 4.0 + 64 * 2.0));
  dim3 grid((W + kSI_T - 1) / kSI_T, (H + kSI_T - 1) / kSI_T, B);
  launch_k(srgan_initial_kernel, grid, dim3(kSI_T, kSI_T), 0, st, x, dw, dwb, pw, pwb, slope, y, H, W, ldy);
  WC_LAUNCH_CHECK();
  return 0;
}

int phase_major_rows(const float* src, float* dst, int cb, int len, int rep_src, cudaStream_t st) {
  const size_t total = static_cast<size_t>(4) * cb * len;
  launch_k(phase_major_rows_kernel, static_cast<int>((total + 255) / 256), 256, 0, st, src, dst, cb, len, rep_src);
  WC_LAUNCH_CHECK();
  return 0;
}
}  // namespace wc

// =====================================================================================================================
// SRGAN input-gradient backward (srgan.cu: wc_srgan_backward_seeded): the elementwise pieces between the data-gradient
// convolutions.  PReLU derivatives read the pre-activation that the with-grad forward keeps (the PReLU output alone does
// not determine the sign of the pre-activation when a slope is <= 0).
namespace wc {
namespace {

// d(pre-tanh) of y = (tanh(z) + 1) / 2:  dz = dy * 2y(1 - y), fp32 NCHW
__global__ void srgan_tanh_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ y, float* __restrict__ dz, size_t n) {
  pdl_prologue();
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float v = y[i];
    dz[i] = dy[i] * (2.f * v * (1.f - v));
  }
}

// wt[ci][co][KK-1-t] = w[co][ci][t]: the data gradient of a stride-1 'same' KxK convolution as a convolution of dy
__global__ void flip_transpose_kk_kernel(const float* __restrict__ w, float* __restrict__ wt, int Co, int Ci, int KK) {
  pdl_prologue();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Co * Ci * KK) return;
  const int t = i % KK, ci = (i / KK) % Ci, co = i / (KK * Ci);
  wt[(static_cast<size_t>(ci) * Co + co) * KK + (KK - 1 - t)] = w[i];
}

// d := (d + add) * (pre > 0 ? 1 : slope[c]), NHWC bf16, 8 channels per thread (C % 8 == 0)
__global__ void prelu_bwd_kernel(__nv_bfloat16* __restrict__ d, const __nv_bfloat16* __restrict__ add,
                                 const __nv_bfloat16* __restrict__ pre, const float* __restrict__ slope, size_t npix, int C, int ldd,
                                 int lda, int ldp) {
  pdl_prologue();
  const int c8n = C / 8;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < npix * c8n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t p = i / c8n;
    const int c0 = static_cast<int>(i % c8n) * 8;
    uint4* dp = reinterpret_cast<uint4*>(d + p * ldd + c0);
    const uint4 u = *dp, m = *reinterpret_cast<const uint4*>(pre + p * ldp + c0);
    const uint4 a = add ? *reinterpret_cast<const uint4*>(add + p * lda + c0) : make_uint4(0, 0, 0, 0);
    const uint32_t uu[4] = {u.x, u.y, u.z, u.w}, mm[4] = {m.x, m.y, m.z, m.w}, aa[4] = {a.x, a.y, a.z, a.w};
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 g = unpack_bf16(uu[k]), s = unpack_bf16(mm[k]), q = unpack_bf16(aa[k]);
      const float gx = g.x + q.x, gy = g.y + q.y;
      o[k] = pack_bf16(s.x > 0.f ? gx : gx * slope[c0 + 2 * k], s.y > 0.f ? gy : gy * slope[c0 + 2 * k + 1]);
    }
    *dp = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// PReLU(PixelShuffle(2)) backward: dconv[b][y][x][4c + 2i + j] = dup[b][2y+i][2x+j][c] * (pre > 0 ? 1 : slope[c]);
// dup / pre: [B][2h][2w][C] (ld C), dconv: [B][h][w][4C].  One thread = 8 consecutive conv channels (two shuffled channels).
__global__ void shuffle_prelu_bwd_kernel(const __nv_bfloat16* __restrict__ dup, const __nv_bfloat16* __restrict__ pre,
                                         const float* __restrict__ slope, __nv_bfloat16* __restrict__ dconv, int B, int h, int w, int C) {
  pdl_prologue();
  const int k8 = C / 2;   // groups of 8 conv channels per pixel
  const size_t total = static_cast<size_t>(B) * h * w * k8;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int k = static_cast<int>(i % k8);
    const size_t pix = i / k8;
    const int x = static_cast<int>(pix % w), y = static_cast<int>((pix / w) % h), b = static_cast<int>(pix / (static_cast<size_t>(w) * h));
    const int c = 2 * k;
    const float s0 = slope[c], s1 = slope[c + 1];
    float v[8];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const size_t off = ((static_cast<size_t>(b) * 2 * h + 2 * y + (q >> 1)) * 2 * w + 2 * x + (q & 1)) * C + c;
      const float2 g = unpack_bf16(*reinterpret_cast<const uint32_t*>(dup + off));
      const float2 m = unpack_bf16(*reinterpret_cast<const uint32_t*>(pre + off));
      v[q] = m.x > 0.f ? g.x : g.x * s0;       // conv channel 4c + q
      v[4 + q] = m.y > 0.f ? g.y : g.y * s1;   // conv channel 4(c+1) + q
    }
    uint4 o;
    o.x = pack_bf16(v[0], v[1]); o.y = pack_bf16(v[2], v[3]); o.z = pack_bf16(v[4], v[5]); o.w = pack_bf16(v[6], v[7]);
    *reinterpret_cast<uint4*>(dconv + pix * (4 * C) + 8 * k) = o;
  }
}

__global__ void fill_f32_kernel(float* __restrict__ p, float v, int n) {
  pdl_prologue();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

}  // namespace

int srgan_tanh_bwd(const float* dy, const float* y, float* dz, size_t n, cudaStream_t st) {
  ProfScope prof(kProfOther, st, 0);
  launch_k(srgan_tanh_bwd_kernel, grid_for(n), 256, 0, st, dy, y, dz, n);
  WC_LAUNCH_CHECK();
  return 0;
}
int flip_transpose_kk(const float* w, float* wt, int Co, int Ci, int KK, cudaStream_t st) {
  launch_k(flip_transpose_kk_kernel, (Co * Ci * KK + 255) / 256, 256, 0, st, w, wt, Co, Ci, KK);
  WC_LAUNCH_CHECK();
  return 0;
}
int prelu_bwd(__nv_bfloat16* d, const __nv_bfloat16* add, const __nv_bfloat16* pre, const float* slope, size_t npix, int C, int ldd,
              int lda, int ldp, cudaStream_t st) {
  WC_REQUIRE(C % 8 == 0 && ldd % 8 == 0 && lda % 8 == 0 && ldp % 8 == 0, "prelu_bwd: channels and pixel strides must be multiples of 8");
  ProfScope prof(kProfOther, st, 0);
  launch_k(prelu_bwd_kernel, grid_for(npix * (C / 8)), 256, 0, st, d, add, pre, slope, npix, C, ldd, lda, ldp);
  WC_LAUNCH_CHECK();
  return 0;
}
int shuffle_prelu_bwd(const __nv_bfloat16* dup, const __nv_bfloat16* pre, const float* slope, __nv_bfloat16* dconv, int B, int h, int w,
                      int C, cudaStream_t st) {
  WC_REQUIRE(C % 2 == 0, "shuffle_prelu_bwd: even channel count");
  ProfScope prof(kProfOther, st, 0);
  launch_k(shuffle_prelu_bwd_kernel, grid_for(static_cast<size_t>(B) * h * w * (C / 2)), 256, 0, st, dup, pre, slope, dconv, B, h, w, C);
  WC_LAUNCH_CHECK();
  return 0;
}
int fill_f32(float* p, float v, int n, cudaStream_t st) {
  launch_k(fill_f32_kernel, (n + 255) / 256, 256, 0, st, p, v, n);
  WC_LAUNCH_CHECK();
  return 0;
}
}  // namespace wc
