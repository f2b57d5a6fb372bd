// Convolution layers expressed as igemm plans: tap lists for stride-1 (dilated) convs, stride-2 convs (phase
// views), transposed / data-gradient convs (one plan per output phase), with weights packed to bf16 K-major.
#pragma once
#include <functional>
#include <memory>
#include <vector>

#include "igemm.cuh"

namespace wc {

// Library-owned device allocations (packed weights, folded biases); freed with the owning object.
class DeviceArena {
 public:
  ~DeviceArena();
  void* alloc(size_t bytes);  // returns nullptr and sets the error on failure
  size_t bytes() const { return total_; }

 private:
  std::vector<void*> ptrs_;
  size_t total_ = 0;
};

// While a recorder is set (training plans), every weight-packing launch issued by build_conv* is also appended to it,
// so the bf16 packed copies can be rebuilt from the fp32 master weights after each optimizer step.
void set_pack_recorder(std::vector<std::function<int(cudaStream_t)>>* recorder);

struct WeightSrc {
  const float* w = nullptr;  // fp32 device tensor, PyTorch layout
  int d0 = 0, d1 = 0;        // dims 0 and 1 of the source tensor
  int KH = 1, KW = 1;
  int transpose = 0;            // 0: out-channel = dim0 (Conv2d fwd); 1: out-channel = dim1 (ConvTranspose2d / dgrad)
  int flip = 0;                 // use tap (KH-1-ky, KW-1-kx): stride-1 data gradient
  const float* scale = nullptr;  // optional per-dim0 scale (folded BatchNorm)
};

struct ConvGeom {
  int K = 3, stride = 1, pad = 1, dil = 1;
};

struct Epilogue {
  const float* bias = nullptr;
  const float* rowbias = nullptr;
  int ldrb = 0;
  const Act* res = nullptr;
  const Act* mask = nullptr;
  int relu = 0;
  int act = 0;  // 2 SiLU, 3 GELU
  const float* prelu = nullptr;
};

struct OutSpec {
  int mode = kOutNHWC;
  Act out;  // kOutNHWC destination (full-resolution grid for transposed convs)
  float* out_f32 = nullptr;
  int n_store = 0;
  __nv_bfloat16 *q = nullptr, *k = nullptr, *vt = nullptr, *v = nullptr;
  int heads = 0, hd = 0;
  // kOutQKV: Q := q_scale * (x W_q + b_q), rounded to bf16 once.  With q_scale = log2(e) / sqrt(hd) the attention kernels run with a
  // unit softmax scale in the log2 domain (attention_forward(.., scale = kAttnScalePrescaled)): same rounding error as storing Q
  // unscaled, one multiply per logit less in the exponential loop.
  float q_scale = 1.f;
  int up = 1, py = 0, px = 0;  // build_conv only: write pixel (y,x) to (y*up+py, x*up+px) of an up-times larger grid
  // build_conv only, with up == 2: the N output columns are FOUR PHASE BLOCKS of N/4 channels; block q goes to (y*2 + q/2, x*2 + q%2)
  // (PixelShuffle with phase-major weight rows: one launch instead of four, the activation tile is read once)
  int phases = 0;
  int bn_max = 0;              // > 0: cap on the N tile (lets a 3x3 layer with N > 128 keep the row-segment mode)
};

// One logical layer = one or more igemm launches (4 for stride-2 transposed / dgrad convs).
struct ConvOp {
  std::vector<IgemmPlan> plans;
  double flops = 0;
  int run(cudaStream_t st) const {
    for (const auto& p : plans)
      if (int e = igemm_launch(p, st)) return e;
    return 0;
  }
};

// Forward convolution y = conv(x, W) (+ fused 1x1 conv of x2 with W2), "same" padding for stride 1,
// Ho = H/2 for stride 2.  N = number of output channels (multiple of 16 after padding by the caller).
int build_conv(ConvOp* op, DeviceArena* arena, const Act& x, const WeightSrc& w, const ConvGeom& g, int N,
               const Act* x2, const WeightSrc* w2, const Epilogue& ep, const OutSpec& out, cudaStream_t st);

// ResNet stem (7x7, stride 2, pad 3, 3 input channels) as an implicit GEMM over a padded NHWC-8 copy of the image (see conv.cu).
// xp: [B][H][W+8][8] bf16 made by stem_prepare(); wprime: [N][64][7] fp32 made by stem_weights().
int build_conv_stem7s2(ConvOp* op, DeviceArena* arena, const __nv_bfloat16* xp, int B, int H, int W, const float* wprime,
                       const float* scale, int N, const Epilogue& ep, const OutSpec& out, cudaStream_t st);
int stem_prepare(const float* x_nchw, __nv_bfloat16* xp, int B, int H, int W, cudaStream_t st);
int stem_weights(const float* w /*[N][3][7][7]*/, float* wprime /*[N][64][7]*/, int N, cudaStream_t st);

// 1 x KW horizontal convolution (w.KH == 1, KW odd), 'same' size: see conv.cu.
int build_conv_hrow(ConvOp* op, DeviceArena* arena, const Act& x, const WeightSrc& w, int N, const Epilogue& ep, const OutSpec& out,
                    cudaStream_t st);

// Transposed convolution with stride 2 (ConvTranspose2d(k, 2, pad), output exactly 2x) or, equivalently, the
// data gradient of a stride-2 convolution: out[2j+q] = sum_{k = (q+pad) mod 2 ...} in[j + (q+pad-k)/2] * W[k].
// Weight source must have transpose = 1 semantics (out-channel = dim1).
int build_conv_transposed_s2(ConvOp* op, DeviceArena* arena, const Act& x, const WeightSrc& w, int K, int pad, int N,
                             const Epilogue& ep, const OutSpec& out, cudaStream_t st);

}  // namespace wc
