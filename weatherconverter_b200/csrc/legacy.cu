// Legacy "old model" UNet forward as a static launch plan (reference: diffusion_model/models/old_modules.py:73-360,
// driven by diffusion_model/sample_integrated.py:40-67).  Eval-mode BatchNorm -> 3x3 conv -> SiLU -> 3x3 conv residual
// blocks, AvgPool2d(2), bilinear x2 up-sampling, LayerNorm + 4-head attention + GELU feed-forward blocks, a
// noise-variance sinusoidal embedding broadcast over the image.  Convolutions / linears / attention reuse the tcgen05
// kernels of the main UNet (igemm.cu, attention.cu); the kernels below are the bandwidth-bound glue.
// Skip tensors are written by the down path straight into the up path's concat buffers (torch.cat at :224 never runs).
#include "plan.cuh"
#include "wc_ptx.cuh"
#include "../../include/wc_b200.h"

namespace wc {
int bn_fold(const float* g, const float* b, const float* mean, const float* var, float eps, float* scale, float* shift,
            int n, int n_pad, cudaStream_t st);
int attention_forward(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, __nv_bfloat16* out, int B,
                      int heads, int ntok, int hd, int ldo, cudaStream_t st, float* lse = nullptr, float scale = 0.f);
double attention_flops(int B, int heads, int ntok, int hd);
int conv_small_cin(const float* x, const float* w, const float* bias, const float* scale, const float* shift,
                   __nv_bfloat16* y, int B, int Cin, int H, int W, int Cout, int K, int stride, int pad, int ldy,
                   int relu, cudaStream_t st, const float* prelu = nullptr);
int conv_small_cout(const __nv_bfloat16* x, const float* w, const float* bias, float* y, int B, int H, int W, int Cin,
                    int Cout, int K, int ldx, int tanh_out, cudaStream_t st);
int bilinear_fwd(const __nv_bfloat16* x, __nv_bfloat16* y, int B, int Hi, int Wi, int Ho, int Wo, int C, int ldx, int ldy,
                 cudaStream_t st);

namespace {

__device__ __forceinline__ void ld8(const __nv_bfloat16* p, float (&f)[8]) {
  const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
  float2 t;
  t = unpack_bf16(u.x); f[0] = t.x; f[1] = t.y;
  t = unpack_bf16(u.y); f[2] = t.x; f[3] = t.y;
  t = unpack_bf16(u.z); f[4] = t.x; f[5] = t.y;
  t = unpack_bf16(u.w); f[6] = t.x; f[7] = t.y;
}
__device__ __forceinline__ void st8(__nv_bfloat16* p, const float (&f)[8]) {
  uint4 w;
  w.x = pack_bf16(f[0], f[1]); w.y = pack_bf16(f[2], f[3]); w.z = pack_bf16(f[4], f[5]); w.w = pack_bf16(f[6], f[7]);
  *reinterpret_cast<uint4*>(p) = w;
}

// eval-mode BatchNorm2d as a per-channel affine map (old_modules.py:146): y = x*scale[c] + shift[c]
__global__ void channel_affine_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, size_t npix, int C,
                                      int ldx, int ldy, const float* __restrict__ scale, const float* __restrict__ shift) {
  pdl_prologue();
  const int vpp = C / 8;
  const size_t total = npix * vpp;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t p = i / vpp;
    const int v = static_cast<int>(i % vpp);
    float f[8];
    ld8(x + p * ldx + v * 8, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = fmaf(f[j], scale[v * 8 + j], shift[v * 8 + j]);
    st8(y + p * ldy + v * 8, f);
  }
}

// nn.LayerNorm([C]) over the channels of every token (old_modules.py:80,82): one warp per token
__global__ void layernorm_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, size_t rows, int C, int ldx,
                                 int ldy, const float* __restrict__ gamma, const float* __restrict__ beta, float eps) {
  pdl_prologue();
  const size_t row = (blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const __nv_bfloat16* xr = x + row * ldx;
  float v[8];  // C <= 256
  int n = 0;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) { v[n] = __bfloat162float(xr[c]); s += v[n]; ++n; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / C;
  float ss = 0.f;
  for (int i = 0; i < n; ++i) { const float d = v[i] - mean; ss += d * d; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float rstd = rsqrtf(ss / C + eps);
  __nv_bfloat16* yr = y + row * ldy;
  n = 0;
  for (int c = lane; c < C; c += 32) { yr[c] = __float2bfloat16_rn((v[n] - mean) * rstd * gamma[c] + beta[c]); ++n; }
}

// nn.AvgPool2d(2) (old_modules.py:183)
__global__ void avgpool2_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, int B, int Ho, int Wo, int C,
                                int ldx, int ldy) {
  pdl_prologue();
  const int vpp = C / 8;
  const size_t total = static_cast<size_t>(B) * Ho * Wo * vpp;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int v = static_cast<int>(i % vpp);
    const size_t p = i / vpp;
    const int ox = static_cast<int>(p % Wo), oy = static_cast<int>((p / Wo) % Ho), b = static_cast<int>(p / (static_cast<size_t>(Wo) * Ho));
    const size_t in0 = (static_cast<size_t>(b) * 2 * Ho + 2 * oy) * (2 * Wo) + 2 * ox;
    float a[8], t[8];
    ld8(x + in0 * ldx + v * 8, a);
    ld8(x + (in0 + 1) * ldx + v * 8, t);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] += t[j];
    ld8(x + (in0 + 2 * Wo) * ldx + v * 8, t);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] += t[j];
    ld8(x + (in0 + 2 * Wo + 1) * ldx + v * 8, t);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = (a[j] + t[j]) * 0.25f;
    st8(y + p * ldy + v * 8, a);
  }
}

// sinusoidal_embedding (old_modules.py:283-307) of the per-sample noise variance + nn.Upsample(nearest) to the image
// (:313-315): 32 channels [sin(2 pi f_j t) | cos(2 pi f_j t)], f_j = exp(linspace(ln 1, ln 1000, 16)), broadcast per pixel
__global__ void embed_broadcast_kernel(const float* __restrict__ t, __nv_bfloat16* __restrict__ y, int HW, int ldy) {
  pdl_prologue();
  __shared__ __align__(16) __nv_bfloat16 emb[32];
  const int b = blockIdx.y;
  if (threadIdx.x < 16) {
    const float step = logf(1000.0f) / 15.0f;
    const float f = expf(threadIdx.x < 8 ? threadIdx.x * step : logf(1000.0f) - (15 - threadIdx.x) * step);
    const float ang = 6.283185307179586f * f * t[b];
    emb[threadIdx.x] = __float2bfloat16_rn(sinf(ang));
    emb[16 + threadIdx.x] = __float2bfloat16_rn(cosf(ang));
  }
  __syncthreads();
  const uint4* e4 = reinterpret_cast<const uint4*>(emb);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < HW * 4; i += gridDim.x * blockDim.x) {
    const int p = i >> 2, q = i & 3;
    *reinterpret_cast<uint4*>(y + (static_cast<size_t>(b) * HW + p) * ldy + q * 8) = e4[q];
  }
}

inline int blocks_for(size_t n) { return static_cast<int>(std::min<size_t>((n + 255) / 256, 148 * 16)); }

}  // namespace

int channel_affine(const __nv_bfloat16* x, __nv_bfloat16* y, size_t npix, int C, int ldx, int ldy, const float* scale,
                   const float* shift, cudaStream_t st) {
  WC_REQUIRE(C % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0, "channel_affine: channel counts must be multiples of 8");
  ProfScope prof(kProfGroupNorm, st, 4.0 * npix * C);
  launch_k(channel_affine_kernel, blocks_for(npix * (C / 8)), 256, 0, st, x, y, npix, C, ldx, ldy, scale, shift);
  WC_LAUNCH_CHECK();
  return 0;
}
int layernorm_rows(const __nv_bfloat16* x, __nv_bfloat16* y, size_t rows, int C, int ldx, int ldy, const float* gamma,
                   const float* beta, float eps, cudaStream_t st) {
  WC_REQUIRE(C <= 256, "layernorm_rows supports C <= 256");
  ProfScope prof(kProfGroupNorm, st, 4.0 * rows * C);
  launch_k(layernorm_kernel, static_cast<int>((rows * 32 + 255) / 256), 256, 0, st, x, y, rows, C, ldx, ldy, gamma, beta, eps);
  WC_LAUNCH_CHECK();
  return 0;
}
int avgpool2(const __nv_bfloat16* x, __nv_bfloat16* y, int B, int Ho, int Wo, int C, int ldx, int ldy, cudaStream_t st) {
  WC_REQUIRE(C % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0, "avgpool2: channel counts must be multiples of 8");
  ProfScope prof(kProfOther, st, 2.5 * B * Ho * Wo * 4.0 * C);
  launch_k(avgpool2_kernel, blocks_for(static_cast<size_t>(B) * Ho * Wo * (C / 8)), 256, 0, st, x, y, B, Ho, Wo, C, ldx, ldy);
  WC_LAUNCH_CHECK();
  return 0;
}
int embed_broadcast(const float* t, __nv_bfloat16* y, int B, int HW, int ldy, cudaStream_t st) {
  ProfScope prof(kProfOther, st, 64.0 * B * HW);
  launch_k(embed_broadcast_kernel, dim3(64, B), 256, 0, st, t, y, HW, ldy);
  WC_LAUNCH_CHECK();
  return 0;
}

}  // namespace wc

struct wc_legacy_unet {
  wc::ParamTable params;
  std::unordered_map<std::string, int64_t> numels;
  std::unique_ptr<wc::DeviceArena> arena;
  struct Geom {
    int B, S;
    bool operator==(const Geom& o) const { return B == o.B && S == o.S; }
  } geom{};
  void* ws = nullptr;
  size_t ws_bytes = 0;
  wc::OpList ops;
  double flops = 0;
  void reset_plan() { ops.clear(); flops = 0; }
  const float* x_in = nullptr;
  const float* t_in = nullptr;
  float* y_out = nullptr;
};

namespace wc {
namespace {

struct LBuilder : PlanBuilder<wc_legacy_unet> {
  using PlanBuilder::PlanBuilder;

  void push(std::function<int(cudaStream_t)> f) {
    if (!dry) net->ops.push_back(std::move(f));
  }

  void conv(const Act& x, const std::string& wname, int cout, int K, const float* bias, int actf, const Act* res, const Act* x2,
            const std::string& w2name, const Act& out, int cin_override = 0) {
    if (dry) return;
    WeightSrc w; w.w = P(wname); w.d0 = cout; w.d1 = cin_override ? cin_override : x.C; w.KH = w.KW = K;
    WeightSrc w2;
    if (x2) { w2.w = P(w2name); w2.d0 = cout; w2.d1 = x2->C; }
    if (err) return;
    ConvGeom g; g.K = K; g.stride = 1; g.pad = (K - 1) / 2; g.dil = 1;
    Epilogue ep; ep.bias = bias; ep.res = res; ep.act = actf;
    OutSpec os; os.mode = kOutNHWC; os.out = out;
    auto op = std::make_shared<ConvOp>();
    if (int e = build_conv(op.get(), arena, x, w, g, cout, x2, x2 ? &w2 : nullptr, ep, os, st)) { err = e; return; }
    net->flops += op->flops;
    push([op](cudaStream_t s) { return op->run(s); });
  }

  // ResidualBlock (old_modules.py:126-160): BN(eval) -> conv3x3 -> SiLU -> conv3x3, + (conv1x1(x) | x)
  void resblock(const Act& x, int cout, const std::string& p, bool residual, const Act& out) {
    const int C = x.C;
    Act t1 = act(x.H, x.W, C), t2 = act(x.H, x.W, cout);
    float *sc = nullptr, *sh = nullptr;
    if (!dry) {
      sc = static_cast<float*>(arena->alloc(C * sizeof(float)));
      sh = static_cast<float*>(arena->alloc(C * sizeof(float)));
      const float *g = P(p + ".double_conv.0.weight"), *b = P(p + ".double_conv.0.bias"), *m = P(p + ".double_conv.0.running_mean"),
                  *v = P(p + ".double_conv.0.running_var");
      if (!sc || !sh || err) { if (!err) err = 1; return; }
      if (int e = bn_fold(g, b, m, v, 1e-5f, sc, sh, C, C, st)) { err = e; return; }
    }
    push([=](cudaStream_t s) { return channel_affine(x.ptr, t1.ptr, x.pixels(), C, x.ld, t1.ld, sc, sh, s); });
    conv(t1, p + ".double_conv.1.weight", cout, 3, nullptr, 2 /*SiLU*/, nullptr, nullptr, "", t2);
    if (residual) {
      conv(t2, p + ".double_conv.3.weight", cout, 3, nullptr, 0, nullptr, &x, p + ".res.weight", out);
    } else {
      if (C != cout && !err) err = fail("internal: identity residual needs equal channel counts");
      conv(t2, p + ".double_conv.3.weight", cout, 3, nullptr, 0, &x, nullptr, "", out);
    }
  }

  // SelfAttention (old_modules.py:73-94) on the [B, s*s, C] token view of an NHWC map
  Act attention(const Act& x, const std::string& p) {
    const int C = x.C, ntok = x.H * x.W, heads = 4;
    int Cp = C;
    if (!dry) {
      auto it = net->numels.find(p + ".mha.in_proj_weight");
      if (it == net->numels.end()) { if (!err) err = fail("missing parameter '" + p + ".mha.in_proj_weight'"); return x; }
      Cp = static_cast<int>(it->second / (3 * static_cast<int64_t>(C)));
    } else {
      const int hd = C / heads;
      Cp = heads * (hd <= 16 ? 16 : hd <= 32 ? 32 : hd <= 64 ? 64 : hd <= 128 ? 128 : 192);
    }
    const int hdp = Cp / heads;
    const size_t rows = static_cast<size_t>(B) * ntok;
    Act a = act(x.H, x.W, C);
    const float *g1 = P(p + ".ln.weight"), *b1 = P(p + ".ln.bias");
    push([=](cudaStream_t s) { return layernorm_rows(x.ptr, a.ptr, rows, C, x.ld, a.ld, g1, b1, 1e-5f, s); });
    auto* q = static_cast<__nv_bfloat16*>(bump.take(rows * Cp * 2));
    auto* k = static_cast<__nv_bfloat16*>(bump.take(rows * Cp * 2));
    auto* vt = static_cast<__nv_bfloat16*>(bump.take(rows * Cp * 2));
    Act o = act(x.H, x.W, Cp), av = act(x.H, x.W, C), f = act(x.H, x.W, C), gl = act(x.H, x.W, C), out = act(x.H, x.W, C);
    if (dry) return out;
    {
      WeightSrc w; w.w = P(p + ".mha.in_proj_weight"); w.d0 = 3 * Cp; w.d1 = C;
      ConvGeom g; g.K = 1; g.stride = 1; g.pad = 0; g.dil = 1;
      Epilogue ep; ep.bias = P(p + ".mha.in_proj_bias");
      OutSpec os; os.mode = kOutQKV; os.q = q; os.k = k; os.vt = vt; os.heads = heads; os.hd = hdp;
      if (err) return out;
      auto op = std::make_shared<ConvOp>();
      if (int e = build_conv(op.get(), arena, a, w, g, 3 * Cp, nullptr, nullptr, ep, os, st)) { err = e; return out; }
      net->flops += op->flops;
      push([op](cudaStream_t s) { return op->run(s); });
    }
    const float scale = 1.f / sqrtf(static_cast<float>(C / heads));
    const int Bc = B;
    net->flops += attention_flops(B, heads, ntok, C / heads);
    push([=](cudaStream_t s) { return attention_forward(q, k, vt, o.ptr, Bc, heads, ntok, hdp, o.ld, s, nullptr, scale); });
    conv(o, p + ".mha.out_proj.weight", C, 1, P(p + ".mha.out_proj.bias"), 0, &x, nullptr, "", av);
    const float *g2 = P(p + ".ff_self.0.weight"), *b2 = P(p + ".ff_self.0.bias");
    push([=](cudaStream_t s) { return layernorm_rows(av.ptr, f.ptr, rows, C, av.ld, f.ld, g2, b2, 1e-5f, s); });
    conv(f, p + ".ff_self.1.weight", C, 1, P(p + ".ff_self.1.bias"), 3 /*GELU*/, nullptr, nullptr, "", gl);
    conv(gl, p + ".ff_self.3.weight", C, 1, P(p + ".ff_self.3.bias"), 0, &av, nullptr, "", out);
    return out;
  }
};

int build(const wc_legacy_unet&, const wc_legacy_unet::Geom& geo, wc_legacy_unet* net, cudaStream_t st, size_t* need) {
  const int B = geo.B, S = geo.S;
  LBuilder b(net, B, st);
  const bool dry = b.dry;
  const int depth = 3;
  struct Level { const char* down; const char* up; int cin_d, cout_d, cin_u, cout_u; };
  // DownBlock(cin_d, cout_d) at size S >> l pairs with UpBlock(cin_u, cout_u, skip = cout_d)  (old_modules.py:252-275)
  const Level lv[4] = {{"down1", "up4", 64, 32, 64, 32}, {"down2", "up3", 32, 64, 96, 64}, {"down3", "up2", 64, 96, 128, 96},
                       {"down4", "up1", 96, 128, 256, 128}};
  // concat buffers of the up path: cat[l][k] = [x_k | skip], k = 0 takes the up-sampled input, k = 1, 2 the previous block
  Act cat[4][3];
  for (int l = 0; l < 4; ++l)
    for (int k = 0; k < depth; ++k) {
      const int cx = (k == 0) ? lv[l].cin_u : lv[l].cout_u;
      cat[l][k] = b.act(S >> l, S >> l, cx + lv[l].cout_d);
    }
  // ---- pre_conv + embedding (forward :311-317)
  Act x0 = b.act(S, S, 64);
  if (!dry) {
    const float* w = b.P("pre_conv.weight");
    if (b.err) return b.err;
    wc_legacy_unet* n = net;
    b.push([=](cudaStream_t s) {
      if (int e = conv_small_cin(n->x_in, w, nullptr, nullptr, nullptr, x0.ptr, B, 3, S, S, 32, 3, 1, 1, x0.ld, 0, s)) return e;
      return embed_broadcast(n->t_in, x0.ptr + 32, B, S * S, x0.ld, s);
    });
    net->flops += 2.0 * B * S * S * 27.0 * 32;
  }
  Act cur = x0;
  // ---- down path (:321-333)
  for (int l = 0; l < 4; ++l) {
    const int s = S >> l;
    if (l == 2) cur = b.attention(cur, "attn_down3");
    if (l == 3) cur = b.attention(cur, "attn_down4");
    for (int i = 0; i < depth; ++i) {
      const int k = depth - 1 - i;  // skip i is popped by up-block layer k
      const int cx = (k == 0) ? lv[l].cin_u : lv[l].cout_u;
      Act dest = slice_act(cat[l][k], cx, lv[l].cout_d);
      b.resblock(cur, lv[l].cout_d, std::string(lv[l].down) + ".residual_blocks." + std::to_string(i), i == 0, dest);
      cur = dest;
    }
    Act pooled = b.act(s / 2, s / 2, lv[l].cout_d);
    const Act src = cur;
    b.push([=](cudaStream_t st2) { return avgpool2(src.ptr, pooled.ptr, B, s / 2, s / 2, src.C, src.ld, pooled.ld, st2); });
    cur = pooled;
    if (b.err) return b.err;
  }
  // ---- bottleneck (:336-340)
  {
    Act t = b.act(cur.H, cur.W, 256);
    b.resblock(cur, 256, "bottleneck1", true, t);
    t = b.attention(t, "attn_bottleneck");
    Act u = b.act(cur.H, cur.W, 256);
    b.resblock(t, 256, "bottleneck2", true, u);
    cur = u;
  }
  // ---- up path (:343-355)
  for (int l = 3; l >= 0; --l) {
    const int s = S >> l;
    Act first = slice_act(cat[l][0], 0, lv[l].cin_u);
    const Act src = cur;
    if (src.C != lv[l].cin_u) return fail("internal: up block input channel mismatch");
    b.push([=](cudaStream_t st2) { return bilinear_fwd(src.ptr, first.ptr, B, s / 2, s / 2, s, s, src.C, src.ld, first.ld, st2); });
    for (int k = 0; k < depth; ++k) {
      Act dest = (k + 1 < depth) ? slice_act(cat[l][k + 1], 0, lv[l].cout_u) : b.act(s, s, lv[l].cout_u);
      b.resblock(cat[l][k], lv[l].cout_u, std::string(lv[l].up) + ".residual_blocks." + std::to_string(k), true, dest);
      cur = dest;
    }
    if (l == 3) cur = b.attention(cur, "attn_up1");
    if (l == 2) cur = b.attention(cur, "attn_up2");
    if (b.err) return b.err;
  }
  // ---- output conv (:357), NHWC bf16 -> NCHW fp32
  if (!dry) {
    const float* w = b.P("output.weight");
    if (b.err) return b.err;
    wc_legacy_unet* n = net;
    const Act fin = cur;
    b.push([=](cudaStream_t s) { return conv_small_cout(fin.ptr, w, nullptr, n->y_out, B, S, S, fin.C, 3, 3, fin.ld, 0, s); });
    net->flops += 2.0 * B * S * S * 9.0 * 32 * 3;
  }
  return b.finish("legacy UNet", need);
}

}  // namespace
}  // namespace wc

using namespace wc;

extern "C" {

int wc_legacy_unet_create(wc_legacy_unet** out, int n_params, const char* const* names, const float* const* ptrs,
                          const int64_t* numels) {
  WC_REQUIRE(out && names && ptrs && numels, "null argument");
  auto net = std::make_unique<wc_legacy_unet>();
  for (int i = 0; i < n_params; ++i) {
    net->params.ptr[names[i]] = ptrs[i];
    net->numels[names[i]] = numels[i];
  }
  *out = net.release();
  return 0;
}
void wc_legacy_unet_destroy(wc_legacy_unet* net) { delete net; }

size_t wc_legacy_unet_workspace_bytes(wc_legacy_unet* net, int batch, int size) {
  return plan_workspace_bytes(*net, {batch, size}, build);
}

int wc_legacy_unet_forward(wc_legacy_unet* net, const float* x, const float* t, float* out, int batch, int size, void* workspace,
                           size_t workspace_bytes, void* stream) {
  WC_REQUIRE(net && x && t && out && workspace, "null argument");
  WC_REQUIRE(size == 128, "the legacy UNet's attention blocks are built for 128 x 128 inputs (old_modules.py:256-270)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = bind(net, {batch, size}, workspace, workspace_bytes, st, build)) return e;
  net->x_in = x; net->t_in = t; net->y_out = out;
  return run_ops(net->ops, st);
}
double wc_legacy_unet_flops(const wc_legacy_unet* net) { return net ? net->flops : 0.0; }
int wc_legacy_unet_launches(const wc_legacy_unet* net) { return net ? static_cast<int>(net->ops.size()) : 0; }

}  // extern "C"
