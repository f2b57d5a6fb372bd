// Swift-SRGAN generator forward as a static launch plan (reference: srgan_model/models.py:5-92,
// srgan_model/inference.py:35-39).  Depthwise 3x3 + pointwise pairs are composed into dense 3x3 convolutions
// (W[o,c,ky,kx] = pw[o,c]*dw[c,ky,kx], eval BatchNorm folded) and run on the tcgen05 implicit-GEMM path with
// PReLU / residual epilogues; PixelShuffle(2) is four output-phase convolutions writing straight into the 2x
// larger tensor; the first (3-channel, 9x9) and last (depthwise 9x9 + 64->3 + tanh) layers are CUDA-core kernels
// that also convert from / to the reference's NCHW fp32 layout.
// wc_srgan_forward_saved / wc_srgan_backward_seeded: the same forward on a with-grad plan, which also keeps what the input
// gradient needs, and a data-gradient backward seeded with dL/dy (torch autograd in srgan_model/models.py).  The parameters are
// constants: no weight gradient is computed.
#include "plan.cuh"
#include "../../include/wc_b200.h"

namespace wc {
int conv_small_cin(const float* x, const float* w, const float* bias, const float* scale, const float* shift,
                   __nv_bfloat16* y, int B, int Cin, int H, int W, int Cout, int K, int stride, int pad, int ldy,
                   int relu, cudaStream_t st, const float* prelu = nullptr);
int bn_fold(const float* g, const float* b, const float* mean, const float* var, float eps, float* scale, float* shift,
            int n, int n_pad, cudaStream_t st);
int compose_sep(const float* dw, const float* pw, const float* dwb, const float* pwb, float* w, float* bias, int Co, int Ci,
                int KK, cudaStream_t st);
int srgan_initial(const float* x, const float* dw, const float* dwb, const float* pw, const float* pwb, const float* slope,
                  __nv_bfloat16* y, int B, int H, int W, int ldy, cudaStream_t st);
int srgan_final(const __nv_bfloat16* x, const float* dw, const float* dwb, const float* pw, const float* pwb, float* y, int B,
                int H, int W, int ldx, cudaStream_t st);
int phase_major_rows(const float* src, float* dst, int cb, int len, int rep_src, cudaStream_t st);
int srgan_final_compose(const float* dw, const float* dwb, const float* pw, const float* pwb, float* wq, float* bias3, cudaStream_t st);
int srgan_final_combine(const float* t, const float* bias3, float* y, int B, int H, int W, cudaStream_t st);
int conv_small_cout(const __nv_bfloat16* x, const float* w, const float* bias, float* y, int B, int H, int W, int Cin,
                    int Cout, int K, int ldx, int tanh_out, cudaStream_t st);
int srgan_tanh_bwd(const float* dy, const float* y, float* dz, size_t n, cudaStream_t st);
int flip_transpose_kk(const float* w, float* wt, int Co, int Ci, int KK, cudaStream_t st);
int prelu_bwd(__nv_bfloat16* d, const __nv_bfloat16* add, const __nv_bfloat16* pre, const float* slope, size_t npix, int C, int ldd,
              int lda, int ldp, cudaStream_t st);
int shuffle_prelu_bwd(const __nv_bfloat16* dup, const __nv_bfloat16* pre, const float* slope, __nv_bfloat16* dconv, int B, int h, int w,
                      int C, cudaStream_t st);
int fill_f32(float* p, float v, int n, cudaStream_t st);
}  // namespace wc

struct wc_srgan {
  int num_blocks = 16, upscale = 4, nc = 64;
  wc::ParamTable params;
  std::unique_ptr<wc::DeviceArena> arena;
  int B = 0, H = 0, W = 0, with_grad = 0;
  void* ws = nullptr;
  size_t ws_bytes = 0;
  wc::OpList ops, bwd_ops;   // bwd_ops: with-grad plans only
  double flops = 0;
  size_t ws_needed = 0;
  int saved_fwd = 0;   // the last call on this handle was wc_srgan_forward_saved
  const float* x_in = nullptr;
  float* y_out = nullptr;
  const float* dy_in = nullptr;
  float* dx_out = nullptr;
};

namespace wc {
namespace {

int build(wc_srgan* net, bool dry, void* ws, size_t ws_bytes, cudaStream_t st) {
  const int B = net->B, H = net->H, W = net->W, NCH = net->nc;
  Bump bump = dry ? Bump::dry() : Bump(ws, ws_bytes);
  DeviceArena* arena = net->arena.get();
  int err = 0;
  auto P = [&](const std::string& n) { return net->params.get(n, &err); };
  auto Popt = [&](const std::string& n) -> const float* {
    auto it = net->params.ptr.find(n);
    return it == net->params.ptr.end() ? nullptr : it->second;
  };
  auto push = [&](std::function<int(cudaStream_t)> f) { if (!dry) net->ops.push_back(std::move(f)); };
  auto pushb = [&](std::function<int(cudaStream_t)> f) { if (!dry) net->bwd_ops.push_back(std::move(f)); };
  const bool grad = net->with_grad;
  auto fa = [&](size_t n) { return static_cast<float*>(arena->alloc(n * sizeof(float))); };

  // composed dense weights of a SeperableConv2d (+ optional folded BN): returns (weights, bias/shift, scale)
  struct Composed { float* w; float* bias; float* scale; };
  auto compose = [&](const std::string& p, int ci, int co, int K, const std::string& bn) -> Composed {
    Composed c{nullptr, nullptr, nullptr};
    c.w = fa(static_cast<size_t>(co) * ci * K * K);
    c.bias = fa(co);
    const float *dw = P(p + ".depthwise.weight"), *pw = P(p + ".pointwise.weight");
    const float *dwb = Popt(p + ".depthwise.bias"), *pwb = Popt(p + ".pointwise.bias");
    if (!c.w || !c.bias || err) { if (!err) err = 1; return c; }
    if (int e = compose_sep(dw, pw, dwb, pwb, c.w, c.bias, co, ci, K * K, st)) { err = e; return c; }
    if (!bn.empty()) {   // conv has no bias when followed by BN (models.py:30): bias := BN shift, weights scaled
      c.scale = fa(co);
      float* shift = fa(co);
      const float *g = P(bn + ".weight"), *b = P(bn + ".bias"), *m = P(bn + ".running_mean"), *v = P(bn + ".running_var");
      if (!c.scale || !shift || err) { if (!err) err = 1; return c; }
      if (int e = bn_fold(g, b, m, v, 1e-5f, c.scale, shift, co, co, st)) { err = e; return c; }
      c.bias = shift;
    }
    return c;
  };
  auto conv3 = [&](const Act& x, const Composed& c, int co, const float* prelu, const Act* res, const Act& out) {
    if (dry || err) return;
    WeightSrc w; w.w = c.w; w.d0 = co; w.d1 = x.C; w.KH = w.KW = 3; w.scale = c.scale;
    ConvGeom g; g.K = 3; g.pad = 1;
    Epilogue ep; ep.bias = c.bias; ep.prelu = prelu; ep.res = res;
    OutSpec os; os.mode = kOutNHWC; os.out = out;
    auto op = std::make_shared<ConvOp>();
    if (int e = build_conv(op.get(), arena, x, w, g, co, nullptr, nullptr, ep, os, st)) { err = e; return; }
    // algorithmic FLOPs = the reference's separable form (depthwise 3x3 + pointwise), not the composed dense conv
    op->flops = 2.0 * x.pixels() * (9.0 * x.C + static_cast<double>(x.C) * co);
    for (auto& pl : op->plans) pl.flops = op->flops / op->plans.size();
    net->flops += op->flops;
    net->ops.push_back([op](cudaStream_t s) { return op->run(s); });
  };
  // data gradient of conv3 (stride 1, 'same'): dx = conv(dz, flipped W^T) (+ res), the folded BN scale applied to W's rows
  auto dgrad3 = [&](const Act& dz, const Composed& c, int ci, const Act* res, const Act& dx) {
    if (dry || err) return;
    WeightSrc w; w.w = c.w; w.d0 = dz.C; w.d1 = ci; w.KH = w.KW = 3; w.transpose = 1; w.flip = 1; w.scale = c.scale;
    ConvGeom g; g.K = 3; g.pad = 1;
    Epilogue ep; ep.res = res;
    OutSpec os; os.mode = kOutNHWC; os.out = dx;
    auto op = std::make_shared<ConvOp>();
    if (int e = build_conv(op.get(), arena, dz, w, g, ci, nullptr, nullptr, ep, os, st)) { err = e; return; }
    net->bwd_ops.push_back([op](cudaStream_t s) { return op->run(s); });
  };

  // ---- initial: SeperableConv2d(3->64, k9) + PReLU, NCHW fp32 in
  Act initial = make_act(bump, B, H, W, NCH);
  // with-grad plans keep the pre-activation of every PReLU: a bf16 copy from a second launch of the same convolution without
  // the PReLU (same accumulators, so the same sign); the PReLU output alone cannot tell the sign when a slope is <= 0
  Act pre_initial = grad ? make_act(bump, B, H, W, NCH) : Act{};
  float* w_initial_t = nullptr;   // [3][64][9][9]: the initial layer's data gradient as a 64 -> 3 convolution
  const float* slope_initial = nullptr;
  if (!dry) {
    const float *dw = P("initial.cnn.depthwise.weight"), *dwb = Popt("initial.cnn.depthwise.bias");
    const float *pw = P("initial.cnn.pointwise.weight"), *pwb = Popt("initial.cnn.pointwise.bias");
    const float* slope = P("initial.act.weight");
    if (err) return err;
    WC_REQUIRE(NCH == 64, "srgan_initial is written for 64 hidden channels");
    wc_srgan* n = net;
    push([=](cudaStream_t s) { return srgan_initial(n->x_in, dw, dwb, pw, pwb, slope, initial.ptr, B, H, W, initial.ld, s); });
    net->flops += 2.0 * B * H * W * (243.0 + 3.0 * NCH);   // separable, as the reference runs it
    if (grad) {
      float* ones = fa(NCH);
      float* w0 = fa(static_cast<size_t>(NCH) * 3 * 81);
      w_initial_t = fa(static_cast<size_t>(NCH) * 3 * 81);
      if (!ones || !w0 || !w_initial_t) return 1;
      if (int e = fill_f32(ones, 1.f, NCH, st)) return e;
      if (int e = compose_sep(dw, pw, nullptr, nullptr, w0, nullptr, NCH, 3, 81, st)) return e;
      if (int e = flip_transpose_kk(w0, w_initial_t, NCH, 3, 81, st)) return e;
      slope_initial = slope;
      push([=](cudaStream_t s) { return srgan_initial(n->x_in, dw, dwb, pw, pwb, ones, pre_initial.ptr, B, H, W, pre_initial.ld, s); });
    }
  }
  // ---- residual trunk
  struct BlockRec { Composed c1, c2; const float* slope; Act pre1; };
  std::vector<BlockRec> blocks(net->num_blocks);
  Act cur = initial;
  for (int i = 0; i < net->num_blocks; ++i) {
    const std::string p = "residual." + std::to_string(i);
    Act t1 = make_act(bump, B, H, W, NCH), out = make_act(bump, B, H, W, NCH);
    if (grad) blocks[i].pre1 = make_act(bump, B, H, W, NCH);
    if (!dry) {
      Composed c1 = compose(p + ".block1.cnn", NCH, NCH, 3, p + ".block1.bn");
      Composed c2 = compose(p + ".block2.cnn", NCH, NCH, 3, p + ".block2.bn");
      const float* slope = P(p + ".block1.act.weight");
      if (err) return err;
      conv3(cur, c1, NCH, slope, nullptr, t1);
      if (grad) conv3(cur, c1, NCH, nullptr, nullptr, blocks[i].pre1);
      conv3(t1, c2, NCH, nullptr, &cur, out);
      blocks[i].c1 = c1; blocks[i].c2 = c2; blocks[i].slope = slope;
    }
    cur = out;
  }
  Act trunk = make_act(bump, B, H, W, NCH);
  Composed c_convblock{nullptr, nullptr, nullptr};
  if (!dry) {
    c_convblock = compose("convblock.cnn", NCH, NCH, 3, "convblock.bn");
    if (err) return err;
    conv3(cur, c_convblock, NCH, nullptr, &initial, trunk);
  }
  cur = trunk;
  // ---- upsamplers: SeperableConv2d(64->256, k3) + PixelShuffle(2) + PReLU(64)
  struct UpRec { Composed c; const float* slope; Act pre; };
  std::vector<UpRec> ups(net->upscale / 2);
  int h = H, w = W;
  for (int u = 0; u < net->upscale / 2; ++u) {
    const std::string p = "upsampler." + std::to_string(u);
    Act up = make_act(bump, B, 2 * h, 2 * w, NCH);
    if (grad) ups[u].pre = make_act(bump, B, 2 * h, 2 * w, NCH);
    if (!dry) {
      Composed c = compose(p + ".conv", NCH, NCH * 4, 3, "");
      const float* slope = P(p + ".act.weight");
      if (err) return err;
      ups[u].c = c; ups[u].slope = slope;
      // ONE launch for the four PixelShuffle phases (out[c, 2y+i, 2x+j] = conv[4c + 2i + j, y, x]): weight rows, bias and PReLU
      // slopes re-ordered phase-major (row q*64 + c = conv channel 4c + q), N tile 128 so that the row-segment mode applies; every
      // 32-channel chunk is stored through the strided map of its phase
      float* wpm = fa(static_cast<size_t>(NCH) * 4 * NCH * 9);
      float* bpm = fa(NCH * 4);
      float* spm = fa(NCH * 4);
      if (!wpm || !bpm || !spm) return 1;
      if (int e = phase_major_rows(c.w, wpm, NCH, NCH * 9, 0, st)) return e;
      if (int e = phase_major_rows(c.bias, bpm, NCH, 1, 0, st)) return e;
      if (int e = phase_major_rows(slope, spm, NCH, 1, 1, st)) return e;
      for (int pass = 0; pass < (grad ? 2 : 1); ++pass) {   // pass 1 (with-grad plans): the pre-activation, without the PReLU
        WeightSrc ws_; ws_.w = wpm; ws_.d0 = NCH * 4; ws_.d1 = NCH; ws_.KH = ws_.KW = 3;
        ConvGeom g; g.K = 3; g.pad = 1;
        Epilogue ep; ep.bias = bpm; ep.prelu = pass ? nullptr : spm;
        OutSpec os; os.mode = kOutNHWC; os.out = pass ? ups[u].pre : up; os.up = 2; os.phases = 4; os.bn_max = 128;
        auto op = std::make_shared<ConvOp>();
        if (int e = build_conv(op.get(), arena, cur, ws_, g, NCH * 4, nullptr, nullptr, ep, os, st)) return e;
        op->flops = 2.0 * cur.pixels() * (9.0 * NCH + static_cast<double>(NCH) * NCH * 4);
        for (auto& pl : op->plans) pl.flops = op->flops / op->plans.size();
        net->flops += op->flops;
        net->ops.push_back([op](cudaStream_t s) { return op->run(s); });
      }
    }
    cur = up; h *= 2; w *= 2;
  }
  // ---- final: depthwise 9x9 + pointwise 64->3 + (tanh + 1)/2, NCHW fp32 out
  // On the tensor core where the output width is a multiple of 4: a 1x9 horizontal convolution with N = (kernel row, output) = 27
  // columns into fp32 planes (igemm), then the vertical shift-add + bias + tanh (seg_kernels.cu: srgan_final_combine).  Otherwise
  // (upscale 2 with an odd latent width) the CUDA-core kernel srgan_final.
  const bool tc = NCH == 64 && w % 4 == 0;
  float* tplanes = tc ? static_cast<float*>(bump.take(static_cast<size_t>(B) * 27 * h * w * sizeof(float))) : nullptr;
  if (!dry) {
    const float *dw = P("final_conv.depthwise.weight"), *dwb = Popt("final_conv.depthwise.bias");
    const float *pw = P("final_conv.pointwise.weight"), *pwb = Popt("final_conv.pointwise.bias");
    if (err) return err;
    wc_srgan* n = net;
    const Act last = cur;
    const int hh = h, ww = w;
    const double fl = 2.0 * B * hh * ww * (81.0 * NCH + 3.0 * NCH);   // algorithmic: the reference's separable form
    if (tc) {
      float* wq = fa(32 * 64 * 9);
      float* bias3 = fa(4);
      if (!wq || !bias3) return 1;
      if (int e = srgan_final_compose(dw, dwb, pw, pwb, wq, bias3, st)) return e;
      WeightSrc ws_; ws_.w = wq; ws_.d0 = 32; ws_.d1 = NCH; ws_.KH = 1; ws_.KW = 9;
      Epilogue ep;
      OutSpec os; os.mode = kOutNCHWf32; os.out_f32 = tplanes; os.n_store = 27;
      auto op = std::make_shared<ConvOp>();
      if (int e = build_conv_hrow(op.get(), arena, last, ws_, 32, ep, os, st)) return e;
      op->flops = fl;
      for (auto& pl : op->plans) pl.flops = fl / op->plans.size();
      net->ops.push_back([op](cudaStream_t s) { return op->run(s); });
      push([=](cudaStream_t s) { return srgan_final_combine(tplanes, bias3, n->y_out, B, hh, ww, s); });
    } else {
      push([=](cudaStream_t s) { return srgan_final(last.ptr, dw, dwb, pw, pwb, n->y_out, B, hh, ww, last.ld, s); });
    }
    net->flops += fl;
  }
  if (grad) {
    // =================================================== backward (data gradients only), in plan order reversed
    const int uh = h, uw = w;
    const size_t ny = static_cast<size_t>(B) * 3 * uh * uw;
    float* y_saved = static_cast<float*>(bump.take(ny * sizeof(float)));   // y, for the tanh derivative
    float* dz = static_cast<float*>(bump.take(ny * sizeof(float)));
    Act dcur = make_act(bump, B, uh, uw, NCH);
    if (!dry) {
      wc_srgan* n = net;
      push([=](cudaStream_t s) {
        return cudaMemcpyAsync(y_saved, n->y_out, ny * sizeof(float), cudaMemcpyDeviceToDevice, s) == cudaSuccess ? 0 : fail("memcpy failed");
      });
      // final layer: d(pre-tanh), then the composed 64 -> 3 9x9 convolution's data gradient as a 3 -> 64 convolution
      const float *dw = P("final_conv.depthwise.weight"), *pw = P("final_conv.pointwise.weight");
      float* wf = fa(static_cast<size_t>(3) * NCH * 81);
      float* wf_t = fa(static_cast<size_t>(3) * NCH * 81);
      if (err) return err;
      if (!wf || !wf_t) return 1;
      if (int e = compose_sep(dw, pw, nullptr, nullptr, wf, nullptr, 3, NCH, 81, st)) return e;
      if (int e = flip_transpose_kk(wf, wf_t, 3, NCH, 81, st)) return e;
      pushb([=](cudaStream_t s) {
        if (int e = srgan_tanh_bwd(n->dy_in, y_saved, dz, ny, s)) return e;
        return conv_small_cin(dz, wf_t, nullptr, nullptr, nullptr, dcur.ptr, B, 3, uh, uw, NCH, 9, 1, 4, dcur.ld, 0, s);
      });
    }
    // up-samplers: PReLU + PixelShuffle backward into the conv's 256 channels (4c + q), then the 64 -> 256 conv's data gradient
    for (int u = net->upscale / 2 - 1; u >= 0; --u) {
      const int hu = h / 2, wu = w / 2;
      Act dconv = make_act(bump, B, hu, wu, 4 * NCH), dx = make_act(bump, B, hu, wu, NCH);
      if (!dry) {
        const Act dup = dcur, pre = ups[u].pre;
        const float* slope = ups[u].slope;
        pushb([=](cudaStream_t s) { return shuffle_prelu_bwd(dup.ptr, pre.ptr, slope, dconv.ptr, B, hu, wu, NCH, s); });
        dgrad3(dconv, ups[u].c, NCH, nullptr, dx);
      }
      dcur = dx; h = hu; w = wu;
    }
    // trunk: d trunk reaches convblock and, through its skip, the initial layer; residual blocks in reverse
    const Act dtrunk = dcur;
    Act gbuf[2] = {make_act(bump, B, H, W, NCH), make_act(bump, B, H, W, NCH)};
    Act dt = make_act(bump, B, H, W, NCH);
    int gi = 0;
    dgrad3(dtrunk, c_convblock, NCH, nullptr, gbuf[gi]);
    for (int i = net->num_blocks - 1; i >= 0; --i) {
      const Act g = gbuf[gi], gn = gbuf[gi ^ 1], pre = blocks[i].pre1;
      dgrad3(g, blocks[i].c2, NCH, nullptr, dt);
      if (!dry) {
        const float* slope = blocks[i].slope;
        pushb([=](cudaStream_t s) { return prelu_bwd(dt.ptr, nullptr, pre.ptr, slope, dt.pixels(), NCH, dt.ld, 0, pre.ld, s); });
      }
      dgrad3(dt, blocks[i].c1, NCH, &g, gn);   // + the identity path of the residual
      gi ^= 1;
    }
    // initial: PReLU backward of (trunk path + skip), then the composed 3 -> 64 9x9 convolution's data gradient into NCHW fp32 dx
    if (!dry) {
      const Act g = gbuf[gi], pre = pre_initial;
      const float *slope = slope_initial, *wt = w_initial_t;
      wc_srgan* n = net;
      pushb([=](cudaStream_t s) {
        if (int e = prelu_bwd(g.ptr, dtrunk.ptr, pre.ptr, slope, g.pixels(), NCH, g.ld, dtrunk.ld, pre.ld, s)) return e;
        return conv_small_cout(g.ptr, wt, nullptr, n->dx_out, B, H, W, NCH, 3, 9, g.ld, 0, s);
      });
    }
  }
  if (dry) net->ws_needed = bump.used() + 4096;
  else if (bump.overflow()) return fail("SRGAN workspace too small");
  return err;
}

// (Re)builds the plan when the geometry, the gradient mode or the workspace differ from the current binding.
int bind_plan(wc_srgan* net, int batch, int h, int w, int with_grad, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (net->B == batch && net->H == h && net->W == w && net->with_grad == with_grad && net->ws == workspace &&
      net->ws_bytes == workspace_bytes)
    return 0;
  net->ops.clear(); net->bwd_ops.clear();
  net->arena = std::make_unique<DeviceArena>();
  net->B = batch; net->H = h; net->W = w; net->with_grad = with_grad; net->ws = workspace; net->ws_bytes = workspace_bytes;
  net->flops = 0;
  if (int e = build(net, false, workspace, workspace_bytes, st)) {
    net->B = 0;
    net->ops.clear(); net->bwd_ops.clear();
    return e;
  }
  return 0;
}

size_t workspace_bytes(wc_srgan* net, int batch, int h, int w, int with_grad) {
  const int sB = net->B, sH = net->H, sW = net->W, sg = net->with_grad;
  net->B = batch; net->H = h; net->W = w; net->with_grad = with_grad;
  size_t need = 0;
  if (build(net, true, nullptr, 0, nullptr) == 0) need = net->ws_needed;
  net->B = sB; net->H = sH; net->W = sW; net->with_grad = sg;
  return need;
}

}  // namespace
}  // namespace wc

using namespace wc;

extern "C" {

int wc_srgan_create(wc_srgan** out, int num_blocks, int upscale, int n_params, const char* const* names,
                    const float* const* ptrs, void* stream) {
  (void)stream;
  WC_REQUIRE(out && names && ptrs, "null argument");
  WC_REQUIRE(upscale == 2 || upscale == 4 || upscale == 8, "upscale must be 2, 4 or 8");
  auto net = std::make_unique<wc_srgan>();
  net->num_blocks = num_blocks; net->upscale = upscale;
  for (int i = 0; i < n_params; ++i) net->params.ptr[names[i]] = ptrs[i];
  *out = net.release();
  return 0;
}
void wc_srgan_destroy(wc_srgan* net) { delete net; }
size_t wc_srgan_workspace_bytes(const wc_srgan* net, int batch, int h, int w) {
  return workspace_bytes(const_cast<wc_srgan*>(net), batch, h, w, 0);
}
size_t wc_srgan_grad_workspace_bytes(const wc_srgan* net, int batch, int h, int w) {
  return workspace_bytes(const_cast<wc_srgan*>(net), batch, h, w, 1);
}
int wc_srgan_forward(wc_srgan* net, const float* x, float* y, int batch, int h, int w, void* workspace,
                     size_t workspace_bytes, void* stream) {
  if (net) net->saved_fwd = 0;
  WC_REQUIRE(net && x && y && workspace, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = bind_plan(net, batch, h, w, 0, workspace, workspace_bytes, st)) return e;
  net->x_in = x; net->y_out = y;
  for (auto& op : net->ops)
    if (int e = op(st)) return e;
  return 0;
}
int wc_srgan_forward_saved(wc_srgan* net, const float* x, float* y, int batch, int h, int w, void* workspace,
                           size_t workspace_bytes, void* stream) {
  if (net) net->saved_fwd = 0;
  WC_REQUIRE(net && x && y && workspace, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = bind_plan(net, batch, h, w, 1, workspace, workspace_bytes, st)) return e;
  net->x_in = x; net->y_out = y;
  for (auto& op : net->ops)
    if (int e = op(st)) return e;
  net->saved_fwd = 1;
  return 0;
}
int wc_srgan_backward_seeded(wc_srgan* net, const float* dy, float* dx, void* stream) {
  WC_REQUIRE(net && dy && dx, "null argument");
  WC_REQUIRE(net->saved_fwd && net->with_grad,
             "wc_srgan_backward_seeded: this handle holds no saved forward; the last call on it must be wc_srgan_forward_saved "
             "(any forward in between discards the saved activations, and so does the backward itself)");
  net->saved_fwd = 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  net->dy_in = dy; net->dx_out = dx;
  for (auto& op : net->bwd_ops)
    if (int e = op(st)) return e;
  return 0;
}
double wc_srgan_flops(const wc_srgan* net) { return net ? net->flops : 0.0; }
int wc_srgan_launches(const wc_srgan* net) { return net ? static_cast<int>(net->ops.size()) : 0; }

}  // extern "C"
