// DeepLabV3+ (ResNet-50/101, output stride 16) forward + cross-entropy + INPUT gradient as a static launch plan.
// Reference: seg_model/network/backbone/resnet.py:78-213, _deeplab.py:28-59,111-162, network/utils.py:7-18,
// modeling.py:32-58 and the guidance call seg_model/inference.py:118-152 (forward, argmax, CE(ignore 255),
// loss.backward(), input.grad).  Only the data gradient is computed (the reference also computes every weight
// gradient and throws it away); eval-mode BatchNorm is folded into the preceding convolution; ReLU derivatives
// are applied as masks in the epilogue of the data-gradient convolution that produces each gradient.
// Per-image semantics (SURVEY D6): the loss of image b is the mean over ITS valid pixels.
// wc_seg_forward / wc_seg_backward_seeded split the same plan at the loss head so that any loss computed by the caller can
// seed the data-gradient backward (torch autograd in seg_model/network/modeling.py).
#include "plan.cuh"
#include "../../include/wc_b200.h"

namespace wc {
int conv_small_cin(const float* x, const float* w, const float* bias, const float* scale, const float* shift,
                   __nv_bfloat16* y, int B, int Cin, int H, int W, int Cout, int K, int stride, int pad, int ldy,
                   int relu, cudaStream_t st, const float* prelu = nullptr);
int bn_fold(const float* g, const float* b, const float* mean, const float* var, float eps, float* scale, float* shift,
            int n, int n_pad, cudaStream_t st);
int maxpool_fwd(const __nv_bfloat16* x, __nv_bfloat16* y, uint8_t* idx, int B, int H, int W, int C, cudaStream_t st);
int maxpool_bwd(const __nv_bfloat16* dy, const uint8_t* idx, const __nv_bfloat16* x, __nv_bfloat16* dx, int B, int H,
                int W, int C, cudaStream_t st);
int gap_fwd(const __nv_bfloat16* x, __nv_bfloat16* y, int B, int HW, int C, int ld, cudaStream_t st);
int broadcast_hw(const __nv_bfloat16* v, __nv_bfloat16* y, int B, int HW, int C, int ldy, cudaStream_t st);
int sum_hw(const __nv_bfloat16* y, const __nv_bfloat16* mask, __nv_bfloat16* v, int B, int HW, int C, int ldy, cudaStream_t st);
int gap_bwd_add(const __nv_bfloat16* g, __nv_bfloat16* dx, int B, int HW, int C, int ld, cudaStream_t st);
int bilinear_fwd(const __nv_bfloat16* x, __nv_bfloat16* y, int B, int Hi, int Wi, int Ho, int Wo, int C, int ldx, int ldy,
                 cudaStream_t st);
int bilinear_bwd(const __nv_bfloat16* dy, const __nv_bfloat16* mask, __nv_bfloat16* dx, int B, int Hi, int Wi, int Ho,
                 int Wo, int C, int ldy, int ldm, int ldx, cudaStream_t st);
int seg_loss_grad(const float* logits_lo, const long long* labels, int* n_valid, long long* pred, float* dlogit_hi,
                  float* loss, float* logits_hi, int B, int h, int w, int H, int W, int nc, int ignore, cudaStream_t st);
int seg_loss_head_fused(const float* logits_lo, const long long* labels, int* n_valid, long long* pred, float* loss,
                        __nv_bfloat16* dlo, int B, int h, int w, int H, int W, int nc, int cp, int ldo, int ignore, cudaStream_t st);
int logits_bilinear_bwd(const float* dhi, __nv_bfloat16* dlo, int B, int h, int w, int H, int W, int nc, int cp, int ldo,
                        cudaStream_t st);
int conv1_dgrad(const __nv_bfloat16* dz, const float* w, const float* scale, float* dx, int B, int H, int W, int Cout,
                cudaStream_t st);
int relu_mask_inplace(__nv_bfloat16* d, const __nv_bfloat16* m, size_t npix, int C, int ldd, int ldm, cudaStream_t st);
int conv1_dgrad_weff(const float* w, const float* scale, float* weff, int P, cudaStream_t st);
int conv1_dgrad_pooled(const __nv_bfloat16* dz, const float* weff, float* out, int B, int H, int W, int P, cudaStream_t st);
}  // namespace wc

struct wc_seg {
  int layers[4];
  int num_classes;
  int output_stride = 16;   // 16: layer4 dilated, ASPP rates 6/12/18; 8: layers 3-4 dilated, rates 12/24/36 (modeling.py:34-39)
  wc::ParamTable params;
  std::unique_ptr<wc::DeviceArena> arena;
  int B = 0, H = 0, W = 0, with_grad = 0, grad_pool = 1;
  void* ws = nullptr;
  size_t ws_bytes = 0;
  wc::OpList fwd_ops, bwd_ops;
  double flops_fwd = 0, flops_bwd = 0;
  size_t ws_needed = 0;
  // seam between the network body and the loss head, for wc_seg_forward / wc_seg_backward_seeded: fwd_ops[0, n_body_ops)
  // end at the low-resolution logits; the backward starts from dlo (NHWC bf16, 32 channels; with_grad plans only)
  size_t n_body_ops = 0;
  float* logits_lo = nullptr;
  __nv_bfloat16* dlo = nullptr;
  int saved_fwd = 0;   // the last call was wc_seg_forward(save_for_backward = 1) on the current binding
  // per-call pointers
  const float* x_in = nullptr;
  const long long* labels = nullptr;
  long long* pred = nullptr;
  float* grad_out = nullptr;
  float* loss = nullptr;
  float* logits_hi = nullptr;
};

namespace wc {
namespace {

struct BlockRec {
  std::string p;
  int inplanes, planes, stride, dil;
  bool has_down;
  Act x_in, y1, y2, out;
};

struct SegBuilder {
  wc_seg* net;
  Bump bump;
  DeviceArena* arena;
  cudaStream_t st;
  bool dry;
  int B;
  int err = 0;
  bool in_bwd = false;
  std::unordered_map<std::string, std::pair<float*, float*>> bn;  // prefix -> (scale, shift)

  const float* P(const std::string& n) { return net->params.get(n, &err); }
  void push(std::function<int(cudaStream_t)> f) {
    if (dry) return;
    (in_bwd ? net->bwd_ops : net->fwd_ops).push_back(std::move(f));
  }
  Act act(int H, int W, int C) { return make_act(bump, B, H, W, C); }

  std::pair<float*, float*> bnfold(const std::string& prefix, int C) {
    auto it = bn.find(prefix);
    if (it != bn.end()) return it->second;
    const int cp = (C + 15) / 16 * 16;
    float* sc = static_cast<float*>(arena->alloc(cp * sizeof(float)));
    float* sh = static_cast<float*>(arena->alloc(cp * sizeof(float)));
    const float *g = P(prefix + ".weight"), *b = P(prefix + ".bias"), *m = P(prefix + ".running_mean"), *v = P(prefix + ".running_var");
    if (!sc || !sh || err) { if (!err) err = 1; return {nullptr, nullptr}; }
    if (int e = bn_fold(g, b, m, v, 1e-5f, sc, sh, C, cp, st)) err = e;
    bn[prefix] = {sc, sh};
    return {sc, sh};
  }

  // forward conv + folded BN (+ residual) (+ ReLU); out may be a channel slice of a concat buffer
  void conv_bn(const Act& x, const std::string& wname, const std::string& bnname, int cin, int cout, int K, int stride,
               int dil, const Act* res, int relu, const Act& out) {
    if (dry) return;
    auto sb = bnfold(bnname, cout);
    WeightSrc w; w.w = P(wname + ".weight"); w.d0 = cout; w.d1 = cin; w.KH = w.KW = K; w.scale = sb.first;
    if (err) return;
    ConvGeom g; g.K = K; g.stride = stride; g.dil = dil;
    g.pad = (stride == 1) ? dil * (K - 1) / 2 : (K == 3 ? 1 : 0);
    Epilogue ep; ep.bias = sb.second; ep.res = res; ep.relu = relu;
    OutSpec os; os.mode = kOutNHWC; os.out = out;
    auto op = std::make_shared<ConvOp>();
    if (int e = build_conv(op.get(), arena, x, w, g, cout, nullptr, nullptr, ep, os, st)) { err = e; return; }
    net->flops_fwd += op->flops;
    push([op](cudaStream_t s) { return op->run(s); });
  }

  // data gradient of a forward conv (weight wname [cout][cin][K][K], BN scale folded): dx = dgrad(dz) (+res) (*mask)
  void dgrad(const Act& dz, const std::string& wname, const std::string& bnname, int cin, int cout, int K, int stride,
             int dil, const Act* res, const Act* mask, const Act& dx, const float* scale_override = nullptr, bool no_bn = false) {
    if (dry) return;
    const float* sc = no_bn ? scale_override : bnfold(bnname, cout).first;
    WeightSrc w; w.w = P(wname + ".weight"); w.d0 = cout; w.d1 = cin; w.KH = w.KW = K; w.transpose = 1; w.scale = sc;
    if (err) return;
    Epilogue ep; ep.res = res; ep.mask = mask;
    OutSpec os; os.mode = kOutNHWC; os.out = dx;
    auto op = std::make_shared<ConvOp>();
    int e;
    if (stride == 1) {
      w.flip = 1;
      ConvGeom g; g.K = K; g.stride = 1; g.dil = dil; g.pad = dil * (K - 1) / 2;
      e = build_conv(op.get(), arena, dz, w, g, cin, nullptr, nullptr, ep, os, st);
    } else {
      e = build_conv_transposed_s2(op.get(), arena, dz, w, K, K == 3 ? 1 : 0, cin, ep, os, st);
    }
    if (e) { err = e; return; }
    net->flops_bwd += op->flops;
    push([op](cudaStream_t s) { return op->run(s); });
  }
};

int build(wc_seg* net, bool dry, void* ws, size_t ws_bytes, cudaStream_t st) {
  const int B = net->B, H = net->H, W = net->W, NC = net->num_classes;
  SegBuilder b{net, dry ? Bump::dry() : Bump(ws, ws_bytes), net->arena.get(), st, dry, B};
  const int H2 = H / 2, W2 = W / 2, H4 = H / 4, W4 = W / 4;
  // ---------------- stem: conv1 7x7 s2 + bn1 + relu (tensor core, from NCHW fp32), maxpool 3x3 s2
  Act c1 = b.act(H2, W2, 64);
  Act p1 = b.act(H4, W4, 64);
  uint8_t* pool_idx = static_cast<uint8_t*>(b.bump.take(p1.pixels() * 64));
  __nv_bfloat16* xpad = static_cast<__nv_bfloat16*>(b.bump.take(static_cast<size_t>(B) * H * (W + 8) * 8 * sizeof(__nv_bfloat16)));
  std::pair<float*, float*> bn1{nullptr, nullptr};
  const float* w_conv1 = nullptr;
  if (!dry) {
    bn1 = b.bnfold("backbone.bn1", 64);
    w_conv1 = b.P("backbone.conv1.weight");
    if (b.err) return b.err;
    wc_seg* n = net;
    const float *sc = bn1.first, *sh = bn1.second;
    // image -> padded NHWC-8 bf16, then an implicit GEMM with overlapping TMA boxes (conv.cu)
    float* wprime = static_cast<float*>(b.arena->alloc(64 * 64 * 7 * sizeof(float)));
    if (!wprime) return 1;
    if (int e = stem_weights(w_conv1, wprime, 64, st)) return e;
    Epilogue ep; ep.bias = sh; ep.relu = 1;
    OutSpec os; os.mode = kOutNHWC; os.out = c1;
    auto op = std::make_shared<ConvOp>();
    if (int e = build_conv_stem7s2(op.get(), b.arena, xpad, B, H, W, wprime, sc, 64, ep, os, st)) return e;
    b.push([=](cudaStream_t s) {
      if (int e = stem_prepare(n->x_in, xpad, B, H, W, s)) return e;
      if (int e = op->run(s)) return e;
      return maxpool_fwd(c1.ptr, p1.ptr, pool_idx, B, H2, W2, 64, s);
    });
    net->flops_fwd += 2.0 * B * H2 * W2 * 147.0 * 64;
  }
  // ---------------- residual layers
  std::vector<BlockRec> blocks;
  {
    int inplanes = 64, dilation = 1;
    const int planes_l[4] = {64, 128, 256, 512}, stride_l[4] = {1, 2, 2, 2};
    const bool os8 = net->output_stride == 8;
    const bool dilate_l[4] = {false, false, os8, true};  // replace_stride_with_dilation: os 16 [F,F,T], os 8 [F,T,T] (modeling.py:34-39)
    for (int li = 0; li < 4; ++li) {
      const int prev = dilation;
      int stride = stride_l[li];
      if (dilate_l[li]) { dilation *= stride; stride = 1; }
      for (int bi = 0; bi < net->layers[li]; ++bi) {
        BlockRec r;
        r.p = "backbone.layer" + std::to_string(li + 1) + "." + std::to_string(bi);
        r.inplanes = inplanes; r.planes = planes_l[li];
        r.stride = bi == 0 ? stride : 1;
        r.dil = bi == 0 ? prev : dilation;
        r.has_down = bi == 0 && (stride != 1 || inplanes != planes_l[li] * 4);
        blocks.push_back(r);
        inplanes = planes_l[li] * 4;
      }
    }
  }
  Act cur = p1;
  Act low;
  for (size_t i = 0; i < blocks.size(); ++i) {
    BlockRec& r = blocks[i];
    r.x_in = cur;
    const int Ho = cur.H / r.stride, Wo = cur.W / r.stride;
    r.y1 = b.act(cur.H, cur.W, r.planes);
    b.conv_bn(cur, r.p + ".conv1", r.p + ".bn1", r.inplanes, r.planes, 1, 1, 1, nullptr, 1, r.y1);
    r.y2 = b.act(Ho, Wo, r.planes);
    b.conv_bn(r.y1, r.p + ".conv2", r.p + ".bn2", r.planes, r.planes, 3, r.stride, r.dil, nullptr, 1, r.y2);
    Act idt = cur;
    if (r.has_down) {
      idt = b.act(Ho, Wo, r.planes * 4);
      b.conv_bn(cur, r.p + ".downsample.0", r.p + ".downsample.1", r.inplanes, r.planes * 4, 1, r.stride, 1, nullptr, 0, idt);
    }
    r.out = b.act(Ho, Wo, r.planes * 4);
    b.conv_bn(r.y2, r.p + ".conv3", r.p + ".bn3", r.planes, r.planes * 4, 1, 1, 1, &idt, 1, r.out);
    cur = r.out;
    if (static_cast<int>(i) + 1 == net->layers[0]) low = cur;
    if (b.err) return b.err;
  }
  const Act feat = cur;  // [B, H/16, W/16, 2048]
  const int h = feat.H, w = feat.W;
  // ---------------- ASPP (_deeplab.py:138-162): five branches written into one 1280-channel buffer
  const std::string c = "classifier";
  Act cat5 = b.act(h, w, 1280);
  b.conv_bn(feat, c + ".aspp.convs.0.0", c + ".aspp.convs.0.1", 2048, 256, 1, 1, 1, nullptr, 1, slice_act(cat5, 0, 256));
  const int rmul = net->output_stride == 8 ? 2 : 1;
  const int rates[3] = {6 * rmul, 12 * rmul, 18 * rmul};   // ASPP dilations (modeling.py:35,38)
  for (int k = 0; k < 3; ++k)
    b.conv_bn(feat, c + ".aspp.convs." + std::to_string(k + 1) + ".0", c + ".aspp.convs." + std::to_string(k + 1) + ".1", 2048,
              256, 3, 1, rates[k], nullptr, 1, slice_act(cat5, 256 * (k + 1), 256));
  Act pooled = b.act(1, 1, 2048), g2 = b.act(1, 1, 256);
  b.push([=](cudaStream_t s) { return gap_fwd(feat.ptr, pooled.ptr, B, h * w, 2048, feat.ld, s); });
  b.conv_bn(pooled, c + ".aspp.convs.4.1", c + ".aspp.convs.4.2", 2048, 256, 1, 1, 1, nullptr, 1, g2);
  {
    Act dst = slice_act(cat5, 1024, 256);
    b.push([=](cudaStream_t s) { return broadcast_hw(g2.ptr, dst.ptr, B, h * w, 256, dst.ld, s); });
  }
  Act aspp = b.act(h, w, 256);
  b.conv_bn(cat5, c + ".aspp.project.0", c + ".aspp.project.1", 1280, 256, 1, 1, 1, nullptr, 1, aspp);
  // ---------------- decoder (_deeplab.py:47-51)
  Act cat2 = b.act(H4, W4, 304);
  Act ll = slice_act(cat2, 0, 48), up = slice_act(cat2, 48, 256);
  b.conv_bn(low, c + ".project.0", c + ".project.1", 256, 48, 1, 1, 1, nullptr, 1, ll);
  b.push([=](cudaStream_t s) { return bilinear_fwd(aspp.ptr, up.ptr, B, h, w, H4, W4, 256, aspp.ld, up.ld, s); });
  Act y = b.act(H4, W4, 256);
  b.conv_bn(cat2, c + ".classifier.0", c + ".classifier.1", 304, 256, 3, 1, 1, nullptr, 1, y);
  const int NCP = 32;
  float* logits_lo = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * NC * H4 * W4 * sizeof(float)));
  if (!dry) {
    float* bias_pad = static_cast<float*>(b.arena->alloc(NCP * sizeof(float)));
    const float* bias = b.P(c + ".classifier.3.bias");
    WeightSrc wsrc; wsrc.w = b.P(c + ".classifier.3.weight"); wsrc.d0 = NC; wsrc.d1 = 256;
    if (!bias_pad || b.err) return b.err ? b.err : 1;
    WC_CHECK_CUDA(cudaMemsetAsync(bias_pad, 0, NCP * sizeof(float), st));
    WC_CHECK_CUDA(cudaMemcpyAsync(bias_pad, bias, NC * sizeof(float), cudaMemcpyDeviceToDevice, st));
    ConvGeom g; g.K = 1; g.pad = 0;
    Epilogue ep; ep.bias = bias_pad;
    OutSpec os; os.mode = kOutNCHWf32; os.out_f32 = logits_lo; os.n_store = NC;
    auto op = std::make_shared<ConvOp>();
    if (int e = build_conv(op.get(), b.arena, y, wsrc, g, NCP, nullptr, nullptr, ep, os, st)) return e;
    net->flops_fwd += op->flops;
    b.push([op](cudaStream_t s) { return op->run(s); });
  }
  // ---------------- loss head: bilinear to the input size, argmax, softmax-CE gradient (inference.py:135-141)
  float* dlogit_hi = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * H * W * NC * sizeof(float)));
  int* n_valid = static_cast<int*>(b.bump.take(B * sizeof(int)));
  // With the input gradient requested, pred / loss / low-resolution d-logits come from ONE kernel and the 19-plane full-resolution
  // d-logit tensor is never written (seg_kernels.cu: seg_loss_head_fused_kernel); geometries it does not take, and requests for the
  // full-resolution logits, go through the two-pass head below.
  Act dlo{};
  if (net->with_grad) dlo = b.act(H4, W4, NCP);
  if (!dry) {
    net->n_body_ops = net->fwd_ops.size();
    net->logits_lo = logits_lo;
    net->dlo = net->with_grad ? dlo.ptr : nullptr;
  }
  {
    wc_seg* n = net;
    const bool with_grad = net->with_grad;
    b.push([=](cudaStream_t s) {
      if (with_grad && !n->logits_hi) {
        const int e = seg_loss_head_fused(logits_lo, n->labels, n_valid, n->pred, n->loss, dlo.ptr, B, H4, W4, H, W, NC, NCP, NCP, 255, s);
        if (e != -1) return e;
      }
      if (int e = seg_loss_grad(logits_lo, n->labels, n_valid, n->pred, dlogit_hi, n->loss, n->logits_hi, B, H4, W4, H, W, NC, 255, s)) return e;
      return with_grad ? logits_bilinear_bwd(dlogit_hi, dlo.ptr, B, H4, W4, H, W, NC, NCP, NCP, s) : 0;
    });
  }
  if (!net->with_grad) {
    if (dry) net->ws_needed = b.bump.used() + 4096;
    else if (b.bump.overflow()) return fail("seg workspace too small");
    return b.err;
  }
  // =================================================== backward (data gradients only)
  b.in_bwd = true;
  Act dlo19 = dlo; dlo19.C = NC;
  Act dy = b.act(H4, W4, 256);
  b.dgrad(dlo19, c + ".classifier.3", "", 256, NC, 1, 1, 1, nullptr, &y, dy, nullptr, true);
  Act dcat2 = b.act(H4, W4, 304);
  b.dgrad(dy, c + ".classifier.0", c + ".classifier.1", 304, 256, 3, 1, 1, nullptr, nullptr, dcat2);
  Act d_ll = slice_act(dcat2, 0, 48), d_up = slice_act(dcat2, 48, 256);
  b.push([=](cudaStream_t s) { return relu_mask_inplace(d_ll.ptr, ll.ptr, d_ll.pixels(), 48, d_ll.ld, ll.ld, s); });
  Act dlow_extra = b.act(H4, W4, 256);  // gradient reaching layer1's output through the decoder
  b.dgrad(d_ll, c + ".project.0", c + ".project.1", 256, 48, 1, 1, 1, nullptr, nullptr, dlow_extra);
  Act daspp = b.act(h, w, 256);
  b.push([=](cudaStream_t s) {
    return bilinear_bwd(d_up.ptr, aspp.ptr, daspp.ptr, B, h, w, H4, W4, 256, d_up.ld, aspp.ld, daspp.ld, s);
  });
  Act dcat5 = b.act(h, w, 1280);
  b.dgrad(daspp, c + ".aspp.project.0", c + ".aspp.project.1", 1280, 256, 1, 1, 1, nullptr, &cat5, dcat5);
  Act dfeat = b.act(h, w, 2048);
  {
    Act d0 = slice_act(dcat5, 0, 256);
    b.dgrad(d0, c + ".aspp.convs.0.0", c + ".aspp.convs.0.1", 2048, 256, 1, 1, 1, nullptr, nullptr, dfeat);
    for (int k = 0; k < 3; ++k) {
      Act dk = slice_act(dcat5, 256 * (k + 1), 256);
      b.dgrad(dk, c + ".aspp.convs." + std::to_string(k + 1) + ".0", c + ".aspp.convs." + std::to_string(k + 1) + ".1", 2048, 256,
              3, 1, rates[k], &dfeat, nullptr, dfeat);
    }
    Act d4 = slice_act(dcat5, 1024, 256);
    Act dg2 = b.act(1, 1, 256), dpooled = b.act(1, 1, 2048);
    b.push([=](cudaStream_t s) { return sum_hw(d4.ptr, nullptr, dg2.ptr, B, h * w, 256, d4.ld, s); });
    b.dgrad(dg2, c + ".aspp.convs.4.1", c + ".aspp.convs.4.2", 2048, 256, 1, 1, 1, nullptr, nullptr, dpooled);
    b.push([=](cudaStream_t s) {
      if (int e = gap_bwd_add(dpooled.ptr, dfeat.ptr, B, h * w, 2048, dfeat.ld, s)) return e;
      return relu_mask_inplace(dfeat.ptr, feat.ptr, dfeat.pixels(), 2048, dfeat.ld, feat.ld, s);
    });
  }
  // ---- residual blocks in reverse; `g` = gradient wrt the block output, ReLU mask already applied
  Act g = dfeat;
  for (int i = static_cast<int>(blocks.size()) - 1; i >= 0; --i) {
    const BlockRec& r = blocks[i];
    const bool first_block = (i == 0);
    const bool feeds_low = (i == net->layers[0]);  // this block's input is layer1's output (the low-level feature)
    Act d2 = b.act(g.H, g.W, r.planes);
    b.dgrad(g, r.p + ".conv3", r.p + ".bn3", r.planes, r.planes * 4, 1, 1, 1, nullptr, &r.y2, d2);
    Act d1 = b.act(r.x_in.H, r.x_in.W, r.planes);
    b.dgrad(d2, r.p + ".conv2", r.p + ".bn2", r.planes, r.planes, 3, r.stride, r.dil, nullptr, &r.y1, d1);
    Act didt = g;
    if (r.has_down) {
      didt = b.act(r.x_in.H, r.x_in.W, r.inplanes);
      const size_t bytes = didt.pixels() * didt.C * sizeof(__nv_bfloat16);
      const bool need_init = (r.stride == 2) || feeds_low;
      if (need_init) {
        if (feeds_low) {
          b.push([=](cudaStream_t s) {
            return cudaMemcpyAsync(didt.ptr, dlow_extra.ptr, bytes, cudaMemcpyDeviceToDevice, s) == cudaSuccess ? 0 : fail("memcpy failed");
          });
        } else {
          b.push([=](cudaStream_t s) { return cudaMemsetAsync(didt.ptr, 0, bytes, s) == cudaSuccess ? 0 : fail("memset failed"); });
        }
      }
      b.dgrad(g, r.p + ".downsample.0", r.p + ".downsample.1", r.inplanes, r.planes * 4, 1, r.stride, 1, need_init ? &didt : nullptr,
              nullptr, didt);
    } else if (feeds_low) {
      return fail("internal: the block after layer1 is expected to have a downsample branch");
    }
    Act dx = b.act(r.x_in.H, r.x_in.W, r.inplanes);
    b.dgrad(d1, r.p + ".conv1", r.p + ".bn1", r.inplanes, r.planes, 1, 1, 1, &didt, first_block ? nullptr : &r.x_in, dx);
    g = dx;
    if (b.err) return b.err;
  }
  // ---- stem backward: maxpool (+ReLU mask of conv1's output), conv1 data gradient to the NCHW fp32 image
  Act dc1 = b.act(H2, W2, 64);
  {
    wc_seg* n = net;
    const Act gp = g;
    const float* sc = bn1.first;
    const int P = net->grad_pool;
    float* weff = nullptr;
    if (!dry && P > 1) {
      const int R = P / 2 + 3;
      weff = static_cast<float*>(b.arena->alloc(static_cast<size_t>(R) * R * 192 * sizeof(float)));
      if (!weff) return 1;
      if (int e = conv1_dgrad_weff(w_conv1, sc, weff, P, st)) return e;
    }
    b.push([=](cudaStream_t s) {
      if (int e = maxpool_bwd(gp.ptr, pool_idx, c1.ptr, dc1.ptr, B, H2, W2, 64, s)) return e;
      if (P > 1) return conv1_dgrad_pooled(dc1.ptr, weff, n->grad_out, B, H, W, P, s);
      return conv1_dgrad(dc1.ptr, w_conv1, sc, n->grad_out, B, H, W, 64, s);
    });
    net->flops_bwd += 2.0 * B * H2 * W2 * 147.0 * 64;
  }
  if (dry) net->ws_needed = b.bump.used() + 4096;
  else if (b.bump.overflow()) return fail("seg workspace too small: need " + std::to_string(b.bump.used()) + " bytes");
  return b.err;
}

// (Re)builds the plan when the geometry, the gradient mode or the workspace differ from the current binding.
int bind_plan(wc_seg* net, int batch, int H, int W, int with_grad, int grad_pool, void* workspace, size_t workspace_bytes,
              cudaStream_t st) {
  if (net->B == batch && net->H == H && net->W == W && net->with_grad == with_grad && net->grad_pool == grad_pool && net->ws == workspace &&
      net->ws_bytes == workspace_bytes)
    return 0;
  net->fwd_ops.clear(); net->bwd_ops.clear();
  net->arena = std::make_unique<DeviceArena>();
  net->B = batch; net->H = H; net->W = W; net->with_grad = with_grad; net->grad_pool = grad_pool; net->ws = workspace; net->ws_bytes = workspace_bytes;
  net->flops_fwd = net->flops_bwd = 0;
  if (int e = build(net, false, workspace, workspace_bytes, st)) {
    net->B = 0;
    net->fwd_ops.clear(); net->bwd_ops.clear();
    return e;
  }
  return 0;
}

}  // namespace
}  // namespace wc

using namespace wc;

extern "C" {

int wc_seg_create(wc_seg** out, const int* blocks_per_layer, int num_classes, int n_params, const char* const* names,
                  const float* const* ptrs, void* stream) {
  (void)stream;
  WC_REQUIRE(out && blocks_per_layer && names && ptrs, "null argument");
  WC_REQUIRE(num_classes == 19, "the loss head is built for 19 classes");
  auto net = std::make_unique<wc_seg>();
  for (int i = 0; i < 4; ++i) net->layers[i] = blocks_per_layer[i];
  net->num_classes = num_classes;
  for (int i = 0; i < n_params; ++i) net->params.ptr[names[i]] = ptrs[i];
  *out = net.release();
  return 0;
}

int wc_seg_set_output_stride(wc_seg* net, int output_stride) {
  WC_REQUIRE(net, "null handle");
  WC_REQUIRE(output_stride == 8 || output_stride == 16, "output_stride must be 8 or 16 (modeling.py:34-39)");
  if (net->output_stride != output_stride) {
    net->output_stride = output_stride;
    net->B = net->H = net->W = 0;   // force a rebuild of the plan on the next call
    net->saved_fwd = 0;
  }
  return 0;
}

void wc_seg_destroy(wc_seg* net) { delete net; }

size_t wc_seg_workspace_bytes(const wc_seg* net_c, int batch, int H, int W, int with_grad) {
  wc_seg* net = const_cast<wc_seg*>(net_c);
  const int sB = net->B, sH = net->H, sW = net->W, sg = net->with_grad;
  net->B = batch; net->H = H; net->W = W; net->with_grad = with_grad;
  size_t need = 0;
  if (build(net, true, nullptr, 0, nullptr) == 0) need = net->ws_needed;
  net->B = sB; net->H = sH; net->W = sW; net->with_grad = sg;
  return need;
}

int wc_seg_infer_pooled(wc_seg* net, const float* x, const int64_t* labels, int64_t* pred, float* input_grad, float* loss,
                        float* logits, int batch, int H, int W, int grad_pool, void* workspace, size_t workspace_bytes,
                        void* stream);

int wc_seg_infer(wc_seg* net, const float* x, const int64_t* labels, int64_t* pred, float* input_grad, float* loss,
                 float* logits, int batch, int H, int W, void* workspace, size_t workspace_bytes, void* stream) {
  return wc_seg_infer_pooled(net, x, labels, pred, input_grad, loss, logits, batch, H, W, 1, workspace, workspace_bytes, stream);
}

int wc_seg_infer_pooled(wc_seg* net, const float* x, const int64_t* labels, int64_t* pred, float* input_grad, float* loss,
                        float* logits, int batch, int H, int W, int grad_pool, void* workspace, size_t workspace_bytes,
                        void* stream) {
  if (net) net->saved_fwd = 0;
  WC_REQUIRE(grad_pool >= 1, "grad_pool must be >= 1");
  WC_REQUIRE(net && x && labels && workspace, "null argument");
  WC_REQUIRE(H % 32 == 0 && W % 32 == 0, "H and W must be multiples of 32 (output stride 16, stride-2 phase views)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int with_grad = input_grad != nullptr;
  if (int e = bind_plan(net, batch, H, W, with_grad, grad_pool, workspace, workspace_bytes, st)) return e;
  net->x_in = x; net->labels = reinterpret_cast<const long long*>(labels);
  net->pred = reinterpret_cast<long long*>(pred); net->grad_out = input_grad; net->loss = loss; net->logits_hi = logits;
  for (auto& op : net->fwd_ops)
    if (int e = op(st)) return e;
  for (auto& op : net->bwd_ops)
    if (int e = op(st)) return e;
  return 0;
}

int wc_seg_forward(wc_seg* net, const float* x, float* logits, int batch, int H, int W, int save_for_backward, void* workspace,
                   size_t workspace_bytes, void* stream) {
  if (net) net->saved_fwd = 0;
  WC_REQUIRE(net && x && logits && workspace, "null argument");
  WC_REQUIRE(H % 32 == 0 && W % 32 == 0, "H and W must be multiples of 32 (output stride 16, stride-2 phase views)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = bind_plan(net, batch, H, W, save_for_backward ? 1 : 0, 1, workspace, workspace_bytes, st)) return e;
  net->x_in = x; net->labels = nullptr; net->pred = nullptr; net->grad_out = nullptr; net->loss = nullptr; net->logits_hi = logits;
  for (size_t i = 0; i < net->n_body_ops; ++i)
    if (int e = net->fwd_ops[i](st)) return e;
  // the loss head's kernel without labels: only the up-sampled logits, the same bits wc_seg_infer writes
  if (int e = seg_loss_grad(net->logits_lo, nullptr, nullptr, nullptr, nullptr, nullptr, logits, batch, H / 4, W / 4, H, W,
                            net->num_classes, 255, st))
    return e;
  net->saved_fwd = save_for_backward ? 1 : 0;
  return 0;
}

int wc_seg_backward_seeded(wc_seg* net, const float* dlogits, float* input_grad, void* stream) {
  WC_REQUIRE(net && dlogits && input_grad, "null argument");
  WC_REQUIRE(net->saved_fwd && net->dlo,
             "wc_seg_backward_seeded: this handle holds no saved forward; the last call on it must be "
             "wc_seg_forward(save_for_backward = 1) (an infer or another forward in between discards the saved activations)");
  net->saved_fwd = 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int B = net->B, H = net->H, W = net->W;
  net->grad_out = input_grad;
  if (int e = logits_bilinear_bwd(dlogits, net->dlo, B, H / 4, W / 4, H, W, net->num_classes, 32, 32, st)) return e;
  for (auto& op : net->bwd_ops)
    if (int e = op(st)) return e;
  return 0;
}

double wc_seg_flops(const wc_seg* net, int backward) { return net ? (backward ? net->flops_bwd : net->flops_fwd) : 0.0; }
int wc_seg_launches(const wc_seg* net) { return net ? static_cast<int>(net->fwd_ops.size() + net->bwd_ops.size()) : 0; }

}  // extern "C"
