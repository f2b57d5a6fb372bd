// Denoising-loss training step of the UNet as static launch plans: forward (activations kept), MSE loss, full
// backward (data + weight gradients of every parameter).  Reference: diffusion_model/train_ddpm.py:95-114
//   noisy = scheduler.add_noise(im, noise, t); pred = model(noisy, t); loss = MSELoss(pred, noise); loss.backward()
// and diffusion_model/models/unet_base.py:372-488 for the network.  The optimizer step (fused Adam) and the gradient
// all-reduce run over flat fp32 buffers owned by the host (weatherconverter_b200/diffusion_model/train_ddpm.py).
//
// The builder walks the network once, emitting forward launches and pushing one closure per layer on a tape; the tape
// is then unwound to emit the backward launches.  Every activation buffer has a same-shaped gradient "shadow"; a
// producer of a gradient accumulates in place when the shadow slice has been written before (skip connections and
// residual branches), so fan-in never needs a separate add kernel.  Weight-dependent device state (bf16 packed
// weights of the forward and data-gradient GEMMs, folded biases, the concatenated t-embedding projection) is rebuilt
// by `repack_ops` at the start of every step because the optimizer changes the fp32 master weights.
//
// The same backward also runs seeded with a caller's dL/dpred (wc_unet_train_backward_seeded: torch autograd of the
// Unet module, diffusion_model/models/unet_base.py), optionally producing dL/dx and optionally skipping every op whose
// only product is a parameter gradient.
#include <map>

#include "plan.cuh"
#include "wgrad.cuh"
#include "../../include/wc_b200.h"

namespace wc {
int groupnorm_silu(const __nv_bfloat16* x, __nv_bfloat16* y, int B, int HW, int C, int ld, int ldy, const float* gamma,
                   const float* beta, float eps, int silu, void* workspace, cudaStream_t st);
size_t groupnorm_workspace_bytes(int B);
int groupnorm_silu_bwd(const __nv_bfloat16* x, const __nv_bfloat16* dy, __nv_bfloat16* dx, int B, int HW, int C, int ld,
                       int ldd, int ldo, const float* gamma, const float* beta, float eps, int silu, const void* stats,
                       const __nv_bfloat16* add1, int lda1, const __nv_bfloat16* add2, int lda2, float* dgamma, float* dbeta,
                       void* workspace, cudaStream_t st);
size_t groupnorm_bwd_workspace_bytes(int B, int Cmax);
int colsum(const __nv_bfloat16* x, int B, int HW, int C, int ld, float* out_rows, int ldo, float* out_total, void* workspace,
           cudaStream_t st);
int attention_forward(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, __nv_bfloat16* out, int B,
                      int heads, int ntok, int hd, int ldo, cudaStream_t st, float* lse = nullptr, float scale = 0.f);
double attention_flops(int B, int heads, int ntok, int hd);
int attention_backward(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* v, const __nv_bfloat16* d_o, int ldd,
                       const float* lse, const float* D, __nv_bfloat16* dqkv, int ld3, int B, int heads, int ntok, int hd,
                       cudaStream_t st);
double attention_bwd_flops(int B, int heads, int ntok, int hd);
int attn_rowdot(const __nv_bfloat16* o, const __nv_bfloat16* d_o, int ldo, int ldd, int B, int ntok, int heads, int hd, float* D,
                cudaStream_t st);
int conv_small_cin(const float* x, const float* w, const float* bias, const float* scale, const float* shift,
                   __nv_bfloat16* y, int B, int Cin, int H, int W, int Cout, int K, int stride, int pad, int ldy,
                   int relu, cudaStream_t st, const float* prelu = nullptr);
int conv_small_cout(const __nv_bfloat16* x, const float* w, const float* bias, float* y, int B, int H, int W, int Cin,
                    int Cout, int K, int ldx, int tanh_out, cudaStream_t st);
int linear_rows(const float* in, int Bt, int dim, const float* w, const float* bias, float* out, int N, cudaStream_t st);
int mse_loss_grad(const float* pred, const float* target, float* dpred, size_t n, float grad_scale, float* loss, void* scratch,
                  cudaStream_t st);
size_t boundary_wgrad_scratch_bytes();
int boundary_wgrad(const __nv_bfloat16* wide, int ldw, const float* narrow, int B, int H, int W, int sign, float* dw,
                   float* dbias, void* scratch, cudaStream_t st);
int flip_transpose_3x3(const float* w, float* wt, int Co, int Ci, cudaStream_t st);
int temb_mlp_train(const long long* t, int Bt, int dim, const float* w1, const float* b1, const float* w2, const float* b2,
                   float* emb, float* h1, float* temb, float* temb_silu, cudaStream_t st);
int temb_backward(const float* dtproj, int total, int B, int dim, const float* wcat, const float* w2, const float* emb,
                  const float* h1, const float* temb, const float* temb_silu, int nsegs, const int* seg_row0,
                  const int* seg_rows, float* const* seg_dw, float* const* seg_db, float* dw1, float* db1, float* dw2,
                  float* db2, float* scratch, cudaStream_t st);
int add_vectors(const float* a, const float* b, float* o, int n, cudaStream_t st);
}  // namespace wc

struct wc_unet_train {
  wc_unet_config cfg;
  wc::ParamTable params;
  std::unordered_map<std::string, float*> grads;
  std::unique_ptr<wc::DeviceArena> arena;
  int B = 0, H = 0, W = 0;
  void* ws = nullptr;
  size_t ws_bytes = 0, ws_needed = 0;
  wc::OpList repack_ops, fwd_ops, bwd_ops;
  std::vector<int> bwd_kind;  // per backward op: what it produces (kOpData / kOpParam / kOpInput)
  std::unordered_map<std::string, int> ready;  // parameter name -> number of backward ops after which its grad is final
  double flops_fwd = 0, flops_bwd = 0;
  // per-call pointers
  const float* x_in = nullptr;
  const float* target = nullptr;
  const long long* t_in = nullptr;
  float* pred_out = nullptr;
  float* loss_out = nullptr;
  float grad_scale = 1.f;
  const float* dpred_seed = nullptr;  // upstream gradient of a seeded backward; NULL: the loss gradient of the forward
  float* dx_out = nullptr;            // dL/dx of a seeded backward, or NULL
};

namespace wc {
namespace {

// What a backward op produces.  A seeded backward without parameter gradients skips every kOpParam op; a kOpInput op
// launches only when the caller asked for dL/dx.
enum { kOpData = 0, kOpParam = 1, kOpInput = 2 };

struct TBuilder {
  wc_unet_train* net;
  Bump bump;
  DeviceArena* arena;
  cudaStream_t st;
  bool dry;
  int B;
  int err = 0;
  bool in_bwd = false;
  float* tproj = nullptr;
  float* dtproj = nullptr;
  int tproj_ld = 0, temb_off = 0;
  float* wg_partial = nullptr;
  void* red_ws = nullptr;
  std::vector<std::function<void()>> tape;

  // ---------------------------------------------------------------- gradient shadows
  struct Alloc {
    __nv_bfloat16* base;
    int ld;
    size_t pixels;
    __nv_bfloat16* shadow;
    std::vector<std::pair<int, int>> written;  // channel ranges [c0, c1)
  };
  std::vector<Alloc> allocs;

  Act new_act(int H, int W, int C) {
    Act a = make_act(bump, B, H, W, C);
    allocs.push_back({a.ptr, C, a.pixels(), nullptr, {}});
    return a;
  }
  Alloc* find(const Act& a, int* c0) {
    for (auto& al : allocs) {
      if (a.ptr >= al.base && a.ptr < al.base + al.ld && a.ld == al.ld) {
        *c0 = static_cast<int>(a.ptr - al.base);
        return &al;
      }
    }
    if (!err) err = fail("internal: activation view without an allocation record");
    return nullptr;
  }
  Act grad(const Act& a) {
    int c0 = 0;
    Alloc* al = find(a, &c0);
    Act g = a;
    if (!al) return g;
    if (!al->shadow) al->shadow = static_cast<__nv_bfloat16*>(bump.take(al->pixels * al->ld * sizeof(__nv_bfloat16)));
    g.ptr = al->shadow ? al->shadow + c0 : nullptr;
    return g;
  }
  bool written(const Act& a) {
    int c0 = 0;
    Alloc* al = find(a, &c0);
    if (!al) return false;
    for (auto& r : al->written)
      if (r.first <= c0 && c0 + a.C <= r.second) return true;
    return false;
  }
  void mark(const Act& a) {
    int c0 = 0;
    Alloc* al = find(a, &c0);
    if (al) al->written.push_back({c0, c0 + a.C});
  }
  Act grad_written(const Act& a) {  // gradient that must already exist (dout of a layer)
    if (!written(a) && !err) err = fail("internal: backward reached a tensor whose gradient was never produced");
    return grad(a);
  }

  // ---------------------------------------------------------------- helpers
  const float* P(const std::string& n) { return dry ? nullptr : net->params.get(n, &err); }
  float* G(const std::string& n) {
    if (dry) return nullptr;
    auto it = net->grads.find(n);
    if (it == net->grads.end()) {
      if (!err) err = fail("missing gradient buffer for '" + n + "'");
      return nullptr;
    }
    return it->second;
  }
  void push(std::function<int(cudaStream_t)> f, int kind = kOpData) {
    if (dry) return;
    if (in_bwd) net->bwd_kind.push_back(kind);
    (in_bwd ? net->bwd_ops : net->fwd_ops).push_back(std::move(f));
  }
  void ready(const std::string& n) {
    if (!dry) net->ready[n] = static_cast<int>(net->bwd_ops.size());
  }

  void* gn_fwd(const Act& x, const Act& y, const std::string& prefix, int silu) {
    void* stats = bump.take(groupnorm_workspace_bytes(B));
    const float *g = P(prefix + ".weight"), *b = P(prefix + ".bias");
    push([=](cudaStream_t s) {
      return groupnorm_silu(x.ptr, y.ptr, x.B, x.H * x.W, x.C, x.ld, y.ld, g, b, 1e-5f, silu, stats, s);
    });
    return stats;
  }
  // dx (= or +=) GN'(dy) (+ add1)
  void gn_bwd(const Act& x, const Act& dy, const std::string& prefix, int silu, const void* stats, const Act* add1) {
    Act gx = grad(x);
    const bool acc = written(x);
    mark(x);
    const float *g = P(prefix + ".weight"), *b = P(prefix + ".bias");
    float *dg = G(prefix + ".weight"), *db = G(prefix + ".bias");
    void* ws = red_ws;
    const __nv_bfloat16* a1 = add1 ? add1->ptr : nullptr;
    const int lda1 = add1 ? add1->ld : 8;
    const __nv_bfloat16* a2 = acc ? gx.ptr : nullptr;
    push([=](cudaStream_t s) {
      return groupnorm_silu_bwd(x.ptr, dy.ptr, gx.ptr, x.B, x.H * x.W, x.C, x.ld, dy.ld, gx.ld, g, b, 1e-5f, silu, stats, a1, lda1,
                                a2, gx.ld, dg, db, ws, s);
    });
    ready(prefix + ".weight");
    ready(prefix + ".bias");
  }

  // forward convolution through the igemm path
  void conv_fwd(const Act& x, const std::string& wname, int cout, int K, int stride, int pad, const float* bias,
                const float* rowbias, int ldrb, const Act* res, const Act* x2, const std::string& w2name, const Act& out,
                bool transposed_up = false) {
    if (dry) return;
    Epilogue ep; ep.bias = bias; ep.rowbias = rowbias; ep.ldrb = ldrb; ep.res = res;
    OutSpec os; os.mode = kOutNHWC; os.out = out;
    auto op = std::make_shared<ConvOp>();
    int e;
    if (transposed_up) {
      WeightSrc w; w.w = P(wname + ".weight"); w.d0 = x.C; w.d1 = cout; w.KH = w.KW = K; w.transpose = 1;
      if (err) return;
      e = build_conv_transposed_s2(op.get(), arena, x, w, K, pad, cout, ep, os, st);
    } else {
      WeightSrc w; w.w = P(wname + ".weight"); w.d0 = cout; w.d1 = x.C; w.KH = w.KW = K;
      WeightSrc w2;
      if (x2) { w2.w = P(w2name + ".weight"); w2.d0 = cout; w2.d1 = x2->C; }
      if (err) return;
      ConvGeom g; g.K = K; g.stride = stride; g.pad = pad; g.dil = 1;
      e = build_conv(op.get(), arena, x, w, g, cout, x2, x2 ? &w2 : nullptr, ep, os, st);
    }
    if (e) { err = e; return; }
    net->flops_fwd += op->flops;
    push([op](cudaStream_t s) { return op->run(s); });
  }

  // data gradient of y = conv(x, W[cout][cin][K][K], stride, pad): gx (= or +=) dgrad(dy)
  void dgrad(const Act& dy, const std::string& wname, int cout, int cin, int K, int stride, const Act& x) {
    Act gx = grad(x);
    const bool acc = written(x);
    mark(x);
    if (dry) return;
    WeightSrc w; w.w = P(wname + ".weight"); w.d0 = cout; w.d1 = cin; w.KH = w.KW = K; w.transpose = 1;
    if (err) return;
    Epilogue ep; ep.res = acc ? &gx : nullptr;
    OutSpec os; os.mode = kOutNHWC; os.out = gx;
    auto op = std::make_shared<ConvOp>();
    int e;
    if (stride == 1) {
      w.flip = 1;
      ConvGeom g; g.K = K; g.stride = 1; g.dil = 1; g.pad = (K - 1) / 2;
      e = build_conv(op.get(), arena, dy, w, g, cin, nullptr, nullptr, ep, os, st);
    } else {
      e = build_conv_transposed_s2(op.get(), arena, dy, w, K, 1, cin, ep, os, st);
    }
    if (e) { err = e; return; }
    net->flops_bwd += op->flops;
    push([op](cudaStream_t s) { return op->run(s); });
  }
  // data gradient of y = conv_transpose2d(x, W[cin][cout][4][4], 2, 1): a stride-2 convolution of dy with W as stored
  void dgrad_convT(const Act& dy, const std::string& wname, int cin, int cout, const Act& x) {
    Act gx = grad(x);
    const bool acc = written(x);
    mark(x);
    if (dry) return;
    WeightSrc w; w.w = P(wname + ".weight"); w.d0 = cin; w.d1 = cout; w.KH = w.KW = 4;
    if (err) return;
    Epilogue ep; ep.res = acc ? &gx : nullptr;
    OutSpec os; os.mode = kOutNHWC; os.out = gx;
    ConvGeom g; g.K = 4; g.stride = 2; g.pad = 1; g.dil = 1;
    auto op = std::make_shared<ConvOp>();
    if (int e = build_conv(op.get(), arena, dy, w, g, cin, nullptr, nullptr, ep, os, st)) { err = e; return; }
    net->flops_bwd += op->flops;
    push([op](cudaStream_t s) { return op->run(s); });
  }
  void wgrad(const Act& x, const Act& dy, int K, int stride, int pad, const std::string& wname, const Act* x2,
             const std::string& w2name, bool transposed = false) {
    if (dry) return;
    float* dw = G(wname + ".weight");
    float* dw2 = x2 ? G(w2name + ".weight") : nullptr;
    if (err) return;
    auto op = std::make_shared<WgradOp>();
    int e = transposed ? build_convT_wgrad(op.get(), x, dy, K, pad, dw, wg_partial)
                       : build_conv_wgrad(op.get(), x, dy, K, stride, pad, 1, dw, x2, dw2, wg_partial);
    if (e) { err = e; return; }
    net->flops_bwd += op->flops;
    push([op](cudaStream_t s) { return op->run(s); }, kOpParam);
    ready(wname + ".weight");
    if (x2) ready(w2name + ".weight");
  }
  // bias gradient(s) = column sums of dy; optionally the per-sample sums (t-embedding projection gradient)
  void bias_grad(const Act& dy, const std::string& bname, const std::string& bname2, float* rows, int ldo) {
    if (dry) return;
    float* db = G(bname);
    float* db2 = bname2.empty() ? nullptr : G(bname2);
    if (err) return;
    void* ws = red_ws;
    const int C = dy.C;
    push([=](cudaStream_t s) {
      if (int e = colsum(dy.ptr, dy.B, dy.H * dy.W, C, dy.ld, rows, ldo, db, ws, s)) return e;
      if (db2) WC_CHECK_CUDA(cudaMemcpyAsync(db2, db, C * sizeof(float), cudaMemcpyDeviceToDevice, s));
      return 0;
    }, kOpParam);
    ready(bname);
    if (db2) ready(bname2);
  }

  // ---------------------------------------------------------------- layers
  // ResNet sub-layer (unet_base.py:146-150): out = conv2(silu(gn2(conv1(silu(gn1(x))) + temb))) + conv1x1(x)
  Act resnet(const Act& x, int cout, const std::string& p, int l, const Act* dest) {
    const std::string ls = std::to_string(l);
    const std::string n1 = p + ".resnet_conv_first." + ls, n2 = p + ".resnet_conv_second." + ls, nr = p + ".residual_input_conv." + ls;
    Act a1 = new_act(x.H, x.W, x.C);
    void* st1 = gn_fwd(x, a1, n1 + ".0", 1);
    Act h = new_act(x.H, x.W, cout);
    const int toff = temb_off;
    temb_off += cout;
    conv_fwd(a1, n1 + ".2", cout, 3, 1, 1, P(n1 + ".2.bias"), dry ? nullptr : tproj + toff, tproj_ld, nullptr, nullptr, "", h);
    Act a2 = new_act(x.H, x.W, cout);
    void* st2 = gn_fwd(h, a2, n2 + ".0", 1);
    Act out = dest ? *dest : new_act(x.H, x.W, cout);
    float* bsum = nullptr;
    if (!dry) {
      bsum = static_cast<float*>(arena->alloc(cout * sizeof(float)));
      const float *b2 = P(n2 + ".2.bias"), *br = P(nr + ".bias");
      if (!bsum || err) { if (!err) err = 1; return out; }
      net->repack_ops.push_back([=](cudaStream_t s) { return add_vectors(b2, br, bsum, cout, s); });
    }
    conv_fwd(a2, n2 + ".2", cout, 3, 1, 1, bsum, nullptr, 0, nullptr, &x, nr, out);
    float* dtp = dtproj;
    const int ldt = tproj_ld;
    tape.push_back([=]() {
      Act dout = grad_written(out);
      dgrad(dout, n2 + ".2", cout, cout, 3, 1, a2);                 // d a2
      dgrad(dout, nr, cout, x.C, 1, 1, x);                           // residual branch -> d x (first contribution)
      wgrad(a2, dout, 3, 1, 1, n2 + ".2", &x, nr);
      bias_grad(dout, n2 + ".2.bias", nr + ".bias", nullptr, 0);
      Act da2 = grad(a2);
      gn_bwd(h, da2, n2 + ".0", 1, st2, nullptr);                    // d h
      Act dh = grad(h);
      bias_grad(dh, n1 + ".2.bias", "", dry ? nullptr : dtp + toff, ldt);   // conv1 bias + per-sample t-emb gradient
      dgrad(dh, n1 + ".2", cout, x.C, 3, 1, a1);                     // d a1
      wgrad(a1, dh, 3, 1, 1, n1 + ".2", nullptr, "");
      Act da1 = grad(a1);
      gn_bwd(x, da1, n1 + ".0", 1, st1, nullptr);                    // d x += GN'(d a1)
    });
    return out;
  }

  // attention sub-layer (unet_base.py:153-161): out = x + out_proj(attn(in_proj(gn(x))))
  Act attention(const Act& x, const std::string& p, int l, int heads, const Act* dest) {
    const std::string ls = std::to_string(l);
    const std::string nn = p + ".attention_norms." + ls, ap = p + ".attentions." + ls;
    const int C = x.C, hd = C / heads, ntok = x.H * x.W;
    Act a = new_act(x.H, x.W, C);
    void* stn = gn_fwd(x, a, nn, 0);
    const size_t per = static_cast<size_t>(B) * ntok * C;
    auto* q = static_cast<__nv_bfloat16*>(bump.take(per * 2));
    auto* k = static_cast<__nv_bfloat16*>(bump.take(per * 2));
    auto* vt = static_cast<__nv_bfloat16*>(bump.take(per * 2));
    auto* v = static_cast<__nv_bfloat16*>(bump.take(per * 2));
    float* lse = static_cast<float*>(bump.take(static_cast<size_t>(B) * heads * ntok * sizeof(float)));
    Act o = new_act(x.H, x.W, C);
    Act out = dest ? *dest : new_act(x.H, x.W, C);
    if (!dry) {
      WeightSrc w; w.w = P(ap + ".in_proj_weight"); w.d0 = 3 * C; w.d1 = C;
      ConvGeom g; g.K = 1; g.stride = 1; g.pad = 0; g.dil = 1;
      Epilogue ep; ep.bias = P(ap + ".in_proj_bias");
      OutSpec os; os.mode = kOutQKV; os.q = q; os.k = k; os.vt = vt; os.v = v; os.heads = heads; os.hd = hd;
      if (err) return out;
      auto op = std::make_shared<ConvOp>();
      if (int e = build_conv(op.get(), arena, a, w, g, 3 * C, nullptr, nullptr, ep, os, st)) { err = e; return out; }
      net->flops_fwd += op->flops;
      push([op](cudaStream_t s) { return op->run(s); });
      const int Bc = B;
      net->flops_fwd += attention_flops(B, heads, ntok, hd);
      push([=](cudaStream_t s) { return attention_forward(q, k, vt, o.ptr, Bc, heads, ntok, hd, o.ld, s, lse); });
    }
    conv_fwd(o, ap + ".out_proj", C, 1, 1, 0, P(ap + ".out_proj.bias"), nullptr, 0, &x, nullptr, "", out);
    tape.push_back([=]() {
      Act dout = grad_written(out);
      dgrad(dout, ap + ".out_proj", C, C, 1, 1, o);
      wgrad(o, dout, 1, 1, 0, ap + ".out_proj", nullptr, "");
      bias_grad(dout, ap + ".out_proj.bias", "", nullptr, 0);
      Act d_o = grad(o);
      Act dqkv = new_act(x.H, x.W, 3 * C);
      float* Dv = static_cast<float*>(bump.take(static_cast<size_t>(B) * heads * ntok * sizeof(float)));
      const int Bc = B;
      if (!dry) net->flops_bwd += attention_bwd_flops(B, heads, ntok, hd);
      push([=](cudaStream_t s) {
        if (int e = attn_rowdot(o.ptr, d_o.ptr, o.ld, d_o.ld, Bc, ntok, heads, hd, Dv, s)) return e;
        return attention_backward(q, k, v, d_o.ptr, d_o.ld, lse, Dv, dqkv.ptr, dqkv.ld, Bc, heads, ntok, hd, s);
      });
      // in-projection: weight [3C][C] (nn.MultiheadAttention.in_proj_weight), a Linear = 1x1 convolution
      {
        Act ga = grad(a);
        mark(a);
        if (!dry) {
          WeightSrc w; w.w = P(ap + ".in_proj_weight"); w.d0 = 3 * C; w.d1 = C; w.transpose = 1;
          Epilogue ep;
          OutSpec os; os.mode = kOutNHWC; os.out = ga;
          ConvGeom g; g.K = 1; g.stride = 1; g.pad = 0; g.dil = 1;
          auto op = std::make_shared<ConvOp>();
          if (!err) {
            if (int e = build_conv(op.get(), arena, dqkv, w, g, C, nullptr, nullptr, ep, os, st)) err = e;
            else { net->flops_bwd += op->flops; push([op](cudaStream_t s) { return op->run(s); }); }
          }
          float* dw = G(ap + ".in_proj_weight");
          auto wop = std::make_shared<WgradOp>();
          if (!err) {
            if (int e = build_conv_wgrad(wop.get(), a, dqkv, 1, 1, 0, 1, dw, nullptr, nullptr, wg_partial)) err = e;
            else { net->flops_bwd += wop->flops; push([wop](cudaStream_t s) { return wop->run(s); }, kOpParam); }
          }
          ready(ap + ".in_proj_weight");
        }
        bias_grad(dqkv, ap + ".in_proj_bias", "", nullptr, 0);
      }
      Act da = grad(a);
      gn_bwd(x, da, nn, 0, stn, &dout);  // d x (+)= GN'(d a) + d out (identity branch)
    });
    return out;
  }
};

int build(wc_unet_train* net, bool dry, void* ws, size_t ws_bytes, cudaStream_t st) {
  const wc_unet_config& c = net->cfg;
  const int B = net->B, H = net->H, W = net->W;
  TBuilder b{net, dry ? Bump::dry() : Bump(ws, ws_bytes), net->arena.get(), st, dry, B};
  const int nlev = c.n_down_channels - 1;
  const int* dc = c.down_channels;
  const int T = c.time_emb_dim;

  // ---- t-embedding layer table (execution order), concatenated projection
  std::vector<std::pair<std::string, int>> tl;
  for (int i = 0; i < nlev; ++i)
    for (int l = 0; l < c.num_down_layers; ++l)
      tl.push_back({"downs." + std::to_string(i) + ".t_emb_layers." + std::to_string(l) + ".1", dc[i + 1]});
  for (int i = 0; i + 1 < c.n_mid_channels; ++i)
    for (int l = 0; l < c.num_mid_layers + 1; ++l)
      tl.push_back({"mids." + std::to_string(i) + ".t_emb_layers." + std::to_string(l) + ".1", c.mid_channels[i + 1]});
  for (int j = 0; j < nlev; ++j) {
    const int i = nlev - 1 - j;
    for (int l = 0; l < c.num_up_layers; ++l)
      tl.push_back({"ups." + std::to_string(j) + ".t_emb_layers." + std::to_string(l) + ".1", i != 0 ? dc[i - 1] : dc[0]});
  }
  int total = 0;
  for (auto& e : tl) total += e.second;

  float* emb = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * T * 4));
  float* h1 = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * T * 4));
  float* temb = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * T * 4));
  float* temb_silu = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * T * 4));
  float* temb_scratch = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * T * 4 * 3));
  b.tproj_ld = total;
  b.tproj = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * total * 4));
  b.dtproj = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * total * 4));
  b.wg_partial = static_cast<float*>(b.bump.take(kWgradPartialBytes));
  int cmax = 3 * 64;
  for (int i = 0; i < c.n_down_channels; ++i) cmax = std::max(cmax, 3 * dc[i]);
  for (int i = 0; i < c.n_mid_channels; ++i) cmax = std::max(cmax, 3 * c.mid_channels[i]);
  b.red_ws = b.bump.take(groupnorm_bwd_workspace_bytes(B, cmax));
  float* dpred = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * c.im_channels * H * W * 4));
  float* pred_ws = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * c.im_channels * H * W * 4));
  void* mse_scratch = b.bump.take(8192);
  void* bw_scratch = b.bump.take(boundary_wgrad_scratch_bytes());

  float *wcat = nullptr, *bcat = nullptr, *w_out_t = nullptr, *w_in_t = nullptr;
  if (!dry) {
    wcat = static_cast<float*>(b.arena->alloc(static_cast<size_t>(total) * T * 4));
    bcat = static_cast<float*>(b.arena->alloc(static_cast<size_t>(total) * 4));
    w_out_t = static_cast<float*>(b.arena->alloc(static_cast<size_t>(dc[0]) * c.im_channels * 9 * 4));
    w_in_t = static_cast<float*>(b.arena->alloc(static_cast<size_t>(dc[0]) * c.im_channels * 9 * 4));
    if (!wcat || !bcat || !w_out_t || !w_in_t) return 1;
    int off = 0;
    for (auto& e : tl) {
      const float *wsrc = b.P(e.first + ".weight"), *bsrc = b.P(e.first + ".bias");
      if (b.err) return b.err;
      const int rows = e.second, o = off;
      net->repack_ops.push_back([=](cudaStream_t s) {
        WC_CHECK_CUDA(cudaMemcpyAsync(wcat + static_cast<size_t>(o) * T, wsrc, static_cast<size_t>(rows) * T * 4, cudaMemcpyDeviceToDevice, s));
        WC_CHECK_CUDA(cudaMemcpyAsync(bcat + o, bsrc, static_cast<size_t>(rows) * 4, cudaMemcpyDeviceToDevice, s));
        return 0;
      });
      off += rows;
    }
    const float *w1 = b.P("t_proj.0.weight"), *b1 = b.P("t_proj.0.bias"), *w2 = b.P("t_proj.2.weight"), *b2 = b.P("t_proj.2.bias");
    if (b.err) return b.err;
    float* tp = b.tproj;
    wc_unet_train* n = net;
    b.push([=](cudaStream_t s) {
      if (int e = temb_mlp_train(n->t_in, B, T, w1, b1, w2, b2, emb, h1, temb, temb_silu, s)) return e;
      return linear_rows(temb_silu, B, T, wcat, bcat, tp, total, s);
    });
  }

  // ---- level geometry and concat buffers
  std::vector<int> LH(nlev + 1), LW(nlev + 1);
  LH[0] = H; LW[0] = W;
  for (int i = 0; i < nlev; ++i) {
    LH[i + 1] = c.down_sample[i] ? LH[i] / 2 : LH[i];
    LW[i + 1] = c.down_sample[i] ? LW[i] / 2 : LW[i];
  }
  std::vector<Act> cat(nlev);
  for (int i = 0; i < nlev; ++i) cat[i] = b.new_act(LH[i], LW[i], 2 * dc[i]);

  // ---- conv_in
  Act skip0 = slice_act(cat[0], dc[0], dc[0]);
  if (!dry) {
    const float *w = b.P("conv_in.weight"), *bias = b.P("conv_in.bias");
    if (b.err) return b.err;
    wc_unet_train* n = net;
    const int cin = c.im_channels, c0 = dc[0];
    b.push([=](cudaStream_t s) {
      return conv_small_cin(n->x_in, w, bias, nullptr, nullptr, skip0.ptr, B, cin, H, W, c0, 3, 1, 1, skip0.ld, 0, s);
    });
    net->flops_fwd += 2.0 * B * H * W * 9.0 * cin * c0;
  }
  b.tape.push_back([&b, skip0, net, B, H, W, bw_scratch, w_in_t]() {
    Act d = b.grad_written(skip0);
    if (b.dry) return;
    const float* w = b.P("conv_in.weight");
    float *dw = b.G("conv_in.weight"), *db = b.G("conv_in.bias");
    if (b.err) return;
    wc_unet_train* n = net;
    const int cin = net->cfg.im_channels, c0 = d.C;
    b.push([=](cudaStream_t s) { return boundary_wgrad(d.ptr, d.ld, n->x_in, B, H, W, +1, dw, db, bw_scratch, s); }, kOpParam);
    b.ready("conv_in.weight");
    b.ready("conv_in.bias");
    // dL/dx: the 64 -> 3 convolution of d(skip0) with the flipped, transposed conv_in weight (conv_out's forward kernel)
    net->repack_ops.push_back([=](cudaStream_t s) { return flip_transpose_3x3(w, w_in_t, c0, cin, s); });
    b.push([=](cudaStream_t s) {
      return n->dx_out ? conv_small_cout(d.ptr, w_in_t, nullptr, n->dx_out, B, H, W, c0, cin, 3, d.ld, 0, s) : 0;
    }, kOpInput);
  });
  Act cur = skip0;

  auto use_attn = [&](int i) {
    const int res = c.im_size >> i;
    for (int k = 0; k < c.n_attn_resolutions; ++k)
      if (c.attn_resolutions[k] == res) return true;
    return false;
  };

  // ---- down path
  for (int i = 0; i < nlev; ++i) {
    const std::string p = "downs." + std::to_string(i);
    const bool ua = use_attn(i);
    const bool has_next_skip = (i + 1 != nlev);
    Act next_skip;
    if (has_next_skip) next_skip = slice_act(cat[i + 1], dc[i + 1], dc[i + 1]);
    for (int l = 0; l < c.num_down_layers; ++l) {
      const bool final_op = (l + 1 == c.num_down_layers) && !c.down_sample[i] && has_next_skip;
      cur = b.resnet(cur, dc[i + 1], p, l, (final_op && !ua) ? &next_skip : nullptr);
      if (ua) cur = b.attention(cur, p, l, c.num_heads, final_op ? &next_skip : nullptr);
    }
    if (c.down_sample[i]) {
      Act out = has_next_skip ? next_skip : b.new_act(LH[i + 1], LW[i + 1], dc[i + 1]);
      const Act xin = cur;
      const int ch = dc[i + 1];
      b.conv_fwd(xin, p + ".down_sample_conv", ch, 4, 2, 1, b.P(p + ".down_sample_conv.bias"), nullptr, 0, nullptr, nullptr, "", out);
      b.tape.push_back([&b, xin, out, p, ch]() {
        Act dout = b.grad_written(out);
        b.dgrad(dout, p + ".down_sample_conv", ch, ch, 4, 2, xin);
        b.wgrad(xin, dout, 4, 2, 1, p + ".down_sample_conv", nullptr, "");
        b.bias_grad(dout, p + ".down_sample_conv.bias", "", nullptr, 0);
      });
      cur = out;
    }
    if (b.err) return b.err;
  }

  // ---- mid blocks
  for (int i = 0; i + 1 < c.n_mid_channels; ++i) {
    const std::string p = "mids." + std::to_string(i);
    const int cout = c.mid_channels[i + 1];
    const bool last_mid = (i + 2 == c.n_mid_channels);
    const int top = nlev - 1;
    const bool direct = last_mid && !c.down_sample[top];
    Act dest = slice_act(cat[top], 0, dc[top]);
    cur = b.resnet(cur, cout, p, 0, nullptr);
    for (int l = 0; l < c.num_mid_layers; ++l) {
      cur = b.attention(cur, p, l, c.num_heads, nullptr);
      const bool final_op = direct && (l + 1 == c.num_mid_layers);
      cur = b.resnet(cur, cout, p, l + 1, final_op ? &dest : nullptr);
    }
    if (b.err) return b.err;
  }

  // ---- up path
  for (int j = 0; j < nlev; ++j) {
    const int i = nlev - 1 - j;
    const std::string p = "ups." + std::to_string(j);
    const bool ua = use_attn(i);
    const int cout = i != 0 ? dc[i - 1] : dc[0];
    Act first_half = slice_act(cat[i], 0, dc[i]);
    if (c.down_sample[i]) {
      const Act xin = cur;
      const int ch = dc[i];
      b.conv_fwd(xin, p + ".up_sample_conv", ch, 4, 2, 1, b.P(p + ".up_sample_conv.bias"), nullptr, 0, nullptr, nullptr, "", first_half, true);
      b.tape.push_back([&b, xin, first_half, p, ch]() {
        Act dout = b.grad_written(first_half);
        b.dgrad_convT(dout, p + ".up_sample_conv", ch, ch, xin);
        b.wgrad(xin, dout, 4, 2, 1, p + ".up_sample_conv", nullptr, "", true);
        b.bias_grad(dout, p + ".up_sample_conv.bias", "", nullptr, 0);
      });
    } else if (cur.ptr != first_half.ptr) {
      return fail("internal: up block without up-sampling expects its input inside the concat buffer");
    }
    cur = cat[i];
    const bool direct = (i > 0) && !c.down_sample[i - 1];
    Act dest = direct ? slice_act(cat[i - 1], 0, dc[i - 1]) : Act();
    for (int l = 0; l < c.num_up_layers; ++l) {
      const bool final_op = direct && (l + 1 == c.num_up_layers);
      cur = b.resnet(cur, cout, p, l, (final_op && !ua) ? &dest : nullptr);
      if (ua) cur = b.attention(cur, p, l, c.num_heads, final_op ? &dest : nullptr);
    }
    if (b.err) return b.err;
  }

  // ---- norm_out + SiLU + conv_out, MSE loss
  Act fin = b.new_act(H, W, dc[0]);
  void* st_out = b.gn_fwd(cur, fin, "norm_out", 1);
  if (!dry) {
    const float *w = b.P("conv_out.weight"), *bias = b.P("conv_out.bias");
    if (b.err) return b.err;
    wc_unet_train* n = net;
    const int cin = dc[0], co = c.im_channels;
    const size_t numel = static_cast<size_t>(B) * co * H * W;
    net->repack_ops.push_back([=](cudaStream_t s) { return flip_transpose_3x3(w, w_out_t, co, cin, s); });
    b.push([=](cudaStream_t s) {
      float* pred = n->pred_out ? n->pred_out : pred_ws;
      if (int e = conv_small_cout(fin.ptr, w, bias, pred, B, H, W, cin, co, 3, fin.ld, 0, s)) return e;
      if (!n->target) return 0;     // no loss: the backward is seeded with dL/dpred by the caller
      return mse_loss_grad(pred, n->target, dpred, numel, n->grad_scale, n->loss_out, mse_scratch, s);
    });
    net->flops_fwd += 2.0 * B * H * W * 9.0 * cin * co;
  }
  if (b.err) return b.err;

  // =========================================================== backward
  b.in_bwd = true;
  {
    Act dfin = b.grad(fin);
    b.mark(fin);
    if (!dry) {
      float *dw = b.G("conv_out.weight"), *db = b.G("conv_out.bias");
      if (b.err) return b.err;
      const int cin = dc[0], co = c.im_channels;
      wc_unet_train* n = net;
      b.push([=](cudaStream_t s) {
        const float* dp = n->dpred_seed ? n->dpred_seed : dpred;
        return conv_small_cin(dp, w_out_t, nullptr, nullptr, nullptr, dfin.ptr, B, co, H, W, cin, 3, 1, 1, dfin.ld, 0, s);
      });
      b.push([=](cudaStream_t s) {
        const float* dp = n->dpred_seed ? n->dpred_seed : dpred;
        return boundary_wgrad(fin.ptr, fin.ld, dp, B, H, W, -1, dw, db, bw_scratch, s);
      }, kOpParam);
      net->flops_bwd += 4.0 * B * H * W * 9.0 * cin * co;
      b.ready("conv_out.weight");
      b.ready("conv_out.bias");
    }
    b.gn_bwd(cur, dfin, "norm_out", 1, st_out, nullptr);
  }
  for (auto it = b.tape.rbegin(); it != b.tape.rend(); ++it) {
    (*it)();
    if (b.err) return b.err;
  }
  // ---- time-embedding MLP and the concatenated projections
  if (!dry) {
    auto segs_row0 = std::make_shared<std::vector<int>>();
    auto segs_rows = std::make_shared<std::vector<int>>();
    auto segs_dw = std::make_shared<std::vector<float*>>();
    auto segs_db = std::make_shared<std::vector<float*>>();
    int off = 0;
    for (auto& e : tl) {
      segs_row0->push_back(off);
      segs_rows->push_back(e.second);
      segs_dw->push_back(b.G(e.first + ".weight"));
      segs_db->push_back(b.G(e.first + ".bias"));
      off += e.second;
    }
    float *dw1 = b.G("t_proj.0.weight"), *db1 = b.G("t_proj.0.bias"), *dw2 = b.G("t_proj.2.weight"), *db2 = b.G("t_proj.2.bias");
    const float* w2 = b.P("t_proj.2.weight");
    if (b.err) return b.err;
    float* dtp = b.dtproj;
    const int nseg = static_cast<int>(tl.size());
    b.push([=](cudaStream_t s) {
      return temb_backward(dtp, total, B, T, wcat, w2, emb, h1, temb, temb_silu, nseg, segs_row0->data(), segs_rows->data(),
                           segs_dw->data(), segs_db->data(), dw1, db1, dw2, db2, temb_scratch, s);
    }, kOpParam);
    for (auto& e : tl) { b.ready(e.first + ".weight"); b.ready(e.first + ".bias"); }
    b.ready("t_proj.0.weight"); b.ready("t_proj.0.bias"); b.ready("t_proj.2.weight"); b.ready("t_proj.2.bias");
  }
  if (b.err) return b.err;
  if (dry) net->ws_needed = b.bump.used() + 4096;
  else if (b.bump.overflow()) return fail("UNet training workspace too small: need " + std::to_string(b.bump.used()) + " bytes");
  return 0;
}

}  // namespace
}  // namespace wc

using namespace wc;

extern "C" {

int wc_unet_train_create(wc_unet_train** out, const wc_unet_config* cfg, int n_params, const char* const* names,
                         float* const* params, float* const* grads) {
  WC_REQUIRE(out && cfg && names && params && grads, "null argument");
  WC_REQUIRE(cfg->im_channels == 3, "UNet boundary kernels support im_channels == 3");
  WC_REQUIRE(cfg->n_down_channels >= 2 && cfg->n_down_channels <= 8 && cfg->n_mid_channels >= 2, "bad channel lists");
  WC_REQUIRE(cfg->down_channels[0] == 64, "the boundary weight-gradient kernels need down_channels[0] == 64");
  for (int i = 0; i < cfg->n_down_channels; ++i) WC_REQUIRE(cfg->down_channels[i] % 64 == 0, "channels must be multiples of 64");
  for (int i = 0; i < cfg->n_mid_channels; ++i) WC_REQUIRE(cfg->mid_channels[i] % 64 == 0, "channels must be multiples of 64");
  auto net = std::make_unique<wc_unet_train>();
  net->cfg = *cfg;
  for (int i = 0; i < n_params; ++i) {
    net->params.ptr[names[i]] = params[i];
    net->grads[names[i]] = grads[i];
  }
  *out = net.release();
  return 0;
}

void wc_unet_train_destroy(wc_unet_train* net) { delete net; }

size_t wc_unet_train_workspace_bytes(wc_unet_train* net, int batch, int H, int W) {
  const int sB = net->B, sH = net->H, sW = net->W;
  net->B = batch; net->H = H; net->W = W;
  size_t need = 0;
  if (build(net, true, nullptr, 0, nullptr) == 0) need = net->ws_needed;
  net->B = sB; net->H = sH; net->W = sW;
  return need;
}

int wc_unet_train_bind(wc_unet_train* net, int batch, int H, int W, void* workspace, size_t workspace_bytes, void* stream) {
  WC_REQUIRE(net && workspace, "null argument");
  int div = 1;
  for (int i = 0; i + 1 < net->cfg.n_down_channels; ++i) if (net->cfg.down_sample[i]) div *= 2;
  WC_REQUIRE(H % div == 0 && W % div == 0, "H and W must be divisible by the total down-sampling factor");
  net->repack_ops.clear(); net->fwd_ops.clear(); net->bwd_ops.clear(); net->bwd_kind.clear(); net->ready.clear();
  net->arena = std::make_unique<DeviceArena>();
  net->B = batch; net->H = H; net->W = W; net->ws = workspace; net->ws_bytes = workspace_bytes;
  net->flops_fwd = net->flops_bwd = 0;
  set_pack_recorder(&net->repack_ops);
  const int e = build(net, false, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
  set_pack_recorder(nullptr);
  if (e) { net->B = 0; net->fwd_ops.clear(); net->bwd_ops.clear(); net->bwd_kind.clear(); net->repack_ops.clear(); }
  return e;
}

int wc_unet_train_forward(wc_unet_train* net, const float* x, const int64_t* t, const float* target, float* pred_out,
                          float* loss_out, float grad_scale, int repack, void* stream) {
  WC_REQUIRE(net && net->B > 0, "wc_unet_train_forward: not bound");
  WC_REQUIRE(x && t && (target ? loss_out != nullptr : pred_out != nullptr), "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  net->x_in = x; net->t_in = reinterpret_cast<const long long*>(t); net->target = target; net->pred_out = pred_out;
  net->loss_out = loss_out; net->grad_scale = grad_scale;
  if (repack)
    for (auto& op : net->repack_ops)
      if (int e = op(st)) return e;
  for (auto& op : net->fwd_ops)
    if (int e = op(st)) return e;
  return 0;
}

int wc_unet_train_num_backward_ops(const wc_unet_train* net) { return net ? static_cast<int>(net->bwd_ops.size()) : 0; }

int wc_unet_train_backward(wc_unet_train* net, int op_begin, int op_end, void* stream) {
  WC_REQUIRE(net && net->B > 0, "wc_unet_train_backward: not bound");
  WC_REQUIRE(op_begin >= 0 && op_end <= static_cast<int>(net->bwd_ops.size()) && op_begin <= op_end, "bad op range");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  net->dpred_seed = nullptr;
  net->dx_out = nullptr;
  for (int i = op_begin; i < op_end; ++i)
    if (int e = net->bwd_ops[i](st)) return e;
  return 0;
}

int wc_unet_train_backward_seeded(wc_unet_train* net, const float* dpred, float* dx, int param_grads, void* stream) {
  WC_REQUIRE(net && net->B > 0, "wc_unet_train_backward_seeded: not bound");
  WC_REQUIRE(dpred, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  net->dpred_seed = dpred;
  net->dx_out = dx;
  int err = 0;
  for (size_t i = 0; i < net->bwd_ops.size() && !err; ++i)
    if (param_grads || net->bwd_kind[i] != kOpParam) err = net->bwd_ops[i](st);
  net->dpred_seed = nullptr;
  net->dx_out = nullptr;
  return err;
}

int wc_unet_train_grad_ready_op(const wc_unet_train* net, const char* name) {
  if (!net || !name) return -1;
  auto it = net->ready.find(name);
  return it == net->ready.end() ? -1 : it->second;
}

double wc_unet_train_flops(const wc_unet_train* net, int backward) {
  return net ? (backward ? net->flops_bwd : net->flops_fwd) : 0.0;
}

}  // extern "C"
