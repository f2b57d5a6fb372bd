// UNet forward as a static launch plan (reference: diffusion_model/models/unet_base.py:372-488).
// The plan is built once per (batch, H, W, workspace) binding: tensor maps, packed weights, epilogue wiring.
// A forward is then a fixed sequence of kernel launches on one stream (CUDA-graph capturable, no host sync).
//
// Dataflow per ResNet sub-layer (unet_base.py:146-150), 4 launches (+2 tiny GN stat launches):
//   GN+SiLU -> conv3x3 [+bias +t-emb row bias] -> GN+SiLU -> conv3x3 [+bias] with the 1x1 residual conv of the
//   block input fused as a tenth tap (its bias folded into the epilogue bias).
// Attention sub-layer (:153-161): GN -> QKV projection (epilogue scatters Q, K, V^T per head) -> flash attention
//   -> out-projection with the residual add fused in the epilogue.
// The topology walk, with the skip routing through the concat buffers, is unet_plan.cuh's.
#include "unet_plan.cuh"

namespace wc {

int groupnorm_silu(const __nv_bfloat16* x, __nv_bfloat16* y, int B, int HW, int C, int ld, int ldy, const float* gamma,
                   const float* beta, float eps, int silu, void* workspace, cudaStream_t st);
size_t groupnorm_workspace_bytes(int B);
int attention_forward(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, __nv_bfloat16* out, int B,
                      int heads, int ntok, int hd, int ldo, cudaStream_t st, float* lse = nullptr, float scale = 0.f);
double attention_flops(int B, int heads, int ntok, int hd);
int conv_small_cin(const float* x, const float* w, const float* bias, const float* scale, const float* shift,
                   __nv_bfloat16* y, int B, int Cin, int H, int W, int Cout, int K, int stride, int pad, int ldy,
                   int relu, cudaStream_t st, const float* prelu = nullptr);
int conv_small_cout(const __nv_bfloat16* x, const float* w, const float* bias, float* y, int B, int H, int W, int Cin,
                    int Cout, int K, int ldx, int tanh_out, cudaStream_t st);
int temb_mlp(const long long* t, int Bt, int dim, const float* w1, const float* b1, const float* w2, const float* b2,
             float* temb, float* temb_silu, cudaStream_t st);
int linear_rows(const float* in, int Bt, int dim, const float* w, const float* bias, float* out, int N, cudaStream_t st);

namespace {

__global__ void add_vec_kernel(const float* a, const float* b, float* o, int n) {
  pdl_prologue();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = a[i] + b[i];
}

}  // namespace

}  // namespace wc

struct wc_unet {
  wc_unet_config cfg;
  wc::ParamTable params;
  std::unique_ptr<wc::DeviceArena> arena;  // packed weights of the current binding
  struct Geom {
    int B, H, W, n_t;
    bool operator==(const Geom& o) const { return B == o.B && H == o.H && W == o.W && n_t == o.n_t; }
  } geom{};
  void* ws = nullptr;
  size_t ws_bytes = 0;
  const float* x_in = nullptr;
  float* y_out = nullptr;
  const long long* t_in = nullptr;
  wc::OpList ops;
  double flops = 0;
  void reset_plan() { ops.clear(); flops = 0; }
};

namespace wc {
namespace {

struct Builder : PlanBuilder<wc_unet> {
  Builder(wc_unet* out, int B, int n_t, cudaStream_t st) : PlanBuilder(out, B, st), n_t(n_t) {}
  int n_t;
  float* tproj = nullptr;
  int tproj_ld = 0;
  int temb_off = 0;
  void* gn_ws = nullptr;

  void push(std::function<int(cudaStream_t)> f) {
    if (!dry) net->ops.push_back(std::move(f));
  }

  void gn(const Act& x, const Act& y, const std::string& prefix, int silu) {
    const float* g = P(prefix + ".weight");
    const float* b = P(prefix + ".bias");
    void* ws = gn_ws;
    push([=](cudaStream_t s) {
      return groupnorm_silu(x.ptr, y.ptr, x.B, x.H * x.W, x.C, x.ld, y.ld, g, b, 1e-5f, silu, ws, s);
    });
  }

  void conv(const Act& x, const std::string& wname, int cout, int K, int stride, int pad, const float* bias,
            const float* rowbias, int ldrb, const Act* res, const Act* x2, const std::string& w2name, const Act& out) {
    if (dry) return;
    WeightSrc w;
    w.w = P(wname + ".weight"); w.d0 = cout; w.d1 = x.C; w.KH = w.KW = K;
    WeightSrc w2;
    if (x2) { w2.w = P(w2name + ".weight"); w2.d0 = cout; w2.d1 = x2->C; }
    if (err) return;
    ConvGeom g; g.K = K; g.stride = stride; g.pad = pad; g.dil = 1;
    Epilogue ep; ep.bias = bias; ep.rowbias = rowbias; ep.ldrb = ldrb; ep.res = res;
    OutSpec os; os.mode = kOutNHWC; os.out = out;
    auto op = std::make_shared<ConvOp>();
    if (int e = build_conv(op.get(), arena, x, w, g, cout, x2, x2 ? &w2 : nullptr, ep, os, st)) { err = e; return; }
    net->flops += op->flops;
    push([op](cudaStream_t s) { return op->run(s); });
  }

  // ---- hooks of walk_unet (unet_plan.cuh)
  // conv_in (NCHW fp32 -> NHWC bf16)
  void conv_in(const Act& skip0) {
    if (dry) return;
    const float *w = P("conv_in.weight"), *bias = P("conv_in.bias");
    if (err) return;
    wc_unet* n = net;
    const int B = skip0.B, H = skip0.H, W = skip0.W, cin = n->cfg.im_channels, c0 = skip0.C;
    push([=](cudaStream_t s) {
      return conv_small_cin(n->x_in, w, bias, nullptr, nullptr, skip0.ptr, B, cin, H, W, c0, 3, 1, 1, skip0.ld, 0, s);
    });
    net->flops += 2.0 * B * H * W * 9.0 * cin * c0;
  }

  // One ResNet sub-layer; writes its output to `dest` if given, else to a fresh buffer.
  Act resnet(const Act& x, int cout, const std::string& p, int l, const Act* dest) {
    const std::string ls = std::to_string(l);
    Act a1 = act(x.H, x.W, x.C);
    gn(x, a1, p + ".resnet_conv_first." + ls + ".0", 1);
    Act h = act(x.H, x.W, cout);
    const float* rb = nullptr;
    if (!dry) {
      rb = tproj + temb_off;
      temb_off += cout;
    }
    conv(a1, p + ".resnet_conv_first." + ls + ".2", cout, 3, 1, 1, P(p + ".resnet_conv_first." + ls + ".2.bias"), rb,
         n_t == 1 ? 0 : tproj_ld, nullptr, nullptr, "", h);
    Act a2 = act(x.H, x.W, cout);
    gn(h, a2, p + ".resnet_conv_second." + ls + ".0", 1);
    Act out = dest ? *dest : act(x.H, x.W, cout);
    float* bsum = nullptr;
    if (!dry) {
      bsum = static_cast<float*>(arena->alloc(cout * sizeof(float)));
      const float* b2 = P(p + ".resnet_conv_second." + ls + ".2.bias");
      const float* br = P(p + ".residual_input_conv." + ls + ".bias");
      if (!bsum || err) { if (!err) err = 1; return out; }
      launch_k(add_vec_kernel, (cout + 255) / 256, 256, 0, st, b2, br, bsum, cout);
    }
    conv(a2, p + ".resnet_conv_second." + ls + ".2", cout, 3, 1, 1, bsum, nullptr, 0, nullptr, &x,
         p + ".residual_input_conv." + ls, out);
    return out;
  }

  Act attention(const Act& x, const std::string& p, int l, int heads, const Act* dest) {
    const std::string ls = std::to_string(l);
    const int C = x.C, hd = C / heads, ntok = x.H * x.W;
    Act a = act(x.H, x.W, C);
    gn(x, a, p + ".attention_norms." + ls, 0);
    const size_t per = static_cast<size_t>(B) * ntok * C;
    auto* q = static_cast<__nv_bfloat16*>(bump.take(per * 2));
    auto* k = static_cast<__nv_bfloat16*>(bump.take(per * 2));
    auto* vt = static_cast<__nv_bfloat16*>(bump.take(per * 2));
    Act o = act(x.H, x.W, C);
    Act out = dest ? *dest : act(x.H, x.W, C);
    if (dry) return out;
    const std::string ap = p + ".attentions." + ls;
    {
      WeightSrc w; w.w = P(ap + ".in_proj_weight"); w.d0 = 3 * C; w.d1 = C;
      ConvGeom g; g.K = 1; g.stride = 1; g.pad = 0; g.dil = 1;
      Epilogue ep; ep.bias = P(ap + ".in_proj_bias");
      OutSpec os; os.mode = kOutQKV; os.q = q; os.k = k; os.vt = vt; os.heads = heads; os.hd = hd;
      os.q_scale = 1.4426950408889634f / sqrtf(static_cast<float>(hd));   // attention then runs with a unit log2-domain scale
      if (err) return out;
      auto op = std::make_shared<ConvOp>();
      if (int e = build_conv(op.get(), arena, a, w, g, 3 * C, nullptr, nullptr, ep, os, st)) { err = e; return out; }
      net->flops += op->flops;
      push([op](cudaStream_t s) { return op->run(s); });
    }
    {
      const int Bc = B;
      net->flops += attention_flops(B, heads, ntok, hd);
      push([=](cudaStream_t s) { return attention_forward(q, k, vt, o.ptr, Bc, heads, ntok, hd, o.ld, s, nullptr, kAttnScalePrescaled); });
    }
    conv(o, ap + ".out_proj", C, 1, 1, 0, P(ap + ".out_proj.bias"), nullptr, 0, &x, nullptr, "", out);
    return out;
  }

  void down_sample(const Act& x, const std::string& p, int ch, const Act& out) {
    conv(x, p + ".down_sample_conv", ch, 4, 2, 1, P(p + ".down_sample_conv.bias"), nullptr, 0, nullptr, nullptr, "", out);
  }

  void up_sample(const Act& x, const std::string& p, int ch, const Act& out) {
    if (dry) return;
    WeightSrc w; w.w = P(p + ".up_sample_conv.weight"); w.d0 = ch; w.d1 = ch; w.KH = w.KW = 4; w.transpose = 1;
    Epilogue ep; ep.bias = P(p + ".up_sample_conv.bias");
    OutSpec os; os.mode = kOutNHWC; os.out = out;
    if (err) return;
    auto op = std::make_shared<ConvOp>();
    if (int e = build_conv_transposed_s2(op.get(), arena, x, w, 4, 1, ch, ep, os, st)) { err = e; return; }
    net->flops += op->flops;
    push([op](cudaStream_t s) { return op->run(s); });
  }
};

int build(const wc_unet& cfg, const wc_unet::Geom& geo, wc_unet* net, cudaStream_t st, size_t* need) {
  const wc_unet_config& c = cfg.cfg;
  const int B = geo.B, H = geo.H, W = geo.W;
  Builder b(net, B, geo.n_t, st);
  const int T = c.time_emb_dim;

  // ---- time embedding: MLP + all t_emb_layers projections (concatenated) in two launches
  const auto tl = temb_layers(c);
  int total = 0;
  for (auto& e : tl) total += e.second;
  float* temb = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * T * 4));
  float* temb_silu = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * T * 4));
  b.tproj_ld = total;
  b.tproj = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * total * 4));
  b.gn_ws = b.bump.take(groupnorm_workspace_bytes(B));
  if (!b.dry) {
    float* wcat = static_cast<float*>(b.arena->alloc(static_cast<size_t>(total) * T * 4));
    float* bcat = static_cast<float*>(b.arena->alloc(static_cast<size_t>(total) * 4));
    if (!wcat || !bcat) return 1;
    int off = 0;
    for (auto& e : tl) {
      const float *wsrc = b.P(e.first + ".weight"), *bsrc = b.P(e.first + ".bias");
      if (b.err) return b.err;
      WC_CHECK_CUDA(cudaMemcpyAsync(wcat + static_cast<size_t>(off) * T, wsrc, static_cast<size_t>(e.second) * T * 4, cudaMemcpyDeviceToDevice, st));
      WC_CHECK_CUDA(cudaMemcpyAsync(bcat + off, bsrc, static_cast<size_t>(e.second) * 4, cudaMemcpyDeviceToDevice, st));
      off += e.second;
    }
    const float *w1 = b.P("t_proj.0.weight"), *b1 = b.P("t_proj.0.bias"), *w2 = b.P("t_proj.2.weight"), *b2 = b.P("t_proj.2.bias");
    if (b.err) return b.err;
    float* tp = b.tproj;
    wc_unet* n = net;
    b.push([=](cudaStream_t s) {
      if (int e = temb_mlp(n->t_in, n->geom.n_t, T, w1, b1, w2, b2, temb, temb_silu, s)) return e;
      return linear_rows(temb_silu, n->geom.n_t, T, wcat, bcat, tp, total, s);
    });
  }

  Act cur = walk_unet(b, c, H, W);
  if (b.err) return b.err;

  // ---- norm_out + SiLU + conv_out (unet_base.py:483-485), NHWC bf16 -> NCHW fp32
  const int* dc = c.down_channels;
  Act fin = b.act(H, W, dc[0]);
  b.gn(cur, fin, "norm_out", 1);
  if (!b.dry) {
    const float *w = b.P("conv_out.weight"), *bias = b.P("conv_out.bias");
    if (b.err) return b.err;
    wc_unet* n = net;
    const int cin = dc[0], co = c.im_channels;
    b.push([=](cudaStream_t s) { return conv_small_cout(fin.ptr, w, bias, n->y_out, B, H, W, cin, co, 3, fin.ld, 0, s); });
    net->flops += 2.0 * B * H * W * 9.0 * cin * co;
  }
  return b.finish("UNet", need);
}

}  // namespace
}  // namespace wc

using namespace wc;

extern "C" {

int wc_unet_create(wc_unet** out, const wc_unet_config* cfg, int n_params, const char* const* names,
                   const float* const* ptrs, const int64_t* numels, void* stream) {
  (void)numels; (void)stream;
  WC_REQUIRE(out && cfg && names && ptrs, "null argument");
  if (int e = check_unet_config(*cfg)) return e;
  auto net = std::make_unique<wc_unet>();
  net->cfg = *cfg;
  for (int i = 0; i < n_params; ++i) net->params.ptr[names[i]] = ptrs[i];
  *out = net.release();
  return 0;
}

void wc_unet_destroy(wc_unet* net) { delete net; }

size_t wc_unet_workspace_bytes(const wc_unet* net, int batch, int H, int W) {
  return plan_workspace_bytes(*net, {batch, H, W, batch}, build);
}

int wc_unet_forward(wc_unet* net, const float* x, const int64_t* t, int n_t, float* out, int batch, int H, int W,
                    void* workspace, size_t workspace_bytes, void* stream) {
  WC_REQUIRE(net && x && t && out && workspace, "null argument");
  WC_REQUIRE(n_t == 1 || n_t == batch, "t must have 1 or batch entries");
  if (int e = check_unet_hw(net->cfg, H, W)) return e;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = bind(net, {batch, H, W, n_t}, workspace, workspace_bytes, st, build)) return e;
  net->x_in = x; net->y_out = out; net->t_in = reinterpret_cast<const long long*>(t);
  return run_ops(net->ops, st);
}

double wc_unet_flops(const wc_unet* net) { return net ? net->flops : 0.0; }
int wc_unet_launches(const wc_unet* net) { return net ? static_cast<int>(net->ops.size()) : 0; }

}  // extern "C"
