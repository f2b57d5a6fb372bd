// UNet forward as a static launch plan (reference: diffusion_model/models/unet_base.py:372-488).
// The plan is built once per (batch, H, W, workspace) binding: tensor maps, packed weights, epilogue wiring.
// A forward is then a fixed sequence of kernel launches on one stream (CUDA-graph capturable, no host sync).
//
// Dataflow per ResNet sub-layer (unet_base.py:146-150), 4 launches (+2 tiny GN stat launches):
//   GN+SiLU -> conv3x3 [+bias +t-emb row bias] -> GN+SiLU -> conv3x3 [+bias] with the 1x1 residual conv of the
//   block input fused as a tenth tap (its bias folded into the epilogue bias).
// Attention sub-layer (:153-161): GN -> QKV projection (epilogue scatters Q, K, V^T per head) -> flash attention
//   -> out-projection with the residual add fused in the epilogue.
// Skip connections are written by their producers directly into the second half of the up-path concat buffers,
// and the up-sampling transposed conv writes the first half (unet_base.py:348-349), so torch.cat never runs.
#include <functional>
#include <string>
#include <unordered_map>

#include "conv.cuh"
#include "../../include/wc_b200.h"

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

class Bump {
 public:
  Bump(void* base, size_t cap) : base_(static_cast<uint8_t*>(base)), cap_(cap) {}
  void* take(size_t bytes) {
    const size_t off = (off_ + 255) & ~static_cast<size_t>(255);
    off_ = off + bytes;
    if (!base_ || off_ > cap_) { overflow_ = true; return nullptr; }
    return base_ + off;
  }
  size_t used() const { return off_; }
  bool overflow() const { return overflow_; }

 private:
  uint8_t* base_;
  size_t cap_, off_ = 0;
  bool overflow_ = false;
};

}  // namespace

}  // namespace wc

struct wc_unet {
  wc_unet_config cfg;
  std::unordered_map<std::string, const float*> params;
  std::unordered_map<std::string, int64_t> numels;
  std::unique_ptr<wc::DeviceArena> static_arena;  // concatenated t-emb weights
  std::unique_ptr<wc::DeviceArena> bind_arena;    // packed conv weights of the current binding
  float* temb_wcat = nullptr;
  float* temb_bcat = nullptr;
  int temb_total = 0;
  std::vector<std::pair<std::string, int>> temb_layers;  // (prefix, Cout) in execution order
  // binding
  int B = 0, H = 0, W = 0, n_t = 0;
  void* ws = nullptr;
  size_t ws_bytes = 0;
  const float* x_in = nullptr;
  float* y_out = nullptr;
  const long long* t_in = nullptr;
  std::vector<std::function<int(cudaStream_t)>> ops;
  double flops = 0;
  size_t ws_needed = 0;
};

namespace wc {
namespace {

struct Builder {
  wc_unet* net;
  Bump bump;
  DeviceArena* arena;
  cudaStream_t st;
  bool dry;  // dry run: only measure workspace
  int B, n_t;
  float* tproj = nullptr;
  int tproj_ld = 0;
  int temb_cursor = 0, temb_off = 0;
  void* gn_ws = nullptr;
  int err = 0;

  const float* P(const std::string& name) {
    auto it = net->params.find(name);
    if (it == net->params.end()) {
      if (!err) err = fail("missing parameter '" + name + "'");
      return nullptr;
    }
    return it->second;
  }
  Act new_act(int H, int W, int C) {
    Act a;
    a.B = B; a.H = H; a.W = W; a.C = C; a.ld = C;
    a.ptr = static_cast<__nv_bfloat16*>(bump.take(a.pixels() * C * sizeof(__nv_bfloat16)));
    return a;
  }
  static Act slice(const Act& a, int c0, int C) {
    Act v = a;
    v.ptr = a.ptr ? a.ptr + c0 : nullptr;
    v.C = C;
    return v;
  }
  void push(std::function<int(cudaStream_t)> f) {
    if (!dry) net->ops.push_back(std::move(f));
  }

  void gn(const Act& x, const Act& y, const std::string& prefix, int silu) {
    const float* g = dry ? nullptr : P(prefix + ".weight");
    const float* b = dry ? nullptr : P(prefix + ".bias");
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

  // One ResNet sub-layer; writes its output to `dest` if given, else to a fresh buffer.
  Act resnet(const Act& x, int cout, const std::string& p, int l, const Act* dest) {
    const std::string ls = std::to_string(l);
    Act a1 = new_act(x.H, x.W, x.C);
    gn(x, a1, p + ".resnet_conv_first." + ls + ".0", 1);
    Act h = new_act(x.H, x.W, cout);
    const float* rb = nullptr;
    if (!dry) {
      rb = tproj + temb_off;
      temb_off += cout;
    }
    conv(a1, p + ".resnet_conv_first." + ls + ".2", cout, 3, 1, 1, dry ? nullptr : P(p + ".resnet_conv_first." + ls + ".2.bias"),
         rb, n_t == 1 ? 0 : tproj_ld, nullptr, nullptr, "", h);
    Act a2 = new_act(x.H, x.W, cout);
    gn(h, a2, p + ".resnet_conv_second." + ls + ".0", 1);
    Act out = dest ? *dest : new_act(x.H, x.W, cout);
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
    Act a = new_act(x.H, x.W, C);
    gn(x, a, p + ".attention_norms." + ls, 0);
    const size_t per = static_cast<size_t>(B) * ntok * C;
    auto* q = static_cast<__nv_bfloat16*>(bump.take(per * 2));
    auto* k = static_cast<__nv_bfloat16*>(bump.take(per * 2));
    auto* vt = static_cast<__nv_bfloat16*>(bump.take(per * 2));
    Act o = new_act(x.H, x.W, C);
    Act out = dest ? *dest : new_act(x.H, x.W, C);
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
};

int build(wc_unet* net, bool dry, void* ws, size_t ws_bytes, cudaStream_t st) {
  const wc_unet_config& c = net->cfg;
  const int B = net->B, H = net->H, W = net->W;
  Builder b{net, Bump(ws, dry ? ~static_cast<size_t>(0) : ws_bytes), net->bind_arena.get(), st, dry, B, net->n_t};
  if (dry) b.bump = Bump(reinterpret_cast<void*>(static_cast<uintptr_t>(4096)), ~static_cast<size_t>(0) >> 1);
  const int nlev = c.n_down_channels - 1;
  const int* dc = c.down_channels;
  const int T = c.time_emb_dim;

  // ---- time embedding: MLP + all t_emb_layers projections in two launches
  float* temb = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * T * 4));
  float* temb_silu = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * T * 4));
  b.tproj_ld = net->temb_total;
  b.tproj = static_cast<float*>(b.bump.take(static_cast<size_t>(B) * net->temb_total * 4));
  b.gn_ws = b.bump.take(groupnorm_workspace_bytes(B));
  if (!dry) {
    const float *w1 = b.P("t_proj.0.weight"), *b1 = b.P("t_proj.0.bias"), *w2 = b.P("t_proj.2.weight"), *b2 = b.P("t_proj.2.bias");
    if (b.err) return b.err;
    float* tp = b.tproj;
    const float *wcat = net->temb_wcat, *bcat = net->temb_bcat;
    const int total = net->temb_total;
    wc_unet* n = net;
    b.push([=](cudaStream_t s) {
      if (int e = temb_mlp(n->t_in, n->n_t, T, w1, b1, w2, b2, temb, temb_silu, s)) return e;
      return linear_rows(temb_silu, n->n_t, T, wcat, bcat, tp, total, s);
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

  // ---- conv_in (NCHW fp32 -> NHWC bf16), written straight into the level-0 skip slot
  Act skip0 = Builder::slice(cat[0], dc[0], dc[0]);
  if (!dry) {
    const float *w = b.P("conv_in.weight"), *bias = b.P("conv_in.bias");
    if (b.err) return b.err;
    wc_unet* n = net;
    const int cin = c.im_channels, c0 = dc[0];
    b.push([=](cudaStream_t s) {
      return conv_small_cin(n->x_in, w, bias, nullptr, nullptr, skip0.ptr, B, cin, H, W, c0, 3, 1, 1, skip0.ld, 0, s);
    });
    net->flops += 2.0 * B * H * W * 9.0 * cin * c0;
  }
  Act cur = skip0;

  auto use_attn = [&](int i) {
    const int res = c.im_size >> i;
    for (int k = 0; k < c.n_attn_resolutions; ++k)
      if (c.attn_resolutions[k] == res) return true;
    return false;
  };

  // ---- down path (unet_base.py:466-468, DownBlock.forward :131-164)
  for (int i = 0; i < nlev; ++i) {
    const std::string p = "downs." + std::to_string(i);
    const bool ua = use_attn(i);
    const bool last_level = (i + 1 == nlev);
    // The block output is the skip of level i+1 (if it exists); route it into that concat buffer.
    Act next_skip;
    const bool has_next_skip = !last_level;
    if (has_next_skip) next_skip = Builder::slice(cat[i + 1], dc[i + 1], dc[i + 1]);
    for (int l = 0; l < c.num_down_layers; ++l) {
      const bool final_op = (l + 1 == c.num_down_layers) && !c.down_sample[i] && has_next_skip;
      cur = b.resnet(cur, dc[i + 1], p, l, (final_op && !ua) ? &next_skip : nullptr);
      if (ua) cur = b.attention(cur, p, l, c.num_heads, final_op ? &next_skip : nullptr);
    }
    if (c.down_sample[i]) {
      Act out = has_next_skip ? next_skip : b.new_act(LH[i + 1], LW[i + 1], dc[i + 1]);
      b.conv(cur, p + ".down_sample_conv", dc[i + 1], 4, 2, 1, dry ? nullptr : b.P(p + ".down_sample_conv.bias"), nullptr, 0,
             nullptr, nullptr, "", out);
      cur = out;
    }
    if (b.err) return b.err;
  }

  // ---- mid blocks (MidBlock.forward :228-268)
  for (int i = 0; i + 1 < c.n_mid_channels; ++i) {
    const std::string p = "mids." + std::to_string(i);
    const int cout = c.mid_channels[i + 1];
    const bool last_mid = (i + 2 == c.n_mid_channels);
    // The last mid output feeds the first up block; if that block does not up-sample it is the first half of
    // its concat buffer.
    const int top = nlev - 1;
    const bool direct = last_mid && !c.down_sample[top];
    Act dest = Builder::slice(cat[top], 0, dc[top]);
    cur = b.resnet(cur, cout, p, 0, nullptr);
    for (int l = 0; l < c.num_mid_layers; ++l) {
      cur = b.attention(cur, p, l, c.num_heads, nullptr);
      const bool final_op = direct && (l + 1 == c.num_mid_layers);
      cur = b.resnet(cur, cout, p, l + 1, final_op ? &dest : nullptr);
    }
    if (b.err) return b.err;
  }

  // ---- up path (UpBlock.forward :336-369)
  for (int j = 0; j < nlev; ++j) {
    const int i = nlev - 1 - j;
    const std::string p = "ups." + std::to_string(j);
    const bool ua = use_attn(i);
    const int cout = i != 0 ? dc[i - 1] : dc[0];
    Act first_half = Builder::slice(cat[i], 0, dc[i]);
    if (c.down_sample[i]) {
      if (!dry) {
        WeightSrc w; w.w = b.P(p + ".up_sample_conv.weight"); w.d0 = dc[i]; w.d1 = dc[i]; w.KH = w.KW = 4; w.transpose = 1;
        Epilogue ep; ep.bias = b.P(p + ".up_sample_conv.bias");
        OutSpec os; os.mode = kOutNHWC; os.out = first_half;
        if (b.err) return b.err;
        auto op = std::make_shared<ConvOp>();
        if (int e = build_conv_transposed_s2(op.get(), b.arena, cur, w, 4, 1, dc[i], ep, os, st)) return e;
        net->flops += op->flops;
        b.push([op](cudaStream_t s) { return op->run(s); });
      }
    } else if (cur.ptr != first_half.ptr) {
      return fail("internal: up block without up-sampling expects its input inside the concat buffer");
    }
    cur = cat[i];
    // If the next (finer) up block does not up-sample, this block's output is the first half of its concat buffer.
    const bool direct = (i > 0) && !c.down_sample[i - 1];
    Act dest = direct ? Builder::slice(cat[i - 1], 0, dc[i - 1]) : Act();
    for (int l = 0; l < c.num_up_layers; ++l) {
      const bool final_op = direct && (l + 1 == c.num_up_layers);
      cur = b.resnet(cur, cout, p, l, (final_op && !ua) ? &dest : nullptr);
      if (ua) cur = b.attention(cur, p, l, c.num_heads, final_op ? &dest : nullptr);
    }
    if (b.err) return b.err;
  }

  // ---- norm_out + SiLU + conv_out (unet_base.py:483-485), NHWC bf16 -> NCHW fp32
  Act fin = b.new_act(H, W, dc[0]);
  b.gn(cur, fin, "norm_out", 1);
  if (!dry) {
    const float *w = b.P("conv_out.weight"), *bias = b.P("conv_out.bias");
    if (b.err) return b.err;
    wc_unet* n = net;
    const int cin = dc[0], co = c.im_channels;
    b.push([=](cudaStream_t s) { return conv_small_cout(fin.ptr, w, bias, n->y_out, B, H, W, cin, co, 3, fin.ld, 0, s); });
    net->flops += 2.0 * B * H * W * 9.0 * cin * co;
  }
  if (b.err) return b.err;
  if (dry) {
    net->ws_needed = b.bump.used() + 4096;
  } else if (b.bump.overflow()) {
    return fail("UNet workspace too small: need " + std::to_string(b.bump.used()) + " bytes");
  }
  return 0;
}

}  // namespace
}  // namespace wc

using namespace wc;

extern "C" {

int wc_unet_create(wc_unet** out, const wc_unet_config* cfg, int n_params, const char* const* names,
                   const float* const* ptrs, const int64_t* numels, void* stream) {
  WC_REQUIRE(out && cfg && names && ptrs, "null argument");
  WC_REQUIRE(cfg->im_channels == 3, "UNet boundary kernels support im_channels == 3");
  WC_REQUIRE(cfg->n_down_channels >= 2 && cfg->n_down_channels <= 8 && cfg->n_mid_channels >= 2, "bad channel lists");
  for (int i = 0; i < cfg->n_down_channels; ++i) WC_REQUIRE(cfg->down_channels[i] % 64 == 0, "channels must be multiples of 64");
  for (int i = 0; i < cfg->n_mid_channels; ++i) WC_REQUIRE(cfg->mid_channels[i] % 64 == 0, "channels must be multiples of 64");
  auto net = std::make_unique<wc_unet>();
  net->cfg = *cfg;
  for (int i = 0; i < n_params; ++i) {
    net->params[names[i]] = ptrs[i];
    net->numels[names[i]] = numels ? numels[i] : 0;
  }
  // Concatenate every t_emb_layers Linear (unet_base.py:96-98) in execution order: one launch projects them all.
  const wc_unet_config& c = *cfg;
  const int nlev = c.n_down_channels - 1;
  for (int i = 0; i < nlev; ++i)
    for (int l = 0; l < c.num_down_layers; ++l)
      net->temb_layers.push_back({"downs." + std::to_string(i) + ".t_emb_layers." + std::to_string(l) + ".1", c.down_channels[i + 1]});
  for (int i = 0; i + 1 < c.n_mid_channels; ++i)
    for (int l = 0; l < c.num_mid_layers + 1; ++l)
      net->temb_layers.push_back({"mids." + std::to_string(i) + ".t_emb_layers." + std::to_string(l) + ".1", c.mid_channels[i + 1]});
  for (int j = 0; j < nlev; ++j) {
    const int i = nlev - 1 - j;
    for (int l = 0; l < c.num_up_layers; ++l)
      net->temb_layers.push_back({"ups." + std::to_string(j) + ".t_emb_layers." + std::to_string(l) + ".1", i != 0 ? c.down_channels[i - 1] : c.down_channels[0]});
  }
  int total = 0;
  for (auto& tl : net->temb_layers) total += tl.second;
  net->temb_total = total;
  net->static_arena = std::make_unique<DeviceArena>();
  const int T = c.time_emb_dim;
  net->temb_wcat = static_cast<float*>(net->static_arena->alloc(static_cast<size_t>(total) * T * 4));
  net->temb_bcat = static_cast<float*>(net->static_arena->alloc(static_cast<size_t>(total) * 4));
  if (!net->temb_wcat || !net->temb_bcat) return 1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int off = 0;
  for (auto& tl : net->temb_layers) {
    auto wi = net->params.find(tl.first + ".weight"), bi = net->params.find(tl.first + ".bias");
    if (wi == net->params.end() || bi == net->params.end()) return fail("missing parameter '" + tl.first + "'");
    WC_CHECK_CUDA(cudaMemcpyAsync(net->temb_wcat + static_cast<size_t>(off) * T, wi->second, static_cast<size_t>(tl.second) * T * 4, cudaMemcpyDeviceToDevice, st));
    WC_CHECK_CUDA(cudaMemcpyAsync(net->temb_bcat + off, bi->second, static_cast<size_t>(tl.second) * 4, cudaMemcpyDeviceToDevice, st));
    off += tl.second;
  }
  *out = net.release();
  return 0;
}

void wc_unet_destroy(wc_unet* net) { delete net; }

size_t wc_unet_workspace_bytes(const wc_unet* net_c, int batch, int H, int W) {
  wc_unet* net = const_cast<wc_unet*>(net_c);
  const int sB = net->B, sH = net->H, sW = net->W, sn = net->n_t;
  net->B = batch; net->H = H; net->W = W; net->n_t = batch;
  size_t need = 0;
  if (build(net, true, nullptr, 0, nullptr) == 0) need = net->ws_needed;
  net->B = sB; net->H = sH; net->W = sW; net->n_t = sn;
  return need;
}

int wc_unet_forward(wc_unet* net, const float* x, const int64_t* t, int n_t, float* out, int batch, int H, int W,
                    void* workspace, size_t workspace_bytes, void* stream) {
  WC_REQUIRE(net && x && t && out && workspace, "null argument");
  WC_REQUIRE(n_t == 1 || n_t == batch, "t must have 1 or batch entries");
  int div = 1;
  for (int i = 0; i + 1 < net->cfg.n_down_channels; ++i) if (net->cfg.down_sample[i]) div *= 2;
  WC_REQUIRE(H % div == 0 && W % div == 0, "H and W must be divisible by the total down-sampling factor");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (net->B != batch || net->H != H || net->W != W || net->n_t != n_t || net->ws != workspace || net->ws_bytes != workspace_bytes) {
    net->ops.clear();
    net->bind_arena = std::make_unique<DeviceArena>();
    net->B = batch; net->H = H; net->W = W; net->n_t = n_t; net->ws = workspace; net->ws_bytes = workspace_bytes;
    net->flops = 0;
    if (int e = build(net, false, workspace, workspace_bytes, st)) {
      net->B = 0;
      net->ops.clear();
      return e;
    }
  }
  net->x_in = x; net->y_out = out; net->t_in = reinterpret_cast<const long long*>(t);
  for (auto& op : net->ops)
    if (int e = op(st)) return e;
  return 0;
}

double wc_unet_flops(const wc_unet* net) { return net ? net->flops : 0.0; }
int wc_unet_launches(const wc_unet* net) { return net ? static_cast<int>(net->ops.size()) : 0; }

}  // extern "C"
