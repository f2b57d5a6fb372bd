#include "conv.cuh"

#include <algorithm>

namespace wc {

int pack_tap(__nv_bfloat16* dst, int ldk, int koff, const float* src, int Nn, int Cc, int Cpad, int KH, int KW, int ky,
             int kx, int transpose, const float* scale, cudaStream_t st);
int pack_taps(__nv_bfloat16* dst, int ldk, int ntaps, const float* const* src, const float* const* scale, const int* params,
              cudaStream_t st);

DeviceArena::~DeviceArena() {
  for (void* p : ptrs_) cudaFree(p);
}
void* DeviceArena::alloc(size_t bytes) {
  void* p = nullptr;
  if (bytes == 0) bytes = 16;
  if (cudaMalloc(&p, bytes) != cudaSuccess) {
    set_error("cudaMalloc of " + std::to_string(bytes) + " bytes failed");
    return nullptr;
  }
  ptrs_.push_back(p);
  total_ += bytes;
  return p;
}

namespace {
thread_local std::vector<std::function<int(cudaStream_t)>>* g_pack_recorder = nullptr;
}
void set_pack_recorder(std::vector<std::function<int(cudaStream_t)>>* recorder) { g_pack_recorder = recorder; }

namespace {

struct TapDef {
  int map, dy, dx;
  const WeightSrc* w;
  int ky, kx;
  int C;  // true input channels of this tap
};

int out_channels_of(const WeightSrc& w) { return w.transpose ? w.d1 : w.d0; }
int in_channels_of(const WeightSrc& w) { return w.transpose ? w.d0 : w.d1; }

// Pack weights for a tap list and fill everything of the plan except the A tensor maps and what igemm_select decides.
// *res_map / *mask_map: the residual / ReLU-mask maps were encoded for the TMA epilogue.
int finish_plan(IgemmPlan* plan, DeviceArena* arena, const std::vector<TapDef>& taps, int B, int H, int W, int tb,
                int th, int tw, int N, const Epilogue& ep, const OutSpec& out, int sy, int sx, int py, int px,
                cudaStream_t st, bool* res_map, bool* mask_map) {
  WC_REQUIRE(N % 16 == 0, "igemm needs N % 16 == 0 (pad the output channels)");
  WC_REQUIRE(static_cast<int>(taps.size()) <= kMaxTaps && !taps.empty(), "tap count out of range");
  IgemmArgs& a = plan->args;
  a = IgemmArgs{};
  *res_map = *mask_map = false;
  a.B = B; a.H = H; a.W = W; a.tb = tb; a.th = th; a.tw = tw;
  a.N = N;
  int total_kb = 0;
  a.ntaps = static_cast<int>(taps.size());
  for (size_t i = 0; i < taps.size(); ++i) {
    const int nkb = (taps[i].C + kIgemmBK - 1) / kIgemmBK;
    a.taps[i].map = static_cast<int8_t>(taps[i].map);
    a.taps[i].dy = static_cast<int8_t>(taps[i].dy);
    a.taps[i].dx = static_cast<int8_t>(taps[i].dx);
    a.taps[i].nkb = nkb;
    total_kb += nkb;
  }
  a.total_kb = total_kb;
  const int ktotal = total_kb * kIgemmBK;
  const long m_tiles = static_cast<long>((W + tw - 1) / tw) * ((H + th - 1) / th) * ((B + tb - 1) / tb);
  a.BN = igemm_pick_bn(N, m_tiles);
  if (out.bn_max > 0 && a.BN > out.bn_max) a.BN = out.bn_max;
  if (out.phases == 4) a.BN = (a.BN + 31) / 32 * 32;   // phase blocks are stored in 32-channel chunks
  if (out.mode == kOutQKV) {
    WC_REQUIRE(out.hd % 16 == 0, "head_dim must be a multiple of 16");
  }
  // ---- weights
  auto* wp = static_cast<__nv_bfloat16*>(arena->alloc(static_cast<size_t>(N) * ktotal * sizeof(__nv_bfloat16)));
  if (!wp) return 1;
  int koff = 0;
  double macs_per_pixel = 0;
  auto rec_src = std::make_shared<std::vector<const float*>>();
  auto rec_scale = std::make_shared<std::vector<const float*>>();
  auto rec_par = std::make_shared<std::vector<int>>();
  for (const TapDef& t : taps) {
    const WeightSrc& w = *t.w;
    const int n_src = out_channels_of(w);
    WC_REQUIRE(n_src <= N, "weight has more output channels than N");
    const int cpad = (t.C + kIgemmBK - 1) / kIgemmBK * kIgemmBK;
    const int ky = w.flip ? w.KH - 1 - t.ky : t.ky, kx = w.flip ? w.KW - 1 - t.kx : t.kx;
    if (int e = pack_tap(wp, ktotal, koff, w.w, n_src, t.C, cpad, w.KH, w.KW, ky, kx, w.transpose, w.scale, st)) return e;
    rec_src->push_back(w.w);
    rec_scale->push_back(w.scale);
    for (int v : {koff, n_src, t.C, cpad, w.KH, w.KW, ky, kx, w.transpose}) rec_par->push_back(v);
    koff += cpad;
    macs_per_pixel += static_cast<double>(t.C) * n_src;
  }
  if (g_pack_recorder) {  // training: one launch re-packs every tap of this plan from the fp32 master weights
    const int nt = static_cast<int>(taps.size());
    g_pack_recorder->push_back([=](cudaStream_t s) {
      return pack_taps(wp, ktotal, nt, rec_src->data(), rec_scale->data(), rec_par->data(), s);
    });
  }
  if (int e = igemm_make_bmap(&plan->maps.b, wp, N, ktotal, a.BN)) return e;
  // zero rows [n_src, N) if any (arena memory is uninitialised)
  {
    const int n_src = out_channels_of(*taps[0].w);
    if (n_src < N)
      WC_CHECK_CUDA(cudaMemsetAsync(wp + static_cast<size_t>(n_src) * ktotal, 0,
                                    static_cast<size_t>(N - n_src) * ktotal * sizeof(__nv_bfloat16), st));
  }
  // ---- epilogue
  a.bias = ep.bias;
  a.rowbias = ep.rowbias; a.ldrb = ep.ldrb;
  if (ep.res) {
    WC_REQUIRE(ep.res->B == B && ep.res->H == H * sy && ep.res->W == W * sx, "residual grid mismatch");
    a.res = ep.res->ptr; a.ldr = ep.res->ld;
  }
  if (ep.mask) {
    WC_REQUIRE(ep.mask->B == B && ep.mask->H == H * sy && ep.mask->W == W * sx, "mask grid mismatch");
    a.mask = ep.mask->ptr; a.ldm = ep.mask->ld;
  }
  a.relu = ep.relu;
  a.act = ep.act;
  a.prelu = ep.prelu;
  a.out_mode = out.mode;
  a.sy = sy; a.sx = sx; a.py = py; a.px = px;
  a.Ho = H * sy; a.Wo = W * sx;
  if (out.mode == kOutNHWC && out.phases == 4) {
    // four phase blocks of N/4 channels, one strided output map per phase; lean epilogue only (igemm.cu)
    const int pn = N / 4;
    WC_REQUIRE(sy == 2 && sx == 2 && N % 128 == 0 && a.BN % 32 == 0, "phase-block output needs up == 2 and N % 128 == 0");
    WC_REQUIRE(out.out.ptr && out.out.B == B && out.out.H == a.Ho && out.out.W == a.Wo && out.out.ld % 8 == 0 && !ep.res && !ep.mask, "phase-block output grid mismatch");
    a.out = out.out.ptr; a.ldc = out.out.ld;
    a.qw = tw < 32 ? tw : 32;
    a.qh = th < 32 / a.qw ? th : 32 / a.qw;
    a.qb = 32 / (a.qw * a.qh);
    WC_REQUIRE(a.qb <= tb, "phase-block output: tile too small");
    for (int q = 0; q < 4; ++q) {
      CUtensorMap* m = q == 0 ? &plan->maps.c : &plan->maps.qkv[q - 1];
      if (int e = igemm_make_cmap(m, out.out, pn, 32, a.qw, a.qh, a.qb, 2, 2, q / 2, q % 2)) return e;
    }
    plan->maps.r = plan->maps.c;
    a.tma_store = 1;
    a.phase_n = pn;
  } else if (out.mode == kOutNHWC) {
    WC_REQUIRE(out.out.ptr && out.out.B == B && out.out.H == a.Ho && out.out.W == a.Wo, "output grid mismatch");
    WC_REQUIRE(out.out.ld % 8 == 0, "output pixel stride must be a multiple of 8");
    a.out = out.out.ptr; a.ldc = out.out.ld;
    // TMA-store epilogue where the box fits the tile; otherwise row-per-lane global stores (epilogue_tile)
    const bool unit = (sy == 1 && sx == 1);
    if (unit || (out.out.H == H * sy && out.out.W == W * sx && (out.out.ld * sx * 2) % 16 == 0)) {
      const int nc = (a.BN % 32 == 0 && N % 32 == 0) ? 32 : 16;   // the epilogue's chunk width (see igemm_kernel)
      a.qw = tw < 32 ? tw : 32;
      a.qh = th < 32 / a.qw ? th : 32 / a.qw;
      a.qb = 32 / (a.qw * a.qh);
      if (a.qb <= tb) {
        if (int e = igemm_make_cmap(&plan->maps.c, out.out, N, nc, a.qw, a.qh, a.qb, sy, sx, py, px)) return e;
        a.tma_store = 1;
        if (ep.res && ep.res->ld % 8 == 0) {
          if (int e = igemm_make_cmap(&plan->maps.r, *ep.res, N, nc, a.qw, a.qh, a.qb, sy, sx, py, px)) return e;
          *res_map = true;
        }
        if (ep.mask && ep.mask->ld % 8 == 0) {
          if (int e = igemm_make_cmap(&plan->maps.m, *ep.mask, N, nc, a.qw, a.qh, a.qb, sy, sx, py, px)) return e;
          *mask_map = true;
        }
      }
    }
  } else if (out.mode == kOutNCHWf32) {
    a.out_f32 = out.out_f32; a.n_store = out.n_store;
    // lean epilogue with bulk-tensor stores of [16 planes][32 pixels] fp32 boxes (igemm.cu) when a TMEM lane quadrant is 32 consecutive
    // pixels of one image row; the map addresses the fp32 planes as bf16 pairs.  Otherwise per-lane stores (epilogue_tile).
    if (sy == 1 && sx == 1 && tw >= 32 && W % 32 == 0 && (W * 2) % 8 == 0 && !ep.res && !ep.mask) {
      uint64_t dims[4] = {static_cast<uint64_t>(2 * W), static_cast<uint64_t>(H), static_cast<uint64_t>(out.n_store), static_cast<uint64_t>(B)};
      uint64_t strides[4] = {1, static_cast<uint64_t>(2 * W), static_cast<uint64_t>(2 * W) * H, static_cast<uint64_t>(2 * W) * H * out.n_store};
      uint32_t box[4] = {64, 1, 16, 1};
      if (int e = encode_tmap_bf16(&plan->maps.c, out.out_f32, 4, dims, strides, box, 0)) return e;
      plan->maps.r = plan->maps.c;
      a.tma_store = 1;
      a.qw = 32; a.qh = 1; a.qb = 1;
    }
  } else {
    a.q = out.q; a.k = out.k; a.vt = out.vt; a.v = out.v; a.heads = out.heads; a.hd = out.hd; a.C = out.heads * out.hd; a.q_scale = out.q_scale;
    WC_REQUIRE(N == 3 * a.C, "QKV epilogue needs N == 3*C");
    WC_REQUIRE((H * W) % 8 == 0, "token count must be a multiple of 8");
    // Lean epilogue with bulk-tensor stores (igemm.cu: the kOutQKV branch of epilogue_tile_lean) when a TMEM lane quadrant is 32
    // consecutive tokens of one image and a 32-channel chunk stays inside q / k / v and inside whole heads.  Otherwise (V stored as
    // well for the training plan, tokens not contiguous) the per-lane scatter stores of epilogue_tile.
    const int qw = tw < 32 ? tw : 32, qh = th < 32 / qw ? th : 32 / qw, qb = 32 / (qw * qh);
    const bool tokens_contiguous = qb == 1 && ((qh == 1 && W % qw == 0) || qw == W);
    if (!out.v && tokens_contiguous && a.C % 32 == 0 && a.BN % 32 == 0 && (out.hd == 16 || out.hd % 32 == 0)) {
      const int hd = out.hd, heads = out.heads, ntok = H * W;
      const uint32_t inner = hd == 16 ? 16u : 32u;
      uint64_t dqk[4] = {static_cast<uint64_t>(hd), static_cast<uint64_t>(ntok), static_cast<uint64_t>(heads), static_cast<uint64_t>(B)};
      uint64_t sqk[4] = {1, static_cast<uint64_t>(hd), static_cast<uint64_t>(ntok) * hd, static_cast<uint64_t>(heads) * ntok * hd};
      uint32_t bqk[4] = {inner, 32, 1, 1};
      if (int e = encode_tmap_bf16(&plan->maps.qkv[0], out.q, 4, dqk, sqk, bqk, inner * 2)) return e;
      if (int e = encode_tmap_bf16(&plan->maps.qkv[1], out.k, 4, dqk, sqk, bqk, inner * 2)) return e;
      uint64_t dv[4] = {static_cast<uint64_t>(ntok), static_cast<uint64_t>(hd), static_cast<uint64_t>(heads), static_cast<uint64_t>(B)};
      uint64_t sv[4] = {1, static_cast<uint64_t>(ntok), static_cast<uint64_t>(ntok) * hd, static_cast<uint64_t>(heads) * ntok * hd};
      uint32_t bv[4] = {32, inner, 1, 1};
      if (int e = encode_tmap_bf16(&plan->maps.qkv[2], out.vt, 4, dv, sv, bv, 0)) return e;
      plan->maps.c = plan->maps.qkv[0];
      plan->maps.r = plan->maps.qkv[0];
      a.tma_store = 1;
      a.qw = qw; a.qh = qh; a.qb = qb;
    }
  }
  const long tiles = m_tiles * ((N + a.BN - 1) / a.BN);
  plan->grid = static_cast<int>(std::min<long>(tiles, num_sms()));
  plan->flops = 2.0 * macs_per_pixel * static_cast<double>(B) * H * W;
  return 0;
}

}  // namespace

int build_conv(ConvOp* op, DeviceArena* arena, const Act& x, const WeightSrc& w, const ConvGeom& g, int N,
               const Act* x2, const WeightSrc* w2, const Epilogue& ep, const OutSpec& out, cudaStream_t st) {
  WC_REQUIRE(x.C == in_channels_of(w), "input channels do not match the weight");
  WC_REQUIRE(x.ld % 8 == 0, "input pixel stride must be a multiple of 8 elements");
  op->plans.clear();
  op->plans.emplace_back();
  IgemmPlan& plan = op->plans.back();
  std::vector<TapDef> taps;
  int window = 0;
  int B = x.B, H, W, tb, th, tw;
  if (g.stride == 1) {
    WC_REQUIRE(2 * g.pad == g.dil * (g.K - 1), "stride-1 convolutions must be 'same' sized");
    H = x.H; W = x.W;
    igemm_pick_tile(B, H, W, &tb, &th, &tw);
    if (int e = igemm_make_amap(&plan.maps.a[0], x, tb, th, tw)) return e;
    for (int ky = 0; ky < g.K; ++ky)
      for (int kx = 0; kx < g.K; ++kx)
        taps.push_back({0, ky * g.dil - g.pad, kx * g.dil - g.pad, &w, ky, kx, x.C});
    int nmaps = 1;
    if (x2) {
      WC_REQUIRE(w2 && x2->B == B && x2->H == H && x2->W == W && x2->C == in_channels_of(*w2), "fused 1x1 input mismatch");
      if (int e = igemm_make_amap(&plan.maps.a[1], *x2, tb, th, tw)) return e;
      taps.push_back({1, 0, 0, w2, 0, 0, x2->C});
      nmaps = 2;
    }
    for (int i = nmaps; i < kMaxMaps; ++i) plan.maps.a[i] = plan.maps.a[0];
    // Row-segment mode: 3x3 / dilation 1 on maps at least 128 pixels wide with narrow N (the L2->SM bound layers)
    if (g.K == 3 && g.dil == 1 && tw == 128 && th == 1 && tb == 1 && (N <= 128 || (out.bn_max > 0 && out.bn_max <= 128))) {
      if (int e = igemm_make_rowseg_map(&plan.maps.a[2], x)) return e;
      window = 3;
    }
  } else {
    WC_REQUIRE(g.stride == 2 && g.dil == 1 && !x2, "only stride 1 or 2 (undilated, unfused) supported");
    WC_REQUIRE(x.H % 2 == 0 && x.W % 2 == 0, "stride-2 convolution needs even input dims");
    H = x.H / 2; W = x.W / 2;
    igemm_pick_tile(B, H, W, &tb, &th, &tw);
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px)
        if (int e = igemm_make_amap(&plan.maps.a[py * 2 + px], x, tb, th, tw, py, 2, px, 2, H, W)) return e;
    plan.maps.a[4] = plan.maps.a[0];
    for (int ky = 0; ky < g.K; ++ky)
      for (int kx = 0; kx < g.K; ++kx) {
        const int oy = ky - g.pad, ox = kx - g.pad;
        const int py = ((oy % 2) + 2) % 2, px = ((ox % 2) + 2) % 2;
        taps.push_back({py * 2 + px, (oy - py) / 2, (ox - px) / 2, &w, ky, kx, x.C});
      }
  }
  bool res_map, mask_map;
  if (int e = finish_plan(&plan, arena, taps, B, H, W, tb, th, tw, N, ep, out, out.up, out.up, out.py, out.px, st, &res_map, &mask_map))
    return e;
  // (resident weights do not pay here: measured on B200 (batch 32, 64 x 128) 3x3 64->64 in row-segment mode 34.7 -> 40.9 us, 1x1
  // 256->64 37.2 -> 35.9 us, 1x1 64->256 unchanged, although they cut the L2->SM traffic of the 3x3 layer 2.4x)
  igemm_select(&plan, window, 0, res_map, mask_map, true);
  op->flops = plan.flops;
  return 0;
}

// 7x7 / stride 2 / pad 3 convolution of a 3-channel image (ResNet stem, resnet.py:142) on the tensor core.  The image is first
// re-laid as NHWC bf16 with 8 channels (3 real) and 4 zero columns on either side: then the 7 taps of one kernel ROW are 56
// CONTIGUOUS elements, and a tensor map whose x stride (16 elements = one stride-2 step) is smaller than its 64-element inner
// box yields, for 128 output pixels, the im2col rows of that kernel row directly in the canonical K-major layout - an implicit
// im2col with overlapping boxes, no gather kernel.  K = 7 kernel rows x 64 (147 real), weights re-laid to match (wprime
// [N][64][7]: element kx*8 + c of kernel row ky).  Input rows alternate between two phase views (stride 2 in y).
int build_conv_stem7s2(ConvOp* op, DeviceArena* arena, const __nv_bfloat16* xp, int B, int H, int W, const float* wprime,
                       const float* scale, int N, const Epilogue& ep, const OutSpec& out, cudaStream_t st) {
  WC_REQUIRE(H % 2 == 0 && W % 2 == 0, "stem: even image dims");
  op->plans.clear();
  op->plans.emplace_back();
  IgemmPlan& plan = op->plans.back();
  const int Ho = H / 2, Wo = W / 2, Wp = W + 8;
  int tb, th, tw;
  igemm_pick_tile(B, Ho, Wo, &tb, &th, &tw);
  for (int ph = 0; ph < 2; ++ph) {
    uint64_t dims[4] = {64, static_cast<uint64_t>(Wo), static_cast<uint64_t>(Ho), static_cast<uint64_t>(B)};
    uint64_t strides[4] = {1, 16, static_cast<uint64_t>(2) * Wp * 8, static_cast<uint64_t>(H) * Wp * 8};
    uint32_t box[4] = {64, static_cast<uint32_t>(tw), static_cast<uint32_t>(th), static_cast<uint32_t>(tb)};
    if (int e = encode_tmap_bf16(&plan.maps.a[ph], xp + (static_cast<size_t>(ph) * Wp + 1) * 8, 4, dims, strides, box, 128)) return e;
  }
  for (int i = 2; i < kMaxMaps; ++i) plan.maps.a[i] = plan.maps.a[0];
  WeightSrc w; w.w = wprime; w.d0 = N; w.d1 = 64; w.KH = 7; w.KW = 1; w.scale = scale;
  std::vector<TapDef> taps;
  for (int ky = 0; ky < 7; ++ky) {
    const int o = ky - 3, dy = (o >= 0) ? o / 2 : -((-o + 1) / 2), ph = o - 2 * dy;   // o = 2 dy + ph, ph in {0, 1}
    taps.push_back({ph, dy, 0, &w, ky, 0, 64});
  }
  bool res_map, mask_map;
  if (int e = finish_plan(&plan, arena, taps, B, Ho, Wo, tb, th, tw, N, ep, out, 1, 1, 0, 0, st, &res_map, &mask_map)) return e;
  igemm_select(&plan, 0, 0, res_map, mask_map, false);
  plan.flops = 2.0 * 147.0 * N * static_cast<double>(B) * Ho * Wo;   // algorithmic (the reference's 7x7x3 taps), not the padded K
  op->flops = plan.flops;
  return 0;
}

// 1 x KW horizontal convolution ('same' size, stride 1): one tap per kernel column.  Used by the SRGAN final layer (srgan.cu), whose
// 9x9 depthwise + 64 -> 3 pointwise pair is run as N = (kernel row, output) columns of a horizontal convolution on the tensor
// core, followed by a vertical shift-add of the 27 fp32 planes (seg_kernels.cu: srgan_final_combine).
int build_conv_hrow(ConvOp* op, DeviceArena* arena, const Act& x, const WeightSrc& w, int N, const Epilogue& ep, const OutSpec& out,
                    cudaStream_t st) {
  WC_REQUIRE(w.KH == 1 && (w.KW & 1) == 1 && w.KW <= kMaxTaps, "build_conv_hrow: 1 x odd kernel with at most kMaxTaps columns");
  WC_REQUIRE(x.C == in_channels_of(w), "input channels do not match the weight");
  WC_REQUIRE(x.ld % 8 == 0, "input pixel stride must be a multiple of 8 elements");
  op->plans.clear();
  op->plans.emplace_back();
  IgemmPlan& plan = op->plans.back();
  int tb, th, tw;
  igemm_pick_tile(x.B, x.H, x.W, &tb, &th, &tw);
  if (int e = igemm_make_amap(&plan.maps.a[0], x, tb, th, tw)) return e;
  for (int i = 1; i < kMaxMaps; ++i) plan.maps.a[i] = plan.maps.a[0];
  std::vector<TapDef> taps;
  for (int kx = 0; kx < w.KW; ++kx) taps.push_back({0, 0, kx - w.KW / 2, &w, 0, kx, x.C});
  bool res_map, mask_map;
  if (int e = finish_plan(&plan, arena, taps, x.B, x.H, x.W, tb, th, tw, N, ep, out, 1, 1, 0, 0, st, &res_map, &mask_map)) return e;
  // Row-segment mode with all KW taps in one stage: one box of 128 + KW - 1 pixels per tile instead of KW boxes of 128, one barrier
  // hand-over per tile instead of KW
  // (the kernel is instantiated for 3 x 3 and 1 x 9 windows: other widths keep one stage per tap)
  int window = 0;
  if (w.KW == 9 && tw == 128 && th == 1 && tb == 1) {
    if (int e = igemm_make_rowseg_map(&plan.maps.a[2], x, w.KW)) return e;
    window = 9;
  }
  // the packed weights of all taps (KW x BN x 64 bf16) are the same for every tile: keep them resident in row-segment mode (one load
  // per CTA) when this is a single N tile - the ring then carries activations only
  const long wb = static_cast<long>(plan.args.BN) * plan.args.total_kb * kIgemmBK * 2;
  igemm_select(&plan, window, plan.args.BN >= N && wb <= kIgemmWresMaxBytes ? static_cast<int>(wb) : 0, res_map, mask_map, false);
  op->flops = plan.flops;
  return 0;
}

int build_conv_transposed_s2(ConvOp* op, DeviceArena* arena, const Act& x, const WeightSrc& w, int K, int pad, int N,
                             const Epilogue& ep, const OutSpec& out, cudaStream_t st) {
  WC_REQUIRE(w.transpose == 1, "transposed conv expects a [Cin][Cout][K][K] weight view");
  WC_REQUIRE(x.C == in_channels_of(w), "input channels do not match the weight");
  op->plans.clear();
  op->flops = 0;
  int tb, th, tw;
  igemm_pick_tile(x.B, x.H, x.W, &tb, &th, &tw);
  for (int qy = 0; qy < 2; ++qy)
    for (int qx = 0; qx < 2; ++qx) {
      std::vector<TapDef> taps;
      for (int ky = (qy + pad) % 2; ky < K; ky += 2)
        for (int kx = (qx + pad) % 2; kx < K; kx += 2)
          taps.push_back({0, (qy + pad - ky) / 2, (qx + pad - kx) / 2, &w, ky, kx, x.C});
      if (taps.empty()) continue;  // e.g. 1x1 stride-2 dgrad: only phase (0,0) receives gradient
      op->plans.emplace_back();
      IgemmPlan& plan = op->plans.back();
      if (int e = igemm_make_amap(&plan.maps.a[0], x, tb, th, tw)) return e;
      for (int i = 1; i < kMaxMaps; ++i) plan.maps.a[i] = plan.maps.a[0];
      bool res_map, mask_map;
      if (int e = finish_plan(&plan, arena, taps, x.B, x.H, x.W, tb, th, tw, N, ep, out, 2, 2, qy, qx, st, &res_map, &mask_map)) return e;
      igemm_select(&plan, 0, 0, res_map, mask_map, false);
      op->flops += plan.flops;
    }
  return 0;
}

int build_conv_dgrad(ConvOp* op, DeviceArena* arena, const Act& dy, const WeightSrc& w, const ConvGeom& g, const Epilogue& ep,
                     const OutSpec& out, cudaStream_t st) {
  WeightSrc wt = w;
  wt.transpose = 1;
  if (g.stride != 1) return build_conv_transposed_s2(op, arena, dy, wt, g.K, g.pad, w.d1, ep, out, st);
  wt.flip = 1;
  return build_conv(op, arena, dy, wt, g, w.d1, nullptr, nullptr, ep, out, st);
}

}  // namespace wc
