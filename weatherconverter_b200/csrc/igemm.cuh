// Implicit-GEMM convolution / linear layer on tcgen05 tensor cores (sm_100a).
//
//   out[pixel, n] = epilogue( sum_{tap} sum_{c} A_tap[pixel + (dy,dx), c] * Wp[n, koff(tap) + c] )
//
// * A operands are NHWC bf16 tensors described by up to kMaxMaps rank-4 TMA tensor maps (C, W, H, B).  One
//   pipeline stage = one (tap, 64-channel block): a TMA box of 128 pixels x 64 channels (128-byte swizzle),
//   zero-filled outside the image, lands in shared memory already in the canonical K-major UMMA layout.
//   Stride-2 convolutions use one map per input phase (strided views); the fused 1x1 residual convolution of
//   a ResNet sub-layer is simply one more tap reading a different tensor.
// * B (weights) are pre-packed bf16 [Npad][Ktotal] K-major, loaded with a 2-D tensor map (box 64 x BN).
// * tcgen05.mma 128 x BN x 16 (cta_group::1), fp32 accumulators double-buffered in TMEM (2 x 256 columns).
// * Persistent CTAs, 10 warps: warp 0 TMA producer, warp 1 MMA issuer (+TMEM alloc), warps 2-9 epilogue
//   (TMEM -> registers -> bias / t-emb / residual / ReLU -> bf16 stores), so the epilogue of tile i overlaps
//   the main loop of tile i+1.
#pragma once
#include "wc_host.h"

namespace wc {

constexpr int kIgemmBM = 128;
constexpr int kIgemmBK = 64;
constexpr int kMaxTaps = 20;
constexpr int kMaxMaps = 5;

struct IgemmTap {
  int8_t map;  // index into IgemmMaps::a
  int8_t dy, dx;
  int8_t pad_;
  int32_t nkb;  // number of 64-channel K blocks for this tap
};

enum IgemmOutMode : int { kOutNHWC = 0, kOutQKV = 1, kOutNCHWf32 = 2 };

struct IgemmArgs {
  int B, H, W;     // logical pixel grid the M tiles walk (== spatial dims of every A map)
  int tb, th, tw;  // tile shape, tb*th*tw == 128
  int N, BN;       // true output channels (multiple of 16) and N tile
  int ntaps, total_kb;
  int nstages;  // depth of the TMA ring (set by igemm_select)
  int row3;  // 1: taps 0..8 form a 3x3 stride-1 window executed in row-segment mode (see igemm.cu)
  IgemmTap taps[kMaxTaps];
  // epilogue
  const float* bias;     // [N] or nullptr
  const float* rowbias;  // [B][ldrb] per-sample additive term (t-embedding projection) or nullptr
  int ldrb;
  const __nv_bfloat16* res;  // residual, NHWC on the OUTPUT grid (B,Ho,Wo), or nullptr
  int ldr;
  const __nv_bfloat16* mask;  // ReLU-derivative mask on the output grid: result zeroed where mask <= 0, or nullptr
  int ldm;
  int relu;
  int act;  // 0 none, 2 SiLU, 3 GELU (exact, erf): applied after bias / residual (legacy UNet, old_modules.py:84,148)
  const float* prelu;  // per-channel PReLU slopes [N] applied after bias/residual, or nullptr
  int out_mode;
  __nv_bfloat16* out;  // kOutNHWC: element (b, y*sy+py, x*sx+px, n) of a [B,Ho,Wo,ldc] buffer
  int ldc, Ho, Wo, sy, sx, py, px;
  float* out_f32;  // kOutNCHWf32: [B, N_store, Ho, Wo] fp32 planes
  int n_store;
  __nv_bfloat16 *q, *k, *vt;  // kOutQKV: Q,K [B,heads,ntok,hd]; V^T [B,heads,hd,ntok]
  __nv_bfloat16* v;           // kOutQKV, optional: V [B,heads,ntok,hd] as well (the attention backward reads it)
  int heads, hd, C;
  int row_nkx;                 // row-segment mode: width of the window (3: 3 x 3, 9: 1 x 9 for build_conv_hrow)
  int phase_n;                 // > 0: kOutNHWC through the lean epilogue with four phase blocks of phase_n channels (maps c, qkv[0..2])
  int res_deep;                // LEAN == 3: load slots per epilogue warp of the residual / mask stream (igemm.cu)
  int stream_res, stream_mask; // LEAN == 3: which boxes a slot carries (residual rows, ReLU-mask rows)
  float q_scale;               // kOutQKV: the Q columns are multiplied by this before the bf16 rounding (1: off); see OutSpec::q_scale
  // kOutNHWC through TMA (tma_store == 1; unit-stride outputs only): every epilogue warp stages its 32 rows x NC channels in
  // shared memory and one lane stores the box (NC, qw, qh, qb) = its TMEM lane quadrant of the tile with IgemmMaps::c
  int tma_store, qw, qh, qb;
  // residual through TMA as well (tma_res == 1): needs tma_store and 16 KiB of the ring area free behind the last stage; every
  // epilogue warp loads the (NC, qw, qh, qb) box of its next chunk with IgemmMaps::r and reads its own row from shared memory
  int tma_res;
  // lean epilogue (igemm.cu: epilogue_tile_lean): TMA store, no ReLU-mask input, residual (if any) through TMA; stage2 = the ring
  // leaves 16 KiB free, i.e. every epilogue warp owns TWO 2 KiB staging buffers and alternates between them
  int lean, stage2;
  // resident weights (wres == 1): the whole packed weight matrix (N == BN, N * Ktotal * 2 bytes <= kIgemmWresMaxBytes) is loaded
  // into shared memory ONCE per persistent CTA and the ring stages carry activations only
  int wres;
};
constexpr int kIgemmWresMaxBytes = 98304;

struct IgemmMaps {
  CUtensorMap a[kMaxMaps];
  CUtensorMap b;
  CUtensorMap c;   // output (tma_store)
  CUtensorMap r;   // residual (tma_res)
  CUtensorMap m;   // ReLU-mask rows through the stream epilogue (same box as c / r)
  CUtensorMap qkv[3];   // kOutQKV through the lean epilogue: Q, K as (hd, N, heads, B), V^T as (N, hd, heads, B)
};

struct IgemmPlan;
using IgemmLaunchFn = int (*)(const IgemmPlan&, cudaStream_t);

struct IgemmPlan {
  IgemmMaps maps;
  IgemmArgs args;
  int grid = 0;
  double flops = 0;  // algorithmic FLOPs (2*MAC) of the convolution this plan implements
  IgemmLaunchFn launch = nullptr;  // the igemm_kernel instantiation igemm_select chose
};

// Completes a plan whose taps, tile, BN, epilogue inputs and output maps are set: row-segment mode, ring depth, residual staging,
// epilogue (generic, lean or residual stream) and the kernel instantiation igemm_launch runs.
//   window:     the row-segment window the builder encoded IgemmMaps::a[2] for: 0 none, 3 (3 x 3) or 9 (1 x 9); taken when
//               BN <= 128 and two ring stages fit
//   wres_bytes: > 0: keep that many bytes of packed weights resident in shared memory if the window is taken
//   res_map / mask_map: IgemmMaps::r / ::m were encoded (residual / ReLU-mask rows can be loaded through TMA)
//   stream:     the residual stream epilogue may be chosen
void igemm_select(IgemmPlan* plan, int window, int wres_bytes, bool res_map, bool mask_map, bool stream);
int igemm_launch(const IgemmPlan& plan, cudaStream_t stream);

// Choose the M-tile shape for a (B,H,W) grid: widest power-of-two span of x, then y, then b.
void igemm_pick_tile(int B, int H, int W, int* tb, int* th, int* tw);
int igemm_pick_bn(int N, long m_tiles);

// Rank-4 (C, W, H, B) bf16 tensor map over an NHWC view, with optional spatial sub-sampling (phase views for
// stride-2 convolutions): element (b, y, x, c) of the view = act(b, y*ys + y0, x*xs + x0, c), view dims Hv x Wv.
int igemm_make_amap(CUtensorMap* out, const Act& act, int tb, int th, int tw, int y0 = 0, int ys = 1, int x0 = 0,
                    int xs = 1, int Hv = -1, int Wv = -1);
// Row-segment A map (box 64 ch x (128 + nkx - 1) pixels of one image row) for the row-segment mode (nkx = 3 or 9).
int igemm_make_rowseg_map(CUtensorMap* out, const Act& act, int nkx = 3);
int igemm_make_bmap(CUtensorMap* out, const __nv_bfloat16* wpacked, int n_rows, int ktotal, int BN);
// Output map for the TMA-store epilogue: channels [0, N) of an NHWC view, box (nc, qw, qh, qb), swizzle = nc*2 bytes.
int igemm_make_cmap(CUtensorMap* out, const Act& act, int N, int nc, int qw, int qh, int qb, int sy = 1, int sx = 1, int py = 0,
                    int px = 0);

}  // namespace wc
