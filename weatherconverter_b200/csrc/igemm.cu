// See igemm.cuh for the design.  Reference ops replaced: every nn.Conv2d / nn.ConvTranspose2d / nn.Linear on
// the hot path (unet_base.py:87-129,293-334,395-449; resnet.py:78-118; _deeplab.py:28-59,111-162).
#include "igemm.cuh"
#include "wc_ptx.cuh"

namespace wc {

namespace {

constexpr int kThreads = 320;  // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue (two groups of 4, one per TMEM lane quadrant)
constexpr uint32_t kABytes = kIgemmBM * kIgemmBK * 2;  // 16 KiB
constexpr uint32_t kPipeBytes = 212992;  // shared-memory budget of the TMA ring (both modes), multiple of 1024; its last 16 KiB double as
                                         // the residual staging of the TMA epilogue when the ring leaves them free (igemm_res_staging_fits)
constexpr int kMaxStages = 8;
// bias / PReLU vectors up to this many channels are staged in shared memory (wider layers: L1-cached broadcast loads); the two
// limits are what is left of the 227 KiB after the ring, the output staging, the barriers and the alignment slack
constexpr int kBiasMaxN = 256, kPreluMaxN = 128;
constexpr uint32_t kVecBytes = (kBiasMaxN + kPreluMaxN) * 4;
// Output staging of the TMA-store epilogue: 2 KiB per epilogue warp (32 rows x 32 channels bf16, 64-byte swizzle).  The
// row-per-lane global stores it replaces touch 32 different 128-byte lines per request (16 bytes each) and keep the L1TEX
// tag stage busy (profiles/r1_ncu_igemm_1x1_64_256.txt); a TMA store reads shared memory directly.
constexpr uint32_t kOutStageBytes = 8 * 2048;
constexpr uint32_t kBarBytes = 512;   // 64 mbarriers: ring (2 x 8), accumulators (4), TMEM slot, residual boxes (8), resident weights,
                                      // and 8 x 4 for the residual stream epilogue (index 32 + 4 * epilogue warp + slot)
constexpr uint32_t kSmemBytes = kPipeBytes + kOutStageBytes + 1024 /*align*/ + kBarBytes + kVecBytes;   // = 227 KiB
constexpr uint32_t kTmemCols = 512;
// Row-segment mode (stride 1, dilation 1, tiles of 128 pixels of ONE image row; ROWK = 3: 3 x 3 window, ROWK = 9: 1 x 9 window): per
// (channel block, kernel row) one TMA box of 128 + nkx - 1 pixels [x0 - nkx/2, ..) is loaded once and the nkx horizontal taps read it
// through UMMA descriptors whose start is shifted by kx*128 bytes (the 128-byte swizzle is a function of the absolute shared-memory
// address, so the shifted start needs no fix-up) -> A traffic / nkx.
constexpr uint32_t kRowABytes = 18432;                       // (128 + 9 - 1) * 128 = 17408, padded to a multiple of 1024

template <int NC>
__device__ __forceinline__ void tmem_ld_n(uint32_t taddr, uint32_t (&r)[NC]) {
  if constexpr (NC == 32) tmem_ld32(taddr, r);
  else tmem_ld16(taddr, r);
}

// Epilogue of one accumulator tile for one thread (= one output pixel row of the tile).  `grp` in {0,1}: the two
// epilogue warpgroups interleave the N chunks.  Residual / ReLU-mask rows are prefetched one chunk ahead so their global
// latency overlaps the TMEM load and the math of the current chunk.
template <int NC, bool TMA_OUT, bool TMA_RES>
__device__ __forceinline__ void epilogue_tile(const IgemmArgs& p, uint32_t tacc, int n0, int b, int y, int x,
                                              bool valid, int grp, const float* s_bias, const float* s_prelu,
                                              uint32_t tfull_addr, uint32_t tfull_parity, const CUtensorMap* cmap,
                                              uint32_t out_stage, int qx, int qy, int qb0, const CUtensorMap* rmap,
                                              uint32_t res_stage, uint32_t res_bar, uint32_t& res_phase) {
  constexpr int NV = NC / 8;
  const int lane = threadIdx.x & 31;
  constexpr bool tma_out = TMA_OUT;
  constexpr bool tma_res = TMA_OUT && TMA_RES;   // the residual box arrives in shared memory through TMA
  const int oy = y * p.sy + p.py, ox = x * p.sx + p.px;
  const size_t opix = (static_cast<size_t>(b) * p.Ho + oy) * p.Wo + ox;
  const uint4* res_row = p.res ? reinterpret_cast<const uint4*>(p.res + opix * p.ldr) : nullptr;
  const uint4* mask_row = p.mask ? reinterpret_cast<const uint4*>(p.mask + opix * p.ldm) : nullptr;
  uint4 res_nxt[NV], mask_nxt[NV];
  auto prefetch = [&](int nb) {
    if (tma_res && nb < p.N && lane == 0) {   // one box (NC channels x this warp's 32 pixels); rows outside the tensor are zero-filled
      mbar_arrive_expect_tx(res_bar, NC * 2 * 32);
      tma_load_4d(res_stage, rmap, res_bar, nb, qx, qy, qb0);
    }
    if (!valid || nb >= p.N) return;
    if (res_row && !tma_res) {
#pragma unroll
      for (int j = 0; j < NV; ++j) res_nxt[j] = __ldg(res_row + (nb >> 3) + j);
    }
    if (mask_row) {
#pragma unroll
      for (int j = 0; j < NV; ++j) mask_nxt[j] = __ldg(mask_row + (nb >> 3) + j);
    }
  };
  if (grp * NC < p.BN) prefetch(n0 + grp * NC);   // issued BEFORE waiting for the accumulator: overlaps the main loop's tail
  mbar_wait(tfull_addr, tfull_parity);
  tc_fence_after();
  for (int c0 = grp * NC; c0 < p.BN; c0 += 2 * NC) {
    const int nb = n0 + c0;
    if (nb >= p.N) break;  // warp-uniform
    uint32_t r[NC];
    tmem_ld_n<NC>(tacc + c0, r);
    uint4 res_cur[NV], mask_cur[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) { res_cur[j] = res_nxt[j]; mask_cur[j] = mask_nxt[j]; }
    if (tma_res) {
      mbar_wait(res_bar, res_phase);
      res_phase ^= 1u;
      const uint32_t mine = res_stage + lane * (NC * 2);
      const uint32_t sw = NC == 32 ? ((lane >> 1) & 3) : ((lane >> 2) & 1);
#pragma unroll
      for (int j = 0; j < NV; ++j)
        asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(res_cur[j].x), "=r"(res_cur[j].y), "=r"(res_cur[j].z), "=r"(res_cur[j].w)
                     : "r"(mine + ((static_cast<uint32_t>(j) ^ sw) << 4)) : "memory");
      // Cross-proxy WAR: the lanes read the staging buffer through the generic proxy and the NEXT residual box is written
      // into the same bytes by the TMA (async proxy).  Without this fence the two are unordered, and on B200 the next box
      // did overtake the reads whenever the epilogue was the bottleneck (1x1 convolutions with several tiles per CTA: a
      // few per cent of the rows picked up the following chunk's residual - found by the batch-invariance tests of
      // round 2, tools/conv_res_sweep.py; a warp barrier alone does not order the proxies).
      fence_proxy_async_smem();
      __syncwarp();   // every lane has read its row before the next box may land
    }
    if (c0 + 2 * NC < p.BN) prefetch(nb + 2 * NC);
    tmem_wait_ld();
    if (!valid && !tma_out) continue;   // TMA store: all lanes stage their row, rows outside the tensor are clipped by the TMA
    float v[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) v[j] = __uint_as_float(r[j]);
    if (p.bias) {
#pragma unroll
      for (int j = 0; j < NC; j += 4) {
        const float4 bv = s_bias ? *reinterpret_cast<const float4*>(s_bias + nb + j)
                                 : __ldg(reinterpret_cast<const float4*>(p.bias + nb + j));
        v[j] += bv.x; v[j + 1] += bv.y; v[j + 2] += bv.z; v[j + 3] += bv.w;
      }
    }
    if (p.rowbias) {
      const float* rb = p.rowbias + static_cast<size_t>(b < p.B ? b : p.B - 1) * p.ldrb + nb;
#pragma unroll
      for (int j = 0; j < NC; j += 4) {
        float4 bv = __ldg(reinterpret_cast<const float4*>(rb + j));
        v[j] += bv.x; v[j + 1] += bv.y; v[j + 2] += bv.z; v[j + 3] += bv.w;
      }
    }
    if (p.res) {
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        const uint4 u = res_cur[j];
        float2 f0 = unpack_bf16(u.x), f1 = unpack_bf16(u.y), f2 = unpack_bf16(u.z), f3 = unpack_bf16(u.w);
        v[8 * j + 0] += f0.x; v[8 * j + 1] += f0.y; v[8 * j + 2] += f1.x; v[8 * j + 3] += f1.y;
        v[8 * j + 4] += f2.x; v[8 * j + 5] += f2.y; v[8 * j + 6] += f3.x; v[8 * j + 7] += f3.y;
      }
    }
    if (p.relu) {
#pragma unroll
      for (int j = 0; j < NC; ++j) v[j] = fmaxf(v[j], 0.f);
    }
    if (p.act == 2) {
#pragma unroll
      for (int j = 0; j < NC; ++j) v[j] = __fdividef(v[j], 1.f + __expf(-v[j]));
    } else if (p.act == 3) {
#pragma unroll
      for (int j = 0; j < NC; ++j) v[j] = 0.5f * v[j] * (1.f + erff(v[j] * 0.70710678118654752f));
    }
    if (p.prelu) {
#pragma unroll
      for (int j = 0; j < NC; j += 4) {
        const float4 sv = s_prelu ? *reinterpret_cast<const float4*>(s_prelu + nb + j)
                                  : __ldg(reinterpret_cast<const float4*>(p.prelu + nb + j));
        v[j] = v[j] > 0.f ? v[j] : v[j] * sv.x; v[j + 1] = v[j + 1] > 0.f ? v[j + 1] : v[j + 1] * sv.y;
        v[j + 2] = v[j + 2] > 0.f ? v[j + 2] : v[j + 2] * sv.z; v[j + 3] = v[j + 3] > 0.f ? v[j + 3] : v[j + 3] * sv.w;
      }
    }
    if (p.mask) {
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        const uint4 u = mask_cur[j];
        float2 f0 = unpack_bf16(u.x), f1 = unpack_bf16(u.y), f2 = unpack_bf16(u.z), f3 = unpack_bf16(u.w);
        if (!(f0.x > 0.f)) v[8 * j + 0] = 0.f;
        if (!(f0.y > 0.f)) v[8 * j + 1] = 0.f;
        if (!(f1.x > 0.f)) v[8 * j + 2] = 0.f;
        if (!(f1.y > 0.f)) v[8 * j + 3] = 0.f;
        if (!(f2.x > 0.f)) v[8 * j + 4] = 0.f;
        if (!(f2.y > 0.f)) v[8 * j + 5] = 0.f;
        if (!(f3.x > 0.f)) v[8 * j + 6] = 0.f;
        if (!(f3.y > 0.f)) v[8 * j + 7] = 0.f;
      }
    }
    if constexpr (tma_out) {
      // the previous chunk's store must have finished READING the staging buffer
      if (lane == 0) tma_store_wait_read0();
      __syncwarp();
      // row `lane` of the box, 16-byte chunk j at j ^ swizzle(row): 64-byte rows -> XOR with bits 1..2 of the row (SWIZZLE_64B),
      // 32-byte rows -> XOR with bit 2 (SWIZZLE_32B); conflict-free per quarter warp
      const uint32_t mine = out_stage + lane * (NC * 2);
      const uint32_t sw = NC == 32 ? ((lane >> 1) & 3) : ((lane >> 2) & 1);
#pragma unroll
      for (int j = 0; j < NV; ++j)
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(mine + ((static_cast<uint32_t>(j) ^ sw) << 4)),
                     "r"(pack_bf16(v[8 * j + 0], v[8 * j + 1])), "r"(pack_bf16(v[8 * j + 2], v[8 * j + 3])),
                     "r"(pack_bf16(v[8 * j + 4], v[8 * j + 5])), "r"(pack_bf16(v[8 * j + 6], v[8 * j + 7])) : "memory");
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_4d(cmap, out_stage, nb, qx, qy, qb0);
        tma_store_commit();
      }
    } else if (p.out_mode == kOutNHWC) {
      uint4* op = reinterpret_cast<uint4*>(p.out + opix * p.ldc + nb);
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        uint4 u;
        u.x = pack_bf16(v[8 * j + 0], v[8 * j + 1]);
        u.y = pack_bf16(v[8 * j + 2], v[8 * j + 3]);
        u.z = pack_bf16(v[8 * j + 4], v[8 * j + 5]);
        u.w = pack_bf16(v[8 * j + 6], v[8 * j + 7]);
        op[j] = u;
      }
    } else if (p.out_mode == kOutNCHWf32) {
      const size_t plane = static_cast<size_t>(p.Ho) * p.Wo;
      float* op = p.out_f32 + (static_cast<size_t>(b) * p.n_store) * plane + static_cast<size_t>(oy) * p.Wo + ox;
#pragma unroll
      for (int j = 0; j < NC; ++j)
        if (nb + j < p.n_store) op[static_cast<size_t>(nb + j) * plane] = v[j];
    } else {  // kOutQKV, NC == 16, hd % 16 == 0: a chunk never straddles a head or the q/k/v boundary
      const int which = nb / p.C, c = nb % p.C, head = c / p.hd, d = c % p.hd;
      if (which == 0 && p.q_scale != 1.f) {
#pragma unroll
        for (int j = 0; j < NC; ++j) v[j] *= p.q_scale;
      }
      const int ntok = p.H * p.W;
      const size_t tok = static_cast<size_t>(y) * p.W + x;
      const size_t bh = static_cast<size_t>(b) * p.heads + head;
      if (which < 2) {
        __nv_bfloat16* dst = (which == 0 ? p.q : p.k) + (bh * ntok + tok) * p.hd + d;
        uint4* op = reinterpret_cast<uint4*>(dst);
#pragma unroll
        for (int j = 0; j < NV; ++j) {
          uint4 u;
          u.x = pack_bf16(v[8 * j + 0], v[8 * j + 1]);
          u.y = pack_bf16(v[8 * j + 2], v[8 * j + 3]);
          u.z = pack_bf16(v[8 * j + 4], v[8 * j + 5]);
          u.w = pack_bf16(v[8 * j + 6], v[8 * j + 7]);
          op[j] = u;
        }
      } else {
        __nv_bfloat16* dst = p.vt + (bh * p.hd + d) * ntok + tok;
#pragma unroll
        for (int j = 0; j < NC; ++j) dst[static_cast<size_t>(j) * ntok] = __float2bfloat16_rn(v[j]);
        if (p.v) {
          uint4* op = reinterpret_cast<uint4*>(p.v + (bh * ntok + tok) * p.hd + d);
#pragma unroll
          for (int j = 0; j < NV; ++j) {
            uint4 u;
            u.x = pack_bf16(v[8 * j + 0], v[8 * j + 1]);
            u.y = pack_bf16(v[8 * j + 2], v[8 * j + 3]);
            u.z = pack_bf16(v[8 * j + 4], v[8 * j + 5]);
            u.w = pack_bf16(v[8 * j + 6], v[8 * j + 7]);
            op[j] = u;
          }
        }
      }
    }
  }
}


// Lean epilogue of one accumulator tile for the common case: bf16 NHWC output through TMA, optional residual through TMA, no
// ReLU-mask input.  Compared with epilogue_tile it has no per-lane global accesses, no look-ahead register arrays and every
// mode decision is a compile-time or tile-uniform choice; ncu on the 1x1 64->256 layer (profiles/r2_ncu_igemm_1x1_64_256_generic.txt)
// showed the generic version executing 320 warp instructions per 32-channel chunk, a quarter of them register moves.
// Staging: every epilogue warp owns two 2 KiB buffers (nbuf == 2 when the ring leaves 16 KiB free) and alternates between them
// chunk by chunk (ectr counts this warp's chunks across tiles): the TMA store of chunk i reads buffer i & 1 while chunk i + 1 is
// staged in the other one.  With a residual the box of chunk i is loaded by TMA INTO the buffer chunk i will be stored from; each
// lane reads its row, adds, and writes the bf16 result back in place.
template <int NC, bool RES>
__device__ __forceinline__ void epilogue_tile_lean(const IgemmArgs& p, uint32_t tacc, int n0, int b, int grp,
                                                   const float* s_bias,
                                                   const float* s_prelu, uint32_t tfull_addr, uint32_t tfull_parity,
                                                   const CUtensorMap* cmap, const CUtensorMap* rmap, uint32_t buf0, uint32_t buf1,
                                                   int nbuf, int qx, int qy, int qb0, uint32_t res_bar, uint32_t& res_phase,
                                                   uint32_t& ectr, const CUtensorMap* qkv_maps = nullptr) {
  constexpr int NV = NC / 8;
  const int lane = threadIdx.x & 31;
  const uint32_t sw = NC == 32 ? ((lane >> 1) & 3) : ((lane >> 2) & 1);
  const uint32_t row_off = static_cast<uint32_t>(lane) * (NC * 2);
  auto buf_of = [&](uint32_t i) { return ((i & 1u) && nbuf == 2) ? buf1 : buf0; };
  auto request = [&](uint32_t i, int nb) {   // residual box of chunk i (channels nb ..) -> its staging buffer
    if (lane == 0) {
      tma_store_wait_read<0>();              // the store that last used this buffer (chunk i - 2) has finished reading it
      mbar_arrive_expect_tx(res_bar, NC * 2 * 32);
      tma_load_4d(buf_of(i), rmap, res_bar, nb, qx, qy, qb0);
    }
  };
  const int c_first = grp * NC;
  if (RES && c_first < p.BN && n0 + c_first < p.N) request(ectr, n0 + c_first);   // before the accumulator is ready: overlaps the main loop
  mbar_wait(tfull_addr, tfull_parity);
  tc_fence_after();
  const float* rb = p.rowbias ? p.rowbias + static_cast<size_t>(b < p.B ? b : p.B - 1) * p.ldrb : nullptr;
  for (int c0 = c_first; c0 < p.BN; c0 += 2 * NC) {
    const int nb = n0 + c0;
    if (nb >= p.N) break;  // warp-uniform
    uint32_t r[NC];
    tmem_ld_n<NC>(tacc + c0, r);
    const uint32_t mine = buf_of(ectr) + row_off;
    uint4 rr[NV];
    if (RES) {
      mbar_wait(res_bar, res_phase);
      res_phase ^= 1u;
#pragma unroll
      for (int j = 0; j < NV; ++j)
        asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(rr[j].x), "=r"(rr[j].y), "=r"(rr[j].z), "=r"(rr[j].w)
                     : "r"(mine + ((static_cast<uint32_t>(j) ^ sw) << 4)) : "memory");
      // the next box goes into the OTHER buffer (last touched, through the generic proxy, one chunk ago and fenced then)
      if (c0 + 2 * NC < p.BN && nb + 2 * NC < p.N) request(ectr + 1, nb + 2 * NC);
    }
    tmem_wait_ld();
    float v[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) v[j] = __uint_as_float(r[j]);
    if (s_bias) {
#pragma unroll
      for (int j = 0; j < NC; j += 4) {
        const float4 bv = *reinterpret_cast<const float4*>(s_bias + nb + j);
        v[j] += bv.x; v[j + 1] += bv.y; v[j + 2] += bv.z; v[j + 3] += bv.w;
      }
    } else if (p.bias) {
#pragma unroll
      for (int j = 0; j < NC; j += 4) {
        const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + nb + j));
        v[j] += bv.x; v[j + 1] += bv.y; v[j + 2] += bv.z; v[j + 3] += bv.w;
      }
    }
    if (rb) {
#pragma unroll
      for (int j = 0; j < NC; j += 4) {
        const float4 bv = __ldg(reinterpret_cast<const float4*>(rb + nb + j));
        v[j] += bv.x; v[j + 1] += bv.y; v[j + 2] += bv.z; v[j + 3] += bv.w;
      }
    }
    if (RES) {
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        const float2 f0 = unpack_bf16(rr[j].x), f1 = unpack_bf16(rr[j].y), f2 = unpack_bf16(rr[j].z), f3 = unpack_bf16(rr[j].w);
        v[8 * j + 0] += f0.x; v[8 * j + 1] += f0.y; v[8 * j + 2] += f1.x; v[8 * j + 3] += f1.y;
        v[8 * j + 4] += f2.x; v[8 * j + 5] += f2.y; v[8 * j + 6] += f3.x; v[8 * j + 7] += f3.y;
      }
    }
    if (p.relu) {
#pragma unroll
      for (int j = 0; j < NC; ++j) v[j] = fmaxf(v[j], 0.f);
    }
    if (p.act == 2) {
#pragma unroll
      for (int j = 0; j < NC; ++j) v[j] = __fdividef(v[j], 1.f + __expf(-v[j]));
    } else if (p.act == 3) {
#pragma unroll
      for (int j = 0; j < NC; ++j) v[j] = 0.5f * v[j] * (1.f + erff(v[j] * 0.70710678118654752f));
    }
    if (p.prelu) {
#pragma unroll
      for (int j = 0; j < NC; j += 4) {
        const float4 sv = s_prelu ? *reinterpret_cast<const float4*>(s_prelu + nb + j)
                                  : __ldg(reinterpret_cast<const float4*>(p.prelu + nb + j));
        v[j] = v[j] > 0.f ? v[j] : v[j] * sv.x; v[j + 1] = v[j + 1] > 0.f ? v[j + 1] : v[j + 1] * sv.y;
        v[j + 2] = v[j + 2] > 0.f ? v[j + 2] : v[j + 2] * sv.z; v[j + 3] = v[j + 3] > 0.f ? v[j + 3] : v[j + 3] * sv.w;
      }
    }
    if (!RES) {   // the store that last read this buffer (two chunks ago with two buffers, the previous one otherwise)
      if (lane == 0) {
        if (nbuf == 2) tma_store_wait_read<1>();
        else tma_store_wait_read<0>();
      }
      __syncwarp();
    }
    if (NC == 16 && !RES && p.out_mode == kOutNCHWf32) {
      // ---- fp32 planes [B, n_store, H, W] through a bulk-tensor store: the staging block is [16 planes][32 pixels] fp32 (2 KiB), the
      // tensor map sees the planes as bf16 pairs (a pure byte mover); planes beyond n_store are clipped by the TMA
      const uint32_t blk = buf_of(ectr);
#pragma unroll
      for (int j = 0; j < NC; ++j)
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(blk + static_cast<uint32_t>(j) * 128u + lane * 4u), "r"(__float_as_uint(v[j])) : "memory");
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_4d(cmap, blk, 2 * qx, qy, nb, qb0);
        tma_store_commit();
      }
      ++ectr;
      continue;
    }
    if (NC == 32 && !RES && p.out_mode == kOutQKV) {
      // ---- QKV projection: the quadrant's 32 pixels are 32 consecutive tokens of image qb0 (host-checked); a 32-channel chunk lies
      // inside q, k or v and covers two heads of 16, one head of 32 or part of a wider head.  Q / K [B,heads,N,hd]: rows of the
      // staging block are tokens (two 1 KiB blocks of 32-byte rows for head_dim 16, else one block of 64-byte rows, as for NHWC);
      // V^T [B,heads,hd,N]: rows of the staging block are channels, 32 tokens = 64 bytes each, written two bytes at a time
      // (conflict-free: the 32 lanes of one store fill one row).
      const int which = nb / p.C, c = nb - which * p.C;
      const int tok0 = qy * p.W + qx;
      const uint32_t blk = buf_of(ectr);
      if (which == 0 && p.q_scale != 1.f) {
#pragma unroll
        for (int j = 0; j < NC; ++j) v[j] *= p.q_scale;
      }
      if (which < 2) {
        if (p.hd == 16) {
          const uint32_t s32 = (lane >> 2) & 1;   // SWIZZLE_32B: 16-byte chunk index ^ bit 7 of the address (row / 4)
#pragma unroll
          for (int j = 0; j < NV; ++j)
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(blk + static_cast<uint32_t>(j >> 1) * 1024u + lane * 32u + ((static_cast<uint32_t>(j & 1) ^ s32) << 4)),
                         "r"(pack_bf16(v[8 * j + 0], v[8 * j + 1])), "r"(pack_bf16(v[8 * j + 2], v[8 * j + 3])),
                         "r"(pack_bf16(v[8 * j + 4], v[8 * j + 5])), "r"(pack_bf16(v[8 * j + 6], v[8 * j + 7])) : "memory");
        } else {
#pragma unroll
          for (int j = 0; j < NV; ++j)
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(mine + ((static_cast<uint32_t>(j) ^ sw) << 4)),
                         "r"(pack_bf16(v[8 * j + 0], v[8 * j + 1])), "r"(pack_bf16(v[8 * j + 2], v[8 * j + 3])),
                         "r"(pack_bf16(v[8 * j + 4], v[8 * j + 5])), "r"(pack_bf16(v[8 * j + 6], v[8 * j + 7])) : "memory");
        }
      } else {
#pragma unroll
        for (int j = 0; j < NC; ++j) {
          const __nv_bfloat16 hv = __float2bfloat16_rn(v[j]);
          asm volatile("st.shared.u16 [%0], %1;" ::"r"(blk + static_cast<uint32_t>(j) * 64u + lane * 2u), "h"(*reinterpret_cast<const uint16_t*>(&hv)) : "memory");
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        const CUtensorMap* m = qkv_maps + which;
        if (p.hd == 16) {
          const int head = c >> 4;
          if (which < 2) {
            tma_store_4d(m, blk, 0, tok0, head, qb0);
            tma_store_4d(m, blk + 1024u, 0, tok0, head + 1, qb0);
          } else {
            tma_store_4d(m, blk, tok0, 0, head, qb0);
            tma_store_4d(m, blk + 1024u, tok0, 0, head + 1, qb0);
          }
        } else {
          const int head = c / p.hd, d0 = c - head * p.hd;
          if (which < 2) tma_store_4d(m, blk, d0, tok0, head, qb0);
          else tma_store_4d(m, blk, tok0, d0, head, qb0);
        }
        tma_store_commit();
      }
      ++ectr;
      continue;
    }
#pragma unroll
    for (int j = 0; j < NV; ++j)
      asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(mine + ((static_cast<uint32_t>(j) ^ sw) << 4)),
                   "r"(pack_bf16(v[8 * j + 0], v[8 * j + 1])), "r"(pack_bf16(v[8 * j + 2], v[8 * j + 3])),
                   "r"(pack_bf16(v[8 * j + 4], v[8 * j + 5])), "r"(pack_bf16(v[8 * j + 6], v[8 * j + 7])) : "memory");
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) {
      if (p.phase_n > 0) {   // phase-block output (PixelShuffle): block nb / phase_n has its own strided map
        const int ph = nb / p.phase_n;
        tma_store_4d(ph == 0 ? cmap : qkv_maps + (ph - 1), buf_of(ectr), nb - ph * p.phase_n, qx, qy, qb0);
      } else {
        tma_store_4d(cmap, buf_of(ectr), nb, qx, qy, qb0);
      }
      tma_store_commit();
    }
    ++ectr;
  }
}

// Residual STREAM epilogue (LEAN == 3) for memory-bound layers with a residual input (1x1 convolutions with K <= 768).  The lean
// epilogue keeps ONE residual box (2 KiB) in flight per epilogue warp: tools/micro/tma_store_rate.cu shows that this pattern moves
// one box per DRAM round trip (~2000 clk) and warp, 2.3 TB/s each way - the bytes in flight bound those layers.  Here the residual
// boxes of a warp form a stream that runs NL - 1 boxes ahead of the accumulators and across tile boundaries: NL load buffers (one
// mbarrier each) separate from two store buffers; after chunk i has been staged for its store, the box of chunk i + NL is requested
// into the load buffer chunk i has just released (its rows were read into registers before the math; every lane fences generic ->
// async before the elected lane issues the load).  The stream's cursor - tile, chunk and the DECODED coordinates of that tile, which
// are recomputed only when the cursor moves to a new tile - is warp-uniform state.  Host guarantees N % BN == 0 and BN % 64 == 0.
struct ResStream {
  int tile, k;             // next box to request: tile index, chunk number of this warp within the tile
  int n0, qx, qy, qb;      // decoded origin of that tile's quadrant box
  uint32_t req_slot;       // slot of the next request (counters instead of issued % nl: no integer division in the chain)
  uint32_t slot, phase;    // slot and mbarrier parity of the next chunk to process
  uint32_t sbuf;           // store buffer (0 / 1) of the next chunk
};

// ROWK: 0 plain taps; 3: row-segment mode for a 3 x 3 window; 9: for a 1 x 9 window (compile-time so that the tap loops of the producer and
// of the MMA issuer unroll - with run-time tap counts the 3 x 3 layers lost 8 %)
template <int ROWK, bool TMA_OUT, bool TMA_RES, int LEAN = 0>   // LEAN: 0 generic epilogue, 1 lean, 3 lean with the residual stream
__global__ void __launch_bounds__(kThreads, 1)
igemm_kernel(const __grid_constant__ IgemmMaps maps, const __grid_constant__ IgemmArgs p) {
  extern __shared__ uint8_t smem_raw[];
  // Pipeline depth is chosen per launch: narrow N tiles have small stages, so more of them fit and more bytes are in
  // flight per SM (these layers are TMA-latency bound, not tensor bound).
  constexpr bool ROW3 = ROWK != 0;
  constexpr int kNky = ROWK == 3 ? 3 : 1, kNkx = ROWK == 0 ? 1 : ROWK;
  constexpr uint32_t kAOff = ROW3 ? kRowABytes : kABytes;   // offset of the B tile(s) inside a stage
  const int kStages = p.nstages;
  const uint32_t kBTile = static_cast<uint32_t>(p.BN) * kIgemmBK * 2;
  const uint32_t kStageSz = kAOff + (p.wres ? 0u : static_cast<uint32_t>(kNkx) * kBTile);
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t wres_base = smem_base + static_cast<uint32_t>(kStages) * kStageSz;   // resident weights sit right behind the ring
  const uint32_t bar_base = smem_base + kPipeBytes + kOutStageBytes;   // [ring | output staging | barriers | bias / PReLU]
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * kStages + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * kStages + 2 + a); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * kStages + 4);
  const uint32_t wfull_bar = bar_base + 8u * (2 * kMaxStages + 13);   // resident weights have landed
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // provably warp-uniform (role dispatch below)
  const int lane = threadIdx.x & 31;
  // bias / PReLU vectors -> shared memory (read once per CTA instead of once per tile from L2)
  float* s_vec = reinterpret_cast<float*>(smem_raw + (bar_base + kBarBytes - smem_u32(smem_raw)));
  const bool bias_in_smem = p.bias && p.N <= kBiasMaxN, prelu_in_smem = p.prelu && p.N <= kPreluMaxN;
  const float* s_bias = bias_in_smem ? s_vec : nullptr;
  const float* s_prelu = prelu_in_smem ? s_vec + kBiasMaxN : nullptr;

  const int tiles_x = (p.W + p.tw - 1) / p.tw, tiles_y = (p.H + p.th - 1) / p.th, tiles_b = (p.B + p.tb - 1) / p.tb;
  const int m_tiles = tiles_x * tiles_y * tiles_b;
  const int n_tiles = (p.N + p.BN - 1) / p.BN;
  const int total_tiles = m_tiles * n_tiles;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < kMaxMaps; ++i) tma_prefetch_desc(&maps.a[i]);
    tma_prefetch_desc(&maps.b);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < kStages; ++s) {
        mbar_init(full_bar(s), 1);
        mbar_init(empty_bar(s), 1);
      }
      for (int a = 0; a < 2; ++a) {
        mbar_init(tfull_bar(a), 1);
        mbar_init(tempty_bar(a), 256);
      }
      for (int w = 0; w < 8; ++w) mbar_init(bar_base + 8u * (2 * kMaxStages + 5 + w), 1);   // residual boxes (tma_res)
      if (LEAN == 3)
        for (int i = 0; i < 32; ++i) mbar_init(bar_base + 8u * (32 + i), 1);                // residual stream (LEAN == 3)
      mbar_init(wfull_bar, 1);
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  // Programmatic dependent launch: everything above (descriptor prefetch, mbarrier init, TMEM allocation) touches no global
  // data and overlaps the tail of the previous kernel; from here on this kernel reads activations / writes outputs.
  pdl_launch_dependents();
  pdl_wait();
  for (int i = threadIdx.x; i < p.N; i += blockDim.x) {
    if (bias_in_smem) s_vec[i] = p.bias[i];
    if (prelu_in_smem) s_vec[kBiasMaxN + i] = p.prelu[i];
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  auto decode = [&](int tile, int& n0, int& b0, int& y0, int& x0) {
    const int nt = tile % n_tiles, mt = tile / n_tiles;
    n0 = nt * p.BN;
    x0 = (mt % tiles_x) * p.tw;
    y0 = ((mt / tiles_x) % tiles_y) * p.th;
    b0 = (mt / (tiles_x * tiles_y)) * p.tb;
  };

  // Producer and MMA warps run their loops in warp-uniform control flow and ONE ELECTED lane issues (elect.sync): the
  // compiler then keeps stage counters / descriptors in uniform registers and emits bare UTCHMMA / UTMALDG sequences.
  // Issuing from inside `if (lane == 0)` wraps every such instruction in an ELECT / PLOP3 / BRA.U.ANY loop plus R2UR moves
  // (~10 SASS instructions per MMA); for the narrow layers (N <= 64) that made the issuing thread the limiter.
  if (warp == 0) {
    {
      // ===================== TMA producer =====================
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t tx_bytes = kABytes + (p.wres ? 0u : kBTile);
      if (p.wres) {   // the whole weight matrix, once: total_kb tiles of BN x 64 (n_tiles == 1)
        if (elect_one_sync()) {
          mbar_arrive_expect_tx(wfull_bar, static_cast<uint32_t>(p.total_kb) * kBTile);
          for (int kb = 0; kb < p.total_kb; ++kb) tma_load_2d(wres_base + kb * kBTile, &maps.b, wfull_bar, kb * kIgemmBK, 0);
        }
        __syncwarp();
      }
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        int n0, b0, y0, x0;
        decode(tile, n0, b0, y0, x0);
        int kb_global = 0;
        int t_first = 0;
        if (ROW3) {
          // taps 0 .. nky*nkx-1 are the window (ky-major) over map 0, all with nkb = p.taps[0].nkb channel blocks; one box of
          // 128 + nkx - 1 pixels of an image row serves the nkx horizontal taps (3x3: nky = nkx = 3; 1x9: nky = 1, nkx = 9)
          const int nkb = p.taps[0].nkb;
          constexpr int nky = kNky, nkx = kNkx;
          const uint32_t b_bytes = static_cast<uint32_t>(p.BN) * kIgemmBK * 2;
          const uint32_t a_bytes = static_cast<uint32_t>(128 + nkx - 1) * 128u;
          for (int ky = 0; ky < nky; ++ky)
            for (int kb = 0; kb < nkb; ++kb) {
              mbar_wait(empty_bar(stage), phase ^ 1u);
              if (elect_one_sync()) {
                const uint32_t sa = smem_base + stage * kStageSz;
                mbar_arrive_expect_tx(full_bar(stage), a_bytes + (p.wres ? 0u : static_cast<uint32_t>(nkx) * b_bytes));
                tma_load_4d(sa, &maps.a[2], full_bar(stage), kb * kIgemmBK, x0 - nkx / 2, y0 + ky - nky / 2, b0);
                for (int kx = 0; kx < nkx && !p.wres; ++kx)
                  tma_load_2d(sa + kAOff + kx * b_bytes, &maps.b, full_bar(stage), ((ky * nkx + kx) * nkb + kb) * kIgemmBK, n0);
              }
              __syncwarp();
              if (++stage == kStages) { stage = 0; phase ^= 1u; }
            }
          t_first = nky * nkx;
          kb_global = nky * nkx * nkb;
        }
        for (int t = t_first; t < p.ntaps; ++t) {
          const IgemmTap tap = p.taps[t];
          const CUtensorMap* amap = &maps.a[tap.map];
          for (int kb = 0; kb < tap.nkb; ++kb, ++kb_global) {
            mbar_wait(empty_bar(stage), phase ^ 1u);
            if (elect_one_sync()) {
              const uint32_t sa = smem_base + stage * kStageSz;
              mbar_arrive_expect_tx(full_bar(stage), tx_bytes);
              tma_load_4d(sa, amap, full_bar(stage), kb * kIgemmBK, x0 + tap.dx, y0 + tap.dy, b0);
              if (!p.wres) tma_load_2d(sa + kAOff, &maps.b, full_bar(stage), kb_global * kIgemmBK, n0);
            }
            __syncwarp();
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    {
      // ===================== MMA issuer =====================
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t idesc = umma_idesc_bf16(kIgemmBM, static_cast<uint32_t>(p.BN));
      // descriptor pieces (see umma_desc_join): constant high word, low words for stage 0, per-stage increment
      const uint64_t d0 = umma_smem_desc(smem_base, 128, 1024);
      const uint32_t dhi = umma_desc_hi(d0), a_lo0 = umma_desc_lo(d0), b_lo0 = a_lo0 + (kAOff >> 4);
      const uint32_t stage16 = kStageSz >> 4, bt16 = kBTile >> 4;
      const uint32_t w_lo0 = a_lo0 + ((wres_base - smem_base) >> 4);   // resident weights: descriptor start of k-block 0
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      if (p.wres) mbar_wait(wfull_bar, 0);
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const int a = it & 1;
        const uint32_t aphase = (it >> 1) & 1u;
        mbar_wait(tempty_bar(a), aphase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_u + static_cast<uint32_t>(a) * 256u;
        int ks_first = 0;
        if (ROW3) {
          constexpr int nkx = kNkx;
          const int nseg = kNky * p.taps[0].nkb;
          for (int sg = 0; sg < nseg; ++sg) {
            mbar_wait(full_bar(stage), phase);
            tc_fence_after();
            if (elect_one_sync()) {
              // stage sg = (ky, kb): its three B tiles are k-blocks (ky*3 + kx) * nkb + kb of the packed weights
              const int nkb3 = p.taps[0].nkb, ky3 = sg / nkb3, kb3 = sg - ky3 * nkb3;
              const uint32_t a_lo = a_lo0 + stage * stage16;
              const uint32_t b_lo = p.wres ? w_lo0 + static_cast<uint32_t>(ky3 * nkx * nkb3 + kb3) * bt16 : b_lo0 + stage * stage16;
              const uint32_t bkx16 = p.wres ? static_cast<uint32_t>(nkb3) * bt16 : bt16;
#pragma unroll
              for (int kx = 0; kx < nkx; ++kx) {
                // window of 128 pixels starting kx pixels (kx*128 B = 8 descriptor units) into the row segment; the
                // UMMA swizzle is a function of the absolute shared-memory address, so the shifted start needs no fix-up
#pragma unroll
                for (int k = 0; k < kIgemmBK / 16; ++k)
                  umma_bf16(d_tmem, umma_desc_join(a_lo + 8u * kx + 2u * k, dhi), umma_desc_join(b_lo + kx * bkx16 + 2u * k, dhi), idesc,
                            (sg | kx | k) != 0 ? 1u : 0u);
              }
              umma_commit(empty_bar(stage));
            }
            __syncwarp();
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
          ks_first = kNky * nkx * p.taps[0].nkb;
        }
        for (int ks = ks_first; ks < p.total_kb; ++ks) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          if (elect_one_sync()) {
            const uint32_t a_lo = a_lo0 + stage * stage16;
            const uint32_t b_lo = p.wres ? w_lo0 + static_cast<uint32_t>(ks) * bt16 : b_lo0 + stage * stage16;
#pragma unroll
            for (int k = 0; k < kIgemmBK / 16; ++k)
              umma_bf16(d_tmem, umma_desc_join(a_lo + 2u * k, dhi), umma_desc_join(b_lo + 2u * k, dhi), idesc, (ks | k) != 0 ? 1u : 0u);
            umma_commit(empty_bar(stage));
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
        if (elect_one_sync()) umma_commit(tfull_bar(a));
        __syncwarp();
      }
    }
  } else {
    // ===================== epilogue warps (2..9) =====================
    const int quad = warp & 3;  // TMEM lane quadrant this warp may access
    const int grp = (warp - 2) >> 2;  // 0 or 1: which half of the interleaved N chunks
    const int row = quad * 32 + lane;
    // TMA-store epilogue: this warp's staging buffer (1024-byte aligned) and the origin of its 32-pixel box inside the tile
    const uint32_t out_stage = smem_base + kPipeBytes + static_cast<uint32_t>(warp - 2) * 2048u;
    // residual staging (tma_res): the last 16 KiB of the ring area (free by construction), one mbarrier per warp
    const uint32_t res_stage = smem_base + kPipeBytes - kOutStageBytes + static_cast<uint32_t>(warp - 2) * 2048u;
    const uint32_t res_bar = bar_base + 8u * (2 * kMaxStages + 5 + (warp - 2));
    uint32_t res_phase = 0;
    uint32_t ectr = 0;     // lean epilogue: this warp's running chunk count (selects the staging buffer)
    const int q_pix = quad * 32;
    const int qx0 = q_pix % p.tw, qy0 = (q_pix / p.tw) % p.th, qb0 = q_pix / (p.tw * p.th);
    // residual stream (LEAN == 3): [2 store blocks | res_deep load blocks] of 16 KiB end where the output staging ends; every warp
    // owns the 2 KiB slice (warp - 2) of each block
    const int nl = p.res_deep;
    const int nbox = p.stream_res + p.stream_mask;   // boxes per slot: residual rows, then ReLU-mask rows
    const uint32_t deep_base = smem_base + kPipeBytes + kOutStageBytes - static_cast<uint32_t>(2 + nl * nbox) * kOutStageBytes + static_cast<uint32_t>(warp - 2) * 2048u;
    const uint32_t lbuf0 = deep_base + 2 * kOutStageBytes;
    const uint32_t lbar0 = bar_base + 8u * (32 + 4 * (warp - 2));
    const int ncw = p.BN / 64;   // chunks of this warp per tile (LEAN == 3: BN % 64 == 0, N % BN == 0)
    ResStream rs{static_cast<int>(blockIdx.x), 0, 0, 0, 0, 0, 0u, 0u, 0u, 0u};
    auto rs_decode = [&]() {
      if (rs.tile < total_tiles) {
        int n0, b0, y0, x0;
        decode(rs.tile, n0, b0, y0, x0);
        rs.n0 = n0; rs.qx = x0 + qx0; rs.qy = y0 + qy0; rs.qb = b0 + qb0;
      }
    };
    auto rs_request = [&]() {
      if (rs.tile >= total_tiles) return;
      const uint32_t slot = rs.req_slot;
      if (lane == 0) {
        mbar_arrive_expect_tx(lbar0 + 8u * slot, static_cast<uint32_t>(nbox) * 32 * 2 * 32);
        uint32_t dstb = lbuf0 + slot * static_cast<uint32_t>(nbox) * kOutStageBytes;
        if (p.stream_res) {
          tma_load_4d(dstb, &maps.r, lbar0 + 8u * slot, rs.n0 + grp * 32 + rs.k * 64, rs.qx, rs.qy, rs.qb);
          dstb += kOutStageBytes;
        }
        if (p.stream_mask) tma_load_4d(dstb, &maps.m, lbar0 + 8u * slot, rs.n0 + grp * 32 + rs.k * 64, rs.qx, rs.qy, rs.qb);
      }
      if (++rs.req_slot == static_cast<uint32_t>(nl)) rs.req_slot = 0;
      if (++rs.k == ncw) {
        rs.k = 0;
        rs.tile += gridDim.x;
        rs_decode();
      }
    };
    const int bb = row / (p.th * p.tw), rem = row % (p.th * p.tw), yy = rem / p.tw, xx = rem % p.tw;
    int it = 0;
    if (LEAN == 3) {
      rs_decode();
      for (int i = 0; i < nl; ++i) rs_request();
    }
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int a = it & 1;
      const uint32_t aphase = (it >> 1) & 1u;
      int n0, b0, y0, x0;
      decode(tile, n0, b0, y0, x0);
      const int b = b0 + bb, y = y0 + yy, x = x0 + xx;
      const bool valid = (b < p.B) && (y < p.H) && (x < p.W);
      const uint32_t tacc = tmem_base + static_cast<uint32_t>(a) * 256u + (static_cast<uint32_t>(quad * 32) << 16);
      if (LEAN == 3) {
        // ---- residual stream: chunks grp*32 + k*64 of this tile; residual rows come from the load ring, results go out through two
        // alternating store buffers
        constexpr int NC = 32, NV = 4;
        const uint32_t sw = (lane >> 1) & 3;
        const uint32_t row_off = static_cast<uint32_t>(lane) * (NC * 2);
        mbar_wait(tfull_bar(a), aphase);
        tc_fence_after();
        const float* rb = p.rowbias ? p.rowbias + static_cast<size_t>(b < p.B ? b : p.B - 1) * p.ldrb : nullptr;
        for (int k = 0; k < ncw; ++k) {
          const int c0 = grp * NC + k * 2 * NC, nb = n0 + c0;
          uint32_t r[NC];
          tmem_ld_n<NC>(tacc + c0, r);
          const uint32_t slot = rs.slot;
          mbar_wait(lbar0 + 8u * slot, rs.phase);
          uint4 rr[NV], mm[NV];
          {
            uint32_t src = lbuf0 + slot * static_cast<uint32_t>(nbox) * kOutStageBytes + row_off;
            if (p.stream_res) {
#pragma unroll
              for (int j = 0; j < NV; ++j)
                asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(rr[j].x), "=r"(rr[j].y), "=r"(rr[j].z), "=r"(rr[j].w)
                             : "r"(src + ((static_cast<uint32_t>(j) ^ sw) << 4)) : "memory");
              src += kOutStageBytes;
            }
            if (p.stream_mask) {
#pragma unroll
              for (int j = 0; j < NV; ++j)
                asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(mm[j].x), "=r"(mm[j].y), "=r"(mm[j].z), "=r"(mm[j].w)
                             : "r"(src + ((static_cast<uint32_t>(j) ^ sw) << 4)) : "memory");
            }
          }
          tmem_wait_ld();
          float v[NC];
#pragma unroll
          for (int j = 0; j < NC; ++j) v[j] = __uint_as_float(r[j]);
          if (s_bias) {
#pragma unroll
            for (int j = 0; j < NC; j += 4) {
              const float4 bv = *reinterpret_cast<const float4*>(s_bias + nb + j);
              v[j] += bv.x; v[j + 1] += bv.y; v[j + 2] += bv.z; v[j + 3] += bv.w;
            }
          } else if (p.bias) {
#pragma unroll
            for (int j = 0; j < NC; j += 4) {
              const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + nb + j));
              v[j] += bv.x; v[j + 1] += bv.y; v[j + 2] += bv.z; v[j + 3] += bv.w;
            }
          }
          if (rb) {
#pragma unroll
            for (int j = 0; j < NC; j += 4) {
              const float4 bv = __ldg(reinterpret_cast<const float4*>(rb + nb + j));
              v[j] += bv.x; v[j + 1] += bv.y; v[j + 2] += bv.z; v[j + 3] += bv.w;
            }
          }
          if (p.stream_res) {
#pragma unroll
            for (int j = 0; j < NV; ++j) {
              const float2 f0 = unpack_bf16(rr[j].x), f1 = unpack_bf16(rr[j].y), f2 = unpack_bf16(rr[j].z), f3 = unpack_bf16(rr[j].w);
              v[8 * j + 0] += f0.x; v[8 * j + 1] += f0.y; v[8 * j + 2] += f1.x; v[8 * j + 3] += f1.y;
              v[8 * j + 4] += f2.x; v[8 * j + 5] += f2.y; v[8 * j + 6] += f3.x; v[8 * j + 7] += f3.y;
            }
          }
          if (p.relu) {
#pragma unroll
            for (int j = 0; j < NC; ++j) v[j] = fmaxf(v[j], 0.f);
          }
          if (p.act == 2) {
#pragma unroll
            for (int j = 0; j < NC; ++j) v[j] = __fdividef(v[j], 1.f + __expf(-v[j]));
          }
          if (p.stream_mask) {   // ReLU derivative of the forward activation (segmentor data gradients)
#pragma unroll
            for (int j = 0; j < NV; ++j) {
              const float2 f0 = unpack_bf16(mm[j].x), f1 = unpack_bf16(mm[j].y), f2 = unpack_bf16(mm[j].z), f3 = unpack_bf16(mm[j].w);
              if (!(f0.x > 0.f)) v[8 * j + 0] = 0.f;
              if (!(f0.y > 0.f)) v[8 * j + 1] = 0.f;
              if (!(f1.x > 0.f)) v[8 * j + 2] = 0.f;
              if (!(f1.y > 0.f)) v[8 * j + 3] = 0.f;
              if (!(f2.x > 0.f)) v[8 * j + 4] = 0.f;
              if (!(f2.y > 0.f)) v[8 * j + 5] = 0.f;
              if (!(f3.x > 0.f)) v[8 * j + 6] = 0.f;
              if (!(f3.y > 0.f)) v[8 * j + 7] = 0.f;
            }
          }
          if (lane == 0) tma_store_wait_read<1>();   // the store that read this store buffer two chunks ago is done with it
          __syncwarp();
          const uint32_t dst = deep_base + rs.sbuf * kOutStageBytes;
#pragma unroll
          for (int j = 0; j < NV; ++j)
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(dst + row_off + ((static_cast<uint32_t>(j) ^ sw) << 4)),
                         "r"(pack_bf16(v[8 * j + 0], v[8 * j + 1])), "r"(pack_bf16(v[8 * j + 2], v[8 * j + 3])),
                         "r"(pack_bf16(v[8 * j + 4], v[8 * j + 5])), "r"(pack_bf16(v[8 * j + 6], v[8 * j + 7])) : "memory");
          fence_proxy_async_smem();   // orders this lane's st.shared AND its earlier ld.shared of the load buffer before the async proxy
          __syncwarp();
          if (lane == 0) {
            tma_store_4d(&maps.c, dst, nb, x0 + qx0, y0 + qy0, b0 + qb0);
            tma_store_commit();
          }
          rs.sbuf ^= 1u;
          if (++rs.slot == static_cast<uint32_t>(nl)) { rs.slot = 0; rs.phase ^= 1u; }
          rs_request();   // box of the chunk nl ahead, into the slot just released
        }
      } else if (LEAN) {
        if ((p.BN % 32 == 0) && (p.N % 32 == 0) && p.out_mode != kOutNCHWf32)
          epilogue_tile_lean<32, TMA_RES>(p, tacc, n0, b, grp, s_bias, s_prelu, tfull_bar(a), aphase, &maps.c, &maps.r, out_stage, res_stage,
                                          p.stage2 ? 2 : 1, x0 + qx0, y0 + qy0, b0 + qb0, res_bar, res_phase, ectr, maps.qkv);
        else
          epilogue_tile_lean<16, TMA_RES>(p, tacc, n0, b, grp, s_bias, s_prelu, tfull_bar(a), aphase, &maps.c, &maps.r, out_stage, res_stage,
                                          p.stage2 ? 2 : 1, x0 + qx0, y0 + qy0, b0 + qb0, res_bar, res_phase, ectr);
      } else if (p.out_mode != kOutQKV && (p.BN % 32 == 0) && (p.N % 32 == 0) && !(p.out_mode == kOutNCHWf32 && p.BN == 32))
        // (fp32 planes with a single 32-column N tile: 16-column chunks keep BOTH epilogue groups busy)
        epilogue_tile<32, TMA_OUT, TMA_RES>(p, tacc, n0, b, y, x, valid, grp, s_bias, s_prelu, tfull_bar(a), aphase, &maps.c, out_stage, x0 + qx0,
                          y0 + qy0, b0 + qb0, &maps.r, res_stage, res_bar, res_phase);
      else
        epilogue_tile<16, TMA_OUT, TMA_RES>(p, tacc, n0, b, y, x, valid, grp, s_bias, s_prelu, tfull_bar(a), aphase, &maps.c, out_stage, x0 + qx0,
                          y0 + qy0, b0 + qb0, &maps.r, res_stage, res_bar, res_phase);
      tc_fence_before();
      mbar_arrive(tempty_bar(a));
    }
    if (TMA_OUT && lane == 0) tma_store_wait_read0();   // shared memory must outlive the last bulk store's read
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace

// wres_bytes > 0: resident weights (that many bytes behind the ring), stages carry activations only; 16 KiB are then always
// left for the second staging buffer of the lean epilogue
int igemm_stages_for(int BN, int row3, int wres_bytes, int row_nkx) {
  if (wres_bytes > 0) {
    const uint32_t stage = row3 ? kRowABytes : kABytes;
    int n = static_cast<int>((kPipeBytes - kOutStageBytes - static_cast<uint32_t>(wres_bytes)) / stage);
    return n > kMaxStages ? kMaxStages : n;
  }
  const uint32_t stage = (row3 ? kRowABytes : kABytes) + (row3 ? static_cast<uint32_t>(row_nkx) : 1u) * static_cast<uint32_t>(BN) * kIgemmBK * 2;
  // stages must stay 1024-byte aligned: BN is a multiple of 16 -> BN*128 is a multiple of 2048
  int n = static_cast<int>(kPipeBytes / stage);
  return n > kMaxStages ? kMaxStages : n;
}

int igemm_res_deep_stages(int BN, int nl) {
  const uint32_t stage = kABytes + static_cast<uint32_t>(BN) * kIgemmBK * 2;
  const uint32_t cap = kPipeBytes + kOutStageBytes - static_cast<uint32_t>(2 + nl) * kOutStageBytes;
  int n = static_cast<int>(cap / stage);
  return n > kMaxStages ? kMaxStages : n;
}

bool igemm_res_staging_fits(int BN, int row3, int nstages, int wres_bytes, int row_nkx) {
  const uint32_t stage = (row3 ? kRowABytes : kABytes) + (wres_bytes > 0 ? 0u : (row3 ? static_cast<uint32_t>(row_nkx) : 1u) * static_cast<uint32_t>(BN) * kIgemmBK * 2);
  return static_cast<uint32_t>(nstages) * stage + static_cast<uint32_t>(wres_bytes > 0 ? wres_bytes : 0) + kOutStageBytes <= kPipeBytes;
}

template <int ROWK, bool TMA_OUT, bool TMA_RES, int LEAN = 0>
static int launch_variant(const IgemmPlan& plan, cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    WC_CHECK_CUDA(cudaFuncSetAttribute(igemm_kernel<ROWK, TMA_OUT, TMA_RES, LEAN>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    attr_set = true;
  }
  launch_k<1>(igemm_kernel<ROWK, TMA_OUT, TMA_RES, LEAN>, plan.grid, kThreads, kSmemBytes, stream, plan.maps, plan.args);
  return 0;
}

int igemm_launch(const IgemmPlan& plan, cudaStream_t stream) {
  ProfScope prof(kProfIgemm, stream, plan.flops);
  prof.note(plan.args.B * plan.args.H * plan.args.W, plan.args.N, plan.args.total_kb * kIgemmBK, plan.args.BN, plan.args.ntaps + 100 * plan.args.row3 + 1000 * (plan.args.lean != 0) + 32000 * (plan.args.lean == 3) + 2000 * (plan.args.mask != nullptr) + 4000 * (plan.args.res != nullptr) +
                8000 * (plan.args.out_mode != kOutNHWC) + 16000 * (plan.args.tma_store == 0), plan.grid);
  const int variant = plan.args.tma_store ? (plan.args.tma_res ? 2 : 1) : 0;   // epilogue: per-lane stores / TMA store / TMA store + TMA residual
  int e = 0;
  if (plan.args.row3 && plan.args.row_nkx == 9) {   // 1 x 9 row-segment mode (build_conv_hrow): fp32 planes, lean or generic epilogue
    e = plan.args.lean ? launch_variant<9, true, false, 1>(plan, stream) : launch_variant<9, false, false>(plan, stream);
  } else if (plan.args.lean == 3) {
    e = launch_variant<0, true, true, 3>(plan, stream);
  } else if (plan.args.lean) {
    if (plan.args.row3) e = plan.args.tma_res ? launch_variant<3, true, true, 1>(plan, stream) : launch_variant<3, true, false, 1>(plan, stream);
    else e = plan.args.tma_res ? launch_variant<0, true, true, 1>(plan, stream) : launch_variant<0, true, false, 1>(plan, stream);
  } else if (plan.args.row3) e = variant == 2 ? launch_variant<3, true, true>(plan, stream) : variant == 1 ? launch_variant<3, true, false>(plan, stream) : launch_variant<3, false, false>(plan, stream);
  else e = variant == 2 ? launch_variant<0, true, true>(plan, stream) : variant == 1 ? launch_variant<0, true, false>(plan, stream) : launch_variant<0, false, false>(plan, stream);
  if (e) return e;
  WC_LAUNCH_CHECK();
  return 0;
}

static int pow2_floor(int v) {
  int p = 1;
  while (p * 2 <= v) p *= 2;
  return p;
}

void igemm_pick_tile(int B, int H, int W, int* tb, int* th, int* tw) {
  int w = pow2_floor(W);
  if (w < W && w * 2 <= 128) w *= 2;  // non power-of-two widths: cover with an over-hanging tile
  if (w > 128) w = 128;
  int rem = 128 / w;
  int h = pow2_floor(H);
  if (h < H && h * 2 <= rem) h *= 2;
  if (h > rem) h = rem;
  *tw = w; *th = h; *tb = 128 / (w * h);
  (void)B;
}

int igemm_pick_bn(int N, long m_tiles) {
  // Candidate N tiles (multiples of 16, <= 256, not wider than the padded N); pick the one minimising
  // waves * per-tile cost, where the per-tile cost has a fixed part that penalises very narrow tiles.
  const int npad = (N + 15) / 16 * 16;
  int cands[9] = {256, 192, 128, 96, 64, 48, 32, 16, npad <= 256 ? npad : 16};
  const int sms = num_sms();
  int best = 16;
  double best_cost = 1e30;
  for (int bn : cands) {
    if (bn > npad) continue;
    const long n_tiles = (N + bn - 1) / bn;
    const long waves = (m_tiles * n_tiles + sms - 1) / sms;
    const double cost = static_cast<double>(waves) * (bn + 48.0);
    if (cost < best_cost - 1e-9) { best_cost = cost; best = bn; }
  }
  return best;
}

int igemm_make_amap(CUtensorMap* out, const Act& act, int tb, int th, int tw, int y0, int ys, int x0, int xs, int Hv,
                    int Wv) {
  if (Hv < 0) Hv = act.H;
  if (Wv < 0) Wv = act.W;
  const __nv_bfloat16* base = act.ptr + (static_cast<size_t>(y0) * act.W + x0) * act.ld;
  uint64_t dims[4] = {static_cast<uint64_t>(act.C), static_cast<uint64_t>(Wv), static_cast<uint64_t>(Hv),
                      static_cast<uint64_t>(act.B)};
  uint64_t strides[4] = {1, static_cast<uint64_t>(act.ld) * xs, static_cast<uint64_t>(act.ld) * act.W * ys,
                         static_cast<uint64_t>(act.ld) * act.W * act.H};
  uint32_t box[4] = {static_cast<uint32_t>(kIgemmBK), static_cast<uint32_t>(tw), static_cast<uint32_t>(th),
                     static_cast<uint32_t>(tb)};
  return encode_tmap_bf16(out, base, 4, dims, strides, box, 128);
}

int igemm_make_rowseg_map(CUtensorMap* out, const Act& act, int nkx) {
  WC_REQUIRE(nkx >= 1 && (128u + nkx - 1) * 128u <= kRowABytes, "row segment does not fit its stage slot");
  uint64_t dims[4] = {static_cast<uint64_t>(act.C), static_cast<uint64_t>(act.W), static_cast<uint64_t>(act.H),
                      static_cast<uint64_t>(act.B)};
  uint64_t strides[4] = {1, static_cast<uint64_t>(act.ld), static_cast<uint64_t>(act.ld) * act.W,
                         static_cast<uint64_t>(act.ld) * act.W * act.H};
  uint32_t box[4] = {static_cast<uint32_t>(kIgemmBK), static_cast<uint32_t>(128 + nkx - 1), 1, 1};
  return encode_tmap_bf16(out, act.ptr, 4, dims, strides, box, 128);
}

int igemm_make_cmap(CUtensorMap* out, const Act& act, int N, int nc, int qw, int qh, int qb, int sy, int sx, int py, int px) {
  // (sy, sx, py, px) != (1, 1, 0, 0): the map covers the phase view act(b, y*sy + py, x*sx + px, c) of an up-sampled output grid
  // (transposed convolutions, stride-2 data gradients, PixelShuffle), so those launches can use the TMA-store epilogue too
  uint64_t dims[4] = {static_cast<uint64_t>(N), static_cast<uint64_t>(act.W / sx), static_cast<uint64_t>(act.H / sy),
                      static_cast<uint64_t>(act.B)};
  uint64_t strides[4] = {1, static_cast<uint64_t>(act.ld) * sx, static_cast<uint64_t>(act.ld) * act.W * sy,
                         static_cast<uint64_t>(act.ld) * act.W * act.H};
  uint32_t box[4] = {static_cast<uint32_t>(nc), static_cast<uint32_t>(qw), static_cast<uint32_t>(qh), static_cast<uint32_t>(qb)};
  const __nv_bfloat16* base = act.ptr + (static_cast<size_t>(py) * act.W + px) * act.ld;
  return encode_tmap_bf16(out, base, 4, dims, strides, box, static_cast<uint32_t>(nc * 2));
}

int igemm_make_bmap(CUtensorMap* out, const __nv_bfloat16* wpacked, int n_rows, int ktotal, int BN) {
  uint64_t dims[2] = {static_cast<uint64_t>(ktotal), static_cast<uint64_t>(n_rows)};
  uint64_t strides[2] = {1, static_cast<uint64_t>(ktotal)};
  uint32_t box[2] = {static_cast<uint32_t>(kIgemmBK), static_cast<uint32_t>(BN)};
  return encode_tmap_bf16(out, wpacked, 2, dims, strides, box, 128);
}

}  // namespace wc
