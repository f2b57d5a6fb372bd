// Flash-style multi-head self-attention on tcgen05 (sm_100a).  Replaces the softmax(QK^T/sqrt(hd))V core of
// nn.MultiheadAttention at unet_base.py:115,159,214,257,320,365 (in/out projections run on the igemm path).
//
// One CTA owns NQ query tiles of 128 rows of one (batch, head) and streams K / V^T tiles of BKV keys:
//   warp 0      TMA producer (Q once, then K_j and V^T_j through 2-stage rings)
//   warp 1      MMA issuer:  S_q = Q_q K_j^T  (128 x BKV x hd)  and  O_q += P_q V_j  (128 x hd x BKV)
//   warp 2      TMEM allocator
//   warps 4-7   softmax for query tile 0 (one thread per query row; no shuffles needed)
//   warps 8-11  softmax for query tile 1 (NQ == 2): while one group exponentiates, the tensor core works for
//               the other group, so MUFU and tcgen05 overlap.
// S, O and P live in TMEM (per query tile: BKV + hd fp32 columns, then BKV / 2 columns of bf16 pairs): the softmax threads write P
// with tcgen05.st (lane = query row) and the PV tcgen05.mma reads it as its A operand; V is consumed as V^T[hd][keys] (K-major B
// operand), which the QKV projection epilogue writes directly.  Head_dim 16 / 32 run on attention_small.cu instead.  Online softmax with lazy rescaling (only when the running max grows
// by more than 2^8), accumulation in fp32.
#include "wc_host.h"
#include "wc_ptx.cuh"

#include <type_traits>

namespace wc {

namespace {

struct AttnArgs {
  int ntok, heads, ldo;
  float scale_log2;  // log2(e) / sqrt(hd)
  __nv_bfloat16* out;
  float* lse;  // optional [B*heads][ntok]: log2-domain log-sum-exp of every row (saved for the backward pass)
};

template <int HD, int BKV, int NQ>
struct AttnCfg {
  static constexpr int kKBlocks = HD >= 64 ? HD / 64 : 1;          // 64-wide K blocks of the QK^T contraction
  static constexpr int kSwz = HD >= 64 ? 128 : HD * 2;             // swizzle span of Q/K rows (bytes)
  static constexpr int kRowBytes = HD >= 64 ? 128 : HD * 2;        // bytes per row within one block
  static constexpr int kKSteps = HD >= 64 ? 4 : HD / 16;           // 16-element MMA K steps per block
  static constexpr uint32_t kQTile = 128 * HD * 2;
  static constexpr uint32_t kKTile = BKV * HD * 2;
  static constexpr uint32_t kVTile = HD * BKV * 2;
  static constexpr int kStages = 2;
  static constexpr uint32_t kSmem = NQ * kQTile + kStages * (kKTile + kVTile) + 1024 + 256;
  static constexpr int kThreads = 128 + 128 * NQ;
  static constexpr int kColsPerQ = BKV + HD + BKV / 2;   // S, O, P (two bf16 per 32-bit column)
  static_assert(NQ * kColsPerQ <= 512, "TMEM budget");
  static constexpr uint32_t kTmemCols = NQ * kColsPerQ <= 256 ? 256 : 512;
};

constexpr int kAttnPoly = 14;   // of every 32 exponentials, this many run on the FMA pipe (even)

template <int HD, int BKV, int NQ>
__global__ void __launch_bounds__(AttnCfg<HD, BKV, NQ>::kThreads, 1)
attention_kernel(const __grid_constant__ AttnMaps maps, const __grid_constant__ AttnArgs p) {
  using Cfg = AttnCfg<HD, BKV, NQ>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t q_smem = base;
  const uint32_t k_smem = q_smem + NQ * Cfg::kQTile;
  const uint32_t v_smem = k_smem + Cfg::kStages * Cfg::kKTile;
  const uint32_t bars = v_smem + Cfg::kStages * Cfg::kVTile;
  // barrier map (8 bytes each)
  const uint32_t q_full = bars;
  auto k_full = [&](int s) { return bars + 8u * (1 + s); };
  auto k_empty = [&](int s) { return bars + 8u * (3 + s); };
  auto v_full = [&](int s) { return bars + 8u * (5 + s); };
  auto v_empty = [&](int s) { return bars + 8u * (7 + s); };
  auto s_full = [&](int q) { return bars + 8u * (9 + q); };
  auto p_full = [&](int q) { return bars + 8u * (12 + q); };
  auto pv_done = [&](int q) { return bars + 8u * (15 + q); };
  const uint32_t tmem_slot = bars + 8u * 18;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp index, provably uniform
  const int bh = blockIdx.y;
  const int q0 = blockIdx.x * (128 * NQ);
  const int nkv = (p.ntok + BKV - 1) / BKV;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&maps.q);
    tma_prefetch_desc(&maps.k);
    tma_prefetch_desc(&maps.vt);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(k_full(s), 1); mbar_init(k_empty(s), 1);
      mbar_init(v_full(s), 1); mbar_init(v_empty(s), 1);
    }
    for (int q = 0; q < NQ; ++q) {
      mbar_init(s_full(q), 1);
      mbar_init(p_full(q), 128);
      mbar_init(pv_done(q), 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, Cfg::kTmemCols);
    tmem_relinquish();
  }
  pdl_launch_dependents();   // programmatic dependent launch: the set-up above overlaps the previous kernel's tail
  pdl_wait();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    if (lane == 0) {
      // ===================== TMA producer =====================
      mbar_arrive_expect_tx(q_full, NQ * Cfg::kQTile);
      for (int q = 0; q < NQ; ++q)
        for (int kb = 0; kb < Cfg::kKBlocks; ++kb)
          tma_load_3d(q_smem + q * Cfg::kQTile + kb * (128 * Cfg::kRowBytes), &maps.q, q_full, kb * 64, q0 + q * 128, bh);
      for (int j = 0; j < nkv; ++j) {
        const int s = j & 1;
        const uint32_t ph = (j >> 1) & 1u;
        mbar_wait(k_empty(s), ph ^ 1u);
        mbar_arrive_expect_tx(k_full(s), Cfg::kKTile);
        for (int kb = 0; kb < Cfg::kKBlocks; ++kb)
          tma_load_3d(k_smem + s * Cfg::kKTile + kb * (BKV * Cfg::kRowBytes), &maps.k, k_full(s), kb * 64, j * BKV, bh);
        mbar_wait(v_empty(s), ph ^ 1u);
        mbar_arrive_expect_tx(v_full(s), Cfg::kVTile);
        for (int vb = 0; vb < BKV / 64; ++vb)
          tma_load_3d(v_smem + s * Cfg::kVTile + vb * (HD * 128), &maps.vt, v_full(s), j * BKV + vb * 64, 0, bh);
      }
    }
  } else if (warp == 1) {
    {
      // ===================== MMA issuer =====================
      // Warp-uniform control flow, one elected lane issues (see igemm.cu): descriptors stay in uniform registers and the
      // UTCHMMA sequences carry no per-instruction ELECT / BRA.U.ANY wrappers.
      const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_ptr, 0);
      const uint32_t idesc_s = umma_idesc_bf16(128, BKV);
      const uint32_t idesc_o = umma_idesc_bf16(128, HD);
      // Descriptors: constant high words, low words advanced with 32-bit adds (the issuing lane's integer work is
      // exposed latency between MMAs).
      const uint64_t dq = umma_smem_desc(q_smem, Cfg::kSwz, 8 * Cfg::kRowBytes);
      const uint64_t dv = umma_smem_desc(v_smem, 128, 1024);
      const uint32_t hi_qk = umma_desc_hi(dq), hi_pv = umma_desc_hi(dv);
      const uint32_t q_lo0 = umma_desc_lo(dq), k_lo0 = q_lo0 + ((k_smem - q_smem) >> 4);
      const uint32_t v_lo0 = umma_desc_lo(dv);
      auto issue_s = [&](int q, int j) {
        const uint32_t d = tmem_base + q * Cfg::kColsPerQ;
        const uint32_t q_lo = q_lo0 + q * (Cfg::kQTile >> 4), k_lo = k_lo0 + (j & 1) * (Cfg::kKTile >> 4);
#pragma unroll
        for (int kb = 0; kb < Cfg::kKBlocks; ++kb) {
#pragma unroll
          for (int k = 0; k < Cfg::kKSteps; ++k)
            umma_bf16(d, umma_desc_join(q_lo + kb * ((128 * Cfg::kRowBytes) >> 4) + 2u * k, hi_qk),
                      umma_desc_join(k_lo + kb * ((BKV * Cfg::kRowBytes) >> 4) + 2u * k, hi_qk), idesc_s, (kb | k) != 0 ? 1u : 0u);
        }
        umma_commit(s_full(q));
      };
      auto issue_pv = [&](int q, int j) {
        const uint32_t d = tmem_base + q * Cfg::kColsPerQ + BKV;
        const uint32_t v_lo = v_lo0 + (j & 1) * (Cfg::kVTile >> 4);
#pragma unroll
        for (int vb = 0; vb < BKV / 64; ++vb) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_ts(d, d + HD + 8u * (vb * 4 + k), umma_desc_join(v_lo + vb * ((HD * 128) >> 4) + 2u * k, hi_pv), idesc_o,
                         (j | vb | k) != 0 ? 1u : 0u);
        }
        umma_commit(pv_done(q));
      };
      mbar_wait(q_full, 0);
      mbar_wait(k_full(0), 0);
      tc_fence_after();
      if (elect_one_sync()) {
        for (int q = 0; q < NQ; ++q) issue_s(q, 0);
        umma_commit(k_empty(0));
      }
      __syncwarp();
      for (int j = 0; j < nkv; ++j) {
        const int s = j & 1;
        const uint32_t ph = (j >> 1) & 1u;
        mbar_wait(v_full(s), ph);
        const bool more = (j + 1 < nkv);
        if (more) mbar_wait(k_full((j + 1) & 1), ((j + 1) >> 1) & 1u);
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
          mbar_wait(p_full(q), j & 1u);
          tc_fence_after();
          if (elect_one_sync()) {
            issue_pv(q, j);
            if (more) issue_s(q, j + 1);
          }
          __syncwarp();
        }
        if (elect_one_sync()) {
          umma_commit(v_empty(s));
          if (more) umma_commit(k_empty((j + 1) & 1));
        }
        __syncwarp();
      }
    }
  } else if (warp >= 4) {
    // ===================== softmax warpgroups =====================
    const int q = (warp - 4) >> 2;
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
    const uint32_t s_tmem = tmem_base + q * Cfg::kColsPerQ + lane_off;
    const uint32_t o_tmem = s_tmem + BKV;
    const float sl2 = p.scale_log2;
    float m = -INFINITY;
    float2 lsum[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
    // One KV tile of the online softmax.  TAIL (compile-time) masks keys >= ntok; only the last tile can need it,
    // so the hot path carries no per-element predicates.  TMEM chunk loads are software-pipelined: the load of
    // chunk c+1 is in flight while chunk c is processed.
    auto tile = [&](int j, auto tail_tag) {
      constexpr bool TAIL = decltype(tail_tag)::value;
      const int kv0 = j * BKV;
      constexpr int NCH = BKV / 32;
      uint32_t ra[32], rb[32];
      // ---- pass 1: tile max
      float tm[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) tm[i] = -INFINITY;   // 8 independent max chains (no serial FMNMX dependency)
      tmem_ld32(s_tmem, ra);
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        tmem_wait_ld();
        uint32_t(&cur)[32] = (c & 1) ? rb : ra;
        if (c + 1 < NCH) tmem_ld32(s_tmem + 32 * (c + 1), (c & 1) ? ra : rb);
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          float a = __uint_as_float(cur[i]), b2 = __uint_as_float(cur[i + 1]);
          if (TAIL) {
            if (kv0 + 32 * c + i >= p.ntok) a = -INFINITY;
            if (kv0 + 32 * c + i + 1 >= p.ntok) b2 = -INFINITY;
          }
          tm[(i >> 1) & 7] = fmaxf(tm[(i >> 1) & 7], fmaxf(a, b2));
        }
      }
      const float tmax = fmaxf(fmaxf(fmaxf(tm[0], tm[1]), fmaxf(tm[2], tm[3])), fmaxf(fmaxf(tm[4], tm[5]), fmaxf(tm[6], tm[7])));
      // start re-reading S for pass 2 while we (possibly) wait for the previous PV and rescale O
      tmem_ld32(s_tmem, ra);
      if (j > 0) mbar_wait(pv_done(q), (j - 1) & 1u);  // O_{j-1} complete, P buffer free
      tc_fence_after();
      if (j == 0) {
        m = tmax;
      } else {
        const bool grow = (tmax - m) * sl2 > 8.0f;
        if (__any_sync(0xffffffffu, grow)) {
          const float m_new = fmaxf(m, tmax);
          const float alpha = ex2_approx((m - m_new) * sl2);
#pragma unroll
          for (int i = 0; i < 2; ++i) { lsum[i].x *= alpha; lsum[i].y *= alpha; }
          m = m_new;
          tmem_wait_ld();  // ra holds chunk 0 of pass 2; keep the TMEM pipe ordered before O traffic
#pragma unroll
          for (int c0 = 0; c0 < HD; c0 += 16) {
            uint32_t r[16];
            tmem_ld16(o_tmem + c0, r);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 16; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * alpha);
            tmem_st16(o_tmem + c0, r);
          }
          tmem_wait_st();
        }
      }
      // ---- pass 2: p = 2^(s*sl2 - m*sl2), row sum, bf16 P into tensor memory behind O
      const float mneg = -m * sl2;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        tmem_wait_ld();
        uint32_t(&cur)[32] = (c & 1) ? rb : ra;
        if (c + 1 < NCH) tmem_ld32(s_tmem + 32 * (c + 1), (c & 1) ? ra : rb);
        float pv[32];
        const float2 sl2v = make_float2(sl2, sl2), mnegv = make_float2(mneg, mneg);
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const float2 xs = ffma2(make_float2(__uint_as_float(cur[i]), __uint_as_float(cur[i + 1])), sl2v, mnegv);
          float2 v;
          if (i < kAttnPoly) {
            v = exp2_poly2(xs);
          } else {
            v.x = ex2_approx(xs.x);
            v.y = ex2_approx(xs.y);
          }
          if (TAIL) {
            if (kv0 + 32 * c + i >= p.ntok) v.x = 0.f;
            if (kv0 + 32 * c + i + 1 >= p.ntok) v.y = 0.f;
          }
          pv[i] = v.x; pv[i + 1] = v.y;
          lsum[(i >> 1) & 1] = fadd2(lsum[(i >> 1) & 1], v);
        }
        uint32_t w[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) w[i] = pack_bf16(pv[2 * i], pv[2 * i + 1]);
        tmem_st16(o_tmem + HD + 16 * c, w);
      }
      tmem_wait_st();
      tc_fence_before();
      mbar_arrive(p_full(q));
    };
    for (int j = 0; j < nkv; ++j) {
      mbar_wait(s_full(q), j & 1u);
      tc_fence_after();
      if (j * BKV + BKV > p.ntok) tile(j, std::true_type{});
      else tile(j, std::false_type{});
    }
    const float l = (lsum[0].x + lsum[0].y) + (lsum[1].x + lsum[1].y);
    // ---- finalize: O / l -> bf16 -> out[b, tok, head*hd + d]
    mbar_wait(pv_done(q), (nkv - 1) & 1u);
    tc_fence_after();
    const int tok = q0 + q * 128 + row;
    const float inv = 1.f / l;
    const int b = bh / p.heads, head = bh % p.heads;
    if (p.lse && tok < p.ntok) p.lse[static_cast<size_t>(bh) * p.ntok + tok] = fmaf(m, sl2, log2f(l));
    __nv_bfloat16* dst = p.out + (static_cast<size_t>(b) * p.ntok + tok) * p.ldo + head * HD;
#pragma unroll
    for (int c0 = 0; c0 < HD; c0 += 16) {
      uint32_t r[16];
      tmem_ld16(o_tmem + c0, r);
      tmem_wait_ld();
      if (tok < p.ntok) {
        uint4 u0, u1;
        u0.x = pack_bf16(__uint_as_float(r[0]) * inv, __uint_as_float(r[1]) * inv);
        u0.y = pack_bf16(__uint_as_float(r[2]) * inv, __uint_as_float(r[3]) * inv);
        u0.z = pack_bf16(__uint_as_float(r[4]) * inv, __uint_as_float(r[5]) * inv);
        u0.w = pack_bf16(__uint_as_float(r[6]) * inv, __uint_as_float(r[7]) * inv);
        u1.x = pack_bf16(__uint_as_float(r[8]) * inv, __uint_as_float(r[9]) * inv);
        u1.y = pack_bf16(__uint_as_float(r[10]) * inv, __uint_as_float(r[11]) * inv);
        u1.z = pack_bf16(__uint_as_float(r[12]) * inv, __uint_as_float(r[13]) * inv);
        u1.w = pack_bf16(__uint_as_float(r[14]) * inv, __uint_as_float(r[15]) * inv);
        *reinterpret_cast<uint4*>(dst + c0) = u0;
        *reinterpret_cast<uint4*>(dst + c0 + 8) = u1;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <int HD, int BKV, int NQ>
int launch_attention(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, __nv_bfloat16* out, int B,
                     int heads, int ntok, int ldo, cudaStream_t st, float* lse, float scale) {
  using Cfg = AttnCfg<HD, BKV, NQ>;
  const int BH = B * heads;
  AttnMaps maps;
  if (int e = encode_attn_maps(&maps, q, k, vt, BH, ntok, HD, BKV)) return e;
  AttnArgs args;
  args.ntok = ntok; args.heads = heads; args.ldo = ldo; args.out = out; args.lse = lse;
  args.scale_log2 = attn_scale_log2(scale, HD);
  static bool attr_set = false;
  if (!attr_set) {
    WC_CHECK_CUDA(cudaFuncSetAttribute(attention_kernel<HD, BKV, NQ>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       Cfg::kSmem));
    attr_set = true;
  }
  dim3 grid((ntok + 128 * NQ - 1) / (128 * NQ), BH);
  ProfScope prof(kProfAttention, st, 4.0 * BH * static_cast<double>(ntok) * ntok * HD);
  prof.note(BH, ntok, HD);
  launch_k<1>(attention_kernel<HD, BKV, NQ>, grid, Cfg::kThreads, Cfg::kSmem, st, maps, args);
  WC_LAUNCH_CHECK();
  return 0;
}

}  // namespace

int attention_small_forward(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, __nv_bfloat16* out, int B,
                            int heads, int ntok, int hd, int ldo, cudaStream_t st, float* lse, float scale);

int encode_attn_maps(AttnMaps* maps, const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, int BH, int ntok,
                     int hd, int bkv) {
  const uint32_t inner = hd >= 64 ? 64 : hd;
  {
    uint64_t dims[3] = {static_cast<uint64_t>(hd), static_cast<uint64_t>(ntok), static_cast<uint64_t>(BH)};
    uint64_t strides[3] = {1, static_cast<uint64_t>(hd), static_cast<uint64_t>(hd) * ntok};
    uint32_t boxq[3] = {inner, 128, 1};
    uint32_t boxk[3] = {inner, static_cast<uint32_t>(bkv), 1};
    if (int e = encode_tmap_bf16(&maps->q, q, 3, dims, strides, boxq, 2 * inner)) return e;
    if (int e = encode_tmap_bf16(&maps->k, k, 3, dims, strides, boxk, 2 * inner)) return e;
  }
  uint64_t dims[3] = {static_cast<uint64_t>(ntok), static_cast<uint64_t>(hd), static_cast<uint64_t>(BH)};
  uint64_t strides[3] = {1, static_cast<uint64_t>(ntok), static_cast<uint64_t>(hd) * ntok};
  uint32_t box[3] = {64, static_cast<uint32_t>(hd), 1};
  return encode_tmap_bf16(&maps->vt, vt, 3, dims, strides, box, 128);
}

// q,k [B,heads,ntok,hd]; vt [B,heads,hd,ntok]; out [B,ntok,ldo] (columns head*hd .. head*hd+hd).
int attention_forward(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, __nv_bfloat16* out, int B,
                      int heads, int ntok, int hd, int ldo, cudaStream_t st, float* lse, float scale) {
  WC_REQUIRE(ntok % 8 == 0, "token count must be a multiple of 8");
  WC_REQUIRE(ldo % 8 == 0, "output row stride must be a multiple of 8");
  if (hd == 16 || hd == 32) return attention_small_forward(q, k, vt, out, B, heads, ntok, hd, ldo, st, lse, scale);
  switch (hd) {
    case 64: return launch_attention<64, 128, 2>(q, k, vt, out, B, heads, ntok, ldo, st, lse, scale);
    case 128: return launch_attention<128, 64, 2>(q, k, vt, out, B, heads, ntok, ldo, st, lse, scale);
    case 192: return launch_attention<192, 64, 1>(q, k, vt, out, B, heads, ntok, ldo, st, lse, scale);
    default: return fail("attention: unsupported head_dim " + std::to_string(hd) + " (supported: 16,32,64,128,192)");
  }
}

double attention_flops(int B, int heads, int ntok, int hd) { return 4.0 * B * heads * static_cast<double>(ntok) * ntok * hd; }

}  // namespace wc
