// Flash attention for SMALL head dims (16, 32) on tcgen05 (sm_100a): the layers of nn.MultiheadAttention at
// unet_base.py:115,159,320,365 whose head_dim is 16 / 32 at N = 8192 tokens are bound by the N^2 exponentials, not by
// the tensor core (the general kernel in attention.cu ran at 52 % FMA-pipe / 44 % MUFU / 62 % issue utilisation there,
// profiles/r1_ncu_attention_hd16_v3.txt).  This kernel removes per-element CUDA-core work by moving it onto the idle
// tensor core:
//   * scale and max subtraction:  log2(e)/sqrt(hd) = 2^k * c with c in [1, 2).  The Q tile is multiplied by 2^k once in
//     shared memory (exact in bf16), and every S MMA gets one extra K = 16 step  S += Qx Kx^T  with Qx[row] = (-E_row, 0, ...)
//     and Kx[key] = (1, 0, ...), so the accumulator already holds  S'' = 2^k q.k - E  with E = (stale row maximum) + 8/c,
//     bf16-rounded (softmax is shift invariant; the same offset is used for P and for the row sum).  P' = 2^(c S''): on the
//     polynomial lanes c rides along in the two FMAs of the range reduction at no cost, the MUFU lanes pay one packed
//     multiply per pair (instead of an FFMA per element and a maximum pass);
//   * no per-tile maximum pass:  P' = 2^(S') is at most 2^-8 while the stale maximum holds; a tile in which any P' >= 2
//     (bit 14 of the packed bf16 words, found with one LOP3 per four elements) or any garbage (sign bit) shows up is
//     recomputed on a slow path that finds the true tile maximum, rescales O and updates Qx.  The first tile and a ragged
//     last tile always take the slow path;
//   * row sums (head_dim 16):  V^T gets a constant row of ones (rows hd..hd+15 of the B operand), so column hd of the
//     O accumulator is l = sum_j P'_j (of the bf16-rounded P' that the PV product really uses); no FADD per element.
//     head_dim 32 has no TMEM columns left for that at three query tiles per CTA and keeps packed fp32 row sums (which also
//     serve as the overflow detector).
//   * head_dim 32: P' in tensor memory too (TP): the tile is read into registers, P' is written over the first 32 columns of the
//     S buffer it came from (tcgen05.st, two bf16 per column) and the PV MMA takes its A operand from there; a tile that needs
//     the slow path is redone from the registers.
//   * S double-buffered in tensor memory (KV tiles of 64 keys: 3 x (2 x 64 + 32) = 480 columns): S(q, j+2) is issued as soon
//     as the softmax group has consumed S(q, j), so the exponentials never wait for the QK^T / PV round trip (in the general
//     kernel the softmax warps spent 36 % of their time waiting for s_full).  A tile that moves the offset leaves the
//     already computed next S tile on the old offset; that tile is corrected in registers on the slow path (`carry`).
// Roles are those of attention.cu: warp 0 TMA, warp 1 MMA issue, warp 2 TMEM alloc, 3 softmax warpgroups (one thread per
// query row), P (double-buffered) through shared memory in the swizzled K-major layout.
#include "wc_host.h"
#include "wc_ptx.cuh"

#include <type_traits>

namespace wc {

namespace {

struct SmallArgs {
  int ntok, heads, ldo;
  float qscale;      // 2^k:  log2(e) * softmax scale = qscale * c
  float c;           // in [1, 2)
  __nv_bfloat16* out;
  float* lse;
};

struct SmallMaps {
  CUtensorMap q, k, vt;
};

constexpr int kBKV = 64;          // keys per tile: S (128 x 64 fp32) is DOUBLE-BUFFERED in tensor memory
constexpr int kNQ = 3;            // query tiles (softmax warpgroups) per CTA
constexpr int kKStages = 4;       // K / V^T TMA ring depth
constexpr float kShift = 8.0f;    // P' = P * 2^-8: the "needs a new maximum" test becomes "exponent bit 7 set"
constexpr float kLazy = 6.0f;

template <int HD, bool TP = false>
struct SmallCfg {
  static constexpr bool kLT = (HD == 16);                       // row sums on the tensor core
  static constexpr int kRowBytes = HD * 2;                      // Q / K rows (one swizzle span)
  static constexpr int kSwz = HD * 2;
  static constexpr int kKSteps = HD / 16;
  static constexpr int kVRows = HD + (kLT ? 16 : 0);            // N of the PV product
  static constexpr uint32_t kQTile = 128 * HD * 2;
  static constexpr uint32_t kXTile = 128 * 32;                  // augmented K = 16 step of Q, 32-byte rows
  static constexpr uint32_t kKxTile = kBKV * 32;                // ... and of K (constant)
  static constexpr uint32_t kKTile = kBKV * HD * 2;
  static constexpr uint32_t kVBlock = kVRows * 128;             // 64 keys x kVRows
  static constexpr uint32_t kVLoad = HD * 128;                  // bytes the TMA writes per stage
  static constexpr uint32_t kPTile = 128 * kBKV * 2;
  // TP: P lives in TENSOR MEMORY, written over the first 32 columns of the S buffer it was computed from (two bf16 per column)
  static constexpr uint32_t kSmem = kNQ * kQTile + kNQ * kXTile + kKxTile + kKStages * (kKTile + kVBlock) + (TP ? 0u : 2 * kNQ * kPTile) + 1024 + 512;
  static constexpr int kThreads = 128 + 128 * kNQ;
  static constexpr int kColsPerQ = 2 * kBKV + kVRows;           // S0 | S1 | O (+ l)
  static_assert(kNQ * kColsPerQ <= 512, "TMEM budget");
  static constexpr uint32_t kTmemCols = 512;
};

__device__ __forceinline__ void lds128(uint32_t addr, uint32_t (&v)[4]) {
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(addr) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void sts16(uint32_t addr, uint16_t v) {
  asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(v) : "memory");
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
__device__ __forceinline__ uint16_t bf16_bits(float x) {
  __nv_bfloat16 h = __float2bfloat16_rn(x);
  return *reinterpret_cast<uint16_t*>(&h);
}

// 2^x for a pair on the FMA / ALU pipes (see exp2_poly2 in wc_ptx.cuh); here the exponent is patched with a shift-add
// (LEA, ALU pipe) instead of an integer multiply-add (FMA pipe), the FMA pipe being the busier one.
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
  unsigned long long ua = *reinterpret_cast<unsigned long long*>(&a), ub = *reinterpret_cast<unsigned long long*>(&b), ud;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(ud) : "l"(ua), "l"(ub));
  return *reinterpret_cast<float2*>(&ud);
}
// 2^(c*x), c in [1, 2): x is clamped at lo = -125/c; n = round(c*x) and f = c*x - n come out of two FMAs.
// Large positive arguments (a row maximum that outgrew the stale one) wrap the exponent field: for c*x < 511.5 the result is
// >= 4, negative or NaN and the caller's "any P' >= 2 / sign bit" test sends the tile to the slow path.  Stated domain limit:
// a logit that exceeds the row's stale maximum by more than 2^511 (354 in natural-log units of the scaled logits - out of
// reach for bf16 q, k of any normalised network) on a polynomial lane would alias to a plausible value undetected.
__device__ __forceinline__ float2 exp2_poly2_scaled(float2 x, float2 c, float lo) {
  const float kMagic = 12582912.f;
  x.x = fmaxf(x.x, lo);
  x.y = fmaxf(x.y, lo);
  const float2 r = ffma2(x, c, make_float2(kMagic, kMagic));
  const float2 nn = ffma2(r, make_float2(-1.f, -1.f), make_float2(kMagic, kMagic));   // -(n), exact
  const float2 f = ffma2(x, c, nn);
  float2 p = ffma2(f, make_float2(0.05517163872718811f, 0.05517163872718811f), make_float2(0.2426111251115799f, 0.2426111251115799f));
  p = ffma2(p, f, make_float2(0.6932609677314758f, 0.6932609677314758f));
  p = ffma2(p, f, make_float2(0.9999280571937561f, 0.9999280571937561f));
  float2 o;
  o.x = __uint_as_float((__float_as_uint(r.x) << 23) + __float_as_uint(p.x));
  o.y = __uint_as_float((__float_as_uint(r.y) << 23) + __float_as_uint(p.y));
  return o;
}

template <int HD, int POLY, bool TP>
__global__ void __launch_bounds__(SmallCfg<HD, TP>::kThreads, 1)
attention_small_kernel(const __grid_constant__ SmallMaps maps, const __grid_constant__ SmallArgs p) {
  using Cfg = SmallCfg<HD, TP>;
  constexpr bool LT = Cfg::kLT;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t q_smem = base;
  const uint32_t qx_smem = q_smem + kNQ * Cfg::kQTile;
  const uint32_t kx_smem = qx_smem + kNQ * Cfg::kXTile;
  const uint32_t k_smem = kx_smem + Cfg::kKxTile;
  const uint32_t v_smem = k_smem + kKStages * Cfg::kKTile;
  const uint32_t p_smem = v_smem + kKStages * Cfg::kVBlock;
  const uint32_t bars = p_smem + (TP ? 0u : 2 * kNQ * Cfg::kPTile);
  const uint32_t q_full = bars;
  auto k_full = [&](int s) { return bars + 8u * (1 + s); };
  auto k_empty = [&](int s) { return bars + 8u * (5 + s); };
  auto v_full = [&](int s) { return bars + 8u * (9 + s); };
  auto v_empty = [&](int s) { return bars + 8u * (13 + s); };
  auto s_full = [&](int q, int b) { return bars + 8u * (17 + 2 * q + b); };
  auto p_full = [&](int q, int b) { return bars + 8u * (23 + 2 * q + b); };
  auto pv_done = [&](int q, int b) { return bars + 8u * (29 + 2 * q + b); };
  auto q_ready = [&](int q) { return bars + 8u * (35 + q); };
  const uint32_t tmem_slot = bars + 8u * 38;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp index, provably uniform
  // head_dim 16: grid = (batch*heads, query blocks), i.e. CTAs are dispatched head-fastest and the short last query block of
  // every head (see nq_valid) fills the tail of the last wave (+2 %).  head_dim 32 keeps query-block-fastest order: K and V of
  // 128 heads (128 MB at N = 8192) would not stay in L2 otherwise (-4 %).
  const int bh = HD == 16 ? blockIdx.x : blockIdx.y;
  const int q0 = (HD == 16 ? blockIdx.y : blockIdx.x) * (128 * kNQ);
  const int nkv = (p.ntok + kBKV - 1) / kBKV;
  // query tiles of this CTA that hold at least one token (8192 = 21 x 384 + 128: the last CTA of every (batch, head) has one);
  // the other softmax groups and their MMAs are skipped, such a CTA finishes in well under half the time
  const int nq_valid = min(kNQ, (p.ntok - q0 + 127) / 128);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&maps.q);
    tma_prefetch_desc(&maps.k);
    tma_prefetch_desc(&maps.vt);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < kKStages; ++s) {
      mbar_init(k_full(s), 1); mbar_init(k_empty(s), 1);
      mbar_init(v_full(s), 1); mbar_init(v_empty(s), 1);
    }
    for (int q = 0; q < kNQ; ++q) {
      for (int b = 0; b < 2; ++b) {
        mbar_init(s_full(q, b), 1);
        mbar_init(p_full(q, b), 128);
        mbar_init(pv_done(q, b), 1);
      }
      mbar_init(q_ready(q), 128);
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
      mbar_arrive_expect_tx(q_full, kNQ * Cfg::kQTile);
      for (int q = 0; q < kNQ; ++q) tma_load_3d(q_smem + q * Cfg::kQTile, &maps.q, q_full, 0, q0 + q * 128, bh);
      for (int j = 0; j < nkv; ++j) {
        const int s = j % kKStages;
        const uint32_t ph = (j / kKStages) & 1u;
        mbar_wait(k_empty(s), ph ^ 1u);
        mbar_arrive_expect_tx(k_full(s), Cfg::kKTile);
        tma_load_3d(k_smem + s * Cfg::kKTile, &maps.k, k_full(s), 0, j * kBKV, bh);
        mbar_wait(v_empty(s), ph ^ 1u);
        mbar_arrive_expect_tx(v_full(s), Cfg::kVLoad);
        tma_load_3d(v_smem + s * Cfg::kVBlock, &maps.vt, v_full(s), j * kBKV, 0, bh);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // The whole warp runs this loop in uniform control flow and one elected lane issues: the compiler then keeps descriptors
    // and counters in uniform registers and emits bare UTCHMMA sequences.  (Issuing from inside `if (lane == 0)` costs ~13
    // SASS instructions per MMA - R2UR moves plus an ELECT / BRA.U.ANY loop around every UTCHMMA - and a single thread
    // executing ~29 instructions per MMA was the limiter of this kernel: 127 clk per MMA.)
    // S(q, j+2) is issued as soon as the softmax group has consumed S(q, j) (p_full(q, j)), i.e. two tiles ahead of the
    // exponentials: the softmax warps do not wait for the tensor core in steady state.
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t idesc_s = umma_idesc_bf16(128, kBKV);
    const uint32_t idesc_o = umma_idesc_bf16(128, Cfg::kVRows);
    const uint64_t dq = umma_smem_desc(q_smem, Cfg::kSwz, 8 * Cfg::kRowBytes);
    const uint64_t dx = umma_smem_desc(qx_smem, 32, 256);
    const uint64_t dp = umma_smem_desc(p_smem, 128, 1024);
    const uint32_t hi_qk = umma_desc_hi(dq), hi_x = umma_desc_hi(dx), hi_pv = umma_desc_hi(dp);
    const uint32_t q_lo0 = umma_desc_lo(dq), k_lo0 = q_lo0 + ((k_smem - q_smem) >> 4);
    const uint32_t qx_lo0 = umma_desc_lo(dx), kx_lo = qx_lo0 + ((kx_smem - qx_smem) >> 4);
    const uint32_t p_lo0 = umma_desc_lo(dp), v_lo0 = p_lo0 - ((p_smem - v_smem) >> 4);
    auto issue_s = [&](int q, int j) {
      const uint32_t d = tmem_u + q * Cfg::kColsPerQ + (j & 1) * kBKV;
      const uint32_t q_lo = q_lo0 + q * (Cfg::kQTile >> 4), k_lo = k_lo0 + (j % kKStages) * (Cfg::kKTile >> 4);
#pragma unroll
      for (int k = 0; k < Cfg::kKSteps; ++k)
        umma_bf16(d, umma_desc_join(q_lo + 2u * k, hi_qk), umma_desc_join(k_lo + 2u * k, hi_qk), idesc_s, k != 0 ? 1u : 0u);
      // S += Qx Kx^T: subtracts the row's offset E inside the accumulator
      umma_bf16(d, umma_desc_join(qx_lo0 + q * (Cfg::kXTile >> 4), hi_x), umma_desc_join(kx_lo, hi_x), idesc_s, 1u);
      umma_commit(s_full(q, j & 1));
    };
    auto issue_pv = [&](int q, int j) {
      const uint32_t d = tmem_u + q * Cfg::kColsPerQ + 2 * kBKV;
      const uint32_t p_lo = p_lo0 + (2 * q + (j & 1)) * (Cfg::kPTile >> 4), v_lo = v_lo0 + (j % kKStages) * (Cfg::kVBlock >> 4);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (TP)   // A = P from tensor memory: 8 columns (16 keys) per K step, in the S buffer the tile came from
          umma_bf16_ts(d, tmem_u + q * Cfg::kColsPerQ + (j & 1) * kBKV + 8u * k, umma_desc_join(v_lo + 2u * k, hi_pv), idesc_o,
                       (j | k) != 0 ? 1u : 0u);
        else
          umma_bf16(d, umma_desc_join(p_lo + 2u * k, hi_pv), umma_desc_join(v_lo + 2u * k, hi_pv), idesc_o, (j | k) != 0 ? 1u : 0u);
      }
      umma_commit(pv_done(q, j & 1));
    };
    const int npro = nkv < 2 ? nkv : 2;
    for (int j = 0; j < npro; ++j) mbar_wait(k_full(j), 0);
#pragma unroll
    for (int q = 0; q < kNQ; ++q) {
      mbar_wait(q_ready(q), 0);   // every group (also one without tokens) has written its share of the constant rows
      tc_fence_after();
      if (q < nq_valid) {
        if (elect_one_sync()) {
          for (int j = 0; j < npro; ++j) issue_s(q, j);
        }
        __syncwarp();
      }
    }
    if (elect_one_sync()) {
      for (int j = 0; j < npro; ++j) umma_commit(k_empty(j));
    }
    __syncwarp();
    for (int j = 0; j < nkv; ++j) {
      const int s = j % kKStages;
      mbar_wait(v_full(s), (j / kKStages) & 1u);
      const bool more = (j + 2 < nkv);
      if (more) mbar_wait(k_full((j + 2) % kKStages), ((j + 2) / kKStages) & 1u);
#pragma unroll
      for (int q = 0; q < kNQ; ++q) {
        if (q < nq_valid) {
          mbar_wait(p_full(q, j & 1), (j >> 1) & 1u);
          tc_fence_after();
          if (elect_one_sync()) {
            issue_pv(q, j);
            if (more) issue_s(q, j + 2);
          }
          __syncwarp();
        }
      }
      if (elect_one_sync()) {
        umma_commit(v_empty(s));
        if (more) umma_commit(k_empty((j + 2) % kKStages));
      }
      __syncwarp();
    }
  } else if (warp >= 4) {
    // ===================== softmax warpgroups =====================
    const int q = (warp - 4) >> 2;
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
    const uint32_t s_tmem = tmem_base + q * Cfg::kColsPerQ + lane_off;
    const uint32_t o_tmem = s_tmem + 2 * kBKV;
    const uint32_t p_row = p_smem + 2 * q * Cfg::kPTile + row * 128;
    const uint32_t qx_row = qx_smem + q * Cfg::kXTile + row * 32;

    const float cs = p.c;
    const float shift = kShift / cs;       // in units of S''
    float E = bf16_round(shift);           // current offset (bf16-representable): S'' = 2^k q.k - E
    // ---- one-time set-up of the constant operands (generic-proxy stores, made visible to the MMA by the fence below)
    {
      const int t = threadIdx.x - 128;  // 0 .. 383
      if (q == 0 && row < kBKV) {
        // Kx: 1.0 in the first element of BOTH 16-byte chunks of every key row; Qx carries its value in the first physical
        // chunk only, so the product is (-E)*1 whichever way the 32-byte swizzle maps the chunks.
        sts128(kx_smem + row * 32, 0x00003F80u, 0u, 0u, 0u);
        sts128(kx_smem + row * 32 + 16, 0x00003F80u, 0u, 0u, 0u);
      }
      if (LT) {
        // rows hd .. hd+15 of every V^T stage: one row of ones (-> column hd of O accumulates the row sums), then zeros
        constexpr int kChunks = kKStages * 16 * 8;  // 16-byte chunks to write
        for (int c = t; c < kChunks; c += 128 * kNQ) {
          const int blk = c >> 7, r = (c >> 3) & 15, ch = c & 7;
          const uint32_t one = r == 0 ? 0x3F803F80u : 0u;
          sts128(v_smem + blk * Cfg::kVBlock + (HD + r) * 128 + ch * 16, one, one, one, one);
        }
      }
      mbar_wait(q_full, 0);
      // Q row *= 2^k (exact; element-wise, so the swizzled chunk order inside the row does not matter)
      const uint32_t q_row = q_smem + q * Cfg::kQTile + row * Cfg::kRowBytes;
      const float qs = p.qscale;
#pragma unroll
      for (int c = 0; c < Cfg::kRowBytes / 16; ++c) {
        uint32_t v[4];
        lds128(q_row + 16 * c, v);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 f = unpack_bf16(v[i]);
          v[i] = pack_bf16(f.x * qs, f.y * qs);
        }
        sts128(q_row + 16 * c, v[0], v[1], v[2], v[3]);
      }
      sts128(qx_row, static_cast<uint32_t>(bf16_bits(-E)), 0u, 0u, 0u);
      sts128(qx_row + 16, 0u, 0u, 0u, 0u);
      fence_proxy_async_smem();
      // the MMA warp waits for q_ready(0..2) before the first S: group 0 wrote Kx, every group its share of the ones rows
      mbar_arrive(q_ready(q));
    }

    float2 lsum[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};   // !LT only
    // S(q, j+1) was issued BEFORE tile j was processed: if tile j moved the offset by `delta`, tile j+1 still carries the
    // old one and is corrected in registers (slow path) by `carry`.
    float carry = 0.f;

    // ---- slow path: true tile maximum, offset update, O rescale, masked tail
    auto slow_tile = [&](int j, auto tail_tag) {
      constexpr bool TAIL = decltype(tail_tag)::value;
      const int kv0 = j * kBKV;
      const int b = j & 1;
      constexpr int NCH = kBKV / 32;
      uint32_t ra[32];
      float tmax = -INFINITY;
#pragma unroll 1
      for (int c = 0; c < NCH; ++c) {
        tmem_ld32(s_tmem + b * kBKV + 32 * c, ra);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float a = __uint_as_float(ra[i]);
          if (TAIL && kv0 + 32 * c + i >= p.ntok) a = -INFINITY;
          tmax = fmaxf(tmax, a);
        }
      }
      tmax -= carry;                       // relative to the CURRENT offset E
      float delta = 0.f;                   // offset change, in units of S''
      // lazy: a row moves its offset only when its maximum has grown by more than 2^kLazy over the stale one (P' stays below
      // 2^(kLazy-8) < 2 otherwise); every update forces the next tile onto this path too (carry), so they must stay rare
      const bool upd = (j == 0) || (tmax > -shift + kLazy / cs);
      if (upd) {
        // S(q, j+1) was issued before this tile and reads Qx: it must have completed before Qx changes
        if (j + 1 < nkv) mbar_wait(s_full(q, b ^ 1), ((j + 1) >> 1) & 1u);
        const float e_new = bf16_round(E + tmax + shift);
        delta = e_new - E;
        E = e_new;
        sts16(qx_row, bf16_bits(-e_new));
      }
      if (j > 0 && __any_sync(0xffffffffu, upd)) {
        mbar_wait(pv_done(q, (j - 1) & 1), ((j - 1) >> 1) & 1u);   // every PV issued so far has completed
        tc_fence_after();
        const float alpha = ex2_approx(-delta * cs);
        if (!LT) {
#pragma unroll
          for (int i = 0; i < 2; ++i) { lsum[i].x *= alpha; lsum[i].y *= alpha; }
        }
#pragma unroll
        for (int c0 = 0; c0 < Cfg::kVRows; c0 += 16) {
          uint32_t r[16];
          tmem_ld16(o_tmem + c0, r);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 16; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * alpha);
          tmem_st16(o_tmem + c0, r);
        }
        tmem_wait_st();
      }
      const float dneg = -(carry + delta) * cs;
      carry = delta;
#pragma unroll 1
      for (int c = 0; c < NCH; ++c) {
        tmem_ld32(s_tmem + b * kBKV + 32 * c, ra);
        tmem_wait_ld();
        float pv[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float v = ex2_approx(fmaf(__uint_as_float(ra[i]), cs, dneg));
          if (TAIL && kv0 + 32 * c + i >= p.ntok) v = 0.f;
          pv[i] = v;
          if (!LT) {
            if (i & 1) lsum[(i >> 1) & 1].y += v; else lsum[(i >> 1) & 1].x += v;
          }
        }
        const uint32_t blk = p_row + b * Cfg::kPTile;
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const int chunk = 4 * c + ch;
          sts128(blk + (static_cast<uint32_t>(chunk ^ (row & 7)) << 4), pack_bf16(pv[8 * ch + 0], pv[8 * ch + 1]),
                 pack_bf16(pv[8 * ch + 2], pv[8 * ch + 3]), pack_bf16(pv[8 * ch + 4], pv[8 * ch + 5]),
                 pack_bf16(pv[8 * ch + 6], pv[8 * ch + 7]));
        }
      }
    };

    // ---- hot path: exponentiate the raw accumulator; returns true (warp-uniform) if the tile has to be redone on the slow path
    auto hot_tile = [&](int b) -> bool {
      constexpr int NCH = kBKV / 32;
      uint32_t ra[32], rb[32];
      uint32_t orw = 0u;
      float2 ts[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
      const float2 cv = make_float2(cs, cs);
      const float lo = -125.f / cs;
      tmem_ld32(s_tmem + b * kBKV, ra);
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        tmem_wait_ld();
        uint32_t(&cur)[32] = (c & 1) ? rb : ra;
        if (c + 1 < NCH) tmem_ld32(s_tmem + b * kBKV + 32 * (c + 1), (c & 1) ? ra : rb);
        uint32_t w[16];
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const float2 xs = make_float2(__uint_as_float(cur[i]), __uint_as_float(cur[i + 1]));
          float2 v;
          if (i < POLY) {
            v = exp2_poly2_scaled(xs, cv, lo);
          } else {
            const float2 y = fmul2(xs, cv);
            v.x = ex2_approx(y.x);
            v.y = ex2_approx(y.y);
          }
          if (!LT) ts[(i >> 1) & 1] = fadd2(ts[(i >> 1) & 1], v);
          w[i >> 1] = pack_bf16(v.x, v.y);
        }
        if (LT) {
#pragma unroll
          for (int i = 0; i < 16; i += 2) orw |= w[i] | w[i + 1];
        }
        const uint32_t blk = p_row + b * Cfg::kPTile;
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const int chunk = 4 * c + ch;
          sts128(blk + (static_cast<uint32_t>(chunk ^ (row & 7)) << 4), w[4 * ch], w[4 * ch + 1], w[4 * ch + 2], w[4 * ch + 3]);
        }
      }
      bool redo;
      if (LT) {
        redo = (orw & 0xC000C000u) != 0u;          // some P' >= 2 (or negative / NaN garbage)
      } else {
        const float tsum = (ts[0].x + ts[0].y) + (ts[1].x + ts[1].y);
        redo = !(tsum < 32.f);                     // all P' <= 2^-8 gives tsum <= 0.25; also catches inf / NaN
      }
      redo = __any_sync(0xffffffffu, redo);
      if (!LT && !redo) { lsum[0] = fadd2(lsum[0], ts[0]); lsum[1] = fadd2(lsum[1], ts[1]); }
      return redo;
    };

    // ---- TP: the whole S tile is read into registers first, P' is written back over its first 32 columns (tcgen05.st) and
    // the PV MMA reads it from there: no shared-memory stores, no fence.proxy.async, no A-operand fetch from shared memory.
    // A tile that has to take the slow path is redone from the registers.
    auto tp_tile = [&](int j, bool force_slow, auto tail_tag) {
      constexpr bool TAIL = decltype(tail_tag)::value;
      const int kv0 = j * kBKV;
      const int b = j & 1;
      // P' is stored 16 words at a time as soon as it is computed (the stores are idempotent: a slow-path redo simply writes the
      // columns again before the PV MMA is released), so only the raw tile (64 registers) and 16 packed words are live at once
      uint32_t ra[32], rb[32], w[16];
      const uint32_t p_tmem = s_tmem + b * kBKV;
      tmem_ld32(s_tmem + b * kBKV, ra);
      tmem_ld32(s_tmem + b * kBKV + 32, rb);
      tmem_wait_ld();
      bool slow = force_slow;
      if (!slow) {
        uint32_t orw = 0u;
        float2 ts[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
        const float2 cv = make_float2(cs, cs);
        const float lo = -125.f / cs;
        auto half = [&](const uint32_t (&cur)[32], uint32_t (&w)[16]) {
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const float2 xs = make_float2(__uint_as_float(cur[i]), __uint_as_float(cur[i + 1]));
            float2 v;
            if (i < POLY) {
              v = exp2_poly2_scaled(xs, cv, lo);
            } else {
              const float2 y = fmul2(xs, cv);
              v.x = ex2_approx(y.x);
              v.y = ex2_approx(y.y);
            }
            if (!LT) ts[(i >> 1) & 1] = fadd2(ts[(i >> 1) & 1], v);
            w[i >> 1] = pack_bf16(v.x, v.y);
          }
          if (LT) {
#pragma unroll
            for (int i = 0; i < 16; i += 2) orw |= w[i] | w[i + 1];
          }
        };
        half(ra, w);
        tmem_st16(p_tmem, w);
        half(rb, w);
        tmem_st16(p_tmem + 16, w);
        bool redo;
        if (LT) {
          redo = (orw & 0xC000C000u) != 0u;
        } else {
          const float tsum = (ts[0].x + ts[0].y) + (ts[1].x + ts[1].y);
          redo = !(tsum < 32.f);
        }
        slow = __any_sync(0xffffffffu, redo);
        if (!LT && !slow) { lsum[0] = fadd2(lsum[0], ts[0]); lsum[1] = fadd2(lsum[1], ts[1]); }
      }
      if (slow) {
        float tmax = -INFINITY;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float a0 = __uint_as_float(ra[i]), a1 = __uint_as_float(rb[i]);
          if (TAIL && kv0 + i >= p.ntok) a0 = -INFINITY;
          if (TAIL && kv0 + 32 + i >= p.ntok) a1 = -INFINITY;
          tmax = fmaxf(tmax, fmaxf(a0, a1));
        }
        tmax -= carry;
        float delta = 0.f;
        const bool upd = (j == 0) || (tmax > -shift + kLazy / cs);
        if (upd) {
          if (j + 1 < nkv) mbar_wait(s_full(q, b ^ 1), ((j + 1) >> 1) & 1u);
          const float e_new = bf16_round(E + tmax + shift);
          delta = e_new - E;
          E = e_new;
          sts16(qx_row, bf16_bits(-e_new));
        }
        if (j > 0 && __any_sync(0xffffffffu, upd)) {
          mbar_wait(pv_done(q, (j - 1) & 1), ((j - 1) >> 1) & 1u);
          tc_fence_after();
          const float alpha = ex2_approx(-delta * cs);
          if (!LT) {
#pragma unroll
            for (int i = 0; i < 2; ++i) { lsum[i].x *= alpha; lsum[i].y *= alpha; }
          }
#pragma unroll
          for (int c0 = 0; c0 < Cfg::kVRows; c0 += 16) {
            uint32_t r[16];
            tmem_ld16(o_tmem + c0, r);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 16; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * alpha);
            tmem_st16(o_tmem + c0, r);
          }
          tmem_wait_st();
        }
        const float dneg = -(carry + delta) * cs;
        carry = delta;
        auto redo_half = [&](const uint32_t (&cur)[32], int k0, float2& acc) {
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            float v0 = ex2_approx(fmaf(__uint_as_float(cur[i]), cs, dneg)), v1 = ex2_approx(fmaf(__uint_as_float(cur[i + 1]), cs, dneg));
            if (TAIL) {
              if (k0 + i >= p.ntok) v0 = 0.f;
              if (k0 + i + 1 >= p.ntok) v1 = 0.f;
            }
            if (!LT) { acc.x += v0; acc.y += v1; }
            w[i >> 1] = pack_bf16(v0, v1);
          }
        };
        tmem_wait_st();
        redo_half(ra, kv0, lsum[0]);
        tmem_st16(p_tmem, w);
        redo_half(rb, kv0 + 32, lsum[1]);
        tmem_st16(p_tmem + 16, w);
        fence_proxy_async_smem();   // Qx may have changed (generic-proxy store read by the next S MMA)
      }
      tmem_wait_st();
    };

    for (int j = 0; j < (q < nq_valid ? nkv : 0); ++j) {
      const int b = j & 1;
      mbar_wait(s_full(q, b), (j >> 1) & 1u);
      if (j >= 2) mbar_wait(pv_done(q, b), ((j - 2) >> 1) & 1u);   // P buffer b free (PV of tile j-2 has read it)
      tc_fence_after();
      const bool tail = (j * kBKV + kBKV > p.ntok);
      if (TP) {
        if (tail) tp_tile(j, true, std::true_type{});
        else tp_tile(j, j == 0 || __any_sync(0xffffffffu, carry != 0.f), std::false_type{});
      } else {
        if (tail) {
          slow_tile(j, std::true_type{});
        } else if (j == 0 || __any_sync(0xffffffffu, carry != 0.f) || hot_tile(b)) {
          slow_tile(j, std::false_type{});
        }
        fence_proxy_async_smem();
      }
      tc_fence_before();
      mbar_arrive(p_full(q, b));
    }

    // ---- finalize: O / l -> bf16 -> out[b, tok, head*hd + d]
    if (q < nq_valid) mbar_wait(pv_done(q, (nkv - 1) & 1), ((nkv - 1) >> 1) & 1u);
    tc_fence_after();
    const int tok = q0 + q * 128 + row;
    const int b = bh / p.heads, head = bh % p.heads;
    __nv_bfloat16* dst = p.out + (static_cast<size_t>(b) * p.ntok + tok) * p.ldo + head * HD;
    uint32_t r[Cfg::kVRows];
#pragma unroll
    for (int c0 = 0; c0 < Cfg::kVRows; c0 += 16) {
      uint32_t t16[16];
      tmem_ld16(o_tmem + c0, t16);
      tmem_wait_ld();
#pragma unroll
      for (int i = 0; i < 16; ++i) r[c0 + i] = t16[i];
    }
    const float l = LT ? __uint_as_float(r[HD]) : (lsum[0].x + lsum[0].y) + (lsum[1].x + lsum[1].y);
    const float inv = 1.f / l;
    if (tok < p.ntok) {
      if (p.lse) p.lse[static_cast<size_t>(bh) * p.ntok + tok] = fmaf(cs, E, log2f(l));
#pragma unroll
      for (int c0 = 0; c0 < HD; c0 += 8) {
        uint4 u;
        u.x = pack_bf16(__uint_as_float(r[c0 + 0]) * inv, __uint_as_float(r[c0 + 1]) * inv);
        u.y = pack_bf16(__uint_as_float(r[c0 + 2]) * inv, __uint_as_float(r[c0 + 3]) * inv);
        u.z = pack_bf16(__uint_as_float(r[c0 + 4]) * inv, __uint_as_float(r[c0 + 5]) * inv);
        u.w = pack_bf16(__uint_as_float(r[c0 + 6]) * inv, __uint_as_float(r[c0 + 7]) * inv);
        *reinterpret_cast<uint4*>(dst + c0) = u;
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

template <int HD, int POLY, bool TP>
int launch_small_p(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, __nv_bfloat16* out, int B, int heads,
                   int ntok, int ldo, cudaStream_t st, float* lse, float scale) {
  using Cfg = SmallCfg<HD, TP>;
  SmallMaps maps;
  const int BH = B * heads;
  {
    uint64_t dims[3] = {static_cast<uint64_t>(HD), static_cast<uint64_t>(ntok), static_cast<uint64_t>(BH)};
    uint64_t strides[3] = {1, static_cast<uint64_t>(HD), static_cast<uint64_t>(HD) * ntok};
    uint32_t boxq[3] = {static_cast<uint32_t>(HD), 128, 1};
    uint32_t boxk[3] = {static_cast<uint32_t>(HD), static_cast<uint32_t>(kBKV), 1};
    if (int e = encode_tmap_bf16(&maps.q, q, 3, dims, strides, boxq, Cfg::kSwz)) return e;
    if (int e = encode_tmap_bf16(&maps.k, k, 3, dims, strides, boxk, Cfg::kSwz)) return e;
  }
  {
    uint64_t dims[3] = {static_cast<uint64_t>(ntok), static_cast<uint64_t>(HD), static_cast<uint64_t>(BH)};
    uint64_t strides[3] = {1, static_cast<uint64_t>(ntok), static_cast<uint64_t>(HD) * ntok};
    uint32_t box[3] = {64, static_cast<uint32_t>(HD), 1};
    if (int e = encode_tmap_bf16(&maps.vt, vt, 3, dims, strides, box, 128)) return e;
  }
  SmallArgs args;
  args.ntok = ntok; args.heads = heads; args.ldo = ldo; args.out = out; args.lse = lse;
  {
    const float sl2 = attn_scale_log2(scale, HD);
    int ex = 0;
    const float mant = frexpf(sl2, &ex);    // sl2 = mant * 2^ex, mant in [0.5, 1)
    args.c = mant * 2.f;
    args.qscale = ldexpf(1.f, ex - 1);
  }
  static bool attr_set = false;
  if (!attr_set) {
    WC_CHECK_CUDA(cudaFuncSetAttribute(attention_small_kernel<HD, POLY, TP>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem));
    attr_set = true;
  }
  const int nqb = (ntok + 128 * kNQ - 1) / (128 * kNQ);
  dim3 grid(HD == 16 ? BH : nqb, HD == 16 ? nqb : BH);
  ProfScope prof(kProfAttention, st, 4.0 * BH * static_cast<double>(ntok) * ntok * HD);
  prof.note(BH, ntok, HD);
  launch_k<1>(attention_small_kernel<HD, POLY, TP>, grid, Cfg::kThreads, Cfg::kSmem, st, maps, args);
  WC_LAUNCH_CHECK();
  return 0;
}

template <int HD>
int launch_small(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, __nv_bfloat16* out, int B, int heads,
                 int ntok, int ldo, cudaStream_t st, float* lse, float scale) {
  // POLY (how many of every 32 exponentials run on the FMA pipe), measured best on B200 (N 8192, batch 32): 12 for head_dim 16
  // (2.46 ms), 8 for head_dim 32 (2.55 ms).
  // TP: P in tensor memory (aliased on the consumed S buffer) instead of shared memory.  Measured on B200 (batch 32, N 8192):
  // head_dim 32: 2.52 -> 2.40 ms; head_dim 16: 2.43 -> 2.48 ms (the whole S tile held in registers spills at 128 registers,
  // which costs more than the saved stores when there are no row-sum FADDs to begin with) -> head_dim 32 only.
  return launch_small_p<HD, HD == 16 ? 12 : 8, HD == 32>(q, k, vt, out, B, heads, ntok, ldo, st, lse, scale);
}

}  // namespace

// Same contract as attention_forward (attention.cu); head_dim 16 or 32 only.
int attention_small_forward(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, __nv_bfloat16* out, int B,
                            int heads, int ntok, int hd, int ldo, cudaStream_t st, float* lse, float scale) {
  switch (hd) {
    case 16: return launch_small<16>(q, k, vt, out, B, heads, ntok, ldo, st, lse, scale);
    case 32: return launch_small<32>(q, k, vt, out, B, heads, ntok, ldo, st, lse, scale);
    default: return fail("attention_small: unsupported head_dim " + std::to_string(hd));
  }
}

}  // namespace wc
