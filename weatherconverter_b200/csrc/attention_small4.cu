// Flash attention for head dims 16 / 32 with FOUR softmax warpgroups per CTA (round 2).  Same arithmetic as attention_small.cu
// (offset folded into the S accumulator through an extra K = 16 MMA step, lazy stale maximum with overflow detection on the
// packed P words / the tile sum, row sums on the tensor core for head_dim 16); what changes is the occupancy model:
//
//   * attention_small.cu runs 3 softmax groups because S is double-buffered in tensor memory (3 x (2 x 64 + 32) = 480 columns).
//     Measured on B200 (batch 32, N 8192, head_dim 16): 2 groups 3.14 ms, 3 groups 2.43 ms, i.e. t = 1.0 + 4.26 / groups ms - a
//     pipe-bound floor plus a latency-bound term that only more resident warps shrink (profiles/r2_pipe_rate.txt: the MUFU +
//     FMA pipes could deliver 31 exponentials / clk / SM, the 3-group kernel reaches 12).
//   * Here S is SINGLE-buffered (4 x (64 + 32) = 384 columns): a group loads its whole 128 x 64 tile into registers (two
//     tcgen05.ld of 32 columns per thread), immediately hands the buffer back (s_free) and the S issuer starts S(q, j+1) while
//     the group exponentiates tile j from registers - the same overlap as double buffering, paid with 64 live registers.
//   * Registers: 640 threads -> 96 per thread at launch (61440 for the CTA); the four service warps shrink to 56
//     (setmaxnreg.dec) and the 16 softmax warps grow to 104 (setmaxnreg.inc): 128 x 56 + 512 x 104 = 60416 (measured: 32 / 112 starves the issuing warps).
//   * Two issuing warps: warp 1 issues the S MMAs (waits on s_free in group order), warp 3 the PV MMAs (waits on p_full), so
//     neither kind of event queues behind the other.
//   * P goes through shared memory (double-buffered).  P' in tensor memory in its own 32 columns per group (4 x (64 + 32 + 32) = 512
//     columns, tcgen05.st + PV with the A operand from tensor memory) was tried and is much slower here: 3.08 vs 2.24 ms
//     (head_dim 16, batch 32, N 8192).
#include "wc_host.h"
#include "wc_ptx.cuh"

#include <type_traits>

namespace wc {

namespace {

struct Small4Args {
  int ntok, heads, ldo;
  float qscale;      // 2^k:  log2(e) * softmax scale = qscale * c
  float c;           // in [1, 2)
  __nv_bfloat16* out;
  float* lse;
};

struct Small4Maps {
  CUtensorMap q, k, vt;
};

constexpr int kBKV = 64;          // keys per tile
constexpr int kNQ = 4;            // query tiles (softmax warpgroups) per CTA
constexpr int kKStages = 4;       // K / V^T TMA ring depth
constexpr float kShift = 8.0f;    // P' = P * 2^-8 while the stale maximum holds
constexpr float kLazy = 6.0f;
// setmaxnreg moves registers inside the CTA's OWN allocation (640 threads x 96 registers = 61440 at launch), so
// 128 * kRegsService + 512 * kRegsSoftmax must not exceed 61440: (32, 112) or (56, 104)
#ifndef WC_S4_SERVICE_REGS
#define WC_S4_SERVICE_REGS 56
#define WC_S4_SOFTMAX_REGS 104
#endif
constexpr int kRegsService = WC_S4_SERVICE_REGS, kRegsSoftmax = WC_S4_SOFTMAX_REGS;
static_assert(128 * kRegsService + 512 * kRegsSoftmax <= 640 * 96, "register pool of the CTA");

template <int HD>
struct Cfg4 {
  static constexpr bool kLT = true;                             // row sums on the tensor core: 4 x (64 + hd + 16) <= 512 columns for hd 16 and 32
  static constexpr int kRowBytes = HD * 2;
  static constexpr int kSwz = HD * 2;
  static constexpr int kKSteps = HD / 16;
  static constexpr int kVRows = HD + (kLT ? 16 : 0);            // N of the PV product
  static constexpr uint32_t kQTile = 128 * HD * 2;
  static constexpr uint32_t kXTile = 128 * 32;                  // augmented K = 16 step of Q, 32-byte rows
  static constexpr uint32_t kKxTile = kBKV * 32;
  static constexpr uint32_t kKTile = kBKV * HD * 2;
  static constexpr uint32_t kVBlock = kVRows * 128;             // 64 keys x kVRows
  static constexpr uint32_t kVLoad = HD * 128;
  static constexpr uint32_t kPTile = 128 * kBKV * 2;
  static constexpr uint32_t kSmem = kNQ * kQTile + kNQ * kXTile + kKxTile + kKStages * (kKTile + kVBlock) + 2 * kNQ * kPTile + 1024 + 512;
  static constexpr int kThreads = 128 + 128 * kNQ;
  static constexpr int kColsPerQ = kBKV + kVRows;               // S | O (+ l)
  static_assert(kNQ * kColsPerQ <= 512, "TMEM budget");
  static constexpr uint32_t kTmemCols = 512;
};

__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void lds128(uint32_t addr, uint32_t (&v)[4]) {
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(addr) : "memory");
}
__device__ __forceinline__ void sts16(uint32_t addr, uint16_t v) {
  asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(v) : "memory");
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
__device__ __forceinline__ uint16_t bf16_bits(float x) {
  __nv_bfloat16 h = __float2bfloat16_rn(x);
  return *reinterpret_cast<uint16_t*>(&h);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
  unsigned long long ua = *reinterpret_cast<unsigned long long*>(&a), ub = *reinterpret_cast<unsigned long long*>(&b), ud;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(ud) : "l"(ua), "l"(ub));
  return *reinterpret_cast<float2*>(&ud);
}
// 2^(c*x) for a pair on the FMA / ALU pipes (see attention_small.cu: exp2_poly2_scaled - same polynomial, same domain limit)
__device__ __forceinline__ float2 exp2_poly2_scaled(float2 x, float2 c, float lo) {
  const float kMagic = 12582912.f;
  x.x = fmaxf(x.x, lo);
  x.y = fmaxf(x.y, lo);
  const float2 r = ffma2(x, c, make_float2(kMagic, kMagic));
  const float2 nn = ffma2(r, make_float2(-1.f, -1.f), make_float2(kMagic, kMagic));
  const float2 f = ffma2(x, c, nn);
  float2 p = ffma2(f, make_float2(0.05517163872718811f, 0.05517163872718811f), make_float2(0.2426111251115799f, 0.2426111251115799f));
  p = ffma2(p, f, make_float2(0.6932609677314758f, 0.6932609677314758f));
  p = ffma2(p, f, make_float2(0.9999280571937561f, 0.9999280571937561f));
  float2 o;
  o.x = __uint_as_float((__float_as_uint(r.x) << 23) + __float_as_uint(p.x));
  o.y = __uint_as_float((__float_as_uint(r.y) << 23) + __float_as_uint(p.y));
  return o;
}

// Of every 32 exponentials, this many run on the FMA pipe.  Measured on B200 (batch 32, N 8192, head_dim 16): 8: 2.245 ms, 12: 2.262,
// 16: 2.427.
constexpr int kSmall4Poly = 8;

template <int HD, bool UNIT>   // UNIT: the softmax scale is exactly 1 in the log2 domain (Q prescaled by the QKV projection)
__global__ void __launch_bounds__(Cfg4<HD>::kThreads, 1)
attention_small4_kernel(const __grid_constant__ Small4Maps maps, const __grid_constant__ Small4Args p) {
  using Cfg = Cfg4<HD>;
  constexpr bool LT = Cfg::kLT;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t q_smem = base;
  const uint32_t qx_smem = q_smem + kNQ * Cfg::kQTile;
  const uint32_t kx_smem = qx_smem + kNQ * Cfg::kXTile;
  const uint32_t k_smem = kx_smem + Cfg::kKxTile;
  const uint32_t v_smem = k_smem + kKStages * Cfg::kKTile;
  const uint32_t p_smem = v_smem + kKStages * Cfg::kVBlock;
  const uint32_t bars = p_smem + 2 * kNQ * Cfg::kPTile;
  const uint32_t q_full = bars;
  auto k_full = [&](int s) { return bars + 8u * (1 + s); };
  auto k_empty = [&](int s) { return bars + 8u * (5 + s); };
  auto v_full = [&](int s) { return bars + 8u * (9 + s); };
  auto v_empty = [&](int s) { return bars + 8u * (13 + s); };
  auto s_full = [&](int q) { return bars + 8u * (17 + q); };
  auto s_free = [&](int q) { return bars + 8u * (21 + q); };
  auto p_full = [&](int q, int b) { return bars + 8u * (25 + 2 * q + b); };
  auto pv_done = [&](int q, int b) { return bars + 8u * (33 + 2 * q + b); };
  auto q_ready = [&](int q) { return bars + 8u * (41 + q); };
  const uint32_t tmem_slot = bars + 8u * 45;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp index, provably uniform
  const int bh = HD == 16 ? blockIdx.x : blockIdx.y;
  const int q0 = (HD == 16 ? blockIdx.y : blockIdx.x) * (128 * kNQ);
  const int nkv = (p.ntok + kBKV - 1) / kBKV;
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
      mbar_init(s_full(q), 1);
      mbar_init(s_free(q), 128);
      for (int b = 0; b < 2; ++b) {
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
  pdl_launch_dependents();
  pdl_wait();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsService));
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
      // ===================== S issuer: S(q, j+1) as soon as group q has loaded S(q, j) into registers =====================
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t idesc_s = umma_idesc_bf16(128, kBKV);
      const uint64_t dq = umma_smem_desc(q_smem, Cfg::kSwz, 8 * Cfg::kRowBytes);
      const uint64_t dx = umma_smem_desc(qx_smem, 32, 256);
      const uint32_t hi_qk = umma_desc_hi(dq), hi_x = umma_desc_hi(dx);
      const uint32_t q_lo0 = umma_desc_lo(dq), k_lo0 = q_lo0 + ((k_smem - q_smem) >> 4);
      const uint32_t qx_lo0 = umma_desc_lo(dx), kx_lo = qx_lo0 + ((kx_smem - qx_smem) >> 4);
      auto issue_s = [&](int q, int j) {
        const uint32_t d = tmem_u + q * Cfg::kColsPerQ;
        const uint32_t q_lo = q_lo0 + q * (Cfg::kQTile >> 4), k_lo = k_lo0 + (j % kKStages) * (Cfg::kKTile >> 4);
#pragma unroll
        for (int k = 0; k < Cfg::kKSteps; ++k)
          umma_bf16(d, umma_desc_join(q_lo + 2u * k, hi_qk), umma_desc_join(k_lo + 2u * k, hi_qk), idesc_s, k != 0 ? 1u : 0u);
        umma_bf16(d, umma_desc_join(qx_lo0 + q * (Cfg::kXTile >> 4), hi_x), umma_desc_join(kx_lo, hi_x), idesc_s, 1u);   // S -= E
        umma_commit(s_full(q));
      };
      mbar_wait(k_full(0), 0);
#pragma unroll
      for (int q = 0; q < kNQ; ++q) {
        mbar_wait(q_ready(q), 0);   // every group (also one without tokens) has written its share of the constant operands
        tc_fence_after();
        if (q < nq_valid) {
          if (elect_one_sync()) issue_s(q, 0);
          __syncwarp();
        }
      }
      if (elect_one_sync()) umma_commit(k_empty(0));
      __syncwarp();
      for (int j = 0; j + 1 < nkv; ++j) {
        const int s1 = (j + 1) % kKStages;
        mbar_wait(k_full(s1), ((j + 1) / kKStages) & 1u);
#pragma unroll
        for (int q = 0; q < kNQ; ++q) {
          if (q < nq_valid) {
            mbar_wait(s_free(q), j & 1u);
            tc_fence_after();
            if (elect_one_sync()) issue_s(q, j + 1);
            __syncwarp();
          }
        }
        if (elect_one_sync()) umma_commit(k_empty(s1));
        __syncwarp();
      }
    } else if (warp == 3) {
      // ===================== PV issuer =====================
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t idesc_o = umma_idesc_bf16(128, Cfg::kVRows);
      const uint64_t dp = umma_smem_desc(p_smem, 128, 1024);
      const uint32_t hi_pv = umma_desc_hi(dp);
      const uint32_t p_lo0 = umma_desc_lo(dp), v_lo0 = p_lo0 - ((p_smem - v_smem) >> 4);
      for (int j = 0; j < nkv; ++j) {
        const int s = j % kKStages;
        mbar_wait(v_full(s), (j / kKStages) & 1u);
#pragma unroll
        for (int q = 0; q < kNQ; ++q) {
          if (q < nq_valid) {
            mbar_wait(p_full(q, j & 1), (j >> 1) & 1u);
            tc_fence_after();
            if (elect_one_sync()) {
              const uint32_t d = tmem_u + q * Cfg::kColsPerQ + kBKV;
              const uint32_t p_lo = p_lo0 + (2 * q + (j & 1)) * (Cfg::kPTile >> 4), v_lo = v_lo0 + s * (Cfg::kVBlock >> 4);
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_bf16(d, umma_desc_join(p_lo + 2u * k, hi_pv), umma_desc_join(v_lo + 2u * k, hi_pv), idesc_o, (j | k) != 0 ? 1u : 0u);
              umma_commit(pv_done(q, j & 1));
            }
            __syncwarp();
          }
        }
        if (elect_one_sync()) umma_commit(v_empty(s));
        __syncwarp();
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsSoftmax));
    // ===================== softmax warpgroups =====================
    const int q = (warp - 4) >> 2;
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
    const uint32_t s_tmem = tmem_base + q * Cfg::kColsPerQ + lane_off;
    const uint32_t o_tmem = s_tmem + kBKV;
    const uint32_t p_row = p_smem + 2 * q * Cfg::kPTile + row * 128;
    const uint32_t qx_row = qx_smem + q * Cfg::kXTile + row * 32;

    const float cs = p.c;
    const float shift = kShift / cs;       // in units of S''
    float E = bf16_round(shift);           // current offset (bf16-representable): S'' = 2^k q.k - E
    {
      const int t = threadIdx.x - 128;  // 0 .. 511
      if (q == 0 && row < kBKV) {
        sts128(kx_smem + row * 32, 0x00003F80u, 0u, 0u, 0u);
        sts128(kx_smem + row * 32 + 16, 0x00003F80u, 0u, 0u, 0u);
      }
      if (LT) {
        constexpr int kChunks = kKStages * 16 * 8;  // rows hd .. hd+15 of every V^T stage: a row of ones, then zeros
        for (int c = t; c < kChunks; c += 128 * kNQ) {
          const int blk = c >> 7, r = (c >> 3) & 15, ch = c & 7;
          const uint32_t one = r == 0 ? 0x3F803F80u : 0u;
          sts128(v_smem + blk * Cfg::kVBlock + (HD + r) * 128 + ch * 16, one, one, one, one);
        }
      }
      mbar_wait(q_full, 0);
      const uint32_t q_row = q_smem + q * Cfg::kQTile + row * Cfg::kRowBytes;
      const float qs = p.qscale;
#pragma unroll
      for (int c = 0; c < (UNIT ? 0 : Cfg::kRowBytes / 16); ++c) {
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
      mbar_arrive(q_ready(q));
    }

    float2 lsum[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};   // !LT only
    float carry = 0.f;   // S(q, j+1) was issued before tile j could move the offset: tile j+1 is corrected in registers

    for (int j = 0; j < (q < nq_valid ? nkv : 0); ++j) {
      const int b = j & 1;
      const int kv0 = j * kBKV;
      mbar_wait(s_full(q), j & 1u);
      if (j >= 2) mbar_wait(pv_done(q, b), ((j - 2) >> 1) & 1u);   // P buffer b free (PV of tile j-2 has read it)
      tc_fence_after();
      uint32_t ra[32], rb[32], w[16];
      tmem_ld32(s_tmem, ra);
      tmem_ld32(s_tmem + 32, rb);
      tmem_wait_ld();
      tc_fence_before();
      mbar_arrive(s_free(q));                 // the S issuer may overwrite the buffer with S(q, j+1) now
      const bool tail = (kv0 + kBKV > p.ntok);
      bool slow = tail || j == 0 || __any_sync(0xffffffffu, carry != 0.f);
      const uint32_t blk = p_row + b * Cfg::kPTile;
      if (!slow) {
        uint32_t orw = 0u;
        float2 ts[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
        const float2 cv = make_float2(cs, cs);
        const float lo = -125.f / cs;
        auto half = [&](const uint32_t (&cur)[32], int c) {
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const float2 xs = make_float2(__uint_as_float(cur[i]), __uint_as_float(cur[i + 1]));
            float2 v;
            if (i < kSmall4Poly) {
              v = exp2_poly2_scaled(xs, cv, lo);
            } else {
              const float2 y = UNIT ? xs : fmul2(xs, cv);
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
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) {
            const int chunk = 4 * c + ch;
            sts128(blk + (static_cast<uint32_t>(chunk ^ (row & 7)) << 4), w[4 * ch], w[4 * ch + 1], w[4 * ch + 2], w[4 * ch + 3]);
          }
        };
        half(ra, 0);
        half(rb, 1);
        bool redo;
        if (LT) {
          redo = (orw & 0xC000C000u) != 0u;          // some P' >= 2 (or negative / NaN garbage)
        } else {
          const float tsum = (ts[0].x + ts[0].y) + (ts[1].x + ts[1].y);
          redo = !(tsum < 32.f);                     // all P' <= 2^-8 gives tsum <= 0.25; also catches inf / NaN
        }
        slow = __any_sync(0xffffffffu, redo);
        if (!LT && !slow) { lsum[0] = fadd2(lsum[0], ts[0]); lsum[1] = fadd2(lsum[1], ts[1]); }
      }
      if (slow) {
        // ---- slow path from the registers: true tile maximum, offset update, O rescale, masked tail
        float tmax = -INFINITY;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float a0 = __uint_as_float(ra[i]), a1 = __uint_as_float(rb[i]);
          if (tail && kv0 + i >= p.ntok) a0 = -INFINITY;
          if (tail && kv0 + 32 + i >= p.ntok) a1 = -INFINITY;
          tmax = fmaxf(tmax, fmaxf(a0, a1));
        }
        tmax -= carry;                       // relative to the CURRENT offset E
        float delta = 0.f;
        const bool upd = (j == 0) || (tmax > -shift + kLazy / cs);
        if (upd) {
          // S(q, j+1) is issued right after this group's s_free arrivals and reads Qx: it must have completed before Qx changes
          if (j + 1 < nkv) mbar_wait(s_full(q), (j + 1) & 1u);
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
        auto redo_half = [&](const uint32_t (&cur)[32], int c, float2& acc) {
          const int k0 = kv0 + 32 * c;
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            float v0 = ex2_approx(fmaf(__uint_as_float(cur[i]), cs, dneg)), v1 = ex2_approx(fmaf(__uint_as_float(cur[i + 1]), cs, dneg));
            if (tail) {
              if (k0 + i >= p.ntok) v0 = 0.f;
              if (k0 + i + 1 >= p.ntok) v1 = 0.f;
            }
            if (!LT) { acc.x += v0; acc.y += v1; }
            w[i >> 1] = pack_bf16(v0, v1);
          }
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) {
            const int chunk = 4 * c + ch;
            sts128(blk + (static_cast<uint32_t>(chunk ^ (row & 7)) << 4), w[4 * ch], w[4 * ch + 1], w[4 * ch + 2], w[4 * ch + 3]);
          }
        };
        redo_half(ra, 0, lsum[0]);
        redo_half(rb, 1, lsum[1]);
      }
      fence_proxy_async_smem();   // P (and possibly Qx) were written through the generic proxy, the MMAs read them through the async one
      tc_fence_before();
      mbar_arrive(p_full(q, b));
    }

    // ---- finalize: O / l -> bf16 -> out[b, tok, head*hd + d]
    if (q < nq_valid) mbar_wait(pv_done(q, (nkv - 1) & 1), ((nkv - 1) >> 1) & 1u);
    tc_fence_after();
    const int tok = q0 + q * 128 + row;
    const int bb = bh / p.heads, head = bh % p.heads;
    __nv_bfloat16* dst = p.out + (static_cast<size_t>(bb) * p.ntok + tok) * p.ldo + head * HD;
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

template <int HD, bool UNIT>
int launch_small4_p(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, __nv_bfloat16* out, int B, int heads,
                    int ntok, int ldo, cudaStream_t st, float* lse, float scale) {
  using Cfg = Cfg4<HD>;
  Small4Maps maps;
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
  Small4Args args;
  args.ntok = ntok; args.heads = heads; args.ldo = ldo; args.out = out; args.lse = lse;
  {
    const float sl2 = attn_scale_log2(scale, HD);   // 1 -> c = 1, qscale = 1 (UNIT)
    int ex = 0;
    const float mant = frexpf(sl2, &ex);
    args.c = mant * 2.f;
    args.qscale = ldexpf(1.f, ex - 1);
  }
  static bool attr_set = false;
  if (!attr_set) {
    WC_CHECK_CUDA(cudaFuncSetAttribute(attention_small4_kernel<HD, UNIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem));
    attr_set = true;
  }
  const int nqb = (ntok + 128 * kNQ - 1) / (128 * kNQ);
  dim3 grid(HD == 16 ? BH : nqb, HD == 16 ? nqb : BH);
  ProfScope prof(kProfAttention, st, 4.0 * BH * static_cast<double>(ntok) * ntok * HD);
  prof.note(BH, ntok, HD);
  launch_k<1>(attention_small4_kernel<HD, UNIT>, grid, Cfg::kThreads, Cfg::kSmem, st, maps, args);
  WC_LAUNCH_CHECK();
  return 0;
}

template <int HD>
int launch_small4(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, __nv_bfloat16* out, int B, int heads,
                  int ntok, int ldo, cudaStream_t st, float* lse, float scale) {
  // inference runs Q prescaled by the QKV projection (unit scale), the training plan unscaled Q
  if (attn_scale_log2(scale, HD) == 1.f) return launch_small4_p<HD, true>(q, k, vt, out, B, heads, ntok, ldo, st, lse, scale);
  return launch_small4_p<HD, false>(q, k, vt, out, B, heads, ntok, ldo, st, lse, scale);
}

}  // namespace

// Same contract as attention_small_forward; four softmax groups per CTA.
int attention_small4_forward(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, __nv_bfloat16* out, int B,
                             int heads, int ntok, int hd, int ldo, cudaStream_t st, float* lse, float scale) {
  switch (hd) {
    case 16: return launch_small4<16>(q, k, vt, out, B, heads, ntok, ldo, st, lse, scale);
    case 32: return launch_small4<32>(q, k, vt, out, B, heads, ntok, ldo, st, lse, scale);
    default: return fail("attention_small4: unsupported head_dim " + std::to_string(hd));
  }
}

}  // namespace wc
