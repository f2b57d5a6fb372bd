// Backward of the flash attention core (attention.cu) on tcgen05: given Q, K, V, dO and the forward's per-row
// log-sum-exp, computes dQ, dK, dV without materialising the N x N probability matrix.  Replaces autograd through
// nn.MultiheadAttention's softmax(QK^T/sqrt(hd))V (unet_base.py:159) in loss.backward() (train_ddpm.py:108).
//
// Two passes of ONE kernel template (no atomics, deterministic):
//   KV pass : a CTA owns 128 keys (K_j, V_j resident) and streams query tiles (Q_i, dO_i):
//               S^T = K_j Q_i^T, dP^T = V_j dO_i^T            (tcgen05, K-major operands, contraction over hd)
//               P^T = exp2(S^T*c - lse_i), dS^T = P^T o (dP^T - D_i)   (softmax warps, one thread per key row)
//               dV_j += P^T dO_i,  dK_j += dS^T Q_i            (A = bf16 P^T/dS^T written to smem K-major,
//                                                               B = the SAME dO_i/Q_i smem tiles read MN-major)
//   Q pass  : a CTA owns 128 queries (Q_i, dO_i resident) and streams key tiles (K_j, V_j):
//               S = Q_i K_j^T, dP = dO_i V_j^T, dS = P o (dP - D_i),  dQ_i += dS K_j   (B = K_j read MN-major)
// D_i = rowsum(dO_i o O_i) is precomputed (attn_rowdot).  Accumulators (S, dP, dV/dK or dQ) live in TMEM.
// Outputs are written as bf16 into one [B, N, 3C] buffer (dQ | dK | dV per token), which is exactly the dY operand
// of the in-projection's data / weight gradients.

#include "wc_host.h"
#include "wc_ptx.cuh"

namespace wc {

namespace {

struct AttnBwdArgs {
  int ntok, heads, C, ld3;  // ld3: row stride of the dqkv buffer (>= 3C)
  float scale_log2, scale;
  const float* lse;  // [B*heads][ntok], log2 domain
  const float* D;    // [B*heads][ntok]
  __nv_bfloat16* dqkv;
};

struct AttnBwdMaps {
  CUtensorMap r1, r2, t1, t2;
};

constexpr int kPoly = 12;             // of every 32 exponentials, this many run on the FMA pipe (exp2_poly2)

// NSW = number of softmax warpgroups.  NSW == 2: one CTA per SM, two warps per TMEM lane quadrant interleave the
// 32-column chunks.  NSW == 1 (head_dim <= 64, BT = 64): the CTA needs <= 256 TMEM columns and <= 113 KB of shared
// memory, so TWO CTAs share an SM and one CTA's exp / dS phase overlaps the other's MMA phase.
// The dQ pass (!KV) keeps its dS' operand in TENSOR MEMORY (written by the softmax threads with tcgen05.st, read by tcgen05.mma as
// its A operand); the KV pass keeps P' and dS' in shared memory.
template <int HD, int BT, int STAGES, bool KV, int NSW>
struct BwdCfg {
  static constexpr int kKBlocks = HD >= 64 ? HD / 64 : 1;
  static constexpr int kRowBytes = HD >= 64 ? 128 : HD * 2;
  static constexpr int kKSteps = HD >= 64 ? 4 : HD / 16;
  static constexpr uint32_t kRTile = 128 * HD * 2;
  static constexpr uint32_t kTTile = BT * HD * 2;
  static constexpr uint32_t kPTile = 128 * BT * 2;
  static constexpr int kNP = KV ? 2 : 1;
  static constexpr uint32_t kVecBytes = KV ? 2 * 2 * BT * 4 : 0;
  static constexpr uint32_t kFixed = 2 * kRTile + STAGES * 2 * kTTile + kVecBytes + 1024 + 256;
  // P'/dS' tiles are double-buffered when shared memory allows it (then the softmax of tile i+1 never waits for the
  // dV/dK/dQ MMAs of tile i)
  static constexpr int kCtasPerSm = NSW == 1 ? 2 : 1;
  static constexpr uint32_t kSmemLimit = NSW == 1 ? 115712 : 232448;
  static constexpr int kColsBase = 2 * BT + (KV ? 2 : 1) * HD;
  static constexpr int kTmemBudget = 512 / kCtasPerSm;
  static constexpr int kPB = !KV ? ((kColsBase + 2 * kNP * (BT / 2) <= kTmemBudget) ? 2 : 1)
                                 : ((kFixed + 2 * kNP * kPTile <= kSmemLimit) ? 2 : 1);
  static constexpr uint32_t kSmem = kFixed + (KV ? kPB * kNP * kPTile : 0);
  static constexpr int kPCol = kColsBase;   // dQ pass: dS' buffer b at kPCol + b*(BT/2)
  static constexpr int kSoftmaxThreads = 128 * NSW;
  static constexpr int kThreads = 128 + kSoftmaxThreads;  // warp 0 TMA, warp 1 MMA, warp 2 TMEM alloc, warps 4.. softmax / epilogue
  static constexpr int kCols = kColsBase + (KV ? 0 : kPB * kNP * (BT / 2));
  static constexpr uint32_t kTmemCols = kCols <= 128 ? 128 : (kCols <= 256 ? 256 : 512);
  static constexpr int kAcc0 = 2 * BT;                  // KV: dV ; Q: dQ
  static constexpr int kAcc1 = 2 * BT + (KV ? HD : 0);  // KV: dK
  static_assert(kCols <= 512 && kTmemCols * kCtasPerSm <= 512, "TMEM budget");
  static_assert(kSmem <= kSmemLimit, "shared memory budget");
};

template <int HD, int BT, int STAGES, bool KV, int NSW>
__global__ void __launch_bounds__(128 + 128 * NSW, NSW == 1 ? 2 : 1)
attention_bwd_kernel(const __grid_constant__ AttnBwdMaps maps, const __grid_constant__ AttnBwdArgs p) {
  using Cfg = BwdCfg<HD, BT, STAGES, KV, NSW>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_u32 = smem_u32(smem_raw);
  const uint32_t base = (raw_u32 + 1023u) & ~1023u;
  const uint32_t r1_smem = base;
  const uint32_t r2_smem = r1_smem + Cfg::kRTile;
  const uint32_t t_smem = r2_smem + Cfg::kRTile;                  // stage s: T1 at t_smem + s*2*kTTile, T2 right after
  const uint32_t p_smem = t_smem + STAGES * 2 * Cfg::kTTile;      // dS' first, then (KV) P'
  const uint32_t vec_smem = p_smem + (KV ? Cfg::kPB * Cfg::kNP * Cfg::kPTile : 0u);
  const uint32_t bars = vec_smem + Cfg::kVecBytes;
  const uint32_t r_full = bars;
  auto t_full = [&](int s) { return bars + 8u * (1 + s); };
  auto t_empty = [&](int s) { return bars + 8u * (3 + s); };
  const uint32_t s_full = bars + 8u * 5, p_full = bars + 8u * 6;
  auto acc_done = [&](int b) { return bars + 8u * (7 + b); };
  const uint32_t tmem_slot = bars + 8u * 9;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw_u32));

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp index, provably uniform
  const int bh = blockIdx.y, b = bh / p.heads, h = bh % p.heads;
  const int r0 = blockIdx.x * 128;
  const int nt = (p.ntok + BT - 1) / BT;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&maps.r1); tma_prefetch_desc(&maps.r2); tma_prefetch_desc(&maps.t1); tma_prefetch_desc(&maps.t2);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(r_full, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(t_full(s), 1); mbar_init(t_empty(s), 1); }
    mbar_init(s_full, 1);
    mbar_init(p_full, Cfg::kSoftmaxThreads);
    mbar_init(acc_done(0), 1);
    mbar_init(acc_done(1), 1);
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
      mbar_arrive_expect_tx(r_full, 2 * Cfg::kRTile);
      for (int kb = 0; kb < Cfg::kKBlocks; ++kb) {
        tma_load_4d(r1_smem + kb * (128 * Cfg::kRowBytes), &maps.r1, r_full, kb * 64, r0, h, b);
        tma_load_4d(r2_smem + kb * (128 * Cfg::kRowBytes), &maps.r2, r_full, kb * 64, r0, h, b);
      }
      for (int i = 0; i < nt; ++i) {
        const int s = i % STAGES;
        const uint32_t ph = (i / STAGES) & 1u;
        mbar_wait(t_empty(s), ph ^ 1u);
        mbar_arrive_expect_tx(t_full(s), 2 * Cfg::kTTile);
        const uint32_t t1 = t_smem + s * 2 * Cfg::kTTile, t2 = t1 + Cfg::kTTile;
        for (int kb = 0; kb < Cfg::kKBlocks; ++kb) {
          tma_load_4d(t1 + kb * (BT * Cfg::kRowBytes), &maps.t1, t_full(s), kb * 64, i * BT, h, b);
          tma_load_4d(t2 + kb * (BT * Cfg::kRowBytes), &maps.t2, t_full(s), kb * 64, i * BT, h, b);
        }
      }
    }
  } else if (warp == 1) {
    {
      // ===================== MMA issuer =====================
      // Warp-uniform control flow, one elected lane issues (see igemm.cu).
      const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_ptr, 0);
      const uint32_t idesc_s = umma_idesc_bf16(128, BT);
      const uint32_t idesc_acc = umma_idesc_bf16(128, HD, 0, 1);  // B operand MN-major
      // K-major descriptors of the hd-contraction operands (R1, R2, T1, T2) and of the P'/dS' tiles
      const uint64_t dk = umma_smem_desc(r1_smem, Cfg::kRowBytes, 8 * Cfg::kRowBytes);
      const uint64_t dp = umma_smem_desc(p_smem, 128, 1024);
      const uint32_t hi_k = umma_desc_hi(dk), hi_p = umma_desc_hi(dp);
      const uint32_t r1_lo = umma_desc_lo(dk), r2_lo = r1_lo + (Cfg::kRTile >> 4), t_lo0 = r1_lo + ((t_smem - r1_smem) >> 4);
      const uint32_t p_lo0 = umma_desc_lo(dp);
      // MN-major view of the T tiles: start address | LBO (stride between 64-column atoms) in the low word; the high word
      // (SBO = 8 rows, swizzle mode) is the same as the K-major one
      const uint32_t lbo_field = (HD >= 64 ? static_cast<uint32_t>(BT * 128) >> 4 : 1u) << 16;
      const uint32_t tmn_lo0 = ((t_smem & 0x3FFFF) >> 4) | lbo_field;
      auto issue_s = [&](int i) {
        const int s = i % STAGES;
        const uint32_t t1_lo = t_lo0 + s * ((2 * Cfg::kTTile) >> 4), t2_lo = t1_lo + (Cfg::kTTile >> 4);
#pragma unroll
        for (int kb = 0; kb < Cfg::kKBlocks; ++kb)
#pragma unroll
          for (int k = 0; k < Cfg::kKSteps; ++k)
            umma_bf16(tmem_base, umma_desc_join(r1_lo + kb * ((128 * Cfg::kRowBytes) >> 4) + 2u * k, hi_k),
                      umma_desc_join(t1_lo + kb * ((BT * Cfg::kRowBytes) >> 4) + 2u * k, hi_k), idesc_s, (kb | k) != 0 ? 1u : 0u);
#pragma unroll
        for (int kb = 0; kb < Cfg::kKBlocks; ++kb)
#pragma unroll
          for (int k = 0; k < Cfg::kKSteps; ++k)
            umma_bf16(tmem_base + BT, umma_desc_join(r2_lo + kb * ((128 * Cfg::kRowBytes) >> 4) + 2u * k, hi_k),
                      umma_desc_join(t2_lo + kb * ((BT * Cfg::kRowBytes) >> 4) + 2u * k, hi_k), idesc_s, (kb | k) != 0 ? 1u : 0u);
        umma_commit(s_full);
      };
      auto issue_acc = [&](int i) {
        const int s = i % STAGES;
        const uint32_t p_lo = p_lo0 + (i % Cfg::kPB) * ((Cfg::kNP * Cfg::kPTile) >> 4);
        const uint32_t t1_mn = tmn_lo0 + s * ((2 * Cfg::kTTile) >> 4), t2_mn = t1_mn + (Cfg::kTTile >> 4);
        constexpr uint32_t kstep16 = (16 * Cfg::kRowBytes) >> 4;  // 16 rows of the T tile per MMA K step
        // dS' is the first P tile, P' (KV pass only) the second
#pragma unroll
        for (int cb = 0; cb < BT / 64; ++cb)
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int kk = cb * 4 + k;
            if (!KV) {
              const uint32_t pa = tmem_base + Cfg::kPCol + (i % Cfg::kPB) * (Cfg::kNP * (BT / 2)) + 8u * kk;
              umma_bf16_ts(tmem_base + Cfg::kAcc1, pa, umma_desc_join(t1_mn + kk * kstep16, hi_k), idesc_acc, (i | kk) != 0 ? 1u : 0u);
            } else {
              umma_bf16(tmem_base + Cfg::kAcc0, umma_desc_join(p_lo + (Cfg::kPTile >> 4) + cb * ((128 * 128) >> 4) + 2u * k, hi_p),
                        umma_desc_join(t2_mn + kk * kstep16, hi_k), idesc_acc, (i | kk) != 0 ? 1u : 0u);
              umma_bf16(tmem_base + Cfg::kAcc1, umma_desc_join(p_lo + cb * ((128 * 128) >> 4) + 2u * k, hi_p),
                        umma_desc_join(t1_mn + kk * kstep16, hi_k), idesc_acc, (i | kk) != 0 ? 1u : 0u);
            }
          }
        umma_commit(acc_done(i % Cfg::kPB));
        umma_commit(t_empty(s));
      };
      mbar_wait(r_full, 0);
      mbar_wait(t_full(0), 0);
      tc_fence_after();
      if (elect_one_sync()) issue_s(0);
      __syncwarp();
      for (int i = 0; i < nt; ++i) {
        mbar_wait(p_full, i & 1u);
        tc_fence_after();
        const bool more = i + 1 < nt;
        if (STAGES >= 2 && more) {
          mbar_wait(t_full((i + 1) % STAGES), ((i + 1) / STAGES) & 1u);
          tc_fence_after();
        }
        if (elect_one_sync()) {
          if (STAGES >= 2 && more) issue_s(i + 1);
          issue_acc(i);
        }
        __syncwarp();
        if (STAGES == 1 && more) {
          mbar_wait(t_full(0), (i + 1) & 1u);
          tc_fence_after();
          if (elect_one_sync()) issue_s(i + 1);
          __syncwarp();
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== softmax-backward warps =====================
    const int quad = warp & 3;
    const int grp = NSW == 2 ? (warp - 4) >> 2 : 0;  // which share of the interleaved 32-column chunks
    const int row = quad * 32 + lane;
    const int tid = threadIdx.x - 128;
    const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
    const uint32_t s_tmem = tmem_base + lane_off, dp_tmem = s_tmem + BT;
    float* vec = reinterpret_cast<float*>(smem_raw + (vec_smem - raw_u32));  // [buf][lse | D][BT]
    const float sl2 = p.scale_log2;
    const size_t voff = static_cast<size_t>(bh) * p.ntok;
    float my_lse = 0.f, my_D = 0.f;
    if (!KV && r0 + row < p.ntok) { my_lse = p.lse[voff + r0 + row]; my_D = p.D[voff + r0 + row]; }
    constexpr int NCH = BT / 32;
    for (int i = 0; i < nt; ++i) {
      const int t0 = i * BT;
      float* vl = vec + (i & 1) * 2 * BT;
      if (KV) {
        if (tid < BT) {
          const int t = t0 + tid;
          vl[tid] = t < p.ntok ? p.lse[voff + t] : INFINITY;
          vl[BT + tid] = t < p.ntok ? p.D[voff + t] : 0.f;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(128 * NSW) : "memory");
      }
      const uint32_t ds_row = p_smem + (i % Cfg::kPB) * (Cfg::kNP * Cfg::kPTile) + row * 128, pp_row = ds_row + Cfg::kPTile;
      mbar_wait(s_full, i & 1u);
      tc_fence_after();
      const bool tail = !KV && (t0 + BT > p.ntok);
      bool p_free = (i < Cfg::kPB);  // first use of a P buffer needs no wait
#pragma unroll
      for (int cc = 0; cc < (NCH + NSW - 1) / NSW; ++cc) {
        const int c = NSW * cc + grp;
        if (c >= NCH) break;
        uint32_t rs[32], rd[32];
        tmem_ld32(s_tmem + 32 * c, rs);
        tmem_ld32(dp_tmem + 32 * c, rd);
        tmem_wait_ld();
        uint32_t wp[16], wd[16];
        const float2 sl2v = make_float2(sl2, sl2);
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          float2 l2, Dc;
          if (KV) {
            l2 = *reinterpret_cast<const float2*>(vl + 32 * c + j);
            Dc = *reinterpret_cast<const float2*>(vl + BT + 32 * c + j);
          } else {
            l2 = make_float2(my_lse, my_lse);
            Dc = make_float2(my_D, my_D);
          }
          const float2 xs = ffma2(make_float2(__uint_as_float(rs[j]), __uint_as_float(rs[j + 1])), sl2v, make_float2(-l2.x, -l2.y));
          float2 pe;
          if (j < kPoly) {
            pe = exp2_poly2(xs);
          } else {
            pe.x = ex2_approx(xs.x);
            pe.y = ex2_approx(xs.y);
          }
          if (tail) {
            if (t0 + 32 * c + j >= p.ntok) pe.x = 0.f;
            if (t0 + 32 * c + j + 1 >= p.ntok) pe.y = 0.f;
          }
          const float2 dd = fadd2(make_float2(__uint_as_float(rd[j]), __uint_as_float(rd[j + 1])), make_float2(-Dc.x, -Dc.y));
          wp[j >> 1] = pack_bf16(pe.x, pe.y);
          wd[j >> 1] = pack_bf16(pe.x * dd.x, pe.y * dd.y);
        }
        if (!p_free) {  // the MMAs that read this P buffer (tile i - kPB) must have completed before it is overwritten
          mbar_wait(acc_done(i % Cfg::kPB), ((i / Cfg::kPB) - 1) & 1u);
          p_free = true;
        }
        if (!KV) {
          tmem_st16(s_tmem + Cfg::kPCol + (i % Cfg::kPB) * (Cfg::kNP * (BT / 2)) + 16 * c, wd);
          continue;
        }
        const uint32_t blk_off = ((32 * c) >> 6) * (128 * 128);
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const int chunk = (((32 * c) & 63) >> 3) + ch;
          const uint32_t sw = static_cast<uint32_t>(chunk ^ (row & 7)) << 4;
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(ds_row + blk_off + sw), "r"(wd[4 * ch]), "r"(wd[4 * ch + 1]),
                       "r"(wd[4 * ch + 2]), "r"(wd[4 * ch + 3]) : "memory");
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(pp_row + blk_off + sw), "r"(wp[4 * ch]), "r"(wp[4 * ch + 1]),
                       "r"(wp[4 * ch + 2]), "r"(wp[4 * ch + 3]) : "memory");
        }
      }
      if (KV) fence_proxy_async_smem();
      else tmem_wait_st();
      tc_fence_before();
      mbar_arrive(p_full);
    }
    // ---- epilogue: accumulators -> bf16 -> dqkv[b, tok, which*C + h*hd + d]; the two warp groups split the columns
    mbar_wait(acc_done((nt - 1) % Cfg::kPB), ((nt - 1) / Cfg::kPB) & 1u);
    tc_fence_after();
    const int tok = r0 + row;
    __nv_bfloat16* orow = p.dqkv + (static_cast<size_t>(b) * p.ntok + tok) * p.ld3 + h * HD;
    auto store_acc = [&](uint32_t taddr, int which, float mul) {
#pragma unroll
      for (int c0 = 0; c0 < HD; c0 += 16) {
        if (NSW == 2 && ((c0 >> 4) & 1) != grp) continue;
        uint32_t r[16];
        tmem_ld16(taddr + c0, r);
        tmem_wait_ld();
        if (tok < p.ntok) {
          uint4 u0, u1;
          u0.x = pack_bf16(__uint_as_float(r[0]) * mul, __uint_as_float(r[1]) * mul);
          u0.y = pack_bf16(__uint_as_float(r[2]) * mul, __uint_as_float(r[3]) * mul);
          u0.z = pack_bf16(__uint_as_float(r[4]) * mul, __uint_as_float(r[5]) * mul);
          u0.w = pack_bf16(__uint_as_float(r[6]) * mul, __uint_as_float(r[7]) * mul);
          u1.x = pack_bf16(__uint_as_float(r[8]) * mul, __uint_as_float(r[9]) * mul);
          u1.y = pack_bf16(__uint_as_float(r[10]) * mul, __uint_as_float(r[11]) * mul);
          u1.z = pack_bf16(__uint_as_float(r[12]) * mul, __uint_as_float(r[13]) * mul);
          u1.w = pack_bf16(__uint_as_float(r[14]) * mul, __uint_as_float(r[15]) * mul);
          __nv_bfloat16* dst = orow + which * p.C + c0;
          *reinterpret_cast<uint4*>(dst) = u0;
          *reinterpret_cast<uint4*>(dst + 8) = u1;
        }
      }
    };
    if (KV) {
      store_acc(s_tmem + Cfg::kAcc0, 2, 1.f);        // dV
      store_acc(s_tmem + Cfg::kAcc1, 1, p.scale);    // dK
    } else {
      store_acc(s_tmem + Cfg::kAcc1, 0, p.scale);    // dQ
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

struct BwdTensors {
  const __nv_bfloat16 *q, *k, *v;  // [B,heads,ntok,hd]
  const __nv_bfloat16* d_o;        // [B,ntok,ldd], head h at columns h*hd
  int ldd;
};

int make_head_map(CUtensorMap* m, const __nv_bfloat16* ptr, int hd, int ntok, int heads, int B, uint64_t s_tok, uint64_t s_head,
                  uint64_t s_b, int rows) {
  uint64_t dims[4] = {static_cast<uint64_t>(hd), static_cast<uint64_t>(ntok), static_cast<uint64_t>(heads), static_cast<uint64_t>(B)};
  uint64_t strides[4] = {1, s_tok, s_head, s_b};
  uint32_t box[4] = {static_cast<uint32_t>(hd >= 64 ? 64 : hd), static_cast<uint32_t>(rows), 1, 1};
  return encode_tmap_bf16(m, ptr, 4, dims, strides, box, hd >= 64 ? 128 : hd * 2);
}

template <int HD, int BT, int STAGES, bool KV, int NSW>
int launch_bwd(const BwdTensors& t, const float* lse, const float* D, __nv_bfloat16* dqkv, int ld3, int B, int heads, int ntok,
               cudaStream_t st) {
  using Cfg = BwdCfg<HD, BT, STAGES, KV, NSW>;
  AttnBwdMaps maps;
  const uint64_t sh = static_cast<uint64_t>(ntok) * HD, sb = sh * heads;
  const uint64_t dsb = static_cast<uint64_t>(ntok) * t.ldd;
  if (KV) {
    if (int e = make_head_map(&maps.r1, t.k, HD, ntok, heads, B, HD, sh, sb, 128)) return e;
    if (int e = make_head_map(&maps.r2, t.v, HD, ntok, heads, B, HD, sh, sb, 128)) return e;
    if (int e = make_head_map(&maps.t1, t.q, HD, ntok, heads, B, HD, sh, sb, BT)) return e;
    if (int e = make_head_map(&maps.t2, t.d_o, HD, ntok, heads, B, t.ldd, HD, dsb, BT)) return e;
  } else {
    if (int e = make_head_map(&maps.r1, t.q, HD, ntok, heads, B, HD, sh, sb, 128)) return e;
    if (int e = make_head_map(&maps.r2, t.d_o, HD, ntok, heads, B, t.ldd, HD, dsb, 128)) return e;
    if (int e = make_head_map(&maps.t1, t.k, HD, ntok, heads, B, HD, sh, sb, BT)) return e;
    if (int e = make_head_map(&maps.t2, t.v, HD, ntok, heads, B, HD, sh, sb, BT)) return e;
  }
  AttnBwdArgs a;
  a.ntok = ntok; a.heads = heads; a.C = heads * HD; a.ld3 = ld3;
  a.scale = 1.f / sqrtf(static_cast<float>(HD));
  a.scale_log2 = 1.4426950408889634f * a.scale;
  a.lse = lse; a.D = D; a.dqkv = dqkv;
  static bool attr_set = false;
  if (!attr_set) {
    WC_CHECK_CUDA(cudaFuncSetAttribute(attention_bwd_kernel<HD, BT, STAGES, KV, NSW>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem));
    attr_set = true;
  }
  dim3 grid((ntok + 127) / 128, B * heads);
  const double flops = (KV ? 8.0 : 6.0) * B * heads * static_cast<double>(ntok) * ntok * HD;
  ProfScope prof(kProfAttention, st, flops);
  launch_k<1>(attention_bwd_kernel<HD, BT, STAGES, KV, NSW>, grid, Cfg::kThreads, Cfg::kSmem, st, maps, a);
  WC_LAUNCH_CHECK();
  return 0;
}

template <int HD, int BT, int SKV, int SQ, int NSW>
int launch_both(const BwdTensors& t, const float* lse, const float* D, __nv_bfloat16* dqkv, int ld3, int B, int heads, int ntok,
                cudaStream_t st) {
  if (int e = launch_bwd<HD, BT, SKV, true, NSW>(t, lse, D, dqkv, ld3, B, heads, ntok, st)) return e;
  return launch_bwd<HD, BT, SQ, false, NSW>(t, lse, D, dqkv, ld3, B, heads, ntok, st);
}

}  // namespace

// q,k,v [B,heads,ntok,hd] bf16; d_o [B,ntok,ldd] bf16; lse (log2 domain), D fp32 [B*heads][ntok];
// dqkv [B,ntok,ld3] bf16 receives dQ | dK | dV at columns 0 | C | 2C (+ head*hd).
int attention_backward(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* v, const __nv_bfloat16* d_o, int ldd,
                       const float* lse, const float* D, __nv_bfloat16* dqkv, int ld3, int B, int heads, int ntok, int hd,
                       cudaStream_t st) {
  WC_REQUIRE(ntok % 8 == 0 && ldd % 8 == 0 && ld3 % 8 == 0, "attention backward: strides / token count must be multiples of 8");
  BwdTensors t{q, k, v, d_o, ldd};
  switch (hd) {
    // head_dim <= 64: two CTAs per SM (NSW == 1, BT = 64)
    case 16: return launch_both<16, 64, 2, 2, 1>(t, lse, D, dqkv, ld3, B, heads, ntok, st);
    case 32: return launch_both<32, 64, 2, 2, 1>(t, lse, D, dqkv, ld3, B, heads, ntok, st);
    case 64: return launch_both<64, 64, 2, 2, 1>(t, lse, D, dqkv, ld3, B, heads, ntok, st);
    case 128: return launch_both<128, 128, 1, 1, 2>(t, lse, D, dqkv, ld3, B, heads, ntok, st);
    case 192: return launch_both<192, 64, 1, 2, 2>(t, lse, D, dqkv, ld3, B, heads, ntok, st);
    default: return fail("attention backward: unsupported head_dim " + std::to_string(hd));
  }
}

double attention_bwd_flops(int B, int heads, int ntok, int hd) { return 14.0 * B * heads * static_cast<double>(ntok) * ntok * hd; }

}  // namespace wc
