// GroupNorm(8 groups, eps 1e-5, affine) with optional fused SiLU on NHWC bf16 activations.
// Reference ops: nn.GroupNorm(8, C) [+ nn.SiLU] at unet_base.py:89-90,101-102,107,155-156,483-484.
// Two bandwidth-bound passes: (1) per-(sample, slab) partial sums, (2) deterministic combine + normalise.
// Statistics are identical for the 4-D [B,C,H,W] and 3-D [B,C,HW] uses (biased variance over C/8 x HW).
#include "wc_host.h"
#include "wc_ptx.cuh"

namespace wc {

namespace {

constexpr int kGroups = 8;

// x * sigmoid(x) = h + h * tanh(h), h = x / 2: ONE MUFU op (tanh.approx, relative error 2^-11 - the result is rounded to bf16,
// 2^-9) instead of two (ex2 + rcp); the apply pass of a 33 MB tensor otherwise spends 7 us of its ~12 us on the MUFU pipe
__device__ __forceinline__ float silu_fast(float x) {
  const float h = 0.5f * x;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

// Each thread owns one 8-channel vector column (fixed group) and strides over pixels.
__global__ void gn_stats_kernel(const __nv_bfloat16* __restrict__ x, int HW, int C, int ld, int nsplit,
                                float2* __restrict__ partial) {
  pdl_prologue();
  extern __shared__ float2 stash[];
  const int vpp = C / 8, gv = (C / kGroups) / 8;  // vectors per pixel, vectors per group
  const int rows = blockDim.x / vpp;
  const int v = threadIdx.x % vpp, r = threadIdx.x / vpp;
  const int b = blockIdx.y, split = blockIdx.x;
  const int p0 = static_cast<int>(static_cast<long long>(HW) * split / nsplit);
  const int p1 = static_cast<int>(static_cast<long long>(HW) * (split + 1) / nsplit);
  const __nv_bfloat16* xb = x + static_cast<size_t>(b) * HW * ld + v * 8;
  float s = 0.f, ss = 0.f;
  auto acc = [&](const uint4& u) {
    const float2 a = unpack_bf16(u.x), bq = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
    s += (a.x + a.y) + (bq.x + bq.y) + (c.x + c.y) + (d.x + d.y);
    ss += (a.x * a.x + a.y * a.y) + (bq.x * bq.x + bq.y * bq.y) + (c.x * c.x + c.y * c.y) + (d.x * d.x + d.y * d.y);
  };
  int p = p0 + r;
  for (; p + 3 * rows < p1; p += 4 * rows) {   // four independent 16-byte loads in flight per thread
    const uint4 u0 = __ldg(reinterpret_cast<const uint4*>(xb + static_cast<size_t>(p) * ld));
    const uint4 u1 = __ldg(reinterpret_cast<const uint4*>(xb + static_cast<size_t>(p + rows) * ld));
    const uint4 u2 = __ldg(reinterpret_cast<const uint4*>(xb + static_cast<size_t>(p + 2 * rows) * ld));
    const uint4 u3 = __ldg(reinterpret_cast<const uint4*>(xb + static_cast<size_t>(p + 3 * rows) * ld));
    acc(u0); acc(u1); acc(u2); acc(u3);
  }
  for (; p < p1; p += rows) acc(__ldg(reinterpret_cast<const uint4*>(xb + static_cast<size_t>(p) * ld)));
  stash[threadIdx.x] = make_float2(s, ss);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nwarps = blockDim.x >> 5;
  for (int g = warp; g < kGroups; g += nwarps) {  // one warp reduces one group in a fixed order (deterministic)
    const int cnt = rows * gv;
    float as = 0.f, ass = 0.f;
    for (int i = lane; i < cnt; i += 32) {
      const int tid = (i / gv) * vpp + g * gv + (i % gv);
      const float2 t = stash[tid];
      as += t.x; ass += t.y;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      as += __shfl_xor_sync(0xffffffffu, as, o);
      ass += __shfl_xor_sync(0xffffffffu, ass, o);
    }
    if (lane == 0) partial[(static_cast<size_t>(b) * nsplit + split) * kGroups + g] = make_float2(as, ass);
  }
}

// Combine the per-slab partial sums of sample b into mean / rstd per group.  Warp g owns group g: lane i takes slab i (<= 32 slabs),
// the sums are added in double precision in a FIXED butterfly order (deterministic, independent of the batch) instead of one thread
// per group looping over up to 32 slabs of dependent FP64 adds.  (Measured neutral on the C3 step: 1.50 vs 1.51 ms for the class.)
__device__ __forceinline__ void combine_partials(const float2* __restrict__ partial, int b, int nsplit_stats, int HW, int C, float eps,
                                                 float* s_mean, float* s_rstd) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int g = warp; g < kGroups; g += (blockDim.x >> 5)) {
    double s = 0.0, ss = 0.0;
    for (int i = lane; i < nsplit_stats; i += 32) {
      const float2 t = partial[(static_cast<size_t>(b) * nsplit_stats + i) * kGroups + g];
      s += t.x; ss += t.y;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s += __shfl_xor_sync(0xffffffffu, s, o);
      ss += __shfl_xor_sync(0xffffffffu, ss, o);
    }
    if (lane == 0) {
      const double n = static_cast<double>(HW) * (C / kGroups);
      const double mean = s / n;
      double var = ss / n - mean * mean;
      if (var < 0.0) var = 0.0;
      s_mean[g] = static_cast<float>(mean);
      s_rstd[g] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
    }
  }
}

__global__ void gn_apply_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, int HW, int C,
                                int ld, int ldy, int nsplit_stats, int nsplit, const float2* __restrict__ partial,
                                const float* __restrict__ gamma, const float* __restrict__ beta, float eps, int silu) {
  pdl_prologue();
  __shared__ float s_mean[kGroups], s_rstd[kGroups];
  const int b = blockIdx.y, split = blockIdx.x;
  combine_partials(partial, b, nsplit_stats, HW, C, eps, s_mean, s_rstd);
  __syncthreads();
  const int vpp = C / 8, cpg = C / kGroups;
  const int rows = blockDim.x / vpp;
  const int v = threadIdx.x % vpp, r = threadIdx.x / vpp;
  const int g = (v * 8) / cpg;
  const float mean = s_mean[g], rstd = s_rstd[g];
  float ga[8], be[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    ga[j] = gamma[v * 8 + j] * rstd;
    be[j] = beta[v * 8 + j] - mean * ga[j];
  }
  const int p0 = static_cast<int>(static_cast<long long>(HW) * split / nsplit);
  const int p1 = static_cast<int>(static_cast<long long>(HW) * (split + 1) / nsplit);
  const __nv_bfloat16* xb = x + static_cast<size_t>(b) * HW * ld + v * 8;
  __nv_bfloat16* yb = y + static_cast<size_t>(b) * HW * ldy + v * 8;
  auto one = [&](const uint4& u, int p) {
    float f[8];
    float2 t;
    t = unpack_bf16(u.x); f[0] = t.x; f[1] = t.y;
    t = unpack_bf16(u.y); f[2] = t.x; f[3] = t.y;
    t = unpack_bf16(u.z); f[4] = t.x; f[5] = t.y;
    t = unpack_bf16(u.w); f[6] = t.x; f[7] = t.y;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float o = fmaf(f[j], ga[j], be[j]);
      if (silu) o = silu_fast(o);
      f[j] = o;
    }
    uint4 w;
    w.x = pack_bf16(f[0], f[1]); w.y = pack_bf16(f[2], f[3]); w.z = pack_bf16(f[4], f[5]); w.w = pack_bf16(f[6], f[7]);
    *reinterpret_cast<uint4*>(yb + static_cast<size_t>(p) * ldy) = w;
  };
  int p = p0 + r;
  for (; p + 3 * rows < p1; p += 4 * rows) {   // four independent 16-byte loads in flight per thread
    const uint4 u0 = __ldg(reinterpret_cast<const uint4*>(xb + static_cast<size_t>(p) * ld));
    const uint4 u1 = __ldg(reinterpret_cast<const uint4*>(xb + static_cast<size_t>(p + rows) * ld));
    const uint4 u2 = __ldg(reinterpret_cast<const uint4*>(xb + static_cast<size_t>(p + 2 * rows) * ld));
    const uint4 u3 = __ldg(reinterpret_cast<const uint4*>(xb + static_cast<size_t>(p + 3 * rows) * ld));
    one(u0, p); one(u1, p + rows); one(u2, p + 2 * rows); one(u3, p + 3 * rows);
  }
  for (; p < p1; p += rows) one(__ldg(reinterpret_cast<const uint4*>(xb + static_cast<size_t>(p) * ld)), p);
}


// ------------------------------------------------------------------------------------------------ backward
// y = act(gamma * xhat + beta), xhat = (x - mean) * rstd, act = SiLU or identity.  With dz = dy * act'(z):
//   dgamma_c = sum dz * xhat,  dbeta_c = sum dz,
//   dx = rstd * (gamma*dz - S1/n - xhat * S2/n),  S1 = sum_group gamma*dz,  S2 = sum_group gamma*dz*xhat.
// (autograd of nn.GroupNorm + nn.SiLU in loss.backward(), diffusion_model/train_ddpm.py:108.)
__device__ __forceinline__ void load8(const __nv_bfloat16* p, float (&f)[8]) {
  const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
  float2 t;
  t = unpack_bf16(u.x); f[0] = t.x; f[1] = t.y;
  t = unpack_bf16(u.y); f[2] = t.x; f[3] = t.y;
  t = unpack_bf16(u.z); f[4] = t.x; f[5] = t.y;
  t = unpack_bf16(u.w); f[6] = t.x; f[7] = t.y;
}

__device__ __forceinline__ void group_stats(const float2* partial, int b, int nsplit_stats, int HW, int C, float eps,
                                            float* s_mean, float* s_rstd) {
  combine_partials(partial, b, nsplit_stats, HW, C, eps, s_mean, s_rstd);   // the same order as the forward pass: identical statistics
  __syncthreads();
}

__device__ __forceinline__ float act_grad(float z, float dy, int silu) {
  if (!silu) return dy;
  const float s = 1.f / (1.f + __expf(-z));
  return dy * s * (1.f + z * (1.f - s));
}

// pass 1: per (sample, slab, channel) sums of dz and dz*xhat
__global__ void gn_bwd_stats_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ dy, int HW, int C,
                                    int ld, int ldd, int nsplit_stats, int nsplit, const float2* __restrict__ partial,
                                    const float* __restrict__ gamma, const float* __restrict__ beta, float eps, int silu,
                                    float2* __restrict__ part) {
  pdl_prologue();
  __shared__ float s_mean[kGroups], s_rstd[kGroups];
  extern __shared__ float2 stash[];  // [rows][C]
  const int b = blockIdx.y, split = blockIdx.x;
  group_stats(partial, b, nsplit_stats, HW, C, eps, s_mean, s_rstd);
  const int vpp = C / 8, cpg = C / kGroups;
  const int rows = blockDim.x / vpp;
  const int v = threadIdx.x % vpp, r = threadIdx.x / vpp;
  const int g = (v * 8) / cpg;
  const float mean = s_mean[g], rstd = s_rstd[g];
  float ga[8], be[8], a0[8], a1[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { ga[j] = gamma[v * 8 + j]; be[j] = beta[v * 8 + j]; a0[j] = 0.f; a1[j] = 0.f; }
  const int p0 = static_cast<int>(static_cast<long long>(HW) * split / nsplit);
  const int p1 = static_cast<int>(static_cast<long long>(HW) * (split + 1) / nsplit);
  const __nv_bfloat16* xb = x + static_cast<size_t>(b) * HW * ld + v * 8;
  const __nv_bfloat16* db = dy + static_cast<size_t>(b) * HW * ldd + v * 8;
  auto accum = [&](const float (&f)[8], const float (&d)[8]) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float xh = (f[j] - mean) * rstd;
      const float dz = act_grad(fmaf(ga[j], xh, be[j]), d[j], silu);
      a0[j] += dz;
      a1[j] = fmaf(dz, xh, a1[j]);
    }
  };
  int p = p0 + r;
  for (; p + rows < p1; p += 2 * rows) {   // four independent 16-byte loads in flight per thread
    float f0[8], d0[8], f1[8], d1[8];
    load8(xb + static_cast<size_t>(p) * ld, f0);
    load8(db + static_cast<size_t>(p) * ldd, d0);
    load8(xb + static_cast<size_t>(p + rows) * ld, f1);
    load8(db + static_cast<size_t>(p + rows) * ldd, d1);
    accum(f0, d0);
    accum(f1, d1);
  }
  for (; p < p1; p += rows) {
    float f[8], d[8];
    load8(xb + static_cast<size_t>(p) * ld, f);
    load8(db + static_cast<size_t>(p) * ldd, d);
    accum(f, d);
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) stash[static_cast<size_t>(r) * C + v * 8 + j] = make_float2(a0[j], a1[j]);
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s0 = 0.f, s1 = 0.f;
    for (int rr = 0; rr < rows; ++rr) { const float2 t = stash[static_cast<size_t>(rr) * C + c]; s0 += t.x; s1 += t.y; }
    part[(static_cast<size_t>(b) * nsplit + split) * C + c] = make_float2(s0, s1);
  }
}

// pass 2: per-sample channel sums bc[b][c] and group sums gs[b][g] = (S1, S2)
__global__ void gn_bwd_reduce_kernel(const float2* __restrict__ part, int C, int nsplit, const float* __restrict__ gamma,
                                     float2* __restrict__ bc, float2* __restrict__ gs) {
  pdl_prologue();
  extern __shared__ float2 prod[];  // [C]
  const int b = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s0 = 0.f, s1 = 0.f;
    for (int i = 0; i < nsplit; ++i) { const float2 t = part[(static_cast<size_t>(b) * nsplit + i) * C + c]; s0 += t.x; s1 += t.y; }
    bc[static_cast<size_t>(b) * C + c] = make_float2(s0, s1);
    const float gm = gamma[c];
    prod[c] = make_float2(gm * s0, gm * s1);
  }
  __syncthreads();
  if (threadIdx.x < kGroups) {
    const int cpg = C / kGroups;
    float s0 = 0.f, s1 = 0.f;
    for (int c = threadIdx.x * cpg; c < (threadIdx.x + 1) * cpg; ++c) { s0 += prod[c].x; s1 += prod[c].y; }
    gs[b * kGroups + threadIdx.x] = make_float2(s0, s1);
  }
}

__global__ void gn_bwd_param_kernel(const float2* __restrict__ bc, int B, int C, float* __restrict__ dgamma,
                                    float* __restrict__ dbeta) {
  pdl_prologue();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s0 = 0.f, s1 = 0.f;
  for (int b = 0; b < B; ++b) { const float2 t = bc[static_cast<size_t>(b) * C + c]; s0 += t.x; s1 += t.y; }
  dbeta[c] = s0;
  dgamma[c] = s1;
}

// pass 3: dx (+ up to two additive gradient inputs)
__global__ void gn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ dy,
                                    __nv_bfloat16* __restrict__ dx, int HW, int C, int ld, int ldd, int ldo, int nsplit_stats,
                                    int nsplit, const float2* __restrict__ partial, const float2* __restrict__ gs,
                                    const float* __restrict__ gamma, const float* __restrict__ beta, float eps, int silu,
                                    const __nv_bfloat16* __restrict__ add1, int lda1, const __nv_bfloat16* __restrict__ add2,
                                    int lda2) {
  pdl_prologue();
  __shared__ float s_mean[kGroups], s_rstd[kGroups];
  const int b = blockIdx.y, split = blockIdx.x;
  group_stats(partial, b, nsplit_stats, HW, C, eps, s_mean, s_rstd);
  const int vpp = C / 8, cpg = C / kGroups;
  const int rows = blockDim.x / vpp;
  const int v = threadIdx.x % vpp, r = threadIdx.x / vpp;
  const int g = (v * 8) / cpg;
  const float mean = s_mean[g], rstd = s_rstd[g];
  const float inv_n = 1.f / (static_cast<float>(HW) * cpg);
  const float2 sg = gs[b * kGroups + g];
  const float m1 = sg.x * inv_n, m2 = sg.y * inv_n;
  float ga[8], be[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { ga[j] = gamma[v * 8 + j]; be[j] = beta[v * 8 + j]; }
  const int p0 = static_cast<int>(static_cast<long long>(HW) * split / nsplit);
  const int p1 = static_cast<int>(static_cast<long long>(HW) * (split + 1) / nsplit);
  const size_t boff = static_cast<size_t>(b) * HW;
  for (int p = p0 + r; p < p1; p += rows) {
    float f[8], d[8], o[8];
    load8(x + (boff + p) * ld + v * 8, f);
    load8(dy + (boff + p) * ldd + v * 8, d);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float xh = (f[j] - mean) * rstd;
      const float dz = act_grad(fmaf(ga[j], xh, be[j]), d[j], silu);
      o[j] = rstd * (ga[j] * dz - m1 - xh * m2);
    }
    if (add1) {
      float t[8];
      load8(add1 + (boff + p) * lda1 + v * 8, t);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] += t[j];
    }
    if (add2) {
      float t[8];
      load8(add2 + (boff + p) * lda2 + v * 8, t);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] += t[j];
    }
    uint4 w;
    w.x = pack_bf16(o[0], o[1]); w.y = pack_bf16(o[2], o[3]); w.z = pack_bf16(o[4], o[5]); w.w = pack_bf16(o[6], o[7]);
    *reinterpret_cast<uint4*>(dx + (boff + p) * ldo + v * 8) = w;
  }
}

// per-sample column sums of an NHWC bf16 tensor: part[b][split][c]
__global__ void colsum_kernel(const __nv_bfloat16* __restrict__ x, int HW, int C, int ld, int nsplit, float* __restrict__ part) {
  pdl_prologue();
  extern __shared__ float cstash[];  // [rows][C]
  const int b = blockIdx.y, split = blockIdx.x;
  const int vpp = C / 8;
  const int rows = blockDim.x / vpp;
  const int v = threadIdx.x % vpp, r = threadIdx.x / vpp;
  float a[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = 0.f;
  const int p0 = static_cast<int>(static_cast<long long>(HW) * split / nsplit);
  const int p1 = static_cast<int>(static_cast<long long>(HW) * (split + 1) / nsplit);
  const __nv_bfloat16* xb = x + static_cast<size_t>(b) * HW * ld + v * 8;
  if (r < rows) {
    int p = p0 + r;
    for (; p + 3 * rows < p1; p += 4 * rows) {   // four independent 16-byte loads in flight per thread
      float f0[8], f1[8], f2[8], f3[8];
      load8(xb + static_cast<size_t>(p) * ld, f0);
      load8(xb + static_cast<size_t>(p + rows) * ld, f1);
      load8(xb + static_cast<size_t>(p + 2 * rows) * ld, f2);
      load8(xb + static_cast<size_t>(p + 3 * rows) * ld, f3);
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] += (f0[j] + f1[j]) + (f2[j] + f3[j]);
    }
    for (; p < p1; p += rows) {
      float f[8];
      load8(xb + static_cast<size_t>(p) * ld, f);
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] += f[j];
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) cstash[static_cast<size_t>(r) * C + v * 8 + j] = a[j];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s = 0.f;
    for (int rr = 0; rr < rows; ++rr) s += cstash[static_cast<size_t>(rr) * C + c];
    part[(static_cast<size_t>(b) * nsplit + split) * C + c] = s;
  }
}

// out_rows[b*ldo + c] = sum_split part (optional), out_total[c] = sum_b sum_split part (optional).  Block = 64 channels x 8
// sample lanes; every sum runs in a fixed order (deterministic).
__global__ void colsum_finish_kernel(const float* __restrict__ part, int B, int C, int nsplit, float* __restrict__ out_rows,
                                     int ldo, float* __restrict__ out_total) {
  pdl_prologue();
  __shared__ float tot[8][64];
  const int cl = threadIdx.x & 63, bl = threadIdx.x >> 6;   // 512 threads
  const int c = blockIdx.x * 64 + cl;
  float t = 0.f;
  if (c < C) {
    for (int b = bl; b < B; b += 8) {
      float s = 0.f;
      for (int i = 0; i < nsplit; ++i) s += part[(static_cast<size_t>(b) * nsplit + i) * C + c];
      if (out_rows) out_rows[static_cast<size_t>(b) * ldo + c] = s;
      t += s;
    }
  }
  tot[bl][cl] = t;
  __syncthreads();
  if (bl == 0 && c < C && out_total) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += tot[k][cl];
    out_total[c] = s;
  }
}


}  // namespace

size_t groupnorm_workspace_bytes(int B) { return static_cast<size_t>(B) * 64 * kGroups * sizeof(float2); }

// Number of per-sample slabs the statistics pass of groupnorm_silu uses for a [B,HW,C] input (the backward pass
// re-combines the same partial sums).
// A function of HW only: the partial sums of a sample are then combined in the same order whatever the batch size, so image b
// of a batch gets bit-identical statistics to the same image processed alone (batch invariance of the whole UNet forward,
// tests/test_gpu_config_shapes.py).  Large batches simply get more, smaller blocks (B * nsplit).
int groupnorm_stats_splits(int B, int HW) {
  (void)B;
  int nsplit = (HW + 127) / 128;     // >= 128 pixels per block (a block of 2048 got 1.5x slower with 32-pixel slabs)
  if (HW <= 2048) {                  // 1, 2, 4 or 8 slabs per sample: this rule fixes the summation order, and with it the bits
    int c = 1;
    while (c * 2 <= nsplit && c < 8) c *= 2;
    return c;
  }
  if (nsplit > 32) nsplit = 32;
  if (nsplit < 1) nsplit = 1;
  return nsplit;
}

// x: [B,HW,C] bf16 with pixel stride ld; y likewise with ldy; workspace >= groupnorm_workspace_bytes(B).
int groupnorm_silu(const __nv_bfloat16* x, __nv_bfloat16* y, int B, int HW, int C, int ld, int ldy, const float* gamma,
                   const float* beta, float eps, int silu, void* workspace, cudaStream_t st) {
  WC_REQUIRE(C % 64 == 0 && C / 8 <= 256, "GroupNorm(8) kernel needs C % 64 == 0 and C <= 2048");
  WC_REQUIRE(ld % 8 == 0 && ldy % 8 == 0, "pixel strides must be multiples of 8 elements");
  const int vpp = C / 8;
  const int threads = (256 / vpp) * vpp;
  const int nsplit = groupnorm_stats_splits(B, HW);
  const int max_split = (HW + 31) / 32;
  float2* partial = reinterpret_cast<float2*>(workspace);
  // Two passes, statistics then apply.  A single-launch variant with one thread-block cluster per sample was measured slower on B200
  // in both regimes: batch 32, GroupNorm 1.55 -> 2.13 ms per C3 step (8 CTAs per sample cannot fill the chip on 25 - 67 MB tensors);
  // batch 1, 0.94 -> 1.61 ms per step (a cluster launch plus two cluster barriers cost more than the second small launch).
  ProfScope prof(kProfGroupNorm, st, 6.0 * B * static_cast<double>(HW) * C);  // algorithmic bytes: 2 reads + 1 write, bf16
  launch_k(gn_stats_kernel, dim3(nsplit, B), threads, threads * sizeof(float2), st, x, HW, C, ld, nsplit, partial);
  WC_LAUNCH_CHECK();
  constexpr int kApplyBlocksPerSm = 8;   // 2 .. 8 measured within 3 % of each other, 16 is 9 % slower; the result does not depend on it
  int asplit = (kApplyBlocksPerSm * num_sms() + B - 1) / B;
  if (asplit > max_split) asplit = max_split;
  if (asplit < 1) asplit = 1;
  launch_k(gn_apply_kernel, dim3(asplit, B), threads, 0, st, x, y, HW, C, ld, ldy, nsplit, asplit, partial, gamma, beta, eps,
                                                       silu);
  WC_LAUNCH_CHECK();
  prof.note(HW, C, ld, ldy, nsplit, asplit);
  return 0;
}

}  // namespace wc

namespace wc {

namespace {
int bwd_splits(int B, int HW) {
  int n = (8 * num_sms() + B - 1) / B;
  const int max_split = (HW + 31) / 32;
  if (n > max_split) n = max_split;
  if (n > 32) n = 32;
  if (n < 1) n = 1;
  return n;
}
}  // namespace

// Scratch for groupnorm_silu_bwd / colsum: part [B][32][C] float2 + bc [B][C] float2 + gs [B][8] float2.
size_t groupnorm_bwd_workspace_bytes(int B, int Cmax) {
  return static_cast<size_t>(B) * 32 * Cmax * sizeof(float2) + static_cast<size_t>(B) * Cmax * sizeof(float2) +
         static_cast<size_t>(B) * kGroups * sizeof(float2) + 1024;
}

// Backward of groupnorm_silu.  `stats` is the workspace the forward call wrote (per-slab partial sums).  dx = dGN(dy)
// (+ add1) (+ add2); dgamma/dbeta fp32 [C] are overwritten.
int groupnorm_silu_bwd(const __nv_bfloat16* x, const __nv_bfloat16* dy, __nv_bfloat16* dx, int B, int HW, int C, int ld,
                       int ldd, int ldo, const float* gamma, const float* beta, float eps, int silu, const void* stats,
                       const __nv_bfloat16* add1, int lda1, const __nv_bfloat16* add2, int lda2, float* dgamma, float* dbeta,
                       void* workspace, cudaStream_t st) {
  WC_REQUIRE(C % 64 == 0 && C / 8 <= 256, "GroupNorm(8) kernel needs C % 64 == 0 and C <= 2048");
  WC_REQUIRE(ld % 8 == 0 && ldd % 8 == 0 && ldo % 8 == 0 && lda1 % 8 == 0 && lda2 % 8 == 0, "pixel strides must be multiples of 8");
  const int vpp = C / 8;
  const int threads = (256 / vpp) * vpp;
  const int rows = threads / vpp;
  const int ns_stats = groupnorm_stats_splits(B, HW);
  const int nsplit = bwd_splits(B, HW);
  float2* part = reinterpret_cast<float2*>(workspace);
  float2* bc = part + static_cast<size_t>(B) * 32 * C;
  float2* gs = bc + static_cast<size_t>(B) * C;
  const float2* partial = reinterpret_cast<const float2*>(stats);
  ProfScope prof(kProfGroupNorm, st, 10.0 * B * static_cast<double>(HW) * C);  // x, dy read twice, dx written (bf16)
  launch_k(gn_bwd_stats_kernel, dim3(nsplit, B), threads, static_cast<size_t>(rows) * C * sizeof(float2), st, 
      x, dy, HW, C, ld, ldd, ns_stats, nsplit, partial, gamma, beta, eps, silu, part);
  WC_LAUNCH_CHECK();
  launch_k(gn_bwd_reduce_kernel, B, 256, C * sizeof(float2), st, part, C, nsplit, gamma, bc, gs);
  WC_LAUNCH_CHECK();
  launch_k(gn_bwd_param_kernel, (C + 127) / 128, 128, 0, st, bc, B, C, dgamma, dbeta);
  WC_LAUNCH_CHECK();
  int asplit = (8 * num_sms() + B - 1) / B;
  const int max_split = (HW + 31) / 32;
  if (asplit > max_split) asplit = max_split;
  if (asplit < 1) asplit = 1;
  launch_k(gn_bwd_apply_kernel, dim3(asplit, B), threads, 0, st, x, dy, dx, HW, C, ld, ldd, ldo, ns_stats, asplit, partial, gs, gamma,
                                                           beta, eps, silu, add1, lda1, add2, lda2);
  WC_LAUNCH_CHECK();
  // strides < 2^16 (C <= 2048 and concat buffers of at most 2C); a missing add term notes stride 0
  prof.note(HW, C, ld | ldd << 16, ldo | (add1 ? lda1 : 0) << 16, add2 ? lda2 : 0, nsplit | asplit << 16);
  return 0;
}

// Column sums of x [B,HW,C] (bf16, pixel stride ld): out_rows[b*ldo + c] per sample (may be null) and out_total[c]
// over the whole batch (may be null) -- the bias gradients of the convolutions / linears and the per-sample gradient
// of the t-embedding projection (unet_base.py:148).  workspace >= groupnorm_bwd_workspace_bytes(B, C).
int colsum(const __nv_bfloat16* x, int B, int HW, int C, int ld, float* out_rows, int ldo, float* out_total, void* workspace,
           cudaStream_t st) {
  WC_REQUIRE(C % 8 == 0 && ld % 8 == 0 && C <= 4096, "colsum: C must be a multiple of 8 (<= 4096)");
  const int vpp = C / 8;
  int threads = vpp >= 256 ? ((vpp + 31) / 32) * 32 : (256 / vpp) * vpp;
  if (threads > 1024) return fail("colsum: too many channels");
  const int rows = threads / vpp > 0 ? threads / vpp : 1;
  const int nsplit = bwd_splits(B, HW);
  float* part = reinterpret_cast<float*>(workspace);
  ProfScope prof(kProfOther, st, 2.0 * B * static_cast<double>(HW) * C);
  launch_k(colsum_kernel, dim3(nsplit, B), threads, static_cast<size_t>(rows) * C * sizeof(float), st, x, HW, C, ld, nsplit, part);
  WC_LAUNCH_CHECK();
  launch_k(colsum_finish_kernel, (C + 63) / 64, 512, 0, st, part, B, C, nsplit, out_rows, ldo, out_total);
  WC_LAUNCH_CHECK();
  // the last field tags the record (class kProfOther is shared): 1 + which outputs are written (2: rows, 4: total)
  prof.note(HW, C, ld, out_rows ? ldo : 0, nsplit, 1 + (out_rows ? 2 : 0) + (out_total ? 4 : 0));
  return 0;
}

}  // namespace wc
