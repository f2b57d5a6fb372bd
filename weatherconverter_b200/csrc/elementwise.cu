// Bandwidth-bound fp32 kernels of the DDPM scheduler (reference: diffusion_model/scheduler/
// linear_noise_scheduler.py:30-116).  Arithmetic is written with explicitly rounded intrinsics in the
// reference's operation order (no FMA contraction), so results are bit-identical to the fp32 PyTorch path.
#include "wc_host.h"

namespace wc {

namespace {

// x_{t-1} = ((x_t - (beta*eps)/s) / sqrt_alpha) + sigma*z     (scheduler.py:96-100,107-116; sample_ddpm.py:44)
struct StepCoef {
  float beta, s, sqrt_alpha, sigma;
};

// timesteps index the [T] tables: a value outside [0, T) (where the reference raises IndexError) is clamped on the device;
// the host wrappers range-check host-side t tensors and raise
__device__ __forceinline__ long long clamp_t(long long t, int T) { return t < 0 ? 0 : (t >= T ? T - 1 : t); }

__device__ __forceinline__ float ddpm_mean(float x, float e, const StepCoef& c) {
  float m = __fsub_rn(x, __fdiv_rn(__fmul_rn(c.beta, e), c.s));
  return __fdiv_rn(m, c.sqrt_alpha);
}

// kMode 0: coefficients by value (host-side scalar t); 1: sample_prev_timestep2 (per-sample t gather, sigma^2 = beta);
// 2: scalar t READ FROM DEVICE MEMORY, coefficients gathered from four host-built [T] tables (betas = {beta, s, sqrt_alpha,
//    sigma} rows) - the same fp32 values mode 0 receives by value, so results are bit-identical, but the launch no longer
//    depends on the step index and a captured CUDA graph of the reverse step can be replayed for every t > 0.
template <int kMode>
__global__ void __launch_bounds__(256)
ddpm_step_kernel(const float4* __restrict__ xt, const float4* __restrict__ eps, const float4* __restrict__ z,
                 float4* __restrict__ out, float4* __restrict__ mean_out, float4* __restrict__ sigz_out,
                 size_t n4_per_sample, int B, StepCoef c, const float* __restrict__ betas,
                 const float* __restrict__ alphas, const float* __restrict__ sqrt_1m_acp,
                 const long long* __restrict__ t, int T) {
  pdl_prologue();
  const size_t total = n4_per_sample * B;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    StepCoef cc = c;
    bool use_z = z != nullptr;
    if (kMode == 2) {
      const long long tb = clamp_t(t[0], T);
      cc.beta = betas[tb];
      cc.s = betas[T + tb];
      cc.sqrt_alpha = betas[2 * T + tb];
      cc.sigma = betas[3 * T + tb];
      use_z = use_z && tb != 0;      // t == 0: x_0 = mean (scheduler.py:102-103)
    }
    if (kMode == 1) {  // sample_prev_timestep2 (scheduler.py:63-77): per-sample gather, sigma^2 = beta
      const long long tb = clamp_t(t[i / n4_per_sample], T);
      cc.beta = betas[tb];
      cc.s = sqrt_1m_acp[tb];
      cc.sqrt_alpha = __fsqrt_rn(alphas[tb]);
      cc.sigma = __fsqrt_rn(cc.beta);
    }
    const float4 x = xt[i], e = eps[i];
    float4 m;
    m.x = ddpm_mean(x.x, e.x, cc); m.y = ddpm_mean(x.y, e.y, cc);
    m.z = ddpm_mean(x.z, e.z, cc); m.w = ddpm_mean(x.w, e.w, cc);
    if (mean_out) mean_out[i] = m;
    if (kMode == 2 && !use_z && sigz_out) sigz_out[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (use_z) {
      const float4 zz = z[i];
      float4 s;
      s.x = __fmul_rn(cc.sigma, zz.x); s.y = __fmul_rn(cc.sigma, zz.y);
      s.z = __fmul_rn(cc.sigma, zz.z); s.w = __fmul_rn(cc.sigma, zz.w);
      if (sigz_out) sigz_out[i] = s;
      m.x = __fadd_rn(m.x, s.x); m.y = __fadd_rn(m.y, s.y); m.z = __fadd_rn(m.z, s.z); m.w = __fadd_rn(m.w, s.w);
    }
    if (out) out[i] = m;
  }
}

// DDIM step tau -> tau' (Song et al., "Denoising Diffusion Implicit Models", eq. 12):
//   x0 = (x - s_t*eps) / a_t ; mean = a_p*x0 + d*eps ; out = mean + sigma*z
// a_t = sqrt(acp_tau), s_t = sqrt(1 - acp_tau), a_p = sqrt(acp_tau'), d = sqrt(1 - acp_tau' - sigma^2); the final step of a
// schedule goes to x0 (a_p = 1, d = 0, sigma = 0).
struct DdimCoef {
  float a_t, s_t, a_p, d, sigma;
};

__device__ __forceinline__ float ddim_mean(float x, float e, const DdimCoef& c) {
  const float x0 = __fdiv_rn(__fsub_rn(x, __fmul_rn(c.s_t, e)), c.a_t);
  return __fadd_rn(__fmul_rn(c.a_p, x0), __fmul_rn(c.d, e));
}

// kMode 0: coefficients by value; 2: scalar tau READ FROM DEVICE MEMORY, coefficients gathered from a host-built [5][T] table
// (rows {a_t, s_t, a_p, d, sigma}, column = the step's current tau), as ddpm_step_kernel<2>.  z == NULL or sigma == 0:
// out = mean and sigz_out = 0.
template <int kMode>
__global__ void __launch_bounds__(256)
ddim_step_kernel(const float4* __restrict__ xt, const float4* __restrict__ eps, const float4* __restrict__ z,
                 float4* __restrict__ out, float4* __restrict__ mean_out, float4* __restrict__ sigz_out,
                 size_t n4_per_sample, int B, DdimCoef c, const float* __restrict__ tables,
                 const long long* __restrict__ t, int T) {
  pdl_prologue();
  const size_t total = n4_per_sample * B;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    DdimCoef cc = c;
    if (kMode == 2) {
      const long long tb = clamp_t(t[0], T);
      cc.a_t = tables[tb];
      cc.s_t = tables[T + tb];
      cc.a_p = tables[2 * T + tb];
      cc.d = tables[3 * T + tb];
      cc.sigma = tables[4 * T + tb];
    }
    const bool use_z = z != nullptr && cc.sigma != 0.f;
    const float4 x = xt[i], e = eps[i];
    float4 m;
    m.x = ddim_mean(x.x, e.x, cc); m.y = ddim_mean(x.y, e.y, cc);
    m.z = ddim_mean(x.z, e.z, cc); m.w = ddim_mean(x.w, e.w, cc);
    if (mean_out) mean_out[i] = m;
    if (!use_z && sigz_out) sigz_out[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (use_z) {
      const float4 zz = z[i];
      float4 s;
      s.x = __fmul_rn(cc.sigma, zz.x); s.y = __fmul_rn(cc.sigma, zz.y);
      s.z = __fmul_rn(cc.sigma, zz.z); s.w = __fmul_rn(cc.sigma, zz.w);
      if (sigz_out) sigz_out[i] = s;
      m.x = __fadd_rn(m.x, s.x); m.y = __fadd_rn(m.y, s.y); m.z = __fadd_rn(m.z, s.z); m.w = __fadd_rn(m.w, s.w);
    }
    if (out) out[i] = m;
  }
}

// x_t = sqrt(acp[t_b]) * x0 + sqrt(1-acp[t_b]) * noise     (scheduler.py:30-35, 37-61)
__global__ void __launch_bounds__(256)
add_noise_kernel(const float4* __restrict__ x0, const float4* __restrict__ noise, float4* __restrict__ out,
                 size_t n4_per_sample, int B, const float* __restrict__ sqrt_acp,
                 const float* __restrict__ sqrt_1m_acp, const long long* __restrict__ t, int T) {
  pdl_prologue();
  const size_t total = n4_per_sample * B;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const long long tb = clamp_t(t[i / n4_per_sample], T);
    const float a = sqrt_acp[tb], b = sqrt_1m_acp[tb];
    const float4 x = x0[i], e = noise[i];
    float4 o;
    o.x = __fadd_rn(__fmul_rn(a, x.x), __fmul_rn(b, e.x));
    o.y = __fadd_rn(__fmul_rn(a, x.y), __fmul_rn(b, e.y));
    o.z = __fadd_rn(__fmul_rn(a, x.z), __fmul_rn(b, e.z));
    o.w = __fadd_rn(__fmul_rn(a, x.w), __fmul_rn(b, e.w));
    out[i] = o;
  }
}

// Semantic-gradient guidance update (sgg/sgg.py:18-22 + seg_model/inference.py:39-43), per image:
//   g4 = avg_pool(grad, pool) ; mag = sqrt(sum_c (g4_c*std_c)^2) in float64 ; x = (mu + lam*sigz*mag) + sigz
// grad is [B,3,Hs,Ws] fp32 (Hs = pool*h); mu, sigz, out are [B,3,h,w] fp32.
__global__ void __launch_bounds__(256)
sgg_update_kernel(const float* __restrict__ grad, const float* __restrict__ mu, const float* __restrict__ sigz,
                  float* __restrict__ out, float* __restrict__ mag_out, int B, int h, int w, int pool, float lam) {
  pdl_prologue();
  const size_t hw = static_cast<size_t>(h) * w;
  const size_t total = hw * B;
  const int Ws = w * pool, Hs = h * pool;
  const double stdv[3] = {0.229, 0.224, 0.225};
  const float area = static_cast<float>(pool * pool);
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int b = static_cast<int>(i / hw);
    const int y = static_cast<int>((i % hw) / w), x = static_cast<int>(i % w);
    double acc = 0.0;
    for (int c = 0; c < 3; ++c) {
      const float* gp = grad + ((static_cast<size_t>(b) * 3 + c) * Hs + static_cast<size_t>(y) * pool) * Ws +
                        static_cast<size_t>(x) * pool;
      float s = 0.f;  // F.avg_pool2d accumulates in fp32 then scales
      for (int dy = 0; dy < pool; ++dy)
        for (int dx = 0; dx < pool; ++dx) s = __fadd_rn(s, gp[static_cast<size_t>(dy) * Ws + dx]);
      const double g = __dmul_rn(static_cast<double>(__fdiv_rn(s, area)), stdv[c]);
      acc = __dadd_rn(acc, __dmul_rn(g, g));  // no FMA contraction: numpy squares, then sums
    }
    const double mag = sqrt(acc);
    if (mag_out) mag_out[i] = static_cast<float>(mag);
    for (int c = 0; c < 3; ++c) {
      const size_t o = (static_cast<size_t>(b) * 3 + c) * hw + static_cast<size_t>(y) * w + x;
      const double sz = static_cast<double>(sigz[o]);
      // reference: (mu + ((lam*sigma) * mag)) + sigma, evaluated in float64 after promotion (D7)
      const double lam_s = static_cast<double>(__fmul_rn(lam, sigz[o]));
      out[o] = static_cast<float>(__dadd_rn(__dadd_rn(static_cast<double>(mu[o]), __dmul_rn(lam_s, mag)), sz));
    }
  }
}

// Local class guidance (sgg/sgg.py:39-58, repaired final sum, see DESIGN.md section 4):
//   prepare: for class c, x_m[b*NC+c] = sr_xt[b] * (gt[b] == c), gt_m[b*NC+c] = (gt[b] == c) ? c : 0
__global__ void __launch_bounds__(256)
lcg_prepare_kernel(const float* __restrict__ sr, const long long* __restrict__ gt, float* __restrict__ xm,
                   long long* __restrict__ gm, int B, int NC, size_t hw) {
  pdl_prologue();
  const size_t total = static_cast<size_t>(B) * NC * hw;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t p = i % hw;
    const int c = static_cast<int>((i / hw) % NC), b = static_cast<int>(i / (hw * NC));
    const bool on = gt[b * hw + p] == c;
    gm[i] = on ? c : 0;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) xm[((static_cast<size_t>(b) * NC + c) * 3 + ch) * hw + p] = on ? sr[(static_cast<size_t>(b) * 3 + ch) * hw + p] : 0.f;
  }
}
//   combine: xt = (mu + (lam*sigz) * sum_c avg_pool(gt == c) * |g4_c|) + sigz, g4 = pooled gradients [B*NC,3,h,w]
__global__ void __launch_bounds__(256)
lcg_combine_kernel(const float* __restrict__ g4, const long long* __restrict__ gt, const float* __restrict__ mu,
                   const float* __restrict__ sigz, float* __restrict__ out, int B, int NC, int h, int w, int pool, float lam) {
  pdl_prologue();
  const size_t hw = static_cast<size_t>(h) * w;
  const double stdv[3] = {0.229, 0.224, 0.225};
  const int Ws = w * pool;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < hw * B;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int b = static_cast<int>(i / hw), y = static_cast<int>((i % hw) / w), x = static_cast<int>(i % w);
    int cnt[32];
    for (int c = 0; c < NC; ++c) cnt[c] = 0;
    for (int dy = 0; dy < pool; ++dy)
      for (int dx = 0; dx < pool; ++dx) {
        const long long l = gt[(static_cast<size_t>(b) * h * pool + y * pool + dy) * Ws + x * pool + dx];
        if (l >= 0 && l < NC) ++cnt[l];
      }
    double acc = 0.0;
    for (int c = 0; c < NC; ++c) {
      if (!cnt[c]) continue;
      double m2 = 0.0;
      for (int ch = 0; ch < 3; ++ch) {
        const double g = __dmul_rn(static_cast<double>(g4[((static_cast<size_t>(b) * NC + c) * 3 + ch) * hw + static_cast<size_t>(y) * w + x]), stdv[ch]);
        m2 = __dadd_rn(m2, __dmul_rn(g, g));
      }
      const double frac = static_cast<double>(__fdiv_rn(static_cast<float>(cnt[c]), static_cast<float>(pool * pool)));
      acc = __dadd_rn(acc, __dmul_rn(frac, sqrt(m2)));
    }
    for (int ch = 0; ch < 3; ++ch) {
      const size_t o = (static_cast<size_t>(b) * 3 + ch) * hw + static_cast<size_t>(y) * w + x;
      const double lam_s = static_cast<double>(__fmul_rn(lam, sigz[o]));
      out[o] = static_cast<float>(__dadd_rn(__dadd_rn(static_cast<double>(mu[o]), __dmul_rn(lam_s, acc)), static_cast<double>(sigz[o])));
    }
  }
}

inline int grid_for(size_t n_items) {
  const size_t blocks = (n_items + 255) / 256;
  const size_t cap = static_cast<size_t>(num_sms()) * 8;
  return static_cast<int>(blocks < cap ? (blocks ? blocks : 1) : cap);
}

}  // namespace

int ddpm_step(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
              size_t n_per_sample, int B, float beta, float s, float sqrt_alpha, float sigma, cudaStream_t st) {
  WC_REQUIRE(n_per_sample % 4 == 0, "elements per sample must be a multiple of 4");
  StepCoef c{beta, s, sqrt_alpha, sigma};
  const size_t n4 = n_per_sample / 4;
  ProfScope prof(kProfScheduler, st, 4.0 * n_per_sample * B * (2 + (z ? 1 : 0) + (out ? 1 : 0) + (mean_out ? 1 : 0) + (sigz_out ? 1 : 0)));
  launch_k(ddpm_step_kernel<0>, grid_for(n4 * B), 256, 0, st, 
      reinterpret_cast<const float4*>(xt), reinterpret_cast<const float4*>(eps), reinterpret_cast<const float4*>(z),
      reinterpret_cast<float4*>(out), reinterpret_cast<float4*>(mean_out), reinterpret_cast<float4*>(sigz_out), n4, B,
      c, nullptr, nullptr, nullptr, nullptr, 1);
  WC_LAUNCH_CHECK();
  return 0;
}

int ddpm_step_indexed(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                      size_t n_per_sample, int B, const float* coef_tables, const long long* t_dev, int T, cudaStream_t st) {
  WC_REQUIRE(n_per_sample % 4 == 0, "elements per sample must be a multiple of 4");
  WC_REQUIRE(T >= 1 && coef_tables && t_dev, "ddpm_step_indexed: tables and the device timestep are required");
  StepCoef c{0, 1, 1, 0};
  const size_t n4 = n_per_sample / 4;
  ProfScope prof(kProfScheduler, st, 4.0 * n_per_sample * B * (2 + (z ? 1 : 0) + (out ? 1 : 0) + (mean_out ? 1 : 0) + (sigz_out ? 1 : 0)));
  launch_k(ddpm_step_kernel<2>, grid_for(n4 * B), 256, 0, st, 
      reinterpret_cast<const float4*>(xt), reinterpret_cast<const float4*>(eps), reinterpret_cast<const float4*>(z),
      reinterpret_cast<float4*>(out), reinterpret_cast<float4*>(mean_out), reinterpret_cast<float4*>(sigz_out), n4, B,
      c, coef_tables, nullptr, nullptr, t_dev, T);
  WC_LAUNCH_CHECK();
  return 0;
}

int ddim_step(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
              size_t n_per_sample, int B, float a_t, float s_t, float a_prev, float d, float sigma, cudaStream_t st) {
  WC_REQUIRE(n_per_sample % 4 == 0, "elements per sample must be a multiple of 4");
  DdimCoef c{a_t, s_t, a_prev, d, sigma};
  const size_t n4 = n_per_sample / 4;
  ProfScope prof(kProfScheduler, st, 4.0 * n_per_sample * B * (2 + (z ? 1 : 0) + (out ? 1 : 0) + (mean_out ? 1 : 0) + (sigz_out ? 1 : 0)));
  launch_k(ddim_step_kernel<0>, grid_for(n4 * B), 256, 0, st,
      reinterpret_cast<const float4*>(xt), reinterpret_cast<const float4*>(eps), reinterpret_cast<const float4*>(z),
      reinterpret_cast<float4*>(out), reinterpret_cast<float4*>(mean_out), reinterpret_cast<float4*>(sigz_out), n4, B,
      c, nullptr, nullptr, 1);
  WC_LAUNCH_CHECK();
  return 0;
}

int ddim_step_indexed(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                      size_t n_per_sample, int B, const float* coef_tables, const long long* t_dev, int T, cudaStream_t st) {
  WC_REQUIRE(n_per_sample % 4 == 0, "elements per sample must be a multiple of 4");
  WC_REQUIRE(T >= 1 && coef_tables && t_dev, "ddim_step_indexed: tables and the device timestep are required");
  DdimCoef c{1, 0, 1, 0, 0};
  const size_t n4 = n_per_sample / 4;
  ProfScope prof(kProfScheduler, st, 4.0 * n_per_sample * B * (2 + (z ? 1 : 0) + (out ? 1 : 0) + (mean_out ? 1 : 0) + (sigz_out ? 1 : 0)));
  launch_k(ddim_step_kernel<2>, grid_for(n4 * B), 256, 0, st,
      reinterpret_cast<const float4*>(xt), reinterpret_cast<const float4*>(eps), reinterpret_cast<const float4*>(z),
      reinterpret_cast<float4*>(out), reinterpret_cast<float4*>(mean_out), reinterpret_cast<float4*>(sigz_out), n4, B,
      c, coef_tables, t_dev, T);
  WC_LAUNCH_CHECK();
  return 0;
}

int ddpm_step_batched(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                      size_t n_per_sample, int B, const float* betas, const float* alphas, const float* sqrt_1m_acp,
                      const long long* t, int T, cudaStream_t st) {
  WC_REQUIRE(n_per_sample % 4 == 0, "elements per sample must be a multiple of 4");
  WC_REQUIRE(T >= 1, "num_timesteps must be positive");
  StepCoef c{0, 1, 1, 0};
  const size_t n4 = n_per_sample / 4;
  launch_k(ddpm_step_kernel<1>, grid_for(n4 * B), 256, 0, st, 
      reinterpret_cast<const float4*>(xt), reinterpret_cast<const float4*>(eps), reinterpret_cast<const float4*>(z),
      reinterpret_cast<float4*>(out), reinterpret_cast<float4*>(mean_out), reinterpret_cast<float4*>(sigz_out), n4, B,
      c, betas, alphas, sqrt_1m_acp, t, T);
  WC_LAUNCH_CHECK();
  return 0;
}

int add_noise(const float* x0, const float* noise, float* out, size_t n_per_sample, int B, const float* sqrt_acp,
              const float* sqrt_1m_acp, const long long* t, int T, cudaStream_t st) {
  WC_REQUIRE(n_per_sample % 4 == 0, "elements per sample must be a multiple of 4");
  WC_REQUIRE(T >= 1, "num_timesteps must be positive");
  const size_t n4 = n_per_sample / 4;
  launch_k(add_noise_kernel, grid_for(n4 * B), 256, 0, st, reinterpret_cast<const float4*>(x0),
                                                      reinterpret_cast<const float4*>(noise),
                                                      reinterpret_cast<float4*>(out), n4, B, sqrt_acp, sqrt_1m_acp, t, T);
  WC_LAUNCH_CHECK();
  return 0;
}

int lcg_prepare(const float* sr, const long long* gt, float* xm, long long* gm, int B, int NC, size_t hw, cudaStream_t st) {
  WC_REQUIRE(NC <= 32, "at most 32 classes");
  launch_k(lcg_prepare_kernel, grid_for(static_cast<size_t>(B) * NC * hw), 256, 0, st, sr, gt, xm, gm, B, NC, hw);
  WC_LAUNCH_CHECK();
  return 0;
}
int lcg_combine(const float* g4, const long long* gt, const float* mu, const float* sigz, float* out, int B, int NC, int h,
                int w, int pool, float lam, cudaStream_t st) {
  WC_REQUIRE(NC <= 32, "at most 32 classes");
  launch_k(lcg_combine_kernel, grid_for(static_cast<size_t>(B) * h * w), 256, 0, st, g4, gt, mu, sigz, out, B, NC, h, w, pool, lam);
  WC_LAUNCH_CHECK();
  return 0;
}

int sgg_update(const float* grad, const float* mu, const float* sigz, float* out, float* mag_out, int B, int h, int w,
               int pool, float lam, cudaStream_t st) {
  ProfScope prof(kProfScheduler, st, static_cast<double>(B) * h * w * (12.0 * pool * pool + 36.0));
  launch_k(sgg_update_kernel, grid_for(static_cast<size_t>(B) * h * w), 256, 0, st, grad, mu, sigz, out, mag_out, B, h, w,
                                                                              pool, lam);
  WC_LAUNCH_CHECK();
  return 0;
}

}  // namespace wc
