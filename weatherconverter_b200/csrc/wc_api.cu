// C ABI (include/wc_b200.h): thin extern "C" wrappers over the kernels' host launchers.
#include "../../include/wc_b200.h"

#include "conv.cuh"
#include "wgrad.cuh"

namespace wc {
int ddpm_step(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
              size_t n_per_sample, int B, float beta, float s, float sqrt_alpha, float sigma, cudaStream_t st);
int ddpm_step_batched(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                      size_t n_per_sample, int B, const float* betas, const float* alphas, const float* sqrt_1m_acp,
                      const long long* t, int T, cudaStream_t st);
int ddpm_step_indexed(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                      size_t n_per_sample, int B, const float* coef_tables, const long long* t_dev, int T, cudaStream_t st);
int ddim_step(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
              size_t n_per_sample, int B, float a_t, float s_t, float a_prev, float d, float sigma, cudaStream_t st);
int ddim_step_indexed(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                      size_t n_per_sample, int B, const float* coef_tables, const long long* t_dev, int T, cudaStream_t st);
int add_noise(const float* x0, const float* noise, float* out, size_t n_per_sample, int B, const float* sqrt_acp,
              const float* sqrt_1m_acp, const long long* t, int T, cudaStream_t st);
int sgg_update(const float* grad, const float* mu, const float* sigz, float* out, float* mag_out, int B, int h, int w,
               int pool, float lam, cudaStream_t st);
int lcg_prepare(const float* sr, const long long* gt, float* xm, long long* gm, int B, int NC, size_t hw, cudaStream_t st);
int lcg_combine(const float* g4, const long long* gt, const float* mu, const float* sigz, float* out, int B, int NC, int h,
                int w, int pool, float lam, cudaStream_t st);
int groupnorm_silu(const __nv_bfloat16* x, __nv_bfloat16* y, int B, int HW, int C, int ld, int ldy, const float* gamma,
                   const float* beta, float eps, int silu, void* workspace, cudaStream_t st);
size_t groupnorm_workspace_bytes(int B);
int conv_small_cin(const float* x, const float* w, const float* bias, const float* scale, const float* shift,
                   __nv_bfloat16* y, int B, int Cin, int H, int W, int Cout, int K, int stride, int pad, int ldy,
                   int relu, cudaStream_t st, const float* prelu = nullptr);
int conv_small_cout(const __nv_bfloat16* x, const float* w, const float* bias, float* y, int B, int H, int W, int Cin,
                    int Cout, int K, int ldx, int tanh_out, cudaStream_t st);
int nchw_f32_to_nhwc_bf16(const float* x, __nv_bfloat16* y, int B, int C, int HW, int ldy, cudaStream_t st);
int nhwc_bf16_to_nchw_f32(const __nv_bfloat16* x, float* y, int B, int C, int HW, int ldx, cudaStream_t st);
void prof_start();
int prof_detail(int cap, int* cls, double* ms, double* work, int* info);
int prof_stop(double* ms, long long* count, double* work);
int attention_forward(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* vt, __nv_bfloat16* out, int B,
                      int heads, int ntok, int hd, int ldo, cudaStream_t st, float* lse = nullptr, float scale = 0.f);
int maxpool_fwd(const __nv_bfloat16* x, __nv_bfloat16* y, uint8_t* idx, int B, int H, int W, int C, cudaStream_t st);
int maxpool_bwd(const __nv_bfloat16* dy, const uint8_t* idx, const __nv_bfloat16* x, __nv_bfloat16* dx, int B, int H,
                int W, int C, cudaStream_t st);
int bilinear_fwd(const __nv_bfloat16* x, __nv_bfloat16* y, int B, int Hi, int Wi, int Ho, int Wo, int C, int ldx, int ldy,
                 cudaStream_t st);
int bilinear_bwd(const __nv_bfloat16* dy, const __nv_bfloat16* mask, __nv_bfloat16* dx, int B, int Hi, int Wi, int Ho,
                 int Wo, int C, int ldy, int ldm, int ldx, cudaStream_t st);
int seg_loss_grad(const float* logits_lo, const long long* labels, int* n_valid, long long* pred, float* dlogit_hi,
                  float* loss, float* logits_hi, int B, int h, int w, int H, int W, int nc, int ignore, cudaStream_t st);
int seg_loss_head_fused(const float* logits_lo, const long long* labels, int* n_valid, long long* pred, float* loss,
                        __nv_bfloat16* dlo, int B, int h, int w, int H, int W, int nc, int cp, int ldo, int ignore, cudaStream_t st);
int logits_bilinear_bwd(const float* dhi, __nv_bfloat16* dlo, int B, int h, int w, int H, int W, int nc, int cp, int ldo,
                        cudaStream_t st);
int conv1_dgrad(const __nv_bfloat16* dz, const float* w, const float* scale, float* dx, int B, int H, int W, int Cout,
                cudaStream_t st);
int groupnorm_silu_bwd(const __nv_bfloat16* x, const __nv_bfloat16* dy, __nv_bfloat16* dx, int B, int HW, int C, int ld,
                       int ldd, int ldo, const float* gamma, const float* beta, float eps, int silu, const void* stats,
                       const __nv_bfloat16* add1, int lda1, const __nv_bfloat16* add2, int lda2, float* dgamma, float* dbeta,
                       void* workspace, cudaStream_t st);
size_t groupnorm_bwd_workspace_bytes(int B, int Cmax);
int colsum(const __nv_bfloat16* x, int B, int HW, int C, int ld, float* out_rows, int ldo, float* out_total, void* workspace,
           cudaStream_t st);
int attention_backward(const __nv_bfloat16* q, const __nv_bfloat16* k, const __nv_bfloat16* v, const __nv_bfloat16* d_o, int ldd,
                       const float* lse, const float* D, __nv_bfloat16* dqkv, int ld3, int B, int heads, int ntok, int hd,
                       cudaStream_t st);
int attn_rowdot(const __nv_bfloat16* o, const __nv_bfloat16* d_o, int ldo, int ldd, int B, int ntok, int heads, int hd, float* D,
                cudaStream_t st);
int mse_loss_grad(const float* pred, const float* target, float* dpred, size_t n, float grad_scale, float* loss, void* scratch,
                  cudaStream_t st);
size_t boundary_wgrad_scratch_bytes();
int boundary_wgrad(const __nv_bfloat16* wide, int ldw, const float* narrow, int B, int H, int W, int sign, float* dw,
                   float* dbias, void* scratch, cudaStream_t st);
int adam_step(float* p, const float* g, float* m, float* v, size_t n, float lr, float beta1, float beta2, float eps, int step,
              float grad_scale, cudaStream_t st);
int time_embedding(const long long* t, int n, int dim, float* out, cudaStream_t st);
int ddpm_grid_u8(const float* x, uint8_t* out, int B, int H, int W, int nrow, int pad, cudaStream_t st);
int postprocess_u8(const float* x, uint8_t* out, int B, int H, int W, const float* mean3, const float* std3, cudaStream_t st);
int label_encode(const uint8_t* lab, int Ws, const int* ytab, const int* xtab, int top, int left, int Hc, int Wc, const long long* lut,
                 int nlut, long long* out, cudaStream_t st);
int resample_u8(const uint8_t* in, uint8_t* tmp, uint8_t* out, int Hin, int Win, int Hout, int Wout, int C, const int* bounds_h,
                const int* kk_h, int ksize_h, const int* bounds_v, const int* kk_v, int ksize_v, cudaStream_t st);
int u8_to_tensor(const uint8_t* in, int Win, int top, int left, int Hc, int Wc, int mode, const float* mean3, const float* std3, float* out,
                 cudaStream_t st);
}  // namespace wc

using namespace wc;
static inline cudaStream_t S(void* s) { return static_cast<cudaStream_t>(s); }
static inline __nv_bfloat16* BF(wc_bf16* p) { return reinterpret_cast<__nv_bfloat16*>(p); }
static inline const __nv_bfloat16* BF(const wc_bf16* p) { return reinterpret_cast<const __nv_bfloat16*>(p); }

extern "C" {

const char* wc_last_error(void) { return last_error_cstr(); }
int wc_abi_version(void) { return 6; }
long long wc_launch_count(void) { return launch_count(); }
void wc_profile_begin(void) { prof_start(); }
int wc_profile_detail(int cap, int* cls, double* ms, double* work, int* info) { return prof_detail(cap, cls, ms, work, info); }
int wc_profile_end(double* ms_by_class, long long* count_by_class, double* work_by_class) {
  return prof_stop(ms_by_class, count_by_class, work_by_class);
}

int wc_ddpm_step(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                 size_t n_per_sample, int batch, float beta, float sqrt_one_minus_acp, float sqrt_alpha, float sigma,
                 void* stream) {
  return ddpm_step(xt, eps, z, out, mean_out, sigz_out, n_per_sample, batch, beta, sqrt_one_minus_acp, sqrt_alpha, sigma,
                   S(stream));
}
int wc_ddpm_step_batched(const float* xt, const float* eps, const float* z, float* out, float* mean_out,
                         float* sigz_out, size_t n_per_sample, int batch, const float* betas, const float* alphas,
                         const float* sqrt_one_minus_acp, const int64_t* t, int num_timesteps, void* stream) {
  return ddpm_step_batched(xt, eps, z, out, mean_out, sigz_out, n_per_sample, batch, betas, alphas, sqrt_one_minus_acp,
                           reinterpret_cast<const long long*>(t), num_timesteps, S(stream));
}
int wc_ddpm_step_indexed(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                         size_t n_per_sample, int batch, const float* coef_tables, const int64_t* t_dev, int num_timesteps,
                         void* stream) {
  return ddpm_step_indexed(xt, eps, z, out, mean_out, sigz_out, n_per_sample, batch, coef_tables,
                           reinterpret_cast<const long long*>(t_dev), num_timesteps, S(stream));
}
int wc_ddim_step(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                 size_t n_per_sample, int batch, float a_t, float s_t, float a_prev, float d, float sigma, void* stream) {
  return ddim_step(xt, eps, z, out, mean_out, sigz_out, n_per_sample, batch, a_t, s_t, a_prev, d, sigma, S(stream));
}
int wc_ddim_step_indexed(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                         size_t n_per_sample, int batch, const float* coef_tables, const int64_t* t_dev, int num_timesteps,
                         void* stream) {
  return ddim_step_indexed(xt, eps, z, out, mean_out, sigz_out, n_per_sample, batch, coef_tables,
                           reinterpret_cast<const long long*>(t_dev), num_timesteps, S(stream));
}
int wc_add_noise(const float* x0, const float* noise, float* out, size_t n_per_sample, int batch,
                 const float* sqrt_acp, const float* sqrt_one_minus_acp, const int64_t* t, int num_timesteps, void* stream) {
  return add_noise(x0, noise, out, n_per_sample, batch, sqrt_acp, sqrt_one_minus_acp,
                   reinterpret_cast<const long long*>(t), num_timesteps, S(stream));
}
int wc_set_time_factor_table(const float* factor_host, int half) { return set_time_factor_table(factor_host, half); }
int wc_time_embedding(const int64_t* t, int n, int dim, float* out, void* stream) {
  return time_embedding(reinterpret_cast<const long long*>(t), n, dim, out, S(stream));
}
int wc_sgg_update(const float* grad, const float* mu, const float* sigz, float* out, float* mag_out, int batch, int h,
                  int w, int pool, float lambda, void* stream) {
  return sgg_update(grad, mu, sigz, out, mag_out, batch, h, w, pool, lambda, S(stream));
}
int wc_lcg_prepare(const float* sr_xt, const int64_t* gt, float* x_masked, int64_t* gt_masked, int batch, int num_classes,
                   int H, int W, void* stream) {
  return lcg_prepare(sr_xt, reinterpret_cast<const long long*>(gt), x_masked, reinterpret_cast<long long*>(gt_masked), batch,
                     num_classes, static_cast<size_t>(H) * W, S(stream));
}
int wc_lcg_combine(const float* pooled_grads, const int64_t* gt, const float* mu, const float* sigz, float* out, int batch,
                   int num_classes, int h, int w, int pool, float lambda, void* stream) {
  return lcg_combine(pooled_grads, reinterpret_cast<const long long*>(gt), mu, sigz, out, batch, num_classes, h, w, pool, lambda,
                     S(stream));
}
size_t wc_groupnorm_workspace_bytes(int batch) { return groupnorm_workspace_bytes(batch); }
int wc_groupnorm_silu(const wc_bf16* x, wc_bf16* y, int batch, int hw, int channels, int ldx, int ldy,
                      const float* gamma, const float* beta, float eps, int silu, void* workspace, void* stream) {
  return groupnorm_silu(BF(x), BF(y), batch, hw, channels, ldx, ldy, gamma, beta, eps, silu, workspace, S(stream));
}

int wc_conv2d(const wc_bf16* x, int batch, int H, int W, int Cin, int ldx, const float* weight, const float* bias,
              int Cout, int K, int stride, int pad, int dil, int transposed, const float* rowbias,
              const wc_bf16* residual, int ldr, const wc_bf16* x2, int Cin2, int ldx2, const float* weight2, int relu,
              wc_bf16* y, int ldy, void* stream) {
  // One-shot convenience entry (unit tests, INTEGRATION.md example): packs weights, runs, frees.  The model-level
  // entries keep their plans and packed weights alive instead.
  cudaStream_t st = S(stream);
  DeviceArena arena;
  ConvOp op;
  Act xin; xin.ptr = const_cast<__nv_bfloat16*>(BF(x)); xin.B = batch; xin.H = H; xin.W = W; xin.C = Cin; xin.ld = ldx;
  const int Ho = transposed ? H * 2 : (stride == 2 ? H / 2 : H), Wo = transposed ? W * 2 : (stride == 2 ? W / 2 : W);
  Act yout; yout.ptr = BF(y); yout.B = batch; yout.H = Ho; yout.W = Wo; yout.C = Cout; yout.ld = ldy;
  Act res; res.ptr = const_cast<__nv_bfloat16*>(BF(residual)); res.B = batch; res.H = Ho; res.W = Wo; res.C = Cout; res.ld = ldr;
  Act x2a; x2a.ptr = const_cast<__nv_bfloat16*>(BF(x2)); x2a.B = batch; x2a.H = H; x2a.W = W; x2a.C = Cin2; x2a.ld = ldx2;
  Epilogue ep; ep.bias = bias; ep.rowbias = rowbias; ep.ldrb = Cout; ep.res = residual ? &res : nullptr; ep.relu = relu;
  OutSpec os; os.mode = kOutNHWC; os.out = yout;
  int e;
  if (transposed) {
    WC_REQUIRE(stride == 2, "transposed convolution supports stride 2");
    WeightSrc w; w.w = weight; w.d0 = Cin; w.d1 = Cout; w.KH = w.KW = K; w.transpose = 1;
    e = build_conv_transposed_s2(&op, &arena, xin, w, K, pad, Cout, ep, os, st);
  } else {
    WeightSrc w; w.w = weight; w.d0 = Cout; w.d1 = Cin; w.KH = w.KW = K;
    WeightSrc w2; w2.w = weight2; w2.d0 = Cout; w2.d1 = Cin2;
    ConvGeom g; g.K = K; g.stride = stride; g.pad = pad; g.dil = dil;
    e = build_conv(&op, &arena, xin, w, g, Cout, x2 ? &x2a : nullptr, x2 ? &w2 : nullptr, ep, os, st);
  }
  if (e) return e;
  if ((e = op.run(st))) return e;
  WC_CHECK_CUDA(cudaStreamSynchronize(st));  // arena (packed weights) is freed on return
  return 0;
}

int wc_conv2d_dgrad(const wc_bf16* dz, int batch, int Ho, int Wo, int Cout, const float* weight, int Cin, int K, int stride,
                    int dil, const wc_bf16* residual, const wc_bf16* mask, wc_bf16* dx, void* stream) {
  // data gradient of y = conv2d(x, weight[Cout,Cin,K,K], stride, pad = dil*(K-1)/2 (stride 1) or K==3 (stride 2))
  cudaStream_t st = S(stream);
  DeviceArena arena;
  ConvOp op;
  const int H = Ho * stride, W = Wo * stride;
  Act g; g.ptr = const_cast<__nv_bfloat16*>(BF(dz)); g.B = batch; g.H = Ho; g.W = Wo; g.C = Cout; g.ld = Cout;
  Act out; out.ptr = BF(dx); out.B = batch; out.H = H; out.W = W; out.C = Cin; out.ld = Cin;
  Act res = out; res.ptr = const_cast<__nv_bfloat16*>(BF(residual));
  Act msk = out; msk.ptr = const_cast<__nv_bfloat16*>(BF(mask));
  WeightSrc w; w.w = weight; w.d0 = Cout; w.d1 = Cin; w.KH = w.KW = K; w.transpose = 1;
  Epilogue ep; ep.res = residual ? &res : nullptr; ep.mask = mask ? &msk : nullptr;
  OutSpec os; os.mode = kOutNHWC; os.out = out;
  int e;
  if (stride == 1) {
    w.flip = 1;
    ConvGeom gg; gg.K = K; gg.stride = 1; gg.dil = dil; gg.pad = dil * (K - 1) / 2;
    e = build_conv(&op, &arena, g, w, gg, Cin, nullptr, nullptr, ep, os, st);
  } else {
    if (!residual) WC_CHECK_CUDA(cudaMemsetAsync(out.ptr, 0, out.pixels() * Cin * 2, st));
    e = build_conv_transposed_s2(&op, &arena, g, w, K, K == 3 ? 1 : 0, Cin, ep, os, st);
  }
  if (e) return e;
  if ((e = op.run(st))) return e;
  WC_CHECK_CUDA(cudaStreamSynchronize(st));
  return 0;
}
int wc_maxpool3x3s2(const wc_bf16* x, wc_bf16* y, uint8_t* idx, int batch, int H, int W, int C, void* stream) {
  return maxpool_fwd(BF(x), BF(y), idx, batch, H, W, C, S(stream));
}
int wc_maxpool3x3s2_bwd(const wc_bf16* dy, const uint8_t* idx, const wc_bf16* x, wc_bf16* dx, int batch, int H, int W, int C,
                        void* stream) {
  return maxpool_bwd(BF(dy), idx, BF(x), BF(dx), batch, H, W, C, S(stream));
}
int wc_bilinear(const wc_bf16* x, wc_bf16* y, int batch, int Hi, int Wi, int Ho, int Wo, int C, void* stream) {
  return bilinear_fwd(BF(x), BF(y), batch, Hi, Wi, Ho, Wo, C, C, C, S(stream));
}
int wc_bilinear_bwd(const wc_bf16* dy, const wc_bf16* mask, wc_bf16* dx, int batch, int Hi, int Wi, int Ho, int Wo, int C,
                    void* stream) {
  return bilinear_bwd(BF(dy), BF(mask), BF(dx), batch, Hi, Wi, Ho, Wo, C, C, C, C, S(stream));
}
int wc_seg_loss_head(const float* logits_lo, const int64_t* labels, int* n_valid_ws, int64_t* pred, float* dlogit_hi,
                     float* loss, float* logits_hi, wc_bf16* dlogit_lo, int batch, int h, int w, int H, int W, void* stream) {
  if (!dlogit_hi) {   // fused path: no full-resolution d-logit tensor (and no up-sampled logits)
    WC_REQUIRE(dlogit_lo && !logits_hi, "wc_seg_loss_head without dlogit_hi needs dlogit_lo and no logits_hi");
    const int e = seg_loss_head_fused(logits_lo, reinterpret_cast<const long long*>(labels), n_valid_ws, reinterpret_cast<long long*>(pred), loss,
                                      BF(dlogit_lo), batch, h, w, H, W, 19, 32, 32, 255, S(stream));
    if (e == -1) return fail("wc_seg_loss_head: the fused path needs integer up-sampling factors; pass dlogit_hi for the two-pass path");
    return e;
  }
  if (int e = seg_loss_grad(logits_lo, reinterpret_cast<const long long*>(labels), n_valid_ws,
                            reinterpret_cast<long long*>(pred), dlogit_hi, loss, logits_hi, batch, h, w, H, W, 19, 255, S(stream)))
    return e;
  if (dlogit_lo) return logits_bilinear_bwd(dlogit_hi, BF(dlogit_lo), batch, h, w, H, W, 19, 32, 32, S(stream));
  return 0;
}
int wc_conv1_dgrad(const wc_bf16* dz, const float* weight, const float* scale, float* dx, int batch, int H, int W, void* stream) {
  return conv1_dgrad(BF(dz), weight, scale, dx, batch, H, W, 64, S(stream));
}
int wc_conv_in(const float* x, const float* weight, const float* bias, const float* scale, const float* shift,
               wc_bf16* y, int batch, int H, int W, int Cout, int K, int stride, int pad, int ldy, int relu,
               void* stream) {
  return conv_small_cin(x, weight, bias, scale, shift, BF(y), batch, 3, H, W, Cout, K, stride, pad, ldy, relu, S(stream));
}
int wc_conv_out(const wc_bf16* x, const float* weight, const float* bias, float* y, int batch, int H, int W, int Cin,
                int K, int ldx, int tanh_out, void* stream) {
  return conv_small_cout(BF(x), weight, bias, y, batch, H, W, Cin, 3, K, ldx, tanh_out, S(stream));
}
int wc_nchw_f32_to_nhwc_bf16(const float* x, wc_bf16* y, int batch, int C, int hw, int ldy, void* stream) {
  return nchw_f32_to_nhwc_bf16(x, BF(y), batch, C, hw, ldy, S(stream));
}
int wc_nhwc_bf16_to_nchw_f32(const wc_bf16* x, float* y, int batch, int C, int hw, int ldx, void* stream) {
  return nhwc_bf16_to_nchw_f32(BF(x), y, batch, C, hw, ldx, S(stream));
}
int wc_attention(const wc_bf16* q, const wc_bf16* k, const wc_bf16* vt, wc_bf16* out, int batch, int heads, int ntok,
                 int hd, int ldo, void* stream) {
  return attention_forward(BF(q), BF(k), BF(vt), BF(out), batch, heads, ntok, hd, ldo, S(stream));
}


int wc_attention_scaled(const wc_bf16* q, const wc_bf16* k, const wc_bf16* vt, wc_bf16* out, int batch, int heads, int ntok,
                        int hd, int ldo, float scale, void* stream) {
  return attention_forward(BF(q), BF(k), BF(vt), BF(out), batch, heads, ntok, hd, ldo, S(stream), nullptr, scale);
}

int wc_attention_lse(const wc_bf16* q, const wc_bf16* k, const wc_bf16* vt, wc_bf16* out, float* lse, int batch, int heads,
                     int ntok, int hd, int ldo, void* stream) {
  return attention_forward(BF(q), BF(k), BF(vt), BF(out), batch, heads, ntok, hd, ldo, S(stream), lse);
}

int wc_attention_bwd(const wc_bf16* q, const wc_bf16* k, const wc_bf16* v, const wc_bf16* o, const wc_bf16* d_o, const float* lse,
                     float* d_scratch, wc_bf16* dqkv, int batch, int heads, int ntok, int hd, void* stream) {
  const int C = heads * hd;
  if (int e = attn_rowdot(BF(o), BF(d_o), C, C, batch, ntok, heads, hd, d_scratch, S(stream))) return e;
  return attention_backward(BF(q), BF(k), BF(v), BF(d_o), C, lse, d_scratch, BF(dqkv), 3 * C, batch, heads, ntok, hd, S(stream));
}

int wc_conv2d_wgrad(const wc_bf16* x, const wc_bf16* dy, int batch, int H, int W, int Cin, int Cout, int K, int stride, int pad,
                    int dil, int transposed, const wc_bf16* x2, int Cin2, float* dw, float* dw2, void* stream) {
  cudaStream_t st = S(stream);
  DeviceArena arena;
  float* partial = static_cast<float*>(arena.alloc(kWgradPartialBytes));
  if (!partial) return 1;
  const int Ho = transposed ? H * 2 : H / stride, Wo = transposed ? W * 2 : W / stride;
  Act xa; xa.ptr = const_cast<__nv_bfloat16*>(BF(x)); xa.B = batch; xa.H = H; xa.W = W; xa.C = Cin; xa.ld = Cin;
  Act dya; dya.ptr = const_cast<__nv_bfloat16*>(BF(dy)); dya.B = batch; dya.H = Ho; dya.W = Wo; dya.C = Cout; dya.ld = Cout;
  Act x2a = xa; x2a.ptr = const_cast<__nv_bfloat16*>(BF(x2)); x2a.C = Cin2; x2a.ld = Cin2;
  WgradOp op;
  int e = transposed ? build_convT_wgrad(&op, xa, dya, K, pad, dw, partial)
                     : build_conv_wgrad(&op, xa, dya, K, stride, pad, dil, dw, x2 ? &x2a : nullptr, dw2, partial);
  if (e) return e;
  if ((e = op.run(st))) return e;
  WC_CHECK_CUDA(cudaStreamSynchronize(st));
  return 0;
}

size_t wc_groupnorm_bwd_workspace_bytes(int batch, int channels) { return groupnorm_bwd_workspace_bytes(batch, channels); }
int wc_groupnorm_silu_bwd(const wc_bf16* x, const wc_bf16* dy, wc_bf16* dx, int batch, int hw, int channels, const float* gamma,
                          const float* beta, float eps, int silu, const void* fwd_workspace, const wc_bf16* add1,
                          const wc_bf16* add2, float* dgamma, float* dbeta, void* workspace, void* stream) {
  return groupnorm_silu_bwd(BF(x), BF(dy), BF(dx), batch, hw, channels, channels, channels, channels, gamma, beta, eps, silu,
                            fwd_workspace, BF(add1), channels, BF(add2), channels, dgamma, dbeta, workspace, S(stream));
}
int wc_colsum(const wc_bf16* x, int batch, int hw, int channels, float* out_rows, float* out_total, void* workspace, void* stream) {
  return colsum(BF(x), batch, hw, channels, channels, out_rows, channels, out_total, workspace, S(stream));
}
int wc_mse_loss_grad(const float* pred, const float* target, float* dpred, size_t n, float grad_scale, float* loss, void* scratch,
                     void* stream) {
  return mse_loss_grad(pred, target, dpred, n, grad_scale, loss, scratch, S(stream));
}
size_t wc_boundary_wgrad_scratch_bytes(void) { return boundary_wgrad_scratch_bytes(); }
int wc_boundary_wgrad(const wc_bf16* wide, const float* narrow, int batch, int H, int W, int sign, float* dw, float* dbias,
                      void* scratch, void* stream) {
  return boundary_wgrad(BF(wide), 64, narrow, batch, H, W, sign, dw, dbias, scratch, S(stream));
}
int wc_adam_step(float* p, const float* g, float* m, float* v, size_t n, float lr, float beta1, float beta2, float eps, int step,
                 float grad_scale, void* stream) {
  return adam_step(p, g, m, v, n, lr, beta1, beta2, eps, step, grad_scale, S(stream));
}


int wc_ddpm_grid_u8(const float* x, uint8_t* out, int batch, int H, int W, int nrow, int padding, void* stream) {
  return ddpm_grid_u8(x, out, batch, H, W, nrow, padding, S(stream));
}
int wc_postprocess_u8(const float* x, uint8_t* out, int batch, int H, int W, const float* mean3_host, const float* std3_host, void* stream) {
  return postprocess_u8(x, out, batch, H, W, mean3_host, std3_host, S(stream));
}
int wc_label_encode(const uint8_t* label_ids, int Ws, const int* ytab, const int* xtab, int top, int left, int Hc, int Wc,
                    const int64_t* lut, int nlut, int64_t* out, void* stream) {
  return label_encode(label_ids, Ws, ytab, xtab, top, left, Hc, Wc, reinterpret_cast<const long long*>(lut), nlut,
                      reinterpret_cast<long long*>(out), S(stream));
}
int wc_resample_u8(const uint8_t* in, uint8_t* tmp, uint8_t* out, int Hin, int Win, int Hout, int Wout, int channels, const int* bounds_h,
                   const int* kk_h, int ksize_h, const int* bounds_v, const int* kk_v, int ksize_v, void* stream) {
  return resample_u8(in, tmp, out, Hin, Win, Hout, Wout, channels, bounds_h, kk_h, ksize_h, bounds_v, kk_v, ksize_v, S(stream));
}
int wc_u8_to_tensor(const uint8_t* in, int Win, int top, int left, int Hc, int Wc, int mode, const float* mean3_host, const float* std3_host,
                    float* out, void* stream) {
  return u8_to_tensor(in, Win, top, left, Hc, Wc, mode, mean3_host, std3_host, out, S(stream));
}

}  // extern "C"
