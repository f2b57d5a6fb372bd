/* wc_b200.h - C ABI of the B200-native WeatherConverter hot path (libwc_b200.so).
 *
 * The reference (xXCoffeeColaXc/WeatherConverter) has no FFI: every arithmetic op on its hot path is a PyTorch
 * call.  These entry points are what a maintainer would bind (ctypes, see INTEGRATION.md) to replace those
 * calls.  Conventions:
 *   - every function returns 0 on success, non-zero on failure; wc_last_error() returns the message
 *     (thread-local).  Nothing falls back to the CPU.
 *   - pointers are raw DEVICE pointers unless the name ends in _host; `stream` is a cudaStream_t passed as
 *     void* (NULL = default stream).  All work is stream-ordered; nothing synchronises the device.
 *   - "nchw_f32" tensors use the reference's layout (fp32, NCHW, contiguous); "nhwc_bf16" tensors are the
 *     internal activation layout: element (b,y,x,c) at ptr[((b*H+y)*W+x)*ld + c].
 * Each entry cites the reference code it replaces (paths relative to the reference root).
 */
#ifndef WC_B200_H_
#define WC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef uint16_t wc_bf16; /* raw bfloat16 bits */

const char* wc_last_error(void);
/* ABI version of this header; bumped on any signature change. */
int wc_abi_version(void);
/* Number of kernel launches issued by this library in the calling process so far (all entry points). */
long long wc_launch_count(void);

/* Per-launch CUDA-event timing (bench.py roofline leg).  Between begin and end every kernel launch of the library is
 * bracketed by events on its stream; end synchronises and returns, per class (0 igemm/tcgen05 conv+linear,
 * 1 flash attention, 2 GroupNorm, 3 boundary convs, 4 scheduler, 5 other; arrays of 8), the summed milliseconds,
 * launch counts and algorithmic work (FLOPs for classes 0-1, bytes for 2-4). */
void wc_profile_begin(void);
int wc_profile_end(double* ms_by_class, long long* count_by_class, double* work_by_class);
/* Per-launch records of the current profiling window (call BEFORE wc_profile_end): class, milliseconds, work and six
 * shape integers (igemm: pixels, N, K, N-tile, taps, grid).  Returns the number of records (may exceed cap). */
int wc_profile_detail(int cap, int* cls, double* ms, double* work, int* info);

/* ---- DDPM scheduler (diffusion_model/scheduler/linear_noise_scheduler.py) ------------------------------ */
/* :79-116 sample_prev_timestep + sample_ddpm.py:44.  mean = (xt - beta*eps/s)/sqrt_alpha ; out = mean + sigma*z.
 * z == NULL -> t == 0 branch (out = mean).  mean_out / sigz_out / out may each be NULL.  Bit-exact vs fp32 torch. */
int wc_ddpm_step(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                 size_t n_per_sample, int batch, float beta, float sqrt_one_minus_acp, float sqrt_alpha, float sigma,
                 void* stream);
/* :63-77 sample_prev_timestep2 (batched t [B] int64, sigma^2 = beta_t), tables are the scheduler's fp32 [T] arrays of
 * num_timesteps entries; a t outside [0, num_timesteps) (IndexError in the reference) is clamped to the table. */
int wc_ddpm_step_batched(const float* xt, const float* eps, const float* z, float* out, float* mean_out,
                         float* sigz_out, size_t n_per_sample, int batch, const float* betas, const float* alphas,
                         const float* sqrt_one_minus_acp, const int64_t* t, int num_timesteps, void* stream);
/* The same update as wc_ddpm_step with the scalar timestep READ FROM DEVICE MEMORY (t_dev: one int64) and the four per-step
 * coefficients gathered from coef_tables [4, num_timesteps] fp32 = rows {beta_t, sqrt(1 - acp_t), sqrt(alpha_t), sigma_t}
 * built on the host exactly as the scalar path builds them (bit-identical results).  The launch parameters do not depend on
 * the step, so ONE captured CUDA graph of a reverse step serves every t > 0 (t == 0: z ignored, sigz_out = 0). */
int wc_ddpm_step_indexed(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                         size_t n_per_sample, int batch, const float* coef_tables, const int64_t* t_dev, int num_timesteps,
                         void* stream);
/* DDIM reverse step from timestep tau to the previous timestep tau' of a strided schedule (Song et al., "Denoising Diffusion
 * Implicit Models"; the reference has no DDIM).  Per element, each op rounded to fp32 in this order (no FMA contraction):
 *   x0 = (xt - s_t*eps) / a_t ; mean = a_p*x0 + d*eps ; sigz = sigma*z ; out = mean + sigz
 * with a_t = sqrt(acp_tau), s_t = sqrt(1 - acp_tau), a_prev = sqrt(acp_tau'),
 * sigma = eta*sqrt((1 - acp_tau')/(1 - acp_tau)*(1 - acp_tau/acp_tau')), d = sqrt(max(0, 1 - acp_tau' - sigma^2)); on the
 * final step of a schedule (to x0) a_prev = 1, d = 0, sigma = 0.  z == NULL or sigma == 0: out = mean, sigz_out = 0.
 * n_per_sample % 4 == 0; out / mean_out / sigz_out may each be NULL. */
int wc_ddim_step(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                 size_t n_per_sample, int batch, float a_t, float s_t, float a_prev, float d, float sigma, void* stream);
/* wc_ddim_step with the timestep READ FROM DEVICE MEMORY (t_dev: one int64, clamped to [0, num_timesteps)) and the five
 * coefficients gathered from coef_tables [5, num_timesteps] fp32 = rows {a_t, s_t, a_prev, d, sigma}, column tau holding
 * the step that STARTS at tau (same values as the scalar path -> bit-identical results).  As wc_ddpm_step_indexed, ONE
 * captured CUDA graph of a reverse step serves every step of any schedule. */
int wc_ddim_step_indexed(const float* xt, const float* eps, const float* z, float* out, float* mean_out, float* sigz_out,
                         size_t n_per_sample, int batch, const float* coef_tables, const int64_t* t_dev, int num_timesteps,
                         void* stream);
/* :30-35 add_noise2 / :37-61 add_noise. */
int wc_add_noise(const float* x0, const float* noise, float* out, size_t n_per_sample, int batch,
                 const float* sqrt_acp, const float* sqrt_one_minus_acp, const int64_t* t, int num_timesteps, void* stream);

/* ---- time embedding (diffusion_model/models/unet_base.py:7-30 get_time_embedding) ------------------------ */
/* factor_host [half] fp32 = the reference's `10000 ** (arange(half) / half)` evaluated by torch on the HOST (:22-24); the
 * library keeps a device copy for the current device and every time-embedding kernel (also inside wc_unet_forward /
 * wc_unet_train_forward) divides by it, so t / factor is bit-identical to the reference's.  Not set -> powf on the device.
 * Synchronous (one small cudaMemcpy); call it at model-load time, not inside a captured region. */
int wc_set_time_factor_table(const float* factor_host, int half);
/* out [n, dim] f32 = cat[sin(t/factor), cos(t/factor)] for t int64 [n] (:27-30). */
int wc_time_embedding(const int64_t* t, int n, int dim, float* out, void* stream);

/* ---- guidance update (sgg/sgg.py:18-22, seg_model/inference.py:36-53) ------------------------------------ */
/* grad [B,3,pool*h,pool*w] f32 ; mu, sigz, out [B,3,h,w] f32 ; mag_out [B,h,w] f32 or NULL. */
int wc_sgg_update(const float* grad, const float* mu, const float* sigz, float* out, float* mag_out, int batch, int h,
                  int w, int pool, float lambda, void* stream);

/* Local class guidance, sgg/sgg.py:27-60 (the shipped final sum raises; repaired as documented in DESIGN.md):
 * prepare builds, for every image b and class c, x_masked[b*NC+c] = sr_xt[b]*(gt[b]==c) and gt_masked = gt[b]*(gt[b]==c)
 * (sgg.py:41-45); after wc_seg_infer_pooled on that batch, combine evaluates
 * xt = mu + lambda*sigz*sum_c avg_pool(gt==c)*|pooled_grad_c| + sigz.  pooled_grads f32 [B*NC,3,h,w]; gt int64 [B,pool*h,pool*w]. */
int wc_lcg_prepare(const float* sr_xt, const int64_t* gt, float* x_masked, int64_t* gt_masked, int batch, int num_classes,
                   int H, int W, void* stream);
int wc_lcg_combine(const float* pooled_grads, const int64_t* gt, const float* mu, const float* sigz, float* out, int batch,
                   int num_classes, int h, int w, int pool, float lambda, void* stream);

/* ---- op-level building blocks (unit-test surface; the model-level calls below use the same kernels) ------ */
/* nn.GroupNorm(8, C) [+ nn.SiLU] on NHWC bf16 (unet_base.py:89-90).  workspace >= wc_groupnorm_workspace_bytes. */
size_t wc_groupnorm_workspace_bytes(int batch);
int wc_groupnorm_silu(const wc_bf16* x, wc_bf16* y, int batch, int hw, int channels, int ldx, int ldy,
                      const float* gamma, const float* beta, float eps, int silu, void* workspace, void* stream);
/* nn.Conv2d / nn.ConvTranspose2d on the tcgen05 implicit-GEMM path (unet_base.py:91-95,129,333; resnet.py:90).
 * x nhwc_bf16 [B,H,W,Cin]; weight fp32 PyTorch layout ([Cout,Cin,K,K], or [Cin,Cout,K,K] when transposed != 0);
 * bias fp32 [Cout] or NULL; rowbias fp32 [B,Cout] or NULL (t-embedding add, unet_base.py:148); residual
 * nhwc_bf16 on the output grid or NULL; x2/weight2 (may be NULL): fused 1x1 convolution of a second input
 * (unet_base.py:150).  stride in {1,2}; stride 1 needs 2*pad == dil*(K-1).  Cout must be a multiple of 16. */
int wc_conv2d(const wc_bf16* x, int batch, int H, int W, int Cin, int ldx, const float* weight, const float* bias,
              int Cout, int K, int stride, int pad, int dil, int transposed, const float* rowbias,
              const wc_bf16* residual, int ldr, const wc_bf16* x2, int Cin2, int ldx2, const float* weight2, int relu,
              wc_bf16* y, int ldy, void* stream);
/* 3-channel boundary convolutions on CUDA cores: conv_in (unet_base.py:399) NCHW f32 -> NHWC bf16, optional
 * folded-BN scale/shift + ReLU (resnet.py:142-145); conv_out (unet_base.py:449) NHWC bf16 -> NCHW f32. */
int wc_conv_in(const float* x, const float* weight, const float* bias, const float* scale, const float* shift,
               wc_bf16* y, int batch, int H, int W, int Cout, int K, int stride, int pad, int ldy, int relu,
               void* stream);
int wc_conv_out(const wc_bf16* x, const float* weight, const float* bias, float* y, int batch, int H, int W, int Cin,
                int K, int ldx, int tanh_out, void* stream);
/* Data gradient of nn.Conv2d (what loss.backward() computes for the conv inputs, seg_model/inference.py:141):
 * dz nhwc_bf16 [B,Ho,Wo,Cout], weight fp32 [Cout,Cin,K,K]; dx nhwc_bf16 [B,Ho*stride,Wo*stride,Cin]
 * (+ residual, then zeroed where mask <= 0: the fused ReLU derivative). */
int wc_conv2d_dgrad(const wc_bf16* dz, int batch, int Ho, int Wo, int Cout, const float* weight, int Cin, int K, int stride,
                    int dil, const wc_bf16* residual, const wc_bf16* mask, wc_bf16* dx, void* stream);
/* nn.MaxPool2d(3,2,1) forward (argmax taps saved in idx, one byte per output element) and backward fused with the
 * ReLU derivative of the pooled activation x (resnet.py:144-145). */
int wc_maxpool3x3s2(const wc_bf16* x, wc_bf16* y, uint8_t* idx, int batch, int H, int W, int C, void* stream);
int wc_maxpool3x3s2_bwd(const wc_bf16* dy, const uint8_t* idx, const wc_bf16* x, wc_bf16* dx, int batch, int H, int W, int C,
                        void* stream);
/* F.interpolate(mode='bilinear', align_corners=False) on nhwc_bf16 and its adjoint (optional ReLU mask). */
int wc_bilinear(const wc_bf16* x, wc_bf16* y, int batch, int Hi, int Wi, int Ho, int Wo, int C, void* stream);
int wc_bilinear_bwd(const wc_bf16* dy, const wc_bf16* mask, wc_bf16* dx, int batch, int Hi, int Wi, int Ho, int Wo, int C,
                    void* stream);
/* Loss head (network/utils.py:17 + inference.py:135-141): low-res logits nchw_f32 [B,19,h,w] -> full-res argmax,
 * per-image CE(ignore 255) and d loss / d logits, full-res (f32 class planes [B,19,H,W]) and pulled back to low-res
 * (nhwc_bf16 [B,h,w,32], optional).  n_valid_ws: int[B] scratch.  dlogit_hi == NULL (then logits_hi must be NULL and
 * dlogit_lo given, H and W integer multiples of h and w): pred, loss and dlogit_lo come from one fused kernel and the
 * full-resolution d-logit tensor is never materialised. */
int wc_seg_loss_head(const float* logits_lo, const int64_t* labels, int* n_valid_ws, int64_t* pred, float* dlogit_hi,
                     float* loss, float* logits_hi, wc_bf16* dlogit_lo, int batch, int h, int w, int H, int W, void* stream);
/* Data gradient of the 7x7/2 stem convolution (64 output channels) to the nchw_f32 image (resnet.py:142). */
int wc_conv1_dgrad(const wc_bf16* dz, const float* weight, const float* scale, float* dx, int batch, int H, int W, void* stream);
/* layout converters between the reference boundary layout and the internal one */
int wc_nchw_f32_to_nhwc_bf16(const float* x, wc_bf16* y, int batch, int C, int hw, int ldy, void* stream);
int wc_nhwc_bf16_to_nchw_f32(const wc_bf16* x, float* y, int batch, int C, int hw, int ldx, void* stream);
/* nn.MultiheadAttention core (unet_base.py:159): softmax(q k^T / sqrt(hd)) v per (batch, head), flash-style on
 * tcgen05.  q,k: [B,heads,ntok,hd] bf16; vt: [B,heads,hd,ntok] bf16; out: [B,ntok,heads*hd] bf16 (ldo). */
int wc_attention(const wc_bf16* q, const wc_bf16* k, const wc_bf16* vt, wc_bf16* out, int batch, int heads, int ntok,
                 int hd, int ldo, void* stream);
/* wc_attention with an explicit softmax scale: scale > 0 replaces 1/sqrt(hd); scale == 0 is wc_attention; scale < 0 says that q
 * already carries log2(e)/sqrt(hd) (what the UNet plan's QKV projection stores), so that exp2(q.k) is the softmax numerator. */
int wc_attention_scaled(const wc_bf16* q, const wc_bf16* k, const wc_bf16* vt, wc_bf16* out, int batch, int heads, int ntok,
                        int hd, int ldo, float scale, void* stream);

/* ---- image / label edges of the loop (SURVEY 8f): byte-exact replacements of the host-side PIL / numpy / torchvision
 * steps right before and after the path.  *_host pointers are HOST memory (three floats). ------------------------------ */
/* sample_ddpm.py:47-51: clamp(-1,1), (x+1)/2, make_grid(nrow, padding 2, pad_value 0), ToPILImage -> HWC uint8 grid
 * [(H+pad)*ceil(B/nrow)+pad][(W+pad)*min(nrow,B)+pad][3] (a batch of one image is returned unpadded, as make_grid does). */
int wc_ddpm_grid_u8(const float* x, uint8_t* out, int batch, int H, int W, int nrow, int padding, void* stream);
/* sample_integrated.py:32-37 postprocess: (x*std + mean)*255 -> clamp(0,255) -> uint8, NCHW. */
int wc_postprocess_u8(const float* x, uint8_t* out, int batch, int H, int W, const float* mean3_host, const float* std3_host, void* stream);
/* seg_model/inference.py:75-78,103 + acdc.py:135-138: labelIds uint8 [Hs,Ws] -> NEAREST resize (source row / column index
 * tables ytab[Hr], xtab[Wr], built on the host exactly as Pillow does) -> centre crop (top, left, Hc, Wc) -> id_to_train_id
 * LUT -> int64 [Hc,Wc]. */
int wc_label_encode(const uint8_t* label_ids, int Ws, const int* ytab, const int* xtab, int top, int left, int Hc, int Wc,
                    const int64_t* lut, int nlut, int64_t* out, void* stream);
/* Pillow's 8-bit two-pass resampling (Image.resize with BILINEAR/antialias; translation.py:140): HWC uint8 in -> HWC uint8
 * out; bounds_* [2*n] and kk_* [n*ksize] are the per-output (first tap, tap count) pairs and the 22-bit fixed-point
 * coefficients (weatherconverter_b200/image_io.py builds them as Resample.c does); tmp is [Hin,Wout,C]. */
int wc_resample_u8(const uint8_t* in, uint8_t* tmp, uint8_t* out, int Hin, int Win, int Hout, int Wout, int channels, const int* bounds_h,
                   const int* kk_h, int ksize_h, const int* bounds_v, const int* kk_v, int ksize_v, void* stream);
/* centre crop + ToTensor (+ x*2-1 when mode == 0, translation.py:141-143; + ExtNormalize(mean, std) when mode == 1,
 * seg_model/inference.py:79-80): HWC uint8 [.,Win,3] -> CHW f32 [3,Hc,Wc]. */
int wc_u8_to_tensor(const uint8_t* in, int Win, int top, int left, int Hc, int Wc, int mode, const float* mean3_host, const float* std3_host,
                    float* out, void* stream);

/* ---- training-step building blocks (diffusion_model/train_ddpm.py:95-114: what loss.backward() and
 * optimizer.step() compute; the model-level wc_unet_train_* calls below use the same kernels) ------------------ */
/* wc_attention that also writes lse [B*heads][ntok] (log2-domain log-sum-exp of every softmax row). */
int wc_attention_lse(const wc_bf16* q, const wc_bf16* k, const wc_bf16* vt, wc_bf16* out, float* lse, int batch, int heads,
                     int ntok, int hd, int ldo, void* stream);
/* Backward of the attention core: q,k,v [B,heads,ntok,hd]; o, d_o [B,ntok,heads*hd]; lse from wc_attention_lse;
 * d_scratch fp32 [B*heads*ntok]; dqkv [B,ntok,3*heads*hd] receives dQ | dK | dV. */
int wc_attention_bwd(const wc_bf16* q, const wc_bf16* k, const wc_bf16* v, const wc_bf16* o, const wc_bf16* d_o, const float* lse,
                     float* d_scratch, wc_bf16* dqkv, int batch, int heads, int ntok, int hd, void* stream);
/* Weight gradient of nn.Conv2d (dw [Cout,Cin,K,K]; optional fused 1x1 second input: dw2 [Cout,Cin2,1,1]) or of
 * nn.ConvTranspose2d (transposed != 0, stride 2: dw [Cin,Cout,K,K]); x [B,H,W,Cin], dy on the output grid. */
int wc_conv2d_wgrad(const wc_bf16* x, const wc_bf16* dy, int batch, int H, int W, int Cin, int Cout, int K, int stride, int pad,
                    int dil, int transposed, const wc_bf16* x2, int Cin2, float* dw, float* dw2, void* stream);
/* Backward of wc_groupnorm_silu: fwd_workspace is the workspace the forward call filled; dx = dGN(dy) (+add1) (+add2).
 * ldx, ldd, ldo, lda1, lda2: pixel strides (elements, multiples of 8) of x, dy, dx, add1, add2; add2 may alias dx (in-place
 * accumulation, lda2 == ldo).  dgamma, dbeta fp32 [C] are overwritten. */
size_t wc_groupnorm_bwd_workspace_bytes(int batch, int channels);
int wc_groupnorm_silu_bwd(const wc_bf16* x, const wc_bf16* dy, wc_bf16* dx, int batch, int hw, int channels, int ldx, int ldd,
                          int ldo, const float* gamma, const float* beta, float eps, int silu, const void* fwd_workspace,
                          const wc_bf16* add1, int lda1, const wc_bf16* add2, int lda2, float* dgamma, float* dbeta,
                          void* workspace, void* stream);
/* Column sums of x [B,hw,C] (pixel stride ldx, a multiple of 8): out_rows[b*ldo + c] (may be NULL), out_total [C] (may be
 * NULL): bias / t-embedding gradients.  workspace >= wc_groupnorm_bwd_workspace_bytes(batch, channels). */
int wc_colsum(const wc_bf16* x, int batch, int hw, int channels, int ldx, float* out_rows, int ldo, float* out_total,
              void* workspace, void* stream);
/* nn.MSELoss (train_ddpm.py:107): loss = mean((pred-target)^2), dpred = grad_scale * 2 (pred-target)/n. scratch: 8 KiB. */
int wc_mse_loss_grad(const float* pred, const float* target, float* dpred, size_t n, float grad_scale, float* loss, void* scratch,
                     void* stream);
/* Weight + bias gradient of the 3-channel boundary convs.  sign +1: conv_in (wide = d(conv_in output) nhwc_bf16 64 ch,
 * narrow = input image nchw_f32; dw [64,3,3,3], dbias [64]); sign -1: conv_out (wide = its input, narrow = dpred;
 * dw [3,64,3,3], dbias [3]). */
size_t wc_boundary_wgrad_scratch_bytes(void);
int wc_boundary_wgrad(const wc_bf16* wide, const float* narrow, int batch, int H, int W, int sign, float* dw, float* dbias,
                      void* scratch, void* stream);
/* torch.optim.Adam step (train_ddpm.py:151,113) over flat fp32 buffers; g is multiplied by grad_scale first. */
int wc_adam_step(float* p, const float* g, float* m, float* v, size_t n, float lr, float beta1, float beta2, float eps, int step,
                 float grad_scale, void* stream);

/* ---- model-level: UNet (diffusion_model/models/unet_base.py:372-488) ------------------------------------- */
typedef struct wc_unet wc_unet;
typedef struct {
  int im_channels, im_size, time_emb_dim, num_down_layers, num_mid_layers, num_up_layers, num_heads;
  int n_down_channels;
  int down_channels[8];
  int n_mid_channels;
  int mid_channels[8];
  int down_sample[8];
  int n_attn_resolutions;
  int attn_resolutions[8];
} wc_unet_config;
/* names/ptrs: the reference state_dict (382 fp32 device tensors for config.yaml), read when a binding
   is built and re-packed. */
int wc_unet_create(wc_unet** out, const wc_unet_config* cfg, int n_params, const char* const* names,
                   const float* const* ptrs, const int64_t* numels, void* stream);
void wc_unet_destroy(wc_unet* net);
/* Bytes of activation workspace needed by wc_unet_forward for a [batch,3,H,W] input. */
size_t wc_unet_workspace_bytes(const wc_unet* net, int batch, int H, int W);
/* Unet.forward(x, t) (unet_base.py:451-488): x, out nchw_f32 [B,3,H,W]; t int64 device [n_t], n_t in {1, B}.
 * The first call for a (batch,H,W,workspace) binds tensor maps; later calls with the same binding only launch. */
int wc_unet_forward(wc_unet* net, const float* x, const int64_t* t, int n_t, float* out, int batch, int H, int W,
                    void* workspace, size_t workspace_bytes, void* stream);
/* Algorithmic FLOPs (2*MAC, conv + linear + attention matmuls) of the last bound forward, per call. */
double wc_unet_flops(const wc_unet* net);
/* Kernel launches per forward of the last bound shape. */
int wc_unet_launches(const wc_unet* net);

/* ---- model-level: denoising-loss training step of the UNet (diffusion_model/train_ddpm.py:95-114) -----------------
 * names / params / grads: the reference state_dict names with fp32 device pointers of every parameter and of its
 * gradient buffer (the host keeps them in flat buffers; see weatherconverter_b200/diffusion_model/train_ddpm.py).
 * bind builds the forward / backward launch plans for one [batch,3,H,W] shape in the given workspace.
 * forward: (repack != 0: rebuild the bf16 packed weights from the fp32 parameters first) pred = Unet(x, t) with
 * t int64 [batch]; loss[0] = mean((pred - target)^2) (nn.MSELoss, :107); pred_out may be NULL.  target == NULL: no
 * loss is computed (loss_out may be NULL, pred_out is required) and the backward must be the seeded one.
 * backward(op_begin, op_end): runs that slice of the backward plan (loss.backward(), :108); running all
 * [0, num_backward_ops) fills every gradient buffer (overwrite, like zero_grad + backward).  grad_ready_op(name) is
 * the op count after which that parameter's gradient is final, so the host can overlap bucketed all-reduces. */
typedef struct wc_unet_train wc_unet_train;
int wc_unet_train_create(wc_unet_train** out, const wc_unet_config* cfg, int n_params, const char* const* names,
                         float* const* params, float* const* grads);
void wc_unet_train_destroy(wc_unet_train* net);
size_t wc_unet_train_workspace_bytes(wc_unet_train* net, int batch, int H, int W);
int wc_unet_train_bind(wc_unet_train* net, int batch, int H, int W, void* workspace, size_t workspace_bytes, void* stream);
int wc_unet_train_forward(wc_unet_train* net, const float* x, const int64_t* t, const float* target, float* pred_out,
                          float* loss_out, float grad_scale, int repack, void* stream);
int wc_unet_train_num_backward_ops(const wc_unet_train* net);
int wc_unet_train_backward(wc_unet_train* net, int op_begin, int op_end, void* stream);
/* Backward of the last wc_unet_train_forward seeded with dpred = dL/d(noise_pred), nchw fp32 [B,3,H,W].
 * dx: nchw fp32 [B,3,H,W] receives dL/dx, or NULL.  param_grads == 0: skip every launch whose only product is a
 * parameter gradient.  Parameter gradients (when computed) go to the grads pointers given at create, overwritten. */
int wc_unet_train_backward_seeded(wc_unet_train* net, const float* dpred, float* dx, int param_grads, void* stream);
int wc_unet_train_grad_ready_op(const wc_unet_train* net, const char* name);
double wc_unet_train_flops(const wc_unet_train* net, int backward);

/* ---- model-level: legacy "old model" UNet (diffusion_model/models/old_modules.py:230-360, used by
 * diffusion_model/sample_integrated.py:40-67).  names/ptrs/numels: the reference state_dict (fp32 device tensors, BN
 * running statistics included); the attention in/out projections may be zero-padded per head to a supported head
 * dimension (the padded size is read from numels; see weatherconverter_b200/diffusion_model/models/old_modules.py).
 * forward: x nchw_f32 [B,3,128,128]; t f32 [B] = the noise variance 1 - alpha_bar_t the reference passes as
 * scheduler.one_minus_cum_prod[t] (sample_integrated.py:60); out nchw_f32 [B,3,128,128]. */
typedef struct wc_legacy_unet wc_legacy_unet;
int wc_legacy_unet_create(wc_legacy_unet** out, int n_params, const char* const* names, const float* const* ptrs,
                          const int64_t* numels);
void wc_legacy_unet_destroy(wc_legacy_unet* net);
size_t wc_legacy_unet_workspace_bytes(wc_legacy_unet* net, int batch, int size);
int wc_legacy_unet_forward(wc_legacy_unet* net, const float* x, const float* t, float* out, int batch, int size, void* workspace,
                           size_t workspace_bytes, void* stream);
double wc_legacy_unet_flops(const wc_legacy_unet* net);
int wc_legacy_unet_launches(const wc_legacy_unet* net);

/* ---- model-level: DeepLabV3+ ResNet-50/101 os16 forward + CE + input gradient ------------------------------
 * (seg_model/network/*, seg_model/inference.py:118-152).  blocks_per_layer = {3,4,6,3} (R50) or {3,4,23,3} (R101).
 * names/ptrs: the reference state_dict (fp32 device tensors; num_batches_tracked entries may be omitted). */
typedef struct wc_seg wc_seg;
int wc_seg_create(wc_seg** out, const int* blocks_per_layer, int num_classes, int n_params, const char* const* names,
                  const float* const* ptrs, void* stream);
/* output_stride of the backbone (seg_model/network/modeling.py:34-39): 16 (default; replace_stride_with_dilation [F,F,T], ASPP
 * rates 6/12/18) or 8 (the reference factories' default argument; [F,T,T], rates 12/24/36).  Call before the first infer. */
int wc_seg_set_output_stride(wc_seg* net, int output_stride);
void wc_seg_destroy(wc_seg* net);
size_t wc_seg_workspace_bytes(const wc_seg* net, int batch, int H, int W, int with_grad);
/* infer(): x nchw_f32 [B,3,H,W]; labels int64 [B,H,W] (255 = ignore); outputs (each may be NULL): pred int64 [B,H,W]
 * (argmax), input_grad nchw_f32 [B,3,H,W] (d loss_b / d x_b, loss_b = CE mean over image b's valid pixels; NULL
 * skips the backward pass), loss f32 [B], logits nchw_f32 [B,19,H,W]. */
int wc_seg_infer(wc_seg* net, const float* x, const int64_t* labels, int64_t* pred, float* input_grad, float* loss,
                 float* logits, int batch, int H, int W, void* workspace, size_t workspace_bytes, void* stream);
/* Same, but input_grad is [B,3,H/grad_pool,W/grad_pool] = F.avg_pool2d(d loss / d x, grad_pool) (sgg/sgg.py:18): the
 * pooling is folded into the stem's data-gradient kernel (both are linear), so the full-resolution gradient is
 * never materialised.  grad_pool in {1 (no pooling), 2, 4, 6, 8}. */
int wc_seg_infer_pooled(wc_seg* net, const float* x, const int64_t* labels, int64_t* pred, float* input_grad, float* loss,
                        float* logits, int batch, int H, int W, int grad_pool, void* workspace, size_t workspace_bytes,
                        void* stream);
/* The plan of wc_seg_infer split at its loss head, so that a caller's own loss can drive the data gradient.
 * wc_seg_forward: x nchw_f32 [B,3,H,W] -> logits nchw_f32 [B,19,H,W], bit-identical to wc_seg_infer's logits; no labels, no
 * argmax, no loss.  save_for_backward = 1 binds the with-grad plan (workspace of wc_seg_workspace_bytes(..., with_grad = 1))
 * and keeps the activations the backward reads in the workspace.
 * wc_seg_backward_seeded: dlogits nchw_f32 [B,19,H,W] contiguous (d L / d logits of the saved forward) -> input_grad nchw_f32
 * [B,3,H,W] = d L / d x.  No pixel is treated specially (ignore labels are the loss's business).  Fails unless the last call
 * on this handle was wc_seg_forward(save_for_backward = 1); any infer or forward call in between discards the saved forward,
 * and so does the backward itself. */
int wc_seg_forward(wc_seg* net, const float* x, float* logits, int batch, int H, int W, int save_for_backward, void* workspace,
                   size_t workspace_bytes, void* stream);
int wc_seg_backward_seeded(wc_seg* net, const float* dlogits, float* input_grad, void* stream);
double wc_seg_flops(const wc_seg* net, int backward);
int wc_seg_launches(const wc_seg* net);

/* ---- model-level: Swift-SRGAN generator (srgan_model/models.py:65-92, inference.py:35-39) ------------------- */
typedef struct wc_srgan wc_srgan;
int wc_srgan_create(wc_srgan** out, int num_blocks, int upscale, int n_params, const char* const* names,
                    const float* const* ptrs, void* stream);
void wc_srgan_destroy(wc_srgan* net);
size_t wc_srgan_workspace_bytes(const wc_srgan* net, int batch, int h, int w);
/* Generator.forward: x nchw_f32 [B,3,h,w] -> y nchw_f32 [B,3,upscale*h,upscale*w] in [0,1]. */
int wc_srgan_forward(wc_srgan* net, const float* x, float* y, int batch, int h, int w, void* workspace,
                     size_t workspace_bytes, void* stream);
/* The input gradient of the generator (the parameters are constants; no weight gradient).
 * wc_srgan_forward_saved: the same ops as wc_srgan_forward, the same bits in y, on the with-grad plan (workspace of
 * wc_srgan_grad_workspace_bytes), which also keeps what the backward reads: every PReLU's pre-activation and a copy of y.
 * wc_srgan_backward_seeded: dy nchw_f32 [B,3,upscale*h,upscale*w] contiguous (d L / d y of the saved forward) -> dx nchw_f32
 * [B,3,h,w] = d L / d x.  Fails unless the last call on this handle was wc_srgan_forward_saved; any forward in between
 * discards the saved forward, and so does the backward itself. */
size_t wc_srgan_grad_workspace_bytes(const wc_srgan* net, int batch, int h, int w);
int wc_srgan_forward_saved(wc_srgan* net, const float* x, float* y, int batch, int h, int w, void* workspace,
                           size_t workspace_bytes, void* stream);
int wc_srgan_backward_seeded(wc_srgan* net, const float* dy, float* dx, void* stream);
double wc_srgan_flops(const wc_srgan* net);
int wc_srgan_launches(const wc_srgan* net);

#ifdef __cplusplus
}
#endif
#endif /* WC_B200_H_ */
