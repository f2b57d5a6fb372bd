// Host-side helpers shared by the C-ABI translation units: error reporting, TMA tensor-map encoding
// through the driver entry point (no link-time dependency on libcuda), tensor views.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <string>

namespace wc {

// Softmax scale of the attention kernels in the log2 domain.  scale > 0: explicit softmax scale; 0: 1/sqrt(head_dim);
// kAttnScalePrescaled (< 0): Q already carries log2(e) * scale (OutSpec::q_scale in the QKV projection) -> exactly 1.
constexpr float kAttnScalePrescaled = -1.f;
inline float attn_scale_log2(float scale, int hd) {
  if (scale < 0.f) return 1.f;
  return 1.4426950408889634f * (scale > 0.f ? scale : 1.f / sqrtf(static_cast<float>(hd)));
}


// ---- error plumbing: every C-ABI entry returns 0 on success, non-zero otherwise; text via wc_last_error()
void set_error(const std::string& msg);
int fail(const std::string& msg);  // sets error, returns 1
#define WC_CHECK_CUDA(expr)                                                                          \
  do {                                                                                               \
    cudaError_t _e = (expr);                                                                         \
    if (_e != cudaSuccess)                                                                           \
      return ::wc::fail(std::string(#expr) + ": " + cudaGetErrorString(_e) + " @" + __FILE__ + ":" + \
                        std::to_string(__LINE__));                                                   \
  } while (0)
#define WC_REQUIRE(cond, msg)                                                                  \
  do {                                                                                         \
    if (!(cond)) return ::wc::fail(std::string("requirement failed: ") + #cond + " - " + msg); \
  } while (0)

// Every kernel launch of the library goes through WC_LAUNCH_CHECK: counts it and surfaces launch errors.
void count_launch();
long long launch_count();
#define WC_LAUNCH_CHECK()               \
  do {                                  \
    ::wc::count_launch();               \
    WC_CHECK_CUDA(cudaGetLastError());  \
  } while (0)

// Optional per-launch timing with CUDA events on the launching stream (bench.py roofline leg).
enum ProfClass : int { kProfIgemm = 0, kProfAttention = 1, kProfGroupNorm = 2, kProfBoundaryConv = 3, kProfScheduler = 4,
                       kProfOther = 5, kProfNumClasses = 8 };
bool profiling_enabled();
void prof_begin_launch(int cls, cudaStream_t st, double work);
void prof_annotate(int a, int b, int c, int d, int e, int f);  // shape info attached to the most recent launch record
void prof_end_launch(cudaStream_t st);
struct ProfScope {
  cudaStream_t st;
  bool on;
  ProfScope(int cls, cudaStream_t s, double work) : st(s), on(profiling_enabled()) {
    if (on) prof_begin_launch(cls, st, work);
  }
  void note(int a, int b = 0, int c = 0, int d = 0, int e = 0, int f = 0) const {
    if (on) prof_annotate(a, b, c, d, e, f);
  }
  ~ProfScope() {
    if (on) prof_end_launch(st);
  }
};

int num_sms();

// ---- programmatic dependent launch (PDL) -----------------------------------------------------------------------------------
// Every kernel of the library is launched through launch_k.  Launches of tcgen05 kernels (KLASS 1) set
// cudaLaunchAttributeProgrammaticStreamSerialization: the kernel may then be scheduled while its predecessor in the stream is still
// draining, and its set-up (block scheduling, shared-memory carve-up, mbarrier init, TMEM allocation, tensor-map prefetch) overlaps
// the predecessor's tail.  Light kernels (KLASS 0) are launched without it.  Measured on B200 (C3, batch 32, graph replay, ms/step):
// no PDL 25.66, tcgen05 kernels only 25.38, light kernels only 25.97, both 26.04 - parked blocks of early-launched light kernels
// next to a running one-CTA-per-SM kernel cost more than the hidden launch gap; a tcgen05 kernel parked next to a light kernel
// hides its mbarrier / TMEM set-up.  (At batch 1, launch-bound, PDL on both classes helped the eager loop: 6.53 -> 5.54 ms/step.)
// Contract: a kernel launched this way executes pdl_prologue() / pdl_wait() (griddepcontrol.wait) BEFORE its first access to
// global memory that any earlier kernel may write or still read; griddepcontrol.launch_dependents lets its own successor in.
// A step is ~440 back-to-back launches (~520 at batch 1), so the per-launch gap is what the small-batch regime is made of.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_prologue() {
  pdl_launch_dependents();
  pdl_wait();
}
template <int KLASS = 0, typename... KArgs, typename... Args>   // KLASS 0: light kernels; 1: tcgen05 kernels (one CTA per SM)
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = KLASS == 1 ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

// Time-embedding factor table (unet_base.py:22-24: 10000 ** (arange(half) / half), fp32): the host evaluates the reference's
// torch expression once and hands the table over, so the embedding's argument t / factor is bit-identical to the reference's.
// time_factor_table(half) returns the device copy for the current device, or nullptr (the kernels then use powf).
int set_time_factor_table(const float* host_table, int half);
const float* time_factor_table(int half);
#ifdef __CUDACC__
__device__ __forceinline__ float time_factor(const float* table, int j, int half) {
  return table ? table[j] : powf(10000.0f, static_cast<float>(j) / static_cast<float>(half));
}
#endif
const char* last_error_cstr();

// NHWC bf16 activation view: element (b,y,x,c) at ptr[((b*H + y)*W + x)*ld + c]; ld >= C lets a view
// address a channel slice of a wider (concatenated) buffer.
struct Act {
  __nv_bfloat16* ptr = nullptr;
  int B = 0, H = 0, W = 0, C = 0, ld = 0;
  size_t pixels() const { return static_cast<size_t>(B) * H * W; }
};

// Encode a tiled bf16 tensor map.  dims/strides are innermost-first; strides in ELEMENTS for dims 1..rank-1
// (dim 0 is contiguous).  swizzle_bytes in {0,32,64,128}.  Returns 0 on success.
int encode_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_elems,
                     const uint32_t* box, uint32_t swizzle_bytes);

}  // namespace wc
