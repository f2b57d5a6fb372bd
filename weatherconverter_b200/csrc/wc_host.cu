// Error plumbing, device queries and TMA tensor-map encoding (driver entry point fetched at run time so the
// library has no link-time dependency on libcuda and loads on a CPU-only build box).
#include "wc_host.h"

#include <cudaTypedefs.h>
#include <atomic>
#include <cstdlib>
#include <mutex>
#include <vector>

namespace wc {

static thread_local std::string g_last_error;

void set_error(const std::string& msg) { g_last_error = msg; }
int fail(const std::string& msg) {
  g_last_error = msg;
  return 1;
}
const char* last_error_cstr() { return g_last_error.c_str(); }

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
long long launch_count() { return g_launches.load(std::memory_order_relaxed); }

namespace {
struct ProfRec { int cls; cudaEvent_t a, b; double work; int info[6]; };
bool g_prof_on = false;
std::vector<ProfRec> g_prof;
}  // namespace
bool profiling_enabled() { return g_prof_on; }
void prof_begin_launch(int cls, cudaStream_t st, double work) {
  ProfRec r{cls, nullptr, nullptr, work, {0, 0, 0, 0, 0, 0}};
  cudaEventCreate(&r.a);
  cudaEventCreate(&r.b);
  cudaEventRecord(r.a, st);
  g_prof.push_back(r);
}
void prof_end_launch(cudaStream_t st) { cudaEventRecord(g_prof.back().b, st); }
void prof_annotate(int a, int b, int c, int d, int e, int f) {
  if (g_prof.empty()) return;
  int* p = g_prof.back().info;
  p[0] = a; p[1] = b; p[2] = c; p[3] = d; p[4] = e; p[5] = f;
}
// Per-launch detail: fills up to `cap` records {cls, ms, work, info[6]}; returns the number of records available.
int prof_detail(int cap, int* cls, double* ms, double* work, int* info) {
  int n = 0;
  for (auto& r : g_prof) {
    if (n < cap) {
      cudaEventSynchronize(r.b);
      float t = 0;
      cudaEventElapsedTime(&t, r.a, r.b);
      cls[n] = r.cls; ms[n] = t; work[n] = r.work;
      for (int i = 0; i < 6; ++i) info[n * 6 + i] = r.info[i];
    }
    ++n;
  }
  return n;
}
void prof_start() {
  for (auto& r : g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  g_prof.clear();
  g_prof_on = true;
}
int prof_stop(double* ms, long long* count, double* work) {
  g_prof_on = false;
  for (int i = 0; i < kProfNumClasses; ++i) { ms[i] = 0; count[i] = 0; work[i] = 0; }
  for (auto& r : g_prof) {
    if (cudaEventSynchronize(r.b) != cudaSuccess) return fail("profiling: event sync failed");
    float t = 0;
    cudaEventElapsedTime(&t, r.a, r.b);
    ms[r.cls] += t; count[r.cls] += 1; work[r.cls] += r.work;
    cudaEventDestroy(r.a); cudaEventDestroy(r.b);
  }
  g_prof.clear();
  return 0;
}

int num_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
      sms = 148;
  }
  return sms;
}

namespace {
struct TimeFactor { float* dev = nullptr; int half = 0; int device = -1; };
TimeFactor g_tf;
}  // namespace
int set_time_factor_table(const float* host_table, int half) {
  WC_REQUIRE(host_table && half > 0 && half <= 4096, "time factor table: bad size");
  int dev = 0;
  WC_CHECK_CUDA(cudaGetDevice(&dev));
  if (g_tf.dev && (g_tf.half != half || g_tf.device != dev)) {
    cudaFree(g_tf.dev);
    g_tf = TimeFactor{};
  }
  if (!g_tf.dev) WC_CHECK_CUDA(cudaMalloc(&g_tf.dev, sizeof(float) * half));
  WC_CHECK_CUDA(cudaMemcpy(g_tf.dev, host_table, sizeof(float) * half, cudaMemcpyHostToDevice));
  g_tf.half = half;
  g_tf.device = dev;
  return 0;
}
const float* time_factor_table(int half) {
  int dev = 0;
  if (!g_tf.dev || g_tf.half != half || cudaGetDevice(&dev) != cudaSuccess || dev != g_tf.device) return nullptr;
  return g_tf.dev;
}

static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  });
  return fn;
}

int encode_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_elems,
                     const uint32_t* box, uint32_t swizzle_bytes) {
  auto fn = get_encode_fn();
  if (!fn) return fail("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)");
  cuuint64_t gdim[5];
  cuuint64_t gstride[5];
  cuuint32_t bdim[5];
  cuuint32_t estride[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bdim[i] = box[i];
    estride[i] = 1;
    if (i > 0) {
      gstride[i - 1] = strides_elems[i] * 2;  // bytes
      if (gstride[i - 1] % 16 != 0) return fail("TMA global stride must be a multiple of 16 bytes");
    }
  }
  if (reinterpret_cast<uintptr_t>(base) % 16 != 0) return fail("TMA base address must be 16-byte aligned");
  CUtensorMapSwizzle sw = swizzle_bytes == 128  ? CU_TENSOR_MAP_SWIZZLE_128B
                          : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                          : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                                : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, static_cast<cuuint32_t>(rank), const_cast<void*>(base), gdim,
                  gstride, bdim, estride, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r)));
  return 0;
}

}  // namespace wc
