// core.cu — library/device plumbing and the host-side filter designers (a1, a7).
#include <math.h>

#include <atomic>
#include <condition_variable>
#include <thread>
#include <vector>
#include <mutex>
#include <set>
#include <utility>

#include "common.cuh"
#include "design.h"

namespace qpsk {

static thread_local std::string tl_cuda_error;
static thread_local int64_t tl_launches = 0;
// Device selection: handles record the ordinal they were created on and every entry point selects it, so the choice below
// only matters at creation time.  qpsk_set_device sets the calling thread's choice and the process-wide default that
// threads which never chose fall back to; two threads driving two GPUs do not see each other's choice.
static std::atomic<int> g_device{0};
static thread_local int tl_device = -1;

void set_cuda_error(cudaError_t e, const char* what, const char* file, int line) {
  char buf[512];
  snprintf(buf, sizeof buf, "%s: %s (%s) at %s:%d", what, cudaGetErrorString(e), cudaGetErrorName(e), file, line);
  tl_cuda_error = buf;
  (void)cudaGetLastError();  // clear the sticky-less error state
}
void set_text_error(const char* text) { tl_cuda_error = text ? text : ""; }
void count_launch(int n) { tl_launches += n; }
int current_device() { return tl_device >= 0 ? tl_device : g_device.load(std::memory_order_relaxed); }

int ensure_device(int dev) {
  if (dev < 0) dev = current_device();
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    if (e != cudaSuccess) set_cuda_error(e, "cudaGetDeviceCount", __FILE__, __LINE__);
    return QPSK_ERR_NO_DEVICE;
  }
  if (dev >= n) return QPSK_ERR_NO_DEVICE;
  QPSK_CUDA_TRY(cudaSetDevice(dev));
  static thread_local int checked_dev = -1;
  if (checked_dev != dev) {
    int major = 0;
    QPSK_CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    if (major != 10) {  // the fatbin holds sm_100a SASS only
      tl_cuda_error = "libqpskcuda is built for sm_100a (B200) only";
      return QPSK_ERR_NO_DEVICE;
    }
    checked_dev = dev;
  }
  return QPSK_OK;
}

int allow_max_dynamic_smem(const void* kernel) {
  static std::mutex mu;
  static std::set<std::pair<const void*, int>> done;
  int dev = 0;
  QPSK_CUDA_TRY(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  if (done.count({kernel, dev})) return QPSK_OK;
  int max_optin = 0;
  QPSK_CUDA_TRY(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  cudaFuncAttributes fa;
  QPSK_CUDA_TRY(cudaFuncGetAttributes(&fa, kernel));
  // the opt-in limit covers static + dynamic shared memory together
  QPSK_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - (int)fa.sharedSizeBytes));
  done.insert({kernel, dev});
  return QPSK_OK;
}

int device_sm_count() {
  static std::atomic<int> cached[64];
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess) d = current_device();
  if (d >= 0 && d < 64) {
    const int c = cached[d].load(std::memory_order_relaxed);
    if (c) return c;
  }
  int n = 148;
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, d);
  if (d >= 0 && d < 64) cached[d].store(n, std::memory_order_relaxed);
  return n;
}

// ---- a1: root-raised-cosine taps (MS/Models/RRC-filter.cs:16-75) ----------------------------
// Same three-branch closed form and unit-energy normalisation; tap count from banker's rounding
// of fs/Rs and of the span (Math.Round).  Compiled without FP contraction so the fp64 results are
// operation-for-operation those of the C# expression tree.
std::vector<double> design_rrc(double span_symbols, double beta, int sample_rate, int symbol_rate) {
  const int sps = (int)nearbyint((double)sample_rate / symbol_rate);
  const int span = (int)nearbyint(span_symbols);
  const int count = span * sps + 1;
  std::vector<double> h((size_t)(count > 0 ? count : 0));
  const int centre = (count - 1) / 2;
  const double tiny = 1e-8;
  for (int n = 0; n < count; ++n) {
    const double t = (n - centre) / (double)sps;  // time in symbols
    double v;
    if (fabs(t) < tiny) {
      v = 1.0 + beta * (4.0 / M_PI - 1.0);
    } else if (fabs(fabs(t) - 1.0 / (4.0 * beta)) < tiny) {
      v = (beta / sqrt(2.0)) * ((1.0 + 2.0 / M_PI) * sin(M_PI / (4.0 * beta)) + (1.0 - 2.0 / M_PI) * cos(M_PI / (4.0 * beta)));
    } else {
      const double numer = sin(M_PI * t * (1.0 - beta)) + 4.0 * beta * t * cos(M_PI * t * (1.0 + beta));
      const double fbt = 4.0 * beta * t;   // Math.Pow(x, 2.0) modelled as the correctly rounded square (DESIGN.md)
      const double denom = M_PI * t * (1.0 - fbt * fbt);
      v = numer / denom;
    }
    h[(size_t)n] = v;
  }
  double e = 0.0;
  for (double v : h) e += v * v;
  const double scale = sqrt(e);
  for (double& v : h) v /= scale;
  return h;
}

std::vector<float> real_taps_as_iq(const std::vector<double>& h) {
  std::vector<float> t(h.size() * 2, 0.0f);
  for (size_t i = 0; i < h.size(); ++i) t[2 * i] = (float)h[i];
  return t;
}

// ---- a7: band-edge filter pair (MS/Models/Band-Edge Filter.cs:132-183) -----------------------
// MathF.Sin/Cos are modelled as the correctly rounded fp32 value (fp64 evaluation rounded once), the
// same definition the device code uses (sincos_f32_exact) — see DESIGN.md "transcendentals".
static inline float cr_sinf(float x) { return (float)sin((double)x); }
static inline float cr_cosf(float x) { return (float)cos((double)x); }
static inline float sinc_pi(float x) {
  if (x == 0.0f) return 1.0f;
  const float a = kPiF * x;
  return cr_sinf(a) / a;
}
void design_band_edge(float sps, float rolloff, int size, std::vector<float>& lower, std::vector<float>& upper) {
  const int centre = (size - 1) / 2;
  std::vector<float> base((size_t)size);
  float total = 0.0f;
  for (int i = 0; i < size; ++i) {
    const float k = (float)(i - centre) / (2.0f * sps);
    const float pos = rolloff * k;
    const float v = sinc_pi(pos - 0.5f) + sinc_pi(pos + 0.5f);
    total += v;
    base[(size_t)i] = v;
  }
  for (float& v : base) v /= total;
  lower.assign((size_t)size * 2, 0.0f);
  upper.assign((size_t)size * 2, 0.0f);
  for (int i = 0; i < size; ++i) {
    const float k = (float)(i - centre) / (2.0f * sps);
    const float ang = -kTwoPiF * (1.0f + rolloff) * k;
    const float re = base[(size_t)i] * cr_cosf(ang);
    const float im = base[(size_t)i] * cr_sinf(ang);
    lower[2 * (size_t)i] = re;
    lower[2 * (size_t)i + 1] = im;
    upper[2 * (size_t)i] = re;
    upper[2 * (size_t)i + 1] = -im;
  }
}

// setupSymbolSync (MS/QPSKDeModulator.cs:39-55)
void mm_gains(double bn, double* kp, double* ki) {
  const double zeta = 1.0 / sqrt(2.0);
  const double wn = ((2.0 * M_PI * bn) / (zeta + 0.25) / zeta);
  const double den = 1.0 + 2.0 * zeta * wn + wn * wn;
  *kp = (4.0 * zeta * wn) / den;
  *ki = (4.0 * wn * wn) / den;
}

// CostasLoopQpsk ctor gains (MS/Models/CostasLoopQpsk.cs:38-44)
void costas_gains(double fs, double bw_hz, double damping, double* alpha, double* beta) {
  const double bw = 2.0 * M_PI * bw_hz / fs;
  const double d = 1.0 + 2.0 * damping * bw + bw * bw;
  *alpha = (4.0 * damping * bw) / d;
  *beta = (4.0 * bw * bw) / d;
}

bool blank_or_null(const char* s) {
  if (!s) return true;
  for (; *s; ++s)
    if (!(*s == ' ' || (*s >= '\t' && *s <= '\r'))) return false;
  return true;
}


// ---- host copy pool -------------------------------------------------------------------------------------------------
bool host_ptr_is_pageable(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();                                  // older runtimes report unknown host memory as an error
    return true;
  }
  return at.type == cudaMemoryTypeUnregistered;
}

namespace {
class HostCopyPool {
 public:
  static HostCopyPool& get() {
    static HostCopyPool pool;
    return pool;
  }
  static constexpr size_t kMinPart = 256 * 1024;         // below that a second thread costs more than it copies
  void copy(char* dst, const char* src, size_t bytes) {
    std::lock_guard<std::mutex> call(call_m_);           // one parallel copy at a time: the pool is per process
    int parts = (int)workers_.size() + 1;
    if ((size_t)parts * kMinPart > bytes) parts = (int)(bytes / kMinPart);
    if (parts <= 1) {
      memcpy(dst, src, bytes);
      return;
    }
    const size_t step = ((bytes + parts - 1) / parts + 63) & ~(size_t)63;
    std::vector<Job> js;
    for (int i = 0; i < parts; ++i) {
      const size_t off = (size_t)i * step;
      if (off >= bytes) break;
      js.push_back({dst + off, src + off, bytes - off < step ? bytes - off : step, 1, 0, 0});
    }
    dispatch(js);
  }
  void copy_rows(char* dst, size_t dpitch, const char* src, size_t spitch, size_t width, size_t rows) {
    std::lock_guard<std::mutex> call(call_m_);
    int parts = (int)workers_.size() + 1;
    if ((size_t)parts * kMinPart > width * rows) parts = (int)(width * rows / kMinPart);
    if (parts < 1) parts = 1;
    const size_t per = (rows + parts - 1) / parts;
    std::vector<Job> js;
    for (size_t r0 = 0; r0 < rows; r0 += per)
      js.push_back({dst + r0 * dpitch, src + r0 * spitch, width, rows - r0 < per ? rows - r0 : per, dpitch, spitch});
    dispatch(js);
  }

 private:
  struct Job {
    char* d;
    const char* s;
    size_t n, rows, dpitch, spitch;
  };
  static void work(const Job& j) {
    for (size_t r = 0; r < j.rows; ++r) memcpy(j.d + r * j.dpitch, j.s + r * j.spitch, j.n);
  }
  // the first job runs on the caller, the rest on the pool; returns when all are done
  void dispatch(const std::vector<Job>& js) {
    if (js.empty()) return;
    {
      std::lock_guard<std::mutex> lk(m_);
      jobs_.assign(js.begin() + 1, js.end());
      next_ = 0;
      pending_ = (int)jobs_.size();
    }
    if (!jobs_.empty()) cv_work_.notify_all();
    work(js[0]);
    std::unique_lock<std::mutex> lk(m_);
    cv_done_.wait(lk, [&] { return pending_ == 0; });
  }
  HostCopyPool() {
    int n = 6;                                           // copy threads, the caller's included
    const int hw = (int)std::thread::hardware_concurrency();
    if (hw > 0 && n > hw) n = hw;
    for (int i = 1; i < n; ++i) workers_.emplace_back([this] { run(); });
  }
  ~HostCopyPool() {
    {
      std::lock_guard<std::mutex> lk(m_);
      stop_ = true;
    }
    cv_work_.notify_all();
    for (std::thread& t : workers_) t.join();
  }
  void run() {
    std::unique_lock<std::mutex> lk(m_);
    for (;;) {
      cv_work_.wait(lk, [&] { return stop_ || next_ < jobs_.size(); });
      if (stop_) return;
      const Job j = jobs_[next_++];
      lk.unlock();
      work(j);
      lk.lock();
      if (--pending_ == 0) cv_done_.notify_all();
    }
  }
  std::vector<std::thread> workers_;
  std::mutex m_, call_m_;
  std::condition_variable cv_work_, cv_done_;
  std::vector<Job> jobs_;
  size_t next_ = 0;
  int pending_ = 0;
  bool stop_ = false;
};
}  // namespace

void host_parallel_copy(void* dst, const void* src, size_t bytes) {
  if (bytes == 0) return;
  HostCopyPool::get().copy((char*)dst, (const char*)src, bytes);
}
void host_parallel_copy_rows(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t rows) {
  if (width == 0 || rows == 0) return;
  HostCopyPool::get().copy_rows((char*)dst, dpitch, (const char*)src, spitch, width, rows);
}

}  // namespace qpsk

using namespace qpsk;

extern "C" {

int qpsk_version(void) { return 200; }

// build stamp (build.py: hash of csrc/, include/qpskcuda.h, the nvcc flags and version); the "QPSK_BUILD_ID=" marker lets
// build.py read it from the file without loading the library
#ifndef QPSK_BUILD_ID_STR
#define QPSK_BUILD_ID_STR "unstamped000000"
#endif
static const char kBuildId[] = "QPSK_BUILD_ID=" QPSK_BUILD_ID_STR;
const char* qpsk_build_id(void) { return kBuildId + 14; }

const char* qpsk_strerror(int s) {
  switch (s) {
    case QPSK_OK: return "ok";
    case QPSK_ERR_NULL: return "null argument (ArgumentNullException)";
    case QPSK_ERR_ARG: return "invalid argument (ArgumentException)";
    case QPSK_ERR_RANGE: return "argument out of range (ArgumentOutOfRangeException)";
    case QPSK_ERR_CUDA: return "CUDA failure";
    case QPSK_ERR_NOMEM: return "out of memory";
    case QPSK_ERR_CAPACITY: return "output buffer too small";
    case QPSK_ERR_UNSUPPORTED: return "unsupported configuration";
    case QPSK_ERR_NO_DEVICE: return "no usable CUDA device (sm_100a required)";
    default: return "unknown status";
  }
}

const char* qpsk_last_cuda_error(void) { return tl_cuda_error.c_str(); }

int qpsk_device_count(int* n) {
  if (!n) return QPSK_ERR_NULL;
  int c = 0;
  cudaError_t e = cudaGetDeviceCount(&c);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    c = 0;
  }
  *n = c;
  return QPSK_OK;
}

int qpsk_set_device(int ordinal) {
  if (ordinal < 0) return QPSK_ERR_RANGE;
  QPSK_TRY(ensure_device(ordinal));
  tl_device = ordinal;
  g_device.store(ordinal, std::memory_order_relaxed);
  return QPSK_OK;
}

int qpsk_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* hbm_bytes) {
  QPSK_TRY(ensure_device());
  cudaDeviceProp p;
  QPSK_CUDA_TRY(cudaGetDeviceProperties(&p, current_device()));
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (cc_major) *cc_major = p.major;
  if (cc_minor) *cc_minor = p.minor;
  if (hbm_bytes) *hbm_bytes = (int64_t)p.totalGlobalMem;
  return QPSK_OK;
}

int qpsk_host_alloc(void** p, int64_t bytes) {
  if (!p) return QPSK_ERR_NULL;
  if (bytes < 0) return QPSK_ERR_RANGE;
  QPSK_TRY(ensure_device());
  QPSK_CUDA_TRY(cudaHostAlloc(p, (size_t)(bytes > 0 ? bytes : 1), cudaHostAllocPortable));
  return QPSK_OK;
}
int qpsk_host_free(void* p) {
  if (!p) return QPSK_OK;
  QPSK_CUDA_TRY(cudaFreeHost(p));
  return QPSK_OK;
}

int qpsk_host_register(void* p, int64_t bytes) {
  if (!p) return QPSK_ERR_NULL;
  if (bytes <= 0) return QPSK_ERR_RANGE;
  QPSK_TRY(ensure_device());
  QPSK_CUDA_TRY(cudaHostRegister(p, (size_t)bytes, cudaHostRegisterPortable));
  return QPSK_OK;
}
int qpsk_host_unregister(void* p) {
  if (!p) return QPSK_OK;
  QPSK_CUDA_TRY(cudaHostUnregister(p));
  return QPSK_OK;
}

int64_t qpsk_launch_count(void) { return tl_launches; }
void qpsk_launch_count_reset(void) { tl_launches = 0; }

int qpsk_rrc_taps(double span_symbols, double beta, int sample_rate, int symbol_rate, double* out, int cap, int* n) {
  if (!n) return QPSK_ERR_NULL;
  if (symbol_rate == 0) return QPSK_ERR_RANGE;
  std::vector<double> h = design_rrc(span_symbols, beta, sample_rate, symbol_rate);
  *n = (int)h.size();
  if (!out) return QPSK_OK;
  if (cap < (int)h.size()) return QPSK_ERR_CAPACITY;
  if (!h.empty()) memcpy(out, h.data(), h.size() * sizeof(double));
  return QPSK_OK;
}

int qpsk_fll_design(float sps, float rolloff, int filter_size, float* lower_iq, float* upper_iq) {
  if (!lower_iq || !upper_iq) return QPSK_ERR_NULL;
  if (!(sps > 0.0f)) return QPSK_ERR_RANGE;
  if (rolloff < 0 || rolloff > 1.0f) return QPSK_ERR_RANGE;
  if (filter_size <= 0) return QPSK_ERR_RANGE;
  std::vector<float> lo, up;
  design_band_edge(sps, rolloff, filter_size, lo, up);
  memcpy(lower_iq, lo.data(), lo.size() * sizeof(float));
  memcpy(upper_iq, up.data(), up.size() * sizeof(float));
  return QPSK_OK;
}

int qpsk_mm_gains_from_bw(double bw, double* kp, double* ki) {
  if (!kp || !ki) return QPSK_ERR_NULL;
  mm_gains(bw, kp, ki);
  return QPSK_OK;
}

}  // extern "C"
