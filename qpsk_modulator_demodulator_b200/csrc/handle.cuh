// handle.cuh — what the block handles (qpsk_fll, qpsk_mm, qpsk_costas, qpsk_eq, qpsk_agc, qpsk_pfb, qpsk_ddc,
// qpsk_resamp, qpsk_conv, qpsk_viterbi, qpsk_rs, qpsk_fsync) share: the engine's device and stream, create / destroy /
// reset, the device-pointer check and the staging of the host entry points.  A handle is a struct with the engine as
// `eng` (and, for the host entry points, its staging DevBufs).
#pragma once
#include <limits.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

namespace qpsk {

// The device an engine was created on and its own stream: host calls and `_dev` calls without a stream run there.
struct EngineBase {
  int device = 0;
  cudaStream_t stream = nullptr;
  ~EngineBase() {
    if (stream) cudaStreamDestroy(stream);
  }
  // the calling thread's device (qpsk_set_device) becomes the engine's, with a new non-blocking stream
  int open() {
    QPSK_TRY(ensure_device());
    device = current_device();
    QPSK_CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    return QPSK_OK;
  }
};

// The start of every create: `out` is checked first and is NULL on every refusal.
template <typename H>
int clear_out(H** out) {
  if (!out) return QPSK_ERR_NULL;
  *out = nullptr;
  return QPSK_OK;
}

// The end of every create, after its own parameter checks: a new handle whose eng.init(args...) succeeded.
template <typename H, typename... A>
int create_handle(H** out, A... args) {
  H* h = new (std::nothrow) H();
  if (!h) return QPSK_ERR_NOMEM;
  const int st = h->eng.init(args...);
  if (st != QPSK_OK) {
    delete h;
    return st;
  }
  *out = h;
  return QPSK_OK;
}

// Work queued on the handle's own stream finishes before its buffers go; destroy(NULL) is QPSK_OK.
template <typename H>
int destroy_handle(H* h) {
  if (h) {
    if (h->eng.stream) cudaStreamSynchronize(h->eng.stream);
    delete h;
  }
  return QPSK_OK;
}

// The state back to what create left, ordered after the handle's queued work and complete on return.
template <typename H>
int reset_handle(H* h) {
  if (!h) return QPSK_ERR_NULL;
  auto& e = h->eng;
  QPSK_TRY(ensure_device(e.device));
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  QPSK_TRY(e.reset(e.stream));
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  return QPSK_OK;
}

// A caller's device pointer the kernels would read or write `a` bytes at a time (a power of two) but that is not
// `a`-byte aligned: the `_dev` calls refuse it with QPSK_ERR_ARG before they launch anything (a misaligned access
// faults and poisons the context).  NULL passes.
inline bool misaligned(const void* p, uintptr_t a = 8) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) != 0; }

// `rows` rows of `width` bytes, `dpitch` / `spitch` bytes apart; one plain copy when both sides are packed
inline cudaError_t copy_rows(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t rows,
                             cudaMemcpyKind kind, cudaStream_t s) {
  if (dpitch == width && spitch == width) return cudaMemcpyAsync(dst, src, width * rows, kind, s);
  return cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, rows, kind, s);
}

// Host rows (`pitch` bytes apart) into `d`, packed, grown to at least one element per row.
template <typename T>
int stage_in(DevBuf<T>& d, const void* src, size_t pitch, size_t width, size_t rows, cudaStream_t s) {
  QPSK_TRY(d.ensure(rows * std::max<size_t>(width / sizeof(T), 1)));
  if (width > 0 && rows > 0) QPSK_CUDA_TRY(copy_rows(d.p, width, src, pitch, width, rows, cudaMemcpyHostToDevice, s));
  return QPSK_OK;
}

// Packed rows of `d` out to the host, `pitch` bytes apart.
template <typename T>
int stage_out(void* dst, size_t pitch, const DevBuf<T>& d, size_t width, size_t rows, cudaStream_t s) {
  if (width > 0 && rows > 0) QPSK_CUDA_TRY(copy_rows(dst, pitch, d.p, width, width, rows, cudaMemcpyDeviceToHost, s));
  return QPSK_OK;
}

// The host form of a block call on the handle's stream: `in_rows` rows of `in_width` bytes from `in` (packed) into
// h->d_in, run(d_in, d_out) (the `_dev` body), `out_rows` rows of `out_width` bytes from h->d_out to `out`, `out_pitch`
// bytes apart; complete on return.
template <typename H, typename Run>
int host_call(H* h, const void* in, size_t in_rows, size_t in_width, void* out, size_t out_pitch, size_t out_rows,
              size_t out_width, Run run) {
  auto& e = h->eng;
  QPSK_TRY(ensure_device(e.device));
  QPSK_TRY(h->d_out.ensure(out_rows * out_width / sizeof(*h->d_out.p)));
  QPSK_TRY(stage_in(h->d_in, in, in_width, in_width, in_rows, e.stream));
  QPSK_TRY(run(h->d_in.p, h->d_out.p));
  QPSK_TRY(stage_out(out, out_pitch, h->d_out, out_width, out_rows, e.stream));
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  return QPSK_OK;
}

// The per-channel symbol counts of a host call that reads [C][stride_floats] symbol rows: each in 0..stride_floats / 2
// (else QPSK_ERR_RANGE); the largest, *max_sym, fits the kernels' int32 counts (else QPSK_ERR_UNSUPPORTED).
inline int host_sym_counts(const int64_t* n_sym, size_t C, int64_t stride_floats, int64_t* max_sym) {
  *max_sym = 0;
  for (size_t c = 0; c < C; ++c) {
    if (n_sym[c] < 0 || n_sym[c] > stride_floats / 2) return QPSK_ERR_RANGE;
    *max_sym = std::max(*max_sym, n_sym[c]);
  }
  return *max_sym > INT_MAX ? QPSK_ERR_UNSUPPORTED : QPSK_OK;
}

// Those rows, max_sym symbols each, into d_sym ([C][max(max_sym, 1)]) and the counts, as int32, into d_n.
inline int upload_syms(DevBuf<float2>& d_sym, DevBuf<int>& d_n, const float* sym, int64_t stride_floats,
                       const int64_t* n_sym, size_t C, int64_t max_sym, cudaStream_t s) {
  QPSK_TRY(stage_in(d_sym, sym, (size_t)stride_floats * 4, (size_t)max_sym * 8, C, s));
  std::vector<int> ns(C);
  for (size_t c = 0; c < C; ++c) ns[c] = (int)n_sym[c];
  return stage_in(d_n, ns.data(), C * sizeof(int), C * sizeof(int), 1, s);
}

}  // namespace qpsk
