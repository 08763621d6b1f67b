// eq.cuh — blind CMA equalizer, symbol-spaced or fractionally spaced (the project's own block: the reference has none).  Arithmetic spec in
// include/qpskcuda.h ("blind CMA equalizer"); eq.cu is compiled with --fmad=false like the other loop kernels, and the
// two CPU restatements in tests/cma_oracle.py (CmaScalar, CmaBatch) agree with it bit for bit; with an update stride,
// FseScalar and FseBatch in tests/fse_oracle.py.
#pragma once
#include "common.cuh"

namespace qpsk {

constexpr int kEqMaxTaps = 64;
constexpr int kEqMaxSps = 8;

struct EqParams {
  int n_taps;
  float mu, modulus;
  int sps;                   // update stride S: the taps update on stream samples n with n % S == 0 (1 = every sample)
};

// the status a parameter set gets: QPSK_ERR_RANGE for mu / modulus, QPSK_ERR_UNSUPPORTED for the tap count or stride
int eq_check_params(int n_taps, float mu, float modulus, int sps);

struct EqEngine {
  int channels = 1;
  int device = 0;
  EqParams P{};
  DevBuf<float2> d_taps;     // [C][N]
  DevBuf<float2> d_win;      // [C][N]: d_win[c][k] = x_{n-k} after the last symbol n (k = N-1 is never read)
  DevBuf<int> d_drop;        // [C] outputs still to discard (process_dev with drop = true)
  DevBuf<int> d_phase;       // [C] stream sample counter mod sps (allocated for sps > 1 only)
  cudaStream_t stream = nullptr;
  ~EqEngine();
  int init(int n_taps, float mu, float modulus, int sps, int channels_in);
  // taps to the centre spike w[(N-1)/2] = 1, window zeroed, drop counter (N-1)/2, sample counter 0
  int reset(cudaStream_t s);
  // x [C][ldx] -> y [C][ldy].  Channel c takes n = d_n_in ? d_n_in[c] : L symbols (samples for sps > 1).  With `drop`, the first outputs of
  // the stream (the counter of reset()) are discarded once: y receives n - dropped outputs, and d_n_out[c] (when not
  // null) that count.  Without, one output per input.
  int process_dev(const float2* x, float2* y, int64_t L, int64_t ldx, int64_t ldy, const int* d_n_in, int* d_n_out,
                  bool drop, cudaStream_t s);
};

}  // namespace qpsk
