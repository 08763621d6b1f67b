// agc.cuh — feed-forward AGC (the project's own block: the reference has none).  Spec in include/qpskcuda.h
// ("feed-forward AGC"); tests/agc_oracle.py restates it (AgcScalar, AgcBatch) and the kernels match it bit for bit.
#pragma once
#include "handle.cuh"

namespace qpsk {

constexpr int kAgcMaxWindow = 4096;

// the status a parameter set gets: QPSK_ERR_UNSUPPORTED for the window, QPSK_ERR_RANGE for ref / max_gain
int agc_check_params(int window, float ref, float max_gain);

struct AgcEngine : EngineBase {
  int channels = 1;
  int W = 1;
  float ref = 1.0f, max_gain = 1.0f;
  int cur = 0;                     // which history buffer is live
  DevBuf<float2> d_hist[2];        // [C][W-1]: the last W-1 input samples of each channel (zero before the stream)
  DevBuf<float> d_gain;            // [C] gain of each channel's last output
  int init(int window, float ref_in, float max_gain_in, int channels_in);
  int reset(cudaStream_t s);       // zero history, gains to max_gain
  // x [C][ldx] -> y [C][ldy], n samples per channel, one output per input (output i carries input i - (W-1) of the
  // stream); y must not overlap x.  State advanced at enqueue.
  int process_dev(const float2* x, int64_t n, int64_t ldx, float2* y, int64_t ldy, cudaStream_t s);
};

}  // namespace qpsk
