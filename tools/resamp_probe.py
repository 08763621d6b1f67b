"""Rational resampler timing on the GPU: qpsk_resamp_process_dev over 2^28 device-resident input samples in total (2 GiB
in: far beyond L2), K = 1, 64 and 2048 channels x L/M = 5/8, 8/5, 125/128, 1/4 x P = 8, 16, 32, 64 taps per branch
(N = P*L).  CUDA events, warm-up, median of --reps calls; the device-to-device copy bandwidth and the FP32 FMA peak are
measured in the same run, and the card name, power limit and max SM clock read there too.  Writes one JSON document to
stdout (and to --out when given).

  python tools/resamp_probe.py --reps 10 --out profiles/r08_resamp_probe_n1.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _median_ms(torch, fn, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2], ts[0], ts[-1]


def _card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]], capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--log2-samples", type=int, default=28)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import qpsk_modulator_demodulator_b200 as Q
    if Q.device_count() < 1:
        raise SystemExit("resamp_probe needs a CUDA device")
    Q.set_device(0)
    torch.cuda.set_device(0)
    ts = torch.cuda.Stream()                 # a real stream: NULL would send the work to the handle's own stream
    torch.cuda.set_stream(ts)
    stream = ts.cuda_stream
    total = 1 << args.log2_samples
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": _card(), "build_id": Q._native.build_id(),
           "reps": args.reps, "warmup": args.warmup, "input_samples_total": total,
           "timing": "CUDA events around one process_dev call over all channels' input, median of reps (min, max beside it)",
           "algorithmic": "per output sample: 8 bytes written + 8*M/L bytes read, 4*P flop (P real taps x complex sample "
                          "as two FMA); totals from the call's shapes",
           "applicable_roofline": "the larger of bytes / copy bandwidth and flop / FMA peak: the limit that would bind a kernel "
                                  "running at peak, not a statement that the kernel reaches it",
           "goals": "0.6 of the copy bandwidth where HBM bounds, 0.5 of the FMA peak where FMA bounds"}

    x = torch.empty(2 * total, dtype=torch.float32, device="cuda")
    Q.fill_uniform_dev(1, 0, 0, x.numel(), x.data_ptr(), stream)
    y = torch.empty(2 * total, dtype=torch.float32, device="cuda")
    ms, lo, hi = _median_ms(torch, lambda: y.copy_(x), args.warmup, args.reps)
    copy_gbs = 2 * x.numel() * 4 / (ms * 1e-3) / 1e9
    peak_tflops = Q.measure_fma_peak()
    res["d2d_copy"] = {"bytes": 2 * x.numel() * 4, "ms": ms, "min_ms": lo, "max_ms": hi, "GB_s": copy_gbs}
    res["fma_peak_tflops"] = peak_tflops
    del y

    rng = np.random.default_rng(1)
    rows = []
    for K in (1, 64, 2048):
        n = total // K
        for L, M in ((5, 8), (8, 5), (125, 128), (1, 4)):
            n_out = (n * L - 1) // M + 1
            stride = 2 * n_out
            y = torch.empty((K, stride), dtype=torch.float32, device="cuda")
            for P in (8, 16, 32, 64):
                h = rng.standard_normal(P * L) / np.sqrt(P)
                r = Q.Resampler(h, L, M, K)

                def call():
                    r.process_dev(x.data_ptr(), 2 * n, y.data_ptr(), stride, stream=stream)

                ms, lo, hi = _median_ms(torch, call, args.warmup, args.reps)
                t = ms * 1e-3
                nbytes = 8 * K * (n + n_out)
                flop = 4 * P * K * n_out
                t_bytes = nbytes / (copy_gbs * 1e9)
                t_flop = flop / (peak_tflops * 1e12)
                bound = "HBM" if t_bytes >= t_flop else "FMA"
                row = dict(K=K, L=L, M=M, P=P, N=P * L, ms=ms, min_ms=lo, max_ms=hi, Gout_s=K * n_out / t / 1e9,
                           GB_s=nbytes / t / 1e9, TFLOP_s=flop / t / 1e12, frac_of_copy_bw=t_bytes / t,
                           frac_of_fma_peak=t_flop / t, applicable_roofline=bound, frac_of_roofline=max(t_bytes, t_flop) / t,
                           goal_met=(t_bytes / t >= 0.6) if bound == "HBM" else (t_flop / t >= 0.5))
                print(json.dumps(row), file=sys.stderr)
                rows.append(row)
                del r
            del y
    res["resamp"] = rows
    torch.cuda.synchronize()
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
