"""Polyphase channelizer timing on the GPU: qpsk_pfb_process_dev over 2^28 device-resident input samples (2 GiB in,
2 GiB out: far beyond L2), M = 16, 64, 256, 1024 channels and P = 8, 16, 32 taps per branch.  CUDA events, warm-up,
median of --reps calls; the device-to-device copy bandwidth and the FP32 FMA peak are measured in the same run, and the
card name and power limit read there too.  Writes one JSON document to stdout (and to --out when given).

  python tools/pfb_probe.py --reps 20 --out profiles/r05_pfb_probe_n1.json
"""
import argparse
import json
import math
import os
import subprocess
import sys

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
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--log2-samples", type=int, default=28)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import qpsk_modulator_demodulator_b200 as Q
    if Q.device_count() < 1:
        raise SystemExit("pfb_probe needs a CUDA device")
    Q.set_device(0)
    torch.cuda.set_device(0)
    ts = torch.cuda.Stream()                 # a real stream: NULL would send the work to the handle's own stream
    torch.cuda.set_stream(ts)
    stream = ts.cuda_stream
    n = 1 << args.log2_samples
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": _card(), "build_id": Q._native.build_id(),
           "reps": args.reps, "warmup": args.warmup, "input_samples": n,
           "timing": "CUDA events around one process_dev call over all input samples, median of reps (min, max beside it)",
           "algorithmic": "bytes 16 per input sample (8 read, 8 written); flop 4P + 5*log2(M) per input sample",
           "applicable_roofline": "the larger of bytes / copy bandwidth and flop / FMA peak: the limit that would bind a kernel "
                                  "running at peak, not a statement that the kernel reaches it"}

    x = torch.empty(2 * n, dtype=torch.float32, device="cuda")
    Q.fill_uniform_dev(1, 0, 0, x.numel(), x.data_ptr(), stream)
    y = torch.empty(2 * n, dtype=torch.float32, device="cuda")

    # roofline references measured here: a 2 GiB device-to-device copy (read + write bytes over time), and the FFMA peak
    ms, lo, hi = _median_ms(torch, lambda: y.copy_(x), args.warmup, args.reps)
    copy_gbs = 2 * x.numel() * 4 / (ms * 1e-3) / 1e9
    peak_tflops = Q.measure_fma_peak()
    res["d2d_copy"] = {"bytes": 2 * x.numel() * 4, "ms": ms, "min_ms": lo, "max_ms": hi, "GB_s": copy_gbs}
    res["fma_peak_tflops"] = peak_tflops

    rows = []
    for M in (16, 64, 256, 1024):
        for P in (8, 16, 32):
            h = Q.pfb_taps(M, P, 0.5 / M, 60.0)
            pfb = Q.PfbChannelizer(h, M)
            stride = 2 * (n // M)

            def call():
                pfb.process_dev(x.data_ptr(), 2 * n, y.data_ptr(), stride, stream)

            ms, lo, hi = _median_ms(torch, call, args.warmup, args.reps)
            t = ms * 1e-3
            flop = (4 * P + 5 * math.log2(M)) * n
            t_bytes = 16 * n / (copy_gbs * 1e9)
            t_flop = flop / (peak_tflops * 1e12)
            roofline = "HBM" if t_bytes >= t_flop else "FMA"     # the limit that would bind at peak, not the one reached
            rows.append({"M": M, "P": P, "ms": ms, "min_ms": lo, "max_ms": hi, "Gsample_s": n / t / 1e9,
                         "GB_s": 16 * n / t / 1e9, "TFLOP_s": flop / t / 1e12,
                         "frac_of_copy_bw": t_bytes / t, "frac_of_fma_peak": t_flop / t, "applicable_roofline": roofline,
                         "frac_of_roofline": max(t_bytes, t_flop) / t})
            del pfb
            print(json.dumps(rows[-1]), file=sys.stderr)
    res["pfb"] = rows
    torch.cuda.synchronize()
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
