"""Down-converter bank timing on the GPU: qpsk_ddc_process_dev over 2^28 device-resident input samples (2 GiB in: far
beyond L2), K = 1, 8, 64, 256 channels, D = 16, 64, 256 and N = 8D taps, and in the same run the polyphase channelizer at
M = 64 and 256 (N = 8M) for the crossover on a full grid.  CUDA events, warm-up, median of --reps calls; the
device-to-device copy bandwidth and the FP32 FMA peak are measured in the same run, and the card name, power limit and
max SM clock read there too.  Writes one JSON document to stdout (and to --out when given).

  python tools/ddc_probe.py --reps 20 --out profiles/r06_ddc_probe_n1.json
"""
import argparse
import json
import math
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
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--log2-samples", type=int, default=28)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import qpsk_modulator_demodulator_b200 as Q
    if Q.device_count() < 1:
        raise SystemExit("ddc_probe needs a CUDA device")
    Q.set_device(0)
    torch.cuda.set_device(0)
    ts = torch.cuda.Stream()                 # a real stream: NULL would send the work to the handle's own stream
    torch.cuda.set_stream(ts)
    stream = ts.cuda_stream
    n = 1 << args.log2_samples
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": _card(), "build_id": Q._native.build_id(),
           "reps": args.reps, "warmup": args.warmup, "input_samples": n,
           "timing": "CUDA events around one process_dev call over all input samples, median of reps (min, max beside it)",
           "algorithmic": "DDC: bytes 8 + 8K/D per input sample (read, written); flop 8*N*K/D per input sample (N complex taps "
                          "x real-imag complex MAC per output).  PFB: bytes 16, flop 4P + 5*log2(M) per input sample",
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

    def row(ms, lo, hi, flop, nbytes, **key):
        t = ms * 1e-3
        t_bytes = nbytes / (copy_gbs * 1e9)
        t_flop = flop / (peak_tflops * 1e12)
        r = dict(key, ms=ms, min_ms=lo, max_ms=hi, Gsample_s=n / t / 1e9, GB_s=nbytes / t / 1e9, TFLOP_s=flop / t / 1e12,
                 frac_of_copy_bw=t_bytes / t, frac_of_fma_peak=t_flop / t,
                 applicable_roofline="HBM" if t_bytes >= t_flop else "FMA", frac_of_roofline=max(t_bytes, t_flop) / t)
        print(json.dumps(r), file=sys.stderr)
        return r

    rng = np.random.default_rng(1)
    rows = []
    for K in (1, 8, 64, 256):
        freqs = list(rng.uniform(-0.5, 0.5, K))
        for D in (16, 64, 256):
            N = 8 * D
            h = rng.standard_normal(N) / np.sqrt(N)
            bank = Q.DdcBank(h, freqs, D)
            stride = 2 * (n // D)
            y = torch.empty((K, stride), dtype=torch.float32, device="cuda")

            def call():
                bank.process_dev(x.data_ptr(), 2 * n, y.data_ptr(), stride, stream)

            ms, lo, hi = _median_ms(torch, call, args.warmup, args.reps)
            rows.append(row(ms, lo, hi, 8 * N * K / D * n, (8 + 8 * K / D) * n, K=K, D=D, N=N))
            del bank, y
    res["ddc"] = rows

    pfb_rows = []
    y = torch.empty(2 * n, dtype=torch.float32, device="cuda")
    for M in (64, 256):
        P = 8
        pfb = Q.PfbChannelizer(Q.pfb_taps(M, P, 0.5 / M, 60.0), M)

        def call():
            pfb.process_dev(x.data_ptr(), 2 * n, y.data_ptr(), 2 * (n // M), stream)

        ms, lo, hi = _median_ms(torch, call, args.warmup, args.reps)
        pfb_rows.append(row(ms, lo, hi, (4 * P + 5 * math.log2(M)) * n, 16 * n, M=M, P=P))
        # the bank on the same grid spacing (D = M, N = 8M): the smallest measured K at which it takes longer than the PFB
        # takes for all M channels (None: faster at every measured K)
        per_k = {r["K"]: r["ms"] for r in rows if r["D"] == M}
        pfb_rows[-1]["ddc_ms_by_K_at_D_eq_M"] = per_k
        pfb_rows[-1]["ddc_slower_than_pfb_from_K"] = min([k for k, t in per_k.items() if t > ms], default=None)
        del pfb
    res["pfb"] = pfb_rows
    torch.cuda.synchronize()
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
