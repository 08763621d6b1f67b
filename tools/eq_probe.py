"""CMA equalizer timing on the GPU: the cma_eq_kernel alone, and demod_bits_dev at the bench chain geometry with and without
the equalizer stage.  CUDA events, warm-up, median of --reps repetitions; the card name and power limit are read in the
same run.  Writes one JSON document to stdout (and to --out when given).

  python tools/eq_probe.py --reps 20 --out profiles/r03_eq_probe_n1.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

TSC = "11001010011101100100100110101100" + "01110100111001011010001101101001"


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
    ap.add_argument("--symbols", type=int, default=4200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    import qpsk_modulator_demodulator_b200 as Q
    if Q.device_count() < 1:
        raise SystemExit("eq_probe needs a CUDA device")
    Q.set_device(0)
    torch.cuda.set_device(0)
    ts = torch.cuda.Stream()                 # a real stream: NULL would send the work to each handle's own stream
    torch.cuda.set_stream(ts)
    stream = ts.cuda_stream
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": _card(), "build_id": Q._native.build_id(),
           "reps": args.reps, "warmup": args.warmup, "timing": "CUDA events, median of reps (min, max beside it)"}

    # --- the kernel alone: [C][S] symbols in HBM, one launch per repetition (state carries on; the timing does not depend
    # on the values) ------------------------------------------------------------------------------------------------------
    S = args.symbols
    kern = []
    for C in (2048, 16384):
        x = torch.empty((C, 2 * S), dtype=torch.float32, device="cuda")
        Q.fill_uniform_dev(1, 0, 0, x.numel(), x.data_ptr(), stream)
        y = torch.empty_like(x)
        for N in (5, 11, 21):
            e = Q.CmaEqualizer(N, 1e-3, channels=C)
            med, lo, hi = _median_ms(torch, lambda: e.process_dev(x.data_ptr(), y.data_ptr(), 2 * S, 0, 0, 0, stream),
                                     args.warmup, args.reps)
            kern.append({"channels": C, "symbols": S, "n_taps": N, "bytes_in_out": 2 * x.numel() * 4,
                         "ms": med, "ms_min": lo, "ms_max": hi,
                         "gsym_per_s": C * S / (med * 1e-3) / 1e9})
            e.close()
        del x, y
    res["eq_kernel"] = kern
    res["eq_kernel_note"] = ("the same rows every repetition: at 2048 channels in + out (138 MB) exceed the 126 MB L2 only "
                             "slightly, so part of the traffic is served from L2; the kernel is bound by its per-symbol "
                             "recurrence, not by memory")

    # --- demod_bits_dev at the bench chain geometry: sps 2, 21-tap RRC, TSC, 2048 channels of 8400-bit bursts, the
    # benchmark's channel (echo -17 dB at 3 samples, AWGN -40 dBFS, two 1 ppm LOs) ----------------------------------------
    fs, rs, alpha, C, n_payload = 10_000_000, 5_000_000, float(np.float32(0.4)), 2048, 1040
    mod = Q.QPSKModulator(fs, rs, alpha, 10, True, TSC)
    pay = torch.empty((C, n_payload), dtype=torch.uint8, device="cuda")
    Q.fill_bytes_dev(3, 0, C, n_payload, pay.data_ptr(), stream)
    ff = mod.frame_floats(n_payload, b"S", b"E")
    tx = torch.empty((C, ff), dtype=torch.float32, device="cuda")
    mod.modulate_frames_dev(pay.data_ptr(), n_payload, C, b"S", b"E", tx.data_ptr(), ff, stream)
    chan = Q.SimChannel(100e6, 100e6, fs, 1, 1, noise_dbfs=-40.0, mode=1, path_gains_iq=(1.0, 0.0, 0.12, 0.08),
                        path_delays=(0, 3), seed=3, channels=C)
    rx = torch.empty_like(tx)
    chan.apply_dev(tx.data_ptr(), ff, ff, rx.data_ptr(), ff, stream)
    legs = {}
    for name, n_taps in (("no_eq", 0), ("eq_n11", 11)):
        dem = Q.QPSKDeModulator(fs, rs, alpha, 10, tsc=TSC, channels=C)
        if n_taps:
            dem.set_equalizer(n_taps, 0.005)
        cap = dem.bits_bound(ff)
        bits = torch.empty((C, cap), dtype=torch.uint8, device="cuda")
        nb = torch.empty(C, dtype=torch.int64, device="cuda")
        legs[name] = (dem, bits, nb, cap)
    out = {}
    for name, (dem, bits, nb, cap) in legs.items():
        med, lo, hi = _median_ms(torch, lambda: dem.demod_bits_dev(rx.data_ptr(), ff, ff, bits.data_ptr(), cap, nb.data_ptr(), stream),
                                 args.warmup, args.reps)
        out[name] = {"ms": med, "ms_min": lo, "ms_max": hi, "gsample_per_s": C * (ff // 2) / (med * 1e-3) / 1e9}
    out["ratio_eq_over_no_eq_time"] = out["eq_n11"]["ms"] / out["no_eq"]["ms"]
    res["demod_bits_dev"] = {"channels": C, "samples_per_channel": ff // 2, "bits_per_burst": 8 * (n_payload + 2) + len(TSC),
                             "geometry": "sps 2, 21-tap RRC (EXACT mode), TSC, differential, no FLL; EQ mu 0.005", **out}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
