"""Fractionally spaced CMA equalizer timing on the GPU: cma_eq_kernel at update stride S = 2 against the symbol-spaced
kernel (S = 1) at the same tap counts, and demod_bits_dev at the bench chain geometry with the fractionally spaced stage
off and on.  CUDA events, warm-up, median of --reps repetitions; the card name and power limit are read in the same run.
Writes one JSON document to stdout (and to --out when given).

  python tools/fse_probe.py --reps 20 --out profiles/r04_fse_probe_n1.json
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from eq_probe import TSC, _card, _median_ms  # noqa: E402


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
        raise SystemExit("fse_probe needs a CUDA device")
    Q.set_device(0)
    torch.cuda.set_device(0)
    ts = torch.cuda.Stream()                 # a real stream: NULL would send the work to each handle's own stream
    torch.cuda.set_stream(ts)
    stream = ts.cuda_stream
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": _card(), "build_id": Q._native.build_id(),
           "reps": args.reps, "warmup": args.warmup, "timing": "CUDA events, median of reps (min, max beside it)"}

    # --- the kernel alone: [C][sps * symbols] inputs in HBM, one launch per repetition (state carries on; the timing does
    # not depend on the values).  Per symbol: S = 2 takes two input samples and makes one tap update per symbol. ---------
    n_sym = args.symbols
    kern = []
    for C in (2048, 16384):
        for sps in (1, 2):
            L = sps * n_sym
            x = torch.empty((C, 2 * L), dtype=torch.float32, device="cuda")
            Q.fill_uniform_dev(1, 0, 0, x.numel(), x.data_ptr(), stream)
            y = torch.empty_like(x)
            for N in (11, 21, 31):
                e = Q.CmaEqualizer(N, 1e-3, channels=C, sps=sps)
                med, lo, hi = _median_ms(torch, lambda: e.process_dev(x.data_ptr(), y.data_ptr(), 2 * L, 0, 0, 0, stream),
                                         args.warmup, args.reps)
                kern.append({"channels": C, "sps": sps, "n_taps": N, "samples": L, "symbols": n_sym,
                             "bytes_in_out": 2 * x.numel() * 4, "ms": med, "ms_min": lo, "ms_max": hi,
                             "gsample_per_s": C * L / (med * 1e-3) / 1e9, "gsym_per_s": C * n_sym / (med * 1e-3) / 1e9})
                e.close()
            del x, y
    res["eq_kernel"] = kern
    res["eq_kernel_note"] = ("the same rows every repetition; at 2048 channels and S = 2 in + out are 275 MB, past the "
                             "126 MB L2; gsym_per_s counts symbols (inputs / sps)")

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
    for name, fse_taps, eq_taps in (("no_stage", 0, 0), ("fse_n21", 21, 0), ("fse_n21_eq_n11", 21, 11)):
        dem = Q.QPSKDeModulator(fs, rs, alpha, 10, tsc=TSC, channels=C)
        if fse_taps:
            dem.set_fractional_equalizer(fse_taps, 0.005)
        if eq_taps:
            dem.set_equalizer(eq_taps, 0.005)
        cap = dem.bits_bound(ff)
        bits = torch.empty((C, cap), dtype=torch.uint8, device="cuda")
        nb = torch.empty(C, dtype=torch.int64, device="cuda")
        legs[name] = (dem, bits, nb, cap)
    out = {}
    for name, (dem, bits, nb, cap) in legs.items():
        med, lo, hi = _median_ms(torch, lambda: dem.demod_bits_dev(rx.data_ptr(), ff, ff, bits.data_ptr(), cap, nb.data_ptr(), stream),
                                 args.warmup, args.reps)
        out[name] = {"ms": med, "ms_min": lo, "ms_max": hi, "gsample_per_s": C * (ff // 2) / (med * 1e-3) / 1e9}
    out["ratio_fse_over_no_stage_time"] = out["fse_n21"]["ms"] / out["no_stage"]["ms"]
    res["demod_bits_dev"] = {"channels": C, "samples_per_channel": ff // 2, "bits_per_burst": 8 * (n_payload + 2) + len(TSC),
                             "geometry": "sps 2, 21-tap RRC (EXACT mode), TSC, differential, no FLL; FSE mu 0.005, EQ mu 0.005",
                             **out}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
