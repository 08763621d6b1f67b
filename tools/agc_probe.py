"""Feed-forward AGC timing on the GPU: qpsk_agc_process_dev over 2^28 device-resident samples (256 rows of 2^20: 2 GiB in,
2 GiB out, far beyond L2) at W = 64, 1024 and 4096, against the device-to-device copy bandwidth measured in the same run
(the AGC moves the same 16 bytes per sample a copy does); then demod_bits_dev at the bench chain geometry with the stage
off and on, without and with the FLL.  CUDA events, warm-up, median of --reps calls; the card name, power limit and max
SM clock are read in the same run.  Writes one JSON document to stdout (and to --out when given).

  python tools/agc_probe.py --reps 20 --out profiles/r07_agc_probe_n1.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
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
    ap.add_argument("--log2-samples", type=int, default=28)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import qpsk_modulator_demodulator_b200 as Q
    if Q.device_count() < 1:
        raise SystemExit("agc_probe needs a CUDA device")
    Q.set_device(0)
    torch.cuda.set_device(0)
    ts = torch.cuda.Stream()                 # a real stream: NULL would send the work to the handle's own stream
    torch.cuda.set_stream(ts)
    stream = ts.cuda_stream
    n = 1 << args.log2_samples
    C = 256
    L = n // C
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": _card(), "build_id": Q._native.build_id(),
           "reps": args.reps, "warmup": args.warmup, "input_samples": n, "rows": C, "samples_per_row": L,
           "timing": "CUDA events around one process_dev call over all samples, median of reps (min, max beside it)",
           "algorithmic": "16 bytes per sample (8 read, 8 written): the copy's traffic; the share is the copy time over the "
                          "AGC time, i.e. the fraction of the measured copy bandwidth reached"}

    x = torch.empty((C, 2 * L), dtype=torch.float32, device="cuda")
    Q.fill_uniform_dev(1, 0, 0, x.numel(), x.data_ptr(), stream)
    y = torch.empty_like(x)
    ms, lo, hi = _median_ms(torch, lambda: y.copy_(x), args.warmup, args.reps)
    copy_gbs = 2 * x.numel() * 4 / (ms * 1e-3) / 1e9
    res["d2d_copy"] = {"bytes": 2 * x.numel() * 4, "ms": ms, "min_ms": lo, "max_ms": hi, "GB_s": copy_gbs}

    rows = []
    for W in (64, 1024, 4096):
        agc = Q.Agc(W, 1.0, 65536.0, C)

        def call():
            agc.process_dev(x.data_ptr(), y.data_ptr(), 2 * L, 2 * L, 2 * L, stream)

        ms, lo, hi = _median_ms(torch, call, args.warmup, args.reps)
        t = ms * 1e-3
        r = {"W": W, "ms": ms, "min_ms": lo, "max_ms": hi, "Gsample_s": n / t / 1e9, "GB_s": 16 * n / t / 1e9,
             "frac_of_copy_bw": 16 * n / (copy_gbs * 1e9) / t}
        print(json.dumps(r), file=sys.stderr)
        rows.append(r)
        del agc
    res["agc"] = rows
    del x, y

    # --- demod_bits_dev at the bench chain geometry: sps 2, 21-tap RRC, TSC, 2048 channels of 8400-bit bursts, the
    # benchmark's channel (echo -17 dB at 3 samples, AWGN -40 dBFS, two 1 ppm LOs) ----------------------------------------
    fs, rs, alpha, Cd, n_payload = 10_000_000, 5_000_000, float(np.float32(0.4)), 2048, 1040
    mod = Q.QPSKModulator(fs, rs, alpha, 10, True, TSC)
    pay = torch.empty((Cd, n_payload), dtype=torch.uint8, device="cuda")
    Q.fill_bytes_dev(3, 0, Cd, n_payload, pay.data_ptr(), stream)
    ff = mod.frame_floats(n_payload, b"S", b"E")
    tx = torch.empty((Cd, ff), dtype=torch.float32, device="cuda")
    mod.modulate_frames_dev(pay.data_ptr(), n_payload, Cd, b"S", b"E", tx.data_ptr(), ff, stream)
    chan = Q.SimChannel(100e6, 100e6, fs, 1, 1, noise_dbfs=-40.0, mode=1, path_gains_iq=(1.0, 0.0, 0.12, 0.08),
                        path_delays=(0, 3), seed=3, channels=Cd)
    rx = torch.empty_like(tx)
    chan.apply_dev(tx.data_ptr(), ff, ff, rx.data_ptr(), ff, stream)
    out = {}
    for fll in (False, True):
        for W in (0, 64):
            dem = Q.QPSKDeModulator(fs, rs, alpha, 10, tsc=TSC, use_fll=fll, channels=Cd)
            if W:
                dem.set_agc(W)
            cap = dem.bits_bound(ff)
            bits = torch.empty((Cd, cap), dtype=torch.uint8, device="cuda")
            nb = torch.empty(Cd, dtype=torch.int64, device="cuda")
            med, lo, hi = _median_ms(torch, lambda: dem.demod_bits_dev(rx.data_ptr(), ff, ff, bits.data_ptr(), cap,
                                                                       nb.data_ptr(), stream), args.warmup, args.reps)
            key = ("fll_" if fll else "") + (f"agc_w{W}" if W else "no_agc")
            out[key] = {"ms": med, "ms_min": lo, "ms_max": hi, "gsample_per_s": Cd * (ff // 2) / (med * 1e-3) / 1e9}
            print(json.dumps({key: out[key]}), file=sys.stderr)
            del dem, bits, nb
    out["ratio_agc_over_no_agc_time"] = out["agc_w64"]["ms"] / out["no_agc"]["ms"]
    out["ratio_agc_over_no_agc_time_fll"] = out["fll_agc_w64"]["ms"] / out["fll_no_agc"]["ms"]
    res["demod_bits_dev"] = {"channels": Cd, "samples_per_channel": ff // 2, "bits_per_burst": 8 * (n_payload + 2) + len(TSC),
                             "geometry": "sps 2, 21-tap RRC (EXACT mode), TSC, differential; AGC ref 1, max_gain 65536",
                             **out}
    torch.cuda.synchronize()
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
