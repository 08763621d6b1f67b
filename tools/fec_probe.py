"""Viterbi decoder probe (csrc/fec.cu): decoder kernel time and decoded bits/s at 1 / 64 / 2048 / 16384 channels of 8192
symbols, as a share of the warp-instruction issue bound; and the coded receive step (constellation_dev + decode +
frame_bits_dev) against the uncoded one (demod_bytes_dev) at the chain shape, 2048 channels of 512-byte payloads.

Issue bound: one warp decodes one channel, and every warp instruction takes one issue slot of one of the 4 schedulers of an
SM, so the least time is  channels * steps * I / (SMs * 4 * f_sm).  I is counted from `cuobjdump -sass` of
viterbi_kernel<true>: the add-compare-select loop (unrolled by 4) issues 124 instructions per 4 steps, 31 per step; per
32-step block the traceback issues 87 per 8 steps of its 64-step walk and 62 per 4 steps of its 32-step read-out, about
1200 per block, 37.5 per step; the per-batch soft-value stage and the block-end reduction add about 3 more.  I = 72.
f_sm is the max SM clock nvidia-smi reports in the same run.  Timing: CUDA events, median of --reps calls after 2 warm-up
calls; inputs are device-resident and written once (the decoder's state advances across calls, as in a stream)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

INSTR_PER_STEP = 72


def smi(q):
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits"], capture_output=True,
                              text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:                                   # noqa: BLE001
        return f"unavailable: {e}"


def timed(fn, reps, torch, stream):
    """median seconds of fn(), every call enqueued on `stream` (a torch.cuda.Stream)"""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import qpsk_modulator_demodulator_b200 as Q
    assert torch.cuda.is_available(), "no CUDA device: nothing to measure"
    props = torch.cuda.get_device_properties(0)
    clk_mhz = smi("clocks.max.sm")
    f_sm = float(clk_mhz) * 1e6
    res = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": smi("power.limit"), "max_sm_clock_mhz": clk_mhz,
           "sms": props.multi_processor_count, "instr_per_step": INSTR_PER_STEP, "decoder": []}
    n_sym = 8192
    stream = torch.cuda.Stream()              # every call on one stream: a NULL stream means each handle's own
    torch.cuda.set_stream(stream)
    s = stream.cuda_stream
    for Cn in (1, 64, 2048, 16384):
        for diff in (False, True):
            g = torch.Generator(device="cuda").manual_seed(Cn)
            sym = (torch.randn((Cn, 2 * n_sym), device="cuda", generator=g) * 0.7).contiguous()
            ns = torch.full((Cn,), n_sym, dtype=torch.int32, device="cuda")
            dec = Q.ViterbiDecoder(Cn, differential=diff)
            cap = dec.bits_bound(n_sym)
            bits = torch.empty((Cn, cap), dtype=torch.uint8, device="cuda")
            nb = torch.empty(Cn, dtype=torch.int64, device="cuda")
            t = timed(lambda: dec.decode_dev(sym.data_ptr(), 2 * n_sym, ns.data_ptr(), bits.data_ptr(), cap, nb.data_ptr(),
                                             s), args.reps, torch, stream)
            bound = Cn * n_sym * INSTR_PER_STEP / (res["sms"] * 4 * f_sm)
            res["decoder"].append({"channels": Cn, "differential": diff, "symbols": n_sym, "kernel_s": t,
                                   "decoded_bits_per_s": Cn * n_sym / t, "issue_bound_s": bound, "share_of_issue_bound": bound / t})
            print(res["decoder"][-1], flush=True)
            dec.close()
            del sym, bits
    # the coded receive step against the uncoded one at the chain shape
    fs, rs, Cn, n_payload = 10_000_000, 5_000_000, 2048, 512
    mod = Q.QPSKModulator(fs, rs, float(np.float32(0.4)), 10, True, None)
    pay = torch.empty((Cn, n_payload), dtype=torch.uint8, device="cuda")
    Q.fill_bytes_dev(5, 0, Cn, n_payload, pay.data_ptr(), s)
    ff = mod.frame_floats(n_payload, b"S", b"E")
    rx = torch.empty((Cn, ff), dtype=torch.float32, device="cuda")
    mod.modulate_frames_dev(pay.data_ptr(), n_payload, Cn, b"S", b"E", rx.data_ptr(), ff, s)
    kw = dict(RrcAlpha=float(np.float32(0.4)), rrcSpan=10, channels=Cn)
    du, dc = Q.QPSKDeModulator(fs, rs, **kw), Q.QPSKDeModulator(fs, rs, **kw)
    d_p = torch.empty((Cn, 1024), dtype=torch.uint8, device="cuda")
    d_np = torch.empty(Cn, dtype=torch.int64, device="cuda")
    ss = dc.bits_bound(ff)
    d_sym = torch.empty((Cn, ss), dtype=torch.float32, device="cuda")
    d_ns = torch.empty(Cn, dtype=torch.int32, device="cuda")
    vit = Q.ViterbiDecoder(Cn, differential=True)
    bc = vit.bits_bound(ss // 2)
    d_b = torch.empty((Cn, bc), dtype=torch.uint8, device="cuda")
    d_nb = torch.empty(Cn, dtype=torch.int64, device="cuda")
    t_unc = timed(lambda: du.demod_bytes_dev(rx.data_ptr(), ff, ff, b"S", b"E", d_p.data_ptr(), 1024, d_np.data_ptr(), s),
                  args.reps, torch, stream)
    t_con = timed(lambda: dc.constellation_dev(rx.data_ptr(), ff, ff, d_sym.data_ptr(), ss, d_ns.data_ptr(), s), args.reps, torch, stream)
    t_dec = timed(lambda: vit.decode_dev(d_sym.data_ptr(), ss, d_ns.data_ptr(), d_b.data_ptr(), bc, d_nb.data_ptr(), s),
                  args.reps, torch, stream)
    t_frm = timed(lambda: dc.frame_bits_dev(d_b.data_ptr(), bc, d_nb.data_ptr(), b"S", b"E", d_p.data_ptr(), 1024,
                                            d_np.data_ptr(), s), args.reps, torch, stream)

    def coded_step():
        dc.constellation_dev(rx.data_ptr(), ff, ff, d_sym.data_ptr(), ss, d_ns.data_ptr(), s)
        vit.decode_dev(d_sym.data_ptr(), ss, d_ns.data_ptr(), d_b.data_ptr(), bc, d_nb.data_ptr(), s)
        dc.frame_bits_dev(d_b.data_ptr(), bc, d_nb.data_ptr(), b"S", b"E", d_p.data_ptr(), 1024, d_np.data_ptr(), s)
    t_step = timed(coded_step, args.reps, torch, stream)
    res["receive_step"] = {"channels": Cn, "payload_bytes": n_payload, "samples_per_channel": ff // 2,
                           "symbols_per_channel": int(d_ns[0].item()),
                           "demod_bytes_dev_s": t_unc, "constellation_dev_s": t_con, "viterbi_decode_dev_s": t_dec,
                           "frame_bits_dev_s": t_frm, "coded_step_s": t_step,
                           "decoder_over_constellation": t_dec / t_con, "goal_decoder_over_constellation": 0.25,
                           "goal_met": t_dec / t_con <= 0.25}
    print(res["receive_step"], flush=True)
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
