"""Frame synchronizer probe (csrc/fsync.cu): process_dev kernel time at 1 / 64 / 2048 / 16384 channels x 8192 symbols with
no frame present (random uncoded QPSK at unit amplitude: the search runs over every position, the worst case), coherent
and differential, START = b"START" (P = 72); the share of the issue bound; the goal, at 2048 channels coherent,
process_dev against ViterbiDecoder.decode_dev on the same rows (at most 0.1); and the receive path after
constellation_dev at the K13 chain shape (2048 channels, 512-byte payloads), marker framer against synchronizer.

Issue bound: one warp per channel, 32 positions per pass; every warp instruction takes one issue slot of one of the 4
schedulers of an SM, so the least time is  channels * symbols / 32 * I / (SMs * 4 * f_sm),  I the warp instructions per
pass of 32 positions estimated from `cuobjdump -sass` as the constants below say; f_sm is the max SM clock nvidia-smi
reports in the same run.  Timing: CUDA events on one stream, median of --reps calls after 2 warm-up calls; every call
continues the stream of the one before (state advances), on device-resident rows."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))

# SASS warp instructions (cuobjdump -sass of fsync_kernel<false> / <true>, sm_100a).  The correlation loop is unrolled to
# 32 pattern words (64 symbols) per iteration: coherent 118 instructions (64 IDP.4A, 48 LDS), differential 102 (32 IDP.4A);
# a position reads P/2 + 1 words rounded up to a multiple of 4 (40 for P = 72).  Per pass of 32 positions the threshold
# test, rotation select, energy difference, ballot and loop control add about 60, and the soft-value fill of 32 new
# symbols (loads, q(), the warp scan of |s0| + |s1|, ring stores) about 110 (130 differential, which loads two symbols).
# An estimate for the issue bound, not a count of executed instructions.
LOOP_PER_32_WORDS = {False: 118, True: 102}
PASS_OVERHEAD = 60
FILL_PER_32 = {False: 110, True: 130}


def instr_per_pass(P, differential):
    words = ((P // 2 + 1) + 3) & ~3
    return words / 32 * LOOP_PER_32_WORDS[differential] + PASS_OVERHEAD + FILL_PER_32[differential]


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


def qpsk_rows(torch, Cn, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    b = torch.randint(0, 2, (Cn, 2 * n), device="cuda", generator=g, dtype=torch.int32)
    return ((2 * b - 1).to(torch.float32) * float(np.float32(np.sqrt(0.5)))).contiguous()


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
           "sms": props.multi_processor_count, "start_marker": "START", "sync": []}
    n_sym = 8192
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    s = stream.cuda_stream
    goal = {}
    for Cn in (1, 64, 2048, 16384):
        sym = qpsk_rows(torch, Cn, n_sym, Cn)
        ns = torch.full((Cn,), n_sym, dtype=torch.int32, device="cuda")
        for diff in (False, True):
            fs = Q.FrameSync(Cn, diff, b"START", 64, 3)
            slots = fs.slots_bound(n_sym)
            ldf = 2 * fs.window_syms
            fr = torch.empty((Cn * slots, ldf), dtype=torch.float32, device="cuda")
            fn = torch.empty(Cn * slots, dtype=torch.int32, device="cuda")
            nb = torch.empty(Cn * slots, dtype=torch.int64, device="cuda")
            info = torch.empty((Cn * slots, 3), dtype=torch.int64, device="cuda")
            t = timed(lambda: fs.process_dev(sym.data_ptr(), 2 * n_sym, ns.data_ptr(), slots, fr.data_ptr(), ldf,
                                             fn.data_ptr(), nb.data_ptr(), info.data_ptr(), s), args.reps, torch, stream)
            frames = int((fn > 0).sum().item())
            I = instr_per_pass(fs.pattern_syms, diff)
            bound = Cn * n_sym / 32 * I / (res["sms"] * 4 * f_sm)
            row = {"channels": Cn, "differential": diff, "symbols": n_sym, "kernel_s": t, "positions_per_s": Cn * n_sym / t,
                   "instr_per_32_positions": I, "issue_bound_s": bound, "share_of_issue_bound": bound / t,
                   "frames_found_last_call": frames}
            res["sync"].append(row)
            print(row, flush=True)
            if Cn == 2048 and not diff:
                goal["process_dev_s"] = t
            fs.close()
            del fr
        if Cn == 2048:
            vit = Q.ViterbiDecoder(Cn, differential=False)
            cap = vit.bits_bound(n_sym)
            bits = torch.empty((Cn, cap), dtype=torch.uint8, device="cuda")
            nbits = torch.empty(Cn, dtype=torch.int64, device="cuda")
            goal["viterbi_decode_dev_s"] = timed(lambda: vit.decode_dev(sym.data_ptr(), 2 * n_sym, ns.data_ptr(),
                                                                        bits.data_ptr(), cap, nbits.data_ptr(), s),
                                                 args.reps, torch, stream)
            vit.close()
        del sym
    goal.update(channels=2048, symbols=n_sym, ratio=goal["process_dev_s"] / goal["viterbi_decode_dev_s"], goal_ratio=0.1)
    goal["goal_met"] = goal["ratio"] <= 0.1
    res["goal"] = goal
    print(goal, flush=True)
    # the receive path after constellation_dev (the same call on both paths) at the chain shape: 2048 channels, one coded
    # frame with a 512-byte payload per row behind 600 lead-in symbols.  Marker path: ViterbiDecoder.flush_dev over the
    # whole row, then frame_bits_dev.  Sync path: process_dev over the row (no frame found: the full search), then
    # ViterbiDecoder(channels * slots).flush_dev over one full window per channel, then pack_bits_dev of the payload.
    Cn, n_pay = 2048, 512
    fs = Q.FrameSync(Cn, True, b"S", n_pay, 1)
    n = 600 + fs.window_syms
    sym = qpsk_rows(torch, Cn, n, 7)
    ns = torch.full((Cn,), n, dtype=torch.int32, device="cuda")
    dem = Q.QPSKDeModulator(10_000_000, 5_000_000, RrcAlpha=float(np.float32(0.4)), rrcSpan=10, channels=Cn)
    vit = Q.ViterbiDecoder(Cn, differential=True)
    bc = vit.bits_bound(n)
    d_b = torch.empty((Cn, bc), dtype=torch.uint8, device="cuda")
    d_nb = torch.empty(Cn, dtype=torch.int64, device="cuda")
    d_p = torch.empty((Cn, 1024), dtype=torch.uint8, device="cuda")
    d_np = torch.empty(Cn, dtype=torch.int64, device="cuda")
    t_vit_row = timed(lambda: vit.flush_dev(sym.data_ptr(), 2 * n, ns.data_ptr(), d_b.data_ptr(), bc, d_nb.data_ptr(), s),
                      args.reps, torch, stream)
    t_frm = timed(lambda: dem.frame_bits_dev(d_b.data_ptr(), bc, d_nb.data_ptr(), b"S", b"E", d_p.data_ptr(), 1024,
                                             d_np.data_ptr(), s), args.reps, torch, stream)
    slots = fs.slots_bound(n)
    ldf = 2 * fs.window_syms
    fr = torch.empty((Cn * slots, ldf), dtype=torch.float32, device="cuda")
    fn = torch.empty(Cn * slots, dtype=torch.int32, device="cuda")
    nbs = torch.empty(Cn * slots, dtype=torch.int64, device="cuda")
    info = torch.empty((Cn * slots, 3), dtype=torch.int64, device="cuda")
    t_sync = timed(lambda: fs.process_dev(sym.data_ptr(), 2 * n, ns.data_ptr(), slots, fr.data_ptr(), ldf, fn.data_ptr(),
                                          nbs.data_ptr(), info.data_ptr(), s), args.reps, torch, stream)
    wn = torch.zeros(Cn * slots, dtype=torch.int32, device="cuda")
    wn.view(Cn, slots)[:, 0] = fs.window_syms                                   # one full window per channel
    fr.view(Cn, slots, ldf)[:, 0] = sym[:, :ldf]
    vw = Q.ViterbiDecoder(Cn * slots, differential=True)
    bw = vw.bits_bound(fs.window_syms)
    w_b = torch.empty((Cn * slots, bw), dtype=torch.uint8, device="cuda")
    w_nb = torch.empty(Cn * slots, dtype=torch.int64, device="cuda")
    w_p = torch.empty((Cn * slots, n_pay), dtype=torch.uint8, device="cuda")
    t_vit_win = timed(lambda: vw.flush_dev(fr.data_ptr(), ldf, wn.data_ptr(), w_b.data_ptr(), bw, w_nb.data_ptr(), s),
                      args.reps, torch, stream)
    L = Q._native.lib()
    t_pack = timed(lambda: Q._native.check(L.qpsk_pack_bits_dev(w_b.data_ptr() + fs.payload_bit_offset, bw, w_nb.data_ptr(),
                                                                8 * n_pay, Cn * slots, w_p.data_ptr(), n_pay, s)),
                   args.reps, torch, stream)
    res["receive_path"] = {"channels": Cn, "payload_bytes": n_pay, "symbols_per_channel": n, "window_symbols": fs.window_syms,
                           "slots": slots, "marker": {"viterbi_flush_dev_row_s": t_vit_row, "frame_bits_dev_s": t_frm,
                                                      "total_s": t_vit_row + t_frm},
                           "sync": {"process_dev_s": t_sync, "viterbi_flush_dev_windows_s": t_vit_win,
                                    "pack_bits_dev_s": t_pack, "total_s": t_sync + t_vit_win + t_pack}}
    print(res["receive_path"], flush=True)
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
