"""Reed-Solomon probe (csrc/rs.cu): encode_dev and decode_dev kernel time at 1 / 64 / 2048 / 16384 rows of one block each,
for RS(255, 223) at depth 1 and 4 and RS(64, 48) at depth 1, decoding with 0 and with t byte errors in every codeword; and
the goal: at 2048 rows of one depth-4 RS(255, 223) block with t errors per codeword, decode_dev against
ViterbiDecoder.decode_dev over the coded symbols of those frames (8 * 1020 trellis steps per row), at most 0.1.

Issue bound: one warp per codeword; every warp instruction takes one issue slot of one of the 4 schedulers of an SM, so the
least time is  codewords * I / (SMs * 4 * f_sm).  I per codeword is estimated from `cuobjdump -sass` of the kernels as
the constants below say; f_sm is the max SM clock nvidia-smi reports in the same run.
Timing: CUDA events on one stream, median of --reps calls after 2 warm-up calls.  The inputs are device-resident and
written once; the largest (16384 rows x 1020 bytes, 16.7 MB) fits in the 126 MB L2, so these are L2-resident times."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))

# SASS warp instructions (cuobjdump -sass of rs_encode_kernel / rs_decode_kernel, sm_100a).  The encoder's byte loop is
# unrolled by 8: 76 instructions, 9.5 per message byte.  The decoder's syndrome loop is unrolled by 16: 85 instructions,
# 5.3 per code byte.  A codeword with errors adds Berlekamp-Massey (about 90 per syndrome, with its 7 shuffles), the Chien
# search (about 16 per locator term and 32 positions, unrolled by 4) and Forney (about 37 per term and 32 positions, for
# the chunks that hold a root: with t random errors in 255 bytes, all of them).  About 60 more per codeword set up the
# warp and write the message; an estimate for the issue bound, not a count of executed instructions.
ENC_PER_BYTE = 9.5
DEC_PER_BYTE = 5.3
DEC_BM_PER_ROOT = 90
DEC_CHIEN_PER_TERM = 16
DEC_FORNEY_PER_TERM = 37


def instr(kind, n, k, nroots, errors):
    if kind == "encode":
        return k * ENC_PER_BYTE + 60
    i = n * DEC_PER_BYTE + 60
    if errors:
        t = nroots // 2
        i += nroots * DEC_BM_PER_ROOT + ((n + 31) // 32) * (t + 1) * (DEC_CHIEN_PER_TERM + DEC_FORNEY_PER_TERM)
    return i


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
    import rs_oracle as R
    assert torch.cuda.is_available(), "no CUDA device: nothing to measure"
    props = torch.cuda.get_device_properties(0)
    clk_mhz = smi("clocks.max.sm")
    f_sm = float(clk_mhz) * 1e6
    res = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": smi("power.limit"), "max_sm_clock_mhz": clk_mhz,
           "sms": props.multi_processor_count, "l2_resident": True, "rows": []}
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    s = stream.cuda_stream
    rng = np.random.default_rng(1)
    goal_in = None
    for nroots, k, depth in ((32, 223, 1), (32, 223, 4), (16, 48, 1)):
        code, rs = R.Code(nroots, k, depth), Q.ReedSolomon(nroots, k, depth)
        mb, bb = depth * k, rs.block_bytes
        for rows in (1, 64, 2048, 16384):
            msg = torch.from_numpy(rng.integers(0, 256, (rows, mb)).astype(np.uint8)).cuda()
            cw = torch.empty((rows, bb), dtype=torch.uint8, device="cuda")
            t_enc = timed(lambda: rs.encode_dev(msg.data_ptr(), mb, rows, 1, cw.data_ptr(), bb, s), args.reps, torch, stream)
            clean = cw.cpu().numpy()
            words = code.deinterleave(clean.reshape(-1))
            noisy = code.interleave(R.add_errors(rng, words, np.full(words.shape[0], code.t))).reshape(rows, bb)
            cnt = torch.full((rows,), bb, dtype=torch.int64, device="cuda")
            out = torch.empty((rows, mb), dtype=torch.uint8, device="cuda")
            nm = torch.empty(rows, dtype=torch.int64, device="cuda")
            st = torch.empty((rows, depth), dtype=torch.int32, device="cuda")
            row = {"nroots": nroots, "k": k, "depth": depth, "rows": rows, "codewords": rows * depth, "encode_s": t_enc}
            for errs, src in ((0, clean), (code.t, noisy)):
                d_src = torch.from_numpy(np.ascontiguousarray(src)).cuda()
                t_dec = timed(lambda: rs.decode_dev(d_src.data_ptr(), bb, cnt.data_ptr(), rows, out.data_ptr(), mb,
                                                    nm.data_ptr(), st.data_ptr(), depth, s), args.reps, torch, stream)
                sts = st.cpu().numpy()
                assert (sts == errs).all(), (nroots, k, depth, rows, errs)
                bound = rows * depth * instr("decode", code.n, k, nroots, errs) / (res["sms"] * 4 * f_sm)
                row[f"decode_{errs}_errors_s"] = t_dec
                row[f"decode_{errs}_errors_share_of_issue_bound"] = bound / t_dec
                if (nroots, k, depth, rows, errs) == (32, 223, 4, 2048, code.t):
                    goal_in = t_dec
            row["encode_share_of_issue_bound"] = rows * depth * instr("encode", code.n, k, nroots, 0) / (res["sms"] * 4 * f_sm) / t_enc
            row["decode_bytes_per_s_t_errors"] = rows * bb / row[f"decode_{code.t}_errors_s"]
            res["rows"].append(row)
            print(row, flush=True)
    # the goal: RS decode against the Viterbi decode of the same frames' coded symbols
    Cn, n_sym = 2048, 8 * 4 * 255
    g = torch.Generator(device="cuda").manual_seed(3)
    sym = (torch.randn((Cn, 2 * n_sym), device="cuda", generator=g) * 0.7).contiguous()
    ns = torch.full((Cn,), n_sym, dtype=torch.int32, device="cuda")
    vit = Q.ViterbiDecoder(Cn, differential=True)
    cap = vit.bits_bound(n_sym)
    bits = torch.empty((Cn, cap), dtype=torch.uint8, device="cuda")
    nb = torch.empty(Cn, dtype=torch.int64, device="cuda")
    t_vit = timed(lambda: vit.decode_dev(sym.data_ptr(), 2 * n_sym, ns.data_ptr(), bits.data_ptr(), cap, nb.data_ptr(), s),
                  args.reps, torch, stream)
    res["goal"] = {"rows": Cn, "code": "RS(255,223) depth 4, t errors per codeword", "rs_decode_dev_s": goal_in,
                   "viterbi_decode_dev_s": t_vit, "symbols_per_row": n_sym, "ratio": goal_in / t_vit, "goal_ratio": 0.1,
                   "goal_met": goal_in / t_vit <= 0.1}
    print(res["goal"], flush=True)
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
