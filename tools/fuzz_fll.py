"""Randomised parity soak of the FLL kernels against the oracle: random tap counts, rates, bandwidths, channel counts,
chunkings and carried state; outputs and loop state must be bit-identical.  usage: python tools/fuzz_fll.py [cases] [seed]
FUZZ_SIZES and FUZZ_CHANNELS restrict the tap and channel counts: FUZZ_SIZES=10,40 FUZZ_CHANNELS=5120,5137 runs the two-lane kernel."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import oracle as O
import qpsk_modulator_demodulator_b200 as Q

Q.set_device(0)
cases = int(sys.argv[1]) if len(sys.argv) > 1 else 60
rng = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 1)
SIZES = [int(v) for v in os.environ["FUZZ_SIZES"].split(",")] if os.environ.get("FUZZ_SIZES") else None
CHANNELS = [int(v) for v in os.environ["FUZZ_CHANNELS"].split(",")] if os.environ.get("FUZZ_CHANNELS") else None


def spread(C, n=33):
    """Channels compared against the oracle: all of a small batch; of a large one n evenly spaced channels (the first and
    the last among them) and both sides of the first and the last 16-stream warp boundary (fll_pair_kernel)."""
    if C <= n:
        return list(range(C))
    last = (C - 1) // 16 * 16
    return sorted(set(np.linspace(0, C - 1, n).astype(int).tolist()) | {15, 16, last - 1, last})


bad = 0
for k in range(cases):
    size = int(rng.choice(SIZES)) if SIZES else int(rng.integers(1, 70))
    sps = float(np.float32(rng.choice([0.7, 1.0, 2.0, 3.0, 4.0, 8.0, 30.0])))
    rolloff = float(np.float32(rng.uniform(0.05, 1.0)))
    bw = float(np.float32(10 ** rng.uniform(-4, -0.3)))
    C = int(rng.choice(CHANNELS)) if CHANNELS else int(rng.choice([1, 2, 3, 4, 5, 9, 33]))
    chk = spread(C)
    L = int(rng.integers(1, 1500))
    amp = float(10 ** rng.uniform(-3, 0.5))
    x = (amp * rng.standard_normal((C, 2 * L))).astype(np.float32)
    if rng.random() < 0.2:
        x[:, : 2 * (L // 3)] = 0.0
    g = Q.FLLBandEdgeFilter(sps, rolloff, size, bw, channels=C)
    os_ = {c: O.FLLBandEdgeFilter(sps, rolloff, size, bw) for c in chk}
    if rng.random() < 0.3:
        ph = rng.uniform(-7, 7, C).astype(np.float32)
        fr = rng.uniform(-0.5, 0.5, C).astype(np.float32)
        g.state = (ph, fr) if C > 1 else (float(ph[0]), float(fr[0]))
        for c in chk:
            os_[c].state = (float(ph[c]), float(fr[c]))
    cuts = sorted(set([0, L] + [int(v) for v in rng.integers(0, L + 1, int(rng.integers(0, 5)))]))
    ok = True
    for a, b in zip(cuts[:-1], cuts[1:]):
        got = g.Process(np.ascontiguousarray(x[:, 2 * a:2 * b]) if C > 1 else x[0, 2 * a:2 * b])
        got = got if C > 1 else got[None, :]
        for c in chk:
            want = os_[c].Process(x[c, 2 * a:2 * b])
            if not np.array_equal(got[c].view(np.uint32), want.view(np.uint32)):
                ok = False
    if not ok:
        bad += 1
        print("MISMATCH", dict(size=size, sps=sps, rolloff=rolloff, bw=bw, C=C, L=L, cuts=cuts))
print(f"fuzz_fll: {cases} cases, {bad} mismatching")
sys.exit(1 if bad else 0)
