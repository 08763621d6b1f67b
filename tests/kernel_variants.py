"""Which instantiation of the FLL, modulator, equalizer and channelizer kernels a call runs, predicted from its public
inputs, listed from the built library, and read back from the profiler.

Every launcher picks a template instantiation from the shape of its input, and each instantiation is separately compiled
code (its own unrolling, tail stages and register window), so each is tested on its own.  Per family:
  * `*_predict` restates the launcher's dispatch in plain Python and returns the instantiation's name, or UNSUPPORTED;
  * `*_ROWS` is the table of public inputs the GPU parity tests run, at least one row per instantiation;
  * `*_launch_rows` runs those rows once each, in order, so that the profiler can list what ran.
`compiled()` lists the instantiations in the built library (cuobjdump -sass | cu++filt).  tests/test_kernel_variants.py
checks on the CPU that the dispatch reaches exactly the compiled set and that the tables cover it; the GPU tests check the
outputs against the oracle and, in a child process (`python kernel_variants.py FAMILY`), the launch list against the
prediction.

Names take one form, whatever prints them: cu++filt's `fll_duo_kernel<(int)5, (int)0, (int)4>` and the profiler's
`fll_duo_kernel<5, 0, 4>` both become `fll_duo_kernel<5, 0, 4>` (`normalise`)."""
import math
import os
import re
import shutil
import subprocess

import numpy as np

UNSUPPORTED = "UNSUPPORTED"

FAMILIES = {
    "fll": ("fll_duo_kernel", "fll_pair_kernel", "fll_group_kernel"),
    "mod": ("mod_shape_kernel",),
    "eq": ("cma_eq_kernel",),
    "pfb": ("pfb_kernel",),
}
_KERNEL_RE = re.compile(r"\b(" + "|".join(k for ks in FAMILIES.values() for k in ks) + r")\b(<[^<>]*>)?")


def normalise(name):
    """'fll_duo_kernel<5, 0, 4>' from a demangled or profiler kernel name, or None for a kernel of no family here."""
    m = _KERNEL_RE.search(name)
    if not m:
        return None
    args = m.group(2) or ""
    if args:
        args = "<" + ", ".join(re.sub(r"\((?:int|bool)\)", "", a).strip() for a in args[1:-1].split(",")) + ">"
    return m.group(1) + args


def family_of(name):
    base = name.split("<")[0]
    for fam, ks in FAMILIES.items():
        if base in ks:
            return fam
    return None


# ---- FLL: FllEngine::init / process_dev, fll_pair_supported, fll_duo_launch (csrc/loops.cu, fll_pair.cu, fll_duo.cu) ------
FLL_PAIR_MIN_STREAMS = 5120
FLL_DUO_PAIRS4_FROM = 1281            # fll_duo_launch: one warp pair per CTA up to 1280 streams, four above
FLL_GROUP_MAX_SMEM = 200 * 1024
TWO_PI_F = np.float32(2.0 * np.pi)


def fll_group_smem(n_taps):
    """Dynamic shared memory of fll_group_kernel: taps (N rounded up to even, + 4), 16 x 8 lane partials (float4), input and
    output staging (16 streams x 32 samples each, float2) and the ring (16 streams x N float2)."""
    np_ = n_taps + (n_taps & 1)
    return (2 * np_ + 4) * 4 + 16 * 8 * 16 + 2 * 16 * 32 * 8 + 16 * n_taps * 8


def fll_max_size():
    n = 1
    while fll_group_smem(n + 1) <= FLL_GROUP_MAX_SMEM:
        n += 1
    return n


def fll_predict(n_taps, channels, phase=0.0, freq=0.0, sps=4.0):
    """The kernel a Process call of an FLL handle runs, the caller-set (phase, freq) of every channel given as scalars."""
    if n_taps < 1 or fll_group_smem(n_taps) > FLL_GROUP_MAX_SMEM:
        return UNSUPPORTED                                                       # refused at creation
    max_freq = TWO_PI_F * (np.float32(2.0) / np.float32(sps))
    wild = not abs(phase) < 1e4 or not abs(freq) < 1e4 or not max_freq < 1e4
    far = not abs(phase) < 32.0
    if not wild and not far and n_taps in (10, 40) and channels >= FLL_PAIR_MIN_STREAMS:
        return f"fll_pair_kernel<{n_taps}>"
    if not wild and 8 <= n_taps <= 55:
        return f"fll_duo_kernel<{n_taps >> 3}, {n_taps & 7}, {1 if channels < FLL_DUO_PAIRS4_FROM else 4}>"
    return "fll_group_kernel"


FLL_DUO_C = (5, 1300)                  # PAIRS = 1 and PAIRS = 4 (82 CTAs of 16 streams, the last with one live pair)
FLL_GENERIC_N = (1, 2, 3, 4, 5, 6, 7, 56, 64, 100, 286, 287, 1000, 1430)
FLL_GENERIC_C = (1, 33)
# (n_taps, channels)
FLL_ROWS = ([(n, c) for c in FLL_DUO_C for n in range(8, 56)] +
            [(23, 1280), (23, 1281)] +                                          # PAIRS 1 -> 4
            [(n, c) for c in FLL_GENERIC_C for n in FLL_GENERIC_N] +
            [(10, 5120), (40, 5120), (40, 5119)])                               # the pair kernel, and one below it


# ---- modulator: ModEngine::init / make_bank / run, mod_pad_taps, mod_shape_pick (csrc/modulator.cu), design_rrc ------------
MOD_MT = (4, 5, 7, 8, 9, 11, 12, 13, 16, 17, 20, 24, 32, 48, 64, 96)
MOD_SPS_KERNELS = (2, 4, 8)            # compile-time samples per symbol, for MT <= 24
MOD_SPS_MAX_MT = 24
MOD_MAX_SPS = 256                      # kModThreads: one thread per phase


def mod_taps(fs, rs, span, pulse=True):
    """Taps of the polyphase bank a Modulate(bits, pulse) call runs: the RRC's N = span * round(fs/rs) + 1 (banker's rounding,
    as nearbyint) with pulse shaping, delay + 1 (a delta at the filter delay) without."""
    n = span * int(round(fs / rs)) + 1
    return n if pulse else (n - 1) // 2 + 1


def mod_predict(fs, rs, span, pulse=True):
    sps = fs // rs
    assert sps >= 1, "fs < rs is refused before any kernel runs"
    if sps > MOD_MAX_SPS:
        return UNSUPPORTED
    m = -(-mod_taps(fs, rs, span, pulse) // sps)
    mt = next((v for v in MOD_MT if v >= m), None)
    if mt is None:
        return UNSUPPORTED
    return f"mod_shape_kernel<{mt}, {sps if sps in MOD_SPS_KERNELS and mt <= MOD_SPS_MAX_MT else 0}>"


def mod_mt(fs, rs, span, pulse=True):
    return int(mod_predict(fs, rs, span, pulse).split("<")[1].split(",")[0])


# (fs, rs, span); every row runs with and without pulse shaping (the second bank has delay + 1 taps)
MOD_ROWS = ([(1000 * s, 1000, mt - 1) for s in MOD_SPS_KERNELS for mt in MOD_MT[:12]] +   # m = span + 1 = MT, SPS = sps
            [(3000, 1000, mt - 1) for mt in MOD_MT[:12]] +                              # sps 3: SPS = 0
            [(2000, 1000, 31), (3000, 1000, 47), (5000, 1000, 63), (2000, 1000, 95)])   # MT 32..96 take SPS = 0 at any rate


# ---- equalizer: EqEngine::process_dev, eq_check_params (csrc/eq.cu) -----------------------------------------------------
EQ_MAX_TAPS, EQ_MAX_SPS = 64, 8


def eq_predict(n_taps, sps):
    if not 1 <= n_taps <= EQ_MAX_TAPS or not 1 <= sps <= EQ_MAX_SPS:
        return UNSUPPORTED
    return f"cma_eq_kernel<{min(-(-n_taps // 8), 8)}, {sps if sps in (1, 2, 4, 8) else 0}>"


EQ_ROWS_C = 37                         # 8 channels per CTA: the last CTA holds five
# (n_taps, sps) per J = 1..8: sps 1, 2, 4, 8 and, for S = 0, 3 and 7
EQ_TAPS_BY_J = {1: (8, 3), 2: (9, 16), 3: (17, 24), 4: (25, 32), 5: (33, 40), 6: (41, 48), 7: (49, 56), 8: (57, 64)}
EQ_ROWS = [(EQ_TAPS_BY_J[j][i % 2], sps) for j in range(1, 9) for i, sps in enumerate((1, 2, 3, 4, 7, 8))]


# ---- channelizer: PfbEngine::init / process_dev (csrc/pfb.cu) ---------------------------------------------------------
PFB_MAX_P = 32


def pfb_predict(n_taps, M):
    if not (2 <= M <= 1024 and M & (M - 1) == 0) or n_taps < 1:
        return UNSUPPORTED
    P = -(-n_taps // M)
    return UNSUPPORTED if P > PFB_MAX_P else f"pfb_kernel<{P}>"


def pfb_taps(P, M):
    """A tap count that is not a multiple of M (the last taps per branch are zero padding), P taps per branch."""
    return P * M - (M // 3 if P > 1 else 0)


PFB_GRID = [(P, M) for P in (1, 2, 8, 16, 32) for M in (2, 4, 8, 16, 32, 64, 128, 256, 512, 1024)]
PFB_ROWS = PFB_GRID + [(P, M) for M in (4, 1024) for P in range(1, PFB_MAX_P + 1) if (P, M) not in PFB_GRID]


# ---- the predicted launch lists of the rows (what *_launch_rows runs) ---------------------------------------------------
def predicted_launches(family):
    if family == "fll":
        return [fll_predict(n, c) for n, c in FLL_ROWS]
    if family == "mod":
        return [mod_predict(fs, rs, span, pulse) for fs, rs, span in MOD_ROWS for pulse in (True, False)]
    if family == "eq":
        return [eq_predict(n, sps) for n, sps in EQ_ROWS]
    if family == "pfb":
        return [pfb_predict(pfb_taps(P, M), M) for P, M in PFB_ROWS]
    raise ValueError(family)


# ---- the compiled instantiations ------------------------------------------------------------------------------------------
def _tool(name):
    for c in (shutil.which(name), os.path.join("/usr/local/cuda/bin", name)):
        if c and os.path.exists(c):
            return c
    raise RuntimeError(f"{name} not found (CUDA toolkit)")


def compiled(lib_path):
    """{family: set of normalised instantiation names} in the library's SASS."""
    sass = subprocess.check_output([_tool("cuobjdump"), "-sass", lib_path], text=True)
    mangled = sorted(set(re.findall(r"Function : (\S+)", sass)))
    demangled = subprocess.run([_tool("cu++filt")], input="\n".join(mangled) + "\n", capture_output=True, text=True,
                               check=True).stdout.splitlines()
    out = {f: set() for f in FAMILIES}
    for d in demangled:
        n = normalise(d)
        if n is not None:
            out[family_of(n)].add(n)
    return out


# ---- GPU side: each family's rows, once each, for the profiler ----------------------------------------------------------
def _fll_launch_rows(Q):
    for n, c in FLL_ROWS:
        x = np.random.default_rng(n).standard_normal((c, 2 * 24)).astype(np.float32)
        Q.FLLBandEdgeFilter(4.0, 0.35, n, 0.05, channels=c).Process(x if c > 1 else x[0])


def _mod_launch_rows(Q):
    bits = "".join(np.random.default_rng(0).choice(["0", "1"], 64))
    for fs, rs, span in MOD_ROWS:
        m = Q.QPSKModulator(fs, rs, 0.35, span)
        m.Modulate(bits, True)
        m.Modulate(bits, False)


def _eq_launch_rows(Q):
    for n, sps in EQ_ROWS:
        x = np.random.default_rng(n).standard_normal((EQ_ROWS_C, 2 * 40)).astype(np.float32)
        Q.CmaEqualizer(n, 0.01, 1.2, channels=EQ_ROWS_C, sps=sps).Process(x)


def _pfb_launch_rows(Q):
    for P, M in PFB_ROWS:
        h = np.random.default_rng(P).standard_normal(pfb_taps(P, M))
        x = np.random.default_rng(M).standard_normal(2 * 2 * M).astype(np.float32)
        Q.PfbChannelizer(h, M).process(x)


LAUNCH_ROWS = {"fll": _fll_launch_rows, "mod": _mod_launch_rows, "eq": _eq_launch_rows, "pfb": _pfb_launch_rows}


def launched_in_child(family, device=0, timeout=900):
    """The family's kernel launches, in order, when its rows run under torch.profiler in a child process (a profiler session
    opened in the pytest process leaves the profiled tests of later files recording no kernels)."""
    import json
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, QPSK_VARIANTS_DEVICE=str(device))
    r = subprocess.run([sys.executable, os.path.join(here, "kernel_variants.py"), family], capture_output=True, text=True,
                       timeout=timeout, env=env)
    assert r.returncode == 0, r.stderr[-4000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("LAUNCHES ")][-1]
    return json.loads(line[len("LAUNCHES "):])


def _child(family):
    import json
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path[:0] = [os.path.dirname(here), here]
    import torch
    import qpsk_modulator_demodulator_b200 as Q
    from torch.profiler import ProfilerActivity, profile
    Q.set_device(int(os.environ.get("QPSK_VARIANTS_DEVICE", "0")))
    torch.cuda.init()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        LAUNCH_ROWS[family](Q)
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert ev, "torch.profiler recorded no CUDA kernel: cannot tell which kernel ran"
    ev.sort(key=lambda e: e.time_range.start)
    names = [normalise(e.name) for e in ev]
    print("LAUNCHES " + json.dumps([n for n in names if n is not None and family_of(n) == family]))


if __name__ == "__main__":
    import sys
    _child(sys.argv[1])
