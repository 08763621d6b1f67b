"""Which instantiation of the FLL, modulator, equalizer, channelizer, DDC bank, resampler and FIR kernels a call runs,
predicted from its public inputs, listed from the built library, and read back from the profiler.

Every launcher picks a template instantiation from the shape of its input, and each instantiation is separately compiled
code (its own unrolling, tail stages and register window), so each is tested on its own.  Per family:
  * `*_predict` restates the launcher's dispatch in plain Python and returns the instantiation's name, or UNSUPPORTED
    (`fir_predict`: the list of kernels the call launches, in order);
  * `*_ROWS` is the table of public inputs the GPU parity tests run, at least one row per instantiation (the DDC,
    resampler and channelizer rows are the ones tests/bank_bounds.py checks against per-output error bounds);
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
    # the history copies next to the DDC and resampler kernels (ddc_history_kernel, resamp_history_kernel) are left out
    "ddc": ("ddc_kernel",),
    "resamp": ("resamp_kernel",),
    # fir_hist_update_kernel (the delay-line copy next to the generic and decimating kernels) is left out
    "fir": ("fir_tma_kernel", "fir_split2_kernel", "fir_exact_real_kernel", "fir_generic_kernel", "fir_dec2_kernel",
            "fir_decim_tma_kernel", "fir_decim_kernel", "fir_subsample_kernel"),
}
_KERNEL_RE = re.compile(r"\b(" + "|".join(k for ks in FAMILIES.values() for k in ks) + r")\b(<[^<>]*>)?")


def _arg(a):
    a = a.strip()
    if a in ("(bool)0", "(bool)1"):
        return "true" if a.endswith("1") else "false"
    return re.sub(r"\((?:int|bool)\)", "", a).strip()


def normalise(name):
    """'fll_duo_kernel<5, 0, 4>' from a demangled or profiler kernel name, or None for a kernel of no family here.
    cu++filt prints a bool template argument as (bool)0 / (bool)1; both become false / true."""
    m = _KERNEL_RE.search(name)
    if not m:
        return None
    args = m.group(2) or ""
    if args:
        args = "<" + ", ".join(_arg(a) for a in args[1:-1].split(",")) + ">"
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


# ---- DDC bank: qpsk_ddc_create, DdcEngine::process_dev (csrc/ddc.cu) ------------------------------------------------------
DDC_MAX_TAPS, DDC_MAX_CHANNELS, DDC_MAX_DECIM = 4096, 2048, 1024
DDC_SMALL_K = 8                         # kDdcSmallK: K <= 8 runs the 4-channel x 1024-output shape
DDC_TILE = {True: 1024, False: 128}     # outputs per CTA, K <= 8 / K > 8


def ddc_predict(n_taps, channels, decim):
    """The kernel a call that completes at least one output runs (the history copy is left out)."""
    if (not 1 <= n_taps <= DDC_MAX_TAPS or not 1 <= channels <= DDC_MAX_CHANNELS or
            not 1 <= decim <= DDC_MAX_DECIM):
        return UNSUPPORTED
    return "ddc_kernel<1, 1, 8>" if channels <= DDC_SMALL_K else "ddc_kernel<4, 2, 32>"


# (K, D, N, taps): both shapes (K = 8 | 9) at D = 1, odd D, D = 16 and 64; taps "rand" (fir_row_taps' recipe) or "kaiser"
# (ddc_oracle.scene_taps, the prototype of the library's scenes)
DDC_ROWS = [(K, D, N, kind) for D, N, kind in ((1, 17, "rand"), (5, 33, "rand"), (16, 100, "rand"), (64, 300, "rand"),
                                               (16, 128, "kaiser")) for K in (8, 9)]


def ddc_row_calls(row):
    """Input samples of a row's two calls: three tiles of outputs and a ragged end each; the first leaves D//2 + 1 samples
    of an open block pending (D > 2), so the second call's first output reads history and pending samples."""
    K, D = row[:2]
    n_out = 3 * DDC_TILE[K <= DDC_SMALL_K] + 37
    return [n_out * D + (D // 2 + 1) % D, n_out * D + 3]


# ---- rational resampler: qpsk_resamp_create, ResampEngine::process_dev (csrc/resamp.cu) ------------------------------------
RESAMP_MAX_TAPS, RESAMP_MAX_FACTOR, RESAMP_MAX_BRANCH, RESAMP_MAX_CHANNELS = 16384, 1024, 64, 16384
RESAMP_SMALL_K = 8                      # kResampSmallK: K <= 8 runs the one-channel x 256-output shape
RESAMP_TILE = {True: 256, False: 32}    # outputs per CTA, K <= 8 / K > 8


def resamp_predict(n_taps, L, M, channels):
    """The kernel a call that completes at least one output runs (the history copy is left out)."""
    if (not 1 <= n_taps <= RESAMP_MAX_TAPS or not 1 <= L <= RESAMP_MAX_FACTOR or not 1 <= M <= RESAMP_MAX_FACTOR or
            not 1 <= channels <= RESAMP_MAX_CHANNELS or -(-n_taps // L) > RESAMP_MAX_BRANCH):
        return UNSUPPORTED
    return "resamp_kernel<1, 1, 1, 2048>" if channels <= RESAMP_SMALL_K else "resamp_kernel<32, 2, 4, 64>"


# (K, L, M, N, taps): both shapes (K = 8 | 9); L < M, L > M, L = 1; P = 1, 24, 64; every ratio coprime, so that every
# branch is used; taps "rand" or "kaiser" (resamp_oracle.resamp_taps)
RESAMP_ROWS = [(K, L, M, N, kind) for L, M, N, kind in ((5, 8, 120, "rand"), (8, 5, 507, "rand"), (1, 3, 1, "rand"),
                                                        (1, 1, 64, "rand"), (3, 1, 190, "rand"), (125, 128, 3000, "kaiser"))
               for K in (8, 9)]
RESAMP_CALL_OUT = 3 * 256 + 37          # outputs per call: >= 3 tiles of either shape, ragged in both


def resamp_row_calls(row):
    """Input samples per channel of a row's two calls, each completing about RESAMP_CALL_OUT outputs."""
    L, M = row[1:3]
    n = RESAMP_CALL_OUT * M // L
    return [n + 3, n + 11]


# ---- FIR: FirEngine::run / decimate_dev, launch_split2 (csrc/fir.cu) ----------------------------------------------------
FIR_MODES = {"FAST": 0, "EXACT": 1, "FMA": 2, "SPLIT": 3}
kMaxG = 1040                            # correlation taps in kernel-parameter space
kR, kNT, kNTWide = 10, 256, 320         # fir_tma_kernel
kSmemBudget = 112 * 1024                # per CTA, two CTAs per SM
kS2R, kS2NT, kS2MinForced, kS2MinFast = 10, 256, 14, 48
kENT = 256                              # fir_exact_real_kernel: 2 outputs per thread, 72 KiB
kET = 2 * kENT
kExactSmem = 72 * 1024
kDec2R, kDec2NT = 14, 256               # fir_dec2_kernel
kDecimRO = 7
kDecimSmemMax = 200 * 1024              # fir_decim_kernel (go)
DECIM_TMA = {4: (128, 2, False), 8: (64, 4, True), 16: (32, 8, True)}   # D: (NTO, NG, repack)
DECIM = {2: (256, 1), 4: (128, 2), 8: (64, 4), 16: (32, 8)}             # D: (NTO, NG)
FIR_TAIL_MOD = {"fir_tma_kernel": 20, "fir_split2_kernel": 7, "fir_exact_real_kernel": 8, "fir_dec2_kernel": 8,
                "fir_decim_tma_kernel": 14, "fir_decim_kernel": 14}
# tap-loop tails: fir_tma_kernel G mod 2R (QPSK_TAIL), fir_split2_kernel G/2 mod (R/2 + 2) (QPSK_TAIL2), fir_exact_real_kernel
# N mod 8 (the scalar tail after the 8-lane blocks; N odd / even is the window lead 0 / 1), fir_dec2_kernel G/2 mod (R/2 + 1)
# (QPSK_TAILD), the decimators K mod 2*RO (QPSK_DTAIL)


def fir_hl(n_taps):
    """FirEngine::init's delay-line length: N - 1 rounded up to even, 2 for a 1-tap filter."""
    hl = (n_taps - 1) + ((n_taps - 1) & 1)
    return hl if hl else 2


def _fir_wide(G, cplx):
    return not cplx and 48 <= G <= 96


def _tma_stages(T, G):
    return min(4, (kSmemBudget - 2 * T * 8 - 128) // ((T + G + 2) * 8))


def _split_fits(hl, G):
    T2 = kS2R * kS2NT
    if hl > T2:
        return False
    stage = (T2 + G + 2) * 8
    fixed = T2 * 8 + (kS2NT // 32) * ((32 * kS2R + G) // 2 + 1) * 8
    return fixed + 128 + 2 * stage <= kSmemBudget


def _fir_run(n, cplx, mode, stateless, rows_ok):
    """(kernel, tail residue) of FirEngine::run; rows_ok: both pointers 16-byte aligned and no odd row stride in a batch."""
    hl = n - 1 if stateless else fir_hl(n)
    G = (hl + 2) & ~1
    wide = _fir_wide(G, cplx)
    T = kR * (kNTWide if wide else kNT)
    use_tma = (mode != "EXACT" or stateless) and G <= kMaxG and hl <= T and rows_ok
    want_split = (mode == "SPLIT" and G >= kS2MinForced) or (mode == "FAST" and G >= kS2MinFast)
    if use_tma and not cplx and want_split and _split_fits(hl, G):
        return f"fir_split2_kernel<{kS2R}, {kS2NT}>", (G // 2) % FIR_TAIL_MOD["fir_split2_kernel"]
    if use_tma and _tma_stages(T, G) >= 2:
        return f"fir_tma_kernel<{kR}, {kNTWide if wide else kNT}, {'true' if cplx else 'false'}>", G % 20
    HL = fir_hl(n)
    if mode == "EXACT" and not stateless and not cplx and n >= 8 and rows_ok:
        GE = (HL + 2) & ~1
        if GE <= kMaxG and HL <= kET and min(4, (kExactSmem - 2 * kET * 8 - 128) // ((kET + GE + 2) * 8)) >= 2:
            return f"fir_exact_real_kernel<{kENT}>", n % 8
    return ("fir_generic_kernel<true>" if mode == "EXACT" and not stateless else "fir_generic_kernel<false>"), None


def _dec2_fits(Gs, HL):
    T2 = kDec2R * kDec2NT
    return (Gs <= kMaxG and HL <= T2 and
            min(4, (kSmemBudget - 2 * (T2 // 2) * 8 - 128) // ((T2 + Gs + 2) * 8)) >= 2)


def _decim_tma_fits(D, Ks):
    NTO, NG, repack = DECIM_TMA[D]
    if Ks * D > kMaxG:
        return False
    T_OUT = kDecimRO * NTO
    E = (T_OUT + Ks) * D
    pad = ((E + 2 * (E // (kDecimRO * D) + 1) + 1) & ~1) if repack else 0
    fixed = NG * T_OUT * 8 + pad * 8
    return fixed + 128 + 2 * (E + 2) * 8 <= kSmemBudget


def _decim_fits(D, K):
    NTO, NG = DECIM[D]
    T_OUT = kDecimRO * NTO
    E = (T_OUT + K) * D
    return (NG * T_OUT + E + (0 if D == 2 else 2) * (E // (kDecimRO * D) + 1)) * 8 <= kDecimSmemMax


def fir_nout(L, D, skip):
    return (L - skip + D - 1) // D if L > skip else 0


def fir_next_skip(L, D, skip):
    """The kept-output phase the next Decimate call with the same D starts from."""
    return skip + fir_nout(L, D, skip) * D - L if L > skip else skip - L


def fir_dispatch(n_taps, cplx=False, mode="FAST", op="filter", L=1000, skip=0, x_off=0, y_off=0, channels=1,
                 ldx=None, ldy=None):
    """[(kernel, tail residue or None)] a call launches, in order.  op: "filter" (streaming Filter), "fft" (stateless
    fftFilter) or a decimation factor D; skip: the kept-output phase carried from earlier Decimate calls with this D;
    x_off / y_off: pointer offsets in samples from a 16-byte boundary; ldx / ldy: row strides in samples (batches)."""
    x_al, y_al = x_off % 2 == 0, y_off % 2 == 0
    ldx = L if ldx is None else ldx
    ldy = L if ldy is None else ldy
    odd_x = channels > 1 and ldx % 2 == 1
    odd_y = channels > 1 and ldy % 2 == 1
    if op in ("filter", "fft"):
        return [_fir_run(n_taps, cplx, mode, op == "fft", x_al and y_al and not odd_x and not odd_y)]
    D = op
    nout = fir_nout(L, D, skip)
    HL = fir_hl(n_taps)
    K = (HL + 1 + D - 1) // D
    if mode != "EXACT" and not cplx and D in (2, 4, 8, 16) and K * D <= kMaxG and nout > 0:
        if D == 2 and x_al and y_al and not odd_x and not odd_y:
            Gs = (HL + 1 + skip + 1) & ~1
            if _dec2_fits(Gs, HL):
                return [(f"fir_dec2_kernel<{kDec2R}, {kDec2NT}>", (Gs // 2) % 8)]
        if D > 2 and x_al and not odd_x:
            Ks = (HL + 1 + (skip & 1) + D - 1) // D
            if _decim_tma_fits(D, Ks):
                NTO, NG, repack = DECIM_TMA[D]
                return [(f"fir_decim_tma_kernel<{kDecimRO}, {NTO}, {NG}, {D}, {'true' if repack else 'false'}>", Ks % 14)]
        if _decim_fits(D, K):
            NTO, NG = DECIM[D]
            return [(f"fir_decim_kernel<{kDecimRO}, {NTO}, {NG}, {D}>", K % 14)]
    # the full-rate streaming filter into an aligned scratch row of even pitch, then the kept samples
    return [_fir_run(n_taps, cplx, mode, False, x_al and not odd_x)] + ([("fir_subsample_kernel", None)] if nout > 0 else [])


def fir_predict(*args, **kw):
    return [k for k, _ in fir_dispatch(*args, **kw)]


# The rows: (n_taps, complex taps, mode, op, layout, phase).  Streaming rows (Filter, Decimate) are two calls on one handle,
# the first of odd length; for a decimator it leaves the kept-output phase `phase` (odd: 1..D-1) for the second.  fftFilter
# rows are two independent calls.  Layouts: dense (one channel), xoff / yoff (input / output pointer one sample past a
# 16-byte boundary), odd3 (three channels, odd row strides), even3 (three channels, even strides, long enough that the
# persistent CTAs' tile walk steps across channel seams).
FIR_L1 = 3 * 3584 + 1001                # three tiles of every kernel (3584 input samples at most) and a ragged end; odd
FIR_L2 = 3 * 3584 + 778
FIR_L_WALK = 110 * 3584 + 1001          # > 2 * 148 tiles over three channels for every tiled kernel
FIR_LAYOUTS = {"dense": (1, 0, 0), "xoff": (1, 1, 0), "yoff": (1, 0, 1), "odd3": (3, 0, 0), "even3": (3, 0, 0)}


def _fir_rows():
    rows = []

    def add(n, cplx=False, mode="FAST", op="filter", layout="dense", phase=0):
        r = (n, cplx, mode, op, layout, phase)
        if r not in rows:
            rows.append(r)

    # fir_tma_kernel<10, 256, true>: every G mod 20, streaming (G = N + 1 for odd N) and stateless (G = N for even N)
    for n in range(19, 39, 2):
        add(n, True)
    for n in range(20, 40, 2):
        add(n, True, op="fft")
    for n in (1, 2, 3, 8, 257):
        add(n, True)
    # fir_tma_kernel<10, 256, false>: every G mod 20 in FMA mode below the ten-warp range, FAST below the split
    for n in range(19, 39, 2):
        add(n, mode="FMA")
    for n in (1, 2, 44, 45):
        add(n)
    # fir_tma_kernel<10, 320, false>: FMA mode, every G mod 20 of G = 48..66; its edges 45 / 46 and 95 / 96 streaming,
    # 46 / 47 and 96 / 97 stateless (FMA and EXACT: a stateless call never takes the exact-order kernels)
    for n in range(47, 67, 2):
        add(n, mode="FMA")
    for n in (45, 46, 95, 96):
        add(n, mode="FMA")
    for n in (46, 47, 96, 97):
        add(n, mode="FMA", op="fft")
        add(n, mode="EXACT", op="fft")
    # fir_split2_kernel: FAST from G = 48 (N 44 / 45 / 46 / 47), SPLIT from G = 14 (N 11 / 12), every G/2 mod 7, the ring's
    # fit at 889 / 890 streaming taps, stateless
    for n in (46, 47, 55, 57, 59, 61, 63, 65, 67, 889, 890):
        add(n)
    for n in (11, 12):
        add(n, mode="SPLIT")
    for n in (48, 890, 891):
        add(n, op="fft")
    # kMaxG: 1039 / 1040 streaming taps, 1040 / 1041 stateless (FMA: the tap-sequential kernel up to the switch)
    for n in (1039, 1040):
        add(n, mode="FMA")
        add(n, True)
    for n in (1040, 1041):
        add(n, mode="FMA", op="fft")
        add(n, True, op="fft")
    # fir_exact_real_kernel: every N mod 8 (window lead 0 and 1), 7 / 8 and 513 / 514 taps (HL = 512: the halo is a tile)
    for n in range(7, 17):
        add(n, mode="EXACT")
    for n in (64, 257, 512, 513, 514, 1039):
        add(n, mode="EXACT")
    add(21, True, mode="EXACT")                                   # complex taps: fir_generic_kernel<true>
    # fir_dec2_kernel: every Gh mod 8, the kept-output phase 1 (a leading zero tap), Gs = kMaxG at 1039 taps; 1040 taps
    # go full-rate
    for n in range(15, 31, 2):
        add(n, op=2, phase=1)
    for n in (1039, 1040):
        add(n, op=2, phase=1)
    # fir_decim_tma_kernel / fir_decim_kernel: every K mod 14 at D = 4, 8, 16 (and 2 for the register-staged kernel), with
    # each odd kept-output phase in turn; the second through a pointer one sample past a 16-byte boundary
    for D in (4, 8, 16):
        for i, K in enumerate(range(14, 28)):
            add(D * (K - 1) + 3, op=D, phase=2 * (i % (D // 2)) + 1)
    for D in (2, 4, 8, 16):
        for i, K in enumerate(range(14, 28)):
            add(D * K - 1, op=D, layout="xoff", phase=2 * (i % (D // 2)) + 1)
    # the TMA ring's fit at D = 8 and 16 (aligned: the register-staged kernel beyond it) and K * D > kMaxG for every D
    for D in (8, 16):
        n = fir_decim_tma_limit(D)
        add(n, op=D, phase=D - 1)
        add(n + 2, op=D, phase=D - 1)
    for D in (2, 4, 8, 16):
        add(1039, op=D, phase=1)
        add(1040, op=D, phase=1)
    # the full-rate path: odd D, D = 1, complex taps, EXACT mode (bit-exact kernels), a split filter
    add(129, op=3, phase=1)
    add(33, op=1)
    add(40, True, op=4, phase=3)
    add(65, mode="EXACT", op=8, phase=5)
    add(600, mode="EXACT", op=2, phase=1)
    # layouts
    add(33, layout="xoff")
    add(33, layout="yoff")
    add(19, True, layout="xoff")
    add(21, mode="EXACT", layout="xoff")
    add(33, op="fft", layout="yoff")
    add(65, op=4, layout="yoff", phase=3)
    add(65, op=2, layout="yoff", phase=1)
    add(65, layout="odd3")
    add(33, True, layout="odd3")
    add(21, mode="EXACT", layout="odd3")
    add(65, op=2, layout="odd3", phase=1)
    add(65, op=8, layout="odd3", phase=3)
    add(33, layout="even3")
    add(129, layout="even3")
    add(21, True, layout="even3")
    add(64, mode="EXACT", layout="even3")
    add(65, mode="FMA", layout="even3")
    add(65, op="fft", layout="even3")
    add(65, op=2, layout="even3", phase=1)
    for D in (4, 8, 16):
        add(65, op=D, layout="even3", phase=D - 1)
    return rows


def fir_decim_tma_limit(D):
    """The longest (odd) tap count whose aligned D-fold decimation still runs on fir_decim_tma_kernel."""
    n = 3
    while _decim_tma_fits(D, (fir_hl(n + 2) + 1 + D - 1) // D):
        n += 2
    return n


def fir_row_calls(row):
    """The calls of a row: [dict(op, L, skip, x_off, y_off, channels, ldx, ldy)] (strides in samples)."""
    n, cplx, mode, op, layout, phase = row
    C, x_off, y_off = FIR_LAYOUTS[layout]
    L1 = FIR_L_WALK if layout == "even3" else FIR_L1
    L2 = FIR_L_WALK - 222 if layout == "even3" else FIR_L2
    if isinstance(op, int) and phase:
        L1 += (-phase - L1) % op                                  # (-L1) mod D = phase; phase odd keeps L1 odd
        assert L1 % 2 == 1 and fir_next_skip(L1, op, 0) == phase, (row, L1)
    calls, skip = [], 0
    for L in (L1, L2):
        m = fir_nout(L, op, skip) if isinstance(op, int) else L
        ldx, ldy = L, m
        if layout == "odd3":
            ldx, ldy = L + 1 + (L & 1), m + 1 + (m & 1)
        elif layout == "even3":
            ldx, ldy = L + 2 - (L & 1), m + 2 - (m & 1)
        calls.append(dict(op=op, L=L, skip=skip, x_off=x_off, y_off=y_off, channels=C, ldx=ldx, ldy=ldy, n_out=m))
        if isinstance(op, int):
            skip = fir_next_skip(L, op, skip)
    return calls


def fir_row_dispatch(row):
    """[[(kernel, tail)] per call] of a row."""
    n, cplx, mode = row[:3]
    return [fir_dispatch(n, cplx, mode, c["op"], c["L"], c["skip"], c["x_off"], c["y_off"], c["channels"], c["ldx"],
                         c["ldy"]) for c in fir_row_calls(row)]


def _seed(*parts):
    import zlib
    return zlib.crc32(repr(parts).encode())


def fir_row_taps(row):
    """Interleaved IQ float32 taps: random signs, magnitudes in [0.5, 1.5] / sqrt(N) (no tap near zero, every one visible),
    and the last two of opposite sign (so that swapping them shows)."""
    n, cplx = row[0], row[1]
    rng = np.random.default_rng(_seed("taps", n, cplx))

    def part():
        v = rng.uniform(0.5, 1.5, n) * rng.choice((-1.0, 1.0), n) / np.sqrt(n)
        if n > 1:
            v[-1] = -np.sign(v[-2]) * abs(v[-1])
        return v

    t = np.zeros(2 * n, np.float32)
    if cplx:
        t[0::2], t[1::2] = part() / np.sqrt(2.0), part() / np.sqrt(2.0)
    else:
        t[0::2] = part()
    return t


def fir_row_inputs(row):
    """Per call a [C, L, 2] float32 input: uniform samples under an envelope that alternates between 1 and 2^-12 every
    N + 97 samples, so that at each step one large sample sits under the first or the last tap next to small ones."""
    calls = fir_row_calls(row)
    C = calls[0]["channels"]
    total = sum(c["L"] for c in calls)
    n = row[0]
    rng = np.random.default_rng(_seed("x", row))
    x = rng.uniform(-1.0, 1.0, (C, total, 2))
    seg = n + 97
    env = np.where(((np.arange(total) + int(rng.integers(seg))) // seg) % 2 == 0, 1.0, 2.0 ** -12)
    x = (x * env[None, :, None]).astype(np.float32)
    out, a = [], 0
    for c in calls:
        out.append(x[:, a: a + c["L"]])
        a += c["L"]
    return out


def fir_reference(taps_iq, xs, op):
    """float64 outputs of the calls (streaming: one stream over all calls; fftFilter: each call alone), and per output the
    sums sum_i |g_i| |x_i| of the real and of the imaginary part, also for the full-rate neighbours n - 1 and n + 1.
    Returns per call (y [C, m] complex, abs_re [C, m], abs_im [C, m], nb_re, nb_im)."""
    h = taps_iq[0::2].astype(np.float64) + 1j * taps_iq[1::2].astype(np.float64)
    ah_r, ah_i = np.abs(h.real), np.abs(h.imag)
    N = h.size

    def full(x):                                                  # x [L] complex128: the convolution and its abs sums
        xr, xi = np.abs(x.real), np.abs(x.imag)
        y = np.convolve(x, h)
        sr = np.convolve(xr, ah_r) + np.convolve(xi, ah_i)
        si = np.convolve(xi, ah_r) + np.convolve(xr, ah_i)
        return y, sr, si

    def nb(s, lo, hi):                                            # s[n - 1] + s[n + 1] over [lo, hi)
        p = np.concatenate([[0.0], s, [0.0]])
        return p[lo: hi] + p[lo + 2: hi + 2]

    C = xs[0].shape[0]
    res = [[None] * C for _ in xs]
    for c in range(C):
        if op == "fft":
            for k, x in enumerate(xs):
                z = x[c, :, 0].astype(np.float64) + 1j * x[c, :, 1].astype(np.float64)
                y, sr, si = full(z)
                L = z.size
                res[k][c] = (y[N - 1: N - 1 + L], sr[N - 1: N - 1 + L], si[N - 1: N - 1 + L],
                             nb(sr, N - 1, N - 1 + L), nb(si, N - 1, N - 1 + L))
            continue
        z = np.concatenate([x[c, :, 0].astype(np.float64) + 1j * x[c, :, 1].astype(np.float64) for x in xs])
        y, sr, si = full(z)
        T = z.size
        y, nr, ni, sr, si = y[:T], nb(sr, 0, T), nb(si, 0, T), sr[:T], si[:T]
        D = op if isinstance(op, int) else 1
        keep = np.arange(0, T, D)
        a = 0
        for k, x in enumerate(xs):
            L = x.shape[1]
            sel = keep[(keep >= a) & (keep < a + L)]
            res[k][c] = (y[sel], sr[sel], si[sel], nr[sel], ni[sel])
            a += L
    return [tuple(np.stack([r[c][j] for c in range(C)]) for j in range(5)) for r in res]


def fir_chain(kernel, n_taps, cplx):
    """(c, w) of the bound c * 2^-24 * (sum|g||x| + w * the neighbours' sums); derived in tests/test_gpu_fir_variants.py."""
    base = kernel.split("<")[0]
    G = fir_hl(n_taps) + 2                                        # >= the G of any call (HL is even)
    if base == "fir_tma_kernel":
        return (n_taps + 1 if cplx else n_taps), 0.0
    if base == "fir_split2_kernel":
        return G // 2 + 4, 2.0
    if base == "fir_exact_real_kernel" or kernel == "fir_generic_kernel<true>":
        return n_taps + 2, 0.0
    if base == "fir_generic_kernel":
        return (2 * n_taps if cplx else n_taps), 0.0
    if base == "fir_dec2_kernel":
        return G // 2 + 1, 0.0
    if base in ("fir_decim_tma_kernel", "fir_decim_kernel"):
        args = [int(a) for a in kernel.split("<")[1].rstrip(">").replace("true", "1").replace("false", "0").split(",")]
        NG, DD = args[2], args[3]
        K = (fir_hl(n_taps) + 2 + DD - 1) // DD
        return 2 * (DD // 2 // NG) * K + NG - 1, 0.0
    raise ValueError(kernel)


def fir_bound(kernel, n_taps, cplx, ref):
    """Per output bounds (re, im) of |kernel - float64 reference|: gamma_c * (own sums + w * neighbours' sums)."""
    c, w = fir_chain(kernel, n_taps, cplx)
    u = 2.0 ** -24
    g = c * u / (1 - c * u)
    _, sr, si, nr, ni = ref
    return g * (sr + w * nr) * (1 + 1e-9) + 1e-300, g * (si + w * ni) * (1 + 1e-9) + 1e-300


FIR_ROWS = _fir_rows()


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
    if family == "ddc":
        return [ddc_predict(N, K, D) for K, D, N, _ in DDC_ROWS for _ in ddc_row_calls((K, D))]
    if family == "resamp":
        return [resamp_predict(N, L, M, K) for K, L, M, N, _ in RESAMP_ROWS for _ in resamp_row_calls((K, L, M))]
    if family == "fir":
        return [k for r in FIR_ROWS for call in fir_row_dispatch(r) for k, _ in call]
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


def fir_run_row(Q, row, xs, taps=None, calls=None):
    """Run a row's calls (fir_row_calls unless given) on one handle through the device entry points, with the row's
    pointer offsets and strides.  Returns per call (y [C, m, 2] float32, whether the row padding and the buffer ends were
    left untouched, last_kernel())."""
    import torch
    n, cplx, mode, op = row[:4]
    calls = fir_row_calls(row) if calls is None else calls
    f = Q.ComplexFIRFilter(fir_row_taps(row) if taps is None else taps, channels=calls[0]["channels"])
    f.set_mode(FIR_MODES[mode])
    out = []
    for c, x in zip(calls, xs):
        C, L, m = c["channels"], c["L"], c["n_out"]
        xb = torch.zeros(2 * (c["x_off"] + C * c["ldx"] + 2), dtype=torch.float32, device="cuda")
        xb[2 * c["x_off"]: 2 * (c["x_off"] + C * c["ldx"])].view(C, c["ldx"], 2)[:, :L] = torch.from_numpy(x).cuda()
        yb = torch.full((2 * (c["y_off"] + C * c["ldy"] + 2),), float("nan"), dtype=torch.float32, device="cuda")
        px, py = xb.data_ptr() + 8 * c["x_off"], yb.data_ptr() + 8 * c["y_off"]
        torch.cuda.synchronize()
        if op == "filter":
            f.filter_dev(px, py, 2 * L, 2 * c["ldx"], 2 * c["ldy"])
        elif op == "fft":
            f.fft_filter_dev(px, py, 2 * L, 2 * c["ldx"], 2 * c["ldy"])
        else:
            got = f.decimate_dev(px, 2 * L, op, py, 2 * m, 2 * c["ldx"], 2 * c["ldy"])
            assert got == 2 * m, (row, got, m)
        torch.cuda.synchronize()
        yh = yb.cpu().numpy()
        rows = yh[2 * c["y_off"]: 2 * (c["y_off"] + C * c["ldy"])].reshape(C, c["ldy"], 2)
        clean = (np.isnan(rows[:, m:]).all() and np.isnan(yh[: 2 * c["y_off"]]).all() and
                 np.isnan(yh[2 * (c["y_off"] + C * c["ldy"]):]).all())
        out.append((rows[:, :m].copy(), clean, f.last_kernel()))
    f.close()
    return out


def _fir_launch_rows(Q):
    for r in FIR_ROWS:
        fir_run_row(Q, r, fir_row_inputs(r))


def _ddc_launch_rows(Q):
    for K, D, N, _ in DDC_ROWS:
        bank = Q.DdcBank(np.ones(N, np.float32) / N, [0.1] * K, D)
        for n in ddc_row_calls((K, D)):
            bank.process(np.ones(n, np.complex64))
        bank.close()


def _resamp_launch_rows(Q):
    for K, L, M, N, _ in RESAMP_ROWS:
        r = Q.Resampler(np.ones(N, np.float32), L, M, K)
        for n in resamp_row_calls((K, L, M)):
            r.process(np.ones((K, n), np.complex64))
        r.close()


LAUNCH_ROWS = {"fir": _fir_launch_rows, "fll": _fll_launch_rows, "mod": _mod_launch_rows, "eq": _eq_launch_rows,
               "pfb": _pfb_launch_rows, "ddc": _ddc_launch_rows, "resamp": _resamp_launch_rows}


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
