"""Which symbol-stage kernel a demodulator call runs, predicted from its public inputs and read back from the profiler.

`predict` restates DemodEngine's dispatch (csrc/demod.cu: can_fuse, can_fuse_mf, mf_warps, launch_symsync and the
kernel's mf_nb / ring_n) in plain Python; `launched_kernels` runs one call under torch.profiler and returns the CUDA
kernels it launched, and `symsync_variants` picks the symsync_decode_kernel<DIFF, MFW, DENSE> instantiations out of them.
`GEOMETRIES` is the table of rate / span rows the parity tests run; tests/test_symsync_dispatch.py checks on the CPU that
it reaches every variant the dispatch can produce."""
import re

K_SS_BLOCK = 32               # samples per round of the symbol-stage kernel
K_MF_MAX_TAPS = 65            # longest matched filter the kernel takes in
K_MF_REG_TAPS = 31            # taps held in registers (NB = 1..3 blocks of eight + a tail)

# (fs, rs, span) -> N = span * round(fs / rs) + 1 taps (banker's rounding, as the reference's Math.Round)
GEOMETRIES = {
    7: (2000, 1000, 3),       # constant bank, tail only
    9: (2000, 1000, 4),       # registers, NB = 1
    25: (2000, 1000, 12),     # registers, NB = 3
    29: (2000, 1000, 14),     # registers, NB = 3; the last tap count with two filter warps at sps 2
    31: (2000, 1000, 15),     # registers, NB = 3 (= K_MF_REG_TAPS); four filter warps
    33: (2000, 1000, 16),     # constant bank; the 96-slot ring exactly full
    34: (3000, 1000, 11),     # constant bank, 128-slot ring
    41: (4000, 1000, 10),     # constant bank, 128-slot ring
    "9w4": (8000, 1000, 1),   # registers, NB = 1, four filter warps
    "17w4": (4000, 1000, 4),  # registers, NB = 2, four filter warps
    65: (8000, 1000, 8),      # constant bank, the longest fused filter
    "65s16": (16000, 1000, 4),
    21: (5000, 2000, 10),     # registers, NB = 2, non-integer rate 2.5
    11: (5000, 4000, 10),     # registers, NB = 1, rate 1.25: the lowest fused rate (sps - 0.1 > 1)
    "33w2": (5000, 4000, 32),  # constant bank, 96-slot ring, two filter warps (rate 1.25)
    "41w2": (5000, 4000, 40),  # constant bank, 128-slot ring, two filter warps (rate 1.25)
    "1w4": (64000, 1000, 0),  # a one-tap filter (span 0) at 64 samples per symbol: constant bank, four filter warps
    81: (8000, 1000, 10),     # not fused: <DIFF, 0> behind the separate exact filter
}

# rows the variant matrix runs at 33 (or 95) channels, and the two-filter-warp rows the DENSE test runs at
# 96 x SM and 96 x SM + 33 channels (DENSE exists only with two filter warps)
MATRIX_ROWS = tuple(GEOMETRIES)
DENSE_ROWS = (7, 9, 21, 25, "33w2", "41w2")

TAPS_CLASSES = ("reg1", "reg2", "reg3", "const_short", "const_long")

# Combinations of (MFW, DENSE, taps class, ring) the kernel cannot run, with the reason.  DIFF is free everywhere.
UNREACHABLE = [
    (lambda mfw, dense, taps, ring: mfw == 4 and dense,
     "DENSE is an instantiation of the two-filter-warp kernel only"),
    (lambda mfw, dense, taps, ring: mfw == 0 and dense,
     "DENSE is an instantiation of the two-filter-warp kernel only"),
    (lambda mfw, dense, taps, ring: mfw == 0 and (taps is not None or ring is not None),
     "without the fused filter there are no filter taps or raw-sample ring in the kernel"),
    (lambda mfw, dense, taps, ring: mfw > 0 and (taps is None or ring is None),
     "the fused filter always has a taps path and a ring"),
    (lambda mfw, dense, taps, ring: taps in ("reg1", "reg2", "reg3", "const_short") and ring == 128,
     "register taps and the short constant-bank path mean N <= 31, so N - 1 <= 32 and the ring has 96 slots"),
]


def n_taps(fs, rs, span):
    return int(span) * int(round(fs / rs)) + 1


def taps_class(n):
    if 8 <= n <= K_MF_REG_TAPS:
        return "reg%d" % (n >> 3)
    return "const_short" if n < 8 else "const_long"


def predict(channels, fs, rs, span, diff=True, exact=True, sm_count=148):
    """-> dict(diff, mfw, dense, taps, ring) of the symsync_decode_kernel a DeModulate call launches, or None when the
    call does not run that kernel (sps - 0.1 <= 1: the separate Mueller-Muller / decode kernels)."""
    sps = fs / rs
    if not (sps - 0.1 > 1.0):
        return None
    n = n_taps(fs, rs, span)
    if channels < 32 or not exact or not (1 <= n <= K_MF_MAX_TAPS):
        return dict(diff=bool(diff), mfw=0, dense=False, taps=None, ring=None)
    round_cycles = 340.0 * K_SS_BLOCK / sps
    mfw = 2 if 110.0 * n <= 0.6 * round_cycles else 4
    grid = (channels + 31) // 32
    dense = mfw == 2 and grid > 3 * sm_count
    return dict(diff=bool(diff), mfw=mfw, dense=dense, taps=taps_class(n), ring=96 if n - 1 <= 32 else 128)


def kernel_name(v):
    """The template arguments as the demangled name prints them."""
    b = lambda x: "true" if x else "false"
    return f"symsync_decode_kernel<{b(v['diff'])}, {v['mfw']}, {b(v['dense'])}>"


def unreachable_reason(mfw, dense, taps, ring):
    for rule, why in UNREACHABLE:
        if rule(mfw, dense, taps, ring):
            return why
    return None


# ---- profiler side (needs a GPU) ------------------------------------------------------------------------------------
SYMSYNC_RE = re.compile(r"symsync_decode_kernel<(true|false), (\d), (true|false)>")


def launched_kernels(fn):
    """Run fn() under torch.profiler (CUDA activity only) and return (fn's result, names of the CUDA kernels launched).
    A trace without a single kernel means the profiler saw nothing, which would make every check on it vacuous."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    names = [n for n in names if not n.startswith("Memcpy") and not n.startswith("Memset")]
    assert names, "torch.profiler recorded no CUDA kernel for this call: cannot tell which kernel ran"
    return out, names


def symsync_variants(names):
    """{'symsync_decode_kernel<DIFF, MFW, DENSE>'} seen in a list of kernel names."""
    out = set()
    for n in names:
        m = SYMSYNC_RE.search(n)
        if m:
            out.add(f"symsync_decode_kernel<{m.group(1)}, {m.group(2)}, {m.group(3)}>")
    return out


# ---- call plan: time chunks and route of one DeModulate call ---------------------------------------------------------
def pipeline_chunks(L, channels):
    """DemodEngine::pipeline_chunks: time chunks of a fused call with the FLL on."""
    n = 6 if channels <= 4096 else 4
    if L < 2048:
        n = 1
    while n > 1 and L < n * 8 * K_SS_BLOCK:
        n -= 1
    return n


def host_chunks(L, channels, cs16):
    """DemodEngine::host_chunks: copy chunks of a fused call on host samples, >= 8 MiB each, at most 6."""
    n = min(max(int(L * channels * (4.0 if cs16 else 8.0) / (8.0 * 1024 * 1024)), 1), 6)
    while n > 1 and L < n * 8 * K_SS_BLOCK:
        n -= 1
    return n


def chunks(L, channels, use_fll, host=False, cs16=False, fused=True):
    """Time chunks one call runs in (DemodEngine::plan); an unfused call is always one."""
    if not fused:
        return 1
    n = pipeline_chunks(L, channels) if use_fll else 1
    return max(n, host_chunks(L, channels, cs16)) if host else n


# rows of tests/test_gpu_demod_routes.py, span 10 and EXACT filter: one call of L samples each
ROUTE_ROWS = {
    "device_fll": dict(channels=256, fs=4000, rs=1000, L=4196, use_fll=True),
    "device": dict(channels=256, fs=4000, rs=1000, L=4196),
    "host_cf32": dict(channels=600, fs=4000, rs=1000, L=7200, host=True),
    "host_cs16": dict(channels=600, fs=4000, rs=1000, L=7200, host=True, cs16=True),
    "mf_separate": dict(channels=16, fs=4000, rs=1000, L=4196),
    "eq": dict(channels=256, fs=4000, rs=1000, L=4196, eq=True),
    "sps_1.05": dict(channels=256, fs=2100, rs=2000, L=4196),
}
ROUTES = ("pipeline_device", "pipeline_host", "single_mf_fused", "single_mf_separate", "unfused")


def route(row):
    """-> (route, chunks) of a ROUTE_ROWS row: the time-chunk pipeline from a device or a host source, a single launch of
    the symbol-stage kernel with the matched filter inside or separate, or the unfused MM -> Costas -> decode chain."""
    fused = not row.get("eq") and predict(row["channels"], row["fs"], row["rs"], 10) is not None
    n = chunks(row["L"], row["channels"], row.get("use_fll", False), row.get("host", False), row.get("cs16", False), fused)
    if not fused:
        return "unfused", n
    if n > 1:
        return ("pipeline_host" if row.get("host") else "pipeline_device"), n
    return ("single_mf_fused" if predict(row["channels"], row["fs"], row["rs"], 10)["mfw"] else "single_mf_separate"), n
