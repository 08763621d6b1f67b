"""GPU parity of every FIR filter and decimator kernel instantiation (tests/kernel_variants.py: FIR_ROWS) against a float64
reference, at every tap-loop tail and on both sides of every dispatch threshold, and the kernel each call ran.

Reference: y in float64 over the float32 taps and inputs (products of two float32 values are exact in float64; the float64
sums are ~2^-29 of the bound below).  Every output must lie within c * u * S of it, u = 2^-24, S = sum_i |g_i| |x_i| over
the output's own products (for the real part |gI||xI| + |gQ||xQ|, for the imaginary part |gI||xQ| + |gQ||xI|).  When every
product is formed exactly or rounded once and then added to a running sum, an output whose terms pass through at most c
roundings is off by at most gamma_c * S, gamma_c = c u / (1 - c u) (Higham, Accuracy and Stability, Thm 3.1 and Lemma 3.1).
Per kernel (kernel_variants.fir_chain; G is the correlation length, HL + 2 with HL the delay line, N the taps):
  * fir_tma_kernel, real taps; fir_generic_kernel<false>, real taps: one FFMA2 / FMA chain per output from +0, one rounding
    per tap; the zero padding tap adds an exact 0.  c = N.
  * fir_tma_kernel, complex taps: two chains of N (gI * x and gQ * x), then one add or subtract.  c = N + 1.
    fir_generic_kernel<false>, complex taps: the four FMAs of a tap on one chain.  c = 2N.
  * fir_dec2_kernel: the even- and odd-tap chains A and B of G/2 sub-taps each, then A + B.  c = G/2 + 1.
  * fir_decim_tma_kernel / fir_decim_kernel <RO, NTO, NG, D>: each of the NG phase groups sums its 2 * PP * K products
    (PP = D/2/NG phase pairs, K taps per phase) on one FFMA2 chain; the NG partial sums are then added in turn.
    c = 2 * PP * K + NG - 1.
  * fir_split2_kernel: even outputs are A + B (c = G/2 + 1).  Odd outputs are (C - A') - B with C = sum fl(h0 + h1) *
    fl(X1 + X0') over G/2 sub-taps: a term of C carries the two roundings of its factors, the chain's, and the two of the
    recombination, so c = G/2 + 4 for both kinds.  The terms of C are |h0 + h1| |X1 + X0'| <= the output's own terms plus
    |h0||X0'| + |h1||X1|, which are the terms of A' and B, met once in C and once in the subtraction.  A' belongs to output
    n + 1 and B to output n - 1, so their sums are bounded by the neighbours' full-rate sums: S_n + 2 (S_{n-1} + S_{n+1}).
  * fir_exact_real_kernel, fir_generic_kernel<true>: each product rounded, 8 lane sums of N/8 terms, the lanes added 0..7,
    then the N mod 8 tail: no term passes through more than N + 2 roundings (a complex product adds one).  c = N + 2.  These
    two must also equal the oracle (ComplexFIRFilter.Filter, subsampled for decimation) bit for bit.
The full-rate decimation path (fir_subsample_kernel after a streaming filter) has the full-rate kernel's bound.  Every
output must also meet the project-wide max|err| <= 1e-5 * max|y|.

Data (kernel_variants.fir_row_taps / fir_row_inputs): taps of random sign with magnitudes in [0.5, 1.5] / sqrt(N), none
near zero, the last two of opposite sign; inputs uniform under an envelope that steps between 1 and 2^-12 every N + 97
samples, so that next to each step a single large sample meets the first or the last tap: dropping, duplicating or
misplacing one tap moves some output by far more than its bound (tests/test_kernel_variants.py checks that on the CPU for
every row).  Every call covers at least three tiles of its kernel and ends partway through one.

Impulse rows: a unit impulse (1, then j) inside a tile and one across a tile seam make every output a single product, so
the output equals the taps (every D-th tap for decimators) exactly; fir_split2_kernel's odd outputs are (h0 + h1) - h0 and
are held to 2e-7 of max|tap| instead (as in test_gpu_fir.py)."""
import os

import numpy as np
import pytest

import kernel_variants as kv

pytestmark = pytest.mark.gpu
REL_TOL = 1e-5

# FirEngine::last_kernel strings -> normalised instantiation names
LIB_NAMES = {
    "fir_tma_kernel<R=10,NT=256,complex taps>": "fir_tma_kernel<10, 256, true>",
    "fir_tma_kernel<R=10,NT=256,real taps>": "fir_tma_kernel<10, 256, false>",
    "fir_tma_kernel<R=10,NT=320,real taps>": "fir_tma_kernel<10, 320, false>",
    "fir_split2_kernel<R=10,NT=256,real taps>": "fir_split2_kernel<10, 256>",
    "fir_exact_real_kernel<NT=256>": "fir_exact_real_kernel<256>",
    "fir_generic_kernel<EXACT>": "fir_generic_kernel<true>",
    "fir_generic_kernel": "fir_generic_kernel<false>",
    "fir_dec2_kernel<R=14,NT=256,D=2>": "fir_dec2_kernel<14, 256>",
    "fir_decim_tma_kernel<RO=7,NTO=128,NG=2,D=4,dense>": "fir_decim_tma_kernel<7, 128, 2, 4, false>",
    "fir_decim_tma_kernel<RO=7,NTO=64,NG=4,D=8,repack>": "fir_decim_tma_kernel<7, 64, 4, 8, true>",
    "fir_decim_tma_kernel<RO=7,NTO=32,NG=8,D=16,repack>": "fir_decim_tma_kernel<7, 32, 8, 16, true>",
    "fir_decim_kernel<RO=7,NTO=256,NG=1,D=2>": "fir_decim_kernel<7, 256, 1, 2>",
    "fir_decim_kernel<RO=7,NTO=128,NG=2,D=4>": "fir_decim_kernel<7, 128, 2, 4>",
    "fir_decim_kernel<RO=7,NTO=64,NG=4,D=8>": "fir_decim_kernel<7, 64, 4, 8>",
    "fir_decim_kernel<RO=7,NTO=32,NG=8,D=16>": "fir_decim_kernel<7, 32, 8, 16>",
}
EXACT_KERNELS = ("fir_exact_real_kernel<256>", "fir_generic_kernel<true>")


def _id(row):
    n, cplx, mode, op, layout, phase = row
    return f"{n}-{'c' if cplx else 'r'}-{mode}-{op}-{layout}" + (f"-p{phase}" if phase else "")


def _oracle_exact(orc, taps, xs, op):
    """The oracle's streaming Filter over the calls, per channel, subsampled for decimation: per call [C, m, 2]."""
    C = xs[0].shape[0]
    per = [[] for _ in xs]
    for c in range(C):
        o = orc.ComplexFIRFilter(taps)
        ys = [o.Filter(np.ascontiguousarray(x[c].reshape(-1))).reshape(-1, 2) for x in xs]
        if isinstance(op, int):
            full = np.concatenate(ys)
            keep = full[::op]
            a, ys = 0, []
            for x in xs:
                L = x.shape[1]
                lo, hi = -(-a // op), -(-(a + L) // op)
                ys.append(keep[lo:hi])
                a += L
        for k, y in enumerate(ys):
            per[k].append(y)
    return [np.stack(p) for p in per]


@pytest.mark.parametrize("row", kv.FIR_ROWS, ids=[_id(r) for r in kv.FIR_ROWS])
def test_fir_variant_matches_reference(gpu, orc, row):
    n, cplx, mode, op = row[:4]
    taps = kv.fir_row_taps(row)
    xs = kv.fir_row_inputs(row)
    want_k = kv.fir_row_dispatch(row)
    got = kv.fir_run_row(gpu, row, xs, taps)
    refs = kv.fir_reference(taps, xs, op)
    scale = max(max(float(np.abs(np.stack([r[0].real, r[0].imag], -1)).max()) for r in refs), 1e-30)
    exact = None
    for k, ((y, clean, lk), ref, pred) in enumerate(zip(got, refs, want_k)):
        kern = pred[0][0]
        assert LIB_NAMES.get(lk) == kern, (k, lk, kern)
        assert clean, (k, "wrote outside its output rows")
        assert y.shape[:2] == ref[0].shape, (k, y.shape, ref[0].shape)
        g = y.astype(np.float64)
        er, ei = np.abs(g[..., 0] - ref[0].real), np.abs(g[..., 1] - ref[0].imag)
        br, bi = kv.fir_bound(kern, n, cplx, ref)
        bad = (er > br) | (ei > bi)
        if bad.any():
            c, m = np.argwhere(bad)[0]
            pytest.fail(f"call {k} ({kern}): {int(bad.sum())} outputs beyond the bound, first channel {c} output {m}: "
                        f"err {er[c, m]:.3e} / {ei[c, m]:.3e}, bound {br[c, m]:.3e} / {bi[c, m]:.3e}")
        assert max(float(er.max()), float(ei.max())) <= REL_TOL * scale, k
        if kern in EXACT_KERNELS:
            if exact is None:
                exact = _oracle_exact(orc, taps, xs, op)
            assert np.array_equal(y.view(np.uint32), exact[k].view(np.uint32)), (k, kern)


def _tile(kernel):
    if kernel.startswith("fir_tma_kernel<10, 320"):
        return 3200
    if kernel.startswith(("fir_tma_kernel", "fir_split2_kernel")):
        return 2560
    if kernel.startswith("fir_exact_real_kernel"):
        return 512
    if kernel.startswith(("fir_dec2_kernel", "fir_decim")):
        return 3584                                           # input samples per tile
    return 256                                                # one-thread-per-output kernels: a CTA


def _impulse_rows():
    """One single-channel row per instantiation (the first in the table), and one of the full-rate decimation path."""
    out = {}
    for r in kv.FIR_ROWS:
        if kv.FIR_LAYOUTS[r[4]][0] != 1:
            continue
        for k, _ in kv.fir_dispatch(r[0], r[1], r[2], r[3], kv.FIR_L1, 0, *kv.FIR_LAYOUTS[r[4]][1:]):
            out.setdefault(k, r)
    return sorted(out.items())


@pytest.mark.parametrize("kernel,row", _impulse_rows(), ids=[k for k, _ in _impulse_rows()])
def test_fir_impulse_gives_the_taps(gpu, kernel, row):
    n, cplx, mode, op, layout, _ = row
    T = _tile(kv.fir_dispatch(n, cplx, mode, op, kv.FIR_L1, 0, *kv.FIR_LAYOUTS[layout][1:])[0][0])
    a = T + T // 2                                            # inside the second tile
    b = -(-(a + n + 8 + 3) // T) * T - 3                      # three samples before a seam, the response across it
    L = b + n + 1001 + ((b + n) % 2)                          # odd
    C, x_off, y_off = kv.FIR_LAYOUTS[layout]
    m = kv.fir_nout(L, op, 0) if isinstance(op, int) else L
    calls = [dict(op=op, L=L, skip=0, x_off=x_off, y_off=y_off, channels=1, ldx=L, ldy=m, n_out=m)]
    taps = kv.fir_row_taps(row)
    for va, vb in ((0, 1), (1, 0)):                           # component 0 = 1, 1 = j
        x = np.zeros((1, L, 2), np.float32)
        x[0, a, va] = 1.0
        x[0, b, vb] = 1.0
        ref = kv.fir_reference(taps, [x], op)[0][0][0]
        y, clean, lk = kv.fir_run_row(gpu, row, [x], taps, calls=calls)[0]
        assert clean
        assert LIB_NAMES.get(lk) == kv.fir_dispatch(n, cplx, mode, op, L, 0, x_off, y_off)[0][0], lk
        assert np.count_nonzero(ref) >= 2 * (n // (op if isinstance(op, int) else 1)), "the impulses fell outside"
        g = y[0, :, 0].astype(np.float64) + 1j * y[0, :, 1].astype(np.float64)
        if kernel == "fir_split2_kernel<10, 256>":
            assert np.abs(y[0] - np.stack([ref.real, ref.imag], -1)).max() <= 2e-7 * np.abs(taps).max()
        else:
            assert np.array_equal(g, ref), (kernel, int(np.argmax(g != ref)))


def test_fir_launches_the_predicted_kernels(gpu):
    got = kv.launched_in_child("fir", int(os.environ.get("LOCAL_RANK", "0")))
    assert got == kv.predicted_launches("fir")
