"""Per-output error bounds of the DDC bank (csrc/ddc.cu), the PFB channelizer (csrc/pfb.cu) and the rational resampler
(csrc/resamp.cu), derived from each kernel's arithmetic; fp64 references on the fp32 taps the kernels receive; the row
tables' taps and inputs; and the tap, history, phase and index slips whose effect the bounds must see.

Notation: u = 2^-24, gamma_n = n u / (1 - n u).  A chain acc = fma(a_q, b_q, acc) from +0 over n terms is off by at most
gamma_n * sum_q |a_q| |b_q| (Higham, Accuracy and Stability, Lemma 3.1 and Thm 3.1; a term whose factor is an exact zero
adds an exact zero).  |.| of a complex number is its modulus.  For a product of computed complex values d (computed) and t
(rounded from fp64) evaluated as (fma(d.re, t.re, -fl(d.im t.im)), fma(d.re, t.im, fl(d.im t.re))) -- the form of the PFB
butterflies and of the DDC epilogue -- each component is (exact + p)(1 + e2) with the inner product rounded once,
p = fl(d.im t.x) - d.im t.x, so the result is within u|d t| + u (1 + u) |d.im| |t| <= u (2 + u) |d| |t| of d t.

Every kernel rounds no input: taps and samples arrive as fp32, and the references below take those fp32 values into fp64,
where each product of two fp32 values is exact.  The references' own error (fp64 sums, fp64 FFT, fp64 angles) is below
2^-40 of the bounds; every bound is multiplied by REF_SLACK = 1 + 2^-20 for it.  FLOOR = 2^-120 covers gradual underflow
(at most 2^-150 per rounding; the kernels are built without flush-to-zero).

Resampler, both shapes (resamp_kernel<CW, CPT, OPT, CJ>).  Output m of channel c is acc = fma((h, h), (x.re, x.im), acc)
from +0 over q = 0..P-1 in increasing q (h = hT[phi_m][q] = h[phi_m + qL], zero past N; x = z[n_m - q]), whatever the tile
shape or chunk: re and im are each one FMA chain of P terms, so
    |dy.re| <= gamma_P * sum_q |h[phi_m + qL]| |x[n_m - q].re|,   and the same for im with x.im.
The sums are upfirdn(|h|, |x.re|, L, M) (resamp_reference forms them with the index arrays of y).

DDC, both shapes (ddc_kernel<CQW, WC, CC>).  The host forms g_k[i] = h_i e^{+j theta_k(i)} in fp64 and rounds each
component to fp32: |g^ - g| <= u_t |h_i| per component, u_t = u + 2^-44 (u for the rounding; the fp64 product, cos / sin
and angle are good to 2^-48 |h_i|).  The kernel forms rr = sum g^.re (x.re, x.im) and ii = sum g^.im (x.re, x.im) as FFMA2
chains over r = 0..NP-1 (tap N-1-r); rows r >= N hold zero taps and zeroed samples, so each chain has N terms.  Then
ur = fl(rr.x - ii.y), ui = fl(rr.y + ii.x).  With A = sum_i |h_i| (|x_i.re| + |x_i.im|) and u_k[m] the exact sum,
each of ur, ui is off by at most u |u_k| + (1 + u) E1, E1 = (u_t + gamma_N (1 + u_t)) A, so the complex error of u^ is
    du <= u |u_k| + sqrt2 (1 + u) E1.
Epilogue: the exact rotation is e^{-j theta}, theta = 2 pi phi / 2^64 with phi = inc_k n_m mod 2^64.  The kernel takes the
top 32 bits of phi (an angle error below pi 2^-31 rad), converts that int to fp32 (|int| < 2^31: half an ulp is 2^6, i.e.
pi 2^-25 rad after the exact scaling by 2^-31), so its angle theta' has |theta' - theta| <= eps_theta = pi (2^-31 + 2^-25).
sincospif is accurate to 1 ulp in each of sin and cos (CUDA C++ Programming Guide 12.9, appendix "Mathematical Functions",
single-precision table: sinpif, cospif, sincospif 1 ulp), so the rounded rotation e^ is within 2u of e^{-j theta'}.  The
product u^ e^ (one rounded product and one FMA per component) adds u (2 + u) |u^| |e^|.  Altogether
    |dy| <= (u (2 + u)(1 + 2u) + 2u + eps_theta) |u_k| + (1 + 2u)(1 + u (2 + u)) du
          = c1 u A + (eps_theta + c2 u) |u_k|,   c1 ~ sqrt2 (N + 1), c2 ~ 5,
and each of re, im is within |dy|.  The bound is the same for re and im.

PFB (pfb_kernel<P>).  Branch sums v_r[m] = sum_q h[qM + r] x[(m-q)M + M-1-r] are FMA chains of P terms from +0 per
component, so v^_r = v_r + e_r with |e_r| <= gamma_P hypot(S_r.re, S_r.im), S_r.re = sum_q |h| |x.re| (the same for im).
The inverse DFT runs log2 M radix-2 decimation-in-frequency stages (the code fuses pairs of them into radix-2^2 passes, after
one lone radix-2 stage when log2 M is odd); each output of a stage is either fl(a + c) (one rounding per component: error
<= u |a + c|) or fl((a - c) t^): a - c rounded per component (|d^ - d| <= u |d|), t^ the twiddle rounded from fp64
(|t^ - t| <= u' = u + 2^-45, |t^| <= 1 + u'), then the product (u (2 + u) |d^| |t^|).  So each stage output is the exact
butterfly on the computed inputs (exact twiddle) plus xi with |xi| <= eta |a -+ c| <= eta (|a| + |c|),
    eta = u (1 + u') + u' + u (2 + u)(1 + u)(1 + u')  (~ 4u).
Each output Y_k depends on the branch sums through a binary tree: 2^(S-s) nodes at stage s, S = log2 M, whose parents are
disjoint and are all the nodes of the tree at stage s-1.  Let A_s be the sum of |computed value| over the tree's nodes at
stage s; then A_s <= (1 + eta) A_{s-1} and the local errors of stage s total at most eta A_{s-1} <= eta (1+eta)^(s-1) A_0.
The exact butterflies carry errors forward with unit-modulus weights, so by induction over the stages
    |dY_k| <= sum_r |e_r| + ((1+eta)^S - 1) A_0,   A_0 = sum_r |v^_r| <= sum_r (|v_r| + |e_r|),
    B_m = (1+eta)^S sum_r gamma_P hypot(S_r.re, S_r.im) + ((1+eta)^S - 1) sum_r |v_r[m]|,
the same for every channel of block m and for re and im.  (sqrt2 max(S.re, S.im) >= hypot(S.re, S.im): the hypot form is the
tighter of the two.)"""
import math

import numpy as np

import kernel_variants as kv
from ddc_oracle import phase_angle, phase_word, scene_taps
from resamp_oracle import resamp_count, resamp_taps

U = 2.0 ** -24
REF_SLACK = 1.0 + 2.0 ** -20
FLOOR = 2.0 ** -120


def gamma(n):
    return n * U / (1.0 - n * U)


# ---- taps and inputs -----------------------------------------------------------------------------------------------------
def kaiser_pfb(M, P):
    """qpsk_pfb_taps(M, P, 0.5 / M, 60): a Kaiser-windowed sinc of P*M taps, unit DC gain (scipy's firwin is the same)."""
    from scipy.signal import firwin, kaiser_beta
    return firwin(P * M, 1.0 / M, window=("kaiser", kaiser_beta(60.0)), scale=True)


def row_taps(N, kind, kaiser):
    """fp32 taps: fir_row_taps' recipe (random signs, magnitudes in [0.5, 1.5] / sqrt(N), the last two of opposite sign) or
    the library's Kaiser prototype `kaiser()`."""
    if kind == "kaiser":
        h = np.asarray(kaiser(), np.float32)
        assert h.size == N
        return h
    return kv.fir_row_taps((N, False))[0::2].copy()


# The envelope's small level.  The Kaiser prototypes' edge taps are 1e-4..1e-8 of their largest: at 2^-12 the small
# samples' own products, rounded, would hide them.  At 2^-36 an edge tap meeting a large sample stands above the rounding
# of everything else (products stay far above the fp32 normal range's end, even at the resampler's 2^-20 rows).
SMALL = {"rand": 2.0 ** -12, "kaiser": 2.0 ** -36}


def _envelope(total, seg, small, seam):
    """1 and `small` in alternate segments of `seg`, placed so that the seam between the calls falls mid-way through a
    segment at 1: the second call's first outputs then read a history whose one-sample slip is large."""
    off = (seg // 2 - seam) % seg
    off += seg * (((seam + off) // seg) % 2)
    return np.where(((np.arange(total) + off) // seg) % 2 == 0, 1.0, small)


def _split(x, ns):
    out, a = [], 0
    for n in ns:
        out.append(np.ascontiguousarray(x[..., a: a + n]))
        a += n
    return out


def _uniform_cx(rng, shape):
    return rng.uniform(-1.0, 1.0, shape) + 1j * rng.uniform(-1.0, 1.0, shape)


# ---- resampler -----------------------------------------------------------------------------------------------------------
def resamp_row_taps(row):
    K, L, M, N, kind = row
    return row_taps(N, kind, lambda: resamp_taps(L, M))


def resamp_row_inputs(row):
    """Per call a [K, n] complex64 input: uniform samples under an envelope that alternates between 1 and SMALL in
    segments of ceil((N + 97) / L) input samples (N + 97 samples of the upsampled stream), channel c scaled by 2^e_c with
    e_c spread over -20..20."""
    K, L, M, N, kind = row
    ns = kv.resamp_row_calls(row)
    rng = np.random.default_rng(kv._seed("resamp x", row))
    env = _envelope(sum(ns), -(-(N + 97) // L), SMALL[kind], ns[0])
    scale = 2.0 ** np.round(np.linspace(-20, 20, K))
    x = (_uniform_cx(rng, (K, sum(ns))) * env[None, :] * scale[:, None]).astype(np.complex64)
    return _split(x, ns)


def _stale(x, a):
    """The stream as a call starting at input a would see it with its history one sample stale."""
    s = x.copy()
    s[..., 1:a] = x[..., : a - 1]
    s[..., :1] = 0
    return s


def _tap_mutation(h, mutation):
    h = h.copy()
    if mutation == "h[0] zeroed":
        h[0] = 0.0
    elif mutation == "h[N-1] zeroed":
        h[-1] = 0.0
    elif mutation == "last two taps swapped":
        h[-2], h[-1] = h[-1], h[-2]
    return h


def resamp_reference(h32, L, M, xs, mutation=None):
    """Per call (y [K, t] complex128, bound_re, bound_im) of the stream xs (the calls' inputs, [K, n] each)."""
    h = _tap_mutation(np.asarray(h32, np.float32).astype(np.float64), mutation)
    N = h.size
    P = -(-N // L)
    hp = np.zeros(P * L)
    hp[:N] = h
    hT = hp.reshape(P, L).T                                      # hT[phi, q] = h[phi + qL]
    x = np.concatenate(xs, axis=1).astype(np.complex128)
    K = x.shape[0]
    out, a = [], 0
    for k, xc in enumerate(xs):
        n = xc.shape[1]
        s = x[:, : a + n]
        if mutation == "history one sample stale" and k > 0:
            s = _stale(s, a)
        m = np.arange(resamp_count(a, L, M), resamp_count(a + n, L, M), dtype=np.int64)
        n_m, phi = m * M // L, m * M % L
        if mutation == "branch + 1":
            phi = (phi + 1) % L
        elif mutation == "n_m - 1":
            n_m = n_m - 1
        z = np.concatenate([np.zeros((K, P + 1)), s], axis=1)
        w = z[:, n_m[:, None] - np.arange(P)[None, :] + P + 1]          # [K, t, P]
        taps = hT[phi]                                                  # [t, P]
        y = np.einsum("tq,ktq->kt", taps, w)
        at = np.abs(taps)
        g = gamma(P) * REF_SLACK
        out.append((y, g * np.einsum("tq,ktq->kt", at, np.abs(w.real)) + FLOOR,
                    g * np.einsum("tq,ktq->kt", at, np.abs(w.imag)) + FLOOR))
        a += n
    return out


RESAMP_MUTATIONS = ("h[0] zeroed", "h[N-1] zeroed", "last two taps swapped", "history one sample stale", "branch + 1",
                    "n_m - 1")


def resamp_mutations(row):
    K, L, M, N, kind = row
    P = -(-N // L)
    skip = {"last two taps swapped"} if N < 2 else set()
    if P == 1:
        skip.add("history one sample stale")             # no history: each output reads one input sample
    if L == 1:
        skip.add("branch + 1")                           # one branch
    return [m for m in RESAMP_MUTATIONS if m not in skip]


# ---- DDC bank ------------------------------------------------------------------------------------------------------------
def ddc_freqs(K):
    """K channel frequencies 0.1037 apart, none closer to 0 than 0.07 cycles per sample, so that a phase slip shows."""
    return [float((0.0731 + 0.1037 * k + 0.5) % 1.0 - 0.5) for k in range(K)]


def ddc_row_taps(row):
    K, D, N, kind = row
    return row_taps(N, kind, lambda: scene_taps(D, N // D))


def ddc_row_inputs(row):
    """Per call one complex64 stream: a 0 dB carrier on channel 0's frequency, a -60 dB carrier on channel 1's and uniform
    noise at -84 dB, under an envelope that alternates between 1 and SMALL in segments of N + 97 samples."""
    K, D, N, kind = row
    ns = kv.ddc_row_calls(row)
    total = sum(ns)
    f = ddc_freqs(K)
    rng = np.random.default_rng(kv._seed("ddc x", row))
    t = np.arange(total)
    with np.errstate(over="ignore"):
        c = (np.exp(1j * phase_angle(phase_word(f[0]), t)) + 1e-3 * np.exp(1j * phase_angle(phase_word(f[1]), t)) +
             2.0 ** -14 * _uniform_cx(rng, total))
    env = _envelope(total, N + 97, SMALL[kind], ns[0])
    return _split((c * env).astype(np.complex64), ns)


def ddc_bound(N, A, au):
    """|dy| bound of one output from A = sum |h| (|x.re| + |x.im|) and |u_k[m]| (module docstring)."""
    ut = U + 2.0 ** -44
    e1 = (ut + gamma(N) * (1 + ut)) * A
    du = U * au + math.sqrt(2.0) * (1 + U) * e1
    eps_theta = math.pi * (2.0 ** -31 + 2.0 ** -25)
    b = (U * (2 + U) * (1 + 2 * U) + 2 * U + eps_theta) * au + (1 + 2 * U) * (1 + U * (2 + U)) * du
    return b * REF_SLACK + FLOOR


def ddc_reference(h32, freqs, D, xs, mutation=None):
    """Per call (y [K, t] complex128, bound, bound) of the stream xs."""
    h = _tap_mutation(np.asarray(h32, np.float32).astype(np.float64), mutation)
    N = h.size
    inc = [phase_word(f) for f in freqs]
    i = np.arange(N)
    with np.errstate(over="ignore"):
        G = np.array([h * np.exp(1j * phase_angle(c, i)) for c in inc])        # [K, N]
    rot_inc = inc[1:] + inc[:1] if mutation == "channel k+1's phase word" else inc
    x = np.concatenate(xs).astype(np.complex128)
    out, a = [], 0
    for k, xc in enumerate(xs):
        n = xc.size
        s = x[: a + n]
        if mutation == "history one sample stale" and k > 0:
            s = _stale(s, a)
        m = np.arange(a // D, (a + n) // D, dtype=np.int64)
        n_m = m * D + D - 1
        z = np.concatenate([np.zeros(N), s])
        W = z[n_m[:, None] - i[None, :] + N]                                  # [t, N]: W[t, i] = x[n_m - i]
        u = G @ W.T
        A = np.abs(h) @ (np.abs(W.real) + np.abs(W.imag)).T
        ph = n_m - 1 if mutation == "phase at n_m - 1" else n_m
        with np.errstate(over="ignore"):
            rot = np.array([np.exp(-1j * phase_angle(c, ph.astype(np.uint64))) for c in rot_inc])
        b = ddc_bound(N, A[None, :], np.abs(u))
        out.append((u * rot, b, b))
        a += n
    return out


DDC_MUTATIONS = ("h[0] zeroed", "h[N-1] zeroed", "last two taps swapped", "history one sample stale", "phase at n_m - 1",
                 "channel k+1's phase word")


def ddc_mutations(row):
    return list(DDC_MUTATIONS)


# ---- PFB channelizer -----------------------------------------------------------------------------------------------------
PFB_TILE_BLOCKS = 8192                  # pfb_run_blocks: T = 8192 / M blocks per CTA at every M
# (P, M, taps): every channelizer row of tests/kernel_variants.py, and the library's prototype at M = 1024, P = 16
PFB_BANK_ROWS = [(P, M, "rand") for P, M in kv.PFB_ROWS] + [(16, 1024, "kaiser")]


def pfb_row_ntaps(row):
    P, M, kind = row
    return P * M if kind == "kaiser" else kv.pfb_taps(P, M)


def pfb_row_calls(row):
    """Input samples of a row's two calls: at least three tiles and four envelope segments of whole blocks each, and a
    ragged end; the first leaves samples of an open block pending."""
    P, M, kind = row
    seg = -(-(pfb_row_ntaps(row) + 97) // M)
    b = max(3 * (PFB_TILE_BLOCKS // M) + 3, 4 * seg + 3)
    return [b * M + max(1, M // 2 - 1), b * M + 3]


def pfb_row_taps(row):
    P, M, kind = row
    return row_taps(pfb_row_ntaps(row), kind, lambda: kaiser_pfb(M, P))


def pfb_row_inputs(row):
    """Per call one complex64 stream: uniform samples under an envelope that alternates between 1 and SMALL in segments of
    ceil((N + 97) / M) whole blocks."""
    P, M, kind = row
    ns = pfb_row_calls(row)
    total = sum(ns)
    rng = np.random.default_rng(kv._seed("pfb x", row))
    seg = -(-(pfb_row_ntaps(row) + 97) // M)
    env = np.repeat(_envelope(-(-total // M), seg, SMALL[kind], ns[0] // M), M)[:total]
    return _split((_uniform_cx(rng, total) * env).astype(np.complex64), ns)


def pfb_twiddles(M):
    return np.exp(2j * np.pi * np.arange(M // 2) / M)


def _bitrev(M):
    bits = M.bit_length() - 1
    return np.array([int(format(k, f"0{bits}b")[::-1], 2) if bits else 0 for k in range(M)])


def pfb_dif(v, tw):
    """The kernel's inverse DFT restated: radix-2 decimation in frequency over the rows of v [t, M] with twiddle table tw
    (span h uses tw[j * M / (2h)]), read out in bit-reversed order: Y[:, k] = sum_r v[:, r] e^{+j 2 pi r k / M}."""
    t, M = v.shape
    w = v.copy()
    h = M // 2
    while h >= 1:
        w = w.reshape(t, M // (2 * h), 2, h)
        a, c = w[:, :, 0, :], w[:, :, 1, :]
        w = np.stack([a + c, (a - c) * tw[np.arange(h) * (M // (2 * h))]], axis=2).reshape(t, M)
        h //= 2
    return w[:, _bitrev(M)]


def pfb_eta():
    up = U + 2.0 ** -45
    return U * (1 + up) + up + U * (2 + U) * (1 + U) * (1 + up)


def pfb_reference(h32, M, xs, mutation=None):
    """Per call (Y [M, t] complex128, bound [1, t], bound [1, t]) of the stream xs."""
    h = _tap_mutation(np.asarray(h32, np.float32).astype(np.float64), mutation)
    N = h.size
    P = -(-N // M)
    hp = np.zeros(P * M)
    hp[:N] = h
    H = hp.reshape(P, M)                                                 # H[q, r] = h[qM + r]
    Hv = H.copy()
    if mutation == "q = P-1 dropped in branch 0":
        Hv[P - 1, 0] = 0.0
    elif mutation == "q = P-1 dropped in branch M-1":
        Hv[P - 1, M - 1] = 0.0
    tw = pfb_twiddles(M)
    if mutation == "twiddle conjugated":
        tw = tw.copy()
        tw[M // 4] = np.conj(tw[M // 4])                                # +j: used once in every stage of span >= 2
    S = M.bit_length() - 1
    g = (1 + pfb_eta()) ** S
    x = np.concatenate(xs).astype(np.complex128)
    out, a = [], 0
    for k, xc in enumerate(xs):
        n = xc.size
        s = x[: a + n]
        if mutation == "history one sample stale" and k > 0:
            s = _stale(s, a)
        m0, m1 = a // M, (a + n) // M
        t = m1 - m0
        j0 = m0 - P + 1                                                  # oldest block read
        Zr = np.zeros((t + P - 1, M), np.complex128)                     # Zr[j - j0, r] = s[jM + M-1-r]
        lo = max(0, j0)
        Zr[lo - j0:] = s[lo * M: m1 * M].reshape(-1, M)[:, ::-1]
        v = np.zeros((t, M), np.complex128)
        sr = np.zeros((t, M))
        si = np.zeros((t, M))
        for q in range(P):
            blk = Zr[P - 1 - q: P - 1 - q + t]
            v += Hv[q] * blk
            sr += np.abs(H[q]) * np.abs(blk.real)
            si += np.abs(H[q]) * np.abs(blk.imag)
        Y = pfb_dif(v, tw)
        if mutation == "channels exchanged":
            k1, k2 = (1, M // 2) if M >= 4 else (0, 1)
            Y[:, [k1, k2]] = Y[:, [k2, k1]]
        b = (g * gamma(P) * np.hypot(sr, si).sum(1) + (g - 1) * np.abs(v).sum(1)) * REF_SLACK + FLOOR
        out.append((Y.T, b[None, :], b[None, :]))
        a += n
    return out


PFB_MUTATIONS = ("h[0] zeroed", "h[N-1] zeroed", "last two taps swapped", "history one sample stale",
                 "q = P-1 dropped in branch 0", "q = P-1 dropped in branch M-1", "channels exchanged", "twiddle conjugated")


def pfb_mutations(row):
    P, M, kind = row
    skip = set()
    if (P - 1) * M + M - 1 >= pfb_row_ntaps(row):
        skip.add("q = P-1 dropped in branch M-1")        # that term is zero padding: dropping it changes nothing
    if M == 2:
        skip.add("twiddle conjugated")                   # the only twiddle is 1
    return [m for m in PFB_MUTATIONS if m not in skip]


# ---- which mutations the Kaiser rows promise to show ---------------------------------------------------------------------
# The random-tap rows promise every mutation that applies.  With the small level at 2^-36, the resampler's and the DDC's
# Kaiser rows show every one too: each edge tap meets a large sample while the rest of its output's terms are small.  The
# channelizer's 16384-tap prototype cannot: an edge tap (1e-8 of the largest) meets its block together with the other
# 1023 taps of its tap row, and the DFT's rounding of that row's branch sums outweighs it whatever the small level.  There
# only the slips that move whole outputs are promised.
KAISER_PROMISED = {
    "resamp": RESAMP_MUTATIONS,
    "ddc": DDC_MUTATIONS,
    "pfb": ("history one sample stale", "channels exchanged", "twiddle conjugated"),
}


# ---- the three blocks behind one interface ---------------------------------------------------------------------------------
def block_rows(block):
    return {"resamp": kv.RESAMP_ROWS, "ddc": kv.DDC_ROWS, "pfb": PFB_BANK_ROWS}[block]


def row_case(block, row):
    """(taps, inputs per call, reference(taps, xs, mutation), mutations) of a row."""
    if block == "resamp":
        K, L, M, N, kind = row
        return (resamp_row_taps(row), resamp_row_inputs(row), lambda h, xs, mu=None: resamp_reference(h, L, M, xs, mu),
                resamp_mutations(row))
    if block == "ddc":
        K, D, N, kind = row
        f = ddc_freqs(K)
        return (ddc_row_taps(row), ddc_row_inputs(row), lambda h, xs, mu=None: ddc_reference(h, f, D, xs, mu),
                ddc_mutations(row))
    P, M, kind = row
    return pfb_row_taps(row), pfb_row_inputs(row), lambda h, xs, mu=None: pfb_reference(h, M, xs, mu), pfb_mutations(row)


def promised(block, row, mutations):
    return [m for m in mutations if row[-1] != "kaiser" or m in KAISER_PROMISED[block]]


def row_id(block, row):
    return f"{block}-" + "-".join(str(v) for v in row)


# ---- GPU side: a row's two calls through the device entry points ----------------------------------------------------------
def run_row(Q, block, row, taps, xs, counts):
    """Run the row's calls on one handle through process_dev, input and output one sample past a 16-byte boundary, output
    rows of odd stride (in samples) and, for the resampler, input rows of odd stride; `counts`: the outputs per channel each
    call must complete.  Returns per call (y [C, t] complex64, whether the row padding and the buffer ends around the rows
    were left untouched)."""
    import torch
    if block == "resamp":
        K, L, M, N, kind = row
        h, C = Q.Resampler(taps, L, M, K), K
    elif block == "ddc":
        K, D, N, kind = row
        h, C = Q.DdcBank(taps, ddc_freqs(K), D), K
    else:
        P, M, kind = row
        h, C = Q.PfbChannelizer(taps, M), M
    out = []
    ts = torch.cuda.Stream()
    with torch.cuda.stream(ts):
        for x, t in zip(xs, counts):
            n = x.shape[-1]
            if block == "resamp":
                ldx = n + 5
                xb = torch.zeros(2 * (1 + K * ldx + 1), dtype=torch.float32, device="cuda")
                xb[2: 2 + 2 * K * ldx].view(K, ldx, 2)[:, :n] = torch.from_numpy(x.view(np.float32).reshape(K, n, 2)).cuda()
            else:
                xb = torch.zeros(2 * (n + 2), dtype=torch.float32, device="cuda")
                xb[2: 2 + 2 * n] = torch.from_numpy(x.view(np.float32)).cuda()
            ldy = t + 3 + (t & 1)
            yb = torch.full((2 * (1 + C * ldy + 1),), float("nan"), dtype=torch.float32, device="cuda")
            px, py = xb.data_ptr() + 8, yb.data_ptr() + 8
            if block == "resamp":
                nf = h.process_dev(px, 2 * n, py, 2 * ldy, in_stride=2 * ldx, stream=ts.cuda_stream)
            else:
                nf = h.process_dev(px, 2 * n, py, 2 * ldy, ts.cuda_stream)
            assert nf == 2 * t, (row, nf, t)
            ts.synchronize()
            yh = yb.cpu().numpy()
            rows = yh[2: 2 + 2 * C * ldy].reshape(C, ldy, 2)
            clean = bool(np.isnan(rows[:, t:]).all() and np.isnan(yh[:2]).all() and np.isnan(yh[2 + 2 * C * ldy:]).all())
            out.append((np.ascontiguousarray(rows[:, :t]).view(np.complex64)[..., 0], clean))
    h.close()
    return out
