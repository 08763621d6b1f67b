"""GPU parity of every mod_shape_kernel<MT, SPS> instantiation (tests/kernel_variants.py: MOD_ROWS) against the oracle, and
the modulator's limits (96 taps per phase, fs/rs <= 256).

Pulse shaping is compared twice: with the oracle (its FFT filter, within the project's 1e-5 * max|y|), and with a float64
restatement of the polyphase sum in the modulator.cu header over the float32 taps, within a bound derived below.  The FFT
comparison alone could hide a dropped edge tap; the direct one cannot.  Without pulse shaping the output is exact.  Every
frame spans at least three tiles of the shaping kernel (n_dibits > 2 * (2048 - HP)) and ends in the middle of one."""
import ctypes as C_
import os

import numpy as np
import pytest

import kernel_variants as kv

pytestmark = pytest.mark.gpu

U32 = np.uint32
REL_TOL = 1e-5
ALPHA = 0.35
TSC = "11001010011101100100100110101100" + "01110100111001011010001101101001"
TILE = 2048                                     # symbols staged per CTA (tile + halo)
N_DIBITS = 2 * (TILE - 8) + 333                 # > 2 * (2048 - HP) for every HP >= 8, and not a multiple of any tile


def _bits(n, seed):
    return "".join(np.random.default_rng(seed).choice(["0", "1"], n))


def _hp(mt):
    return (mt + 7) & ~7


def _direct(h32, fs, rs, sym):
    """y[i] = sum_d sym[d] * h[i + (N-1-delay) - d*sps] in float64 (modulator.cu header), and per sample the sum of |terms|.
    Polyphase: with j = i + N-1-delay = q*sps + p, y[i] = (sym * h[p::sps])[q]."""
    sps = fs // rs
    n = h32.size
    D = n - 1 - (n - 1) // 2
    total = 2 * ((n - 1) // 2) + sym.size * sps
    h = h32.astype(np.float64)
    Q = sym.size + -(-2 * n // sps) + 1                                  # rows of q: past D + total for every delay
    y = np.zeros((Q, sps), np.complex128)
    a = np.zeros((Q, sps), np.float64)
    for p in range(min(sps, n)):
        hp = h[p::sps]
        c = np.convolve(sym, hp)
        y[: c.size, p] = c
        ca = np.convolve(np.abs(sym.real), np.abs(hp))                    # |sym.real| == |sym.imag| == 1/sqrt2
        a[: ca.size, p] = ca
    return y.reshape(-1)[D: D + total], a.reshape(-1)[D: D + total]


def _symbols(x0, fs, rs, n_taps):
    """the complex symbols from the exact no-pulse-shaping output: up[delay + d*sps] = sym[d]"""
    sps = fs // rs
    z = x0[0::2].astype(np.float64) + 1j * x0[1::2].astype(np.float64)
    return z[(n_taps - 1) // 2::sps]


@pytest.mark.parametrize("diff", [True, False])
@pytest.mark.parametrize("fs,rs,span", kv.MOD_ROWS)
def test_mod_variant_matches_oracle(gpu, orc, fs, rs, span, diff):
    bits = _bits(2 * N_DIBITS, fs + span)
    mt = kv.mod_mt(fs, rs, span)
    assert N_DIBITS > 2 * (TILE - _hp(mt)) and N_DIBITS > 2 * (TILE - _hp(kv.mod_mt(fs, rs, span, False)))
    o = orc.QPSKModulator(fs, rs, ALPHA, span, diff)
    g = gpu.QPSKModulator(fs, rs, ALPHA, span, diff)
    taps = g.getCoeef()
    assert np.array_equal(taps, o.getCoeef()) and taps.size == kv.mod_taps(fs, rs, span)
    # no pulse shaping: the zero-stuffed symbol train, exact
    got0, want0 = g.Modulate(bits, False), o.Modulate(bits, False)
    assert np.array_equal(got0.view(U32), want0.view(U32))
    # pulse shaping: the oracle's FFT filter
    got, want = g.Modulate(bits), o.Modulate(bits)
    assert got.shape == want.shape
    assert np.abs(got - want).max() <= REL_TOL * np.abs(want).max()
    # ... and the direct sum.  The kernel adds the MT products of a phase to a zero accumulator with fused multiply-adds, one
    # rounding each, so |error| <= gamma_MT * sum|terms|, gamma_MT = MT u / (1 - MT u), u = 2^-24 (Higham, Thm 3.1); the
    # symbols and the float32 taps are exact in float64.
    sym = _symbols(got0, fs, rs, taps.size)
    assert sym.size == N_DIBITS
    y, absum = _direct(taps.astype(np.float32), fs, rs, sym)
    u = 2.0 ** -24
    gamma = mt * u / (1 - mt * u)
    g64 = got[0::2].astype(np.float64) + 1j * got[1::2].astype(np.float64)
    assert g64.size == y.size
    bound = gamma * absum * (1 + 1e-9) + 1e-300
    bad = (np.abs(g64.real - y.real) > bound) | (np.abs(g64.imag - y.imag) > bound)
    assert not bad.any(), (int(np.argmax(bad)), int(bad.sum()))


@pytest.mark.parametrize("fs,rs,span", [(2000, 1000, 10), (4000, 1000, 10), (8000, 1000, 10), (3000, 1000, 10)])
def test_frame_batch_store_paths(gpu, orc, fs, rs, span):
    """modulate_frames_dev at SPS = 2, 4, 8 and 0 with an even and an odd row stride (in complex samples): rows at odd
    offsets take the staging path's 8-byte stores, the others the 16-byte ones.  Nothing lands in the row padding."""
    import torch
    n_payload, frames = 1100, 3                                         # 32 + 8 + 4400 dibits: three tiles and a part
    m = gpu.QPSKModulator(fs, rs, ALPHA, span, True, TSC)
    om = orc.QPSKModulator(fs, rs, ALPHA, span, True, TSC)
    assert TSC and len(TSC) // 2 + 4 * (n_payload + 2) > 2 * (TILE - _hp(kv.mod_mt(fs, rs, span)))
    ts = torch.cuda.Stream()
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream
    pay = torch.from_numpy(np.random.default_rng(fs).integers(0, 256, (frames, n_payload), dtype=np.uint8)).cuda()
    ff = m.frame_floats(n_payload, b"S", b"E")
    fc = ff // 2
    for stride_c in (fc + (fc & 1), fc + 1 - (fc & 1)):
        out = torch.full((frames * 2 * stride_c + 64,), float("nan"), dtype=torch.float32, device="cuda")
        assert m.modulate_frames_dev(pay.data_ptr(), n_payload, frames, b"S", b"E", out.data_ptr(), 2 * stride_c, s) == ff
        torch.cuda.synchronize()
        rows = out[: frames * 2 * stride_c].view(frames, 2 * stride_c).cpu().numpy()
        for f in range(frames):
            want = om.ModulateBytes(pay[f].cpu().numpy().tobytes(), b"S", b"E")
            assert want.size == ff
            assert np.abs(rows[f, :ff] - want).max() <= REL_TOL * np.abs(want).max(), (stride_c, f)
            assert np.isnan(rows[f, ff:]).all(), (stride_c, f)
        assert np.isnan(out[frames * 2 * stride_c:].cpu().numpy()).all()


def _modulate_raw(gpu, m, bits, pulse, out):
    n = C_.c_int64(0)
    b = bits.encode("latin-1")
    return gpu._native.lib().qpsk_mod_modulate_bits(m._h, b, len(b), int(pulse), out.ctypes.data_as(C_.POINTER(C_.c_float)),
                                                    out.size, C_.byref(n))


def test_modulator_limits(gpu, orc):
    bits = _bits(2 * N_DIBITS, 5)
    # 96 taps per phase is the last supported (span 95 at sps 2 is in MOD_ROWS); span 96 needs 97
    m = gpu.QPSKModulator(2000, 1000, ALPHA, 96)
    assert kv.mod_predict(2000, 1000, 96) == kv.UNSUPPORTED
    with pytest.raises(gpu.QpskCudaError, match="status -7"):
        m.Modulate(bits)
    n_out = 2 * (2 * 96 + N_DIBITS * 2)
    out = np.full(n_out, 7.25, np.float32)
    assert _modulate_raw(gpu, m, bits, True, out) == gpu._native.ERR_UNSUPPORTED
    assert (out == 7.25).all()                                             # the output is not written
    # the delta bank of the same handle has 97 taps, 49 per phase: supported
    o = orc.QPSKModulator(2000, 1000, ALPHA, 96)
    assert np.array_equal(m.Modulate(bits, False).view(U32), o.Modulate(bits, False).view(U32))
    # fs / rs = 256: one thread per phase in the 256-thread CTA
    bits_s = _bits(2 * 300, 6)
    g, o = gpu.QPSKModulator(256000, 1000, ALPHA, 4), orc.QPSKModulator(256000, 1000, ALPHA, 4)
    got, want = g.Modulate(bits_s), o.Modulate(bits_s)
    assert got.shape == want.shape and np.abs(got - want).max() <= REL_TOL * np.abs(want).max()
    assert np.array_equal(g.Modulate(bits_s, False).view(U32), o.Modulate(bits_s, False).view(U32))
    # 257 is refused, with and without pulse shaping, and writes nothing
    g = gpu.QPSKModulator(257000, 1000, ALPHA, 4)
    for pulse in (True, False):
        with pytest.raises(gpu.QpskCudaError, match="status -7"):
            g.Modulate(bits_s, pulse)
        out = np.full(2 * (257 * 300 + 2 * 1028), 7.25, np.float32)
        assert _modulate_raw(gpu, g, bits_s, pulse, out) == gpu._native.ERR_UNSUPPORTED
        assert (out == 7.25).all()


def test_modulator_launches_the_predicted_kernels(gpu):
    got = kv.launched_in_child("mod", int(os.environ.get("LOCAL_RANK", "0")))
    assert got == kv.predicted_launches("mod")
