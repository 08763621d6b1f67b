"""GPU parity of the decimate-by-D matched filter (north_star item (2); SURVEY §8d) through the C ABI.

The reference's matched filter is non-decimating (FIRFilter.cs:80-91), so the oracle is ComplexFIRFilter.Filter()'s output
kept at stream indices 0, D, 2D, ...  Tolerance: max |err| <= 1e-5 * max|y| in QPSK_FIR_FAST (fir_decim_kernel), bit-exact
in QPSK_FIR_EXACT."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
REL_TOL = 1e-5


def _taps(q, span, sps, alpha=0.35):
    return q.real_taps_to_iq(q.RRCFilter.generateCoefficents(span, alpha, sps * 1000, 1000))


def _close(got, want):
    return got.shape == want.shape and float(np.abs(got - want).max()) <= REL_TOL * float(np.abs(want).max())


def _sub(y, d, skip=0):
    import oracle
    return oracle.decimate(y, d, skip)                          # Filter()'s output kept at indices skip, skip + d, ...


@pytest.mark.parametrize("span,sps,dec", [(16, 2, 2), (16, 4, 4), (16, 8, 8), (16, 16, 16), (16, 4, 2), (10, 2, 2), (16, 16, 4),
                                          (4, 2, 2), (6, 4, 16)])
def test_decimate_matches_subsampled_oracle(gpu, orc, span, sps, dec):
    taps = _taps(gpu, span, sps)
    L = 40013                                                   # several tiles of every geometry, ragged end, odd length
    x = orc.fill_uniform(5, 0, 0, 2 * L)
    want = _sub(orc.ComplexFIRFilter(taps).Filter(x), dec)
    f = gpu.ComplexFIRFilter(taps)
    got = f.Decimate(x, dec)
    assert _close(got, want)
    # D = 2 rides the TMA pipeline (fir_dec2_kernel); D = 4, 8, 16 the padded register-staged kernel
    assert f.last_kernel().startswith("fir_dec2_kernel" if dec == 2 else "fir_decim_tma_kernel"), f.last_kernel()


def test_decimate_streaming_any_chunking(gpu, orc):
    """The kept indices are counted across calls: chunk lengths that are not multiples of D (odd ones, shorter than D,
    shorter than the filter) give the same decimated stream, and the delay line is shared with Filter()."""
    taps = _taps(gpu, 16, 4)                                    # 65 taps
    L = 9001
    x = orc.fill_uniform(6, 1, 0, 2 * L)
    full = orc.ComplexFIRFilter(taps).Filter(x)
    rng = np.random.default_rng(4)
    for dec in (2, 4, 8, 3):
        want = _sub(full, dec)
        cuts = sorted(set([0, L, 1, 2, 3, 7, 8, 70] + [int(v) for v in rng.integers(0, L, 9)]))
        f = gpu.ComplexFIRFilter(taps)
        parts = [f.Decimate(x[2 * a:2 * b], dec) for a, b in zip(cuts[:-1], cuts[1:])]
        assert _close(np.concatenate(parts), want), dec
    # mixed with Filter(): the stream position and the delay line carry over
    f = gpu.ComplexFIRFilter(taps)
    a = f.Filter(x[: 2 * 1000])
    b = f.Decimate(x[2 * 1000:2 * 5000], 4)                     # decimation phase starts at its first sample
    c = f.Filter(x[2 * 5000:])
    assert _close(a, full[: 2 * 1000]) and _close(c, full[2 * 5000:])
    assert _close(b, _sub(full[2 * 1000:2 * 5000], 4))
    f.reset()
    assert _close(f.Decimate(x, 2), _sub(full, 2))


def test_decimate_batch_exact_and_fallbacks(gpu, orc):
    taps = _taps(gpu, 16, 2)                                    # 33 taps
    C, L = 5, 6007
    x = orc.fill_uniform(7, 2, 0, 2 * L * C).reshape(C, 2 * L)
    fulls = [orc.ComplexFIRFilter(taps).Filter(x[c]) for c in range(C)]
    f = gpu.ComplexFIRFilter(taps, channels=C)
    got = f.Decimate(x, 2)
    for c in range(C):
        assert _close(got[c], _sub(fulls[c], 2)), c
    fe = gpu.ComplexFIRFilter(taps, channels=C)                 # QPSK_FIR_EXACT: bit-identical to the subsampled exact filter
    fe.set_mode(gpu.FIR_EXACT)
    ge = fe.Decimate(x, 2)
    for c in range(C):
        assert np.array_equal(ge[c].view(np.uint32), _sub(fulls[c], 2).view(np.uint32)), c
    rng = np.random.default_rng(9)
    ct = (0.1 * rng.standard_normal(2 * 40)).astype(np.float32)  # complex taps -> full-rate path
    want = _sub(orc.ComplexFIRFilter(ct).Filter(x[0]), 4)
    assert _close(gpu.ComplexFIRFilter(ct).Decimate(x[0], 4), want)
    assert _close(gpu.ComplexFIRFilter(taps).Decimate(x[0], 5), _sub(fulls[0], 5))    # odd D
    assert _close(gpu.ComplexFIRFilter(taps).Decimate(x[0], 1), fulls[0])             # D = 1 is Filter()


def test_decimate_argument_errors_leave_the_stream_untouched(gpu, orc):
    taps = _taps(gpu, 16, 2)
    x = orc.fill_uniform(8, 0, 0, 2 * 3000)
    full = orc.ComplexFIRFilter(taps).Filter(x)
    f = gpu.ComplexFIRFilter(taps)
    with pytest.raises(gpu.ArgumentException):
        f.Decimate(np.zeros(3, np.float32), 2)                  # odd float count (:82)
    with pytest.raises(gpu.ArgumentOutOfRangeException):
        f.Decimate(x, 0)
    with pytest.raises(gpu.QpskCudaError):
        f.Decimate(x, 2, out_cap_floats=100)                    # QPSK_ERR_CAPACITY, nothing consumed
    assert _close(f.Decimate(x, 2), _sub(full, 2))
    assert f.Decimate(np.zeros(0, np.float32), 2).size == 0


def test_decimate_dev_full_size_properties(gpu, orc):
    """2^26 samples on the device: oracle windows at the start, at tile seams and at the end; exact homogeneity."""
    import torch
    taps = _taps(gpu, 16, 8)                                    # 129 taps
    n = 1 << 26
    ts = torch.cuda.Stream()
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream
    x = torch.empty(2 * n, dtype=torch.float32, device="cuda")
    gpu.fill_uniform_dev(1, 0, 0, 2 * n, x.data_ptr(), s)
    for dec in (2, 8):
        y = torch.zeros(2 * (n // dec), dtype=torch.float32, device="cuda")
        f = gpu.ComplexFIRFilter(taps)
        assert f.decimate_dev(x.data_ptr(), 2 * n, dec, y.data_ptr(), y.numel(), stream=s) == y.numel()
        torch.cuda.synchronize()
        tile = 7 * (256 if dec == 2 else 64)                    # decimated outputs per tile
        for m0 in (0, tile - 3, 5 * tile - 3, n // dec - 300):
            a = max(0, m0 * dec - 200)                          # input window with 200 samples of run-in (> 128 taps)
            b = min(n, (m0 + 300) * dec)
            xin = x[2 * a:2 * b].cpu().numpy()
            if a > 0:
                w = orc.ComplexFIRFilter(taps).Filter(xin).reshape(-1, 2)[m0 * dec - a:][::dec][:300].reshape(-1)
            else:
                w = _sub(orc.ComplexFIRFilter(taps).Filter(xin), dec)[: 2 * 300]
            g = y[2 * m0:2 * m0 + w.size].cpu().numpy()
            assert _close(g, w), (dec, m0)
        x2 = x * 2.0
        y2 = torch.zeros_like(y)
        f2 = gpu.ComplexFIRFilter(taps)
        f2.decimate_dev(x2.data_ptr(), 2 * n, dec, y2.data_ptr(), y2.numel(), stream=s)
        torch.cuda.synchronize()
        assert torch.equal(y2, y * 2.0)                         # scaling by 2 is exact in fp32
        del y, y2, x2


@pytest.mark.parametrize("aligned", [False, True])
def test_decimate_by_2_kernels_agree_across_an_odd_cut(gpu, orc, aligned):
    """Bulk copies need 16-byte aligned rows: a device pointer that starts on an odd sample falls back to the register-staged
    fir_decim_kernel<D=2>, an aligned one takes fir_dec2_kernel.  Either way two calls with an odd first length give the
    decimated stream of one call (on the TMA kernel the kept-output phase of 1 is a leading zero tap)."""
    import torch
    taps = _taps(gpu, 16, 4)                                    # 65 taps
    L, cut = 30001, 10001
    x = orc.fill_uniform(9, 2, 0, 2 * (L + 2))
    off = 2 if aligned else 1                                   # first sample of the stream inside the device buffer
    want = _sub(orc.ComplexFIRFilter(taps).Filter(x[2 * off: 2 * (off + L)]), 2)
    dx = torch.from_numpy(x).cuda()
    dy = torch.zeros(2 * (L + 4), dtype=torch.float32, device="cuda")
    f = gpu.ComplexFIRFilter(taps)
    p = dx.data_ptr() + 8 * off
    n1 = f.decimate_dev(p, 2 * cut, 2, dy.data_ptr(), 2 * (L + 4))
    k1 = f.last_kernel()
    # the second call's output row starts right after the first one's: aligned only if n1 is even, so give it its own buffer
    dz = torch.zeros(2 * (L + 4), dtype=torch.float32, device="cuda")
    n2 = f.decimate_dev(p + 8 * cut, 2 * (L - cut), 2, dz.data_ptr(), 2 * (L + 4))
    k2 = f.last_kernel()
    torch.cuda.synchronize()
    assert k1.startswith("fir_dec2_kernel" if aligned else "fir_decim_kernel"), k1
    # the second call starts on an odd sample of an aligned buffer (cut is odd): the pointer is misaligned exactly when the
    # first one was aligned
    assert k2.startswith("fir_decim_kernel" if aligned else "fir_dec2_kernel"), k2
    got = np.concatenate([dy.cpu().numpy()[:n1], dz.cpu().numpy()[:n2]])          # the counts are in floats
    assert n1 + n2 == want.size
    assert _close(got, want)


@pytest.mark.parametrize("layout", ["offset_pointer", "odd_stride_batch"])
@pytest.mark.parametrize("span,sps,dec", [(16, 4, 4), (16, 4, 8), (16, 4, 16), (16, 8, 4), (16, 8, 8), (16, 8, 16)])
def test_register_staged_decimators_match_the_subsampled_oracle(gpu, orc, span, sps, dec, layout):
    """D = 4, 8, 16 leave the bulk-copy pipeline for the register-staged fir_decim_kernel when the rows rule out bulk
    copies: an input pointer one sample into the buffer, or a 3-channel batch whose rows are an odd number of samples
    apart.  65 and 129 taps, over more than two tiles of every D with a ragged end."""
    import torch
    taps = _taps(gpu, span, sps)
    L = 40010                                                   # 11+ tiles at every D; L + 3 is odd
    C = 1 if layout == "offset_pointer" else 3
    x = orc.fill_uniform(11 + dec, sps, 0, 2 * L * C).reshape(C, 2 * L)
    if layout == "offset_pointer":
        ld = 2 * L
        buf = torch.zeros(2 + ld + 2, dtype=torch.float32, device="cuda")
        buf[2:2 + ld] = torch.from_numpy(x[0]).cuda()
        p = buf.data_ptr() + 8
    else:
        ld = 2 * (L + 3)                                        # floats: an odd number of samples per row
        buf = torch.zeros(C * ld, dtype=torch.float32, device="cuda")
        buf.view(C, ld)[:, : 2 * L] = torch.from_numpy(x).cuda()
        p = buf.data_ptr()
    n_out = (L + dec - 1) // dec
    ldo = 2 * n_out + 6
    y = torch.zeros(C * ldo, dtype=torch.float32, device="cuda")
    f = gpu.ComplexFIRFilter(taps, channels=C)
    torch.cuda.synchronize()
    n = f.decimate_dev(p, 2 * L, dec, y.data_ptr(), 2 * n_out, in_stride=ld, out_stride=ldo)
    torch.cuda.synchronize()
    assert f.last_kernel().startswith("fir_decim_kernel<"), f.last_kernel()
    assert n == 2 * n_out
    yh = y.view(C, ldo).cpu().numpy()
    for c in range(C):
        assert _close(yh[c, :n], _sub(orc.ComplexFIRFilter(taps).Filter(x[c]), dec)), c
