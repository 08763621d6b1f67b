"""GPU parity of the demodulator with the matched filter fused into the symbol-stage kernel
(symsync_decode_kernel<DIFF, MFW, DENSE>, the default path for 32 or more channels: QPSK_FIR_EXACT, real taps, <= 65 taps).
Everything is compared with the oracle bit for bit: bits, constellation points (which go through the SEPARATE
matched-filter kernel on the same delay line) and loop state.  Which instantiation ran is read from torch.profiler and must
be the one tests/symsync_dispatch.py predicts from the public inputs; its geometry table reaches every variant the dispatch
can produce (checked on the CPU by tests/test_symsync_dispatch.py)."""
import numpy as np
import pytest

import symsync_dispatch as sd

pytestmark = pytest.mark.gpu

TSC = "11001010011101100100100110101100" + "01110100111001011010001101101001"
ALPHA = float(np.float32(0.35))


def _stream(orc, fs, rs, alpha, span, n_bursts, n_payload, seed, tsc=None, noise=-45.0):
    rng = np.random.default_rng(seed)
    mod = orc.QPSKModulator(fs, rs, alpha, span, True, tsc)
    tx, rx = orc.NCO(100e6, fs, 1, seed=seed, stream=0), orc.NCO(100e6, fs, 1, seed=seed, stream=1)
    parts = []
    for b in range(n_bursts):
        s = mod.ModulateBytes(rng.integers(0, 256, n_payload, dtype=np.uint8).tobytes(), b"S", b"E")
        nz = orc.noise_iq(noise, s.size // 2, seed, 2, first_sample=b * 100000)
        parts.append(orc.channel_apply(tx, rx, 1, s, nz))
    return np.concatenate(parts)


def _scene(orc, fs, rs, span, C, L, diff, seed, tsc=None):
    """[C, 2L] float32: every channel its own stream — its own bits, carrier phase and drift, and noise.  Integer rates
    carry real modulated bursts (differential encoding as the demodulator's, the TSC when given); non-integer rates (and
    the one-tap filter) a noisy +-0.7 corner signal held for sps samples with a timing drift."""
    rng = np.random.default_rng(seed)
    sps = fs / rs
    mod = orc.QPSKModulator(fs, rs, ALPHA, span, diff, tsc) if fs % rs == 0 and span > 0 else None
    x = np.empty((C, 2 * L), np.float32)
    for c in range(C):
        if mod is not None:
            parts, n = [], 0
            while n < L:
                y = mod.Modulate("".join(rng.choice(["0", "1"], 2 * int(rng.integers(100, 400)))), True)
                parts.append(y)
                n += y.size // 2
            y = np.concatenate(parts)[: 2 * L]
            z = y[0::2] + 1j * y[1::2]
        else:
            t = (np.arange(L) / (sps * (1 + rng.uniform(-0.01, 0.01)))).astype(np.int64)
            sym = rng.choice([-0.7, 0.7], (t.max() + 1, 2))
            z = sym[t, 0] + 1j * sym[t, 1]
        ph = rng.uniform(-3, 3) + rng.uniform(-2e-3, 2e-3) * np.arange(L)
        z = z * np.exp(1j * ph) + 0.02 * (rng.standard_normal(L) + 1j * rng.standard_normal(L))
        x[c, 0::2], x[c, 1::2] = z.real, z.imag
    return x


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _assert_variant(names, C, fs, rs, span, diff, what=""):
    want = sd.kernel_name(sd.predict(C, fs, rs, span, diff=diff, sm_count=_sm_count()))
    got = sd.symsync_variants(names)
    print(f"[kernel] {what} C={C} fs/rs={fs}/{rs} span={span} diff={diff}: {sorted(got)}")
    assert got == {want}, (want, names)


def _assert_loop_state(gd, ods):
    gs = gd.loop_state()
    for c, od in enumerate(ods):
        ws = od.loop_state()
        for k in ("costas_theta", "costas_freq", "mm_mu", "mm_integral"):
            g = gs[k] if np.ndim(gs[k]) == 0 else gs[k][c]
            assert abs(ws[k] - g) <= 1e-5 * max(1.0, abs(ws[k])), (k, c)


def _chunkings(L, seed):
    """One call; cuts at odd positions, shorter than a round (32 samples) and than the filter, with an empty call; random."""
    rng = np.random.default_rng(seed)
    return [[0, L],
            [0, 5, 31, 31, 33, 64, 1001, 1002, 1003, 2047, L - 1, L],
            sorted([0, L] + [int(v) for v in rng.integers(0, L, 12)])]


def _compare_chunkings(gpu, orc, fs, rs, kw, x, seed):
    C, L = x.shape[0], x.shape[1] // 2
    for trial, cuts in enumerate(_chunkings(L, seed)):
        gd = gpu.QPSKDeModulator(fs, rs, channels=C, **kw)
        ods = [orc.QPSKDeModulator(fs, rs, **kw) for _ in range(C)]
        for a, b in zip(cuts[:-1], cuts[1:]):
            xs = np.ascontiguousarray(x[:, 2 * a:2 * b])
            got = gd.DeModulate(xs if C > 1 else xs[0])
            got = got if C > 1 else [got]
            for c in range(C):
                assert got[c] == ods[c].DeModulate(xs[c]), (trial, a, b, c)
        _assert_loop_state(gd, ods)


# every row of the geometry table at 33 channels (one full CTA and one with a single live lane); some also at 95, and the
# 33- / 41- / 65-tap rows also with the TSC strip and the FLL (a call of 2048+ samples runs the FLL time-chunk pipeline,
# the kernel's append path)
MATRIX = [(row, 33, False) for row in sd.MATRIX_ROWS] + [(row, 95, False) for row in (9, 21, 41, "65s16")] + \
         [(row, 33, True) for row in (33, 41, 65)]


@pytest.mark.parametrize("diff", [True, False])
@pytest.mark.parametrize("row,C,tsc_fll", MATRIX)
def test_fused_variant_matrix(gpu, orc, row, C, tsc_fll, diff):
    fs, rs, span = sd.GEOMETRIES[row]
    L = max(4000, int(300 * fs / rs))
    tsc = TSC if tsc_fll else None
    x = _scene(orc, fs, rs, span, C, L, diff, seed=1000 + 7 * C + span, tsc=tsc)
    kw = dict(RrcAlpha=ALPHA, rrcSpan=span, SymbolSyncBandwith=0.002, differentialEncoding=diff, tsc=tsc, use_fll=tsc_fll)
    probe = gpu.QPSKDeModulator(fs, rs, channels=C, **kw)
    _, names = sd.launched_kernels(lambda: probe.DeModulate(x))
    _assert_variant(names, C, fs, rs, span, diff, f"matrix row={row} tsc_fll={tsc_fll}")
    _compare_chunkings(gpu, orc, fs, rs, kw, x, seed=span)


@pytest.mark.parametrize("fs,rs,span,alpha", [(10_000_000, 5_000_000, 10, 0.4), (4000, 1000, 10, 0.35), (8000, 1000, 8, 0.5),
                                               (3000, 1000, 6, 0.9), (16000, 1000, 6, 0.35)])
def test_fused_mf_bits_any_chunking(gpu, orc, fs, rs, span, alpha):
    """33 channels of framed bursts: 21 / 41 / 65 / 19 taps run fused (2 or 4 matched-filter warps), 97 taps (sps 16) take
    <DIFF, 0> behind the separate exact filter; chunk cuts at odd positions, shorter than a round (32 samples) and shorter
    than the filter."""
    alpha = float(np.float32(alpha))
    C = 33
    x = np.stack([_stream(orc, fs, rs, alpha, span, 3, 120, seed=fs % 97 + c) for c in range(C)])
    L = x.shape[1] // 2
    kw = dict(RrcAlpha=alpha, rrcSpan=span, SymbolSyncBandwith=0.002, tsc=None)
    probe = gpu.QPSKDeModulator(fs, rs, channels=C, **kw)
    _, names = sd.launched_kernels(lambda: probe.DeModulate(x))
    _assert_variant(names, C, fs, rs, span, True, "any_chunking")
    rng = np.random.default_rng(3)
    for trial in range(3):
        cuts = [0, L] if trial == 0 else sorted(set([0, L, 5, 31, 33, 64, 1000] + [int(v) for v in rng.integers(0, L, 12)]))
        ods = [orc.QPSKDeModulator(fs, rs, **kw) for _ in range(C)]
        gd = gpu.QPSKDeModulator(fs, rs, channels=C, **kw)
        for a, b in zip(cuts[:-1], cuts[1:]):
            got = gd.DeModulate(np.ascontiguousarray(x[:, 2 * a:2 * b]))
            for c in range(C):
                assert got[c] == ods[c].DeModulate(x[c, 2 * a:2 * b]), (trial, a, b, c)
        _assert_loop_state(gd, ods)


def test_fused_mf_shares_the_delay_line_with_the_separate_filter(gpu, orc):
    """DeModulate (fused matched filter) and deModulateConstellation (separate matched-filter kernel) alternate on one
    handle: both advance the same delay line, MM queue and Costas state, exactly as the reference object's calls do.  At 33
    channels with 25 taps (registers, NB = 3) and 41 taps (four filter warps, 128-slot ring); one channel keeps <DIFF, 0>
    and the separate filter for both calls."""
    for row, C in ((25, 33), (41, 33), (41, 1)):
        fs, rs, span = sd.GEOMETRIES[row]
        L = 4000
        x = np.stack([_stream(orc, fs, rs, ALPHA, span, 4, 90, seed=8 + c)[: 2 * L] for c in range(C)])
        kw = dict(RrcAlpha=ALPHA, rrcSpan=span, SymbolSyncBandwith=0.002, tsc=None)
        ods = [orc.QPSKDeModulator(fs, rs, **kw) for _ in range(C)]
        gd = gpu.QPSKDeModulator(fs, rs, channels=C, **kw)
        cuts = [0, 700, 701, 1500, 2222, 2240, 3001, L]
        for i, (a, b) in enumerate(zip(cuts[:-1], cuts[1:])):
            seg = np.ascontiguousarray(x[:, 2 * a:2 * b])
            arg = seg if C > 1 else seg[0]
            if i % 2 == 0:
                if i == 0:
                    got, names = sd.launched_kernels(lambda: gd.DeModulate(arg))
                    _assert_variant(names, C, fs, rs, span, True, f"delay line row={row}")
                else:
                    got = gd.DeModulate(arg)
                got = got if C > 1 else [got]
                for c in range(C):
                    assert got[c] == ods[c].DeModulate(seg[c]), (row, C, i, c)
            else:
                g = gd.deModulateConstellation(arg)
                g = g if C > 1 else [g]
                for c in range(C):
                    w = ods[c].deModulateConstellation(seg[c])
                    assert np.array_equal(g[c].view(np.uint32), w.view(np.uint32)), (row, C, i, c)


@pytest.mark.parametrize("row", [25, 41])
def test_fused_mf_device_entry_offset_pointer_and_odd_stride(gpu, orc, row):
    """demod_bits_dev on rows that start one sample into the buffer, `in_stride` longer than the row by an odd number of
    samples, two calls cut at an odd sample: the bits equal the host call's and the oracle's (96- and 128-slot ring)."""
    import torch
    fs, rs, span = sd.GEOMETRIES[row]
    C, L, cut, pad = 33, 5001, 1777, 3
    x = _scene(orc, fs, rs, span, C, L, True, seed=77 + row)
    kw = dict(RrcAlpha=ALPHA, rrcSpan=span, SymbolSyncBandwith=0.002, tsc=None)
    ld = 2 * (L + pad)                                          # floats per row
    buf = torch.zeros(2 + C * ld + 2, dtype=torch.float32, device="cuda")
    buf[2:2 + C * ld].view(C, ld)[:, : 2 * L] = torch.from_numpy(x).cuda()
    dem = gpu.QPSKDeModulator(fs, rs, channels=C, **kw)
    host = gpu.QPSKDeModulator(fs, rs, channels=C, **kw)
    ods = [orc.QPSKDeModulator(fs, rs, **kw) for _ in range(C)]
    cap = dem.bits_bound(2 * L)
    bits = torch.zeros((C, cap), dtype=torch.uint8, device="cuda")
    nb = torch.zeros(C, dtype=torch.int64, device="cuda")
    for k, (a, b) in enumerate(((0, cut), (cut, L))):
        bits.zero_()
        torch.cuda.synchronize()
        call = lambda: dem.demod_bits_dev(buf.data_ptr() + 8 * (1 + a), 2 * (b - a), ld, bits.data_ptr(), cap, nb.data_ptr())
        if k == 0:
            _, names = sd.launched_kernels(call)
            _assert_variant(names, C, fs, rs, span, True, f"device entry row={row}")
        else:
            call()
        torch.cuda.synchronize()
        bits_h, nb_h = (bits & 1).cpu().numpy(), nb.cpu().numpy()
        xs = np.ascontiguousarray(x[:, 2 * a:2 * b])
        hb = host.DeModulate(xs)
        for c in range(C):
            got = "".join("1" if v else "0" for v in bits_h[c, : nb_h[c]])
            assert got == hb[c], (k, c)
            assert got == ods[c].DeModulate(xs[c]), (k, c)


@pytest.mark.parametrize("diff", [True, False])
@pytest.mark.parametrize("row", sd.DENSE_ROWS)
def test_dense_variant_on_both_sides_of_its_threshold(gpu, orc, row, diff):
    """DENSE (the two-filter-warp kernel compiled for four CTAs per SM) runs when the grid exceeds 3 x SM CTAs: 96 x SM
    channels (exactly 3 x SM CTAs) must run the ordinary kernel, 96 x SM + 33 the DENSE one.  37 distinct streams tiled
    over the channels (channel c carries stream c mod 37; 37 is coprime to 32, so a mix-up between the lanes of a CTA or
    between neighbouring CTAs changes the stream), every channel compared with its stream's oracle bits and loop state,
    over two calls cut at an odd sample (the second call's rows start on an odd sample)."""
    import torch
    K = 37
    fs, rs, span = sd.GEOMETRIES[row]
    L, cut = 3000, 1001
    base = _scene(orc, fs, rs, span, K, L, diff, seed=500 + span)
    kw = dict(RrcAlpha=ALPHA, rrcSpan=span, SymbolSyncBandwith=0.002, differentialEncoding=diff, tsc=None)
    calls = ((0, cut), (cut, L))
    ods = [orc.QPSKDeModulator(fs, rs, **kw) for _ in range(K)]
    want = [[ods[k].DeModulate(base[k, 2 * a:2 * b]) for k in range(K)] for a, b in calls]
    wstate = {n: np.array([od.loop_state()[n] for od in ods]) for n in ("costas_theta", "costas_freq", "mm_mu", "mm_integral")}
    sm = _sm_count()
    dbase = torch.from_numpy(base).cuda()
    for C in (96 * sm, 96 * sm + 33):
        idx = torch.arange(C, device="cuda") % K
        x = dbase[idx].contiguous()
        dem = gpu.QPSKDeModulator(fs, rs, channels=C, **kw)
        cap = dem.bits_bound(2 * L)
        bits = torch.zeros((C, cap), dtype=torch.uint8, device="cuda")
        nb = torch.zeros(C, dtype=torch.int64, device="cuda")
        for k, (a, b) in enumerate(calls):
            bits.zero_()
            torch.cuda.synchronize()
            call = lambda: dem.demod_bits_dev(x.data_ptr() + 8 * a, 2 * (b - a), 2 * L, bits.data_ptr(), cap, nb.data_ptr())
            if k == 0:
                _, names = sd.launched_kernels(call)
                _assert_variant(names, C, fs, rs, span, diff, f"dense row={row}")
            else:
                call()
            torch.cuda.synchronize()
            wn = torch.tensor([len(w) for w in want[k]], dtype=torch.int64, device="cuda")
            wb = torch.zeros((K, cap), dtype=torch.uint8, device="cuda")
            for j, w in enumerate(want[k]):
                if w:
                    wb[j, : len(w)] = torch.from_numpy(np.frombuffer(w.encode("ascii"), np.uint8) - 48).cuda()
            bad = (nb != wn[idx]).nonzero()
            assert bad.numel() == 0, ("bit counts differ", C, k, bad[:8].flatten().tolist())
            m = int(wn.max())
            live = torch.arange(m, device="cuda")[None, :] < nb[:, None]
            diffs = (((bits[:, :m] & 1) != wb[idx, :m]) & live).any(dim=1).nonzero()
            assert diffs.numel() == 0, ("bits differ", C, k, diffs[:8].flatten().tolist())
        st = dem.loop_state()
        ih = idx.cpu().numpy()
        for n, w in wstate.items():
            err = np.abs(st[n] - w[ih]) > 1e-5 * np.maximum(1.0, np.abs(w[ih]))
            assert not err.any(), (n, C, np.nonzero(err)[0][:8])
        del x, bits


@pytest.mark.parametrize("use_fll", [False, True])
def test_fused_mf_batch_ragged_channel_count(gpu, orc, use_fll):
    """70 channels (two full 32-channel CTAs and a partial one), TSC strip and framer behind the fused kernel, three bursts
    with state carried; with the FLL on the call is long enough for the time-chunk pipeline."""
    fs, rs = 10_000_000, 5_000_000
    alpha = float(np.float32(0.4))
    C = 70
    om = orc.QPSKModulator(fs, rs, alpha, 10, True, TSC)
    rng = np.random.default_rng(12)
    n_payload = 300 if use_fll else 64
    rx = []
    for c in range(C):
        s = om.ModulateBytes(rng.integers(0, 256, n_payload, dtype=np.uint8).tobytes(), b"S", b"E")
        a, b = orc.NCO(100e6, fs, 1, seed=31, stream=4 * c), orc.NCO(100e6, fs, 1, seed=31, stream=4 * c + 1)
        rx.append(orc.channel_apply(a, b, 1, s, orc.noise_iq(-40.0, s.size // 2, 31, 4 * c + 2)))
    rx = np.stack(rx)
    gd = gpu.QPSKDeModulator(fs, rs, alpha, 10, tsc=TSC, use_fll=use_fll, channels=C)
    ods = [orc.QPSKDeModulator(fs, rs, alpha, 10, tsc=TSC, use_fll=use_fll) for _ in range(C)]
    for rep in range(3):
        got = gd.DeModulateBytes(rx, b"S", b"E")
        for c in range(C):
            assert got[c] == ods[c].DeModulateBytes(rx[c], b"S", b"E"), (rep, c)
    assert sum(bool(g) for g in got) > C // 2
