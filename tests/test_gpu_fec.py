"""GPU: the convolutional encoder and the Viterbi decoder (csrc/fec.cu) bit-identical to tests/fec_oracle.py: both modes,
1 to 16384 channels, noise levels that leave decoding errors, saturating and tiny scales, ragged counts with 0 and 1 symbol
and flushes mid-row; the same bits under any chunking, for host and device calls, strided and offset rows, after reset()
and for a subset of channels; untouched guard bands; argument checks, and a refused call that leaves the state alone; every
compiled instantiation seen running; qpsk_demod_frame_bits_dev against the host framer; and the coded receive path end to
end: at a noise level where uncoded frames are lost, coded frames decode."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import fec_oracle as F
import kernel_variants as kv

pytestmark = pytest.mark.gpu

KERNELS = ("viterbi_kernel", "conv_encode_kernel")
INSTANTIATIONS = {"viterbi_kernel<false>", "viterbi_kernel<true>", "conv_encode_kernel"}
_KRE = re.compile(r"\b(" + "|".join(KERNELS) + r")\b(<[^<>]*>)?")


def _norm(name):
    m = _KRE.search(name)
    if not m:
        return None
    args = m.group(2) or ""
    return m.group(1) + ("<" + ", ".join(kv._arg(a) for a in args[1:-1].split(",")) + ">" if args else "")


def _noisy(rng, Cn, n, differential, ebn0_db, amp=1.0):
    """ConvEncoder-coded random bits as unit-amplitude symbols (x amp) with AWGN at ebn0_db per information bit; a random
    carrier phase per channel in differential mode"""
    bits = rng.integers(0, 2, (Cn, n)).astype(np.uint8)
    y = F.qpsk_symbols(F.encode(bits)[0], differential)[:, :n]
    if differential:
        y = y * np.exp(1j * rng.uniform(0, 2 * np.pi, (Cn, 1)))
    sig = np.sqrt(0.5 / 10 ** (ebn0_db / 10))
    y = amp * y + amp * sig * (rng.standard_normal(y.shape) + 1j * rng.standard_normal(y.shape))
    return y.astype(np.complex64), bits


def _calls(rng, Cn, n, n_calls):
    """per call: symbols used per channel (ragged, 0 and 1 included, rarely a multiple of 32), summing to at most n"""
    left = np.full(Cn, n, np.int64)
    out = []
    for k in range(n_calls):
        c = rng.integers(0, max(2, 2 * n // n_calls), Cn)
        c[rng.random(Cn) < 0.15] = 0
        c[rng.random(Cn) < 0.1] = 1
        c = np.minimum(c, left)
        out.append(c)
        left -= c
    return out


def _run_both(gpu, y, calls, differential, scale=None, flush_at=()):
    """the same call sequence on the GPU (host entry points) and on the oracle; returns per-channel bit streams of both"""
    Cn = y.shape[0]
    g = gpu.ViterbiDecoder(Cn, differential, scale)
    o = F.Viterbi(Cn, differential, g.scale)
    gs, os_ = [[] for _ in range(Cn)], [[] for _ in range(Cn)]
    pos = np.zeros(Cn, np.int64)
    for k, c in enumerate(calls):
        w = max(int(c.max()), 1)
        seg = np.zeros((Cn, w), np.complex64)
        for ch in range(Cn):
            seg[ch, : c[ch]] = y[ch, pos[ch]: pos[ch] + c[ch]]
        pos += c
        fl = k in flush_at or k == len(calls) - 1
        got = g.flush(seg, c) if fl else g.decode(seg, c)
        want = o.flush(seg, c) if fl else o.decode(seg, c)
        for ch in range(Cn):
            gs[ch].append(got[ch])
            os_[ch].append(want[ch])
    g.close()
    return [np.concatenate(a) for a in gs], [np.concatenate(a) for a in os_]


@pytest.mark.parametrize("differential", [False, True])
@pytest.mark.parametrize("Cn", [1, 31, 32, 33, 2048, 16384])
def test_decoder_bit_identical_to_oracle(gpu, Cn, differential):
    rng = np.random.default_rng(Cn * 2 + differential)
    n = 700 if Cn <= 2048 else 160
    y, bits = _noisy(rng, Cn, n, differential, 1.0 if not differential else 3.0)
    calls = _calls(rng, Cn, n, 6)
    got, want = _run_both(gpu, y, calls, differential, flush_at=(3,))
    bad = [c for c in range(Cn) if not np.array_equal(got[c], want[c])]
    assert not bad, (bad[:10], len(bad))
    assert sum(w.size for w in want) > 0


@pytest.mark.parametrize("scale", [1e5, 4000.0, 0.02, 1e-30])
@pytest.mark.parametrize("differential", [False, True])
def test_decoder_saturating_and_tiny_scale(gpu, scale, differential):
    rng = np.random.default_rng(int(scale) % 97 + differential)
    Cn, n = 33, 500
    y, _ = _noisy(rng, Cn, n, differential, 2.0)
    got, want = _run_both(gpu, y, _calls(rng, Cn, n, 4), differential, scale=scale)
    for c in range(Cn):
        assert np.array_equal(got[c], want[c]), c


def test_decoder_non_finite_symbols(gpu):
    rng = np.random.default_rng(9)
    Cn, n = 5, 300
    for diff in (False, True):
        y, _ = _noisy(rng, Cn, n, diff, 2.0)
        y[0, 10] = np.complex64(complex(np.nan, 1.0))
        y[1, 50] = np.complex64(complex(np.inf, -np.inf))
        y[2, 90] = np.complex64(complex(3e38, 3e38))
        got, want = _run_both(gpu, y, _calls(rng, Cn, n, 3), diff)
        for c in range(Cn):
            assert np.array_equal(got[c], want[c]), (diff, c)


def test_decoder_errors_are_real(gpu):
    """At the noise of the parity tests, decoding leaves errors (so ties and survivor choices are exercised) while the
    noiseless round trip is exact."""
    rng = np.random.default_rng(5)
    Cn, n = 64, 2000
    for diff, eb in ((False, 1.0), (True, 3.0)):
        y, bits = _noisy(rng, Cn, n, diff, eb)
        g = gpu.ViterbiDecoder(Cn, diff)
        got = g.flush(y)
        nerr = sum(int((a != b[: n - diff]).sum()) for a, b in zip(got, bits))   # differential: n - 1 steps
        assert nerr > 0, diff
        y0, bits0 = _noisy(rng, Cn, n, diff, 300.0)
        for a, b in zip(g.flush(y0), bits0):
            assert np.array_equal(a, b[: n - diff])


def test_encoder_bit_identical_chunked_and_reset(gpu):
    import torch
    rng = np.random.default_rng(11)
    for Cn in (1, 33, 2048):
        n = 300
        bits = rng.integers(0, 2, (Cn, n)).astype(np.uint8)
        want = F.encode(bits)[0]
        e = gpu.ConvEncoder(Cn)
        assert np.array_equal(e.encode(bits), want)
        e.reset()
        parts = [e.encode(np.ascontiguousarray(bits[:, a:b])) for a, b in ((0, 0), (0, 1), (1, 97), (97, 300))]
        assert np.array_equal(np.concatenate(parts, axis=1), want)
        # device: offset, strided rows, guard bands
        e.reset()
        ld_in, ld_out = n + 5, 2 * n + 9
        d_in = torch.zeros((Cn, ld_in), dtype=torch.uint8, device="cuda")
        d_in[:, 3:3 + n] = torch.from_numpy(bits).cuda()
        d_out = torch.full((Cn * ld_out + 16,), 0xAB, dtype=torch.uint8, device="cuda")
        col = 0
        for a, b in ((0, 50), (50, 50), (50, 300)):
            e.encode_dev(d_in.data_ptr() + 3 + a, b - a, d_out.data_ptr() + 8 + col, ld_out, bits_stride=ld_in)
            col += 2 * (b - a)
        torch.cuda.synchronize()
        h = d_out.cpu().numpy()
        rows = h[8: 8 + Cn * ld_out].reshape(Cn, ld_out)
        assert np.array_equal(rows[:, : 2 * n], want)
        assert (rows[:, 2 * n:] == 0xAB).all() and (h[:8] == 0xAB).all() and (h[8 + Cn * ld_out:] == 0xAB).all()
        e.close()


def _dev_rows(torch, y, ld, off):
    """complex rows [C, n] into a device buffer of [C][ld] complex at `off` complex from its start"""
    Cn, n = y.shape
    buf = torch.zeros(2 * (off + Cn * ld + 1), dtype=torch.float32, device="cuda")
    rows = np.zeros((Cn, ld), np.complex64)
    rows[:, :n] = y
    buf[2 * off: 2 * (off + Cn * ld)] = torch.from_numpy(rows.view(np.float32).ravel()).cuda()
    return buf, buf.data_ptr() + 8 * off


@pytest.mark.parametrize("differential", [False, True])
def test_device_path_chunked_strided_offset_subset_reset(gpu, differential):
    import torch
    rng = np.random.default_rng(21 + differential)
    Cn, n = 40, 600
    y, _ = _noisy(rng, Cn, n, differential, 2.0)
    calls = _calls(rng, Cn, n, 5)
    tot = np.sum(calls, axis=0)
    whole = gpu.ViterbiDecoder(Cn, differential).flush(y, tot)
    ld = n + 3                                                   # odd complex stride: rows start at 8-byte offsets only
    for rep in range(2):
        dec = gpu.ViterbiDecoder(Cn, differential)
        if rep:
            dec.decode(y[:, :100])                               # state to be discarded
            dec.reset()
        outs = [[] for _ in range(Cn)]
        pos = np.zeros(Cn, np.int64)
        ts = torch.cuda.Stream()
        for k, c in enumerate(calls + [np.zeros(Cn, np.int64)]):
            seg = np.zeros((Cn, n), np.complex64)
            for ch in range(Cn):
                seg[ch, : c[ch]] = y[ch, pos[ch]: pos[ch] + c[ch]]
            pos += c
            buf, p = _dev_rows(torch, seg, ld, 3)
            d_n = torch.from_numpy(c.astype(np.int32)).cuda()
            cap = dec.bits_bound(ld) + 6
            guard = 24
            d_bits = torch.full((Cn * cap + 2 * guard,), 0xAB, dtype=torch.uint8, device="cuda")
            d_nb = torch.full((Cn,), -7, dtype=torch.int64, device="cuda")
            torch.cuda.synchronize()
            fn = dec.flush_dev if k == len(calls) else dec.decode_dev
            fn(p, 2 * ld, d_n.data_ptr(), d_bits.data_ptr() + guard, cap, d_nb.data_ptr(), ts.cuda_stream)
            ts.synchronize()
            h, nb = d_bits.cpu().numpy(), d_nb.cpu().numpy()
            assert (h[:guard] == 0xAB).all() and (h[guard + Cn * cap:] == 0xAB).all()
            rows = h[guard: guard + Cn * cap].reshape(Cn, cap)
            for ch in range(Cn):
                assert (rows[ch, nb[ch]:] == 0xAB).all()
                outs[ch].append(rows[ch, : nb[ch]].copy())
        for ch in range(Cn):
            assert np.array_equal(np.concatenate(outs[ch]), whole[ch]), (rep, ch)
    # a subset of the channels on its own handle gives the rows of the full batch
    sub = gpu.ViterbiDecoder(7, differential)
    got = sub.flush(np.ascontiguousarray(y[11:18]), tot[11:18])
    for k in range(7):
        assert np.array_equal(got[k], whole[11 + k])


def test_argument_checks_and_refusal_keeps_state(gpu):
    import torch
    L = gpu._native.lib()
    E = gpu._native
    h = C.c_void_p()
    for ch, st in ((0, E.ERR_UNSUPPORTED), (16385, E.ERR_UNSUPPORTED)):
        assert L.qpsk_viterbi_create(ch, 1, 24.0, C.byref(h)) == st
        assert L.qpsk_conv_create(ch, C.byref(h)) == st
    for sc in (0.0, -1.0, float("inf"), float("nan")):
        assert L.qpsk_viterbi_create(4, 0, sc, C.byref(h)) == E.ERR_RANGE
    assert L.qpsk_viterbi_create(4, 0, 24.0, None) == E.ERR_NULL
    Cn, n = 4, 200
    rng = np.random.default_rng(31)
    y, _ = _noisy(rng, Cn, n, False, 2.0)
    want = gpu.ViterbiDecoder(Cn, False).flush(y)
    dec = gpu.ViterbiDecoder(Cn, False)
    buf, p = _dev_rows(torch, y, n, 0)
    d_n = torch.full((Cn,), n, dtype=torch.int32, device="cuda")
    cap = dec.bits_bound(n)
    assert cap == n + 96 - (n & 1)
    d_bits = torch.zeros((Cn, cap), dtype=torch.uint8, device="cuda")
    d_nb = torch.zeros(Cn, dtype=torch.int64, device="cuda")
    f = L.qpsk_viterbi_decode_dev
    a = (dec._h, p, 2 * n, d_n.data_ptr(), d_bits.data_ptr(), cap, d_nb.data_ptr(), None)
    assert f(None, *a[1:]) == E.ERR_NULL
    assert f(a[0], None, *a[2:]) == E.ERR_NULL
    assert f(*a[:3], None, *a[4:]) == E.ERR_NULL
    assert f(*a[:4], None, *a[5:]) == E.ERR_NULL
    assert f(*a[:6], None, None) == E.ERR_NULL
    assert f(a[0], a[1], 2 * n + 1, *a[3:]) == E.ERR_ARG                    # odd stride
    assert f(*a[:5], cap - 1, *a[6:]) == E.ERR_ARG                          # odd capacity
    assert f(a[0], a[1] + 4, *a[2:]) == E.ERR_ARG                           # misaligned
    assert f(*a[:4], a[4] + 1, *a[5:]) == E.ERR_ARG
    assert f(a[0], a[1], -2, *a[3:]) == E.ERR_RANGE
    assert f(*a[:5], cap - 2, *a[6:]) == E.ERR_CAPACITY                     # refused before any state advances
    assert L.qpsk_viterbi_flush_dev(*a[:5], cap - 2, *a[6:]) == E.ERR_CAPACITY
    assert L.qpsk_viterbi_flush_dev(*a) == 0
    torch.cuda.synchronize()
    nb = d_nb.cpu().numpy()
    rows = d_bits.cpu().numpy()
    for c in range(Cn):
        assert np.array_equal(rows[c, : nb[c]], want[c])
    # host forms
    ns = np.full(Cn, n, np.int64)
    yy = np.ascontiguousarray(y).view(np.float32)
    out = np.zeros((Cn, cap), np.uint8)
    nbh = np.zeros(Cn, np.int64)
    ptr = lambda v: C.c_void_p(v.ctypes.data)                                # noqa: E731
    assert L.qpsk_viterbi_decode(dec._h, ptr(yy), 2 * n, ptr(ns), ptr(out), cap - 2, ptr(nbh)) == E.ERR_CAPACITY
    assert (nbh == cap).all()
    bad = ns.copy()
    bad[2] = n + 1
    assert L.qpsk_viterbi_decode(dec._h, ptr(yy), 2 * n, ptr(bad), ptr(out), cap, ptr(nbh)) == E.ERR_RANGE
    bad[2] = -1
    assert L.qpsk_viterbi_decode(dec._h, ptr(yy), 2 * n, ptr(bad), ptr(out), cap, ptr(nbh)) == E.ERR_RANGE
    assert L.qpsk_viterbi_decode(dec._h, ptr(yy), 2 * n + 1, ptr(ns), ptr(out), cap, ptr(nbh)) == E.ERR_ARG
    assert L.qpsk_viterbi_flush(dec._h, ptr(yy), 2 * n, ptr(ns), ptr(out), cap, ptr(nbh)) == 0
    for c in range(Cn):
        assert np.array_equal(out[c, : nbh[c]], want[c])
    b = C.c_int64(0)
    assert L.qpsk_viterbi_bits_bound(dec._h, -1, C.byref(b)) == E.ERR_RANGE
    assert L.qpsk_viterbi_bits_bound(None, 5, C.byref(b)) == E.ERR_NULL
    # encoder
    enc = gpu.ConvEncoder(2)
    d_in = torch.zeros((2, 16), dtype=torch.uint8, device="cuda")
    d_out = torch.zeros((2, 32), dtype=torch.uint8, device="cuda")
    g = L.qpsk_conv_encode_dev
    assert g(enc._h, d_in.data_ptr(), 16, 16, d_out.data_ptr(), 31, None) == E.ERR_CAPACITY
    assert g(enc._h, d_in.data_ptr(), 16, 15, d_out.data_ptr(), 32, None) == E.ERR_ARG
    assert g(enc._h, d_in.data_ptr(), -1, 16, d_out.data_ptr(), 32, None) == E.ERR_RANGE
    assert g(None, d_in.data_ptr(), 16, 16, d_out.data_ptr(), 32, None) == E.ERR_NULL
    assert g(enc._h, None, 16, 16, d_out.data_ptr(), 32, None) == E.ERR_NULL


_CHILD = r"""
import json, os, sys
sys.path[:0] = [sys.argv[1], sys.argv[2]]
import numpy as np, torch
import qpsk_modulator_demodulator_b200 as Q
from torch.profiler import ProfilerActivity, profile
Q.set_device(int(sys.argv[3]))
torch.cuda.init(); torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    Q.ConvEncoder(3).encode(np.ones((3, 40), np.uint8))
    for diff in (False, True):
        Q.ViterbiDecoder(3, diff).flush(np.ones((3, 40), np.complex64))
    torch.cuda.synchronize()
ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA), key=lambda e: e.time_range.start)
print("LAUNCHES " + json.dumps([e.name for e in ev]))
"""


def test_every_instantiation_is_compiled_and_runs(gpu):
    """The FEC kernels of the library (cuobjdump -sass | cu++filt) are exactly the three instantiations, and the profiler,
    in a child process, sees each run for the calls that select it.  (The FEC kernels are listed here rather than in
    tests/kernel_variants.py, whose family table the dispatch tests of the other blocks enumerate.)"""
    sass = subprocess.check_output([kv._tool("cuobjdump"), "-sass", gpu._native.LIB_PATH], text=True)
    mangled = sorted(set(re.findall(r"Function : (\S+)", sass)))
    dem = subprocess.run([kv._tool("cu++filt")], input="\n".join(mangled) + "\n", capture_output=True, text=True,
                         check=True).stdout.splitlines()
    compiled = {n for n in map(_norm, dem) if n}
    assert compiled == INSTANTIATIONS, compiled
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-c", _CHILD, os.path.dirname(here), here, os.environ.get("LOCAL_RANK", "0")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    import json
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("LAUNCHES ")][-1]
    ran = [n for n in map(_norm, json.loads(line[len("LAUNCHES "):])) if n]
    assert ran == ["conv_encode_kernel", "viterbi_kernel<false>", "viterbi_kernel<true>"], ran


def test_frame_bits_dev_matches_host_framer(gpu):
    import torch
    rng = np.random.default_rng(41)
    Cn = 37
    start, end = b"START", b"END"
    streams = []
    for c in range(Cn):
        parts = []
        for f in range(int(rng.integers(0, 4))):
            pay = rng.integers(0, 256, int(rng.integers(1, 40)), dtype=np.uint8).tobytes()
            parts.append(np.unpackbits(np.frombuffer(start + pay + end, np.uint8)))
            parts.append(rng.integers(0, 2, int(rng.integers(0, 50))).astype(np.uint8))
        lead = rng.integers(0, 2, int(rng.integers(0, 30))).astype(np.uint8)
        streams.append(np.concatenate([lead] + parts) if parts else lead)
    kw = dict(channels=Cn, tsc=None)
    host = gpu.QPSKDeModulator(4000, 1000, **kw)
    dev = gpu.QPSKDeModulator(4000, 1000, **kw)
    pos = np.zeros(Cn, np.int64)
    cap, ld = 256, 700
    for k in range(4):                                           # ragged chunks: frames cross calls
        take = np.array([min(int(rng.integers(0, 300)), streams[c].size - pos[c]) for c in range(Cn)], np.int64)
        if k == 3:
            take = np.array([streams[c].size - pos[c] for c in range(Cn)], np.int64)
        rows = np.zeros((Cn, ld), np.uint8)
        for c in range(Cn):
            rows[c, : take[c]] = streams[c][pos[c]: pos[c] + take[c]]
        pos += take
        want = host.FrameBits(["".join(map(str, rows[c, : take[c]])) for c in range(Cn)], start, end, cap=cap)
        d_b = torch.from_numpy(rows).cuda()
        d_n = torch.from_numpy(take).cuda()
        d_p = torch.zeros((Cn, cap), dtype=torch.uint8, device="cuda")
        d_np = torch.full((Cn,), -1, dtype=torch.int64, device="cuda")
        dev.frame_bits_dev(d_b.data_ptr(), ld, d_n.data_ptr(), start, end, d_p.data_ptr(), cap, d_np.data_ptr())
        torch.cuda.synchronize()
        p, npb = d_p.cpu().numpy(), d_np.cpu().numpy()
        for c in range(Cn):
            assert p[c, : npb[c]].tobytes() == want[c], (k, c)
    L = gpu._native.lib()
    E = gpu._native
    z = torch.zeros(64, dtype=torch.int64, device="cuda")
    a = (dev._h, z.data_ptr(), 8, z.data_ptr())
    s, e = np.frombuffer(start, np.uint8).copy(), np.frombuffer(end, np.uint8).copy()
    ps, pe = C.c_void_p(s.ctypes.data), C.c_void_p(e.ctypes.data)
    assert L.qpsk_demod_frame_bits_dev(*a, ps, 0, pe, 3, z.data_ptr(), 8, z.data_ptr(), None) == E.ERR_ARG
    assert L.qpsk_demod_frame_bits_dev(*a, ps, 5, pe, 3, z.data_ptr(), 0, z.data_ptr(), None) == E.ERR_RANGE
    assert L.qpsk_demod_frame_bits_dev(*a, ps, 5, pe, 3, None, 8, z.data_ptr(), None) == E.ERR_NULL
    assert L.qpsk_demod_frame_bits_dev(dev._h, None, 8, z.data_ptr(), ps, 5, pe, 3, z.data_ptr(), 8, z.data_ptr(),
                                       None) == E.ERR_NULL
    assert L.qpsk_demod_frame_bits_dev(dev._h, z.data_ptr(), -1, z.data_ptr(), ps, 5, pe, 3, z.data_ptr(), 8,
                                       z.data_ptr(), None) == E.ERR_RANGE


# ---- end to end: coded against uncoded frames through the same channel ----------------------------------------------------
E2E_FS, E2E_RS = 8000, 2000                      # 4 samples per symbol
E2E_C = 256
E2E_PAYLOAD = 48
E2E_LEAD_BITS = 1200                             # uncoded random lead-in ahead of each frame: the loops lock on it
E2E_OFFSET_HZ = 8.0                              # carrier offset Costas tracks
E2E_START, E2E_END = b"START", b"END"
E2E_NOISE_DBFS = -13.0                           # pinned: see test_coded_frames_survive_where_uncoded_are_lost


def e2e_scene(gpu, noise_dbfs, seed=2024):
    """-> (fraction of uncoded payloads recovered, fraction of coded payloads recovered, rms of the Costas output).
    Per channel one burst: random lead-in, then the frame; uncoded: START payload END, coded: coded_frame_bits of the same
    payload.  Both go through the same SimChannel (seeded AWGN per channel, a small carrier offset); the uncoded burst to
    demod_bytes_dev, the coded one to constellation_dev -> ViterbiDecoder(differential=True).flush_dev -> frame_bits_dev.
    At one symbol rate the coded frame takes twice the symbols: the coding gain is paid for in throughput."""
    import torch
    rng = np.random.default_rng(seed)
    pays = [rng.integers(0, 256, E2E_PAYLOAD, dtype=np.uint8).tobytes() for _ in range(E2E_C)]
    mod = gpu.QPSKModulator(E2E_FS, E2E_RS, 0.35, 8, True, None)

    def bursts(coded):
        rows = []
        for c in range(E2E_C):
            lead = "".join(map(str, rng.integers(0, 2, E2E_LEAD_BITS)))
            if coded:
                frame = gpu.coded_frame_bits(pays[c], E2E_START, E2E_END)
            else:
                frame = gpu.BitPacker.BytesToBitString(E2E_START + pays[c] + E2E_END)
            rows.append(mod.Modulate(lead + frame + "0" * 64))
        n = max(r.size for r in rows)
        out = np.zeros((E2E_C, n), np.float32)
        for c, r in enumerate(rows):
            out[c, : r.size] = r
        return out

    results, rms = [], None
    ts = torch.cuda.Stream()                     # every call on one stream: a NULL stream means each handle's own
    st = ts.cuda_stream
    for coded in (False, True):
        with torch.cuda.stream(ts):
            tx = torch.from_numpy(bursts(coded)).cuda()
            nf = tx.shape[1]
            rx = torch.empty_like(tx)
            cap = 256
            d_p = torch.zeros((E2E_C, cap), dtype=torch.uint8, device="cuda")
            d_np = torch.zeros(E2E_C, dtype=torch.int64, device="cuda")
        ch = gpu.SimChannel(0.0, -E2E_OFFSET_HZ, E2E_FS, noise_dbfs=noise_dbfs, mode=1, seed=seed, channels=E2E_C)
        ch.apply_dev(tx.data_ptr(), nf, nf, rx.data_ptr(), nf, st)
        dem = gpu.QPSKDeModulator(E2E_FS, E2E_RS, 0.35, 8, channels=E2E_C, tsc=None)
        if not coded:
            dem.demod_bytes_dev(rx.data_ptr(), nf, nf, E2E_START, E2E_END, d_p.data_ptr(), cap, d_np.data_ptr(), st)
        else:
            ss = dem.bits_bound(nf)
            vit = gpu.ViterbiDecoder(E2E_C, differential=True)
            bc = vit.bits_bound(ss // 2)
            with torch.cuda.stream(ts):
                d_sym = torch.zeros((E2E_C, ss), dtype=torch.float32, device="cuda")
                d_ns = torch.zeros(E2E_C, dtype=torch.int32, device="cuda")
                d_b = torch.zeros((E2E_C, bc), dtype=torch.uint8, device="cuda")
                d_nb = torch.zeros(E2E_C, dtype=torch.int64, device="cuda")
            dem.constellation_dev(rx.data_ptr(), nf, nf, d_sym.data_ptr(), ss, d_ns.data_ptr(), st)
            vit.flush_dev(d_sym.data_ptr(), ss, d_ns.data_ptr(), d_b.data_ptr(), bc, d_nb.data_ptr(), st)
            dem.frame_bits_dev(d_b.data_ptr(), bc, d_nb.data_ptr(), E2E_START, E2E_END, d_p.data_ptr(), cap, d_np.data_ptr(),
                               st)
            ts.synchronize()
            sym, ns = d_sym.cpu().numpy(), d_ns.cpu().numpy()
            tail = np.concatenate([sym[c, ns[c]: 2 * ns[c]] for c in range(E2E_C)])   # second half of each burst: locked
            rms = float(np.sqrt(np.mean(tail.astype(np.float64) ** 2) * 2))
        ts.synchronize()
        p, npb = d_p.cpu().numpy(), d_np.cpu().numpy()
        results.append(np.mean([p[c, : npb[c]].tobytes() == pays[c] for c in range(E2E_C)]))
    return results[0], results[1], rms


def test_coded_frames_survive_where_uncoded_are_lost(gpu):
    """At E2E_NOISE_DBFS (seeded) the uncoded path loses at least a quarter of the frames and the coded path recovers
    every payload.  The coded frame is twice as long at one symbol rate: the gain is paid for in throughput."""
    unc, cod, rms = e2e_scene(gpu, E2E_NOISE_DBFS)
    assert unc <= 0.75, unc
    assert cod == 1.0, (cod, unc)
    assert 0.5 < rms < 2.0, rms                  # Costas output near unit amplitude, the level the default scale assumes
