"""GPU: the frame synchronizer (csrc/fsync.cu) bit-identical to tests/fsync_oracle.py: frame rows, counts and info at 1 to
16384 channels in both modes, at noise levels that put the metric near the threshold; ragged, zero, negative and
out-of-range counts, chunk invariance, strides and offsets, untouched guard bands, NaN input and reset; every argument
check and a slot-capacity refusal that leaves the state unchanged; the host form; the compiled and running kernels; and
end to end, the sync path against the marker framer on the K14 scene's bursts, differential and coherent."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import fec_oracle as V
import fsync_oracle as S
import kernel_variants as kv
from fsync_oracle import awgn, frame_bits, stream

pytestmark = pytest.mark.gpu

KERNELS = ("fsync_kernel<true>", "fsync_kernel<false>")
_KRE = re.compile(r"\bfsync_kernel\b(<[^<>]*>)")
GUARD = -7.0


def _norm(name):
    m = _KRE.search(name)
    return "fsync_kernel<" + kv._arg(m.group(1)[1:-1]) + ">" if m else None


class DevCall:
    """device buffers for one handle: process() runs process_dev on [C][lds] rows at a float offset, checks the guard
    bands around and inside every output, and returns per channel the list of (window, info) like the oracle"""

    def __init__(self, torch, fs, lds, slots=None, ldf=None, off=2):
        self.t, self.fs, self.lds, self.off = torch, fs, lds, off
        self.slots = slots if slots is not None else fs.slots_bound(lds // 2)
        self.ldf = ldf or 2 * fs.window_syms + 6
        Cn, Sn = fs.channels, fs.channels * self.slots
        self.d_sym = torch.zeros(off + Cn * lds + 8, dtype=torch.float32, device="cuda")
        self.d_n = torch.zeros(Cn, dtype=torch.int32, device="cuda")
        self.d_f = torch.full((Sn * self.ldf + 16,), GUARD, dtype=torch.float32, device="cuda")
        self.d_fn = torch.full((Sn + 2,), -5, dtype=torch.int32, device="cuda")
        self.d_nb = torch.full((Sn + 1,), -5, dtype=torch.int64, device="cuda")
        self.d_info = torch.full((Sn * 3 + 3,), -5, dtype=torch.int64, device="cuda")

    def process(self, Y, counts, stream=0):
        t, fs = self.t, self.fs
        Cn = fs.channels
        rows = np.zeros((Cn, self.lds), np.float32)
        w = min(Y.shape[1], self.lds // 2)
        rows[:, : 2 * w] = np.ascontiguousarray(Y[:, :w]).view(np.float32).reshape(Cn, -1)
        self.d_sym[self.off: self.off + Cn * self.lds] = t.from_numpy(rows.reshape(-1)).cuda()
        self.d_n.copy_(t.from_numpy(np.asarray(counts, np.int32)))
        self.d_f.fill_(GUARD)
        t.cuda.synchronize()
        fs.process_dev(self.d_sym.data_ptr() + 4 * self.off, self.lds, self.d_n.data_ptr(), self.slots,
                       self.d_f.data_ptr() + 8 * 4, self.ldf, self.d_fn.data_ptr(), self.d_nb.data_ptr(),
                       self.d_info.data_ptr(), stream)
        t.cuda.synchronize()
        f, fn, nb = self.d_f.cpu().numpy(), self.d_fn.cpu().numpy(), self.d_nb.cpu().numpy()
        info = self.d_info.cpu().numpy()[: 3 * Cn * self.slots].view(S.INFO)
        Sn = Cn * self.slots
        assert (f[:8] == GUARD).all() and (f[8 + Sn * self.ldf:] == GUARD).all()
        assert (fn[Sn:] == -5).all() and nb[Sn] == -5 and (self.d_info.cpu().numpy()[3 * Sn:] == -5).all()
        rows = f[8: 8 + Sn * self.ldf].reshape(max(Sn, 1), self.ldf) if Sn else np.zeros((0, self.ldf), np.float32)
        out = [[] for _ in range(Cn)]
        for c in range(Cn):
            for j in range(self.slots):
                k = c * self.slots + j
                assert info[k]["channel"] == c
                if fn[k] == 0:
                    assert nb[k] == 0 and info[k]["position"] == -1
                    assert (rows[k] == GUARD).all()                          # empty slot: row untouched
                    continue
                assert fn[k] == fs.window_syms and nb[k] == fs.payload_bytes
                assert all(fn[c * self.slots + i] > 0 for i in range(j))      # filled slots come first
                assert (rows[k, 2 * fn[k]:] == GUARD).all()
                out[c].append((rows[k, : 2 * fn[k]].copy().view(np.complex64), info[k]))
        return out


def _same(got, want):
    assert len(got) == len(want)
    for c, (g, w) in enumerate(zip(got, want)):
        assert len(g) == len(w), (c, [int(i["position"]) for _, i in g], [int(i["position"]) for _, i in w])
        for (wg, ig), (ww, iw) in zip(g, w):
            assert ig.tobytes() == iw.tobytes(), (c, ig, iw)
            assert np.array_equal(wg.view(np.uint32), ww.view(np.uint32)), c


def _scene(rng, Cn, differential, start, pay, end, n, levels):
    """per channel random pairs and frames from a pool of 16 payloads, rotated by j^(c mod 4), at a noise level cycling
    through `levels` (None = clean), trimmed to n symbols"""
    pool = [V.encode(frame_bits(start, rng.integers(0, 256, pay, dtype=np.uint8).tobytes(), end)[None])[0][0]
            for _ in range(16)]
    Y = np.zeros((Cn, n), np.complex64)
    for c in range(Cn):
        parts, m = [], 0
        while m < n:
            g = int(rng.integers(0, 120))
            f = pool[int(rng.integers(0, 16))]
            parts += [rng.integers(0, 2, 2 * g).astype(np.uint8), f]
            m += g + f.size // 2
        y = V.qpsk_symbols(np.concatenate(parts)[None], differential)[0][:n] * np.complex64(1j ** (c % 4))
        lvl = levels[c % len(levels)]
        Y[c] = y if lvl is None else awgn(rng, y, lvl)
    return Y


# near-miss levels: M / E at the true position straddles rho / 256 (DESIGN.md §3 K15)
LEVELS = {True: [None, -2.0, -1.0, 0.0], False: [None, -6.0, -5.0, -4.0]}
CASES = [(1, True), (1, False), (33, True), (33, False), (2048, True), (2048, False), (16384, True), (16384, False)]


@pytest.mark.parametrize("channels,differential", CASES)
def test_bit_identical_to_oracle(gpu, channels, differential):
    import torch
    rng = np.random.default_rng(channels + differential)
    start, pay, end = (b"ST", 4, b"E") if channels >= 2048 else (b"START", 12, b"END")
    n = 700 if channels >= 2048 else 2400
    Y = _scene(rng, channels, differential, start, pay, end, n, LEVELS[differential])
    fs = gpu.FrameSync(channels, differential, start, pay, len(end))
    ref = S.FrameSync(channels, differential, start, pay, len(end))
    assert (fs.pattern_syms, fs.frame_syms, fs.window_syms, fs.rho) == (ref.P, ref.F, ref.window, ref.rho)
    # two calls, ragged: the first ends inside frames and peak windows
    cut = rng.integers(0, n + 1, channels)
    cut[: min(channels, 4)] = [0, n, 1, n // 2][: min(channels, 4)]
    lds = 2 * n + 6
    dc = DevCall(torch, fs, lds)
    A = np.zeros_like(Y)
    B = np.zeros_like(Y)
    for c in range(channels):
        A[c, : cut[c]] = Y[c, : cut[c]]
        B[c, : n - cut[c]] = Y[c, cut[c]:]
    for X, k in ((A, cut), (B, n - cut)):
        got = dc.process(X, k)
        want = ref.process(X, k)
        _same(got, want)
    assert sum(len(w) for w in want) + sum(len(w) for w in got) > 0


def test_chunking_counts_strides_nan_and_reset(gpu):
    """any chunking gives the frames of one call; zero, negative and past-the-stride counts; NaN symbols; reset"""
    import torch
    rng = np.random.default_rng(4)
    Cn, n = 9, 1500
    for differential in (True, False):
        Y = _scene(rng, Cn, differential, b"AB", 3, b"Z", n, [None, -1.0 if differential else -4.0])
        Y[3, 200:230] = np.nan
        Y[4, 500] = np.complex64(complex(np.inf, -np.inf))
        ref = S.FrameSync(Cn, differential, b"AB", 3, 1)
        whole = ref.process(Y)
        assert sum(len(w) for w in whole) > 2 * Cn
        fs = gpu.FrameSync(Cn, differential, b"AB", 3, 1)
        for trial in range(2):
            lds = 2 * 160 + 2 * trial
            dc = DevCall(torch, fs, lds, off=2 * trial)
            got = [[] for _ in range(Cn)]
            at = np.zeros(Cn, np.int64)
            while (at < n).any():
                k = rng.integers(0, 161, Cn)
                k[rng.integers(0, Cn)] = 0
                X = np.zeros((Cn, 161), np.complex64)
                for c in range(Cn):
                    k[c] = min(k[c], n - at[c])
                    X[c, : k[c]] = Y[c, at[c]: at[c] + k[c]]
                big = rng.integers(0, Cn)
                k[big] = min(lds // 2, n - at[big])
                X[big, : k[big]] = Y[big, at[big]: at[big] + k[big]]
                dev_k = k.copy()
                if k[big] == lds // 2:
                    dev_k[big] = 10 ** 6                                       # past the stride: read as the stride
                neg = (k == 0) & (rng.random(Cn) < 0.5)
                dev_k[neg] = -3                                                # negative: read as 0
                for c, fr in enumerate(dc.process(X, dev_k)):
                    got[c] += fr
                at += k
            _same(got, whole)
            fs.reset()


def test_argument_checks_and_capacity_refusal(gpu):
    import torch
    L = gpu._native.lib()
    E = gpu._native
    h = C.c_void_p()
    st = (C.c_uint8 * 24)(*range(24))
    for args, code in (((0, 1, 24.0, st, 5, 8, 3, 0), E.ERR_UNSUPPORTED), ((16385, 1, 24.0, st, 5, 8, 3, 0), E.ERR_UNSUPPORTED),
                       ((1, 1, 0.0, st, 5, 8, 3, 0), E.ERR_RANGE), ((1, 1, float("nan"), st, 5, 8, 3, 0), E.ERR_RANGE),
                       ((1, 1, 24.0, st, 0, 8, 3, 0), E.ERR_RANGE), ((1, 1, 24.0, st, 25, 8, 3, 0), E.ERR_RANGE),
                       ((1, 1, 24.0, st, 5, 0, 3, 0), E.ERR_RANGE), ((1, 1, 24.0, st, 5, 65537, 3, 0), E.ERR_RANGE),
                       ((1, 1, 24.0, st, 5, 8, -1, 0), E.ERR_RANGE), ((1, 1, 24.0, st, 5, 8, 33, 0), E.ERR_RANGE),
                       ((1, 1, 24.0, st, 5, 8, 3, -1), E.ERR_RANGE), ((1, 1, 24.0, st, 5, 8, 3, 257), E.ERR_RANGE),
                       ((1, 1, 24.0, None, 5, 8, 3, 0), E.ERR_NULL)):
        assert L.qpsk_fsync_create(*args, C.byref(h)) == code, args
    assert L.qpsk_fsync_create(1, 0, 32.0, st, 24, 65536, 32, 256, C.byref(h)) == 0
    L.qpsk_fsync_destroy(h)
    assert L.qpsk_fsync_create(1, 0, 32.0, st, 5, 8, 3, 0, None) == E.ERR_NULL
    with pytest.raises(gpu.ArgumentOutOfRangeException):
        gpu.FrameSync(2, True, b"", 8, 3)
    fs = gpu.FrameSync(3, True, b"START", 8, 3)                       # F = 32 + 8 * 16 + 6 = 166, window 167
    assert fs.layout() == dict(P=72, F=166, window=167, payload_bit_offset=72, rho=S.RHO_DEFAULT)
    assert [fs.slots_bound(m) for m in (0, 1, 166, 167, 1000)] == [0, 1, 1, 2, 7]
    b = C.c_int64(0)
    assert L.qpsk_fsync_slots_bound(fs._h, -1, C.byref(b)) == E.ERR_RANGE
    assert L.qpsk_fsync_slots_bound(fs._h, 5, None) == E.ERR_NULL
    # a stream with one frame; the refused calls between the two halves must not move the state
    rng = np.random.default_rng(1)
    y, pos, _ = stream(rng, b"START", [bytes(8)], b"END", [60, 40], True)     # 267 symbols, the frame at 61
    ref = S.FrameSync(3, True, b"START", 8, 3)
    Y = np.tile(y, (3, 1))
    dc = DevCall(torch, fs, 2 * 300)
    _same(dc.process(Y[:, :150], [150] * 3), ref.process(Y[:, :150], 150))
    f = dc.d_f.data_ptr() + 32
    a = [fs._h, dc.d_sym.data_ptr(), 600, dc.d_n.data_ptr(), 2, f, 334, dc.d_fn.data_ptr(), dc.d_nb.data_ptr(),
         dc.d_info.data_ptr(), None]

    def call(**kw):
        b = list(a)
        for i, v in kw.items():
            b[int(i[1:])] = v
        return L.qpsk_fsync_process_dev(*b)
    before = [x.clone() for x in (dc.d_f, dc.d_fn, dc.d_nb, dc.d_info)]
    assert call(a4=1) == E.ERR_CAPACITY                                 # slots_bound(300) = 2
    assert call(a6=332) == E.ERR_CAPACITY                               # below 2 * window
    assert call(a2=-2) == E.ERR_RANGE and call(a4=-1) == E.ERR_RANGE and call(a6=-2) == E.ERR_RANGE
    assert call(a2=601) == E.ERR_ARG and call(a6=335) == E.ERR_ARG
    assert call(a1=a[1] + 4) == E.ERR_ARG and call(a3=a[3] + 4) == E.ERR_ARG and call(a5=f + 4) == E.ERR_ARG
    assert call(a7=a[7] + 4) == E.ERR_ARG and call(a8=a[8] + 4) == E.ERR_ARG and call(a9=a[9] + 4) == E.ERR_ARG
    for i in (0, 1, 3, 5, 7, 8, 9):
        assert call(**{f"a{i}": None}) == E.ERR_NULL, i
    torch.cuda.synchronize()
    for x, y0 in zip((dc.d_f, dc.d_fn, dc.d_nb, dc.d_info), before):
        assert torch.equal(x, y0)
    _same(dc.process(Y[:, 150:], [117] * 3), ref.process(Y[:, 150:], 117))
    assert ref.next[0] > pos[0]
    # host form: the same frames, and its own checks
    fs.reset()
    ref.reset()
    got = fs.process(Y)
    want = ref.process(Y)
    assert [[(w.view(np.uint32).tolist(), i.tobytes()) for w, i in g] for g in got] == \
           [[(w.view(np.uint32).tolist(), i.tobytes()) for w, i in g] for g in want]
    need = C.c_int64(0)
    hs = np.zeros(6, np.float32)
    hn = np.array([1, 4, 2], np.int64)
    ptr = lambda v: C.c_void_p(v.ctypes.data)                                # noqa: E731
    assert L.qpsk_fsync_process(fs._h, ptr(hs), 6, ptr(hn), 0, None, 334, None, None, None, C.byref(need)) == E.ERR_RANGE
    hn[1] = 3
    assert L.qpsk_fsync_process(fs._h, ptr(hs), 6, ptr(hn), 0, None, 334, None, None, None, C.byref(need)) == E.ERR_CAPACITY
    assert need.value == 1


def test_pattern_matches_coded_frame_bits(gpu):
    for start in (b"START", b"\x02", bytes(range(24))):
        bits = np.frombuffer(gpu.coded_frame_bits(b"\x5a" * 9, start, b"END").encode("ascii"), np.uint8) - ord("0")
        fs = gpu.FrameSync(1, False, start, 9, 3)
        assert bits.size == 2 * fs.frame_syms
        assert np.array_equal(bits[: 2 * fs.pattern_syms], S.pattern(start))


_CHILD = r"""
import json, sys
sys.path[:0] = [sys.argv[1], sys.argv[2]]
import numpy as np, torch
import qpsk_modulator_demodulator_b200 as Q
from torch.profiler import ProfilerActivity, profile
Q.set_device(int(sys.argv[3]))
torch.cuda.init(); torch.cuda.synchronize()
a, b = Q.FrameSync(2, True, b"ST", 4, 1), Q.FrameSync(2, False, b"ST", 4, 1)
y = np.zeros((2, 300), np.complex64)
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    a.process(y)
    b.process(y)
    torch.cuda.synchronize()
ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA), key=lambda e: e.time_range.start)
print("LAUNCHES " + json.dumps([e.name for e in ev]))
"""


def test_every_kernel_is_compiled_and_runs(gpu):
    """The synchronizer kernels of the library (cuobjdump -sass | cu++filt) are exactly the two modes, and the profiler,
    in a child process, sees each run.  (Listed here rather than in tests/kernel_variants.py, whose family table the
    dispatch tests of the other blocks enumerate.)"""
    sass = subprocess.check_output([kv._tool("cuobjdump"), "-sass", gpu._native.LIB_PATH], text=True)
    mangled = sorted(set(re.findall(r"Function : (\S+)", sass)))
    dem = subprocess.run([kv._tool("cu++filt")], input="\n".join(mangled) + "\n", capture_output=True, text=True,
                         check=True).stdout.splitlines()
    assert {n for n in map(_norm, dem) if n} == set(KERNELS)
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-c", _CHILD, os.path.dirname(here), here, os.environ.get("LOCAL_RANK", "0")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("LAUNCHES ")][-1]
    assert [n for n in map(_norm, json.loads(line[len("LAUNCHES "):])) if n] == list(KERNELS)


# ---- end to end: the K14 scene's bursts through the marker framer and through the synchronizer ---------------------------
E2E_FS, E2E_RS, E2E_C, E2E_PAYLOAD, E2E_LEAD_BITS, E2E_OFFSET_HZ = 8000, 2000, 256, 48, 1200, 8.0
E2E_START, E2E_END = b"START", b"END"


def sync_scene(gpu, noise_dbfs, differential=True, rotate=False, seed=2024):
    """The bursts of tests/test_gpu_rs.py::e2e_scene (same seed, payloads, lead-ins and channel), conv+RS frames,
    RS(64, 48).  differential=False sends and receives without differential encoding; rotate multiplies channel c's burst
    by j^(c mod 4).  -> dict: payloads recovered by the sync path (constellation_dev -> FrameSync.process_dev ->
    ViterbiDecoder(C * slots).flush_dev -> pack_bits_dev -> ReedSolomon.decode_dev, one stream) and by the marker framer
    path (differential only), each with its losses at the sync / framer and at RS, RS-accepted wrong payloads, and the
    rotations the synchronizer reported."""
    import torch
    rng = np.random.default_rng(seed)
    pays = [rng.integers(0, 256, E2E_PAYLOAD, dtype=np.uint8).tobytes() for _ in range(E2E_C)]
    rs = gpu.ReedSolomon(16, E2E_PAYLOAD, 1)
    mod = gpu.QPSKModulator(E2E_FS, E2E_RS, 0.35, 8, differential, None)
    leads = ["".join(map(str, rng.integers(0, 2, E2E_LEAD_BITS))) for _ in range(E2E_C)]
    rows = [mod.Modulate(leads[c] + gpu.coded_frame_bits(rs.encode(pays[c]), E2E_START, E2E_END) + "0" * 64)
            for c in range(E2E_C)]
    tx_h = np.zeros((E2E_C, max(r.size for r in rows)), np.float32)
    for c, r in enumerate(rows):
        z = r.view(np.complex64) * np.complex64(1j ** (c % 4) if rotate else 1)
        tx_h[c, : r.size] = z.view(np.float32)
    res = {}
    ts = torch.cuda.Stream()
    st = ts.cuda_stream
    with torch.cuda.stream(ts):
        tx = torch.from_numpy(tx_h).cuda()
        nf = tx.shape[1]
        rx = torch.empty_like(tx)
    ch = gpu.SimChannel(0.0, -E2E_OFFSET_HZ, E2E_FS, noise_dbfs=noise_dbfs, mode=1, seed=seed, channels=E2E_C)
    ch.apply_dev(tx.data_ptr(), nf, nf, rx.data_ptr(), nf, st)
    dem = gpu.QPSKDeModulator(E2E_FS, E2E_RS, 0.35, 8, channels=E2E_C, tsc=None, differentialEncoding=differential)
    ss = dem.bits_bound(nf)
    with torch.cuda.stream(ts):
        d_sym = torch.zeros((E2E_C, ss), dtype=torch.float32, device="cuda")
        d_ns = torch.zeros(E2E_C, dtype=torch.int32, device="cuda")
    dem.constellation_dev(rx.data_ptr(), nf, nf, d_sym.data_ptr(), ss, d_ns.data_ptr(), st)
    fs = gpu.FrameSync(E2E_C, differential, E2E_START, rs.n, len(E2E_END))
    slots = fs.slots_bound(ss // 2)
    Sn, ldf = E2E_C * slots, 2 * fs.window_syms
    vit = gpu.ViterbiDecoder(Sn, differential=differential)
    bc = vit.bits_bound(fs.window_syms)
    with torch.cuda.stream(ts):
        d_f = torch.zeros((Sn, ldf), dtype=torch.float32, device="cuda")
        d_fn = torch.zeros(Sn, dtype=torch.int32, device="cuda")
        d_nb = torch.zeros(Sn, dtype=torch.int64, device="cuda")
        d_info = torch.zeros((Sn, 3), dtype=torch.int64, device="cuda")
        d_b = torch.zeros((Sn, bc), dtype=torch.uint8, device="cuda")
        d_nbits = torch.zeros(Sn, dtype=torch.int64, device="cuda")
        d_p = torch.zeros((Sn, rs.n), dtype=torch.uint8, device="cuda")
        d_m = torch.zeros((Sn, rs.k), dtype=torch.uint8, device="cuda")
        d_nm = torch.zeros(Sn, dtype=torch.int64, device="cuda")
        d_s = torch.zeros((Sn, 1), dtype=torch.int32, device="cuda")
    fs.process_dev(d_sym.data_ptr(), ss, d_ns.data_ptr(), slots, d_f.data_ptr(), ldf, d_fn.data_ptr(), d_nb.data_ptr(),
                   d_info.data_ptr(), st)
    vit.flush_dev(d_f.data_ptr(), ldf, d_fn.data_ptr(), d_b.data_ptr(), bc, d_nbits.data_ptr(), st)
    gpu._native.check(gpu._native.lib().qpsk_pack_bits_dev(d_b.data_ptr() + fs.payload_bit_offset, bc, d_nbits.data_ptr(),
                                                           8 * rs.n, Sn, d_p.data_ptr(), rs.n, st))
    rs.decode_dev(d_p.data_ptr(), rs.n, d_nb.data_ptr(), Sn, d_m.data_ptr(), rs.k, d_nm.data_ptr(), d_s.data_ptr(), 1, st)
    ts.synchronize()
    fn, info = d_fn.cpu().numpy(), d_info.cpu().numpy().view(S.INFO).reshape(-1)
    m, nm, s = d_m.cpu().numpy(), d_nm.cpu().numpy(), d_s.cpu().numpy()[:, 0]
    good = np.zeros(E2E_C, bool)
    accepted = np.zeros(E2E_C, bool)
    wrong = 0
    for k in range(Sn):
        c = k // slots
        if fn[k] > 0 and nm[k] == rs.k and s[k] >= 0:
            ok = m[k].tobytes() == pays[c]
            good[c] |= ok
            accepted[c] = True
            wrong += not ok
    found = np.array([(fn[c * slots: (c + 1) * slots] > 0).any() for c in range(E2E_C)])
    rot = np.array([int(info[c * slots]["rotation"]) if fn[c * slots] > 0 else -1 for c in range(E2E_C)])
    res.update(sync=float(good.mean()), lost_sync=float((~found).mean()), lost_rs=float((found & ~accepted).mean()),
               wrong=int(wrong), frames=int((fn > 0).sum()), rotations=rot.tolist())
    if differential and not rotate:
        import test_gpu_rs
        r = test_gpu_rs.e2e_scene(gpu, noise_dbfs, seed)
        res.update(marker=r["conv_rs"], lost_framer=r["lost_framer"], marker_lost_rs=r["lost_rs"])
    return res


E2E_NOISE_DBFS = -8.0


def test_sync_path_beats_the_marker_framer(gpu):
    """the K14 scene at -8 dBFS, differential: the sync path recovers more payloads than the marker framer, loses clearly
    fewer at the sync than the framer does, and RS accepts no wrong payload (DESIGN.md §3 K15 has the table)"""
    r = sync_scene(gpu, E2E_NOISE_DBFS)
    print("E2E", json.dumps(r))
    assert r["sync"] > r["marker"], r
    assert r["lost_sync"] < 0.5 * r["lost_framer"], r
    assert r["wrong"] == 0, r


def test_coherent_sync_resolves_the_lock_phase(gpu):
    """coherent at -30 dBFS with channel c's burst multiplied by j^(c mod 4): every payload is recovered, so every
    reported rotation is the lock phase of its channel; and against the same bursts unrotated, the reported rotation of
    channel c steps by c mod 4 (compared channel by channel: where the Costas loop locks depends on the channel, and on
    a rare channel the rotated burst makes the loop lock one quadrant apart)"""
    r = sync_scene(gpu, -30.0, differential=False, rotate=True)
    plain = sync_scene(gpu, -30.0, differential=False, rotate=False)
    print("E2E", json.dumps({k: v for k, v in r.items() if k != "rotations"}))
    assert r["sync"] == 1.0 and plain["sync"] == 1.0 and r["wrong"] == 0, r
    rot, rot0 = np.array(r["rotations"]), np.array(plain["rotations"])
    step = (rot - rot0) % 4 == np.arange(E2E_C) % 4
    print("E2E rotation steps", json.dumps({"fraction": float(step.mean()), "off": np.nonzero(~step)[0].tolist(),
                                            "rot": rot[~step].tolist(), "rot0": rot0[~step].tolist()}))
    assert step.mean() >= 0.98, step.mean()                                # measured: 255 of 256 (DESIGN.md §3 K15)
