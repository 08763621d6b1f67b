"""GPU: the Reed-Solomon outer code (csrc/rs.cu) bit-identical to tests/rs_oracle.py: encoder and decoder bytes, statuses
and counts, miscorrections included, at 1 to 16384 rows with error loads of 0, t, t + 1 and heavy, and on real Viterbi
burst patterns of the oracle chain; ragged device counts (0, partial blocks, past the stride, negative), strides, offsets,
row subsets and untouched guard bands; every argument check and a capacity refusal that enqueues nothing; the compiled and
running kernels; and end to end, conv+RS frames against conv-only frames through the same noisy channel."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import kernel_variants as kv
import rs_oracle as R

pytestmark = pytest.mark.gpu

KERNELS = ("rs_encode_kernel", "rs_decode_kernel")
_KRE = re.compile(r"\b(" + "|".join(KERNELS) + r")\b")
GUARD = 0xAB


def _norm(name):
    m = _KRE.search(name)
    return m.group(1) if m else None


def _loads(rng, code, N):
    """per codeword an error count cycling through 0, t, t + 1 and heavy (up to n)"""
    kinds = rng.integers(0, 4, N)
    heavy = rng.integers(code.t + 2, code.n + 1, N)
    return np.select([kinds == 0, kinds == 1, kinds == 2], [0, code.t, code.t + 1], heavy)


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _decode_dev(torch, rs, rows_u8, counts, ldc, off=0, ldm=None, lds=None, stream=0):
    """rows_u8 [R, ldc] at byte offset `off` of a buffer -> (msg rows, n_msg, status rows); the outputs are pre-filled
    with GUARD / -7 and the guard bands around them are checked"""
    Rn = rows_u8.shape[0]
    nb = ldc // rs.block_bytes
    ldm = ldm or max(nb * rs.depth * rs.k, 1)
    lds = lds or max(nb * rs.depth, 1)
    buf = torch.zeros(off + Rn * ldc + 16, dtype=torch.uint8, device="cuda")
    buf[off: off + Rn * ldc] = _dev(torch, rows_u8.reshape(-1))
    d_n = _dev(torch, np.asarray(counts, np.int64))
    d_m = torch.full((Rn * ldm + 64,), GUARD, dtype=torch.uint8, device="cuda")
    d_nm = torch.full((Rn,), -7, dtype=torch.int64, device="cuda")
    d_s = torch.full((Rn * lds + 16,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    rs.decode_dev(buf.data_ptr() + off, ldc, d_n.data_ptr(), Rn, d_m.data_ptr() + 32, ldm, d_nm.data_ptr(),
                  d_s.data_ptr() + 8 * 4, lds, stream)
    torch.cuda.synchronize()
    m, s = d_m.cpu().numpy(), d_s.cpu().numpy()
    assert (m[:32] == GUARD).all() and (m[32 + Rn * ldm:] == GUARD).all()
    assert (s[:8] == -7).all() and (s[8 + Rn * lds:] == -7).all()
    return m[32: 32 + Rn * ldm].reshape(Rn, ldm), d_nm.cpu().numpy(), s[8: 8 + Rn * lds].reshape(Rn, lds)


def _check_rows(code, rows, counts, msg, n_msg, status):
    want = code.decode_rows(rows, counts)
    for r, (wm, ws) in enumerate(want):
        assert n_msg[r] == wm.size, r
        assert np.array_equal(msg[r, : wm.size], wm), r
        assert (msg[r, wm.size:] == GUARD).all(), r                        # past the count: untouched
        assert np.array_equal(status[r, : ws.size], ws), r
        assert (status[r, ws.size:] == -7).all(), r
    return want


CASES = [(1, (32, 223, 4)), (1, (2, 10, 3)), (31, (16, 48, 1)), (32, (32, 223, 1)), (33, (2, 10, 3)), (33, (4, 1, 8)),
         (33, (32, 223, 8)), (2048, (32, 223, 4)), (2048, (16, 48, 1)), (16384, (16, 48, 1))]


@pytest.mark.parametrize("rows,params", CASES)
def test_bit_identical_to_oracle(gpu, rows, params):
    import torch
    code = R.Code(*params)
    rs = gpu.ReedSolomon(*params)
    assert (rs.n, rs.t, rs.block_bytes) == (code.n, code.t, code.depth * code.n)
    rng = np.random.default_rng(rows * 7 + params[0] + params[1])
    nb = 1 if rows * rs.block_bytes > 1 << 21 else 3
    mb = nb * rs.depth * rs.k
    ldm_in, ldc = mb + 5, nb * rs.block_bytes + 7
    msgs = rng.integers(0, 256, (rows, mb)).astype(np.uint8)
    # encoder: strided, offset message rows; guard bands around and between the code rows
    d_in = torch.zeros(rows * ldm_in + 3, dtype=torch.uint8, device="cuda")
    d_in[3:] = _dev(torch, np.pad(msgs, ((0, 0), (0, ldm_in - mb))).reshape(-1))
    d_c = torch.full((rows * ldc + 40,), GUARD, dtype=torch.uint8, device="cuda")
    rs.encode_dev(d_in.data_ptr() + 3, ldm_in, rows, nb, d_c.data_ptr() + 20, ldc)
    torch.cuda.synchronize()
    h = d_c.cpu().numpy()
    assert (h[:20] == GUARD).all() and (h[20 + rows * ldc:] == GUARD).all()
    sent = h[20: 20 + rows * ldc].reshape(rows, ldc)
    want = np.stack([code.encode(m) for m in msgs]) if rows <= 64 else code.encode(msgs.reshape(-1)).reshape(rows, -1)
    assert np.array_equal(sent[:, : nb * rs.block_bytes], want)
    assert (sent[:, nb * rs.block_bytes:] == GUARD).all()
    # decoder: every error load, ragged counts
    words = code.deinterleave(want.reshape(-1))
    rx = R.add_errors(rng, words, _loads(rng, code, words.shape[0]))
    # every fifth codeword a miscorrection: t + 1 errors on the support of a weight nroots + 1 codeword (the generator)
    gcw = code.encode_words(np.eye(1, code.k, code.k - 1, dtype=np.int64))[0]
    sup = np.nonzero(gcw)[0][: code.t + 1]
    rx[::5] = words[::5]
    rx[::5, sup] ^= gcw[sup]
    rows_rx = np.full((rows, ldc), 0x5A, np.uint8)
    rows_rx[:, : nb * rs.block_bytes] = code.interleave(rx).reshape(rows, -1)
    counts = np.full(rows, nb * rs.block_bytes, np.int64)
    if rows > 1:
        pick = rng.integers(0, 6, rows)
        counts = np.select([pick == 0, pick == 1, pick == 2, pick == 3],
                           [0, rng.integers(0, nb * rs.block_bytes + 1, rows), ldc + 1000, -5], counts)
    msg, n_msg, status = _decode_dev(torch, rs, rows_rx, counts, ldc, off=1)
    got = _check_rows(code, rows_rx, counts, msg, n_msg, status)
    st = np.concatenate([g[1] for g in got])
    assert st.size > 0 and (st == 0).any() or rows == 1
    dec, dst = code.decode_words(rx)
    assert ((dst == code.t) & (dec != words).any(axis=1)).any()              # miscorrections are among the words


@pytest.mark.parametrize("params", [(32, 223, 1), (32, 223, 4), (16, 48, 1), (2, 1, 2)])
def test_host_forms(gpu, params):
    code = R.Code(*params)
    rs = gpu.ReedSolomon(*params)
    rng = np.random.default_rng(params[1])
    msg = rng.integers(0, 256, 5 * rs.depth * rs.k).astype(np.uint8)
    enc = rs.encode(msg.tobytes())
    assert np.array_equal(np.frombuffer(enc, np.uint8), code.encode(msg))
    words = R.add_errors(rng, code.deinterleave(np.frombuffer(enc, np.uint8)), _loads(rng, code, 5 * rs.depth))
    rx = np.concatenate([code.interleave(words), np.full(rs.block_bytes - 1, 9, np.uint8)])   # remainder ignored
    got, st = rs.decode(rx.tobytes())
    wm, ws = code.decode(rx)
    assert np.frombuffer(got, np.uint8).tolist() == wm.tolist() and np.array_equal(st, ws)
    assert rs.encode(b"") == b"" and rs.decode(b"\x00" * (rs.block_bytes - 1))[0] == b""


@pytest.mark.parametrize("depth,ebn0", [(1, 2.0), (4, 2.0), (4, 2.5)])
def test_viterbi_burst_patterns(gpu, depth, ebn0):
    """the byte errors the oracle Viterbi decoder leaves on coherent AWGN: bursts, across interleaved codewords, at levels
    where some codewords fail"""
    import torch
    code = R.Code(32, 223, depth)
    rs = gpu.ReedSolomon(32, 223, depth)
    rows, nb = 64, 4 // depth
    msg, sent, got = R.viterbi_chain(np.random.default_rng(int(10 * ebn0) + depth), code, rows, ebn0, nb)
    assert (got != sent).any()
    ldc = got.shape[1]
    m, n_msg, st = _decode_dev(torch, rs, got, np.full(rows, ldc), ldc)
    want = _check_rows(code, got, np.full(rows, ldc), m, n_msg, st)
    allst = np.concatenate([w[1] for w in want])
    assert (allst > 0).any()
    if ebn0 == 2.0:
        assert (allst < 0).any()


def test_row_subsets_offsets_and_streams(gpu):
    """a subset of the rows decoded from an offset pointer, on a side stream, gives the rows of the full call"""
    import torch
    code = R.Code(16, 48, 2)
    rs = gpu.ReedSolomon(16, 48, 2)
    rng = np.random.default_rng(77)
    rows, ldc = 40, 3 * rs.block_bytes + 3
    msgs = rng.integers(0, 256, (rows, 3 * 2 * 48)).astype(np.uint8)
    rx = np.zeros((rows, ldc), np.uint8)
    for r in range(rows):
        w = R.add_errors(rng, code.deinterleave(code.encode(msgs[r])), rng.integers(0, 10, 6))
        rx[r, : 3 * rs.block_bytes] = code.interleave(w)
    counts = rng.integers(0, ldc + 1, rows)
    full = _decode_dev(torch, rs, rx, counts, ldc)
    ts = torch.cuda.Stream()
    sub = _decode_dev(torch, rs, rx[11:29], counts[11:29], ldc, off=5, stream=ts.cuda_stream)
    for a, b in zip(full, sub):
        assert np.array_equal(a[11:29], b)
    _check_rows(code, rx, counts, *full)


def test_argument_checks_and_capacity_refusal(gpu):
    import torch
    L = gpu._native.lib()
    E = gpu._native
    h = C.c_void_p()
    for nr, k, d, st in ((0, 10, 1, E.ERR_UNSUPPORTED), (3, 10, 1, E.ERR_UNSUPPORTED), (34, 10, 1, E.ERR_UNSUPPORTED),
                         (4, 10, 0, E.ERR_UNSUPPORTED), (4, 10, 9, E.ERR_UNSUPPORTED), (4, 0, 1, E.ERR_RANGE),
                         (32, 224, 1, E.ERR_RANGE), (2, 254, 1, E.ERR_RANGE)):
        assert L.qpsk_rs_create(nr, k, d, C.byref(h)) == st, (nr, k, d)
    assert L.qpsk_rs_create(2, 253, 8, C.byref(h)) == 0
    L.qpsk_rs_destroy(h)
    assert L.qpsk_rs_create(4, 10, 1, None) == E.ERR_NULL
    with pytest.raises(gpu.ArgumentOutOfRangeException):
        gpu.ReedSolomon(32, 224)
    rs = gpu.ReedSolomon(4, 10, 2)                                          # block: 28 code bytes, 20 message bytes
    z = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    p = z.data_ptr()
    enc = L.qpsk_rs_encode_dev
    assert enc(rs._h, p, 40, 2, 2, p + 1024, 56, None) == 0
    assert enc(rs._h, p, 39, 2, 2, p + 1024, 56, None) == E.ERR_ARG
    assert enc(rs._h, p, 40, 2, 2, p + 1024, 55, None) == E.ERR_CAPACITY
    assert enc(rs._h, p, 40, -1, 2, p + 1024, 56, None) == E.ERR_RANGE
    assert enc(rs._h, p, 40, 2, -1, p + 1024, 56, None) == E.ERR_RANGE
    assert enc(None, p, 40, 2, 2, p + 1024, 56, None) == E.ERR_NULL
    assert enc(rs._h, None, 40, 2, 2, p + 1024, 56, None) == E.ERR_NULL
    assert enc(rs._h, None, 40, 0, 2, None, 56, None) == 0                  # nothing to do
    # decode: a refused call enqueues nothing
    cnt = torch.full((2,), 56, dtype=torch.int64, device="cuda")
    d_m = torch.full((100,), GUARD, dtype=torch.uint8, device="cuda")
    d_nm = torch.full((2,), -7, dtype=torch.int64, device="cuda")
    d_s = torch.full((16,), -7, dtype=torch.int32, device="cuda")
    dec = L.qpsk_rs_decode_dev
    a = [rs._h, p, 56, cnt.data_ptr(), 2, d_m.data_ptr(), 40, d_nm.data_ptr(), d_s.data_ptr(), 4, None]

    def call(**kw):
        b = list(a)
        for i, v in kw.items():
            b[int(i[1:])] = v
        return dec(*b)
    assert call(a6=39) == E.ERR_CAPACITY
    assert call(a9=3) == E.ERR_CAPACITY
    assert call(a2=-1) == E.ERR_RANGE and call(a4=-1) == E.ERR_RANGE and call(a9=-1) == E.ERR_RANGE
    assert call(a0=None) == E.ERR_NULL and call(a1=None) == E.ERR_NULL and call(a3=None) == E.ERR_NULL
    assert call(a5=None) == E.ERR_NULL and call(a7=None) == E.ERR_NULL and call(a8=None) == E.ERR_NULL
    assert call(a3=a[3] + 4) == E.ERR_ARG and call(a7=a[7] + 4) == E.ERR_ARG and call(a8=a[8] + 2) == E.ERR_ARG
    torch.cuda.synchronize()
    assert (d_m.cpu().numpy() == GUARD).all() and (d_nm.cpu().numpy() == -7).all() and (d_s.cpu().numpy() == -7).all()
    # a stride below one block: counts are still written, nothing else
    assert call(a2=27, a6=0, a9=0) == 0
    torch.cuda.synchronize()
    assert (d_nm.cpu().numpy() == 0).all() and (d_m.cpu().numpy() == GUARD).all() and (d_s.cpu().numpy() == -7).all()
    assert call() == 0
    torch.cuda.synchronize()
    assert (d_nm.cpu().numpy() == 40).all()
    hm, hs = np.zeros(40, np.uint8), np.zeros(4, np.int32)
    hc = np.zeros(56, np.uint8)
    ptr = lambda v: C.c_void_p(v.ctypes.data)                                # noqa: E731
    assert L.qpsk_rs_decode(rs._h, ptr(hc), -1, ptr(hm), ptr(hs)) == E.ERR_RANGE
    assert L.qpsk_rs_decode(rs._h, ptr(hc), 2, ptr(hm), None) == E.ERR_NULL
    assert L.qpsk_rs_encode(rs._h, None, 2, ptr(hc)) == E.ERR_NULL
    assert L.qpsk_rs_decode(rs._h, ptr(hc), 2, ptr(hm), ptr(hs)) == 0 and (hs == 0).all()


_CHILD = r"""
import json, sys
sys.path[:0] = [sys.argv[1], sys.argv[2]]
import numpy as np, torch
import qpsk_modulator_demodulator_b200 as Q
from torch.profiler import ProfilerActivity, profile
Q.set_device(int(sys.argv[3]))
torch.cuda.init(); torch.cuda.synchronize()
rs = Q.ReedSolomon(4, 10, 1)
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    code = rs.encode(bytes(20))
    rs.decode(code)
    torch.cuda.synchronize()
ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA), key=lambda e: e.time_range.start)
print("LAUNCHES " + json.dumps([e.name for e in ev]))
"""


def test_every_kernel_is_compiled_and_runs(gpu):
    """The RS kernels of the library (cuobjdump -sass | cu++filt) are exactly the two, and the profiler, in a child
    process, sees each run.  (Listed here rather than in tests/kernel_variants.py, whose family table the dispatch tests of
    the other blocks enumerate.)"""
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
    assert [n for n in map(_norm, json.loads(line[len("LAUNCHES "):])) if n] == ["rs_encode_kernel", "rs_decode_kernel"]


# ---- end to end: conv-only against conv+RS frames through the same channel ------------------------------------------------
E2E_FS, E2E_RS = 8000, 2000                      # 4 samples per symbol
E2E_C = 256
E2E_PAYLOAD = 48                                 # conv+RS: the same 48 bytes as one RS(64, 48) codeword
E2E_LEAD_BITS = 1200
E2E_OFFSET_HZ = 8.0
E2E_START, E2E_END = b"START", b"END"
E2E_NOISE_DBFS = -8.0                            # pinned: see test_rs_frames_survive_where_conv_only_are_lost


def e2e_scene(gpu, noise_dbfs, seed=2024):
    """-> dict: fraction of payloads recovered by conv-only and by conv+RS frames, and for conv+RS the fractions lost at the
    framer (d_n_bytes other than 64) and at RS (a status of -1 on a whole frame), plus `wrong`, rows whose every status is
    >= 0 but whose message differs from the payload sent.  Per channel one burst: random lead-in, then the frame; conv-only:
    coded_frame_bits(payload), conv+RS: coded_frame_bits(ReedSolomon(16, 48).encode(payload)), 64 bytes between the
    markers.  Both go through the same SimChannel and constellation_dev -> ViterbiDecoder.flush_dev -> frame_bits_dev; the
    RS frames then through ReedSolomon.decode_dev, all on one stream."""
    import torch
    rng = np.random.default_rng(seed)
    pays = [rng.integers(0, 256, E2E_PAYLOAD, dtype=np.uint8).tobytes() for _ in range(E2E_C)]
    rs = gpu.ReedSolomon(16, E2E_PAYLOAD, 1)
    mod = gpu.QPSKModulator(E2E_FS, E2E_RS, 0.35, 8, True, None)
    leads = ["".join(map(str, rng.integers(0, 2, E2E_LEAD_BITS))) for _ in range(E2E_C)]

    def bursts(outer):
        rows = [mod.Modulate(leads[c] + gpu.coded_frame_bits(rs.encode(pays[c]) if outer else pays[c], E2E_START, E2E_END)
                             + "0" * 64) for c in range(E2E_C)]
        out = np.zeros((E2E_C, max(r.size for r in rows)), np.float32)
        for c, r in enumerate(rows):
            out[c, : r.size] = r
        return out

    res = {}
    ts = torch.cuda.Stream()
    st = ts.cuda_stream
    for outer in (False, True):
        with torch.cuda.stream(ts):
            tx = torch.from_numpy(bursts(outer)).cuda()
            nf = tx.shape[1]
            rx = torch.empty_like(tx)
            cap = 256
            d_p = torch.zeros((E2E_C, cap), dtype=torch.uint8, device="cuda")
            d_np = torch.zeros(E2E_C, dtype=torch.int64, device="cuda")
        ch = gpu.SimChannel(0.0, -E2E_OFFSET_HZ, E2E_FS, noise_dbfs=noise_dbfs, mode=1, seed=seed, channels=E2E_C)
        ch.apply_dev(tx.data_ptr(), nf, nf, rx.data_ptr(), nf, st)
        dem = gpu.QPSKDeModulator(E2E_FS, E2E_RS, 0.35, 8, channels=E2E_C, tsc=None)
        ss = dem.bits_bound(nf)
        vit = gpu.ViterbiDecoder(E2E_C, differential=True)
        bc = vit.bits_bound(ss // 2)
        with torch.cuda.stream(ts):
            d_sym = torch.zeros((E2E_C, ss), dtype=torch.float32, device="cuda")
            d_ns = torch.zeros(E2E_C, dtype=torch.int32, device="cuda")
            d_b = torch.zeros((E2E_C, bc), dtype=torch.uint8, device="cuda")
            d_nb = torch.zeros(E2E_C, dtype=torch.int64, device="cuda")
            d_m = torch.zeros((E2E_C, cap), dtype=torch.uint8, device="cuda")
            d_nm = torch.zeros(E2E_C, dtype=torch.int64, device="cuda")
            d_s = torch.zeros((E2E_C, cap // rs.n), dtype=torch.int32, device="cuda")
        dem.constellation_dev(rx.data_ptr(), nf, nf, d_sym.data_ptr(), ss, d_ns.data_ptr(), st)
        vit.flush_dev(d_sym.data_ptr(), ss, d_ns.data_ptr(), d_b.data_ptr(), bc, d_nb.data_ptr(), st)
        dem.frame_bits_dev(d_b.data_ptr(), bc, d_nb.data_ptr(), E2E_START, E2E_END, d_p.data_ptr(), cap, d_np.data_ptr(), st)
        if outer:
            rs.decode_dev(d_p.data_ptr(), cap, d_np.data_ptr(), E2E_C, d_m.data_ptr(), cap, d_nm.data_ptr(), d_s.data_ptr(),
                          cap // rs.n, st)
        ts.synchronize()
        p, npb = d_p.cpu().numpy(), d_np.cpu().numpy()
        if not outer:
            res["conv"] = float(np.mean([p[c, : npb[c]].tobytes() == pays[c] for c in range(E2E_C)]))
            continue
        m, nm, s = d_m.cpu().numpy(), d_nm.cpu().numpy(), d_s.cpu().numpy()
        framed = npb == rs.n
        okrs = framed & (nm == E2E_PAYLOAD) & (s[:, 0] >= 0)
        good = np.array([m[c, : nm[c]].tobytes() == pays[c] for c in range(E2E_C)])
        res.update(conv_rs=float(np.mean(good & okrs)), lost_framer=float(np.mean(~framed)),
                   lost_rs=float(np.mean(framed & (s[:, 0] < 0))), wrong=int((okrs & ~good).sum()),
                   corrected=int(s[okrs, 0].sum()))
    return res


def test_rs_frames_survive_where_conv_only_are_lost(gpu):
    """At E2E_NOISE_DBFS (seeded) conv+RS frames recover at least twice the payloads of conv-only frames, and every frame
    RS accepts carries the payload sent.  The RS frame is 64 payload bytes against 48: n/k more symbols per frame."""
    r = e2e_scene(gpu, E2E_NOISE_DBFS)
    assert r["conv_rs"] >= 2 * r["conv"] and r["conv_rs"] > 0.2, r
    assert r["wrong"] == 0, r
