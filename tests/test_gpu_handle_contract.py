"""The lifecycle and refusal contract shared by the block handles (qpsk_fll, qpsk_mm, qpsk_costas, qpsk_eq, qpsk_agc,
qpsk_pfb, qpsk_ddc, qpsk_resamp, qpsk_conv, qpsk_viterbi, qpsk_rs, qpsk_fsync), one table row per handle:

  * a NULL handle is refused with QPSK_ERR_NULL by every entry point that takes one, and destroy(NULL) is QPSK_OK;
  * a NULL `out` is refused by every create;
  * reset() leaves a handle that gives the same outputs as a fresh one;
  * a refused call consumes nothing: after it, a valid call gives what it gives on a fresh handle;
  * a `_dev` call refuses a float2 row pointer that is not 8-byte aligned with QPSK_ERR_ARG, before it launches anything.

The per-block files test each block's arithmetic; this file tests what the handles have in common."""
import ctypes as C

import numpy as np
import pytest

from fsync_oracle import stream

pytestmark = pytest.mark.gpu

CH = 3


def _p(a):
    return a.ctypes.data


def _bits(v):
    """a call's output as one flat byte string (lists and tuples of arrays concatenated)"""
    if isinstance(v, (list, tuple)):
        return b"".join(_bits(u) for u in v)
    if isinstance(v, (bytes, np.void)):
        return bytes(v)
    return np.ascontiguousarray(v).tobytes()


class Block:
    """one handle: `make` builds it through api.py, `run` is a valid host call on fixed inputs, `refusals(L, obj)` are
    (status, expected, label) triples of calls that must be refused.  Blocks with float2-row `_dev` calls also give
    `dev_call(L, obj, d_in, d_out)`, a valid call over device buffers of the `dev_sizes()` floats."""
    name = ""
    has_reset = True
    creates = ()                          # (function, args before `out`)

    def __init__(self, q, torch):
        self.q, self.torch = q, torch

    @property
    def rng(self):
        """the same inputs for every handle `make` builds"""
        return np.random.default_rng(sum(map(ord, self.name)))

    def dev(self, n_floats):
        return self.torch.zeros(int(n_floats), dtype=self.torch.float32, device="cuda")


def _iq(rng, rows, n):
    return (rng.standard_normal((rows, 2 * n)) * 0.5).astype(np.float32)


class _Loop(Block):
    """fll / costas / eq: [channels][2n] floats in, the same shape out"""
    has_reset = False
    n = 600

    def setup(self):
        self.x = _iq(self.rng, CH, self.n)
        self.y = np.zeros_like(self.x)

    def run(self, obj):
        return obj.Process(self.x)

    def host_refusals(self, L, h, fn, cap_status):
        x, y, nf = _p(self.x), _p(self.y), 2 * self.n
        return [(fn(h, x, y, nf - 1, nf), self.q._native.ERR_ARG, "odd count"),
                (fn(h, x, y, nf, nf - 2), cap_status, "short output"),
                (fn(h, x, y, -2, nf), self.q._native.ERR_RANGE, "negative count"),
                (fn(h, None, y, nf, nf), self.q._native.ERR_NULL, "NULL input")]

    def dev_refusals(self, fn, extra):
        N = self.q._native
        nf = 2 * self.n
        dx, dy = self.dev(CH * nf), self.dev(CH * nf)
        x, y = dx.data_ptr(), dy.data_ptr()
        return [(fn(self.h, x, y, -2, nf, nf, *extra), N.ERR_RANGE, "dev negative count"),
                (fn(self.h, x, y, nf - 1, nf, nf, *extra), N.ERR_ARG, "dev odd count"),
                (fn(self.h, x, y, nf, nf + 1, nf, *extra), N.ERR_ARG, "dev odd in stride"),
                (fn(self.h, x, y, nf, nf, nf + 1, *extra), N.ERR_ARG, "dev odd out stride"),
                (fn(self.h, None, y, nf, nf, nf, *extra), N.ERR_NULL, "dev NULL input")]

    def dev_sizes(self):
        return 2 * self.n * CH, 2 * self.n * CH


class Fll(_Loop):
    name = "fll"
    creates = (("qpsk_fll_create", (4.0, 0.35, 40, 0.05)), ("qpsk_fll_create_batch", (4.0, 0.35, 40, 0.05, CH)))

    def make(self):
        self.setup()
        return self.q.FLLBandEdgeFilter(4.0, 0.35, 40, 0.05, channels=CH)

    def refusals(self, L, obj):
        self.h = obj._h
        return (self.host_refusals(L, obj._h, L.qpsk_fll_process, self.q._native.ERR_ARG) +
                self.dev_refusals(L.qpsk_fll_process_dev, (None,)))

    def dev_call(self, L, obj, d_in, d_out):
        nf = 2 * self.n
        return L.qpsk_fll_process_dev(obj._h, d_in, d_out, nf, nf, nf, None)


class Costas(_Loop):
    name = "costas"
    creates = (("qpsk_costas_create", (1e5, 500.0, 0.707)), ("qpsk_costas_create_batch", (1e5, 500.0, 0.707, CH)))

    def make(self):
        self.setup()
        return self.q.CostasLoopQpsk(1e5, 500.0, 0.707, channels=CH)

    def refusals(self, L, obj):
        self.h = obj._h
        return (self.host_refusals(L, obj._h, L.qpsk_costas_process, self.q._native.ERR_ARG) +
                self.dev_refusals(L.qpsk_costas_process_dev, (None, None)))

    def dev_call(self, L, obj, d_in, d_out):
        nf = 2 * self.n
        return L.qpsk_costas_process_dev(obj._h, d_in, d_out, nf, nf, nf, None, None)


class Eq(_Loop):
    name = "eq"
    has_reset = True
    creates = (("qpsk_eq_create", (7, 1e-3, 1.0)), ("qpsk_eq_create_batch", (7, 1e-3, 1.0, CH)),
               ("qpsk_eq_create_fractional", (7, 1e-3, 1.0, 2, CH)))

    def make(self):
        self.setup()
        return self.q.CmaEqualizer(7, 1e-3, channels=CH)

    def refusals(self, L, obj):
        self.h = obj._h
        return (self.host_refusals(L, obj._h, L.qpsk_eq_process, self.q._native.ERR_CAPACITY) +
                self.dev_refusals(L.qpsk_eq_process_dev, (None, None)))

    def dev_call(self, L, obj, d_in, d_out):
        nf = 2 * self.n
        return L.qpsk_eq_process_dev(obj._h, d_in, d_out, nf, nf, nf, None, None)


class Mm(Block):
    name = "mm"
    has_reset = False
    creates = (("qpsk_mm_create", (4.0, 0.01, 1e-4)), ("qpsk_mm_create_batch", (4.0, 0.01, 1e-4, CH)))
    n = 800

    def make(self):
        self.x = _iq(self.rng, CH, self.n)
        self.y = np.zeros_like(self.x)
        self.ns = np.zeros(CH, np.int32)
        return self.q.MuellerMuller(4.0, 0.01, 1e-4, channels=CH)

    def run(self, obj):
        return obj.Process(self.x)

    def refusals(self, L, obj):
        N = self.q._native
        h, x, y, ns, nf = obj._h, _p(self.x), _p(self.y), self.ns.ctypes.data_as(N.i32p), 2 * self.n
        dx, dy, dn = self.dev(CH * nf), self.dev(CH * nf), self.dev(CH)
        X, Y, D = dx.data_ptr(), dy.data_ptr(), dn.data_ptr()
        f, g = L.qpsk_mm_process, L.qpsk_mm_process_dev
        return [(f(h, x, nf, y, nf, None), N.ERR_NULL, "NULL n_sym"),
                (f(h, x, -2, y, nf, ns), N.ERR_RANGE, "negative count"),
                (f(h, x, nf, y, -2, ns), N.ERR_RANGE, "negative capacity"),
                (f(h, x, nf - 1, y, nf, ns), N.ERR_ARG, "odd count"),
                (f(h, None, nf, y, nf, ns), N.ERR_NULL, "NULL input"),
                (f(h, x, nf, None, nf, ns), N.ERR_NULL, "NULL output"),
                (g(h, X, -2, nf, Y, nf, nf, D, None), N.ERR_RANGE, "dev negative count"),
                (g(h, X, nf, nf, Y, -2, nf, D, None), N.ERR_RANGE, "dev negative capacity"),
                (g(h, X, nf - 1, nf, Y, nf, nf, D, None), N.ERR_ARG, "dev odd count"),
                (g(h, X, nf, nf + 1, Y, nf, nf, D, None), N.ERR_ARG, "dev odd in stride"),
                (g(h, X, nf, nf, Y, nf, nf + 1, D, None), N.ERR_ARG, "dev odd out stride"),
                (g(h, X, nf, nf, Y, nf, nf, None, None), N.ERR_NULL, "dev NULL n_sym"),
                (g(h, None, nf, nf, Y, nf, nf, D, None), N.ERR_NULL, "dev NULL input"),
                (g(h, X, nf, nf, None, nf, nf, D, None), N.ERR_NULL, "dev NULL output")]

    def dev_sizes(self):
        return 2 * self.n * CH, 2 * self.n * CH + CH

    def dev_call(self, L, obj, d_in, d_out):
        nf = 2 * self.n
        return L.qpsk_mm_process_dev(obj._h, d_in, nf, nf, d_out, nf, nf, d_out + 4 * CH * nf, None)


class Agc(Block):
    name = "agc"
    creates = (("qpsk_agc_create_batch", (16, 1.0, 65536.0, CH)),)
    n = 700

    def make(self):
        self.x = _iq(self.rng, CH, self.n)
        self.y = np.zeros_like(self.x)
        return self.q.Agc(16, channels=CH)

    def run(self, obj):
        return obj.process(self.x)

    def refusals(self, L, obj):
        N = self.q._native
        h, x, y, nf = obj._h, _p(self.x), _p(self.y), 2 * self.n
        dx, dy = self.dev(CH * nf), self.dev(CH * nf)
        X, Y = dx.data_ptr(), dy.data_ptr()
        f, g = L.qpsk_agc_process, L.qpsk_agc_process_dev
        return [(f(h, x, y, nf - 1, nf), N.ERR_ARG, "odd count"),
                (f(h, x, y, nf, nf - 2), N.ERR_CAPACITY, "short output"),
                (f(h, x, y, -2, nf), N.ERR_RANGE, "negative count"),
                (f(h, None, y, nf, nf), N.ERR_NULL, "NULL input"),
                (g(h, X, Y, nf, nf - 2, nf, None), N.ERR_ARG, "dev rows overlap"),
                (g(h, X, Y, nf, nf, nf - 2, None), N.ERR_CAPACITY, "dev short output"),
                (g(h, X + 4, Y, nf, nf, nf, None), N.ERR_ARG, "dev misaligned input"),
                (g(h, X, None, nf, nf, nf, None), N.ERR_NULL, "dev NULL output")]


class _Bank(Block):
    """pfb / ddc: one wideband stream in, [channels][n_out] out"""
    n = 1024

    def setup(self):
        self.x = _iq(self.rng, 1, self.n)[0]
        self.y = np.zeros(1 << 16, np.float32)
        self.no = C.c_int64(0)

    def run(self, obj):
        return obj.process(self.x)

    def bank_refusals(self, L, obj, f, g):
        N = self.q._native
        h, x, y, nf, no = obj._h, _p(self.x), _p(self.y), 2 * self.n, C.byref(self.no)
        dx, dy = self.dev(nf), self.dev(self.y.size)
        X, Y = dx.data_ptr(), dy.data_ptr()
        return [(f(h, x, nf - 1, y, nf, no), N.ERR_ARG, "odd count"),
                (f(h, x, -2, y, nf, no), N.ERR_RANGE, "negative count"),
                (f(h, x, nf, y, 0, no), N.ERR_CAPACITY, "short output"),
                (f(h, None, nf, y, nf, no), N.ERR_NULL, "NULL input"),
                (f(h, x, nf, y, nf, None), N.ERR_NULL, "NULL count"),
                (g(h, X, nf - 1, Y, nf, no, None), N.ERR_ARG, "dev odd count"),
                (g(h, X, nf, Y, nf + 1, no, None), N.ERR_ARG, "dev odd stride"),
                (g(h, X, nf, Y, 0, no, None), N.ERR_CAPACITY, "dev short output"),
                (g(h, None, nf, Y, nf, no, None), N.ERR_NULL, "dev NULL input")]

    def dev_sizes(self):
        return 2 * self.n, self.y.size

    def dev_call(self, L, obj, d_in, d_out, fn):
        nf = 2 * self.n
        return fn(obj._h, d_in, nf, d_out, nf, C.byref(self.no), None)


class Pfb(_Bank):
    name = "pfb"

    @property
    def creates(self):
        return (("qpsk_pfb_create", (self.taps.ctypes.data_as(self.q._native.f32p), self.taps.size, 8)),)

    def make(self):
        self.setup()
        self.taps = self.q.pfb_taps(8, 4, 0.5 / 8).astype(np.float32)
        return self.q.PfbChannelizer(self.taps, 8)

    def refusals(self, L, obj):
        return self.bank_refusals(L, obj, L.qpsk_pfb_process, L.qpsk_pfb_process_dev)

    def dev_call(self, L, obj, d_in, d_out):
        return _Bank.dev_call(self, L, obj, d_in, d_out, L.qpsk_pfb_process_dev)


class Ddc(_Bank):
    name = "ddc"

    @property
    def creates(self):
        N = self.q._native
        return (("qpsk_ddc_create", (self.taps.ctypes.data_as(N.f32p), self.taps.size, self.freqs.ctypes.data_as(N.f64p),
                                     self.freqs.size, 4)),)

    def make(self):
        self.setup()
        self.taps = (np.hanning(33) / np.hanning(33).sum()).astype(np.float32)
        self.freqs = np.array([0.1, -0.2, 0.3], np.float64)
        return self.q.DdcBank(self.taps, self.freqs, 4)

    def refusals(self, L, obj):
        return self.bank_refusals(L, obj, L.qpsk_ddc_process, L.qpsk_ddc_process_dev)

    def dev_call(self, L, obj, d_in, d_out):
        return _Bank.dev_call(self, L, obj, d_in, d_out, L.qpsk_ddc_process_dev)


class Resamp(Block):
    name = "resamp"
    n = 500

    @property
    def creates(self):
        return (("qpsk_resamp_create", (self.taps.ctypes.data_as(self.q._native.f32p), self.taps.size, 3, 2, CH)),)

    def make(self):
        self.taps = (3 * np.hanning(24) / np.hanning(24).sum()).astype(np.float32)
        self.x = _iq(self.rng, CH, self.n)
        self.y = np.zeros((CH, 4 * self.n), np.float32)
        self.no = C.c_int64(0)
        return self.q.Resampler(self.taps, 3, 2, CH)

    def run(self, obj):
        return obj.process(self.x)

    def refusals(self, L, obj):
        N = self.q._native
        h, x, y, nf, no = obj._h, _p(self.x), _p(self.y), 2 * self.n, C.byref(self.no)
        f = L.qpsk_resamp_process
        return [(f(h, x, nf - 1, y, 4 * self.n, no), N.ERR_ARG, "odd count"),
                (f(h, x, -2, y, 4 * self.n, no), N.ERR_RANGE, "negative count"),
                (f(h, x, nf, y, 0, no), N.ERR_CAPACITY, "short output"),
                (f(h, None, nf, y, 4 * self.n, no), N.ERR_NULL, "NULL input")]


class Conv(Block):
    name = "conv"
    creates = (("qpsk_conv_create", (CH,)),)
    n = 300

    def make(self):
        self.x = self.rng.integers(0, 2, (CH, self.n)).astype(np.uint8)
        self.y = np.zeros((CH, 2 * self.n), np.uint8)
        return self.q.ConvEncoder(CH)

    def run(self, obj):
        return obj.encode(self.x)

    def refusals(self, L, obj):
        N = self.q._native
        h, x, y = obj._h, _p(self.x), _p(self.y)
        return [(L.qpsk_conv_encode(h, x, -1, y), N.ERR_RANGE, "negative count"),
                (L.qpsk_conv_encode(h, None, self.n, y), N.ERR_NULL, "NULL input"),
                (L.qpsk_conv_encode(h, x, self.n, None), N.ERR_NULL, "NULL output")]


def _coded(rng):
    """CH rows of differential QPSK symbols that carry one coded frame each"""
    rows = [stream(rng, b"START", [rng.integers(0, 256, 16, dtype=np.uint8).tobytes()], b"END", [37 + 11 * c, 200],
                   True)[0] for c in range(CH)]
    n = min(r.size for r in rows)
    return np.stack([r[:n] for r in rows]).astype(np.complex64)


class Viterbi(Block):
    name = "viterbi"
    creates = (("qpsk_viterbi_create", (CH, 1, 24.0)),)

    def make(self):
        self.s = _coded(self.rng)
        self.sf = np.ascontiguousarray(self.s).view(np.float32)
        self.ns = np.full(CH, self.s.shape[1], np.int64)
        self.bits = np.zeros((CH, self.s.shape[1] + 200), np.uint8)
        self.nb = np.zeros(CH, np.int64)
        return self.q.ViterbiDecoder(CH, differential=True)

    def run(self, obj):
        return obj.decode(self.s) + obj.flush()

    def refusals(self, L, obj):
        N = self.q._native
        h, s, st, bits, cap = obj._h, _p(self.sf), self.sf.shape[1], _p(self.bits), self.bits.shape[1]
        f = L.qpsk_viterbi_decode
        big = self.ns + 1
        return [(f(h, s, st, _p(big), bits, cap, _p(self.nb)), N.ERR_RANGE, "count past the stride"),
                (f(h, s, st + 1, _p(self.ns), bits, cap, _p(self.nb)), N.ERR_ARG, "odd stride"),
                (f(h, s, st, _p(self.ns), bits, 8, _p(self.nb)), N.ERR_CAPACITY, "short output"),
                (f(h, s, st, _p(self.ns), None, cap, _p(self.nb)), N.ERR_NULL, "NULL output"),
                (f(h, None, st, _p(self.ns), bits, cap, _p(self.nb)), N.ERR_NULL, "NULL input")]


class Fsync(Block):
    name = "fsync"

    @property
    def creates(self):
        return (("qpsk_fsync_create", (CH, 1, 24.0, _p(self.start), 5, 16, 3, 0)),)

    def make(self):
        self.start = np.frombuffer(b"START", np.uint8).copy()
        self.s = _coded(self.rng)
        self.sf = np.ascontiguousarray(self.s).view(np.float32)
        self.ns = np.full(CH, self.s.shape[1], np.int64)
        fs = self.q.FrameSync(CH, True, b"START", 16, 3)
        self.slots = fs.slots_bound(self.s.shape[1])
        S = CH * self.slots
        self.frames = np.zeros((S, fs.window_syms), np.complex64)
        self.fn, self.nb = np.zeros(S, np.int32), np.zeros(S, np.int64)
        self.info = np.zeros(S, self.q.api.FSYNC_INFO)
        self.need = C.c_int64(0)
        return fs

    def run(self, obj):
        got = obj.process(self.s)
        assert sum(len(g) for g in got) == CH
        return [[w for f in g for w in f] for g in got]

    def refusals(self, L, obj):
        N = self.q._native
        st, L2 = self.sf.shape[1], 2 * self.frames.shape[1]
        rest = (_p(self.frames), L2, _p(self.fn), _p(self.nb), _p(self.info), C.byref(self.need))
        f = L.qpsk_fsync_process
        big = self.ns + 1
        return [(f(obj._h, _p(self.sf), st, _p(big), self.slots, *rest), N.ERR_RANGE, "count past the stride"),
                (f(obj._h, _p(self.sf), st + 1, _p(self.ns), self.slots, *rest), N.ERR_ARG, "odd stride"),
                (f(obj._h, _p(self.sf), st, _p(self.ns), 0, *rest), N.ERR_CAPACITY, "too few slots"),
                (f(obj._h, None, st, _p(self.ns), self.slots, *rest), N.ERR_NULL, "NULL input")]


class Rs(Block):
    name = "rs"
    has_reset = False
    creates = (("qpsk_rs_create", (4, 16, 2)),)

    def make(self):
        rs = self.q.ReedSolomon(4, 16, 2)
        msg = self.rng.integers(0, 256, 3 * 32, dtype=np.uint8).tobytes()
        code = np.frombuffer(rs.encode(msg), np.uint8).copy()
        code[[3, 50, 77]] ^= 0x5A
        self.code = code
        self.msg, self.st = np.zeros(3 * 32, np.uint8), np.zeros(6, np.int32)
        return rs

    def run(self, obj):
        return obj.decode(self.code.tobytes())

    def refusals(self, L, obj):
        N = self.q._native
        c, m, s = _p(self.code), _p(self.msg), _p(self.st)
        return [(L.qpsk_rs_decode(obj._h, c, -1, m, s), N.ERR_RANGE, "negative count"),
                (L.qpsk_rs_decode(obj._h, None, 3, m, s), N.ERR_NULL, "NULL input"),
                (L.qpsk_rs_encode(obj._h, m, 3, None), N.ERR_NULL, "NULL output")]


BLOCKS = [Fll, Mm, Costas, Eq, Agc, Pfb, Ddc, Resamp, Conv, Viterbi, Rs, Fsync]
IDS = [b.name for b in BLOCKS]
ALIGN = [Fll, Mm, Costas, Eq, Pfb, Ddc]      # the float2-row _dev calls this file checks for alignment


@pytest.fixture
def mk(gpu):
    import torch

    def make(cls):
        return cls(gpu, torch)
    return make


@pytest.mark.parametrize("cls", BLOCKS, ids=IDS)
def test_null_handle_and_null_out(gpu, mk, cls):
    N = gpu._native
    L = N.lib()
    prefix = f"qpsk_{cls.name}_"
    entry = [n for n, (_, args) in N._signatures().items()
             if n.startswith(prefix) and args and args[0] is C.c_void_p and not n.endswith("_destroy")]
    assert entry
    for name in entry:
        args = [None if (t is C.c_void_p or isinstance(t, type) and issubclass(t, C._Pointer)) else 0
                for t in N._signatures()[name][1]]
        assert getattr(L, name)(*args) == N.ERR_NULL, name
    assert getattr(L, prefix + "destroy")(None) == N.OK
    b = mk(cls)
    b.make()
    for fn, args in b.creates:
        assert getattr(L, fn)(*args, None) == N.ERR_NULL, fn
        h = C.c_void_p(1)
        assert getattr(L, fn)(*args, C.byref(h)) == N.OK, fn       # the same arguments are valid
        assert getattr(L, prefix + "destroy")(h) == N.OK


@pytest.mark.parametrize("cls", [b for b in BLOCKS if b.has_reset], ids=[b.name for b in BLOCKS if b.has_reset])
def test_reset_matches_a_fresh_handle(gpu, mk, cls):
    b = mk(cls)
    obj = b.make()
    first = _bits(b.run(obj))
    b.run(obj)
    obj.reset()
    assert _bits(b.run(obj)) == first
    fresh = b.make()
    assert _bits(b.run(fresh)) == first


@pytest.mark.parametrize("cls", BLOCKS, ids=IDS)
def test_refused_calls_consume_nothing(gpu, mk, cls):
    import torch
    b = mk(cls)
    obj = b.make()
    L = gpu._native.lib()
    for got, want, label in b.refusals(L, obj):
        assert got == want, (cls.name, label, got)
    torch.cuda.synchronize()
    after = [_bits(b.run(obj)), _bits(b.run(obj))]
    fresh = b.make()
    assert after == [_bits(b.run(fresh)), _bits(b.run(fresh))]


@pytest.mark.parametrize("cls", ALIGN, ids=[b.name for b in ALIGN])
def test_dev_calls_refuse_misaligned_rows(gpu, mk, cls):
    """Each of these calls checks alignment before it launches a kernel: a 4-byte-aligned float2 row pointer is refused
    with QPSK_ERR_ARG and leaves the handle as it was."""
    import torch
    N = gpu._native
    L = N.lib()
    b = mk(cls)
    obj = b.make()
    n_in, n_out = b.dev_sizes()
    d_in, d_out = b.dev(n_in + 2), b.dev(n_out + 2)
    x, y = d_in.data_ptr(), d_out.data_ptr()
    assert b.dev_call(L, obj, x + 4, y) == N.ERR_ARG
    assert b.dev_call(L, obj, x, y + 4) == N.ERR_ARG
    torch.cuda.synchronize()
    fresh = b.make()
    assert _bits(b.run(obj)) == _bits(b.run(fresh))
