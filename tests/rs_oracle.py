"""CPU restatement of the Reed-Solomon outer code of csrc/rs.cu (definition in include/qpskcuda.h).

Written from the definition, not from the kernel: the GPU must be bit-identical to it.
  * field GF(2^8), primitive polynomial x^8 + x^4 + x^3 + x^2 + 1 (0x11d), alpha = 0x02;
  * generator g(x) = prod_{j=0}^{nroots-1} (x - alpha^j); n = k + nroots <= 255 (a shortened code when n < 255);
  * codeword bytes c_0..c_{n-1}, c_0 first and the coefficient of x^{n-1}; message in c_0..c_{k-1}, parity in c_k..c_{n-1}
    the coefficients of m(x) x^nroots mod g(x);
  * a block interleaves I = depth codewords byte by byte: block byte p is byte p // I of codeword p % I;
  * decoding: a received codeword within Hamming distance t = nroots / 2 of a codeword of the shortened code becomes that
    codeword, status = the distance; otherwise status -1 and the received bytes pass through.  Implemented as
    Berlekamp-Massey + Chien + Forney with the checks the header lists (L <= t, deg Lambda = L, exactly L roots among the
    n valid positions, every Forney magnitude nonzero); `brute_decode` states the rule directly for tests.
Everything is vectorised over codewords."""
import itertools

import numpy as np

import fec_oracle as F

PRIM = 0x11D
EXP = np.zeros(512, np.int64)
LOG = np.zeros(256, np.int64)
_x = 1
for _i in range(255):
    EXP[_i] = _x
    LOG[_x] = _i
    _x <<= 1
    if _x & 0x100:
        _x ^= PRIM
EXP[255:510] = EXP[:255]
EXP[510:] = EXP[:2]


def gmul(a, b):
    a, b = np.asarray(a, np.int64), np.asarray(b, np.int64)
    return np.where((a == 0) | (b == 0), 0, EXP[LOG[a] + LOG[b]])


def gdiv(a, b):
    """a / b, b nonzero"""
    a, b = np.asarray(a, np.int64), np.asarray(b, np.int64)
    return np.where(a == 0, 0, EXP[(LOG[a] - LOG[b]) % 255])


def gpow(e):
    return EXP[np.asarray(e, np.int64) % 255]


def generator(nroots):
    """coefficients g[0..nroots] of g(x), g[i] the coefficient of x^i (g[nroots] = 1)"""
    g = np.array([1], np.int64)
    for j in range(nroots):
        # g(x) (x + alpha^j): shift up, plus alpha^j g
        g = np.concatenate([[0], g]) ^ np.concatenate([gmul(g, gpow(j)), [0]])
    return g


def poly_eval(coef_high_first, x):
    """sum_i c_i x^(len-1-i) by Horner; coef [..., m], x broadcast against coef[..., 0]"""
    coef = np.asarray(coef_high_first, np.int64)
    acc = np.zeros(np.broadcast(coef[..., 0], x).shape, np.int64)
    for i in range(coef.shape[-1]):
        acc = gmul(acc, x) ^ coef[..., i]
    return acc


class Code:
    def __init__(self, nroots=32, k=223, depth=1):
        assert nroots % 2 == 0 and 2 <= nroots <= 32 and k >= 1 and k + nroots <= 255 and 1 <= depth <= 8
        self.nroots, self.k, self.depth = nroots, k, depth
        self.n, self.t = k + nroots, nroots // 2
        self.g = generator(nroots)

    # ---- single codewords, [N, k] -> [N, n] ----
    def encode_words(self, msg):
        msg = np.atleast_2d(np.asarray(msg, np.int64))
        p = np.zeros((msg.shape[0], self.nroots), np.int64)      # p[:, 0] the coefficient of x^(nroots-1)
        gr = self.g[::-1][1:]                                      # g_{nroots-1} .. g_0
        for j in range(self.k):
            fb = msg[:, j] ^ p[:, 0]
            p = np.concatenate([p[:, 1:], np.zeros((p.shape[0], 1), np.int64)], axis=1) ^ gmul(fb[:, None], gr[None])
        return np.concatenate([msg, p], axis=1).astype(np.uint8)

    def syndromes(self, words):
        """[N, n] -> [N, nroots]: S_j = r(alpha^j)"""
        words = np.atleast_2d(np.asarray(words, np.int64))
        return poly_eval(words[:, None, :], gpow(np.arange(self.nroots))[None, :])

    def decode_words(self, words):
        """[N, n] received -> ([N, n] decoded (received where it fails), int32 status [N])"""
        r = np.atleast_2d(np.asarray(words, np.int64))
        N, nr, t, n = r.shape[0], self.nroots, self.t, self.n
        S = self.syndromes(r)
        out, status = r.copy(), np.zeros(N, np.int32)
        bad = np.nonzero(S.any(axis=1))[0]
        if bad.size == 0:
            return out.astype(np.uint8), status
        S = S[bad]
        M = bad.size
        W = nr + 1
        # Berlekamp-Massey over all bad words at once
        lam = np.zeros((M, W), np.int64)
        lam[:, 0] = 1
        B = lam.copy()
        L = np.zeros(M, np.int64)
        m = np.ones(M, np.int64)
        b = np.ones(M, np.int64)
        for rr in range(nr):
            d = S[:, rr].copy()
            for i in range(1, rr + 1):
                d ^= gmul(lam[:, i], S[:, rr - i])
            nz = d != 0
            coef = gdiv(d, b)
            src = np.arange(W)[None] - m[:, None]                  # x^m B
            shifted = np.where(src >= 0, np.take_along_axis(B, np.clip(src, 0, W - 1), axis=1), 0)
            upd = lam ^ gmul(coef[:, None], shifted)
            grow = nz & (2 * L <= rr)
            B = np.where(grow[:, None], lam, B)
            b = np.where(grow, d, b)
            L = np.where(grow, rr + 1 - L, L)
            m = np.where(grow, 1, m + 1)
            lam = np.where(nz[:, None], upd, lam)
        deg = W - 1 - np.argmax(lam[:, ::-1] != 0, axis=1)          # lam[:, 0] = 1 throughout
        ok = (L <= t) & (deg == L)
        # Chien: roots alpha^-e over the valid exponents e = 0..n-1 (byte n-1-e)
        e = np.arange(n)
        xinv = gpow(-e)                                            # [n]
        val = np.zeros((M, n), np.int64)
        for i in range(W - 1, -1, -1):
            val = gmul(val, xinv[None]) ^ lam[:, i:i + 1]
        roots = val == 0
        ok &= roots.sum(axis=1) == L
        # Forney: Omega = S Lambda mod x^nroots; e_l = X Omega(X^-1) / Lambda'(X^-1)
        om = np.zeros((M, nr), np.int64)
        for i in range(nr):
            for j in range(i + 1):
                om[:, i] ^= gmul(lam[:, j], S[:, i - j])
        num = np.zeros((M, n), np.int64)
        for i in range(nr - 1, -1, -1):
            num = gmul(num, xinv[None]) ^ om[:, i:i + 1]
        dlam = np.zeros((M, W), np.int64)
        dlam[:, 0:W - 1:2] = lam[:, 1::2][:, : (W // 2)]           # Lambda'(x) = sum_{i odd} Lambda_i x^(i-1)
        den = np.zeros((M, n), np.int64)
        for i in range(W - 1, -1, -1):
            den = gmul(den, xinv[None]) ^ dlam[:, i:i + 1]
        ok &= ~(roots & ((num == 0) | (den == 0))).any(axis=1)
        mag = np.where(roots & (den != 0), gmul(gpow(e)[None], gdiv(num, np.where(den == 0, 1, den))), 0)
        fix = np.nonzero(ok)[0]
        out[bad[fix]] ^= mag[fix][:, ::-1]                         # exponent e is byte n-1-e
        status[bad] = np.where(ok, L, -1)
        return out.astype(np.uint8), status

    # ---- blocks ----
    def encode(self, msg):
        """bytes or uint8 [n_blocks * I * k] -> uint8 [n_blocks * I * n]"""
        a = np.frombuffer(bytes(msg), np.uint8) if isinstance(msg, (bytes, bytearray)) else np.asarray(msg, np.uint8)
        I, k, n = self.depth, self.k, self.n
        nb = a.size // (I * k)
        assert a.size == nb * I * k
        words = a.reshape(nb, k, I).transpose(0, 2, 1).reshape(nb * I, k)
        return self.interleave(self.encode_words(words))

    def interleave(self, words):
        """[n_blocks * I, n] codewords in block order -> the block bytes"""
        I = self.depth
        w = np.asarray(words, np.uint8)
        nb = w.shape[0] // I
        return w.reshape(nb, I, w.shape[-1]).transpose(0, 2, 1).reshape(-1)

    def deinterleave(self, code):
        """block bytes [n_blocks * I * n] -> [n_blocks * I, n] codewords in block order"""
        I, n = self.depth, self.n
        a = np.asarray(code, np.uint8)
        nb = a.size // (I * n)
        return a[: nb * I * n].reshape(nb, n, I).transpose(0, 2, 1).reshape(nb * I, n)

    def decode(self, code):
        """block bytes (whole blocks; a remainder is ignored) -> (message bytes [n_blocks * I * k], status [n_blocks * I])"""
        I, k = self.depth, self.k
        words, status = self.decode_words(self.deinterleave(code))
        nb = words.shape[0] // I
        msg = words[:, :k].reshape(nb, I, k).transpose(0, 2, 1).reshape(-1)
        return msg.astype(np.uint8), status

    def decode_rows(self, rows, counts):
        """the device layout: rows [R, stride], counts [R] (read as clamp(count, 0, stride)) -> per row
        (message bytes, status), whole blocks only; decoded as one batch"""
        rows = np.asarray(rows, np.uint8)
        bb, mb = self.depth * self.n, self.depth * self.k
        nb = np.clip(np.asarray(counts, np.int64), 0, rows.shape[1]) // bb
        msg, st = self.decode(np.concatenate([rows[r, : nb[r] * bb] for r in range(rows.shape[0])] + [np.zeros(0, np.uint8)]))
        mo, so = np.concatenate([[0], np.cumsum(nb)]) * mb, np.concatenate([[0], np.cumsum(nb)]) * self.depth
        return [(msg[mo[r]: mo[r + 1]], st[so[r]: so[r + 1]]) for r in range(rows.shape[0])]


def brute_decode(code, words):
    """the decoding rule by enumeration (codes with k <= 2 only): the nearest of all 256^k codewords, taken when it lies
    within distance t -> (decoded words, status), as decode_words"""
    assert code.k <= 2
    msgs = np.array(list(itertools.product(range(256), repeat=code.k)), np.int64)
    book = code.encode_words(msgs).astype(np.int64)                  # [256^k, n]
    words = np.atleast_2d(np.asarray(words, np.int64))
    out, status = words.copy(), np.full(words.shape[0], -1, np.int32)
    for w in range(words.shape[0]):
        dist = (book != words[w][None]).sum(axis=1)
        j = int(np.argmin(dist))
        if dist[j] <= code.t:
            out[w], status[w] = book[j], dist[j]
    return out.astype(np.uint8), status


def viterbi_chain(rng, code, rows, ebn0_db, blocks=1):
    """rows x `blocks` RS blocks of random messages, each row ConvEncoder-coded (6 zero tail bits) onto coherent
    unit-amplitude symbols with AWGN at ebn0_db per information bit of the concatenated code (rate 1/2 x k/n), decoded by
    the oracle Viterbi decoder -> (messages [rows, blocks*I*k], sent code bytes [rows, L], Viterbi's bytes [rows, L])"""
    msg = rng.integers(0, 256, (rows, blocks * code.depth * code.k)).astype(np.uint8)
    sent = np.stack([code.encode(m) for m in msg])
    bits = np.concatenate([np.unpackbits(sent, axis=1), np.zeros((rows, 6), np.uint8)], axis=1)
    y = F.qpsk_symbols(F.encode(bits)[0], False)
    sig = np.sqrt(0.5 * code.n / code.k / 10 ** (ebn0_db / 10))
    y = (y + sig * (rng.standard_normal(y.shape) + 1j * rng.standard_normal(y.shape))).astype(np.complex64)
    dec = F.Viterbi(rows, False).flush(y, y.shape[1])
    got = np.stack([np.packbits(d[: sent.shape[1] * 8]) for d in dec])
    return msg, sent, got


def add_errors(rng, words, counts):
    """words [N, n] with counts[w] random nonzero symbol errors at distinct random positions"""
    out = np.asarray(words, np.uint8).copy()
    for w, c in enumerate(counts):
        pos = rng.choice(out.shape[1], int(c), replace=False)
        out[w, pos] ^= rng.integers(1, 256, int(c)).astype(np.uint8)
    return out
