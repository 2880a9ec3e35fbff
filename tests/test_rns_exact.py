"""Exact RNS basis conversion and scale-and-round (Halevi-Polyakov-Shoup): nttb200_rns_base_convert_exact
(the centred value of x mod B in the target basis) and nttb200_rns_scale_round (round(t X / B) on the
target channels).  The FP64 model of the correction against big-integer CRT on the CPU, including the
rounding band; on the GPU the results against Python-int CRT, the relation to the fast conversion,
the buffer rules, one call over 2^31 words, and a BFV multiplication and decryption at N = 4096 and
2^14 bit-identical to a big-integer reference."""
import math
import random
from fractions import Fraction

import numpy as np
import pytest

from test_rns_conv import (CONVERT_CASES, L2_WORDS, Consts, convert_ref, crt, overshoot, residues,
                           sample_cols, split_primes, to_dev)
from test_rns_eval import SENTINEL, Guarded, _status, channel_tables, host, ones_plan, rand_rns, rows_of

OK, INVALID_ARG, UNSUPPORTED = 0, 1, 7
T_VALUES = [1, 3, 1 << 16, 65537, (1 << 32) - 1]


# ------------------------------------------------------------------ CPU: argument checks
def test_null_arguments_without_device(lib):
    L = lib.load_library()
    assert L.nttb200_rns_base_convert_exact(None, 16, 0, 16, 0, 1, None) == INVALID_ARG
    assert L.nttb200_rns_base_convert_exact(None, None, 0, None, 0, 0, None) == INVALID_ARG
    assert L.nttb200_rns_scale_round(None, 16, 16, 1, 3, None) == INVALID_ARG
    assert L.nttb200_rns_scale_round(None, None, None, 0, 1, None) == INVALID_ARG
    assert L.nttb200_rns_scale_round(None, 16, 16, 1, 0, None) == INVALID_ARG


# --------------------------------------------------- CPU: the FP64 model of the correction
def fma(a, b, c):
    """IEEE double fma: exact a*b + c, rounded once (Python's int / int division rounds correctly)."""
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def model_v(ys, bs):
    """v as the kernel computes it: sum_i fma(y_i, fl(1/b_i), .) in order, then rint (half to even)."""
    f = 0.0
    for y, b in zip(ys, bs):
        f = fma(float(y), 1.0 / b, f)
    return int(f + 2.0 ** 52) - (1 << 52)


def model_exact(x, k):
    """The exact conversion of x in [0, B) through the model, as an integer (before mod c_j)."""
    ys = [(x % b) * w % b for b, w in zip(k.bs, k.w)]
    return sum(y * (k.B // b) for y, b in zip(ys, k.bs)) - model_v(ys, k.bs) * k.B


def centred(x, m):
    r = x % m
    return r - m if r > m // 2 else r


@pytest.mark.parametrize("S", [1, 2, 8, 16, 17, 32])
def test_model_against_crt(S):
    """Random x, small +-x, every y_i = b_i - 1 and x at B (1/2 -+ 2^-40): all exact."""
    bs, = split_primes(S)
    k = Consts(bs, [])
    rng = random.Random(1000 + S)
    xs = [rng.randrange(k.B) for _ in range(200)] + [0, 1, 2, 77, k.B - 1, k.B - 2, k.B - 77]
    xs.append(crt([(-(k.B // b)) % b for b in bs], bs))                       # y_i = b_i - 1
    lo, hi = (k.B * ((1 << 39) - 1)) >> 40, -((-k.B * ((1 << 39) + 1)) >> 40)   # floor / ceil
    xs += [lo, lo - 1, hi, hi + 1]
    for x in xs:
        assert model_exact(x, k) == centred(x, k.B), x


def test_model_band():
    """Inside the band either neighbour may come back: x = B/2 - 5 at S = 16 lies within 2^-40 of
    1/2, and the model returns x_c or x_c - B."""
    bs, = split_primes(16)
    k = Consts(bs, [])
    x = k.B // 2 - 5
    assert abs(Fraction(x, k.B) - Fraction(1, 2)) < Fraction(1, 1 << 40)
    assert model_exact(x, k) in (x, x - k.B)


def test_decryption_identity():
    """round(t X / Q) = -[t X]_Q Q^-1 (mod t), the decryption route through the exact conversion."""
    rng = random.Random(7)
    Q = math.prod(split_primes(3)[0])
    for t in (65537, 1 << 16, 257):
        for _ in range(200):
            X = rng.randrange(-Q, 2 * Q)
            assert (2 * t * X + Q) // (2 * Q) % t == -centred(t * X, Q) * pow(Q, -1, t) % t


# ------------------------------------------------------------------------ GPU helpers
def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"
    return torch


def exact_ref(x, k):
    """numpy: the fast conversion less v (B mod c_j), v = rint(sum y_i / b_i) in float64 (exact
    outside the band, which random data does not meet)."""
    bc = np.array(k.bs, dtype=np.uint64)[:, None]
    y = x % bc * np.array(k.w, dtype=np.uint64)[:, None] % bc
    v = np.rint((y.astype(np.float64) / bc.astype(np.float64)).sum(axis=-2)).astype(np.uint64)
    out = convert_ref(x, k)
    for j, c in enumerate(k.cs):
        out[..., j, :] = (out[..., j, :] + np.uint64(c) - v * np.uint64(k.B % c) % np.uint64(c)) % np.uint64(c)
    return out


def scale_round_ref(x, k, t):
    """numpy: round(t X / B) mod c_j on [..., T+S, N] (target channels first)."""
    T = len(k.cs)
    bc = np.array(k.bs, dtype=np.uint64)[:, None]
    tw = np.array([w * t % b for w, b in zip(k.w, k.bs)], dtype=np.uint64)[:, None]
    y = x[..., T:, :] % bc * tw % bc
    v = np.rint((y.astype(np.float64) / bc.astype(np.float64)).sum(axis=-2)).astype(np.uint64)
    out = np.empty(x.shape[:-2] + (T, x.shape[-1]), dtype=np.uint64)
    for j, c in enumerate(k.cs):
        c64 = np.uint64(c)
        acc = np.zeros_like(v)
        for i in range(len(k.bs)):
            acc = (acc + y[..., i, :] * np.uint64(k.m[j][i])) % c64
        acc = (acc + c64 - v * np.uint64(k.B % c) % c64) % c64
        tx = x[..., j, :] * np.uint64(t % c) % c64
        out[..., j, :] = (tx + c64 - acc) % c64 * np.uint64(k.binv[j]) % c64
    return out


def shape_of(logn, S, T, batch, rows):
    n = 1 << logn
    return n, (L2_WORDS // (rows * n) if batch == "l2" else batch)


# -------------------------------------------------------------------- convert(exact=True)
@pytest.mark.gpu
@pytest.mark.parametrize("logn,S,T,batch", CONVERT_CASES)
def test_convert_exact(lib, logn, S, T, batch):
    """Against numpy on every (above L2: sampled) polynomial and against the Python-int centred
    CRT on sampled columns; the fast result differs by alpha B or (alpha + 1) B."""
    torch = _torch()
    n, batch = shape_of(logn, S, T, batch, S)
    bs, cs = split_primes(S, T)
    k = Consts(bs, cs)
    seed = 71000 + 100 * logn + S * 33 + T
    x = rand_rns((batch, S, n), bs, seed)
    out = torch.empty((batch, T, n), dtype=torch.int32, device="cuda")
    fast = torch.empty_like(out)
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        cv.convert(x, out, batch, exact=True)
        cv.convert(x, fast, batch)
    rows = rows_of(batch, seed)
    hx, got, hf = host(x, rows), host(out, rows), host(fast, rows)
    assert np.array_equal(got, exact_ref(hx, k))
    for c in sample_cols(n, seed, 8):
        xv = crt(hx[-1, :, c], bs)
        assert [int(v) for v in got[-1, :, c]] == [centred(xv, k.B) % cj for cj in cs], c
        _, alpha = overshoot(xv, k)
        for j, cj in enumerate(cs):
            d = (int(hf[-1, j, c]) - int(got[-1, j, c])) % cj
            assert d in (alpha * k.B % cj, (alpha + 1) * k.B % cj), (c, j)


@pytest.mark.gpu
@pytest.mark.parametrize("S,T", [(1, 31), (8, 8), (16, 4), (17, 3), (32, 32)])
def test_convert_exact_special_values(lib, S, T):
    """x = 0, +-1, +-small, B (1/2 -+ 2^-40) and every y_i = b_i - 1 are exact; x = B/2 + d for
    small d lies within 2^-40 of 1/2 (for S > 1), where either representative may come back."""
    torch = _torch()
    logn = 12
    n = 1 << logn
    bs, cs = split_primes(S, T)
    k = Consts(bs, cs)
    lo, hi = (k.B * ((1 << 39) - 1)) >> 40, -((-k.B * ((1 << 39) + 1)) >> 40)
    vals = [0, 1, -1, 2, -2, 12345, -12345, (1 << 40) + 3, -(1 << 40) - 3, lo, lo - 1, hi, hi + 1,
            crt([(-(k.B // b)) % b for b in bs], bs)]
    vals += [k.B // 2 + d for d in (-(1 << 20), -1, 0, 1, 2, 1 << 20)]
    rng = random.Random(S * 100 + T)
    xs = (vals + [rng.randrange(k.B) for _ in range(n)])[:n]
    x = to_dev(residues(xs, bs)[None])
    out = torch.empty((1, T, n), dtype=torch.int32, device="cuda")
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        cv.convert(x, out, 1, exact=True)
    got = host(out)[0]
    band = 0
    for col, v in enumerate(xs):
        xc = centred(v, k.B)
        g = [int(r) for r in got[:, col]]
        if abs(Fraction(v % k.B, k.B) - Fraction(1, 2)) < Fraction(1, 1 << 40):
            band += 1
            other = xc - k.B if xc > 0 else xc + k.B
            assert g in ([xc % c for c in cs], [other % c for c in cs]), col
        else:
            assert g == [xc % c for c in cs], col
    assert band == (6 if S > 1 else 0)


@pytest.mark.gpu
def test_convert_exact_strided_pq(lib):
    """Q -> P into the P rows of a [batch][P | Q] buffer with equal strides (no copy), and a
    middle digit of a ciphertext into a separate buffer; every other word untouched."""
    torch = _torch()
    logn, batch, Lq, K = 12, 3, 6, 4
    n = 1 << logn
    qs, ps = split_primes(Lq, K)
    ct = rand_rns((batch, Lq, n), qs, 72000)
    hct = host(ct)
    with ones_plan(lib, logn, qs) as pq, ones_plan(lib, logn, ps) as pp, ones_plan(lib, logn, qs[2:4]) as pd:
        buf = Guarded(batch * (K + Lq) * n)
        bv = buf.view.view(batch, K + Lq, n)
        bv[:, K:] = ct
        with lib.RnsConv(pq, pp) as cv:
            cv.convert(buf.view[K * n:], buf.view, batch, in_stride=(K + Lq) * n, out_stride=(K + Lq) * n, exact=True)
        assert np.array_equal(host(bv[:, :K]), exact_ref(hct, Consts(qs, ps)))
        assert torch.equal(bv[:, K:], ct) and buf.guards_intact()
        dst = Guarded(batch * (K + Lq) * n)
        with lib.RnsConv(pd, pp) as cv:
            cv.convert(ct[:, 2:], dst.view, batch, in_stride=Lq * n, out_stride=(K + Lq) * n, exact=True)
        dv = dst.view.view(batch, K + Lq, n)
        assert np.array_equal(host(dv[:, :K]), exact_ref(hct[:, 2:4], Consts(qs[2:4], ps)))
        assert bool((dv[:, K:] == SENTINEL).all()) and dst.guards_intact()


# --------------------------------------------------------------------------- scale_round
@pytest.mark.gpu
@pytest.mark.parametrize("logn,S,T,batch", CONVERT_CASES)
def test_scale_round(lib, logn, S, T, batch):
    """round(t X / B) mod c_j for every t of T_VALUES: numpy on every (sampled) polynomial,
    Python ints on sampled columns."""
    torch = _torch()
    n, batch = shape_of(logn, S, T, batch, S + T)
    bs, cs = split_primes(S, T)
    k = Consts(bs, cs)
    seed = 73000 + 100 * logn + S * 33 + T
    x = rand_rns((batch, T + S, n), cs + bs, seed)
    out = torch.empty((batch, T, n), dtype=torch.int32, device="cuda")
    rows = rows_of(batch, seed)
    hx = host(x, rows)
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        for t in T_VALUES:
            cv.scale_round(x, out, batch, t)
            got = host(out, rows)
            assert np.array_equal(got, scale_round_ref(hx, k, t)), t
            for c in sample_cols(n, seed + t, 6):
                X = crt(hx[-1, :, c], cs + bs)
                want = (2 * t * X + k.B) // (2 * k.B)
                assert [int(v) for v in got[-1, :, c]] == [want % cj for cj in cs], (t, c)
    assert np.array_equal(host(x, rows), hx)


@pytest.mark.gpu
@pytest.mark.parametrize("logn,T", [(12, 31), (16, 5), (13, 1)])
def test_scale_round_t1_s1_equals_mod_down(lib, logn, T):
    """t = 1, S = 1 (an odd prime): bit for bit the result of mod_down(ROUND), on every column."""
    torch = _torch()
    n, batch = 1 << logn, 3
    cs, bs = split_primes(T, 1)
    x = rand_rns((batch, T + 1, n), cs + bs, 74000 + logn)
    a = torch.empty((batch, T, n), dtype=torch.int32, device="cuda")
    b = torch.empty_like(a)
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        cv.scale_round(x, a, batch, 1)
        cv.mod_down(x, b, batch, round=True)
    assert torch.equal(a, b)


@pytest.mark.gpu
def test_scale_round_centred_and_multi_prime_rescale(lib):
    """A centred X (X < 0 stored as X + CB) gives round(t X / B) too; t = 1 with S = 3 is the
    exact rounded division by three primes at once."""
    torch = _torch()
    logn, S, T = 12, 3, 4
    n = 1 << logn
    cs, bs = split_primes(T, S)
    B, C = math.prod(bs), math.prod(cs)
    rng = random.Random(75000)
    xs = [rng.randrange(-(C * B) // 2, (C * B) // 2) for _ in range(n)]
    # t X / B stays about 1/6 or more from a half-integer for these (the band is 2^-40 wide)
    xs[:6] = [0, -1, 1, -(B // 4), B // 3, -(C * B) // 3]
    x = to_dev(residues(xs, cs + bs)[None])
    out = torch.empty((1, T, n), dtype=torch.int32, device="cuda")
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        for t in (1, 65537):
            cv.scale_round(x, out, 1, t)
            want = residues([(2 * t * v + B) // (2 * B) for v in xs], cs)
            assert np.array_equal(host(out)[0], want), t


# ------------------------------------------------------------------------ buffer rules
@pytest.mark.gpu
def test_buffer_rules(lib):
    """Unaligned -> UNSUPPORTED, overlaps and t == 0 -> INVALID_ARG (t == 0 also at batch 0), nothing
    written and nothing launched; batch == 0 launches nothing."""
    torch = _torch()
    logn, batch, S, T = 12, 2, 3, 2
    n = 1 << logn
    bs, cs = split_primes(S, T)
    k = Consts(bs, cs)
    x = rand_rns((batch, T + S, n), cs + bs, 76000)
    hx = host(x)
    row = (T + S) * n
    L = lib.load_library()
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        before = lib.kernel_launches()
        for kk in (1, 2, 3):
            for ki, ko in ((kk, 0), (0, kk)):
                gi, go = Guarded(batch * row, ki, x), Guarded(batch * T * n, ko)
                snap = gi.raw.clone()
                calls = [lambda: cv.convert(gi.view[T * n:], go.view, batch, in_stride=row, exact=True),
                         lambda: cv.scale_round(gi.view, go.view, batch, 65537)]
                for i, call in enumerate(calls):
                    assert _status(lib, call) == UNSUPPORTED, (kk, ki, ko, i)
                torch.cuda.synchronize()
                assert go.untouched() and torch.equal(gi.raw, snap)
        big = Guarded(4 * row, 0, torch.cat([x.reshape(-1), x.reshape(-1)]))
        snap = big.raw.clone()
        v = big.view
        bad = [lambda: cv.scale_round(v, v, batch, 3),
               lambda: cv.scale_round(v, v[row + T * n:], batch, 3),
               lambda: cv.scale_round(v[T * n:], v[n:], 1, 3),
               lambda: cv.scale_round(x, big.view, batch, 0),
               lambda: cv.convert(v, v[(S - 1) * n:], batch, in_stride=row, out_stride=row, exact=True),
               lambda: cv.convert(v[row:], v, batch, in_stride=row, out_stride=row, exact=True),
               lambda: cv.convert(v, v[S * n:], batch, in_stride=2 * row, out_stride=row, exact=True),
               lambda: cv.convert(v, big.view, batch, in_stride=S * n - n, exact=True)]
        for i, call in enumerate(bad):
            assert _status(lib, call) == INVALID_ARG, i
        assert L.nttb200_rns_scale_round(cv._h, None, None, 0, 0, None) == INVALID_ARG
        assert L.nttb200_rns_scale_round(cv._h, x.data_ptr(), None, batch, 3, None) == INVALID_ARG
        assert L.nttb200_rns_base_convert_exact(cv._h, None, 0, big.view.data_ptr(), 0, batch, None) == INVALID_ARG
        torch.cuda.synchronize()
        assert torch.equal(big.raw, snap)
        assert L.nttb200_rns_scale_round(cv._h, None, None, 0, 3, None) == OK
        assert L.nttb200_rns_base_convert_exact(cv._h, None, 0, None, 0, 0, None) == OK
        cv.convert(x, x, 0, exact=True)
        cv.scale_round(x, x, 0, 5)
        assert lib.kernel_launches() == before
        out = Guarded(batch * T * n)
        cv.scale_round(x, out.view, batch, 65537)
        assert np.array_equal(host(out.view.view(batch, T, n)), scale_round_ref(hx, k, 65537)) and out.guards_intact()
        cv.convert(x[:, T:], out.view, batch, in_stride=row, exact=True)
        assert np.array_equal(host(out.view.view(batch, T, n)), exact_ref(hx[:, T:], k)) and out.guards_intact()
    assert np.array_equal(host(x), hx)


@pytest.mark.gpu
def test_beyond_2_31_words(lib):
    """One call over 2^31 + 2^16 words each way (S = T = 1, N = 2^16, batch 2^15 + 1): the exact
    conversion from channel 1 of a [batch][2][N] buffer into its channel 0, then scale_round of that
    buffer; checked on sampled polynomials including the last."""
    torch = _torch()
    logn, batch = 16, (1 << 15) + 1
    n = 1 << logn
    cs, bs = split_primes(1, 1)
    k = Consts(bs, cs)
    gen = torch.Generator(device="cuda").manual_seed(77000)
    x = torch.randint(0, min(bs[0], cs[0]), (batch, 2, n), dtype=torch.int32, device="cuda", generator=gen)
    rows = np.array([0, 1, batch // 2, batch - 2, batch - 1])
    src = host(x[:, 1], rows)[:, None]
    out = torch.empty((batch, 1, n), dtype=torch.int32, device="cuda")
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        cv.convert(x[:, 1], x, batch, in_stride=2 * n, out_stride=2 * n, exact=True)
        assert np.array_equal(host(x[:, :1], rows), exact_ref(src, k))
        cv.scale_round(x, out, batch, 65537)
    assert np.array_equal(host(out, rows), scale_round_ref(host(x, rows), k, 65537))


# ------------------------------------------------------------------------ end-to-end BFV
def negacyclic_small(a, b, n):
    """a * b mod (X^N + 1) over the integers for int64 operands whose products and sums fit."""
    full = np.convolve(a, b)
    out = full[:n].copy()
    out[:n - 1] -= full[n:]
    return out


W = 256   # Kronecker slot width in bits: |coefficients of a product| < 2^(W-1)


def kron(poly):
    """sum_i poly[i] 2^(W i) for signed coefficients: the positive and the negative parts packed
    through bytes, then one subtraction."""
    def pack(vals):
        return int.from_bytes(b"".join(v.to_bytes(W // 8, "little") for v in vals), "little")
    return pack([max(v, 0) for v in poly]) - pack([max(-v, 0) for v in poly])


def negacyclic_big(a, b, n):
    """Exact a * b mod (X^N + 1) for Python-int coefficient lists (any sign): one big-integer
    product by Kronecker substitution, slots read back with an offset that makes them positive."""
    prod = kron(a) * kron(b)
    off = sum(1 << (W * i + W - 1) for i in range(2 * n))
    raw = (prod + off).to_bytes(2 * n * W // 8 + 1, "little")
    step = W // 8
    coef = [int.from_bytes(raw[i * step:(i + 1) * step], "little") - (1 << (W - 1)) for i in range(2 * n)]
    return [coef[i] - coef[i + n] for i in range(n)]


def bfv_setup(n, t, qs, seed):
    """Host-built secret and two encryptions: c = (-a s + e + floor(Q/t) m, a) mod Q, residues [2][L][N]."""
    rng = np.random.default_rng(seed)
    Q = math.prod(qs)
    delta = Q // t
    s = rng.integers(-1, 2, n).astype(np.int64)
    ms, cts = [], []
    for _ in range(2):
        m = rng.integers(0, t, n).astype(np.int64)
        e = rng.integers(-4, 5, n).astype(np.int64)
        a = np.stack([rng.integers(0, q, n) for q in qs]).astype(np.int64)
        c0 = np.stack([(-negacyclic_small(a[l], s, n) + e + (delta % q) * m % q) % q for l, q in enumerate(qs)])
        ms.append(m)
        cts.append(np.stack([c0, a]))
    return s, ms, cts


def bfv_mul_ref(c, cp, qs, t, n):
    """round(t/Q * (c (x) c')) mod Q with centred lifts of c and c', residues [3][L][N]."""
    Q = math.prod(qs)

    def lift(res):
        return [centred(crt([int(res[l][i]) for l in range(len(qs))], qs), Q) for i in range(n)]

    a0, a1, b0, b1 = lift(c[0]), lift(c[1]), lift(cp[0]), lift(cp[1])
    d1 = [u + v for u, v in zip(negacyclic_big(a0, b1, n), negacyclic_big(a1, b0, n))]
    out = []
    for d in (negacyclic_big(a0, b0, n), d1, negacyclic_big(a1, b1, n)):
        out.append(residues([(2 * t * v + Q) // (2 * Q) for v in d], qs))
    return np.stack(out)


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 14])
@pytest.mark.parametrize("t", [65537, 1 << 16])
def test_bfv_multiply_and_decrypt(lib, logn, t):
    """BFV: the INTEGRATION multiplication sequence on a [P | Q] plan (convert exact Q -> P, ct,
    tensor product, gs_scaled, scale_round Q -> P, convert exact P -> Q) bit-identical to the
    big-integer reference, and the 3-component result decrypted on the GPU (rns_scale by t, convert
    exact Q -> {t}, rns_scale by -Q^-1 mod t) to m1 m2 mod (X^N + 1, t)."""
    torch = _torch()
    n, Lq = 1 << logn, 4
    K = Lq + 2
    qs, ps = split_primes(Lq, K)
    Q = math.prod(qs)
    s, (m1, m2), (c, cp) = bfv_setup(n, t, qs, 78000 + logn + t)
    want = bfv_mul_ref(c, cp, qs, t, n)
    fwd, inv, _ = channel_tables(lib, n, ps + qs)
    qfwd, qinv = fwd[K:], inv[K:]
    qp = torch.empty((2, K + Lq, n), dtype=torch.int32, device="cuda")
    A, Bt = torch.empty_like(qp), torch.empty_like(qp)
    d = torch.empty((3, K + Lq, n), dtype=torch.int32, device="cuda")
    dp = torch.empty((3, K, n), dtype=torch.int32, device="cuda")
    res = torch.empty((3, Lq, n), dtype=torch.int32, device="cuda")
    with lib.RnsPlan(ps + qs, fwd, logn=logn) as pf, lib.RnsPlan(ps + qs, inv, logn=logn) as pi, \
            ones_plan(lib, logn, qs) as pq, ones_plan(lib, logn, ps) as pp, \
            lib.RnsConv(pq, pp) as up, lib.RnsConv(pp, pq) as back:
        for ev, ct in ((A, c), (Bt, cp)):
            qp[:, K:] = to_dev(ct)                                                     # 1
            up.convert(qp[:, K:], qp, 2, in_stride=(K + Lq) * n, out_stride=(K + Lq) * n, exact=True)  # 2
            pf.ct(qp, ev, 2)                                                           # 3
        pf.pointwise(lib.RNS_MUL, A[0], Bt[0], d[0], 1)                                # 4
        pf.pointwise(lib.RNS_MUL, A[0], Bt[1], d[1], 1)
        lib.rns_dot(pf, A[1], Bt[0], d[1], 1, 1, accumulate=True)
        pf.pointwise(lib.RNS_MUL, A[1], Bt[1], d[2], 1)
        pi.gs_scaled(d, d, 3)                                                          # 5
        up.scale_round(d, dp, 3, t)                                                    # 6
        back.convert(dp, res, 3, exact=True)                                           # 7
    assert np.array_equal(host(res), want)

    # decryption on the GPU: X = d0 + d1 s + d2 s^2 mod Q, then round(t X / Q) mod t
    s_res = to_dev(residues([int(v) for v in s], qs)[None])
    ev = torch.empty_like(res)
    se = torch.empty_like(s_res)
    s2 = torch.empty_like(s_res)
    x = torch.empty_like(s_res)
    mt = torch.empty((1, 1, n), dtype=torch.int32, device="cuda")
    with lib.RnsPlan(qs, qfwd, logn=logn) as qf, lib.RnsPlan(qs, qinv, logn=logn) as qi, \
            ones_plan(lib, logn, qs) as pq, ones_plan(lib, logn, [t]) as ptt, lib.RnsConv(pq, ptt) as to_t:
        qf.ct(res, ev, 3)
        qf.ct(s_res, se, 1)
        qf.pointwise(lib.RNS_MUL, se, se, s2, 1)
        qf.pointwise(lib.RNS_MUL, ev[1], se, x, 1)
        qf.pointwise(lib.RNS_ADD, x, ev[0], x, 1)
        qf.pointwise(lib.RNS_MUL, ev[2], s2, s2, 1)
        qf.pointwise(lib.RNS_ADD, x, s2, x, 1)
        qi.gs_scaled(x, x, 1)
        qf.scale(x, x, 1, [t % q for q in qs])
        to_t.convert(x, mt, 1, exact=True)
        ptt.scale(mt, mt, 1, [(-pow(Q, -1, t)) % t])
    prod = negacyclic_small(m1, m2, n) % t
    assert np.array_equal(host(mt)[0, 0].astype(np.int64), prod)
