"""Basis conversion between the primes of two RNS plans (coefficient domain): nttb200_rns_conv_create,
nttb200_rns_base_convert (fast base conversion, ModUp) and nttb200_rns_mod_down (division by B with
or without rounding: rescale, modulus drop, ModDown).  Results against numpy residues in uint64 with
the constants computed here from Python ints, and the integer-level contracts (the alpha bound,
floor / round of X / B) against exact CRT on sampled columns.  Guard bands check that nothing is
stored outside the written rows.  The null-conv argument checks run without a device."""
import ctypes
import math

import numpy as np
import pytest

from test_rns_eval import SENTINEL, Guarded, _status, channel_tables, host, ones_plan, rand_rns, rows_of
from test_rns_sizes import ntt_primes

OK, INVALID_ARG, MODULUS, UNSUPPORTED = 0, 1, 2, 7
ROUND = 1
L2_WORDS = 1 << 26   # 256 MiB per operand: twice the B200's L2


# ------------------------------------------------------------------ CPU: argument checks
def test_null_arguments_without_device(lib):
    L = lib.load_library()
    h = ctypes.c_void_p()
    assert L.nttb200_rns_conv_create(None, None, None, 0) == INVALID_ARG
    assert L.nttb200_rns_conv_create(ctypes.byref(h), None, None, 0) == INVALID_ARG and h.value is None
    assert L.nttb200_rns_conv_create(ctypes.byref(h), None, None, 1) == INVALID_ARG
    assert L.nttb200_rns_conv_destroy(None) == OK
    assert L.nttb200_rns_base_convert(None, 16, 0, 16, 0, 1, None) == INVALID_ARG
    assert L.nttb200_rns_base_convert(None, None, 0, None, 0, 0, None) == INVALID_ARG
    assert L.nttb200_rns_base_convert(None, 16, 3, 16, 5, 1, None) == INVALID_ARG
    assert L.nttb200_rns_mod_down(None, 16, 16, 1, ROUND, None) == INVALID_ARG
    assert L.nttb200_rns_mod_down(None, None, None, 0, 0, None) == INVALID_ARG
    assert L.nttb200_rns_mod_down(None, 16, 16, 1, 2, None) == INVALID_ARG
    assert lib.RNS_ROUND == ROUND


# ---------------------------------------------------------------- host constants, oracle
def split_primes(*counts):
    """Disjoint lists of NTT-friendly primes below 2^30 (2^17 | q - 1)."""
    qs = ntt_primes(sum(counts))
    out, at = [], 0
    for k in counts:
        out.append(qs[at:at + k])
        at += k
    return out


class Consts:
    def __init__(self, bs, cs):
        self.bs, self.cs = list(bs), list(cs)
        self.B, self.C = math.prod(bs), math.prod(cs)
        self.w = [pow(self.B // b % b, -1, b) for b in bs]            # (B/b_i)^-1 mod b_i
        self.m = [[self.B // b % c for b in bs] for c in cs]          # (B/b_i) mod c_j
        self.binv = [pow(self.B % c, -1, c) for c in cs]
        self.h = self.B // 2


def col(vals):
    return np.array(vals, dtype=np.uint64)[:, None]


def convert_ref(x, k, h=0):
    """x: uint64 [..., S, N] -> [..., T, N]; h: the offset added to the source value first."""
    bc = col(k.bs)
    y = (x + col([h % b for b in k.bs])) % bc * col(k.w) % bc
    out = np.empty(x.shape[:-2] + (len(k.cs), x.shape[-1]), dtype=np.uint64)
    for j, c in enumerate(k.cs):
        acc = np.zeros(x.shape[:-2] + x.shape[-1:], dtype=np.uint64)
        for i in range(len(k.bs)):
            acc = (acc + y[..., i, :] * np.uint64(k.m[j][i])) % np.uint64(c)
        out[..., j, :] = acc
    return out


def mod_down_ref(x, k, rnd):
    """x: uint64 [..., T+S, N] (target channels first) -> [..., T, N]."""
    t = len(k.cs)
    h = k.h if rnd else 0
    cc = col(k.cs)
    s = convert_ref(x[..., t:, :], k, h)
    v = (x[..., :t, :] + col([h % c for c in k.cs])) % cc
    return (v + cc - s) % cc * col(k.binv) % cc


def crt(res, mods):
    M = math.prod(mods)
    return sum(int(r) * (M // m) * pow(M // m % m, -1, m) for r, m in zip(res, mods)) % M


def overshoot(x, k):
    """(sum_i y_i B/b_i, alpha) of the fast conversion of x in [0, B)."""
    total = sum((x % b) * w % b * (k.B // b) for b, w in zip(k.bs, k.w))
    assert (total - x) % k.B == 0
    return total, (total - x) // k.B


def sample_cols(n, seed, count=24):
    rng = np.random.default_rng(seed)
    return np.unique(np.concatenate([[0, 1, n - 1], rng.integers(0, n, count)]))


def residues(values, mods):
    """Python ints -> uint64 [len(mods), len(values)]."""
    return np.array([[v % m for v in values] for m in mods], dtype=np.uint64)


def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"
    return torch


def to_dev(a):
    torch = _torch()
    return torch.from_numpy(np.ascontiguousarray(a).astype(np.int32)).cuda()


# ------------------------------------------------------------------------- base_convert
CONVERT_CASES = [(12, 1, 31, 3), (12, 4, 28, 2), (12, 16, 3, 5), (12, 17, 3, 5), (12, 32, 32, 2),
                 (12, 31, 1, 3), (16, 1, 1, 2), (16, 8, 32, 1), (16, 17, 16, 2), (12, 8, 8, "l2")]


@pytest.mark.gpu
@pytest.mark.parametrize("logn,S,T,batch", CONVERT_CASES)
def test_convert(lib, logn, S, T, batch):
    """Against numpy on every (or, above L2, on sampled) polynomials; the integer contract
    sum y_i B/b_i = x + alpha B, 0 <= alpha < S, with exact CRT on sampled columns."""
    torch = _torch()
    n = 1 << logn
    if batch == "l2":
        batch = L2_WORDS // (S * n)
    bs, cs = split_primes(S, T)
    k = Consts(bs, cs)
    seed = 91000 + 100 * logn + S * 33 + T
    x = rand_rns((batch, S, n), bs, seed)
    out = torch.empty((batch, T, n), dtype=torch.int32, device="cuda")
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        cv.convert(x, out, batch)
    rows = rows_of(batch, seed)
    hx, got = host(x, rows), host(out, rows)
    assert np.array_equal(got, convert_ref(hx, k))
    for c in sample_cols(n, seed, 8):
        xv = crt(hx[0, :, c], bs)
        total, alpha = overshoot(xv, k)
        assert 0 <= alpha < S
        assert [int(v) for v in got[0, :, c]] == [total % cj for cj in cs]


@pytest.mark.gpu
@pytest.mark.parametrize("S,T", [(16, 4), (17, 4), (32, 32)])
def test_convert_alpha_worst_case(lib, S, T):
    """Every y_i = b_i - 1 (x_i = -(B/b_i) mod b_i): the largest terms the 64-bit sum sees, and
    the largest overshoot; out_j = (x + alpha B) mod c_j with 0 <= alpha < S."""
    torch = _torch()
    logn, batch = 12, 2
    n = 1 << logn
    bs, cs = split_primes(S, T)
    k = Consts(bs, cs)
    xi = [(-(k.B // b)) % b for b in bs]
    x = torch.tensor(xi, dtype=torch.int32, device="cuda").view(1, S, 1).repeat(batch, 1, n)
    x[1, :, n // 2:] = rand_rns((1, S, n // 2), bs, 92000 + S)[0]
    out = torch.empty((batch, T, n), dtype=torch.int32, device="cuda")
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        cv.convert(x, out, batch)
    hx, got = host(x), host(out)
    assert np.array_equal(got, convert_ref(hx, k))
    xv = crt(xi, bs)
    total, alpha = overshoot(xv, k)
    assert total == sum((b - 1) * (k.B // b) for b in bs) and 0 <= alpha < S
    assert [int(v) for v in got[0, :, 0]] == [(xv + alpha * k.B) % cj for cj in cs]


@pytest.mark.gpu
def test_convert_strided(lib):
    """Different strides: a middle digit of a [batch][L][N] ciphertext into the P channels of a
    separate [batch][L+K][N] buffer.  Equal strides: the Q channels of a [batch][L+K][N] buffer
    into its own P channels (interleaved rows).  Every other word stays as it was."""
    torch = _torch()
    logn, batch, Lq, K = 12, 3, 6, 3
    n = 1 << logn
    qs, ps = split_primes(Lq, K)
    ct = rand_rns((batch, Lq, n), qs, 93000)
    hct = host(ct)
    with ones_plan(lib, logn, qs[2:4]) as pd, ones_plan(lib, logn, qs) as pq, ones_plan(lib, logn, ps) as pp:
        # a digit (channels 2, 3) -> P channels of a separate QP buffer
        src = Guarded(batch * Lq * n, 0, ct)
        dst = Guarded(batch * (Lq + K) * n)
        with lib.RnsConv(pd, pp) as cv:
            cv.convert(src.view[2 * n:], dst.view[Lq * n:], batch, in_stride=Lq * n, out_stride=(Lq + K) * n)
        want = convert_ref(hct[:, 2:4], Consts(qs[2:4], ps))
        got = dst.view.view(batch, Lq + K, n)
        assert np.array_equal(host(got[:, Lq:]), want)
        assert bool((got[:, :Lq] == SENTINEL).all()) and dst.guards_intact()
        assert torch.equal(src.view, ct.reshape(-1)) and src.guards_intact()
        # Q channels -> P channels of the same buffer
        qp = Guarded(batch * (Lq + K) * n)
        qpv = qp.view.view(batch, Lq + K, n)
        qpv[:, :Lq] = ct
        with lib.RnsConv(pq, pp) as cv:
            cv.convert(qp.view, qp.view[Lq * n:], batch, in_stride=(Lq + K) * n, out_stride=(Lq + K) * n)
        assert np.array_equal(host(qpv[:, Lq:]), convert_ref(hct, Consts(qs, ps)))
        assert torch.equal(qpv[:, :Lq], ct) and qp.guards_intact()


# ----------------------------------------------------------------------------- mod_down
@pytest.mark.gpu
@pytest.mark.parametrize("logn,S,T,batch", [(12, 1, 31, 3), (12, 8, 24, 2), (16, 3, 5, 2), (12, 17, 2, 2)])
def test_mod_down(lib, logn, S, T, batch):
    """With and without ROUND against the formula (numpy) and the contract
    out = (floor(X'/B) - alpha) mod c_j, X' = (X + h) mod CB, on sampled columns."""
    torch = _torch()
    n = 1 << logn
    bs, cs = split_primes(S, T)
    k = Consts(bs, cs)
    seed = 94000 + 100 * logn + S
    x = rand_rns((batch, T + S, n), cs + bs, seed)
    hx = host(x)
    out = torch.empty((batch, T, n), dtype=torch.int32, device="cuda")
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        for rnd in (False, True):
            cv.mod_down(x, out, batch, round=rnd)
            got = host(out)
            assert np.array_equal(got, mod_down_ref(hx, k, rnd)), rnd
            h = k.h if rnd else 0
            for c in sample_cols(n, seed, 8):
                X = (crt(hx[1, :, c], cs + bs) + h) % (k.C * k.B)
                _, alpha = overshoot(X % k.B, k)
                assert 0 <= alpha < S
                assert [int(v) for v in got[1, :, c]] == [(X // k.B - alpha) % cj for cj in cs], (rnd, c)
    assert np.array_equal(host(x), hx)


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 16])
def test_rescale_exact(lib, logn):
    """S = 1 is exact: ROUND gives round(X / q) for X in [0, CB - floor(B/2)), without it
    floor(X / q); X at 0, at the top of the range and random, as Python ints."""
    torch = _torch()
    n, batch, T = 1 << logn, 2, 5
    cs, bs = split_primes(T, 1)
    B, C = bs[0], math.prod(cs)
    top = C * B - B // 2
    rng = np.random.default_rng(95000 + logn)
    xs = [int.from_bytes(rng.bytes(24), "little") % top for _ in range(batch * n)]
    xs[:6] = [0, 1, B // 2, B // 2 + 1, top - 1, top - 2]
    xs[n:n + 3] = [top - 1 - B, C * B - 1 - B // 2, B - 1]
    res = residues(xs, cs + bs).reshape(T + 1, batch, n).transpose(1, 0, 2)
    x = to_dev(res)
    out = torch.empty((batch, T, n), dtype=torch.int32, device="cuda")
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        for rnd in (True, False):
            cv.mod_down(x, out, batch, round=rnd)
            want = [(2 * v + B) // (2 * B) if rnd else v // B for v in xs]
            assert np.array_equal(host(out), residues(want, cs).reshape(T, batch, n).transpose(1, 0, 2)), rnd


@pytest.mark.gpu
def test_mod_up_mod_down_identity(lib):
    """x on Q, converted to P straight into the P channels of a [batch][L+K][N] buffer, x in its
    Q channels, rns_scale by (P mod q_l on Q, 0 on P): the value is P x, and mod_down by P
    without ROUND returns x bit for bit."""
    torch = _torch()
    logn, batch, Lq, K = 13, 3, 5, 3
    n = 1 << logn
    qs, ps = split_primes(Lq, K)
    P = math.prod(ps)
    x = rand_rns((batch, Lq, n), qs, 96000)
    qp = torch.empty((batch, Lq + K, n), dtype=torch.int32, device="cuda")
    out = torch.empty_like(x)
    with ones_plan(lib, logn, qs) as pq, ones_plan(lib, logn, ps) as pp, ones_plan(lib, logn, qs + ps) as pqp:
        with lib.RnsConv(pq, pp) as up, lib.RnsConv(pp, pq) as down:
            up.convert(x, qp[:, Lq:], batch, out_stride=(Lq + K) * n)
            assert np.array_equal(host(qp[:, Lq:]), convert_ref(host(x), Consts(qs, ps)))
            qp[:, :Lq] = x
            pqp.scale(qp, qp, batch, [P % q for q in qs] + [0] * K)
            down.mod_down(qp, out, batch)
    assert torch.equal(out, x)


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 16])
def test_ntt_domain_rescale(lib, logn):
    """ct_L(X) -> gs_scaled_L -> mod_down(ROUND) -> ct_(L-1) equals ct_(L-1) of round(X / q_(L-1)),
    computed on the host with Python ints."""
    torch = _torch()
    n, batch, Lq = 1 << logn, 2, 5
    qs = ntt_primes(Lq)
    Q, ql = math.prod(qs), qs[-1]
    rng = np.random.default_rng(97000 + logn)
    xs = [int.from_bytes(rng.bytes(20), "little") % (Q - ql // 2) for _ in range(batch * n)]
    xs[:2] = [0, Q - ql // 2 - 1]
    want = [(2 * v + ql) // (2 * ql) for v in xs]
    x = to_dev(residues(xs, qs).reshape(Lq, batch, n).transpose(1, 0, 2))
    e = to_dev(residues(want, qs[:-1]).reshape(Lq - 1, batch, n).transpose(1, 0, 2))
    fwd, inv, _ = channel_tables(lib, n, qs)
    ev, low, got, exp = torch.empty_like(x), torch.empty_like(e), torch.empty_like(e), torch.empty_like(e)
    with lib.RnsPlan(qs, fwd, logn=logn) as pf, lib.RnsPlan(qs, inv, logn=logn) as pi, \
            lib.RnsPlan(qs[:-1], fwd[:-1], logn=logn) as pf1, ones_plan(lib, logn, qs[-1:]) as plast, \
            lib.RnsConv(plast, pf1) as cv:
        pf.ct(x, ev, batch)                 # the ciphertext in the NTT domain
        pi.gs_scaled(ev, ev, batch)
        cv.mod_down(ev, low, batch, round=True)
        pf1.ct(low, got, batch)
        pf1.ct(e, exp, batch)
    assert torch.equal(low, e) and torch.equal(got, exp)


# ------------------------------------------------------------------------ documented errors
@pytest.mark.gpu
def test_create_errors(lib):
    logn = 12
    (a, b, c) = split_primes(2, 2, 2)
    L = lib.load_library()
    h = ctypes.c_void_p()
    with ones_plan(lib, logn, a) as pa, ones_plan(lib, logn, b) as pb, ones_plan(lib, logn, [b[0]] + c) as pbc, \
            ones_plan(lib, 13, c) as p13, ones_plan(lib, logn, [1 << 20]) as peven, \
            ones_plan(lib, logn, [3 * 5, 7 * 11]) as pcomp, ones_plan(lib, logn, [5 * 13]) as pshare:
        for src, dst, status in ((pa, pbc, OK), (pb, pbc, MODULUS), (pa, pa, MODULUS), (pa, p13, INVALID_ARG),
                                 (peven, pa, OK), (pcomp, pa, OK), (pcomp, pshare, MODULUS)):
            rc = L.nttb200_rns_conv_create(ctypes.byref(h), src._h, dst._h, 0)
            assert rc == status, (src.qs, dst.qs)
            assert (h.value is not None) == (status == OK)
            L.nttb200_rns_conv_destroy(h)
        assert L.nttb200_rns_conv_create(ctypes.byref(h), pa._h, pb._h, 1) == INVALID_ARG
        assert L.nttb200_rns_conv_create(ctypes.byref(h), pa._h, None, 0) == INVALID_ARG
        assert _status(lib, lambda: lib.RnsConv(pb, pbc)) == MODULUS


@pytest.mark.gpu
def test_composite_and_even_moduli(lib):
    """The moduli need not be prime, and floor(B/2) is right with an even modulus in B."""
    torch = _torch()
    logn, batch = 12, 2
    n = 1 << logn
    bs, cs = [1 << 20, 3 * 5 * 7 * 11 * 13 * 17], ntt_primes(3)
    k = Consts(bs, cs)
    x = rand_rns((batch, 3 + 2, n), cs + bs, 98000)
    out = torch.empty((batch, 3, n), dtype=torch.int32, device="cuda")
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        cv.convert(x[:, 3:], out, batch, in_stride=5 * n)
        assert np.array_equal(host(out), convert_ref(host(x[:, 3:]), k))
        for rnd in (False, True):
            cv.mod_down(x, out, batch, round=rnd)
            assert np.array_equal(host(out), mod_down_ref(host(x), k, rnd)), rnd


@pytest.mark.gpu
def test_buffer_rules(lib):
    """Unaligned views -> UNSUPPORTED, overlaps -> INVALID_ARG, bad strides and flags ->
    INVALID_ARG, nothing written and nothing launched; batch == 0 launches nothing; the conv
    works after both plans are destroyed."""
    torch = _torch()
    logn, batch, S, T = 12, 2, 3, 2
    n = 1 << logn
    bs, cs = split_primes(S, T)
    k = Consts(bs, cs)
    pb, pc = ones_plan(lib, logn, bs), ones_plan(lib, logn, cs)
    cv = lib.RnsConv(pb, pc)
    pb.close()
    pc.close()
    x = rand_rns((batch, T + S, n), cs + bs, 99000)
    hx = host(x)
    want_c, want_d = convert_ref(hx[:, T:], k), mod_down_ref(hx, k, True)
    # unaligned views: UNSUPPORTED, every buffer untouched
    for kk in (1, 2, 3):
        for ki, ko in ((kk, 0), (0, kk)):
            gi, go = Guarded(batch * (T + S) * n, ki, x), Guarded(batch * T * n, ko)
            snap = gi.raw.clone()
            calls = [lambda: cv.convert(gi.view[T * n:], go.view, batch, in_stride=(T + S) * n),
                     lambda: cv.mod_down(gi.view, go.view, batch, round=True)]
            for i, call in enumerate(calls):
                assert _status(lib, call) == UNSUPPORTED, (kk, ki, ko, i)
            torch.cuda.synchronize()
            assert go.untouched() and torch.equal(gi.raw, snap)
    # overlaps: INVALID_ARG, nothing written
    big = Guarded(4 * (T + S) * n, 0, torch.cat([x.reshape(-1), x.reshape(-1)]))
    snap = big.raw.clone()
    row = (T + S) * n
    v = big.view
    bad = [lambda: cv.mod_down(v, v, batch),                                  # in place
           lambda: cv.mod_down(v, v[row + T * n:], batch),                    # into row 1's source channels
           lambda: cv.mod_down(v[T * n:], v[n:], 1),                          # output ends inside the input
           lambda: cv.convert(v, v[(S - 1) * n:], batch, in_stride=row, out_stride=row),     # same stride, collides
           lambda: cv.convert(v, v[(S + 1) * n:], batch, in_stride=row, out_stride=row),     # runs into row b+1
           lambda: cv.convert(v[row:], v, batch, in_stride=row, out_stride=row),            # row 0 out hits row 0 in
           lambda: cv.convert(v, v[S * n:], batch, in_stride=2 * row, out_stride=row)]       # rows apart, extents overlap
    for i, call in enumerate(bad):
        assert _status(lib, call) == INVALID_ARG, i
    # bad strides and flags
    L = lib.load_library()
    A, C = x.data_ptr(), big.view.data_ptr()
    for ins, outs in ((S * n - n, 0), (S * n + 1, 0), (0, T * n - n), (0, T * n + 4), (n // 2, 0)):
        assert L.nttb200_rns_base_convert(cv._h, A, ins, C, outs, batch, None) == INVALID_ARG, (ins, outs)
    assert L.nttb200_rns_mod_down(cv._h, A, C, batch, 2, None) == INVALID_ARG
    assert L.nttb200_rns_mod_down(cv._h, A, None, batch, 0, None) == INVALID_ARG
    assert L.nttb200_rns_base_convert(cv._h, None, 0, C, 0, batch, None) == INVALID_ARG
    torch.cuda.synchronize()
    assert torch.equal(big.raw, snap)
    # accepted: equal strides, rows interleaved without a shared word (batch 1 may run past row 0)
    cv.convert(v, v[(S + 1) * n:], 1, in_stride=row, out_stride=row)
    assert np.array_equal(host(v[(S + 1) * n:(S + 1 + T) * n].view(1, T, n)),
                          convert_ref(hx[:1, :S], k))
    # batch == 0: OK, nothing launched
    before = lib.kernel_launches()
    assert L.nttb200_rns_base_convert(cv._h, None, 0, None, 0, 0, None) == OK
    assert L.nttb200_rns_mod_down(cv._h, None, None, 0, ROUND, None) == OK
    cv.convert(x, x, 0)
    assert lib.kernel_launches() == before
    # still usable, with both plans gone
    out = Guarded(batch * T * n)
    cv.convert(x[:, T:], out.view, batch, in_stride=row)
    assert np.array_equal(host(out.view.view(batch, T, n)), want_c) and out.guards_intact()
    cv.mod_down(x, out.view, batch, round=True)
    assert np.array_equal(host(out.view.view(batch, T, n)), want_d) and out.guards_intact()
    assert np.array_equal(host(x), hx)
    cv.close()


@pytest.mark.gpu
def test_beyond_2_31_words(lib):
    """One call over 2^31 + 2^16 words each way (S = T = 1, N = 2^16, batch 2^15 + 1): convert
    from channel 1 of a [batch][2][N] buffer into its channel 0, then mod_down of that buffer;
    checked on sampled polynomials including the last."""
    torch = _torch()
    logn, batch = 16, (1 << 15) + 1
    n = 1 << logn
    cs, bs = split_primes(1, 1)
    k = Consts(bs, cs)
    gen = torch.Generator(device="cuda").manual_seed(99500)
    x = torch.randint(0, min(bs[0], cs[0]), (batch, 2, n), dtype=torch.int32, device="cuda", generator=gen)
    rows = np.array([0, 1, batch // 2, batch - 2, batch - 1])
    src = host(x[:, 1], rows)[:, None]
    out = torch.empty((batch, 1, n), dtype=torch.int32, device="cuda")
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        cv.convert(x[:, 1], x, batch, in_stride=2 * n, out_stride=2 * n)
        assert np.array_equal(host(x[:, :1], rows), convert_ref(src, k))
        cv.mod_down(x, out, batch, round=True)
    assert np.array_equal(host(out, rows), mod_down_ref(host(x, rows), k, True))
