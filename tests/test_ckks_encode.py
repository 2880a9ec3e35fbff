"""CKKS slot encoding and decoding on RNS batches: nttb200_ckks_encode / nttb200_ckks_decode.
On the CPU: a numpy reference written from the convention in include/nttb200.h, checked against
direct evaluation m(zeta^(5^j)) in long double, the rotation and conjugation identities on it, and
the null-argument checks.  On the GPU: encode against the reference through the residues of every
channel, the |a| >= 2^64 branch, decode of known centred integers at both ends of the range, the
round trip, rotation / conjugation / product / rescale through the existing kernels, the buffer
rules, the launch counts and one call over 2^31 output words."""
import ctypes
import math
import random

import numpy as np
import pytest

from test_rns_conv import split_primes
from test_rns_eval import Guarded, _status, channel_tables, ones_plan, rows_of

OK, INVALID_ARG, MODULUS, UNSUPPORTED = 0, 1, 2, 7
L2_BYTES = 160 << 20     # more than the B200's 126 MB L2


# ------------------------------------------------------------------------- numpy reference
def slot_perm(N):
    """s_j = (5^j mod 2N - 1) / 4 for j < N/2."""
    return np.array([(pow(5, j, 2 * N) - 1) // 4 for j in range(N // 2)], dtype=np.int64)


def zeta_pows(N, sign=1):
    k = np.arange(N // 2)
    return np.exp(sign * 1j * np.pi * k / N)


def decode_ref(x, scale):
    """x: float64 [..., N] coefficients -> complex128 [..., N/2] slots."""
    N = x.shape[-1]
    n = N // 2
    y = (x[..., :n] + 1j * x[..., n:]) * zeta_pows(N)
    Y = np.fft.ifft(y, axis=-1) * n            # sum_k y_k e^(+2 pi i s k / n)
    return Y[..., slot_perm(N)] / scale


def encode_unrounded(z, scale):
    """z: complex128 [..., n] -> scale * m (float64 [..., 2n]) before rounding."""
    n = z.shape[-1]
    N = 2 * n
    v = np.empty_like(z)
    v[..., slot_perm(N)] = z
    y = np.fft.fft(v, axis=-1) / n             # (1/n) sum_s v_s e^(-2 pi i s k / n)
    m = y * zeta_pows(N, -1)
    return np.concatenate([m.real, m.imag], axis=-1) * scale


def fft_tau(n, scale, z):
    """The FFT error bound of DESIGN 3.6 on one encoded coefficient: 8 (log2 n + 1) 2^-53 scale
    ||z||_rms, per polynomial (z [..., n])."""
    rms = np.sqrt(np.mean(np.abs(z) ** 2, axis=-1, keepdims=True))
    return 8 * (math.log2(n) + 1) * 2.0 ** -53 * scale * rms


def decode_tau(x, scale):
    """The bound on one decoded slot: 8 (log2 n + 1) 2^-53 sqrt(n) ||x||_2 / scale (x [..., N])."""
    n = x.shape[-1] // 2
    return 8 * (math.log2(n) + 1) * 2.0 ** -53 * math.sqrt(n) * np.linalg.norm(x, axis=-1, keepdims=True) / scale


def rand_slots(shape, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(-1, 1, shape) + 1j * rng.uniform(-1, 1, shape)


def negacyclic_sigma(x, g):
    """a(X) -> a(X^g) mod X^N + 1 on integer / float coefficients."""
    N = x.shape[-1]
    e = np.arange(N) * g % (2 * N)
    out = np.zeros_like(x)
    out[..., e % N] = np.where(e < N, 1, -1) * x
    return out


# ------------------------------------------------------------------ CPU: the reference itself
def test_reference_matches_direct_evaluation():
    """N = 4096: decode_ref equals m(zeta^(5^j)) evaluated in long double (order and sign)."""
    N = 4096
    rng = np.random.default_rng(5)
    x = rng.integers(-1000, 1000, N)
    z = decode_ref(x.astype(np.float64), 1.0)
    ld = np.longdouble
    pi = ld(np.pi)
    k = np.arange(N, dtype=ld)
    for j in list(range(8)) + [1000, N // 2 - 1]:
        e = pow(5, j, 2 * N)
        ang = (pi * e / N) * k
        re, im = np.sum(x * np.cos(ang)), np.sum(x * np.sin(ang))
        assert abs(complex(float(re), float(im)) - z[j]) < 1e-6 * np.linalg.norm(x), j


def test_reference_encode_inverts_decode():
    N = 4096
    z = rand_slots(N // 2, 6)
    m = encode_unrounded(z, 1.0)
    assert np.max(np.abs(decode_ref(m, 1.0) - z)) < 1e-12
    x = np.random.default_rng(7).integers(-2 ** 20, 2 ** 20, N).astype(np.float64)
    assert np.max(np.abs(encode_unrounded(decode_ref(x, 1.0), 1.0) - x)) < 1e-6


@pytest.mark.parametrize("r", [1, -1, 7, 1024])
def test_reference_rotation_and_conjugation(lib, r):
    N = 4096
    x = np.random.default_rng(8).integers(-1000, 1000, N).astype(np.float64)
    z = decode_ref(x, 1.0)
    rot = decode_ref(negacyclic_sigma(x, lib.galois_rotation(N, r)), 1.0)
    assert np.max(np.abs(rot - np.roll(z, -r))) < 1e-7
    conj = decode_ref(negacyclic_sigma(x, lib.galois_conjugate(N)), 1.0)
    assert np.max(np.abs(conj - np.conj(z))) < 1e-7


def test_null_arguments_without_device(lib):
    L = lib.load_library()
    h = ctypes.c_void_p()
    assert L.nttb200_ckks_encoder_create(None, None, 0) == INVALID_ARG
    assert L.nttb200_ckks_encoder_create(ctypes.byref(h), None, 0) == INVALID_ARG and not h.value
    assert L.nttb200_ckks_encoder_destroy(None) == OK
    assert L.nttb200_ckks_encode(None, 16, 1.0, 16, 1, None) == INVALID_ARG
    assert L.nttb200_ckks_encode(None, None, 1.0, None, 0, None) == INVALID_ARG
    assert L.nttb200_ckks_decode(None, 16, 0, 1, 1.0, 16, 1, None) == INVALID_ARG
    assert L.nttb200_ckks_decode(None, None, 0, 1, 1.0, None, 0, None) == INVALID_ARG


# ------------------------------------------------------------------------------ GPU helpers
def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"
    return torch


def centred_crt(res, qs):
    """res: int [L, cols] residues -> list of centred Python ints."""
    B = math.prod(qs)
    out = []
    for col in np.asarray(res).T:
        x = sum(int(r) * (B // q) * pow(B // q % q, -1, q) for r, q in zip(col, qs)) % B
        out.append(x - B if x > B // 2 else x)
    return out


def check_encoded(res, qs, ref, tau):
    """res: uint64 [L, N] residues of one polynomial, ref: float64 [N] unrounded scale * m.
    Every channel holds c mod q_l for one integer c with |c - ref| <= 1/2 + tau, and c = rint(ref)
    wherever ref lies more than tau from a half-integer."""
    lo = np.floor(ref - 0.5 - tau).astype(np.int64)
    ok = np.zeros(ref.shape, dtype=bool)
    for d in range(4):
        c = lo + d
        inside = np.abs(c - ref) <= 0.5 + tau
        match = np.all([(c % q).astype(np.uint64) == res[l] for l, q in enumerate(qs)], axis=0)
        ok |= inside & match
    assert ok.all(), np.nonzero(~ok)[0][:8]
    sure = np.abs(ref - np.floor(ref) - 0.5) > tau
    r = np.rint(ref).astype(np.int64)
    for l, q in enumerate(qs):
        assert np.array_equal(res[l][sure], (r[sure] % q).astype(np.uint64))


def batch_of(batch, n, L):
    return -(-L2_BYTES // (16 * n + 8 * L * n)) if batch == "l2" else batch


ENCODE_CASES = [(logn, L, batch) for logn in (12, 13, 14, 15, 16) for L in (1, 3, 32) for batch in (1, 5, "l2")]


@pytest.mark.gpu
@pytest.mark.parametrize("logn,L,batch", ENCODE_CASES)
def test_encode(lib, logn, L, batch):
    torch = _torch()
    N, n = 1 << logn, 1 << (logn - 1)
    qs = split_primes(L)[0]
    batch = batch_of(batch, n, L)
    z = rand_slots((batch, n), 100 + logn + L)
    d_z = torch.from_numpy(z).cuda()
    out = torch.empty((batch, L, N), dtype=torch.int32, device="cuda")
    rows = rows_of(batch, logn)
    with lib.CkksEncoder(ones_plan(lib, logn, qs)) as enc:
        for scale in (2.0 ** 20, 2.0 ** 40):
            l0 = lib.kernel_launches()
            enc.encode(d_z, out, batch, scale)
            torch.cuda.synchronize()
            assert lib.kernel_launches() - l0 == (1 if logn <= 14 else 2)
            ref = encode_unrounded(z[rows], scale)
            tau = fft_tau(n, scale, z[rows])
            got = out[torch.from_numpy(rows).cuda()].cpu().numpy().astype(np.uint64)
            for i in range(len(rows)):
                check_encoded(got[i], qs, ref[i], tau[i])


@pytest.mark.gpu
def test_encode_beyond_2_64(lib):
    """scale 2^75 on four channels: |a| >= 2^64, CRT'd a_k is a double's exact integer value
    within 1/2 + tau of the reference."""
    torch = _torch()
    logn, N, n = 12, 4096, 2048
    qs = split_primes(4)[0]
    z = rand_slots((2, n), 11)
    out = torch.empty((2, 4, N), dtype=torch.int32, device="cuda")
    scale = 2.0 ** 75
    with lib.CkksEncoder(ones_plan(lib, logn, qs)) as enc:
        enc.encode(torch.from_numpy(z).cuda(), out, 2, scale)
    res = out.cpu().numpy()
    ref = encode_unrounded(z, scale)
    tau = fft_tau(n, scale, z)
    big = 0
    for b in range(2):
        a = centred_crt(res[b], qs)
        for k in range(N):
            assert float(a[k]) == a[k]
            assert abs(a[k] - int(ref[b, k])) <= 1 + tau[b, 0]
            big += abs(a[k]) >= 1 << 64
    assert big > N


DECODE_CASES = [(logn, L, batch) for logn in (12, 13, 14, 15, 16) for L in (1, 3, 32) for batch in (1, 5, "l2")]


@pytest.mark.gpu
@pytest.mark.parametrize("logn,L,batch", DECODE_CASES)
def test_decode(lib, logn, L, batch):
    """Residues of known centred integers on the moduli 2^30, 3 and NTT primes, every channel count;
    coefficients 0 and 1 at floor(B/2) and -floor((B-1)/2)."""
    torch = _torch()
    N, n = 1 << logn, 1 << (logn - 1)
    qs = ([1 << 30, 3] + split_primes(L)[0])[:L]
    batch = batch_of(batch, n, L)
    rows = rows_of(batch, logn)
    rnd = random.Random(logn * 7 + L)
    with lib.CkksEncoder(ones_plan(lib, logn, qs)) as enc:
        for C in range(1, min(L, 4) + 1):
            B = math.prod(qs[:C])
            x = [[B // 2, -((B - 1) // 2)] + [rnd.randrange(B) - (B - 1) // 2 for _ in range(N - 2)] for _ in rows]
            res = np.zeros((batch, L, N), dtype=np.int64)
            for i, r in enumerate(rows):
                res[r, :C] = np.array([[v % q for v in x[i]] for q in qs[:C]])
            d_in = torch.from_numpy(res.astype(np.int32)).cuda()
            d_z = torch.empty((batch, n), dtype=torch.complex128, device="cuda")
            scale = 2.0 ** 40
            l0 = lib.kernel_launches()
            enc.decode(d_in, d_z, batch, scale, channels=C, in_stride=L * N)
            torch.cuda.synchronize()
            assert lib.kernel_launches() - l0 == (1 if logn <= 14 else 2)
            got = d_z.cpu().numpy()[rows]
            xf = np.array([[float(v) for v in xr] for xr in x])
            want = decode_ref(xf, scale)
            tol = decode_tau(xf, scale) + 2.0 ** -51 * np.abs(want)
            assert np.all(np.abs(got - want) <= tol), (C, np.max(np.abs(got - want) / tol))


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 13, 14, 15, 16])
def test_round_trip(lib, logn):
    torch = _torch()
    N, n, batch = 1 << logn, 1 << (logn - 1), 3
    qs = split_primes(3)[0]
    z = rand_slots((batch, n), 40 + logn)
    out = torch.empty((batch, 3, N), dtype=torch.int32, device="cuda")
    back = torch.empty((batch, n), dtype=torch.complex128, device="cuda")
    with lib.CkksEncoder(ones_plan(lib, logn, qs)) as enc:
        for scale in (2.0 ** 20, 2.0 ** 40):
            enc.encode(torch.from_numpy(z).cuda(), out, batch, scale)
            enc.decode(out, back, batch, scale)
            err = np.abs(back.cpu().numpy() - z)
            assert np.all(err <= N / (2 * scale) + 2 * fft_tau(n, 1.0, z)), np.max(err)


class Ckks:
    """Forward / inverse plans on NTT primes and an encoder."""

    def __init__(self, lib, logn, L):
        self.lib, self.logn, self.N, self.n = lib, logn, 1 << logn, 1 << (logn - 1)
        self.qs = split_primes(L)[0]
        fwd, inv, _ = channel_tables(lib, self.N, self.qs)
        self.fwd = lib.RnsPlan(self.qs, fwd, logn=logn)
        self.inv = lib.RnsPlan(self.qs, inv, logn=logn)
        self.enc = lib.CkksEncoder(self.fwd)

    def encode(self, z, scale):
        torch = _torch()
        out = torch.empty((z.shape[0], len(self.qs), self.N), dtype=torch.int32, device="cuda")
        self.enc.encode(torch.from_numpy(z).cuda(), out, z.shape[0], scale)
        return out

    def decode(self, a, scale, channels=None):
        torch = _torch()
        out = torch.empty((a.shape[0], self.n), dtype=torch.complex128, device="cuda")
        self.enc.decode(a, out, a.shape[0], scale, channels=channels)
        return out.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 14, 16])
def test_rotation_and_conjugation_through_automorphism(lib, logn):
    """automorphism(galois_rotation(N, r)) moves slot j + r to slot j, galois_conjugate conjugates,
    on coefficients and in the rns_ct order."""
    torch = _torch()
    c = Ckks(lib, logn, 3)
    N, scale = c.N, 2.0 ** 40
    z = rand_slots((2, c.n), 60 + logn)
    a = c.encode(z, scale)
    rs = [1, -1, 7, N // 4]
    gs = [lib.galois_rotation(N, r) for r in rs] + [lib.galois_conjugate(N)]
    want = [np.roll(z, -r, axis=-1) for r in rs] + [np.conj(z)]
    tol = N / (2 * scale) + 4 * fft_tau(c.n, 1.0, z)
    coeff = torch.empty((len(gs), 2, 3, N), dtype=torch.int32, device="cuda")
    c.fwd.automorphism(a, coeff, 2, gs, domain=lib.AUTO_COEFF)
    ev = torch.empty_like(a)
    c.fwd.ct(a, ev, 2)
    evo = torch.empty_like(coeff)
    c.fwd.automorphism(ev, evo, 2, gs, domain=lib.AUTO_EVAL)
    back = torch.empty_like(a)
    for i, w in enumerate(want):
        assert np.all(np.abs(c.decode(coeff[i], scale) - w) <= tol), gs[i]
        c.inv.gs_scaled(evo[i], back, 2)
        assert np.all(np.abs(c.decode(back, scale) - w) <= tol), gs[i]


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 15])
def test_product_and_rescale(lib, logn):
    """rns_polymul_negacyclic of two encodings decodes with scale^2 to z1 z2; after mod_down(ROUND)
    by the last prime, with scale^2 / q_last."""
    torch = _torch()
    c = Ckks(lib, logn, 4)
    N, scale = c.N, 2.0 ** 30
    z1, z2 = rand_slots((2, c.n), 70 + logn), rand_slots((2, c.n), 80 + logn)
    a1, a2 = c.encode(z1, scale), c.encode(z2, scale)
    prod = torch.empty_like(a1)
    lib.rns_polymul_negacyclic(c.fwd, c.inv, a1, a2, prod, 2)
    want = z1 * z2
    tol = 2 * N / (2 * scale) * 2 + 8 * fft_tau(c.n, 1.0, want)
    assert np.all(np.abs(c.decode(prod, scale * scale) - want) <= tol)
    q_last = c.qs[-1]
    src = lib.RnsPlan([q_last], [np.ones(N, dtype=np.int32)], logn=logn)
    dst = lib.RnsPlan(c.qs[:-1], [np.ones(N, dtype=np.int32)] * 3, logn=logn)
    down = torch.empty((2, 3, N), dtype=torch.int32, device="cuda")
    with lib.RnsConv(src, dst) as conv:
        conv.mod_down(prod, down, 2, round=True)
    tol2 = tol + N * q_last / (2 * scale * scale)
    got = c.decode(down, scale * scale / q_last, channels=3)
    assert np.all(np.abs(got - want) <= tol2), np.max(np.abs(got - want))


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 15])
def test_buffers_and_errors(lib, logn):
    torch = _torch()
    N, n, batch = 1 << logn, 1 << (logn - 1), 3
    qs = split_primes(3)[0]
    z = rand_slots((batch, n), 90)
    zi = torch.from_numpy(z).cuda().view(torch.int32).reshape(-1)
    with lib.CkksEncoder(ones_plan(lib, logn, qs)) as enc:
        L = lib.load_library()
        h = enc._h
        zin = Guarded(batch * 4 * n, data=zi)
        out = Guarded(batch * 3 * N)
        assert L.nttb200_ckks_encode(h, zin.view.data_ptr(), 2.0 ** 30, out.view.data_ptr(), batch, None) == OK
        torch.cuda.synchronize()
        assert out.guards_intact() and zin.guards_intact() and torch.equal(zin.view, zi)
        res = out.view.clone()
        dec = Guarded(batch * 4 * n)
        assert L.nttb200_ckks_decode(h, out.view.data_ptr(), 0, 3, 2.0 ** 30, dec.view.data_ptr(), batch, None) == OK
        torch.cuda.synchronize()
        assert dec.guards_intact() and torch.equal(out.view, res)
        # strided decode: read the first 2 channels of the [batch][3][N] rows
        dec2 = torch.empty((batch, n), dtype=torch.complex128, device="cuda")
        enc.decode(out.view, dec2, batch, 2.0 ** 30, channels=2, in_stride=3 * N)
        assert np.max(np.abs(dec2.cpu().numpy() - z)) < 1e-6
        # argument errors: nothing written
        fresh = Guarded(batch * 3 * N)
        p_in, p_out = zin.view.data_ptr(), fresh.view.data_ptr()
        for scale in (0.0, -1.0, float("inf"), float("nan")):
            assert L.nttb200_ckks_encode(h, p_in, scale, p_out, batch, None) == INVALID_ARG
            assert L.nttb200_ckks_decode(h, p_out, 0, 1, scale, p_in, batch, None) == INVALID_ARG
            assert L.nttb200_ckks_encode(h, p_in, scale, p_out, 0, None) == INVALID_ARG
        assert L.nttb200_ckks_encode(h, None, 1.0, p_out, batch, None) == INVALID_ARG
        assert L.nttb200_ckks_encode(h, None, 1.0, None, 0, None) == OK
        assert L.nttb200_ckks_encode(h, p_in, 1.0, p_in + 16, batch, None) == INVALID_ARG      # overlap
        assert L.nttb200_ckks_encode(h, p_in + 4, 1.0, p_out, batch, None) == UNSUPPORTED
        assert L.nttb200_ckks_encode(h, p_in, 1.0, p_out + 4, batch, None) == UNSUPPORTED
        src = out.view.data_ptr()
        for ch in (0, 4):
            assert L.nttb200_ckks_decode(h, src, 0, ch, 1.0, p_out, batch, None) == INVALID_ARG
        for stride in (N + 1, N, 4 * N - 1):
            assert L.nttb200_ckks_decode(h, src, stride, 2, 1.0, p_out, batch, None) == INVALID_ARG
        assert L.nttb200_ckks_decode(h, src, 0, 2, 1.0, src + 16, batch, None) == INVALID_ARG     # overlap
        assert L.nttb200_ckks_decode(h, src + 4, 0, 2, 1.0, p_out, batch, None) == UNSUPPORTED
        assert L.nttb200_ckks_decode(h, src, 0, 2, 1.0, p_out + 8, batch, None) == UNSUPPORTED
        assert L.nttb200_ckks_decode(h, None, 0, 2, 1.0, None, 0, None) == OK
        torch.cuda.synchronize()
        assert fresh.untouched() and zin.guards_intact() and torch.equal(zin.view, zi)
    hh = ctypes.c_void_p()
    assert L.nttb200_ckks_encoder_create(ctypes.byref(hh), ones_plan(lib, logn, qs)._h, 1) == INVALID_ARG
    with lib.CkksEncoder(ones_plan(lib, logn, [6, 35, 9])) as enc:
        d = torch.zeros((1, 3, N), dtype=torch.int32, device="cuda")
        zz = torch.empty((1, n), dtype=torch.complex128, device="cuda")
        assert _status(lib, lambda: enc.decode(d, zz, 1, 1.0, channels=2)) == OK
        assert _status(lib, lambda: enc.decode(d, zz, 1, 1.0, channels=3)) == MODULUS
        assert _status(lib, lambda: enc.decode(d, zz, 0, 1.0, channels=3)) == MODULUS


@pytest.mark.gpu
def test_encode_beyond_2_31_words(lib):
    """One encode of 1025 polynomials at N = 2^16, L = 32: 2^31 + 2^21 output words."""
    torch = _torch()
    logn, L, batch = 16, 32, 1025
    N, n = 1 << logn, 1 << (logn - 1)
    qs = split_primes(L)[0]
    z = rand_slots((2, n), 12)
    d_z = torch.from_numpy(z).cuda()[torch.arange(batch, device="cuda") % 2].contiguous()
    out = torch.empty((batch, L, N), dtype=torch.int32, device="cuda")
    with lib.CkksEncoder(ones_plan(lib, logn, qs)) as enc:
        enc.encode(d_z, out, batch, 2.0 ** 40)
    torch.cuda.synchronize()
    assert torch.equal(out[batch - 1], out[0]) and torch.equal(out[batch - 2], out[1])
    ref = encode_unrounded(z[:1], 2.0 ** 40)
    check_encoded(out[batch - 1].cpu().numpy().astype(np.uint64), qs, ref[0], fft_tau(n, 2.0 ** 40, z[:1])[0])
