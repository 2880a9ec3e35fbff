"""Hybrid key switching on RNS batches: nttb200_rns_keyswitch_create / _apply (Python KeySwitcher).
On the CPU: the argument checks that need no device, and a residue-wise numpy reference of the
operation checked against direct big-integer evaluation (ragged last digit included).  On the GPU:
bit-exactness against the composed sequence of existing calls (rns_gs_scaled, base_convert, rns_ct,
automorphism, rns_dot, rns_gs_scaled, mod_down, rns_ct) for N = 2^12..2^16, five (L, K, alpha),
count 1, 3 and 64, all four COEFF_IN / COEFF_OUT combinations, batch 1 and the strided c1 of a
ciphertext batch, and one shape beyond the L2; CKKS rotations (single and hoisted) and
relinearisation with host-built keys decoded on the device; a BFV product relinearised in the
coefficient domain; the buffer rules, the create errors and the launch counts."""
import ctypes
import math

import numpy as np
import pytest

from test_packed_encode import Keys, bfv_tensor, channels, decrypt_to_t, rand_slots, signed, to_dev, valid_t
from test_rns_automorph import negamul, sigma_int
from test_rns_eval import Guarded, _status, channel_tables, ones_plan, rand_rns
from test_rns_sizes import channel_primes

OK, INVALID_ARG, MODULUS, UNSUPPORTED = 0, 1, 2, 7
COEFF_IN, COEFF_OUT = 1, 2
ADD, MUL = 0, 2
CONFIGS = [(3, 1, 1), (24, 8, 8), (24, 8, 24), (20, 4, 6), (31, 1, 31)]


def digits_of(L, alpha):
    return [(lo, min(lo + alpha, L)) for lo in range(0, L, alpha)]


def launches(logn, dnum, coeff_in=False, coeff_out=False):
    t = 1 if logn == 12 else 2
    return 2 * dnum + 1 + 4 * t - (t if coeff_in else 0) - (t if coeff_out else 0)


# ------------------------------------------------------------------ CPU: argument checks
def test_null_arguments_without_device(lib):
    L = lib.load_library()
    h = ctypes.c_void_p()
    g = (ctypes.c_uint32 * 2)(5, 1)
    assert L.nttb200_rns_keyswitch_create(None, 16, 16, 1, 1, 0) == INVALID_ARG
    assert L.nttb200_rns_keyswitch_create(ctypes.byref(h), None, 16, 1, 1, 0) == INVALID_ARG and not h.value
    assert L.nttb200_rns_keyswitch_create(ctypes.byref(h), 16, None, 1, 1, 0) == INVALID_ARG
    assert L.nttb200_rns_keyswitch_destroy(None) == OK
    assert L.nttb200_rns_keyswitch_apply(None, 16, 0, 16, g, 1, 16, 1, 0, None) == INVALID_ARG
    assert L.nttb200_rns_keyswitch_apply(None, None, 0, None, g, 1, None, 0, 0, None) == INVALID_ARG
    assert (lib.KS_COEFF_IN, lib.KS_COEFF_OUT) == (COEFF_IN, COEFF_OUT)
    assert [launches(12, 3), launches(13, 3), launches(16, 1, True, True)] == [11, 15, 7]


# ------------------------------------------------------------ CPU: the reference
def crt(res, ms):
    M = math.prod(ms)
    return sum(int(r) * (M // m) * pow(M // m % m, -1, m) for r, m in zip(res, ms)) % M


def negamul_obj(a, b):
    """a (*) b mod X^N + 1 for object (Python-int) arrays; b sparse"""
    n = len(a)
    out = np.zeros(n, dtype=object)
    for e in np.nonzero(b)[0]:
        r = np.roll(a, e) * b[e]
        r[:e] = -r[:e]
        out = out + r
    return out


def ks_reference(x, keys, qs, L, alpha, g):
    """Residue-wise hybrid key switching in the coefficient domain: x [L][N] residues on Q, keys
    [dnum][2][L+K][N] coefficient residues on Q P (sparse), -> (u0, u1) [2][L][N] on Q."""
    n, LK = x.shape[-1], len(qs)
    acc = np.zeros((2, LK, n), dtype=object)
    for i, (lo, hi) in enumerate(digits_of(L, alpha)):
        dq = qs[lo:hi]
        D = math.prod(dq)
        y = [x[lo + k].astype(object) * pow(D // q % q, -1, q) % q for k, q in enumerate(dq)]
        for j, m in enumerate(qs):   # fast conversion of digit i into every channel, own rows exact
            up = x[j].astype(object) if lo <= j < hi else sum(yk * (D // q % m) for yk, q in zip(y, dq)) % m
            up = sigma_int(up, g) % m
            for p in range(2):
                acc[p, j] = (acc[p, j] + negamul_obj(up, keys[i, p, j].astype(object))) % m
    P = qs[L:]
    B = math.prod(P)
    out = np.zeros((2, L, n), dtype=object)
    for p in range(2):   # mod_down(ROUND): fast conversion of (x + floor(B/2)) on P, subtracted, times B^-1
        yp = [(acc[p, L + k] + B // 2) % b * pow(B // b % b, -1, b) % b for k, b in enumerate(P)]
        for j in range(L):
            c = qs[j]
            conv = sum(yk * (B // b % c) for yk, b in zip(yp, P)) % c
            out[p, j] = (acc[p, j] + B // 2 - conv) % c * pow(B % c, -1, c) % c
    return out


def test_reference_against_big_integers():
    """The residue-wise reference equals the big-integer evaluation: digit values Y_i = sum_j
    y_j (D_i / q_j) as integers, sigma_g, products with the keys mod Q P, and
    ((X + floor(P/2)) - sum_k y'_k (P / p_k)) / P exactly; L = 5, alpha = 2 (digits 2, 2, 1), K = 2."""
    n, L, alpha = 4096, 5, 2
    qs = channel_primes(L + 2)
    QP, P = math.prod(qs), math.prod(qs[L:])
    rng = np.random.default_rng(4242)
    x = np.stack([rng.integers(0, q, n) for q in qs[:L]])
    x[:, :8] = np.array(qs[:L])[:, None] - 1
    dn = len(digits_of(L, alpha))
    keys = np.zeros((dn, 2, L + 2, n), dtype=np.int64)
    for i in range(dn):
        for p in range(2):
            for e in rng.choice(n, 3, replace=False):   # sparse keys keep the big-integer products cheap
                v = int(rng.integers(0, 1 << 62)) * int(rng.integers(1, 1 << 62)) % QP
                keys[i, p, :, e] = [v % m for m in qs]
    for g in (1, 5, 2 * n - 1):
        ref = ks_reference(x, keys, qs, L, alpha, g)
        acc = [np.zeros(n, dtype=object) for _ in range(2)]
        for i, (lo, hi) in enumerate(digits_of(L, alpha)):
            dq = qs[lo:hi]
            D = math.prod(dq)
            Y = sum((x[lo + k].astype(object) * pow(D // q % q, -1, q) % q) * (D // q) for k, q in enumerate(dq))
            Y = sigma_int(Y, g)
            for p in range(2):
                kv = np.array([crt(keys[i, p, :, e], qs) for e in range(n)], dtype=object)
                acc[p] = acc[p] + negamul_obj(Y, kv)
        for p in range(2):
            X = acc[p] % QP
            yp = [(X + P // 2) % b * pow(P // b % b, -1, b) % b for b in qs[L:]]
            conv = sum(yk * (P // b) for yk, b in zip(yp, qs[L:]))
            V = X + P // 2 - conv
            assert all(v % P == 0 for v in V)
            V = V // P
            for j in range(L):
                assert np.array_equal(V % qs[j], ref[p, j]), (g, p, j)


# ------------------------------------------------------------------------- GPU helpers
def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"
    return torch


class Env:
    """[Q | P] plans, the KeySwitcher and the conversions of the composed sequence."""

    def __init__(self, lib, logn, L, K, alpha, qs=None):
        self.lib, self.logn, self.n = lib, logn, 1 << logn
        self.L, self.K, self.alpha = L, K, alpha
        self.qs = qs or channel_primes(L + K)
        fwd, inv, _ = channel_tables(lib, self.n, self.qs)
        self.qpf = lib.RnsPlan(self.qs, fwd, logn=logn)
        self.qpi = lib.RnsPlan(self.qs, inv, logn=logn)
        self.qf = lib.RnsPlan(self.qs[:L], fwd[:L], logn=logn)
        self.qi = lib.RnsPlan(self.qs[:L], inv[:L], logn=logn)
        self.ks = lib.KeySwitcher(self.qpf, self.qpi, L, alpha)
        self.dig = digits_of(L, alpha)
        assert self.ks.dnum == len(self.dig)
        self.up = []
        for lo, hi in self.dig:
            rest = [j for j in range(L + K) if not lo <= j < hi]
            with ones_plan(lib, logn, self.qs[lo:hi]) as a, ones_plan(lib, logn, [self.qs[j] for j in rest]) as b:
                self.up.append((lib.RnsConv(a, b), rest))
        with ones_plan(lib, logn, self.qs[L:]) as a, ones_plan(lib, logn, self.qs[:L]) as b:
            self.down = lib.RnsConv(a, b)

    def composed(self, x, keys, gs, batch):
        """The existing calls: x [batch][L][N] in the rns_ct order -> (coefficients, rns_ct order) of
        [count][batch][2][L][N]."""
        torch, lib = _torch(), self.lib
        L, LK, n, dn, cnt = self.L, self.L + self.K, self.n, len(self.dig), len(gs)
        xc = torch.empty_like(x)
        self.qi.gs_scaled(x, xc, batch)
        d = torch.empty((dn, batch, LK, n), dtype=torch.int32, device="cuda")
        for i, ((lo, hi), (conv, rest)) in enumerate(zip(self.dig, self.up)):
            tmp = torch.empty((batch, len(rest), n), dtype=torch.int32, device="cuda")
            conv.convert(xc[:, lo:hi], tmp, batch, in_stride=L * n)
            d[i][:, rest] = tmp
            d[i][:, lo:hi] = xc[:, lo:hi]
        self.qpf.ct(d, d, dn * batch)
        rot = torch.empty((cnt, dn, batch, LK, n), dtype=torch.int32, device="cuda")
        self.qpf.automorphism(d, rot, dn * batch, gs)
        u = torch.empty((cnt, batch, 2, LK, n), dtype=torch.int32, device="cuda")
        part = torch.empty((batch, LK, n), dtype=torch.int32, device="cuda")
        for c in range(cnt):
            for p in range(2):
                lib.rns_dot(self.qpf, rot[c], keys[c, :, p].contiguous(), part, dn, batch, w_batch=1)
                u[c, :, p] = part
        del rot
        self.qpi.gs_scaled(u, u, cnt * batch * 2)
        out = torch.empty((cnt, batch, 2, L, n), dtype=torch.int32, device="cuda")
        self.down.mod_down(u, out, cnt * batch * 2, round=True)
        ev = torch.empty_like(out)
        self.qf.ct(out, ev, cnt * batch * 2)
        return out, ev

    def close(self):
        for o in [self.ks, self.qpf, self.qpi, self.qf, self.qi, self.down] + [c for c, _ in self.up]:
            o.close()


def element_sets(lib, n, seed):
    rng = np.random.default_rng(seed)
    rot, back, conj = lib.galois_rotation(n, 1), lib.galois_rotation(n, -3), lib.galois_conjugate(n)
    g64 = [1, rot, back, conj] + [int(v) * 2 + 1 for v in rng.integers(0, n, 60)]
    return [[1], [rot], [back], [conj], [rot, back, conj], g64]


# ------------------------------------------------------------ GPU: bit-exact, composed
@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 13, 14, 15, 16])
@pytest.mark.parametrize("L,K,alpha", CONFIGS)
def test_bit_exact_against_composed(lib, logn, L, K, alpha):
    """One call equals the composed sequence bit for bit: batch 1 and the strided c1 of a batch of
    three [2][L][N] ciphertexts, element sets of count 1 (1, a rotation, a negative rotation,
    conjugation), 3 and 64, all four COEFF_IN / COEFF_OUT combinations; guard bands around the
    output; the input and the keys unchanged; the launch count of the formula."""
    torch = _torch()
    env = Env(lib, logn, L, K, alpha)
    n, LK, dn = env.n, L + K, env.ks.dnum
    seed = 97000 + 100 * logn + L
    ct = rand_rns((3, 2, L, n), env.qs[:L], seed)
    keys = rand_rns((64, dn, 2, LK, n), env.qs, seed + 1)
    ksnap, csnap = keys.clone(), ct.clone()
    for gs in element_sets(lib, n, seed):
        for batch, src, stride in ((1, ct[0, 1:2], 0), (3, ct[:, 1], 2 * L * n)):
            x = src.contiguous()
            want_c, want_e = env.composed(x, keys, gs, batch)
            xc = torch.empty_like(x)
            env.qi.gs_scaled(x, xc, batch)
            words = len(gs) * batch * 2 * L * n
            for flags in range(4):
                inp = xc if flags & COEFF_IN else src
                out = Guarded(words)
                before = lib.kernel_launches()
                env.ks.switch(inp, keys, out.view, batch, gs, in_stride=0 if flags & COEFF_IN else stride,
                              coeff_in=bool(flags & COEFF_IN), coeff_out=bool(flags & COEFF_OUT))
                assert lib.kernel_launches() - before == launches(logn, dn, flags & COEFF_IN, flags & COEFF_OUT)
                want = want_c if flags & COEFF_OUT else want_e
                assert torch.equal(out.view.view(want.shape), want), (gs[:3], batch, flags)
                assert out.guards_intact()
    assert torch.equal(keys, ksnap) and torch.equal(ct, csnap)
    env.close()


@pytest.mark.gpu
def test_bit_exact_beyond_l2(lib):
    """N = 2^16, (L, K, alpha) = (24, 8, 8), batch 86, two elements: 2^29 output words."""
    torch = _torch()
    logn, L, K, alpha, batch = 16, 24, 8, 8, 86
    env = Env(lib, logn, L, K, alpha)
    x = rand_rns((batch, L, env.n), env.qs[:L], 98000)
    keys = rand_rns((2, env.ks.dnum, 2, L + K, env.n), env.qs, 98001)
    gs = [lib.galois_rotation(env.n, 5), 1]
    assert 2 * batch * 2 * L * env.n >= 1 << 28
    _, want = env.composed(x, keys, gs, batch)
    out = torch.empty_like(want)
    env.ks.switch(x, keys, out, batch, gs)
    assert torch.equal(out, want)
    env.close()


# ------------------------------------------------------------- GPU: end to end
def host_keys(env, s, sps, seed):
    """[count][dnum][2][L+K][N] on Q P in the rns_ct order: b_i + a_i s = e_i + P (Q/D_i)
    [(Q/D_i)^-1]_{D_i} s'  with s' = sps[c]."""
    rng = np.random.default_rng(seed)
    qs, L, n = env.qs, env.L, env.n
    Q, P = math.prod(qs[:L]), math.prod(qs[L:])
    k = np.zeros((len(sps), env.ks.dnum, 2, len(qs), n), dtype=np.int64)
    for c, sp in enumerate(sps):
        for i, (lo, hi) in enumerate(env.dig):
            D = math.prod(qs[lo:hi])
            gad = P * (Q // D) * pow(Q // D % D, -1, D)
            e = rng.integers(-4, 5, n)
            for j, m in enumerate(qs):
                a = rng.integers(0, m, n)
                k[c, i, 1, j] = a
                k[c, i, 0, j] = (e - negamul(a, s, m) + (gad % m) * (sp % m)) % m
    d = to_dev(k)
    env.qpf.ct(d, d, len(sps) * env.ks.dnum * 2)
    return d


def square(s):
    """s^2 mod X^N + 1 for a small integer polynomial"""
    n = len(s)
    full = np.convolve(s, s)
    r = full[:n].copy()
    r[:n - 1] -= full[n:]
    return r


def ckks_setup(lib, logn, seed):
    L, K, alpha = 3, 2, 2   # digits of 2 and 1 primes; P > D_i
    env = Env(lib, logn, L, K, alpha)
    keys = Keys(lib, logn, env.qs[:L], seed)
    return env, keys


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 13])
def test_ckks_rotation_end_to_end(lib, logn):
    """Encoded slots, encrypted with a host secret, rotated by 1 and -3 and conjugated through one
    call each and through one hoisted call; the hoisted outputs equal the single ones bit for bit
    and every result decodes to the rotated slots."""
    torch = _torch()
    env, keys = ckks_setup(lib, logn, 99000 + logn)
    n, L, slots = env.n, env.L, env.n // 2
    rng = np.random.default_rng(99100 + logn)
    z = rng.uniform(-1, 1, slots) + 1j * rng.uniform(-1, 1, slots)
    scale = 2.0 ** 34
    gs = [lib.galois_rotation(n, 1), lib.galois_rotation(n, -3), lib.galois_conjugate(n)]
    wants = [np.roll(z, -1), np.roll(z, 3), np.conj(z)]
    rk = host_keys(env, keys.s, [sigma_int(keys.s, g) for g in gs], 99200 + logn)
    with lib.CkksEncoder(keys.pf) as enc:
        m = torch.empty((1, L, n), dtype=torch.int32, device="cuda")
        enc.encode(torch.from_numpy(z[None].astype(np.complex128)).cuda(), m, 1, scale)
        ct = keys.encrypt(m, 1)
        env.qf.ct(ct, ct, 2)
        hoisted = torch.empty((3, 1, 2, L, n), dtype=torch.int32, device="cuda")
        env.ks.switch(ct[1:2], rk, hoisted, 1, gs)
        for c, (g, want) in enumerate(zip(gs, wants)):
            single = torch.empty((1, 1, 2, L, n), dtype=torch.int32, device="cuda")
            env.ks.switch(ct[1:2], rk[c:c + 1].contiguous(), single, 1, g)
            assert torch.equal(single, hoisted[c:c + 1]), g
            out = single[0, 0].clone()
            s0 = torch.empty((1, L, n), dtype=torch.int32, device="cuda")
            env.qf.automorphism(ct[0:1], s0, 1, g)
            env.qf.pointwise(ADD, out[0:1], s0, out[0:1], 1)
            env.qi.gs_scaled(out, out, 2)
            dec = torch.empty((1, slots), dtype=torch.complex128, device="cuda")
            enc.decode(keys.decrypt(out), dec, 1, scale)
            err = np.abs(dec.cpu().numpy()[0] - want).max()
            assert err < 1e-3, (g, err)   # hybrid key-switching noise over Delta = 2^34
    keys.close()
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 14])
def test_ckks_relinearisation_end_to_end(lib, logn):
    """The tensor product of two ciphertexts, relinearised with the s^2 key (g = 1) and rescaled by
    the last prime (mod_down ROUND), decodes to the slotwise product."""
    torch = _torch()
    env, keys = ckks_setup(lib, logn, 99300 + logn)
    n, L, slots, qs = env.n, env.L, env.n // 2, env.qs
    rng = np.random.default_rng(99400 + logn)
    z1, z2 = (rng.uniform(-1, 1, slots) + 1j * rng.uniform(-1, 1, slots) for _ in range(2))
    scale = 2.0 ** 28
    rk = host_keys(env, keys.s, [square(keys.s)], 99500 + logn)
    with lib.CkksEncoder(keys.pf) as enc:
        cts = []
        for z in (z1, z2):
            m = torch.empty((1, L, n), dtype=torch.int32, device="cuda")
            enc.encode(torch.from_numpy(z[None].astype(np.complex128)).cuda(), m, 1, scale)
            ct = keys.encrypt(m, 1)
            env.qf.ct(ct, ct, 2)
            cts.append(ct)
    a, b = cts
    d = torch.empty((3, L, n), dtype=torch.int32, device="cuda")
    tmp = torch.empty((1, L, n), dtype=torch.int32, device="cuda")
    env.qf.pointwise(MUL, a[0:1], b[0:1], d[0:1], 1)
    env.qf.pointwise(MUL, a[0:1], b[1:2], d[1:2], 1)
    env.qf.pointwise(MUL, a[1:2], b[0:1], tmp, 1)
    env.qf.pointwise(ADD, d[1:2], tmp, d[1:2], 1)
    env.qf.pointwise(MUL, a[1:2], b[1:2], d[2:3], 1)
    u = torch.empty((1, 1, 2, L, n), dtype=torch.int32, device="cuda")
    env.ks.switch(d[2:3], rk, u, 1)
    r = d[0:2].clone()
    env.qf.pointwise(ADD, r, u[0, 0], r, 2)
    env.qi.gs_scaled(r, r, 2)
    res = torch.empty((2, L - 1, n), dtype=torch.int32, device="cuda")
    with ones_plan(lib, logn, qs[L - 1:L]) as top, ones_plan(lib, logn, qs[:L - 1]) as low, \
            lib.RnsConv(top, low) as rescale:
        rescale.mod_down(r, res, 2, round=True)
    k2 = Keys(lib, logn, qs[:L - 1], 1)
    k2.s = keys.s
    k2.s_res = to_dev(np.stack([keys.s % q for q in qs[:L - 1]])[None])
    with lib.CkksEncoder(k2.pf) as enc2:
        dec = torch.empty((1, slots), dtype=torch.complex128, device="cuda")
        enc2.decode(k2.decrypt(res), dec, 1, scale * scale / qs[L - 1])
    err = np.abs(dec.cpu().numpy()[0] - z1 * z2).max()
    assert err < 1e-3, err
    k2.close()
    keys.close()
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 13])
def test_bfv_relinearisation_end_to_end(lib, logn):
    """The INTEGRATION BFV multiplication ([P | Q] plan, steps 1-7) gives (d0, d1, d2) in
    coefficients; one call with COEFF_IN | COEFF_OUT and the s^2 key relinearises d2, and the
    two-part ciphertext decrypts exactly to the slotwise product mod t."""
    torch = _torch()
    N, Lq, Km = 1 << logn, 4, 6
    t = valid_t(logn)
    primes = channels(Lq + Km + 2, t)
    qs, ps, sp = primes[:Lq], primes[Lq:Lq + Km], primes[Lq + Km:]
    s1, s2 = rand_slots(1, N, t, 99600 + logn), rand_slots(1, N, t, 99700 + logn)
    want = signed(s1) % t * (signed(s2) % t) % t
    keys = Keys(lib, logn, qs, 99800 + logn)
    env = Env(lib, logn, Lq, 2, 2, qs=qs + sp)
    rk = host_keys(env, keys.s, [square(keys.s)], 99900 + logn)
    pt1, pt2 = (torch.empty((1, Lq, N), dtype=torch.int32, device="cuda") for _ in range(2))
    z = torch.empty_like(s1)
    fwd, inv, _ = channel_tables(lib, N, ps + qs)
    with lib.PackedEncoder(keys.pf, t) as enc:
        enc.encode(s1, pt1, 1)
        enc.encode(s2, pt2, 1)
        c, cp = keys.encrypt(pt1, 1), keys.encrypt(pt2, 1)
        prod = bfv_tensor(lib, logn, t, qs, ps, fwd, inv, c, cp)
        u = torch.empty((1, 1, 2, Lq, N), dtype=torch.int32, device="cuda")
        before = lib.kernel_launches()
        env.ks.switch(prod[2:3], rk, u, 1, coeff_in=True, coeff_out=True)
        assert lib.kernel_launches() - before == launches(logn, env.ks.dnum, True, True)
        r = prod[0:2].clone()
        keys.pf.pointwise(ADD, r, u[0, 0], r, 2)   # coefficient-domain sum: any plan of Q
        enc.decode(decrypt_to_t(lib, keys.decrypt(r), qs, t, True), z, 1)
        assert np.array_equal(signed(z), want)
    keys.close()
    env.close()


# --------------------------------------------------------------- GPU: buffers, errors
@pytest.mark.gpu
def test_create_errors(lib):
    """INVALID_ARG and MODULUS cases of create, all before a device allocation."""
    logn, L, K = 12, 3, 2
    n = 1 << logn
    qs = channel_primes(L + K)
    fwd, inv, _ = channel_tables(lib, n, qs)
    Lb = lib.load_library()
    h = ctypes.c_void_p()
    other = [q for q in channel_primes(L + K + 1) if q not in qs][0]
    with lib.RnsPlan(qs, fwd, logn=logn) as pf, lib.RnsPlan(qs, inv, logn=logn) as pi, \
            ones_plan(lib, logn, qs[:4]) as short, ones_plan(lib, logn, qs[:4] + [other]) as diff, \
            ones_plan(lib, 13, qs) as wide:
        for args in ((pf._h, pi._h, L, 1, 1), (pf._h, pi._h, 0, 1, 0), (pf._h, pi._h, L + K, 1, 0),
                     (pf._h, pi._h, L + K + 1, 1, 0), (pf._h, pi._h, L, 0, 0), (pf._h, pi._h, L, L + 1, 0),
                     (pf._h, short._h, L, 1, 0), (pf._h, wide._h, L, 1, 0), (pf._h, diff._h, L, 1, 0)):
            assert Lb.nttb200_rns_keyswitch_create(ctypes.byref(h), *args) == INVALID_ARG, args
            assert not h.value
        for mods in ([15, 7, 11, 13, 3], [qs[0], qs[1], qs[2], qs[3], 1 << 20]):   # a shared factor, an even modulus
            with ones_plan(lib, logn, mods) as bad:
                assert Lb.nttb200_rns_keyswitch_create(ctypes.byref(h), bad._h, bad._h, L, 1, 0) == MODULUS, mods
                assert not h.value
        with lib.KeySwitcher(pf, pi, L, L) as ks:
            assert ks.dnum == 1
        with lib.KeySwitcher(pf, pi, L, 2) as ks:
            assert ks.dnum == 2


@pytest.mark.gpu
def test_buffers_and_errors(lib):
    """Bad elements, counts and flags (also at batch 0), null buffers, bad strides, overlap of the
    output with the input or the keys -> INVALID_ARG; unaligned buffers -> UNSUPPORTED; nothing
    written, nothing launched; batch 0 -> OK; the plans may be closed after create."""
    torch = _torch()
    logn, L, K, alpha, batch = 13, 3, 2, 2, 2
    env = Env(lib, logn, L, K, alpha)
    n, LK, dn = env.n, L + K, env.ks.dnum
    env.qpf.close()
    env.qpi.close()
    x = rand_rns((batch, L, n), env.qs[:L], 99990)
    keys = rand_rns((2, dn, 2, LK, n), env.qs, 99991)
    words = 2 * batch * 2 * L * n
    ks = env.ks
    out = Guarded(words)
    before = lib.kernel_launches()
    for gs in ([2], [0], [2 * n], [2 * n + 1], [5, 4], [], [5] * 65):
        assert _status(lib, lambda: ks.switch(x, keys, out.view, batch, gs)) == INVALID_ARG, gs
        assert _status(lib, lambda: ks.switch(x, keys, out.view, 0, gs)) == INVALID_ARG, gs
    Lb = lib.load_library()
    g2 = (ctypes.c_uint32 * 2)(5, 1)
    for flags in (4, 8, 1 << 31):
        assert Lb.nttb200_rns_keyswitch_apply(ks._h, x.data_ptr(), 0, keys.data_ptr(), g2, 2, out.view.data_ptr(),
                                              batch, flags, None) == INVALID_ARG
    for args in ((None, keys.data_ptr(), out.view.data_ptr()), (x.data_ptr(), None, out.view.data_ptr()),
                 (x.data_ptr(), keys.data_ptr(), None)):
        assert Lb.nttb200_rns_keyswitch_apply(ks._h, args[0], 0, args[1], g2, 2, args[2], batch, 0, None) == INVALID_ARG
    assert Lb.nttb200_rns_keyswitch_apply(ks._h, None, 0, None, g2, 2, None, 0, 3, None) == OK
    for stride in (L * n - n, L * n + 1, L * n + n // 2):
        assert _status(lib, lambda: ks.switch(x, keys, out.view, batch, [5, 1], in_stride=stride)) == INVALID_ARG
    big = Guarded(words + batch * L * n + 2 * dn * 2 * LK * n)
    v = big.view
    ik, ko = batch * L * n, 2 * dn * 2 * LK * n
    bad = [lambda: ks.switch(v[:ik], keys, v[ik - 4:ik - 4 + words], batch, [5, 1]),
           lambda: ks.switch(v[words:words + ik], keys, v[4:4 + words], batch, [5, 1]),
           lambda: ks.switch(x, v[:ko], v[ko - 4:ko - 4 + words], batch, [5, 1]),
           lambda: ks.switch(x, v[words - 4:words - 4 + ko], v[:words], batch, [5, 1])]
    for i, call in enumerate(bad):
        assert _status(lib, call) == INVALID_ARG, i
    for k in (1, 2, 3):
        ux, uk, uo = Guarded(batch * L * n, k, x), Guarded(keys.numel(), k, keys), Guarded(words, k)
        for call in (lambda: ks.switch(ux.view, keys, out.view, batch, [5, 1]),
                     lambda: ks.switch(x, uk.view, out.view, batch, [5, 1]),
                     lambda: ks.switch(x, keys, uo.view, batch, [5, 1])):
            assert _status(lib, call) == UNSUPPORTED, k
        torch.cuda.synchronize()
        assert uo.untouched()
    assert lib.kernel_launches() == before
    torch.cuda.synchronize()
    assert out.untouched() and big.untouched()
    ks.switch(x, keys, out.view, batch, [5, 1])
    assert out.guards_intact() and not out.untouched()
    env.close()
