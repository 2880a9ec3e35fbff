"""Galois automorphisms on RNS batches: nttb200_rns_automorphism in the coefficient domain and in
the evaluation (rns_ct) order, several elements per call, and galois_rotation / galois_conjugate.
The numpy references of both domains are pinned to the oracle's CT network on the CPU; on the GPU
both domains against them, the commutation with rns_ct / rns_gs_scaled and the composition rules
bit for bit, the buffer rules, and an end-to-end CKKS-style rotation and conjugation (RLWE
ciphertext, Galois keys, hybrid key switching with the library's primitives, decryption on the
host).  The null-plan argument checks run without a device."""
import ctypes
import math

import numpy as np
import pytest

from test_rns_eval import Guarded, _status, channel_tables, host, ones_plan, rand_rns, rows_of
from test_rns_sizes import channel_primes, psi_of

OK, INVALID_ARG, UNSUPPORTED = 0, 1, 7
COEFF, EVAL = 0, 1
ADD = 0
L2_WORDS = 1 << 26   # 256 MiB per operand: twice the B200's L2


# ----------------------------------------------------------------------- references
def brev(x, bits):
    """bit reversal of the integers in the array x over `bits` bits"""
    x = np.asarray(x, dtype=np.int64)
    out = np.zeros_like(x)
    for b in range(bits):
        out |= ((x >> b) & 1) << (bits - 1 - b)
    return out


def coeff_index(n, g):
    """(source index, negate) of every output coefficient: e = j g^-1 mod 2N"""
    e = np.arange(n, dtype=np.int64) * pow(g, -1, 2 * n) % (2 * n)
    return e % n, e >= n


def eval_index(n, g):
    """source index of every output word in the rns_ct order"""
    logn = n.bit_length() - 1
    return brev((g * brev(np.arange(n), logn) + (g - 1) // 2) % n, logn)


def sigma_coeff(x, g, q):
    """x: [..., L, N] residues (uint64 or int64), q: column [L, 1] of the same dtype"""
    src, neg = coeff_index(x.shape[-1], g)
    y = x[..., src]
    return np.where(neg, (q - y) % q, y)


def sigma_eval(x, g):
    return x[..., eval_index(x.shape[-1], g)]


def sigma_int(a, g):
    """the automorphism of an integer polynomial (int64 or Python-int object array)"""
    src, neg = coeff_index(len(a), g)
    y = a[src]
    return np.where(neg, -y, y)


# ------------------------------------------------------------------ CPU: argument checks
def test_null_arguments_without_device(lib):
    L = lib.load_library()
    g1 = (ctypes.c_uint32 * 1)(5)
    assert L.nttb200_rns_automorphism(None, 16, 16, 1, g1, 1, EVAL, None) == INVALID_ARG
    assert L.nttb200_rns_automorphism(None, None, None, 0, g1, 1, COEFF, None) == INVALID_ARG
    assert L.nttb200_rns_automorphism(None, 16, 16, 1, None, 1, EVAL, None) == INVALID_ARG
    assert L.nttb200_rns_automorphism(None, 16, 16, 1, g1, 0, EVAL, None) == INVALID_ARG
    assert L.nttb200_rns_automorphism(None, 16, 16, 1, g1, 1, 2, None) == INVALID_ARG
    assert (lib.AUTO_COEFF, lib.AUTO_EVAL) == (COEFF, EVAL)


# ------------------------------------------------------------- CPU: the conventions
@pytest.mark.parametrize("logn", [12, 13])
def test_references_commute_with_oracle_ct(oracle_mod, logn):
    """ntt_ct(sigma_coeff(x)) == sigma_eval(ntt_ct(x)) with psi^bitrev tables: the evaluation-domain
    permutation matches the library's CT order; also for a second root psi^3 of the same prime."""
    n = 1 << logn
    rng = np.random.default_rng(91000 + logn)
    for q in channel_primes(2):
        qc = np.array([[q]], dtype=np.int64)
        x = rng.integers(0, q, (2, n)).astype(np.int64)
        x[0, :16], x[0, 16:32] = q - 1, 0
        for psi in (psi_of(n, q), pow(psi_of(n, q), 3, q)):
            table = oracle_mod.make_bitrev_table(n, q, psi)
            ex = oracle_mod.ntt_ct(x, table, q).astype(np.int64)
            for g in (1, 3, 5, pow(5, 77, 2 * n), pow(5, -1, 2 * n), 2 * n - 1):
                lhs = oracle_mod.ntt_ct(sigma_coeff(x[:, None], g, qc)[:, 0], table, q)
                assert np.array_equal(lhs, sigma_eval(ex, g)), (q, psi, g)


def test_galois_elements(lib):
    for n in (1 << 12, 1 << 13, 1 << 16):
        two_n = 2 * n
        assert lib.galois_rotation(n, 0) == 1 and lib.galois_rotation(n, 1) == 5
        assert lib.galois_rotation(n, n // 2) == 1          # 5 has order N/2 ...
        assert pow(5, n // 4, two_n) != 1                   # ... exactly
        for r in (1, 3, 100, n // 2 - 1):
            assert lib.galois_rotation(n, r) * lib.galois_rotation(n, -r) % two_n == 1
            assert lib.galois_rotation(n, -r) == lib.galois_rotation(n, n // 2 - r)
            assert lib.galois_rotation(n, r) * lib.galois_rotation(n, 7) % two_n == lib.galois_rotation(n, r + 7)
        assert lib.galois_conjugate(n) == two_n - 1
        assert lib.galois_conjugate(n) ** 2 % two_n == 1
    # the references compose like the group: sigma_g sigma_h = sigma_gh, conjugation an involution
    n, q = 1 << 12, channel_primes(1)[0]
    qc = np.array([[q]], dtype=np.int64)
    x = np.random.default_rng(5).integers(0, q, (1, n)).astype(np.int64)
    g, h = lib.galois_rotation(n, 3), lib.galois_rotation(n, -11)
    assert np.array_equal(sigma_coeff(sigma_coeff(x, h, qc), g, qc), sigma_coeff(x, g * h % (2 * n), qc))
    assert np.array_equal(sigma_eval(sigma_eval(x, h), g), sigma_eval(x, g * h % (2 * n)))
    c = lib.galois_conjugate(n)
    assert np.array_equal(sigma_coeff(sigma_coeff(x, c, qc), c, qc), x)


# ------------------------------------------------------------------------- GPU helpers
def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"
    return torch


def elements(n, seed):
    """1, 5, 5^-1, 2N - 1 and a random odd g"""
    rng = np.random.default_rng(seed)
    return [1, 5, pow(5, -1, 2 * n), 2 * n - 1, int(rng.integers(0, n)) * 2 + 1]


def reference(x, gs, qs, domain):
    """x: uint64 [rows, L, N] -> [len(gs), rows, L, N]"""
    q = np.array(qs, dtype=np.uint64)[:, None]
    return np.stack([sigma_eval(x, g) if domain == EVAL else sigma_coeff(x, g, q) for g in gs])


# --------------------------------------------------------------- GPU: against numpy
CASES = [(logn, limbs, batch) for logn in (12, 13, 14, 15, 16) for limbs in (1, 3, 32) for batch in (1, 5, "l2")]


@pytest.mark.gpu
@pytest.mark.parametrize("logn,limbs,batch", CASES)
def test_automorphism(lib, logn, limbs, batch):
    """Both domains against numpy for count 1 (each of 1, 5, 5^-1, 2N-1, a random g), 3 and 64;
    inputs pinned at 0 and q - 1; guard bands around the output; the input unchanged; one launch
    per call.  batch "l2" makes the input 256 MiB, twice the L2."""
    torch = _torch()
    n = 1 << logn
    if batch == "l2":
        batch = L2_WORDS // (limbs * n)
    qs = channel_primes(limbs)
    seed = 92000 + 100 * logn + limbs
    words = batch * limbs * n
    x = rand_rns((batch, limbs, n), qs, seed)
    rows = rows_of(batch, seed)
    hx = host(x, rows)
    gs = elements(n, seed)
    rng = np.random.default_rng(seed)
    g64 = gs + [int(v) * 2 + 1 for v in rng.integers(0, n, 64 - len(gs))]
    calls = [[g] for g in gs] + [gs[1:4], g64]
    with ones_plan(lib, logn, qs) as rp:
        for domain in (COEFF, EVAL):
            for elems in calls:
                out = Guarded(len(elems) * words)
                before = lib.kernel_launches()
                rp.automorphism(x, out.view, batch, elems, domain)
                assert lib.kernel_launches() == before + 1
                got = out.view.view(len(elems), batch, limbs, n)[:, rows].cpu().numpy().astype(np.uint64)
                assert np.array_equal(got, reference(hx, elems, qs, domain)), (domain, elems[:3])
                assert out.guards_intact(), (domain, len(elems))
                del out
        assert np.array_equal(host(x, rows), hx)
        before = lib.kernel_launches()
        rp.automorphism(0, 0, 0, 5)
        assert lib.kernel_launches() == before


# ------------------------------------------------------------- GPU: commutation, group
@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 13, 14, 15, 16])
def test_commutes_with_transforms(lib, logn):
    """rns_ct . sigma_coeff == sigma_eval . rns_ct and rns_gs_scaled . sigma_eval == sigma_coeff .
    rns_gs_scaled bit for bit; sigma_g . sigma_h == sigma_gh and conjugation twice is the
    identity in both domains."""
    torch = _torch()
    n, limbs, batch = 1 << logn, 3, 2
    qs = channel_primes(limbs)
    fwd, inv, _ = channel_tables(lib, n, qs)
    gs = elements(n, 93000 + logn)
    k = len(gs)
    x = rand_rns((batch, limbs, n), qs, 93000 + logn)
    y = rand_rns((batch, limbs, n), qs, 93100 + logn)
    with lib.RnsPlan(qs, fwd, logn=logn) as pf, lib.RnsPlan(qs, inv, logn=logn) as pi:
        sx = torch.empty((k, batch, limbs, n), dtype=torch.int32, device="cuda")
        lhs, ex, rhs = torch.empty_like(sx), torch.empty_like(x), torch.empty_like(sx)
        pf.automorphism(x, sx, batch, gs, COEFF)
        pf.ct(sx, lhs, k * batch)
        pf.ct(x, ex, batch)
        pf.automorphism(ex, rhs, batch, gs, EVAL)
        assert torch.equal(lhs, rhs)
        pi.automorphism(y, sx, batch, gs, EVAL)    # either plan of the pair will do
        pi.gs_scaled(sx, lhs, k * batch)
        py = torch.empty_like(y)
        pi.gs_scaled(y, py, batch)
        pi.automorphism(py, rhs, batch, gs, COEFF)
        assert torch.equal(lhs, rhs)
        g, h, c = lib.galois_rotation(n, 5), lib.galois_rotation(n, -9), lib.galois_conjugate(n)
        for domain in (COEFF, EVAL):
            one, two, gh = torch.empty_like(x), torch.empty_like(x), torch.empty_like(x)
            pf.automorphism(x, one, batch, h, domain)
            pf.automorphism(one, two, batch, g, domain)
            pf.automorphism(x, gh, batch, g * h % (2 * n), domain)
            assert torch.equal(two, gh), domain
            pf.automorphism(x, one, batch, c, domain)
            pf.automorphism(one, two, batch, c, domain)
            assert torch.equal(two, x), domain
            pf.automorphism(x, one, batch, 1, domain)
            assert torch.equal(one, x), domain


# ---------------------------------------------------------------------- buffer rules
@pytest.mark.gpu
def test_buffers_and_errors(lib):
    """Overlap and in place -> INVALID_ARG, views 4/8/12 bytes past alignment -> UNSUPPORTED,
    bad elements, counts and domains -> INVALID_ARG; nothing written, nothing launched."""
    torch = _torch()
    logn, batch, limbs = 13, 3, 3
    n = 1 << logn
    qs = channel_primes(limbs)
    words = batch * limbs * n
    x = rand_rns((batch, limbs, n), qs, 94000)
    with ones_plan(lib, logn, qs) as rp:
        before = lib.kernel_launches()
        big = Guarded(3 * words, data=torch.cat([x.reshape(-1)] * 3))
        snap = big.raw.clone()
        bad = [lambda: rp.automorphism(big.view[:words], big.view[:words], batch, 5),
               lambda: rp.automorphism(big.view[:words], big.view[words - 4:2 * words - 4], batch, 5),
               lambda: rp.automorphism(big.view[words:2 * words], big.view[4:words + 4], batch, 5, COEFF),
               lambda: rp.automorphism(big.view[words:2 * words], big.view[:2 * words], batch, [5, 3])]
        for i, call in enumerate(bad):
            assert _status(lib, call) == INVALID_ARG, i
        for k in (1, 2, 3):
            for ki, ko in ((k, 0), (0, k)):
                ui, uo = Guarded(words, ki, x), Guarded(2 * words, ko)
                si = ui.raw.clone()
                for domain in (COEFF, EVAL):
                    assert _status(lib, lambda: rp.automorphism(ui.view, uo.view, batch, [5, 7], domain)) \
                        == UNSUPPORTED, (k, ki, ko, domain)
                torch.cuda.synchronize()
                assert uo.untouched() and torch.equal(ui.raw, si)
        out = Guarded(words)
        for gs in ([2], [0], [2 * n], [2 * n + 1], [1 << 31 | 1], [5, 4]):
            assert _status(lib, lambda: rp.automorphism(x, out.view, batch, gs)) == INVALID_ARG, gs
            assert _status(lib, lambda: rp.automorphism(x, out.view, 0, gs)) == INVALID_ARG, gs
        assert _status(lib, lambda: rp.automorphism(x, out.view, batch, [])) == INVALID_ARG
        assert _status(lib, lambda: rp.automorphism(x, out.view, batch, [5] * 65)) == INVALID_ARG
        for domain in (2, 7):
            assert _status(lib, lambda: rp.automorphism(x, out.view, batch, 5, domain)) == INVALID_ARG
        L = lib.load_library()
        g1 = (ctypes.c_uint32 * 1)(5)
        assert L.nttb200_rns_automorphism(rp._h, None, out.view.data_ptr(), batch, g1, 1, EVAL, None) == INVALID_ARG
        assert L.nttb200_rns_automorphism(rp._h, x.data_ptr(), None, batch, g1, 1, EVAL, None) == INVALID_ARG
        assert L.nttb200_rns_automorphism(rp._h, None, None, 0, g1, 1, EVAL, None) == OK
        assert L.nttb200_rns_automorphism(rp._h, None, None, 0, g1, 1, COEFF, None) == OK
        assert lib.kernel_launches() == before
        torch.cuda.synchronize()
        assert torch.equal(big.raw, snap) and out.untouched()
        rp.automorphism(x, out.view, batch, 5)   # still usable
        want = reference(host(x), [5], qs, EVAL)[0]
        assert np.array_equal(host(out.view.view(x.shape)), want) and out.guards_intact()


@pytest.mark.gpu
def test_beyond_2_31_words(lib):
    """One call over 2^31 + 2^16 words (L = 1, N = 2^16, batch 2^15 + 1: 8 GiB in, 8 GiB out) in
    each domain, checked on sampled polynomials including the last."""
    torch = _torch()
    logn, batch = 16, (1 << 15) + 1
    n = 1 << logn
    qs = channel_primes(1)
    gen = torch.Generator(device="cuda").manual_seed(95000)
    x = torch.randint(0, qs[0], (batch, 1, n), dtype=torch.int32, device="cuda", generator=gen)
    out = torch.empty_like(x)
    rows = np.array([0, 1, batch // 2, batch - 2, batch - 1])
    hx = host(x, rows)
    g = lib.galois_rotation(n, 3)
    with ones_plan(lib, logn, qs) as rp:
        for domain in (EVAL, COEFF):
            rp.automorphism(x, out, batch, g, domain)
            assert np.array_equal(host(out, rows), reference(hx, [g], qs, domain)[0]), domain


# ------------------------------------------------------------- GPU: end-to-end rotation
def negamul(a, s, q):
    """a * s mod (X^N + 1, q) for a in [0, q) and a small integer s (int64 numpy, exact)"""
    n = len(a)
    full = np.convolve(a.astype(np.int64), s.astype(np.int64))
    r = full[:n].copy()
    r[:n - 1] -= full[n:]
    return r % q


class Rotation:
    """RLWE ciphertexts mod Q = 3 primes, one special prime P > max(Q), digit i = channel i, and
    the key-switching sequence of INTEGRATION.md built from the library's primitives."""

    def __init__(self, lib, logn, seed):
        torch = _torch()
        self.lib, self.torch = lib, torch
        self.n = n = 1 << logn
        primes = channel_primes(4)
        self.P, self.Q = primes[0], primes[1:]
        self.QP = self.Q + [self.P]
        self.rng = np.random.default_rng(seed)
        fq, iq, _ = channel_tables(lib, n, self.Q)
        fqp, iqp, _ = channel_tables(lib, n, self.QP)
        self.qf, self.qi = lib.RnsPlan(self.Q, fq, logn=logn), lib.RnsPlan(self.Q, iq, logn=logn)
        self.pf, self.pi = lib.RnsPlan(self.QP, fqp, logn=logn), lib.RnsPlan(self.QP, iqp, logn=logn)
        # ModUp of digit i: {q_i} -> the other Q primes and P; ModDown: P -> Q
        self.up = []
        for i, qv in enumerate(self.Q):
            rest = [m for j, m in enumerate(self.Q) if j != i] + [self.P]
            with ones_plan(lib, logn, [qv]) as a, ones_plan(lib, logn, rest) as b:
                self.up.append(lib.RnsConv(a, b))
        with ones_plan(lib, logn, [self.P]) as a, ones_plan(lib, logn, self.Q) as b:
            self.down = lib.RnsConv(a, b)
        self.s = self.rng.integers(-1, 2, n).astype(np.int64)
        self.keys = {}

    def dev(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a).astype(np.int32)).cuda()

    def encrypt(self, m):
        """(c0, c1) in the NTT domain on the Q plan: [2][3][N]"""
        e = self.rng.integers(-20, 21, self.n)
        c1 = np.stack([self.rng.integers(0, q, self.n) for q in self.Q])
        c0 = np.stack([(m + e - negamul(c1[j], self.s, q)) % q for j, q in enumerate(self.Q)])
        ct = self.dev(np.stack([c0, c1]))
        self.qf.ct(ct, ct, 2)
        return ct

    def decrypt(self, ct):
        """centred integers of c0 + c1 s mod Q (ct in the NTT domain, [2][3][N])"""
        c = self.torch.empty_like(ct)
        self.qi.gs_scaled(ct, c, 2)
        c = c.cpu().numpy().astype(np.int64)
        res = [(c[0, j] + negamul(c[1, j], self.s, q)) % q for j, q in enumerate(self.Q)]
        Qp = math.prod(self.Q)
        basis = [(Qp // q) * pow(Qp // q % q, -1, q) for q in self.Q]
        out = []
        for k in range(self.n):
            v = sum(int(res[j][k]) * basis[j] for j in range(3)) % Qp
            out.append(v - Qp if v > Qp // 2 else v)
        return np.array(out, dtype=object)

    def galois_key(self, g):
        """NTT-domain (b_i, a_i) on QP with b_i + a_i s = e_i + P g_i sigma_g(s), g_i the CRT gadget
        (Q/q_i) [(Q/q_i)^-1]_{q_i}: ([3][1][4][N], [3][1][4][N])"""
        if g not in self.keys:
            Qp = math.prod(self.Q)
            sg = sigma_int(self.s, g)
            b = np.zeros((3, 4, self.n), dtype=np.int64)
            a = np.zeros((3, 4, self.n), dtype=np.int64)
            for i, qv in enumerate(self.Q):
                gadget = self.P * (Qp // qv) * pow(Qp // qv % qv, -1, qv)
                e = self.rng.integers(-20, 21, self.n)
                for j, m in enumerate(self.QP):
                    a[i, j] = self.rng.integers(0, m, self.n)
                    b[i, j] = (e - negamul(a[i, j], self.s, m) + gadget % m * (sg % m)) % m
            kb, ka = self.dev(b), self.dev(a)
            self.pf.ct(kb, kb, 3)
            self.pf.ct(ka, ka, 3)
            self.keys[g] = (kb, ka)
        return self.keys[g]

    def mod_up(self, c1):
        """coefficients [1][3][N] -> NTT-domain digits [3][1][4][N] on QP"""
        torch = self.torch
        d = torch.empty((3, 1, 4, self.n), dtype=torch.int32, device="cuda")
        tmp = torch.empty((1, 3, self.n), dtype=torch.int32, device="cuda")
        for i in range(3):
            self.up[i].convert(c1[:, i], tmp, 1)
            rest = [j for j in range(3) if j != i] + [3]
            d[i, 0, i] = c1[0, i]
            d[i, 0, rest] = tmp[0]
        self.pf.ct(d, d, 3)
        return d

    def switch(self, s0, digits, g):
        """steps 5-9: sigma(c0) in the NTT domain [1][3][N], NTT-domain digits [3][1][4][N] of
        sigma(c1) under sigma(s) -> the ciphertext [2][3][N] under s"""
        torch = self.torch
        kb, ka = self.galois_key(g)
        u = torch.empty((2, 4, self.n), dtype=torch.int32, device="cuda")
        self.lib.rns_dot(self.pf, digits, kb, u[0:1], 3, 1, w_batch=1)
        self.lib.rns_dot(self.pf, digits, ka, u[1:2], 3, 1, w_batch=1)
        self.pi.gs_scaled(u, u, 2)
        v = torch.empty((2, 3, self.n), dtype=torch.int32, device="cuda")
        self.down.mod_down(u, v, 2, round=True)
        self.qf.ct(v, v, 2)
        self.qf.pointwise(ADD, v[0:1], s0, v[0:1], 1)
        return v

    def rotate(self, ct, g, coeff_route=False):
        """steps 1-9 for one element g; the coefficient-domain route applies sigma to the
        coefficients of c1 instead of step 1 on c1.  Returns the ciphertext and sigma(c1)."""
        torch = self.torch
        s0, s1, sc1 = (torch.empty((1, 3, self.n), dtype=torch.int32, device="cuda") for _ in range(3))
        self.qf.automorphism(ct[0:1], s0, 1, g)
        if coeff_route:
            self.qi.gs_scaled(ct[1:2], s1, 1)
            self.qi.automorphism(s1, sc1, 1, g, COEFF)
        else:
            self.qf.automorphism(ct[1:2], s1, 1, g)
            self.qi.gs_scaled(s1, sc1, 1)
        return self.switch(s0, self.mod_up(sc1), g), sc1

    def rotate_hoisted(self, ct, gs):
        torch = self.torch
        c1 = torch.empty((1, 3, self.n), dtype=torch.int32, device="cuda")
        self.qi.gs_scaled(ct[1:2], c1, 1)
        digits = self.mod_up(c1)
        r = len(gs)
        rot = torch.empty((r, 3, 1, 4, self.n), dtype=torch.int32, device="cuda")
        self.pf.automorphism(digits, rot, 3, gs)   # [r][dnum][batch][L+K][N]
        s0 = torch.empty((r, 1, 3, self.n), dtype=torch.int32, device="cuda")
        self.qf.automorphism(ct[0:1], s0, 1, gs)
        return [self.switch(s0[c], rot[c], g) for c, g in enumerate(gs)]

    def close(self):
        for x in [self.qf, self.qi, self.pf, self.pi, self.down] + self.up:
            x.close()


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 13])
def test_end_to_end_rotation(lib, logn):
    """Rotation by one slot and conjugation of an RLWE ciphertext decrypt to sigma_g(m) within the
    key-switching noise bound; the hoisted form (one ModUp, count = 3) as well; the
    coefficient-domain route gives a bit-identical ciphertext."""
    torch = _torch()
    rot = Rotation(lib, logn, 96000 + logn)
    n = rot.n
    bound = 1 << 22
    m = rot.rng.integers(-(1 << 40), 1 << 40, n).astype(np.int64)
    ct = rot.encrypt(m)
    dec = rot.decrypt(ct)
    assert max(abs(int(v)) for v in dec - m.astype(object)) <= 20
    mo = m.astype(object)
    g_rot, g_back, g_conj = lib.galois_rotation(n, 1), lib.galois_rotation(n, -3), lib.galois_conjugate(n)
    singles = {}
    for g in (g_rot, g_conj):
        out, sc1 = rot.rotate(ct, g)
        err = max(abs(int(v)) for v in rot.decrypt(out) - sigma_int(mo, g))
        assert err < bound, (g, err)
        out_c, sc1_c = rot.rotate(ct, g, coeff_route=True)
        assert torch.equal(sc1_c, sc1) and torch.equal(out_c, out), g
        singles[g] = out
    hoisted = rot.rotate_hoisted(ct, [g_rot, g_back, g_conj])
    for g, out in zip((g_rot, g_back, g_conj), hoisted):
        err = max(abs(int(v)) for v in rot.decrypt(out) - sigma_int(mo, g))
        assert err < bound, (g, err)
    rot.close()
