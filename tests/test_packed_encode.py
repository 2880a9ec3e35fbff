"""Packed integer slots mod t for BFV and BGV: nttb200_packed_encode / nttb200_packed_decode.
On the CPU: a numpy reference written from the convention in include/nttb200.h, checked against
direct evaluation m(psi^e) mod t and against the oracle's CT order, the rotation and row-swap
identities on it, the lift formulas against Python-int round(Q m / t), and the null-argument checks.
On the GPU: encode (both forms) and decode against the reference, the round trips through the
BFV and BGV decryption steps, rotations and the row swap through `automorphism`, end-to-end BFV
and BGV products, the buffer rules, the launch counts and one call over 2^31 output words."""
import ctypes
import math

import numpy as np
import pytest

from test_ckks_encode import negacyclic_sigma
from test_rns_eval import Guarded, _status, channel_tables, host, ones_plan, rows_of
from test_rns_sizes import ntt_primes

OK, INVALID_ARG, MODULUS, UNSUPPORTED = 0, 1, 2, 7
SCALED, CENTRED = 0, 1
L2_BYTES = 160 << 20     # more than the B200's 126 MB L2
SPECIAL = [-(1 << 31), (1 << 31) - 1, -1, 0]   # then t - 1 and t


# ------------------------------------------------------------------------- numpy reference
def is_prime(t):
    return t >= 2 and all(t % d for d in range(2, math.isqrt(t) + 1))


def valid_t(logn, largest=False):
    """The smallest or the largest prime t < 2^30 with t = 1 (mod 2N)."""
    two_n = 2 << logn
    ks = range((2 ** 30 - 2) // two_n, 0, -1) if largest else range(1, 2 ** 30 // two_n)
    return next(k * two_n + 1 for k in ks if is_prime(k * two_n + 1))


def channels(L, t, edge=False):
    """L NTT-friendly primes below 2^30 other than t; with edge, 2^30 and 3 first."""
    qs = [q for q in ntt_primes(L + 1) if q != t]
    return ([1 << 30, 3] + qs)[:L] if edge else qs[:L]


def powers(x, count, t):
    out = np.empty(count, dtype=np.int64)
    v = 1
    for i in range(count):
        out[i] = v
        v = v * x % t
    return out


def brev(x, bits):
    return int(format(x, f"0{bits}b")[::-1], 2)


def smallest_psi(N, t):
    x = 2
    while pow(x, (t - 1) // 2, t) != t - 1:
        x += 1
    psi0 = pow(x, (t - 1) // (2 * N), t)
    return int(np.min(powers(psi0 * psi0 % t, N, t) * psi0 % t))


def slot_exponents(N):
    """e_i: 5^j mod 2N for row 0, 2N - (5^j mod 2N) for row 1."""
    g = np.array([pow(5, j, 2 * N) for j in range(N // 2)], dtype=np.int64)
    return np.concatenate([g, 2 * N - g])


def dft_mod(x, w, t):
    """X_k = sum_c x_c w^(ck) mod t along the last axis (iterative radix-2, int64)."""
    N = x.shape[-1]
    logn = N.bit_length() - 1
    perm = np.array([brev(i, logn) for i in range(N)]) if logn else np.zeros(1, dtype=np.int64)
    a = x[..., perm] % t
    wp = powers(w, N // 2, t)
    lead = a.shape[:-1]
    m = 2
    while m <= N:
        a = a.reshape(lead + (N // m, m))
        o = a[..., m // 2:] * wp[::N // m][:m // 2] % t
        e = a[..., :m // 2]
        a = np.concatenate([(e + o) % t, (e - o) % t], axis=-1).reshape(lead + (N,))
        m *= 2
    return a


class Ref:
    """Encode and decode of one ring degree N and plaintext modulus t, from the convention."""

    def __init__(self, N, t):
        self.N, self.t = N, t
        self.psi = smallest_psi(N, t)
        psi_inv = pow(self.psi, -1, t)
        self.w, self.w_inv = self.psi * self.psi % t, psi_inv * psi_inv % t
        self.twist, self.untwist = powers(self.psi, N, t), powers(psi_inv, N, t)
        self.n_inv = pow(N, -1, t)
        self.pos = (slot_exponents(N) - 1) // 2      # v_j = m(psi^(2j + 1)): slot i is v_pos[i]
        logn = N.bit_length() - 1
        self.k = np.array([brev(int(p), logn) for p in self.pos])   # index in the rns_ct order

    def decode(self, m):
        """m int [..., N] (any integers) -> slots in [0, t)."""
        return dft_mod(np.asarray(m, dtype=np.int64) % self.t * self.twist % self.t, self.w, self.t)[..., self.pos]

    def encode(self, s):
        """s int [..., N] (any integers) -> m in [0, t) with decode(m) = s mod t."""
        s = np.asarray(s, dtype=np.int64)
        v = np.empty_like(s)
        v[..., self.pos] = s % self.t
        y = dft_mod(v, self.w_inv, self.t) * self.n_inv % self.t
        return y * self.untwist % self.t


def centre(m, t):
    return np.where(m > t // 2, m - t, m)


def lift(m, qs, t, centred):
    """The documented lift in int64: (delta_l m + rho) mod q_l, or m_c mod q_l; [..., L, N]."""
    m = np.asarray(m, dtype=np.int64)
    if centred:
        mc = centre(m, t)
        return np.stack([mc % q for q in qs], axis=-2)
    r = math.prod(qs) % t
    rho = (r * m + t // 2) // t
    return np.stack([((-r * pow(t, -1, q)) % q * m + rho) % q for q in qs], axis=-2)


def rows_rotated(s, r):
    N = s.shape[-1]
    return np.roll(s.reshape(s.shape[:-1] + (2, N // 2)), -r, axis=-1).reshape(s.shape)


def rows_swapped(s):
    N = s.shape[-1]
    return np.concatenate([s[..., N // 2:], s[..., :N // 2]], axis=-1)


# ------------------------------------------------------------------ CPU: the reference itself
@pytest.mark.parametrize("largest", [False, True])
def test_reference_matches_direct_evaluation(largest):
    """N = 4096: slot i of decode equals m(psi^e_i) mod t evaluated with Python ints, on sampled
    slots of both rows; psi is the least primitive 2N-th root; encode inverts decode."""
    N = 4096
    t = valid_t(12, largest)
    ref = Ref(N, t)
    assert pow(ref.psi, N, t) == t - 1
    assert min(pow(ref.psi, 2 * i + 1, t) for i in range(N)) == ref.psi
    rng = np.random.default_rng(3 + largest)
    m = rng.integers(0, t, N)
    s = ref.decode(m)
    e = slot_exponents(N)
    for i in [0, 1, 2, 5, 1000, N // 2 - 1, N // 2, N // 2 + 1, N // 2 + 777, N - 1]:
        pe = pow(ref.psi, int(e[i]), t)
        want = 0
        for c in reversed(range(N)):
            want = (want * pe + int(m[c])) % t
        assert int(s[i]) == want, i
    assert np.array_equal(ref.encode(s), m)
    x = rng.integers(-2 ** 31, 2 ** 31, N)
    assert np.array_equal(ref.decode(ref.encode(x)), x % t)


@pytest.mark.parametrize("logn", [12, 13])
def test_reference_order_is_oracle_ct_order(oracle_mod, logn):
    """The oracle's CT network on a psi^bitrev table holds slot i at index brev((e_i - 1) / 2)."""
    N = 1 << logn
    t = valid_t(logn, True)
    ref = Ref(N, t)
    m = np.random.default_rng(logn).integers(0, t, (2, N))
    ct = oracle_mod.ntt_ct(m, oracle_mod.make_bitrev_table(N, t, ref.psi), t).astype(np.int64)
    assert np.array_equal(ct[:, ref.k], ref.decode(m))


@pytest.mark.parametrize("r", [1, -1, 7, 1024])
def test_reference_rotation_and_row_swap(lib, r):
    """sigma_(5^r) rotates both rows left by r, sigma_(2N - 1) swaps them."""
    N = 4096
    t = valid_t(12)
    ref = Ref(N, t)
    m = np.random.default_rng(8).integers(0, t, N)
    s = ref.decode(m)
    assert np.array_equal(ref.decode(negacyclic_sigma(m, lib.galois_rotation(N, r))), rows_rotated(s, r))
    assert np.array_equal(ref.decode(negacyclic_sigma(m, lib.galois_conjugate(N))), rows_swapped(s))


@pytest.mark.parametrize("largest", [False, True])
def test_lift_against_python_ints(largest):
    """(delta_l m + rho) mod q_l = round(Q m / t) mod q_l and m_c mod q_l, channels including 2, 3,
    2^30 and composites coprime to t; m at 0, 1, (t - 1) / 2, (t + 1) / 2, t - 1 and random."""
    t = valid_t(14, largest)
    qs = [1 << 30, 3, 2, 1 << 29, 999999999] + [q for q in ntt_primes(6) if q != t][:5]
    Q = math.prod(qs)
    m = np.concatenate([[0, 1, (t - 1) // 2, (t + 1) // 2, t - 1],
                        np.random.default_rng(9 + largest).integers(0, t, 3000)])
    got, gotc = lift(m, qs, t, False), lift(m, qs, t, True)
    for c, v in enumerate(m.tolist()):
        want = (2 * Q * v + t) // (2 * t)
        assert abs(Q * v - t * want) * 2 < t
        vc = v - t if v > t // 2 else v
        for l, q in enumerate(qs):
            assert got[l, c] == want % q and gotc[l, c] == vc % q


def test_null_arguments_without_device(lib):
    L = lib.load_library()
    h = ctypes.c_void_p()
    assert L.nttb200_packed_encoder_create(None, None, 65537, 0) == INVALID_ARG
    assert L.nttb200_packed_encoder_create(ctypes.byref(h), None, 65537, 0) == INVALID_ARG and not h.value
    assert L.nttb200_packed_encoder_destroy(None) == OK
    for mode in (SCALED, CENTRED, 2):
        assert L.nttb200_packed_encode(None, 16, mode, 16, 1, None) == INVALID_ARG
        assert L.nttb200_packed_encode(None, None, mode, None, 0, None) == INVALID_ARG
        assert L.nttb200_packed_decode(None, 16, mode, 16, 1, None) == INVALID_ARG
        assert L.nttb200_packed_decode(None, None, mode, None, 0, None) == INVALID_ARG
    assert (lib.PACK_SCALED, lib.PACK_CENTRED) == (SCALED, CENTRED)


# ------------------------------------------------------------------------------ GPU helpers
def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"
    return torch


def to_dev(a):
    return _torch().from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.int64) % (1 << 32))
                               .astype(np.uint32).view(np.int32)).cuda()


def rand_slots(batch, N, t, seed):
    """int32 [batch][N] on the device: random words of the whole int32 range, every row starting
    with INT32_MIN, INT32_MAX, -1, 0, t - 1, t."""
    torch = _torch()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randint(-(1 << 31), (1 << 31) - 1, (batch, N), dtype=torch.int64, device="cuda", generator=gen)
    x[:, :6] = torch.tensor(SPECIAL + [t - 1, t], dtype=torch.int64, device="cuda")
    return x.to(torch.int32)


def signed(x, rows=None):
    y = x if rows is None else x[rows]
    return y.cpu().numpy().astype(np.int64)


def batch_of(batch, N, L):
    return L2_BYTES // (4 * N * (L + 1)) + 1 if batch == "l2" else batch


def encode_launches(logn):
    return 3 if logn == 12 else 4


def decode_launches(logn):
    return 2 if logn == 12 else 3


ENCODE_CASES = [(logn, L, batch) for logn in (12, 13, 14, 15, 16) for L in (1, 3, 32) for batch in (1, 5, "l2")]


@pytest.mark.gpu
@pytest.mark.parametrize("logn,L,batch", ENCODE_CASES)
def test_encode(lib, logn, L, batch):
    """Both forms against the reference on every channel, for the smallest and the largest t; the
    3-channel set is {2^30, 3, q}."""
    torch = _torch()
    N = 1 << logn
    batch = batch_of(batch, N, L)
    rows = rows_of(batch, logn)
    for largest in (False, True):
        t = valid_t(logn, largest)
        qs = channels(L, t, edge=L == 3)
        ref = Ref(N, t)
        d_s = rand_slots(batch, N, t, 100 * logn + L + largest)
        out = torch.empty((batch, L, N), dtype=torch.int32, device="cuda")
        m = ref.encode(signed(d_s, rows))
        with lib.PackedEncoder(ones_plan(lib, logn, qs), t) as enc:
            for centred in (False, True):
                l0 = lib.kernel_launches()
                enc.encode(d_s, out, batch, centred=centred)
                torch.cuda.synchronize()
                assert lib.kernel_launches() - l0 == encode_launches(logn)
                assert np.array_equal(host(out, rows), lift(m, qs, t, centred)), (t, centred)


DECODE_CASES = [(logn, batch) for logn in (12, 13, 14, 15, 16) for batch in (1, 5, "l2")]


@pytest.mark.gpu
@pytest.mark.parametrize("logn,batch", DECODE_CASES)
def test_decode(lib, logn, batch):
    """Canonical residues mod t in, slots in [0, t) and centred out, for the smallest and the
    largest t; rows of t - 1 and of 0 included."""
    torch = _torch()
    N = 1 << logn
    batch = batch_of(batch, N, 1)
    rows = rows_of(batch, logn)
    for largest in (False, True):
        t = valid_t(logn, largest)
        ref = Ref(N, t)
        gen = torch.Generator(device="cuda").manual_seed(logn * 3 + largest)
        x = torch.randint(0, t, (batch, N), dtype=torch.int32, device="cuda", generator=gen)
        x[0, :N // 2], x[-1, N // 2:] = t - 1, 0
        want = ref.decode(signed(x, rows))
        z = torch.empty_like(x)
        with lib.PackedEncoder(ones_plan(lib, logn, channels(2, t)), t) as enc:
            for centred in (False, True):
                l0 = lib.kernel_launches()
                enc.decode(x, z, batch, centred=centred)
                torch.cuda.synchronize()
                assert lib.kernel_launches() - l0 == decode_launches(logn)
                assert np.array_equal(signed(z, rows), centre(want, t) if centred else want), (t, centred)


def decrypt_to_t(lib, x, qs, t, bfv):
    """Plaintext residues mod t of X on the channels qs (coefficient domain, [batch][L][N]): BFV
    round(t X / Q) through rns_scale by t, convert exact to {t} and rns_scale by -Q^-1 mod t;
    BGV X_c mod t through convert exact."""
    torch = _torch()
    batch, _, N = x.shape
    logn = N.bit_length() - 1
    mt = torch.empty((batch, 1, N), dtype=torch.int32, device="cuda")
    with ones_plan(lib, logn, qs) as pq, ones_plan(lib, logn, [t]) as ptt, lib.RnsConv(pq, ptt) as to_t:
        if bfv:
            xs = torch.empty_like(x)
            pq.scale(x, xs, batch, [t % q for q in qs])
            to_t.convert(xs, mt, batch, exact=True)
            ptt.scale(mt, mt, batch, [(-pow(math.prod(qs), -1, t)) % t])
        else:
            to_t.convert(x, mt, batch, exact=True)
    return mt


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 13, 14, 15, 16])
def test_round_trips(lib, logn):
    """With zero noise: CENTRED encode -> convert exact to {t} -> decode, and SCALED encode -> the
    BFV decryption steps -> decode, both give the slots mod t back."""
    torch = _torch()
    N, batch = 1 << logn, 3
    t = valid_t(logn, True)
    qs = channels(3, t)
    s = rand_slots(batch, N, t, 500 + logn)
    want = signed(s) % t
    out = torch.empty((batch, 3, N), dtype=torch.int32, device="cuda")
    z = torch.empty_like(s)
    with lib.PackedEncoder(ones_plan(lib, logn, qs), t) as enc:
        for bfv in (False, True):
            enc.encode(s, out, batch, centred=not bfv)
            mt = decrypt_to_t(lib, out, qs, t, bfv)
            enc.decode(mt, z, batch)
            assert np.array_equal(signed(z), want), bfv


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 14, 16])
def test_rotation_and_row_swap_through_automorphism(lib, logn):
    """automorphism by galois_rotation(N, r) rotates both rows left by r, galois_conjugate(N) swaps
    them, on coefficients and in the rns_ct order (plans on psi^bitrev / psi^-bitrev tables)."""
    torch = _torch()
    N, batch = 1 << logn, 2
    t = valid_t(logn)
    qs = channels(3, t)
    s = rand_slots(batch, N, t, 600 + logn)
    want0 = signed(s) % t
    rs = [1, -1, 7, N // 4]
    gs = [lib.galois_rotation(N, r) for r in rs] + [lib.galois_conjugate(N)]
    want = [rows_rotated(want0, r) for r in rs] + [rows_swapped(want0)]
    fwd, inv, _ = channel_tables(lib, N, qs)
    a = torch.empty((batch, 3, N), dtype=torch.int32, device="cuda")
    coeff = torch.empty((len(gs), batch, 3, N), dtype=torch.int32, device="cuda")
    ev, evo = torch.empty_like(a), torch.empty_like(coeff)
    back, z = torch.empty_like(a), torch.empty_like(s)
    with lib.RnsPlan(qs, fwd, logn=logn) as pf, lib.RnsPlan(qs, inv, logn=logn) as pi, \
            lib.PackedEncoder(pf, t) as enc:
        enc.encode(s, a, batch, centred=True)
        pf.automorphism(a, coeff, batch, gs, domain=lib.AUTO_COEFF)
        pf.ct(a, ev, batch)
        pf.automorphism(ev, evo, batch, gs, domain=lib.AUTO_EVAL)
        for i, w in enumerate(want):
            enc.decode(decrypt_to_t(lib, coeff[i], qs, t, False), z, batch)
            assert np.array_equal(signed(z), w), ("coeff", gs[i])
            pi.gs_scaled(evo[i], back, batch)
            enc.decode(decrypt_to_t(lib, back, qs, t, False), z, batch)
            assert np.array_equal(signed(z), w), ("eval", gs[i])


class Keys:
    """Host-drawn secret, noise and uniform a; products through rns_polymul_negacyclic on Q."""

    def __init__(self, lib, logn, qs, seed):
        self.lib, self.N, self.qs = lib, 1 << logn, qs
        self.rng = np.random.default_rng(seed)
        fwd, inv, _ = channel_tables(lib, self.N, qs)
        self.qfwd, self.qinv = fwd, inv
        self.pf = lib.RnsPlan(qs, fwd, logn=logn)
        self.pi = lib.RnsPlan(qs, inv, logn=logn)
        self.s = self.rng.integers(-1, 2, self.N)
        self.s_res = to_dev(np.stack([self.s % q for q in qs])[None])

    def mul(self, a, b):
        """a (*) b mod (X^N + 1, q_l), [batch][L][N] each."""
        c = _torch().empty_like(a)
        self.lib.rns_polymul_negacyclic(self.pf, self.pi, a, b, c, a.shape[0])
        return c

    def encrypt(self, pt, noise_mult):
        """(c0, c1) = (-a s + noise_mult e + pt, a) mod Q, [2][L][N]."""
        torch = _torch()
        qcol = np.array(self.qs, dtype=np.int64)[:, None]
        a = np.stack([self.rng.integers(0, q, self.N) for q in self.qs])
        e = self.rng.integers(-4, 5, self.N) * noise_mult
        a_s = signed(self.mul(to_dev(a[None]), self.s_res))[0]
        c0 = (signed(pt)[0] + e % qcol - a_s) % qcol
        return torch.stack([to_dev(c0), to_dev(a)])

    def decrypt(self, d):
        """X = d0 + d1 s + d2 s^2 + ... mod Q, [1][L][N]."""
        torch = _torch()
        x = d[0:1].clone()
        sp = self.s_res
        for i in range(1, d.shape[0]):
            term = self.mul(d[i:i + 1], sp)
            self.pf.pointwise(self.lib.RNS_ADD, x, term, x, 1)
            if i + 1 < d.shape[0]:
                sp = self.mul(sp, self.s_res)
        return x

    def close(self):
        self.pf.close()
        self.pi.close()


def bfv_tensor(lib, logn, t, qs, ps, qp_fwd, qp_inv, c, cp):
    """The INTEGRATION BFV multiplication on a [P | Q] plan: convert exact Q -> P, ct, tensor
    product, gs_scaled, scale_round Q -> P, convert exact P -> Q; [3][L][N]."""
    torch = _torch()
    n, Lq, K = 1 << logn, len(qs), len(ps)
    qp = torch.empty((2, K + Lq, n), dtype=torch.int32, device="cuda")
    A, Bt = torch.empty_like(qp), torch.empty_like(qp)
    d = torch.empty((3, K + Lq, n), dtype=torch.int32, device="cuda")
    dp = torch.empty((3, K, n), dtype=torch.int32, device="cuda")
    res = torch.empty((3, Lq, n), dtype=torch.int32, device="cuda")
    with lib.RnsPlan(ps + qs, qp_fwd, logn=logn) as pf, lib.RnsPlan(ps + qs, qp_inv, logn=logn) as pi, \
            ones_plan(lib, logn, qs) as pq, ones_plan(lib, logn, ps) as pp, \
            lib.RnsConv(pq, pp) as up, lib.RnsConv(pp, pq) as back:
        for ev, ct in ((A, c), (Bt, cp)):
            qp[:, K:] = ct
            up.convert(qp[:, K:], qp, 2, in_stride=(K + Lq) * n, out_stride=(K + Lq) * n, exact=True)
            pf.ct(qp, ev, 2)
        pf.pointwise(lib.RNS_MUL, A[0], Bt[0], d[0], 1)
        pf.pointwise(lib.RNS_MUL, A[0], Bt[1], d[1], 1)
        lib.rns_dot(pf, A[1], Bt[0], d[1], 1, 1, accumulate=True)
        pf.pointwise(lib.RNS_MUL, A[1], Bt[1], d[2], 1)
        pi.gs_scaled(d, d, 3)
        up.scale_round(d, dp, 3, t)
        back.convert(dp, res, 3, exact=True)
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("logn,largest", [(12, False), (14, True)])
def test_bfv_end_to_end(lib, logn, largest):
    """Encode (SCALED) -> encrypt with host keys -> the INTEGRATION multiplication -> decrypt ->
    decode equals the slotwise product mod t; a ciphertext times a CENTRED plaintext as well."""
    torch = _torch()
    N, Lq = 1 << logn, 4
    K = Lq + 2
    t = valid_t(logn, largest)
    primes = channels(Lq + K, t)
    qs, ps = primes[:Lq], primes[Lq:]
    s1, s2 = rand_slots(1, N, t, 700 + logn), rand_slots(1, N, t, 800 + logn)
    want = signed(s1) % t * (signed(s2) % t) % t
    keys = Keys(lib, logn, qs, 900 + logn)
    pt1, pt2, p2c = (torch.empty((1, Lq, N), dtype=torch.int32, device="cuda") for _ in range(3))
    z = torch.empty_like(s1)
    fwd, inv, _ = channel_tables(lib, N, ps + qs)
    with lib.PackedEncoder(keys.pf, t) as enc:
        enc.encode(s1, pt1, 1)
        enc.encode(s2, pt2, 1)
        enc.encode(s2, p2c, 1, centred=True)
        c, cp = keys.encrypt(pt1, 1), keys.encrypt(pt2, 1)
        prod = bfv_tensor(lib, logn, t, qs, ps, fwd, inv, c, cp)
        enc.decode(decrypt_to_t(lib, keys.decrypt(prod), qs, t, True), z, 1)
        assert np.array_equal(signed(z), want)
        cpt = keys.mul(c, torch.cat([p2c, p2c]))
        enc.decode(decrypt_to_t(lib, keys.decrypt(cpt), qs, t, True), z, 1)
        assert np.array_equal(signed(z), want)
    keys.close()


@pytest.mark.gpu
@pytest.mark.parametrize("logn,largest", [(12, True), (14, False)])
def test_bgv_end_to_end(lib, logn, largest):
    """Encode (CENTRED) -> encrypt with t e noise -> tensor product mod Q -> decrypt through
    convert exact Q -> {t} -> decode equals the slotwise product mod t."""
    torch = _torch()
    N, Lq = 1 << logn, 4
    t = valid_t(logn, largest)
    qs = channels(Lq, t)
    s1, s2 = rand_slots(1, N, t, 1000 + logn), rand_slots(1, N, t, 1100 + logn)
    want = signed(s1) % t * (signed(s2) % t) % t
    keys = Keys(lib, logn, qs, 1200 + logn)
    pt1, pt2 = (torch.empty((1, Lq, N), dtype=torch.int32, device="cuda") for _ in range(2))
    z = torch.empty_like(s1)
    with lib.PackedEncoder(keys.pf, t) as enc:
        enc.encode(s1, pt1, 1, centred=True)
        enc.encode(s2, pt2, 1, centred=True)
        c, cp = keys.encrypt(pt1, t), keys.encrypt(pt2, t)
        d = torch.empty((3, Lq, N), dtype=torch.int32, device="cuda")
        d[0:1] = keys.mul(c[0:1], cp[0:1])
        d[1:2] = keys.mul(c[0:1], cp[1:2])
        keys.pf.pointwise(lib.RNS_ADD, d[1:2], keys.mul(c[1:2], cp[0:1]), d[1:2], 1)
        d[2:3] = keys.mul(c[1:2], cp[1:2])
        enc.decode(decrypt_to_t(lib, keys.decrypt(d), qs, t, False), z, 1)
        assert np.array_equal(signed(z), want)
    keys.close()


def two_n_prime_above_2_30(logn):
    two_n = 2 << logn
    k = (1 << 30) // two_n + 1
    while not is_prime(k * two_n + 1):
        k += 1
    return k * two_n + 1


@pytest.mark.gpu
def test_create_errors(lib):
    """Each bad t gives MODULUS: not prime, not 1 mod 2N, >= 2^30, dividing a channel (prime or
    composite); flags != 0 gives INVALID_ARG."""
    L = lib.load_library()
    logn = 13
    two_n = 2 << logn
    t = valid_t(logn)
    qs = channels(3, t)
    composite = next(k * two_n + 1 for k in range(1, 100) if not is_prime(k * two_n + 1))
    bad = [0, 1, 2, 3, 12289, composite, two_n_prime_above_2_30(logn), (1 << 31) - 1, (1 << 32) - 1]
    assert is_prime(12289) and 12289 % two_n != 1
    h = ctypes.c_void_p()
    with ones_plan(lib, logn, qs) as p:
        for b in bad:
            assert L.nttb200_packed_encoder_create(ctypes.byref(h), p._h, b, 0) == MODULUS, b
            assert not h.value
        assert L.nttb200_packed_encoder_create(ctypes.byref(h), p._h, t, 1) == INVALID_ARG
        assert L.nttb200_packed_encoder_create(ctypes.byref(h), None, t, 0) == INVALID_ARG
    for chans in ([qs[0], t], [3 * t, qs[0]]):
        with ones_plan(lib, logn, chans) as p:
            assert L.nttb200_packed_encoder_create(ctypes.byref(h), p._h, t, 0) == MODULUS
    with ones_plan(lib, logn, [3, 2, 1 << 30]) as p:
        assert L.nttb200_packed_encoder_create(ctypes.byref(h), p._h, t, 0) == OK
        assert L.nttb200_packed_encoder_destroy(h) == OK


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 15])
def test_buffers_and_errors(lib, logn):
    torch = _torch()
    N, batch, Lq = 1 << logn, 3, 3
    t = valid_t(logn)
    qs = channels(Lq, t)
    s = rand_slots(batch, N, t, 1300 + logn)
    with lib.PackedEncoder(ones_plan(lib, logn, qs), t) as enc:
        L = lib.load_library()
        h = enc._h
        sin = Guarded(batch * N, data=s)
        out = Guarded(batch * Lq * N)
        for mode in (SCALED, CENTRED):
            l0 = lib.kernel_launches()
            assert L.nttb200_packed_encode(h, sin.view.data_ptr(), mode, out.view.data_ptr(), batch, None) == OK
            torch.cuda.synchronize()
            assert lib.kernel_launches() - l0 == encode_launches(logn)
            assert out.guards_intact() and sin.guards_intact() and torch.equal(sin.view, s.reshape(-1))
        mt = Guarded(batch * N, data=decrypt_to_t(lib, out.view.reshape(batch, Lq, N), qs, t, False))
        mt_copy = mt.view.clone()
        dec = Guarded(batch * N)
        for flags in (0, CENTRED):
            l0 = lib.kernel_launches()
            assert L.nttb200_packed_decode(h, mt.view.data_ptr(), flags, dec.view.data_ptr(), batch, None) == OK
            torch.cuda.synchronize()
            assert lib.kernel_launches() - l0 == decode_launches(logn)
            assert dec.guards_intact() and mt.guards_intact() and torch.equal(mt.view, mt_copy)
        want = centre(signed(s).reshape(-1) % t, t)
        assert np.array_equal(signed(dec.view), want)
        # argument errors and batch == 0: nothing written, nothing launched
        fresh = Guarded(batch * Lq * N)
        p_in, p_out = sin.view.data_ptr(), fresh.view.data_ptr()
        l0 = lib.kernel_launches()
        for mode in (2, 3, 0xffffffff):
            assert L.nttb200_packed_encode(h, p_in, mode, p_out, batch, None) == INVALID_ARG
            assert L.nttb200_packed_encode(h, p_in, mode, p_out, 0, None) == INVALID_ARG
            assert L.nttb200_packed_decode(h, p_in, mode, p_out, batch, None) == INVALID_ARG
            assert L.nttb200_packed_decode(h, p_in, mode, p_out, 0, None) == INVALID_ARG
        for mode in (SCALED, CENTRED):
            assert L.nttb200_packed_encode(h, None, mode, p_out, batch, None) == INVALID_ARG
            assert L.nttb200_packed_encode(h, p_in, mode, None, batch, None) == INVALID_ARG
            assert L.nttb200_packed_encode(h, None, mode, None, 0, None) == OK
            assert L.nttb200_packed_encode(h, p_in, mode, p_in + 4 * N, batch, None) == INVALID_ARG   # overlap
            assert L.nttb200_packed_encode(h, p_out + 4 * (batch * Lq * N - 4), mode, p_out, batch, None) == INVALID_ARG
            assert L.nttb200_packed_encode(h, p_in + 4, mode, p_out, batch, None) == UNSUPPORTED
            assert L.nttb200_packed_encode(h, p_in, mode, p_out + 8, batch, None) == UNSUPPORTED
            assert L.nttb200_packed_encode(h, 1 << 40, mode, 1 << 46, 1 << 31, None) == UNSUPPORTED
        for flags in (0, CENTRED):
            assert L.nttb200_packed_decode(h, None, flags, p_out, batch, None) == INVALID_ARG
            assert L.nttb200_packed_decode(h, None, flags, None, 0, None) == OK
            assert L.nttb200_packed_decode(h, p_out, flags, p_out + 4 * (N - 4), batch, None) == INVALID_ARG
            assert L.nttb200_packed_decode(h, p_in, flags, p_in, batch, None) == INVALID_ARG
            assert L.nttb200_packed_decode(h, p_in + 12, flags, p_out, batch, None) == UNSUPPORTED
            assert L.nttb200_packed_decode(h, p_in, flags, p_out + 4, batch, None) == UNSUPPORTED
        torch.cuda.synchronize()
        assert lib.kernel_launches() == l0
        assert fresh.untouched() and sin.guards_intact() and torch.equal(sin.view, s.reshape(-1))
        assert _status(lib, lambda: enc.encode(s, fresh.view, 0)) == OK


@pytest.mark.gpu
def test_encode_beyond_2_31_words(lib):
    """One SCALED encode of 1025 polynomials at N = 2^16, L = 32: 2^31 + 2^21 output words."""
    torch = _torch()
    logn, L, batch = 16, 32, 1025
    N = 1 << logn
    t = valid_t(logn, True)
    qs = channels(L, t)
    s = rand_slots(2, N, t, 1400)
    d_s = s[torch.arange(batch, device="cuda") % 2].contiguous()
    out = torch.empty((batch, L, N), dtype=torch.int32, device="cuda")
    with lib.PackedEncoder(ones_plan(lib, logn, qs), t) as enc:
        enc.encode(d_s, out, batch)
    torch.cuda.synchronize()
    assert torch.equal(out[batch - 1], out[0]) and torch.equal(out[batch - 2], out[1])
    want = lift(Ref(N, t).encode(signed(s[:1])), qs, t, False)[0]
    assert np.array_equal(host(out[batch - 1]), want)
