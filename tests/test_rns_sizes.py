"""RNS batches at N = 2^13..2^16: [batch][L][N], channel l of polynomial b at (b*L + l)*N,
modulo its own prime with its own table.  GS, CT and the negacyclic product per channel
against the CPU oracle (integer equality), device-generated channel tables against host
tables, N = 4096 through the new constructors against the existing RnsPlan, and the
documented errors.  The argument checks of the two constructors run without a device."""
import ctypes

import numpy as np
import pytest

from conftest import Q29, Q30

OK, INVALID_ARG, MODULUS, TABLE, UNSUPPORTED = 0, 1, 2, 3, 7
GEN_BITREV = 1
GUARD = 64
SENTINEL = -1


def ntt_primes(count, two_n=1 << 17, below=1 << 30):
    """Primes q < 2^30 with two_n | q-1, largest first; 2^17 | q-1 serves every N <= 2^16."""
    out, k = [], (below - 1) // two_n
    while len(out) < count and k > 0:
        q = k * two_n + 1
        if q < below and all(q % d for d in range(3, int(q ** 0.5) + 1, 2)):
            out.append(q)
        k -= 1
    return out


def psi_of(n, q):
    """An element of order 2n modulo the prime q."""
    for x in range(2, 1000):
        psi = pow(x, (q - 1) // (2 * n), q)
        if pow(psi, n, q) == q - 1:
            return psi
    raise AssertionError("no 2n-th root found")


def channel_primes(limbs):
    """L primes below 2^30, largest first, with Q29 as the last channel when L > 1."""
    return ntt_primes(1) if limbs == 1 else ntt_primes(limbs - 1) + [Q29]


# ------------------------------------------------------------------ CPU: argument checks
def _u32(vals):
    return (ctypes.c_uint32 * len(vals))(*vals)


def _tables(lib, n, qs, mutate=None):
    tabs = [np.ones(n, dtype=np.int32) for _ in qs]
    if mutate:
        mutate(tabs)
    i32p = ctypes.POINTER(ctypes.c_int32)
    return tabs, (i32p * len(tabs))(*[t.ctypes.data_as(i32p) for t in tabs])


def test_create_logn_argument_checks_without_device(lib):
    L = lib.load_library()
    h = ctypes.c_void_p()
    qs = [Q30, Q29]

    def create(logn, limbs=2, q=qs, mutate=None, out=True, tables=True, flags=0):
        n = 1 << logn if 1 <= logn <= 16 else 1
        _, parr = _tables(lib, n, q, mutate)
        return L.nttb200_rns_plan_create_logn(ctypes.byref(h) if out else None, 0, logn, limbs, _u32(q),
                                              parr if tables else None, flags)

    for logn in (11, 17, 1, 27):
        assert create(logn) == UNSUPPORTED, logn
    for logn in (0, 28):
        assert create(logn) == INVALID_ARG, logn
    assert create(13, limbs=0) == INVALID_ARG
    assert create(13, limbs=33) == INVALID_ARG
    assert create(13, out=False) == INVALID_ARG
    assert create(13, tables=False) == INVALID_ARG
    assert create(13, flags=1) == INVALID_ARG
    assert L.nttb200_rns_plan_create_logn(ctypes.byref(h), 0, 13, 2, None, _tables(lib, 8192, qs)[1], 0) \
        == INVALID_ARG
    i32p = ctypes.POINTER(ctypes.c_int32)
    assert L.nttb200_rns_plan_create_logn(ctypes.byref(h), 0, 13, 2, _u32(qs), (i32p * 2)(), 0) == INVALID_ARG
    for bad_q in (0, 1, 1 << 31, 0xffffffff):
        assert create(14, q=[Q30, bad_q]) == MODULUS, bad_q
    for logn in (12, 13, 16):
        def big(t, n=1 << logn):
            t[1][n - 1] = Q29
        assert create(logn, mutate=big) == TABLE, logn

        def neg(t):
            t[0][5] = -1
        assert create(logn, mutate=neg) == TABLE, logn
    assert h.value is None


def test_create_generated_argument_checks_without_device(lib):
    L = lib.load_library()
    h = ctypes.c_void_p()
    qs = [Q30, Q29]

    def create(logn, limbs=2, q=qs, bases=(3, 3), kind=GEN_BITREV, out=True, flags=0):
        return L.nttb200_rns_plan_create_generated(ctypes.byref(h) if out else None, 0, logn, limbs, _u32(q),
                                                   kind, _u32(bases) if bases is not None else None, flags)

    for logn in (11, 17, 1, 27):
        assert create(logn) == UNSUPPORTED, logn
    for logn in (0, 28):
        assert create(logn) == INVALID_ARG, logn
    assert create(13, limbs=0) == INVALID_ARG
    assert create(13, limbs=33) == INVALID_ARG
    assert create(13, out=False) == INVALID_ARG
    assert create(13, bases=None) == INVALID_ARG
    assert create(13, kind=2) == INVALID_ARG
    assert create(13, flags=4) == INVALID_ARG
    assert L.nttb200_rns_plan_create_generated(ctypes.byref(h), 0, 13, 2, None, GEN_BITREV, _u32([3, 3]), 0) \
        == INVALID_ARG
    for bad_q in (0, 1, 1 << 31):
        assert create(15, q=[Q30, bad_q]) == MODULUS, bad_q
    assert create(16, bases=(3, Q29)) == TABLE
    assert create(12, bases=(Q30 + 1, 3)) == TABLE
    assert h.value is None


def test_rns_plan_table_size_is_checked(lib):
    with pytest.raises(ValueError):
        lib.RnsPlan([Q29], [np.ones(8192, dtype=np.int32)])               # default logn = 12
    with pytest.raises(ValueError):
        lib.RnsPlan([Q29], [np.ones(4096, dtype=np.int32)], logn=13)


# ------------------------------------------------------------------------- GPU helpers
def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"
    return torch


def dev(a):
    torch = _torch()
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).cuda()


def channel_tables(lib, n, qs):
    fwd, inv, psis = [], [], []
    for q in qs:
        psi = psi_of(n, q)
        psis.append(psi)
        fwd.append(lib.make_bitrev_table(n, q, psi))
        inv.append(lib.make_bitrev_table(n, q, pow(psi, q - 2, q)))
    return fwd, inv, psis


def rns_data(rng, batch, qs, n):
    """[batch][L][n] residues, polynomial 0 pinned at q_l - 1 on every channel."""
    a = np.stack([rng.integers(0, q, (batch, n), dtype=np.int32) for q in qs], axis=1)
    a[0] = np.array(qs, dtype=np.int32)[:, None] - 1
    return a


def oracle_product(om, a, b, fwd, inv, q):
    n = a.shape[-1]
    prod = om.pointwise(om.ntt_ct(a, fwd, q), om.ntt_ct(b, fwd, q), q)
    return om.scale(om.ntt_gs(prod, inv, q), om.powmod(n, q - 2, q), q)


def sampled(batch, rng, limit):
    if batch <= limit:
        return np.arange(batch)
    return np.unique(np.concatenate([[0, 1, batch // 2, batch - 1], rng.integers(0, batch, 4)]))


# (logn, L, batch): every size with 1, 3 and 32 channels, batches 1, 2, 7, and batches
# >= 64 whose CTA ranges cross position changes of the shared-memory table segments
SHAPES = [(13, 1, 7), (13, 3, 2), (13, 32, 1), (13, 3, 70),
          (14, 3, 7), (14, 32, 2), (14, 1, 1),
          (15, 3, 2), (15, 32, 1), (15, 1, 7),
          (16, 3, 2), (16, 32, 1), (16, 1, 2), (16, 2, 65)]


@pytest.mark.gpu
@pytest.mark.parametrize("logn,limbs,batch", SHAPES)
def test_rns_transforms_and_product(lib, oracle_mod, logn, limbs, batch):
    """GS and CT per channel against ntt_gs / ntt_ct with that channel's table; the product
    per channel against the oracle pipeline; in place, d_c aliasing d_a, operands unchanged."""
    torch = _torch()
    om = oracle_mod
    n = 1 << logn
    qs = channel_primes(limbs)
    rng = np.random.default_rng(71000 + 100 * logn + limbs + batch)
    fwd, inv, _ = channel_tables(lib, n, qs)
    a, b = rns_data(rng, batch, qs, n), rns_data(rng, batch, qs, n)
    rows = sampled(batch, rng, 8)
    d_a, d_b = dev(a), dev(b)
    d_o = torch.empty_like(d_a)
    with lib.RnsPlan(qs, fwd, logn=logn) as pf, lib.RnsPlan(qs, inv, logn=logn) as pi:
        assert (pf.logn, pf.n) == (logn, n)
        pi.gs(d_a, d_o, batch)
        got = d_o.cpu().numpy()
        for l, q in enumerate(qs):
            assert np.array_equal(got[rows, l], om.ntt_gs(a[rows, l], inv[l], q)), ("gs", l)
        pf.ct(d_a, d_o, batch)
        got = d_o.cpu().numpy()
        for l, q in enumerate(qs):
            assert np.array_equal(got[rows, l], om.ntt_ct(a[rows, l], fwd[l], q)), ("ct", l)
        lib.rns_polymul_negacyclic(pf, pi, d_a, d_b, d_o, batch)
        got = d_o.cpu().numpy()
        want = {l: oracle_product(om, a[rows, l], b[rows, l], fwd[l], inv[l], q) for l, q in enumerate(qs)}
        for l in want:
            assert np.array_equal(got[rows, l], want[l]), ("polymul", l)
        if logn == 13 and limbs == 3 and batch == 2:
            assert np.array_equal(got[1, 2], om.negacyclic_schoolbook(a[1, 2], b[1, 2], qs[2]))
        assert np.array_equal(d_a.cpu().numpy(), a) and np.array_equal(d_b.cpu().numpy(), b)
        # d_c aliasing d_a, then both transforms in place
        d_x = d_a.clone()
        lib.rns_polymul_negacyclic(pf, pi, d_x, d_b, d_x, batch)
        got = d_x.cpu().numpy()
        for l in want:
            assert np.array_equal(got[rows, l], want[l]), ("polymul aliased", l)
        assert np.array_equal(d_b.cpu().numpy(), b)
        d_x = d_a.clone()
        pi.gs(d_x, d_x, batch)
        pf.ct(d_x, d_x, batch)
        got = d_x.cpu().numpy()
        for l, q in enumerate(qs):
            want_l = om.ntt_ct(om.ntt_gs(a[rows, l], inv[l], q), fwd[l], q)
            assert np.array_equal(got[rows, l], want_l), ("in place", l)


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [13, 14, 15, 16])
def test_rns_tables_pinned_at_q_minus_1(lib, oracle_mod, logn):
    """Every table entry and every input word at q - 1 (the largest operands of every
    butterfly) on one channel, a 30-bit prime beside it."""
    torch = _torch()
    n = 1 << logn
    qs = [ntt_primes(1)[0], Q29]
    rng = np.random.default_rng(72000 + logn)
    tabs = [rng.integers(0, qs[0], n, dtype=np.int32), np.full(n, qs[1] - 1, dtype=np.int32)]
    a = rns_data(rng, 2, qs, n)
    a[1, 1] = qs[1] - 1
    d_a = dev(a)
    d_o = torch.empty_like(d_a)
    with lib.RnsPlan(qs, tabs, logn=logn) as rp:
        rp.gs(d_a, d_o, 2)
        got = d_o.cpu().numpy()
        for l, q in enumerate(qs):
            assert np.array_equal(got[:, l], oracle_mod.ntt_gs(a[:, l], tabs[l], q)), ("gs", l)
        rp.ct(d_a, d_o, 2)
        got = d_o.cpu().numpy()
        for l, q in enumerate(qs):
            assert np.array_equal(got[:, l], oracle_mod.ntt_ct(a[:, l], tabs[l], q)), ("ct", l)


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 13, 14, 15, 16])
def test_generated_plans_equal_host_table_plans(lib, oracle_mod, logn):
    """RnsPlan.generated(logn, qs, GEN_BITREV, psi_l / psi_l^-1) computes exactly what plans
    built from make_bitrev_table(n, q, psi_l) / (psi_l^-1) compute."""
    torch = _torch()
    n, batch = 1 << logn, 3
    qs = channel_primes(4)
    rng = np.random.default_rng(73000 + logn)
    fwd, inv, psis = channel_tables(lib, n, qs)
    psis_inv = [pow(p, q - 2, q) for p, q in zip(psis, qs)]
    a, b = rns_data(rng, batch, qs, n), rns_data(rng, batch, qs, n)
    d_a, d_b = dev(a), dev(b)
    outs = []
    host = (lib.RnsPlan(qs, fwd, logn=logn), lib.RnsPlan(qs, inv, logn=logn))
    gen = (lib.RnsPlan.generated(logn, qs, GEN_BITREV, psis), lib.RnsPlan.generated(logn, qs, GEN_BITREV, psis_inv))
    for pf, pi in (host, gen):
        assert pf.n == n
        o = [torch.empty_like(d_a) for _ in range(3)]
        pi.gs(d_a, o[0], batch)
        pf.ct(d_a, o[1], batch)
        lib.rns_polymul_negacyclic(pf, pi, d_a, d_b, o[2], batch)
        outs.append([x.cpu().numpy() for x in o])
        pf.close()
        pi.close()
    for k in range(3):
        assert np.array_equal(outs[0][k], outs[1][k]), k
    want = oracle_product(oracle_mod, a[:, 1], b[:, 1], fwd[1], inv[1], qs[1])
    assert np.array_equal(outs[1][2][:, 1], want)


@pytest.mark.gpu
def test_n4096_new_constructors_match_rns_plan_create(lib):
    """logn = 12 through nttb200_rns_plan_create_logn and through RnsPlan.generated equals the
    plan of nttb200_rns_plan_create bit for bit (GS, CT, product)."""
    torch = _torch()
    n, batch = 4096, 5
    qs = channel_primes(5)
    rng = np.random.default_rng(74000)
    fwd, inv, psis = channel_tables(lib, n, qs)
    a, b = rns_data(rng, batch, qs, n), rns_data(rng, batch, qs, n)
    d_a, d_b = dev(a), dev(b)
    L = lib.load_library()
    i32p = ctypes.POINTER(ctypes.c_int32)

    def legacy(tabs):
        plan = lib.RnsPlan.__new__(lib.RnsPlan)
        plan._lib, plan.limbs, plan.qs = L, len(qs), qs
        h = ctypes.c_void_p()
        parr = (i32p * len(qs))(*[t.ctypes.data_as(i32p) for t in tabs])
        assert L.nttb200_rns_plan_create(ctypes.byref(h), 0, len(qs), _u32(qs), parr, 0) == OK
        plan._h = h
        return plan

    def run(pf, pi):
        o = [torch.empty_like(d_a) for _ in range(3)]
        pi.gs(d_a, o[0], batch)
        pf.ct(d_a, o[1], batch)
        lib.rns_polymul_negacyclic(pf, pi, d_a, d_b, o[2], batch)
        res = [x.cpu().numpy() for x in o]
        pf.close()
        pi.close()
        return res

    ref = run(legacy(fwd), legacy(inv))
    new = run(lib.RnsPlan(qs, fwd, logn=12), lib.RnsPlan(qs, inv, logn=12))
    gen = run(lib.RnsPlan.generated(12, qs, GEN_BITREV, psis),
              lib.RnsPlan.generated(12, qs, GEN_BITREV, [pow(p, q - 2, q) for p, q in zip(psis, qs)]))
    for k in range(3):
        assert np.array_equal(ref[k], new[k]), k
        assert np.array_equal(ref[k], gen[k]), k


class Guarded:
    """`words` int32 between two sentinel guard bands; the view starts k words past a
    16-byte boundary."""

    def __init__(self, words, k=0, data=None):
        torch = _torch()
        self.raw = torch.full((words + 2 * GUARD,), SENTINEL, dtype=torch.int32, device="cuda")
        self.view = self.raw[GUARD + k:GUARD + k + words]
        if data is not None:
            self.view.copy_(torch.from_numpy(np.ascontiguousarray(data, dtype=np.int32)).reshape(-1))

    def untouched(self):
        return bool((self.raw == SENTINEL).all())


def _status(lib, call):
    try:
        call()
    except lib.NttError as err:
        return err.status
    return OK


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [13, 16])
def test_rns_documented_errors(lib, oracle_mod, logn):
    """Unaligned input, operand or output -> UNSUPPORTED with nothing stored and the plan
    still usable; fwd / inv of different N -> INVALID_ARG; an empty batch is OK; more than
    2^31 - 1 tiles -> UNSUPPORTED before anything runs."""
    torch = _torch()
    n, batch = 1 << logn, 2
    qs = channel_primes(3)
    rng = np.random.default_rng(75000 + logn)
    fwd, inv, _ = channel_tables(lib, n, qs)
    a, b = rns_data(rng, batch, qs, n), rns_data(rng, batch, qs, n)
    with lib.RnsPlan(qs, fwd, logn=logn) as pf, lib.RnsPlan(qs, inv, logn=logn) as pi:
        for k_in, k_out in ((1, 0), (0, 3), (2, 1)):
            for fn in (pi.gs, pf.ct):
                src, dst = Guarded(a.size, k_in, a), Guarded(a.size, k_out)
                assert _status(lib, lambda: fn(src.view, dst.view, batch)) == UNSUPPORTED
                torch.cuda.synchronize()
                assert dst.untouched()
                assert np.array_equal(src.view.cpu().numpy().reshape(a.shape), a)
        for ka, kb, kc in ((1, 0, 0), (0, 2, 0), (0, 0, 3)):
            ga, gb, gc = Guarded(a.size, ka, a), Guarded(b.size, kb, b), Guarded(a.size, kc)
            assert _status(lib, lambda: lib.rns_polymul_negacyclic(pf, pi, ga.view, gb.view, gc.view,
                                                                   batch)) == UNSUPPORTED
            torch.cuda.synchronize()
            assert gc.untouched(), (ka, kb, kc)
        # the plans are still usable
        d_a, d_o = dev(a), torch.empty(a.shape, dtype=torch.int32, device="cuda")
        pi.gs(d_a, d_o, batch)
        assert np.array_equal(d_o.cpu().numpy()[:, 0], oracle_mod.ntt_gs(a[:, 0], inv[0], qs[0]))
        # empty batch
        pi.gs(d_a, d_o, 0)
        lib.rns_polymul_negacyclic(pf, pi, d_a, d_a, d_o, 0)
        # tile count: batch * L * N / 4096 must stay below 2^31 (nothing is launched)
        huge = ((1 << 31) >> (logn - 12)) // len(qs) + 1
        assert _status(lib, lambda: pi.gs(d_a, d_o, huge)) == UNSUPPORTED
        assert _status(lib, lambda: pf.ct(d_a, d_o, huge)) == UNSUPPORTED
        assert _status(lib, lambda: lib.rns_polymul_negacyclic(pf, pi, d_a, d_a, d_o, huge)) == UNSUPPORTED
        # fwd and inv of different N
        other_n = 1 << (logn - 1)
        with lib.RnsPlan(qs, channel_tables(lib, other_n, qs)[1], logn=logn - 1) as po:
            assert _status(lib, lambda: lib.rns_polymul_negacyclic(pf, po, d_a, d_a, d_o, 1)) == INVALID_ARG
        torch.cuda.synchronize()
