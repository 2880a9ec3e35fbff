"""Evaluation-domain arithmetic on RNS batches ([batch][L][N], channel l of polynomial b at
(b*L + l)*N modulo q_l): nttb200_rns_pointwise (add / sub / mul, own or broadcast operand),
nttb200_rns_scale, nttb200_rns_dot and nttb200_rns_gs_scaled_batch.  Results against numpy
residues in uint64; the scaled inverse against rns_gs + rns_scale and as the inverse of rns_ct;
ct, ct, mul, gs_scaled against rns_polymul_negacyclic.  Guard bands around every buffer check
that nothing is stored outside the output.  The null-plan argument checks run without a device."""
import ctypes

import numpy as np
import pytest

from conftest import Q29
from test_rns_sizes import channel_primes, psi_of

OK, INVALID_ARG, MODULUS, UNSUPPORTED = 0, 1, 2, 7
ADD, SUB, MUL = 0, 1, 2
GEN_BITREV = 1
GUARD = 64        # sentinel words on each side of a view (256 B: the view base stays 16 B aligned)
SENTINEL = -1     # 0xffffffff: >= q for every modulus, never a result
L2_WORDS = 1 << 26   # 256 MiB per operand: twice the B200's L2


# ------------------------------------------------------------------ CPU: argument checks
def test_null_arguments_without_device(lib):
    L = lib.load_library()
    s = (ctypes.c_uint32 * 1)(1)
    assert L.nttb200_rns_pointwise(None, MUL, None, None, None, 1, 1, None) == INVALID_ARG
    assert L.nttb200_rns_pointwise(None, ADD, None, None, None, 0, 0, None) == INVALID_ARG
    assert L.nttb200_rns_pointwise(None, 3, 16, 16, 16, 1, 1, None) == INVALID_ARG
    assert L.nttb200_rns_scale(None, 16, 16, 1, s, None) == INVALID_ARG
    assert L.nttb200_rns_scale(None, 16, 16, 1, None, None) == INVALID_ARG
    assert L.nttb200_rns_scale(None, None, None, 0, s, None) == INVALID_ARG
    assert L.nttb200_rns_dot(None, 16, 16, 16, 1, 1, 1, 0, None) == INVALID_ARG
    assert L.nttb200_rns_dot(None, 16, 16, 16, 0, 1, 1, 0, None) == INVALID_ARG
    assert L.nttb200_rns_dot(None, 16, 16, 16, 65, 1, 1, 0, None) == INVALID_ARG
    assert L.nttb200_rns_gs_scaled_batch(None, 16, 16, 1, None) == INVALID_ARG
    assert L.nttb200_rns_gs_scaled_batch(None, None, None, 0, None) == INVALID_ARG
    assert (lib.RNS_ADD, lib.RNS_SUB, lib.RNS_MUL) == (ADD, SUB, MUL)


# ------------------------------------------------------------------------- GPU helpers
def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"
    return torch


def rand_rns(shape, qs, seed, pin=True):
    """Residues of shape [..., L, N] on the device; with pin, coefficients 0..15 of every row
    at q_l - 1 and 16..31 at 0 (with the other operand's pins: every pair of extremes)."""
    torch = _torch()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    qt = torch.tensor(qs, dtype=torch.int32, device="cuda").view(len(qs), 1)
    x = torch.randint(0, 1 << 30, shape, dtype=torch.int32, device="cuda", generator=gen)
    x.remainder_(qt)
    if pin:
        x[..., :16] = qt - 1
        x[..., 16:32] = 0
    return x


def rows_of(batch, seed):
    if batch <= 5:
        return np.arange(batch)
    rng = np.random.default_rng(seed)
    return np.unique(np.concatenate([[0, 1, batch // 2, batch - 1], rng.integers(0, batch, 3)]))


def host(x, rows=None):
    y = x if rows is None else x[rows]
    return y.cpu().numpy().astype(np.uint64)


def qcol(qs):
    return np.array(qs, dtype=np.uint64)[:, None]


def channel_tables(lib, n, qs):
    fwd, inv, psis = [], [], []
    for q in qs:
        psi = psi_of(n, q)
        psis.append(psi)
        fwd.append(lib.make_bitrev_table(n, q, psi))
        inv.append(lib.make_bitrev_table(n, q, pow(psi, q - 2, q)))
    return fwd, inv, psis


def ones_plan(lib, logn, qs):
    """A plan whose tables are all ones: the operators do not read tables."""
    return lib.RnsPlan(qs, [np.ones(1 << logn, dtype=np.int32) for _ in qs], logn=logn)


class Guarded:
    """`words` int32 on the device between two guard bands of the sentinel; `view` starts
    k words (4k bytes) past a 16-byte boundary."""

    def __init__(self, words, k=0, data=None):
        torch = _torch()
        self.raw = torch.full((words + 2 * GUARD,), SENTINEL, dtype=torch.int32, device="cuda")
        self.k, self.words = k, words
        self.view = self.raw[GUARD + k:GUARD + k + words]
        assert self.view.data_ptr() % 16 == 4 * k
        if data is not None:
            self.view.copy_(data.reshape(-1))

    def guards_intact(self):
        head = self.raw[:GUARD + self.k]
        tail = self.raw[GUARD + self.k + self.words:]
        return bool((head == SENTINEL).all()) and bool((tail == SENTINEL).all())

    def untouched(self):
        return bool((self.raw == SENTINEL).all())


def _status(lib, call):
    try:
        call()
    except lib.NttError as err:
        return err.status
    return OK


# ---------------------------------------------------------------- streaming operators
OP_CASES = [(logn, limbs, batch) for logn in (12, 13, 16) for limbs in (1, 3, 32) for batch in (1, 5, "l2")]


@pytest.mark.gpu
@pytest.mark.parametrize("logn,limbs,batch", OP_CASES)
def test_pointwise_and_scale(lib, logn, limbs, batch):
    """add / sub / mul with an own and with a broadcast operand, scale with scalars 0, 1 and
    q_l - 1 on every channel; batch "l2" makes each operand 256 MiB, twice the L2."""
    torch = _torch()
    n = 1 << logn
    if batch == "l2":
        batch = L2_WORDS // (limbs * n)
    qs = channel_primes(limbs)
    seed = 81000 + 100 * logn + limbs
    a = rand_rns((batch, limbs, n), qs, seed)
    b = rand_rns((batch, limbs, n), qs, seed + 1)
    b[..., 8:16] = 0
    b[..., 16:24] = torch.tensor(qs, dtype=torch.int32, device="cuda").view(limbs, 1) - 1
    c = torch.empty_like(a)
    rows = rows_of(batch, seed)
    ha, hb, q = host(a, rows), host(b, rows), qcol(qs)
    hb0 = host(b[:1])
    want = {ADD: lambda y: (ha + y) % q, SUB: lambda y: (ha + q - y) % q, MUL: lambda y: ha * y % q}
    with ones_plan(lib, logn, qs) as rp:
        for op in (ADD, SUB, MUL):
            rp.pointwise(op, a, b, c, batch)
            assert np.array_equal(host(c, rows), want[op](hb)), ("own", op)
            rp.pointwise(op, a, b[:1], c, batch, b_batch=1)
            assert np.array_equal(host(c, rows), want[op](hb0)), ("broadcast", op)
        for j in range(3):
            scalars = [(0, 1, qv - 1)[(l + j) % 3] for l, qv in enumerate(qs)]
            rp.scale(a, c, batch, scalars)
            want_s = ha * np.array(scalars, dtype=np.uint64)[:, None] % q
            assert np.array_equal(host(c, rows), want_s), ("scale", j)
        assert np.array_equal(host(a, rows), ha) and np.array_equal(host(b, rows), hb)


# --------------------------------------------------------------------------- rns_dot
def dot_reference(a, w, q, acc0):
    """a: [K][rows][L][N], w: [K][rows or 1][L][N] (uint64), reduced per term."""
    acc = acc0.copy() if acc0 is not None else np.zeros(a.shape[1:], dtype=np.uint64)
    for k in range(a.shape[0]):
        acc = (acc + a[k] * w[k] % q) % q
    return acc


@pytest.mark.gpu
@pytest.mark.parametrize("terms", [1, 2, 16, 17, 64])
@pytest.mark.parametrize("shared_key", [False, True])
def test_dot(lib, terms, shared_key):
    """Random and all-(q_l - 1) inputs (the largest sums before a fold), accumulate off and on,
    one key per polynomial or one shared key; batch 11 leaves ragged polynomial groups."""
    torch = _torch()
    logn, batch = 12, 11
    n = 1 << logn
    qs = channel_primes(3)
    q = qcol(qs)
    w_batch = 1 if shared_key else batch
    seed = 82000 + terms * 2 + shared_key
    with ones_plan(lib, logn, qs) as rp:
        for extreme in (False, True):
            a = rand_rns((terms, batch, 3, n), qs, seed)
            w = rand_rns((terms, w_batch, 3, n), qs, seed + 1)
            c0 = rand_rns((batch, 3, n), qs, seed + 2)
            if extreme:
                qm1 = torch.tensor(qs, dtype=torch.int32, device="cuda").view(3, 1) - 1
                for x in (a, w, c0):
                    x.copy_(qm1.expand_as(x))
            ha, hw, hc0 = host(a), host(w), host(c0)
            if shared_key:
                hw = np.broadcast_to(hw, (terms, batch, 3, n))
            for accumulate in (False, True):
                c = c0.clone()
                lib.rns_dot(rp, a, w, c, terms, batch, w_batch=w_batch, accumulate=accumulate)
                want = dot_reference(ha, hw, q, hc0 if accumulate else None)
                assert np.array_equal(host(c), want), (extreme, accumulate)
            assert np.array_equal(host(a), ha) and np.array_equal(host(w)[:, :w_batch], hw[:, :w_batch])


@pytest.mark.gpu
def test_dot_large_n_and_channels(lib):
    """N = 2^16 with 16 channels, 17 terms (one fold inside the sum), both key layouts."""
    torch = _torch()
    logn, limbs, batch, terms = 16, 16, 2, 17
    n = 1 << logn
    qs = channel_primes(limbs)
    q = qcol(qs)
    a = rand_rns((terms, batch, limbs, n), qs, 83000)
    w = rand_rns((terms, batch, limbs, n), qs, 83001)
    c = torch.empty((batch, limbs, n), dtype=torch.int32, device="cuda")
    ha, hw = host(a), host(w)
    with ones_plan(lib, logn, qs) as rp:
        lib.rns_dot(rp, a, w, c, terms, batch)
        assert np.array_equal(host(c), dot_reference(ha, hw, q, None))
        lib.rns_dot(rp, a, w[:, :1].contiguous(), c, terms, batch, w_batch=1)
        assert np.array_equal(host(c), dot_reference(ha, np.broadcast_to(hw[:, :1], ha.shape), q, None))


# -------------------------------------------------------------------- scaled inverse
@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 13, 14, 15, 16])
def test_gs_scaled(lib, logn):
    """gs_scaled == gs then scale by N^-1, bit for bit (batch 2 and a batch of 65, which takes
    the per-segment table mode); gs_scaled(ct(x)) == x with host-table and device-generated
    plans; in place."""
    torch = _torch()
    n = 1 << logn
    qs = channel_primes(3)
    fwd, inv, psis = channel_tables(lib, n, qs)
    ninv = [pow(n, q - 2, q) for q in qs]
    host_plans = (lib.RnsPlan(qs, fwd, logn=logn), lib.RnsPlan(qs, inv, logn=logn))
    gen_plans = (lib.RnsPlan.generated(logn, qs, GEN_BITREV, psis),
                 lib.RnsPlan.generated(logn, qs, GEN_BITREV, [pow(p, q - 2, q) for p, q in zip(psis, qs)]))
    for batch in (2, 65):
        x = rand_rns((batch, 3, n), qs, 84000 + logn + batch)
        want, got, y = torch.empty_like(x), torch.empty_like(x), torch.empty_like(x)
        pf, pi = host_plans
        pi.gs(x, want, batch)
        pi.scale(want, want, batch, ninv)
        pi.gs_scaled(x, got, batch)
        assert torch.equal(got, want), batch
        for pf, pi in (host_plans, gen_plans):
            pf.ct(x, y, batch)
            pi.gs_scaled(y, y, batch)
            assert torch.equal(y, x), batch
    for p in host_plans + gen_plans:
        p.close()


@pytest.mark.gpu
def test_gs_scaled_even_modulus(lib):
    torch = _torch()
    d = torch.zeros((1, 2, 8192), dtype=torch.int32, device="cuda")
    with ones_plan(lib, 13, [Q29, 1 << 20]) as rp:
        before = lib.kernel_launches()
        assert _status(lib, lambda: rp.gs_scaled(d, d, 1)) == MODULUS
        assert _status(lib, lambda: rp.gs_scaled(d, d, 0)) == MODULUS
        assert lib.kernel_launches() == before
        rp.gs(d, d, 1)   # the unscaled network needs no N^-1


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 13, 14, 15, 16])
def test_eval_domain_product_equals_polymul(lib, oracle_mod, logn):
    """ct(a), ct(b), pointwise MUL, gs_scaled == rns_polymul_negacyclic(a, b) bit for bit; at
    N <= 8192 one channel also against the schoolbook product."""
    torch = _torch()
    n, batch, limbs = 1 << logn, 3, 4
    qs = channel_primes(limbs)
    fwd, inv, _ = channel_tables(lib, n, qs)
    a = rand_rns((batch, limbs, n), qs, 85000 + logn)
    b = rand_rns((batch, limbs, n), qs, 85100 + logn)
    ea, eb, want = torch.empty_like(a), torch.empty_like(a), torch.empty_like(a)
    with lib.RnsPlan(qs, fwd, logn=logn) as pf, lib.RnsPlan(qs, inv, logn=logn) as pi:
        lib.rns_polymul_negacyclic(pf, pi, a, b, want, batch)
        pf.ct(a, ea, batch)
        pf.ct(b, eb, batch)
        pf.pointwise(MUL, ea, eb, ea, batch)
        pi.gs_scaled(ea, ea, batch)
        assert torch.equal(ea, want)
    if logn <= 13:
        ha, hb, got = a.cpu().numpy(), b.cpu().numpy(), ea.cpu().numpy()
        assert np.array_equal(got[1, 3], oracle_mod.negacyclic_schoolbook(ha[1, 3], hb[1, 3], qs[3]))


# ---------------------------------------------------------------------- buffer rules
@pytest.mark.gpu
def test_buffers_aliasing_and_errors(lib):
    """Guard bands hold and out-of-place inputs are unchanged; in place and the documented
    aliasing work; other overlaps -> INVALID_ARG and views 4/8/12 bytes past alignment ->
    UNSUPPORTED, nothing written and the plan still usable; bad options and batch == 0
    launch nothing."""
    torch = _torch()
    logn, batch, limbs = 13, 3, 3
    n = 1 << logn
    qs = channel_primes(limbs)
    fwd, inv, _ = channel_tables(lib, n, qs)
    words = batch * limbs * n
    q = qcol(qs)
    a = rand_rns((batch, limbs, n), qs, 86000)
    b = rand_rns((batch, limbs, n), qs, 86001)
    ha, hb = host(a), host(b)
    prod = ha * hb % q
    with lib.RnsPlan(qs, fwd, logn=logn) as pf, lib.RnsPlan(qs, inv, logn=logn) as rp:
        def fresh(x=None, k=0, w=words):
            return Guarded(w, k, x)

        # out of place: guards hold, inputs unchanged
        ga, gb, gc = fresh(a), fresh(b), fresh()
        rp.pointwise(MUL, ga.view, gb.view, gc.view, batch)
        rp.pointwise(SUB, ga.view, gb.view[:limbs * n], gc.view, batch, b_batch=1)
        torch.cuda.synchronize()
        assert np.array_equal(host(gc.view.view(a.shape)), (ha + q - hb[:1]) % q)
        rp.scale(ga.view, gc.view, batch, [2] * limbs)
        assert np.array_equal(host(gc.view.view(a.shape)), ha * 2 % q)
        want_gs = torch.empty_like(a)
        rp.gs(a, want_gs, batch)
        rp.scale(want_gs, want_gs, batch, [pow(n, qv - 2, qv) for qv in qs])
        rp.gs_scaled(ga.view, gc.view, batch)
        assert torch.equal(gc.view.view(a.shape), want_gs)
        ka = fresh(torch.stack([a, b]), w=2 * words)
        kw = fresh(torch.stack([b[0], a[0]]), w=2 * limbs * n)
        lib.rns_dot(rp, ka.view, kw.view, gc.view, 2, batch, w_batch=1)
        assert np.array_equal(host(gc.view.view(a.shape)), (ha * hb[0] % q + hb * ha[0] % q) % q)
        for g in (ga, gb, gc, ka, kw):
            assert g.guards_intact()
        assert torch.equal(ka.view, torch.stack([a, b]).reshape(-1))
        assert torch.equal(ga.view, a.reshape(-1)) and torch.equal(gb.view, b.reshape(-1))
        # in place and the documented aliasing
        gx = fresh(a)
        rp.pointwise(MUL, gx.view, gb.view, gx.view, batch)
        assert np.array_equal(host(gx.view.view(a.shape)), prod)
        gx = fresh(b)
        rp.pointwise(MUL, ga.view, gx.view, gx.view, batch)
        assert np.array_equal(host(gx.view.view(a.shape)), prod)
        gx = fresh(a)
        rp.scale(gx.view, gx.view, batch, [3] * limbs)
        assert np.array_equal(host(gx.view.view(a.shape)), ha * 3 % q)
        gx = fresh(a)
        rp.gs_scaled(gx.view, gx.view, batch)
        assert torch.equal(gx.view.view(a.shape), want_gs) and gx.guards_intact()
        # disallowed overlaps: INVALID_ARG, nothing written
        big = fresh(torch.cat([a.reshape(-1), b.reshape(-1)]), w=2 * words)
        snap = big.raw.clone()
        half, one = big.view[:words], limbs * n
        shifted = big.view[one:one + words]
        bad = [lambda: rp.pointwise(ADD, half, big.view[words:], shifted, batch),
               lambda: rp.pointwise(ADD, big.view[words:], half, shifted, batch),
               lambda: rp.pointwise(ADD, big.view[words:], half, half, batch, b_batch=1),
               lambda: rp.scale(half, shifted, batch, [1] * limbs),
               lambda: lib.rns_dot(rp, half, gb.view, shifted, 1, batch),
               lambda: lib.rns_dot(rp, ga.view, half, half, 1, batch),
               lambda: lib.rns_dot(rp, ga.view, big.view, half, 1, 1, w_batch=1)]
        for i, call in enumerate(bad):
            assert _status(lib, call) == INVALID_ARG, i
        torch.cuda.synchronize()
        assert torch.equal(big.raw, snap)
        # unaligned views: UNSUPPORTED, nothing written
        for k in (1, 2, 3):
            for ka, kb, kc in ((k, 0, 0), (0, k, 0), (0, 0, k)):
                ua, ub, uc = fresh(a, ka), fresh(b, kb), fresh(None, kc)
                sa, sb = ua.raw.clone(), ub.raw.clone()
                calls = [lambda: rp.pointwise(MUL, ua.view, ub.view, uc.view, batch),
                         lambda: rp.pointwise(ADD, ua.view, ub.view[:one], uc.view, batch, b_batch=1),
                         lambda: lib.rns_dot(rp, ua.view, ub.view, uc.view, 1, batch)]
                if kb == 0:
                    calls += [lambda: rp.scale(ua.view, uc.view, batch, [1] * limbs),
                              lambda: rp.gs_scaled(ua.view, uc.view, batch)]
                for i, call in enumerate(calls):
                    assert _status(lib, call) == UNSUPPORTED, (k, ka, kb, kc, i)
                torch.cuda.synchronize()
                assert uc.untouched() and torch.equal(ua.raw, sa) and torch.equal(ub.raw, sb)
        gx = fresh()
        rp.pointwise(MUL, a, b, gx.view, batch)   # still usable
        assert np.array_equal(host(gx.view.view(a.shape)), prod) and gx.guards_intact()
        # bad options and empty batches launch nothing
        before = lib.kernel_launches()
        L = lib.load_library()
        h = rp._h
        s_ok = (ctypes.c_uint32 * limbs)(*[1] * limbs)
        s_big = (ctypes.c_uint32 * limbs)(*qs)
        A, B, C = a.data_ptr(), b.data_ptr(), gx.view.data_ptr()
        assert L.nttb200_rns_pointwise(h, 3, A, B, C, batch, batch, None) == INVALID_ARG
        assert L.nttb200_rns_pointwise(h, MUL, A, B, C, batch, 2, None) == INVALID_ARG
        assert L.nttb200_rns_pointwise(h, MUL, A, B, C, batch, 0, None) == INVALID_ARG
        assert L.nttb200_rns_pointwise(h, MUL, A, None, C, batch, batch, None) == INVALID_ARG
        assert L.nttb200_rns_scale(h, A, C, batch, None, None) == INVALID_ARG
        assert L.nttb200_rns_scale(h, A, C, batch, s_big, None) == INVALID_ARG
        assert L.nttb200_rns_scale(h, None, C, batch, s_ok, None) == INVALID_ARG
        for terms in (0, 65):
            assert L.nttb200_rns_dot(h, A, B, C, terms, 1, 1, 0, None) == INVALID_ARG
        assert L.nttb200_rns_dot(h, A, B, C, 1, batch, 2, 0, None) == INVALID_ARG
        assert L.nttb200_rns_dot(h, A, None, C, 1, batch, batch, 0, None) == INVALID_ARG
        assert L.nttb200_rns_gs_scaled_batch(h, A, None, batch, None) == INVALID_ARG
        assert L.nttb200_rns_pointwise(h, MUL, None, None, None, 0, 0, None) == OK
        assert L.nttb200_rns_pointwise(h, MUL, None, None, None, 0, 1, None) == OK
        assert L.nttb200_rns_scale(h, None, None, 0, s_ok, None) == OK
        assert L.nttb200_rns_dot(h, None, None, None, 64, 0, 1, 1, None) == OK
        assert L.nttb200_rns_gs_scaled_batch(h, None, None, 0, None) == OK
        assert lib.kernel_launches() == before
        torch.cuda.synchronize()
        assert np.array_equal(host(gx.view.view(a.shape)), prod)


@pytest.mark.gpu
def test_pointwise_beyond_2_31_words(lib):
    """One call over 2^31 + 2^16 words (L = 1, N = 2^16, batch 2^15 + 1: 8 GiB per operand),
    checked on sampled polynomials including the last."""
    torch = _torch()
    logn, batch = 16, (1 << 15) + 1
    n = 1 << logn
    qs = channel_primes(1)
    q = qcol(qs)
    gen = torch.Generator(device="cuda").manual_seed(87000)
    a = torch.randint(0, qs[0], (batch, 1, n), dtype=torch.int32, device="cuda", generator=gen)
    b = torch.randint(0, qs[0], (batch, 1, n), dtype=torch.int32, device="cuda", generator=gen)
    rows = np.array([0, 1, batch // 2, batch - 2, batch - 1])
    want = host(a, rows) * host(b, rows) % q
    with ones_plan(lib, logn, qs) as rp:
        rp.pointwise(MUL, a, b, a, batch)
        assert np.array_equal(host(a, rows), want)
