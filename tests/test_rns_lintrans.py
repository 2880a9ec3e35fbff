"""Plaintext matrix-vector products on RNS ciphertext batches: nttb200_rns_lintrans_keys / _apply
(Python lintrans_galois, KeySwitcher.linear_transform).  On the CPU: the key list against a direct
enumeration, the baby-step giant-step identity on numpy slot vectors against M z, and the argument
checks that need no device.  On the GPU: bit-exactness against the composed sequence of existing
calls (keyswitch_apply over the babies, automorphism and ADD of c0, automorphism of each diagonal,
MUL / ADD per term, keyswitch_apply per giant, automorphism of W_i.c0 and the adds) for N =
2^12..2^16 and the key-switch (L, K, alpha), offset sets {0}, babies only, giants only, banded,
random sparse, all N/2 offsets and more than 64 giants, batch 1 and 3, one shape beyond the L2;
CKKS and BFV end to end with host-built keys; the errors, batch 0, unaligned buffers and the
launch counts."""
import ctypes
import math

import numpy as np
import pytest

from test_packed_encode import Keys, channels, decrypt_to_t, signed, to_dev
from test_rns_automorph import sigma_int
from test_rns_eval import Guarded, _status, rand_rns
from test_rns_keyswitch import CONFIGS, Env, host_keys

OK, INVALID_ARG, UNSUPPORTED = 0, 1, 7
ADD, MUL = 0, 2


def schedule(offsets, n1):
    """babies j >= 1 and giants i >= 1 that occur, ascending, and the terms {i: [(j, index)]}"""
    terms = {}
    for c, k in enumerate(offsets):
        terms.setdefault(k // n1, []).append((k % n1, c))
    babies = sorted({k % n1 for k in offsets} - {0})
    return babies, sorted(set(terms) - {0}), {i: sorted(t) for i, t in sorted(terms.items())}


def launches(logn, dnum, offsets, n1):
    """[nb > 0] P + 1 + [ng > 0] (ceil(ng / 64) P + 1), P = 2 dnum + 5 (+ 4 above N = 4096)"""
    babies, giants, _ = schedule(offsets, n1)
    p = 2 * dnum + (5 if logn == 12 else 9)
    return (p if babies else 0) + 1 + ((-(-len(giants) // 64)) * p + 1 if giants else 0)


def banded(n, w):
    return sorted({k % n for k in range(-w, w + 1)})


def offset_sets(n, seed):
    """(offsets, n1): {0} alone, babies only, giants only (n1 = 1), banded +-40, random sparse"""
    rng = np.random.default_rng(seed)
    sparse = sorted(int(k) for k in rng.choice(n, 12, replace=False))
    return [([0], 8), ([1, 2, 5, 7], 8), ([0, 3, 7, n - 2], 1), (banded(n, 40), 9), (sparse, 16)]


# ------------------------------------------------------------------ CPU: the schedule
def test_lintrans_galois_against_enumeration(lib):
    for n, offs, n1 in ((4096, [0], 1), (4096, [0, 1, 2, 17, 40], 8), (8192, banded(4096, 40), 9),
                        (4096, list(range(2048)), 64), (65536, [5, 32767, 100], 1), (16384, [3, 64, 129], 64)):
        babies = sorted({k % n1 for k in offs} - {0})
        giants = sorted({k // n1 for k in offs} - {0})
        want = [pow(5, j, 2 * n) for j in babies] + [pow(5, n1 * i, 2 * n) for i in giants]
        assert lib.lintrans_galois(n, offs, n1) == want
        assert want == [lib.galois_rotation(n, r) for r in babies + [n1 * i for i in giants]]
    assert launches(12, 3, [0], 8) == 1 and launches(13, 1, list(range(4096)), 32) == 11 + 1 + 2 * 11 + 1


@pytest.mark.parametrize("n1", [1, 7, 16, 64])
def test_bsgs_identity_on_slots(lib, n1):
    """W_i = sum_j rot_{-n1 i}(d_{n1 i + j}) * rot_j(z), y = W_0 + sum_i rot_{n1 i}(W_i) equals
    M z, the rotations read from the key list (5^r mod 2N -> r); dense, banded and random sparse
    diagonal sets (negative offsets written mod n), each of the two packed rows with its own M."""
    N = 4096
    n = N // 2
    dlog = {pow(5, r, 2 * N): r for r in range(n)}
    rng = np.random.default_rng(4100 + n1)
    rot = lambda v, r: np.roll(v, -r)   # rot_r(v)[s] = v[(s + r) mod n]
    for offs in (list(range(n)), banded(n, 40), sorted({int(k) % n for k in rng.integers(-n, n, 30)})):
        babies, giants, terms = schedule(offs, n1)
        gal = lib.lintrans_galois(N, offs, n1)
        assert [dlog[g] for g in gal] == babies + [n1 * i for i in giants]
        for _row in range(2):
            M = np.zeros((n, n), dtype=np.complex128)
            s = np.arange(n)
            for k in offs:
                M[s, (s + k) % n] = rng.normal(size=n) + 1j * rng.normal(size=n)
            d = {k: M[s, (s + k) % n] for k in offs}
            z = rng.normal(size=n) + 1j * rng.normal(size=n)
            y = np.zeros(n, dtype=np.complex128)
            for i, tl in terms.items():
                w = sum(rot(d[offs[c]], -n1 * i) * rot(z, j) for j, c in tl)
                y += rot(w, n1 * i)
            assert np.allclose(y, M @ z, rtol=0, atol=1e-9 * n)


def test_argument_checks_without_device(lib):
    Lb = lib.load_library()
    u32 = ctypes.c_uint32
    offs = (u32 * 3)(0, 1, 9)
    nk = u32(77)
    assert Lb.nttb200_rns_lintrans_keys(12, offs, 3, 8, None, ctypes.byref(nk)) == OK and nk.value == 2
    for args in ((12, None, 3, 8), (12, offs, 0, 8), (12, offs, 3, 0), (12, offs, 3, 65), (11, offs, 3, 8),
                 (17, offs, 3, 8), (12, (u32 * 3)(0, 1, 1), 3, 8), (12, (u32 * 2)(0, 2048), 2, 8),
                 (13, (u32 * 2)(4095, 4096), 2, 8)):
        assert Lb.nttb200_rns_lintrans_keys(*args, None, ctypes.byref(nk)) == INVALID_ARG, args
    assert Lb.nttb200_rns_lintrans_keys(12, offs, 3, 8, None, None) == INVALID_ARG
    assert Lb.nttb200_rns_lintrans_apply(None, 16, 16, offs, 3, 8, 16, 2, 16, 1, None) == INVALID_ARG
    assert Lb.nttb200_rns_lintrans_apply(None, None, None, offs, 3, 8, None, 2, None, 0, None) == INVALID_ARG
    with pytest.raises(lib.NttError):
        lib.lintrans_galois(4096, [0, 0], 4)


# ------------------------------------------------------------------------- GPU helpers
def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"
    return torch


def composed(env, ct, diags, offs, n1, keys, batch):
    """The existing calls: ct [batch][2][L][N], diags [count][L][N], keys in the lintrans_galois
    order, all in the rns_ct order -> y [batch][2][L][N]."""
    torch, lib = _torch(), env.lib
    L, n = env.L, env.n
    babies, giants, terms = schedule(offs, n1)
    gal = lib.lintrans_galois(n, offs, n1)
    nb = len(babies)
    new = lambda *shape: torch.empty(shape, dtype=torch.int32, device="cuda")

    def rotate_ct(c0, u, g):   # (sigma_g(c0) + u0, u1)
        r = new(batch, 2, L, n)
        s0 = new(batch, L, n)
        env.qf.automorphism(c0.contiguous(), s0, batch, g)
        u0 = u[:, 0].contiguous()
        env.qf.pointwise(ADD, s0, u0, u0, batch)
        r[:, 0], r[:, 1] = u0, u[:, 1]
        return r

    R = {0: ct}
    if nb:
        U = new(nb, batch, 2, L, n)
        env.ks.switch(ct[:, 1], keys[:nb], U, batch, gal[:nb], in_stride=2 * L * n)
        for b, j in enumerate(babies):
            R[j] = rotate_ct(ct[:, 0], U[b], gal[b])
    W = {}
    for i, tl in terms.items():
        acc = torch.zeros((batch, 2, L, n), dtype=torch.int32, device="cuda")
        pd = new(1, L, n)
        prod = new(batch, 2, L, n)
        for j, c in tl:
            env.qf.automorphism(diags[c:c + 1], pd, 1, lib.galois_rotation(n, -n1 * i))
            env.qf.pointwise(MUL, R[j].contiguous(), pd, prod, 2 * batch, b_batch=1)
            env.qf.pointwise(ADD, acc, prod, acc, 2 * batch)
        W[i] = acc
    y = W.get(0, torch.zeros((batch, 2, L, n), dtype=torch.int32, device="cuda"))
    for c, i in enumerate(giants):
        V = new(1, batch, 2, L, n)
        env.ks.switch(W[i][:, 1], keys[nb + c:nb + c + 1].contiguous(), V, batch, gal[nb + c], in_stride=2 * L * n)
        env.qf.pointwise(ADD, y, rotate_ct(W[i][:, 0], V[0], gal[nb + c]), y, 2 * batch)
    return y


def check_call(env, ct, diags, offs, n1, keys, batch):
    """one call into a guarded output against the composed sequence, inputs unchanged, launches"""
    torch, lib = _torch(), env.lib
    want = composed(env, ct, diags, offs, n1, keys, batch)
    snaps = [x.clone() for x in (ct, diags, keys)]
    out = Guarded(batch * 2 * env.L * env.n)
    before = lib.kernel_launches()
    env.ks.linear_transform(ct, diags, offs, n1, keys, out.view, batch)
    assert lib.kernel_launches() - before == launches(env.logn, env.ks.dnum, offs, n1)
    assert torch.equal(out.view.view(want.shape), want), (offs[:4], n1, batch)
    assert out.guards_intact()
    assert all(torch.equal(a, b) for a, b in zip((ct, diags, keys), snaps))


# ------------------------------------------------------------ GPU: bit-exact, composed
@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 13, 14, 15, 16])
@pytest.mark.parametrize("L,K,alpha", CONFIGS)
def test_bit_exact_against_composed(lib, logn, L, K, alpha):
    """{0} alone, babies only, giants only, banded +-40 and random sparse, batch 1 and 3, random
    (not necessarily valid) keys."""
    env = Env(lib, logn, L, K, alpha)
    n, LK, dn = env.n, L + K, env.ks.dnum
    seed = 71000 + 100 * logn + L
    ct = rand_rns((3, 2, L, n), env.qs[:L], seed)
    for s, (offs, n1) in enumerate(offset_sets(n // 2, seed)):
        nk = len(lib.lintrans_galois(n, offs, n1))
        diags = rand_rns((len(offs), L, n), env.qs[:L], seed + 10 + s)
        keys = rand_rns((max(nk, 1), dn, 2, LK, n), env.qs, seed + 20 + s)
        for batch in (1, 3):
            check_call(env, ct[:batch], diags, offs, n1, keys, batch)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("logn,n1", [(12, 64), (13, 32)])
def test_bit_exact_dense(lib, logn, n1):
    """All N/2 offsets: at N = 4096 with n1 = 64 (63 babies, 31 giants), at N = 2^13 with n1 = 32
    (127 giants: two key-switch passes of the giants)."""
    L, K, alpha = 3, 1, 1
    env = Env(lib, logn, L, K, alpha)
    n = env.n
    offs = list(range(n // 2))
    nk = len(lib.lintrans_galois(n, offs, n1))
    assert (logn == 12) or len(schedule(offs, n1)[1]) > 64
    ct = rand_rns((3, 2, L, n), env.qs[:L], 72000 + logn)
    diags = rand_rns((len(offs), L, n), env.qs[:L], 72001 + logn)
    keys = rand_rns((nk, env.ks.dnum, 2, L + K, n), env.qs, 72002 + logn)
    for batch in (1, 3):
        check_call(env, ct[:batch], diags, offs, n1, keys, batch)
    env.close()


@pytest.mark.gpu
def test_bit_exact_beyond_l2(lib):
    """N = 2^16, (L, K, alpha) = (24, 8, 8), batch 4, 16 banded diagonals with n1 = 4."""
    logn, L, K, alpha, batch = 16, 24, 8, 8, 4
    env = Env(lib, logn, L, K, alpha)
    n = env.n
    offs = banded(n // 2, 8)[:16]
    nk = len(lib.lintrans_galois(n, offs, 4))
    ct = rand_rns((batch, 2, L, n), env.qs[:L], 73000)
    diags = rand_rns((len(offs), L, n), env.qs[:L], 73001)
    keys = rand_rns((nk, env.ks.dnum, 2, L + K, n), env.qs, 73002)
    assert (ct.numel() + diags.numel() + keys.numel()) * 4 > 126 << 20
    check_call(env, ct, diags, offs, 4, keys, batch)
    env.close()


# ------------------------------------------------------------- GPU: end to end
def matrix_diagonals(M, offs):
    n = M.shape[0]
    s = np.arange(n)
    return np.stack([M[s, (s + k) % n] for k in offs])


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 13])
@pytest.mark.parametrize("shape", ["dense", "banded"])
def test_ckks_end_to_end(lib, logn, shape):
    """Encode, encrypt, transform, rescale by the last prime, decode: y = M z within 1e-3.  Noise
    estimate: the fresh and key-switching noise is below 2^16 per coefficient at Delta = 2^34, so
    below 2^-18 sqrt(N) per slot after the product with |d_k| <= 1/sqrt(count) summed over the
    terms; the encoding of the diagonals at Delta_pt = 2^30 adds below sqrt(N) 2^-31 per term and
    the rescale below sqrt(N) 2^-34: together below 1e-4."""
    torch = _torch()
    L, K, alpha = 3, 2, 2
    env = Env(lib, logn, L, K, alpha)
    keys = Keys(lib, logn, env.qs[:L], 74000 + logn)
    n, slots, qs = env.n, env.n // 2, env.qs
    rng = np.random.default_rng(74100 + logn)
    offs = list(range(slots)) if shape == "dense" else banded(slots, 20)
    n1 = 64 if shape == "dense" else 6
    M = np.zeros((slots, slots), dtype=np.complex128)
    s = np.arange(slots)
    for k in offs:
        M[s, (s + k) % slots] = (rng.uniform(-1, 1, slots) + 1j * rng.uniform(-1, 1, slots)) / (2 * len(offs))
    z = rng.uniform(-1, 1, slots) + 1j * rng.uniform(-1, 1, slots)
    gal = lib.lintrans_galois(n, offs, n1)
    rk = host_keys(env, keys.s, [sigma_int(keys.s, g) for g in gal], 74200 + logn)
    scale, pscale = 2.0 ** 34, 2.0 ** 30
    with lib.CkksEncoder(keys.pf) as enc:
        m = torch.empty((1, L, n), dtype=torch.int32, device="cuda")
        enc.encode(torch.from_numpy(z[None]).cuda(), m, 1, scale)
        ct = keys.encrypt(m, 1)
        env.qf.ct(ct, ct, 2)
        d = matrix_diagonals(M, offs)
        diags = torch.empty((len(offs), L, n), dtype=torch.int32, device="cuda")
        enc.encode(torch.from_numpy(d).cuda(), diags, len(offs), pscale)
        env.qf.ct(diags, diags, len(offs))
    y = torch.empty((1, 2, L, n), dtype=torch.int32, device="cuda")
    env.ks.linear_transform(ct[None], diags, offs, n1, rk, y, 1)
    r = y[0].clone()
    env.qi.gs_scaled(r, r, 2)
    from test_rns_eval import ones_plan
    res = torch.empty((2, L - 1, n), dtype=torch.int32, device="cuda")
    with ones_plan(lib, logn, qs[L - 1:L]) as top, ones_plan(lib, logn, qs[:L - 1]) as low, \
            lib.RnsConv(top, low) as rescale:
        rescale.mod_down(r, res, 2, round=True)
    k2 = Keys(lib, logn, qs[:L - 1], 1)
    k2.s = keys.s
    k2.s_res = to_dev(np.stack([keys.s % q for q in qs[:L - 1]])[None])
    with lib.CkksEncoder(k2.pf) as enc2:
        dec = torch.empty((1, slots), dtype=torch.complex128, device="cuda")
        enc2.decode(k2.decrypt(res), dec, 1, scale * pscale / qs[L - 1])
    err = np.abs(dec.cpu().numpy()[0] - M @ z).max()
    assert err < 1e-3, err
    k2.close()
    keys.close()
    env.close()


@pytest.mark.gpu
def test_bfv_end_to_end(lib):
    """BFV at N = 4096, t = 65537: one random N/2 x N/2 matrix per packed row, diagonals encoded
    centred; decryption and decode give exactly M_r z_r mod t for both rows."""
    torch = _torch()
    logn, t, Lq = 12, 65537, 4
    N, n = 1 << logn, 1 << (logn - 1)
    primes = channels(Lq + 2, t)
    qs, sp = primes[:Lq], primes[Lq:]
    keys = Keys(lib, logn, qs, 75000)
    env = Env(lib, logn, Lq, 2, 2, qs=qs + sp)
    rng = np.random.default_rng(75100)
    offs, n1 = list(range(n)), 64
    Ms = [rng.integers(0, t, (n, n)) for _ in range(2)]
    zs = [rng.integers(0, t, n) for _ in range(2)]
    want = np.concatenate([(M.astype(object) @ z.astype(object)) % t for M, z in zip(Ms, zs)]).astype(np.int64)
    d = np.concatenate([matrix_diagonals(M, offs) for M in Ms], axis=1)   # [count][2 n]: both rows
    gal = lib.lintrans_galois(N, offs, n1)
    rk = host_keys(env, keys.s, [sigma_int(keys.s, g) for g in gal], 75200)
    with lib.PackedEncoder(keys.pf, t) as enc:
        pt = torch.empty((1, Lq, N), dtype=torch.int32, device="cuda")
        enc.encode(torch.from_numpy(np.concatenate(zs).astype(np.int32)[None]).cuda(), pt, 1)
        ct = keys.encrypt(pt, 1)
        env.qf.ct(ct, ct, 2)
        diags = torch.empty((len(offs), Lq, N), dtype=torch.int32, device="cuda")
        enc.encode(torch.from_numpy(d.astype(np.int32)).cuda(), diags, len(offs), centred=True)
        env.qf.ct(diags, diags, len(offs))
        y = torch.empty((1, 2, Lq, N), dtype=torch.int32, device="cuda")
        env.ks.linear_transform(ct[None], diags, offs, n1, rk, y, 1)
        r = y[0].clone()
        env.qi.gs_scaled(r, r, 2)
        out = torch.empty((1, N), dtype=torch.int32, device="cuda")
        enc.decode(decrypt_to_t(lib, keys.decrypt(r), qs, t, True), out, 1)
    assert np.array_equal(signed(out)[0], want)
    keys.close()
    env.close()


# --------------------------------------------------------------- GPU: rules
@pytest.mark.gpu
def test_errors_batch_zero_and_alignment(lib):
    """Every error code, each with nothing launched and nothing written; batch 0 -> OK."""
    torch = _torch()
    logn, L, K, alpha, batch = 12, 3, 2, 2, 2
    env = Env(lib, logn, L, K, alpha)
    n, LK, dn, ks = env.n, L + K, env.ks.dnum, env.ks
    offs, n1 = [0, 1, 9], 8
    nk = len(lib.lintrans_galois(n, offs, n1))
    ct = rand_rns((batch, 2, L, n), env.qs[:L], 76000)
    diags = rand_rns((3, L, n), env.qs[:L], 76001)
    keys = rand_rns((nk, dn, 2, LK, n), env.qs, 76002)
    words = batch * 2 * L * n
    out = Guarded(words)
    Lb = lib.load_library()
    u32 = ctypes.c_uint32
    arr = lambda v: (u32 * len(v))(*v)
    call = lambda c, d, o, cnt, m, k, nkeys, y, b: Lb.nttb200_rns_lintrans_apply(
        ks._h, c, d, arr(o), cnt, m, k, nkeys, y, b, None)
    p = lambda x: x.data_ptr()
    before = lib.kernel_launches()
    for b in (batch, 0):
        assert call(p(ct), p(diags), offs, 3, n1, p(keys), nk - 1, p(out.view), b) == INVALID_ARG   # a missing key
        assert call(p(ct), p(diags), offs, 3, n1, p(keys), nk + 1, p(out.view), b) == INVALID_ARG   # a surplus key
        assert call(p(ct), p(diags), offs, 3, 0, p(keys), nk, p(out.view), b) == INVALID_ARG
        assert call(p(ct), p(diags), offs, 3, 65, p(keys), nk, p(out.view), b) == INVALID_ARG
        assert call(p(ct), p(diags), [0, 1, 1], 3, n1, p(keys), nk, p(out.view), b) == INVALID_ARG
        assert call(p(ct), p(diags), [0, 1, n // 2], 3, n1, p(keys), nk, p(out.view), b) == INVALID_ARG
        assert call(p(ct), p(diags), offs, 0, n1, p(keys), nk, p(out.view), b) == INVALID_ARG
        assert Lb.nttb200_rns_lintrans_apply(ks._h, p(ct), p(diags), None, 3, n1, p(keys), nk, p(out.view), b,
                                             None) == INVALID_ARG
    for c, d, k, y in ((None, p(diags), p(keys), p(out.view)), (p(ct), None, p(keys), p(out.view)),
                       (p(ct), p(diags), None, p(out.view)), (p(ct), p(diags), p(keys), None)):
        assert call(c, d, offs, 3, n1, k, nk, y, batch) == INVALID_ARG
    assert call(None, None, offs, 3, n1, None, nk, None, 0) == OK
    big = Guarded(2 * words + 3 * L * n + nk * dn * 2 * LK * n)
    v = big.view
    ck, dk, kk = words, 3 * L * n, nk * dn * 2 * LK * n
    for c, d, k, y in ((v[:ck], diags, keys, v[ck - 4:]), (ct, v[:dk], keys, v[dk - 4:]),
                       (ct, diags, v[:kk], v[kk - 4:]), (v[words:], diags, keys, v[4:])):
        assert call(p(c), p(d), offs, 3, n1, p(k), nk, p(y), batch) == INVALID_ARG
    for kw in (1, 2, 3):
        uc, ud, uk, uo = (Guarded(ct.numel(), kw, ct), Guarded(diags.numel(), kw, diags),
                          Guarded(keys.numel(), kw, keys), Guarded(words, kw))
        for c, d, k, y in ((uc.view, diags, keys, out.view), (ct, ud.view, keys, out.view),
                           (ct, diags, uk.view, out.view), (ct, diags, keys, uo.view)):
            assert call(p(c), p(d), offs, 3, n1, p(k), nk, p(y), batch) == UNSUPPORTED, kw
        torch.cuda.synchronize()
        assert uo.untouched()
    assert lib.kernel_launches() == before
    torch.cuda.synchronize()
    assert out.untouched() and big.untouched()
    ks.linear_transform(ct, diags, offs, n1, keys, out.view, batch)
    assert out.guards_intact() and not out.untouched()
    # one diagonal at offset 0 needs no key and is one launch
    before = lib.kernel_launches()
    ks.linear_transform(ct, diags[:1], [0], 1, None, out.view, batch)
    assert lib.kernel_launches() - before == 1
    assert _status(lib, lambda: ks.linear_transform(ct, diags, [0, 1, 1], n1, keys, out.view, batch)) == INVALID_ARG
    env.close()
