"""Every transform, product and RNS kernel at the edges of its modulus range.

Each kernel is correct because of a range argument: the classic butterflies keep values in
[0, 2q) / [0, 4q), which touches 2^32 at q = 2^30; the 4q-lazy (L4) butterflies let sums grow to
8q, which touches 2^32 at q = 2^29 - 3; rns_dot and the conversion kernel fold 64-bit sums whose
bounds are tightest at q = 2^30; RNS channels may be any modulus in [2, 2^30].  This file runs
every kernel family at the moduli where those arguments are tight:

  2^30             top of the classic domain, 4q = 2^32 (even: transforms only)
  2^30 - 35        odd, classic
  2^29, 2^29 + 1   the first moduli back on the classic kernels (2^29 even)
  2^29 - 1, 2^29 - 3   the L4 limit, 8q within 24 of 2^32
  2, 3             tiny moduli, where the lazy offsets dominate

with tables that have every other entry at q - 1 and a few at 0 (the kernels do not care which
table they get), and inputs with rows all q - 1, all 0 and random.  Every result is compared for
integer equality with the C oracle, numpy uint64 or Python-int CRT, and every single-modulus case
asserts the kernel path that ran: a case that lands on the generic kernel tests nothing.  The
helpers (moduli, tables, inputs, the fold bounds) are checked on the CPU."""
import math
import random
from fractions import Fraction

import numpy as np
import pytest

from test_gpu_parity import dev, run_gs
from test_multigpu_cpu import gs_stage_range_numpy
from test_rns_automorph import COEFF, EVAL, reference as automorph_reference
from test_rns_conv import Consts, convert_ref, crt, mod_down_ref, overshoot, residues, to_dev
from test_rns_eval import Guarded, host, ones_plan, rand_rns
from test_rns_exact import centred, exact_ref, scale_round_ref

ADD, SUB, MUL = 0, 1, 2

# ---------------------------------------------------------------------------- the moduli
EDGES = {
    "2^30": 1 << 30,
    "2^30-35": (1 << 30) - 35,
    "2^29+1": (1 << 29) + 1,
    "2^29": 1 << 29,
    "2^29-1": (1 << 29) - 1,
    "2^29-3": (1 << 29) - 3,
    "3": 3,
    "2": 2,
}
NAME = {q: name for name, q in EDGES.items()}
ALL = list(EDGES.values())
ODD = [q for q in ALL if q & 1]
L4_LIMIT = [(1 << 29) - 1, (1 << 29) - 3]


def is_prime(n):
    """Deterministic Miller-Rabin for n < 3.3 * 10^24."""
    if n < 2:
        return False
    small = (2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37, 41)
    for p in small:
        if n % p == 0:
            return n == p
    d, s = n - 1, 0
    while d % 2 == 0:
        d, s = d // 2, s + 1
    for a in small:
        x = pow(a, d, n)
        if x in (1, n - 1):
            continue
        for _ in range(s - 1):
            x = x * x % n
            if x == n - 1:
                break
        else:
            return False
    return True


def primes_below(limit, count):
    """The `count` largest primes below `limit`, largest first."""
    out, k = [], limit - 1
    while len(out) < count:
        if is_prime(k):
            out.append(k)
        k -= 1
    return out


# RNS channel sets: odd moduli for every operation; with the even ones for GS and CT; 32 channels
# that alternate odd moduli near 2^30 with small odd moduli (a channel-indexing mix-up between
# neighbours cannot go unnoticed there)
RNS_ODD = [(1 << 30) - 35, (1 << 30) - 1, (1 << 29) + 1, (1 << 29) - 1, (1 << 29) - 3, 3, 12289]
RNS_FULL = RNS_ODD + [1 << 30, 1 << 29, 2]
RNS_MIXED = [x for k in range(16) for x in ((1 << 30) - 1 - 2 * k, 3 + 2 * k)]
RNS_SETS = {"odd": RNS_ODD, "full": RNS_FULL, "mixed32": RNS_MIXED}
# the evaluation-domain operators: the top of the domain, an odd classic modulus, the tiny ones
EVAL_QS = [1 << 30, (1 << 30) - 35, 3, 2]


def edge_table(rng, n, q):
    """A table in [0, q): random, every other entry at q - 1, a few at 0."""
    t = rng.integers(0, q, n, dtype=np.int64)
    t[1::2] = q - 1
    t[rng.integers(0, n, 4) & ~1] = 0
    return t.astype(np.int32)


def edge_rows(rng, batch, n, q):
    """[batch][n]: row 0 all q - 1, row 1 all 0, the others random; a single row is q - 1 in its
    first half and random in its second."""
    a = rng.integers(0, q, (batch, n), dtype=np.int64).astype(np.int32)
    if batch == 1:
        a[0, :n // 2] = q - 1
        return a
    a[0] = q - 1
    a[1] = 0
    return a


def oracle_product(om, a, b, fwd, inv, q):
    """The negacyclic product pipeline of the oracle: CT, CT, pointwise, GS, N^-1."""
    n = a.shape[-1]
    prod = om.pointwise(om.ntt_ct(a, fwd, q), om.ntt_ct(b, fwd, q), q)
    return om.scale(om.ntt_gs(prod, inv, q), pow(n, -1, q), q)


def dot_fold_peak(q):
    """The largest 64-bit sum rns_dot reaches: an accumulator below q plus 16 products."""
    return (q - 1) + 16 * (q - 1) ** 2


# ------------------------------------------------------------------- CPU: the helpers
def test_edge_moduli_sit_where_the_range_arguments_are_tight():
    assert ALL == sorted(ALL, reverse=True) and len(set(ALL)) == len(ALL)
    assert max(ALL) == 1 << 30 and 4 * max(ALL) == 1 << 32            # classic: 4q fills a word
    assert [q for q in ALL if q & 1 == 0] == [1 << 30, 1 << 29, 2]
    for q in L4_LIMIT:                                                 # L4: 8q within 24 of 2^32
        assert q < 1 << 29 and 0 < (1 << 32) - 8 * q <= 24
    assert min(q for q in ALL if q >= 1 << 29) == 1 << 29              # first classic modulus
    assert 8 * ((1 << 29) + 1) > 1 << 32                               # where 8q no longer fits
    assert NAME[(1 << 29) - 3] == "2^29-3" and NAME[2] == "2"


def test_rns_channel_sets():
    for name, qs in RNS_SETS.items():
        assert all(2 <= q <= 1 << 30 for q in qs), name
        assert len(qs) <= 32
    assert all(q & 1 for q in RNS_ODD + RNS_MIXED)
    assert set(RNS_FULL) - set(RNS_ODD) == {1 << 30, 1 << 29, 2}
    assert len(RNS_MIXED) == 32 and len(set(RNS_MIXED)) == 32
    assert all(q > (1 << 30) - 64 for q in RNS_MIXED[0::2]) and all(q < 64 for q in RNS_MIXED[1::2])


@pytest.mark.parametrize("q", ALL, ids=lambda q: f"q={NAME[q]}")
def test_edge_tables_and_rows(q):
    rng = np.random.default_rng(q)
    n = 1 << 12
    t = edge_table(rng, n, q)
    assert t.dtype == np.int32 and t.min() >= 0 and t.max() == q - 1
    assert (t[1::2] == q - 1).all() and (t == 0).any()
    a = edge_rows(rng, 5, n, q)
    assert (a[0] == q - 1).all() and (a[1] == 0).all()
    assert a.min() >= 0 and a.max() < q
    one = edge_rows(rng, 1, n, q)
    assert (one[0, :n // 2] == q - 1).all() and one.max() < q


def test_primes_and_conversion_bases():
    assert [is_prime(x) for x in (2, 3, 4, 12289, 469762049, (1 << 31) - 1, 1 << 30, 561)] == \
        [True, True, False, True, True, True, False, False]
    assert primes_below(1 << 30, 3) == [(1 << 30) - 35, (1 << 30) - 41, (1 << 30) - 83]
    bs, cs = conv_bases()
    assert len(bs) == 32 and len(set(bs)) == 32 and max(bs) < 1 << 30
    assert cs[0] == 1 << 30 and cs[1] == 3 and cs[2] < min(bs) and is_prime(cs[2])
    assert all(math.gcd(b, c) == 1 for b in bs for c in cs)


def test_dot_fold_bound_is_tightest_at_2_30():
    """The 16-term fold of rns_dot: q + 16 (q-1)^2 fits 64 bits for every q <= 2^30, with the
    least room at 2^30 (2^64 - 2^35 + 2^30 + 15); 17 terms would not fit there."""
    assert dot_fold_peak(1 << 30) == (1 << 64) - (1 << 35) + (1 << 30) + 15
    for q in ALL + RNS_MIXED:
        assert dot_fold_peak(q) <= dot_fold_peak(1 << 30) < 1 << 64
    assert 17 * ((1 << 30) - 1) ** 2 > 1 << 64


# --------------------------------------------------------------------- GPU helpers
def _torch():
    import torch
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"
    return torch


def device_rows(rng_seed, batch, n, q):
    """Like edge_rows, generated on the device (the persistent kernels need 896 rows)."""
    torch = _torch()
    gen = torch.Generator(device="cuda").manual_seed(rng_seed)
    a = torch.randint(0, q, (batch, n), dtype=torch.int32, device="cuda", generator=gen)
    a[0] = q - 1
    a[1] = 0
    return a


def sample(batch):
    return sorted({0, 1, batch // 2, batch - 1} & set(range(batch)))


def case_id(q, logn, batch, op):
    return f"q={NAME[q]}-logn={logn}-batch={batch}-{op}"


# ------------------------------------------------- A. single modulus, N >= 2^17
A_SHAPES = [(17, 3), (17, 65), (18, 3), (20, 3)]
A_CASES = [(q, logn, batch, op) for logn, batch in A_SHAPES for q in ALL
           for op in ("gs", "ct", "polymul", "gs_inplace") + (("stage_range",) if q in (1 << 30, (1 << 29) - 3) else ())
           if op != "polymul" or q & 1]
A_CASES += [(q, 22, 1, op) for q in (1 << 30, (1 << 29) - 3) for op in ("gs", "ct")]
A_PATH = {"gs": "tile_tma + column_passes", "gs_inplace": "tile_tma + column_passes",
          "ct": "column_passes_ct + tile_tma_ct", "polymul": "tile_tma_dual + column_passes",
          "stage_range": "column_passes"}


@pytest.mark.gpu
@pytest.mark.parametrize("q,logn,batch,op", A_CASES, ids=[case_id(*c) for c in A_CASES])
def test_large_n_single_modulus(lib, oracle_mod, q, logn, batch, op):
    """The tile pass and the column passes (logn 17: one column pass of 5 stages, 18: one of 6,
    20: two of 4; batch 65 takes the per-segment shared-memory twiddles) at every edge modulus."""
    torch = _torch()
    om = oracle_mod
    n = 1 << logn
    rng = np.random.default_rng(40000 + 97 * logn + batch + q % 1009)
    table = edge_table(rng, n, q)
    a = edge_rows(rng, batch, n, q)
    if op in ("gs", "gs_inplace"):
        got, path = run_gs(lib, a, table, q, inplace=(op == "gs_inplace"))
        want = om.ntt_gs(a, table, q)
    elif op == "ct":
        d_a = dev(a)
        d_o = torch.empty_like(d_a)
        with lib.Plan(logn, q, table) as plan:
            plan.ct(d_a, d_o, batch)
            torch.cuda.synchronize()
            path = plan.last_path
        got, want = d_o.cpu().numpy(), om.ntt_ct(a, table, q)
    elif op == "polymul":
        inv = edge_table(rng, n, q)
        b = edge_rows(rng, batch, n, q)[::-1].copy()
        d_c = torch.empty(batch, n, dtype=torch.int32, device="cuda")
        with lib.Plan(logn, q, table) as pf, lib.Plan(logn, q, inv) as pi:
            lib.polymul_negacyclic(pf, pi, dev(a), dev(b), d_c, batch)
            torch.cuda.synchronize()
            path = pi.last_path
        got, want = d_c.cpu().numpy(), oracle_product(om, a, b, table, inv, q)
    else:
        d_a = dev(a)
        d_o = torch.empty_like(d_a)
        with lib.Plan(logn, q, table) as plan:
            for sb, se in ((2, logn), (12, logn), (3, logn - 1)):
                plan.gs_stage_range(d_a, d_o, batch, sb, se)
                torch.cuda.synchronize()
                assert plan.last_path == A_PATH[op], plan.last_path
                want = np.stack([gs_stage_range_numpy(x, table, q, sb, se) for x in a])
                assert np.array_equal(d_o.cpu().numpy(), want), (sb, se)
        return
    assert path == A_PATH[op], path
    assert np.array_equal(got, want)


# ------------------------------------------------- B. single modulus, smaller N
B_CT = [(q, logn) for logn in (6, 7, 8, 9, 10, 11, 13, 15, 16) for q in ALL]
B_MUL = [(q, logn) for logn in (6, 7, 8, 9, 10, 11, 14, 15, 16) for q in ((1 << 30) - 35,) + tuple(L4_LIMIT)]
PERSISTENT_BATCH = 896   # 12 tiles per team * 148 SMs * 8 teams / 16 tiles = 888 at least


def small_path(logn, kind):
    if logn <= 11:
        return {"ct": "fused_ct_small_warp_tma", "polymul": "fused_gs_small_warp_tma_dual"}[kind]
    if logn <= 15:
        return {"ct": "poly_tmem_3round_ct", "polymul": "poly_tmem_3round_dual"}[kind]
    return {"ct": "tilecol_persistent_ct", "polymul": "tilecol_persistent_dual", "gs": "tilecol_persistent"}[kind]


def b_batch(logn, kind):
    """logn <= 11: two blocks of 2048 coefficients, plus one polynomial (a ragged tail) for CT;
    the product needs whole blocks.  logn 16: the persistent kernel's batch."""
    if logn <= 11:
        return 2 * (2048 >> logn) + (kind == "ct")
    return PERSISTENT_BATCH if logn == 16 else 3


def run_sampled(lib, om, q, logn, kind, table, inv=None, seed=0):
    """One call at b_batch(logn, kind); returns (path, got, want) on the compared rows (all rows
    below logn 16, sampled rows of the persistent kernel's batch)."""
    torch = _torch()
    n, batch = 1 << logn, b_batch(logn, kind)
    rng = np.random.default_rng(seed)
    if logn == 16:
        d_a = device_rows(seed, batch, n, q)
        d_b = device_rows(seed + 1, batch, n, q).flip(0).contiguous()
        rows = sample(batch)
    else:
        d_a, d_b = dev(edge_rows(rng, batch, n, q)), dev(edge_rows(rng, batch, n, q)[::-1].copy())
        rows = list(range(batch))
    d_o = torch.empty_like(d_a)
    idx = torch.tensor(rows, device="cuda")
    a, b = d_a[idx].cpu().numpy(), d_b[idx].cpu().numpy()
    if kind == "ct":
        with lib.Plan(logn, q, table) as plan:
            plan.ct(d_a, d_o, batch)
            torch.cuda.synchronize()
            path = plan.last_path
        want = om.ntt_ct(a, table, q)
    elif kind == "gs":
        with lib.Plan(logn, q, table) as plan:
            plan.gs(d_a, d_o, batch)
            torch.cuda.synchronize()
            path = plan.last_path
        want = om.ntt_gs(a, table, q)
    else:
        with lib.Plan(logn, q, table) as pf, lib.Plan(logn, q, inv) as pi:
            lib.polymul_negacyclic(pf, pi, d_a, d_b, d_o, batch)
            torch.cuda.synchronize()
            path = pi.last_path
        want = oracle_product(om, a, b, table, inv, q)
    return path, d_o[idx].cpu().numpy(), want


@pytest.mark.gpu
@pytest.mark.parametrize("q,logn", B_CT, ids=[case_id(q, l, b_batch(l, "ct"), "ct") for q, l in B_CT])
def test_forward_kernels_small_n(lib, oracle_mod, q, logn):
    """The warp-per-block forward kernel (logn 6-11, ragged tail), the one-pass tensor-memory
    kernel (13, 15) and the persistent kernel (16) at every edge modulus."""
    rng = np.random.default_rng(41000 + 31 * logn + q % 997)
    path, got, want = run_sampled(lib, oracle_mod, q, logn, "ct", edge_table(rng, 1 << logn, q),
                                  seed=41000 + logn)
    assert path == small_path(logn, "ct"), path
    assert np.array_equal(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("q,logn", B_MUL, ids=[case_id(q, l, b_batch(l, "polymul"), "polymul") for q, l in B_MUL])
def test_products_small_n(lib, oracle_mod, q, logn):
    """The small product kernels (logn 6-11), the DUAL one-pass product (14, 15) and the persistent
    DUAL kernel (16) at the classic edge and at the L4 limit."""
    rng = np.random.default_rng(42000 + 31 * logn + q % 997)
    n = 1 << logn
    path, got, want = run_sampled(lib, oracle_mod, q, logn, "polymul", edge_table(rng, n, q),
                                  edge_table(rng, n, q), seed=42000 + logn)
    assert path == small_path(logn, "polymul"), path
    assert np.array_equal(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("q", [1 << 30, 1 << 29], ids=lambda q: case_id(q, 16, PERSISTENT_BATCH, "gs"))
def test_persistent_gs_classic(lib, oracle_mod, q):
    """The persistent N = 2^16 transform on its classic butterflies: at the top of the domain and
    at the first modulus above the L4 kernels."""
    rng = np.random.default_rng(43000 + q % 997)
    path, got, want = run_sampled(lib, oracle_mod, q, 16, "gs", edge_table(rng, 1 << 16, q), seed=43000)
    assert path == small_path(16, "gs"), path
    assert np.array_equal(got, want)


# ------------------------------------------------------------------ C. RNS transforms
C_CASES = [(s, logn, batch) for s in RNS_SETS for logn in (12, 13, 14, 15, 16) for batch in (1, 7, 65)]


def rns_tables(lib_seed, n, qs):
    rng = np.random.default_rng(lib_seed)
    return [edge_table(rng, n, q) for q in qs], [edge_table(rng, n, q) for q in qs]


def rns_edge_data(shape, qs, seed):
    """rand_rns with polynomial 0 at q_l - 1 and polynomial 1 at 0 on every channel (a single
    polynomial: q_l - 1 in its first half); every other row pinned at its first 32 coefficients."""
    torch = _torch()
    x = rand_rns(shape, qs, seed)
    qm1 = torch.tensor(qs, dtype=torch.int32, device="cuda").view(len(qs), 1) - 1
    if shape[0] == 1:
        x[0, :, :shape[-1] // 2] = qm1
        return x
    x[0] = qm1
    x[1] = 0
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("chan,logn,batch", C_CASES, ids=[f"{s}-logn={l}-batch={b}" for s, l, b in C_CASES])
def test_rns_transforms_at_the_edges(lib, oracle_mod, chan, logn, batch):
    """gs, ct, gs_scaled and rns_polymul_negacyclic (odd sets) per channel against the oracle, on
    sampled polynomials; one launch per transform at N = 4096 and two above, one per channel for
    the N = 4096 product."""
    torch = _torch()
    om = oracle_mod
    qs = RNS_SETS[chan]
    limbs, n = len(qs), 1 << logn
    odd = all(q & 1 for q in qs)
    fwd, inv = rns_tables(44000 + logn, n, qs)
    seed = 44000 + 100 * logn + batch + limbs
    a = rns_edge_data((batch, limbs, n), qs, seed)
    b = rns_edge_data((batch, limbs, n), qs, seed + 1).flip(0).contiguous()
    rows = sample(batch)
    idx = torch.tensor(rows, device="cuda")
    ha, hb = a[idx].cpu().numpy(), b[idx].cpu().numpy()
    out = torch.empty_like(a)
    per_transform = 1 if logn == 12 else 2
    with lib.RnsPlan(qs, fwd, logn=logn) as pf, lib.RnsPlan(qs, inv, logn=logn) as pi:
        ops = [("gs", pi.gs, lambda x, l: om.ntt_gs(x, inv[l], qs[l]), per_transform),
               ("ct", pf.ct, lambda x, l: om.ntt_ct(x, fwd[l], qs[l]), per_transform)]
        if odd:
            ops.append(("gs_scaled", pi.gs_scaled,
                        lambda x, l: om.scale(om.ntt_gs(x, inv[l], qs[l]), pow(n, -1, qs[l]), qs[l]),
                        per_transform))
        for name, call, ref, launches in ops:
            out.fill_(-1)
            before = lib.kernel_launches()
            call(a, out, batch)
            torch.cuda.synchronize()
            assert lib.kernel_launches() - before == launches, name
            got = out[idx].cpu().numpy()
            for l in range(limbs):
                assert np.array_equal(got[:, l], ref(ha[:, l], l)), (name, l, qs[l])
        if odd:
            out.fill_(-1)
            before = lib.kernel_launches()
            lib.rns_polymul_negacyclic(pf, pi, a, b, out, batch)
            torch.cuda.synchronize()
            assert lib.kernel_launches() - before == (limbs if logn == 12 else 3 * per_transform)
            got = out[idx].cpu().numpy()
            for l, q in enumerate(qs):
                want = oracle_product(om, ha[:, l], hb[:, l], fwd[l], inv[l], q)
                assert np.array_equal(got[:, l], want), ("polymul", l, q)


# ---------------------------------------------- D. RNS operators at 2^30 and tiny moduli
def qcol(qs):
    return np.array(qs, dtype=np.uint64)[:, None]


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 16])
def test_pointwise_and_scale_at_the_edges(lib, logn):
    """add / sub / mul with an own and a broadcast operand; scale by 0, 1 and q - 1."""
    torch = _torch()
    qs, n, batch = EVAL_QS, 1 << logn, 3
    a = rns_edge_data((batch, len(qs), n), qs, 45000 + logn)
    b = rns_edge_data((batch, len(qs), n), qs, 45001 + logn)
    b[0, :, n // 2:] = 0                 # q - 1 against 0 as well as against q - 1
    b[1, :, n // 2:] = torch.tensor(qs, dtype=torch.int32, device="cuda").view(-1, 1) - 1
    c = torch.empty_like(a)
    ha, hb, q = host(a), host(b), qcol(qs)
    want = {ADD: lambda y: (ha + y) % q, SUB: lambda y: (ha + q - y) % q, MUL: lambda y: ha * y % q}
    with ones_plan(lib, logn, qs) as rp:
        for op in (ADD, SUB, MUL):
            rp.pointwise(op, a, b, c, batch)
            assert np.array_equal(host(c), want[op](hb)), ("own", op)
            rp.pointwise(op, a, b[:1], c, batch, b_batch=1)
            assert np.array_equal(host(c), want[op](hb[:1])), ("broadcast", op)
        for j in range(3):
            scalars = [(0, 1, qv - 1)[(l + j) % 3] for l, qv in enumerate(qs)]
            rp.scale(a, c, batch, scalars)
            assert np.array_equal(host(c), ha * np.array(scalars, dtype=np.uint64)[:, None] % q), j


@pytest.mark.gpu
@pytest.mark.parametrize("terms", [16, 17, 64])
@pytest.mark.parametrize("shared_key", [False, True])
def test_dot_at_the_fold_bound(lib, terms, shared_key):
    """Every input at q - 1 (the largest sum before each fold: 2^64 - 2^35 + 2^30 + 15 on the 2^30
    channel) and random pinned inputs, accumulate off and on, against numpy reduced per term."""
    torch = _torch()
    qs, logn, batch = EVAL_QS, 12, 3
    n, limbs = 1 << logn, len(EVAL_QS)
    q = qcol(qs)
    w_batch = 1 if shared_key else batch
    qm1 = torch.tensor(qs, dtype=torch.int32, device="cuda").view(limbs, 1) - 1
    with ones_plan(lib, logn, qs) as rp:
        for extreme in (True, False):
            a = rand_rns((terms, batch, limbs, n), qs, 46000 + terms)
            w = rand_rns((terms, w_batch, limbs, n), qs, 46001 + terms)
            c0 = rand_rns((batch, limbs, n), qs, 46002 + terms)
            if extreme:
                for x in (a, w, c0):
                    x.copy_(qm1.expand_as(x))
            ha, hw, hc0 = host(a), np.broadcast_to(host(w), (terms, batch, limbs, n)), host(c0)
            for accumulate in (False, True):
                c = c0.clone()
                lib.rns_dot(rp, a, w, c, terms, batch, w_batch=w_batch, accumulate=accumulate)
                acc = hc0.copy() if accumulate else np.zeros_like(hc0)
                for k in range(terms):
                    acc = (acc + ha[k] * hw[k] % q) % q
                assert np.array_equal(host(c), acc), (extreme, accumulate)


@pytest.mark.gpu
@pytest.mark.parametrize("logn", [12, 13, 16])
def test_automorphism_at_the_edges(lib, logn):
    """Both domains on channels 2^30, 3 and 2: a 0 coefficient negates to 0, never to q."""
    torch = _torch()
    qs, batch = [1 << 30, 3, 2], 3
    n = 1 << logn
    x = rns_edge_data((batch, len(qs), n), qs, 47000 + logn)
    hx = host(x)
    gs = [5, pow(5, -1, 2 * n), 2 * n - 1, 2 * n - 3]
    with ones_plan(lib, logn, qs) as rp:
        for domain in (COEFF, EVAL):
            out = Guarded(len(gs) * x.numel())
            rp.automorphism(x, out.view, batch, gs, domain)
            got = out.view.view(len(gs), batch, len(qs), n).cpu().numpy().astype(np.uint64)
            assert np.array_equal(got, automorph_reference(hx, gs, qs, domain)), domain
            assert (got < qcol(qs)).all() and out.guards_intact()
            assert (got[:, 1] == 0).all()      # polynomial 1 is all zeros


# the conversion: 32 sources (the largest primes below 2^30), targets 2^30, 3 and a 30-bit prime
def conv_bases():
    ps = primes_below(1 << 30, 33)
    return ps[:32], [1 << 30, 3, ps[32]]


def in_band(num, den):
    """num / den within 2^-40 of 1/2 modulo 1: either neighbour may come back (DESIGN 3.6)."""
    return abs(Fraction(num % den, den) - Fraction(1, 2)) < Fraction(1, 1 << 40)


def conv_columns(k, n, seed, t=1):
    """Python ints in [0, B), one per column: the special values of the exact conversion, the
    columns whose y_i = [x_i t (B/b_i)^-1]_{b_i} are all b_i - 1 (the largest start of the HPS
    accumulator, v = S), and random values."""
    B = k.B
    lo, hi = (B * ((1 << 39) - 1)) >> 40, -((-B * ((1 << 39) + 1)) >> 40)
    top = crt([(b - 1) * pow(t * w, -1, b) % b for b, w in zip(k.bs, k.w)], k.bs)
    vals = [0, 1, -1, 2, -2, 12345, -12345, (1 << 40) + 3, -(1 << 40) - 3, lo, lo - 1, hi, hi + 1,
            top, B - 1, B // 2 + 1]
    vals += [B // 2 + d for d in (-(1 << 20), -1, 0, 1, 2, 1 << 20)]
    rng = random.Random(seed)
    return [v % B for v in vals] + [rng.randrange(B) for _ in range(n - len(vals))]


@pytest.mark.gpu
def test_conversion_at_the_edges(lib):
    """convert (fast and exact), mod_down (with and without ROUND) and scale_round (t = 1, 65537,
    2^32 - 1) from 32 primes just below 2^30 to {2^30, 3, a 30-bit prime}: numpy references on the
    columns outside the rounding band, Python-int CRT on every column."""
    torch = _torch()
    logn = 12
    n = 1 << logn
    bs, cs = conv_bases()
    k = Consts(bs, cs)
    C = math.prod(cs)
    xs = conv_columns(k, n, 48000)
    outside = np.array([not in_band(x, k.B) for x in xs])
    x = to_dev(residues(xs, bs)[None])
    out = torch.empty((1, 3, n), dtype=torch.int32, device="cuda")
    with ones_plan(lib, logn, bs) as pb, ones_plan(lib, logn, cs) as pc, lib.RnsConv(pb, pc) as cv:
        # fast: (x + alpha B) mod c_j, 0 <= alpha < S
        cv.convert(x, out, 1)
        got = host(out)[0]
        hx = host(x)
        assert np.array_equal(got, convert_ref(hx, k)[0])
        for col in range(0, n, 97):
            total, alpha = overshoot(xs[col], k)
            assert 0 <= alpha < 32 and [int(v) for v in got[:, col]] == [total % c for c in cs], col
        # exact: the centred x; inside the band either representative
        cv.convert(x, out, 1, exact=True)
        got = host(out)[0]
        assert np.array_equal(got[:, outside], exact_ref(hx, k)[0][:, outside])
        for col, v in enumerate(xs):
            xc = centred(v, k.B)
            want = [[xc % c for c in cs]]
            if not outside[col]:
                want.append([(xc - k.B if xc > 0 else xc + k.B) % c for c in cs])
            assert [int(r) for r in got[:, col]] in want, col
        # mod_down / scale_round read [T + S] channels, the targets first: X = x + B * y
        ys = [random.Random(48001 + col).randrange(C) for col in range(n)]
        ys[:4] = [0, C - 1, C - 1, 0]
        Xs = [xv + k.B * yv for xv, yv in zip(xs, ys)]
        X = to_dev(residues(Xs, cs + bs)[None])
        hX = host(X)
        for rnd in (False, True):
            cv.mod_down(X, out, 1, round=rnd)
            got = host(out)[0]
            assert np.array_equal(got, mod_down_ref(hX, k, rnd)[0]), rnd
            h = k.B // 2 if rnd else 0
            for col in range(0, n, 61):
                Xh = (Xs[col] + h) % (C * k.B)
                _, alpha = overshoot(Xh % k.B, k)
                assert [int(v) for v in got[:, col]] == [(Xh // k.B - alpha) % c for c in cs], (rnd, col)
        for t in (1, 65537, (1 << 32) - 1):
            Xt = [xv + k.B * yv for xv, yv in zip(conv_columns(k, n, 48002, t), ys)]
            Xd = to_dev(residues(Xt, cs + bs)[None])
            cv.scale_round(Xd, out, 1, t)
            got = host(out)[0]
            ok = np.array([not in_band(t * v, k.B) for v in Xt])
            assert np.array_equal(got[:, ok], scale_round_ref(host(Xd), k, t)[0][:, ok]), t
            for col, v in enumerate(Xt):
                r = (2 * t * v + k.B) // (2 * k.B)
                want = [[r % c for c in cs]]
                if not ok[col]:
                    want += [[(r - 1) % c for c in cs], [(r + 1) % c for c in cs]]
                assert [int(s) for s in got[:, col]] in want, (t, col)
