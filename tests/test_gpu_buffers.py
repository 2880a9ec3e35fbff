"""Offset views, guard bands and the AIE device order on every kernel path.

The ABI takes plain int32_t * device pointers, so callers pass views such as t[1:], chunks
at odd offsets or one RNS channel.  Every buffer here is a view inside a larger allocation
filled with a sentinel.  After each call, the words before and after every view must still
hold the sentinel, every out-of-place input must be unchanged and the result must equal the
CPU oracle.  Each case also asserts the kernel path that ran, which proves that both the
fast kernel (every view 16-byte aligned) and its fallback (a view 4, 8 or 12 bytes past
alignment) were exercised."""
import numpy as np
import pytest
import torch

from conftest import Q29, Q30, load_golden

pytestmark = pytest.mark.gpu

GUARD = 64        # sentinel words on each side of a view (256 B: the view base stays 16 B aligned)
SENTINEL = -1     # 0xffffffff as uint32 is >= q for every modulus: never a result
BIG = 1 << 23     # batches of more words than this are checked on sampled rows (CPU oracle cost)

# (layout, word offset of the input view, word offset of the output view); "aligned" first:
# for large batches its result is the reference of the other layouts
LAYOUTS = (("aligned", 0, 0), ("in", 1, 0), ("out", 0, 3), ("both", 2, 1),
           ("inplace", 0, 0), ("inplace", 3, 3))

GENERIC = "generic_stage_pass"
FUSED = "fused_gs4096_tma"
FUSED_BR = "fused_gs4096_tma_bitrev"
SMALL = "fused_gs_small_warp_tma"


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"


class Guarded:
    """`words` int32 on the device between two guard bands of the sentinel; `view` starts
    k words (4k bytes) past a 16-byte boundary."""

    def __init__(self, words, k=0, data=None):
        self.raw = torch.full((words + 2 * GUARD,), SENTINEL, dtype=torch.int32, device="cuda")
        self.k, self.words = k, words
        self.view = self.raw[GUARD + k:GUARD + k + words]
        assert self.view.data_ptr() % 16 == 4 * k
        if data is not None:
            if isinstance(data, np.ndarray):
                data = torch.from_numpy(np.ascontiguousarray(data, dtype=np.int32))
            self.view.copy_(data.reshape(-1))

    def guards_intact(self):
        head = self.raw[:GUARD + self.k]
        tail = self.raw[GUARD + self.k + self.words:]
        return bool((head == SENTINEL).all()) and bool((tail == SENTINEL).all())

    def untouched(self):
        return bool((self.raw == SENTINEL).all())


def run_checked(call, outs, ins):
    """call(), synchronise; the guards of every buffer hold and every input that is not
    also an output is unchanged."""
    snaps = [(b, b.view.clone()) for b in ins if all(b is not o for o in outs)]
    call()
    torch.cuda.synchronize()
    for b in list(ins) + list(outs):
        assert b.guards_intact(), "store outside the view"
    for b, s in snaps:
        assert torch.equal(b.view, s), "input modified"


def device_rows(batch, n, q, seed):
    """batch x n residues on the device, row 0 pinned at q - 1."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    a = torch.randint(0, q, (batch, n), dtype=torch.int32, device="cuda", generator=gen)
    a[0] = q - 1
    return a


def sample_rows(batch, n):
    """None (every row) when the oracle can take the whole batch, else a few rows
    including both ends."""
    if batch * n <= BIG:
        return None
    return sorted({0, 1, batch // 2, batch - 1})


def check_result(out, want, rows, ref, what):
    """out: [batch][n] device view.  want: oracle result of every row (rows None) or of
    `rows`; ref: the aligned run's whole result (or None for that run itself)."""
    if rows is None:
        assert np.array_equal(out.cpu().numpy(), want), what
    else:
        assert np.array_equal(out[rows].cpu().numpy(), want), what
        if ref is not None:
            assert torch.equal(out, ref), what


def check_layouts(plan, run, a, path, want, rows, layouts=LAYOUTS):
    """run(src_view, dst_view) for every layout; path(k_in, k_out) is the kernel path the
    plan must report."""
    ref = None
    for name, k_in, k_out in layouts:
        src = Guarded(a.numel(), k_in, a)
        dst = src if name == "inplace" else Guarded(a.numel(), k_out)
        run_checked(lambda: run(src.view, dst.view), [dst], [src])
        assert plan.last_path == path(k_in, k_out), (name, plan.last_path)
        out = dst.view.view(a.shape)
        check_result(out, want, rows, ref, name)
        if rows is not None and ref is None:
            ref = out.clone()
        del src, dst


def fast_when_aligned(fast):
    return lambda k_in, k_out: fast if k_in == 0 and k_out == 0 else GENERIC


def bitrev_index(n):
    logn = n.bit_length() - 1
    idx = np.arange(n)
    rev = np.zeros(n, dtype=np.int64)
    for b in range(logn):
        rev |= ((idx >> b) & 1) << (logn - 1 - b)
    return rev


def gs_stage_range_numpy(a, table, p, sb, se):
    """Stages [sb, se) of the golden network on the rows of a, vectorised (int64)."""
    a = a.astype(np.int64).copy()
    n = a.shape[-1]
    for s in range(sb, se):
        t, h = 1 << s, n >> (s + 1)
        v = a.reshape(-1, h, 2, t)
        w = table[h:2 * h].astype(np.int64)[None, :, None]
        x, y = v[:, :, 0, :].copy(), v[:, :, 1, :].copy()
        v[:, :, 0, :] = (x + y) % p
        v[:, :, 1, :] = ((x + p - y) % p) * w % p
    return a.astype(np.int32)


# ------------------------------------------------------------------- offset matrix
# (logn, batch, path with every view 16-byte aligned).  Batches are ragged around each kernel's
# grouping: 148 SMs x 8 teams (N = 4096), x 16 warps (N <= 2048), x 4 polynomials (N = 2^13),
# and the persistent N = 2^16 kernel needs >= 888 polynomials.
GS_CASES = [
    (12, 1, FUSED), (12, 7, FUSED), (12, 33, FUSED), (12, 1190, FUSED),
    (6, 33, SMALL), (6, 70, SMALL), (9, 1, GENERIC), (9, 7, SMALL), (9, 33, SMALL),
    (11, 1, SMALL), (11, 33, SMALL), (11, 2373, SMALL),
    (13, 1, "poly_tmem_3round"), (13, 7, "poly_tmem_3round"), (13, 600, "poly_tmem_3round"),
    (14, 33, "poly_tmem_3round"), (15, 3, "poly_tmem_3round"),
    (16, 896, "tilecol_persistent"), (16, 1, "tile_tma + column_passes"),
    (16, 7, "tile_tma + column_passes"), (18, 2, "tile_tma + column_passes"),
]


@pytest.mark.parametrize("logn,batch,fast", GS_CASES)
def test_gs_offset_views(lib, oracle_mod, logn, batch, fast):
    """nttb200_gs_batch on offset input / output views.  Every fast kernel needs 16-byte
    aligned views and declines others to the generic passes -- except the N = 4096 kernel,
    which loads by TMA (16-byte aligned input) but stores words, so an offset output still
    takes it."""
    n, q = 1 << logn, Q29
    rng = np.random.default_rng(40000 + logn * 7 + batch)
    table = rng.integers(0, q, n, dtype=np.int32)
    a = device_rows(batch, n, q, 40000 + logn * 7 + batch)
    rows = sample_rows(batch, n)
    want = oracle_mod.ntt_gs(a.cpu().numpy() if rows is None else a[rows].cpu().numpy(), table, q)
    if logn == 12:
        path = lambda k_in, k_out: FUSED if k_in == 0 else GENERIC
    else:
        path = fast_when_aligned(fast)
    with lib.Plan(logn, q, table) as plan:
        check_layouts(plan, lambda s, d: plan.gs(s, d, batch), a, path, want, rows)


def _flag_path(logn, flags):
    """Kernel path of the flagged golden network for (k_in, k_out) word offsets."""
    core = FUSED if logn == 12 else "poly_tmem_3round"
    in_br, out_br = bool(flags & 8), bool(flags & 16)
    if logn == 12 and (in_br or out_br):
        def path(k_in, k_out):
            # TMA load of d_in; the bit-reversed store writes 16-byte rows of d_out
            if k_in == 0 and (k_out == 0 or not out_br):
                return FUSED_BR
            if in_br:                            # permutation pass d_in -> d_out, core on d_out
                return core if k_out == 0 else GENERIC
            return core if k_in == 0 else GENERIC   # core d_in -> d_out, permutation pass after
        return path
    if in_br or flags & 4:                       # reduction / permutation into d_out first
        return lambda k_in, k_out: core if k_out == 0 else GENERIC
    return fast_when_aligned(core)


@pytest.mark.parametrize("flags", [8, 16, 24, 4])
@pytest.mark.parametrize("logn,batch", [(12, 33), (13, 7)])
def test_gs_flags_offset_views(lib, oracle_mod, logn, batch, flags):
    """INPUT_BITREV / OUTPUT_BITREV / REDUCE_INPUT on offset views: at N = 4096 the adapters
    leave the fused bit-reversing kernel for a permutation pass + the core kernel, or the
    generic passes; the reduction runs into the output first."""
    n, q = 1 << logn, Q29
    rng = np.random.default_rng(41000 + logn + flags)
    table = rng.integers(0, q, n, dtype=np.int32)
    rev = bitrev_index(n)
    if flags & 4:
        src = rng.integers(-(1 << 31), (1 << 31) - 1, (batch, n), dtype=np.int64).astype(np.int32)
        want = oracle_mod.ntt_gs((src.astype(np.int64) % q).astype(np.int32), table, q)
    else:
        a = rng.integers(0, q, (batch, n), dtype=np.int32)
        want = oracle_mod.ntt_gs(a, table, q)
        src = a[:, rev] if flags & 8 else a
        if flags & 16:
            want = want[:, rev]
    with lib.Plan(logn, q, table, flags=flags) as plan:
        check_layouts(plan, lambda s, d: plan.gs(s, d, batch), torch.from_numpy(src).cuda(),
                      _flag_path(logn, flags), want, None)


CT_CASES = [
    (12, 1, "tile_tma_ct"), (12, 7, "tile_tma_ct"), (12, 33, "tile_tma_ct"),
    (12, 1190, "tile_tma_ct"), (9, 7, "fused_ct_small_warp_tma"), (11, 33, "fused_ct_small_warp_tma"),
    (13, 7, "poly_tmem_3round_ct"), (13, 600, "poly_tmem_3round_ct"),
    (16, 896, "tilecol_persistent_ct"),
]


@pytest.mark.parametrize("logn,batch,fast", CT_CASES)
def test_ct_offset_views(lib, oracle_mod, logn, batch, fast):
    """nttb200_ct_batch on offset views; in place through the persistent N = 2^16 kernel
    (which keeps a lazy intermediate and reloads tiles by TMA) included."""
    n, q = 1 << logn, Q29
    rng = np.random.default_rng(42000 + logn * 7 + batch)
    table = rng.integers(0, q, n, dtype=np.int32)
    a = device_rows(batch, n, q, 42000 + logn * 7 + batch)
    rows = sample_rows(batch, n)
    want = oracle_mod.ntt_ct(a.cpu().numpy() if rows is None else a[rows].cpu().numpy(), table, q)
    with lib.Plan(logn, q, table) as plan:
        check_layouts(plan, lambda s, d: plan.ct(s, d, batch), a, fast_when_aligned(fast), want, rows)


@pytest.mark.parametrize("sb,se", [(2, 14), (5, 9), (0, 14), (0, 3)])
def test_stage_range_offset_views(lib, oracle_mod, sb, se):
    """nttb200_gs_stage_range: column passes (stage_begin >= 2) on aligned views, the
    generic passes otherwise."""
    logn, batch, q = 14, 3, Q29
    n = 1 << logn
    rng = np.random.default_rng(43000 + sb * 16 + se)
    table = rng.integers(0, q, n, dtype=np.int32)
    a = rng.integers(0, q, (batch, n), dtype=np.int32)
    want = gs_stage_range_numpy(a, table, q, sb, se)
    if (sb, se) == (0, logn):
        assert np.array_equal(want, oracle_mod.ntt_gs(a, table, q))   # the restatement is the golden
    path = fast_when_aligned("column_passes") if sb >= 2 else (lambda k_in, k_out: GENERIC)
    with lib.Plan(logn, q, table) as plan:
        check_layouts(plan, lambda s, d: plan.gs_stage_range(s, d, batch, sb, se),
                      torch.from_numpy(a).cuda(), path, want, None)


# (logn, batch, path of the aligned product, path of the inverse transform when the product
# falls back to the generic pipeline with an aligned d_c)
POLYMUL_CASES = [
    (12, 7, "polymul4096_one_kernel_tmem", FUSED),
    (12, 1190, "polymul4096_one_kernel_tmem", FUSED),
    (10, 34, "fused_gs_small_warp_tma_dual", SMALL),
    (13, 7, "poly_tmem_3round_dual", "poly_tmem_3round"),
    (16, 896, "tilecol_persistent_dual", "tilecol_persistent"),
]


@pytest.mark.parametrize("logn,batch,fast,inv_fast", POLYMUL_CASES)
def test_polymul_offset_views(lib, oracle_mod, logn, batch, fast, inv_fast):
    """nttb200_polymul_negacyclic with each operand offset on its own and d_c aliasing an
    offset operand.  The fast products need 16-byte aligned views (the N = 4096 one-kernel
    product only a 4-byte aligned d_c); otherwise the generic pipeline CT, CT, pointwise,
    GS, scale runs, its pointwise product and scaling on d_c itself."""
    n, q = 1 << logn, Q29
    rng = np.random.default_rng(44000 + logn)
    fwd = rng.integers(0, q, n, dtype=np.int32)      # the kernels are table-agnostic
    inv = rng.integers(0, q, n, dtype=np.int32)
    a = device_rows(batch, n, q, 44000 + logn)
    b = device_rows(batch, n, q, 44100 + logn)
    rows = sample_rows(batch, n)
    av, bv = (a.cpu().numpy(), b.cpu().numpy()) if rows is None else (a[rows].cpu().numpy(),
                                                                      b[rows].cpu().numpy())
    prod = oracle_mod.pointwise(oracle_mod.ntt_ct(av, fwd, q), oracle_mod.ntt_ct(bv, fwd, q), q)
    want = oracle_mod.scale(oracle_mod.ntt_gs(prod, inv, q), oracle_mod.powmod(n, q - 2, q), q)
    # (layout, k_a, k_b, k_c, expected path); alias layouts reuse the operand's view as d_c
    layouts = [("aligned", 0, 0, 0, fast),
               ("c", 0, 0, 3, fast if logn == 12 else GENERIC),
               ("c=a", 1, 0, None, GENERIC), ("c=b", 0, 2, None, GENERIC)]
    if batch * n <= BIG:
        layouts += [("a", 1, 0, 0, inv_fast), ("b", 0, 2, 0, inv_fast)]
    ref = None
    with lib.Plan(logn, q, fwd) as pf, lib.Plan(logn, q, inv) as pi:
        for name, ka, kb, kc, path in layouts:
            ga, gb = Guarded(a.numel(), ka, a), Guarded(b.numel(), kb, b)
            gc = ga if name == "c=a" else gb if name == "c=b" else Guarded(a.numel(), kc)
            run_checked(lambda: lib.polymul_negacyclic(pf, pi, ga.view, gb.view, gc.view, batch),
                        [gc], [ga, gb])
            assert pi.last_path == path, (name, pi.last_path)
            out = gc.view.view(batch, n)
            check_result(out, want, rows, ref, name)
            if rows is not None and ref is None:
                ref = out.clone()
            del ga, gb, gc


@pytest.mark.parametrize("q", [3329, Q29, 1 << 30, (1 << 31) - 1])
def test_pointwise_scale_offset_views(lib, oracle_mod, q):
    """nttb200_pointwise / nttb200_scale with each of a, b, c offset on its own and in place
    on an offset view: the 128-bit loop needs all pointers 16-byte aligned, any other view
    takes the word loop; ragged counts around the 4-word vector."""
    rng = np.random.default_rng(45000 + q % 1000)
    with lib.Plan(4, q, np.zeros(16, np.int32)) as plan:
        for count in (1, 3, 4, 5, 4099):
            a = rng.integers(0, q, count, dtype=np.int64).astype(np.int32)
            b = rng.integers(0, q, count, dtype=np.int64).astype(np.int32)
            a[0] = b[0] = q - 1
            s = int(rng.integers(0, q))
            want_pw, want_sc = oracle_mod.pointwise(a, b, q), oracle_mod.scale(a, s, q)
            for ka, kb, kc in ((0, 0, 0), (1, 0, 0), (0, 2, 0), (0, 0, 3), (1, 1, None)):
                ga, gb = Guarded(count, ka, a), Guarded(count, kb, b)
                gc = ga if kc is None else Guarded(count, kc)
                run_checked(lambda: plan.pointwise(ga.view, gb.view, gc.view, count), [gc], [ga, gb])
                assert np.array_equal(gc.view.cpu().numpy(), want_pw), (count, ka, kb, kc)
                if kc is None or kb == 0:      # scale reads a, writes c
                    ga = Guarded(count, ka, a)
                    gc = ga if kc is None else Guarded(count, kc)
                    run_checked(lambda: plan.scale(ga.view, gc.view, count, s), [gc], [ga])
                    assert np.array_equal(gc.view.cpu().numpy(), want_sc), (count, ka, kc, "scale")


def test_adapters_offset_views(lib):
    """nttb200_bitrev_permute (in place too) and nttb200_transpose (out of place only) on
    offset views: word kernels, no alignment requirement."""
    logn, batch = 11, 5
    n = 1 << logn
    rng = np.random.default_rng(46000)
    a = rng.integers(0, Q29, (batch, n), dtype=np.int32)
    want = a[:, bitrev_index(n)]
    with lib.Plan(logn, Q29, np.zeros(n, np.int32)) as plan:
        for name, k_in, k_out in LAYOUTS:
            src = Guarded(a.size, k_in, a)
            dst = src if name == "inplace" else Guarded(a.size, k_out)
            run_checked(lambda: plan.bitrev_permute(src.view, dst.view, batch), [dst], [src])
            assert np.array_equal(dst.view.cpu().numpy().reshape(batch, n), want), name
        for name, k_in, k_out in LAYOUTS[:4]:
            src = Guarded(a.size, k_in, a)
            dst = Guarded(a.size, k_out)
            run_checked(lambda: plan.transpose(src.view, dst.view, batch, True), [dst], [src])
            assert np.array_equal(dst.view.cpu().numpy().reshape(n, batch), a.T), name
            back = Guarded(a.size, k_in)
            run_checked(lambda: plan.transpose(dst.view, back.view, batch, False), [back], [dst])
            assert np.array_equal(back.view.cpu().numpy().reshape(batch, n), a), name


def _host_view(words, k):
    """numpy int32 view of `words` starting 4k bytes past a 16-byte boundary, inside an
    array whose other words hold the sentinel: (whole array, view)."""
    whole = np.full(words + 2 * GUARD, SENTINEL, dtype=np.int32)
    start = GUARD - (whole.ctypes.data // 4) % 4 + k
    view = whole[start:start + words]
    assert view.ctypes.data % 16 == 4 * k
    return whole, view


def test_gs_host_offset_views_aie_order_two_chunks(lib, oracle_mod):
    """nttb200_gs_host with ORDER_AIE_DEVICE on host views at word offsets (and in place),
    over more than one 32 MiB staging chunk (2048 polynomials of N = 4096): unreduced
    inputs, every row against the permuted golden, nothing written around the output."""
    logn, q, batch = 12, Q29, 2048 + 3
    n = 1 << logn
    rng = np.random.default_rng(47000)
    table = rng.integers(0, q, n, dtype=np.int32)
    a = rng.integers(0, (1 << 31) - 1, (batch, n), dtype=np.int32)
    want = oracle_mod.ans_order_permute(oracle_mod.ntt_gs(a % q, table, q))
    with lib.Plan(logn, q, table, flags=lib.ORDER_AIE_DEVICE) as plan:
        for name, k_in, k_out in (("aligned", 0, 0), ("both", 1, 3), ("inplace", 2, 2)):
            win, vin = _host_view(a.size, k_in)
            vin[:] = a.reshape(-1)
            if name == "inplace":
                wout, vout = win, vin
            else:
                wout, vout = _host_view(a.size, k_out)
            plan.gs_host(vin, vout, batch)
            assert plan.last_path == FUSED, plan.last_path
            assert np.array_equal(vout.reshape(batch, n), want), name
            lo = vout.ctypes.data // 4 - wout.ctypes.data // 4
            assert (wout[:lo] == SENTINEL).all() and (wout[lo + a.size:] == SENTINEL).all(), name
            if name != "inplace":
                assert np.array_equal(vin.reshape(batch, n), a), name


# ------------------------------------------------------------------- RNS and scatter
def _rns_setup(rng, batch):
    qs = [Q29, Q30]
    n = 4096
    fwd = [rng.integers(0, q, n, dtype=np.int32) for q in qs]
    inv = [rng.integers(0, q, n, dtype=np.int32) for q in qs]
    a = np.stack([rng.integers(0, q, (batch, n), dtype=np.int32) for q in qs], axis=1)
    b = np.stack([rng.integers(0, q, (batch, n), dtype=np.int32) for q in qs], axis=1)
    return qs, fwd, inv, a, b


def _expect_status(lib, status, call):
    with pytest.raises(lib.NttError) as err:
        call()
    assert err.value.status == status, str(err.value)


def test_rns_offset_views(lib, oracle_mod):
    """The RNS entry points need 16-byte aligned buffers: an offset input / operand / output
    returns NTTB200_ERR_UNSUPPORTED with the output and the guards untouched, and the next
    aligned call on the same plans is correct (no sticky error).  An offset d_c alone still
    computes the product (the strided one-kernel product stores words)."""
    rng = np.random.default_rng(48000)
    batch = 3
    qs, fwd_t, inv_t, a, b = _rns_setup(rng, batch)
    n = 4096
    want_gs = np.stack([oracle_mod.ntt_gs(a[:, l], inv_t[l], q) for l, q in enumerate(qs)], axis=1)
    want_ct = np.stack([oracle_mod.ntt_ct(a[:, l], fwd_t[l], q) for l, q in enumerate(qs)], axis=1)
    want_mul = np.stack([
        oracle_mod.scale(oracle_mod.ntt_gs(oracle_mod.pointwise(oracle_mod.ntt_ct(a[:, l], fwd_t[l], q),
                                                                oracle_mod.ntt_ct(b[:, l], fwd_t[l], q), q),
                                           inv_t[l], q), oracle_mod.powmod(n, q - 2, q), q)
        for l, q in enumerate(qs)], axis=1)
    UNSUPPORTED = 7
    with lib.RnsPlan(qs, fwd_t) as pf, lib.RnsPlan(qs, inv_t) as pi:
        for k_in, k_out in ((1, 0), (0, 3)):
            for plan, fn, want in ((pi, pi.gs, want_gs), (pf, pf.ct, want_ct)):
                src, dst = Guarded(a.size, k_in, a), Guarded(a.size, k_out)
                run_checked(lambda: _expect_status(lib, UNSUPPORTED, lambda: fn(src.view, dst.view, batch)),
                            [dst], [src])
                assert dst.untouched()
                src, dst = Guarded(a.size, 0, a), Guarded(a.size, 0)
                run_checked(lambda: fn(src.view, dst.view, batch), [dst], [src])
                assert np.array_equal(dst.view.cpu().numpy().reshape(a.shape), want), (k_in, k_out)
        for ka, kb, kc in ((1, 0, 0), (0, 2, 0), (0, 0, 3)):
            ga, gb, gc = Guarded(a.size, ka, a), Guarded(b.size, kb, b), Guarded(a.size, kc)
            call = lambda: lib.rns_polymul_negacyclic(pf, pi, ga.view, gb.view, gc.view, batch)
            if kc:
                run_checked(call, [gc], [ga, gb])
                assert np.array_equal(gc.view.cpu().numpy().reshape(a.shape), want_mul), "offset d_c"
                continue
            run_checked(lambda: _expect_status(lib, UNSUPPORTED, call), [gc], [ga, gb])
            assert gc.untouched(), (ka, kb)
            ga, gb, gc = Guarded(a.size, 0, a), Guarded(b.size, 0, b), Guarded(a.size, 0)
            run_checked(lambda: lib.rns_polymul_negacyclic(pf, pi, ga.view, gb.view, gc.view, batch),
                        [gc], [ga, gb])
            assert np.array_equal(gc.view.cpu().numpy().reshape(a.shape), want_mul), (ka, kb)


def test_scatter_offset_views(lib, oracle_mod):
    """nttb200_gs_stage_range_scatter: an offset d_buf returns NTTB200_ERR_UNSUPPORTED, an
    offset peer buffer NTTB200_ERR_INVALID_ARG, both before anything is written; the aligned
    call that follows stores exactly this rank's slice of every peer and nothing else."""
    logn, world, q = 13, 2, Q29
    n, c = 1 << logn, (1 << logn) // 2
    rng = np.random.default_rng(49000)
    table = rng.integers(0, q, n, dtype=np.int32)
    x = rng.integers(0, q, n, dtype=np.int32)
    y = oracle_mod.ntt_gs(x, table, q)
    with lib.Plan(logn, q, table) as plan:
        for rank in range(world):
            for k_buf, k_peer, status in ((1, 0, 7), (0, 2, 1)):
                buf = Guarded(n, k_buf, x)
                peers = [Guarded(n, k_peer) for _ in range(world)]
                run_checked(lambda: _expect_status(
                    lib, status, lambda: plan.gs_stage_range_scatter(
                        buf.view, 0, logn, [p.view.data_ptr() for p in peers], rank)), peers, [buf])
                assert all(p.untouched() for p in peers)
            buf = Guarded(n, 0, x)
            peers = [Guarded(n, 0) for _ in range(world)]
            plan.gs_stage_range_scatter(buf.view, 0, logn, [p.view.data_ptr() for p in peers], rank)
            torch.cuda.synchronize()
            assert plan.last_path == "passes + peer scatter", plan.last_path
            assert buf.guards_intact()
            for k, p in enumerate(peers):
                got = p.view.cpu().numpy()
                assert np.array_equal(got[rank * c:(rank + 1) * c], y[k * c:(k + 1) * c]), (rank, k)
                rest = np.delete(got, np.s_[rank * c:(rank + 1) * c])
                assert (rest == SENTINEL).all() and p.guards_intact(), (rank, k)


# ------------------------------------------------------------------- AIE device order
@pytest.mark.parametrize("q", [3329, Q29, (1 << 29) - 3, 1 << 30])
def test_aie_order_n4096_fused(lib, oracle_mod, q):
    """ORDER_AIE_DEVICE through the device-order variant of the N = 4096 kernel (classic
    butterflies where the default takes the 4q-lazy ones): batches 1, 3 and one beyond
    148 SMs x 8 teams (every team loops), out of place, on an offset output and in place,
    tables and one row pinned at q - 1; the generic passes (flags 3) agree."""
    n = 4096
    rng = np.random.default_rng(50000 + q % 1000)
    table = rng.integers(0, q, n, dtype=np.int32)
    table[1::2] = q - 1
    a = rng.integers(0, q, (1190, n), dtype=np.int32)
    a[0] = q - 1
    want = oracle_mod.ans_order_permute(oracle_mod.ntt_gs(a, table, q))
    layouts = (("aligned", 0, 0), ("out", 0, 1), ("inplace", 0, 0))
    for flags, path in ((1, FUSED), (3, GENERIC)):
        with lib.Plan(12, q, table, flags=flags) as plan:
            for batch in (1, 3, 1190):
                check_layouts(plan, lambda s, d: plan.gs(s, d, batch), torch.from_numpy(a[:batch]).cuda(),
                              lambda k_in, k_out: path, want[:batch], None, layouts)


@pytest.mark.parametrize("logn,batch,path", [
    (4, 5, GENERIC), (5, 5, GENERIC), (9, 5, GENERIC), (11, 33, SMALL), (13, 3, GENERIC),
    (15, 3, GENERIC), (16, 3, GENERIC), (18, 2, GENERIC)])
def test_aie_order_all_paths(lib, oracle_mod, logn, batch, path):
    """ORDER_AIE_DEVICE at the other sizes, batch > 1, in place and out of place, q <= 2^30:
    the N = 2048 warp kernel's permuted store, and the generic passes whose last pass is
    widened to the four stages the permuted store needs (at logn = 13 it runs one stage and
    borrows three)."""
    n = 1 << logn
    rng = np.random.default_rng(51000 + logn)
    for q in (Q29, 1 << 30):
        table = rng.integers(0, q, n, dtype=np.int32)
        a = rng.integers(0, q, (batch, n), dtype=np.int32)
        a[0] = q - 1
        want = oracle_mod.ans_order_permute(oracle_mod.ntt_gs(a, table, q))
        with lib.Plan(logn, q, table, flags=lib.ORDER_AIE_DEVICE) as plan:
            check_layouts(plan, lambda s, d: plan.gs(s, d, batch), torch.from_numpy(a).cuda(),
                          lambda k_in, k_out: path, want, None,
                          (("aligned", 0, 0), ("inplace", 0, 0)))


def test_aie_order_with_reduce_input(lib, oracle_mod):
    """ORDER_AIE_DEVICE | REDUCE_INPUT on the reference harness's unreduced a[i] = i at
    N = 4096 (fused kernel) and 8192 (generic passes), in place and out of place."""
    g = load_golden("unreduced_inputs.npz")
    for n, path in ((4096, FUSED), (8192, GENERIC)):
        a = np.arange(n, dtype=np.int32)[None, :]
        want = oracle_mod.ans_order_permute(g[f"out_{n}"])[None, :]
        with lib.Plan(n.bit_length() - 1, 3329, g[f"roots_{n}"],
                      flags=lib.ORDER_AIE_DEVICE | lib.REDUCE_INPUT) as plan:
            check_layouts(plan, lambda s, d: plan.gs(s, d, 1), torch.from_numpy(a).cuda(),
                          lambda k_in, k_out: path, want, None,
                          (("aligned", 0, 0), ("inplace", 0, 0)))


@pytest.mark.parametrize("logn", [12, 13])
def test_aie_order_applies_to_full_depth_gs_only(lib, oracle_mod, logn):
    """On an ORDER_AIE_DEVICE plan a partial depth, nttb200_ct_batch and
    nttb200_gs_stage_range return the golden (unpermuted) order."""
    n, q, batch = 1 << logn, Q29, 3
    rng = np.random.default_rng(52000 + logn)
    table = rng.integers(0, q, n, dtype=np.int32)
    a = rng.integers(0, q, (batch, n), dtype=np.int32)
    d_a = torch.from_numpy(a).cuda()
    with lib.Plan(logn, q, table, flags=lib.ORDER_AIE_DEVICE) as plan:
        for stage in (0, logn // 2, logn - 2):
            out = torch.empty_like(d_a)
            plan.gs(d_a, out, batch, stage)
            assert np.array_equal(out.cpu().numpy(), oracle_mod.ntt_gs(a, table, q, stage)), stage
        out = torch.empty_like(d_a)
        plan.ct(d_a, out, batch)
        assert np.array_equal(out.cpu().numpy(), oracle_mod.ntt_ct(a, table, q))
        plan.gs_stage_range(d_a, out, batch, 0, logn)
        assert np.array_equal(out.cpu().numpy(), oracle_mod.ntt_gs(a, table, q))
        plan.gs_stage_range(d_a, out, batch, 2, logn)
        assert np.array_equal(out.cpu().numpy(), gs_stage_range_numpy(a, table, q, 2, logn))
        plan.gs(d_a, out, batch)                  # while full depth is permuted
        assert np.array_equal(out.cpu().numpy(), oracle_mod.ans_order_permute(oracle_mod.ntt_gs(a, table, q)))
