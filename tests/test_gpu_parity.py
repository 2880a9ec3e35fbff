"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the
committed golden fixtures.  Bit-exact: every comparison is integer equality."""
import os
import numpy as np
import pytest
import torch

from conftest import Q29, Q30, load_golden

pytestmark = pytest.mark.gpu


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).cuda()


def run_gs(lib, a, roots, p, stage=-1, flags=0, inplace=False):
    a = np.ascontiguousarray(a, dtype=np.int32)
    n = a.shape[-1]
    batch = a.size // n
    d_in = dev(a)
    d_out = d_in if inplace else torch.empty_like(d_in)
    with lib.Plan(n.bit_length() - 1, p, roots, flags=flags) as plan:
        plan.gs(d_in, d_out, batch, stage)
        torch.cuda.synchronize()
        path = plan.last_path
    return d_out.cpu().numpy(), path


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    assert torch.cuda.is_available(), "gpu-marked tests need a CUDA device"


def test_library_is_loaded_and_counts_launches(lib):
    before = lib.kernel_launches()
    g = load_golden("default_n2048_p3329.npz")
    out, _ = run_gs(lib, g["a"], g["roots"], int(g["p"]), 10)
    assert np.array_equal(out, g["out"])
    assert lib.kernel_launches() > before


@pytest.mark.parametrize("flags", [0, 2])
def test_reference_default_config(lib, flags):
    """N=2048, p=3329, g=3, a[i]=i, full depth == golden (src/test.cpp:203-235)."""
    g = load_golden("default_n2048_p3329.npz")
    roots = lib.make_roots(2048, 3329, 3)
    assert np.array_equal(roots, g["roots"])
    out, _ = run_gs(lib, g["a"], roots, 3329, 10, flags=flags)
    assert np.array_equal(out, g["out"])


def test_reference_default_config_device_order(lib, oracle_mod):
    """ORDER_AIE_DEVICE reproduces what the AIE leaves in bo_outC: the golden permuted
    by ans_order (src/test.cpp:69-71,212-219)."""
    g = load_golden("default_n2048_p3329.npz")
    for flags in (1, 3):
        out, _ = run_gs(lib, g["a"], g["roots"], 3329, 10, flags=flags)
        assert np.array_equal(out, oracle_mod.ans_order_permute(g["out"]))
        out, _ = run_gs(lib, g["a"], g["roots"], 3329, 10, flags=flags, inplace=True)
        assert np.array_equal(out, oracle_mod.ans_order_permute(g["out"]))


def test_stage_early_exit(lib, oracle_mod):
    """Every partial depth of the default config (src/test.cpp:55-58)."""
    g = load_golden("default_n2048_p3329.npz")
    for s in range(11):
        out, _ = run_gs(lib, g["a"], g["roots"], 3329, s)
        assert np.uint64(oracle_mod.fnv1a64_words(out)) == g["stage_digest"][s], f"stage {s}"


@pytest.mark.parametrize("name", ["n4096_q29.npz", "n4096_p3329.npz"])
@pytest.mark.parametrize("flags", [0, 1, 2, 3])
def test_n4096_fixtures(lib, oracle_mod, name, flags):
    """flags 1: the device-order variant of the fused kernel, 3: the generic passes' permuted
    store."""
    g = load_golden(name)
    out, path = run_gs(lib, g["a"], g["roots"], int(g["p"]), flags=flags)
    want = oracle_mod.ans_order_permute(g["out"]) if flags & 1 else g["out"]
    assert np.array_equal(out, want)
    assert path == ("generic_stage_pass" if flags & 2 else "fused_gs4096_tma"), path


def test_small_fixtures(lib):
    g = load_golden("small.npz")
    for logn in range(1, 7):
        for p, tag in ((Q29, "q29"), (3329, "p3329")):
            out, _ = run_gs(lib, g[f"a_{tag}_{logn}"], g[f"roots_{tag}_{logn}"], p)
            assert np.array_equal(out, g[f"out_{tag}_{logn}"]), (logn, tag)


def test_n65536_digest(lib, oracle_mod):
    g = load_golden("n65536_q29_digest.npz")
    n, p = int(g["n"]), int(g["p"])
    a = np.random.default_rng(int(g["seed"])).integers(0, p, n, dtype=np.int32)
    out, _ = run_gs(lib, a, lib.make_roots(n, p, 3), p)
    assert np.uint64(oracle_mod.fnv1a64_words(out)) == g["digest"]
    assert np.array_equal(out[:16], g["head"]) and np.array_equal(out[-16:], g["tail"])


@pytest.mark.parametrize("logn", list(range(1, 17)))
@pytest.mark.parametrize("flags", [0, 2])
def test_gs_vs_oracle_all_sizes(lib, oracle_mod, logn, flags):
    """N = 2..65536 x {reference w^i table, psi^-bitrev table, arbitrary table} x
    {random, a[i]=i, all q-1, zeros}, ragged batch sizes."""
    n = 1 << logn
    rng = np.random.default_rng(1000 + logn)
    for p in (Q29, 3329, Q30):
        tables = [lib.make_roots(n, p, 3), rng.integers(0, p, n, dtype=np.int32)]
        if p == Q29:
            tables.append(lib.negacyclic_tables(n, p, 3)[1])
        batch = 3 if logn > 12 else 5
        a = rng.integers(0, p, (batch, n), dtype=np.int32)
        a[0] = np.arange(n) % p
        a[1] = p - 1
        a[2] = 0
        for table in tables:
            out, _ = run_gs(lib, a, table, p, flags=flags)
            assert np.array_equal(out, oracle_mod.ntt_gs(a, table, p)), (logn, p)


@pytest.mark.parametrize("logn", [3, 7, 12, 14])
def test_gs_partial_depth_and_inplace(lib, oracle_mod, logn):
    n = 1 << logn
    rng = np.random.default_rng(2000 + logn)
    table = rng.integers(0, Q29, n, dtype=np.int32)
    a = rng.integers(0, Q29, (4, n), dtype=np.int32)
    for stage in (0, 1, logn // 2, logn - 2, logn - 1, logn + 5, -1):
        out, _ = run_gs(lib, a, table, Q29, stage, inplace=(stage % 2 == 0))
        assert np.array_equal(out, oracle_mod.ntt_gs(a, table, Q29, stage)), (logn, stage)


@pytest.mark.parametrize("logn", [1, 4, 9, 12, 13, 16, 18, 19])
def test_ct_vs_oracle(lib, oracle_mod, logn):
    n = 1 << logn
    rng = np.random.default_rng(3000 + logn)
    fwd, inv = lib.negacyclic_tables(n, Q29, 3)
    a = rng.integers(0, Q29, (3, n), dtype=np.int32)
    d_in = dev(a)
    d_out = torch.empty_like(d_in)
    with lib.Plan(logn, Q29, fwd) as pf, lib.Plan(logn, Q29, inv) as pi:
        for stage in (-1, 0, logn // 2):
            pf.ct(d_in, d_out, 3, stage)
            assert np.array_equal(d_out.cpu().numpy(), oracle_mod.ntt_ct(a, fwd, Q29, stage))
        # round trip: GS(inv) o CT(fwd) = n * identity
        pf.ct(d_in, d_out, 3)
        pi.gs(d_out, d_out, 3)
        assert np.array_equal(d_out.cpu().numpy(), oracle_mod.scale(a, n % Q29, Q29))


def test_pointwise_and_scale(lib, oracle_mod):
    rng = np.random.default_rng(5)
    for p in (3329, Q29, Q30, 1 << 30, 2):
        for count in (1, 3, 4, 1023, 4096 * 3 + 1):
            a = rng.integers(0, p, count, dtype=np.int32)
            b = rng.integers(0, p, count, dtype=np.int32)
            a[0] = p - 1
            b[0] = p - 1
            with lib.Plan(4, p, np.zeros(16, np.int32)) as plan:
                d_c = torch.empty(count, dtype=torch.int32, device="cuda")
                plan.pointwise(dev(a), dev(b), d_c, count)
                assert np.array_equal(d_c.cpu().numpy(), oracle_mod.pointwise(a, b, p))
                s = int(rng.integers(0, p))
                plan.scale(dev(a), d_c, count, s)
                assert np.array_equal(d_c.cpu().numpy(), oracle_mod.scale(a, s, p))


@pytest.mark.parametrize("logn", [1, 5, 8, 10])
def test_polymul_vs_schoolbook(lib, oracle_mod, logn):
    n = 1 << logn
    rng = np.random.default_rng(6000 + logn)
    fwd, inv = lib.negacyclic_tables(n, Q29, 3)
    a = rng.integers(0, Q29, (3, n), dtype=np.int32)
    b = rng.integers(0, Q29, (3, n), dtype=np.int32)
    want = np.stack([oracle_mod.negacyclic_schoolbook(x, y, Q29) for x, y in zip(a, b)])
    with lib.Plan(logn, Q29, fwd) as pf, lib.Plan(logn, Q29, inv) as pi:
        d_a, d_b = dev(a), dev(b)
        d_c = torch.empty_like(d_a)
        lib.polymul_negacyclic(pf, pi, d_a, d_b, d_c, 3)
        assert np.array_equal(d_c.cpu().numpy(), want)
        assert np.array_equal(d_a.cpu().numpy(), a) and np.array_equal(d_b.cpu().numpy(), b)
        lib.polymul_negacyclic(pf, pi, d_a, d_b, d_b, 3)    # output aliases b
        assert np.array_equal(d_b.cpu().numpy(), want)


@pytest.mark.parametrize("logn", [12, 13, 14, 16, 19])
def test_polymul_vs_oracle_pipeline(lib, oracle_mod, logn):
    n = 1 << logn
    rng = np.random.default_rng(7000 + logn)
    fwd, inv = lib.negacyclic_tables(n, Q29, 3)
    a = rng.integers(0, Q29, (2, n), dtype=np.int32)
    b = rng.integers(0, Q29, (2, n), dtype=np.int32)
    prod = oracle_mod.pointwise(oracle_mod.ntt_ct(a, fwd, Q29), oracle_mod.ntt_ct(b, fwd, Q29), Q29)
    want = oracle_mod.scale(oracle_mod.ntt_gs(prod, inv, Q29), oracle_mod.powmod(n, Q29 - 2, Q29), Q29)
    with lib.Plan(logn, Q29, fwd) as pf, lib.Plan(logn, Q29, inv) as pi:
        d_c = torch.empty(2, n, dtype=torch.int32, device="cuda")
        lib.polymul_negacyclic(pf, pi, dev(a), dev(b), d_c, 2)
        assert np.array_equal(d_c.cpu().numpy(), want)


def test_batch_independence(lib, oracle_mod):
    """Polynomial k is unaffected by its neighbours; ragged batch sizes around the
    kernel's grouping factors."""
    n, p = 4096, Q29
    rng = np.random.default_rng(8)
    roots = lib.make_roots(n, p, 3)
    a = rng.integers(0, p, (67, n), dtype=np.int32)
    want = oracle_mod.ntt_gs(a, roots, p)
    for batch in (1, 2, 7, 8, 9, 63, 67):
        out, _ = run_gs(lib, a[:batch], roots, p)
        assert np.array_equal(out, want[:batch]), batch
    out, _ = run_gs(lib, a[:0].reshape(0, n), roots, p)   # empty batch
    assert out.size == 0


def test_host_buffer_entry_point(lib, oracle_mod):
    """nttb200_gs_host: host in, host out (the reference's sync + launch + sync)."""
    n, p = 4096, Q29
    rng = np.random.default_rng(9)
    roots = lib.make_roots(n, p, 3)
    batch = 2100      # > one 32 MiB staging chunk (2048 polys), not a multiple
    a = rng.integers(0, p, (batch, n), dtype=np.int32)
    out = np.empty_like(a)
    with lib.Plan(12, p, roots) as plan:
        plan.gs_host(a, out, batch)
    idx = [0, 1, 2047, 2048, 2049, batch - 1] + rng.integers(0, batch, 26).tolist()
    assert np.array_equal(out[idx], oracle_mod.ntt_gs(a[idx], roots, p))
    # the golden-signature wrapper
    g = load_golden("default_n2048_p3329.npz")
    assert np.array_equal(lib.ntt(g["a"], 2048, g["roots"], 3329, 10), g["out"])


def test_full_size_properties(lib, oracle_mod):
    """BASELINE config 2 shape (65,536 x N=4096): sampled rows against the oracle,
    plus size-independent properties over the whole batch: linearity of the network
    (NTT(a+b) = NTT(a)+NTT(b) mod q) and the CT o GS round trip = n * x."""
    n, p, batch = 4096, Q29, 65536
    roots = lib.make_roots(n, p, 3)
    gen = torch.Generator(device="cuda").manual_seed(0x5EED0001)
    a = torch.randint(0, p, (batch, n), dtype=torch.int32, device="cuda", generator=gen)
    b = torch.randint(0, p, (batch, n), dtype=torch.int32, device="cuda", generator=gen)
    fa, fb, fs = torch.empty_like(a), torch.empty_like(a), torch.empty_like(a)
    with lib.Plan(12, p, roots) as plan:
        plan.gs(a, fa, batch)
        plan.gs(b, fb, batch)
        s = (a + b) % p
        plan.gs(s, fs, batch)
        torch.cuda.synchronize()
        assert plan.last_path != "none"
    assert torch.equal(fs, (fa + fb) % p)
    rng = np.random.default_rng(10)
    idx = [0, 1, batch - 1] + rng.integers(0, batch, 253).tolist()
    assert np.array_equal(fa[idx].cpu().numpy(), oracle_mod.ntt_gs(a[idx].cpu().numpy(), roots, p))
    del fb, fs, s, b
    fwd, inv = lib.negacyclic_tables(n, p, 3)
    with lib.Plan(12, p, fwd) as pf, lib.Plan(12, p, inv) as pi:
        pf.ct(a, fa, batch)
        pi.gs(fa, fa, batch)
        torch.cuda.synchronize()
    assert torch.equal(fa, ((a.to(torch.int64) * n) % p).to(torch.int32))


def test_cpp_host_harness(lib):
    """tests/host/ntt_test: the C++ successor of the reference's src/test.cpp main() --
    default config, AIE device order, and a 29-bit batch -- prints PASS! and exits 0."""
    import os
    import subprocess
    import sys
    sys.path.insert(0, os.path.dirname(lib.lib_path()))
    root = os.path.dirname(os.path.dirname(os.path.dirname(lib.lib_path())))
    exe = os.path.join(root, "tests", "host", "ntt_test")
    if not os.path.exists(exe):
        import importlib.util
        spec = importlib.util.spec_from_file_location(
            "nttb200_build", os.path.join(root, "ntt-aie_b200", "build.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.build_host_harness()
    for extra in ([], ["--aie-order"], ["--logn", "12", "--p", "469762049", "--batch", "33",
                                        "--random", "--iters", "2"],
                  ["--stage", "4"], ["--logn", "12"], ["--logn", "13"]):   # a[i] = i >= p there
        res = subprocess.run([exe] + extra, capture_output=True, text=True, timeout=120)
        assert res.returncode == 0 and "PASS!" in res.stdout, res.stdout + res.stderr


def _free_port():
    import socket
    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        return sock.getsockname()[1]


def test_fourstep_on_available_gpus(lib):
    """tools/fourstep_run.py under torchrun on min(2, #GPUs) ranks: the whole N=2^18
    vector bit-exact against the golden, for the reference table and an arbitrary one."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.dirname(lib.lib_path())))
    world = min(2, torch.cuda.device_count())
    variants = [[], ["--arbitrary-table"], ["--generated"]]
    if world > 1:
        variants.append(["--fused", "--arbitrary-table"])   # transposes fused into peer stores
        variants.append(["--fused", "--generated"])
    for extra in variants:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
               f"--nproc-per-node={world}", "--master-addr", "127.0.0.1", "--master-port",
               str(_free_port()),
               os.path.join(root, "tools", "fourstep_run.py"), "--logn", "18", "--verify",
               "--steps", "1", "--warmup", "1"] + extra
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stdout + res.stderr
        line = json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][-1])
        assert line["bit_exact_vs_golden"] is True and line["n_gpus"] == world
        assert line["bit_exact_transposed_order"] is True


@pytest.mark.parametrize("logn", [6, 13, 17, 20])
def test_stage_range_vs_restatement(lib, oracle_mod, logn):
    """nttb200_gs_stage_range against the vectorised restatement of src/test.cpp:36-59
    (itself pinned to the oracle in tests/test_multigpu_cpu.py), incl. in place and the
    column-pass path (stage_begin >= 2)."""
    from test_multigpu_cpu import gs_stage_range_numpy
    n = 1 << logn
    rng = np.random.default_rng(9000 + logn)
    table = rng.integers(0, Q29, n, dtype=np.int32)
    a = rng.integers(0, Q29, (2, n), dtype=np.int32)
    ranges = [(0, logn), (0, 1), (2, logn), (logn - 3, logn), (3, 3), (logn // 2, logn // 2 + 1),
              (1, logn - 1), (logn - 1, logn)]
    with lib.Plan(logn, Q29, table) as plan:
        for sb, se in ranges:
            d = dev(a)
            out = torch.empty_like(d)
            plan.gs_stage_range(d, out, 2, sb, se)
            want = np.stack([gs_stage_range_numpy(x, table, Q29, sb, se) for x in a])
            assert np.array_equal(out.cpu().numpy(), want), (logn, sb, se, plan.last_path)
            plan.gs_stage_range(d, d, 2, sb, se)
            assert np.array_equal(d.cpu().numpy(), want), (logn, sb, se, "in place")


@pytest.mark.parametrize("logn", [13, 15, 16, 18, 21])
def test_large_n_multi_pass_path(lib, oracle_mod, logn):
    """logn >= 13 takes the tile pass + column passes; batch sizes around the CTA
    range partition, arbitrary tables."""
    n = 1 << logn
    rng = np.random.default_rng(9500 + logn)
    table = rng.integers(0, Q29, n, dtype=np.int32)
    for batch in ((1, 3, 40) if logn <= 16 else (1, 2)):
        a = rng.integers(0, Q29, (batch, n), dtype=np.int32)
        out, path = run_gs(lib, a, table, Q29)
        assert "tile" in path or "poly" in path, path
        assert np.array_equal(out, oracle_mod.ntt_gs(a, table, Q29)), (logn, batch)
        out, _ = run_gs(lib, a, table, Q29, inplace=True)
        assert np.array_equal(out, oracle_mod.ntt_gs(a, table, Q29)), (logn, batch, "in place")


@pytest.mark.parametrize("logn", [6, 7, 8, 9, 10, 11])
def test_small_n_warp_kernel_ragged_batches(lib, oracle_mod, logn):
    """N = 512..2048 run one warp per 2048-coefficient block; batches that are not a
    multiple of the block (tail through the generic pass), in place, 12-bit and
    30-bit moduli, AIE device order at N=2048 with a batch."""
    n = 1 << logn
    rng = np.random.default_rng(11000 + logn)
    for p in (3329, Q30):
        table = rng.integers(0, p, n, dtype=np.int32)
        a = rng.integers(0, p, (70, n), dtype=np.int32)
        want = oracle_mod.ntt_gs(a, table, p)
        for batch in (1, 2, 3, 4, 5, 31, 32, 33, 70):
            out, path = run_gs(lib, a[:batch], table, p, inplace=(batch % 2 == 0))
            assert np.array_equal(out, want[:batch]), (logn, p, batch, path)
    if logn == 11:
        g = load_golden("default_n2048_p3329.npz")
        a = np.stack([g["a"], (g["a"] * 7) % 3329, np.zeros(2048, np.int32)]).astype(np.int32)
        out, path = run_gs(lib, a, g["roots"], 3329, flags=1)
        assert "small" in path
        assert np.array_equal(out, oracle_mod.ans_order_permute(oracle_mod.ntt_gs(a, g["roots"], 3329)))


@pytest.mark.parametrize("logn", [10, 12, 14])
def test_extreme_moduli_on_fast_paths(lib, oracle_mod, logn):
    """q = 2^30 (the largest modulus of the golden's domain, where the lazy ranges
    [0,2q) / [0,4q) touch 2^32), q = 2^29 - 1 and 2^29 - 3 (the largest moduli of the 4q-lazy
    kernels, whose ranges [0,4q) / [0,8q) touch 2^32 there), q = 2^29 (the first modulus back
    on the classic kernels), q = 2 and q = 3 through the register-radix kernels, GS and CT,
    inputs pinned at q-1."""
    n = 1 << logn
    rng = np.random.default_rng(12000 + logn)
    for q in (1 << 30, (1 << 30) - 35, (1 << 29) - 1, (1 << 29) - 3, 1 << 29, 2, 3):
        table = rng.integers(0, q, n, dtype=np.int32)
        a = rng.integers(0, q, (4, n), dtype=np.int32)
        a[0] = q - 1
        table[1::2] = q - 1
        out, path = run_gs(lib, a, table, q)
        assert path != "generic_stage_pass" or logn < 9
        assert np.array_equal(out, oracle_mod.ntt_gs(a, table, q)), (logn, q, path)
        if logn >= 12:
            d_in = dev(a)
            d_out = torch.empty_like(d_in)
            with lib.Plan(logn, q, table) as plan:
                plan.ct(d_in, d_out, 4)
                assert "ct" in plan.last_path
            assert np.array_equal(d_out.cpu().numpy(), oracle_mod.ntt_ct(a, table, q)), (logn, q)


def _ntt_primes(count, two_n=8192, below=1 << 30):
    """Primes q < 2^30 with 2N | q-1, largest first (deterministic trial division)."""
    out, k = [], (below - 1) // two_n
    while len(out) < count and k > 0:
        q = k * two_n + 1
        if q < below and all(q % d for d in range(3, int(q ** 0.5) + 1, 2)) and q % 2:
            out.append(q)
        k -= 1
    return out


def _psi(n, q):
    """An element of order 2n modulo the prime q."""
    for x in range(2, 1000):
        psi = pow(x, (q - 1) // (2 * n), q)
        if pow(psi, n, q) == q - 1:
            return psi
    raise AssertionError("no 2n-th root found")


def test_rns_large_batch(lib, oracle_mod):
    """A large RNS batch: the transform through the all-channel tile kernel with per-segment
    tables, the product through one strided launch of the one-kernel product per channel
    (tile = poly * L + channel): sampled rows against the oracle, in place too.  (Measured and
    not adopted: one strided launch of the N=4096 transform kernel per channel, 0.611 against
    0.626 of the HBM roofline for the tile kernel at 8 channels x 8192 polynomials.)"""
    n, limbs, batch = 4096, 3, 1024 + 5
    qs = _ntt_primes(limbs - 1) + [Q29]          # the last channel runs the 4q-lazy kernel
    rng = np.random.default_rng(13100)
    fwd_t, inv_t = [], []
    for q in qs:
        psi = _psi(n, q)
        fwd_t.append(lib.make_bitrev_table(n, q, psi))
        inv_t.append(lib.make_bitrev_table(n, q, pow(psi, q - 2, q)))
    a = np.stack([rng.integers(0, q, (batch, n), dtype=np.int32) for q in qs], axis=1)
    b = np.stack([rng.integers(0, q, (batch, n), dtype=np.int32) for q in qs], axis=1)
    a[0] = np.array(qs, dtype=np.int32)[:, None] - 1
    rows = np.unique(np.concatenate([[0, 1, batch - 1], rng.integers(0, batch, 40)]))
    d_a, d_b = dev(a), dev(b)
    d_o = torch.empty_like(d_a)
    with lib.RnsPlan(qs, fwd_t) as pf, lib.RnsPlan(qs, inv_t) as pi:
        pi.gs(d_a, d_o, batch)
        got = d_o.cpu().numpy()
        for l, q in enumerate(qs):
            assert np.array_equal(got[rows, l], oracle_mod.ntt_gs(a[rows, l], inv_t[l], q)), ("gs", l)
        lib.rns_polymul_negacyclic(pf, pi, d_a, d_b, d_o, batch)
        got = d_o.cpu().numpy()
        for l, q in enumerate(qs):
            prod = oracle_mod.pointwise(oracle_mod.ntt_ct(a[rows, l], fwd_t[l], q),
                                        oracle_mod.ntt_ct(b[rows, l], fwd_t[l], q), q)
            want = oracle_mod.scale(oracle_mod.ntt_gs(prod, inv_t[l], q),
                                    oracle_mod.powmod(n, q - 2, q), q)
            assert np.array_equal(got[rows, l], want), ("polymul", l)
        assert np.array_equal(d_a.cpu().numpy(), a)
        pi.gs(d_a, d_a, batch)
        got = d_a.cpu().numpy()
        for l, q in enumerate(qs):
            assert np.array_equal(got[rows, l], oracle_mod.ntt_gs(a[rows, l], inv_t[l], q)), ("in place", l)


def test_rns_batches(lib, oracle_mod):
    """SURVEY 8f.1: N=4096 polynomials in RNS form, [batch][L][4096], one launch for all
    channels, each channel with its own prime and table.  GS and CT per channel against
    the oracle; the negacyclic product per channel against the oracle pipeline and, for
    one channel, the O(N^2) schoolbook product."""
    n, limbs, batch = 4096, 5, 7
    qs = _ntt_primes(limbs - 1) + [Q29]
    rng = np.random.default_rng(13000)
    fwd_t, inv_t = [], []
    for q in qs:
        psi = _psi(n, q)
        fwd_t.append(lib.make_bitrev_table(n, q, psi))
        inv_t.append(lib.make_bitrev_table(n, q, pow(psi, q - 2, q)))
    a = np.stack([np.stack([rng.integers(0, q, n, dtype=np.int32) for q in qs]) for _ in range(batch)])
    b = np.stack([np.stack([rng.integers(0, q, n, dtype=np.int32) for q in qs]) for _ in range(batch)])
    a[0, :, :] = np.array(qs, dtype=np.int32)[:, None] - 1
    d_a, d_b = dev(a), dev(b)
    d_o = torch.empty_like(d_a)
    with lib.RnsPlan(qs, fwd_t) as pf, lib.RnsPlan(qs, inv_t) as pi:
        pi.gs(d_a, d_o, batch)
        got = d_o.cpu().numpy()
        for l, q in enumerate(qs):
            assert np.array_equal(got[:, l], oracle_mod.ntt_gs(a[:, l], inv_t[l], q)), ("gs", l)
        pf.ct(d_a, d_o, batch)
        got = d_o.cpu().numpy()
        for l, q in enumerate(qs):
            assert np.array_equal(got[:, l], oracle_mod.ntt_ct(a[:, l], fwd_t[l], q)), ("ct", l)
        lib.rns_polymul_negacyclic(pf, pi, d_a, d_b, d_o, batch)
        got = d_o.cpu().numpy()
        for l, q in enumerate(qs):
            prod = oracle_mod.pointwise(oracle_mod.ntt_ct(a[:, l], fwd_t[l], q),
                                        oracle_mod.ntt_ct(b[:, l], fwd_t[l], q), q)
            want = oracle_mod.scale(oracle_mod.ntt_gs(prod, inv_t[l], q),
                                    oracle_mod.powmod(n, q - 2, q), q)
            assert np.array_equal(got[:, l], want), ("polymul", l)
        assert np.array_equal(got[1, 0], oracle_mod.negacyclic_schoolbook(a[1, 0], b[1, 0], qs[0]))
        # in place, and the operands were left untouched above
        assert np.array_equal(d_a.cpu().numpy(), a)
        pi.gs(d_a, d_a, batch)
        for l, q in enumerate(qs):
            assert np.array_equal(d_a.cpu().numpy()[:, l], oracle_mod.ntt_gs(a[:, l], inv_t[l], q))


@pytest.mark.parametrize("logn", [6, 7, 8, 9, 10, 11])
def test_small_n_ct_and_polymul_fast_paths(lib, oracle_mod, logn):
    """N = 512..2048: warp-per-block forward (CT) kernel and the product kernel
    (pointwise + inverse + N^-1 in one launch), whole and ragged batches, q = 3329-like
    small prime (12289 for N <= 2048 negacyclic needs 2N | q-1) and 29-bit q."""
    n = 1 << logn
    rng = np.random.default_rng(14000 + logn)
    for q, g in ((Q29, 3), (12289, 11)):
        fwd, inv = lib.negacyclic_tables(n, q, g)
        for batch in (32, 33, 64):
            a = rng.integers(0, q, (batch, n), dtype=np.int32)
            b = rng.integers(0, q, (batch, n), dtype=np.int32)
            a[0] = q - 1
            d_a, d_b = dev(a), dev(b)
            d_c = torch.empty_like(d_a)
            with lib.Plan(logn, q, fwd) as pf, lib.Plan(logn, q, inv) as pi:
                pf.ct(d_a, d_c, batch)
                assert "ct_small" in pf.last_path, pf.last_path
                assert np.array_equal(d_c.cpu().numpy(), oracle_mod.ntt_ct(a, fwd, q)), (logn, q, batch)
                lib.polymul_negacyclic(pf, pi, d_a, d_b, d_c, batch)
                if batch % (2048 >> logn) == 0:
                    assert "dual" in pi.last_path, pi.last_path
                prod = oracle_mod.pointwise(oracle_mod.ntt_ct(a, fwd, q), oracle_mod.ntt_ct(b, fwd, q), q)
                want = oracle_mod.scale(oracle_mod.ntt_gs(prod, inv, q), oracle_mod.powmod(n, q - 2, q), q)
                assert np.array_equal(d_c.cpu().numpy(), want), (logn, q, batch)
                if logn <= 10:
                    assert np.array_equal(want[1], oracle_mod.negacyclic_schoolbook(a[1], b[1], q))
                assert np.array_equal(d_a.cpu().numpy(), a) and np.array_equal(d_b.cpu().numpy(), b)


def test_segmented_table_path(lib, oracle_mod):
    """Batches >= 64 of N >= 2^16 (and RNS batches) stage each tile position's twiddle
    table in shared memory per segment of the CTA's work range: whole-batch parity with
    a ragged batch that makes ranges straddle position changes."""
    rng = np.random.default_rng(15000)
    for logn, batch in ((16, 70), (17, 65)):
        n = 1 << logn
        table = rng.integers(0, Q29, n, dtype=np.int32)
        a = rng.integers(0, Q29, (batch, n), dtype=np.int32)
        out, path = run_gs(lib, a, table, Q29)
        assert "tile" in path
        assert np.array_equal(out, oracle_mod.ntt_gs(a, table, Q29)), logn
    n, limbs, batch = 4096, 3, 67
    qs = _ntt_primes(limbs)
    tabs = [rng.integers(0, q, n, dtype=np.int32) for q in qs]
    a = np.stack([np.stack([rng.integers(0, q, n, dtype=np.int32) for q in qs]) for _ in range(batch)])
    d_a = dev(a)
    d_o = torch.empty_like(d_a)
    with lib.RnsPlan(qs, tabs) as rp:
        rp.gs(d_a, d_o, batch)
    got = d_o.cpu().numpy()
    for l, q in enumerate(qs):
        assert np.array_equal(got[:, l], oracle_mod.ntt_gs(a[:, l], tabs[l], q)), l


# ------------------------------------------------------------------ round 2 additions
def _golden_dir():
    import os
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("logn,world", [(16, 2), (16, 4), (16, 8), (18, 4), (17, 8)])
def test_scatter_kernels_with_self_peers(lib, oracle_mod, logn, world):
    """nttb200_gs_stage_range_scatter on ONE GPU: every "peer" buffer lives on this device,
    the ranks run one after the other.  Exercises column_kernel<.., SCATTER=true>, its peer
    index math, the tile pass + scatter (stage_begin == 0) and the cross-device pass +
    return scatter (stage_begin == log2(S/G)); the reassembled vector must equal the golden
    transform of the whole input, the intermediate the transposed local results."""
    from test_multigpu_cpu import gs_stage_range_numpy
    import ntt_aie_b200.fourstep as fs
    n, s = 1 << logn, (1 << logn) // world
    logs, c = logn - (world.bit_length() - 1), s // world
    rng = np.random.default_rng(16000 + logn + world)
    table = rng.integers(0, Q29, n, dtype=np.int32)
    a = rng.integers(0, Q29, n, dtype=np.int32)
    want = oracle_mod.ntt_gs(a, table, Q29)
    recv = [torch.zeros(s, dtype=torch.int32, device="cuda") for _ in range(world)]
    final = [torch.zeros(s, dtype=torch.int32, device="cuda") for _ in range(world)]
    recv_ptrs, final_ptrs = [t.data_ptr() for t in recv], [t.data_ptr() for t in final]
    local_results = []
    for r in range(world):                       # steps 1+2 of every rank
        t_local = fs.local_table(table, world, r)
        shard = dev(a[r * s:(r + 1) * s])
        with lib.Plan(logs, Q29, t_local) as plan:
            plan.gs_stage_range_scatter(shard, 0, logs, recv_ptrs, r)
            torch.cuda.synchronize()
            assert "scatter" in plan.last_path
        local_results.append(oracle_mod.ntt_gs(a[r * s:(r + 1) * s], t_local, Q29))
    for k in range(world):                       # rank k holds slice k of every shard
        exp = np.concatenate([local_results[r][k * c:(k + 1) * c] for r in range(world)])
        assert np.array_equal(recv[k].cpu().numpy(), exp), ("transpose", k)
    t_cross = fs.cross_table(table, world, s)
    logc = logs - (world.bit_length() - 1)
    for k in range(world):                       # steps 3+4
        exp3 = gs_stage_range_numpy(recv[k].cpu().numpy(), t_cross, Q29, logc, logs)
        with lib.Plan(logs, Q29, t_cross) as plan:
            plan.gs_stage_range_scatter(recv[k], logc, logs, final_ptrs, k)
            torch.cuda.synchronize()
        # the pass ran in place on everything but its scattered last stage group; compare
        # through the reassembled result below and the stage-range restatement here
        for r in range(world):
            assert np.array_equal(final[r].cpu().numpy()[k * c:(k + 1) * c], exp3[r * c:(r + 1) * c])
    got = np.concatenate([t.cpu().numpy() for t in final])
    assert np.array_equal(got, want)


@pytest.mark.parametrize("logn", [22, 24, 26, 27])
def test_large_transforms_against_reference_digests(lib, logn):
    """One N = 2^22 / 2^24 / 2^26 (BASELINE configs[4] size) / 2^27 transform against the
    digest of the reference's own golden output (tests/golden/make_golden_large.py); table
    shipped from the host AND generated on the device."""
    import os
    from tools.digest import as_unsigned, digest_numpy, digest_torch
    g = np.load(os.path.join(_golden_dir(), "large_digests.npz"))
    n, q = 1 << logn, int(g["q"])
    a = np.random.default_rng(int(g["seed"]) + logn).integers(0, q, n, dtype=np.int32)
    assert digest_numpy(a) == tuple(int(v) for v in g[f"in_digest_{logn}"])
    d_in = dev(a)
    d_out = torch.empty_like(d_in)
    want = tuple(int(v) for v in g[f"digest_{logn}"])
    w = lib.powmod(int(g["g"]), (q - 1) // n, q)
    plans = [lambda: lib.Plan.generated(logn, q, lib.GEN_POWERS, w)]
    if logn <= 26:
        plans.append(lambda: lib.Plan(logn, q, lib.make_roots(n, q, int(g["g"]))))
    for make in plans:
        d_out.zero_()
        with make() as plan:
            plan.gs(d_in, d_out, 1)
            torch.cuda.synchronize()
            assert "tile" in plan.last_path, plan.last_path
        assert as_unsigned(digest_torch(d_out)) == want, logn
        assert np.array_equal(d_out[:16].cpu().numpy(), g[f"head_{logn}"])
        assert np.array_equal(d_out[-16:].cpu().numpy(), g[f"tail_{logn}"])
    # in place
    with plans[0]() as plan:
        plan.gs(d_in, d_in, 1)
        torch.cuda.synchronize()
    assert as_unsigned(digest_torch(d_in)) == want


@pytest.mark.parametrize("logn", [1, 4, 11, 12, 13, 16, 20])
def test_generated_tables_match_host_tables(lib, logn):
    """nttb200_plan_create_generated: tables built on the device equal make_roots /
    make_bitrev_table / the four-step derived tables built on the host, word for word,
    and transform identically."""
    import ntt_aie_b200.fourstep as fs
    n = 1 << logn
    for q, g in ((Q29, 3), (3329, 3), (Q30, 7)):
        w = lib.powmod(g, (q - 1) // n, q)
        with lib.Plan.generated(logn, q, lib.GEN_POWERS, w) as plan:
            assert np.array_equal(plan.table(), lib.make_roots(n, q, g)), (logn, q)
        base = 12345 % q
        with lib.Plan.generated(logn, q, lib.GEN_BITREV, base) as plan:
            assert np.array_equal(plan.table(), lib.make_bitrev_table(n, q, base)), (logn, q)
    # four-step derived tables of a global transform of length 2^(logn+3) on 8 ranks
    world, glog = 8, logn + 3
    if glog <= 22:
        w = lib.powmod(3, (Q29 - 1) >> glog, Q29)
        table = lib.make_roots(1 << glog, Q29, 3)
        bt = lib.make_bitrev_table(1 << glog, Q29, 777)
        for r in (0, 5, 7):
            with lib.Plan.generated(logn, Q29, lib.GEN_POWERS, w, gen_logn=glog, block_mult=world + r) as p:
                assert np.array_equal(p.table()[1:], fs.local_table(table, world, r)[1:])
            with lib.Plan.generated(logn, Q29, lib.GEN_BITREV, 777, gen_logn=glog, block_mult=world + r) as p:
                assert np.array_equal(p.table()[1:], fs.local_table(bt, world, r)[1:])
        if n >= world:
            with lib.Plan.generated(logn, Q29, lib.GEN_POWERS, w, gen_logn=glog) as p:
                assert np.array_equal(p.table()[1:world], table[1:world])
    a = np.random.default_rng(17000 + logn).integers(0, Q29, (3, n), dtype=np.int32)
    w = lib.powmod(3, (Q29 - 1) // n, Q29)
    d_in, d_out = dev(a), torch.empty(3, n, dtype=torch.int32, device="cuda")
    with lib.Plan.generated(logn, Q29, lib.GEN_POWERS, w) as plan:
        plan.gs(d_in, d_out, 3)
    assert np.array_equal(d_out.cpu().numpy(), oracle_ntt(a, lib.make_roots(n, Q29, 3), Q29))


def oracle_ntt(a, roots, p):
    import oracle
    return oracle.ntt_gs(a, roots, p)


def test_unreduced_inputs_like_the_reference_harness(lib, oracle_mod):
    """The reference harness feeds a[i] = i (src/test.cpp:141); at its larger sizes
    (N = 4096, 8192 with p = 3329) that is not reduced and the golden takes it mod p on
    first touch.  nttb200_gs_host / ntt() reduce always; device entry points with the
    REDUCE_INPUT plan flag; nttb200_reduce by itself."""
    import os
    g = np.load(os.path.join(_golden_dir(), "unreduced_inputs.npz"))
    for n in (4096, 8192):
        a = np.arange(n, dtype=np.int32)
        roots = g[f"roots_{n}"]
        assert np.array_equal(lib.ntt(a, n, roots, 3329), g[f"out_{n}"]), n
        for flags in (lib.REDUCE_INPUT, lib.REDUCE_INPUT | lib.FORCE_GENERIC):
            out, _ = run_gs(lib, a, roots, 3329, flags=flags)
            assert np.array_equal(out, g[f"out_{n}"]), (n, flags)
            out, _ = run_gs(lib, a, roots, 3329, flags=flags, inplace=True)
            assert np.array_equal(out, g[f"out_{n}"]), (n, flags, "in place")
    assert np.array_equal(lib.ntt(g["a_q29"], 4096, g["roots_q29"], Q29), g["out_q29"])
    out, _ = run_gs(lib, g["a_q29"], g["roots_q29"], Q29, flags=lib.REDUCE_INPUT)
    assert np.array_equal(out, g["out_q29"])
    # nttb200_reduce: any int32, incl. negative (mapped to the mathematical residue), ragged
    rng = np.random.default_rng(18000)
    for q in (3329, Q29, 1 << 30, 2):
        for count in (1, 5, 4096 + 3):
            x = rng.integers(-(1 << 31), (1 << 31) - 1, count, dtype=np.int64).astype(np.int32)
            with lib.Plan(4, q, np.zeros(16, np.int32)) as plan:
                d = dev(x)
                o = torch.empty_like(d)
                plan.reduce(d, o, count)
                assert np.array_equal(o.cpu().numpy(), (x.astype(np.int64) % q).astype(np.int32))
                plan.reduce(d[1:], o[1:], count - 1)      # unaligned views
                assert np.array_equal(o.cpu().numpy()[1:], (x[1:].astype(np.int64) % q).astype(np.int32))
    # forward network with the flag
    n = 4096
    fwd, _ = lib.negacyclic_tables(n, Q29, 3)
    a = g["a_q29"]
    d_in, d_out = dev(a), torch.empty(n, dtype=torch.int32, device="cuda")
    with lib.Plan(12, Q29, fwd, flags=lib.REDUCE_INPUT) as plan:
        plan.ct(d_in, d_out, 1)
    assert np.array_equal(d_out.cpu().numpy(), oracle_mod.ntt_ct((a.astype(np.int64) % Q29).astype(np.int32), fwd, Q29))


def test_concurrent_launches_on_one_plan(lib, oracle_mod):
    """SURVEY 8b: one plan, several host threads, each on its own stream."""
    import threading
    n, p, batch = 4096, Q29, 64
    roots = lib.make_roots(n, p, 3)
    rng = np.random.default_rng(19000)
    a = rng.integers(0, p, (4, batch, n), dtype=np.int32)
    want = [oracle_mod.ntt_gs(a[k], roots, p) for k in range(4)]
    outs = [None] * 4
    with lib.Plan(12, p, roots) as plan:
        def work(k):
            st = torch.cuda.Stream()
            d_in = dev(a[k])
            d_out = torch.empty_like(d_in)
            for _ in range(20):
                plan.gs(d_in, d_out, batch, -1, st)
                _ = plan.last_path
            st.synchronize()
            outs[k] = d_out.cpu().numpy()
        threads = [threading.Thread(target=work, args=(k,)) for k in range(4)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
    for k in range(4):
        assert np.array_equal(outs[k], want[k]), k


def test_stage_range_empty_batch_and_scatter_limits(lib):
    n = 1 << 14
    table = np.random.default_rng(3).integers(0, Q29, n, dtype=np.int32)
    with lib.Plan(14, Q29, table) as plan:
        plan.gs_stage_range(0, 0, 0, 2, 14)          # batch 0 with a column-pass range: OK, no launch
        plan.gs_stage_range(0, 0, 0, 0, 14)
        plan.gs(0, 0, 0)
        plan.ct(0, 0, 0)


def test_lazy_range_limits_in_products_and_the_persistent_kernel(lib, oracle_mod):
    """The 4q-lazy ranges at their limit: q = 2^29 - 3 (8q within 24 of 2^32) and q = 2^29 - 1,
    tables and inputs pinned at q - 1 / random, through the one-kernel product (N = 4096), the
    DUAL one-pass product (N = 2^13) and the persistent tile/column kernel (N = 2^16, a batch
    large enough to take it).  The kernels are table-agnostic, so arbitrary tables stand in for
    the transform pair; the oracle pipeline is CT, CT, pointwise, GS, N^-1."""
    rng = np.random.default_rng(20500)
    for q in ((1 << 29) - 3, (1 << 29) - 1):
        for logn, batch in ((12, 24), (13, 9)):
            n = 1 << logn
            fwd = rng.integers(0, q, n, dtype=np.int32)
            inv = rng.integers(0, q, n, dtype=np.int32)
            fwd[1::3] = q - 1
            inv[1::2] = q - 1
            a = rng.integers(0, q, (batch, n), dtype=np.int32)
            b = rng.integers(0, q, (batch, n), dtype=np.int32)
            a[0] = q - 1
            b[0] = q - 1
            b[1] = q - 1
            prod = oracle_mod.pointwise(oracle_mod.ntt_ct(a, fwd, q), oracle_mod.ntt_ct(b, fwd, q), q)
            want = oracle_mod.scale(oracle_mod.ntt_gs(prod, inv, q), oracle_mod.powmod(n, q - 2, q), q)
            with lib.Plan(logn, q, fwd) as pf, lib.Plan(logn, q, inv) as pi:
                d_c = torch.zeros(batch, n, dtype=torch.int32, device="cuda")
                lib.polymul_negacyclic(pf, pi, dev(a), dev(b), d_c, batch)
                assert np.array_equal(d_c.cpu().numpy(), want), (q, logn, pi.last_path)
        # N = 2^16: 12 tiles per team * 148 SMs * 8 teams / 16 tiles = 888 polynomials at least
        n, batch = 1 << 16, 896
        table = rng.integers(0, q, n, dtype=np.int32)
        table[1::2] = q - 1
        a = rng.integers(0, q, (batch, n), dtype=np.int32)
        a[0] = q - 1
        rows = np.array([0, 1, 500, batch - 1])
        d_a = dev(a)
        d_o = torch.empty_like(d_a)
        with lib.Plan(16, q, table) as plan:
            plan.gs(d_a, d_o, batch)
            path = plan.last_path
        assert np.array_equal(d_o[torch.from_numpy(rows).cuda()].cpu().numpy(),
                              oracle_mod.ntt_gs(a[rows], table, q)), (q, path)


def test_polymul4096_one_kernel(lib, oracle_mod):
    """N = 4096 products in ONE kernel (operands parked in tensor memory): ragged batches
    around the team/grid sizes, three moduli (29-bit, 30-bit, 16-bit), output aliasing a or
    b, against the oracle pipeline CT, CT, pointwise, GS, N^-1 and one schoolbook row."""
    n = 4096
    rng = np.random.default_rng(20000)
    for q in (Q29, _ntt_primes(1)[0], 40961):
        psi = _psi(n, q)
        fwd = lib.make_bitrev_table(n, q, psi)
        inv = lib.make_bitrev_table(n, q, pow(psi, q - 2, q))
        big = 1190 if q == Q29 else 19
        a = rng.integers(0, q, (big, n), dtype=np.int32)
        b = rng.integers(0, q, (big, n), dtype=np.int32)
        a[0] = q - 1
        b[0] = q - 1
        a[1] = 0
        prod = oracle_mod.pointwise(oracle_mod.ntt_ct(a, fwd, q), oracle_mod.ntt_ct(b, fwd, q), q)
        want = oracle_mod.scale(oracle_mod.ntt_gs(prod, inv, q), oracle_mod.powmod(n, q - 2, q), q)
        assert np.array_equal(want[2], oracle_mod.negacyclic_schoolbook(a[2], b[2], q))
        with lib.Plan(12, q, fwd) as pf, lib.Plan(12, q, inv) as pi:
            for batch in (1, 7, 8, 9, big):
                d_a, d_b = dev(a[:batch]), dev(b[:batch])
                d_c = torch.zeros_like(d_a)
                lib.polymul_negacyclic(pf, pi, d_a, d_b, d_c, batch)
                assert "one_kernel" in pi.last_path, pi.last_path
                assert np.array_equal(d_c.cpu().numpy(), want[:batch]), (q, batch)
                assert np.array_equal(d_a.cpu().numpy(), a[:batch])
                assert np.array_equal(d_b.cpu().numpy(), b[:batch])
                lib.polymul_negacyclic(pf, pi, d_a, d_b, d_a, batch)      # c aliases a
                assert np.array_equal(d_a.cpu().numpy(), want[:batch]), (q, batch, "alias a")
                d_a = dev(a[:batch])
                lib.polymul_negacyclic(pf, pi, d_a, d_b, d_b, batch)      # c aliases b
                assert np.array_equal(d_b.cpu().numpy(), want[:batch]), (q, batch, "alias b")
            # twice in a row on one stream (TMEM is allocated and released per launch)
            d_a, d_b = dev(a), dev(b)
            d_c = torch.zeros_like(d_a)
            for _ in range(3):
                lib.polymul_negacyclic(pf, pi, d_a, d_b, d_c, big)
            assert np.array_equal(d_c.cpu().numpy(), want)


@pytest.mark.parametrize("logn", [3, 9, 12, 14, 17])
def test_wide_moduli(lib, oracle_mod, logn):
    """SURVEY 8f.4: 2^30 < q < 2^31 (outside the reference's int32 domain; oracle = the
    widened restatement).  GS with arbitrary tables, CT, partial depth, AIE order, the
    negacyclic product and pointwise/scale, at an NTT prime (15*2^27+1), the Mersenne prime
    2^31-1 and 2^30+3; inputs pinned at q-1."""
    n = 1 << logn
    rng = np.random.default_rng(21000 + logn)
    for q in (2013265921, 2147483647, (1 << 30) + 3):
        table = rng.integers(0, q, n, dtype=np.int64).astype(np.int32)
        a = rng.integers(0, q, (3, n), dtype=np.int64).astype(np.int32)
        a[0] = q - 1
        table[1::2] = q - 1
        out, path = run_gs(lib, a, table, q)
        assert path == "generic_stage_pass"
        assert np.array_equal(out, oracle_mod.ntt_gs(a, table, q)), (logn, q)
        out, _ = run_gs(lib, a, table, q, stage=logn // 2, inplace=True)
        assert np.array_equal(out, oracle_mod.ntt_gs(a, table, q, logn // 2)), (logn, q, "partial")
        d_in = dev(a)
        d_out = torch.empty_like(d_in)
        with lib.Plan(logn, q, table) as plan:
            plan.ct(d_in, d_out, 3)
            assert np.array_equal(d_out.cpu().numpy(), oracle_mod.ntt_ct(a, table, q)), (logn, q, "ct")
            b = rng.integers(0, q, (3, n), dtype=np.int64).astype(np.int32)
            plan.pointwise(d_in, dev(b), d_out, 3 * n)
            assert np.array_equal(d_out.cpu().numpy(), oracle_mod.pointwise(a, b, q))
            plan.scale(d_in, d_out, 3 * n, q - 2)
            assert np.array_equal(d_out.cpu().numpy(), oracle_mod.scale(a, q - 2, q))
        if logn >= 4:
            out, _ = run_gs(lib, a, table, q, flags=1)
            assert np.array_equal(out, oracle_mod.ans_order_permute(oracle_mod.ntt_gs(a, table, q)))
    # negacyclic product at the NTT prime 2013265921 (primitive root 31)
    q, g = 2013265921, 31
    fwd, inv = lib.negacyclic_tables(n, q, g)
    a = rng.integers(0, q, (2, n), dtype=np.int64).astype(np.int32)
    b = rng.integers(0, q, (2, n), dtype=np.int64).astype(np.int32)
    prod = oracle_mod.pointwise(oracle_mod.ntt_ct(a, fwd, q), oracle_mod.ntt_ct(b, fwd, q), q)
    want = oracle_mod.scale(oracle_mod.ntt_gs(prod, inv, q), pow(n, q - 2, q), q)
    if logn <= 9:
        assert np.array_equal(want[0], oracle_mod.negacyclic_schoolbook(a[0], b[0], q))
    with lib.Plan(logn, q, fwd) as pf, lib.Plan(logn, q, inv) as pi:
        d_c = torch.empty(2, n, dtype=torch.int32, device="cuda")
        lib.polymul_negacyclic(pf, pi, dev(a), dev(b), d_c, 2)
        assert np.array_equal(d_c.cpu().numpy(), want), logn
    # generated tables on the wide range
    w = lib.powmod(g, (q - 1) // n, q)
    with lib.Plan.generated(logn, q, lib.GEN_POWERS, w) as plan:
        assert np.array_equal(plan.table(), lib.make_roots(n, q, g))


def _bitrev_index(n):
    logn = n.bit_length() - 1
    idx = np.arange(n)
    rev = np.zeros(n, dtype=np.int64)
    for b in range(logn):
        rev |= ((idx >> b) & 1) << (logn - 1 - b)
    return rev


@pytest.mark.parametrize("logn", [1, 5, 11, 12, 13, 16])
def test_bitrev_layout_adapters(lib, oracle_mod, logn):
    """SURVEY 8f.2: input stored in bit-reversed order / output delivered in bit-reversed
    order.  At N = 4096 both adapters are fused into the golden kernel's load and store
    (path fused_gs4096_tma_bitrev); elsewhere they are one permutation pass.  Also the
    standalone permutation, out of place and in place, and the forward network."""
    n = 1 << logn
    rev = _bitrev_index(n)
    rng = np.random.default_rng(22000 + logn)
    table = rng.integers(0, Q29, n, dtype=np.int32)
    a = rng.integers(0, Q29, (11, n), dtype=np.int32)
    a[0] = np.arange(n) % Q29
    want = oracle_mod.ntt_gs(a, table, Q29)
    for flags, src, exp in ((lib.OUTPUT_BITREV, a, want[:, rev]),
                            (lib.INPUT_BITREV, a[:, rev], want),
                            (lib.INPUT_BITREV | lib.OUTPUT_BITREV, a[:, rev], want[:, rev])):
        for inplace in (False, True):
            out, path = run_gs(lib, src, table, Q29, flags=flags, inplace=inplace)
            assert np.array_equal(out, exp), (logn, flags, inplace, path)
            if logn == 12:
                assert path == "fused_gs4096_tma_bitrev"
        out, _ = run_gs(lib, src, table, Q29, flags=flags | lib.FORCE_GENERIC)
        assert np.array_equal(out, exp), (logn, flags, "generic")
    with lib.Plan(logn, Q29, table, flags=lib.OUTPUT_BITREV) as plan:
        d_in, d_out = dev(a), torch.empty(11, n, dtype=torch.int32, device="cuda")
        plan.ct(d_in, d_out, 11)
        assert np.array_equal(d_out.cpu().numpy(), oracle_mod.ntt_ct(a, table, Q29)[:, rev])
        plan.bitrev_permute(d_in, d_out, 11)
        assert np.array_equal(d_out.cpu().numpy(), a[:, rev])
        plan.bitrev_permute(d_in, d_in, 11)
        assert np.array_equal(d_in.cpu().numpy(), a[:, rev])
    if logn >= 4:
        with pytest.raises(lib.NttError):
            lib.Plan(logn, Q29, table, flags=lib.OUTPUT_BITREV | lib.ORDER_AIE_DEVICE)


def test_persistent_tile_column_kernel_full_batch(lib, oracle_mod):
    """N = 2^16 with a batch large enough for the persistent tile-item / column-item kernel
    (kernels_tilecol.cu; smaller batches take the two passes): sampled rows against the oracle,
    linearity over the whole batch, in place, and the product tail (DUAL) via polymul."""
    logn, batch = 16, 1000
    n = 1 << logn
    rng = np.random.default_rng(23000)
    table = rng.integers(0, Q29, n, dtype=np.int32)
    gen = torch.Generator(device="cuda").manual_seed(23000)
    a = torch.randint(0, Q29, (batch, n), dtype=torch.int32, device="cuda", generator=gen)
    fa, f2 = torch.empty_like(a), torch.empty_like(a)
    with lib.Plan(logn, Q29, table) as plan:
        plan.gs(a, fa, batch)
        torch.cuda.synchronize()
        assert "tilecol" in plan.last_path, plan.last_path
        a2 = ((a.to(torch.int64) * 3) % Q29).to(torch.int32)
        plan.gs(a2, f2, batch)
        assert torch.equal(f2.to(torch.int64), (fa.to(torch.int64) * 3) % Q29)
        idx = [0, 1, 499, batch - 1] + rng.integers(0, batch, 4).tolist()
        assert np.array_equal(fa[idx].cpu().numpy(), oracle_mod.ntt_gs(a[idx].cpu().numpy(), table, Q29))
        plan.gs(a2, a2, batch)                      # in place
        assert torch.equal(a2, f2)
    fwd, inv = lib.negacyclic_tables(n, Q29, 3)
    b = torch.randint(0, Q29, (batch, n), dtype=torch.int32, device="cuda", generator=gen)
    b[0].zero_()
    b[0, 5] = 1                                      # x^5: a negacyclic shift
    with lib.Plan(logn, Q29, fwd) as pf, lib.Plan(logn, Q29, inv) as pi:
        lib.polymul_negacyclic(pf, pi, a, b, fa, batch)
        assert "tilecol" in pi.last_path, pi.last_path
    a0 = a[0].to(torch.int64)
    assert torch.equal(fa[0].to(torch.int64), torch.cat([(Q29 - a0[n - 5:]) % Q29, a0[:n - 5]]))
    i = batch - 1
    av, bv = a[i:i + 1].cpu().numpy(), b[i:i + 1].cpu().numpy()
    prod = oracle_mod.pointwise(oracle_mod.ntt_ct(av, fwd, Q29), oracle_mod.ntt_ct(bv, fwd, Q29), Q29)
    want = oracle_mod.scale(oracle_mod.ntt_gs(prod, inv, Q29), oracle_mod.powmod(n, Q29 - 2, Q29), Q29)
    assert np.array_equal(fa[i:i + 1].cpu().numpy(), want)


def test_batch_minor_layout_adapter(lib, oracle_mod):
    """SURVEY 8f.2: batch-minor [N][batch] data through the transposing adapter, then the
    transform, then back: equals the golden on every polynomial; ragged shapes."""
    rng = np.random.default_rng(24000)
    for logn, batch in ((12, 37), (6, 1000), (10, 1), (13, 5)):
        n = 1 << logn
        table = rng.integers(0, Q29, n, dtype=np.int32)
        a = rng.integers(0, Q29, (batch, n), dtype=np.int32)
        minor = np.ascontiguousarray(a.T)                 # [N][batch]
        with lib.Plan(logn, Q29, table) as plan:
            d_minor = dev(minor)
            d_major = torch.empty(batch, n, dtype=torch.int32, device="cuda")
            plan.transpose(d_minor, d_major, batch, False)
            assert np.array_equal(d_major.cpu().numpy(), a)
            plan.gs(d_major, d_major, batch)
            d_back = torch.empty(n, batch, dtype=torch.int32, device="cuda")
            plan.transpose(d_major, d_back, batch, True)
            assert np.array_equal(d_back.cpu().numpy(), oracle_mod.ntt_gs(a, table, Q29).T), (logn, batch)


def test_persistent_forward_kernel_n65536(lib, oracle_mod):
    """N = 2^16 forward transform in one persistent kernel (C-items first, T-items trailing; the
    tile comes back from L2 by TMA behind a counter): a batch large enough to take it, a 4q-lazy
    and a classic modulus, tables and one row pinned at q - 1; sampled rows against the oracle,
    the whole batch against the two-pass path (small sub-batches), and in place."""
    n = 1 << 16
    rng = np.random.default_rng(31000)
    for q, batch in ((Q29, 896), ((1 << 30) - 35, 890)):
        table = rng.integers(0, q, n, dtype=np.int32)
        table[1::2] = q - 1
        a = rng.integers(0, q, (batch, n), dtype=np.int32)
        a[0] = q - 1
        rows = [0, 1, 447, batch - 1]
        d_a = dev(a)
        d_o = torch.empty_like(d_a)
        d_c = torch.empty_like(d_a)
        with lib.Plan(16, q, table) as plan:
            plan.ct(d_a, d_o, batch)
            torch.cuda.synchronize()
            assert plan.last_path == "tilecol_persistent_ct", plan.last_path
            assert np.array_equal(d_o.cpu().numpy()[rows], oracle_mod.ntt_ct(a[rows], table, q)), q
            for s in range(0, batch, 128):
                e = min(batch, s + 128)
                plan.ct(d_a[s:e], d_c[s:e], e - s)
            torch.cuda.synchronize()
            assert plan.last_path != "tilecol_persistent_ct"
            assert torch.equal(d_c, d_o), q
            plan.ct(d_a, d_a, batch)
            torch.cuda.synchronize()
            assert torch.equal(d_a, d_o), (q, "in place")
