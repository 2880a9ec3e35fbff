#!/usr/bin/env python
"""bench.py -- batched NTT throughput on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input.  Workload
(BASELINE.json configs[1]): 65,536 independent polynomials, N=4096, 32-bit prime
q = 469762049 (7*2^26+1), twiddle table in the reference's convention
(roots[i] = w^i, w = 3^((q-1)/N), src/test.cpp:27-32), golden GS network
(src/test.cpp:34-60).  Per-GPU work is fixed as N grows (weak scaling, batched
polynomials shard with no communication).

Numbers on the one JSON line rank 0 prints:
  value      polys/s, whole job, inputs resident in HBM, device-timed (CUDA events on
             the launching stream, max over ranks);
  e2e        the same metric through the host-buffer entry point nttb200_gs_host
             (pinned host buffers, H2D + kernel + D2H every step inside the timed region),
             with the box's measured concurrent H2D+D2H copy ceiling beside it;
  roofline   algorithmic bytes (8 B per coefficient: 4 read + 4 written) per launch /
             mean launch duration, against MEASURED_PEAKS.json hbm_gbs;
  cpu_baseline  the reference's own golden ntt() (oracle/_ref, compiled from
             /root/reference/src/test.cpp:15-60) on the host cores, bounded sample;
  polymul_sweep  (N=1) BASELINE configs[2]: negacyclic products N = 2^12..2^16;
  cfg4_strong    BASELINE configs[3]: 4096 polynomials of N = 2^16 sharded over the ranks;
  fourstep       BASELINE configs[4]: one N = 2^26 transform over the ranks (NCCL all-to-all
             and the fused peer-store exchange), checked against the digest of the
             reference's own golden output.

--impl reference times only that CPU golden (all host threads) and prints the same
line with "impl": "reference".

--dump-outputs DIR writes, after the timed steps, what the last timed step returned: a fixed,
seeded sample of DUMP_ROWS output polynomials (whole rows, spread over the ranks) as
DIR/ntt_out.npy (DIR/ntt_out_rank<r>.npy on several GPUs), float64 (every residue < 2^31 is
exact), 32 MiB in all.  The inputs are seeded, so two builds run with the same arguments can
be compared output for output.  Compare dumps of the same arm only: the GPU arm draws its
inputs on the device (torch.Generator seeded 0x5EED0001 + rank), --impl reference with numpy
(default_rng(0x5EED0001)), so the two arms transform different polynomials.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LOGN = 12
N = 1 << LOGN
Q = 469762049
G = 3
BATCH = 65536
METRIC = "batched NTT polys/sec (N=4096, 32-bit q)"
BYTES_PER_POLY = 8 * N                 # algorithmic: 4 B read + 4 B written per coefficient
BFLY_PER_POLY = (N // 2) * LOGN
FALLBACK_HBM_GBS = 6650.0              # B200_PROFILING.md fallback
DUMP_ROWS = 1024                       # --dump-outputs: 1024 x 4096 float64 = 32 MiB
DUMP_SEED = 0x5EED00D0


def workload_config(polys_per_gpu: int) -> dict:
    """Identical in both arms (the driver compares them)."""
    return {"workload": "batched forward NTT: 65,536 independent polynomials per GPU, N=4096, "
                        "q=469762049",
            "logn": LOGN, "q": Q, "polys_per_gpu": polys_per_gpu,
            "table": "reference convention roots[i]=w^i (src/test.cpp:27-32)",
            "l2": "inputs larger than L2 (1 GiB in + 1 GiB out per step)"}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic_per_launch():
    """dram bytes per launch of the dominant kernel -- NOT measured in this run: read from
    the committed `ncu --set full` capture (profiles/traffic.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get("fused_gs4096_bytes_per_launch")
    except Exception:
        return None


def dump_rows(batch: int, world: int) -> np.ndarray:
    """Row indices of the --dump-outputs sample on each rank (the same on every run)."""
    k = min(batch, max(1, DUMP_ROWS // world))
    return np.sort(np.random.default_rng(DUMP_SEED).choice(batch, k, replace=False))


def dump_outputs(out_dir: str, rank: int, world: int, sample: np.ndarray) -> None:
    os.makedirs(out_dir, exist_ok=True)
    name = "ntt_out" if world == 1 else f"ntt_out_rank{rank}"
    np.save(os.path.join(out_dir, name + ".npy"), sample.astype(np.float64))


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons while the timed region runs."""

    def __init__(self, index: int, period_s: float = 0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = statistics.median(self.samples) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def gpu_numa_cpus(phys_index: int):
    """(numa node, cpus of that node this process may run on) of a GPU, or (None, None)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(phys_index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(":", 1)
        path = f"/sys/bus/pci/devices/{dom[-4:].lower()}:{rest.lower()}/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None, None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        mine = cpus & os.sched_getaffinity(0)
        return node, (mine or None)
    except Exception:
        return None, None


# --------------------------------------------------------------------- CPU golden
def _golden_fn():
    import oracle
    if oracle.have_ref():
        return "reference", oracle.ref_ntt_batch_inplace
    oracle.build()
    return "port", oracle.ntt_gs_batch_inplace


def cpu_golden_rate(sample_polys: int, threads: int, repeats: int = 2):
    """polys/s of the reference's golden ntt() on `threads` host threads."""
    import oracle
    roots = oracle.make_roots(N, Q, G)
    rng = np.random.default_rng(0x5EED0001)
    a = rng.integers(0, Q, (sample_polys, N), dtype=np.int32)
    kind, fn = _golden_fn()
    best = None
    for _ in range(repeats):
        work = a.copy()
        t0 = time.perf_counter()
        fn(work, roots, Q, threads)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return sample_polys / best, kind, best


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    sample = args.batch                       # the same 65,536 polynomials per step as the GPU arm
    import oracle
    roots = oracle.make_roots(N, Q, G)
    kind, fn = _golden_fn()
    rng = np.random.default_rng(0x5EED0001)
    a = rng.integers(0, Q, (sample, N), dtype=np.int32)
    work = a.copy()
    # ~10 core-seconds per step: the warm-up is bounded to ~20 s on small hosts
    t0 = time.perf_counter()
    fn(work, roots, Q, threads)
    per_step = time.perf_counter() - t0
    warmup = max(0, min(args.warmup, int(20.0 / per_step)) - 1)
    steps = args.steps
    for _ in range(warmup):
        np.copyto(work, a)
        fn(work, roots, Q, threads)
    total = 0.0
    for _ in range(steps):
        np.copyto(work, a)                    # untimed: restore canonical inputs
        t0 = time.perf_counter()
        fn(work, roots, Q, threads)
        total += time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, 0, 1, work[dump_rows(sample, 1)])
    value = sample * steps / total
    sample_txt = (f"{sample} polys/step x {steps} timed steps of the same workload "
                  f"(N={N}, q={Q}) on {threads} host threads, g++ -O2")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "polys/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "i32", "data": "synthetic",
        "config": workload_config(sample),
        "note": f"CPU golden ntt() (src/test.cpp:34-60), kind {kind}; host only",
        "butterflies_per_s": value * BFLY_PER_POLY,
        "cpu_baseline": {"value": value, "unit": "polys/s", "cores": threads, "kind": kind,
                         "sample": sample_txt},
        "e2e": {"value": value, "unit": "polys/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------ GPU arm
class Ctx:
    """Rank plumbing shared by the measurement blocks."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the product has no CPU path")
        torch.cuda.set_device(self.local_rank)
        self.distributed = self.world > 1
        if self.distributed:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.distributed:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.distributed:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x: float) -> float:
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.distributed:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def all_true(self, ok: bool) -> bool:
        return self.sum_over_ranks(0.0 if ok else 1.0) == 0.0


def time_launches(ctx: Ctx, fn, reps: int, warmup: int = 3):
    """Device time of `reps` back-to-back calls (CUDA events on the current stream),
    bracketed by barriers; returns (max-over-ranks total ms, per-launch ms on this rank)."""
    torch = ctx.torch
    for _ in range(warmup):
        fn()
    ctx.barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    ev[0].record()
    for k in range(reps):
        fn()
        ev[k + 1].record()
    ctx.barrier()
    total = ctx.max_over_ranks(ev[0].elapsed_time(ev[-1]))
    return total, [ev[k].elapsed_time(ev[k + 1]) for k in range(reps)]


def pcie_ceiling(ctx: Ctx, h_in, h_out, d_a, d_b, reps: int = 3):
    """The box's raw copy ceiling: every rank copies 1 GiB host->device and 1 GiB
    device->host AT THE SAME TIME (plain cudaMemcpyAsync on two streams, pinned buffers),
    all ranks together.  This is what bounds e2e: nttb200_gs_host moves exactly these bytes."""
    torch = ctx.torch
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    nbytes = h_in.numel() * 4

    def one(h2d: bool, d2h: bool) -> float:
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            if h2d:
                with torch.cuda.stream(s1):
                    d_a.copy_(h_in, non_blocking=True)
            if d2h:
                with torch.cuda.stream(s2):
                    h_out.copy_(d_b, non_blocking=True)
        torch.cuda.synchronize()
        return ctx.max_over_ranks(time.perf_counter() - t0)

    one(True, True)  # warm-up
    t_h2d, t_d2h, t_both = one(True, False), one(False, True), one(True, True)
    agg = ctx.world * reps * nbytes / 1e9
    return {"h2d_alone_GBps": agg / t_h2d, "d2h_alone_GBps": agg / t_d2h,
            "bidir_GBps_each_way": agg / t_both,
            "what": f"aggregate over {ctx.world} GPU(s), 1 GiB pinned copies each way at once, "
                    "plain cudaMemcpyAsync"}


def block_polymul_sweep(ctx: Ctx, nt, peak: float, reps: int):
    """BASELINE configs[2]: c = a (*) b mod (x^N + 1, q), N = 2^12..2^16, 2^26 coefficients
    per operand; algorithmic traffic 12 N bytes per product.  Checked on the device through
    a size-independent property: multiplying by the monomial x^k is a negacyclic shift."""
    torch = ctx.torch
    out = []
    for logn in range(12, 17):
        n = 1 << logn
        batch = (1 << 26) // n
        fwd, inv = nt.negacyclic_tables(n, Q, G)
        gen = torch.Generator(device="cuda").manual_seed(100 + logn)
        d_a = torch.randint(0, Q, (batch, n), dtype=torch.int32, device="cuda", generator=gen)
        d_b = torch.randint(0, Q, (batch, n), dtype=torch.int32, device="cuda", generator=gen)
        d_c = torch.empty_like(d_a)
        ks = [0, 1, n // 2 + 3, n - 1]
        for i, k in enumerate(ks):                 # b_i = x^k for the first few products
            d_b[i].zero_()
            d_b[i, k] = 1
        with nt.Plan(logn, Q, fwd) as pf, nt.Plan(logn, Q, inv) as pi:
            launches0 = nt.kernel_launches()
            nt.polymul_negacyclic(pf, pi, d_a, d_b, d_c, batch)
            per_call = nt.kernel_launches() - launches0
            _, ms = time_launches(ctx, lambda: nt.polymul_negacyclic(pf, pi, d_a, d_b, d_c, batch), reps)
            path = pi.last_path
        ok = True
        for i, k in enumerate(ks):
            a = d_a[i].to(torch.int64)
            want = torch.cat([(Q - a[n - k:]) % Q, a[:n - k]]) if k else a
            ok = ok and bool(torch.equal(d_c[i].to(torch.int64), want))
        ms.sort()
        t = statistics.mean(ms[1:-1]) * 1e-3
        gbs = batch * n * 12 / t / 1e9
        out.append({"logn": logn, "batch": batch, "products_per_s": batch / t, "ms": t * 1e3,
                    "algorithmic_GBps": gbs, "frac_of_measured_hbm": gbs / peak,
                    "butterflies_per_s": 3 * batch * (n // 2) * logn / t,
                    "kernel_launches_per_call": int(per_call), "kernel_path": path,
                    "monomial_shift_property_ok": ok})
        del d_a, d_b, d_c
    return out


def block_cfg4_strong(ctx: Ctx, nt, peak: float, reps: int):
    """BASELINE configs[3]: 4096 polynomials of N = 2^16 (2^28 coefficients in total),
    sharded 4096/G per GPU, no communication; strong scaling (total work fixed).  Row 0 of
    rank 0 is the fixture polynomial of tests/golden/n65536_q29_digest.npz (the reference's
    own golden output: first/last words and the word sum are compared)."""
    torch = ctx.torch
    logn, total = 16, 4096
    n = 1 << logn
    batch = total // ctx.world
    roots = nt.make_roots(n, Q, G)
    gen = torch.Generator(device="cuda").manual_seed(16 + ctx.rank)
    d_in = torch.randint(0, Q, (batch, n), dtype=torch.int32, device="cuda", generator=gen)
    fx = np.load(os.path.join(ROOT, "tests", "golden", "n65536_q29_digest.npz"))
    d_in[0].copy_(torch.from_numpy(
        np.random.default_rng(int(fx["seed"])).integers(0, Q, n, dtype=np.int32)))
    d_out = torch.empty_like(d_in)
    with nt.Plan(logn, Q, roots, device=ctx.local_rank) as plan:
        total_ms, ms = time_launches(ctx, lambda: plan.gs(d_in, d_out, batch), reps)
        path = plan.last_path
    row = d_out[0]
    ok = (bool(np.array_equal(row[:16].cpu().numpy(), fx["head"])) and
          bool(np.array_equal(row[-16:].cpu().numpy(), fx["tail"])) and
          int(row.to(torch.int64).sum().item()) == int(fx["total"]))
    # linearity over the whole shard: NTT(2a) = 2 NTT(a)
    d_2 = ((d_in.to(torch.int64) * 2) % Q).to(torch.int32)
    d_o2 = torch.empty_like(d_2)
    with nt.Plan(logn, Q, roots, device=ctx.local_rank) as plan:
        plan.gs(d_2, d_o2, batch)
        torch.cuda.synchronize()
    ok = ok and bool(torch.equal(d_o2.to(torch.int64), (d_out.to(torch.int64) * 2) % Q))
    ok = ctx.all_true(ok)
    t = total_ms / reps * 1e-3
    ms.sort()
    per_gpu_gbs = batch * n * 8 / (statistics.mean(ms[1:-1]) * 1e-3) / 1e9   # trimmed like the other blocks
    return {"workload": "4096 polys x N=2^16 (2^28 coefficients), batch-sharded, no communication",
            "n_gpus": ctx.world, "polys_per_gpu": batch, "scaling": "strong",
            "polys_per_s": total / t, "ms": t * 1e3,
            "butterflies_per_s": total * (n // 2) * logn / t,
            "per_gpu_algorithmic_GBps": per_gpu_gbs, "per_gpu_frac_of_measured_hbm": per_gpu_gbs / peak,
            "kernel_path": path, "fixture_row_and_linearity_ok": ok}


def block_fourstep(ctx: Ctx, steps: int):
    """BASELINE configs[4]: one N = 2^26 transform over the ranks."""
    from tools import fourstep_run
    torch = ctx.torch
    out = {}
    if ctx.world == 1:
        r = fourstep_run.run(26, steps, 2, verify_digest=True, generated=True, detail=False)
        out["one_gpu"] = r
        return out
    out["nccl"] = fourstep_run.run(26, steps, 2, verify_digest=True, generated=True)
    try:
        out["fused"] = fourstep_run.run(26, steps, 2, verify_digest=True, generated=True, fused=True,
                                        detail=False)
    except Exception as exc:  # symmetric memory unavailable on this box
        out["fused"] = {"unavailable": repr(exc)[:200]}
    # the same transform on one GPU (rank 0 alone), for the speed-up
    one_ms = None
    if ctx.rank == 0:
        import ntt_aie_b200 as nt
        n = 1 << 26
        w = nt.powmod(G, (Q - 1) // n, Q)
        d = torch.randint(0, Q, (n,), dtype=torch.int32, device="cuda")
        with nt.Plan.generated(26, Q, nt.GEN_POWERS, w, device=ctx.local_rank) as plan:
            for _ in range(2):
                plan.gs(d, d, 1)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                plan.gs(d, d, 1)
            e1.record()
            torch.cuda.synchronize()
            one_ms = e0.elapsed_time(e1) / steps
        del d
    ctx.barrier()
    if ctx.rank == 0:
        out["one_gpu_ms"] = one_ms
        for key in ("nccl", "fused"):
            r = out.get(key)
            if r and "ms_natural_order" in r:
                r["speedup_vs_one_gpu_natural"] = one_ms / r["ms_natural_order"]
                r["speedup_vs_one_gpu_transposed"] = one_ms / r["ms_transposed_order"]
    return out


def run_ours(args) -> None:
    ctx = Ctx()
    torch = ctx.torch
    world, rank, local_rank = ctx.world, ctx.rank, ctx.local_rank

    import ntt_aie_b200 as nt
    nt.load_library()                          # fails loudly if the .so is missing

    batch = args.batch
    roots = nt.make_roots(N, Q, G)
    plan = nt.Plan(LOGN, Q, roots, device=local_rank)
    gen = torch.Generator(device="cuda").manual_seed(0x5EED0001 + rank)
    d_in = torch.randint(0, Q, (batch, N), dtype=torch.int32, device="cuda", generator=gen)
    d_out = torch.empty_like(d_in)
    stream = torch.cuda.current_stream()

    # ---- device-resident throughput -------------------------------------------------
    for _ in range(args.warmup):
        plan.gs(d_in, d_out, batch, -1, stream)
    ctx.barrier()
    path = plan.last_path
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    launches0 = nt.kernel_launches()
    ctx.barrier()
    ev[0].record(stream)
    for k in range(args.steps):
        plan.gs(d_in, d_out, batch, -1, stream)
        ev[k + 1].record(stream)
    ctx.barrier()
    launches = nt.kernel_launches() - launches0
    clocks = sampler.stop()
    total_ms = ev[0].elapsed_time(ev[-1])
    per_launch_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    total_ms_max = ctx.max_over_ranks(total_ms)
    value = world * batch * args.steps / (total_ms_max * 1e-3)
    if args.dump_outputs:                      # d_out holds the last timed step's result
        rows = torch.from_numpy(dump_rows(batch, world)).to(d_out.device)
        dump_outputs(args.dump_outputs, rank, world, d_out[rows].cpu().numpy())

    # ---- end to end through the host-buffer entry point -----------------------------
    e2e_steps = 0 if args.no_e2e else max(3, min(args.steps, 10))
    e2e_value, same, ceiling, numa = None, None, None, None
    if e2e_steps:
        # pinned buffers from the library, allocated and first touched by a thread bound to
        # the CPUs of this GPU's NUMA node
        affinity0 = os.sched_getaffinity(0)
        node, cpus = gpu_numa_cpus(physical_gpu_index(local_rank))
        if cpus:
            os.sched_setaffinity(0, cpus)
        numa = {"node": node, "bound_cpus": len(cpus) if cpus else None}
        hb_in, hb_out = nt.HostBuffer(batch * N), nt.HostBuffer(batch * N)
        h_in = torch.from_numpy(hb_in.array).view(batch, N)
        h_out = torch.from_numpy(hb_out.array).view(batch, N)
        h_in.copy_(d_in)
        plan.gs_host(h_in, h_out, batch)      # warm-up (allocates the staging ring)
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            plan.gs_host(h_in, h_out, batch)  # synchronous: returns when h_out is complete
        torch.cuda.synchronize()
        e2e_s = ctx.max_over_ranks(time.perf_counter() - t0)
        e2e_value = world * batch * e2e_steps / e2e_s
        # cheap integrity check of the e2e result against the device-resident one
        same = bool(torch.equal(h_out[:64].cuda(), d_out[:64])) and bool(
            torch.equal(h_out[-64:].cuda(), d_out[-64:]))
        ceiling = pcie_ceiling(ctx, h_in, h_out, d_in, d_out)
        ceiling["polys_per_s_at_ceiling"] = ceiling["bidir_GBps_each_way"] * 1e9 / (N * 4)
        ceiling["e2e_frac_of_ceiling"] = e2e_value / ceiling["polys_per_s_at_ceiling"]
        del h_in, h_out
        hb_in.free()
        hb_out.free()
        os.sched_setaffinity(0, affinity0)

    peak, peak_src = measured_peaks()
    line = None
    if rank == 0:
        mean_launch_ms = statistics.mean(per_launch_ms)
        achieved = batch * BYTES_PER_POLY / (mean_launch_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": "polys/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": workload_config(batch),
            "kernel_path": path, "sharding": f"batch x{world} GPU(s), no communication",
            "butterflies_per_s": value * BFLY_PER_POLY,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "polys/s",
                    "h2d_bytes_per_step": batch * N * 4, "d2h_bytes_per_step": batch * N * 4,
                    "steps": e2e_steps, "api": "nttb200_gs_host (pinned host buffers)",
                    "matches_device_result": same, "pcie_ceiling": ceiling, "numa": numa},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": ncu_traffic_per_launch(),
                         "traffic_source": "committed ncu --set full capture (profiles/), not this run",
                         "peak_source": peak_src, "kernel": path,
                         "algorithmic_bytes_per_launch": batch * BYTES_PER_POLY,
                         "mean_launch_ms": mean_launch_ms,
                         "frac_of_nominal_8TBs": achieved / 8000.0},
        }
    plan.close()
    del d_in, d_out
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs, under the same clock ----------------------------
    if not args.no_extras:
        extras = {}
        try:
            if world == 1:
                extras["polymul_sweep"] = block_polymul_sweep(ctx, nt, peak, 10)
            torch.cuda.empty_cache()
            extras["cfg4_strong"] = block_cfg4_strong(ctx, nt, peak, 10)
            torch.cuda.empty_cache()
            extras["fourstep"] = block_fourstep(ctx, 5)
        except Exception as exc:
            extras["error"] = repr(exc)[:300]
        if line is not None:
            line.update(extras)

    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            threads = host_threads()
            sample = BATCH                        # the full workload: ~10 core-seconds
            rate, kind, secs = cpu_golden_rate(sample, threads)
            rate1, _, secs1 = cpu_golden_rate(1024, 1, repeats=1)
            line["cpu_baseline"] = {
                "value": rate, "unit": "polys/s", "cores": threads, "kind": kind,
                "sample": f"{sample} polys of the same workload (N={N}, q={Q}), best of 2, "
                          f"{secs:.3f} s wall on {threads} threads",
                "single_thread_polys_per_s": rate1}
        print(json.dumps(line), flush=True)
    if ctx.distributed:
        ctx.dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--batch", type=int, default=BATCH, help="polynomials per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs: skip the host-buffer leg")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the polymul / cfg4 / four-step blocks (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed sample of the last timed step's output to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
