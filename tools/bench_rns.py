#!/usr/bin/env python
"""RNS batches at N = 2^13..2^16: GS, CT and the negacyclic product, all channels per call.

    python tools/bench_rns.py [--logns 13,14,15,16] [--reps 20]

Two workloads per N, one JSON line per (workload, operation) on stdout:
  bulk    L = 8 primes below 2^30, 2^28 coefficients per operand (1 GiB, far above the
          126 MB L2): channel transforms (products) per second, algorithmic GB/s (8 N bytes
          per channel transform, 12 N per channel product) and its fraction of the HBM copy
          bandwidth measured in the same run.
  ct1     one ciphertext pair: L = 32, batch = 2.  It fits in L2, so it is a latency figure,
          not a roofline fraction.  Beside it, the same work done the way a caller without
          RNS plans has to: 32 single-modulus Plan calls, each on a contiguous 2-polynomial
          batch of channel-major data, timed with the same events.
Every line carries the GPU name and power limit read in the same run and a sampled
bit-exactness check against the CPU oracle.  Device-timed with CUDA events, 3 warm-ups,
trimmed mean (min and max dropped)."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ntt_aie_b200 as nt  # noqa: E402
import oracle  # noqa: E402


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "not read"
    return {"gpu": name, "power_limit": out}


def trimmed(ms):
    ms = sorted(ms)
    return statistics.mean(ms[1:-1]) if len(ms) > 2 else statistics.mean(ms)


def time_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    ev[0].record()
    for k in range(reps):
        fn()
        ev[k + 1].record()
    torch.cuda.synchronize()
    return trimmed([ev[k].elapsed_time(ev[k + 1]) for k in range(reps)])


def hbm_copy_gbps(reps):
    """Device-to-device copy of 1 GiB: bytes read + written over time."""
    x = torch.empty(1 << 28, dtype=torch.int32, device="cuda")
    y = torch.empty_like(x)
    ms = time_ms(lambda: y.copy_(x), reps)
    del x, y
    return 2 * (1 << 30) / (ms * 1e-3) / 1e9


def primes(count, two_n=1 << 17, below=1 << 30):
    out, k = [], (below - 1) // two_n
    while len(out) < count:
        q = k * two_n + 1
        if all(q % d for d in range(3, int(q ** 0.5) + 1, 2)):
            out.append(q)
        k -= 1
    return out


def tables(n, qs):
    fwd, inv = [], []
    for q in qs:
        psi = next(pow(x, (q - 1) // (2 * n), q) for x in range(2, 1000)
                   if pow(pow(x, (q - 1) // (2 * n), q), n, q) == q - 1)
        fwd.append(nt.make_bitrev_table(n, q, psi))
        inv.append(nt.make_bitrev_table(n, q, pow(psi, q - 2, q)))
    return fwd, inv


def check(d_out, d_a, d_b, kind, fwd, inv, qs, rows, chans):
    """Sampled (polynomial, channel) pairs of the [batch][L][N] output against the oracle."""
    a = d_a[rows].cpu().numpy()
    b = d_b[rows].cpu().numpy()
    got = d_out[rows].cpu().numpy()
    n = a.shape[-1]
    for l in chans:
        q = qs[l]
        if kind == "gs":
            want = oracle.ntt_gs(a[:, l], inv[l], q)
        elif kind == "ct":
            want = oracle.ntt_ct(a[:, l], fwd[l], q)
        else:
            prod = oracle.pointwise(oracle.ntt_ct(a[:, l], fwd[l], q), oracle.ntt_ct(b[:, l], fwd[l], q), q)
            want = oracle.scale(oracle.ntt_gs(prod, inv[l], q), oracle.powmod(n, q - 2, q), q)
        if not np.array_equal(got[:, l], want):
            return False
    return True


def operations(pf, pi, d_a, d_b, d_c, batch):
    return {"gs": lambda: pi.gs(d_a, d_c, batch), "ct": lambda: pf.ct(d_a, d_c, batch),
            "polymul": lambda: nt.rns_polymul_negacyclic(pf, pi, d_a, d_b, d_c, batch)}


def bulk(logn, reps, hbm, info):
    n, limbs = 1 << logn, 8
    batch = (1 << 28) // (limbs * n)
    qs = primes(limbs)
    fwd, inv = tables(n, qs)
    gen = torch.Generator(device="cuda").manual_seed(1000 + logn)
    d_a = torch.randint(0, min(qs), (batch, limbs, n), dtype=torch.int32, device="cuda", generator=gen)
    d_b = torch.randint(0, min(qs), (batch, limbs, n), dtype=torch.int32, device="cuda", generator=gen)
    d_c = torch.empty_like(d_a)
    rows = [0, batch // 2, batch - 1]
    with nt.RnsPlan(qs, fwd, logn=logn) as pf, nt.RnsPlan(qs, inv, logn=logn) as pi:
        for kind, fn in operations(pf, pi, d_a, d_b, d_c, batch).items():
            ms = time_ms(fn, reps)
            ok = check(d_c, d_a, d_b, kind, fwd, inv, qs, rows, [0, limbs - 1])
            work = batch * limbs
            gbs = work * n * (12 if kind == "polymul" else 8) / (ms * 1e-3) / 1e9
            print(json.dumps({"workload": "bulk", "op": kind, "logn": logn, "limbs": limbs, "batch": batch,
                              "ms": ms, ("channel_products_per_s" if kind == "polymul"
                                         else "channel_transforms_per_s"): work / (ms * 1e-3),
                              "algorithmic_GBps": gbs, "hbm_copy_GBps": hbm, "frac_of_measured_hbm": gbs / hbm,
                              "bit_exact_sampled": ok, **info}), flush=True)
    del d_a, d_b, d_c


def one_ciphertext(logn, reps, info):
    n, limbs, batch = 1 << logn, 32, 2
    qs = primes(limbs)
    fwd, inv = tables(n, qs)
    gen = torch.Generator(device="cuda").manual_seed(2000 + logn)
    d_a = torch.randint(0, min(qs), (batch, limbs, n), dtype=torch.int32, device="cuda", generator=gen)
    d_b = torch.randint(0, min(qs), (batch, limbs, n), dtype=torch.int32, device="cuda", generator=gen)
    d_c = torch.empty_like(d_a)
    # channel-major copies [L][batch][N] for the per-modulus calls
    c_a, c_b = d_a.transpose(0, 1).contiguous(), d_b.transpose(0, 1).contiguous()
    c_c = torch.empty_like(c_a)
    pfs = [nt.Plan(logn, q, t) for q, t in zip(qs, fwd)]
    pis = [nt.Plan(logn, q, t) for q, t in zip(qs, inv)]
    single = {
        "gs": lambda: [pis[l].gs(c_a[l], c_c[l], batch) for l in range(limbs)],
        "ct": lambda: [pfs[l].ct(c_a[l], c_c[l], batch) for l in range(limbs)],
        "polymul": lambda: [nt.polymul_negacyclic(pfs[l], pis[l], c_a[l], c_b[l], c_c[l], batch)
                            for l in range(limbs)],
    }
    with nt.RnsPlan(qs, fwd, logn=logn) as pf, nt.RnsPlan(qs, inv, logn=logn) as pi:
        for kind, fn in operations(pf, pi, d_a, d_b, d_c, batch).items():
            ms = time_ms(fn, reps)
            ok = check(d_c, d_a, d_b, kind, fwd, inv, qs, [0, 1], [0, 17, limbs - 1])
            ms_single = time_ms(single[kind], reps)
            same = bool(torch.equal(c_c.transpose(0, 1), d_c))
            print(json.dumps({"workload": "one ciphertext (L2-resident latency, not a roofline figure)",
                              "op": kind, "logn": logn, "limbs": limbs, "batch": batch,
                              "ms_one_rns_call": ms, "ms_32_single_modulus_calls": ms_single,
                              "speedup": ms_single / ms, "bit_exact_sampled": ok,
                              "single_modulus_results_equal": same, **info}), flush=True)
    for p in pfs + pis:
        p.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--logns", default="13,14,15,16")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rns.py needs a CUDA device; nothing was measured")
    torch.cuda.set_device(0)
    info = gpu_info()
    hbm = hbm_copy_gbps(args.reps)
    print(json.dumps({"hbm_copy_GBps": hbm, "bytes": 2 << 30, **info}), flush=True)
    for logn in (int(x) for x in args.logns.split(",")):
        bulk(logn, args.reps, hbm, info)
        one_ciphertext(logn, args.reps, info)


if __name__ == "__main__":
    main()
