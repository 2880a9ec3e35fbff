#!/usr/bin/env python
"""Packed integer slots mod t for BFV and BGV (nttb200_packed_encode / nttb200_packed_decode).

    python tools/bench_packed_encode.py [--reps 20] [--out profiles/r9_bench_packed.jsonl]

One JSON line per measurement on stdout (and appended to --out when given):
  encode   N = 2^12, 2^14, 2^16, L = 1, 8 and 32 primes below 2^30, t the largest prime below 2^30
           with t = 1 (mod 2N), both forms (SCALED, CENTRED), a batch of at least 512 MiB of slots
           plus residues (far above the 126 MB L2).  Algorithmic bytes 4 + 4 L per coefficient.
           Next to the CENTRED row the route that existed before, on the same data: a torch
           index_select of the slots into the rns_ct order and a remainder mod t, rns_gs_scaled on
           a plan of modulus t, convert(exact=True) from {t} to Q.  It is bit-identical to the
           CENTRED form; the outputs are compared before timing.
  decode   the same N and t, slots in [0, t).  Algorithmic bytes 8 per coefficient.
Fractions are of the device-to-device copy bandwidth measured in the same run.  Every line carries
the GPU name and power limit read in the same run.  CUDA events, 3 warm-ups, trimmed mean."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ntt_aie_b200 as nt  # noqa: E402
from tools.bench_rns import gpu_info, hbm_copy_gbps, primes, time_ms  # noqa: E402

BULK_BYTES = 512 << 20


def ones_plan(logn, qs):
    return nt.RnsPlan(qs, [np.ones(1 << logn, dtype=np.int32) for _ in qs], logn=logn)


def emit(out, info, hbm, **kw):
    kw["frac_of_measured_copy"] = kw["algorithmic_GBps"] / hbm
    kw["copy_GBps"] = hbm
    line = json.dumps({**kw, **info})
    print(line, flush=True)
    if out:
        with open(out, "a") as f:
            f.write(line + "\n")


def largest_t(logn):
    two_n = 2 << logn
    k = (2 ** 30 - 2) // two_n
    while any((k * two_n + 1) % d == 0 for d in range(2, int((k * two_n + 1) ** 0.5) + 1)):
        k -= 1
    return k * two_n + 1


def smallest_psi(n, t):
    """the least primitive 2n-th root of unity mod t: the odd powers of psi_0"""
    x = 2
    while pow(x, (t - 1) // 2, t) != t - 1:
        x += 1
    psi0 = pow(x, (t - 1) // (2 * n), t)
    best, w, sq = psi0, psi0, psi0 * psi0 % t
    for _ in range(n - 1):
        w = w * sq % t
        best = min(best, w)
    return best


def rns_ct_index_of_slots(logn):
    """k_i = brev((e_i - 1) / 2): e_i = 5^j mod 2N (row 0), 2N - 5^j mod 2N (row 1)"""
    n = 1 << logn
    g = [pow(5, j, 2 * n) for j in range(n // 2)]
    e = g + [2 * n - x for x in g]
    return np.array([int(format((x - 1) // 2, f"0{logn}b")[::-1], 2) for x in e], dtype=np.int64)


def rand_slots(batch, n, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randint(-(1 << 31), (1 << 31) - 1, (batch, n), dtype=torch.int64, device="cuda",
                         generator=gen).to(torch.int32)


def bench_encode(logn, L, reps, hbm, info, out):
    N = 1 << logn
    t = largest_t(logn)
    qs = [q for q in primes(L + 1) if q != t][:L]
    batch = max(1, BULK_BYTES // (4 * N * (1 + L)))
    s = rand_slots(batch, N, logn + L)
    res = torch.empty((batch, L, N), dtype=torch.int32, device="cuda")
    base_out = torch.empty_like(res)
    k = rns_ct_index_of_slots(logn)
    islot = np.empty(N, dtype=np.int64)
    islot[k] = np.arange(N)
    idx = torch.from_numpy(islot).cuda()
    psi = smallest_psi(N, t)
    m = torch.empty((batch, 1, N), dtype=torch.int32, device="cuda")
    with nt.PackedEncoder(ones_plan(logn, qs), t) as enc, \
            nt.RnsPlan.generated(logn, [t], nt.GEN_BITREV, [pow(psi, -1, t)]) as pinv, \
            ones_plan(logn, [t]) as pt, ones_plan(logn, qs) as pq, nt.RnsConv(pt, pq) as conv:

        def baseline():
            torch.remainder(s.index_select(1, idx), t, out=m.view(batch, N))
            pinv.gs_scaled(m, m, batch)
            conv.convert(m, base_out, batch, exact=True)

        baseline()
        enc.encode(s, res, batch, centred=True)
        torch.cuda.synchronize()
        identical = bool(torch.equal(res, base_out))
        base_ms = time_ms(baseline, reps)
        for centred in (False, True):
            ms = time_ms(lambda: enc.encode(s, res, batch, centred=centred), reps)
            gbps = batch * N * (4 + 4 * L) / (ms * 1e-3) / 1e9
            extra = {"baseline_ms": base_ms, "speedup_vs_baseline": base_ms / ms,
                     "baseline_bit_identical": identical} if centred else {}
            emit(out, info, hbm, op="encode", mode="centred" if centred else "scaled", N=N, L=L, t=t, batch=batch,
                 ms=ms, algorithmic_GBps=gbps, launches=3 if logn == 12 else 4, **extra)


def bench_decode(logn, reps, hbm, info, out):
    N = 1 << logn
    t = largest_t(logn)
    qs = [q for q in primes(2) if q != t][:1]
    batch = max(1, BULK_BYTES // (8 * N))
    gen = torch.Generator(device="cuda").manual_seed(logn)
    x = torch.randint(0, t, (batch, N), dtype=torch.int32, device="cuda", generator=gen)
    z = torch.empty_like(x)
    with nt.PackedEncoder(ones_plan(logn, qs), t) as enc:
        ms = time_ms(lambda: enc.decode(x, z, batch), reps)
    gbps = batch * N * 8 / (ms * 1e-3) / 1e9
    emit(out, info, hbm, op="decode", N=N, t=t, batch=batch, ms=ms, algorithmic_GBps=gbps,
         launches=2 if logn == 12 else 3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    info = gpu_info()
    hbm = hbm_copy_gbps(args.reps)
    for logn in (12, 14, 16):
        for L in (1, 8, 32):
            bench_encode(logn, L, args.reps, hbm, info, args.out)
        bench_decode(logn, args.reps, hbm, info, args.out)


if __name__ == "__main__":
    main()
