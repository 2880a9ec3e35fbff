#!/usr/bin/env python
"""CKKS slot encoding and decoding on RNS batches (nttb200_ckks_encode / nttb200_ckks_decode).

    python tools/bench_ckks_encode.py [--reps 20] [--out profiles/r8_bench_ckks.jsonl]

One JSON line per measurement on stdout (and appended to --out when given):
  encode   N = 2^12, 2^14, 2^16, L = 1, 8 and 32 primes below 2^30, a batch of at least 512 MiB of
           slots plus residues (far above the 126 MB L2).  Algorithmic bytes 8 + 4 L per
           coefficient (16 bytes per slot in, 4 L bytes per coefficient out).  Next to each row the
           torch baseline on the same data: index gather of the slots, torch.fft.fft, the twist,
           the round and an int64 remainder per prime; its residues are compared with the
           library's (equal, or one apart where the value lies at a half-integer within the FFT
           error).
  decode   the same N, channels = 1 and 4 of an L = 8 batch read in place (in_stride = 8 N).
           Algorithmic bytes 4 channels + 8 per coefficient.
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
SCALE = 2.0 ** 40


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


def rand_slots(batch, n, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return torch.complex(torch.rand((batch, n), dtype=torch.float64, device="cuda", generator=gen) * 2 - 1,
                         torch.rand((batch, n), dtype=torch.float64, device="cuda", generator=gen) * 2 - 1)


def baseline_encode(z, qs, logn):
    """the torch route: inverse permutation gather, FFT, twist, round, remainder per prime"""
    N, n = 1 << logn, 1 << (logn - 1)
    s = np.array([(pow(5, j, 2 * N) - 1) // 4 for j in range(n)])
    inv = np.empty(n, dtype=np.int64)
    inv[s] = np.arange(n)
    idx = torch.from_numpy(inv).cuda()
    k = torch.arange(n, device="cuda", dtype=torch.float64)
    twist = torch.exp(torch.complex(torch.zeros_like(k), -torch.pi * k / N)) * (SCALE / n)
    qcol = torch.tensor(qs, dtype=torch.int64, device="cuda").view(len(qs), 1)

    def run():
        m = torch.fft.fft(z[:, idx], dim=-1) * twist
        a = torch.round(torch.cat([m.real, m.imag], dim=-1)).to(torch.int64)
        return torch.remainder(a.unsqueeze(1), qcol).to(torch.int32)
    return run


def bench_encode(logn, L, reps, hbm, info, out):
    N, n = 1 << logn, 1 << (logn - 1)
    qs = primes(L)
    batch = max(1, BULK_BYTES // (16 * n + 4 * L * N))
    z = rand_slots(batch, n, logn + L)
    res = torch.empty((batch, L, N), dtype=torch.int32, device="cuda")
    with nt.CkksEncoder(ones_plan(logn, qs)) as enc:
        ms = time_ms(lambda: enc.encode(z, res, batch, SCALE), reps)
        base = baseline_encode(z, qs, logn)
        base_ms = time_ms(base, reps)
        rows = torch.tensor([0, batch - 1], device="cuda")
        want = base()[rows].long()
        got = res[rows].long()
        d = (got - want).remainder(torch.tensor(qs, device="cuda").view(1, L, 1))
        qv = torch.tensor(qs, device="cuda").view(1, L, 1).expand_as(d)
        agree = bool(((d == 0) | (d == 1) | (d == qv - 1)).all())
        exact_frac = float((d == 0).double().mean())
    gbps = batch * N * (8 + 4 * L) / (ms * 1e-3) / 1e9
    emit(out, info, hbm, op="encode", N=N, L=L, batch=batch, ms=ms, algorithmic_GBps=gbps,
         launches=1 if logn <= 14 else 2, torch_ms=base_ms, speedup_vs_torch=base_ms / ms,
         torch_agrees_within_one=agree, torch_equal_fraction=exact_frac)


def bench_decode(logn, C, reps, hbm, info, out):
    N, n, L = 1 << logn, 1 << (logn - 1), 8
    qs = primes(L)
    batch = max(1, BULK_BYTES // (4 * C * N + 16 * n))
    gen = torch.Generator(device="cuda").manual_seed(logn * 10 + C)
    x = torch.randint(0, 1 << 30, (batch, L, N), dtype=torch.int32, device="cuda", generator=gen)
    x.remainder_(torch.tensor(qs, dtype=torch.int32, device="cuda").view(L, 1))
    z = torch.empty((batch, n), dtype=torch.complex128, device="cuda")
    with nt.CkksEncoder(ones_plan(logn, qs)) as enc:
        ms = time_ms(lambda: enc.decode(x, z, batch, SCALE, channels=C, in_stride=L * N), reps)
    gbps = batch * N * (4 * C + 8) / (ms * 1e-3) / 1e9
    emit(out, info, hbm, op="decode", N=N, channels=C, batch=batch, ms=ms, algorithmic_GBps=gbps,
         launches=1 if logn <= 14 else 2)


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
        for C in (1, 4):
            bench_decode(logn, C, args.reps, hbm, info, args.out)


if __name__ == "__main__":
    main()
