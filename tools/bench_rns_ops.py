#!/usr/bin/env python
"""Evaluation-domain operators on RNS batches: pointwise add / sub / mul (own and broadcast
operand), per-channel scale, rns_dot and the scaled inverse transform.

    python tools/bench_rns_ops.py [--logns 12,13,14,15,16] [--reps 20]

One JSON line per measurement on stdout:
  bulk    L = 8 primes below 2^30.  Streaming operators and rns_dot at N = 4096 and 2^16 with
          2^28 coefficients per operand (1 GiB, far above the 126 MB L2); algorithmic bytes:
          12 per coefficient for pointwise, 8 + the operand once for a broadcast, 8 for scale,
          4 L N (K batch + K w_batch + batch (1 + accumulate)) for rns_dot (2^26 output
          coefficients, so the K = 16 operand is 4 GiB).  Fractions are of the HBM copy
          bandwidth measured in the same run.  rns_gs_scaled next to rns_gs at every N, the two
          timed alternately.
  ct1     one ciphertext pair, L = 32, batch 2 (L2-resident: a latency figure).  rns_pointwise MUL
          next to the batch * L Plan.pointwise calls on L single-modulus plans that were the only
          way before it, and the ct, ct, mul, gs_scaled pipeline next to rns_polymul_negacyclic.
Every line carries the GPU name and power limit read in the same run and a sampled
bit-exactness check against numpy.  CUDA events, 3 warm-ups, trimmed mean (min and max dropped)."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ntt_aie_b200 as nt  # noqa: E402
from tools.bench_rns import gpu_info, hbm_copy_gbps, primes, tables, time_ms  # noqa: E402

ADD, SUB, MUL = nt.RNS_ADD, nt.RNS_SUB, nt.RNS_MUL


def rand_rns(shape, qs, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randint(0, 1 << 30, shape, dtype=torch.int32, device="cuda", generator=gen)
    return x.remainder_(torch.tensor(qs, dtype=torch.int32, device="cuda").view(len(qs), 1))


def h64(x):
    return x.cpu().numpy().astype(np.uint64)


def emit(info, hbm, **kw):
    if "algorithmic_GBps" in kw:
        kw["frac_of_measured_hbm"] = kw["algorithmic_GBps"] / hbm
        kw["hbm_copy_GBps"] = hbm
    print(json.dumps({**kw, **info}), flush=True)


def ones_plan(logn, qs):
    return nt.RnsPlan(qs, [np.ones(1 << logn, dtype=np.int32) for _ in qs], logn=logn)


def bulk_stream(logn, reps, hbm, info):
    n, limbs = 1 << logn, 8
    batch = (1 << 28) // (limbs * n)
    qs = primes(limbs)
    q = np.array(qs, dtype=np.uint64)[:, None]
    a, b = rand_rns((batch, limbs, n), qs, 3000 + logn), rand_rns((batch, limbs, n), qs, 3100 + logn)
    c = torch.empty_like(a)
    rows = [0, batch // 2, batch - 1]
    ha, hb = h64(a[rows]), h64(b[rows])
    words = batch * limbs * n
    scalars = [qv // 3 for qv in qs]
    cases = [
        ("add", lambda rp: rp.pointwise(ADD, a, b, c, batch), 12 * words, (ha + hb) % q),
        ("sub", lambda rp: rp.pointwise(SUB, a, b, c, batch), 12 * words, (ha + q - hb) % q),
        ("mul", lambda rp: rp.pointwise(MUL, a, b, c, batch), 12 * words, ha * hb % q),
        ("mul_broadcast", lambda rp: rp.pointwise(MUL, a, b[:1], c, batch, b_batch=1),
         8 * words + 4 * limbs * n, ha * hb[:1] % q),
        ("scale", lambda rp: rp.scale(a, c, batch, scalars), 8 * words,
         ha * np.array(scalars, dtype=np.uint64)[:, None] % q),
    ]
    with ones_plan(logn, qs) as rp:
        for op, fn, nbytes, want in cases:
            ms = time_ms(lambda: fn(rp), reps)
            ok = bool(np.array_equal(h64(c[rows]), want))
            emit(info, hbm, workload="bulk", op=op, logn=logn, limbs=limbs, batch=batch, ms=ms,
                 algorithmic_GBps=nbytes / (ms * 1e-3) / 1e9, bit_exact_sampled=ok)
    del a, b, c


def bulk_dot(logn, reps, hbm, info):
    n, limbs = 1 << logn, 8
    batch = (1 << 26) // (limbs * n)
    qs = primes(limbs)
    q = np.array(qs, dtype=np.uint64)[:, None]
    rows = [0, batch - 1]
    with ones_plan(logn, qs) as rp:
        for terms in (4, 16):
            a = rand_rns((terms, batch, limbs, n), qs, 4000 + terms)
            w = rand_rns((terms, batch, limbs, n), qs, 4100 + terms)
            c = rand_rns((batch, limbs, n), qs, 4200 + terms)
            ha, hw, hc = h64(a[:, rows]), h64(w[:, rows]), h64(c[rows])
            for w_batch, accumulate in ((batch, False), (1, False), (1, True)):
                wk = w if w_batch == batch else w[:, :1].contiguous()
                c0 = c.clone()
                lib_call = (lambda: nt.rns_dot(rp, a, wk, c0, terms, batch, w_batch=w_batch,
                                               accumulate=accumulate))
                # correctness from the untimed first call (accumulate changes c on every call)
                lib_call()
                hwk = hw if w_batch == batch else np.broadcast_to(hw[:, :1], hw.shape)
                acc = hc.copy() if accumulate else np.zeros_like(hc)
                for k in range(terms):
                    acc = (acc + ha[k] * hwk[k] % q) % q
                ok = bool(np.array_equal(h64(c0[rows]), acc))
                ms = time_ms(lib_call, reps)
                nbytes = 4 * limbs * n * (terms * batch + terms * w_batch + batch * (1 + accumulate))
                emit(info, hbm, workload="bulk", op="dot", logn=logn, limbs=limbs, batch=batch, terms=terms,
                     w_batch=w_batch, accumulate=accumulate, ms=ms,
                     algorithmic_GBps=nbytes / (ms * 1e-3) / 1e9, bit_exact_sampled=ok)
                del c0
            del a, w, c


def bulk_gs_scaled(logn, reps, hbm, info):
    n, limbs = 1 << logn, 8
    batch = (1 << 28) // (limbs * n)
    qs = primes(limbs)
    q = np.array(qs, dtype=np.uint64)[:, None]
    _, inv = tables(n, qs)
    a = rand_rns((batch, limbs, n), qs, 5000 + logn)
    c_gs, c_sc = torch.empty_like(a), torch.empty_like(a)
    rows = [0, batch // 2, batch - 1]
    with nt.RnsPlan(qs, inv, logn=logn) as pi:
        ms = {"gs": [], "gs_scaled": []}
        for _ in range(3):   # alternate the two, three rounds each
            ms["gs"].append(time_ms(lambda: pi.gs(a, c_gs, batch), reps))
            ms["gs_scaled"].append(time_ms(lambda: pi.gs_scaled(a, c_sc, batch), reps))
        ninv = np.array([pow(n, qv - 2, qv) for qv in qs], dtype=np.uint64)[:, None]
        ok = bool(np.array_equal(h64(c_sc[rows]), h64(c_gs[rows]) * ninv % q))
        for op in ("gs", "gs_scaled"):
            t = float(np.median(ms[op]))
            emit(info, hbm, workload="bulk", op=op, logn=logn, limbs=limbs, batch=batch, ms=t,
                 ms_rounds=ms[op], algorithmic_GBps=8 * batch * limbs * n / (t * 1e-3) / 1e9,
                 bit_exact_sampled=ok)
    del a, c_gs, c_sc


def one_ciphertext(logn, reps, info):
    n, limbs, batch = 1 << logn, 32, 2
    qs = primes(limbs)
    fwd, inv = tables(n, qs)
    q = np.array(qs, dtype=np.uint64)[:, None]
    a, b = rand_rns((batch, limbs, n), qs, 6000 + logn), rand_rns((batch, limbs, n), qs, 6100 + logn)
    c, c1 = torch.empty_like(a), torch.empty_like(a)
    ta, tb = torch.empty_like(a), torch.empty_like(a)
    singles = [nt.Plan(logn, qv, t) for qv, t in zip(qs, fwd)]
    with nt.RnsPlan(qs, fwd, logn=logn) as pf, nt.RnsPlan(qs, inv, logn=logn) as pi:
        ms = time_ms(lambda: pf.pointwise(MUL, a, b, c, batch), reps)
        ms_single = time_ms(lambda: [singles[l].pointwise(a[k, l], b[k, l], c1[k, l], n)
                                     for k in range(batch) for l in range(limbs)], reps)
        ok = bool(np.array_equal(h64(c), h64(a) * h64(b) % q)) and bool(torch.equal(c, c1))
        emit(info, 0, workload="one ciphertext (L2-resident latency, not a roofline figure)", op="mul",
             logn=logn, limbs=limbs, batch=batch, ms_one_rns_call=ms,
             ms_64_single_modulus_calls=ms_single, speedup=ms_single / ms, bit_exact_sampled=ok)

        def pipeline():
            pf.ct(a, ta, batch)
            pf.ct(b, tb, batch)
            pf.pointwise(MUL, ta, tb, ta, batch)
            pi.gs_scaled(ta, ta, batch)

        ms_pipe = time_ms(pipeline, reps)
        ms_fused = time_ms(lambda: nt.rns_polymul_negacyclic(pf, pi, a, b, c, batch), reps)
        emit(info, 0, workload="one ciphertext (L2-resident latency, not a roofline figure)",
             op="ct,ct,mul,gs_scaled vs polymul", logn=logn, limbs=limbs, batch=batch,
             ms_eval_domain_pipeline=ms_pipe, ms_rns_polymul_negacyclic=ms_fused,
             bit_exact_sampled=bool(torch.equal(ta, c)))
    for p in singles:
        p.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--logns", default="12,13,14,15,16")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rns_ops.py needs a CUDA device; nothing was measured")
    torch.cuda.set_device(0)
    info = gpu_info()
    hbm = hbm_copy_gbps(args.reps)
    print(json.dumps({"hbm_copy_GBps": hbm, "bytes": 2 << 30, **info}), flush=True)
    logns = [int(x) for x in args.logns.split(",")]
    for logn in (12, 16):
        if logn in logns:
            bulk_stream(logn, args.reps, hbm, info)
            bulk_dot(logn, args.reps, hbm, info)
    for logn in logns:
        bulk_gs_scaled(logn, args.reps, hbm, info)
    for logn in logns:
        one_ciphertext(logn, args.reps, info)


if __name__ == "__main__":
    main()
