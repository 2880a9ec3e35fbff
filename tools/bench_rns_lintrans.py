"""Plaintext matrix-vector products on one B200: one nttb200_rns_lintrans_apply call against the
composed sequence of existing calls that a caller would otherwise write (keyswitch_apply hoisted over
the babies, automorphism(EVAL) of c0 and ADD, automorphism(EVAL) of each diagonal, MUL / ADD per
term, one keyswitch_apply per giant, automorphism of W_i.c0 and the adds; the reference of
tests/test_rns_lintrans.py), timed alternately in the same run with outputs compared word for word.
N = 2^16, (L, K, alpha) = (24, 8, 8), the sizes of a bootstrapping-scale ciphertext; 16 banded
(offsets -8..7), 64 and 256 consecutive diagonals with n1 = 8, 8 and 16, at batch 1 and 8.  The
diagonals alone are 100 MiB to 1.6 GiB, so most shapes run beyond the 126 MB L2.  Writes one JSON line
per row to --out (default profiles/r11_bench_lintrans.jsonl).

    python tools/bench_rns_lintrans.py [--out PATH] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import ntt_aie_b200 as nt  # noqa: E402
from test_rns_eval import rand_rns  # noqa: E402
from test_rns_keyswitch import Env  # noqa: E402
from test_rns_lintrans import composed, launches, schedule  # noqa: E402

LOGN, L, K, ALPHA = 16, 24, 8, 8


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:
        pl = "unknown"
    return name, pl


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def kernel_ms(fn, names, reps):
    """mean device time per call of the kernels whose names contain one of `names`"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    tot = {}
    for ev in prof.key_averages():
        for nm in names:
            if nm in ev.key:
                tot[nm] = tot.get(nm, 0.0) + ev.device_time_total / 1000.0 / reps
    return tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_bench_lintrans.jsonl"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    name, plim = card()
    env = Env(nt, LOGN, L, K, ALPHA)
    n, LK, dn, half = env.n, L + K, env.ks.dnum, env.n // 2
    shapes = [("banded16", [k % half for k in range(-8, 8)], 8), ("dense64", list(range(64)), 8),
              ("dense256", list(range(256)), 16)]
    rows = []
    for label, offs, n1 in shapes:
        gal = nt.lintrans_galois(n, offs, n1)
        babies, giants, terms = schedule(offs, n1)
        diags = rand_rns((len(offs), L, n), env.qs[:L], 3000 + len(offs))
        keys = rand_rns((len(gal), dn, 2, LK, n), env.qs, 4000 + len(offs))
        for batch in (1, 8):
            ct = rand_rns((batch, 2, L, n), env.qs[:L], 5000 + batch)
            out = torch.empty((batch, 2, L, n), dtype=torch.int32, device="cuda")
            res = {}
            one = lambda: env.ks.linear_transform(ct, diags, offs, n1, keys, out, batch)
            many = lambda: res.__setitem__("y", composed(env, ct, diags, offs, n1, keys, batch))
            one(), many()
            torch.cuda.synchronize()
            l0 = nt.kernel_launches()
            one()
            l1 = nt.kernel_launches()
            many()
            l2 = nt.kernel_launches()
            assert l1 - l0 == launches(LOGN, dn, offs, n1)
            assert torch.equal(out, res["y"]), (label, batch)
            t1, t2 = [], []
            for _ in range(args.reps):
                t1.append(timed(one))
                t2.append(timed(many))
            k1 = kernel_ms(one, ["rns_lt_kernel", "rns_ks_dot_kernel"], 3)
            nb, ng, nw = len(babies), len(giants), len(terms)
            ctw = 2 * L * n
            scratch = 4 * ((nb + (nw if ng else 0) + ng) * batch * ctw) + 16 * (2 * nw + len(offs) + 1)
            row = dict(card=name, power_limit=plim, logn=LOGN, L=L, K=K, alpha=ALPHA, dnum=dn, shape=label,
                       diagonals=len(offs), n1=n1, babies=nb, giants=ng, batch=batch,
                       one_call_ms=float(np.median(t1)), composed_ms=float(np.median(t2)),
                       speedup=float(np.median(t2) / np.median(t1)), one_call_launches=l1 - l0,
                       composed_launches=l2 - l1, one_call_scratch_bytes=scratch,
                       lt_kernels_ms=k1.get("rns_lt_kernel", float("nan")),
                       ks_dot_kernels_ms=k1.get("rns_ks_dot_kernel", float("nan")), outputs_equal=True)
            print(json.dumps(row), flush=True)
            rows.append(row)
            del ct, out, res
            torch.cuda.empty_cache()
        del diags, keys
    env.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
