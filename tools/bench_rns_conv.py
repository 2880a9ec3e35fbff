#!/usr/bin/env python
"""RNS basis conversion: fast base conversion (ModUp) and mod_down (rescale, ModDown).

    python tools/bench_rns_conv.py [--logns 12,16] [--reps 20]

One JSON line per measurement on stdout:
  bulk    Operands far above the 126 MB L2: 2^28 coefficients over the S + T input and output
          channels (1 GiB moved per call).  convert at (S, T) = (1, 31), (4, 28), (8, 32),
          (16, 16), (32, 8), (32, 32); mod_down with ROUND at S = 1, T = 31 (rescale) and S = 8,
          T = 24 (ModDown).  Algorithmic bytes: 4 (S + T) per column for convert, 4 (2T + S) for
          mod_down; MACs: S T per column.  Two ceilings are measured in the same run, each
          independently of the conversion kernel: the HBM copy bandwidth, and the rate of the
          32x32->64 multiply-accumulate the kernel's sums are made of (profiles/microbench/mac64.cu,
          compiled with nvcc into a temporary directory).  Each row carries its fraction of both;
          "bound" names the ceiling whose least time (bytes / copy bandwidth or MACs / MAC rate) is
          the larger.
  exact   convert_exact at every convert shape and scale_round (t = 65537) at every mod_down
          shape, each timed alternately with its fast counterpart (convert, mod_down with ROUND) at
          the same shape and batch, three rounds in one run; the row carries both times and their
          ratio.  Same byte and MAC counts as bulk.
  bfv_mul one BFV ciphertext product, N = 2^14, Q = 8 primes, P = 10 primes on a [P | Q] plan:
          the seven steps of INTEGRATION's BFV multiplication (copy into the Q rows, exact Q -> P,
          ct, tensor product, gs_scaled, scale_round, exact P -> Q), timed as one unit.
  ct1     one ciphertext, L = 32, batch 2 (L2-resident: a latency figure).  The NTT-domain rescale
          gs_scaled (L) -> mod_down(ROUND) -> ct (L - 1), and ModUp (Q = 32 primes -> P = 8
          primes, written into the P channels of a [batch][40][N] buffer) with the ModDown back.
Every line carries the GPU name and power limit read in the same run and a sampled
bit-exactness check against numpy.  CUDA events, 3 warm-ups, trimmed mean (min and max dropped)."""
import argparse
import json
import math
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ntt_aie_b200 as nt  # noqa: E402
from tools.bench_rns import gpu_info, hbm_copy_gbps, primes, tables, time_ms  # noqa: E402

CONVERT_SHAPES = [(1, 31), (4, 28), (8, 32), (16, 16), (32, 8), (32, 32)]
MOD_DOWN_SHAPES = [(1, 31), (8, 24)]


def mac_ceiling():
    """Multiply-accumulates per second of profiles/microbench/mac64.cu, built here and run once."""
    nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    src = os.path.join(ROOT, "profiles", "microbench", "mac64.cu")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "mac64")
        subprocess.run([nvcc, "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe, src], check=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    return json.loads(out.strip().splitlines()[-1])


def rand_rns(shape, qs, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randint(0, 1 << 30, shape, dtype=torch.int32, device="cuda", generator=gen)
    return x.remainder_(torch.tensor(qs, dtype=torch.int32, device="cuda").view(len(qs), 1))


def h64(x):
    return x.cpu().numpy().astype(np.uint64)


def ones_plan(logn, qs):
    return nt.RnsPlan(qs, [np.ones(1 << logn, dtype=np.int32) for _ in qs], logn=logn)


def convert_ref(x, bs, cs, h=0):
    """numpy reference of the fast conversion of x [..., S, N] (offset h added first)."""
    B = math.prod(bs)
    bc = np.array(bs, dtype=np.uint64)[:, None]
    w = np.array([pow(B // b % b, -1, b) for b in bs], dtype=np.uint64)[:, None]
    y = (x + np.array([h % b for b in bs], dtype=np.uint64)[:, None]) % bc * w % bc
    out = np.empty(x.shape[:-2] + (len(cs), x.shape[-1]), dtype=np.uint64)
    for j, c in enumerate(cs):
        acc = np.zeros(x.shape[:-2] + x.shape[-1:], dtype=np.uint64)
        for i, b in enumerate(bs):
            acc = (acc + y[..., i, :] * np.uint64(B // b % c)) % np.uint64(c)
        out[..., j, :] = acc
    return out


def mod_down_ref(x, bs, cs, rnd):
    B, t = math.prod(bs), len(cs)
    h = B // 2 if rnd else 0
    cc = np.array(cs, dtype=np.uint64)[:, None]
    s = convert_ref(x[..., t:, :], bs, cs, h)
    v = (x[..., :t, :] + np.array([h % c for c in cs], dtype=np.uint64)[:, None]) % cc
    binv = np.array([pow(B % c, -1, c) for c in cs], dtype=np.uint64)[:, None]
    return (v + cc - s) % cc * binv % cc


def bulk(logn, reps, hbm):
    """Rows without the bound yet (it needs every row's MAC rate)."""
    n, out = 1 << logn, []
    cases = [("convert", s, t) for s, t in CONVERT_SHAPES] + [("mod_down", s, t) for s, t in MOD_DOWN_SHAPES]
    for op, S, T in cases:
        qs = primes(S + T)
        bs, cs = qs[:S], qs[S:]
        words_in = (S if op == "convert" else S + T)
        batch = max(1, (1 << 28) // ((words_in + T) * n))
        x = rand_rns((batch, words_in, n), bs if op == "convert" else cs + bs, 7000 + 64 * S + T + logn)
        y = torch.empty((batch, T, n), dtype=torch.int32, device="cuda")
        rows = [0, batch // 2, batch - 1]
        with ones_plan(logn, bs) as pb, ones_plan(logn, cs) as pc, nt.RnsConv(pb, pc) as cv:
            if op == "convert":
                fn = lambda: cv.convert(x, y, batch)  # noqa: E731
            else:
                fn = lambda: cv.mod_down(x, y, batch, round=True)  # noqa: E731
            ms = time_ms(fn, reps)
        hx = h64(x[rows])
        want = convert_ref(hx, bs, cs) if op == "convert" else mod_down_ref(hx, bs, cs, True)
        ok = bool(np.array_equal(h64(y[rows]), want))
        cols = batch * n
        nbytes = 4 * cols * (words_in + T)
        out.append({"workload": "bulk", "op": op, "round": op == "mod_down", "logn": logn, "S": S, "T": T,
                    "batch": batch, "ms": ms, "algorithmic_GBps": nbytes / (ms * 1e-3) / 1e9,
                    "frac_of_measured_hbm": nbytes / (ms * 1e-3) / 1e9 / hbm, "hbm_copy_GBps": hbm,
                    "macs_per_s": S * T * cols / (ms * 1e-3), "bytes": nbytes, "macs": S * T * cols,
                    "bit_exact_sampled": ok})
        del x, y
    return out


def exact_ref(x, bs, cs):
    """numpy: the exact conversion of x [..., S, N], the fast one less rint(sum y_i / b_i) B."""
    B = math.prod(bs)
    bc = np.array(bs, dtype=np.uint64)[:, None]
    w = np.array([pow(B // b % b, -1, b) for b in bs], dtype=np.uint64)[:, None]
    v = np.rint((x % bc * w % bc / bc.astype(np.float64)).sum(axis=-2)).astype(np.uint64)
    out = convert_ref(x, bs, cs)
    for j, c in enumerate(cs):
        out[..., j, :] = (out[..., j, :] + np.uint64(c) - v * np.uint64(B % c) % np.uint64(c)) % np.uint64(c)
    return out


def scale_round_ref(x, bs, cs, t):
    """numpy: round(t X / B) mod c_j of x [..., T+S, N]: t X less the centred [t X]_B (the exact
    conversion of t x_B) is B round(t X / B), divided by B on each target prime."""
    B, T = math.prod(bs), len(cs)
    bc = np.array(bs, dtype=np.uint64)[:, None]
    s = exact_ref(x[..., T:, :] * np.array([t % b for b in bs], dtype=np.uint64)[:, None] % bc, bs, cs)
    out = np.empty(x.shape[:-2] + (T, x.shape[-1]), dtype=np.uint64)
    for j, c in enumerate(cs):
        c64 = np.uint64(c)
        out[..., j, :] = (x[..., j, :] * np.uint64(t % c) % c64 + c64 - s[..., j, :]) % c64 * \
            np.uint64(pow(B % c, -1, c)) % c64
    return out


def exact_rows(logn, reps, hbm):
    """convert_exact / scale_round rows, each alternated with its fast counterpart at the same shape."""
    n, out = 1 << logn, []
    cases = [("convert_exact", s, t) for s, t in CONVERT_SHAPES] + [("scale_round", s, t) for s, t in MOD_DOWN_SHAPES]
    for op, S, T in cases:
        qs = primes(S + T)
        bs, cs = qs[:S], qs[S:]
        words_in = (S if op == "convert_exact" else S + T)
        batch = max(1, (1 << 28) // ((words_in + T) * n))
        x = rand_rns((batch, words_in, n), bs if op == "convert_exact" else cs + bs, 7500 + 64 * S + T + logn)
        y = torch.empty((batch, T, n), dtype=torch.int32, device="cuda")
        rows = [0, batch // 2, batch - 1]
        with ones_plan(logn, bs) as pb, ones_plan(logn, cs) as pc, nt.RnsConv(pb, pc) as cv:
            if op == "convert_exact":
                fast = lambda: cv.convert(x, y, batch)  # noqa: E731
                new = lambda: cv.convert(x, y, batch, exact=True)  # noqa: E731
            else:
                fast = lambda: cv.mod_down(x, y, batch, round=True)  # noqa: E731
                new = lambda: cv.scale_round(x, y, batch, 65537)  # noqa: E731
            ms_fast, ms_new = [], []
            for _ in range(3):
                ms_fast.append(time_ms(fast, reps))
                ms_new.append(time_ms(new, reps))
            new()
        hx = h64(x[rows])
        want = exact_ref(hx, bs, cs) if op == "convert_exact" else scale_round_ref(hx, bs, cs, 65537)
        ok = bool(np.array_equal(h64(y[rows]), want))
        cols = batch * n
        nbytes = 4 * cols * (words_in + T)
        ms, msf = min(ms_new), min(ms_fast)
        out.append({"workload": "exact", "op": op, "fast_op": "convert" if op == "convert_exact" else "mod_down(ROUND)",
                    "logn": logn, "S": S, "T": T, "batch": batch, "ms": ms, "ms_fast": msf,
                    "ratio_to_fast": ms / msf, "ms_rounds": ms_new, "ms_fast_rounds": ms_fast,
                    "algorithmic_GBps": nbytes / (ms * 1e-3) / 1e9,
                    "frac_of_measured_hbm": nbytes / (ms * 1e-3) / 1e9 / hbm, "hbm_copy_GBps": hbm,
                    "macs_per_s": S * T * cols / (ms * 1e-3), "bytes": nbytes, "macs": S * T * cols,
                    "bit_exact_sampled": ok})
        del x, y
    return out


def bfv_mul(reps, info):
    """Steps 1-7 of INTEGRATION's BFV multiplication on one ciphertext pair (random residues:
    the timing does not depend on the values)."""
    logn, L, K = 14, 8, 10
    n = 1 << logn
    qs = primes(L + K)
    ps, qq = qs[L:], qs[:L]
    fwd, inv = tables(n, ps + qq)
    c = rand_rns((2, L, n), qq, 8500)
    cp = rand_rns((2, L, n), qq, 8501)
    qp = torch.empty((2, K + L, n), dtype=torch.int32, device="cuda")
    A, Bt = torch.empty_like(qp), torch.empty_like(qp)
    d = torch.empty((3, K + L, n), dtype=torch.int32, device="cuda")
    dp = torch.empty((3, K, n), dtype=torch.int32, device="cuda")
    res = torch.empty((3, L, n), dtype=torch.int32, device="cuda")
    with nt.RnsPlan(ps + qq, fwd, logn=logn) as pf, nt.RnsPlan(ps + qq, inv, logn=logn) as pi, \
            ones_plan(logn, qq) as pq, ones_plan(logn, ps) as pp, nt.RnsConv(pq, pp) as up, \
            nt.RnsConv(pp, pq) as back:
        def pipeline():
            for ev, ct in ((A, c), (Bt, cp)):
                qp[:, K:] = ct
                up.convert(qp[:, K:], qp, 2, in_stride=(K + L) * n, out_stride=(K + L) * n, exact=True)
                pf.ct(qp, ev, 2)
            pf.pointwise(nt.RNS_MUL, A[0], Bt[0], d[0], 1)
            pf.pointwise(nt.RNS_MUL, A[0], Bt[1], d[1], 1)
            nt.rns_dot(pf, A[1], Bt[0], d[1], 1, 1, accumulate=True)
            pf.pointwise(nt.RNS_MUL, A[1], Bt[1], d[2], 1)
            pi.gs_scaled(d, d, 3)
            up.scale_round(d, dp, 3, 65537)
            back.convert(dp, res, 3, exact=True)

        ms = time_ms(pipeline, reps)
        ms_scale = time_ms(lambda: up.scale_round(d, dp, 3, 65537), reps)
        ms_back = time_ms(lambda: back.convert(dp, res, 3, exact=True), reps)
    print(json.dumps({"workload": "bfv_mul (one ciphertext pair, L2-resident latency, not a roofline figure)",
                      "op": "BFV multiplication steps 1-7", "logn": logn, "limbs_q": L, "limbs_p": K, "t": 65537,
                      "ms_pipeline": ms, "ms_scale_round": ms_scale, "ms_convert_exact_p_to_q": ms_back,
                      **info}), flush=True)


def one_ciphertext(logn, reps, info):
    n, L, batch, K = 1 << logn, 32, 2, 8
    qs = primes(L + K)
    qL, ps = qs[:L], qs[L:]
    fwd, inv = tables(n, qL)
    x = rand_rns((batch, L, n), qL, 8000 + logn)
    low = torch.empty((batch, L - 1, n), dtype=torch.int32, device="cuda")
    low_ev = torch.empty_like(low)
    qp = torch.empty((batch, L + K, n), dtype=torch.int32, device="cuda")
    back = torch.empty((batch, L, n), dtype=torch.int32, device="cuda")
    ev = torch.empty_like(x)
    with nt.RnsPlan(qL, inv, logn=logn) as pi, nt.RnsPlan(qL[:-1], fwd[:-1], logn=logn) as pf1, \
            ones_plan(logn, qL[-1:]) as plast, nt.RnsConv(plast, pf1) as rescale, \
            ones_plan(logn, qL) as pq, ones_plan(logn, ps) as pp, nt.RnsConv(pq, pp) as up, \
            nt.RnsConv(pp, pq) as down:
        def pipeline():
            pi.gs_scaled(x, ev, batch)
            rescale.mod_down(ev, low, batch, round=True)
            pf1.ct(low, low_ev, batch)

        ms_pipe = time_ms(pipeline, reps)
        ms_md = time_ms(lambda: rescale.mod_down(ev, low, batch, round=True), reps)
        ok = bool(np.array_equal(h64(low), mod_down_ref(h64(ev), qL[-1:], qL[:-1], True)))
        print(json.dumps({"workload": "one ciphertext (L2-resident latency, not a roofline figure)",
                          "op": "rescale: gs_scaled -> mod_down(ROUND) -> ct", "logn": logn, "limbs": L,
                          "batch": batch, "ms_pipeline": ms_pipe, "ms_mod_down": ms_md,
                          "bit_exact_sampled": ok, **info}), flush=True)

        qp[:, :L] = x
        ms_up = time_ms(lambda: up.convert(x, qp[:, L:], batch, out_stride=(L + K) * n), reps)
        ms_down = time_ms(lambda: down.mod_down(qp, back, batch), reps)
        ms_pair = time_ms(lambda: (up.convert(x, qp[:, L:], batch, out_stride=(L + K) * n),
                                   down.mod_down(qp, back, batch)), reps)
        hqp = h64(qp)
        ok = bool(np.array_equal(hqp[:, L:], convert_ref(h64(x), qL, ps))) and \
            bool(np.array_equal(h64(back), mod_down_ref(hqp, ps, qL, False)))
        print(json.dumps({"workload": "one ciphertext (L2-resident latency, not a roofline figure)",
                          "op": "ModUp (Q 32 -> P 8) + ModDown", "logn": logn, "limbs": L, "special": K,
                          "batch": batch, "ms_mod_up": ms_up, "ms_mod_down": ms_down, "ms_pair": ms_pair,
                          "bit_exact_sampled": ok, **info}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--logns", default="12,16")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rows", default="bulk,exact,bfv_mul,ct1", help="which row groups to run")
    args = ap.parse_args()
    groups = set(args.rows.split(","))
    if not torch.cuda.is_available():
        raise SystemExit("bench_rns_conv.py needs a CUDA device; nothing was measured")
    torch.cuda.set_device(0)
    info = gpu_info()
    hbm = hbm_copy_gbps(args.reps)
    mac = mac_ceiling()
    print(json.dumps({"hbm_copy_GBps": hbm, "bytes": 2 << 30, "mac64_microbench": mac, **info}), flush=True)
    peak = mac["mac64_per_s"]
    logns = [int(v) for v in args.logns.split(",")]
    for logn in logns:
        rows = (bulk(logn, args.reps, hbm) if "bulk" in groups else []) + \
            (exact_rows(logn, args.reps, hbm) if "exact" in groups else [])
        for r in rows:
            t_hbm, t_mac = r["bytes"] / (hbm * 1e9), r["macs"] / peak
            r.update(mac_ceiling_per_s=peak, frac_of_mac_ceiling=r["macs_per_s"] / peak,
                     bound="hbm" if t_hbm >= t_mac else "integer multiplier")
            print(json.dumps({**r, **info}), flush=True)
    if "bfv_mul" in groups:
        bfv_mul(args.reps, info)
    if "ct1" in groups:
        for logn in logns:
            one_ciphertext(logn, args.reps, info)


if __name__ == "__main__":
    main()
