#!/usr/bin/env python
"""Galois automorphisms on RNS batches (nttb200_rns_automorphism), both domains.

    python tools/bench_rns_automorph.py [--reps 20]

One JSON line per measurement on stdout:
  bulk     L = 8 primes below 2^30, 2^28 coefficients per input (1 GiB, far above the 126 MB L2),
           N = 4096 and 2^16, count 1 and 8 (hoisted: count outputs from one read of the input).
           Algorithmic bytes 4 words (1 + count); fractions are of the HBM copy bandwidth
           measured in the same run.  Next to each row the torch baseline on the same
           [batch * L][N] view: index_select along N with a precomputed index (and a torch.where
           negation in the coefficient domain), run count times.
  forms    the coefficient-domain design decision, at every N, count 1 and 8, timed alternately,
           outputs compared word for word: the library kernel (the row staged in one CTA's shared
           memory for N <= 2^13, every word gathered from L2 above) next to the form it does not
           use there (profiles/microbench/automorph_coeff_forms.cu, compiled with nvcc into a
           temporary directory): the L2 gather for N <= 2^13, and for N >= 2^14 the row staged
           across a cluster of N / 2^13 CTAs and gathered through distributed shared memory.
  latency  one ciphertext, L = 32, batch 2 (L2-resident), count 1, both domains, and the baseline.
Every line carries the GPU name and power limit read in the same run and a sampled
bit-exactness check against numpy.  CUDA events, 3 warm-ups, trimmed mean (min and max dropped)."""
import argparse
import ctypes
import json
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
from tools.bench_rns import gpu_info, hbm_copy_gbps, primes, time_ms  # noqa: E402

COEFF, EVAL = nt.AUTO_COEFF, nt.AUTO_EVAL
DOMAIN = {COEFF: "coeff", EVAL: "eval"}


def rand_rns(shape, qs, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randint(0, 1 << 30, shape, dtype=torch.int32, device="cuda", generator=gen)
    return x.remainder_(torch.tensor(qs, dtype=torch.int32, device="cuda").view(len(qs), 1))


def brev(x, bits):
    out = np.zeros_like(x)
    for b in range(bits):
        out |= ((x >> b) & 1) << (bits - 1 - b)
    return out


def index_of(n, g, domain):
    """(source index, negate mask or None) of every output word"""
    j = np.arange(n, dtype=np.int64)
    if domain == EVAL:
        logn = n.bit_length() - 1
        return brev((g * brev(j, logn) + (g - 1) // 2) % n, logn), None
    e = j * pow(g, -1, 2 * n) % (2 * n)
    return e % n, e >= n


def reference(x, n, g, domain, q):
    """x: uint64 [rows, L, N], q: uint64 column [L, 1]"""
    src, neg = index_of(n, g, domain)
    y = x[..., src]
    return y if neg is None else np.where(neg, (q - y) % q, y)


def baseline(x, out, batch, limbs, n, gs, domain, qs):
    """the torch route a user had: index_select along N (+ a torch.where negation), per element"""
    idx = [index_of(n, g, domain) for g in gs]
    src = [torch.from_numpy(s).cuda() for s, _ in idx]
    neg = [None if m is None else torch.from_numpy(m).cuda() for _, m in idx]
    x2 = x.view(batch * limbs, n)
    qcol = torch.tensor(qs, dtype=torch.int32, device="cuda").repeat(batch).view(batch * limbs, 1)
    o2 = out.view(len(gs), batch * limbs, n)

    def run():
        for c in range(len(gs)):
            if neg[c] is None:
                torch.index_select(x2, 1, src[c], out=o2[c])
            else:
                y = torch.index_select(x2, 1, src[c])
                torch.where(neg[c], (qcol - y) % qcol, y, out=o2[c])
    return run


def ones_plan(logn, qs):
    return nt.RnsPlan(qs, [np.ones(1 << logn, dtype=np.int32) for _ in qs], logn=logn)


def element_list(n, count):
    """count 1: rotation by one slot; count > 1: rotations by 1 .. count - 1 slots and conjugation
    (a reversal of the row in the coefficient domain, so it is never timed alone)"""
    rot = [nt.galois_rotation(n, r + 1) for r in range(max(count - 1, 1))]
    return rot if count == 1 else rot + [nt.galois_conjugate(n)]


def emit(info, hbm, **kw):
    if "algorithmic_GBps" in kw and hbm:
        kw["frac_of_measured_hbm"] = kw["algorithmic_GBps"] / hbm
        kw["hbm_copy_GBps"] = hbm
    print(json.dumps({**kw, **info}), flush=True)


def sampled_ok(out, x, rows, n, gs, domain, qs):
    q = np.array(qs, dtype=np.uint64)[:, None]
    hx = x[rows].cpu().numpy().astype(np.uint64)
    got = out[:, rows].cpu().numpy().astype(np.uint64)
    return all(np.array_equal(got[c], reference(hx, n, g, domain, q)) for c, g in enumerate(gs))


def bulk(logn, reps, hbm, info):
    n, limbs = 1 << logn, 8
    batch = (1 << 28) // (limbs * n)
    qs = primes(limbs)
    x = rand_rns((batch, limbs, n), qs, 7000 + logn)
    rows = [0, batch // 2, batch - 1]
    words = batch * limbs * n
    with ones_plan(logn, qs) as rp:
        for count in (1, 8):
            gs = element_list(n, count)
            out = torch.empty((count, batch, limbs, n), dtype=torch.int32, device="cuda")
            for domain in (EVAL, COEFF):
                ms = time_ms(lambda: rp.automorphism(x, out, batch, gs, domain), reps)
                ok = sampled_ok(out, x, rows, n, gs, domain, qs)
                out.fill_(-1)
                base = baseline(x, out, batch, limbs, n, gs, domain, qs)
                ms_base = time_ms(base, reps)
                ok_base = sampled_ok(out, x, rows, n, gs, domain, qs)
                nbytes = 4 * words * (1 + count)
                emit(info, hbm, workload="bulk", domain=DOMAIN[domain], logn=logn, limbs=limbs, batch=batch,
                     count=count, ms=ms, algorithmic_GBps=nbytes / (ms * 1e-3) / 1e9, bit_exact_sampled=ok,
                     ms_torch_index_select=ms_base, speedup_vs_torch=ms_base / ms, torch_bit_exact_sampled=ok_base)
            del out
    del x


def build_forms(tmp):
    nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    src = os.path.join(ROOT, "profiles", "microbench", "automorph_coeff_forms.cu")
    so = os.path.join(tmp, "automorph_coeff_forms.so")
    subprocess.run([nvcc, "-O3", "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a",
                    "-o", so, src], check=True)
    lib = ctypes.CDLL(so)
    u32p = ctypes.POINTER(ctypes.c_uint32)
    for fn in (lib.auto_coeff_cluster, lib.auto_coeff_l2):
        fn.restype = ctypes.c_int
        fn.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32,
                       u32p, u32p, ctypes.c_uint32, ctypes.c_int]
    return lib


def coeff_forms(forms, logn, reps, hbm, info):
    """the library's coefficient-domain kernel next to the forms it does not use at this N"""
    n, limbs = 1 << logn, 8
    batch = (1 << 28) // (limbs * n)
    qs = primes(limbs)
    x = rand_rns((batch, limbs, n), qs, 8000 + logn)
    words = batch * limbs * n
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rows = [0, batch // 2, batch - 1]
    library_form = "one-CTA shared-memory staging" if logn <= 13 else "l2_gather"
    alts = {"l2_gather": forms.auto_coeff_l2} if logn <= 13 else {"cluster_dsmem": forms.auto_coeff_cluster}
    with ones_plan(logn, qs) as rp:
        for count in (1, 8):
            gs = element_list(n, count)
            garr = (ctypes.c_uint32 * count)(*gs)
            qarr = (ctypes.c_uint32 * limbs)(*qs)
            a = torch.empty((count, batch, limbs, n), dtype=torch.int32, device="cuda")
            b = torch.full_like(a, -1)

            def alt_call(fn):
                rc = fn(x.data_ptr(), b.data_ptr(), batch * limbs, logn, limbs, qarr, garr, count, sms)
                if rc:
                    raise RuntimeError(f"microbench: CUDA error {rc}")

            calls = {"library": lambda: rp.automorphism(x, a, batch, gs, COEFF)}
            for name, fn in alts.items():
                calls[name] = (lambda f=fn: alt_call(f))
            ms = {name: [] for name in calls}
            for _ in range(3):   # alternate, three rounds each
                for name, fn in calls.items():
                    ms[name].append(time_ms(fn, reps))
            same = bool(torch.equal(a, b))
            ok = sampled_ok(a, x, rows, n, gs, COEFF, qs)
            nbytes = 4 * words * (1 + count)
            for name in calls:
                t = float(np.median(ms[name]))
                emit(info, hbm, workload="coefficient-domain forms", form=name,
                     library_form=library_form, domain="coeff", logn=logn, limbs=limbs, batch=batch, count=count,
                     ms=t, ms_rounds=ms[name], algorithmic_GBps=nbytes / (t * 1e-3) / 1e9, bit_exact_sampled=ok,
                     outputs_identical=same)
            del a, b
    del x


def latency(logn, reps, info):
    n, limbs, batch = 1 << logn, 32, 2
    qs = primes(limbs)
    x = rand_rns((batch, limbs, n), qs, 9000 + logn)
    out = torch.empty_like(x)
    g = nt.galois_rotation(n, 1)
    with ones_plan(logn, qs) as rp:
        for domain in (EVAL, COEFF):
            ms = time_ms(lambda: rp.automorphism(x, out, batch, g, domain), reps)
            ok = sampled_ok(out.view(1, batch, limbs, n), x, [0, 1], n, [g], domain, qs)
            ms_base = time_ms(baseline(x, out, batch, limbs, n, [g], domain, qs), reps)
            emit(info, 0, workload="one ciphertext (L2-resident latency, not a roofline figure)",
                 domain=DOMAIN[domain], logn=logn, limbs=limbs, batch=batch, count=1, ms=ms,
                 ms_torch_index_select=ms_base, speedup_vs_torch=ms_base / ms, bit_exact_sampled=ok)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--logns", default="12,13,14,15,16")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rns_automorph.py needs a CUDA device; nothing was measured")
    torch.cuda.set_device(0)
    info = gpu_info()
    hbm = hbm_copy_gbps(args.reps)
    print(json.dumps({"hbm_copy_GBps": hbm, "bytes": 2 << 30, **info}), flush=True)
    logns = [int(v) for v in args.logns.split(",")]
    for logn in (12, 16):
        if logn in logns:
            bulk(logn, args.reps, hbm, info)
    with tempfile.TemporaryDirectory() as tmp:
        forms = build_forms(tmp)
        for logn in logns:
            coeff_forms(forms, logn, args.reps, hbm, info)
    for logn in logns:
        latency(logn, args.reps, info)


if __name__ == "__main__":
    main()
