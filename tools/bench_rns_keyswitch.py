"""Hybrid key switching on one B200: one nttb200_rns_keyswitch_apply call against the composed
sequence of existing calls (rns_gs_scaled, base_convert into the digit rows, rns_ct,
automorphism(EVAL) of the digits, rns_dot for b and a, rns_gs_scaled, mod_down(ROUND), rns_ct),
timed alternately in the same run with outputs compared word for word; and the fused kernel alone
(torch.profiler) against the automorphism + 2 x rns_dot it replaces, as a fraction of the copy
bandwidth measured in the same run.  N = 2^16, (L, K, alpha) = (24, 8, 8); batch 1 (the working
set of a count-1 call, about 100 MiB, is L2-resident) and batch 16 (digits alone 384 MiB, beyond
the 126 MB L2).  Writes one JSON line per row to --out (default profiles/r10_bench_keyswitch.jsonl).

    python tools/bench_rns_keyswitch.py [--out PATH] [--reps 20]
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
from test_rns_eval import channel_tables, ones_plan, rand_rns  # noqa: E402
from test_rns_sizes import channel_primes  # noqa: E402

LOGN, L, K, ALPHA = 16, 24, 8, 8


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:
        pl = "unknown"
    return name, pl


class Composed:
    def __init__(self, qs, fwd, inv):
        n = 1 << LOGN
        self.n, self.qs = n, qs
        self.qpf = nt.RnsPlan(qs, fwd, logn=LOGN)
        self.qpi = nt.RnsPlan(qs, inv, logn=LOGN)
        self.qf = nt.RnsPlan(qs[:L], fwd[:L], logn=LOGN)
        self.qi = nt.RnsPlan(qs[:L], inv[:L], logn=LOGN)
        self.dig = [(lo, min(lo + ALPHA, L)) for lo in range(0, L, ALPHA)]
        self.lo, self.hi = [], []
        for lo, hi in self.dig:
            with ones_plan(nt, LOGN, qs[lo:hi]) as a:
                if lo:
                    with ones_plan(nt, LOGN, qs[:lo]) as b:
                        self.lo.append(nt.RnsConv(a, b))
                else:
                    self.lo.append(None)
                with ones_plan(nt, LOGN, qs[hi:]) as b:
                    self.hi.append(nt.RnsConv(a, b))
        with ones_plan(nt, LOGN, qs[L:]) as a, ones_plan(nt, LOGN, qs[:L]) as b:
            self.down = nt.RnsConv(a, b)

    def run(self, x, keys_b, keys_a, gs, batch, out, buf):
        """keys_b / keys_a: [count][dnum][L+K][N] contiguous; u and out [count][2][batch][..][N] (the
        part-major order rns_dot writes)"""
        n, LK, dn, cnt = self.n, L + K, len(self.dig), len(gs)
        xc, d, rot, u = buf
        self.qi.gs_scaled(x, xc, batch)
        for i, (lo, hi) in enumerate(self.dig):
            if self.lo[i]:
                self.lo[i].convert(xc[:, lo:hi], d[i], batch, in_stride=L * n, out_stride=LK * n)
            self.hi[i].convert(xc[:, lo:hi], d[i][:, hi:], batch, in_stride=L * n, out_stride=LK * n)
            d[i][:, lo:hi].copy_(xc[:, lo:hi])
        self.qpf.ct(d, d, dn * batch)
        self.qpf.automorphism(d, rot, dn * batch, gs)
        for c in range(cnt):
            nt.rns_dot(self.qpf, rot[c], keys_b[c], u[c, 0], dn, batch, w_batch=1)
            nt.rns_dot(self.qpf, rot[c], keys_a[c], u[c, 1], dn, batch, w_batch=1)
        self.qpi.gs_scaled(u, u, cnt * batch * 2)
        self.down.mod_down(u, out, cnt * batch * 2, round=True)
        self.qf.ct(out, out, cnt * batch * 2)


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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_bench_keyswitch.jsonl"))
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    name, plim = card()
    n, LK = 1 << LOGN, L + K
    qs = channel_primes(LK)
    fwd, inv, _ = channel_tables(nt, n, qs)
    comp = Composed(qs, fwd, inv)
    rows = []
    # copy bandwidth of this run: 1 GiB device-to-device
    src = torch.empty(1 << 28, dtype=torch.int32, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    copy_ms = min(timed(lambda: dst.copy_(src)) for _ in range(10))
    copy_bw = 2 * src.numel() * 4 / copy_ms / 1e6   # GB/s
    del src, dst
    with nt.RnsPlan(qs, fwd, logn=LOGN) as pf, nt.RnsPlan(qs, inv, logn=LOGN) as pi:
        ks = nt.KeySwitcher(pf, pi, L, ALPHA)
    dn = ks.dnum
    for batch in (1, 16):
        x = rand_rns((batch, L, n), qs[:L], 1000 + batch)
        for count in (1, 8, 32):
            gs = [nt.galois_rotation(n, r + 1) for r in range(count)]
            keys = rand_rns((count, dn, 2, LK, n), qs, 2000 + count)
            kb, ka = keys[:, :, 0].contiguous(), keys[:, :, 1].contiguous()
            out1 = torch.empty((count, batch, 2, L, n), dtype=torch.int32, device="cuda")
            out2 = torch.empty_like(out1)
            buf = (torch.empty((batch, L, n), dtype=torch.int32, device="cuda"),
                   torch.empty((dn, batch, LK, n), dtype=torch.int32, device="cuda"),
                   torch.empty((count, dn, batch, LK, n), dtype=torch.int32, device="cuda"),
                   torch.empty((count, 2, batch, LK, n), dtype=torch.int32, device="cuda"))
            one = lambda: ks.switch(x, keys, out1, batch, gs)
            many = lambda: comp.run(x, kb, ka, gs, batch, out2, buf)
            one(), many()
            torch.cuda.synchronize()
            l0 = nt.kernel_launches()
            one()
            l1 = nt.kernel_launches()
            many()
            l2 = nt.kernel_launches()
            assert torch.equal(out1, out2.view(count, 2, batch, L, n).transpose(1, 2)), (batch, count)
            t1, t2 = [], []
            for _ in range(args.reps):
                t1.append(timed(one))
                t2.append(timed(many))
            k1 = kernel_ms(one, ["rns_ks_dot_kernel"], 5)
            k2 = kernel_ms(many, ["rns_auto_eval_kernel", "rns_dot_kernel"], 5)
            E = batch * LK * n
            fused_words = count * (dn * E + 2 * dn * LK * n + 2 * E)
            old_words = count * (dn * E / count + dn * E + 2 * (dn * E + dn * LK * n) + 2 * E)
            fused_ms = k1.get("rns_ks_dot_kernel", float("nan"))
            old_ms = sum(k2.values())
            row = dict(card=name, power_limit=plim, logn=LOGN, L=L, K=K, alpha=ALPHA, dnum=dn, batch=batch,
                       count=count, one_call_ms=float(np.median(t1)), composed_ms=float(np.median(t2)),
                       speedup=float(np.median(t2) / np.median(t1)), one_call_launches=l1 - l0,
                       composed_launches=l2 - l1,
                       one_call_scratch_bytes=4 * (dn * batch + 2 * count * batch) * LK * n,
                       composed_buffer_bytes=4 * (batch * L * n + dn * batch * LK * n + count * dn * batch * LK * n
                                                  + 2 * count * batch * LK * n),
                       fused_kernel_ms=fused_ms, fused_algorithmic_bytes=4 * fused_words,
                       fused_copy_bw_fraction=4 * fused_words / fused_ms / 1e6 / copy_bw,
                       replaced_kernels_ms=old_ms, replaced_algorithmic_bytes=4 * old_words,
                       replaced_copy_bw_fraction=4 * old_words / old_ms / 1e6 / copy_bw,
                       copy_bw_gbs=copy_bw, outputs_equal=True)
            print(json.dumps(row), flush=True)
            rows.append(row)
            del buf, keys, kb, ka, out1, out2
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
