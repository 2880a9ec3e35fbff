"""Device time of nttb200_polymul_negacyclic per N (one line each)."""
import json, os, sys, statistics
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import ntt_aie_b200 as nt
Q = 469762049
peak = 6539.5
for logn in [int(x) for x in (sys.argv[1] if len(sys.argv) > 1 else "12").split(",")]:
    n = 1 << logn
    batch = (1 << 26) // n
    fwd, inv = nt.negacyclic_tables(n, Q, 3)
    a = torch.randint(0, Q, (batch, n), dtype=torch.int32, device="cuda")
    b = torch.randint(0, Q, (batch, n), dtype=torch.int32, device="cuda")
    c = torch.empty_like(a)
    with nt.Plan(logn, Q, fwd) as pf, nt.Plan(logn, Q, inv) as pi:
        for _ in range(3):
            nt.polymul_negacyclic(pf, pi, a, b, c, batch)
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(21)]
        ev[0].record()
        for k in range(20):
            nt.polymul_negacyclic(pf, pi, a, b, c, batch)
            ev[k + 1].record()
        torch.cuda.synchronize()
        ms = sorted(ev[k].elapsed_time(ev[k + 1]) for k in range(20))
        t = statistics.mean(ms[1:-1])
        print(json.dumps({"logn": logn, "ms": t, "frac": batch * n * 12 / (t * 1e-3) / 1e9 / peak,
                          "path": pi.last_path}), flush=True)
