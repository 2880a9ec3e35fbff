import os, sys, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import ntt_aie_b200 as nt
Q, n, batch = 469762049, 1 << 16, 2100
roots = nt.make_roots(n, Q, 3)
h_in = torch.randint(0, Q, (batch, n), dtype=torch.int32).pin_memory()
h_out = torch.empty_like(h_in).pin_memory()
with nt.Plan(16, Q, roots) as p:
    p.gs_host(h_in.numpy(), h_out.numpy(), batch)
    path_host = p.last_path
    d = h_in.cuda(); o = torch.empty_like(d)
    for s in range(0, batch, 100):
        e = min(batch, s + 100); p.gs(d[s:e], o[s:e], e - s)
    torch.cuda.synchronize()
    print("host path", path_host, "equal", bool(torch.equal(o.cpu(), h_out)))
