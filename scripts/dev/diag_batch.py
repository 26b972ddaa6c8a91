import os, sys, torch, numpy as np
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', '..'))
from oracle import tpspp_oracle as O
import tps_pp_b200 as T
DEV='cuda:0'
sd = O.trained_like_state(3)
m = T.TPS_PP().to(DEV).eval(); m.load_state_dict(sd, strict=True)
B = 1024
g = torch.Generator(device=DEV).manual_seed(5)
x = torch.randn((B, 64, 16, 64), device=DEV, generator=g)
o0 = torch.randn((B, 32, 32, 128), device=DEV, generator=g)
o1 = torch.randn((B, 32, 32, 128), device=DEV, generator=g)
with torch.no_grad():
    full = m(x, [o0, o1]); out_full = full["output"].clone(); sc_full = full["pc_score"].clone()
    full2 = m(x, [o0, o1])
    print('rerun equal', torch.equal(full2["output"], out_full), torch.equal(full2["pc_score"], sc_full), float((full2["pc_score"]-sc_full).abs().max()))
    for lo in (0, 300, 1000):
        hi = min(B, lo + 24)
        part = m(x[lo:hi], [o0[lo:hi], o1[lo:hi]])
        d = (part["pc_score"] - sc_full[lo:hi]).abs()
        print(lo, 'out', float((part["output"] - out_full[lo:hi]).abs().max()), 'score', float(d.max()), 'nbad', int((d > 0).sum()), 'where', torch.nonzero(d > 0)[:5].tolist())
