"""Dev tool: run the native head twice on the same inputs and report which workspace intermediates differ."""
import os, sys, torch, numpy as np
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', '..'))
from oracle import tpspp_oracle as O
import tps_pp_b200 as T
from tps_pp_b200 import _native as N, functional as TF
DEV = 'cuda:0'
B = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
sd = O.trained_like_state(3)
m = T.TPS_PP().to(DEV).eval(); m.load_state_dict(sd, strict=True)
g = torch.Generator(device=DEV).manual_seed(5)
x = torch.randn((B, 64, 16, 64), device=DEV, generator=g)
o0 = torch.randn((B, 32, 32, 128), device=DEV, generator=g)
o1 = torch.randn((B, 32, 32, 128), device=DEV, generator=g)
cfg = TF.head_cfg(B, 16, 64, (2, 16), 2, N.HEAD_TC)
offs = TF.head_workspace_offsets(cfg)
names = sorted(offs, key=lambda k: offs[k])
runs = []
for r in range(3):
    fg, cp, sc, ws = TF.head_forward(x, o0, o1, list(m.parameters()), (2, 16), 2, N.HEAD_TC, None)
    torch.cuda.synchronize()
    runs.append((fg.clone(), cp.clone(), sc.clone(), ws.clone()))
for r in (1, 2):
    print('run', r, 'fg', torch.equal(runs[0][0], runs[r][0]), 'cp', torch.equal(runs[0][1], runs[r][1]), 'sc', torch.equal(runs[0][2], runs[r][2]))
    a, b = runs[0][3], runs[r][3]
    for i, nm in enumerate(names):
        lo = offs[nm]; hi = offs[names[i + 1]] if i + 1 < len(names) else a.numel()
        if hi <= lo: continue
        fa = a[lo:hi].view(torch.float32); fb = b[lo:hi].view(torch.float32)
        ne = (fa != fb) & ~(torch.isnan(fa) & torch.isnan(fb))
        if ne.any():
            idx = torch.nonzero(ne)[:, 0]
            print('   differs:', nm, 'count', int(ne.sum()), 'of', fa.numel(), 'first idx', int(idx[0]), 'last', int(idx[-1]), 'maxdiff', float((fa - fb)[ne].abs().max()))
