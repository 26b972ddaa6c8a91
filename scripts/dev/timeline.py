"""Dev tool: prints the clock64 timeline written by an INSTRUMENTED build of libtpspp.so (a temporary g_tl device array +
tpspp_dbg_read export patched into conv_tma_kernel by hand; see profiles/r02_conv_experiments.md).  The last conv_tma launch
of the forward (dec3: 18 chunks per tile) is what remains in the buffer.  It does not work against the shipped library."""
import os, sys, ctypes, torch, numpy as np
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', '..'))
import tps_pp_b200 as T
from tps_pp_b200 import _native as N
DEV = 'cuda:0'
m = T.TPS_PP().to(DEV).eval()
B = 256
g = torch.Generator(device=DEV).manual_seed(5)
x = torch.randn((B, 64, 16, 64), device=DEV, generator=g); o0 = torch.randn((B, 32, 32, 128), device=DEV, generator=g); o1 = torch.randn((B, 32, 32, 128), device=DEV, generator=g)
with torch.no_grad():
    for _ in range(3): m(x, [o0, o1])
torch.cuda.synchronize()
buf = (ctypes.c_longlong * 2048)()
lib = ctypes.CDLL(N.LIB_PATH)
print('rc', lib.tpspp_dbg_read(buf))
a = np.array(buf[:]).reshape(64, 32)
t0 = a[0, 0]
print('chunk | MMA: top a_full w_full issued (probe bits) | P warp0: lds_done split_done a_empty st_issued arrived | TMA: top a_empty')
for i in range(0, 44):
    r = a[i] - t0
    print(128 + i, r[0:4].tolist(), int(a[i, 30]), '|', r[8:13].tolist(), '|', r[16:18].tolist())
