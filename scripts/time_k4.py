"""Per-kernel timings of the K4 passes on a 4096 x 4096 log-joint."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from probayes_b200.engine import get_engine
eng = get_engine(0)
M = S = 4096
lj = (torch.randn(M, S, dtype=torch.float64, device=eng.device) * 30 - 4e5)
def t(fn, n=5):
    for _ in range(2): fn()
    ms = []
    for _ in range(n):
        fn(); ms.append(eng.last_kernel_ms())
    return float(np.median(ms))
print("max_sumexp       %.4f ms" % t(lambda: eng.grid_max_sumexp(lj)))
ms = eng.grid_max_sumexp(lj)
print("posterior2       %.4f ms" % t(lambda: eng.grid_posterior2(lj, ms[0:1], ms[1:2])))
print("posterior2 inpl  %.4f ms" % t(lambda: eng.grid_posterior2(lj.clone(), ms[0:1], ms[1:2], inplace=True)))
print("posterior2 nopost %.4f ms" % t(lambda: eng.grid_posterior2(lj, ms[0:1], ms[1:2], want_post=False)))
ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for _ in range(3): eng.grid_conditionalise(lj)
torch.cuda.synchronize(); ev0.record()
for _ in range(10): eng.grid_conditionalise(lj)
ev1.record(); torch.cuda.synchronize()
print("conditionalise (2 passes, 3 launches + memset) %.4f ms" % (ev0.elapsed_time(ev1) / 10))
