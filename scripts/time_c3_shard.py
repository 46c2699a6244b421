"""C3 shards (N = 10^6 observations): ms per MH step for 2048 / 4096 / 8192 / 16384 chains."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from probayes_b200.engine import get_engine
eng = get_engine(0); rng = np.random.default_rng(2024)
N = 1_000_000
x = rng.normal(0, 1, N); y = rng.normal(-1 + 1.5 * x, 0.5)
xd, yd = eng.to_device(x), eng.to_device(y)
lims = np.array([[-6., 6.], [-6., 6.], [0.001, 10.]]); ex = np.array([[0, 0], [0, 0], [1, 0]]); lg = np.zeros(3, int)
sd = 0.5 / np.sqrt(N)
for C in (2048, 4096, 8192, 16384):
    st = eng.to_device(np.tile(np.array([[-1.], [1.5], [.5]]), (1, C)))
    T = 10
    ms = []
    for _ in range(4):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(eng.stream)
        eng.mh_normreg(st, yd, xd, T, lims, ex, lg, [2.4 * sd] * 3, seed=1, variant=1, record=True)
        ev1.record(eng.stream); torch.cuda.synchronize()
        ms.append(ev0.elapsed_time(ev1) / T)
    m = float(np.median(ms[1:]))
    print("C=%5d: %.4f ms per MH step, %.3e terms/s" % (C, m, C * N / (m * 1e-3)))
