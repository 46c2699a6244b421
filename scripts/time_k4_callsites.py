"""Device-event timings of the two K4 call sites outside Engine.grid_conditionalise:
the normalisation inside dist.omc_sharded and PD.marginalise over every axis of a
log-pscale device PD.

    python scripts/time_k4_callsites.py [--trees DIR ...] [--rounds R] [--reps N]

Every tree (default: this one) is timed in a process of its own, the trees alternating
for R rounds, so that two builds of the library can be compared in one run.  Only the
public calls are timed.  The omc_sharded normalisation is the time of omc_sharded minus
the time of the same draws, log-joint and weighted sums without it (one observation, so
that the log-joint pass stays small).  10^3 and 10^6 entries are L2-resident; 2^24
entries and the 4096^2 grid (134 MB each) are not.  Prints one JSON line per tree and
round with median milliseconds per call."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OMC_SIZES = [10 ** 6, 1 << 24]
MARG_SHAPES = [(10 ** 3,), (10 ** 6,), (1 << 24,), (4096, 4096)]


def _child(reps):
    import numpy as np
    import torch
    from probayes_b200 import dist
    from probayes_b200.engine import get_engine
    import probayes_b200 as pb
    eng = get_engine(0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def t(fn):
        for _ in range(3):
            fn()
        ms = []
        for _ in range(reps):
            torch.cuda.synchronize()
            ev0.record()
            fn()
            ev1.record()
            torch.cuda.synchronize()
            ms.append(ev0.elapsed_time(ev1))
        return float(np.median(ms))

    res = {}
    lims, logu, ex = np.array([[40., 60.], [5., 20.]]), np.array([0, 1]), np.ones((2, 2), int)
    y = np.array([50.])
    for n in OMC_SIZES:
        def rest():
            th = eng.box_sample(lims, logu, n, seed=3)
            lp = eng.normreg_logjoint(th, eng.to_device(y), None, lims, ex, logu)
            eng.expectation_sums(lp, True, None, th).cpu()
        res["omc_sharded_%d" % n] = t(lambda: dist.omc_sharded(eng, y, lims, ex, logu, n, seed=3))
        res["omc_rest_%d" % n] = t(rest)
        res["omc_norm_%d" % n] = res["omc_sharded_%d" % n] - res["omc_rest_%d" % n]
    g = torch.Generator(device=eng.device).manual_seed(5)
    for shape in MARG_SHAPES:
        p = torch.randn(*shape, dtype=torch.float64, device=eng.device, generator=g) * 30 - 700
        vals = {k: np.arange(m, dtype=float) for k, m in zip("xy", shape)}
        pd = pb.PD(",".join(vals), vals, prob=p, pscale='log')
        keys = list(vals)
        res["marginalise_" + "x".join(map(str, shape))] = t(lambda: pd.marginalise(keys))
    dev = torch.cuda.get_device_properties(0).name
    return dict(device=dev, ms=res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trees", nargs="+", default=[ROOT])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        print(json.dumps(_child(a.reps)))
        return
    for r in range(a.rounds):
        for tree in a.trees:
            tree = os.path.abspath(tree)
            env = dict(os.environ, PYTHONPATH=tree)
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--child",
                                  "--reps", str(a.reps)], env=env, cwd=tree,
                                 capture_output=True, text=True)
            if out.returncode:
                sys.stderr.write(out.stderr)
                raise SystemExit(out.returncode)
            line = json.loads(out.stdout.strip().splitlines()[-1])
            print(json.dumps(dict(tree=tree, round=r, **line)), flush=True)


if __name__ == "__main__":
    main()
