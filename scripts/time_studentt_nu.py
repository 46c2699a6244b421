"""K2 with the sampled-nu Student-t (theta = (mu, sigma, nu), logc(nu) on the device every step)
against the fixed-nu t (df = 4, logc from the host) on one GPU.

    python scripts/time_studentt_nu.py [--reps 7]

Shapes: the tiles MH step at C3 shape (16384 chains, N = 1e6); the streaming step at N = 2^27
with 1, 4 and 8 chains; the one-launch walk with 64 chains at N = 1000 over 2000 steps, and with
1 chain at N = 60.  Both kinds run on the same (mu, sigma) data and start (nu = 4 for the sampled
kind), alternated rep by rep; medians of CUDA-event kernel times (Engine.last_kernel_ms).  The
sampled kind's per-step extra is one logc(nu) and one load of nu per chain, against C * N terms.
Prints the card's name and power limit first; one JSON line per result.
"""
import argparse
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from probayes_b200 import catalogue  # noqa: E402
from probayes_b200.engine import get_engine  # noqa: E402
import time_normreg_cov_tran  # noqa: E402

T4 = catalogue.likelihood('t', 4.)
NU = dict(family='t', df_param='nu')
LIMS = np.array([[40., 60.], [0.001, 20.], [0.5, 100.]])


def shapes():
    """name -> (chains, N, steps per call)."""
    return {"tiles_c16384_n1e6": (16384, 10 ** 6, 10),
            "stream_c1_n2e27": (1, 1 << 27, 4),
            "stream_c4_n2e27": (4, 1 << 27, 4),
            "stream_c8_n2e27": (8, 1 << 27, 4),
            "walk_c64_n1000": (64, 1000, 2000),
            "walk_c1_n60": (1, 60, 2000)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    print(json.dumps({"card": time_normreg_cov_tran.card()}), flush=True)
    eng = get_engine(0)
    rng = np.random.default_rng(0)
    for name, (C, N, T) in shapes().items():
        y = eng.to_device(50. + 0.5 * rng.standard_t(4., N))
        kinds = {"fixed_nu": (2, T4), "sampled_nu": (3, NU)}
        times = {k: [] for k in kinds}
        for rep in range(args.reps + 1):                       # rep 0 warms up
            for tag, (P, lik) in kinds.items():
                st = eng.to_device(np.tile(np.array([50., 0.5, 4.])[:P], (C, 1)).T)
                eng.mh_normreg(st, y, None, T, LIMS[:P], np.zeros((P, 2), int),
                               np.zeros(P, int), np.full(P, 1e-3), seed=rep, record=False,
                               stats=False, lik=lik)
                eng.sync()
                if rep:
                    times[tag].append(eng.last_kernel_ms() / T)
        out = {"name": name, "chains": C, "n_obs": N, "steps": T}
        for tag, v in times.items():
            ms = float(np.median(v))
            out[tag + "_ms_per_step"] = ms
            out[tag + "_spread_ms"] = [float(min(v)), float(max(v))]
            out[tag + "_terms_per_s"] = C * N / (ms * 1e-3)
        out["sampled_over_fixed"] = out["sampled_nu_ms_per_step"] / out["fixed_nu_ms_per_step"]
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
