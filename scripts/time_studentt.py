"""K2 / K3 with the Student-t likelihood against the normal one on one GPU.

    python scripts/time_studentt.py [--baseline-lib OLD/libpbx.so] [--reps 7]

Shapes: the tiles MH step at C3 shape (16384 chains, N = 1e6, (b0, b1, sigma)); the streaming
step at N = 2^27 with 1, 4 and 8 chains ((mu, sigma)); the one-launch walk (64 chains, N = 1000,
(b0, b1, sigma), 2000 steps); K3 on a 1024 x 1024 grid at N = 1e5.  For each: the t and the
normal kernels alternated rep by rep (medians), and with --baseline-lib the normal kernels of
another build too (same inputs, same alternation).  Terms are (chain or cell) x observation
evaluations; the fraction of the FP64 issue rate is FP64 instructions per term (counted in the
cuobjdump -sass of the t instantiation's inner loop, passed in INSTR_PER_TERM) x terms/s / 32
against 581.6 G warp-instructions/s.  Kernel times are CUDA events around each call's launches
(Engine.last_kernel_ms).  Prints the card's name and power limit first; one JSON line per result.
"""
import argparse
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from probayes_b200 import _lib, catalogue  # noqa: E402
from probayes_b200.engine import get_engine  # noqa: E402
import time_normreg_cov_tran  # noqa: E402

ISSUE_RATE = 581.6e9            # FP64-pipe warp-instructions / s of one B200 (148 SMs)
# FP64-pipe SASS instructions (DFMA / DMUL / DADD) per term of the t instantiations on the
# small-argument path of log1p (z^2/nu < 2/3; all instructions: ~57; the large-argument path takes
# 31 more, and lanes that disagree run both): DESIGN section 3
INSTR_PER_TERM = {"tiles": 27, "stream": 26, "walk": 27, "grid": 24}
T4 = catalogue.likelihood('t', 4.)
LIMS3 = np.array([[-6., 6.], [-6., 6.], [0.001, 10.]])
LIMS2 = np.array([[40., 60.], [0.001, 20.]])


def baseline_engine(path, eng):
    """time_normreg_cov_tran.engine_on for a library built before pbx_grid_t_logjoint: the
    signatures it does not export are left unbound (only the normal kernels are timed there)."""
    import ctypes as C
    have = C.CDLL(os.path.abspath(path))
    full = _lib.SIGNATURES
    _lib.SIGNATURES = {k: v for k, v in full.items() if hasattr(have, k)}
    try:
        return time_normreg_cov_tran.engine_on(path, eng)
    finally:
        _lib.SIGNATURES = full


def walks(eng):
    """name -> (kind, chains, P, N, steps per call)."""
    return {"tiles_c16384_n1e6": ("tiles", 16384, 3, 10 ** 6, 10),
            "stream_c1_n2e27": ("stream", 1, 2, 1 << 27, 4),
            "stream_c4_n2e27": ("stream", 4, 2, 1 << 27, 4),
            "stream_c8_n2e27": ("stream", 8, 2, 1 << 27, 4),
            "walk_c64_n1000": ("walk", 64, 3, 1000, 2000)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib")
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    print(json.dumps({"card": time_normreg_cov_tran.card()}), flush=True)
    eng = get_engine(0)
    engines = {"t": eng, "normal": eng}
    if args.baseline_lib:
        engines["normal_baseline"] = baseline_engine(args.baseline_lib, eng)
    rng = np.random.default_rng(0)
    data = {}
    for name, (kind, C, P, N, T) in walks(eng).items():
        key = (P, N)
        if key not in data:
            x = rng.normal(0., 1., N)
            y = (-1. + 1.5 * x if P == 3 else 50.) + 0.5 * rng.standard_t(4., N)
            data[key] = (eng.to_device(y), eng.to_device(x) if P == 3 else None)
        y, x = data[key]
        lims = LIMS3 if P == 3 else LIMS2
        init = np.array([-1., 1.5, 0.5]) if P == 3 else np.array([50., 0.5])
        scale = np.full(P, 1e-3)
        ex, lg = np.zeros((P, 2), int), np.zeros(P, int)
        times = {k: [] for k in engines}
        for rep in range(args.reps + 1):                       # rep 0 warms up
            for tag, e in engines.items():
                st = eng.to_device(np.tile(init, (C, 1)).T)
                e.mh_normreg(st, y, x, T, lims, ex, lg, scale, seed=rep, record=False,
                             stats=False, lik=T4 if tag == "t" else None)
                eng.sync()
                if rep:
                    times[tag].append(e.last_kernel_ms() / T)
        out = {"name": name, "chains": C, "n_obs": N}
        for tag, v in times.items():
            ms = float(np.median(v))
            out[tag + "_ms_per_step"] = ms
            out[tag + "_spread_ms"] = [float(min(v)), float(max(v))]
            out[tag + "_terms_per_s"] = C * N / (ms * 1e-3)
        out["t_fp64_issue_fraction"] = \
            INSTR_PER_TERM[kind] * out["t_terms_per_s"] / 32. / ISSUE_RATE
        out["t_hbm_TBps"] = 8. * N * (2 if P == 3 else 1) / (out["t_ms_per_step"] * 1e-3) / 1e12
        print(json.dumps(out), flush=True)
    # K3: 1024 x 1024 grid, N = 1e5
    M, N = 1024, 10 ** 5
    xo = eng.to_device(rng.normal(50., 10., N))
    mu, sg = eng.to_device(np.linspace(40., 60., M)), eng.to_device(np.linspace(5., 20., M))
    lp = eng.to_device(np.zeros(M))
    times = {k: [] for k in engines}
    for rep in range(args.reps + 1):
        for tag, e in engines.items():
            e.grid_norm_logjoint(xo, mu, sg, lp, lp, lik=T4 if tag == "t" else None)
            eng.sync()
            if rep:
                times[tag].append(e.last_kernel_ms())
    out = {"name": "grid_1024x1024_n1e5", "cells": M * M, "n_obs": N}
    for tag, v in times.items():
        ms = float(np.median(v))
        out[tag + "_ms"] = ms
        out[tag + "_spread_ms"] = [float(min(v)), float(max(v))]
        out[tag + "_terms_per_s"] = M * M * N / (ms * 1e-3)
    out["t_fp64_issue_fraction"] = \
        INSTR_PER_TERM["grid"] * out["t_terms_per_s"] / 32. / ISSUE_RATE
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
