"""K2 with and without a covariance-matrix transition (set_tran(covariance)) on one GPU.

    python scripts/time_normreg_cov_tran.py [--baseline-lib OLD/libpbx.so] [--reps 7] [--quick]

(a) with --baseline-lib (a libpbx.so built from another commit): the uncoloured kernels of
    both libraries on the same inputs, alternated rep by rep -- C3 MH step (16384 chains,
    N = 1e6, tiles), the N = 2^27 4-chain streaming step, the one-launch walk (64 chains,
    N = 1000, 2000 steps) and the sufficient-statistics walk (16384 chains, 1000 steps);
(b) the coloured proposal against the uncoloured one on every walk path;
(c) mixing on y = -1 + 1.5 x + N(0, 0.5^2), x ~ N(5, 1), N = 1e5 (corr(b0, b1) ~ -0.98):
    effective samples per second of b0 and b1 for a single uniform [delta] tuned to ~25 %
    acceptance, against a normal proposal coloured by 2.38^2 / 3 times the covariance of a
    pilot run (batch-means ESS summed over chains, over the kernel time of the walk).
Kernel times are CUDA events around each call's launches (Engine.last_kernel_ms).  Prints the
card's name and power limit first; every result is one JSON line."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from probayes_b200 import _lib  # noqa: E402
from probayes_b200.engine import Engine, get_engine  # noqa: E402

LIMS = np.array([[-6., 6.], [-6., 6.], [0.001, 10.]])
EX = np.array([[0, 0], [0, 0], [1, 0]])
LG = np.zeros(3, int)
L_TEST = np.linalg.cholesky(np.array([[1., -.6, .3], [-.6, 1., -.4], [.3, -.4, 1.]]))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "nvidia-smi unavailable"


def engine_on(path, eng):
    """An Engine on ``eng``'s device and stream whose calls go to the library at ``path``."""
    lib = C.CDLL(os.path.abspath(path))
    for name, (res, args) in _lib.SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    other = Engine.__new__(Engine)
    other.lib, other.device_index, other.device, other.stream, other.info = \
        lib, eng.device_index, eng.device, eng.stream, eng.info
    h = C.c_void_p()
    _lib.check(lib.pbx_ctx_create(eng.device_index, C.c_void_p(eng.stream.cuda_stream), 0,
                                  C.byref(h)), "pbx_ctx_create")
    other.ctx = h
    return other


def workloads(eng, quick):
    """The timed walks (name -> chains, data, steps per call, delta, variant, divisor of the
    call's time) and a builder of their start states."""
    import torch
    rng = np.random.default_rng(2024)
    N = 100_000 if quick else 1_000_000
    x = eng.to_device(rng.normal(0, 1, N))
    y = eng.to_device(-1 + 1.5 * x.cpu().numpy() + rng.normal(0, .5, N))
    Ns = (1 << 22) if quick else (1 << 27)
    xs = torch.randn(Ns, dtype=torch.float64, device=eng.device)
    ys = -1 + 1.5 * xs + 0.5 * torch.randn(Ns, dtype=torch.float64, device=eng.device)
    xm, ym = x[:1000].contiguous(), y[:1000].contiguous()

    def state(C_):
        return eng.to_device(np.tile(np.array([[-1.], [1.5], [.5]]), (1, C_)))

    sd, sds, sdm = 0.5 / np.sqrt(N), 0.5 / np.sqrt(Ns), 0.5 / np.sqrt(1000)
    return {
        "c3_tiles_step": dict(C=16384, y=y, x=x, T=10, scale=2.4 * sd, variant=0, steps=10),
        "stream_c4_step": dict(C=4, y=ys, x=xs, T=6, scale=2.4 * sds, variant=2, steps=6),
        "small_walk_c64": dict(C=64, y=ym, x=xm, T=2000, scale=2.4 * sdm, variant=0, steps=1),
        "suffstat_walk": dict(C=16384, y=y, x=x, T=1000, scale=2.4 * sd, variant=3, steps=1),
    }, state


def time_call(e, w, state, chol=None, prop="uniform"):
    st = state(w["C"])
    e.mh_normreg(st, w["y"], w["x"], 2, LIMS, EX, LG, [w["scale"]] * 3, seed=1,
                 variant=w["variant"], record=False, prop=prop, prop_chol=chol)
    e.sync()

    def run():
        e.mh_normreg(st, w["y"], w["x"], w["T"], LIMS, EX, LG, [w["scale"]] * 3, seed=1,
                     variant=w["variant"], record=True, prop=prop, prop_chol=chol)
        return e.last_kernel_ms() / w["steps"]
    return run


def spread(v):
    v = np.asarray(v)
    return dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()), n=len(v))


def ab(eng, base, ws, state, reps):
    res = {}
    for name, w in ws.items():
        fns = {"parent": time_call(base, w, state), "this": time_call(eng, w, state)}
        for f in fns.values():
            f()
        t = {k: [] for k in fns}
        for _ in range(reps):
            for k, f in fns.items():
                t[k].append(f())
        res[name] = {k: spread(v) for k, v in t.items()}
        print(json.dumps(dict(section="a_parent_vs_this_uncoloured", workload=name,
                              unit="ms per step" if w["steps"] > 1 else "ms per walk",
                              **res[name])), flush=True)
    return res


def coloured_cost(eng, ws, state, reps):
    for name, w in ws.items():
        fns = {"uncoloured": time_call(eng, w, state),
               "coloured": time_call(eng, w, state, chol=L_TEST)}
        for f in fns.values():
            f()
        t = {k: [] for k in fns}
        for _ in range(reps):
            for k, f in fns.items():
                t[k].append(f())
        print(json.dumps(dict(section="b_coloured_vs_uncoloured", workload=name,
                              unit="ms per step" if w["steps"] > 1 else "ms per walk",
                              ratio=float(np.median(t["coloured"]) / np.median(t["uncoloured"])),
                              **{k: spread(v) for k, v in t.items()})), flush=True)


def ess_batch_means(x):
    """x [n, C]: batch-means effective sample size, summed over the chains."""
    n = x.shape[0]
    b = int(np.sqrt(n))
    m = n // b
    xb = x[:m * b].reshape(m, b, -1).mean(axis=1)
    var, var_b = x.var(axis=0, ddof=1), xb.var(axis=0, ddof=1)
    return float(np.sum(n * var / (b * var_b)))


def mixing(eng, quick):
    rng = np.random.default_rng(7)
    N, Cn = 100_000, 128
    T = 1000 if quick else 6000
    xo = rng.normal(5., 1., N)
    yo = rng.normal(-1. + 1.5 * xo, 0.5)
    X = np.stack([np.ones(N), xo], 1)
    b_ols = np.linalg.lstsq(X, yo, rcond=None)[0]
    s2 = float(np.mean((yo - X @ b_ols) ** 2))
    post = np.zeros((3, 3))
    post[:2, :2] = s2 * np.linalg.inv(X.T @ X)
    post[2, 2] = s2 / (2 * N)
    init = rng.multivariate_normal([b_ols[0], b_ols[1], np.sqrt(s2)], post, Cn).T
    yd, xd = eng.to_device(yo), eng.to_device(xo)
    burn = T // 5

    def walk(steps, **kw):
        st = eng.to_device(init)
        out = eng.mh_normreg(st, yd, xd, steps, LIMS, EX, LG, seed=3, **kw)
        ms = eng.last_kernel_ms()
        return out["x"].cpu().numpy(), ms, out["accept_count"].cpu().numpy().sum() / (Cn * steps)

    lo, hi = 1e-5, 1e-1                       # [delta] (every parameter) for ~25 % acceptance
    for _ in range(14):
        d = np.sqrt(lo * hi)
        rate = walk(400, prop_scale=[d] * 3, prop="uniform")[2]
        lo, hi = (d, hi) if rate > 0.25 else (lo, d)
    d = np.sqrt(lo * hi)
    res = {}
    xs, ms, rate = walk(T, prop_scale=[d] * 3, prop="uniform")
    res["uncoloured_delta"] = (xs, ms, rate, dict(delta=d))
    pilot = xs[burn:].transpose(0, 2, 1).reshape(-1, 3)
    Lp = np.linalg.cholesky(2.38 ** 2 / 3 * np.cov(pilot.T))
    xs, ms, rate = walk(T, prop_scale=[1.] * 3, prop="normal", prop_chol=Lp)
    res["coloured_pilot_cov"] = (xs, ms, rate, dict(pilot="covariance of the uncoloured run"))
    for k, (xs, ms, rate, extra) in res.items():
        ess = [ess_batch_means(xs[burn:, j, :]) for j in range(2)]
        print(json.dumps(dict(section="c_mixing_x_N5_1", proposal=k, N=N, chains=Cn, steps=T,
                              kept_steps=T - burn, accept_rate=float(rate), walk_ms=ms,
                              ess_b0=ess[0], ess_b1=ess[1],
                              ess_per_s_b0=ess[0] / (ms * 1e-3 * (T - burn) / T),
                              ess_per_s_b1=ess[1] / (ms * 1e-3 * (T - burn) / T), **extra)),
              flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", help="libpbx.so of the commit to compare against")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--quick", action="store_true", help="small sizes (a smoke run)")
    args = ap.parse_args()
    import torch
    eng = get_engine(0)
    print(json.dumps(dict(card=card(), torch_name=torch.cuda.get_device_name(0))), flush=True)
    ws, state = workloads(eng, args.quick)
    if args.baseline_lib:
        ab(eng, engine_on(args.baseline_lib, eng), ws, state, args.reps)
    else:
        print(json.dumps(dict(section="a_parent_vs_this_uncoloured",
                              result="not measured: no --baseline-lib")))
    coloured_cost(eng, ws, state, args.reps)
    mixing(eng, args.quick)


if __name__ == "__main__":
    main()
