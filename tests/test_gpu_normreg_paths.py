"""K2: every walk path against the numpy oracle, for everything a step does besides the
likelihood sum -- the ufun move, the bound rule, the accept rule, per-step outputs,
thinned records, running sums and the final write-back.

Paths (C ABI ``variant``): 1 one launch per step, chains in registers (KC = 1, 2, 4 chains
per thread, selected by the chain count); 2 the same for <= 8 chains (KS = 1, 2, 4, 8);
3 the whole walk in one launch from sufficient statistics; 4 the whole walk in one launch,
one warp per chain.  Every case also runs once without per-step outputs and without the
bound rule, which for variants 1 and 2 selects the kernels without the per-step extras.
Accept decisions identical; values within 1e-12 relative for injected streams and 1e-11
for the native Philox stream (device libm against glibc); scores within 1e-9 absolute."""
import functools
import zlib

import numpy as np
import pytest
from conftest import relerr
from gpu_util import engine, dev, tcd_to_tdc, host
from oracle import np_oracle as o
from oracle import philox

pytestmark = pytest.mark.gpu
THIN = 3
SEED = 4242
CHAIN0 = 11
RADIUS = 1.0

# (variant, C, P): C selects KC for variant 1 (>= 4096: 4, >= 2048: 2) and KS for variant 2
PATHS = {
    "tiles_kc1": (1, 37, 3), "tiles_kc2": (1, 2100, 2), "tiles_kc4": (1, 4100, 3),
    "stream_ks1": (2, 1, 2), "stream_ks2": (2, 2, 3), "stream_ks4": (2, 4, 2),
    "stream_ks8": (2, 8, 3),
    "suffstat_slope": (3, 37, 3), "suffstat": (3, 37, 2),
    "warp_slope": (4, 37, 3), "warp": (4, 37, 2),
}
# accept rule, accept_coef, stream ("inj" or the native proposal), bound, log-ufun sigma, N
CASES = {
    "reference_coef": ("reference", 0.7, "inj", False, False, 40),
    "log_logufun": ("log", 1.0, "inj", False, True, 2500),
    "bound_mixed": ("log", 1.0, "inj", True, True, 2500),
    "native_uniform": ("log", 1.0, "uniform", False, False, 2500),
    "native_normal": ("reference", 1.0, "normal", False, True, 60),
    "native_spherical": ("log", 1.0, "spherical", False, False, 2500),
}


def _problem(P, N, logufun, bound, C, rng):
    """Data, prior box, proposal scale and a dispersed start for (b0, b1, sigma) or (mu, sigma).
    With ``bound`` the box is tight around the start so that proposals reach every end; the
    first proposal, which is always accepted, stays inside it even without the bound rule."""
    x = rng.normal(0., 1., N)
    if P == 3:
        y = rng.normal(-1. + 1.5 * x, 0.5)
        lims = np.array([[-6., 6.], [-6., 6.], [0.001, 10.]])
        ex = np.array([[0, 0], [0, 0], [1, 0]])
        sd = 0.5 / np.sqrt(N)
        init = np.stack([rng.normal(-1., sd, C), rng.normal(1.5, sd, C),
                         rng.uniform(.45, .55, C)], axis=1)
        scale = np.array([2.5 * sd, 2.5 * sd, 2. * sd])
        if bound:                  # closed | open below | open above
            lims = np.array([[-1. - 3.2 * sd, -1. + 3.2 * sd], [1.5 - 3.2 * sd, 1.5 + 3.2 * sd],
                             [0.42, 0.58]])
            ex = np.array([[0, 0], [1, 0], [0, 1]])
            init[:, :2] = [-1., 1.5] + rng.uniform(-sd / 2, sd / 2, (C, 2))
    else:
        y = rng.normal(50., 10., N)
        lims = np.array([[40., 60.], [5., 20.]])
        ex = np.array([[1, 1], [0, 0]])
        sd = 10. / np.sqrt(N)
        init = np.stack([rng.uniform(50. - sd, 50. + sd, C), rng.uniform(9., 11., C)], axis=1)
        scale = np.array([2.5 * sd, 2. * sd])
        if bound:                  # open at both ends | open above
            lims = np.array([[50. - 3.2 * sd, 50. + 3.2 * sd], [8.5, 11.5]])
            ex = np.array([[1, 1], [0, 1]])
            init[:, 0] = 50. + rng.uniform(-sd / 2, sd / 2, C)
    lg = np.zeros(P, int)
    if logufun:                    # sigma moves in log space
        lg[-1] = 1
        scale[-1] = scale[-1] / 0.5 if P == 3 else scale[-1] / 10.
    return x, y, lims, ex, lg, scale, init


def _native_delta(prop, scale, radius, T, chains, P, step0=0):
    """The device's proposal deltas, restated from the Philox stream."""
    if prop == "uniform":
        return -scale + 2. * scale * philox.uniforms(SEED, T, chains, P, step0)
    if prop == "normal":
        return philox.normals(SEED, T, chains, P, step0) * scale
    d = -radius + (2. * radius) * philox.uniforms(SEED, T, chains, P, step0)
    nrm = np.sqrt(np.sum(d * d, axis=2, keepdims=True))
    return ((d * radius) / nrm) * scale


@functools.lru_cache(maxsize=None)
def _problem_and_ref(path, case, bound):
    """The inputs of one case and the oracle's trajectory for them (``bound`` applied or not)."""
    variant, C, P = PATHS[path]
    accept, coef, stream, tight, logufun, N = CASES[case]
    rng = np.random.default_rng(zlib.crc32((path + "/" + case).encode()))
    x, y, lims, ex, lg, scale, init = _problem(P, N, logufun, tight, C, rng)
    T = _steps(path)
    chains = np.arange(CHAIN0, CHAIN0 + C)
    if stream == "inj":
        delta = (rng.random((T, C, P)) * 2 - 1) * scale
        thresh = rng.random((T, C))
    else:
        delta = _native_delta(stream, scale, RADIUS, T, chains, P)
        thresh = philox.thresholds(SEED, T, chains)
    ref = o.mh_normreg_walk(init, delta, thresh, x if P == 3 else None, y, lims, ex.astype(bool),
                            lg.astype(bool), has_slope=P == 3, accept=accept, coef=coef,
                            bound=bound)
    return dict(x=x, y=y, lims=lims, ex=ex, lg=lg, scale=scale, init=init, delta=delta,
                thresh=thresh), ref


def _run(eng, path, case, per_step, bound, step0=0, n_steps=None, state=None, state_lp=None):
    """Runs steps step0 .. step0 + n_steps - 1 of a case on the device."""
    variant, C, P = PATHS[path]
    accept, coef, stream = CASES[case][:3]
    pb, _ = _problem_and_ref(path, case, False)
    n_steps = _steps(path) if n_steps is None else n_steps
    if stream == "inj":
        inj = dict(inj_delta=dev(eng, tcd_to_tdc(pb["delta"][step0:step0 + n_steps])),
                   inj_thresh=dev(eng, pb["thresh"][step0:step0 + n_steps]))
        prop = "uniform"
    else:
        inj, prop = {}, stream
    st = dev(eng, pb["init"].T) if state is None else state
    out = eng.mh_normreg(st, dev(eng, pb["y"]), dev(eng, pb["x"]) if P == 3 else None, n_steps,
                         pb["lims"], pb["ex"], pb["lg"], pb["scale"], thin=THIN, seed=SEED,
                         step0=step0, chain0=CHAIN0, accept=accept, accept_coef=coef, prop=prop,
                         variant=variant, state_lp=state_lp, per_step=per_step, stats=True,
                         prop_radius=RADIUS, prop_bound=bound, **inj)
    eng.sync()
    return out, st


def _tol(case):
    return 1e-12 if CASES[case][2] == "inj" else 1e-11


def _check(out, st, ref, tol, per_step):
    X = ref["x"]
    assert np.array_equal(host(out["accept_count"]), ref["u"].sum(axis=0))
    assert relerr(host(out["x"]), tcd_to_tdc(X[THIN - 1::THIN])) <= tol
    assert relerr(host(out["prob"]), ref["prob"][THIN - 1::THIN]) <= tol
    assert relerr(host(out["stat_sum"]), X.sum(axis=0).T) <= tol
    assert relerr(host(out["stat_sumsq"]), (X * X).sum(axis=0).T) <= tol
    assert relerr(host(st), X[-1].T) <= tol
    assert relerr(host(out["state_lp"]), ref["prob"][-1]) <= tol
    if per_step:
        assert np.array_equal(host(out["accept"]).astype(bool), ref["u"])
        s = host(out["score"])
        assert np.isnan(s[0]).all() and not np.isnan(s[1:]).any()
        assert np.abs(s[1:] - ref["s"][1:]).max() <= 1e-9
        assert relerr(host(out["xprop"]), tcd_to_tdc(ref["xprop"])) <= tol
        # a proposal outside the prior box in two coordinates sums two -huge priors to -inf:
        # those entries must match exactly, the rest within tol
        pp, want = host(out["pprop"]), ref["pprop"]
        fin = np.isfinite(want)
        assert np.array_equal(pp[~fin], want[~fin])
        assert relerr(pp[fin], want[fin]) <= tol


def _steps(path):
    # variant 4 draws 32 steps at a time: cross one such batch
    return 40 if PATHS[path][0] == 4 else 15


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("path", list(PATHS))
def test_path_matches_oracle(path, case):
    eng = engine()
    bound = CASES[case][3]
    _, ref = _problem_and_ref(path, case, bound)
    out, st = _run(eng, path, case, True, bound)
    _check(out, st, ref, _tol(case), True)
    # no per-step outputs, no bound rule
    _, plain = _problem_and_ref(path, case, False)
    if bound:                                   # the bound rule changed some proposals
        assert not np.array_equal(ref["xprop"], plain["xprop"])
    out, st = _run(eng, path, case, False, False)
    _check(out, st, plain, _tol(case), False)


@pytest.mark.parametrize("path", list(PATHS))
def test_path_resume_equals_one_call(path):
    """Native stream, nonzero chain0: two calls split at a record boundary give the records,
    per-step outputs, final state and accept counts of one call."""
    eng = engine()
    T = _steps(path)
    T1 = THIN * (T // (2 * THIN))
    one, st = _run(eng, path, "native_uniform", True, False)
    a, st2 = _run(eng, path, "native_uniform", True, False, n_steps=T1)
    b, _ = _run(eng, path, "native_uniform", True, False, step0=T1, n_steps=T - T1, state=st2,
                state_lp=a["state_lp"])
    for k in ("x", "prob", "accept", "score", "xprop", "pprop"):
        assert np.array_equal(np.concatenate([host(a[k]), host(b[k])]), host(one[k]),
                              equal_nan=True), k
    assert not np.isnan(host(b["score"])[0]).any()
    assert np.array_equal(host(st2), host(st))
    assert np.array_equal(host(b["state_lp"]), host(one["state_lp"]))
    assert np.array_equal(host(a["accept_count"]) + host(b["accept_count"]),
                          host(one["accept_count"]))
    for k in ("stat_sum", "stat_sumsq"):
        assert relerr(host(a[k]) + host(b[k]), host(one[k])) <= 1e-14
