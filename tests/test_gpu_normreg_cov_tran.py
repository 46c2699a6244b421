"""K2 with a covariance-matrix transition (set_tran(covariance), rf.py:209-220,346-348): every
delta -- injected, or drawn, scaled and spherically rescaled -- is multiplied by the Cholesky
factor L before the ufun move and the bound rule.  Every walk path and case of
test_gpu_normreg_paths against the numpy oracle fed the coloured deltas, with that file's
problems, native streams and checks; resume; the public API; and the ABI's refusal of a
malformed factor."""
import functools
import zlib
import ctypes as C

import numpy as np
import pytest
import scipy.stats
from conftest import relerr
from gpu_util import engine, dev, tcd_to_tdc, host
from oracle import np_oracle as o
from oracle import philox
import probayes_b200 as pb
from probayes_b200 import _lib
import test_gpu_normreg_paths as tp

pytestmark = pytest.mark.gpu

# full (non-diagonal) factors: correlations -0.6 / 0.3 / -0.4 between the coordinates
_CORR = {3: np.array([[1., -.6, .3], [-.6, 1., -.4], [.3, -.4, 1.]]),
         2: np.array([[1., -.6], [-.6, 1.]])}
HUGE = np.finfo(float).max


def _chol(scale):
    """diag(scale) chol(R) diag(scale)^-1 (lower-triangular): a delta with spread scale_j in
    coordinate j keeps those spreads, whose units differ between the parameters, and gains
    the correlations R."""
    scale = np.asarray(scale, dtype=float)
    return np.linalg.cholesky(_CORR[len(scale)]) * scale[:, None] / scale[None, :]


def _check(out, st, ref, tol, per_step):
    """tp._check, with log-joints of -inf (a first proposal -- always accepted -- outside the
    prior box in two coordinates) required at the same places and then compared as -HUGE."""
    lp, want = host(out["prob"]), ref["prob"][tp.THIN - 1::tp.THIN]
    assert np.array_equal(np.isneginf(lp), np.isneginf(want))
    assert np.array_equal(np.isneginf(host(out["state_lp"])), np.isneginf(ref["prob"][-1]))
    out = dict(out, prob=out["prob"].nan_to_num(nan=np.nan, neginf=-HUGE),
               state_lp=out["state_lp"].nan_to_num(nan=np.nan, neginf=-HUGE))
    ref = dict(ref, prob=np.nan_to_num(ref["prob"], nan=np.nan, neginf=-HUGE))
    tp._check(out, st, ref, tol, per_step)


@functools.lru_cache(maxsize=None)
def _problem_and_ref(path, case, bound):
    """The inputs of one case (raw deltas, as the device takes them) and the oracle's
    trajectory for the coloured deltas."""
    variant, Cn, P = tp.PATHS[path]
    accept, coef, stream, tight, logufun, N = tp.CASES[case]
    rng = np.random.default_rng(zlib.crc32(("coloured/" + path + "/" + case).encode()))
    x, y, lims, ex, lg, scale, init = tp._problem(P, N, logufun, tight, Cn, rng)
    T = tp._steps(path)
    chains = np.arange(tp.CHAIN0, tp.CHAIN0 + Cn)
    if stream == "inj":
        delta = (rng.random((T, Cn, P)) * 2 - 1) * scale
        thresh = rng.random((T, Cn))
    else:
        delta = tp._native_delta(stream, scale, tp.RADIUS, T, chains, P)
        thresh = philox.thresholds(tp.SEED, T, chains)
    coloured = delta @ _chol(scale).T
    ref = o.mh_normreg_walk(init, coloured, thresh, x if P == 3 else None, y, lims,
                            ex.astype(bool), lg.astype(bool), has_slope=P == 3, accept=accept,
                            coef=coef, bound=bound)
    return dict(x=x, y=y, lims=lims, ex=ex, lg=lg, scale=scale, init=init, delta=delta,
                thresh=thresh), ref


def _run(eng, path, case, per_step, bound, step0=0, n_steps=None, state=None, state_lp=None):
    variant, Cn, P = tp.PATHS[path]
    accept, coef, stream = tp.CASES[case][:3]
    pb_, _ = _problem_and_ref(path, case, False)
    n_steps = tp._steps(path) if n_steps is None else n_steps
    if stream == "inj":
        inj = dict(inj_delta=dev(eng, tcd_to_tdc(pb_["delta"][step0:step0 + n_steps])),
                   inj_thresh=dev(eng, pb_["thresh"][step0:step0 + n_steps]))
        prop = "uniform"
    else:
        inj, prop = {}, stream
    st = dev(eng, pb_["init"].T) if state is None else state
    out = eng.mh_normreg(st, dev(eng, pb_["y"]), dev(eng, pb_["x"]) if P == 3 else None,
                         n_steps, pb_["lims"], pb_["ex"], pb_["lg"], pb_["scale"], thin=tp.THIN,
                         seed=tp.SEED, step0=step0, chain0=tp.CHAIN0, accept=accept,
                         accept_coef=coef, prop=prop, variant=variant, state_lp=state_lp,
                         per_step=per_step, stats=True, prop_radius=tp.RADIUS, prop_bound=bound,
                         prop_chol=_chol(pb_["scale"]), **inj)
    eng.sync()
    return out, st


@pytest.mark.parametrize("case", list(tp.CASES))
@pytest.mark.parametrize("path", list(tp.PATHS))
def test_coloured_path_matches_oracle(path, case):
    eng = engine()
    bound = tp.CASES[case][3]
    _, ref = _problem_and_ref(path, case, bound)
    out, st = _run(eng, path, case, True, bound)
    _check(out, st, ref, tp._tol(case), True)
    # no per-step outputs, no bound rule
    _, plain = _problem_and_ref(path, case, False)
    if bound:                                   # the bound rule changed some proposals
        assert not np.array_equal(ref["xprop"], plain["xprop"])
    out, st = _run(eng, path, case, False, False)
    _check(out, st, plain, tp._tol(case), False)


@pytest.mark.parametrize("path", list(tp.PATHS))
def test_coloured_resume_equals_one_call(path):
    """Native stream, nonzero chain0, split at a record boundary: bit-equal to one call."""
    eng = engine()
    T = tp._steps(path)
    T1 = tp.THIN * (T // (2 * tp.THIN))
    one, st = _run(eng, path, "native_uniform", True, False)
    a, st2 = _run(eng, path, "native_uniform", True, False, n_steps=T1)
    b, _ = _run(eng, path, "native_uniform", True, False, step0=T1, n_steps=T - T1, state=st2,
                state_lp=a["state_lp"])
    for k in ("x", "prob", "accept", "score", "xprop", "pprop"):
        assert np.array_equal(np.concatenate([host(a[k]), host(b[k])]), host(one[k]),
                              equal_nan=True), k
    assert np.array_equal(host(st2), host(st))
    assert np.array_equal(host(b["state_lp"]), host(one["state_lp"]))
    assert np.array_equal(host(a["accept_count"]) + host(b["accept_count"]),
                          host(one["accept_count"]))
    for k in ("stat_sum", "stat_sumsq"):
        assert relerr(host(a[k]) + host(b[k]), host(one[k])) <= 1e-14


def _linreg_process(cov, delta, log_sigma=False):
    """The gibbs_linreg.py model (C3) driven as MH with paras.set_tran(cov)."""
    x = pb.RV('x', vtype=float, vset=[-np.inf, np.inf])
    y = pb.RV('y', vtype=float, vset=[-np.inf, np.inf])
    beta_0 = pb.RV('beta_0', vtype=float, vset=[-6., 6.], pscale='log')
    beta_1 = pb.RV('beta_1', vtype=float, vset=[-6., 6.], pscale='log')
    y_sigma = pb.RV('y_sigma', vtype=float, vset=[(0.001), 10.], pscale='log')
    if log_sigma:
        y_sigma.set_ufun((np.log, np.exp))

    def norm_reg(x, y, beta_0, beta_1, y_sigma):
        return scipy.stats.norm.logpdf(y, loc=beta_0 + beta_1 * x, scale=y_sigma)

    paras = beta_0 & beta_1 & y_sigma
    process = pb.SP(x & y, paras)
    process.set_prob(norm_reg, pscale='log')
    paras.set_tran(np.asarray(cov, dtype=float))
    paras.set_delta(delta)
    process.set_tran(paras)
    process.set_delta(paras)
    process.set_scores('metropolis')
    return process


def _uncentred_data(N, seed):
    rng = np.random.default_rng(seed)
    xo = rng.normal(5., 1., N)
    return xo, rng.normal(-1. + 1.5 * xo, 0.5)


@pytest.mark.filterwarnings("ignore:probayes_b200. the Python likelihood")
def test_public_api_single_chain_proposals_are_coloured():
    """summary.p of a reference-shaped run is ufun^-1(ufun(x) + L delta) of its predecessor,
    for the injected delta (log-ufun sigma, so the move is not a plain sum)."""
    engine()
    T, N = 60, 80
    xo, yo = _uncentred_data(N, 11)
    X = np.stack([np.ones(N), xo], 1)
    b_ols = np.linalg.lstsq(X, yo, rcond=None)[0]
    cov = np.zeros((3, 3))                   # twice the posterior covariance, log(sigma) last
    cov[:2, :2] = 2 * np.mean((yo - X @ b_ols) ** 2) * np.linalg.inv(X.T @ X)
    cov[2, 2] = 2 / (2 * N)
    L = np.linalg.cholesky(cov)
    rng = np.random.default_rng(12)
    delta, thresh = rng.standard_normal((T, 3)), rng.random(T)
    process = _linreg_process(cov, [0.02], log_sigma=True)
    init = np.array([b_ols[0], b_ols[1], 0.5])
    sampler = process.sampler({'beta_0': init[0], 'beta_1': init[1], 'y_sigma': init[2]},
                              {'x,y': [xo, yo]}, stop=T, iid=True, joint=True,
                              inj_delta=delta, inj_thresh=thresh)
    summary = process(process.walk(sampler))
    keys = ['beta_0', 'beta_1', 'y_sigma']
    prop = np.stack([summary.p[k] for k in keys], 1)
    state = np.stack([summary.v[k] for k in keys], 1)
    pred = np.concatenate([init[None], state[:-1]])
    step = delta @ L.T
    want = pred + step
    want[:, 2] = np.exp(np.log(pred[:, 2]) + step[:, 2])
    assert relerr(prop, want) <= 1e-12
    u = np.array([v is True for v in summary.u])
    assert 0 < u.sum() < T                          # some moves accepted, some not
    assert np.array_equal(state[u], prop[u]) and np.array_equal(state[~u], pred[~u])
    ref = o.mh_normreg_walk(init[None], step[:, None], thresh[:, None], xo, yo,
                            np.array([[-6., 6.], [-6., 6.], [0.001, 10.]]),
                            np.zeros((3, 2), bool), np.array([0, 0, 1], bool))
    assert np.array_equal(ref["u"][:, 0], u)
    assert relerr(summary.v.prob, ref["prob"][:, 0]) <= 1e-12


@pytest.mark.filterwarnings("ignore:probayes_b200. the Python likelihood")
def test_public_api_batched_posterior_uncentred_x():
    """Native draws, 1024 chains, x ~ N(5, 1) (posterior corr(b0, b1) ~ -0.98), proposal
    covariance 2.38^2 / 3 times the large-N posterior covariance.  Reference: with the flat box
    priors, (b0, b1) | sigma ~ N(b_ols, sigma^2 (X'X)^-1) and sigma^2 | y is inverse gamma, so
    E[b] = b_ols, Cov[b] = E[sigma^2] (X'X)^-1 with E[sigma^2] = RSS / (N - 5), and E[sigma] by
    quadrature of p(sigma | y) ~ sigma^-(N-2) exp(-RSS / (2 sigma^2)).  Monte Carlo error: the
    chains are independent, so the standard error of a pooled mean (or covariance) is the
    standard deviation of the per-chain values over sqrt(chains); each check allows 5 of them,
    and the standard errors are asserted to be below 5 % of the posterior sd."""
    engine()
    N, Cn, T, thin, burn = 4000, 1024, 1200, 4, 50
    xo, yo = _uncentred_data(N, 21)
    X = np.stack([np.ones(N), xo], 1)
    XtXi = np.linalg.inv(X.T @ X)
    b_ols = XtXi @ X.T @ yo
    rss = float(np.sum((yo - X @ b_ols) ** 2))
    s2 = rss / N
    post = np.zeros((3, 3))
    post[:2, :2] = s2 * XtXi
    post[2, 2] = s2 / (2 * N)
    assert post[0, 1] / np.sqrt(post[0, 0] * post[1, 1]) < -0.95
    process = _linreg_process(2.38 ** 2 / 3 * post, scipy.stats.norm(0., 1.))
    sampler = process.sampler({'beta_0': b_ols[0], 'beta_1': b_ols[1], 'y_sigma': np.sqrt(s2)},
                              {'x,y': [xo, yo]}, stop=T, iid=True, joint=True, chains=Cn,
                              thin=thin, seed=8)
    summary = process(process.walk(sampler))
    assert 0.15 < summary.u.rate() < 0.6
    V = np.stack([summary.v[k][:, burn:] for k in ['beta_0', 'beta_1', 'y_sigma']])  # [3, C, R]
    # reference values
    e_s2 = rss / (N - 5)
    sg = np.sqrt(s2) * np.linspace(0.8, 1.2, 40001)
    logw = -(N - 2) * np.log(sg) - rss / (2 * sg * sg)
    w = np.exp(logw - logw.max())
    e_sigma = float(np.sum(w * sg) / np.sum(w))
    want_mean = np.array([b_ols[0], b_ols[1], e_sigma])
    want_cov = e_s2 * XtXi
    sd = np.sqrt(np.diag(post))
    chain_means = V.mean(axis=2)                                        # [3, C]
    se = chain_means.std(axis=1, ddof=1) / np.sqrt(Cn)
    assert np.all(se < 0.05 * sd)
    assert np.all(np.abs(chain_means.mean(axis=1) - want_mean) < 5 * se)
    dev_ = V[:2] - V[:2].mean(axis=(1, 2), keepdims=True)
    for i, j in ((0, 0), (0, 1), (1, 1)):
        per_chain = (dev_[i] * dev_[j]).mean(axis=1)                     # [C]
        se_c = per_chain.std(ddof=1) / np.sqrt(Cn)
        assert se_c < 0.05 * abs(want_cov[i, j])
        assert abs(per_chain.mean() - want_cov[i, j]) < 5 * se_c, (i, j)


def _params(eng, L, y):
    p = eng._normreg_params(4, 2, None, y, [[40., 60.], [5., 20.]], [[0, 0], [0, 0]], [0, 0],
                            [0.1, 0.1], prop_chol=L)
    st, lp = eng.to_device(np.tile([[50.], [10.]], (1, 4))), eng.zeros(4)
    p.n_steps, p.thin, p.state, p.state_lp = 3, 1, st.data_ptr(), lp.data_ptr()
    return p, st, lp


@pytest.mark.parametrize("what,L", [
    ("upper", [[1., 0.2], [0., 1.]]), ("nan", [[1., 0.], [np.nan, 1.]]),
    ("inf", [[np.inf, 0.], [0.1, 1.]]), ("zero_diag", [[1., 0.], [0.3, 0.]]),
    ("negative_diag", [[-1., 0.], [0.3, 1.]])])
def test_malformed_factor_is_refused(what, L):
    """pbx_mh_normreg_run returns PBX_ERR_INVALID for a factor that is not lower-triangular,
    finite and positive on the diagonal; pbx_normreg_logjoint ignores it."""
    eng = engine()
    y = eng.to_device(np.random.default_rng(1).normal(50., 10., 100))
    p, st, lp = _params(eng, np.array(L), y)
    rc = eng.lib.pbx_mh_normreg_run(eng.ctx, C.byref(p))
    assert rc == -1                                       # PBX_ERR_INVALID
    assert b"prop_mat" in eng.lib.pbx_last_error()
    out = eng.empty(4)
    assert eng.lib.pbx_normreg_logjoint(eng.ctx, C.byref(p), C.c_void_p(st.data_ptr()),
                                        C.c_void_p(out.data_ptr())) == 0
    eng.sync()
    good, st, lp = _params(eng, np.array([[1., 0.], [0.3, 1.]]), y)
    _lib.check(eng.lib.pbx_mh_normreg_run(eng.ctx, C.byref(good)), "pbx_mh_normreg_run")
    eng.sync()
    with pytest.raises(_lib.PbxError, match="prop_mat"):
        eng.mh_normreg(eng.to_device(np.tile([[50.], [10.]], (1, 4))), y, None, 3,
                       [[40., 60.], [5., 20.]], [[0, 0], [0, 0]], [0, 0], [0.1, 0.1],
                       prop_chol=np.array(L))
