"""Student-t and Cauchy likelihoods on the device: every K2 walk path against the oracle (the
cases of test_gpu_normreg_paths, a covariance-coloured case and Cauchy data 1e6 sigma out), the
evaluate-only path random sampling uses, K3, the kernel instantiation each case launches, the
public API on data with outliers, and the sharded helpers on one rank."""
import functools
import zlib

import numpy as np
import pytest
import scipy.special
import scipy.stats
from conftest import relerr
from gpu_util import engine, dev, tcd_to_tdc, host
from oracle import philox
import probayes_b200 as pb
from probayes_b200 import catalogue
import studentt_oracle as to
import test_gpu_normreg_paths as tp

pytestmark = pytest.mark.gpu

T4 = catalogue.likelihood('t', 4.)
CAUCHY = catalogue.likelihood('cauchy')
# every walk path but the sufficient statistics (refused for the t)
PATHS = {k: v for k, v in tp.PATHS.items() if v[0] != 3}
# test_gpu_normreg_paths' cases (df = 4), a coloured one, and Cauchy data 1e6 sigma out
CASES = dict(tp.CASES, coloured=("log", 1.0, "inj", False, True, 2500),
             cauchy_far=("log", 1.0, "inj", False, True, 2501))
CORR = {3: np.array([[1., -.6, .3], [-.6, 1., -.4], [.3, -.4, 1.]]),
        2: np.array([[1., -.6], [-.6, 1.]])}


def _lik(case):
    return CAUCHY if case == "cauchy_far" else T4


def _chol(case, scale):
    if case != "coloured":
        return None
    return np.linalg.cholesky(CORR[len(scale)]) * scale[:, None] / scale[None, :]


@functools.lru_cache(maxsize=None)
def _problem_and_ref(path, case, bound):
    variant, C, P = PATHS[path]
    accept, coef, stream, tight, logufun, N = CASES[case]
    rng = np.random.default_rng(zlib.crc32(("studentt/" + path + "/" + case).encode()))
    x, y, lims, ex, lg, scale, init = tp._problem(P, N, logufun, tight, C, rng)
    if case == "cauchy_far":             # log1p at arguments ~1e12
        sg = 0.5 if P == 3 else 10.
        y = y.copy()
        y[::97] += 1e6 * sg * rng.choice([-1., 1.], len(y[::97]))
    T = tp._steps(path)
    chains = np.arange(tp.CHAIN0, tp.CHAIN0 + C)
    if stream == "inj":
        delta = (rng.random((T, C, P)) * 2 - 1) * scale
        thresh = rng.random((T, C))
    else:
        delta = tp._native_delta(stream, scale, tp.RADIUS, T, chains, P)
        thresh = philox.thresholds(tp.SEED, T, chains)
    L = _chol(case, scale)
    ref = to.mh_normreg_walk(init, delta if L is None else delta @ L.T, thresh,
                             x if P == 3 else None, y, lims, ex.astype(bool), lg.astype(bool),
                             has_slope=P == 3, accept=accept, coef=coef, bound=bound,
                             lik=_lik(case))
    return dict(x=x, y=y, lims=lims, ex=ex, lg=lg, scale=scale, init=init, delta=delta,
                thresh=thresh, chol=L), ref


def _run(eng, path, case, per_step, bound, step0=0, n_steps=None, state=None, state_lp=None):
    variant, C, P = PATHS[path]
    accept, coef, stream = CASES[case][:3]
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
                         per_step=per_step, stats=True, prop_radius=tp.RADIUS,
                         prop_bound=bound, prop_chol=pb_["chol"], lik=_lik(case), **inj)
    eng.sync()
    return out, st


def _check(out, st, ref, tol, per_step):
    """tp._check, with log-joints of -inf (a proposal outside the prior box in two coordinates)
    required at the same places and then compared as -huge."""
    huge = np.finfo(float).max
    lp, want = host(out["prob"]), ref["prob"][tp.THIN - 1::tp.THIN]
    assert np.array_equal(np.isneginf(lp), np.isneginf(want))
    out = dict(out, prob=out["prob"].nan_to_num(nan=np.nan, neginf=-huge),
               state_lp=out["state_lp"].nan_to_num(nan=np.nan, neginf=-huge))
    ref = dict(ref, prob=np.nan_to_num(ref["prob"], nan=np.nan, neginf=-huge))
    tp._check(out, st, ref, tol, per_step)


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("path", list(PATHS))
def test_t_path_matches_oracle(path, case):
    eng = engine()
    bound = CASES[case][3]
    tol = 1e-12 if CASES[case][2] == "inj" else 1e-11
    _, ref = _problem_and_ref(path, case, bound)
    out, st = _run(eng, path, case, True, bound)
    _check(out, st, ref, tol, True)
    _, plain = _problem_and_ref(path, case, False)
    out, st = _run(eng, path, case, False, False)
    _check(out, st, plain, tol, False)


@pytest.mark.parametrize("path", list(PATHS))
def test_t_path_resume_equals_one_call(path):
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


def test_t_suffstat_refused_by_the_abi():
    eng = engine()
    pb_, _ = _problem_and_ref("warp", "log_logufun", False)
    th = dev(eng, pb_["init"].T)
    with pytest.raises(pb.PbxError, match="variant 3"):
        eng.mh_normreg(th, dev(eng, pb_["y"]), None, 4, pb_["lims"], pb_["ex"], pb_["lg"],
                       pb_["scale"], variant=3, lik=T4)
    with pytest.raises(pb.PbxError, match="variant 3"):
        eng.normreg_logjoint(th, dev(eng, pb_["y"]), None, pb_["lims"], pb_["ex"], pb_["lg"],
                             variant=3, lik=T4)
    with pytest.raises(pb.PbxError, match="lik_df"):
        eng.normreg_logjoint(th, dev(eng, pb_["y"]), None, pb_["lims"], pb_["ex"], pb_["lg"],
                             lik=dict(df=np.nan, logc=0.))
    with pytest.raises(pb.PbxError, match="df"):
        y = dev(eng, pb_["y"])
        eng.grid_norm_logjoint(y, y[:3], y[:3], y[:3], y[:3], lik=dict(df=-1., logc=0.))


@pytest.mark.parametrize("lik", [T4, CAUCHY, catalogue.likelihood('t', 1e6)],
                         ids=["t4", "cauchy", "t1e6"])
@pytest.mark.parametrize("C,P", [(37, 2), (3000, 3), (5, 3)])
def test_t_logjoint_matches_scipy(lik, C, P):
    """The evaluate-only path random sampling uses (tiles for 37 / 3000 chains, stream for 5),
    at N = 1e5 with 1 % gross outliers, against the scipy sums."""
    eng = engine()
    rng = np.random.default_rng(C + P)
    N = 100001
    x = rng.normal(0., 1., N)
    y = (-1. + 1.5 * x if P == 3 else 50.) + rng.normal(0., 0.5, N)
    y[::100] += 1e4
    lims = np.array([[-6., 6.], [-6., 6.], [0.001, 10.]]) if P == 3 else \
        np.array([[40., 60.], [0.001, 10.]])
    ex, lg = np.zeros((P, 2), int), np.zeros(P, int)
    theta = np.stack([rng.uniform(lo, hi, C) for lo, hi in lims], axis=1)
    got = host(eng.normreg_logjoint(dev(eng, theta.T), dev(eng, y),
                                    dev(eng, x) if P == 3 else None, lims, ex, lg, lik=lik))
    want = to.normreg_logjoint(theta, x, y, lims, ex.astype(bool), lg.astype(bool), P == 3, lik)
    assert relerr(got, want) <= 1e-12


@pytest.mark.parametrize("lik", [T4, CAUCHY], ids=["t4", "cauchy"])
def test_t_grid_matches_scipy(lik):
    eng = engine()
    rng = np.random.default_rng(5)
    # all cells of a small grid, odd N (the ragged tail), aligned and unaligned observations
    N = 1001
    xo = np.concatenate([[0.], rng.normal(50., 10., N)])
    xo[5::50] += 1e5
    mu, sg = np.linspace(40., 60., 37), np.linspace(5., 20., 53)
    lpm, lps = rng.normal(0., 1., 37), rng.normal(0., 1., 53)
    want = to.grid_logjoint(xo[1:], mu, sg, lpm, lps, lik)
    xd = dev(eng, xo)
    for xs in (xd[1:], dev(eng, xo[1:])):
        got = host(eng.grid_norm_logjoint(xs, dev(eng, mu), dev(eng, sg), dev(eng, lpm),
                                          dev(eng, lps), lik=lik))
        assert relerr(got, want) <= 1e-12
    # sampled cells of 1024 x 1024 at N = 1e5
    N, M = 100000, 1024
    xo = rng.normal(50., 10., N)
    xo[::1000] -= 1e5
    mu, sg = np.linspace(40., 60., M), np.linspace(5., 20., M)
    lpm, lps = np.full(M, -np.log(20.)), -np.log(15.) - np.log(sg)
    got = host(eng.grid_norm_logjoint(dev(eng, xo), dev(eng, mu), dev(eng, sg), dev(eng, lpm),
                                      dev(eng, lps), lik=lik))
    ii, jj = rng.integers(0, M, 64), rng.integers(0, M, 64)
    for i, j in zip(ii, jj):
        w = to.grid_logjoint(xo, mu[i:i + 1], sg[j:j + 1], lpm[i:i + 1], lps[j:j + 1], lik)
        assert relerr(got[i, j], w[0, 0]) <= 1e-12


LAUNCHES = [
    ("tiles_kc1", "nr_tiles_kernel<1, true, false, 1>"),
    ("tiles_kc2", "nr_tiles_kernel<2, false, false, 1>"),
    ("tiles_kc4", "nr_tiles_kernel<4, true, false, 1>"),
    ("stream_ks1", "nr_stream_kernel<1, false, false, 1>"),
    ("stream_ks2", "nr_stream_kernel<2, true, false, 1>"),
    ("stream_ks4", "nr_stream_kernel<4, false, false, 1>"),
    ("stream_ks8", "nr_stream_kernel<8, true, false, 1>"),
    ("warp_slope", "rw_walk_kernel<true, false, 1>"),
    ("warp", "rw_walk_kernel<false, false, 1>"),
]


def test_t_launches_its_instantiation():
    """Every t case launches the Student-t instantiation of its path (the coloured case the one
    with the per-step extras / colouring) and no normal one; one profiler session for all, as
    test_gpu_mh_mvn_kernels does."""
    import re
    import torch
    from torch.profiler import profile, ProfilerActivity
    eng = engine()
    runs = [(path, case) for path, _ in LAUNCHES for case in ("log_logufun", "coloured")]
    for path, case in runs:                      # inputs and oracle outside the session
        _problem_and_ref(path, case, False)
    x = dev(eng, np.linspace(0., 1., 100))
    eng.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        probe = torch.ones(1024, device=eng.device, dtype=torch.float64) * 3.0
        for path, case in runs:
            _run(eng, path, case, False, False)
        eng.grid_norm_logjoint(x, x[:4], x[1:5], x[:4], x[:4], lik=T4)
        eng.sync()
        torch.cuda.synchronize()
    del probe
    kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    if not kern:
        pytest.skip("the profiler recorded no device events, not even the probe's torch kernel")
    kern.sort(key=lambda e: e.time_range.start)
    names = []
    for e in kern:
        m = re.search(r"((?:nr_tiles|nr_stream|rw_walk|grid_logjoint)_kernel<[^>]*>)", e.name)
        if m:
            names.append(re.sub(r"\s+", " ", m.group(1)))
    # the sequence of instantiations, one entry per run (a run of the per-step paths launches
    # its kernel once per step; the profiler can miss the first launches of a session)
    seq = [n for i, n in enumerate(names) if i == 0 or n != names[i - 1]]
    want = [w for _, inst in LAUNCHES for w in (inst, inst.replace("false, 1>", "true, 1>"))]
    assert seq == want + ["grid_logjoint_kernel<1>"], seq


# ---- the public API on data with outliers ------------------------------------------------------
MU_LIMS, SIGMA_LIMS = (40., 60.), (5., 20.)


def _outlier_data():
    rng = np.random.default_rng(2024)
    data = rng.normal(50., 10., 200)
    data[:6] = [900., 1200., -800., 2500., 1500., -3000.]      # gross outliers
    return data


def _rvs():
    mu = pb.RV('mu', vtype=float, vset=MU_LIMS)
    sigma = pb.RV('sigma', vtype=float, vset=SIGMA_LIMS)
    x = pb.RV('x', vtype=float, vset={-np.inf, np.inf})
    sigma.set_ufun((np.log, np.exp))
    return mu, sigma, x


def _grid_posterior(M=256, S=256):
    mu, sigma, x = _rvs()
    model = pb.SD(pb.RF(x), pb.RF(mu, sigma))
    model.set_prob(scipy.stats.t.logpdf, order={'x': 0, 'mu': 'loc', 'sigma': 'scale'},
                   df=4., pscale='log')
    joint = model({x: _outlier_data(), 'mu': {M}, 'sigma': {S}}, iid=True, joint=True)
    return model, joint, joint.conditionalise('x')


def test_t_dgei_posterior_against_numpy():
    engine()
    model, joint, post = _grid_posterior()
    data = _outlier_data()
    mus, sgs = np.ravel(post['mu']), np.ravel(post['sigma'])
    from probayes_b200.pscales import rescale
    lpm = rescale(np.asarray(model._roots['mu'].eval_prob(mus), float),
                  model._roots['mu'].pscale, 'log')
    lps = rescale(np.asarray(model._roots['sigma'].eval_prob(sgs), float),
                  model._roots['sigma'].pscale, 'log')
    lj = to.grid_logjoint(data, mus, sgs, lpm, lps, T4)
    assert relerr(joint.prob, lj) <= 1e-12
    lpost = lj - scipy.special.logsumexp(lj)
    keep = lpost > -600.
    assert np.abs(post.prob[keep] - lpost[keep]).max() <= 1e-10
    p = np.exp(lpost)
    assert np.abs(post.marginal('mu').prob - np.log(p.sum(axis=1))).max() <= 1e-10
    assert np.abs(post.marginal('sigma').prob - np.log(p.sum(axis=0))).max() <= 1e-10
    e = post.expectation()
    assert abs(e['mu'] - (p.sum(axis=1) * mus).sum()) <= 1e-9
    assert abs(e['sigma'] - (p.sum(axis=0) * sgs).sum()) <= 1e-9
    # the t posterior ignores the outliers; the normal's is dragged far from the bulk
    assert abs(e['mu'] - np.median(data)) < 2.


def test_t_mh_posterior_agrees_with_the_grid():
    """1024 MH chains of the same (mu, sigma) model: means and sds within a Monte Carlo error
    estimated from the spread of the per-chain means (chains are independent)."""
    engine()
    _, _, post = _grid_posterior(512, 512)
    p = np.exp(post.prob)
    mus, sgs = np.ravel(post['mu']), np.ravel(post['sigma'])
    grid = {}
    for k, v, w in (('mu', mus, p.sum(axis=1)), ('sigma', sgs, p.sum(axis=0))):
        m = (w * v).sum()
        grid[k] = (m, np.sqrt((w * (v - m) ** 2).sum()))
    mu, sigma, x = _rvs()
    paras = pb.RF(mu, sigma)
    process = pb.SP(pb.RF(x), paras)
    process.set_prob(scipy.stats.t.logpdf, order={'x': 0, 'mu': 'loc', 'sigma': 'scale'},
                     df=4., pscale='log')
    paras.set_delta([0.06], scale=True)
    process.set_tran(paras)
    process.set_delta(paras)
    process.set_scores('metropolis')
    sampler = process.sampler({'mu': 50., 'sigma': 10.}, {x: _outlier_data()}, stop=6000,
                              iid=True, joint=True, chains=1024, thin=4, seed=17)
    v = process(process.walk(sampler)).v
    for k in ('mu', 'sigma'):
        s = np.asarray(v[k])[:, 250:]                  # [chains, records] after burn-in
        cm = s.mean(axis=1)
        se = cm.std(ddof=1) / np.sqrt(len(cm))
        m, sd = grid[k]
        assert abs(cm.mean() - m) <= 5. * se + 1e-3 * sd, (k, cm.mean(), m, se)
        sd_mh = s.std()
        csd = s.std(axis=1)
        assert abs(sd_mh - sd) <= 5. * csd.std(ddof=1) / np.sqrt(len(csd)) + 0.01 * sd, \
            (k, sd_mh, sd)


def test_t_sharded_helpers_on_one_rank_equal_unsharded():
    from probayes_b200 import dist as pd_
    eng = engine()
    data = _outlier_data()
    mu, sg = np.linspace(40., 60., 96), np.linspace(5., 20., 80)
    lpm, lps = np.full(96, -np.log(20.)), -np.log(15.) - np.log(sg)
    r = pd_.dgei_sharded(eng, data, mu, sg, lpm, lps, lik=T4)
    lj = eng.grid_norm_logjoint(dev(eng, data), dev(eng, mu), dev(eng, sg), dev(eng, lpm),
                                dev(eng, lps), lik=T4)
    w = eng.grid_conditionalise(lj)
    assert np.array_equal(host(r["post"]), host(w["post"]))
    assert np.array_equal(host(r["marg_mu"]), host(w["marg_mu"]))
    lims, ex, lg = np.array([MU_LIMS, SIGMA_LIMS]), np.zeros((2, 2), int), np.array([0, 1])
    ro = pd_.omc_sharded(eng, data, lims, ex, lg, 5000, seed=21, lik=CAUCHY)
    th = eng.box_sample(lims, lg, 5000, seed=21)
    lp = eng.normreg_logjoint(th, dev(eng, data), None, lims, ex, lg, lik=CAUCHY)
    assert np.array_equal(host(ro["theta"]), host(th))
    w1 = eng.grid_conditionalise(lp.reshape(1, -1))
    s1 = host(eng.expectation_sums(w1["post"].reshape(-1), True, None, th))
    assert np.allclose(ro["expectation"], s1[1:] / s1[0], rtol=1e-12, atol=0.)
