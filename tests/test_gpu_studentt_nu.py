"""Student-t likelihood with nu sampled on the device (PBX_LIK_STUDENT_T_NU, theta = (mu, sigma,
nu)): every K2 walk path against the oracle, the instantiation each case launches, the device
logc(nu) against mpmath, the evaluate-only path and random sampling against the scipy sums, and
posterior recovery on t_4 data against a stack of fixed-nu grids."""
import functools
import zlib

import mpmath
import numpy as np
import pytest
import scipy.stats
from conftest import relerr
from gpu_util import engine, dev, tcd_to_tdc, host
from oracle import np_oracle as o
from oracle import philox
import probayes_b200 as pb
from probayes_b200 import _lib, catalogue
import studentt_nu_oracle as tno
import test_gpu_normreg_paths as tp
import test_gpu_studentt as ts

pytestmark = pytest.mark.gpu

NU = dict(family='t', df_param='nu')
# (variant, C): C selects KC for the tiles (>= 4096: 4, >= 2048: 2) and KS for the stream
PATHS = {
    "tiles_kc1": (1, 37), "tiles_kc2": (1, 2100), "tiles_kc4": (1, 4100),
    "stream_ks1": (2, 1), "stream_ks2": (2, 2), "stream_ks4": (2, 4), "stream_ks8": (2, 8),
    "warp": (4, 37),
}
# accept rule, accept_coef, stream ("inj" or the native proposal), bound, log-ufun sigma and
# nu, coloured (a 3x3 covariance transition), N
CASES = {
    "reference_coef": ("reference", 0.7, "inj", False, False, False, 40),
    "log_logufun": ("log", 1.0, "inj", False, True, False, 2500),
    "bound_mixed": ("log", 1.0, "inj", True, True, False, 2500),
    "native_uniform": ("log", 1.0, "uniform", False, False, False, 2500),
    "native_normal": ("reference", 1.0, "normal", False, True, False, 60),
    "coloured": ("log", 1.0, "inj", False, True, True, 2500),
    "native_coloured": ("log", 1.0, "normal", False, True, True, 2500),
}
CORR = np.array([[1., -.5, .3], [-.5, 1., -.4], [.3, -.4, 1.]])


def _problem(N, logufun, tight, C, rng):
    """t_4 data around (mu, sigma) = (1, 2), the prior box, proposal scales and a start near the
    bulk.  ``tight``: a box around the start that proposals leave at every end (closed | open
    below | open above)."""
    y = 1. + 2. * rng.standard_t(4., N)
    sd = 2. / np.sqrt(N)
    lims = np.array([[-5., 7.], [0.2, 10.], [0.5, 60.]])
    ex = np.array([[0, 0], [1, 0], [0, 0]])
    init = np.stack([rng.uniform(1. - sd, 1. + sd, C), rng.uniform(1.9, 2.1, C),
                     rng.uniform(3.5, 5., C)], axis=1)
    scale = np.array([2.5 * sd, 2. * sd, 0.3])
    if tight:
        lims = np.array([[1. - 3.2 * sd, 1. + 3.2 * sd], [1.8, 2.2], [3., 6.]])
        ex = np.array([[0, 0], [1, 0], [0, 1]])
    lg = np.array([0, 1, 1]) if logufun else np.zeros(3, int)
    if logufun:
        scale[1:] = [scale[1] / 2., 0.08]
    return y, lims, ex, lg, scale, init


@functools.lru_cache(maxsize=None)
def _problem_and_ref(path, case, bound):
    variant, C = PATHS[path]
    accept, coef, stream, tight, logufun, coloured, N = CASES[case]
    rng = np.random.default_rng(zlib.crc32(("studentt_nu/" + path + "/" + case).encode()))
    y, lims, ex, lg, scale, init = _problem(N, logufun, tight, C, rng)
    T = tp._steps(path)
    chains = np.arange(tp.CHAIN0, tp.CHAIN0 + C)
    if stream == "inj":
        delta = (rng.random((T, C, 3)) * 2 - 1) * scale
        thresh = rng.random((T, C))
    else:
        delta = tp._native_delta(stream, scale, tp.RADIUS, T, chains, 3)
        thresh = philox.thresholds(tp.SEED, T, chains)
    L = np.linalg.cholesky(CORR) * scale[:, None] / scale[None, :] if coloured else None
    ref = tno.mh_walk(init, delta if L is None else delta @ L.T, thresh, y, lims,
                      ex.astype(bool), lg.astype(bool), accept=accept, coef=coef, bound=bound)
    return dict(y=y, lims=lims, ex=ex, lg=lg, scale=scale, init=init, delta=delta,
                thresh=thresh, chol=L), ref


def _run(eng, path, case, per_step, bound, step0=0, n_steps=None, state=None, state_lp=None):
    variant, C = PATHS[path]
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
    out = eng.mh_normreg(st, dev(eng, pb_["y"]), None, n_steps, pb_["lims"], pb_["ex"],
                         pb_["lg"], pb_["scale"], thin=tp.THIN, seed=tp.SEED, step0=step0,
                         chain0=tp.CHAIN0, accept=accept, accept_coef=coef, prop=prop,
                         variant=variant, state_lp=state_lp, per_step=per_step, stats=True,
                         prop_radius=tp.RADIUS, prop_bound=bound, prop_chol=pb_["chol"], lik=NU,
                         **inj)
    eng.sync()
    return out, st


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("path", list(PATHS))
def test_nu_path_matches_oracle(path, case):
    """Accept decisions identical; records, running sums, final state and log-joints within
    1e-12 (injected streams) / 1e-11 (native Philox replay); with and without the per-step
    outputs and the bound rule."""
    eng = engine()
    bound = CASES[case][3]
    tol = 1e-12 if CASES[case][2] == "inj" else 1e-11
    _, ref = _problem_and_ref(path, case, bound)
    out, st = _run(eng, path, case, True, bound)
    ts._check(out, st, ref, tol, True)
    _, plain = _problem_and_ref(path, case, False)
    if bound:
        assert not np.array_equal(ref["xprop"], plain["xprop"])
    out, st = _run(eng, path, case, False, False)
    ts._check(out, st, plain, tol, False)


@pytest.mark.parametrize("path", list(PATHS))
def test_nu_path_resume_equals_one_call(path):
    """Two calls split at step0 > 0 give one call's records, per-step outputs and state, which
    test_nu_path_matches_oracle pins to the oracle."""
    eng = engine()
    T = tp._steps(path)
    T1 = tp.THIN * (T // (2 * tp.THIN))
    one, st = _run(eng, path, "native_coloured", True, False)
    a, st2 = _run(eng, path, "native_coloured", True, False, n_steps=T1)
    b, _ = _run(eng, path, "native_coloured", True, False, step0=T1, n_steps=T - T1, state=st2,
                state_lp=a["state_lp"])
    for k in ("x", "prob", "accept", "score", "xprop", "pprop"):
        assert np.array_equal(np.concatenate([host(a[k]), host(b[k])]), host(one[k]),
                              equal_nan=True), k
    assert np.array_equal(host(st2), host(st))
    assert np.array_equal(host(b["state_lp"]), host(one["state_lp"]))
    assert np.array_equal(host(a["accept_count"]) + host(b["accept_count"]),
                          host(one["accept_count"]))


def test_nu_abi_refusals():
    eng = engine()
    y = dev(eng, np.zeros(10))
    th = dev(eng, np.array([[0.], [1.], [4.]]))
    lims = np.array([[-1., 1.], [0.5, 2.], [0.5, 60.]])
    ex, lg = np.zeros((3, 2), int), np.zeros(3, int)
    with pytest.raises(pb.PbxError, match="variant 3"):
        eng.normreg_logjoint(th, y, None, lims, ex, lg, variant=3, lik=NU)
    bad = lims.copy()
    bad[2, 0] = 0.                             # closed at 0: admits nu = 0
    with pytest.raises(pb.PbxError, match="nu > 0"):
        eng.normreg_logjoint(th, y, None, bad, ex, lg, lik=NU)
    ex0 = ex.copy()
    ex0[2, 0] = 1                              # open at 0: nu > 0 only
    assert np.isfinite(host(eng.normreg_logjoint(th, y, None, bad, ex0, lg, lik=NU))).all()
    # structs the engine never builds, filled by hand: each is refused with its own message
    import ctypes as C
    out = eng.empty(1)
    for field, value, msg in (("lik_df", 4., "lik_df and lik_logc must be 0"),
                              ("lik_logc", -1., "lik_df and lik_logc must be 0"),
                              ("has_slope", 1, "3 params \\(mu, sigma, nu\\) and no slope"),
                              ("n_params", 2, "3 params \\(mu, sigma, nu\\) and no slope")):
        p = eng._normreg_params(1, 3, None, y, lims, ex, lg, 0.0, lik=NU)
        setattr(p, field, value)
        if field == "has_slope":
            p.x_obs = p.y_obs
        with pytest.raises(pb.PbxError, match=msg):
            _lib.check(eng.lib.pbx_normreg_logjoint(eng.ctx, C.byref(p), eng._ptr(th),
                                                    eng._ptr(out)), "pbx_normreg_logjoint")


def _mp_logc(nu):
    with mpmath.workdps(40):
        v = mpmath.mpf(nu)
        return float(mpmath.loggamma((v + 1) / 2) - mpmath.loggamma(v / 2) -
                     mpmath.log(v * mpmath.pi) / 2)


def test_device_logc_against_mpmath():
    """logc(nu) as the kernels compute it, read through pbx_normreg_logjoint at N = 1 with y = mu
    and sigma = 1 (the sum is log1p(0) = 0) and every prior box of unit length (its log density
    is 0), so the log-joint IS logc.  Within 1e-14 absolute of mpmath over nu in [1e-3, 1e12];
    measured on a B200: 1.2e-15 at most (at nu = 11.9, the lgamma side of the crossover)."""
    eng = engine()
    nus = np.concatenate([np.geomspace(1e-3, 1e12, 601), [15.999999, 16., 16.000001]])
    y = dev(eng, np.zeros(1))
    lg = np.zeros(3, int)
    got = np.empty(len(nus))
    for i, v in enumerate(nus):
        lo = np.floor(v)                       # a unit box [lo, lo + 1], (0, 1] below nu = 1
        lims = np.array([[-0.5, 0.5], [0.5, 1.5], [lo, lo + 1.]])
        ex = np.array([[0, 0], [0, 0], [1 if lo == 0. else 0, 0]])
        th = dev(eng, np.array([[0.], [1.], [v]]))
        got[i] = host(eng.normreg_logjoint(th, y, None, lims, ex, lg, lik=NU))[0]
    want = np.array([_mp_logc(v) for v in nus])
    err = np.abs(got - want)
    print("device logc: max abs error %.3g at nu = %.6g" % (err.max(), nus[err.argmax()]))
    assert err.max() <= 1e-14, (err.max(), nus[err.argmax()])
    # no cancellation at large nu: within a few ulp of the normal's constant's neighbourhood
    assert np.abs(got[nus > 1e6] - want[nus > 1e6]).max() <= 2e-16


@pytest.mark.parametrize("C", [37, 3000, 5])
def test_nu_logjoint_matches_scipy(C):
    """The evaluate-only path random sampling uses (tiles for 37 / 3000 chains, stream for 5),
    at N = 1e5 with 1 % gross outliers, nu over [0.5, 1e5], against the scipy sums."""
    eng = engine()
    rng = np.random.default_rng(C)
    N = 100001
    y = 50. + 10. * rng.standard_t(3., N)
    y[::100] += 1e4
    lims = np.array([[40., 60.], [0.5, 30.], [0.5, 1e5]])
    ex, lg = np.zeros((3, 2), int), np.array([0, 1, 1])
    theta = np.stack([rng.uniform(40., 60., C), rng.uniform(0.5, 30., C),
                      np.exp(rng.uniform(np.log(0.5), np.log(1e5), C))], axis=1)
    got = host(eng.normreg_logjoint(dev(eng, theta.T), dev(eng, y), None, lims, ex, lg, lik=NU))
    want = tno.logjoint(theta, y, lims, ex.astype(bool), lg.astype(bool))
    assert relerr(got, want) <= 1e-12


LIMS_RS, LOGU_RS = np.array([[40., 60.], [5., 20.], [1., 50.]]), np.array([0, 1, 1])


def _nu_process(nu_order=1):
    mu = pb.RV('mu', vtype=float, vset=[40., 60.])
    sigma = pb.RV('sigma', vtype=float, vset=[5., 20.])
    nu = pb.RV('nu', vtype=float, vset=[1., 50.])
    sigma.set_ufun((np.log, np.exp))
    nu.set_ufun((np.log, np.exp))
    x = pb.RV('x', vtype=float, vset=(-np.inf, np.inf))
    process = pb.SP(pb.RF(x), mu & sigma & nu)
    process.set_prob(scipy.stats.t.logpdf,
                     order={'x': 0, 'nu': nu_order, 'mu': 'loc', 'sigma': 'scale'}, pscale='log')
    return process


def test_nu_random_sampling_matches_oracle():
    """SP random sampling ({0} requests: box draws, then the evaluate-only path) against the
    oracle on the replayed Philox uniforms, and dist.omc_sharded on one rank."""
    from probayes_b200 import dist as pd_
    eng = engine()
    data = 50. + 10. * np.random.default_rng(9).standard_t(4., 300)
    T = 20000
    process = _nu_process('df')
    sampler = process.sampler({'mu': {0}, 'sigma': {0}, 'nu': {0}, 'x': data}, iid=True,
                              joint=True, stop=T, seed=5)
    summary = process(process.walk(sampler))
    th = o.box_sample(LIMS_RS, LOGU_RS, philox.uniforms(5, T, 1, 3)[:, 0, :])
    got = np.stack([summary['mu'], summary['sigma'], summary['nu']])
    assert np.array_equal(got[0], th[0]) and relerr(got[1:], th[1:]) <= 4e-16
    ex = np.zeros((3, 2), int)
    lj = tno.logjoint(got.T[:3000], data, LIMS_RS, ex.astype(bool), LOGU_RS.astype(bool))
    assert relerr(summary.prob[:3000], lj) <= 1e-12
    ro = pd_.omc_sharded(eng, data, LIMS_RS, ex, LOGU_RS, 5001, seed=21, lik=NU)
    theta = host(ro["theta"])
    lj = tno.logjoint(theta.T, data, LIMS_RS, ex.astype(bool), LOGU_RS.astype(bool))
    w = np.exp(lj - lj.max())
    assert np.allclose(ro["expectation"], (theta * w).sum(axis=1) / w.sum(), rtol=1e-10, atol=0.)


LAUNCHES = [
    ("tiles_kc1", "nr_tiles_kernel<1, false, {}, 2>"),
    ("tiles_kc2", "nr_tiles_kernel<2, false, {}, 2>"),
    ("tiles_kc4", "nr_tiles_kernel<4, false, {}, 2>"),
    ("stream_ks1", "nr_stream_kernel<1, false, {}, 2>"),
    ("stream_ks2", "nr_stream_kernel<2, false, {}, 2>"),
    ("stream_ks4", "nr_stream_kernel<4, false, {}, 2>"),
    ("stream_ks8", "nr_stream_kernel<8, false, {}, 2>"),
    ("warp", "rw_walk_kernel<false, {}, 2>"),
]


def test_nu_launches_its_instantiation():
    """Every case of every path launches the sampled-nu instantiation of its path: with the
    extras / colouring exactly when it has a covariance transition, and no other likelihood's."""
    import re
    import torch
    from torch.profiler import profile, ProfilerActivity
    eng = engine()
    runs = [(path, case) for path, _ in LAUNCHES for case in CASES]
    for path, case in runs:
        _problem_and_ref(path, case, False)
    eng.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        probe = torch.ones(1024, device=eng.device, dtype=torch.float64) * 3.0
        for path, case in runs:
            _run(eng, path, case, False, False)
        eng.sync()
        torch.cuda.synchronize()
    del probe
    kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    if not kern:
        pytest.skip("the profiler recorded no device events, not even the probe's torch kernel")
    kern.sort(key=lambda e: e.time_range.start)
    names = []
    for e in kern:
        m = re.search(r"((?:nr_tiles|nr_stream|rw_walk)_kernel<[^>]*>)", e.name)
        if m:
            names.append(re.sub(r"\s+", " ", m.group(1)))
    seq = [n for i, n in enumerate(names) if i == 0 or n != names[i - 1]]
    # per_step off, bound off: the extras (tiles, stream) / the colouring (walk) are the
    # covariance transition's alone
    want = [inst.format("true" if CASES[case][5] else "false") for path, inst in LAUNCHES
            for case in CASES]
    want = [n for i, n in enumerate(want) if i == 0 or n != want[i - 1]]
    assert seq == want, seq


# ---- posterior recovery on t_4 data --------------------------------------------------------
BOX = dict(mu=[0., 2.], sigma=[1., 4.], nu=[1., 50.])


def _recovery_data():
    rng = np.random.default_rng(44)
    return 1. + 2. * rng.standard_t(4., 2000)


def _recovery_rvs():
    mu = pb.RV('mu', vtype=float, vset=BOX['mu'])
    sigma = pb.RV('sigma', vtype=float, vset=BOX['sigma'])
    nu = pb.RV('nu', vtype=float, vset=BOX['nu'])
    sigma.set_ufun((np.log, np.exp))
    nu.set_ufun((np.log, np.exp))
    x = pb.RV('x', vtype=float, vset=(-np.inf, np.inf))
    return mu, sigma, nu, x


def _reference_posterior(data, n_nu=240, M=301, S=241):
    """Means and sds of (mu, sigma, nu) from a stack of (mu, sigma) grids of the fixed-nu t
    (pbx_grid_t_logjoint), one per nu of nu.evaluate({n_nu}): uniform in nu's ufun space, as
    the sigma grid is in sigma's, so that every point weighs its log-joint alone -- the walk's
    stationary law, whose box priors carry no Jacobian (rv.py:161-163)."""
    eng = engine()
    mu_rv, sigma_rv, nu_rv, _ = _recovery_rvs()
    nus = np.ravel(nu_rv.evaluate({n_nu}))
    mus = np.linspace(0.5, 1.5, M)
    sgs = np.exp(np.linspace(np.log(1.5), np.log(2.6), S))
    xd, md, sd = dev(eng, data), dev(eng, mus), dev(eng, sgs)
    z = dev(eng, np.zeros(max(M, S)))
    lj = np.stack([host(eng.grid_norm_logjoint(xd, md, sd, z[:M], z[:S],
                                               lik=catalogue.likelihood('t', v))) for v in nus])
    p = np.exp(lj - lj.max())
    p /= p.sum()
    for ax in ((1, 2), (0, 2), (0, 1)):        # nothing of weight at the edges of the stack
        m = p.sum(axis=ax)
        assert max(m[0], m[-1]) <= 1e-7 * m.max()
    out = {}
    for k, v, w in (('mu', mus, p.sum(axis=(0, 2))), ('sigma', sgs, p.sum(axis=(0, 1))),
                    ('nu', nus, p.sum(axis=(1, 2)))):
        m = (w * v).sum()
        out[k] = (m, np.sqrt((w * (v - m) ** 2).sum()))
    return out


def test_nu_posterior_recovery():
    """The issue's model through the public API: 1024 MH chains on t_4 data (mu = 1, sigma = 2,
    N = 2000); the means and sds of mu, sigma and nu agree with the grid stack within 5 Monte
    Carlo standard errors (from the spread of the independent chains), and nu is near 4."""
    data = _recovery_data()
    ref = _reference_posterior(data)
    assert abs(ref['nu'][0] - 4.) < 1.5 and abs(ref['mu'][0] - 1.) < 0.2
    mu, sigma, nu, x = _recovery_rvs()
    paras = mu & sigma & nu
    process = pb.SP(pb.RF(x), paras)
    process.set_prob(scipy.stats.t.logpdf, order={'x': 0, 'nu': 1, 'mu': 'loc', 'sigma': 'scale'},
                     pscale='log')
    paras.set_delta([0.04], scale=True)
    process.set_tran(paras)
    process.set_delta(paras)
    process.set_scores('metropolis')
    sampler = process.sampler({'mu': 1., 'sigma': 2., 'nu': 4.}, {'x': data}, stop=8000,
                              iid=True, joint=True, chains=1024, thin=4, seed=23)
    v = process(process.walk(sampler)).v
    for k in ('mu', 'sigma', 'nu'):
        s = np.asarray(v[k])[:, 250:]                  # [chains, records] after burn-in
        cm = s.mean(axis=1)
        se = cm.std(ddof=1) / np.sqrt(len(cm))
        m, sd = ref[k]
        assert abs(cm.mean() - m) <= 5. * se + 1e-3 * sd, (k, cm.mean(), m, se)
        csd = s.std(axis=1)
        assert abs(s.std() - sd) <= 5. * csd.std(ddof=1) / np.sqrt(len(csd)) + 0.01 * sd, \
            (k, s.std(), sd)


def test_nu_dgei_at_a_scalar_nu_is_the_fixed_nu_grid():
    """SD with nu a model parameter, given nu = 4: the fixed-nu t grid plus nu's prior."""
    eng = engine()
    mu, sigma, nu, x = _recovery_rvs()
    model = pb.SD(pb.RF(x), mu & sigma & nu)
    model.set_prob(scipy.stats.t.logpdf, order={'x': 0, 'nu': 'df', 'mu': 'loc',
                                                 'sigma': 'scale'}, pscale='log')
    data = _recovery_data()[:500]
    joint = model({x: data, 'mu': {64}, 'sigma': {48}, 'nu': 4.}, iid=True, joint=True)
    mus, sgs = np.ravel(joint['mu']), np.ravel(joint['sigma'])
    lpn = -np.log(np.log(50.))
    lpm = np.full(64, -np.log(2.) + lpn)
    lps = np.full(48, -np.log(np.log(4.)))
    want = host(eng.grid_norm_logjoint(dev(eng, data), dev(eng, mus), dev(eng, sgs),
                                       dev(eng, lpm), dev(eng, lps),
                                       lik=catalogue.likelihood('t', 4.)))
    assert relerr(joint.prob, want) <= 1e-15
