"""K6 parity (GPU, through the C ABI): PD post-processing -- argsort / gather,
cumulative probability / digitize, expectation sums -- and the box sampler of
ordinary Monte Carlo random sampling, against the numpy oracle and the fixture
generated from the live reference (examples/omc/omc_rs_sp_norm1d.py).
Index work is bit-exact; fp64 sums <= 1e-12 relative."""
import numpy as np
import pytest
import scipy.stats
from conftest import load_golden, relerr
from gpu_util import engine, dev, host
from oracle import np_oracle as o
from oracle import philox

pytestmark = pytest.mark.gpu
TOL = 1e-12


def _keys(kind, n, rng):
    if kind == "normal":
        return rng.standard_normal(n)
    if kind == "unit":                      # one exponent: the top digit passes are skipped
        return 1.0 + rng.random(n)
    if kind == "ties":                      # heavy duplication: stability matters
        return rng.integers(-5, 6, n).astype(float)
    if kind == "wide":                      # every magnitude, both signs, infinities
        k = rng.standard_normal(n) * 10.0 ** rng.integers(-300, 300, n)
        k[rng.integers(0, n, max(1, n // 50))] = np.inf
        k[rng.integers(0, n, max(1, n // 50))] = -np.inf
        return k
    if kind == "const":
        return np.full(n, 3.25)
    raise ValueError(kind)


@pytest.mark.parametrize("kind", ["normal", "unit", "ties", "wide", "const"])
@pytest.mark.parametrize("n", [1, 2, 33, 4095, 4096, 4097, 100003, (1 << 21) + 17])
def test_argsort_matches_stable_numpy(kind, n):
    eng = engine()
    rng = np.random.default_rng(n * 7 + len(kind))
    k = _keys(kind, n, rng)
    order, ks = eng.argsort(dev(eng, k), want_keys=True)
    eng.sync()
    want = o.pd_sorted_order(k)
    assert np.array_equal(host(order).astype(np.int64), want)       # bit-exact, stable
    assert np.array_equal(host(ks), k[want])


def test_argsort_order_only_and_empty():
    eng = engine()
    k = np.random.default_rng(3).standard_normal(5000)
    order = eng.argsort(dev(eng, k))
    assert np.array_equal(host(order), o.pd_sorted_order(k))
    import torch
    e = eng.argsort(torch.empty(0, dtype=torch.float64, device=eng.device))
    assert e.numel() == 0


def test_argsort_signed_zero_and_nan_last():
    eng = engine()
    k = np.array([0.0, -0.0, 1.0, np.nan, -1.0, 0.0, -0.0, -np.inf, np.inf])
    order, ks = eng.argsort(dev(eng, k), want_keys=True)
    ks = host(ks)
    assert np.isnan(ks[-1]) and ks[-2] == np.inf and ks[0] == -np.inf
    assert np.array_equal(ks[:-1], np.sort(k)[:-1])                  # -0.0 == 0.0 by value
    assert np.array_equal(np.signbit(ks[2:6]), [True, True, False, False])   # -0 before +0
    assert sorted(host(order).tolist()) == list(range(len(k)))


def test_argsort_bad_arguments():
    import torch
    from probayes_b200 import _lib
    eng = engine()
    k = dev(eng, np.arange(10.))
    out = torch.empty(10, dtype=torch.int32, device=eng.device)
    with pytest.raises(_lib.PbxError, match="workspace"):
        _lib.check(eng.lib.pbx_argsort_f64(eng.ctx, k.data_ptr(), 10, out.data_ptr(), 0, 0, 0))
    with pytest.raises(_lib.PbxError, match="2\\^31"):
        _lib.check(eng.lib.pbx_argsort_f64(eng.ctx, k.data_ptr(), 1 << 31, out.data_ptr(), 0, 0, 0))


def test_gather_and_take_axis():
    eng = engine()
    rng = np.random.default_rng(5)
    src = rng.standard_normal(70001)
    perm = rng.permutation(70001).astype(np.int32)
    import torch
    got = eng.gather(dev(eng, src), torch.from_numpy(perm).to(eng.device))
    assert np.array_equal(host(got), src[perm])
    a = rng.standard_normal((37, 1001))
    p0 = rng.permutation(37).astype(np.int32)
    p1 = rng.permutation(1001).astype(np.int32)
    g0 = eng.take_axis(dev(eng, a), torch.from_numpy(p0).to(eng.device), 0)
    g1 = eng.take_axis(dev(eng, a), torch.from_numpy(p1).to(eng.device), 1)
    assert np.array_equal(host(g0), a[p0]) and np.array_equal(host(g1), a[:, p1])


@pytest.mark.parametrize("log_pscale", [False, True])
@pytest.mark.parametrize("n", [1, 7, 2047, 2048, 2049, 300001, (1 << 22) + 5])
def test_cumprob_and_digitize(n, log_pscale):
    eng = engine()
    rng = np.random.default_rng(n + int(log_pscale))
    p = rng.random(n) ** 3
    if log_pscale:
        p = np.log(p + 1e-300) - 250.0          # tiny linear values, still above the clamp
        p[rng.integers(0, n, 1 + n // 100)] = o.NEARLY_NEGATIVE_INF     # clamped cells -> 0
    cum, total = eng.cumprob(dev(eng, p), log_pscale)
    eng.sync()
    want, rav = o.pd_cumprob(p, log_pscale)
    c = host(cum)
    assert relerr(c, want) <= TOL
    assert relerr(host(total), np.sum(rav)) <= TOL
    assert np.all(np.diff(c) >= 0.0)             # truly non-decreasing (np.digitize needs it)
    assert c[-1] == (1.0 if np.sum(rav) >= o.NEARLY_POSITIVE_ZERO else 0.0)
    cum2, _ = eng.cumprob(dev(eng, p), log_pscale)
    assert np.array_equal(host(cum2), c)         # bit-reproducible
    qs = np.array([0.0, 1e-9, 0.025, 0.5, 0.975, 1.0 - 1e-12, 1.0, 1.5])
    idx = host(eng.digitize(cum, qs))
    assert np.array_equal(idx, o.pd_quantile_index(c, qs))          # bit-exact on the same cum


def test_cumprob_in_place():
    eng = engine()
    p = np.random.default_rng(9).random(50000)
    t = dev(eng, p)
    cum, _ = eng.cumprob(t, False, out=t)
    assert relerr(host(cum), o.pd_cumprob(p, False)[0]) <= TOL


@pytest.mark.parametrize("shape", [(1, 100000), (64, 81), (513, 2050), (3000, 1)])
@pytest.mark.parametrize("log_pscale", [False, True])
def test_expectation_sums(shape, log_pscale):
    eng = engine()
    rng = np.random.default_rng(shape[0] + shape[1])
    rows, cols = shape
    p = rng.random(shape)
    if log_pscale:
        p = np.log(p) - 30.0
    rv = rng.standard_normal((2, rows))
    cv = rng.standard_normal((3, cols)) + 2.0
    got = host(eng.expectation_sums(dev(eng, p), log_pscale, dev(eng, rv), dev(eng, cv)))
    tot, r, c = o.pd_expectation(p, log_pscale, rv, cv)
    lin = o.to_linear(p, log_pscale)
    # absolute bound from the size of the summed terms (cancellation in sum p*v)
    scale = np.array([tot] + [np.sum(lin * np.abs(v)[:, None]) for v in rv] +
                     [np.sum(lin * np.abs(v)[None, :]) for v in cv])
    assert np.all(np.abs(got - np.array([tot] + r + c)) <= TOL * scale)
    again = host(eng.expectation_sums(dev(eng, p), log_pscale, dev(eng, rv), dev(eng, cv)))
    assert np.array_equal(again, got)
    only = host(eng.expectation_sums(dev(eng, p), log_pscale, None, dev(eng, cv[:1])))
    assert abs(only[0] - tot) <= TOL * tot and abs(only[1] - c[0]) <= TOL * scale[3]


# ---- ordinary Monte Carlo random sampling -----------------------------------------------
LIMS = np.array([[40., 60.], [5., 20.]])
LOGU = np.array([0, 1])


def test_box_sample_injected_matches_reference():
    eng = engine()
    g = load_golden("omc_rs_norm1d")
    th = host(eng.box_sample(LIMS, LOGU, len(g["runif"]), inj_unif=dev(eng, g["runif"])))
    assert np.array_equal(th[0], g["mu"])                      # affine map: bit-exact
    assert relerr(th[1], g["sigma"]) <= 4e-16                  # exp(): within 2 ulp of libm


def test_box_sample_philox_replay():
    eng = engine()
    T, P = 5000, 3
    lims = np.array([[-6., 6.], [0.001, 10.], [2., 3.]])
    logu = np.array([0, 1, 0])
    th = host(eng.box_sample(lims, logu, T, seed=77, sample0=1234))
    r = philox.uniforms(77, T, 1, P, step0=1234)[:, 0, :]
    want = o.box_sample(lims, logu, r)
    assert np.array_equal(th[0], want[0]) and np.array_equal(th[2], want[2])
    assert relerr(th[1], want[1]) <= 4e-16
    assert np.all((th > lims[:, :1]) & (th < lims[:, 1:]))


def test_box_sample_needs_finite_limits():
    from probayes_b200._lib import PbxError
    eng = engine()
    with pytest.raises(PbxError, match="finite"):
        eng.box_sample(np.array([[-np.inf, 1.]]), np.array([0]), 10)


def _omc_process(pb, data):
    mu = pb.RV('mu', vtype=float, vset=(40, 60))
    sigma = pb.RV('sigma', vtype=float, vset=(5, 20.))
    x = pb.RV('x', vtype=float, vset=[-np.inf, np.inf])
    sigma.set_ufun((np.log, np.exp))
    process = pb.SP(pb.RF(x), pb.RF(mu, sigma))
    process.set_prob(scipy.stats.norm.logpdf,
                     order={'x': 0, 'mu': 'loc', 'sigma': 'scale'}, pscale='log')
    return process


def test_api_omc_random_sampling_golden():
    """examples/omc/omc_rs_sp_norm1d.py through the public API with the reference's
    prior draws injected: per-step PDs, summary, rescaled / sorted / quantile /
    expectation against the live-reference fixture."""
    engine()
    import probayes_b200 as pb
    g = load_golden("omc_rs_norm1d")
    T = len(g["runif"])
    process = _omc_process(pb, g["data"])
    sampler = process.sampler({'mu': {0}, 'sigma': {0}, 'x': g["data"]}, iid=True, joint=True,
                              stop=T, inj_unif=g["runif"])
    samples = [s for s in sampler]
    assert len(samples) == T
    first = str(g["first_name"])                 # "mu=55.83...,sigma=19.06...,x={60}"
    assert samples[0].name.split(',')[0] == first.split(',')[0]
    assert samples[0].name.split(',')[2] == first.split(',')[2]
    assert abs(samples[0].prob - g["logp"][0]) <= TOL * abs(g["logp"][0])
    summary = process(samples)
    assert summary.name == str(g["name"]) and summary.shape == [T] and summary.pscale == 0j
    assert summary.prob_device is not None
    assert np.array_equal(summary['mu'], g["mu"])
    assert relerr(summary['sigma'], g["sigma"]) <= 4e-16
    assert relerr(summary.prob, g["logp"]) <= TOL
    inference = summary.rescaled()
    assert inference.prob_device is not None
    assert relerr(inference.prob, g["lin"]) <= 1e-11            # exp amplifies |logp| * eps
    mu_sort = inference.sorted('mu')
    assert mu_sort.prob_device is not None
    assert np.array_equal(mu_sort['mu'], g["mu_sorted"])
    assert relerr(mu_sort['sigma'], g["mu_sorted_sigma"]) <= 4e-16
    assert relerr(mu_sort.prob, g["mu_sorted_prob"]) <= 1e-11
    qs = g["qs"].tolist()
    q = mu_sort.quantile(qs)
    assert relerr([v['mu'] for v in q], g["q_mu"]) <= 1e-10
    assert q[0]['sigma'] == {T} and q[0]['x'] == {T * len(g["data"])}   # unsorted -> {size}
    assert abs(mu_sort.quantile(0.5)['mu'] - g["med_mu"]) <= 1e-10 * g["med_mu"]
    sig_sort = inference.sorted('sigma')
    assert relerr(sig_sort['sigma'], g["sigma_sorted"]) <= 4e-16
    assert relerr([v['sigma'] for v in sig_sort.quantile(qs)], g["q_sigma"]) <= 1e-10
    e = inference.expectation()
    assert relerr([e['mu'], e['sigma']], g["expt"]) <= 1e-10
    e2 = inference.expectation(['mu', 'sigma'], exponent=2)
    assert relerr([e2['mu'], e2['sigma']], g["expt2"]) <= 1e-10
    # straight from the log-pscale summary (rescale folded into the kernels)
    e = summary.expectation()
    assert relerr([e['mu'], e['sigma']], g["expt"]) <= 1e-10


def test_api_omc_large_native_rng():
    """2e5 samples with the Philox stream: the device summary against the oracle fed
    with the replayed uniforms; the posterior mean must sit near the data's."""
    eng = engine()
    import probayes_b200 as pb
    rng = np.random.default_rng(8)
    data = rng.normal(50., 10., size=300)
    T = 200000
    process = _omc_process(pb, data)
    sampler = process.sampler({'mu': {0}, 'sigma': {0}, 'x': data}, iid=True, joint=True,
                              stop=T, seed=5)
    walk = process.walk(sampler)
    summary = process(walk)
    r = philox.uniforms(5, T, 1, 2)[:, 0, :]
    th = o.box_sample(LIMS, LOGU, r)
    assert np.array_equal(summary['mu'], th[0]) and relerr(summary['sigma'], th[1]) <= 4e-16
    lj = o.normreg_logjoint(np.stack([summary['mu'], summary['sigma']], 1)[:2000], None, data,
                            LIMS, np.ones((2, 2), int), LOGU, has_slope=False)
    assert relerr(summary.prob[:2000], lj) <= TOL
    post = summary.conditionalise('x')
    assert post.prob_device is not None
    srt = post.sorted('mu')
    med = srt.quantile(0.5)['mu']
    lin = o.exp_logp(summary.prob - summary.prob.max())
    order = np.argsort(summary['mu'], kind='stable')
    want = o.pd_quantile_1d(summary['mu'][order], lin[order], False, [0.5])[0]
    assert abs(med - want) <= 1e-9 * want
    e = post.expectation()
    assert abs(e['mu'] - np.sum(lin * summary['mu']) / np.sum(lin)) <= 1e-9 * e['mu']
    assert abs(e['mu'] - data.mean()) < 0.5


def test_omc_sharded_single_rank_matches_oracle():
    """dist.omc_sharded outside a process group: the Philox draws, the log posterior
    normalised over all samples (an odd count, off every CTA tile) and the posterior means
    against the oracle on the replayed stream."""
    from probayes_b200 import dist as pd_
    eng = engine()
    data = np.random.default_rng(4).normal(50., 10., 300)
    T, seed, ex = 100003, 21, np.ones((2, 2), int)
    r = pd_.omc_sharded(eng, data, LIMS, ex, LOGU, T, seed=seed)
    eng.sync()
    assert r["samples"] == (0, T)
    th = o.box_sample(LIMS, LOGU, philox.uniforms(seed, T, 1, 2)[:, 0, :])
    got = host(r["theta"])
    assert np.array_equal(got[0], th[0]) and relerr(got[1], th[1]) <= 4e-16
    lj = o.normreg_logjoint(th.T, None, data, LIMS, ex, LOGU, has_slope=False)
    want = o.grid_conditionalise(lj)
    post = host(r["logpost"])
    clamp = want == o.NEARLY_NEGATIVE_INF
    assert np.array_equal(post == o.NEARLY_NEGATIVE_INF, clamp) and not clamp.all()
    assert np.abs(post[~clamp] - want[~clamp]).max() <= TOL * np.abs(lj).max()
    lin = o.exp_logp(want)
    assert relerr(r["expectation"], (lin * th).sum(axis=1) / lin.sum()) <= 1e-10


def test_api_dgei_posterior_postprocessing():
    """The steps right after the DGEI posterior (dgei_norm1d_improved.py:38-46) on the
    device-backed grid PD: expectation over both axes, quantiles of the marginals and
    of the ravelled 2-D posterior, sorted() along an axis -- against the fixture."""
    engine()
    import probayes_b200 as pb
    g = load_golden("dgei_small")
    mu = pb.RV('mu', vtype=float, vset=(40, 60))
    sigma = pb.RV('sigma', vtype=float, vset=(5, 20.))
    x = pb.RV('x', vtype=float, vset={-np.inf, np.inf})
    sigma.set_ufun((np.log, np.exp))
    model = pb.SD(pb.RF(x), pb.RF(mu, sigma))
    model.set_prob(scipy.stats.norm.logpdf, order={'x': 0, 'mu': 'loc', 'sigma': 'scale'},
                   pscale='log')
    M, S = len(g["mu"]), len(g["sigma"])
    joint = model({x: g["data"], 'mu': {M}, 'sigma': {S}}, iid=True, joint=True)
    posterior = joint.conditionalise('x')
    assert posterior.prob_device is not None
    e = posterior.expectation()
    assert abs(e['mu'] - g["expt_mu"]) <= 1e-10 * g["expt_mu"]
    assert abs(e['sigma'] - g["expt_sigma"]) <= 1e-10 * g["expt_sigma"]
    pm, ps = posterior.marginal('mu'), posterior.marginal('sigma')
    assert pm.prob_device is not None
    assert abs(pm.quantile()['mu'] - g["med_mu"]) <= 1e-10 * g["med_mu"]
    assert abs(ps.quantile()['sigma'] - g["med_sigma"]) <= 1e-10 * g["med_sigma"]
    assert relerr([q['mu'] for q in pm.quantile([0.025, 0.5, 0.975])], g["q3_mu"]) <= 1e-10
    # 2-D: ravelled cumulative probability; mu (axis 0) takes the cell value, sigma (last
    # axis) is interpolated -- compared with the same arithmetic on the fixture's posterior
    q2 = posterior.quantile(0.5)
    lin = o.exp_logp(g["posterior"])
    cum, rav = o.pd_cumprob(lin, False)
    i = int(o.pd_quantile_index(cum, 0.5)[0])
    r, c = np.unravel_index(i, lin.shape)
    assert q2['mu'] == g["mu"][r]
    assert g["sigma"][c] <= q2['sigma'] <= g["sigma"][min(c + 1, S - 1)]
    # sorted along sigma with a descending key: columns reverse
    rev = pb.PD(posterior.name, collections_copy(posterior, 'sigma', g["sigma"][::-1].copy()),
                dims=posterior.dims, prob=posterior.prob_device, pscale=posterior.pscale)
    srt = rev.sorted('sigma')
    assert np.array_equal(srt['sigma'], g["sigma"])
    assert np.array_equal(srt.prob, posterior.prob[:, ::-1])


def collections_copy(pd, key, newval):
    import collections
    vals = collections.OrderedDict(pd)
    vals[key] = newval
    return vals


# ---- joint-product / division algebra -------------------------------------------------------
@pytest.mark.parametrize("op", ["mul", "div"])
@pytest.mark.parametrize("a_shape,b_shape", [
    ((37, 53), (37, 53)), ((37, 1), (1, 53)), ((37, 53), (1, 53)), ((37, 53), (37, 1)),
    ((1, 7000), (1, 7000)), ((1, 1), (300, 200)), ((1300, 1), (1300, 1))])
@pytest.mark.parametrize("a_log,b_log", [(False, False), (True, True), (False, True), (True, False)])
def test_pd_binary_kernel(op, a_shape, b_shape, a_log, b_log):
    eng = engine()
    rng = np.random.default_rng(a_shape[0] * 31 + b_shape[1] + 2 * a_log + b_log)

    def draw(shape, lg):
        p = rng.random(shape) + 0.01
        p.flat[rng.integers(0, p.size, max(1, p.size // 20))] = 0.0       # clamp edge: log(0)
        if not lg:
            return p
        with np.errstate(divide="ignore"):
            l = np.log(p) - 300.0 * rng.random(shape)
        l[~np.isfinite(l)] = o.NEARLY_NEGATIVE_INF
        return l
    a, b = draw(a_shape, a_log), draw(b_shape, b_log)
    if op == "mul":
        want, out_log = o.pd_product(a, a_log, b, b_log)
    else:
        want, out_log = o.pd_divide(a, a_log, b, b_log), a_log
    got = host(eng.pd_binary(op, dev(eng, a), a_log, dev(eng, b), b_log, out_log))
    want = np.broadcast_to(want, got.shape)
    # clamped cells (-1.797e308) and the -inf two of them add up to (as in numpy) match
    # exactly; everything else to 1e-12
    special = (want == o.NEARLY_NEGATIVE_INF) | np.isneginf(want)
    assert np.array_equal(got[special], want[special])
    assert np.all(np.isfinite(got[~special]))
    assert relerr(got[~special], want[~special]) <= TOL


def test_pd_binary_rejects_bad_shapes():
    from probayes_b200 import _lib
    eng = engine()
    a, b = dev(eng, np.ones((3, 4))), dev(eng, np.ones((2, 4)))
    out = eng.empty(3, 4)
    with pytest.raises(_lib.PbxError, match="rows or 1"):
        _lib.check(eng.lib.pbx_pd_binary_f64(eng.ctx, 0, a.data_ptr(), 3, 4, 0, b.data_ptr(), 2, 4,
                                             0, 3, 4, 0, out.data_ptr()))
    with pytest.raises(_lib.PbxError, match="log pscale iff"):
        _lib.check(eng.lib.pbx_pd_binary_f64(eng.ctx, 0, a.data_ptr(), 3, 4, 1, a.data_ptr(), 3, 4,
                                             0, 3, 4, 0, out.data_ptr()))


def test_api_pd_algebra_golden():
    """prior * likelihood, joint / evidence and joint / p(mu, x) with device-backed PDs
    against the live-reference fixture (pd.py:564-615)."""
    engine()
    import probayes_b200 as pb
    g = load_golden("pd_algebra")
    names = [str(n) for n in g["names"]]
    M, S = len(g["mu"]), len(g["sigma"])
    mu = pb.RV('mu', vtype=float, vset=(40, 60))
    sigma = pb.RV('sigma', vtype=float, vset=(5, 20.))
    x = pb.RV('x', vtype=float, vset={-np.inf, np.inf})
    sigma.set_ufun((np.log, np.exp))
    paras = pb.RF(mu, sigma)
    model = pb.SD(pb.RF(x), paras)
    model.set_prob(scipy.stats.norm.logpdf, order={'x': 0, 'mu': 'loc', 'sigma': 'scale'},
                   pscale='log')
    grid = {'mu': {M}, 'sigma': {S}}
    joint = model({x: g["data"], **grid}, iid=True, joint=True)
    like = model({x: g["data"], **grid}, iid=True, joint=False)
    assert like.name == names[3] and like.prob_device is not None
    assert relerr(like.prob, g["like"]) <= TOL
    prior = paras(dict(grid))
    j2 = prior * like
    assert j2.name == names[4] and j2.prob_device is not None and j2.pscale == 0j
    assert relerr(j2.prob, g["prior_like"]) <= TOL and relerr(joint.prob, g["joint"]) <= TOL
    ev = joint.marginal('x')
    assert ev.name == names[5] and abs(float(ev.prob) - g["evidence"]) <= 1e-11 * abs(g["evidence"])
    post = joint / ev
    assert post.name == names[6] and post.prob_device is not None
    assert np.abs(post.prob - g["post"]).max() <= 1e-12 * np.abs(g["joint"]).max()
    mm = joint.marginal(['mu', 'x'])
    assert mm.name == names[7] and relerr(mm.prob, g["marg_mu_x"]) <= 1e-11
    pc = joint / mm
    assert pc.name == names[8]
    assert np.abs(pc.prob - g["cond_sigma"]).max() <= 1e-12 * np.abs(g["joint"]).max()


def _dgei_model():
    import probayes_b200 as pb
    mu = pb.RV('mu', vtype=float, vset=(40, 60))
    sigma = pb.RV('sigma', vtype=float, vset=(5, 20.))
    x = pb.RV('x', vtype=float, vset={-np.inf, np.inf})
    sigma.set_ufun((np.log, np.exp))
    model = pb.SD(pb.RF(x), pb.RF(mu, sigma))
    model.set_prob(scipy.stats.norm.logpdf, order={'x': 0, 'mu': 'loc', 'sigma': 'scale'},
                   pscale='log')
    return model, x


def test_api_conditionalise_on_array_keys_golden():
    """PD.conditionalise on array-valued keys (pd.py:214-295) with device-backed PDs, log
    and linear pscale, against the live-reference fixture: values, names, axis moves."""
    engine()
    g = load_golden("pd_cond_array")
    names = [str(n) for n in g["names"]]
    M, S = len(g["mu"]), len(g["sigma"])
    model, x = _dgei_model()
    joint = model({x: g["data"], 'mu': {M}, 'sigma': {S}}, iid=True, joint=True)
    atol = 1e-12 * np.abs(g["joint"]).max()
    cases = [('sigma', "c_sig"), ('mu', "c_mu"), (['sigma', 'x'], "c_sx")]
    for i, (keys, k) in enumerate(cases):
        c = joint.conditionalise(keys)
        assert c.prob_device is not None and c.name == names[i]
        assert [c.dims['mu'], c.dims['sigma']] == list(g["dims"][i])
        assert np.abs(c.prob - g[k]).max() <= atol
    c_mu = joint.conditionalise('mu')
    assert np.shape(c_mu['mu']) == tuple(g["shapes"][0])
    assert np.shape(c_mu['sigma']) == tuple(g["shapes"][1])
    lin = joint.conditionalise('x').rescaled()
    assert lin.prob_device is not None and lin.pscale == 1.
    assert np.abs(lin.prob - g["lin"]).max() <= atol * g["lin"].max()
    for i, (keys, k) in enumerate([('sigma', "l_sig"), ('mu', "l_mu")]):
        c = lin.conditionalise(keys)
        assert c.prob_device is not None and c.name == names[3 + i]
        assert [c.dims['mu'], c.dims['sigma']] == list(g["dims"][3 + i])
        assert np.abs(c.prob - g[k]).max() <= atol * g[k].max()


def test_linear_pscale_device_pds_stay_on_the_device():
    """A device-backed PD in LINEAR pscale (after .rescaled()) is normalised and
    marginalised by the linear-pscale kernel variants -- no host copy -- with the values
    numpy gives on the same arrays; other pscales raise instead of falling back."""
    eng = engine()
    import probayes_b200 as pb
    rng = np.random.default_rng(3)
    data = rng.normal(50., 10., 30)
    model, x = _dgei_model()
    joint = model({x: data, 'mu': {37}, 'sigma': {29}}, iid=True, joint=True)
    lin = joint.rescaled()                               # un-normalised linear joint
    assert lin.prob_device is not None and lin._prob is None
    post = lin.conditionalise('x')
    assert post.prob_device is not None and lin._prob is None and post.pscale == 1.
    p = np.exp(joint.prob)
    want = p / p.sum()
    assert relerr(post.prob, want) <= 1e-12
    mm = post.marginal('mu')
    ms = post.marginal('sigma')
    assert mm.prob_device is not None
    assert relerr(np.ravel(mm.prob), want.sum(axis=1)) <= 1e-12
    assert relerr(np.ravel(ms.prob), want.sum(axis=0)) <= 1e-12
    tot = lin.marginalise(['mu', 'sigma'])
    assert abs(float(tot.prob) - p.sum()) <= 1e-12 * p.sum()
    # log-pscale twin: identical normalised values
    lpost = joint.conditionalise('x')
    assert np.abs(np.exp(lpost.prob) - want).max() <= 1e-12 * want.max()
    odd = pb.PD(joint.name, dict(joint), dims=joint.dims, prob=joint.prob_device, pscale=2.0)
    with pytest.raises(NotImplementedError):
        odd.conditionalise('x')
    with pytest.raises(NotImplementedError):
        odd.marginalise('mu')


@pytest.mark.parametrize("shape", [(1,), (1000,), (5000,), (37, 29), (3, 5000)])
def test_full_marginalise_log_pscale_matches_oracle(shape):
    """PD.marginalise over every array axis of a log-pscale device PD (1-D and 2-D, one and
    several 1024-column blocks): log_prob(sum exp_logp(p)) without a max shift, against the
    oracle.  Ordinary values; every term underflowing (-> -1.797e308); a subnormal total;
    subnormal terms with a normal total; one term above log(huge) (clamped to huge); two of
    them (the sum overflows -> inf)."""
    eng = engine()
    import probayes_b200 as pb
    n = int(np.prod(shape))
    rng = np.random.default_rng(n)
    vals = {k: np.arange(m, dtype=float) for k, m in zip("xy", shape)}
    name = ",".join(vals)
    cases = {"ordinary": rng.normal(-3., 2., n),
             "underflow": np.concatenate([[o.NEARLY_NEGATIVE_INF, -np.inf],
                                          rng.uniform(-3000., -746., n)])[:n],
             "subnormal_total": rng.uniform(-745., -720., n),
             "subnormal_terms": rng.uniform(-712., -709.5, n),
             "huge_term": np.concatenate([[1e4], rng.normal(-3., 2., n)])[:n]}
    if n > 1:
        cases["overflow"] = np.concatenate([[709.9, 1e4], rng.normal(-3., 2., n)])[:n]
    for case, p in cases.items():
        p = rng.permutation(p)
        pd = pb.PD(name, dict(vals), prob=dev(eng, p.reshape(shape)), pscale='log')
        got = float(pd.marginalise(list(vals)).prob)
        with np.errstate(over='ignore'):
            want = float(o.log_prob(o.exp_logp(p).sum()))
        if case in ("underflow", "subnormal_total"):
            assert want == o.NEARLY_NEGATIVE_INF, case
        if case == "overflow":
            assert want == np.inf, case
        assert got == want or abs(got - want) <= 1e-13, (case, got, want)


# ---- full-size properties (no CPU oracle at these sizes) --------------------------------------
def test_argsort_full_size_properties():
    """2^26 keys: the result is sorted, is a permutation, is stable for ties, and sorting
    the sorted keys again is the identity (size-independent properties of PD.sorted)."""
    import torch
    eng = engine()
    n = 1 << 26
    g = torch.Generator(device=eng.device).manual_seed(7)
    keys = torch.randn(n, dtype=torch.float64, device=eng.device, generator=g)
    keys[::3] = torch.round(keys[::3]) + 0.0                # a third of the keys are heavy ties
    # (+ 0.0 turns round()'s -0.0 into +0.0: the sort orders -0.0 before +0.0, == does not)
    order, ks = eng.argsort(keys, want_keys=True)
    assert bool((ks[1:] >= ks[:-1]).all())                  # sorted
    assert bool(torch.equal(ks, keys[order.long()]))        # consistent with the order
    seen = torch.zeros(n, dtype=torch.int32, device=eng.device)
    seen.index_add_(0, order.long(), torch.ones(n, dtype=torch.int32, device=eng.device))
    assert int(seen.min()) == 1 and int(seen.max()) == 1    # a permutation
    ties = ks[1:] == ks[:-1]
    assert bool((order[1:][ties] > order[:-1][ties]).all()) # stable: input order among equals
    order2, ks2 = eng.argsort(ks, want_keys=True)
    assert bool(torch.equal(ks2, ks))
    assert bool(torch.equal(order2, torch.arange(n, dtype=torch.int32, device=eng.device)))


def test_cumprob_and_expectation_full_size_properties():
    """2^26 cells: cum is non-decreasing, ends at exactly 1, its increments are the
    normalised cells; expectation of a constant is the constant, and linear in the values."""
    import torch
    eng = engine()
    n = 1 << 26
    g = torch.Generator(device=eng.device).manual_seed(11)
    p = torch.rand(n, dtype=torch.float64, device=eng.device, generator=g)
    cum, total = eng.cumprob(p, False)
    assert bool((cum[1:] >= cum[:-1]).all()) and float(cum[-1]) == 1.0
    assert abs(float(total) - float(p.sum())) <= 1e-12 * float(total)
    inc = cum[1:] - cum[:-1]
    assert float((inc - p[1:] / total).abs().max()) <= 5e-15         # a few ulp of cum ~ 1 (increments ~ 1e-8)
    v = torch.rand(n, dtype=torch.float64, device=eng.device, generator=g)
    vals = torch.stack([torch.full_like(v, 3.25), v, 2.0 * v - 1.0])
    s = eng.expectation_sums(p, False, None, vals).cpu().numpy()
    e = s[1:] / s[0]
    assert abs(e[0] - 3.25) <= 1e-12 and abs(e[2] - (2.0 * e[1] - 1.0)) <= 1e-12
    lp = torch.log(p) - 500.0                                # same weights in log pscale
    s2 = eng.expectation_sums(lp, True, None, vals).cpu().numpy()
    assert np.abs(s2[1:] / s2[0] - e).max() <= 1e-11
