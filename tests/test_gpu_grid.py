"""K3/K4 parity (GPU, through the C ABI): discrete grid exact inference against
the golden fixtures (live reference) and the oracles.  fp64, <= 1e-12 relative."""
import numpy as np
import pytest
from conftest import load_golden, relerr
from gpu_util import engine, dev, host
from oracle import np_oracle as o

pytestmark = pytest.mark.gpu
TOL = 1e-12
NNI = o.NEARLY_NEGATIVE_INF


def _priors(M, S):
    return np.full(M, -np.log(20.)), np.full(S, -np.log(np.log(20.) - np.log(5.)))


def _rel_masked(a, b):
    """relative error over the cells both sides did not clamp; clamp masks equal."""
    ca, cb = a == NNI, b == NNI
    assert np.array_equal(ca, cb)
    return relerr(a[~ca], b[~cb])


def _abs_masked(a, b):
    ca, cb = a == NNI, b == NNI
    assert np.array_equal(ca, cb)
    return float(np.abs(a[~ca] - b[~cb]).max())


# The posterior / marginals are DIFFERENCES of log-joints of magnitude |lj| ~ N, so
# they inherit an absolute error |lj|*eps from the summation order of either side
# (SURVEY.md "DGEI conditioning", probe B.8).  The 1e-12 relative bound of the
# log-densities therefore translates into an absolute bound 1e-12 * max|lj| here.


@pytest.mark.parametrize("name", ["dgei_small", "dgei_peaked"])
def test_golden(name):
    eng = engine()
    g = load_golden(name)
    M, S = len(g["mu"]), len(g["sigma"])
    lpm, lps = _priors(M, S)
    lj = eng.grid_norm_logjoint(dev(eng, g["data"]), dev(eng, g["mu"]), dev(eng, g["sigma"]),
                                dev(eng, lpm), dev(eng, lps))
    r = eng.grid_conditionalise(lj)
    eng.sync()
    assert relerr(host(lj), g["joint"]) <= TOL
    atol = TOL * np.abs(g["joint"]).max()
    assert _abs_masked(host(r["post"]), g["posterior"]) <= atol
    assert _abs_masked(host(r["marg_mu"]), g["marg_mu"]) <= atol
    assert _abs_masked(host(r["marg_sigma"]), g["marg_sigma"]) <= atol
    lin = host(eng.exp_logp_(r["post"].clone()))
    eng.sync()
    # linear cells: relative error = absolute error of the log cell
    assert np.abs(lin - g["post_linear"]).max() <= atol * g["post_linear"].max()


@pytest.mark.parametrize("N,M,S", [(1, 3, 5), (1023, 7, 1030), (4097, 33, 257), (20000, 64, 96),
                                   (5, 1, 1), (50, 5, 1024), (50, 6, 2050), (10, 1027, 8),
                                   (20, 600, 1024)])
def test_oracle_ragged(N, M, S):
    """Ragged observation counts (below / across the 1024-obs tile) and grid edges
    that do not fill a CTA tile: single cells, row counts off the 4-row tile, column counts on
    and off the 1024-column block (interior and edge variants of the posterior pass), more
    4-row tiles than resident CTAs."""
    from oracle.c import liboracle as lo
    eng = engine()
    rng = np.random.default_rng(N + M + S)
    data = rng.normal(50., 10., N)
    mu = o.uniform_grid(40, 60, M, True, True)
    sg = np.exp(o.uniform_grid(np.log(5), np.log(20), S, True, True))
    lpm, lps = rng.normal(-3, .1, M), rng.normal(-1, .1, S)
    want = lo.grid_norm_logjoint(data, mu, sg, lpm, lps)
    lj = eng.grid_norm_logjoint(dev(eng, data), dev(eng, mu), dev(eng, sg), dev(eng, lpm),
                                dev(eng, lps))
    r = eng.grid_conditionalise(lj)
    eng.sync()
    assert relerr(host(lj), want) <= TOL
    post = o.grid_conditionalise(want)
    atol = TOL * np.abs(want).max()
    assert _abs_masked(host(r["post"]), post) <= atol
    assert _abs_masked(host(r["marg_mu"]), o.grid_marginal(post, 1)) <= atol
    assert _abs_masked(host(r["marg_sigma"]), o.grid_marginal(post, 0)) <= atol


def test_slab_sharded_two_pass_equals_whole():
    """mu-row slabs (the multi-GPU partitioning) reproduce the whole-grid result:
    max of maxes, sum of sums, summed sigma marginal, concatenated mu marginal."""
    import torch
    eng = engine()
    rng = np.random.default_rng(3)
    N, M, S = 3000, 96, 130
    data = rng.normal(50., 10., N)
    mu = o.uniform_grid(40, 60, M, True, True)
    sg = np.exp(o.uniform_grid(np.log(5), np.log(20), S, True, True))
    lpm, lps = _priors(M, S)
    xd, sd, lpsd = dev(eng, data), dev(eng, sg), dev(eng, lps)
    whole = eng.grid_conditionalise(eng.grid_norm_logjoint(xd, dev(eng, mu), sd, dev(eng, lpm),
                                                          lpsd))
    slabs = [eng.grid_norm_logjoint(xd, dev(eng, mu[a:b]), sd, dev(eng, lpm[a:b]), lpsd)
             for a, b in [(0, 40), (40, 41), (41, 96)]]
    pairs = [eng.grid_max_sumexp(s) for s in slabs]
    gmax = torch.stack([p[0:1] for p in pairs]).max(dim=0).values
    gsum = torch.stack([eng.grid_rescale_sumexp_(p[0:1], gmax, p[1:2]) for p in pairs]).sum(dim=0)
    parts = [eng.grid_posterior2(s, gmax, gsum, marg_log=1) for s in slabs]
    post = torch.cat([p[0] for p in parts])
    mm = torch.cat([p[1] for p in parts])
    ms = eng.log_prob_(torch.stack([p[2] for p in parts]).sum(dim=0))
    eng.sync()
    assert float(gmax) == float(whole["gmax"])
    assert _rel_masked(host(post), host(whole["post"])) <= 1e-13
    assert relerr(host(mm), host(whole["marg_mu"])) <= 1e-13
    assert relerr(host(ms), host(whole["marg_sigma"])) <= 1e-13


def test_full_size_properties():
    """BASELINE config C4 shape at reduced N (4096 x 4096 grid, N = 2000): the
    posterior is normalised, marginals agree with row/column sums of the
    posterior, and a random sample of cells matches the C restatement."""
    from oracle.c import liboracle as lo
    eng = engine()
    rng = np.random.default_rng(7)
    N, M, S = 2000, 4096, 4096
    data = rng.normal(50., 10., N)
    mu = o.uniform_grid(40, 60, M, True, True)
    sg = np.exp(o.uniform_grid(np.log(5), np.log(20), S, True, True))
    lpm, lps = _priors(M, S)
    lj = eng.grid_norm_logjoint(dev(eng, data), dev(eng, mu), dev(eng, sg), dev(eng, lpm),
                                dev(eng, lps))
    r = eng.grid_conditionalise(lj)
    eng.sync()
    ljh = host(lj)
    rows = rng.choice(M, 6, replace=False); cols = rng.choice(S, 7, replace=False)
    want = lo.grid_norm_logjoint(data, mu[rows], sg[cols], lpm[rows], lps[cols])
    assert relerr(ljh[np.ix_(rows, cols)], want) <= TOL
    post = host(r["post"])
    lin = np.where(post == NNI, 0.0, np.exp(np.maximum(post, -745.)))
    assert abs(lin.sum() - 1.0) <= 1e-10
    mm, ms = host(r["marg_mu"]), host(r["marg_sigma"])
    ok = mm > -700
    assert relerr(np.exp(mm[ok]), lin.sum(axis=1)[ok]) <= 1e-10
    ok = ms > -700
    assert relerr(np.exp(ms[ok]), lin.sum(axis=0)[ok]) <= 1e-10
    assert np.unravel_index(np.argmax(ljh), ljh.shape) == \
        np.unravel_index(np.argmax(post), post.shape)


def test_clamped_exp_edge_cases_through_the_two_pass_path():
    """The branch-free table exp of the two K4 passes over its whole range: entries far below
    the maximum (subnormal / underflowing exp), the reference's clamp decision q < tiny ->
    -1.797e308, and the marginalise path (no max shift) with arguments up to and beyond
    log(huge) (pscales.py:44-65)."""
    import torch
    eng = engine()
    tail = np.array([0., -1., -37.25, -600.5, -650., -699., -700.5, -701., -707., -708.3,
                     -708.39, -708.4, -720., -744.4, -745.2, -760., -1e4, NNI])
    rng = np.random.default_rng(5)
    lj = np.concatenate([tail, -rng.uniform(0., 760., 4096 - len(tail))]).reshape(64, 64) - 3e5
    r = eng.grid_conditionalise(dev(eng, lj))
    eng.sync()
    want = o.grid_conditionalise(lj)
    post = host(r["post"])
    clamp = want == NNI
    assert np.array_equal(post == NNI, clamp)
    assert np.abs(post[~clamp] - want[~clamp]).max() <= 1e-12 * 3e5
    wm = o.grid_marginal(want, axis=1)
    ok = wm > -690
    assert np.abs(host(r["marg_mu"])[ok] - wm[ok]).max() <= 1e-10
    # marginalise path: exp_logp without a shift, incl. overflow clamp and subnormal results
    big = np.array([[700., 705.5, 709.7, 709.9, 1e4], [-800., -744., -710., -50., 0.]])
    zero = torch.zeros(1, dtype=torch.float64, device=eng.device)
    one = torch.ones(1, dtype=torch.float64, device=eng.device)
    _, rows, cols = eng.grid_posterior2(dev(eng, big), zero, one, want_post=False, marg_log=4)
    eng.sync()
    lin = o.exp_logp(big)
    assert relerr(host(cols), lin.sum(axis=0)) <= 1e-12       # 1.8e308 clamps included
    assert host(rows)[0] == np.inf and abs(host(rows)[1] - lin[1].sum()) <= 1e-15
    # a row of tiny values only: subnormal results survive (one rounded multiply)
    small = np.array([[-800., -744.5, -720., -710., -705.]])
    _, r2, c2 = eng.grid_posterior2(dev(eng, small), zero, one, want_post=False, marg_log=4)
    eng.sync()
    want = o.exp_logp(small)
    assert np.abs(host(c2) - want[0]).max() <= 1e-15 * want.max() + 1e-323
