"""Student-t and Cauchy likelihoods on the host: the catalogue's spellings and refusals, the
per-observation constant, the engine's ABI struct and export, and the oracle's sums."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest
import scipy.stats

import probayes_b200 as pb
from probayes_b200 import _lib, catalogue
import studentt_oracle as to

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORDER = {'x': 0, 'mu': 'loc', 'sigma': 'scale'}


def _mu_sigma_sp():
    mu = pb.RV('mu', vtype=float, vset=(40, 60), pscale='log')
    sigma = pb.RV('sigma', vtype=float, vset=(5, 20.), pscale='log')
    x = pb.RV('x', vtype=float, vset=(-np.inf, np.inf))
    return pb.SP(pb.RF(x), pb.RF(mu, sigma))


def _spec(sp):
    return catalogue.identify_target(sp, sp.leafs, sp.roots)


def test_catalogue_recognises_t_and_cauchy():
    sp = _mu_sigma_sp()
    sp.set_prob(scipy.stats.norm.logpdf, order=ORDER)
    normal = _spec(sp)
    assert 'lik' not in normal
    sp.set_prob(scipy.stats.t.logpdf, order=ORDER, df=4.)
    spec = _spec(sp)
    assert spec['lik'] == dict(family='t', df=4.0, logc=catalogue.t_logc(4.))
    assert {k: v for k, v in spec.items() if k != 'lik'} == normal
    sp.set_prob(scipy.stats.cauchy.logpdf, order=ORDER)
    spec = _spec(sp)
    assert spec['lik'] == dict(family='cauchy', df=1.0, logc=-np.log(np.pi))
    # df = inf is the normal, as scipy's t_gen._logpdf
    sp.set_prob(scipy.stats.t.logpdf, order=ORDER, df=np.inf)
    assert _spec(sp) == normal


def test_student_t_regression_spec():
    xx = pb.RV('x', vtype=float, vset=[-3, 3])
    yy = pb.RV('y', vtype=float, vset=[-np.inf, np.inf])
    b0 = pb.RV('beta_0', vtype=float, vset=[-6., 6.], pscale='log')
    b1 = pb.RV('beta_1', vtype=float, vset=[-6., 6.], pscale='log')
    ys = pb.RV('y_sigma', vtype=float, vset=[(0.001), 10.], pscale='log')
    proc = pb.SP(xx & yy, b0 & b1 & ys)
    proc.set_prob(pb.StudentTRegression('x', 'y', 'beta_0', 'beta_1', 'y_sigma', df=4.),
                  pscale='log')
    spec = _spec(proc)
    assert spec == dict(kind='normreg', has_slope=True, obs_y='y', obs_x='x',
                        params=['beta_0', 'beta_1', 'y_sigma'], log_pscale=True,
                        lik=dict(family='t', df=4.0, logc=catalogue.t_logc(4.)))
    proc.set_prob(pb.StudentTRegression('x', 'y', 'beta_0', 'beta_1', 'y_sigma', df=np.inf),
                  pscale='log')
    assert 'lik' not in _spec(proc)
    with pytest.raises(ValueError):
        proc.set_prob(pb.StudentTRegression('x', 'y', 'beta_0', 'beta_1', 'y_sigma'),
                      pscale='log')
        _spec(proc)


@pytest.mark.parametrize("df", [None, 0., -2., np.nan, "four"])
def test_catalogue_refuses_bad_df(df):
    sp = _mu_sigma_sp()
    kw = {} if df is None else dict(df=df)
    sp.set_prob(scipy.stats.t.logpdf, order=ORDER, **kw)
    with pytest.raises(ValueError, match="df"):
        _spec(sp)


@pytest.mark.parametrize("family", ["t", "cauchy"])
def test_catalogue_refuses_pdf_and_suffstat(family):
    sp = _mu_sigma_sp()
    dist = getattr(scipy.stats, family)
    kw = dict(df=4.) if family == "t" else {}
    sp.set_prob(dist.pdf, order=ORDER, **kw)
    with pytest.raises(NotImplementedError, match="log pscale"):
        _spec(sp)
    sp.set_prob(dist.logpdf, order=ORDER, **kw)
    spec = _spec(sp)
    with pytest.raises(NotImplementedError, match="sufficient statistics"):
        catalogue.refuse_suffstat(spec, 3)
    catalogue.refuse_suffstat(spec, 0)
    sp.set_prob(scipy.stats.norm.logpdf, order=ORDER)
    catalogue.refuse_suffstat(_spec(sp), 3)


def test_suffstat_refused_before_any_device_call():
    """SD.__call__ and SP walks refuse suffstat=True with a t likelihood (host-side)."""
    mu = pb.RV('mu', vtype=float, vset=(40, 60), pscale='log')
    sigma = pb.RV('sigma', vtype=float, vset=(5, 20.), pscale='log')
    x = pb.RV('x', vtype=float, vset=(-np.inf, np.inf))
    sd = pb.SD(pb.RF(x), pb.RF(mu, sigma))
    sd.set_prob(scipy.stats.t.logpdf, order=ORDER, df=4.)
    with pytest.raises(NotImplementedError, match="sufficient statistics"):
        sd({'x': np.ones(10), 'mu': {8}, 'sigma': {8}}, iid=True, joint=True, suffstat=True)


@pytest.mark.parametrize("df", [1., 4., 1e3, 1e6])
def test_logc_equals_scipy_constant(df):
    # t.logpdf(0) = logc - (df + 1)/2 * log1p(0) - log(1): scipy's constant, bit for bit
    assert catalogue.t_logc(df) == float(scipy.stats.t.logpdf(0., df))


def test_cauchy_constant():
    assert catalogue.likelihood('cauchy')['logc'] == float(scipy.stats.cauchy.logpdf(0.))


def test_abi_fields_at_header_offsets():
    src = r'''
#include <stddef.h>
#include <stdio.h>
#include "pbx.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %d %d\n", offsetof(pbx_mh_normreg_params, prop_mat),
         offsetof(pbx_mh_normreg_params, lik_kind), offsetof(pbx_mh_normreg_params, lik_df),
         offsetof(pbx_mh_normreg_params, lik_logc), sizeof(pbx_mh_normreg_params),
         PBX_LIK_NORMAL, PBX_LIK_STUDENT_T);
  return 0;
}'''
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "p.c"), "w").write(src)
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "p.c"),
                        "-o", os.path.join(d, "p")], check=True)
        out = subprocess.run([os.path.join(d, "p")], capture_output=True, text=True,
                             check=True).stdout.split()
    P = _lib.MhNormregParams
    assert [int(v) for v in out] == [P.prop_mat.offset, P.lik_kind.offset, P.lik_df.offset,
                                     P.lik_logc.offset, C.sizeof(P), _lib.LIK_NORMAL,
                                     _lib.LIK_STUDENT_T]
    # the new fields follow the old ones: a zeroed tail is the normal likelihood
    assert P.lik_kind.offset == P.prop_mat.offset + 9 * 8
    assert P().lik_kind == _lib.LIK_NORMAL


def test_grid_export_bound():
    res, args = _lib.SIGNATURES["pbx_grid_t_logjoint"]
    assert args[:10] == _lib.SIGNATURES["pbx_grid_norm_logjoint"][1]
    assert args[10:] == [C.c_double, C.c_double]
    from probayes_b200 import build
    build.build()
    assert hasattr(_lib.load(), "pbx_grid_t_logjoint")


class _FakeEngine:
    """Records the likelihood the engine entry points are handed."""

    def __init__(self):
        self.calls = []

    def to_device(self, a):
        import torch
        return torch.as_tensor(np.asarray(a, dtype=np.float64))

    def box_sample(self, lims, lg, n, seed=0, sample0=0, inj_unif=None):
        raise _Reached(None)

    def grid_norm_logjoint(self, *args, **kw):
        raise _Reached(kw.get('lik'))

    def mh_normreg(self, *args, **kw):
        raise _Reached(kw.get('lik'))


class _Reached(Exception):
    def __init__(self, lik):
        self.lik = lik


def test_student_t_regression_reaches_the_engine(monkeypatch):
    import probayes_b200.engine as engine_mod
    fake = _FakeEngine()
    monkeypatch.setattr(engine_mod, "get_engine", lambda device=None: fake)
    xx = pb.RV('x', vtype=float, vset=[-3, 3])
    yy = pb.RV('y', vtype=float, vset=[-np.inf, np.inf])
    b0 = pb.RV('beta_0', vtype=float, vset=[-6., 6.], pscale='log')
    b1 = pb.RV('beta_1', vtype=float, vset=[-6., 6.], pscale='log')
    ys = pb.RV('y_sigma', vtype=float, vset=[(0.001), 10.], pscale='log')
    proc = pb.SP(xx & yy, b0 & b1 & ys)
    proc.set_prob(pb.StudentTRegression('x', 'y', 'beta_0', 'beta_1', 'y_sigma', df=4.),
                  pscale='log')
    proc.set_delta([0.01])
    proc.set_scores('metropolis')
    x = np.linspace(-1, 1, 20)
    sampler = proc.sampler({'beta_0': 0., 'beta_1': 0., 'y_sigma': 1.}, {'x': x, 'y': x},
                           stop=5, iid=True, joint=True)
    with pytest.raises(_Reached) as e:
        proc.walk(sampler)
    assert e.value.lik == dict(family='t', df=4.0, logc=catalogue.t_logc(4.))


def test_oracle_logjoint_is_the_scipy_sum():
    rng = np.random.default_rng(3)
    x = rng.normal(0., 1., 200)
    y = -1. + 1.5 * x + 0.5 * rng.standard_t(3., 200)
    theta = np.array([[-1., 1.5, 0.5], [-0.9, 1.4, 0.7]])
    lims = np.array([[-6., 6.], [-6., 6.], [0.001, 10.]])
    ex = np.zeros((3, 2), bool)
    lg = np.zeros(3, bool)
    prior = -np.log(12.) - np.log(12.) - np.log(10. - 0.001)
    for lik in (catalogue.likelihood('t', 3.), catalogue.likelihood('cauchy')):
        got = to.normreg_logjoint(theta, x, y, lims, ex, lg, True, lik)
        dist = scipy.stats.t(lik['df']) if lik['family'] == 't' else scipy.stats.cauchy()
        for c in range(2):
            want = prior + np.sum(dist.logpdf((y - theta[c, 0] - theta[c, 1] * x) / theta[c, 2])
                                  - np.log(theta[c, 2]))
            assert abs(got[c] - want) <= 1e-12 * abs(want)
    # the walk's recorded log-joints are the same sums
    delta = rng.uniform(-0.02, 0.02, (6, 2, 3))
    walk = to.mh_normreg_walk(theta, delta, rng.random((6, 2)), x, y, lims, ex, lg, True,
                              accept="log", lik=catalogue.likelihood('t', 3.))
    for k in range(6):
        want = to.normreg_logjoint(walk["x"][k], x, y, lims, ex, lg, True,
                                   catalogue.likelihood('t', 3.))
        assert np.array_equal(walk["prob"][k], want)
