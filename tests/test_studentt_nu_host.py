"""Student-t likelihood with nu sampled, on the host: the catalogue's two spellings and its
refusals, the engine's ABI struct, the device logc method restated in numpy against mpmath, the
spec reaching the engine from SP and SD, and the oracle's sums."""
import ctypes as C
import os
import subprocess
import tempfile

import mpmath
import numpy as np
import pytest
import scipy.stats

import probayes_b200 as pb
from probayes_b200 import _lib, catalogue
import studentt_nu_oracle as tno
import studentt_oracle as to

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORDER = {'x': 0, 'nu': 1, 'mu': 'loc', 'sigma': 'scale'}
NU_LIK = dict(family='t', df_param='nu')


def _model(nu_vset=(0.5, 100.), cls=pb.SP, pscale='log'):
    mu = pb.RV('mu', vtype=float, vset=[40., 60.], pscale=pscale)
    sigma = pb.RV('sigma', vtype=float, vset=[5., 20.], pscale=pscale)
    nu = pb.RV('nu', vtype=float, vset=nu_vset, pscale=pscale)
    x = pb.RV('x', vtype=float, vset=(-np.inf, np.inf))
    return cls(pb.RF(x), mu & sigma & nu)


def _spec(sp):
    return catalogue.identify_target(sp, sp.leafs, sp.roots)


@pytest.mark.parametrize("role", [1, 'df'])
def test_catalogue_recognises_sampled_nu(role):
    sp = _model([0.5, 100.])
    sp.set_prob(scipy.stats.t.logpdf, order=dict(ORDER, nu=role), pscale='log')
    assert _spec(sp) == dict(kind='normreg', has_slope=False, obs_y='x', obs_x=None,
                             params=['mu', 'sigma', 'nu'], log_pscale=True, lik=NU_LIK)
    # an open lower end at 0 admits nu > 0 only
    sp = _model((0., 100.))
    sp.set_prob(scipy.stats.t.logpdf, order=dict(ORDER, nu=role), pscale='log')
    assert _spec(sp)['lik'] == NU_LIK


def test_fixed_nu_spec_unchanged():
    """Without a df role the t is the fixed-nu spec (df = inf: the normal), nu an unused RV."""
    sp = _model()
    order = {'x': 0, 'mu': 'loc', 'sigma': 'scale'}
    sp.set_prob(scipy.stats.t.logpdf, order=order, df=4., pscale='log')
    assert _spec(sp) == dict(kind='normreg', has_slope=False, obs_y='x', obs_x=None,
                             params=['mu', 'sigma'], log_pscale=True,
                             lik=dict(family='t', df=4.0, logc=catalogue.t_logc(4.)))
    sp.set_prob(scipy.stats.t.logpdf, order=order, df=np.inf, pscale='log')
    assert 'lik' not in _spec(sp)


def test_catalogue_refusals():
    sp = _model()
    sp.set_prob(scipy.stats.t.logpdf, order=ORDER, df=4., pscale='log')
    with pytest.raises(ValueError, match="given twice"):
        _spec(sp)
    sp.set_prob(scipy.stats.cauchy.logpdf, order=ORDER, pscale='log')
    with pytest.raises(NotImplementedError, match="cauchy.logpdf has no degrees of freedom"):
        _spec(sp)
    sp.set_prob(scipy.stats.t.pdf, order=ORDER)
    with pytest.raises(NotImplementedError, match="log pscale"):
        _spec(sp)
    lin = _model(pscale=None)
    lin.set_prob(scipy.stats.t.logpdf, order=ORDER)
    with pytest.raises(NotImplementedError, match="log pscale"):
        _spec(lin)
    # the df role on a stats (observation) RV
    x = pb.RV('x', vtype=float, vset=(-np.inf, np.inf))
    w = pb.RV('w', vtype=float, vset=(0., 10.))
    mu = pb.RV('mu', vtype=float, vset=[40., 60.], pscale='log')
    sigma = pb.RV('sigma', vtype=float, vset=[5., 20.], pscale='log')
    sp = pb.SP(x & w, mu & sigma)
    sp.set_prob(scipy.stats.t.logpdf, order={'x': 0, 'w': 'df', 'mu': 'loc', 'sigma': 'scale'},
                pscale='log')
    with pytest.raises(NotImplementedError, match="stats \\(observation\\) RV"):
        _spec(sp)
    # suffstat=True
    sp = _model()
    sp.set_prob(scipy.stats.t.logpdf, order=ORDER, pscale='log')
    with pytest.raises(NotImplementedError, match="sufficient statistics"):
        catalogue.refuse_suffstat(_spec(sp), 3)


@pytest.mark.parametrize("vset", [[0., 100.], [-1., 100.], (-1., 100.)])
def test_catalogue_refuses_nu_box_admitting_nonpositive(vset):
    sp = _model(vset)
    sp.set_prob(scipy.stats.t.logpdf, order=ORDER, pscale='log')
    with pytest.raises(ValueError, match="nu > 0 only"):
        _spec(sp)


def test_normreg_params_fill():
    """The ctypes struct of the sampled-nu t: lik_kind 2, three parameters, no slope, a zero
    lik_df / lik_logc; the regression and the fixed-nu t keep their fill."""
    import torch
    from probayes_b200.engine import Engine
    y = torch.zeros(10, dtype=torch.float64)
    lims = [[40., 60.], [5., 20.], [0.5, 100.]]
    p = Engine._normreg_params(None, 16, 3, None, y, lims, np.zeros((3, 2)), np.zeros(3), 0.1,
                               lik=NU_LIK)
    assert (p.lik_kind, p.n_params, p.has_slope, p.lik_df, p.lik_logc, p.x_obs) == \
        (_lib.LIK_STUDENT_T_NU, 3, 0, 0.0, 0.0, None)
    assert [list(p.lims[j]) for j in range(3)] == lims
    t4 = catalogue.likelihood('t', 4.)
    p = Engine._normreg_params(None, 16, 3, y, y, lims, np.zeros((3, 2)), np.zeros(3), 0.1,
                               lik=t4)
    assert (p.lik_kind, p.has_slope, p.lik_df, p.lik_logc) == \
        (_lib.LIK_STUDENT_T, 1, 4.0, t4['logc'])
    with pytest.raises(ValueError, match="mu, sigma, nu"):
        Engine._normreg_params(None, 16, 2, None, y, lims[:2], np.zeros((2, 2)), np.zeros(2),
                               0.1, lik=NU_LIK)


def test_header_constant():
    src = r'''
#include <stdio.h>
#include "pbx.h"
int main(void) { printf("%d\n", PBX_LIK_STUDENT_T_NU); return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "p.c"), "w").write(src)
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "p.c"),
                        "-o", os.path.join(d, "p")], check=True)
        out = subprocess.run([os.path.join(d, "p")], capture_output=True, text=True,
                             check=True).stdout
    assert int(out) == _lib.LIK_STUDENT_T_NU == 2
    assert C.sizeof(_lib.MhNormregParams) == _lib.MhNormregParams.lik_logc.offset + 8


def _mp_logc(nu):
    nu = mpmath.mpf(nu)
    return mpmath.loggamma((nu + 1) / 2) - mpmath.loggamma(nu / 2) - mpmath.log(nu * mpmath.pi) / 2


def test_series_coefficients():
    c = tno.series_coefficients()
    assert [c[k] for k in (1, 3, 5, 7)] == [-1 / tno.Fraction(8), 1 / tno.Fraction(192),
                                           -1 / tno.Fraction(640), 17 / tno.Fraction(14336)]
    # the series the kernel hard-codes, term by term
    src = open(os.path.join(ROOT, "probayes_b200", "csrc", "pbx_mh_normreg.cu")).read()
    for k, v in c.items():
        lit = "{}.0 / {}.0".format(abs(v.numerator), v.denominator) if v.denominator != 8 \
            else "0.125"
        assert lit in src, (k, v)


def test_logc_method_against_mpmath():
    """The device method restated in numpy: within 1e-14 absolute of mpmath over nu in
    [1e-3, 1e12] (measured here: ~5e-15, from glibc's lgamma below nu = 16; the series part
    alone is within 1e-16), and continuous at the crossover."""
    nus = np.concatenate([np.geomspace(1e-3, 1e12, 1500), [15.999999, 16., 16.000001]])
    with mpmath.workdps(40):
        err = np.array([abs(tno.device_logc(v) - float(_mp_logc(v))) for v in nus])
    assert err.max() <= 1e-14, (err.max(), nus[err.argmax()])
    series = nus >= 16.
    assert err[series].max() <= 2e-16, err[series].max()
    # the normal's constant as nu -> inf, without cancellation
    with mpmath.workdps(40):
        assert tno.device_logc(1e300) == -float(mpmath.log(2 * mpmath.pi) / 2)
    assert tno.device_logc(4.) == pytest.approx(catalogue.t_logc(4.), abs=1e-15)


class _FakeEngine:
    def to_device(self, a):
        import torch
        return torch.as_tensor(np.asarray(a, dtype=np.float64))

    def box_sample(self, lims, lg, n, seed=0, sample0=0, inj_unif=None):
        import torch
        return torch.zeros(len(lims), n, dtype=torch.float64)

    def normreg_logjoint(self, *args, **kw):
        raise _Reached(kw.get('lik'), args)

    def grid_norm_logjoint(self, *args, **kw):
        raise _Reached(kw.get('lik'), args)

    def mh_normreg(self, *args, **kw):
        raise _Reached(kw.get('lik'), args)


class _Reached(Exception):
    def __init__(self, lik, args):
        self.lik, self.args = lik, args


def test_spec_reaches_the_engine(monkeypatch):
    """MH walks and random sampling hand the engine the sampled-nu likelihood, state (mu, sigma,
    nu) and no x; SD's grid turns a scalar nu into the fixed-nu t and refuses a nu grid."""
    import probayes_b200.engine as engine_mod
    fake = _FakeEngine()
    monkeypatch.setattr(engine_mod, "get_engine", lambda device=None: fake)
    data = np.linspace(-1., 1., 20)
    sp = _model()
    sp.set_prob(scipy.stats.t.logpdf, order=ORDER, pscale='log')
    sp.set_delta([0.01])
    sp.set_scores('metropolis')
    sampler = sp.sampler({'mu': 50., 'sigma': 10., 'nu': 4.}, {'x': data}, stop=5, iid=True,
                         joint=True)
    with pytest.raises(_Reached) as e:
        sp.walk(sampler)
    state, y, x = e.value.args[:3]
    assert e.value.lik == NU_LIK and tuple(state.shape) == (3, 1) and x is None
    assert np.array_equal(state[:, 0].cpu().numpy(), [50., 10., 4.])
    sp = _model()                              # random sampling: no transition, no delta
    sp.set_prob(scipy.stats.t.logpdf, order=ORDER, pscale='log')
    sampler = sp.sampler({'mu': {0}, 'sigma': {0}, 'nu': {0}, 'x': data}, stop=8, iid=True,
                         joint=True)
    with pytest.raises(_Reached) as e:
        sp.walk(sampler)
    assert e.value.lik == NU_LIK and tuple(e.value.args[0].shape) == (3, 8)
    sd = _model(cls=pb.SD)
    sd.set_prob(scipy.stats.t.logpdf, order=ORDER, pscale='log')
    with pytest.raises(_Reached) as e:
        sd({'x': data, 'mu': {8}, 'sigma': {8}, 'nu': 4.}, iid=True, joint=True)
    assert e.value.lik == catalogue.likelihood('t', 4.)
    # nu's prior joins the mu prior, the same for every cell
    lpm = e.value.args[3].numpy()
    assert np.allclose(lpm, -np.log(20.) - np.log(99.5), rtol=1e-15, atol=0.)
    for bad in ({4}, np.array([3., 4.])):
        with pytest.raises(NotImplementedError, match="three-axis"):
            sd({'x': data, 'mu': {8}, 'sigma': {8}, 'nu': bad}, iid=True, joint=True)
    with pytest.raises(NotImplementedError, match="sufficient statistics"):
        sd({'x': data, 'mu': {8}, 'sigma': {8}, 'nu': 4.}, iid=True, joint=True, suffstat=True)


def test_oracle_is_the_per_chain_fixed_nu_sum():
    rng = np.random.default_rng(7)
    y = 1. + 2. * rng.standard_t(4., 300)
    theta = np.array([[1., 2., 4.], [0.8, 2.3, 0.7], [1.1, 1.9, 1e6]])
    lims = np.array([[-5., 5.], [0.1, 10.], [0.5, 1e7]])
    ex, lg = np.zeros((3, 2), bool), np.array([False, True, True])
    got = tno.logjoint(theta, y, lims, ex, lg)
    for c in range(3):
        nu = theta[c, 2]
        want = to.normreg_logjoint(theta[c:c + 1, :2], None, y, lims[:2], ex[:2], lg[:2], False,
                                   catalogue.likelihood('t', nu))[0]
        want += -np.log(np.log(lims[2, 1]) - np.log(lims[2, 0]))
        assert got[c] == pytest.approx(want, rel=1e-14)
