"""A covariance-matrix transition (``set_tran(ndarray)``, rf.py:209-220) on a normal-likelihood
sampler reaches the K2 kernel: SP hands the Cholesky factor to ``Engine.mh_normreg`` on every
call of a walk, resumed calls included, and the engine writes it into the C ABI parameters.
No GPU: the engine is replaced by a recorder, and the ABI struct is only filled, not passed."""
import types

import numpy as np
import pytest
import scipy.stats
import probayes_b200 as pb
from probayes_b200 import engine as engine_mod
from probayes_b200._lib import MhNormregParams

COV = np.array([[4e-3, -7.6e-4, 0.], [-7.6e-4, 1.5e-4, 0.], [0., 0., 1e-5]])


def _linreg_process(cov):
    x = pb.RV('x', vtype=float, vset=[-np.inf, np.inf])
    y = pb.RV('y', vtype=float, vset=[-np.inf, np.inf])
    beta_0 = pb.RV('beta_0', vtype=float, vset=[-6., 6.], pscale='log')
    beta_1 = pb.RV('beta_1', vtype=float, vset=[-6., 6.], pscale='log')
    y_sigma = pb.RV('y_sigma', vtype=float, vset=[(0.001), 10.], pscale='log')

    def norm_reg(x, y, beta_0, beta_1, y_sigma):
        return scipy.stats.norm.logpdf(y, loc=beta_0 + beta_1 * x, scale=y_sigma)

    paras = beta_0 & beta_1 & y_sigma
    process = pb.SP(x & y, paras)
    process.set_prob(norm_reg, pscale='log')
    paras.set_tran(cov)
    paras.set_delta(scipy.stats.norm(0., 1.))
    process.set_tran(paras)
    process.set_delta(paras)
    process.set_scores('metropolis')
    return process


class _Recorder:
    """Stands in for the device engine: keeps host arrays and records each mh_normreg call."""

    def __init__(self):
        self.calls = []

    def to_device(self, a):                      # host tensors stand in for device ones
        import torch
        return torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.float64)))

    def sync(self):
        pass

    def mh_normreg(self, state, y, x, T, *args, thin=1, **kw):
        self.calls.append(dict(kw, T=T))
        P, C = state.shape
        R = T // thin
        return dict(x=np.zeros((R, P, C)), prob=np.zeros((R, C)), state_lp=np.zeros(C),
                    accept_count=np.zeros(C, np.int64), stat_sum=np.zeros((P, C)),
                    stat_sumsq=np.zeros((P, C)))


@pytest.mark.filterwarnings("ignore:probayes_b200. the Python likelihood")
def test_set_tran_covariance_reaches_mh_normreg(monkeypatch):
    pytest.importorskip("torch")
    rec = _Recorder()
    monkeypatch.setattr(engine_mod, "get_engine", lambda *a, **k: rec)
    process = _linreg_process(COV)
    rng = np.random.default_rng(3)
    xo = rng.normal(5., 1., 200)
    yo = rng.normal(-1. + 1.5 * xo, 0.5)
    sampler = process.sampler({'beta_0': -1., 'beta_1': 1.5, 'y_sigma': 0.5},
                              {'x,y': [xo, yo]}, stop=40, iid=True, joint=True, chains=8,
                              chain0=16, seed=5)
    process.walk(sampler, stop=24)
    process.walk(sampler, stop=16)                     # resumes at step 24
    assert [(c['T'], c['step0'], c['chain0']) for c in rec.calls] == [(24, 0, 16), (16, 24, 16)]
    for c in rec.calls:
        assert np.array_equal(c['prop_chol'], np.linalg.cholesky(COV))
        assert c['prop'] == 'normal'
    assert rec.calls[1]['state_lp'] is not None


def test_normreg_params_carry_the_factor():
    """The ctypes mirror: prop_mat is the row-major [P][P] factor and has_prop_mat is set;
    without a factor both stay zero; a factor of the wrong shape is refused."""
    fake = types.SimpleNamespace(numel=lambda: 10, data_ptr=lambda: 4096)
    args = (5, 3, fake, fake, [[-6., 6.]] * 3, [[0, 0]] * 3, [0, 0, 1], [0.1] * 3)
    L = np.linalg.cholesky(COV)
    p = engine_mod.Engine._normreg_params(None, *args, prop_chol=L)
    assert isinstance(p, MhNormregParams) and p.has_prop_mat == 1
    assert np.array_equal(np.array(p.prop_mat[:]), L.ravel())
    p0 = engine_mod.Engine._normreg_params(None, *args)
    assert p0.has_prop_mat == 0 and not any(p0.prop_mat[:])
    with pytest.raises(ValueError, match=r"\[P, P\]"):
        engine_mod.Engine._normreg_params(None, *args, prop_chol=np.eye(2))
