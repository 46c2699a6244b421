"""The numpy oracle of the Student-t / Cauchy likelihoods: oracle.np_oracle's walk, proposal and
box priors with the likelihood sum replaced by the sum of scipy.stats.t.logpdf (or
cauchy.logpdf) -- the reference's own arithmetic.  ``lik`` is the catalogue's likelihood entry:
None (the normal: np_oracle's functions unchanged) or dict(family, df, logc)."""
import numpy as np
import scipy.stats

from oracle import np_oracle as o


def lik_logpdf(y, loc, scale, lik):
    """Per-observation log-density of y ~ family(loc, scale)."""
    if lik is None:
        return o.norm_logpdf(y, loc, scale)
    if lik["family"] == "cauchy":
        return scipy.stats.cauchy.logpdf(y, loc=loc, scale=scale)
    return scipy.stats.t.logpdf(y, lik["df"], loc=loc, scale=scale)


def normreg_logjoint(theta, x_obs, y_obs, lims, ex, log_ufun, has_slope=True, lik=None):
    """np_oracle.normreg_logjoint with the iid likelihood of ``lik``."""
    if lik is None:
        return o.normreg_logjoint(theta, x_obs, y_obs, lims, ex, log_ufun, has_slope)
    theta = np.asarray(theta, dtype=float)
    C, P = theta.shape
    out = np.empty(C)
    y = np.asarray(y_obs, dtype=float)[None, :]
    for c0 in range(0, C, 64):                 # row c sums observation axis 1 of chain c
        th = theta[c0:c0 + 64]
        loc = th[:, :1] + th[:, 1:2] * np.asarray(x_obs)[None, :] if has_slope else th[:, :1]
        with np.errstate(invalid="ignore", divide="ignore"):
            out[c0:c0 + 64] = np.sum(lik_logpdf(y, loc, th[:, P - 1:], lik), axis=1)
    prior = np.zeros(C)
    with np.errstate(over="ignore"):           # two -huge priors sum to -inf, as np_oracle's
        for j in range(P):
            prior = prior + o.box_log_prior(theta[:, j], lims[j][0], lims[j][1], ex[j][0],
                                            ex[j][1], log_ufun[j])
    return prior + out


def mh_normreg_walk(init, delta, thresh, x_obs, y_obs, lims, ex, log_ufun, has_slope=True,
                    accept="reference", coef=1.0, bound=False, lik=None):
    """np_oracle.mh_normreg_walk with the iid likelihood of ``lik``."""
    def target(th):
        return normreg_logjoint(th, x_obs, y_obs, lims, ex, log_ufun, has_slope, lik)

    def propose(th, dl):
        return o.ufun_propose(th, dl, log_ufun, (lims, ex) if bound else None)

    return o.mh_walk(init, delta, thresh, target, propose, True, accept, coef)


def grid_logjoint(x_obs, mu, sigma, logprior_mu, logprior_sigma, lik=None, chunk=16):
    """np_oracle.grid_norm_logjoint with the iid likelihood of ``lik`` (observation axis 0
    summed, priors added first)."""
    if lik is None:
        return o.grid_norm_logjoint(x_obs, mu, sigma, logprior_mu, logprior_sigma)
    x_obs = np.asarray(x_obs, dtype=float)
    M, S = len(mu), len(sigma)
    out = np.empty((M, S))
    xs = x_obs[:, None, None]
    sg = np.asarray(sigma, dtype=float)[None, None, :]
    for m0 in range(0, M, chunk):
        mm = np.asarray(mu[m0:m0 + chunk], dtype=float)[None, :, None]
        out[m0:m0 + chunk] = np.sum(lik_logpdf(xs, mm, sg, lik), axis=0)
    prior = np.asarray(logprior_mu, dtype=float).reshape(-1, 1) + \
        np.asarray(logprior_sigma, dtype=float).reshape(1, -1)
    return prior + out
