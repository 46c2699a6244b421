"""The numpy oracle of the Student-t likelihood with nu sampled: studentt_oracle's walk and
log-joint for theta = (mu, sigma, nu), each chain summing scipy.stats.t.logpdf(y, nu_c, loc=mu_c,
scale=sigma_c) with its own nu -- the reference's own arithmetic."""
import math
from fractions import Fraction

import numpy as np
import scipy.stats

from oracle import np_oracle as o


def logjoint(theta, y_obs, lims, ex, log_ufun):
    """Box priors + sum_i t.logpdf(y_i; nu, mu, sigma) of every row (mu, sigma, nu) of theta."""
    theta = np.asarray(theta, dtype=float)
    C = theta.shape[0]
    y = np.asarray(y_obs, dtype=float)[None, :]
    out = np.empty(C)
    for c0 in range(0, C, 64):
        th = theta[c0:c0 + 64]
        with np.errstate(invalid="ignore", divide="ignore"):
            out[c0:c0 + 64] = np.sum(scipy.stats.t.logpdf(y, th[:, 2:3], loc=th[:, :1],
                                                          scale=th[:, 1:2]), axis=1)
    prior = np.zeros(C)
    with np.errstate(over="ignore"):           # two -huge priors sum to -inf, as np_oracle's
        for j in range(3):
            prior = prior + o.box_log_prior(theta[:, j], lims[j][0], lims[j][1], ex[j][0],
                                            ex[j][1], log_ufun[j])
    return prior + out


def mh_walk(init, delta, thresh, y_obs, lims, ex, log_ufun, accept="reference", coef=1.0,
            bound=False):
    """np_oracle.mh_walk of the (mu, sigma, nu) target; delta [T, C, 3] already coloured."""
    def target(th):
        return logjoint(th, y_obs, lims, ex, log_ufun)

    def propose(th, dl):
        return o.ufun_propose(th, dl, log_ufun, (lims, ex) if bound else None)

    return o.mh_walk(init, delta, thresh, target, propose, True, accept, coef)


def series_coefficients(kmax=17):
    """c_k of R(z) = lgamma(z + 1/2) - lgamma(z) - log(z)/2 ~ sum_k c_k z^-k (odd k): from
    lgamma(z + a) - lgamma(z) - a log z ~ sum_k (-1)^(k+1) (B_{k+1}(a) - B_{k+1}) / (k (k+1) z^k)
    and B_n(1/2) = -(1 - 2^(1-n)) B_n, so c_k = -(2 - 2^-k) B_{k+1} / (k (k+1)); exact."""
    B = [Fraction(1)]
    for m in range(1, kmax + 2):
        B.append(-sum(math.comb(m + 1, j) * B[j] for j in range(m)) / Fraction(m + 1))
    return {k: -(2 - Fraction(1, 2 ** k)) * B[k + 1] / (k * (k + 1)) for k in range(1, kmax + 1, 2)}


def device_logc(nu):
    """nr_t_logc of pbx_mh_normreg.cu restated in numpy (glibc lgamma below z = 8)."""
    c = series_coefficients()
    z = 0.5 * float(nu)
    if z < 8.0:
        R = math.lgamma(z + 0.5) - math.lgamma(z) - 0.5 * math.log(z)
    else:
        w = 1.0 / (z * z)
        s = float(c[17])
        for k in range(15, 0, -2):
            s = s * w + float(c[k])
        R = s / z
    return R - 0.91893853320467274178
