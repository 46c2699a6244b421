"""The device catalogue: maps what the user configured through the reference API
(set_prob / set_tran / set_delta / set_scores ...) onto a libpbx kernel, or refuses.

The reference accepts arbitrary Python callables everywhere (probayes/prob.py:
125-189, expression.py:376-452); a callable cannot run on the GPU, so the drop-in
*recognises* the cases the reference's own examples use and raises
``NotImplementedError`` for the rest -- there is no CPU fallback.

Targets
  mvn      scipy.stats.multivariate_normal(mean, cov)        (mcmc_prob4a, gibbs_norm2d)
  norm     scipy.stats.norm.logpdf + order={'x': 0, 'mu': 'loc', 'sigma': 'scale'}
           with iid=True                                      (metrohast_norm1d, dgei_*)
           -- or scipy.stats.t.logpdf with df=nu, or scipy.stats.cauchy.logpdf, in the
           same call: the spec's ``lik`` entry names the family; or t.logpdf with order
           mapping a parameter RV nu to 1 or 'df': nu is sampled, params (loc, scale, nu)
  normreg  a Python callable that IS norm.logpdf(y, loc=b0 + b1*x, scale=s) -- verified
           numerically by probing it against every role assignment (gibbs_linreg's
           ``norm_reg``), or an explicit ``NormalRegression`` / ``StudentTRegression`` spec
Proposals (field.py:220-317, variable.py:600-638, rf.py:209-220)
  [d] uniform per RV, (d,) spherical, frozen scipy.stats.norm, covariance-matrix tran
Rejection sampling (set_prop + custom scores / thresh / update, omc_rejection_sp_circle)
  target    BallIndicator (1.0 inside a ball, 0.0 outside)
  proposal  NormalProduct (prod_j norm.pdf(x_j; loc_j, scale_j)) or BoxUniform
  scores    opqr.p.prob  or  opqr.p.prob / opqr.q.prob ;  thresh np.random.uniform(low, high) ;
  update    stu.s >= stu.t   -- Python callables are recognised by probing (with a warning)
"""
import inspect
import itertools
import numpy as np
import scipy.special
import scipy.stats

from .pscales import iscomplex, rescale


class NormalRegression:
    """Explicit catalogue spec of y ~ N(intercept + slope*x, scale) (log-density)."""

    def __init__(self, x, y, intercept, slope, scale):
        self.x, self.y, self.intercept, self.slope, self.scale = x, y, intercept, slope, scale


class StudentTRegression:
    """Explicit catalogue spec of y ~ t_df(intercept + slope*x, scale) (log-density,
    scipy.stats.t.logpdf); ``df=np.inf`` is the normal regression."""

    def __init__(self, x, y, intercept, slope, scale, df=None):
        self.x, self.y, self.intercept, self.slope, self.scale = x, y, intercept, slope, scale
        self.df = df


def t_logc(df):
    """The per-observation constant of scipy.stats.t.logpdf, computed as scipy's t_gen._logpdf
    does: log(poch(df/2, 1/2)) - (log df + log pi)/2.  (lgamma((df+1)/2) - lgamma(df/2)
    cancels: 6e-10 relative at df = 1e6, which N observations multiply.)"""
    df = np.float64(df)
    return float(np.log(scipy.special.poch(0.5 * df, 0.5)) - 0.5 * (np.log(df) + np.log(np.pi)))


def likelihood(family, df=None):
    """The ``lik`` entry of a target spec: None for the normal, else dict(family, df, logc)
    for the Student-t (df = nu) or the Cauchy (df = 1, logc = -log pi as cauchy.logpdf).
    A t with df = inf is the normal, as in scipy (t_gen._logpdf calls norm._logpdf)."""
    if family == 'norm':
        return None
    if family == 'cauchy':
        return dict(family='cauchy', df=1.0, logc=float(-np.log(np.pi)))
    if df is None:
        raise ValueError("the Student-t likelihood needs its degrees of freedom: "
                         "set_prob(scipy.stats.t.logpdf, ..., df=nu)")
    try:
        df = float(df)
    except (TypeError, ValueError):
        raise ValueError("df must be a positive number, got {!r}".format(df))
    if df == np.inf:
        return None
    if not df > 0:
        raise ValueError("df must be positive (and not NaN), got {!r}".format(df))
    return dict(family='t', df=df, logc=t_logc(df))


def _df_role(order, family, kwds, stats, paras):
    """The parameter RV an order of t.logpdf maps to df (positional 1 or 'df'), or None.  Only
    t.logpdf takes a df; for the normal, whose catalogue entry predates this, a role 1 stays
    unread as before."""
    names = [k for k, v in order.items() if isinstance(v, (int, str)) and not isinstance(v, bool)
             and v in (1, 'df')]
    if not names or family == 'norm':
        return None
    if family == 'cauchy':
        raise NotImplementedError("scipy.stats.cauchy.logpdf has no degrees of freedom: use "
                                  "scipy.stats.t.logpdf to sample nu (order maps {!r} to {!r})"
                                  .format(names[0], order[names[0]]))
    if len(names) > 1:
        raise NotImplementedError("order maps more than one RV to the degrees of freedom: "
                                  "{}".format(names))
    nu = names[0]
    if 'df' in (kwds or {}):
        raise ValueError("the degrees of freedom are given twice: by df= and by order "
                         "({!r} -> {!r}); drop one".format(nu, order[nu]))
    if paras is None or nu not in paras.keyset:
        where = "a stats (observation) RV" if nu in stats.keyset else "not a parameter RV"
        raise NotImplementedError("order maps {!r} to the degrees of freedom, but {!r} is {}: a "
                                  "sampled nu must be a parameter RV".format(nu, nu, where))
    lo, (lo_open, _) = float(paras[nu].vlims[0]), paras[nu].open_ends
    if not (lo > 0 or (lo == 0 and lo_open)):
        raise ValueError("the prior box of the degrees of freedom {!r} must admit nu > 0 only: "
                         "its lower end is {} ({}); use vset=[a, b] with a > 0, or (0, b)"
                         .format(nu, lo, "open" if lo_open else "closed"))
    return nu


def _with_lik(spec, lik):
    """A normreg spec carries a ``lik`` entry for a non-normal likelihood only: the normal spec
    (df = inf included) is the one the catalogue has always returned."""
    if lik is not None:
        spec['lik'] = lik
    return spec


def refuse_suffstat(spec, variant):
    """suffstat=True (K2 variant 3) evaluates the normal likelihood from sufficient statistics,
    which the Student-t likelihood does not have: refused before any device call."""
    if variant == 3 and spec.get('lik') is not None:
        raise NotImplementedError("suffstat=True needs the normal likelihood: the {} likelihood "
                                  "has no sufficient statistics".format(spec['lik']['family']))


def is_scipy_mvn(obj):
    return obj is scipy.stats.multivariate_normal or \
        type(obj).__name__ in ('multivariate_normal_gen', 'multivariate_normal_frozen')


def mvn_args(args, kwds):
    args = list(args)
    mean = kwds.get('mean', args.pop(0) if args else None)
    cov = kwds.get('cov', args.pop(0) if args else None)
    if mean is None or cov is None:
        raise ValueError("multivariate_normal needs (mean, cov)")
    return np.atleast_1d(np.asarray(mean, dtype=float)), np.atleast_2d(np.asarray(cov, dtype=float))


_LOC_SCALE = {'norm': scipy.stats.norm, 't': scipy.stats.t, 'cauchy': scipy.stats.cauchy}


def _loc_scale_method(prob):
    """(family, 'logpdf' / 'pdf') if prob is that bound method of scipy.stats.norm, .t or
    .cauchy, else (None, None)."""
    owner = getattr(prob, '__self__', None)
    for family, dist in _LOC_SCALE.items():
        if owner is dist or type(owner).__name__ == family + '_gen':
            name = getattr(prob, '__name__', None)
            if name in ('logpdf', 'pdf'):
                return family, name
    return None, None


def identify_target(holder, stats, paras):
    """holder: the object set_prob was called on (SD/SP).  Returns a spec dict."""
    prob, args, kwds = holder._prob, holder._prob_args, holder._prob_kwds
    log_pscale = iscomplex(holder.pscale)
    if prob is None:
        raise NotImplementedError("no probability set: call set_prob() first")
    if is_scipy_mvn(prob):
        if type(prob).__name__ == 'multivariate_normal_frozen':
            mean, cov = np.atleast_1d(prob.mean), np.atleast_2d(prob.cov)
        else:
            mean, cov = mvn_args(args, kwds)
        names = [rv.name for rv in (stats.varlist if paras is None else
                                    stats.varlist + paras.varlist)]
        if len(mean) != len(names):
            raise ValueError("multivariate_normal over {} variables but {} means".format(
                len(names), len(mean)))
        return dict(kind='mvn', mean=mean, cov=cov, names=names, log_pscale=log_pscale)
    family, method = _loc_scale_method(prob)
    if method is not None:
        order = holder._order
        if not isinstance(order, dict):
            raise NotImplementedError(
                "scipy.stats.{}.{} needs order={{obs: 0, mean: 'loc', sd: 'scale'}}".format(
                    family, method))
        roles = {v: k for k, v in order.items()}
        try:
            obs, loc, scale = roles[0], roles['loc'], roles['scale']
        except KeyError:
            raise NotImplementedError("unrecognised order mapping {}".format(order))
        if method == 'pdf' or not log_pscale:
            raise NotImplementedError(
                "the iid {} likelihood is in the catalogue in log pscale only "
                "(set_prob(scipy.stats.{}.logpdf, ..., pscale='log'))".format(family, family))
        if paras is None or obs not in stats.keyset or {loc, scale} - paras.keyset:
            raise NotImplementedError("order must map a stats RV to 0 and parameter RVs "
                                      "to 'loc'/'scale'")
        nu = _df_role(order, family, kwds, stats, paras)
        if nu is not None:
            # theta = (loc, scale, nu): the parameter order of the kernels' sampled-nu t
            return dict(kind='normreg', has_slope=False, obs_y=obs, obs_x=None,
                        params=[loc, scale, nu], log_pscale=True,
                        lik=dict(family='t', df_param=nu))
        return _with_lik(dict(kind='normreg', has_slope=False, obs_y=obs, obs_x=None,
                              params=[loc, scale], log_pscale=True),
                         likelihood(family, (kwds or {}).get('df')))
    if isinstance(prob, (NormalRegression, StudentTRegression)):
        lik = None
        if isinstance(prob, StudentTRegression):
            if not log_pscale:
                raise NotImplementedError("StudentTRegression is in the catalogue in log pscale "
                                          "only (set_prob(..., pscale='log'))")
            lik = likelihood('t', prob.df)
        return _with_lik(dict(kind='normreg', has_slope=True, obs_y=prob.y, obs_x=prob.x,
                              params=[prob.intercept, prob.slope, prob.scale], log_pscale=True),
                         lik)
    if callable(prob):
        spec = _probe_normreg(prob, stats, paras, log_pscale)
        if spec is not None:
            import warnings
            warnings.warn(
                "probayes_b200: the Python likelihood {!r} was recognised BY PROBING as the normal "
                "linear-regression log-density log N({} | {} + {} * {}, {}) and is replaced by "
                "the device kernel; it is never called during the walk.  Pass "
                "probayes_b200.catalogue.NormalRegression(...) to state this explicitly (a "
                "function that only coincides with norm.logpdf on the probed range would be "
                "evaluated wrongly).".format(getattr(prob, '__name__', prob), spec['obs_y'],
                                             spec['params'][0], spec['params'][1], spec['obs_x'],
                                             spec['params'][2]), stacklevel=3)
            return spec
    raise NotImplementedError(
        "target {!r} is outside the device catalogue (multivariate_normal, "
        "norm.logpdf with order=..., or a normal linear-regression log-likelihood)".format(prob))


def _probe_normreg(func, stats, paras, log_pscale):
    """Is ``func`` (called by keyword with the RV names, as the reference does) the
    log-density of y ~ N(a + b*x, s)?  Checked on random probes to 1e-12."""
    if paras is None or not log_pscale or stats.nvars != 2 or paras.nvars != 3:
        return None
    try:
        sig = inspect.signature(func)
    except (TypeError, ValueError):
        return None
    names = stats.keylist + paras.keylist
    if not set(names).issubset(sig.parameters.keys()):
        return None
    rng = np.random.default_rng(12345)
    n_probe, n_obs = 24, 7

    def par_draw(rv):
        # across the variable's own range (finite limits), else a wide default
        lo, hi = (float(v) for v in rv.vlims)
        lo = lo if np.isfinite(lo) else -50.
        hi = hi if np.isfinite(hi) else 50.
        return lo + (hi - lo) * rng.uniform(0.02, 0.98, n_probe)

    obs_sets = [{k: rng.normal(0., 1., n_obs) * sc + off for k in stats.keylist}
                for sc, off in zip(rng.uniform(0.1, 30., n_probe), rng.normal(0., 20., n_probe))]
    par_sets = {k: par_draw(paras[k]) for k in paras.keylist}
    got = []
    for i in range(n_probe):
        pars = {k: float(par_sets[k][i]) for k in paras.keylist}
        try:
            g = np.asarray(func(**obs_sets[i], **pars), dtype=float)
        except Exception:
            return None
        if g.shape != (n_obs,):
            return None
        got.append(g)
    for (xk, yk) in itertools.permutations(stats.keylist, 2):
        for (a, b, s) in itertools.permutations(paras.keylist, 3):
            ok = True
            for i in range(n_probe):
                sd = par_sets[s][i]
                if not sd > 0:
                    continue
                want = scipy.stats.norm.logpdf(obs_sets[i][yk], loc=par_sets[a][i] +
                                               par_sets[b][i] * obs_sets[i][xk], scale=sd)
                if not np.allclose(got[i], want, rtol=1e-12, atol=1e-12, equal_nan=True):
                    ok = False
                    break
            if ok:
                return dict(kind='normreg', has_slope=True, obs_y=yk, obs_x=xk,
                            params=[a, b, s], log_pscale=True)
    return None


# ---------------------------------------------------------------------------
def _frozen_norm_scale(obj):
    if type(obj).__name__ == 'rv_continuous_frozen' and getattr(obj.dist, 'name', '') == 'norm':
        loc = obj.kwds.get('loc', obj.args[0] if len(obj.args) > 0 else 0.)
        scale = obj.kwds.get('scale', obj.args[1] if len(obj.args) > 1 else 1.)
        if float(loc) != 0.:
            raise NotImplementedError("normal proposals must be centred (loc=0)")
        return float(scale)
    return None


def identify_proposal(rf, target_pscale, injected=False):
    """rf: the RF whose set_delta / set_tran describe the proposal.
    Returns dict(kind, scale[D], radius, chol, coef)."""
    D = rf.nvars
    delta, kw = rf._delta, rf._delta_kwds
    lengths = rf.lengths
    out = dict(kind='normal', scale=np.ones(D), radius=0.0, chol=None, coef=1.0,
               bound=bool(kw.get('bound')))
    if isinstance(rf._tfun, np.ndarray):
        out['chol'] = np.asarray(rf._tfun, dtype=float)
    fro = _frozen_norm_scale(delta)
    if fro is not None:
        out.update(kind='normal', scale=np.full(D, fro))
    elif isinstance(delta, list):
        assert len(delta) == 1, "List delta requires a single element"
        d = float(delta[0])
        scale = np.full(D, d)
        if kw.get('scale'):
            assert np.all(np.isfinite(lengths)), "Cannot scale by infinite length"
            scale = d * lengths
        if rf._delta_args:
            unscale = rf._delta_args[0]
            assert isinstance(unscale, dict), \
                "Optional positional arguments must comprises a single dict"
            for i, key in enumerate(rf.keylist):
                if key in unscale:
                    v = unscale[key]
                    scale[i] = float(v[0] if isinstance(v, list) else v)
        out.update(kind='uniform', scale=scale)
    elif isinstance(delta, tuple):
        assert len(delta) == 1, "Tuple delta must contain one element"
        d = float(delta[0])
        assert np.all(np.isfinite(lengths)), "Cannot spherise Variable with infinite length"
        if kw.get('scale'):
            rss = float(np.sqrt(np.sum(lengths ** 2)))
            out.update(kind='spherical', radius=d * rss, scale=lengths.copy())
        else:
            out.update(kind='spherical', radius=d, scale=np.ones(D))
    elif delta is None or callable(delta):
        if not injected:
            raise NotImplementedError(
                "a Python-callable (or missing) delta cannot run on the device: use [d], (d,), "
                "a frozen scipy.stats.norm(0, s), or inject the draws (inj_delta=...)")
    else:
        raise NotImplementedError("unrecognised delta specification {!r}".format(delta))
    # asymmetric (q, r) pair: hastings_scores multiplies the linear proposal density
    # into the target *in the target's pscale* (sp_utils.py:52-64, rf.py:531-536)
    tran = rf._tran
    if isinstance(tran, tuple):
        assert len(tran) == 2 and all(callable(t) for t in tran), \
            "tuple transitions must be a (q, r) pair of callables"
        vals = _probe_constant(tran[0], rf)
        if vals is None:
            raise NotImplementedError("state-dependent asymmetric proposal densities are not "
                                      "in the device catalogue")
        out['coef'] = float(rescale(vals, rf.pscale, 1.)) if iscomplex(target_pscale) else 1.0
    return out


def _probe_constant(func, rf):
    rng = np.random.default_rng(99)
    seen = []
    for _ in range(3):
        kwds = {}
        for rv in rf.varlist:
            lo, hi = rv.vlims
            lo = lo if np.isfinite(lo) else -1.
            hi = hi if np.isfinite(hi) else 1.
            a, b = rng.uniform(lo, hi, 2)
            kwds[rv.name] = float(a)
            kwds[rv.name + "'"] = float(b)
        try:
            seen.append(float(func(**kwds)))
        except Exception:
            return None
    return seen[0] if max(seen) == min(seen) else None


# ---------------------------------------------------------------------------
# rejection sampling (examples/omc/omc_rejection_sp_circle.py:26-39)
# ---------------------------------------------------------------------------
class BallIndicator:
    """Explicit target spec: 1.0 where sum_j (x_j - centre_j)^2 <= radius^2, else 0.0."""

    def __init__(self, radius, centre=0.):
        self.radius, self.centre = float(radius), centre


class NormalProduct:
    """Explicit proposal-density spec: prod_j scipy.stats.norm.pdf(x_j, loc_j, scale_j)."""

    def __init__(self, loc=0., scale=1.):
        self.loc, self.scale = loc, scale


class BoxUniform:
    """Explicit proposal-density spec: the box-uniform density prod_j 1 / length_j."""


def _warn_probed(what, func, as_what):
    import warnings
    warnings.warn("probayes_b200: the Python {} {!r} was recognised BY PROBING as {} and is "
                  "replaced by the device kernel; it is never called during the walk.  Pass the "
                  "explicit probayes_b200.catalogue spec to state this."
                  .format(what, getattr(func, '__name__', func), as_what), stacklevel=4)


def _sig(x, digits=12):
    return float(('%.' + str(digits) + 'g') % x)


def identify_rejection_target(prob, args, kwds, rvs):
    """-> dict(kind='ball', radius, centre [P]) or NotImplementedError."""
    P = len(rvs)
    names = [rv.name for rv in rvs]
    if isinstance(prob, BallIndicator):
        return dict(kind='ball', radius=prob.radius,
                    centre=np.broadcast_to(np.asarray(prob.centre, float), (P,)).copy())
    if callable(prob):
        lims = np.array([rv.vlims for rv in rvs], dtype=float)
        if np.isfinite(lims).all():
            f = lambda pt: float(np.asarray(prob(*args, **dict(zip(names, pt)), **kwds)))
            try:
                centre = lims.mean(axis=1)
                if f(centre) == 1.0:
                    # radius by bisection along the first axis, then verified on random points
                    lo, hi = 0.0, float(lims[0, 1] - centre[0]) * 4.0
                    for _ in range(80):
                        mid = 0.5 * (lo + hi)
                        pt = centre.copy()
                        pt[0] += mid
                        lo, hi = (mid, hi) if f(pt) == 1.0 else (lo, mid)
                    radius = _sig(lo)
                    rng = np.random.default_rng(2468)
                    pts = lims[:, 0] + (lims[:, 1] - lims[:, 0]) * rng.random((256, P))
                    want = (((pts - centre) ** 2).sum(axis=1) <= radius ** 2).astype(float)
                    got = np.array([f(pt) for pt in pts])
                    if np.array_equal(got, want) and 0 < want.sum() < len(want):
                        _warn_probed('target', prob, 'the indicator of a ball of radius {} '
                                     'centred at {}'.format(radius, list(centre)))
                        return dict(kind='ball', radius=radius, centre=centre)
            except Exception:
                pass
    raise NotImplementedError("rejection-sampling target {!r} is outside the device catalogue "
                              "(BallIndicator)".format(prob))


def identify_rejection_prop(prop, args, kwds, rvs):
    """-> dict(kind='normal', loc [P], scale [P]) | dict(kind='box')."""
    P = len(rvs)
    names = [rv.name for rv in rvs]
    if isinstance(prop, BoxUniform):
        return dict(kind='box')
    if isinstance(prop, NormalProduct):
        return dict(kind='normal', loc=np.broadcast_to(np.asarray(prop.loc, float), (P,)).copy(),
                    scale=np.broadcast_to(np.asarray(prop.scale, float), (P,)).copy())
    if callable(prop):
        f = lambda pt: float(np.asarray(prop(*args, **dict(zip(names, pt)), **kwds)))
        try:
            base = np.zeros(P)
            g0 = np.log(f(base))
            loc, scale = np.zeros(P), np.ones(P)
            for j in range(P):
                e = np.zeros(P)
                e[j] = 1.0
                gp, gm = np.log(f(base + e)), np.log(f(base - e))
                inv_var = -(gp - 2.0 * g0 + gm)               # second difference = -1 / s^2
                if not inv_var > 0:
                    raise ValueError
                scale[j] = _sig(1.0 / np.sqrt(inv_var))
                loc[j] = _sig(0.5 * (gp - gm) / inv_var) if abs(gp - gm) > 1e-13 else 0.0
            rng = np.random.default_rng(1357)
            pts = loc + scale * rng.standard_normal((64, P)) * 1.5
            want = np.prod(scipy.stats.norm.pdf(pts, loc=loc, scale=scale), axis=1)
            got = np.array([f(pt) for pt in pts])
            if np.allclose(got, want, rtol=1e-12, atol=0.0):
                _warn_probed('proposal density', prop, 'the product of normal pdfs with loc {} '
                             'and scale {}'.format(list(loc), list(scale)))
                return dict(kind='normal', loc=loc, scale=scale)
        except Exception:
            pass
    raise NotImplementedError("proposal density {!r} is outside the device catalogue "
                              "(NormalProduct, BoxUniform)".format(prop))


class _Obj:
    def __init__(self, **kw):
        self.__dict__.update(kw)


def identify_scores(func, args=(), kwds=None):
    """'p' for opqr -> opqr.p.prob, 'p/q' for opqr -> opqr.p.prob / opqr.q.prob."""
    kwds = kwds or {}
    try:
        a = func(_Obj(o=None, p=_Obj(prob=0.37), q=_Obj(prob=0.11), r=None), *args, **kwds)
        b = func(_Obj(o=None, p=_Obj(prob=0.05), q=_Obj(prob=0.4), r=None), *args, **kwds)
        if np.isclose(a, 0.37, rtol=1e-14) and np.isclose(b, 0.05, rtol=1e-14):
            return 'p'
        if np.isclose(a, 0.37 / 0.11, rtol=1e-14) and np.isclose(b, 0.05 / 0.4, rtol=1e-14):
            return 'p/q'
    except Exception:
        pass
    raise NotImplementedError("scores must be 'metropolis' | 'hastings' | 'gibbs', or a function "
                              "equal to opqr.p.prob or opqr.p.prob / opqr.q.prob (custom Python "
                              "score functions cannot run in the kernel)")


def identify_thresh(func, args=(), kwds=None):
    """('uniform', low, high) for np.random.uniform(low=, high=)."""
    kwds = dict(kwds or {})
    if getattr(func, '__name__', '') == 'uniform' and \
            'random' in str(getattr(func, '__module__', None) or
                            type(getattr(func, '__self__', None)).__module__):
        a = list(args)
        low = kwds.pop('low', a.pop(0) if a else 0.0)
        high = kwds.pop('high', a.pop(0) if a else 1.0)
        if not kwds and not a:
            return ('uniform', float(low), float(high))
    raise NotImplementedError("thresh must be one of the MCMC sampler names or "
                              "np.random.uniform with low / high")


def identify_update(func, args=(), kwds=None):
    """'s>=t' for stu -> stu.s >= stu.t."""
    kwds = kwds or {}
    try:
        probes = [(0.7, 0.2, True), (0.1, 0.2, False), (0.2, 0.2, True), (0.0, 1e-300, False)]
        if all(bool(func(_Obj(s=s_, t=t_, u=None, v=None), *args, **kwds)) is w
               for s_, t_, w in probes):
            return 's>=t'
    except Exception:
        pass
    raise NotImplementedError("update must be one of the MCMC sampler names or a function equal "
                              "to stu.s >= stu.t")
