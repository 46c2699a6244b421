"""SD -- stochastic dependence between a field of observed statistics (leafs) and
a field of parameters (roots), or a single joint field.

Mirror of the reference interface on the hot path (probayes/sd.py:39-42,71-116,
148-161): ``SD(stats, paras)`` / ``SD(x & y)``, ``set_prob``, ``set_tran``,
``set_delta``, ``set_tfun`` (accepting one of the member fields as proxy, as the
reference does) and ``__call__(values, iid=, joint=)`` -- the discrete-grid exact
inference entry point, which here runs as the K3 kernel and returns a
device-backed ``PD``.
"""
import collections
import numpy as np

from .rv import RV
from .rf import RF
from .pd import PD
from .pscales import eval_pscale, prod_pscale, iscomplex
from .vtypes import isunitsetint
from . import catalogue


class SD:

    def __init__(self, *args):
        fields = []
        for arg in args:
            if isinstance(arg, RV):
                arg = RF(arg)
            assert isinstance(arg, RF), \
                "SD arguments must be RV / RF instances, not {}".format(type(arg))
            fields.append(arg)
        assert fields, "SD needs at least one field"
        if len(fields) == 1:
            self._leafs, self._roots = fields[0], None
        elif len(fields) == 2:
            self._leafs, self._roots = fields[0], fields[1]
        else:
            raise NotImplementedError("SD(stats, paras) or SD(field) only")
        allvars = self._leafs.varlist + (self._roots.varlist if self._roots else [])
        self._all = RF(*allvars)
        self._id = '_and_'.join(rv.name for rv in allvars)
        # the field whose values are sampled / proposed
        self._state_rf = self._roots if self._roots is not None else self._leafs
        self._own_rf = RF(*self._state_rf.varlist)       # proposal specs set on the SD itself
        self._tran_obj = self._own_rf
        self._delta_obj = self._own_rf
        self._prob, self._prob_args, self._prob_kwds, self._order = None, (), {}, None
        self._prop, self._prop_args, self._prop_kwds = None, (), {}
        self._pscale = self._all.pscale
        self.Delta = self._state_rf.Delta
        self.opqr = collections.namedtuple(self._id, ['o', 'p', 'q', 'r'])

    # ---- members --------------------------------------------------------------------------
    @property
    def leafs(self):
        return self._leafs

    @property
    def roots(self):
        return self._roots

    @property
    def pscale(self):
        return self._pscale

    @property
    def prob(self):
        return self._prob

    @property
    def _cond_cov(self):
        return self._tran_obj._cond_cov

    def _member(self, spec):
        """The member field ``spec`` refers to (sd.py:88-116 / leafs_roots), if any."""
        if isinstance(spec, RF):
            for rf in (self._leafs, self._roots):
                if rf is not None and (spec is rf or spec.keyset == rf.keyset):
                    return spec
            raise ValueError("Field {} is not a member of this dependence".format(spec))
        return None

    def set_prob(self, prob=None, *args, **kwds):
        kwds = dict(kwds)
        if 'pscale' in kwds:
            self._pscale = eval_pscale(kwds.pop('pscale'))
        else:
            self._pscale = prod_pscale([rv.pscale for rv in self._all.varlist])
        self._order = kwds.pop('order', None)
        kwds.pop('passdims', None)
        self._prob, self._prob_args, self._prob_kwds = prob, tuple(args), kwds

    @property
    def prop(self):
        return self._prop

    def set_prop(self, prop=None, *args, **kwds):
        """Proposal DENSITY for ordinary Monte Carlo / rejection sampling (rf.py:146-161):
        a callable of the variables, or a catalogue spec (NormalProduct, BoxUniform)."""
        if prop is not None:
            assert self._tran_obj.tran is None, \
                "Cannot assign both proposition and transition probabilities"
        kwds = dict(kwds)
        kwds.pop('deps', None)
        self._prop, self._prop_args, self._prop_kwds = prop, tuple(args), kwds

    def set_tran(self, tran=None, *args, **kwds):
        member = self._member(tran)
        if member is not None:
            self._tran_obj = member
            return member.tran
        self._tran_obj = self._own_rf
        self._own_rf.set_tran(tran, *args, **kwds)
        return self._own_rf.tran

    def set_tfun(self, tfun=None, *args, **kwds):
        member = self._member(tfun)
        if member is not None:
            self._tran_obj = member
            return member.tfun
        self._tran_obj = self._own_rf
        self._own_rf.set_tfun(tfun, *args, **kwds)
        return self._own_rf.tfun

    def set_delta(self, delta=None, *args, **kwds):
        member = self._member(delta)
        if member is not None:
            self._delta_obj = member
            return
        self._delta_obj = self._own_rf
        self._own_rf.set_delta(delta, *args, **kwds)

    def _proposal_rf(self):
        """One RF view carrying the delta of ``_delta_obj`` and the tran of ``_tran_obj``."""
        rf = self._delta_obj
        if self._tran_obj is not rf:
            merged = RF(*rf.varlist)
            merged._delta, merged._delta_args, merged._delta_kwds = \
                rf._delta, rf._delta_args, rf._delta_kwds
            t = self._tran_obj
            merged._tran, merged._tfun, merged._sym_tran = t._tran, t._tfun, t._sym_tran
            merged._tsteps, merged._cond_cov = t._tsteps, t._cond_cov
            return merged
        return rf

    def parse_values(self, values):
        """RV-object keys -> names; 'x,y' joint keys -> separate entries."""
        out = collections.OrderedDict()
        for key, val in values.items():
            key = key.name if isinstance(key, RV) else key
            if ',' in key:
                names = key.split(',')
                assert len(names) == len(val), "Joint key {} needs {} arrays".format(key, len(names))
                for n, v in zip(names, val):
                    out[n] = v
            else:
                out[key] = val
        return out

    # ---- discrete grid exact inference ---------------------------------------------------------
    def __call__(self, values=None, iid=False, joint=False, **kwds):
        """model({x: data, 'mu': {M}, 'sigma': {S}}, iid=True, joint=True) -> PD of the
        log-joint over the (mu, sigma) grid (examples/dgei/dgei_norm1d_improved.py:36-37).
        A Student-t whose nu is a model parameter takes nu as a scalar value ('nu': 4.) and
        gives the (mu, sigma) grid at that nu, its prior included when ``joint``.
        ``suffstat=True`` (new, opt-in): evaluate it from centred sufficient statistics of
        the observations -- O(M S) instead of O(N M S), same values to fp64 round-off."""
        suffstat = bool(kwds.pop('suffstat', False))
        from .engine import get_engine
        assert isinstance(values, dict), "values must be a dictionary keyed by variable"
        values = self.parse_values(values)
        spec = catalogue.identify_target(self, self._leafs, self._roots)
        if spec['kind'] != 'normreg' or spec['has_slope']:
            raise NotImplementedError("grid evaluation is in the catalogue for the iid normal, "
                                      "Student-t or Cauchy (mu, sigma) likelihood only")
        if not iid:
            raise NotImplementedError("the un-reduced [N, M, S] likelihood tensor is never "
                                      "materialised on the device: call with iid=True")
        catalogue.refuse_suffstat(spec, 3 if suffstat else 0)
        obs, (kmu, ksg) = spec['obs_y'], spec['params'][:2]
        lik = spec.get('lik')
        knu = (lik or {}).get('df_param')
        if knu is not None:
            nu = values.get(knu)
            if nu is None:
                raise ValueError("values must give the degrees of freedom '{}' a scalar".format(knu))
            if isunitsetint(nu) or np.ndim(nu) > 0:
                raise NotImplementedError("a grid over '{}' would be a three-axis (mu, sigma, nu) "
                                          "grid: give it a scalar value".format(knu))
            nu = float(nu)
            lik = catalogue.likelihood('t', nu)        # the fixed-nu grid at this nu
        data = np.ascontiguousarray(np.ravel(np.asarray(values[obs], dtype=np.float64)))
        grids = {}
        for key in (kmu, ksg):
            rv = self._roots[key]
            v = values[key]
            grids[key] = np.ravel(rv.evaluate(v)) if isunitsetint(v) else \
                np.ravel(np.asarray(v, dtype=np.float64))
        M, S = len(grids[kmu]), len(grids[ksg])
        if joint:
            lpm = np.asarray(self._roots[kmu].eval_prob(grids[kmu]), dtype=np.float64)
            lps = np.asarray(self._roots[ksg].eval_prob(grids[ksg]), dtype=np.float64)
            from .pscales import rescale
            lpm = rescale(lpm, self._roots[kmu].pscale, 'log')
            lps = rescale(lps, self._roots[ksg].pscale, 'log')
            if knu is not None:                        # nu's prior: the same for every cell
                lpm = lpm + float(rescale(self._roots[knu].eval_prob(nu),
                                          self._roots[knu].pscale, 'log'))
        else:
            lpm, lps = np.zeros(M), np.zeros(S)
        eng = get_engine()
        lj = eng.grid_norm_logjoint(eng.to_device(data), eng.to_device(grids[kmu]),
                                    eng.to_device(grids[ksg]), eng.to_device(lpm),
                                    eng.to_device(lps), suffstat=suffstat, lik=lik)
        order = [k for k in self._roots.keylist if k in (kmu, ksg)]
        vals = collections.OrderedDict()
        dims = collections.OrderedDict()
        for key in order:
            vals[key] = grids[key]
            dims[key] = 0 if key == kmu else 1
        if order[0] != kmu:
            lj = lj.t().contiguous()
            dims = collections.OrderedDict((k, 1 - d) for k, d in dims.items())
        fixed = []
        if knu is not None:
            vals[knu], dims[knu] = nu, None
            fixed = ["{}={}".format(knu, nu)]
        vals[obs] = {len(data)}
        dims[obs] = None
        names = [k + "=[]" for k in order] + fixed + ["{}={{{}}}".format(obs, len(data))]
        cond = "" if joint else "|" + ",".join([k + "=[]" for k in order] + fixed)
        name = ",".join(names) if joint else names[-1] + cond
        return PD(name, vals, dims=dims, prob=lj, pscale=self._pscale)
