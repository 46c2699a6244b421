"""PD -- probability distribution: named values + dims + prob + pscale.

Host-side mirror of the reference's result container (probayes/pd.py,
distribution.py, named_dict.py) for what the hot path returns, with the
array algebra of the path running in libpbx:

  * ``prob`` may be backed by a device tensor (a DGEI grid of 134 MB stays in HBM;
    ``.prob`` copies to the host on first access, ``.prob_device`` does not);
  * ``conditionalise`` / ``marginal`` / ``marginalise`` / ``rescaled`` on a
    2-D device-backed PD are the K4 kernels (probayes/pd.py:136-165,168-211,
    214-295,496-499);
  * ``expectation`` / ``quantile`` / ``sorted`` on a device-backed PD (1-D sample
    sets / marginals, 2-D grids) are the K6 kernels: radix argsort + gathers,
    reduce-then-scan cumulative probability + digitize, one-pass weighted sums
    (probayes/pd.py:373-405,408-461,464-493); only the O(1) bracket interpolation
    and the name/dims bookkeeping stay in Python.  Host-backed PDs (scalars, small
    user-built arrays) keep the reference's numpy arithmetic.

Names follow the reference: ``"mu=[],sigma=[]|x={60}"`` -- ``key=[]`` for array
values, ``key={n}`` for an iid-reduced set, ``key=value`` for scalars; marginal
keys before the ``|``, conditional keys after it.
"""
import collections
import numpy as np

from .pscales import eval_pscale, iscomplex, rescale, div_prob, log_prob, exp_logp, prod_rule
from .vtypes import isscalar, isunitset, isunitsetint


def str_margcond(name):
    marg, cond = collections.OrderedDict(), collections.OrderedDict()
    if not name:
        return marg, cond
    left, _, right = name.partition('|')
    for part, dst in ((left, marg), (right, cond)):
        for item in (part.split(',') if part else []):
            key = item.split('=')[0]
            dst[key] = item
    return marg, cond


def margcond_str(marg, cond):
    m = ','.join(marg.values() if isinstance(marg, dict) else marg)
    c = ','.join(cond.values() if isinstance(cond, dict) else cond)
    return m + '|' + c if c else m


def _label(key, val):
    if isinstance(val, set):
        return "{}={}".format(key, val)
    if isscalar(val):
        return "{}={}".format(key, val)
    return key + "=[]"


def _is_tensor(a):
    return type(a).__module__.startswith("torch")


class PD(collections.OrderedDict):
    """PD(name, vals, dims=None, prob=None, pscale=None)."""

    def __init__(self, name, vals=None, dims=None, prob=None, pscale=None, **kwds):
        super().__init__()
        if vals is not None:
            self.update(vals)
        self.update(kwds)
        self._marg, self._cond = str_margcond(name)
        for key in self.keys():
            assert key in self._marg or key in self._cond, \
                "Variable {} not accounted for in name {}".format(key, name)
        self._set_dims(dims)
        self._pscale = eval_pscale(pscale)
        self._prob_dev = None
        self._prob = None
        self._cache = {}            # device-side by-products (marginals of a posterior)
        self._vals_dev = {}         # key -> 1-D device tensor mirroring an array value
        self._monotonic = {}        # key -> True where known (set by sorted())
        self.prob = prob

    # ---- bookkeeping ------------------------------------------------------------
    def _set_dims(self, dims):
        self._aresingleton = [isscalar(v) or isunitset(v) for v in self.values()]
        if dims is None:
            dims, k = collections.OrderedDict(), 0
            for key, single in zip(self.keys(), self._aresingleton):
                dims[key] = None if single else k
                k += 0 if single else 1
        self._dims = collections.OrderedDict((k, dims.get(k)) for k in self.keys())
        sizes = {}
        for key, single in zip(self.keys(), self._aresingleton):
            if single:
                continue
            shp = np.shape(self[key])
            if len(shp) > 1 and int(np.prod(shp)) != max(shp):
                # batched samples [C, R]: the array spans consecutive dims from dims[key]
                for off, n in enumerate(shp):
                    sizes[self._dims[key] + off] = int(n)
            else:
                sizes[self._dims[key]] = int(np.size(self[key]))
        self._shape = [sizes[k] for k in sorted(sizes)]
        # refresh labels of scalar / set values in the name
        for key, single in zip(self.keys(), self._aresingleton):
            label = _label(key, self[key]) if single else None
            for group in (self._marg, self._cond):
                if key in group and label is not None:
                    group[key] = label
        self._name = margcond_str(self._marg, self._cond)

    @property
    def name(self):
        return self._name

    @property
    def marg(self):
        return self._marg

    @property
    def cond(self):
        return self._cond

    @property
    def dims(self):
        return self._dims

    @property
    def shape(self):
        return self._shape

    @property
    def ndim(self):
        return len(self._shape)

    @property
    def size(self):
        return int(np.prod(self._shape)) if self._shape else 1

    @property
    def issingleton(self):
        return all(self._aresingleton)

    @property
    def short_name(self):
        m, c = ','.join(self._marg.keys()), ','.join(self._cond.keys())
        return m + '|' + c if c else m

    @property
    def pscale(self):
        return self._pscale

    # ---- probabilities ------------------------------------------------------------
    @property
    def prob(self):
        """numpy array / scalar (device-backed grids are copied on first access)."""
        if self._prob is None and self._prob_dev is not None:
            self._prob = self._prob_dev.detach().cpu().numpy()
        return self._prob

    @prob.setter
    def prob(self, prob):
        self._prob, self._prob_dev = None, None
        if prob is None:
            return
        if _is_tensor(prob):
            if prob.is_cuda:
                self._prob_dev = prob
            else:
                self._prob = prob.numpy()
            shape = list(prob.shape)
        else:
            self._prob = prob
            shape = [] if isscalar(prob) else list(np.shape(prob))
        if self.issingleton:
            assert shape == [], "Singleton vals with non-scalar prob"
        else:
            assert shape == self._shape, \
                "Mismatch in dimensions between values {} and probabilities {}".format(
                    self._shape, shape)

    @property
    def prob_device(self):
        """The device tensor behind ``prob`` (None for host-backed PDs)."""
        return self._prob_dev

    def set_device_vals(self, vals_dev):
        """Registers device mirrors of array values (so sorted() / expectation() need
        no upload).  vals_dev: {key: 1-D fp64 device tensor}."""
        for k, t in vals_dev.items():
            assert k in self and int(t.numel()) == int(np.size(self[k]))
            self._vals_dev[k] = t

    def _dev_val(self, key, exponent=None):
        """1-D device tensor of the values of ``key`` (uploaded on first use)."""
        eng = self._engine()
        if exponent:
            return eng.to_device(np.ravel(np.asarray(self[key], dtype=float)) ** exponent)
        if key not in self._vals_dev:
            self._vals_dev[key] = eng.to_device(np.ravel(np.asarray(self[key], dtype=float)))
        return self._vals_dev[key]

    def _new(self, name, vals, dims, prob, pscale=None):
        return PD(name, vals, dims=dims, prob=prob,
                  pscale=self._pscale if pscale is None else pscale)

    # ---- device helpers ---------------------------------------------------------------
    def _engine(self):
        from .engine import get_engine
        return get_engine(self._prob_dev.device.index)

    def rescaled(self, pscale=None):
        """PD with prob converted to ``pscale`` (default linear): pd.py:496-499."""
        dst = eval_pscale(pscale)
        if self._prob_dev is not None and iscomplex(self._pscale) != iscomplex(dst) \
                and self._pscale in (0j, 1.) and dst in (0j, 1.):
            eng = self._engine()
            out = self._prob_dev.clone()
            out = eng.exp_logp_(out) if iscomplex(self._pscale) else eng.log_prob_(out)
            res = self._new(self._name, collections.OrderedDict(self), self._dims, out, dst)
            res._vals_dev, res._monotonic = dict(self._vals_dev), dict(self._monotonic)
            return res
        prob = rescale(np.copy(self.prob), self._pscale, dst)
        return self._new(self._name, collections.OrderedDict(self), self._dims, prob, dst)

    # ---- marginal-sum algebra ----------------------------------------------------------
    def _device_linear(self, what):
        """True / False for a device-backed PD in linear (1.) / log (0j) pscale; any other
        pscale has no kernel and raises instead of falling back to the host."""
        if iscomplex(self._pscale) and self._pscale == 0j:
            return False
        if not iscomplex(self._pscale) and self._pscale == 1.:
            return True
        raise NotImplementedError("{} of a device-backed PD with pscale {} is outside the "
                                  "device catalogue (log and linear pscales are): call "
                                  ".rescaled() first".format(what, self._pscale))

    def _split_keys(self, keys):
        if isinstance(keys, str):
            keys = [keys]
        for key in keys:
            assert key in self._marg, \
                "Key {} not marginal in distribution {}".format(key, self._name)
        return set(keys)

    def marginalise(self, keys):
        """from p(A, key | B) returns p(A | B): exp -> sum over key axes -> clamped
        log (pd.py:136-165)."""
        keys = self._split_keys(keys)
        marg = collections.OrderedDict(self._marg)
        vals, dims, axes, shift = collections.OrderedDict(), collections.OrderedDict(), set(), 0
        for key, single in zip(self.keys(), self._aresingleton):
            if key in keys:
                assert not single, "Cannot marginalise along scalar for key {}".format(key)
                axes.add(self._dims[key])
                marg.pop(key)
                shift += 1
            else:
                if not single:
                    dims[key] = self._dims[key] - shift
                vals[key] = self[key]
        name = margcond_str(marg, self._cond)
        cached = self._cache.get(("marginalise", frozenset(keys)))
        if cached is not None:
            return self._new(name, vals, dims, cached)
        if self._prob_dev is not None:
            # device-backed: kernels only (no silent host path).  log (0j) and linear (1.)
            # pscales, 1-D / 2-D arrays -- everything the device catalogue produces
            linear = self._device_linear("marginalise")
            eng = self._engine()
            import torch
            if len(axes) == self.ndim:
                # every array axis goes: log_prob(sum exp_logp(p)) without a max shift, as
                # the reference evaluates it (underflows like the reference for large |log p|)
                if linear:
                    tot = eng.grid_max_sumexp(self._prob_dev.reshape(-1), linear=True)[1:2]
                else:
                    one = torch.ones(1, dtype=torch.float64, device=self._prob_dev.device)
                    zero = torch.zeros(1, dtype=torch.float64, device=self._prob_dev.device)
                    # row sums of exp_logp(prob) from the posterior pass (max = 0, sum = 1,
                    # marginalise semantics), then their plain sum.  A 2-D PD keeps its rows:
                    # one warp finishes a row, from one partial per 128 columns
                    p2 = self._prob_dev if self.ndim == 2 else self._prob_dev.reshape(1, -1)
                    _, rows, _ = eng.grid_posterior2(p2, zero, one, want_post=False, marg_log=4)
                    tot = eng.log_prob_(eng.grid_max_sumexp(rows, linear=True)[1:2])
                return self._new(name, vals, dims, float(tot.item()))
            if self.ndim == 2 and len(axes) == 1:
                one = torch.ones(1, dtype=torch.float64, device=self._prob_dev.device)
                zero = torch.zeros(1, dtype=torch.float64, device=self._prob_dev.device)
                # sum_axis exp_logp(prob): the posterior pass with max = 0, sum = 1 and no
                # posterior output; row / column sums, through the clamped log for log pscale
                _, rows, cols = eng.grid_posterior2(self._prob_dev, zero, one, linear,
                                                    want_post=False, marg_log=4 if linear else 7)
                return self._new(name, vals, dims, rows if 1 in axes else cols)
            if not axes:
                return self._new(name, vals, dims, self._prob_dev)
            raise NotImplementedError("marginalise of a device-backed PD with {} array axes "
                                      "over {} of them is outside the device catalogue"
                                      .format(self.ndim, len(axes)))
        prob = rescale(self.prob, self._pscale, 1.)
        prob = rescale(np.sum(prob, axis=tuple(axes), keepdims=False), 1., self._pscale)
        return self._new(name, vals, dims, prob)

    def marginal(self, keys):
        """from p(A, key | B) returns p(key | B) (pd.py:168-211)."""
        keys = self._split_keys(keys)
        others = set()
        for key, single in zip(self.keys(), self._aresingleton):
            if key in self._marg and not single and key not in keys:
                others.add(key)
        scalars = {k for k, s in zip(self.keys(), self._aresingleton) if s and k in self._marg}
        if scalars:
            assert scalars.issubset(keys), \
                "If evaluating marginal, must include all marginal scalars in {}".format(
                    list(self._marg.keys()))
        return self.marginalise(others)

    def conditionalise(self, keys):
        """from p(A, key | B) returns p(A | B, key).  Conditioning on a scalar /
        iid-reduced key normalises the whole array: prob - max; exp; / max(tiny,
        sum); clamped log (pd.py:214-295, arithmetic 285-295)."""
        keys = self._split_keys(keys)
        marg = collections.OrderedDict(self._marg)
        cond = collections.OrderedDict(self._cond)
        normalise = False
        array_keys = []
        for key, single in zip(self.keys(), self._aresingleton):
            if key in keys:
                cond[key] = marg.pop(key)
                if single:
                    normalise = True
                else:
                    array_keys.append(key)
        name = margcond_str(marg, cond)
        if array_keys:
            return self._conditionalise_array(name, array_keys, normalise)
        vals = collections.OrderedDict(self)
        if not normalise:
            return self._new(name, vals, self._dims, self._prob_dev
                             if self._prob_dev is not None else self.prob)
        if self._prob_dev is not None:
            linear = self._device_linear("conditionalise")
            eng = self._engine()
            if self.ndim == 1:
                r = eng.grid_conditionalise(self._prob_dev.reshape(1, -1), linear=linear)
                out = self._new(name, vals, self._dims, r["post"].reshape(-1))
                out._vals_dev = dict(self._vals_dev)
                return out
            if self.ndim == 2:
                r = eng.grid_conditionalise(self._prob_dev, linear=linear)
                out = self._new(name, vals, self._dims, r["post"])
                # the posterior pass already produced both marginal sums
                akeys = [k for k, s in zip(self.keys(), self._aresingleton) if not s]
                k0 = [k for k in akeys if self._dims[k] == 0]
                k1 = [k for k in akeys if self._dims[k] == 1]
                out._cache[("marginalise", frozenset(k1))] = r["marg_mu"]
                out._cache[("marginalise", frozenset(k0))] = r["marg_sigma"]
                return out
            raise NotImplementedError("conditionalise of a device-backed PD with {} array "
                                      "axes is outside the device catalogue".format(self.ndim))
        prob = np.asarray(self.prob, dtype=float)
        if iscomplex(self._pscale):
            prob = prob - prob.max()
        prob = rescale(prob, self._pscale, 1.)
        prob = div_prob(prob, np.sum(prob))
        return self._new(name, vals, self._dims, rescale(prob, 1., self._pscale))

    def _conditionalise_array(self, name, array_keys, normalise):
        """p(A, K | B) -> p(A | B, K) for an ARRAY-valued key K (pd.py:214-295): K's axis
        moves behind the remaining marginal axis and every slice along it is divided by its
        sum over that axis (pd.py:285-295: to linear, [normalise,] div_prob by the keepdims
        sum, back to the PD's pscale).  2-D arrays with one conditioned array key."""
        akeys = [k for k, sg in zip(self.keys(), self._aresingleton) if not sg]
        if self.ndim != 2 or len(array_keys) != 1 or len(akeys) != 2:
            raise NotImplementedError("conditionalising on array-valued keys is in the "
                                      "catalogue for 2-D PDs and one such key")
        key = array_keys[0]
        other = [k for k in akeys if k != key][0]
        assert other in self._marg, \
            "Key {} must stay marginal when conditionalising on {}".format(other, key)
        ax = self._dims[key]                              # axis of K in the stored array
        dims = collections.OrderedDict(self._dims)
        dims[other], dims[key] = 0, 1
        vals = collections.OrderedDict()
        for k, v in self.items():
            if k in akeys:
                shp = [1, 1]
                shp[dims[k]] = int(np.size(v))
                vals[k] = np.reshape(np.asarray(v), shp)
            else:
                vals[k] = v
        if self._prob_dev is not None:
            linear = self._device_linear("conditionalise")
            eng = self._engine()
            import torch
            base = self._prob_dev
            if normalise:
                base = eng.grid_conditionalise(base, linear=linear)["post"]
            one = torch.ones(1, dtype=torch.float64, device=base.device)
            zero = torch.zeros(1, dtype=torch.float64, device=base.device)
            # linear sums over the remaining marginal axis, one per value of K
            _, rows, cols = eng.grid_posterior2(base, zero, one, linear, want_post=False,
                                                marg_log=0)
            den = cols.reshape(1, -1) if ax == 1 else rows.reshape(-1, 1)
            out = eng.pd_binary('div', base, not linear, den, False, not linear)
            if ax == 0:
                out = out.t().contiguous()                # K's axis goes last (layout only)
            return self._new(name, vals, dims, out)
        prob = np.asarray(self.prob, dtype=float)
        if ax == 0:
            prob = prob.T
        if normalise and iscomplex(self._pscale):
            prob = prob - prob.max()
        prob = rescale(prob, self._pscale, 1.)
        if normalise:
            prob = div_prob(prob, np.sum(prob))
        prob = div_prob(prob, np.sum(prob, axis=0, keepdims=True))
        return self._new(name, vals, dims, rescale(prob, 1., self._pscale))

    def prod(self, keys):
        """iid product over ``keys``: sum (log pscale) / product (linear) along their
        axis; the values become the set {n} (pd.py:332-370)."""
        keys = self._split_keys(keys)
        marg = collections.OrderedDict(self._marg)
        vals, dims, axes, shift = collections.OrderedDict(), collections.OrderedDict(), [], 0
        for key, single in zip(self.keys(), self._aresingleton):
            if key in keys:
                assert not single, "Cannot apply product along scalar for key {}".format(key)
                if self._dims[key] not in axes:
                    axes.append(self._dims[key])
                    shift += 1
                marg[key] = key + "={}"
                vals[key] = {int(np.size(self[key]))}
            else:
                if not single:
                    dims[key] = self._dims[key] - shift
                vals[key] = self[key]
        prob = np.sum(self.prob, axis=tuple(axes)) if iscomplex(self._pscale) \
            else np.prod(self.prob, axis=tuple(axes))
        return self._new(margcond_str(marg, self._cond), vals, dims, prob)

    def _log_flag(self):
        if self._pscale == 0j:
            return True
        if self._pscale == 1.:
            return False
        raise NotImplementedError("device post-processing handles pscale 'log' and 1 only")

    def expectation(self, keys=None, exponent=None):
        """E[key] = sum(prob*val) / max(tiny, sum(prob)) over all array axes
        (pd.py:373-405)."""
        keys = list(self._marg.keys()) if keys is None else \
            ([keys] if isinstance(keys, str) else list(keys))
        for key in keys:
            assert key in self._marg, \
                "Key {} not marginal in distribution {}".format(key, self._name)
        akeys = [k for k, single in zip(self.keys(), self._aresingleton)
                 if k in keys and not single]
        sums = {}
        if self._prob_dev is not None and akeys:
            # K6: one pass over prob for the total and every numerator
            if self.ndim > 2:
                raise NotImplementedError("device expectation handles 1-D and 2-D PDs")
            if {self._dims[k] for k in akeys} != set(range(self.ndim)):
                raise NotImplementedError("device expectation sums over every array axis: "
                                          "request keys on all of them")
            import torch
            last = self.ndim - 1                       # 1-D: everything is a 'column' value
            rk = [k for k in akeys if self._dims[k] != last]
            ck = [k for k in akeys if self._dims[k] == last]
            if len(rk) > 4 or len(ck) > 4:
                raise NotImplementedError("at most 4 array keys per axis")
            rv = torch.stack([self._dev_val(k, exponent) for k in rk]) if rk else None
            cv = torch.stack([self._dev_val(k, exponent) for k in ck]) if ck else None
            res = self._engine().expectation_sums(self._prob_dev, self._log_flag(), rv, cv)
            res = res.cpu().numpy()
            total = res[0]
            for j, k in enumerate(rk + ck):
                sums[k] = res[1 + j]
        elif akeys:
            prob = rescale(self.prob, self._pscale, 1.)
            total = np.sum(prob)
            for key in akeys:
                val = self[key] if not exponent else self[key] ** exponent
                shape = [1] * self.ndim
                shape[self._dims[key]] = -1
                sums[key] = np.sum(prob * np.asarray(val, dtype=float).reshape(shape))
        out = collections.OrderedDict()
        for key, single in zip(self.keys(), self._aresingleton):
            if key in keys:
                if single:
                    out[key] = self[key] if not exponent or isinstance(self[key], set) \
                        else self[key] ** exponent
                else:
                    out[key] = div_prob(sums[key], total)
            elif key in self._cond:
                out[key] = self[key]
        return out

    def _ismonotonic(self, key):
        if key in self._monotonic:
            return self._monotonic[key]
        v = np.ravel(self[key])
        ge = v[1:] >= v[:-1]
        self._monotonic[key] = bool(v.size < 2 or np.all(ge) or not np.any(ge))
        return self._monotonic[key]

    def _cum_brackets(self, quants):
        """For each quantile: (ravelled index i of the bracketing cell, linear probs of
        cells i, i+1, cumulative probs of cells i, i+1) -- pd.py:426-430."""
        n = self.size
        if self._prob_dev is not None:
            eng = self._engine()
            flat = self._prob_dev.reshape(-1)
            cum, _ = eng.cumprob(flat, self._log_flag())
            idx = eng.digitize(cum, quants).cpu().numpy()
            out = []
            for i in idx:
                i = int(i)
                j = min(i + 2, n)
                rav = rescale(flat[i:j].cpu().numpy(), self._pscale, 1.)
                out.append((i, rav, cum[i:j].cpu().numpy()))
            return out
        rav = rescale(np.ravel(self.prob), self._pscale, 1.)
        cum = np.cumsum(rav)
        cum = div_prob(cum, cum[-1])
        idx = np.maximum(0, np.digitize(np.array(quants), cum) - 1).tolist()
        return [(int(i), rav[int(i):int(i) + 2], cum[int(i):int(i) + 2]) for i in idx]

    def quantile(self, q=0.5):
        """Quantiles from the cumulative probability of the ravelled distribution;
        values of the last axis are interpolated inside the bracketing cell, other
        axes take the cell's value, non-monotonic values are returned as the set
        {size} (pd.py:408-461)."""
        quants = [q] if isscalar(q) else list(q)
        if self.issingleton:
            res = [collections.OrderedDict(self)] * len(quants)
            return res[0] if isscalar(q) else res
        unsorted = {k for k, single in zip(self.keys(), self._aresingleton)
                    if not single and not self._ismonotonic(k)}
        res = []
        for qq, (rav_idx, ravp, cump) in zip(quants, self._cum_brackets(quants)):
            unr_idx = np.unravel_index(rav_idx, self._shape)
            item = collections.OrderedDict()
            for key, single in zip(self.keys(), self._aresingleton):
                if single:
                    item[key] = self[key]
                    continue
                if key in unsorted:
                    item[key] = {int(np.size(self[key]))}
                    continue
                dim = self._dims[key]
                val = np.ravel(self[key])
                i = int(min(unr_idx[dim], len(val) - 1))
                if dim < self.ndim - 1 or i == len(val) - 1:
                    item[key] = val[i]
                elif abs(ravp[1] - ravp[0]) < min(qq, 1. - qq):
                    item[key] = np.interp(qq, cump, val[i:i + 2])
                else:
                    item[key] = np.sum(ravp * val[i:i + 2]) / np.sum(ravp)
            res.append(item)
        return res[0] if isscalar(q) else res

    def sorted(self, key):
        """Distribution re-ordered by ascending ``key`` (pd.py:464-493)."""
        dim = self._dims[key]
        if dim is None:
            return self._new(self._name, collections.OrderedDict(self), self._dims,
                             self._prob_dev if self._prob_dev is not None else self.prob)
        if self._prob_dev is not None:
            # K6: radix argsort of the key, gathers of prob and of the values on that axis
            if self.ndim > 2:
                raise NotImplementedError("device sorted() handles 1-D and 2-D PDs")
            eng = self._engine()
            order, ks = eng.argsort(self._dev_val(key), want_keys=True)
            prob = eng.gather(self._prob_dev, order) if self.ndim == 1 else \
                eng.take_axis(self._prob_dev, order, dim)
            vals, vdev = collections.OrderedDict(), {}
            for k, v in self.items():
                if self._dims[k] != dim:
                    vals[k] = v
                    if k in self._vals_dev:
                        vdev[k] = self._vals_dev[k]
                    continue
                vdev[k] = ks if k == key else eng.gather(self._dev_val(k), order)
                vals[k] = vdev[k].cpu().numpy()
            out = self._new(self._name, vals, self._dims, prob)
            out._vals_dev = vdev
            out._monotonic = {k: m for k, m in self._monotonic.items() if self._dims[k] != dim}
            out._monotonic[key] = True
            return out
        order = np.argsort(np.ravel(self[key]))
        vals = collections.OrderedDict()
        for k, v in self.items():
            vals[k] = np.ravel(v)[order] if self._dims[k] == dim else v
        prob = np.take(self.prob, order, axis=dim)
        return self._new(self._name, vals, self._dims, prob)

    # ---- joint-product algebra -----------------------------------------------------------
    def __mul__(self, other):
        """Product rule: p(A | ..) * p(B | A, ..) -> p(A, B | ..) (pd.py:564-565)."""
        return product(self, other)

    def __truediv__(self, other):
        """If self is p(A, B | C) and other is p(A | C), returns p(B | C, A): the safe
        division ``num / max(tiny, den)`` in linear space (pd.py:572-615,
        pscales.py:219-236).  For log-pscale grids of large |log p| the reference's linear
        detour underflows -- use conditionalise() there, as its examples do."""
        assert set(self._cond.keys()) == set(other.cond.keys()), "Conditionals must match"
        divs = other.issingleton
        if divs:
            scalars = {k for k, single in zip(self.keys(), self._aresingleton)
                       if k in self._marg and single}
            assert scalars == set(other.marg.keys()), \
                "For divisor singletons, scalar marginals must match"
        keys = list(other.marg.keys())
        marg = collections.OrderedDict(self._marg)
        cond = collections.OrderedDict(self._cond)
        vals = collections.OrderedDict((k, self[k]) for k in self._cond)
        re_shape = [1] * self.ndim
        for key, single in zip(self.keys(), self._aresingleton):
            if key in keys:
                cond[key] = marg.pop(key)
                if not single and not divs:
                    re_shape[self._dims[key]] = int(np.size(other[key]))
            elif key not in vals:
                vals[key] = self[key]
        for key in self.keys():
            if key in keys:
                vals[key] = self[key]
        name = margcond_str(marg, cond)
        dims = collections.OrderedDict((k, self._dims[k]) for k in vals)
        a_log, b_log = _log_flag_of(self._pscale), _log_flag_of(other.pscale)
        if self._prob_dev is not None or other.prob_device is not None:
            if self.ndim > 2:
                raise NotImplementedError("device division handles 1-D and 2-D PDs")
            eng = (self if self._prob_dev is not None else other)._engine()
            a = self._prob_dev if self._prob_dev is not None else eng.to_device(self.prob)
            b = other.prob_device if other.prob_device is not None else \
                eng.to_device(np.atleast_1d(np.asarray(other.prob, dtype=float)))
            a2 = a.reshape(1, -1) if self.ndim < 2 else a
            shape_b = [1, 1] if divs else ([1] + re_shape if self.ndim < 2 else re_shape)
            out = eng.pd_binary('div', a2, a_log, b.reshape(shape_b), b_log, a_log)
            return self._new(name, vals, dims, out.reshape(self._shape))
        divp = other.prob if divs else np.reshape(other.prob, re_shape)
        prob = div_prob(self.prob, divp, self._pscale, other.pscale)
        return self._new(name, vals, dims, prob)

    def serialise(self):
        """{short name: {key: value, ..., 'attrs': dims, 'prob': prob, 'pscale':
        pscale}} (distribution.py:286-290, pd.py:698-703); a device-backed ``prob`` is copied
        to the host."""
        name = self.short_name
        d = {}
        for key, val in self.items():
            dim = self._dims.get(key)
            if dim is not None and self.ndim > 1 and np.ndim(val) == 1:
                # the reference keeps grid values in their broadcast shape ([M, 1], [1, S])
                shape = [1] * self.ndim
                shape[dim] = -1
                val = np.reshape(val, shape)
            d[key] = val
        d['attrs'] = self.dims
        d['prob'] = self.prob
        d['pscale'] = self.pscale
        return {name: d}

    def __repr__(self):
        return "PD({!r}, shape={}, pscale={})".format(self._name, self._shape, self._pscale)


def _log_flag_of(pscale):
    if pscale == 0j:
        return True
    if pscale == 1.:
        return False
    raise NotImplementedError("the joint-product algebra handles pscale 'log' and 1 only")


def product(*args):
    """Product rule over PDs with distinct marginal variables (pd_utils.py:85-328):
    conditionals that another factor carries as marginals become marginals of the
    product, the remaining conditionals must agree, array values get consecutive axes
    in name order (keys that share an axis in a factor keep sharing it), iid-reduced sets
    ``{n}`` add up, and the probabilities are combined by the product rule of
    pscales.py:160-216 -- on the device as soon as one factor is device-backed.
    Products of up to two array axes are in the device catalogue."""
    assert args, "product() needs at least one distribution"
    if len(args) == 1:
        return args[0]
    all_marg = [k for a in args for k in a.marg.keys()]
    assert len(all_marg) == len(set(all_marg)), \
        "Non-unique marginal variables for currently not supported: {}".format(all_marg)
    logs = [_log_flag_of(a.pscale) for a in args]
    out_log = any(logs)
    marg_names = [name for a in args for name in a.marg.values()]
    marg_keys = set(all_marg)
    cond_items = [(k, name) for a in args for k, name in a.cond.items()]
    prod_cond = collections.OrderedDict((k, n) for k, n in cond_items if k not in marg_keys)
    for a in args:
        rest = {k for k in a.cond.keys() if k not in marg_keys}
        if rest:
            assert rest == set(prod_cond.keys()), \
                "Incompatible product conditional {} for conditional set {}".format(
                    set(prod_cond.keys()), rest)
    prod_keys = all_marg + list(prod_cond.keys())
    # values: the first factor that has the key provides it; {n} sets add up
    vals = collections.OrderedDict()
    for key in prod_keys:
        found = [a[key] for a in args if key in a]
        assert found, "Values for key {} not found".format(key)
        if isunitsetint(found[0]):
            assert all(isunitsetint(v) for v in found), "Mismatch in variables"
            vals[key] = {sum(list(v)[0] for v in found)}
        else:
            vals[key] = found[0]
            for v in found[1:]:
                if not np.allclose(np.ravel(v), np.ravel(found[0])):
                    raise ValueError("Mismatch in values for condition {}".format(key))
    # axes: consecutive in key order; keys sharing an axis inside a factor share it here
    dims, ndim, groups = collections.OrderedDict(), 0, {}
    for key in prod_keys:
        if isscalar(vals[key]) or isunitset(vals[key]):
            dims[key] = None
            continue
        tag = None
        for ai, a in enumerate(args):
            if key in a and a.dims[key] is not None:
                tag = (ai, a.dims[key])
                break
        if tag in groups:
            dims[key] = groups[tag]
        else:
            dims[key] = groups[tag] = ndim
            ndim += 1
    # product labels ("mu=[]", "x={40}", "mu=50.0") are refreshed by the constructor
    name = ','.join(marg_names)
    if prod_cond:
        name += '|' + ','.join(prod_cond.values())
    pscale = 0j if out_log else 1.
    if ndim == 0:
        prob, _ = prod_rule(*[a.prob for a in args], pscales=[a.pscale for a in args])
        return PD(name, vals, dims=dims, prob=float(prob), pscale=pscale)
    if ndim > 2:
        raise NotImplementedError("products of more than two array axes are outside the "
                                  "device catalogue")
    shape = [0] * ndim
    for key, d in dims.items():
        if d is not None:
            shape[d] = int(np.size(vals[key]))

    def aligned(a):
        """(array-like prob of factor a, its shape broadcast into the product axes)"""
        olddims = sorted({d for d in a.dims.values() if d is not None})
        newdims = []
        for od in olddims:
            key = next(k for k, d in a.dims.items() if d == od)
            newdims.append(dims[key])
        tgt = [1] * ndim
        for nd in newdims:
            tgt[nd] = shape[nd]
        return olddims, newdims, tgt

    device = any(a.prob_device is not None for a in args)
    if not device:
        probs = []
        for a in args:
            _, newdims, tgt = aligned(a)
            p = a.prob
            if not isscalar(p):
                p = np.asarray(p, dtype=float)
                if len(newdims) == 2 and newdims[0] > newdims[1]:
                    p = p.T
                p = p.reshape(tgt)
            probs.append(p)
        prob, _ = prod_rule(*probs, pscales=[a.pscale for a in args])
        return PD(name, vals, dims=dims, prob=np.broadcast_to(prob, shape).copy(), pscale=pscale)
    eng = next(a for a in args if a.prob_device is not None)._engine()
    acc, acc_log = None, None
    for a, lg in zip(args, logs):
        _, newdims, tgt = aligned(a)
        t = a.prob_device if a.prob_device is not None else \
            eng.to_device(np.atleast_1d(np.asarray(a.prob, dtype=float)))
        if len(newdims) == 2 and newdims[0] > newdims[1]:
            t = t.t().contiguous()
        t = t.reshape(tgt if ndim == 2 else [1] + tgt)
        if acc is None:
            acc, acc_log = t, lg
            continue
        step_log = acc_log or lg
        acc = eng.pd_binary('mul', acc, acc_log, t, lg, step_log)
        acc_log = step_log
    if acc_log != out_log:                       # single log factor among linear ones, last
        acc = eng.log_prob_(acc.clone())
    return PD(name, vals, dims=dims, prob=acc.reshape(shape), pscale=pscale)
