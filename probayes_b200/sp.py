"""SP -- stochastic process: the Metropolis-Hastings / Gibbs sampler front end.

Mirror of the reference interface (probayes/sp.py:57-100,131-198,221-295;
sp_utils.py:8-91): ``set_scores`` / ``set_thresh`` / ``set_update`` with the
``MCMC_SAMPLERS`` names, ``sampler(init, [obs], stop=, iid=, joint=)``,
``walk(sampler)``, ``process(samples)`` -> ``opqrstuv`` summary.  The step loop
itself (sp.py:221-258) never runs in Python: ``walk`` hands the whole walk to the
batched-chain kernels of libpbx.

New keyword arguments of ``sampler`` (everything else keeps its meaning):
  chains=C      run C independent chains (default: one, reference-shaped results)
  thin=k        record every k-th step
  seed=s        Philox seed of the native RNG
  chain0=g      global id of this process's first chain (the Philox stream is keyed on
                chain0 + c).  Default: 0, or rank * chains when a torch.distributed
                process group is initialised, so that the ranks of a sharded run draw
                DIFFERENT chains and their concatenation equals the single-process run
  accept=       'log' (default for native RNG) | 'reference' (the reference's
                linear-space ratio with its clamps; default for injected streams)
  inj_delta=, inj_thresh=   injected proposal / threshold streams ([T, D] or
                [T, C, D] and [T] or [T, C]) for bit-parity runs
  host_stream=True   stream samples straight into pinned host buffers (K1)
  host_buffers=dict  a dict the sampler fills with its pinned host buffers and reuses on
                later walks / other samplers of the same shape (the streamed K1 outputs
                with host_stream, the final device-to-host copy of samples and densities
                otherwise); the returned arrays are then views into them
  inj_unif=     injected prior draws [T, P] for ordinary Monte Carlo random sampling
  suffstat=True (opt-in, normal-likelihood targets) evaluate the likelihood from centred
                sufficient statistics of the observations: one reduction over the data,
                then O(1) per evaluation and the whole walk in one launch; same values as
                the term-by-term kernels to fp64 round-off

Ordinary Monte Carlo random sampling (sp.py:229-234, the no-proposal branch of
``SP.next``; examples/omc/omc_rs_sp_norm1d.py): with neither transition nor delta set,
``sampler({'mu': {0}, 'sigma': {0}, 'x': data}, iid=True, joint=True, stop=T)`` draws
every parameter afresh from its box (uniform in ufun space) at each step and evaluates
the joint; ``process(samples)`` is then ONE PD over the T samples (summate,
pd_utils.py:332-383), device-backed, whose ``rescaled / sorted / quantile /
expectation`` run as K6 kernels.
"""
import collections
import numpy as np

from .sd import SD
from .pd import PD
from .pscales import iscomplex
from .vtypes import isunitsetint
from . import catalogue

MCMC_SAMPLERS = ('metropolis', 'hastings', 'gibbs')


class AcceptRecord:
    """``summary.u`` of a batched run: behaves like the reference's list of
    True/None for the one thing examples do with it -- ``u.count(True)``."""

    def __init__(self, counts, steps):
        self.counts = np.asarray(counts)
        self.steps = int(steps)

    def count(self, value=True):
        total = int(self.counts.sum())
        if value is True:
            return total
        if value is None:
            return self.counts.size * self.steps - total
        return 0

    def __len__(self):
        return self.counts.size * self.steps

    def rate(self):
        return self.count(True) / float(len(self))


class Walk(list):
    """Result of ``SP.walk``: a list of per-step ``opqrstuv`` tuples for
    reference-shaped single-chain runs, plus the raw arrays (``.arrays``).  The per-step
    tuples (three scalar PDs each) are built on first use of the list -- iteration, indexing,
    ``len`` -- because ``process(walk)`` works from the arrays and never looks at them:
    building 12288 of them eagerly was 95 % of the wall clock of the reference's own
    single-chain example."""
    arrays = None
    sampler = None
    _builder = None

    def _fill(self):
        builder, self._builder = self._builder, None
        if builder is not None:
            list.extend(self, builder())


def _lazy(name):
    base = getattr(list, name)

    def method(self, *args, **kwds):
        self._fill()
        return base(self, *args, **kwds)
    method.__name__ = name
    return method


for _name in ('__iter__', '__len__', '__getitem__', '__contains__', '__reversed__', '__eq__',
              '__ne__', '__repr__', '__add__', '__mul__', 'count', 'index', 'copy', 'pop',
              'append', 'extend', 'insert', 'remove', 'reverse', 'sort', '__setitem__',
              '__delitem__', '__iadd__'):
    setattr(Walk, _name, _lazy(_name))
Walk.__hash__ = None


class Sampler:
    """Returned by ``SP.sampler``; iterating it (or ``SP.walk``) runs the walk."""

    def __init__(self, sp, init, obs, stop, opts):
        self.sp, self.init, self.obs, self.stop, self.opts = sp, init, obs, stop, opts
        self.counter = 0
        self.state = None           # device state between calls (resume)
        self.state_lp = None

    def __iter__(self):
        return iter(self.sp.walk(self))


class SP(SD):

    def __init__(self, *args):
        super().__init__(*args)
        self._scores = self._thresh = self._update = None
        self._samplers = []
        self.stuv = collections.namedtuple(self._id, ['s', 't', 'u', 'v'])
        self.opqrstuv = collections.namedtuple(self._id,
                                               ['o', 'p', 'q', 'r', 's', 't', 'u', 'v'])

    # ---- scores / thresh / update ------------------------------------------------------------
    @property
    def scores(self):
        return self._scores

    @property
    def thresh(self):
        return self._thresh

    @property
    def update(self):
        return self._update

    def _check_spec(self, spec, what, args=(), kwds=None):
        """MCMC sampler names pass through; Python callables are mapped onto the kernel
        modes the catalogue knows (rejection sampling: scores opqr.p.prob [/ opqr.q.prob],
        thresh np.random.uniform(low, high), update stu.s >= stu.t) or refused."""
        if spec is None:
            return None
        if isinstance(spec, str) and spec in MCMC_SAMPLERS:
            assert not args and not kwds, \
                "Neither args nor kwds permitted with spec '{}'".format(spec)
            return spec
        if callable(spec):
            fn = {'scores': catalogue.identify_scores, 'thresh': catalogue.identify_thresh,
                  'update': catalogue.identify_update}[what]
            return fn(spec, args, kwds)
        raise NotImplementedError(
            "{} must be one of {} or a catalogue-recognised function on the device path"
            .format(what, MCMC_SAMPLERS))

    def set_scores(self, scores=None, *args, **kwds):
        self._scores = self._check_spec(scores, 'scores', args, kwds)
        if self._scores in MCMC_SAMPLERS:       # the reference chains these (sp.py:61-66)
            self.set_thresh(scores)

    def set_thresh(self, thresh=None, *args, **kwds):
        self._thresh = self._check_spec(thresh, 'thresh', args, kwds)
        if self._thresh in MCMC_SAMPLERS:
            self.set_update(thresh)

    def set_update(self, update=None, *args, **kwds):
        self._update = self._check_spec(update, 'update', args, kwds)

    # ---- sampler bookkeeping --------------------------------------------------------------------
    def reset(self, sampler_id=None, reset_last=True):
        if sampler_id is None:
            self._samplers = []
            return
        s = self.get_sampler(sampler_id)
        s.counter = 0
        if reset_last:
            s.state = s.state_lp = None

    def get_sampler(self, sampler_id=None):
        if sampler_id is None:
            return self._samplers
        return self._samplers[sampler_id] if isinstance(sampler_id, int) else sampler_id

    def get_counter(self, sampler_id=None):
        if sampler_id is None:
            return {s: s.counter for s in self._samplers}
        return self.get_sampler(sampler_id).counter

    def sampler(self, *args, **kwds):
        """sampler(init_state, [observations], stop=T, iid=, joint=, **new_kwargs)."""
        kwds = dict(kwds)
        stop = kwds.pop('stop', None)
        if len(args) == 1 and type(args[0]) is int and stop is None:
            stop, args = args[0], ()
        if self._prop is not None:
            # proposal DENSITY set: every step draws afresh ({0}) -- rejection sampling
            assert not args or (isinstance(args[0], set) and list(args[0]) == [0]), \
                "a sampler with a proposal density draws {0} per step"
            opts = dict(rejection=True, omc=False, seed=kwds.pop('seed', None),
                        inj_unif=kwds.pop('inj_unif', None), sample0=kwds.pop('sample0', None))
            assert not kwds, "Unknown sampler keywords: {}".format(list(kwds))
            s = Sampler(self, None, None, stop, opts)
            self._samplers.append(s)
            return s
        if not args:
            raise NotImplementedError("random initial states ({0}) are not in the device "
                                      "catalogue: pass an initial-state dictionary")
        init = self.parse_values(args[0])
        obs = self.parse_values(args[1]) if len(args) > 1 else None
        omc = self._is_random_sampling(init)
        if omc:                     # one dict holds the {0} requests and the observations
            obs = collections.OrderedDict((k, v) for k, v in init.items()
                                          if k not in self._state_rf.keyset)
        opts = dict(iid=kwds.pop('iid', False), joint=kwds.pop('joint', False),
                    chains=kwds.pop('chains', None), thin=int(kwds.pop('thin', 1)),
                    seed=kwds.pop('seed', None), accept=kwds.pop('accept', None),
                    chain0=kwds.pop('chain0', None),
                    inj_delta=kwds.pop('inj_delta', None),
                    inj_thresh=kwds.pop('inj_thresh', None),
                    host_stream=kwds.pop('host_stream', False),
                    host_buffers=kwds.pop('host_buffers', None),
                    variant=kwds.pop('variant', 0),
                    inj_unif=kwds.pop('inj_unif', None), omc=omc)
        if kwds.pop('suffstat', False):
            opts['variant'] = 3
        assert not kwds, "Unknown sampler keywords: {}".format(list(kwds))
        s = Sampler(self, init, obs, stop, opts)
        self._samplers.append(s)
        return s

    def _is_random_sampling(self, init):
        """No proposal configured and every sampled variable requested as {0}
        (sp.py:227-234: such a sampler is a plain distribution call per step)."""
        rf = self._proposal_rf()
        if rf._delta is not None or rf._tran is not None or rf._tfun is not None:
            return False
        req = [init.get(k) for k in self._state_rf.keylist]
        if not all(isunitsetint(v) for v in req):
            return False
        if any(list(v)[0] != 0 for v in req):
            raise NotImplementedError("random sampling draws one value per step: use {0}")
        return True

    # ---- the walk ----------------------------------------------------------------------------------
    def walk(self, sampler, stop=None):
        """Runs the sampler for ``stop`` steps (default: its own ``stop``) on the
        device and returns a :class:`Walk`."""
        assert isinstance(sampler, Sampler), \
            'Sampler must be a sampler instance returned by SP.sampler()'
        T = stop if stop is not None else sampler.stop
        if T is None:
            raise ValueError("No stop specification set - a device walk needs a finite length")
        if sampler.stop is not None:
            T = min(T, sampler.stop - sampler.counter)
        if sampler.opts.get('rejection'):
            arrays = self._run_rejection(sampler, int(T))
            sampler.counter += int(T)
            if sampler.stop is not None and sampler.counter >= sampler.stop:
                sampler.counter = 0
            out = Walk()
            out.arrays, out.sampler = arrays, sampler
            if arrays['T'] <= 200000:
                out._builder = lambda: self._rejection_per_step(arrays)
            return out
        arrays = self._run_omc(sampler, int(T)) if sampler.opts['omc'] \
            else self._run(sampler, int(T))
        sampler.counter += int(T)
        if sampler.stop is not None and sampler.counter >= sampler.stop:
            sampler.counter = 0                  # auto-reset (sp_utils.py:15-16)
        out = Walk()
        out.arrays, out.sampler = arrays, sampler
        if arrays.get('omc'):
            if arrays['T'] <= 200000:
                out._builder = lambda: self._omc_per_step(arrays)
            return out
        if arrays['chains'] is None and arrays['R'] <= 200000:
            out._builder = lambda: self._per_step(arrays)
        return out

    # ---- ordinary Monte Carlo with rejection sampling -----------------------------------------
    def _run_rejection(self, sampler, T):
        """examples/omc/omc_rejection_sp_circle.py:26-39 as ONE kernel launch: T proposals
        from the variables' boxes, proposal density q, target p, score, threshold, update."""
        from .engine import get_engine
        from .dist import world
        eng = get_engine()
        opts = sampler.opts
        rvs = self._state_rf.varlist
        keys = self._state_rf.keylist
        for rv in rvs:
            assert rv.isfinite, "Cannot evaluate {{0}} values for bounds: {}".format(rv.ulims)
        if not (self._scores in ('p', 'p/q') and isinstance(self._thresh, tuple)
                and self._update == 's>=t'):
            raise NotImplementedError(
                "rejection sampling needs set_scores(opqr.p.prob [/ opqr.q.prob]), "
                "set_thresh(np.random.uniform, low=, high=) and set_update(stu.s >= stu.t)")
        target = catalogue.identify_rejection_target(self._prob, self._prob_args,
                                                     self._prob_kwds, rvs)
        prop = catalogue.identify_rejection_prop(self._prop, self._prop_args, self._prop_kwds,
                                                 rvs)
        lims = np.array([rv.vlims for rv in rvs])
        lg = np.array([rv.log_ufun for rv in rvs], dtype=int)
        inj = None
        if opts['inj_unif'] is not None:
            u = np.asarray(opts['inj_unif'], dtype=np.float64)[sampler.counter:sampler.counter + T]
            assert u.shape == (T, len(keys) + 1), "injected uniform stream must be [T, P + 1]"
            inj = eng.to_device(u)
        seed = opts['seed']
        if seed is None:
            seed = int(np.random.randint(0, 2 ** 31 - 1))
        sample0 = opts['sample0']
        if sample0 is None:                      # sharded run: disjoint global sample ids
            rank, ws = world()
            sample0 = rank * (sampler.stop or T)
        out = eng.rejection_sample(lims, lg, T, target, prop, self._scores, self._thresh[1:],
                                   seed=seed, sample0=int(sample0) + sampler.counter,
                                   inj_unif=inj)
        eng.sync()
        host = {k: v.detach().cpu().numpy() for k, v in out.items()}
        return dict(rejection=True, keys=keys, T=T, pscale=self._pscale, chains=None,
                    dev=out, **host)

    def _rejection_pd(self, arrays, sel, primed=False, prob_key='p'):
        """PD over the samples ``sel`` (an index -> scalar PD, a mask / slice -> arrays)."""
        keys = arrays['keys']
        names = [k + "'" for k in keys] if primed else list(keys)
        th, pr = arrays['theta'], arrays[prob_key]
        if np.ndim(sel) == 0 and not isinstance(sel, slice):
            vals = collections.OrderedDict((n, float(th[j, sel])) for j, n in enumerate(names))
            name = ','.join("{}={}".format(n, vals[n]) for n in names)
            return PD(name, vals, dims=collections.OrderedDict((n, None) for n in names),
                      prob=float(pr[sel]), pscale=arrays['pscale'])
        vals = collections.OrderedDict((n, th[j][sel]) for j, n in enumerate(names))
        return PD(','.join(names), vals, dims=collections.OrderedDict((n, 0) for n in names),
                  prob=pr[sel], pscale=arrays['pscale'])

    def _rejection_per_step(self, arrays):
        """Reference-shaped tuples (sp.py:244-258): p the target PD at the proposal, q the
        proposal-density PD (primed names, rf.py:584-602), s, t, u; v = p when kept."""
        out = []
        for i in range(arrays['T']):
            p = self._rejection_pd(arrays, i)
            q = self._rejection_pd(arrays, i, primed=True, prob_key='q')
            out.append(self.opqrstuv(None, p, q, None, float(arrays['s'][i]),
                                     float(arrays['t'][i]), bool(arrays['u'][i]),
                                     p if (arrays['u'][i] or i == 0) else None))
        return out

    def _rejection_summary(self, arrays):
        """process(samples) of a rejection run (sp.py:131-198): samples with u == False are
        dropped, the rest summated."""
        keep = arrays['u'].astype(bool)
        p = self._rejection_pd(arrays, keep)
        q = self._rejection_pd(arrays, keep, primed=True, prob_key='q')
        return self.opqrstuv(None, p, q, None, list(arrays['s'][keep]), list(arrays['t'][keep]),
                             [True] * int(keep.sum()), p)

    # ---- ordinary Monte Carlo random sampling ------------------------------------------------
    def _run_omc(self, sampler, T):
        from .engine import get_engine
        opts = sampler.opts
        eng = get_engine()
        spec = catalogue.identify_target(self, self._leafs, self._roots)
        if spec['kind'] != 'normreg':
            raise NotImplementedError("random sampling is in the device catalogue for the iid "
                                      "normal likelihood targets")
        if not (opts['iid'] and opts['joint']):
            raise NotImplementedError("random sampling needs iid=True, joint=True")
        keys = self._state_rf.keylist
        assert spec['params'] == keys, \
            "parameter field order {} must be {}".format(keys, spec['params'])
        rvs = [self._state_rf[k] for k in keys]
        for rv in rvs:
            assert rv.isfinite, "Cannot evaluate {{0}} values for bounds: {}".format(rv.ulims)
        lims = np.array([rv.vlims for rv in rvs])
        ex = np.array([rv.open_ends for rv in rvs], dtype=int)
        lg = np.array([rv.log_ufun for rv in rvs], dtype=int)
        if sampler.obs is None or spec['obs_y'] not in sampler.obs:
            raise ValueError("observations for '{}' are required".format(spec['obs_y']))
        if 'obs_dev' not in sampler.__dict__:
            y = eng.to_device(np.ravel(np.asarray(sampler.obs[spec['obs_y']], np.float64)))
            x = None
            if spec['has_slope']:
                x = eng.to_device(np.ravel(np.asarray(sampler.obs[spec['obs_x']], np.float64)))
            sampler.obs_dev = (y, x)
        y, x = sampler.obs_dev
        inj = None
        if opts['inj_unif'] is not None:
            u = np.asarray(opts['inj_unif'], dtype=np.float64)[sampler.counter:sampler.counter + T]
            assert u.shape == (T, len(keys)), "injected uniform stream shape mismatch"
            inj = eng.to_device(u)
        seed = opts['seed']
        if seed is None:
            seed = int(np.random.randint(0, 2 ** 31 - 1))
        theta = eng.box_sample(lims, lg, T, seed=seed, sample0=sampler.counter, inj_unif=inj)
        catalogue.refuse_suffstat(spec, opts['variant'])
        logp = eng.normreg_logjoint(theta, y, x, lims, ex, lg,
                                    variant=3 if opts['variant'] == 3 else 0,
                                    lik=spec.get('lik'))
        return dict(omc=True, keys=keys, T=T, spec=spec, theta=theta, logp=logp,
                    n_obs=int(y.numel()), pscale=self._pscale, chains=None)

    def _omc_names(self, arrays, n):
        spec = arrays['spec']
        return ["{}={{{}}}".format(ok, n) for ok in (spec['obs_x'], spec['obs_y']) if ok], \
            [ok for ok in (spec['obs_x'], spec['obs_y']) if ok]

    def _omc_per_step(self, arrays):
        """One scalar PD per step, named like the reference's per-step joint call
        ("mu=55.8,sigma=19.1,x={60}")."""
        th = arrays['theta'].detach().cpu().numpy()
        lp = arrays['logp'].detach().cpu().numpy()
        arrays['theta_host'], arrays['logp_host'] = th, lp
        labels, okeys = self._omc_names(arrays, arrays['n_obs'])
        out = []
        for t in range(arrays['T']):
            vals = collections.OrderedDict((k, th[j, t]) for j, k in enumerate(arrays['keys']))
            for ok in okeys:
                vals[ok] = {arrays['n_obs']}
            name = ','.join(["{}={}".format(k, vals[k]) for k in arrays['keys']] + labels)
            out.append(PD(name, vals, dims=collections.OrderedDict((k, None) for k in vals),
                          prob=float(lp[t]), pscale=arrays['pscale']))
            out[-1]._origin = (arrays, t)       # lets process([...]) find the device arrays
        return out

    def _omc_summary(self, arrays):
        """summate() of the per-step PDs (pd_utils.py:332-383): arrays on dim 0, the
        iid sets added up, prob device-backed."""
        th = arrays.get('theta_host')
        if th is None:
            th = arrays['theta'].detach().cpu().numpy()
        n = arrays['n_obs'] * arrays['T']
        labels, okeys = self._omc_names(arrays, n)
        vals = collections.OrderedDict((k, th[j]) for j, k in enumerate(arrays['keys']))
        dims = collections.OrderedDict((k, 0) for k in arrays['keys'])
        for ok in okeys:
            vals[ok] = {n}
            dims[ok] = None
        pd = PD(','.join(list(arrays['keys']) + labels), vals, dims=dims, prob=arrays['logp'],
                pscale=arrays['pscale'])
        pd.set_device_vals({k: arrays['theta'][j] for j, k in enumerate(arrays['keys'])})
        return pd

    def _run(self, sampler, T):
        from .engine import get_engine
        if self._scores is None:
            raise NotImplementedError("set_scores('metropolis' | 'hastings' | 'gibbs') first")
        opts = sampler.opts
        eng = get_engine()
        state_rf = self._state_rf
        keys = state_rf.keylist
        D = len(keys)
        Cn = opts['chains']
        C = 1 if Cn is None else int(Cn)
        spec = catalogue.identify_target(self, self._leafs, self._roots)
        injected = opts['inj_delta'] is not None
        seed = opts['seed']
        if seed is None:
            seed = int(np.random.randint(0, 2 ** 31 - 1))     # the reference draws from np.random
        thin = opts['thin']
        step0 = sampler.counter
        chain0 = opts['chain0']
        if chain0 is None:                       # sharded run: rank r owns chains [r*C, (r+1)*C)
            from .dist import default_chain0
            chain0 = default_chain0(C)
        chain0 = int(chain0)
        # ---- initial / resumed state [D, C] ------------------------------------------------
        if sampler.state is None or step0 == 0:
            init = np.empty((D, C))
            for j, k in enumerate(keys):
                init[j] = np.broadcast_to(np.asarray(sampler.init[k], dtype=np.float64), (C,))
            sampler.state, sampler.state_lp = eng.to_device(init), None
        state = sampler.state
        inj_d = inj_t = None
        if opts['inj_thresh'] is not None:       # thresholds (MH) / cdf uniforms (Gibbs)
            t = np.asarray(opts['inj_thresh'], dtype=np.float64)
            t = (t[:, None] if t.ndim == 1 else t)[step0:step0 + T]
            gibbs_k = (self._tran_obj.tsteps or D) if self._scores == 'gibbs' else 1
            assert t.shape == (T, C) or gibbs_k > 1, "injected threshold stream shape mismatch"
            inj_t = eng.to_device(t)
        if injected:
            assert inj_t is not None, "inj_delta needs inj_thresh"
            d = np.asarray(opts['inj_delta'], dtype=np.float64)
            d = (d[:, None, :] if d.ndim == 2 else d)[step0:step0 + T]
            assert d.shape == (T, C, D), "injected delta stream shape mismatch"
            inj_d = eng.to_device(np.ascontiguousarray(np.transpose(d, (0, 2, 1))))
        accept = opts['accept'] or ('reference' if injected else 'log')
        per_step = Cn is None and T <= 200000
        gibbs = self._scores == 'gibbs'
        res = dict(keys=keys, chains=Cn, T=T, thin=thin, R=T // thin, spec=spec,
                   inj_thresh=None if inj_t is None else np.asarray(opts['inj_thresh']),
                   gibbs=gibbs, pscale=self._pscale)
        if per_step and not gibbs:
            # the state this call starts from: the first predecessor of summary.q
            res['init'] = state.detach().cpu().numpy()[:, 0].copy()
        if gibbs:
            cc = self._cond_cov
            if spec['kind'] != 'mvn' or cc is None:
                raise NotImplementedError("Gibbs needs a scipy.stats.multivariate_normal "
                                          "transition (set_tran(mvn, mean, cov, tsteps=1))")
            # tsteps coordinates are updated per step, cursor wrapping at D (rf.py:446-452);
            # no tsteps = the whole sweep.  The kernel counts single-coordinate updates.
            k = self._tran_obj.tsteps or D
            if D % k != 0:
                raise NotImplementedError("tsteps must divide the number of variables "
                                          "({} does not divide {})".format(k, D))
            if inj_t is not None and k > 1:
                # k cdf uniforms per step, in update order
                t = np.asarray(opts['inj_thresh'], dtype=np.float64)
                t = (t[:, None] if t.ndim == 1 else t)[step0 * k:(step0 + T) * k]
                assert t.shape == (T * k, C), "injected uniform stream shape mismatch"
                inj_t = eng.to_device(t)
            out = eng.gibbs_mvn(state, cc, T * k, thin=thin * k, seed=seed, step0=step0 * k,
                                chain0=chain0, log_pscale=spec['log_pscale'],
                                inj_runif=inj_t)
            res.update(x=out['x'], prob=out['prob'], accept_count=None, accept=None, score=None)
            return self._finish(res, eng, opts.get('host_buffers'))
        prop = catalogue.identify_proposal(self._proposal_rf(), self._pscale, injected)
        coef = prop['coef'] if self._scores == 'hastings' else 1.0
        if spec['kind'] == 'mvn':
            assert spec['names'] == keys
            bound = None
            if prop['bound'] and any(np.isfinite(state_rf[k].vlims).any() for k in keys):
                # set_delta(..., bound=True) on bounded RVs (variable.py:700-739)
                bound = (np.array([state_rf[k].vlims for k in keys]),
                         np.array([state_rf[k].open_ends for k in keys], dtype=int))
            if opts['host_stream'] and not injected and not per_step:
                h = eng.mh_mvn_walk_host(state.cpu().numpy(), spec['mean'], spec['cov'], T,
                                         thin=thin, seed=seed, step0=step0,
                                         log_pscale=spec['log_pscale'], accept=accept,
                                         prop=prop['kind'], prop_scale=prop['scale'],
                                         prop_radius=prop['radius'], prop_chol=prop['chol'],
                                         state_lp=None if sampler.state_lp is None
                                         else sampler.state_lp.cpu().numpy(),
                                         chain0=chain0, bound=bound,
                                         **self._host_bufs(opts, T // thin, D, C))
                sampler.state = eng.to_device(h['state'])
                sampler.state_lp = eng.to_device(h['state_lp'])
                res.update(x=h['x'], prob=h['prob'], accept_count=h['accept_count'],
                           accept=None, score=None, stat_sum=h['stat_sum'],
                           stat_sumsq=h['stat_sumsq'])
                return self._finish(res, eng)
            out = eng.mh_mvn(state, spec['mean'], spec['cov'], T, thin=thin, seed=seed,
                             step0=step0, log_pscale=spec['log_pscale'], accept=accept,
                             prop=prop['kind'], prop_scale=prop['scale'],
                             prop_radius=prop['radius'], prop_chol=prop['chol'],
                             inj_delta=inj_d, inj_thresh=inj_t, state_lp=sampler.state_lp,
                             per_step=per_step, variant=opts['variant'], chain0=chain0,
                             bound=bound)
        else:
            if not opts['iid']:
                raise NotImplementedError("the normal-likelihood target needs iid=True")
            catalogue.refuse_suffstat(spec, opts['variant'])
            if sampler.obs is None or spec['obs_y'] not in sampler.obs:
                raise ValueError("observations for '{}' are required".format(spec['obs_y']))
            assert spec['params'] == keys, \
                "parameter field order {} must be {}".format(keys, spec['params'])
            if 'obs_dev' not in sampler.__dict__:
                y = eng.to_device(np.ravel(np.asarray(sampler.obs[spec['obs_y']], np.float64)))
                x = None
                if spec['has_slope']:
                    x = eng.to_device(np.ravel(np.asarray(sampler.obs[spec['obs_x']],
                                                          np.float64)))
                sampler.obs_dev = (y, x)
            y, x = sampler.obs_dev
            rvs = [state_rf[k] for k in keys]
            lims = np.array([rv.vlims for rv in rvs])
            ex = np.array([rv.open_ends for rv in rvs], dtype=int)
            lg = np.array([rv.log_ufun for rv in rvs], dtype=int)
            if not opts['joint']:
                raise NotImplementedError("likelihood-only sampling (joint=False) is not in the "
                                          "device catalogue: the box priors are part of K2")
            out = eng.mh_normreg(state, y, x, T, lims, ex, lg, prop['scale'], thin=thin,
                                 seed=seed, step0=step0, accept=accept, accept_coef=coef,
                                 prop=prop['kind'], prop_radius=prop['radius'],
                                 prop_bound=prop['bound'], prop_chol=prop['chol'],
                                 inj_delta=inj_d, inj_thresh=inj_t,
                                 state_lp=sampler.state_lp, per_step=per_step,
                                 variant=opts['variant'], chain0=chain0, lik=spec.get('lik'))
            res['n_obs'] = int(y.numel())
        sampler.state_lp = out['state_lp']
        res.update(x=out['x'], prob=out['prob'], accept_count=out['accept_count'],
                   accept=out.get('accept'), score=out.get('score'),
                   xprop=out.get('xprop'), pprop=out.get('pprop'),
                   stat_sum=out.get('stat_sum'), stat_sumsq=out.get('stat_sumsq'))
        return self._finish(res, eng, opts.get('host_buffers'))

    @staticmethod
    def _host_bufs(opts, R, D, C):
        """Pinned output buffers cached in the user-supplied ``host_buffers`` dict."""
        cache = opts.get('host_buffers')
        if cache is None:
            return {}
        import torch
        key = (R, D, C)
        if cache.get('key') != key:
            cache['key'] = key
            cache['x'] = torch.empty((R, D, C), dtype=torch.float64, pin_memory=True)
            cache['prob'] = torch.empty((R, C), dtype=torch.float64, pin_memory=True)
        return dict(out_x=cache['x'], out_prob=cache['prob'])

    @staticmethod
    def _finish(res, eng, cache=None):
        """Device results -> host arrays ([R, D, C] / [R, C]).  With the user-supplied
        ``host_buffers`` dict the two large arrays (samples, densities) go through pinned
        buffers kept in it (asynchronous copies at PCIe rate instead of a pageable staging
        copy into freshly faulted memory); the arrays returned then alias those buffers
        until the next walk that uses the same dict."""
        import torch
        pinned = {}

        def host(k, a):
            if a is None or isinstance(a, np.ndarray):
                return a
            if cache is not None and k in ('x', 'prob') and a.numel() > 0:
                key = ('finish', k, tuple(a.shape), str(a.dtype))
                buf = cache.get(key)
                if buf is None:
                    buf = cache[key] = torch.empty(tuple(a.shape), dtype=a.dtype, pin_memory=True)
                with torch.cuda.stream(eng.stream):
                    buf.copy_(a.detach(), non_blocking=True)
                pinned[k] = buf
                return buf
            return a.detach().cpu().numpy()
        eng.sync()
        for k in ('x', 'prob', 'accept_count', 'accept', 'score', 'stat_sum', 'stat_sumsq',
                  'xprop', 'pprop'):
            res[k] = host(k, res.get(k))
        if pinned:
            eng.sync()
            for k, buf in pinned.items():
                res[k] = buf.numpy()
        return res

    # ---- result marshalling --------------------------------------------------------------------------
    def _value_pd(self, arrays, sel=None, x=None, prob=None):
        """PD of the retained states (or, with ``x`` / ``prob``, of any [R, D, C] / [R, C]
        pair such as the proposals): arrays [R] per variable (single chain) or [C, R]
        (batched), named like the reference's summate() result."""
        keys = arrays['keys']
        x = arrays['x'] if x is None else x
        prob = arrays['prob'] if prob is None else prob
        single = arrays['chains'] is None
        vals = collections.OrderedDict()
        for j, k in enumerate(keys):
            v = x[:, j, 0] if single else x[:, j, :].T
            vals[k] = v if sel is None else v[sel]
        p = prob[:, 0] if single else prob.T
        if sel is not None:
            p = p[sel]
        names = list(keys)
        dims = collections.OrderedDict((k, 0) for k in keys)
        spec = arrays['spec']
        if spec['kind'] == 'normreg':
            n = arrays['n_obs'] * (1 if sel is not None and np.ndim(p) == 0 else x.shape[0])
            for ok in [k for k in (spec['obs_x'], spec['obs_y']) if k]:
                vals[ok] = {n}
                dims[ok] = None
                names.append("{}={{{}}}".format(ok, n))
        if sel is not None and np.ndim(p) == 0:
            names = ["{}={}".format(k, vals[k]) if k in keys else n_
                     for k, n_ in zip(list(vals.keys()), names)]
            dims = collections.OrderedDict((k, None) for k in vals)
            p = float(p)
        return PD(','.join(names), vals, dims=dims, prob=p, pscale=arrays['pscale'])

    @staticmethod
    def _has_proposals(arrays):
        return arrays.get('xprop') is not None and arrays['thin'] == 1

    def _q_pd(self, arrays, sel=None, reverse=False):
        """The proposal-density PD of the reference's ``opqr.q`` / ``summary.q`` (sd.py:253-288,
        sp.py:170-198) for a reference-shaped single-chain run: named ``x',y'|x,y``, the
        proposals under the primed keys, their predecessors (the state the call started from,
        then the retained states) under the plain keys, and the user's transition callable
        evaluated on them -- on the host, vectorised, after the walk: with a single callable
        the Hastings score does not use q (sp_utils.py:40-64), it is only recorded.  None for
        transitions that are not callables.  A ``(q, r)`` pair (constants in the device
        catalogue) also yields ``r`` (``reverse=True``): the same values under
        ``x,y|x',y'`` with ``r`` evaluated on them."""
        tran = self._proposal_rf()._tran
        if isinstance(tran, tuple) and len(tran) == 2:
            tran = tran[1] if reverse else tran[0]
        elif reverse:
            return None
        if not callable(tran) or arrays.get('xprop') is None or arrays.get('init') is None \
                or arrays['thin'] != 1:
            return None
        keys = arrays['keys']
        prop = np.asarray(arrays['xprop'])[:, :, 0]                     # [T, D]
        pred = np.concatenate([arrays['init'][None, :], np.asarray(arrays['x'])[:-1, :, 0]])
        ckey = '_r_prob' if reverse else '_q_prob'
        cache = arrays.get(ckey)
        if cache is None:
            kw = {}
            for j, k in enumerate(keys):
                kw[k] = pred[:, j]
                kw[k + "'"] = prop[:, j]
            try:
                cache = np.asarray(tran(**kw), dtype=float)
                if cache.ndim == 0:
                    cache = np.full(prop.shape[0], float(cache))
                assert cache.shape == (prop.shape[0],)
            except Exception:                       # a callable that only takes scalars
                cache = np.array([float(tran(**{n: float(v[i]) for n, v in kw.items()}))
                                  for i in range(prop.shape[0])])
            arrays[ckey] = cache
        vals = collections.OrderedDict()
        primed, plain = [k + "'" for k in keys], list(keys)
        marg, cond = (plain, primed) if reverse else (primed, plain)
        if sel is None:
            for k in marg + cond:
                j = keys.index(k.rstrip("'"))
                vals[k] = prop[:, j] if k.endswith("'") else pred[:, j]
            name = ','.join(marg) + '|' + ','.join(cond)
            dims = collections.OrderedDict((k, 0) for k in vals)
            return PD(name, vals, dims=dims, prob=cache, pscale=self._proposal_rf().pscale)
        for j, k in enumerate(keys):
            vals[k] = pred[sel, j]
        for j, k in enumerate(keys):
            vals[k + "'"] = prop[sel, j]
        name = ','.join("{}={}".format(k, vals[k]) for k in marg) + '|' + \
            ','.join("{}={}".format(k, vals[k]) for k in cond)
        return PD(name, vals, dims=collections.OrderedDict((k, None) for k in vals),
                  prob=float(cache[sel]), pscale=self._proposal_rf().pscale)

    @staticmethod
    def _stu_lists(arrays):
        """Per-step ``s / t / u`` of a single-chain run as three lists (sp.py:244-258):
        Gibbs keeps every step with nan scores; MH has them where the records align with the
        steps (thin == 1)."""
        R = arrays['R']
        acc, score, thr = arrays.get('accept'), arrays.get('score'), arrays.get('inj_thresh')
        if arrays['gibbs']:
            return [np.nan] * R, [np.nan] * R, [True] * R
        if arrays['thin'] == 1 and acc is not None:
            us = [True if a else None for a in np.asarray(acc)[:R, 0].tolist()]
            ss = [None] * R if score is None else \
                [None if v != v else v for v in np.asarray(score, dtype=float)[:R, 0].tolist()]
            ts = [None] * R if thr is None else [float(v) for v in np.ravel(thr)[:R].tolist()]
            return ss, ts, us
        return [None] * R, [None] * R, [None] * R

    def _per_step(self, arrays):
        """Reference-shaped per-step tuples for a single chain: ``v`` the retained state,
        and (thin == 1) ``p`` the proposal with its target density, ``o`` the predecessor
        (None on the first step of a fresh sampler), ``s / t / u`` (sp.py:244-258)."""
        out = []
        R = arrays['R']
        aligned = arrays['thin'] == 1
        props = self._has_proposals(arrays)
        ss, ts, us = self._stu_lists(arrays)
        prev = None
        for i in range(R):
            v = self._value_pd(arrays, sel=i)
            s, t, u, p = ss[i], ts[i], us[i], None
            q = r = None
            if props:
                p = self._value_pd(arrays, sel=i, x=arrays['xprop'], prob=arrays['pprop'])
                q = self._q_pd(arrays, sel=i)
                r = self._q_pd(arrays, sel=i, reverse=True)
            out.append(self.opqrstuv(prev if aligned else None, p, q, r, s, t, u, v))
            prev = v
        return out

    def __call__(self, *args, **kwds):
        """process(samples) -> opqrstuv summary with array-valued ``v``; other
        call signatures are the SD grid evaluation."""
        conditionalise = kwds.pop('conditionalise', None)
        samples = args[0] if args else None
        if isinstance(samples, Walk) or (isinstance(samples, (list, tuple, collections.deque))
                                         and len(samples)
                                         and isinstance(samples[0], self.opqrstuv)):
            return self._summary(samples, conditionalise)
        if isinstance(samples, (list, tuple, collections.deque)) and len(samples) \
                and isinstance(samples[0], PD):
            # [sample for sample in sampler] of a random-sampling run: all T per-step PDs
            # of one walk, in order -> the device-backed summary; anything else is outside
            # the catalogue (a host-side concatenation would be a CPU path)
            first, last = getattr(samples[0], '_origin', None), getattr(samples[-1], '_origin', None)
            if first is None or last is None or first[0] is not last[0] or first[1] != 0 \
                    or last[1] != first[0]['T'] - 1 or len(samples) != first[0]['T']:
                raise NotImplementedError("process(list of PDs) needs the complete, ordered "
                                          "output of one sampler (or pass SP.walk(sampler))")
            pd = self._omc_summary(first[0])
            return pd.conditionalise(self._leafs.keyset) if conditionalise else pd
        return super().__call__(*args, **kwds)

    def _summary(self, samples, conditionalise=None):
        arrays = samples.arrays if isinstance(samples, Walk) else None
        if arrays is not None and arrays.get('rejection'):
            return self._rejection_summary(arrays)
        if arrays is not None and arrays.get('omc'):
            pd = self._omc_summary(arrays)
            return pd.conditionalise(self._leafs.keyset) if conditionalise else pd
        if arrays is None:
            # a plain list of per-step tuples: concatenate their scalar PDs
            def concat(pds):
                pds = [d for d in pds if d is not None]
                if not pds:
                    return None
                keys = list(pds[0].keys())
                cond = list(pds[0].cond.keys())
                if cond:                         # a proposal density x',y'|x,y: primed keys first
                    keys = [k for k in keys if k not in cond] + [k for k in keys if k in cond]
                vals = collections.OrderedDict()
                for k in keys:
                    if isinstance(pds[0][k], set):
                        vals[k] = {sum(list(d[k])[0] for d in pds)}
                    else:
                        vals[k] = np.array([d[k] for d in pds])
                dims = collections.OrderedDict((k, None if isinstance(vals[k], set) else 0)
                                               for k in keys)
                names = [k if not isinstance(vals[k], set) else "{}={}".format(k, vals[k])
                         for k in keys]
                name = ','.join(names)
                if cond:
                    name = ','.join(n for n, k in zip(names, keys) if k not in cond) + '|' + \
                        ','.join(n for n, k in zip(names, keys) if k in cond)
                return PD(name, vals, dims=dims,
                          prob=np.array([d.prob for d in pds]), pscale=pds[0].pscale)
            kept = [s for s in samples if s.u is not False]
            v = concat([s.v for s in kept])
            if conditionalise:
                v = v.conditionalise([k for k in self._leafs.keylist if k in v.marg])
            u = [s.u for s in kept]
            s_ = [s.s for s in kept if s.s is not None]      # sp.py:181-190: dropped samples
            t_ = [s.t for s in kept if s.t is not None]      # contribute nothing
            return self.opqrstuv(concat([s.o for s in kept]), concat([s.p for s in kept]),
                                 concat([s.q for s in kept]), concat([s.r for s in kept]),
                                 s_ or None, t_ or None, u, v)
        v = self._value_pd(arrays)
        if conditionalise:                      # sp.py:194-196: condition on the leaf (data) keys
            v = v.conditionalise([k for k in self._leafs.keylist if k in v.marg])
        o = p = q = r = None
        if self._has_proposals(arrays) and not conditionalise:
            q = self._q_pd(arrays)
            r = self._q_pd(arrays, reverse=True)
            # summate() of the per-step p / o PDs (sp.py:170-198): every proposal, and the
            # predecessor of every step but the first
            p = self._value_pd(arrays, x=arrays['xprop'], prob=arrays['pprop'])
            if arrays['R'] > 1:
                o = self._value_pd(arrays, x=arrays['x'][:-1], prob=arrays['prob'][:-1])
        if arrays['chains'] is None and arrays['R'] <= 200000 and arrays['R'] > 0:
            # reference-shaped single chain: s / t / u straight from the arrays (the per-step
            # tuples of the Walk are not built for this)
            ss, ts, u = self._stu_lists(arrays)
            s_ = [x for x in ss if x is not None]
            t_ = [x for x in ts if x is not None]
            return self.opqrstuv(o, p, q, r, s_ or None, t_ or None, u, v)
        if arrays['gibbs']:
            C = 1 if arrays['chains'] is None else arrays['chains']
            u = AcceptRecord(np.full(C, arrays['T']), arrays['T'])
        else:
            u = AcceptRecord(arrays['accept_count'], arrays['T'])
        return self.opqrstuv(None, None, None, None, None, None, u, v)

    # ---- chain diagnostics (new) -------------------------------------------------------------------------
    @staticmethod
    def rhat(summary_v):
        """Gelman-Rubin R-hat per variable from a batched summary ``v`` ([C, R] arrays)."""
        out = collections.OrderedDict()
        for k, a in summary_v.items():
            if isinstance(a, set) or np.ndim(a) != 2:
                continue
            T = a.shape[1]
            W = a.var(axis=1, ddof=1).mean()
            B = T * a.mean(axis=1).var(ddof=1)
            out[k] = float(np.sqrt(((T - 1) / T * W + B / T) / W))
        return out
