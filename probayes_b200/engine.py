"""Device engine: thin Python layer between the host mirror (SP/SD/PD objects) and
the C ABI of libpbx.  PyTorch is used only for device memory, streams and
``torch.distributed``; every computation on the path is a libpbx kernel.

All device arrays are fp64 and chain-minor: state ``[D, C]``, samples
``[R, D, C]``, per-step scalars ``[T, C]``.
"""
import ctypes as C
import math
import numpy as np

from . import _lib
from ._lib import (PbxError, MhMvnParams, MhNormregParams, GibbsMvnParams, DevInfo,
                   RejectionParams,
                   ACCEPT_REFERENCE, ACCEPT_LOG, PROP_NORMAL, PROP_UNIFORM, PROP_SPHERICAL,
                   PBX_MAX_DIMS)

LOG_2PI = math.log(2.0 * math.pi)

_ACCEPT = {"reference": ACCEPT_REFERENCE, "log": ACCEPT_LOG}
_PROP = {"normal": PROP_NORMAL, "uniform": PROP_UNIFORM, "spherical": PROP_SPHERICAL}


def _torch():
    import torch
    return torch


def mvn_value_order(d):
    """Order in which the reference hands the variables of a scipy multivariate
    target to scipy (probayes/prob.py:349-358): reversed, and rotated for d > 2."""
    if d == 1:
        return [0]
    order = list(range(d))[::-1]
    if d > 2:
        order = order[1:] + [order[0]]
    return order


def mvn_setup(mean, cov, reorder=True):
    """Host-side constants of the mvn target in natural variable order:
    whitening matrix (scipy _PSD: U = u * sqrt(1/s) from eigh) with the value
    permutation folded in, permuted mean, and norm_c = d log 2pi + log_pdet."""
    mean = np.atleast_1d(np.asarray(mean, dtype=np.float64))
    cov = np.atleast_2d(np.asarray(cov, dtype=np.float64))
    d = mean.shape[0]
    if cov.shape != (d, d):
        raise ValueError("Means and covariance matrix incommensurate")
    s, u = np.linalg.eigh(cov)
    if np.min(s) <= 0:
        raise ValueError("covariance matrix must be positive definite")
    U = u * np.sqrt(1.0 / s)
    norm_c = d * LOG_2PI + float(np.sum(np.log(s)))
    order = mvn_value_order(d) if reorder else list(range(d))
    # scipy sees point y with y[j] = x[order[j]]; dev = y - mean; maha = |dev @ U|^2.
    # In natural order: dev_nat[i] = x[i] - mean_nat[i] with mean_nat[order[j]] = mean[j],
    # W[order[j], :] = U[j, :].
    W = np.empty_like(U)
    mean_nat = np.empty_like(mean)
    for j, i in enumerate(order):
        W[i, :] = U[j, :]
        mean_nat[i] = mean[j]
    return mean_nat, W, norm_c


class Engine:
    """One libpbx context on one GPU (one per process, as torch.distributed
    launches them).  Not thread-safe, like the reference's global RNG state."""

    def __init__(self, device=0, stream=None):
        self.lib = _lib.load()
        torch = _torch()
        if not torch.cuda.is_available():
            raise PbxError("probayes_b200 needs a CUDA device (no CPU fallback)")
        self.device_index = int(device)
        self.device = torch.device("cuda", self.device_index)
        torch.cuda.set_device(self.device)
        self.stream = stream if stream is not None else torch.cuda.current_stream(self.device)
        h = C.c_void_p()
        # run on torch's current stream (0 = the default stream), never on a private one
        _lib.check(self.lib.pbx_ctx_create(self.device_index,
                                           C.c_void_p(self.stream.cuda_stream), 0, C.byref(h)),
                   "pbx_ctx_create")
        self.ctx = h
        info = DevInfo()
        _lib.check(self.lib.pbx_device_info(self.device_index, C.byref(info)), "pbx_device_info")
        self.info = info
        # The context runs on torch's current stream, so torch's stream-ordered
        # caching allocator keeps every tensor handed to a kernel valid until
        # that kernel has run; no extra keep-alive list is needed.

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.pbx_ctx_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ utils
    def sync(self):
        _lib.check(self.lib.pbx_ctx_sync(self.ctx), "pbx_ctx_sync")

    @property
    def launches(self):
        return int(self.lib.pbx_ctx_launch_count(self.ctx))

    def last_kernel_ms(self):
        ms = C.c_float()
        _lib.check(self.lib.pbx_ctx_last_kernel_ms(self.ctx, C.byref(ms)), "last_kernel_ms")
        return float(ms.value)

    def fp64_peak_tflops(self):
        v = C.c_double()
        _lib.check(self.lib.pbx_fp64_peak(self.ctx, C.byref(v)), "pbx_fp64_peak")
        return float(v.value)

    def fp64_dep_latency(self):
        """(DFMA, DADD) dependent-issue latency in SM cycles."""
        a, b = C.c_double(), C.c_double()
        _lib.check(self.lib.pbx_fp64_dep_latency(self.ctx, C.byref(a), C.byref(b)),
                   "pbx_fp64_dep_latency")
        return float(a.value), float(b.value)

    def empty(self, *shape, dtype=None):
        torch = _torch()
        return torch.empty(*shape, dtype=dtype or torch.float64, device=self.device)

    def zeros(self, *shape, dtype=None):
        torch = _torch()
        return torch.zeros(*shape, dtype=dtype or torch.float64, device=self.device)

    def to_device(self, a):
        """numpy / tensor -> contiguous fp64 device tensor."""
        torch = _torch()
        if isinstance(a, torch.Tensor):
            return a.to(self.device, torch.float64).contiguous()
        a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
        return torch.from_numpy(a).to(self.device)

    @staticmethod
    def _ptr(t):
        return C.c_void_p(0 if t is None else t.data_ptr())

    def _dev(self, t, shape, what, dtype=None):
        """Checks a tensor whose pointer crosses the C ABI: on this engine's device,
        contiguous, ``dtype`` (fp64 by default) and exactly ``shape``.  The kernels read
        raw pointers as contiguous arrays; anything else would be silent garbage or an
        out-of-bounds write, so it raises."""
        torch = _torch()
        if t is None:
            return None
        dtype = dtype or torch.float64
        if not isinstance(t, torch.Tensor):
            raise TypeError("%s must be a torch tensor on %s" % (what, self.device))
        if not t.is_cuda or t.device.index != self.device_index:
            raise ValueError("%s must live on %s (got %s)" % (what, self.device, t.device))
        if t.dtype != dtype:
            raise TypeError("%s must be %s (got %s)" % (what, dtype, t.dtype))
        if not t.is_contiguous():
            raise ValueError("%s must be contiguous (got strides %s)" % (what, t.stride()))
        if shape is not None and tuple(t.shape) != tuple(shape):
            raise ValueError("%s must have shape %s (got %s)" % (what, tuple(shape),
                                                                 tuple(t.shape)))
        return t

    # ------------------------------------------------------------ K1: mh mvn
    def _mvn_params(self, D, C_, T, thin, step0, chain0, seed, log_pscale, accept,
                    prop, prop_scale, prop_chol, mean, cov, reorder, variant=0,
                    prop_radius=0.0, bound=None):
        if not 1 <= D <= PBX_MAX_DIMS:
            raise NotImplementedError(
                "mh_mvn supports 1..%d dimensions (got %d)" % (PBX_MAX_DIMS, D))
        if int(thin) < 1:
            raise ValueError("thin must be >= 1")
        if accept not in _ACCEPT or prop not in _PROP:
            raise ValueError("unknown accept/prop mode: %r / %r" % (accept, prop))
        p = MhMvnParams()
        p.kernel_variant = int(variant)
        p.prop_radius = float(prop_radius)
        p.n_chains, p.n_dims, p.n_steps, p.thin = C_, D, T, thin
        p.step0, p.chain0, p.seed = step0, chain0, seed & 0xFFFFFFFFFFFFFFFF
        p.log_pscale = 1 if log_pscale else 0
        p.accept_mode = _ACCEPT[accept]
        p.prop_kind = _PROP[prop]
        mean_nat, W, norm_c = mvn_setup(mean, cov, reorder)
        for j in range(D):
            p.mean[j] = mean_nat[j]
        for i, v in enumerate(W.ravel()):
            p.whiten[i] = v
        p.norm_c = norm_c
        scale = np.broadcast_to(np.asarray(prop_scale, dtype=np.float64), (D,))
        for j in range(D):
            p.prop_scale[j] = scale[j]
        if prop_chol is not None:
            L = np.asarray(prop_chol, dtype=np.float64)
            if L.shape != (D, D):
                raise ValueError("prop_chol must be [D, D]")
            p.has_prop_mat = 1
            for i, v in enumerate(L.ravel()):
                p.prop_mat[i] = v
        if bound is not None:                  # (lims [D, 2], open_end [D, 2])
            lims = np.asarray(bound[0], dtype=np.float64).reshape(D, 2)
            ex = np.asarray(bound[1]).reshape(D, 2)
            p.prop_bound = 1
            for j in range(D):
                p.lims[j][0], p.lims[j][1] = lims[j]
                p.open_end[j][0], p.open_end[j][1] = int(ex[j][0]), int(ex[j][1])
        return p

    def _walk_outputs(self, p, out, state, state_lp, accept_count, stats, T, thin, record,
                      per_step, inj_delta, inj_thresh):
        """Fills ``out`` with the output tensors of a walk of ``T`` steps and sets the
        matching pointer fields of the ABI params ``p`` (K1 and K2 share the field names).
        ``out`` may already hold "x" / "prob" buffers to reuse; ``stats`` is a zero-filled
        [2, D, C] tensor (stat_sum, stat_sumsq) or None."""
        torch = _torch()
        D, C_ = state.shape
        R = T // thin
        if record:
            if "x" not in out:
                out["x"] = self.empty(R, D, C_)
            if "prob" not in out:
                out["prob"] = self.empty(R, C_)
            self._dev(out["x"], (R, D, C_), "out['x']")
            self._dev(out["prob"], (R, C_), "out['prob']")
        if per_step:
            out["accept"] = self.empty(T, C_, dtype=torch.uint8)
            out["score"] = self.empty(T, C_)
            out["xprop"] = self.empty(T, D, C_)
            out["pprop"] = self.empty(T, C_)
        out["accept_count"] = accept_count
        if stats is not None:
            out["stat_sum"], out["stat_sumsq"] = stats[0], stats[1]
        out["state_lp"] = state_lp
        if inj_delta is not None:
            if tuple(inj_delta.shape) != (T, D, C_) or tuple(inj_thresh.shape) != (T, C_):
                raise ValueError("injected streams must be delta[T, D, C], thresh[T, C]")
        p.state, p.state_lp = state.data_ptr(), state_lp.data_ptr()
        p.inj_delta = 0 if inj_delta is None else inj_delta.data_ptr()
        p.inj_thresh = 0 if inj_thresh is None else inj_thresh.data_ptr()
        p.out_x = out["x"].data_ptr() if record else 0
        p.out_prob = out["prob"].data_ptr() if record else 0
        p.out_accept = out["accept"].data_ptr() if per_step else 0
        p.out_score = out["score"].data_ptr() if per_step else 0
        p.out_xprop = out["xprop"].data_ptr() if per_step else 0
        p.out_pprop = out["pprop"].data_ptr() if per_step else 0
        p.accept_count = accept_count.data_ptr()
        p.stat_sum = stats[0].data_ptr() if stats is not None else 0
        p.stat_sumsq = stats[1].data_ptr() if stats is not None else 0

    def mh_mvn(self, state, mean, cov, steps, thin=1, seed=0, step0=0, chain0=0,
               log_pscale=False, accept="reference", prop="normal", prop_scale=1.0,
               prop_chol=None, reorder=True, inj_delta=None, inj_thresh=None,
               state_lp=None, record=True, per_step=False, stats=True, variant=0,
               out=None, prop_radius=0.0, events=None, bound=None):
        """Runs ``steps`` MH steps for all chains of ``state`` ([D, C] device fp64,
        updated in place).  Returns a dict of device tensors:
        x [R, D, C], prob [R, C] (record), accept [T, C] uint8 + score [T, C]
        (per_step), accept_count [C] int64, stat_sum/stat_sumsq [D, C] (stats),
        state_lp [C].  ``bound`` = (lims [D, 2], open_end [D, 2]) applies
        set_delta(..., bound=True): closed limits clip the proposal, open ones bounce it
        back (one-thread-per-chain kernel).  ``out`` may carry preallocated "x"/"prob" buffers to
        reuse; ``variant`` 0 picks the kernel (native RNG + log rule + D <= 4: the
        warp-specialised kernel that decides on the whitened state), 1 forces the
        one-thread-per-chain kernel, 2 the warp-specialised kernel with the reference's
        arithmetic in the decision, 4 the whitened-decision kernel."""
        torch = _torch()
        D, C_ = state.shape
        T = int(steps)
        self._dev(state, (D, C_), "state")
        self._dev(state_lp, (C_,), "state_lp")
        self._dev(inj_delta, (T, D, C_), "inj_delta")
        self._dev(inj_thresh, (T, C_), "inj_thresh")
        p = self._mvn_params(D, C_, T, thin, step0, chain0, seed, log_pscale, accept,
                             prop, prop_scale, prop_chol, mean, cov, reorder, variant,
                             prop_radius, bound)
        out = dict(out) if out else {}
        if state_lp is None and step0 != 0:
            raise ValueError("state_lp is required when resuming (step0 > 0)")
        # one zero-fill for every accumulator of the walk: [state_lp | accept_count |
        # stat_sum | stat_sumsq]
        zbuf = self.zeros(C_ * (2 + (2 * D if stats else 0)))
        if state_lp is None:
            state_lp = zbuf[:C_]
        self._walk_outputs(p, out, state, state_lp, zbuf[C_:2 * C_].view(torch.int64),
                           zbuf[2 * C_:].view(2, D, C_) if stats else None, T, thin, record,
                           per_step, inj_delta, inj_thresh)
        if events is not None:                 # torch events bracketing the kernel launch only
            events[0].record(self.stream)
        _lib.check(self.lib.pbx_mh_mvn_run(self.ctx, C.byref(p)), "pbx_mh_mvn_run")
        if events is not None:
            events[1].record(self.stream)
        return out

    def mh_mvn_walk_host(self, state, mean, cov, steps, thin=1, seed=0, step0=0, chain0=0,
                         log_pscale=False, accept="reference", prop="normal",
                         prop_scale=1.0, prop_chol=None, reorder=True, state_lp=None,
                         chunk_steps=1000, out_x=None, out_prob=None, prop_radius=0.0,
                         bound=None):
        """Whole walk through the host-buffer entry point: ``state`` is a HOST
        ndarray [D, C] (updated in place); samples are streamed back into pinned
        host buffers while the next chunk runs.  Returns dict of ndarrays."""
        torch = _torch()
        state = np.ascontiguousarray(state, dtype=np.float64)
        D, C_ = state.shape
        T = int(steps)
        R = T // thin
        p = self._mvn_params(D, C_, T, thin, step0, chain0, seed, log_pscale, accept,
                             prop, prop_scale, prop_chol, mean, cov, reorder, 0, prop_radius,
                             bound)
        if out_x is None:
            out_x = torch.empty((R, D, C_), dtype=torch.float64, pin_memory=True)
        if out_prob is None:
            out_prob = torch.empty((R, C_), dtype=torch.float64, pin_memory=True)
        for t, shp, what in ((out_x, (R, D, C_), "out_x"), (out_prob, (R, C_), "out_prob")):
            if t.is_cuda or t.dtype != torch.float64 or not t.is_contiguous() \
                    or tuple(t.shape) != shp:
                raise ValueError("%s must be a contiguous host fp64 tensor of shape %s"
                                 % (what, shp))
        lp = np.zeros(C_) if state_lp is None else np.ascontiguousarray(state_lp, np.float64)
        if lp.shape != (C_,):
            raise ValueError("state_lp must have shape (%d,)" % C_)
        acc = np.zeros(C_, dtype=np.int64)
        ssum = np.zeros((D, C_))
        ssq = np.zeros((D, C_))
        p.state, p.state_lp = state.ctypes.data, lp.ctypes.data
        p.out_x, p.out_prob = out_x.data_ptr(), out_prob.data_ptr()
        p.accept_count, p.stat_sum, p.stat_sumsq = acc.ctypes.data, ssum.ctypes.data, \
            ssq.ctypes.data
        _lib.check(self.lib.pbx_mh_mvn_walk_host(self.ctx, C.byref(p), int(chunk_steps)),
                   "pbx_mh_mvn_walk_host")
        return dict(x=out_x.numpy(), prob=out_prob.numpy(), state=state, state_lp=lp,
                    accept_count=acc, stat_sum=ssum, stat_sumsq=ssq)

    # ------------------------------------------------- K2: streaming normal MH
    def _normreg_params(self, C_, P, x_obs, y_obs, lims, open_end, log_ufun, prop_scale,
                        accept="log", accept_coef=1.0, prop="uniform", variant=0,
                        prop_radius=0.0, prop_bound=False, prop_chol=None, lik=None):
        if P not in (2, 3):
            raise NotImplementedError("normal-likelihood MH supports (mu, sigma) or "
                                      "(b0, b1, sigma) parameters, got %d" % P)
        if accept not in _ACCEPT or prop not in _PROP:
            raise ValueError("unknown accept/prop mode: %r / %r" % (accept, prop))
        # a sampled nu is the third parameter of (mu, sigma, nu); otherwise three are a slope's
        sampled_nu = lik is not None and lik.get("df_param") is not None
        has_slope = P == 3 and not sampled_nu
        if sampled_nu and P != 3:
            raise ValueError("the sampled-nu Student-t needs parameters (mu, sigma, nu)")
        if has_slope and x_obs is None:
            raise ValueError("x_obs is required for the regression likelihood")
        p = MhNormregParams()
        p.n_chains, p.n_params = C_, P
        p.has_slope = 1 if has_slope else 0
        p.accept_mode, p.accept_coef = _ACCEPT[accept], float(accept_coef)
        p.prop_kind, p.variant = _PROP[prop], int(variant)
        p.prop_radius = float(prop_radius)
        p.prop_bound = 1 if prop_bound else 0
        p.n_obs = int(y_obs.numel())
        if has_slope and int(x_obs.numel()) != p.n_obs:
            raise ValueError("x_obs and y_obs differ in length")
        p.x_obs = x_obs.data_ptr() if has_slope else 0
        p.y_obs = y_obs.data_ptr()
        lims = np.asarray(lims, dtype=np.float64).reshape(P, 2)
        open_end = np.asarray(open_end).reshape(P, 2)
        log_ufun = np.asarray(log_ufun).reshape(P)
        scale = np.broadcast_to(np.asarray(prop_scale, dtype=np.float64), (P,))
        for j in range(P):
            p.lims[j][0], p.lims[j][1] = lims[j]
            p.open_end[j][0], p.open_end[j][1] = int(open_end[j][0]), int(open_end[j][1])
            p.log_ufun[j] = int(log_ufun[j])
            p.prop_scale[j] = scale[j]
        if prop_chol is not None:
            L = np.asarray(prop_chol, dtype=np.float64)
            if L.shape != (P, P):
                raise ValueError("prop_chol must be [P, P]")
            p.has_prop_mat = 1
            for i, v in enumerate(L.ravel()):
                p.prop_mat[i] = v
        if sampled_nu:
            p.lik_kind = _lib.LIK_STUDENT_T_NU          # nu and logc(nu) per chain, on the device
        elif lik is not None:
            p.lik_kind = _lib.LIK_STUDENT_T
            p.lik_df, p.lik_logc = float(lik["df"]), float(lik["logc"])
        return p

    def mh_normreg(self, state, y_obs, x_obs, steps, lims, open_end, log_ufun, prop_scale,
                   thin=1, seed=0, step0=0, chain0=0, accept="log", accept_coef=1.0,
                   prop="uniform", variant=0, inj_delta=None, inj_thresh=None, state_lp=None,
                   record=True, per_step=False, stats=True, prop_radius=0.0,
                   prop_bound=False, prop_chol=None, lik=None):
        """MH on the iid-normal posterior; ``state`` [P, C] device fp64 (in place),
        ``y_obs``/``x_obs`` device fp64 [N].  Same outputs as :meth:`mh_mvn`; the
        recorded ``prob`` is the log-joint (log pscale).  ``prop_chol`` [P, P]: the
        lower-triangular factor every delta is multiplied by before the ufun move
        (set_tran(covariance), rf.py:346-348), injected deltas included.  ``lik``: the
        likelihood family, None (normal) or a Student-t dict(df=nu, logc=...) as
        ``catalogue.likelihood`` returns, or dict(family='t', df_param=name) for a t whose nu
        is sampled as the third parameter of (mu, sigma, nu); the t has no sufficient
        statistics (no variant 3)."""
        torch = _torch()
        P, C_ = state.shape
        T = int(steps)
        if int(thin) < 1:
            raise ValueError("thin must be >= 1")
        self._dev(state, (P, C_), "state")
        self._dev(state_lp, (C_,), "state_lp")
        self._dev(y_obs, None, "y_obs")
        self._dev(x_obs, None, "x_obs")
        self._dev(inj_delta, (T, P, C_), "inj_delta")
        self._dev(inj_thresh, (T, C_), "inj_thresh")
        p = self._normreg_params(C_, P, x_obs, y_obs, lims, open_end, log_ufun, prop_scale,
                                 accept, accept_coef, prop, variant, prop_radius, prop_bound,
                                 prop_chol, lik)
        p.n_steps, p.thin, p.step0, p.chain0 = T, thin, step0, chain0
        p.seed = seed & 0xFFFFFFFFFFFFFFFF
        if state_lp is None:
            if step0 != 0:
                raise ValueError("state_lp is required when resuming (step0 > 0)")
            state_lp = self.zeros(C_)
        out = {}
        self._walk_outputs(p, out, state, state_lp, self.zeros(C_, dtype=torch.int64),
                           self.zeros(2, P, C_) if stats else None, T, thin, record, per_step,
                           inj_delta, inj_thresh)
        _lib.check(self.lib.pbx_mh_normreg_run(self.ctx, C.byref(p)), "pbx_mh_normreg_run")
        return out

    def normreg_logjoint(self, theta, y_obs, x_obs, lims, open_end, log_ufun, variant=0,
                         lik=None):
        """log-joint (likelihood + box priors) of theta [P, C] -> [C] device; ``lik`` as
        :meth:`mh_normreg`'s."""
        P, C_ = theta.shape
        self._dev(theta, (P, C_), "theta")
        self._dev(y_obs, None, "y_obs")
        self._dev(x_obs, None, "x_obs")
        p = self._normreg_params(C_, P, x_obs, y_obs, lims, open_end, log_ufun, 0.0,
                                 variant=variant, lik=lik)
        out = self.empty(C_)
        _lib.check(self.lib.pbx_normreg_logjoint(self.ctx, C.byref(p), self._ptr(theta),
                                                 self._ptr(out)), "pbx_normreg_logjoint")
        return out

    # ------------------------------------------------------ K3/K4: grid (DGEI)
    def grid_norm_logjoint(self, x_obs, mu, sigma, logprior_mu, logprior_sigma, out=None,
                           suffstat=False, lik=None):
        """log-joint [M, S] = priors + sum_i norm.logpdf(x_i; mu_m, sigma_s); all
        arguments device fp64 vectors.  ``suffstat=True`` (opt-in) evaluates it from
        centred sufficient statistics of the observations: O(M S) instead of O(N M S).
        ``lik``: as :meth:`mh_normreg`'s; a Student-t sums t.logpdf and has no suffstat."""
        M, S = int(mu.numel()), int(sigma.numel())
        extra = ()
        if lik is not None and lik.get("df_param") is not None:
            raise NotImplementedError("the (mu, sigma) grid needs a fixed nu: a grid over nu "
                                      "would be a three-axis grid")
        if lik is not None:
            if suffstat:
                raise ValueError("suffstat=True needs the normal likelihood: the Student-t "
                                 "likelihood has no sufficient statistics")
            fn, what = self.lib.pbx_grid_t_logjoint, "pbx_grid_t_logjoint"
            extra = (float(lik["df"]), float(lik["logc"]))
        elif suffstat:
            fn, what = self.lib.pbx_grid_norm_logjoint_ss, "pbx_grid_norm_logjoint_ss"
        else:
            fn, what = self.lib.pbx_grid_norm_logjoint, "pbx_grid_norm_logjoint"
        if out is None:
            out = self.empty(M, S)
        row_cap = 65535
        for m0 in range(0, M, row_cap):                     # slab very tall grids
            m1 = min(M, m0 + row_cap)
            _lib.check(fn(
                self.ctx, self._ptr(x_obs), int(x_obs.numel()), self._ptr(mu[m0:m1]), m1 - m0,
                self._ptr(sigma), S, self._ptr(logprior_mu[m0:m1]), self._ptr(logprior_sigma),
                self._ptr(out[m0:m1]), *extra), what)
        return out

    def log_prob_(self, v):
        """In-place clamped log (probayes/pscales.py:44-53)."""
        _lib.check(self.lib.pbx_log_prob_inplace(self.ctx, self._ptr(v), int(v.numel())),
                   "pbx_log_prob_inplace")
        return v

    def exp_logp_(self, v):
        """In-place clamped exp (probayes/pscales.py:56-65)."""
        _lib.check(self.lib.pbx_exp_logp_inplace(self.ctx, self._ptr(v), int(v.numel())),
                   "pbx_exp_logp_inplace")
        return v

    def grid_max_sumexp(self, v, linear=False):
        """[2] device tensor (max, sum exp_logp(v - max)) of all entries of ``v`` from ONE
        read (online rescaling); linear-pscale input: (0, sum v)."""
        out = self.empty(2)
        _lib.check(self.lib.pbx_grid_max_sumexp(self.ctx, self._ptr(v), int(v.numel()),
                                                1 if linear else 0, self._ptr(out)),
                   "pbx_grid_max_sumexp")
        return out

    def grid_rescale_sumexp_(self, lmax, gmax, gsum):
        """gsum = sum exp(v - lmax) -> sum exp(v - gmax) in place (1-element device tensors;
        a zero sum stays zero): a slab's sum against the maximum over all slabs."""
        _lib.check(self.lib.pbx_grid_rescale_sumexp(self.ctx, self._ptr(lmax), self._ptr(gmax),
                                                    self._ptr(gsum)), "pbx_grid_rescale_sumexp")
        return gsum

    def grid_posterior2(self, prob, gmax, gsum, linear=False, want_post=True, inplace=False,
                        marg_log=3):
        """(post [M, S] or None, marg_mu [M], marg_sigma [S]); ``marg_log`` bit 0 / 1: pass
        marg_mu / marg_sigma through the clamped log (log-pscale results)."""
        M, S = prob.shape
        post = (prob if inplace else self.empty(M, S)) if want_post else None
        mm, ms = self.empty(M), self.empty(S)
        _lib.check(self.lib.pbx_grid_posterior2(
            self.ctx, self._ptr(prob), M, S, self._ptr(gmax), self._ptr(gsum),
            1 if linear else 0, self._ptr(post), self._ptr(mm), self._ptr(ms), int(marg_log)),
            "pbx_grid_posterior2")
        return post, mm, ms

    def grid_conditionalise(self, lj, want_post=True, inplace=False, group=None, linear=False):
        """PD.conditionalise + both PD.marginal calls on a joint slab [M_local, S] in two
        passes over the grid: (max, sum-exp) with online rescaling, then posterior + both
        marginals.  ``linear``: the slab holds linear-pscale probabilities (results linear
        too).  With ``group`` (a torch.distributed group over mu-row slabs) the normaliser
        and the sigma marginal are all-reduced; the mu marginal stays a local slab.
        Returns dict(post, marg_mu, marg_sigma, gmax, gsum) in the input's pscale."""
        ms = self.grid_max_sumexp(lj, linear)
        gmax, gsum = ms[0:1], ms[1:2]
        if group is not None:
            from .dist import allreduce_max_sumexp
            allreduce_max_sumexp(gmax, gsum, self.grid_rescale_sumexp_, linear, group)
        log_bits = 0 if linear else (1 if group is not None else 3)
        post, mm, msig = self.grid_posterior2(lj, gmax, gsum, linear, want_post, inplace, log_bits)
        if group is not None:
            import torch.distributed as dist
            dist.all_reduce(msig, op=dist.ReduceOp.SUM, group=group)
            if not linear:
                self.log_prob_(msig)
        return dict(post=post, marg_mu=mm, marg_sigma=msig, gmax=gmax, gsum=gsum)

    # ------------------------------------------------------------ K5: Gibbs
    def mvn_logpdf(self, x, mean, cov, log_pscale=True, reorder=True):
        """Batched mvn density of x [d, n] (device) -> [n]; d = 64 runs the
        whitening product on the FP64 tensor cores."""
        d, n = x.shape
        mean_nat, W, norm_c = mvn_setup(mean, cov, reorder)
        md, Wd = self.to_device(mean_nat), self.to_device(W)
        out = self.empty(n)
        _lib.check(self.lib.pbx_mvn_logpdf(self.ctx, self._ptr(x), d, n, self._ptr(md),
                                           self._ptr(Wd), norm_c, 1 if log_pscale else 0,
                                           self._ptr(out)), "pbx_mvn_logpdf")
        return out

    def ndtri(self, u):
        """ndtri(u) of a device array as the Gibbs kernel evaluates it (pbx_ndtri.cuh)."""
        u = u.contiguous()
        self._dev(u, tuple(u.shape), "u")
        out = self.empty(*u.shape)
        _lib.check(self.lib.pbx_ndtri(self.ctx, self._ptr(u), u.numel(), self._ptr(out)),
                   "pbx_ndtri")
        return out

    def gibbs_mvn(self, state, cond_cov, steps, thin=1, seed=0, step0=0, chain0=0,
                  log_pscale=False, reorder=True, inj_runif=None, record=True, want_prob=True,
                  stats=False):
        """``steps`` single-coordinate Gibbs updates (coordinate = step mod d) of
        all chains of ``state`` [d, C] (device, in place) for the mvn described by
        ``cond_cov`` (a :class:`probayes_b200.cond_cov.CondCov`).  Returns dict
        with x [R, d, C] and prob [R, C] (the mvn target evaluated on every kept
        state, as the reference's SP.next does)."""
        d, C_ = state.shape
        self._dev(state, (d, C_), "state")
        self._dev(inj_runif, (int(steps), C_), "inj_runif")
        if d != cond_cov.n:
            raise ValueError("state has %d dims, CondCov has %d" % (d, cond_cov.n))
        if d > 128:
            raise NotImplementedError("gibbs_mvn supports up to 128 dimensions")
        if int(thin) < 1:
            raise ValueError("thin must be >= 1")
        T = int(steps)
        R = T // thin
        p = GibbsMvnParams()
        p.n_chains, p.n_dims, p.n_steps, p.thin = C_, d, T, thin
        p.step0, p.chain0, p.seed = step0, chain0, seed & 0xFFFFFFFFFFFFFFFF
        p.log_pscale = 1 if log_pscale else 0
        consts = getattr(cond_cov, "_dev", None)
        if consts is None or consts[0] is not self or consts[1] != reorder:
            mean_nat, W, norm_c = mvn_setup(cond_cov.mean, cond_cov.cov, reorder)
            consts = (self, reorder, dict(
                mean=self.to_device(cond_cov.mean), coef=self.to_device(cond_cov.coef_matrix()),
                stdv=self.to_device(cond_cov.stdv), lo=self.to_device(cond_cov.cdfs[:, 0]),
                hi=self.to_device(cond_cov.cdfs[:, 1]), W=self.to_device(W),
                dmean=self.to_device(mean_nat), norm_c=norm_c))
            cond_cov._dev = consts
        k = consts[2]
        p.mean, p.coef, p.stdv = k["mean"].data_ptr(), k["coef"].data_ptr(), k["stdv"].data_ptr()
        p.cdf_lo, p.cdf_hi = k["lo"].data_ptr(), k["hi"].data_ptr()
        p.whiten, p.dens_mean, p.norm_c = k["W"].data_ptr(), k["dmean"].data_ptr(), k["norm_c"]
        out = {}
        if record:
            out["x"] = self.empty(R, d, C_)
            if want_prob:
                out["prob"] = self.empty(R, C_)
        if stats:
            out["stat_sum"] = self.zeros(d, C_)
            out["stat_sumsq"] = self.zeros(d, C_)
        p.state = state.data_ptr()
        p.inj_runif = 0 if inj_runif is None else inj_runif.data_ptr()
        p.out_x = out["x"].data_ptr() if record else 0
        p.out_prob = out["prob"].data_ptr() if (record and want_prob) else 0
        p.want_prob = 1 if (record and want_prob) else 0
        p.stat_sum = out["stat_sum"].data_ptr() if stats else 0
        p.stat_sumsq = out["stat_sumsq"].data_ptr() if stats else 0
        _lib.check(self.lib.pbx_gibbs_mvn_run(self.ctx, C.byref(p)), "pbx_gibbs_mvn_run")
        return out

    # ------------------------------------------------- K6: PD post-processing
    def _workspace(self, nbytes):
        torch = _torch()
        return torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)

    def argsort(self, keys, want_keys=False):
        """Ascending stable argsort of a 1-D fp64 device tensor -> int32 order
        (and the sorted keys): np.argsort of PD.sorted (pd.py:473-474)."""
        torch = _torch()
        n = int(keys.numel())
        nb = C.c_size_t()
        _lib.check(self.lib.pbx_argsort_workspace_bytes(n, C.byref(nb)), "pbx_argsort_workspace_bytes")
        ws = self._workspace(max(nb.value, 1))
        order = torch.empty(n, dtype=torch.int32, device=self.device)
        ks = self.empty(n) if want_keys else None
        _lib.check(self.lib.pbx_argsort_f64(self.ctx, self._ptr(keys), n, order.data_ptr(),
                                            0 if ks is None else ks.data_ptr(),
                                            ws.data_ptr(), nb.value), "pbx_argsort_f64")
        return (order, ks) if want_keys else order

    def gather(self, src, order):
        out = self.empty(int(order.numel()))
        _lib.check(self.lib.pbx_gather_f64(self.ctx, self._ptr(src), order.data_ptr(),
                                           int(order.numel()), out.data_ptr()), "pbx_gather_f64")
        return out

    def take_axis(self, src, order, axis):
        rows, cols = src.shape
        out = self.empty(rows, cols)
        _lib.check(self.lib.pbx_take_axis_f64(self.ctx, self._ptr(src), rows, cols, int(axis),
                                              order.data_ptr(), out.data_ptr()),
                   "pbx_take_axis_f64")
        return out

    def _scan_ws(self, n):
        nb = C.c_size_t()
        _lib.check(self.lib.pbx_scan_workspace_bytes(int(n), C.byref(nb)), "pbx_scan_workspace_bytes")
        return self._workspace(nb.value), nb.value

    def cumprob(self, prob, log_pscale, out=None):
        """Normalised cumulative probability of the ravelled ``prob`` and the
        un-normalised total (1-element device tensor): pd.py:426-429."""
        n = int(prob.numel())
        ws, nb = self._scan_ws(n)
        cum = self.empty(n) if out is None else out
        total = self.empty(1)
        _lib.check(self.lib.pbx_cumprob_f64(self.ctx, self._ptr(prob), n, int(bool(log_pscale)),
                                            cum.data_ptr(), total.data_ptr(), ws.data_ptr(), nb),
                   "pbx_cumprob_f64")
        return cum, total

    def digitize(self, cum, q):
        """np.maximum(0, np.digitize(q, cum) - 1) -> int64 device tensor (pd.py:430)."""
        torch = _torch()
        q = np.ascontiguousarray(np.atleast_1d(np.asarray(q, dtype=np.float64)))
        out = torch.empty(q.size, dtype=torch.int64, device=self.device)
        _lib.check(self.lib.pbx_digitize_f64(self.ctx, self._ptr(cum), int(cum.numel()),
                                             q.ctypes.data_as(C.POINTER(C.c_double)), q.size,
                                             out.data_ptr()), "pbx_digitize_f64")
        return out

    def expectation_sums(self, prob, log_pscale, row_vals=None, col_vals=None):
        """[1 + KR + KC] device sums: total, sum p*row_vals[k][i], sum p*col_vals[k][j]
        over a [rows, cols] (or 1-D = [1, n]) prob tensor (pd.py:387-402)."""
        if prob.dim() == 1:
            rows, cols = 1, int(prob.numel())
        else:
            rows, cols = prob.shape
        kr = 0 if row_vals is None else int(row_vals.shape[0])
        kc = 0 if col_vals is None else int(col_vals.shape[0])
        ws, nb = self._scan_ws(rows * cols)
        out = self.empty(1 + kr + kc)
        _lib.check(self.lib.pbx_expectation_f64(
            self.ctx, self._ptr(prob), rows, cols, int(bool(log_pscale)),
            0 if kr == 0 else self._ptr(row_vals), kr,
            0 if kc == 0 else self._ptr(col_vals), kc, out.data_ptr(), ws.data_ptr(), nb),
            "pbx_expectation_f64")
        return out

    def pd_binary(self, op, a, a_log, b, b_log, out_log):
        """Product rule (op='mul') / safe division (op='div') of two probability
        tensors of shapes [rows or 1, cols or 1] -> [rows, cols] device tensor."""
        a2 = a.reshape(1, -1) if a.dim() < 2 else a
        b2 = b.reshape(1, -1) if b.dim() < 2 else b
        a2, b2 = a2.contiguous(), b2.contiguous()       # kept alive until after the launch
        rows, cols = max(a2.shape[0], b2.shape[0]), max(a2.shape[1], b2.shape[1])
        out = self.empty(rows, cols)
        _lib.check(self.lib.pbx_pd_binary_f64(
            self.ctx, 0 if op == 'mul' else 1, self._ptr(a2), a2.shape[0], a2.shape[1],
            int(bool(a_log)), self._ptr(b2), b2.shape[0], b2.shape[1], int(bool(b_log)),
            rows, cols, int(bool(out_log)), out.data_ptr()), "pbx_pd_binary_f64")
        return out

    def box_sample(self, lims, log_ufun, n_samples, seed=0, sample0=0, inj_unif=None):
        """theta [P, T] device: uniform draws in ufun space mapped back
        (variable.py:558-583); inj_unif [T, P] device or None = Philox."""
        lims = np.ascontiguousarray(np.asarray(lims, dtype=np.float64))
        P = lims.shape[0]
        lg = np.ascontiguousarray(np.asarray(log_ufun, dtype=np.int32))
        out = self.empty(P, int(n_samples))
        _lib.check(self.lib.pbx_box_sample(
            self.ctx, P, int(n_samples), lims.ctypes.data_as(C.POINTER(C.c_double)),
            lg.ctypes.data_as(C.POINTER(C.c_int32)), int(seed), int(sample0),
            0 if inj_unif is None else self._ptr(inj_unif), out.data_ptr()), "pbx_box_sample")
        return out

    def rejection_sample(self, lims, log_ufun, n_samples, target, prop, score_mode, thresh,
                         seed=0, sample0=0, inj_unif=None):
        """Ordinary Monte Carlo with rejection sampling (sp.py:221-258 with a proposal
        density): returns dict(theta [P, T], p, q, s, t [T], u [T] uint8) device tensors.
        target = dict(kind='ball', radius, centre); prop = dict(kind='normal', loc, scale) |
        dict(kind='box'); score_mode 'p' | 'p/q'; thresh = (low, high); inj_unif [T, P + 1]."""
        torch = _torch()
        lims = np.asarray(lims, dtype=np.float64)
        P, T = lims.shape[0], int(n_samples)
        p = RejectionParams()
        p.n_params, p.n_samples, p.sample0 = P, T, int(sample0)
        p.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        if target['kind'] != 'ball':
            raise NotImplementedError("rejection target kind %r" % target['kind'])
        p.target_kind, p.target_radius = 0, float(target['radius'])
        p.prop_kind = {'normal': 0, 'box': 1}[prop['kind']]
        p.score_mode = {'p': 0, 'p/q': 1}[score_mode]
        p.thresh_lo, p.thresh_hi = float(thresh[0]), float(thresh[1])
        for j in range(P):
            p.lims[j][0], p.lims[j][1] = lims[j]
            p.log_ufun[j] = int(np.asarray(log_ufun)[j])
            p.target_centre[j] = float(np.asarray(target['centre'])[j])
            p.prop_loc[j] = float(prop['loc'][j]) if prop['kind'] == 'normal' else 0.0
            p.prop_scale[j] = float(prop['scale'][j]) if prop['kind'] == 'normal' else 1.0
        out = dict(theta=self.empty(P, T), p=self.empty(T), q=self.empty(T), s=self.empty(T),
                   t=self.empty(T), u=self.empty(T, dtype=torch.uint8))
        self._dev(inj_unif, (T, P + 1), "inj_unif")
        p.inj_unif = 0 if inj_unif is None else inj_unif.data_ptr()
        p.out_theta, p.out_p, p.out_q = out['theta'].data_ptr(), out['p'].data_ptr(), \
            out['q'].data_ptr()
        p.out_s, p.out_t, p.out_u = out['s'].data_ptr(), out['t'].data_ptr(), out['u'].data_ptr()
        _lib.check(self.lib.pbx_rejection_sample(self.ctx, C.byref(p)), "pbx_rejection_sample")
        return out

    # ------------------------------------------------------- chain summaries
    def chain_stats(self, stat_sum, stat_sumsq, n_steps):
        """[D, 4] device tensor (sum_c mean, sum_c mean^2, sum_c var, C)."""
        D, C_ = stat_sum.shape
        self._dev(stat_sum, (D, C_), "stat_sum")
        self._dev(stat_sumsq, (D, C_), "stat_sumsq")
        out = self.empty(D, 4)
        _lib.check(self.lib.pbx_reduce_chain_stats(self.ctx, self._ptr(stat_sum),
                                                   self._ptr(stat_sumsq), D, C_, int(n_steps),
                                                   self._ptr(out)), "pbx_reduce_chain_stats")
        return out


_engines = {}


def get_engine(device=None):
    """Process-wide engine for ``device`` (default: the current CUDA device)."""
    torch = _torch()
    if device is None:
        if not torch.cuda.is_available():
            raise PbxError("probayes_b200 needs a CUDA device (no CPU fallback)")
        device = torch.cuda.current_device()
    device = int(device)
    if device not in _engines:
        _engines[device] = Engine(device)
    return _engines[device]
