"""K1 MH on a multivariate-normal target, one compiled kernel at a time, against the numpy oracle.

``launch_mh_mvn<D>`` picks one of 72 instantiations: the per-thread ``mh_mvn_kernel<D, kInjected>``
(16), the warp-specialised ``mh_mvn_ws_kernel<D, kRefAccept, kFast, kZeroMean>`` (5 flag
combinations for each D = 1..8, 40) and the whitened-decision ``mh_mvn_wd_kernel<D, kFast,
kZeroMean>`` (4 for each D = 1..4, 16).  ``_instantiation`` restates that choice.  Every case
replays its chains on the CPU: native-RNG runs from ``oracle/philox.py`` (normal, uniform and
spherical proposals, per-dimension scales, Cholesky colouring) through ``np_oracle.mh_mvn_walk``
at arbitrary ``step0`` / ``chain0``, so no kernel is only compared with another kernel.

Tolerances (DESIGN section 4): accept decisions identical; native-RNG trajectories <= 1e-11
absolute, injected ones <= 1e-12; densities within 1e-11 relative (1e-12 injected) or, for linear
densities that underflow into the subnormal range, 2 ulp; running sums |d| <= 1e-11 * sum |x|."""
import re
from collections import namedtuple

import numpy as np
import pytest
from gpu_util import engine, dev, tcd_to_tdc, host
from oracle import np_oracle as o
from oracle import philox

NTOL = 1e-11           # native-RNG trajectories (table log / sincos / sqrt against glibc)
ITOL = 1e-12           # injected streams: the same arithmetic as the oracle up to fma contraction
SUM_TOL = 1e-11        # running sums, relative to sum |x| (sum x^2)
# scores of the reference rule divide a linear density by max(tiny, lin): where the density is
# subnormal, one ulp of it (2^-1074, libm exp on either side) is 2.2e-16 of the score
SCORE_ATOL = 4.5e-16
HI = 2 ** 32 - 5       # a walk from here crosses into the Philox step high word
RADIUS = 0.9           # spherical proposals

PT, WS, WD = "mh_mvn_kernel", "mh_mvn_ws_kernel", "mh_mvn_wd_kernel"


# ---------------------------------------------------------------------------------------------
# dispatch mirror (pbx_mh_mvn_run -> launch_mh_mvn<D>)
# ---------------------------------------------------------------------------------------------
def _instantiation(D, accept, prop, chol, mean, injected, per_step, bound, variant):
    """(kernel, D, template flags...) launched for a walk in ``D`` dimensions, or None where the
    call is refused (variant 4 outside the whitened-decision kernel's domain).  ``chol``: a
    proposal Cholesky factor is given; ``mean`` is the target mean (kZeroMean when every entry
    is exactly 0)."""
    use_ws = not injected and not per_step and variant != 1 and not bound
    wd_ok = use_ws and D <= 4 and accept == "log"
    if variant == 4 and not wd_ok:
        return None
    fast = prop == "normal" and not chol
    zero = bool(np.all(np.asarray(mean, dtype=float) == 0.0))
    if wd_ok and variant != 2:
        return (WD, D, fast, zero)
    if use_ws:
        if accept == "reference":
            return (WS, D, True, fast, False)
        return (WS, D, False, fast, fast and zero)
    return (PT, D, bool(injected))


def _wd_cpc(C, sm_count):
    """wd_pick_cpc: the chains per CTA that fill whole waves of SMs at the least cost
    waves * cpc; ties go to the earlier candidate."""
    best, best_cost = 32, None
    for cand in (32, 28, 16, 8, 4):
        ctas = -(-C // cand)
        cost = -(-ctas // sm_count) * cand
        if best_cost is None or cost < best_cost:
            best, best_cost = cand, cost
    return best


CPCS = (32, 28, 16, 8, 4)
WS_FLAGS = [(True, True, False), (True, False, False), (False, True, True), (False, True, False),
            (False, False, False)]
REACHABLE = {(PT, D, inj) for D in range(1, 9) for inj in (False, True)} | \
            {(WS, D) + f for D in range(1, 9) for f in WS_FLAGS} | \
            {(WD, D, f, z) for D in range(1, 5) for f in (False, True) for z in (False, True)}


def _name(inst):
    """The demangled template-id of an instantiation, e.g. mh_mvn_ws_kernel<4, false, true, true>."""
    args = ["true" if a is True else "false" if a is False else str(a) for a in inst[1:]]
    return "%s<%s>" % (inst[0], ", ".join(args))


def _cpc_chains(cpc, sm_count):
    """The smallest chain count >= 97 for which the host picks ``cpc`` and whose last CTA is
    partial."""
    for C in range(97, 40 * 32 * sm_count):
        if _wd_cpc(C, sm_count) == cpc and C % cpc:
            return C
    raise AssertionError("no chain count picks cpc = %d on %d SMs" % (cpc, sm_count))


def _wd_batch(cpc):
    """Steps per batch of the whitened-decision kernel: 448 / cpc pairs."""
    return 2 * (448 // cpc)


def _sample(C, width, n=96, seed=0):
    """Chains replayed on the CPU: all of them when there are few, else chain 0, the last chain,
    both sides of three CTA boundaries (the first, one in the middle and the start of the
    partial last CTA) and random others."""
    if C <= n:
        return np.arange(C)
    nb = C // width
    must = {0, C - 1, width - 1, width, nb // 2 * width - 1, nb // 2 * width,
            nb * width - 1, min(nb * width, C - 1)}
    rest = np.setdiff1d(np.arange(C), sorted(must))
    pick = np.random.default_rng(seed).choice(rest, n - len(must), replace=False)
    return np.sort(np.concatenate([sorted(must), pick]))


# ---------------------------------------------------------------------------------------------
# cases
# ---------------------------------------------------------------------------------------------
Case = namedtuple("Case", "D accept logp prop chol zero injected per_step bound variant C T thin "
                          "step0 chain0 reorder")
Case.__new__.__defaults__ = ("log", True, "normal", False, False, False, False, False, 0, 101, 97,
                             1, 0, 0, True)

# (step0, chain0), cycled over the cases: the unconditional first step, the Philox high word
# with chain ids offset, and odd resumes
STARTS = [(0, 0), (HI, 1000003), (13, 0), (HI, 7), (0, 4099), (7, 250)]
PROPS = ["normal", "uniform", "spherical"]


def _parity_cases():
    """One case per reachable instantiation.  Across the list: both accept rules, both pscales,
    every proposal, Cholesky colouring, zero and nonzero mean, reorder on and off, thin 1 and 3,
    T not a multiple of the ws slot length or the wd batch, ragged chain counts."""
    cases = []
    for D in range(1, 9):
        odd = D % 2 == 1
        nonfast = PROPS[1 + D % 2]                               # uniform or spherical
        # per-thread kernel: native stream (with per-step outputs) and injected streams
        cases.append(Case(D, accept="reference" if odd else "log", logp=D % 3 != 1,
                          prop=PROPS[D % 3], chol=D in (3, 6, 7), per_step=True, bound=D == 2,
                          C=45 + 7 * D, thin=1 + 2 * (D % 2)))
        cases.append(Case(D, accept="log" if odd else "reference", logp=D % 3 != 0,
                          chol=D in (1, 4, 8), injected=True, per_step=True, C=40 + 9 * D,
                          thin=3 - 2 * (D % 2)))
        # warp-specialised kernel: the five flag sets (variant 2 keeps D <= 4 off wd)
        cases.append(Case(D, accept="reference", logp=odd, C=70 + 3 * D, thin=1))
        cases.append(Case(D, accept="reference", logp=not odd, prop=nonfast if D % 3 else "normal",
                          chol=D % 3 == 0, C=75 + 3 * D, thin=3))
        cases.append(Case(D, logp=not odd, zero=True, variant=2, C=80 + 3 * D, thin=1))
        cases.append(Case(D, logp=odd, variant=2, C=85 + 3 * D, thin=3, reorder=not odd))
        cases.append(Case(D, logp=D % 4 < 2, prop=nonfast if D != 4 else "normal",
                          chol=D in (4, 5, 8), zero=D % 4 == 0, variant=2, C=90 + 3 * D,
                          thin=1 + 2 * (D % 2)))
        if D <= 4:
            for fast in (True, False):
                for zero in (True, False):
                    cases.append(Case(D, logp=fast != zero, prop="normal" if fast else
                                      PROPS[1 + (D + zero) % 2], chol=not fast and D == 3 and zero,
                                      zero=zero, C=101 + 2 * D, T=2 * _wd_batch(4) + 3,
                                      thin=1 if zero else 3))
    return [c._replace(step0=STARTS[i % len(STARTS)][0], chain0=STARTS[i % len(STARTS)][1])
            for i, c in enumerate(cases)]


CASES = _parity_cases()


def _inst(k):
    return _instantiation(k.D, k.accept, k.prop, k.chol, np.zeros(k.D) if k.zero else np.ones(k.D),
                          k.injected, k.per_step, k.bound, k.variant)


def _case_id(k):
    return "%s-%s-%s-%s" % (_name(_inst(k)), k.accept[:3], "logp" if k.logp else "lin", k.prop)


def test_dispatch_mirror_rules():
    assert len(REACHABLE) == 72
    z2, m2 = np.zeros(2), np.array([0.0, 0.5])
    cases = [
        ((2, "log", "normal", False, z2, False, False, False, 0), (WD, 2, True, True)),
        ((2, "log", "normal", False, m2, False, False, False, 0), (WD, 2, True, False)),
        ((2, "log", "normal", True, z2, False, False, False, 4), (WD, 2, False, True)),
        ((4, "log", "uniform", False, m2, False, False, False, 0), (WD, 4, False, False)),
        ((4, "log", "normal", False, z2, False, False, False, 2), (WS, 4, False, True, True)),
        ((3, "log", "spherical", False, z2, False, False, False, 2), (WS, 3, False, False, False)),
        ((4, "reference", "normal", False, z2, False, False, False, 0), (WS, 4, True, True, False)),
        ((1, "reference", "uniform", False, m2, False, False, False, 0), (WS, 1, True, False, False)),
        ((5, "log", "normal", False, np.zeros(5), False, False, False, 0), (WS, 5, False, True, True)),
        ((8, "log", "normal", False, np.ones(8), False, False, False, 0), (WS, 8, False, True, False)),
        ((6, "log", "normal", True, np.zeros(6), False, False, False, 0), (WS, 6, False, False, False)),
        ((2, "log", "normal", False, z2, False, False, False, 1), (PT, 2, False)),
        ((2, "log", "normal", False, z2, False, True, False, 0), (PT, 2, False)),     # per-step
        ((2, "log", "normal", False, z2, False, False, True, 0), (PT, 2, False)),     # bound
        ((7, "reference", "uniform", False, z2, True, False, False, 0), (PT, 7, True)),
        ((2, "reference", "normal", False, z2, False, False, False, 4), None),
        ((5, "log", "normal", False, np.zeros(5), False, False, False, 4), None),
        ((2, "log", "normal", False, z2, False, True, False, 4), None),
    ]
    for args, want in cases:
        assert _instantiation(*args) == want, args
    # exhaustively over the arguments: exactly the 72 compiled instantiations are reached
    seen = set()
    for D in range(1, 9):
        for accept in ("reference", "log"):
            for prop in PROPS:
                for chol in (False, True):
                    for mean in (np.zeros(D), np.ones(D)):
                        for inj, ps, bd in ((False, False, False), (True, True, False),
                                            (False, True, False), (False, False, True)):
                            for variant in (0, 1, 2, 4):
                                got = _instantiation(D, accept, prop, chol, mean, inj, ps, bd,
                                                     variant)
                                if got is not None:
                                    seen.add(got)
    assert seen == REACHABLE
    # the demangled names the profiler reports
    assert _name((WS, 4, False, True, True)) == "mh_mvn_ws_kernel<4, false, true, true>"
    assert _name((PT, 7, True)) == "mh_mvn_kernel<7, true>"
    # wd_pick_cpc on 148 SMs
    for C, cpc in ((1, 4), (100, 4), (592, 4), (593, 8), (1184, 8), (1185, 4), (1776, 4),
                   (1777, 16), (2368, 16), (2369, 4), (2961, 8), (3553, 28), (4096, 28),
                   (4144, 28), (4145, 32), (4736, 32), (4737, 4), (5000, 4)):
        assert _wd_cpc(C, 148) == cpc, C
    for cpc in CPCS:
        C = _cpc_chains(cpc, 148)
        assert _wd_cpc(C, 148) == cpc and C % cpc and C >= 97


def _reaches(sm_count):
    got = {_inst(k) for k in CASES}
    assert got == REACHABLE, sorted(REACHABLE - got)
    assert len(CASES) == len(REACHABLE)
    assert {_wd_cpc(_cpc_chains(cpc, sm_count), sm_count) for cpc in CPCS} == set(CPCS)
    for k in CASES:                      # every wd parity case has one whole batch and a tail
        if _inst(k)[0] == WD:
            S = _wd_batch(_wd_cpc(k.C, sm_count))
            assert k.T > S and k.T % S and k.C % _wd_cpc(k.C, sm_count)


def test_case_list_reaches_every_instantiation_on_148_sms():
    _reaches(148)
    kinds = {(k.accept, k.logp, k.prop, k.chol, k.zero, k.reorder) for k in CASES}
    for accept in ("reference", "log"):
        for logp in (False, True):
            assert any(a == accept and lp == logp for a, lp, *_ in kinds)
    assert {k.prop for k in CASES} == set(PROPS) and any(k.chol for k in CASES)
    assert {k.step0 for k in CASES} >= {0, HI} and any(k.step0 % 2 for k in CASES)


@pytest.mark.gpu
def test_case_list_reaches_every_instantiation():
    _reaches(engine().info.sm_count)


# ---------------------------------------------------------------------------------------------
# models, device runs and the CPU replay
# ---------------------------------------------------------------------------------------------
def _model(D, seed, zero=False):
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((D, D))
    cov = A @ A.T / D + np.eye(D)
    mean = np.zeros(D) if zero else rng.standard_normal(D)
    return mean, cov, rng


def _scale(D):
    return 0.45 + 0.1 * np.arange(D)


def _chol(k, cov):
    return np.linalg.cholesky(0.3 * cov) if k.chol else None


def _bound(D):
    """Closed and open ends mixed; a proposal past an open end bounces back."""
    lims = np.tile([-1.5, 1.4], (D, 1))
    ex = np.array([[j % 2, (j + 1) % 2] for j in range(D)])
    return lims, ex


def _logpdf(x, mean, cov, reorder):
    U, lpd = o.mvn_whiten(cov)
    order = o.mvn_value_order(len(mean)) if reorder else list(range(len(mean)))
    return o.mvn_logpdf(x[..., order], np.asarray(mean, dtype=float), U, lpd)


def _deltas(k, seed, chains, scale=None):
    """The native proposal deltas [T, n, D] of the chain ids ``chains``."""
    scale = _scale(k.D) if scale is None else scale
    if k.prop == "normal":
        return philox.normals(seed, k.T, chains, k.D, k.step0) * scale
    if k.prop == "uniform":
        return -scale + (2.0 * scale) * philox.uniforms(seed, k.T, chains, k.D, k.step0)
    return philox.spherical(seed, k.T, chains, k.D, RADIUS, scale, k.step0)


def _replay(k, init, mean, cov, seed, sel, delta=None, thresh=None, scale=None):
    """The oracle's walk of chains ``sel`` (ids ``chain0 + sel``) from ``init[sel]``.  A walk
    from ``step0 > 0`` decides at its first step, from the density passed as ``state_lp``: the
    oracle gets a zero move in front, which it accepts, so that it starts from that density.
    The log rule is replayed in log pscale (the oracle's form of it) and its densities are
    exponentiated for linear-pscale runs."""
    chains = sel.astype(np.uint64) + np.uint64(k.chain0)
    if delta is None:
        delta = _deltas(k, seed, chains, scale)
        thresh = philox.thresholds(seed, k.T, chains, k.step0)
    lp_walk = k.logp or k.accept == "log"
    if k.step0 > 0:
        delta = np.concatenate([np.zeros((1,) + delta.shape[1:]), delta])
        thresh = np.concatenate([np.full((1, len(sel)), 0.5), thresh])
    ref = o.mh_mvn_walk(init[sel], delta, thresh, mean, cov, tran_chol=_chol(k, cov),
                        log_pscale=lp_walk, reorder=k.reorder, accept=k.accept,
                        bound=_bound(k.D) if k.bound else None)
    if k.step0 > 0:
        ref = {key: v[1:] for key, v in ref.items()}
    if lp_walk and not k.logp:
        ref["prob"], ref["pprop"] = np.exp(ref["prob"]), np.exp(ref["pprop"])
    return ref


def _run(eng, k, init, mean, cov, seed, inj=None, scale=None, **kw):
    """Runs case ``k`` from ``init`` [C, D]; returns (out, state)."""
    state = dev(eng, init.T)
    if k.step0 > 0 and "state_lp" not in kw:
        kw["state_lp"] = dev(eng, _logpdf(init, mean, cov, k.reorder))
    if inj is not None:
        kw.update(inj_delta=dev(eng, tcd_to_tdc(inj[0])), inj_thresh=dev(eng, inj[1]))
    out = eng.mh_mvn(state, mean, cov, k.T, thin=k.thin, seed=seed, step0=k.step0,
                     chain0=k.chain0, log_pscale=k.logp, accept=k.accept, prop=k.prop,
                     prop_scale=_scale(k.D) if scale is None else scale,
                     prop_chol=_chol(k, cov), reorder=k.reorder, per_step=k.per_step,
                     variant=k.variant, prop_radius=RADIUS,
                     bound=_bound(k.D) if k.bound else None, **kw)
    return out, state


def _fetch(out, state, sel, last=None):
    """Host copies of the outputs of chains ``sel`` (the last ``last`` records only), sliced on
    the device."""
    import torch
    idx = torch.as_tensor(sel, device=state.device)
    got = {"state": host(state[:, idx])}
    for key in ("x", "prob", "accept", "score", "xprop", "pprop"):
        if key in out:
            t = out[key] if last is None else out[key][-last:]
            got[key] = host(t.index_select(t.dim() - 1, idx))
    for key in ("accept_count", "state_lp"):
        got[key] = host(out[key][idx])
    for key in ("stat_sum", "stat_sumsq"):
        got[key] = host(out[key][:, idx])
    return got


def _dens_close(got, want, rtol, what):
    """Within ``rtol`` relative, or 2 ulp of the reference where it is subnormal or 0."""
    got, want = np.asarray(got, dtype=float), np.asarray(want, dtype=float)
    assert got.shape == want.shape, what
    tol = np.maximum(rtol * np.abs(want), 2 * np.spacing(np.abs(want)))
    bad = ~(np.abs(got - want) <= tol)
    assert not bad.any(), "%s: %d off, e.g. %r vs %r" % (what, bad.sum(), got[bad][:3], want[bad][:3])


def _check(k, got, ref, mean, cov, injected=False, last=None):
    """Every output of the chains in ``got`` (from ``_fetch``) against the oracle walk ``ref``."""
    tol = ITOL if injected else NTOL
    X = ref["x"]                                                   # [T, n, D]
    recs = slice(k.thin - 1, None, k.thin)
    Xr = tcd_to_tdc(X)[recs]
    Pr = ref["prob"][recs]
    if last is not None:
        Xr, Pr = Xr[-last:], Pr[-last:]
    assert got["x"].shape == Xr.shape
    if Xr.size:
        assert np.abs(got["x"] - Xr).max() <= tol
        _dens_close(got["prob"], Pr, tol, "prob")
    assert np.array_equal(got["accept_count"], ref["u"].sum(axis=0))
    assert np.abs(got["state"] - X[-1].T).max() <= tol
    _dens_close(got["state_lp"], _logpdf(X[-1], mean, cov, k.reorder), tol, "state_lp")
    s1, s2 = X.sum(axis=0).T, (X * X).sum(axis=0).T
    assert (np.abs(got["stat_sum"] - s1) <= SUM_TOL * np.abs(X).sum(axis=0).T).all()
    assert (np.abs(got["stat_sumsq"] - s2) <= SUM_TOL * s2).all()
    if "accept" in got:                                            # per-step outputs
        assert np.array_equal(got["accept"].astype(bool), ref["u"])
        assert np.abs(got["xprop"] - tcd_to_tdc(ref["xprop"])).max() <= tol
        _dens_close(got["pprop"], ref["pprop"], tol, "pprop")
        s, want = got["score"], ref["s"]
        assert np.array_equal(np.isnan(s), np.isnan(want))
        ok = ~np.isnan(want)
        assert (np.abs(s[ok] - want[ok]) <= tol * np.abs(want[ok]) + SCORE_ATOL).all()
        if k.step0 == 0:
            assert np.isnan(s[0]).all()


def _injected_streams(k, rng, C):
    return rng.standard_normal((k.T, C, k.D)) * _scale(k.D), rng.random((k.T, C))


@pytest.mark.gpu
@pytest.mark.parametrize("k", CASES, ids=[_case_id(k) for k in CASES])
def test_every_instantiation_against_oracle(k):
    eng = engine()
    mean, cov, rng = _model(k.D, 1000 * k.D + k.C, k.zero)
    init = mean + rng.standard_normal((k.C, k.D))
    if k.bound:
        init = rng.uniform(-1.0, 1.0, (k.C, k.D))
    seed = 0x51A0 + 17 * k.C
    inj = _injected_streams(k, rng, k.C) if k.injected else None
    sel = np.arange(k.C)
    out, state = _run(eng, k, init, mean, cov, seed, inj)
    eng.sync()
    ref = _replay(k, init, mean, cov, seed, sel, *(inj or ()))
    assert ref["u"][1:].any() and not ref["u"][1:].all()          # decisions go both ways
    _check(k, _fetch(out, state, sel), ref, mean, cov, injected=k.injected)


# ---------------------------------------------------------------------------------------------
# geometry and counter edges
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cpc", CPCS)
@pytest.mark.parametrize("D", [1, 2, 3, 4])
def test_whitened_decision_every_cpc(D, cpc):
    """wd at each chains-per-CTA shape: two whole batches and a tail, ragged last CTA.  At
    cpc = 32 a batch has 14 pairs, so the D <= 2 decision loop ends every whole batch with its
    remainder code."""
    eng = engine()
    sm = eng.info.sm_count
    C = _cpc_chains(cpc, sm)
    k = Case(D, logp=D % 2 == 0, prop="normal" if D != 3 else "uniform", zero=D in (1, 3), C=C,
             T=2 * _wd_batch(cpc) + 5, thin=1 if cpc in (32, 16, 4) else 3,
             step0=(0, 9, HI)[cpc % 3], chain0=31 * cpc)
    assert _inst(k)[0] == WD and _wd_cpc(C, sm) == cpc
    mean, cov, rng = _model(D, 7 * cpc + D, k.zero)
    init = mean + rng.standard_normal((C, D))
    seed = 1234567 + cpc
    out, state = _run(eng, k, init, mean, cov, seed)
    eng.sync()
    sel = _sample(C, cpc)
    _check(k, _fetch(out, state, sel), _replay(k, init, mean, cov, seed, sel), mean, cov)


# (family, T, thin, C, step0): a single step (that decides: step0 > 0), thin > T (no records)
# and a single chain, for each kernel family
TINY = [(fam, T, thin, C, step0) for fam in ("pt", "ws", "wd")
        for T, thin, C, step0 in ((1, 1, 37, 5), (7, 9, 40, 0), (29, 2, 1, 3))]
FAMILY = {"pt": dict(variant=1), "ws": dict(variant=2), "wd": dict(variant=0)}


@pytest.mark.gpu
@pytest.mark.parametrize("fam,T,thin,C,step0", TINY)
def test_tiny_walks(fam, T, thin, C, step0):
    eng = engine()
    k = Case(3, logp=fam != "ws", C=C, T=T, thin=thin, step0=step0, chain0=11, **FAMILY[fam])
    assert _inst(k)[0] == {"pt": PT, "ws": WS, "wd": WD}[fam]
    mean, cov, rng = _model(3, 50 + T)
    init = mean + rng.standard_normal((C, 3))
    out, state = _run(eng, k, init, mean, cov, 99)
    eng.sync()
    assert host(out["x"]).shape == (T // thin, 3, C)
    sel = np.arange(C)
    _check(k, _fetch(out, state, sel), _replay(k, init, mean, cov, 99, sel), mean, cov)


# resume at an odd step into the walk: ws at D = 4 (384-thread CTA) and D = 6, the reference
# rule in linear pscale (the consumer re-derives lin from state_lp), wd, and the per-thread kernel
RESUME = {"ws4": Case(4, variant=2), "ws6": Case(6, logp=False),
          "ws-ref-lin": Case(3, accept="reference", logp=False),
          "pt-ref-lin": Case(2, accept="reference", logp=False, variant=1),
          "wd": Case(2, logp=False, zero=True)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(RESUME))
def test_resume_at_odd_step_is_bit_exact(name):
    eng = engine()
    k = RESUME[name]._replace(C=150, T=97, chain0=3)
    mean, cov, rng = _model(k.D, 60 + k.D, k.zero)
    init = mean + rng.standard_normal((k.C, k.D))
    seed, h = 777, 37
    one, s_one = _run(eng, k, init, mean, cov, seed)
    a, s_two = _run(eng, k._replace(T=h), init, mean, cov, seed)
    state_lp = a["state_lp"].clone()
    b = eng.mh_mvn(s_two, mean, cov, k.T - h, seed=seed, step0=h, chain0=k.chain0,
                   log_pscale=k.logp, accept=k.accept, prop_scale=_scale(k.D),
                   variant=k.variant, state_lp=state_lp)
    eng.sync()
    assert np.array_equal(host(s_two), host(s_one))
    assert np.array_equal(host(state_lp), host(one["state_lp"]))
    for key in ("x", "prob"):
        assert np.array_equal(np.concatenate([host(a[key]), host(b[key])]), host(one[key])), key
    assert np.array_equal(host(a["accept_count"]) + host(b["accept_count"]),
                          host(one["accept_count"]))
    for key in ("stat_sum", "stat_sumsq"):
        tot = host(one[key])
        assert (np.abs(host(a[key]) + host(b[key]) - tot) <= SUM_TOL * np.abs(tot)).all()
    sel = np.arange(k.C)
    _check(k, _fetch(one, s_one, sel), _replay(k, init, mean, cov, seed, sel), mean, cov)


# ---------------------------------------------------------------------------------------------
# density edges: chains 37-40 sigma out, log densities down to -800
# ---------------------------------------------------------------------------------------------
EDGES = [("pt", acc, lp) for acc in ("reference", "log") for lp in (False, True)] + \
        [("ws", acc, lp) for acc in ("reference", "log") for lp in (False, True)] + \
        [("wd", "log", lp) for lp in (False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("fam,accept,logp", EDGES)
def test_density_edges(fam, accept, logp):
    """Linear densities below exp(-700) (libm past the table exp), subnormal and 0; the reference
    rule with an underflowing density (the max(tiny, lin) clamp and the clamped exp): chains
    whose density is 0 stay where they are, exactly as in the oracle."""
    eng = engine()
    D = 4 if fam == "ws" else 2
    k = Case(D, accept=accept, logp=logp, C=96, T=61, step0=11, chain0=5,
             per_step=fam == "pt", variant=FAMILY[fam]["variant"])
    assert _inst(k)[0] == {"pt": PT, "ws": WS, "wd": WD}[fam]
    mean, cov, rng = _model(D, 400 + D)
    u = rng.standard_normal((k.C, D))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    r = np.linspace(37.0, 40.0, k.C)
    r[::8] = 0.5                                   # and a few chains in the bulk
    y = mean + r[:, None] * (u @ np.linalg.cholesky(cov).T)     # the point scipy sees
    init = np.empty_like(y)
    init[:, o.mvn_value_order(D)] = y
    seed = 2718
    scale = np.full(D, 0.25)
    out, state = _run(eng, k, init, mean, cov, seed, scale=scale)
    eng.sync()
    sel = np.arange(k.C)
    ref = _replay(k, init, mean, cov, seed, sel, scale=scale)
    lp = _logpdf(ref["x"], mean, cov, k.reorder)                  # of every recorded state
    for lo, hi in ((-np.inf, -745.2), (-745.1, -708.5), (-708.3, -700.0), (-699.0, -600.0)):
        assert ((lp > lo) & (lp < hi)).any(), (lo, hi)
    if not logp:
        assert (ref["prob"] == 0).any() and ((ref["prob"] > 0) & (ref["prob"] < 2.2e-308)).any()
    if accept == "reference":
        stuck = ref["u"].sum(axis=0) == 0
        assert stuck.any() and (~stuck).any()
        assert (ref["x"][:, stuck] == init[stuck]).all()
    _check(k, _fetch(out, state, sel), ref, mean, cov)


# ---------------------------------------------------------------------------------------------
# host-streamed walk and 64-bit output offsets
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("D", [3, 4, 6])
def test_walk_host_equals_one_device_call(D):
    """pbx_mh_mvn_walk_host in chunks of an odd number of steps (39: 37 rounded up to whole
    records of thin = 3) equals one device call bit for bit."""
    eng = engine()
    C, T, seed, chain0 = 130, 230, 4321, 9
    mean, cov, rng = _model(D, 70 + D)
    init = rng.standard_normal((D, C))
    kw = dict(seed=seed, thin=3, chain0=chain0, accept="log" if D <= 4 else "reference",
              log_pscale=D != 4, prop_scale=_scale(D))
    st = dev(eng, init)
    d = eng.mh_mvn(st, mean, cov, T, **kw)
    eng.sync()
    h = eng.mh_mvn_walk_host(init.copy(), mean, cov, T, chunk_steps=37, **kw)
    for key in ("x", "prob", "accept_count", "state_lp"):
        assert np.array_equal(h[key], host(d[key])), key
    assert np.array_equal(h["state"], host(st))
    for key in ("stat_sum", "stat_sumsq"):
        want = host(d[key])
        assert (np.abs(h[key] - want) <= SUM_TOL * np.abs(want)).all(), key


@pytest.mark.gpu
@pytest.mark.parametrize("fam", ["pt", "ws", "wd"])
def test_output_offsets_beyond_2_31(fam):
    """R * D * C > 2^31 elements of x (17 GB): the last records of the last 32 chains lie past
    2^31 and are replayed through the oracle with their chain ids."""
    import torch
    eng = engine()
    D, C, T = 4, 32768 + 37, 16384
    assert T * D * C > 2 ** 31
    k = Case(D, logp=True, C=C, T=T, **FAMILY[fam])
    assert _inst(k)[0] == {"pt": PT, "ws": WS, "wd": WD}[fam]
    mean, cov, rng = _model(D, 90)
    init = mean + rng.standard_normal((C, D))
    seed = 8080
    out = state = None
    try:
        out, state = _run(eng, k, init, mean, cov, seed)
        sel = np.arange(C - 32, C)
        got = _fetch(out, state, sel, last=3)
        eng.sync()
    finally:
        del out, state
        torch.cuda.empty_cache()
    _check(k, got, _replay(k, init, mean, cov, seed, sel), mean, cov, last=3)


# ---------------------------------------------------------------------------------------------
# each case really launches the instantiation the mirror names
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_each_case_launches_its_instantiation():
    import torch
    from torch.profiler import profile, ProfilerActivity
    eng = engine()
    runs = []
    for k in CASES:
        k = k._replace(T=6, C=40)
        mean, cov, rng = _model(k.D, 5, k.zero)
        init = mean + rng.standard_normal((k.C, k.D))
        if k.bound:
            init = rng.uniform(-1.0, 1.0, (k.C, k.D))
        runs.append((k, init, mean, cov, _injected_streams(k, rng, k.C) if k.injected else None))
    eng.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        probe = torch.ones(1024, device=eng.device, dtype=torch.float64) * 3.0
        for k, init, mean, cov, inj in runs:
            _run(eng, k, init, mean, cov, 42, inj)
        eng.sync()
        torch.cuda.synchronize()
    del probe
    kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    if not kern:
        pytest.skip("the profiler recorded no device events, not even the probe's torch kernel")
    kern.sort(key=lambda e: e.time_range.start)
    names = []
    for e in kern:
        m = re.search(r"(mh_mvn(?:_ws|_wd)?_kernel<[^>]*>)", e.name)
        if m:
            names.append(re.sub(r"\s+", " ", m.group(1)))
    want = [_name(_inst(k)) for k, *_ in runs]
    assert names == want
    assert len(set(names)) == 72
