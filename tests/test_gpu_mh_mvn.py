"""K1 parity (GPU, through the C ABI): batched-chain MH on a multivariate-normal
target against the golden fixtures (live reference) and the numpy oracle.
Tolerances: accept decisions identical; trajectories / densities within 1e-12
(north_star, fp64)."""
import numpy as np
import pytest
from conftest import load_golden, relerr
from gpu_util import engine, dev, tcd_to_tdc, host
from oracle import np_oracle as o
from oracle import philox

pytestmark = pytest.mark.gpu
TOL = 1e-12
COV = np.array([[2.0, 1.2], [1.2, 2.0]])


@pytest.mark.parametrize("name", ["mh_mvn_c1", "mh_mvn_c1_b", "mh_mvn_log", "mh_mvn_3d"])
def test_golden_injected(name):
    eng = engine()
    g = load_golden(name)
    T = len(g["thresh"])
    state = dev(eng, g["init"][:, None])
    out = eng.mh_mvn(state, g["mean"], g["cov"], T, log_pscale=bool(g["log_pscale"]),
                     inj_delta=dev(eng, tcd_to_tdc(g["delta"][:, None, :])),
                     inj_thresh=dev(eng, g["thresh"][:, None]), per_step=True)
    eng.sync()
    assert np.array_equal(host(out["accept"])[:, 0].astype(bool), g["u"])
    assert np.abs(host(out["x"])[:, :, 0] - g["x"]).max() <= TOL
    assert relerr(host(out["prob"])[:, 0], g["prob"]) <= TOL
    s = host(out["score"])[:, 0]
    assert np.isnan(s[0]) and relerr(s[1:], g["s"][1:]) <= TOL
    assert int(host(out["accept_count"])[0]) == int(g["u"].sum())


def test_bounded_delta_golden_and_native():
    """K1 with set_delta(..., bound=True) (variable.py:700-739): the live-reference fixture
    with injected streams (decisions identical, trajectory <= 1e-12), then native RNG on
    many chains against the Philox replay through the oracle."""
    eng = engine()
    g = load_golden("mh_mvn_bound")
    T = len(g["thresh"])
    bound = (g["lims"], g["ex"])
    state = dev(eng, g["init"][:, None])
    out = eng.mh_mvn(state, g["mean"], g["cov"], T, prop="uniform", prop_scale=float(g["step"]),
                     inj_delta=dev(eng, tcd_to_tdc(g["delta"][:, None, :])),
                     inj_thresh=dev(eng, g["thresh"][:, None]), per_step=True, bound=bound)
    eng.sync()
    assert np.array_equal(host(out["accept"])[:, 0].astype(bool), g["u"])
    assert np.abs(host(out["x"])[:, :, 0] - g["x"]).max() <= TOL
    assert relerr(host(out["prob"])[:, 0], g["prob"]) <= TOL
    assert np.abs(host(out["xprop"])[:, :, 0] - g["xprop"]).max() <= TOL
    # native RNG, uniform proposal, 70 chains: Philox replay
    C, T2, seed = 70, 200, 424242
    init = np.tile(g["init"], (C, 1))
    t = np.arange(T2, dtype=np.uint64)[:, None]
    c = np.arange(C, dtype=np.uint64)[None, :]
    r0, r1 = philox.uniform_pair(seed, t, c, 0)
    step = float(g["step"])
    delta = np.stack([-step + (2 * step) * r0, -step + (2 * step) * r1], axis=-1)
    ref = o.mh_mvn_walk(init, delta, philox.thresholds(seed, T2, C), g["mean"], g["cov"],
                        accept="log", log_pscale=True, bound=bound)
    out = eng.mh_mvn(dev(eng, init.T), g["mean"], g["cov"], T2, seed=seed, accept="log",
                     log_pscale=True, prop="uniform", prop_scale=step, bound=bound)
    eng.sync()
    assert np.array_equal(host(out["accept_count"]), ref["u"].sum(axis=0))
    assert np.abs(host(out["x"]) - tcd_to_tdc(ref["x"])).max() <= 1e-11
    x = host(out["x"])
    assert x.min() >= -1.5 and x.max() <= 1.5 and (np.abs(x[:, 0]) == 1.5).any()


@pytest.mark.parametrize("D,C,T,log_pscale,chol", [
    (2, 257, 300, False, False), (2, 64, 200, True, False), (3, 33, 150, False, True),
    (5, 100, 120, True, False), (8, 40, 100, False, True), (1, 31, 100, False, False)])
def test_oracle_injected(D, C, T, log_pscale, chol):
    eng = engine()
    rng = np.random.default_rng(100 + D)
    A = rng.standard_normal((D, D))
    cov = A @ A.T / D + np.eye(D)
    mean = rng.standard_normal(D)
    init = rng.standard_normal((C, D)) * 2
    delta = rng.standard_normal((T, C, D)) * 0.8
    thresh = rng.random((T, C))
    L = None
    if chol:
        B = rng.standard_normal((D, D))
        L = np.linalg.cholesky(B @ B.T / D + 0.5 * np.eye(D))
    ref = o.mh_mvn_walk(init, delta, thresh, mean, cov, tran_chol=L, log_pscale=log_pscale)
    state = dev(eng, init.T)
    out = eng.mh_mvn(state, mean, cov, T, log_pscale=log_pscale, prop_chol=L,
                     inj_delta=dev(eng, tcd_to_tdc(delta)), inj_thresh=dev(eng, thresh),
                     per_step=True)
    eng.sync()
    assert np.array_equal(host(out["accept"]).astype(bool), ref["u"])
    assert np.abs(host(out["x"]) - tcd_to_tdc(ref["x"])).max() <= TOL
    assert relerr(host(out["prob"]), ref["prob"]) <= TOL
    assert relerr(host(out["score"])[1:], ref["s"][1:]) <= 1e-11
    assert np.abs(host(state) - ref["x"][-1].T).max() <= TOL
    assert np.array_equal(host(out["accept_count"]), ref["u"].sum(axis=0))
    # running sums feed R-hat
    assert relerr(host(out["stat_sum"]), ref["x"].sum(axis=0).T) <= 1e-11


@pytest.mark.parametrize("accept", ["reference", "log"])
def test_philox_replay(accept):
    """Native-RNG run == injected-stream restatement fed with the same Philox
    stream generated on the CPU (oracle/philox.py)."""
    eng = engine()
    C, T, seed = 96, 250, 20240607
    init = np.tile(np.array([0., 1.]), (C, 1))
    Z = philox.normals(seed, T, C, 2)
    U = philox.thresholds(seed, T, C)
    ref = o.mh_mvn_walk(init, Z, U, [0., 0.], COV, log_pscale=(accept == "log"),
                        accept=accept)
    state = dev(eng, init.T)
    out = eng.mh_mvn(state, [0., 0.], COV, T, seed=seed, accept=accept,
                     log_pscale=(accept == "log"), per_step=True)
    eng.sync()
    same = host(out["accept"]).astype(bool) == ref["u"]
    assert same.all()
    assert np.abs(host(out["x"]) - tcd_to_tdc(ref["x"])).max() <= 1e-11
    assert relerr(host(out["prob"]), ref["prob"]) <= 1e-11


@pytest.mark.parametrize("D,C,T,accept,logp,prop,chol", [
    (2, 4096, 333, "log", False, "normal", False), (2, 100, 257, "reference", False, "normal", False),
    (2, 33, 100, "log", True, "uniform", False), (3, 65, 130, "log", True, "normal", True),
    (5, 40, 90, "reference", True, "normal", False), (8, 64, 64, "log", False, "normal", True),
    (1, 50, 77, "log", False, "normal", False), (7, 48, 70, "log", False, "normal", False),
    (6, 33, 50, "log", True, "normal", False), (8, 40, 61, "reference", True, "uniform", False)])
def test_warp_specialised_equals_per_thread_kernel(D, C, T, accept, logp, prop, chol):
    """The warp-specialised fast path is bit-identical to the per-thread kernel
    (same Philox stream, same arithmetic), for every D and both accept rules."""
    eng = engine()
    rng = np.random.default_rng(7 * D + C)
    A = rng.standard_normal((D, D))
    cov = A @ A.T / D + np.eye(D)
    mean = rng.standard_normal(D)
    init = rng.standard_normal((D, C))
    L = np.linalg.cholesky(0.3 * cov) if chol else None
    kw = dict(seed=31337, accept=accept, log_pscale=logp, prop=prop, prop_scale=0.7,
              prop_chol=L, thin=3)
    s1, s2 = dev(eng, init), dev(eng, init)
    a = eng.mh_mvn(s1, mean, cov, T, variant=1, **kw)
    b = eng.mh_mvn(s2, mean, cov, T, variant=2, **kw)
    eng.sync()
    for key in ("x", "prob", "accept_count", "stat_sum", "stat_sumsq", "state_lp"):
        assert np.array_equal(host(a[key]), host(b[key])), key
    assert np.array_equal(host(s1), host(s2))


@pytest.mark.parametrize("D,C,T,logp,prop,chol,thin", [
    (2, 4096, 333, False, "normal", False, 1), (2, 4096, 1000, True, "normal", False, 1),
    (2, 100, 257, False, "normal", False, 3), (2, 33, 101, True, "uniform", False, 1),
    (3, 65, 130, True, "normal", True, 2), (1, 50, 77, False, "normal", False, 1),
    (4, 48, 95, False, "normal", False, 1), (4, 300, 64, True, "spherical", False, 5),
    (2, 5000, 129, False, "normal", False, 1), (3, 7, 40, False, "normal", False, 1)])
def test_whitened_decision_kernel_equals_per_thread_kernel(D, C, T, logp, prop, chol, thin):
    """The default native-RNG kernel (decisions taken on the incrementally tracked whitened
    state, kernel_variant 4) against the exact-arithmetic per-thread kernel: same Philox
    stream, identical decisions, and therefore bit-identical trajectories and densities
    (x is advanced by the same x + delta, the density recomputed from the recorded x).
    Covers odd walk lengths and partial batches.  On 148 SMs these chain counts give 4 or 28
    chains per CTA only; test_gpu_mh_mvn_kernels.py runs every chains-per-CTA choice against
    the oracle."""
    eng = engine()
    rng = np.random.default_rng(11 * D + C)
    A = rng.standard_normal((D, D))
    cov = A @ A.T / D + np.eye(D)
    mean = rng.standard_normal(D) if C % 2 else np.zeros(D)
    init = rng.standard_normal((D, C))
    L = np.linalg.cholesky(0.3 * cov) if chol else None
    kw = dict(seed=99173, accept="log", log_pscale=logp, prop=prop, prop_scale=0.7,
              prop_chol=L, thin=thin, prop_radius=0.9 if prop == "spherical" else 0.0)
    s1, s2 = dev(eng, init), dev(eng, init)
    a = eng.mh_mvn(s1, mean, cov, T, variant=1, **kw)
    b = eng.mh_mvn(s2, mean, cov, T, variant=4, **kw)
    eng.sync()
    for key in ("x", "prob", "accept_count", "state_lp"):
        assert np.array_equal(host(a[key]), host(b[key])), key
    assert np.array_equal(host(s1), host(s2))
    # running sums: the same terms in a different (fixed) order
    assert relerr(host(a["stat_sum"]) + 1e3, host(b["stat_sum"]) + 1e3) <= 1e-12
    assert relerr(host(a["stat_sumsq"]), host(b["stat_sumsq"])) <= 1e-12
    # resumed in two launches == one launch (y is re-derived from x at the resume point)
    s3 = dev(eng, init)
    h = (T // 2) // thin * thin
    c1 = eng.mh_mvn(s3, mean, cov, h, variant=4, **kw)
    c2 = eng.mh_mvn(s3, mean, cov, T - h, variant=4, step0=h, state_lp=c1["state_lp"], **kw)
    eng.sync()
    assert np.array_equal(np.concatenate([host(c1["x"]), host(c2["x"])])[:host(b["x"]).shape[0]],
                          host(b["x"]))


def test_whitened_decision_variant_is_refused_where_it_does_not_apply():
    eng = engine()
    st = dev(eng, np.zeros((2, 8)))
    with pytest.raises(Exception):
        eng.mh_mvn(st, [0., 0.], COV, 10, seed=1, accept="reference", variant=4)
    st5 = dev(eng, np.zeros((5, 8)))
    with pytest.raises(Exception):
        eng.mh_mvn(st5, np.zeros(5), np.eye(5), 10, seed=1, accept="log", variant=4)


def test_warp_specialised_philox_replay_general_d():
    """Fast path vs the CPU restatement fed with the CPU-generated Philox stream."""
    eng = engine()
    D, C, T, seed = 3, 70, 140, 4242
    rng = np.random.default_rng(3)
    A = rng.standard_normal((D, D))
    cov = A @ A.T / D + np.eye(D)
    mean = rng.standard_normal(D)
    init = rng.standard_normal((C, D))
    Z = philox.normals(seed, T, C, D) * 0.9
    U = philox.thresholds(seed, T, C)
    ref = o.mh_mvn_walk(init, Z, U, mean, cov, log_pscale=True, accept="log")
    out = eng.mh_mvn(dev(eng, init.T), mean, cov, T, seed=seed, accept="log",
                     log_pscale=True, prop_scale=0.9, variant=2)
    eng.sync()
    assert np.abs(host(out["x"]) - tcd_to_tdc(ref["x"])).max() <= 1e-11
    assert relerr(host(out["prob"]), ref["prob"]) <= 1e-11
    assert np.array_equal(host(out["accept_count"]), ref["u"].sum(axis=0))


def test_resume_thin_and_sharding():
    eng = engine()
    C, T, seed = 70, 120, 5
    init = np.random.default_rng(1).standard_normal((2, C))
    full = eng.mh_mvn(dev(eng, init), [0., 0.], COV, T, seed=seed)
    eng.sync()
    X = host(full["x"])
    # resume: 2 calls of T/2 with step0
    st = dev(eng, init)
    a = eng.mh_mvn(st, [0., 0.], COV, T // 2, seed=seed)
    b = eng.mh_mvn(st, [0., 0.], COV, T // 2, seed=seed, step0=T // 2,
                   state_lp=a["state_lp"])
    eng.sync()
    assert np.array_equal(np.concatenate([host(a["x"]), host(b["x"])]), X)
    # thinning keeps every 5th recorded state
    th = eng.mh_mvn(dev(eng, init), [0., 0.], COV, T, seed=seed, thin=5)
    eng.sync()
    assert np.array_equal(host(th["x"]), X[4::5])
    assert np.array_equal(host(th["prob"]), host(full["prob"])[4::5])
    # sharding: chains 32.. as a separate call with chain0=32
    lo = eng.mh_mvn(dev(eng, init[:, :32]), [0., 0.], COV, T, seed=seed)
    hi = eng.mh_mvn(dev(eng, init[:, 32:]), [0., 0.], COV, T, seed=seed, chain0=32)
    eng.sync()
    assert np.array_equal(np.concatenate([host(lo["x"]), host(hi["x"])], axis=2), X)


def test_walk_host_matches_device():
    eng = engine()
    C, T, seed = 130, 230, 9
    init = np.random.default_rng(2).standard_normal((2, C))
    d = eng.mh_mvn(dev(eng, init), [0., 0.], COV, T, seed=seed, thin=2)
    eng.sync()
    h = eng.mh_mvn_walk_host(init.copy(), [0., 0.], COV, T, seed=seed, thin=2,
                             chunk_steps=64)
    assert np.array_equal(h["x"], host(d["x"]))
    assert np.array_equal(h["prob"], host(d["prob"]))
    assert np.array_equal(h["accept_count"], host(d["accept_count"]))
    assert relerr(h["stat_sum"], host(d["stat_sum"])) <= 1e-11    # chunked partial sums


def test_philox_posterior_moments():
    """Native RNG: pooled moments of the 2-D target within Monte Carlo error and
    R-hat ~ 1 (config C2 at reduced length)."""
    eng = engine()
    C, T = 4096, 2000
    state = dev(eng, np.tile(np.array([[0.], [1.]]), (1, C)))
    burn = eng.mh_mvn(state, [0., 0.], COV, 500, seed=77, record=False)   # burn-in
    out = eng.mh_mvn(state, [0., 0.], COV, T, seed=77, step0=500, accept="log",
                     state_lp=burn["state_lp"], thin=10)
    eng.sync()
    X = host(out["x"])                              # [R, 2, C]
    flat = X.transpose(1, 0, 2).reshape(2, -1)
    assert np.abs(flat.mean(axis=1)).max() < 0.02
    assert np.abs(np.cov(flat) - COV).max() < 0.05
    acc = host(out["accept_count"]).sum() / (C * T)
    assert 0.55 < acc < 0.68                        # reference run: 0.614
    st = host(eng.chain_stats(out["stat_sum"], out["stat_sumsq"], T))
    eng.sync()
    Cn = st[:, 3]
    W = st[:, 2] / Cn
    B = T * (st[:, 1] - st[:, 0] ** 2 / Cn) / (Cn - 1)
    rhat = np.sqrt(((T - 1) / T * W + B / T) / W)
    assert np.all(np.abs(rhat - 1) < 0.02)


def test_errors_are_loud():
    from probayes_b200._lib import PbxError
    eng = engine()
    with pytest.raises(NotImplementedError):
        eng.mh_mvn(eng.zeros(9, 4), np.zeros(9), np.eye(9), 10)
    with pytest.raises(ValueError):
        eng.mh_mvn(eng.zeros(2, 4), np.zeros(2), np.eye(2), 10, thin=0)
    with pytest.raises(PbxError):          # the C ABI validates too
        eng.mh_mvn(eng.zeros(2, 4), np.zeros(2), np.eye(2), 10, step0=-1,
                   state_lp=eng.zeros(4))


def test_table_driven_math_accuracy():
    """The RNG path's -2 log / sqrt / sincos(2 pi .) / exp replacements stay within a few
    ulp of libm over the ranges the kernels feed them (uniforms, 32-bit angle words)."""
    import torch
    from probayes_b200 import _lib
    eng = engine()
    rng = np.random.default_rng(123)
    n = 1 << 20
    u = rng.random(n)
    u[:4] = [2.0 ** -53, 1.0 - 2.0 ** -53, 0.5, 2.0 ** -45]
    u[4:68] = 1.0 - (2.0 * np.arange(64) + 1.0) * 2.0 ** -53      # the 64 largest uniforms
    w = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    w[:4] = [0, 0xFFFFFFFF, 0x80000000, 0x40000000]
    ud = dev(eng, u)
    wd = torch.from_numpy(w.view(np.int32)).to(eng.device)
    out = eng.empty(5, n)
    _lib.check(eng.lib.pbx_selftest_fastmath(eng.ctx, ud.data_ptr(), wd.data_ptr(), n,
                                             out.data_ptr()))
    o5 = host(out)
    l = -2.0 * np.log(u)
    ulp = lambda got, want: np.max(np.abs(got - want) / np.spacing(np.abs(want)))
    # -2 log u: table value + polynomial, so the error is absolute (~1 ulp of 1) for u near 1
    # -- the normal variates built from it are O(1) quantities
    assert np.max(np.abs(o5[0] - l) / np.spacing(np.maximum(1.0, l))) <= 2.0
    # sqrt of the value it was given, clamped at tiny as the kernel does: for u within an
    # ulp of 1 the table log may return 0 (absolute accuracy), which must not become NaN
    assert np.all(np.isfinite(o5)) and o5[0].min() >= -2.3e-16
    assert ulp(o5[1], np.sqrt(np.maximum(o5[0], 2.2250738585072014e-308))) <= 1.0
    # extended-precision reference: in fp64 the argument 2 pi u alone carries 4e-16
    ang = 2.0 * np.longdouble("3.14159265358979323846264338327950288") * \
        ((w.astype(np.longdouble) + 0.5) / np.longdouble(2.0 ** 32))
    # absolute error (the functions are O(1); near their zeros an ulp bound is meaningless)
    assert float(np.max(np.abs(o5[2] - np.sin(ang)))) <= 4e-16
    assert float(np.max(np.abs(o5[3] - np.cos(ang)))) <= 4e-16
    assert ulp(o5[4], np.exp(-700.0 * u)) <= 2.0
