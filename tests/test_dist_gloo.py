"""Multi-rank host logic on CPU with the gloo backend (world_size 2 and 3): chain
sharding, summary all-reduce -> R-hat, slab-sharded grid normaliser and marginal
gathering.  The device kernels are not involved (no GPU here); the per-rank slab
arithmetic, including the rescaling of a local sum to the global maximum, is stood in for
by the numpy oracle."""
import os
import sys
import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, fn, ret):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ret[rank] = fn(rank, world)
    finally:
        dist.destroy_process_group()


def _spawn(fn, world, port):
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, port, fn, ret), nprocs=world, join=True)
    return [ret[r] for r in range(world)]


def _rhat_job(rank, world):
    from probayes_b200 import dist as pd_
    from oracle import np_oracle as o
    rng = np.random.default_rng(5)
    T, C, D = 400, 37, 3
    X = rng.standard_normal((T, C, D)).cumsum(axis=0) * 0.05 + rng.standard_normal((1, C, D))
    start, count = pd_.shard_range(C, rank, world)
    Xl = X[:, start:start + count]
    m, v = o.chain_moments(Xl)
    st = torch.tensor(np.stack([m.sum(0), (m ** 2).sum(0), v.sum(0),
                                np.full(D, float(count))], axis=1))
    st = pd_.allreduce_chain_stats(st)
    return pd_.rhat_from_stats(st, T), o.rhat(X), pd_.pooled_moments(st)[0], X.mean(axis=(0, 1))


@pytest.mark.parametrize("world,port", [(2, 29611), (3, 29613)])
def test_rhat_allreduce(world, port):
    for got, want, pm, wm in _spawn(_rhat_job, world, port):
        assert np.allclose(got, want, rtol=1e-12)
        assert np.allclose(pm, wm, rtol=1e-12)


def _rescale(lmax, gmax, gsum):
    """Engine.grid_rescale_sumexp_ (grid_rescale_sumexp_kernel) on host tensors."""
    s = float(gsum[0])
    gsum[0] = 0.0 if s == 0 else s * np.exp(float(lmax[0]) - float(gmax[0]))


def _local_max_sumexp(v):
    """This rank's (max, sum exp(v - max)) pair, as Engine.grid_max_sumexp returns it."""
    from oracle import np_oracle as o
    return torch.tensor([v.max()]), torch.tensor([o.exp_logp(v - v.max()).sum()])


def _grid_job(rank, world):
    from probayes_b200 import dist as pd_
    from oracle import np_oracle as o
    rng = np.random.default_rng(9)
    M, S = 23, 17
    lj = rng.normal(-500, 30, (M, S))
    start, count = pd_.shard_range(M, rank, world)
    slab = lj[start:start + count]
    gmax, gsum = pd_.allreduce_max_sumexp(*_local_max_sumexp(slab), _rescale)
    # linear-pscale slabs: only the plain sum is reduced
    p = np.exp(lj - lj.max())
    lin_max, lin_sum = pd_.allreduce_max_sumexp(
        torch.zeros(1), torch.tensor([p[start:start + count].sum()]), _rescale, linear=True)
    lin_ok = float(lin_max) == 0.0 and abs(float(lin_sum) - p.sum()) <= 1e-12 * p.sum()
    post = o.log_prob(o.exp_logp(slab - float(gmax)) / max(o.NEARLY_POSITIVE_ZERO, float(gsum)))
    lin = o.exp_logp(post)
    ms = torch.tensor(lin.sum(axis=0))
    dist.all_reduce(ms)
    counts = [pd_.shard_range(M, r, world)[1] for r in range(world)]
    mm = pd_.gather_slabs(torch.tensor(lin.sum(axis=1)), counts)
    whole = o.grid_conditionalise(lj)
    return (np.abs(post - whole[start:start + count]).max(),
            np.abs(o.log_prob(mm.numpy()) - o.grid_marginal(whole, 1)).max(),
            np.abs(o.log_prob(ms.numpy()) - o.grid_marginal(whole, 0)).max(),
            float(gmax) == lj.max(), lin_ok)


@pytest.mark.parametrize("world,port", [(2, 29615), (3, 29617)])
def test_slab_sharded_allreduce_max_sumexp(world, port):
    for e_post, e_mm, e_ms, max_ok, lin_ok in _spawn(_grid_job, world, port):
        assert max_ok and e_post <= 1e-9 and e_mm <= 1e-9 and e_ms <= 1e-9
        assert lin_ok


def _omc_job(rank, world):
    """Per-rank arithmetic of dist.omc_sharded stood in for by the oracle: the global
    Philox sample stream is cut into contiguous ranges, the normaliser and the weighted
    sums are all-reduced."""
    from probayes_b200 import dist as pd_
    from oracle import np_oracle as o, philox
    T, seed = 1001, 17
    lims = np.array([[40., 60.], [5., 20.]]); logu = np.array([0, 1])
    data = np.random.default_rng(3).normal(50., 10., 40)
    start, count = pd_.shard_range(T, rank, world)
    th = o.box_sample(lims, logu, philox.uniforms(seed, count, 1, 2, step0=start)[:, 0, :])
    lj = o.normreg_logjoint(th.T, None, data, lims, np.ones((2, 2), int), logu, has_slope=False)
    gmax, gsum = pd_.allreduce_max_sumexp(*_local_max_sumexp(lj), _rescale)
    lin = o.exp_logp(lj - float(gmax)) / max(o.NEARLY_POSITIVE_ZERO, float(gsum))
    sums = torch.tensor([lin.sum(), (lin * th[0]).sum(), (lin * th[1]).sum()])
    e = pd_.allreduce_expectation(sums)
    # single-process answer over the whole stream
    tha = o.box_sample(lims, logu, philox.uniforms(seed, T, 1, 2)[:, 0, :])
    lja = o.normreg_logjoint(tha.T, None, data, lims, np.ones((2, 2), int), logu, has_slope=False)
    w = o.exp_logp(lja - lja.max())
    want = np.array([(w * tha[0]).sum(), (w * tha[1]).sum()]) / w.sum()
    return e, want, np.array_equal(th, tha[:, start:start + count])


@pytest.mark.parametrize("world,port", [(2, 29619), (3, 29621)])
def test_sample_sharded_omc_expectation_allreduce_max_sumexp(world, port):
    for e, want, same_stream in _spawn(_omc_job, world, port):
        assert same_stream                       # results do not depend on the rank count
        assert np.allclose(e, want, rtol=1e-12)


def _chain0_job(rank, world):
    from probayes_b200 import dist as pd_
    return pd_.default_chain0(4096)


def test_default_chain0_is_rank_times_chains():
    """SP.sampler's default chain offset under a process group (ADVICE r1: all ranks
    used to draw the same chains)."""
    from probayes_b200 import dist as pd_
    assert pd_.default_chain0(4096) == 0                    # no process group
    assert _spawn(_chain0_job, 2, 29617) == [0, 4096]


def test_shard_range_covers_everything():
    from probayes_b200.dist import shard_range
    for n in (1, 7, 4096, 16384, 65537):
        for world in (1, 2, 3, 4, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and sum(c for _, c in spans) == n
            for (s0, c0), (s1, _) in zip(spans, spans[1:]):
                assert s0 + c0 == s1
            assert max(c for _, c in spans) - min(c for _, c in spans) <= 1
