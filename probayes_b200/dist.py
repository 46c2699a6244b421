"""Multi-GPU partitioning of the hot path: one process per GPU, launched with
``torch.distributed`` (NCCL on the GPU box, gloo in the CPU tests).

The path shards without any data-path collective (SURVEY.md section 8e):
  * MH / Gibbs chains are independent -> contiguous chain ranges per rank, the
    Philox stream is keyed on the GLOBAL chain id so results do not depend on the
    number of ranks; only the per-chain summaries (for R-hat) are all-reduced,
    once, after the walk.
  * DGEI grids shard by mu-row slabs; the normaliser needs all-reduce(max) and
    all-reduce(sum) of two scalars, the sigma marginal an all-reduce(sum) of an
    S-vector, the mu marginal an all-gather of the slabs.
  * Ordinary-MC random samples are independent -> contiguous sample ranges per rank
    (Philox keyed on the GLOBAL sample id); posterior expectations need the same
    two-scalar normaliser plus one all-reduce of the 1 + P weighted sums.
The reference has no parallelism of any kind; all of this is new.
"""
import numpy as np


def shard_range(n, rank, world):
    """Contiguous even split of n units: returns (start, count) for ``rank``; the
    first n % world ranks get one extra unit."""
    assert 0 <= rank < world
    base, extra = divmod(int(n), int(world))
    start = rank * base + min(rank, extra)
    return start, base + (1 if rank < extra else 0)


def world():
    """(rank, world_size) of the default process group, (0, 1) when not initialised."""
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size()
    except ImportError:
        pass
    return 0, 1


def default_chain0(chains):
    """Global id of this rank's first chain when every rank runs ``chains`` chains
    through ``SP.sampler`` without an explicit ``chain0``: rank * chains (0 outside a
    process group), so that sharded public-API runs never duplicate chains."""
    return world()[0] * int(chains)


def _sharded(group=None):
    """``torch.distributed`` when ``group`` (None: the default group) has more than one
    rank, else None."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        return dist
    return None


def allreduce_chain_stats(stats, group=None):
    """stats [D, 4] = (sum_c mean, sum_c mean^2, sum_c var, C) per dimension, as
    produced by ``Engine.chain_stats`` on this rank's chains -> summed over ranks
    (in place)."""
    dist = _sharded(group)
    if dist is not None:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    return stats


def rhat_from_stats(stats, n_steps):
    """Gelman-Rubin R-hat per dimension from the (all-reduced) [D, 4] summaries:
    W = mean_c var_c;  B = T * var_c(mean_c);  R = sqrt(((T-1)/T W + B/T) / W)."""
    st = np.asarray(stats.detach().cpu().numpy() if hasattr(stats, "detach") else stats,
                    dtype=np.float64)
    T = float(n_steps)
    C = st[:, 3]
    W = st[:, 2] / C
    B = T * (st[:, 1] - st[:, 0] ** 2 / C) / (C - 1.0)
    return np.sqrt(((T - 1.0) / T * W + B / T) / W)


def pooled_moments(stats):
    """Pooled mean per dimension and the mean within-chain variance."""
    st = np.asarray(stats.detach().cpu().numpy() if hasattr(stats, "detach") else stats,
                    dtype=np.float64)
    return st[:, 0] / st[:, 3], st[:, 2] / st[:, 3]


def allreduce_max_sumexp(gmax, gsum, rescale, linear=False, group=None):
    """Normaliser of a slab-sharded log-joint: (gmax, gsum) = this slab's (max, sum exp(v -
    max)) as 1-element tensors, updated in place to the same pair over all ranks.

    All-reduce(max) of gmax; rescale(local_max, gmax, gsum) turns the local sum into the
    sum against the global maximum (``Engine.grid_rescale_sumexp_`` on the device: 0 stays
    0, else gsum * exp(local_max - gmax)); all-reduce(sum) of gsum.  ``linear`` input (plain
    sums): only gsum is reduced.  Identical on every rank; a no-op on one rank."""
    dist = _sharded(group)
    if dist is not None:
        if not linear:
            lmax = gmax.clone()
            dist.all_reduce(gmax, op=dist.ReduceOp.MAX, group=group)
            rescale(lmax, gmax, gsum)
        dist.all_reduce(gsum, op=dist.ReduceOp.SUM, group=group)
    return gmax, gsum


def gather_slabs(local, counts, group=None):
    """All-gather of per-rank 1-D slabs of (possibly) different lengths ``counts``
    into one vector (the mu marginal of a slab-sharded grid)."""
    import torch
    dist = _sharded(group)
    if dist is None:
        return local
    m = max(counts)
    pad = torch.zeros(m, dtype=local.dtype, device=local.device)
    pad[:local.numel()] = local
    parts = [torch.empty_like(pad) for _ in counts]
    dist.all_gather(parts, pad, group=group)
    return torch.cat([p[:c] for p, c in zip(parts, counts)])


def dgei_sharded(engine, x_obs, mu, sigma, logprior_mu, logprior_sigma, group=None, lik=None):
    """Slab-sharded discrete grid exact inference: every rank evaluates the
    log-joint of its mu rows, the ranks agree on the normaliser, and each returns
    dict(post=[M_local, S] slab, marg_mu=[M] (gathered), marg_sigma=[S], rows=(start,
    count)).  All inputs are full-size host arrays; ``lik`` as Engine.mh_normreg's."""
    rank, ws = world()
    M = len(mu)
    start, count = shard_range(M, rank, ws)
    sl = slice(start, start + count)
    lj = engine.grid_norm_logjoint(engine.to_device(x_obs), engine.to_device(mu[sl]),
                                   engine.to_device(sigma), engine.to_device(logprior_mu[sl]),
                                   engine.to_device(logprior_sigma), lik=lik)
    dist = _sharded(group)
    if dist is not None and group is None:
        group = dist.group.WORLD
    r = engine.grid_conditionalise(lj, want_post=True, inplace=True,
                                   group=group if dist is not None else None)
    counts = [shard_range(M, q, ws)[1] for q in range(ws)]
    mm = gather_slabs(r["marg_mu"], counts, group)
    return dict(post=r["post"], marg_mu=mm, marg_sigma=r["marg_sigma"], rows=(start, count),
                gmax=r["gmax"], gsum=r["gsum"])


def allreduce_expectation(sums, group=None):
    """sums [1 + K] = (sum p, sum p*v_1, ...) over this rank's cells (Engine.
    expectation_sums) -> expectations [K] over all ranks: all-reduce(sum), then the
    reference's safe division (probayes/pd.py:402, pscales.py:219-236)."""
    dist = _sharded(group)
    if dist is not None:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    st = np.asarray(sums.detach().cpu().numpy() if hasattr(sums, "detach") else sums,
                    dtype=np.float64)
    return st[1:] / max(2.2250738585072014e-308, st[0])


def omc_sharded(engine, y_obs, lims, open_end, log_ufun, n_samples, seed=0, x_obs=None,
                group=None, lik=None):
    """Sample-sharded ordinary Monte Carlo random sampling of a normal-likelihood
    posterior: rank r draws samples [start, start + count) of the global Philox stream,
    evaluates their log-joint, the ranks agree on the normaliser, and the posterior
    means of the parameters are all-reduced.  Returns dict(theta [P, count], logpost
    [count] (normalised over ALL ranks), expectation [P], samples=(start, count)).  ``lik``
    as Engine.mh_normreg's."""
    rank, ws = world()
    start, count = shard_range(n_samples, rank, ws)
    theta = engine.box_sample(lims, log_ufun, count, seed=seed, sample0=start)
    y = engine.to_device(np.ravel(np.asarray(y_obs, dtype=np.float64)))
    x = None if x_obs is None else engine.to_device(np.ravel(np.asarray(x_obs, np.float64)))
    logp = engine.normreg_logjoint(theta, y, x, lims, open_end, log_ufun, lik=lik)
    ms = engine.grid_max_sumexp(logp)
    gmax, gsum = allreduce_max_sumexp(ms[0:1], ms[1:2], engine.grid_rescale_sumexp_,
                                      group=group)
    # Engine.grid_conditionalise without its marginals: the per-sample "column" sums differ
    # in length from rank to rank and must not be all-reduced
    post, _, _ = engine.grid_posterior2(logp.reshape(1, -1), gmax, gsum, inplace=True,
                                        marg_log=0)
    sums = engine.expectation_sums(post.reshape(-1), True, None, theta)
    return dict(theta=theta, logpost=post.reshape(-1), samples=(start, count),
                expectation=allreduce_expectation(sums, group))
