"""Multi-GPU plumbing: one process per GPU (torchrun), samples sharded by rows of X with no
data-path collective; the only exchange is at the end -- an all-gather of the per-sample lnL
(8 bytes per sample) and a global log-sum-exp (max + sum all-reduces) for the posterior
normalisation (Visualization/utils.py:157-166).  NCCL on GPUs, gloo in the CPU tests."""
import numpy as np
import torch
import torch.distributed as dist


def shard_bounds(n, rank, world):
    """Contiguous, balanced row range [lo, hi) of rank `rank`."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def gather_rows(local, n_total, rank=None, world=None):
    """All-gather contiguous shards (last dim = samples) back into the full table on every rank."""
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return local
    rank = dist.get_rank() if rank is None else rank
    world = dist.get_world_size() if world is None else world
    sizes = [shard_bounds(n_total, r, world) for r in range(world)]
    width = max(hi - lo for lo, hi in sizes)
    pad = torch.zeros(local.shape[:-1] + (width,), dtype=local.dtype, device=local.device)
    pad[..., :local.shape[-1]] = local
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad)
    return torch.cat([p[..., :hi - lo] for p, (lo, hi) in zip(parts, sizes)], dim=-1)


def global_logsumexp(local_max_sum):
    """Combine shard-local (max, sum exp(x-max)) pairs [..., 2] into log sum_i exp(x_i) over all
    ranks: all-reduce(MAX) of the maxima, rescale, all-reduce(SUM)."""
    m = local_max_sum[..., 0].clone()
    s = local_max_sum[..., 1].clone()
    if dist.is_initialized() and dist.get_world_size() > 1:
        gm = m.clone()
        dist.all_reduce(gm, op=dist.ReduceOp.MAX)
        s = s * torch.exp(m - gm)
        s = torch.where(torch.isfinite(m), s, torch.zeros_like(s))
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
        m = gm
    return m + torch.log(s)


def normalize_posterior(lnP, lse):
    """exp(lnP - logsumexp): posterior weights that sum to one over ALL ranks' samples (the
    shift-invariant result of Visualization/utils.normalize)."""
    return torch.exp(lnP - lse)


def merge_block_cyclic(P_local):
    """Sum the per-rank likelihood tables of the reference's block-cyclic layout (each rank
    leaves zeros outside its own blocks, bayes_io.py:134) into the full table."""
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return P_local
    t = P_local if isinstance(P_local, torch.Tensor) else torch.from_numpy(np.asarray(P_local))
    if dist.get_backend() == "nccl":
        t = t.cuda()
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


class TorchExchange:
    """The exchange points of a run (parallel_bayes_gpu.run) over torch.distributed, or none on a single
    rank: the default.  nccl.Communicator offers the same methods over the C ABI, without a process group."""

    def rank_world(self):
        return (dist.get_rank(), dist.get_world_size()) if dist.is_initialized() else (0, 1)

    def gather_rows(self, local, n_total):
        return gather_rows(local, n_total)

    def merge_block_cyclic(self, P_local):
        return merge_block_cyclic(P_local)

    def posterior_weights_full(self, lnP):
        """Weights of a full table [S] on the device, normalised on this rank."""
        from . import engine
        ms = engine.lse_partial(lnP)
        return normalize_posterior(lnP, ms[0] + torch.log(ms[1]))
