"""Multi-GPU sharding of the particle push: one process per GPU, particles split by index.

No hot-path element couples particles (``iscollective = False`` on every element,
``xline/base_classes.py:57``; beam-beam and space-charge lenses are frozen), so the path
shards into independent units: rank ``r`` owns the contiguous block
``[r*N/W, (r+1)*N/W)``, the packed lattice (<= a few MB) is replicated, and there is no
data-path collective.  ``torch.distributed`` (NCCL over NVLink on GPUs, gloo in the CPU
tests) is used only after the kernel: a SUM all-reduce of the per-element loss tallies and
a gather of BeamMonitor slabs / survivor counts, and a fold of the per-rank beam-moment sums.
"""
import torch
import torch.distributed as dist


def shard_bounds(n_total, rank, world_size):
    """Contiguous, balanced index block of ``rank``: sizes differ by at most one."""
    base, rem = divmod(int(n_total), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_columns(cols, rank, world_size):
    """Slice every per-particle column of a dict to this rank's block; ``particle_id`` is
    kept global so results do not depend on the GPU count."""
    n = len(next(iter(cols.values())))
    lo, hi = shard_bounds(n, rank, world_size)
    out = {k: v[lo:hi] for k, v in cols.items()}
    if "particle_id" not in out:
        import numpy as np

        out["particle_id"] = np.arange(lo, hi)
    return out


def _initialized():
    return dist.is_available() and dist.is_initialized()


def allreduce_loss_tally(tally):
    """SUM of ``int64[n_elements]`` loss tallies over all ranks (in place)."""
    if _initialized() and dist.get_world_size() > 1:
        dist.all_reduce(tally, op=dist.ReduceOp.SUM)
    return tally


def global_counts(p):
    """(alive, lost, particle-turns done) summed over ranks, as Python ints."""
    t = torch.stack([(p.state == 1).sum(), (p.state != 1).sum(), p.at_turn.sum()]).to(torch.int64)
    if _initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return tuple(int(v) for v in t.tolist())


def merge_monitor(data, dst=0):
    """Combine BeamMonitor slabs written by different ranks.  Every rank holds the full
    ``[num_stores, n_ids]`` slab with NaN where it owns no particle; the merged slab takes
    the (unique) non-NaN entry.  Returns the merged tensor on every rank."""
    if not (_initialized() and dist.get_world_size() > 1):
        return data
    filled = torch.nan_to_num(data, nan=0.0)
    count = (~torch.isnan(data)).to(data.dtype)
    dist.all_reduce(filled, op=dist.ReduceOp.SUM)
    dist.all_reduce(count, op=dist.ReduceOp.SUM)
    out = torch.where(count > 0, filled, torch.full_like(filled, float("nan")))
    return out


def merge_moments(m):
    """Global beam moments from the per-rank ``BeamMoments`` ``m``: all-gathers the stores of every
    rank and folds them in rank order (counts exactly, the double-double sums with the addition of
    the device reduction), so every rank holds the same bits.  Returns a new ``BeamMoments``."""
    from .moments import BeamMoments, dd_add

    out = BeamMoments(m.num_stores, m.start, m.skip, device=m.data.device)
    out.beta0gamma0 = m.beta0gamma0
    if not (_initialized() and dist.get_world_size() > 1):
        out.data.copy_(m.data)
        return out
    parts = [torch.empty_like(m.data) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, m.data.contiguous())
    acc = parts[0].clone()
    for w in parts[1:]:
        acc[:, :2] += w[:, :2]
        hi, lo = dd_add(acc[:, 2::2], acc[:, 3::2], w[:, 2::2], w[:, 3::2])
        acc[:, 2::2], acc[:, 3::2] = hi, lo
    out.data.copy_(acc)
    return out


def gather_columns(p, names=("x", "px", "y", "py", "zeta", "delta", "state", "at_element", "at_turn",
                             "particle_id")):
    """All-gather the listed particle columns (ragged shards allowed); returns a dict of
    full-length tensors ordered by rank, i.e. by global particle index."""
    if not (_initialized() and dist.get_world_size() > 1):
        return {k: (p.delta if k == "delta" else getattr(p, k)) for k in names}
    world = dist.get_world_size()
    n_local = torch.tensor([len(p)], dtype=torch.int64, device=p.x.device)
    sizes = [torch.zeros_like(n_local) for _ in range(world)]
    dist.all_gather(sizes, n_local)
    sizes = [int(s.item()) for s in sizes]
    nmax = max(sizes)
    out = {}
    for k in names:
        t = p.delta if k == "delta" else getattr(p, k)
        pad = torch.zeros(nmax, dtype=t.dtype, device=t.device)
        pad[: len(t)] = t
        parts = [torch.zeros_like(pad) for _ in range(world)]
        dist.all_gather(parts, pad)
        out[k] = torch.cat([parts[r][: sizes[r]] for r in range(world)])
    return out
