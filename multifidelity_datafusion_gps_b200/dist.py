"""Multi-GPU plumbing (SURVEY.md section 8e): one process per GPU, torch.distributed.

Only the naturally sharded work is partitioned -- test points x MC samples and acquisition
candidates -- by contiguous ranges with no data-path collective.  NCCL is used for broadcasting the
factorised training state after a fit, gathering one (value, global index) pair per rank for the
arg-max, and (batch acquisition) broadcasting the winner's small pivot record from the rank that owns
it.  The same code runs on gloo for CPU tests.
"""
import numpy as np
import torch
import torch.distributed as tdist


def is_dist():
    return tdist.is_available() and tdist.is_initialized()


def rank_world():
    return (tdist.get_rank(), tdist.get_world_size()) if is_dist() else (0, 1)


def shard_range(n, rank, world):
    """Contiguous [lo, hi) of n items for `rank`; the first n % world ranks get one extra item."""
    base, extra = divmod(int(n), int(world))
    lo = rank * base + min(rank, extra)
    hi = lo + base + (1 if rank < extra else 0)
    return lo, hi


def combine_argmax(vals, idxs):
    """Deterministic winner of per-shard (value, global index) pairs: max value, lowest index."""
    best_v, best_i = -np.inf, np.iinfo(np.int64).max
    for v, i in zip(vals, idxs):
        if i < 0:
            continue            # empty shard
        if v > best_v or (v == best_v and i < best_i):
            best_v, best_i = float(v), int(i)
    return best_v, best_i


def coll_device(device=None):
    """Where the small collectives stage their tensors: the rank's GPU under NCCL, the host under gloo
    (gloo has no CUDA all_gather; the CPU tests and the one-GPU two-rank test run on it)."""
    if device is None or not is_dist() or tdist.get_backend() != "nccl":
        return "cpu"
    return device


def gather_argmax(local_val, local_idx, device=None):
    """all_gather of one (f64 value, i64 global index) pair per rank, then combine_argmax."""
    if not is_dist():
        return float(local_val), int(local_idx)
    dev = coll_device(device)
    v = torch.tensor([float(local_val)], dtype=torch.float64, device=dev)
    i = torch.tensor([int(local_idx)], dtype=torch.int64, device=dev)
    world = tdist.get_world_size()
    vs = [torch.empty_like(v) for _ in range(world)]
    is_ = [torch.empty_like(i) for _ in range(world)]
    tdist.all_gather(vs, v)
    tdist.all_gather(is_, i)
    return combine_argmax([t.item() for t in vs], [t.item() for t in is_])


def shard_owner(index, n, world):
    """Rank whose shard_range(n, rank, world) holds the global `index`."""
    base, extra = divmod(int(n), int(world))
    index = int(index)
    if index < extra * (base + 1):
        return index // (base + 1)
    return extra + (index - extra * (base + 1)) // base


def broadcast_record(rec, src, device=None):
    """The f64 vector `rec` of rank `src` on every rank, bit for bit (the batch acquisition's pivot record: every rank
    conditions its shard on the global winner).  Every rank passes a vector of the same length."""
    rec = np.ascontiguousarray(rec, dtype=np.float64)
    if not is_dist():
        return rec.copy()
    t = torch.from_numpy(rec.copy()).to(coll_device(device))
    tdist.broadcast(t, src=int(src))
    return t.cpu().numpy()


def restart_share(num_restarts, rank, world):
    """Restart indices rank `rank` runs: round-robin, so that run 0 (the warm start) is on rank 0."""
    return [i for i in range(int(num_restarts)) if i % int(world) == int(rank)]


def gather_runs(local_runs):
    """all_gather of per-rank lists of (run index, objective, x_opt) -> one list ordered by run index
    on every rank.  Small host objects; the object channel is enough (no data-path collective)."""
    if not is_dist():
        return sorted(local_runs, key=lambda r: r[0])
    gathered = [None] * tdist.get_world_size()
    tdist.all_gather_object(gathered, list(local_runs))
    return sorted((r for part in gathered for r in part), key=lambda r: r[0])


def best_run(runs):
    """np.argmin semantics over runs ordered by index: lowest objective, lowest run index on ties;
    NaN objectives never win unless every run is NaN."""
    best = None
    for r in sorted(runs, key=lambda r: r[0]):
        f = r[1]
        if best is None or (f < best[1]) or (best[1] != best[1] and f == f):
            best = r
    return best


def broadcast_tensors(tensors, src=0):
    if not is_dist():
        return
    for t in tensors:
        tdist.broadcast(t, src=src)


def allreduce_sum_scalar(x, device=None):
    if not is_dist():
        return float(x)
    t = torch.tensor([float(x)], dtype=torch.float64, device=coll_device(device))
    tdist.all_reduce(t, op=tdist.ReduceOp.SUM)
    return float(t.item())
