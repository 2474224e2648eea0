"""Multi-GPU plumbing: trajectories are independent given the model (maximum_likelihood.py:383-385,
bayesian_sampling.py:288-290), so they are partitioned across ranks -- contiguous blocks balanced by frame count, one
block per GPU, resident for the whole fit -- and the only exchange per iteration is ONE sum-all-reduce of the packed
sufficient statistics (1 + N + N^2 + 3N doubles; plus the N x M B-numerator for discrete models).  The reference
has no counterpart (single process).  One process per GPU; torch.distributed (NCCL on GPUs, gloo in CPU tests) is
the transport."""
import numpy as np


def _td():
    import torch.distributed as td
    return td


def initialized():
    td = _td()
    return td.is_available() and td.is_initialized()


def rank():
    return _td().get_rank() if initialized() else 0


def world_size():
    return _td().get_world_size() if initialized() else 1


def shard_bounds(lengths, r, world):
    """Contiguous block [lo, hi) of trajectories for rank r, cut where the cumulative frame count crosses
    r/world of the total.  Deterministic, covers every trajectory exactly once; a rank may get an empty block
    when there are fewer trajectories than ranks."""
    lengths = np.asarray(lengths, dtype=np.int64)
    K = len(lengths)
    if world <= 1:
        return 0, K
    cum = np.concatenate([[0], np.cumsum(lengths)])
    total = cum[-1]
    # boundary b (1..world-1): first trajectory index whose start offset is >= b*total/world (rounded to nearest)
    cuts = [0]
    for b in range(1, world):
        target = total * b / float(world)
        k = int(np.searchsorted(cum, target, side='left'))
        if k > 0 and k <= K and (target - cum[k - 1]) < (cum[min(k, K)] - target):
            k -= 1
        cuts.append(min(max(k, cuts[-1]), K))
    cuts.append(K)
    return cuts[r], cuts[r + 1]


def tune_for_world():
    """Make certification failures rarer on multi-rank jobs: a failed hand-over costs a repair sweep on one rank and a wait in
    the all-reduce on all the others (measured at 8 GPUs: the slowest rank ran 6 extra launches in 30 iterations, about a third
    of the scaling loss), so the adaptive warm-up keeps 0.04 log2(W) more head-room above the measured need on W ranks."""
    import math
    from ._lib import lib
    w = world_size()
    lib.bhmm_b200_set_warm_margin(0.04 * math.log2(w) if w > 1 else 0.0)


def allreduce_sum(tensor):
    """In-place sum over ranks of a (device) tensor; identity when torch.distributed is not initialised."""
    if initialized() and world_size() > 1:
        _td().all_reduce(tensor, op=_td().ReduceOp.SUM)
    return tensor


def broadcast_int(value, src=0):
    """The integer `value` of rank `src` on every rank (identity without torch.distributed).  Used to agree on the seed of
    the host-side parameter draws of the Gibbs sampler: every rank must draw the SAME model from the all-reduced
    statistics, or the shards silently sample different chains."""
    if not (initialized() and world_size() > 1):
        return int(value)
    import torch
    td = _td()
    dev = 'cuda' if td.get_backend() == 'nccl' else 'cpu'
    t = torch.tensor([int(value)], dtype=torch.int64, device=dev)
    td.broadcast(t, src=src)
    return int(t.item())


def _device():
    import torch
    return torch.device('cuda', torch.cuda.current_device()) if _td().get_backend() == 'nccl' else torch.device('cpu')


def allreduce_max(tensor):
    """In-place maximum over ranks of a tensor; identity when torch.distributed is not initialised."""
    if initialized() and world_size() > 1:
        _td().all_reduce(tensor, op=_td().ReduceOp.MAX)
    return tensor


def broadcast_array(array, src=0):
    """Rank `src`'s copy of a numpy array on every rank, bit for bit (identity without torch.distributed).  Every rank passes
    an array of the same shape and dtype; only `src`'s contents matter.  The initial-model builders send the packed model
    this way, so that all ranks start from identical parameters."""
    array = np.ascontiguousarray(array)
    if not (initialized() and world_size() > 1):
        return array
    import torch
    t = torch.from_numpy(array.copy()).to(_device())
    _td().broadcast(t, src=src)
    return t.cpu().numpy()


def allgather_varlen(tensor):
    """Every rank's 1-D tensor, of any length, as a list of host arrays in rank order (the local one alone without
    torch.distributed): one all_gather of the lengths, one of the pieces padded to the longest."""
    if not (initialized() and world_size() > 1):
        return [tensor.cpu().numpy()]
    import torch
    td, dev = _td(), _device()
    n = torch.tensor([tensor.numel()], dtype=torch.int64, device=dev)
    ns = [torch.empty_like(n) for _ in range(world_size())]
    td.all_gather(ns, n)
    ns = [int(x.item()) for x in ns]
    pad = torch.zeros(max(max(ns), 1), dtype=tensor.dtype, device=dev)
    pad[:tensor.numel()] = tensor.to(dev)
    got = [torch.empty_like(pad) for _ in ns]
    td.all_gather(got, pad)
    return [g[:m].cpu().numpy() for g, m in zip(got, ns)]
