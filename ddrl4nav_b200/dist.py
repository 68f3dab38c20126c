"""Host-side data-parallel plumbing of the learner / predictor (SURVEY 8e).  torch.distributed only
(NCCL on the GPU box, gloo in the CPU tests); no collective is invented where the path has none:

  learner   rows of each full-batch iteration are sharded over ranks; every rank scales its local
            gradient SUMS by 1/B_global, ONE all-reduce(sum) of the flat gradient buffer (the 4 loss
            sums ride in its tail) per iteration, then the identical fused clip+Adam on every rank.
  inference env rows are independent: shard, no collective (weights are replicated by broadcast).
  GAE       env columns are independent: shard, no collective.
"""
from typing import Optional, Tuple

import torch


def world(group=None) -> Tuple[int, int]:
    """(rank, world_size); (0, 1) when torch.distributed is not initialised."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return 0, 1
    return dist.get_rank(group), dist.get_world_size(group)


def shard_rows(n_rows: int, rank: int, world_size: int) -> Tuple[int, int]:
    """Contiguous [begin, end) row range of `rank`; sizes differ by at most one row."""
    base, rem = divmod(n_rows, world_size)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def global_rows(local_rows: int, device, group=None) -> int:
    """Sum of the per-rank row counts (the 1/B_global every rank must scale by)."""
    import torch.distributed as dist
    _, ws = world(group)
    if ws == 1:
        return local_rows
    t = torch.tensor([local_rows], dtype=torch.int64, device=device)
    dist.all_reduce(t, group=group)
    return int(t.item())


def global_chunk_rows(chunk_rows, device, group=None):
    """Per minibatch k: the sum over ranks of the local chunk-k row counts (the 1/B_global of step k), all M sums from ONE
    int64 all-reduce.  Raises DDRLError on every rank together when some global chunk is empty."""
    import torch.distributed as dist
    from ._lib import DDRLError
    sums = [int(x) for x in chunk_rows]
    _, ws = world(group)
    if ws > 1:
        t = torch.tensor(sums, dtype=torch.int64, device=device)
        dist.all_reduce(t, group=group)
        sums = [int(x) for x in t.tolist()]
    if any(x < 1 for x in sums):
        raise DDRLError("minibatch plan has an empty global chunk (rows per chunk over all ranks: %s); lower MINI_BATCH_NUM"
                        % sums)
    return sums


def allreduce_grads(flat_grads_with_tail: torch.Tensor, n_params: int, group=None, tail: int = 4) -> None:
    """In-place sum over ranks of grads[0 : P+tail]: P parameters + the loss sums {actor, v, entropy, -} (tail 4), or
    {actor, v, entropy, approx KL, clip fraction} (tail 5, PPO_STATS), + the behaviour KL (tail 6, PPO_STATS with
    DECOUPLED_PPO)."""
    import torch.distributed as dist
    _, ws = world(group)
    if ws > 1:
        dist.all_reduce(flat_grads_with_tail[:n_params + tail], group=group)


def global_moments(m3: torch.Tensor, group=None) -> torch.Tensor:
    """In-place sum over ranks of the float64 advantage moments {n, sum a, sum a^2} (kernels.adv_moments): afterwards every
    rank normalises its rows with the statistics of the global minibatch (NORM_ADV)."""
    import torch.distributed as dist
    _, ws = world(group)
    if ws > 1:
        dist.all_reduce(m3, group=group)
    return m3


def global_obs_sums(sums: torch.Tensor, group=None) -> torch.Tensor:
    """In-place sum over ranks of the float64 observation moments of every normalised slot, concatenated into ONE buffer
    (kernels.obs_moments, NORM_OBS): every rank shifts by the same running mean, so the sums add, and every rank then merges
    the same global batch into its statistics.  With NORM_VALUE the two sums of critic 0's return targets follow the
    observation sums in the same buffer (nn/obs_rms.share_sums), or are the whole buffer without NORM_OBS.  One collective per
    learn call."""
    import torch.distributed as dist
    _, ws = world(group)
    if ws > 1:
        dist.all_reduce(sums, group=group)
    return sums


def broadcast_params(flat_params: torch.Tensor, src: int = 0, group=None) -> None:
    import torch.distributed as dist
    _, ws = world(group)
    if ws > 1:
        dist.broadcast(flat_params, src=src, group=group)


def max_over_ranks(value: float, device, group=None) -> float:
    """Timing convention of bench.py: a multi-GPU step takes as long as its slowest rank."""
    import torch.distributed as dist
    _, ws = world(group)
    if ws == 1:
        return value
    t = torch.tensor([value], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item())


def bind_host_to_device(device_index: int):
    """Pins the calling thread (and the threads it starts later) to the CPUs of the NUMA node the GPU hangs off, so that the
    pinned staging buffers it allocates from now on are local to the GPU's PCIe root: DMA from the far socket's memory runs at
    about half the bandwidth, which is what made the host->device legs bimodal from run to run (23 vs 46 GB/s).  Does nothing
    when the node is unknown, the allowed CPU set does not intersect it, or anything about sysfs is unexpected.  Returns
    (previous affinity, node) for the caller to restore / report, or None."""
    import os
    try:
        p = torch.cuda.get_device_properties(device_index)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as fh:
            node = int(fh.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as fh:
            cpus = set()
            for part in fh.read().strip().split(","):
                if not part:
                    continue
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        old = os.sched_getaffinity(0)
        new = old & cpus
        if not new or new == old:
            return None
        os.sched_setaffinity(0, new)
        return sorted(old), node
    except Exception:
        return None
