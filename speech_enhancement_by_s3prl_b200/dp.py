"""Data-parallel plumbing: one process per GPU, utterances sharded by rank, NCCL (gloo in the
CPU tests) used only to all-reduce loss / metric partial sums and head gradients
(SURVEY.md 8e).  No collective touches the audio itself -- the path has no exchange step.
"""
import os

import torch
import torch.distributed as dist


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def init_from_env(backend=None):
    """Initialise torch.distributed from RANK / WORLD_SIZE / MASTER_* (torchrun).  No-op for world size 1."""
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    if ws <= 1 or dist.is_initialized():
        return world()
    if backend is None:
        backend = "nccl" if torch.cuda.is_available() else "gloo"
    if backend == "nccl":
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    dist.init_process_group(backend=backend)
    return world()


def bind_to_gpu_numa_node(device_index):
    """Pin this process (and the pinned host buffers it allocates afterwards: first touch) to the CPUs of the NUMA node the
    GPU hangs off.  With one process per GPU on an 8-GPU box the host-to-device copies of every rank then come from local
    memory instead of crossing the inter-socket link (round 1: the e2e feed of 8 ranks reached 0.47 of linear).
    Returns the node number, or None when the topology cannot be read (nothing is changed then)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(int(device_index))).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bdf = bus.lower()[-12:]                                        # 0000:1b:00.0
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None


def shard_bounds(n_utt, rank, world_size):
    """Contiguous split of the batch dimension: rank r owns [lo, hi)."""
    base, rem = divmod(n_utt, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_batch(lengths, wavs, rank, world_size):
    lo, hi = shard_bounds(lengths.shape[0], rank, world_size)
    return lengths[lo:hi], wavs[lo:hi]


def reduce_sums(vec):
    """All-reduce (sum) a small vector of partial sums in place; returns it."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(vec, op=dist.ReduceOp.SUM)
    return vec


def global_max(t):
    """All-reduce (max) a small tensor in place; returns it.  objective.WSD thresholds voicing against the loudest frame of
    the WHOLE batch (objective.py:132-133), so every rank needs the maximum over all shards.  No-op at world size 1; under NCCL
    it may run inside CUDA-graph capture."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t


def global_means(per_utt_loss, per_utt_metric):
    """Batch means exactly as the single-process reference defines them (objective.py:100,
    runner.py:602): sum the per-utterance terms locally, all-reduce [sum_loss, sum_metric, count],
    divide by the GLOBAL utterance count."""
    vec = torch.stack([per_utt_loss.double().sum(), per_utt_metric.double().sum(),
                       torch.tensor(float(per_utt_loss.numel()), dtype=torch.float64, device=per_utt_loss.device)])
    vec = reduce_sums(vec)
    return (vec[0] / vec[2]), (vec[1] / vec[2]), int(vec[2].item())


def means_from_acc(metric_acc):
    """Global (mean loss, mean metric, utterances) from the device-side running sums [sum loss, sum metric, n] that
    ``se_finalize_metrics_acc`` keeps over an evaluation pass: ONE all-reduce of three doubles on the current stream and
    no host synchronisation -- the returned values are device tensors."""
    vec = reduce_sums(metric_acc.clone())
    return vec[0] / vec[2], vec[1] / vec[2], vec[2]


def global_l1(acc2):
    """objective.L1 under DP: all-reduce numerator AND element count before dividing (objective.py:113-116)."""
    acc2 = reduce_sums(acc2.clone())
    return acc2[0] / acc2[1]


def allreduce_gradients(parameters, world_size=None):
    """Average head gradients across ranks (one flat bucket: the head is <= a few MB, latency-bound)."""
    params = [p for p in parameters if p.grad is not None]
    if not params or not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    world_size = world_size or dist.get_world_size()
    flat = torch.cat([p.grad.reshape(-1) for p in params])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    flat /= world_size
    off = 0
    for p in params:
        n = p.grad.numel()
        p.grad.copy_(flat[off:off + n].view_as(p.grad))
        off += n
