"""Batch sharding across the GPUs of one box (SURVEY.md 8(e)).

Static-PTQ and fp32 outputs are per-image independent, so rank ``r`` of ``R`` simply takes images
``[r*N/R, (r+1)*N/R)``; weights are replicated; there is no collective on the hot path.  The only exchange is one
all-reduce of the int64 counters at the end of a sweep (NCCL over NVLink on GPUs, gloo in the CPU tests): three
``[top1, top5, total]`` for ``sharded_accuracy`` (any model, ``topk`` counting), five for ``evaluate_sharded`` (the
static-PTQ net's counting head, tie rule of ``include/b200q.h``).  The reference has no multi-process code at all;
this mirrors what ``utils/model_evaluator.py:15-55`` computes in one process.
"""
from __future__ import annotations

import os

import torch
import torch.distributed as dist


def parse_cpulist(text: str) -> set[int]:
    """``"0-3,8,10-11"`` (sysfs ``local_cpulist`` syntax) -> ``{0,1,2,3,8,10,11}``."""
    cpus: set[int] = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def gpu_numa_info(device_index: int) -> dict:
    """NUMA node and local CPUs of a GPU as the kernel reports them (``/sys/bus/pci/devices/<bdf>/``)."""
    info = {"pci_bus_id": None, "numa_node": None, "local_cpus": None}
    try:
        prop = torch.cuda.get_device_properties(device_index)
        bdf = f"{prop.pci_domain_id:04x}:{prop.pci_bus_id:02x}:{prop.pci_device_id:02x}.0"
        info["pci_bus_id"] = bdf
        base = f"/sys/bus/pci/devices/{bdf}"
        with open(f"{base}/numa_node") as f:
            info["numa_node"] = int(f.read().strip())
        with open(f"{base}/local_cpulist") as f:
            info["local_cpus"] = sorted(parse_cpulist(f.read()))
    except (OSError, AttributeError, ValueError, RuntimeError):
        pass
    return info


def bind_to_gpu_numa(device_index: int) -> dict:
    """Pin the calling process to the CPUs that are local to ``device_index`` (when the container's CPU set contains
    any), BEFORE it allocates pinned host buffers: page placement follows the allocating thread, and a rank whose
    staging buffers sit on the other socket pays a UPI hop on every host->device copy.  One process per GPU, so this
    is per rank.  Returns what was found and what was done (bench.py reports it)."""
    info = gpu_numa_info(device_index)
    allowed = os.sched_getaffinity(0)
    info["allowed_cpus"] = len(allowed)
    info["bound_cpus"] = None
    local = set(info["local_cpus"] or ()) & allowed
    if local and local != allowed:
        os.sched_setaffinity(0, local)
        info["bound_cpus"] = len(local)
    info["local_cpus"] = len(info["local_cpus"]) if info["local_cpus"] is not None else None
    return info


def shard_range(n: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous, balanced ``[lo, hi)`` of ``n`` images for ``rank`` (first ``n % world`` ranks get one extra)."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    base, extra = divmod(n, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def topk_counts(logits: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
    """int64 ``[top1 hits, top5 hits, images]`` of one shard — the arithmetic of ``evaluate_accuracy``."""
    top5 = logits.topk(min(5, logits.shape[1]), dim=1).indices
    hit = top5.eq(labels.view(-1, 1))
    return torch.stack([hit[:, 0].sum(), hit.sum(), torch.tensor(labels.numel(), device=logits.device)]).to(torch.int64)


def rank_rule_hits(logits: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
    """bool ``[B, 4]``: (top-1 hit, top-5 hit, top-1 tied, top-5 tied) per image under the counting rule of
    ``b200q_static_evaluate`` (``include/b200q.h``), restated with torch ops on any device: hits follow the order of
    ``torch.sort(logits, 1, descending=True, stable=True)``; "tied" means some order of the classes tied with the label
    would flip the hit; a label outside ``[0, n)`` is a miss and not tied."""
    n = logits.shape[1]
    k5 = min(5, n)
    valid = (labels >= 0) & (labels < n)
    lab = torch.where(valid, labels, torch.zeros_like(labels)).view(-1, 1)
    v = logits.gather(1, lab)
    g = (logits > v).sum(1)
    same = logits == v
    e = same.sum(1) - 1
    rank = g + (same & (torch.arange(n, device=logits.device).view(1, -1) < lab)).sum(1)
    return torch.stack([valid & (rank < 1), valid & (rank < k5),
                        valid & (g < 1) & (g + e >= 1), valid & (g < k5) & (g + e >= k5)], 1)


def rank_rule_counts(logits: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
    """int64 ``[top1, top5, images, top1_tied, top5_tied]`` of ``rank_rule_hits`` (the counters' layout)."""
    h = rank_rule_hits(logits, labels).sum(0)
    return torch.stack([h[0], h[1], torch.tensor(labels.numel(), device=logits.device), h[2], h[3]]).to(torch.int64)


def allreduce_counts(counts: torch.Tensor) -> torch.Tensor:
    """Sum the per-rank counters over the default process group (no-op without one)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
    return counts


def sharded_accuracy(model, images: torch.Tensor, labels: torch.Tensor, rank: int, world: int, batch: int = 4096):
    """Evaluate this rank's shard in oracle-sized batches and return global ``(top1 %, top5 %, total)``."""
    lo, hi = shard_range(images.shape[0], rank, world)
    counts = torch.zeros(3, dtype=torch.int64, device=labels.device)
    with torch.no_grad():
        for i in range(lo, hi, batch):
            j = min(hi, i + batch)
            counts += topk_counts(model(images[i:j]), labels[i:j]).to(counts.device)
    counts = allreduce_counts(counts)
    t1, t5, n = (int(v) for v in counts.tolist())
    return 100.0 * t1 / max(n, 1), 100.0 * t5 / max(n, 1), n


def evaluate_sharded(model, images: torch.Tensor, labels: torch.Tensor, rank: int, world: int, u8: bool = False) -> dict:
    """This rank's shard through ``model.evaluate`` (``evaluate_uint8`` with ``u8``: uint8 NHWC pixels), then one
    all-reduce of the five counters over the default process group (NCCL on GPUs).  Returns the global counts as
    ``model.evaluate`` does; every rank gets the same result."""
    from .engine import eval_result
    lo, hi = shard_range(images.shape[0], rank, world)
    counts = model.eval_counters(images[lo:hi], labels[lo:hi], u8=u8)
    return eval_result(allreduce_counts(counts))
