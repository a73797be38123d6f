"""Multi-GPU plumbing (one process per GPU, torch.distributed): where the hot path shards.

SURVEY.md section 8(e): batched inference shards over images with NO collective (GroupNorm statistics are per
sample); data-parallel training adds exactly one exchange step per optimisation step -- a sum all-reduce of the
flat gradient (486,409 floats = 1.95 MB for the shipped model), latency-bound over NVSwitch, so ONE bucket.
The reference has no distributed code at all (optimized_train.py:383 is single-device); the hook point is between
`loss.backward()` (:226/:210) and `clip_grad_norm_` (:230/:215).
"""
import torch
import torch.distributed as dist

from .train import _alias_grads, _zero_grads


def shard_range(n_items, rank, world):
    """Contiguous [start, stop) slice of `n_items` independent units (images / tiles) owned by `rank`.
    Sizes differ by at most one; ranks beyond n_items get an empty range."""
    if world < 1 or not 0 <= rank < world:
        raise ValueError(f"bad rank/world {rank}/{world}")
    base, rem = divmod(n_items, world)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def bind_to_gpu_numa_node(device_index):
    """Pin the calling process to the CPUs NVML reports as local to `device_index` (its NUMA node), so that the pinned host
    buffers it allocates afterwards are first-touched next to that GPU's PCIe root.  One process per GPU on a two-socket box:
    without this, half of the ranks stream their host buffers across the inter-socket link and the 8-GPU end-to-end rate with
    fp32 I/O (2 x 67 MB per 64-image batch per GPU) collapsed to 2.9x of one GPU (measured; uint8 I/O, a quarter of the bytes,
    scaled 7.9x).  Returns the CPU set, or None if NVML / affinity control is unavailable (never raises)."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        try:
            props = torch.cuda.get_device_properties(device_index)
            bus = "%08x:%02x:%02x.0" % (getattr(props, "pci_domain_id", 0), props.pci_bus_id, props.pci_device_id)
            h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:
        return None


class FlatGradBucket:
    """One flat fp32 buffer aliasing every parameter's .grad, so the data-parallel exchange is a single all-reduce.

    After `attach()`, each `p.grad` is a view into `self.flat`; autograd (and this package's fused backward) write
    gradients straight into the bucket.  `allreduce_mean()` sums over ranks and divides by the world size -- with equal
    local batches the mean of per-rank L1 means equals the global L1 mean (optimized_train.py:439, nn.L1Loss mean)."""

    def __init__(self, params):
        self.params = [p for p in params if p.requires_grad]
        if not self.params:
            raise ValueError("no trainable parameters")
        dev = self.params[0].device
        n = sum(p.numel() for p in self.params)
        self.flat = torch.zeros(n, dtype=torch.float32, device=dev)
        self.attach()

    def attach(self):
        _alias_grads(self.flat, self.params)

    def zero_(self):
        _zero_grads(self.flat, self.params)   # lets the fused backward write straight into the bucket

    def allreduce_mean(self, group=None):
        if dist.is_available() and dist.is_initialized():
            world = dist.get_world_size(group)
            if world > 1:
                dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group)
                self.flat.mul_(1.0 / world)
        return self.flat
