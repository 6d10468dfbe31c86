"""torch.distributed plumbing for the stage drivers: bins are sharded across ranks (one process per GPU,
launched with torchrun); the only exchange of the path is the all-reduce of the integer expected tables and
the gather of per-rank score rows to the writing rank.  Without an initialised process group everything is
a single-rank no-op.  This replaces the reference's SLURM job fan-out (run.py:193-279)."""
import torch
import torch.distributed as dist


_solo = False


def initialised():
    return (not _solo) and dist.is_available() and dist.is_initialized()


class solo:
    """Inside this context the calling rank behaves as a single-rank job (rank 0 of 1: no all-reduce, no gather, no
    barrier), although a process group exists.  Used when whole input FILES, not row ranges, are dealt to the ranks: every
    rank then runs the unsharded stage code on its own files and the ranks only meet at the barriers between stages."""

    def __enter__(self):
        global _solo
        self.prev = _solo
        _solo = True
        return self

    def __exit__(self, *exc):
        global _solo
        _solo = self.prev
        return False


def group_rank():
    """Rank in the process group, also inside solo()."""
    return dist.get_rank() if dist.is_available() and dist.is_initialized() else 0


def group_world_size():
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def world_size():
    return dist.get_world_size() if initialised() else 1


def rank():
    return dist.get_rank() if initialised() else 0


def all_reduce_sum(t):
    """In-place sum over ranks of an integer table (order independent => bit-exact for any world size)."""
    if initialised() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def all_reduce_max(t):
    """In-place maximum over ranks of an integer tensor (order independent => bit-exact for any world size)."""
    if initialised() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t


def halo_rows(head, need):
    """The first `need` rows that follow this rank's rows (ranks own consecutive row ranges): every rank passes its first
    `need` host rows (numpy [<= need, ...]; fewer when it holds fewer) and gets the concatenation of those of the ranks
    after it, cut to `need` rows.  Collective (an all-gather of at most world x need rows); None on a single rank."""
    import numpy as np
    if not initialised() or dist.get_world_size() == 1:
        return None
    parts = [None] * dist.get_world_size()
    dist.all_gather_object(parts, np.ascontiguousarray(head[:need]))
    after = parts[dist.get_rank() + 1:]
    if not after:
        return None
    return np.concatenate(after, axis=0)[:need]


def gather_rows(t, total_rows, dst=0):
    """Concatenate per-rank row blocks (ranks own consecutive row ranges) on rank `dst`; other ranks get None."""
    if not initialised() or dist.get_world_size() == 1:
        return t
    ws = dist.get_world_size()
    sizes = [torch.zeros(1, dtype=torch.int64, device=t.device) for _ in range(ws)]
    dist.all_gather(sizes, torch.tensor([t.shape[0]], dtype=torch.int64, device=t.device))
    sizes = [int(s.item()) for s in sizes]
    assert sum(sizes) == total_rows, (sizes, total_rows)
    maxr = max(sizes)
    pad = torch.zeros((maxr,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    pad[: t.shape[0]] = t
    outs = [torch.empty_like(pad) for _ in range(ws)] if dist.get_rank() == dst else None
    dist.gather(pad, outs, dst=dst)
    if dist.get_rank() != dst:
        return None
    return torch.cat([o[:n] for o, n in zip(outs, sizes)], dim=0)


def deal_rows(full, ranges, src, pitch, pinned=False):
    """Rank `src` holds `full`, an int8 [total, pitch] numpy matrix; every rank gets its rows ranges[rank] = (lo, hi) as an
    int8 [hi - lo, pitch] numpy matrix (pinned when asked).  Point-to-point sends in rank order (NCCL: through the GPUs,
    i.e. one upload on the reader and NVLink to the peers; gloo: host tensors)."""
    import numpy as np
    me = dist.get_rank()
    lo, hi = ranges[me]
    cuda = dist.get_backend() == "nccl"

    def alloc(n):
        if pinned:
            return torch.empty((n, pitch), dtype=torch.int8, pin_memory=True)
        return torch.empty((n, pitch), dtype=torch.int8)
    mine = alloc(hi - lo)
    if me == src:
        t = torch.from_numpy(full)
        dev = t.cuda(non_blocking=True) if cuda else t
        for dst, (a, b) in enumerate(ranges):
            if dst != src and b > a:
                dist.send(dev[a:b], dst=dst)
        mine.copy_(t[lo:hi])
    elif hi > lo:
        if cuda:
            buf = torch.empty((hi - lo, pitch), dtype=torch.int8, device="cuda")
            dist.recv(buf, src=src)
            mine.copy_(buf)
        else:
            dist.recv(mine, src=src)
    out = mine.numpy()
    return out if isinstance(out, np.ndarray) else np.asarray(out)


def init_from_env():
    """Join the NCCL process group when launched by torchrun (RANK / WORLD_SIZE / LOCAL_RANK in the environment):
    one process per GPU, pinned to the GPU's NUMA node.  A plain `python` launch stays single-rank."""
    import os
    if "RANK" in os.environ and "WORLD_SIZE" in os.environ and not initialised():
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        bind_to_gpu_numa(local)
        dist.init_process_group("nccl")


def barrier():
    if initialised():
        dist.barrier()


def bind_to_gpu_numa(device_index):
    """Pin this process (one per GPU) to the CPUs that are NUMA-local to its GPU, so that the pinned host buffers it
    allocates afterwards (first touch) and its H2D / D2H copies stay on the GPU's own socket.  With several ranks streaming
    13 GB matrices over PCIe at once, remote-socket buffers cost end-to-end bandwidth.  Best effort: returns the CPU list or
    None when NVML or the affinity call is not available."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(device_index))
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:
        return None
