"""Sharding of independent subints across GPUs (no data-path collective).

Every subint (and every archive) is fit independently (pptoas.py:247, 344), so
the batch is split into contiguous ranges, one per GPU.  Two launch styles:

* one process per GPU under ``torch.distributed`` (bench.py, large campaigns):
  :func:`shard_range` + :func:`gather_results` (a host-side gather of the small
  result arrays; the only collective, and not on the data path);
* one host thread per GPU inside a single process (:class:`MultiGPUFitter`),
  the style the Python facade uses for interactive sessions.
"""
from __future__ import annotations

import threading

import numpy as np


def gpu_local_cpus(device):
    """CPUs that share a NUMA node / PCIe root with CUDA device ``device`` (sysfs ``local_cpulist`` of
    its PCI function), or None when that cannot be read."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(device)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bus) as fh:
            text = fh.read().strip()
        cpus = set()
        for part in text.split(","):
            if not part:
                continue
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        return sorted(cpus) or None
    except Exception:  # noqa: BLE001
        return None


def bind_to_gpu_numa(device):
    """Pin the calling thread to the CPUs local to ``device`` so that page-locked buffers allocated
    afterwards (first touch) and the copies out of them stay on the GPU's own NUMA node and PCIe root.
    Returns {"cpus": n, "bound": bool}."""
    import os
    cpus = gpu_local_cpus(device)
    if not cpus:
        return {"cpus": 0, "bound": False}
    try:
        allowed = set(os.sched_getaffinity(0))
        use = sorted(allowed.intersection(cpus))
        if not use:
            return {"cpus": 0, "bound": False}
        os.sched_setaffinity(0, use)
        return {"cpus": len(use), "bound": True}
    except (AttributeError, OSError):
        return {"cpus": 0, "bound": False}


def shard_range(n, rank, world):
    """Contiguous [start, stop) of n items for ``rank`` of ``world`` (sizes
    differ by at most one; earlier ranks take the remainder)."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("bad rank/world %r/%r" % (rank, world))
    base, rem = divmod(int(n), int(world))
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def gather_results(local, group=None, dst=0):
    """Concatenate per-rank result dicts (numpy arrays, first axis = subint) on
    rank ``dst`` in rank order.  Returns the merged dict on ``dst``, None
    elsewhere.  Works with any torch.distributed backend (gloo on CPU, nccl)."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    bucket = [None] * world if rank == dst else None
    dist.gather_object(local, bucket, dst=dst, group=group)
    if rank != dst:
        return None
    return merge_results([b for b in bucket if b is not None and len(b)])


class SharedGather(object):
    """Host-side gather for the one-process-per-GPU launch on ONE node: every rank copies its packed
    per-subint results (float64 [n_local, width]) into its slot of a POSIX shared-memory segment and
    rank ``dst`` reads the slots in rank order.  No network stack and no NCCL: a few MB of memcpy per
    rank and one (gloo) barrier.  ``group`` is a torch.distributed group used for the barriers only."""

    def __init__(self, max_rows, width, group=None, dst=0, tag="g"):
        import os
        import torch.distributed as dist
        from multiprocessing import shared_memory
        self.dist, self.group, self.dst = dist, group, dst
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.max_rows, self.width = int(max_rows), int(width)
        self.slot = self.max_rows * self.width
        name = "ppb200_%s_%s_%s" % (os.environ.get("MASTER_PORT", "0"), os.getppid(), tag)
        nbytes = 8 * (self.world * (self.slot + 1))
        if self.rank == dst:
            try:                                   # a stale segment of a killed run
                old = shared_memory.SharedMemory(name=name)
                old.close()
                old.unlink()
            except FileNotFoundError:
                pass
            self.shm = shared_memory.SharedMemory(name=name, create=True, size=nbytes)
            dist.barrier(group=group)
        else:
            dist.barrier(group=group)
            self.shm = shared_memory.SharedMemory(name=name)
            try:       # only the creating rank owns the segment: keep this process's resource tracker out of it
                from multiprocessing import resource_tracker
                resource_tracker.unregister(self.shm._name, "shared_memory")
            except Exception:  # noqa: BLE001
                pass
        buf = np.ndarray((self.world, self.slot + 1), dtype=np.float64, buffer=self.shm.buf)
        self.buf = buf

    def gather(self, local):
        """local: float64 [n, width] (n <= max_rows).  Returns the rows of all ranks in rank order on
        ``dst``, None elsewhere."""
        local = np.ascontiguousarray(local, dtype=np.float64)
        n = local.shape[0]
        if n > self.max_rows or (n and local.shape[1] != self.width):
            raise ValueError("gather: got %r, slots are [%d, %d]" % (local.shape, self.max_rows, self.width))
        row = self.buf[self.rank]
        row[0] = n
        row[1:1 + n * self.width] = local.ravel()
        self.dist.barrier(group=self.group)        # every slot is written
        out = None
        if self.rank == self.dst:
            parts = []
            for r in range(self.world):
                m = int(self.buf[r, 0])
                parts.append(self.buf[r, 1:1 + m * self.width].reshape(m, self.width).copy())
            out = np.concatenate(parts, axis=0)
        self.dist.barrier(group=self.group)        # the slots may be overwritten
        return out

    def close(self):
        self.buf = None
        try:
            self.shm.close()
            self.dist.barrier(group=self.group)
            if self.rank == self.dst:
                self.shm.unlink()
        except Exception:  # noqa: BLE001
            pass


class MultiGPUFitter(object):
    """Fit one batch on several GPUs from one process: one plan, one stream and
    one host thread per device; results are concatenated on the host."""

    def __init__(self, nchan, nbin, devices):
        from .engine import WidebandPlan
        self.devices = list(devices)
        self.plans = [WidebandPlan(nchan, nbin, d) for d in self.devices]

    def set_model(self, model, freqs):
        for p in self.plans:
            p.set_model(model, freqs)

    def set_models(self, models, freqs):
        """Every plan holds every model (WidebandPlan.set_models); model_index is sliced with the subints."""
        for p in self.plans:
            p.set_models(models, freqs)

    def close(self):
        for p in self.plans:
            p.close()

    # keyword arguments of WidebandPlan.fit_batch that carry one row per subint
    PER_SUBINT = ("errs", "chan_mask", "weights", "init", "DM_guess", "snrs", "nu_fits", "nu_outs",
                  "scat_guess", "dat_scl", "dat_offs", "model_index")
    # results that are sums over the subints of a shard (the fused ppalign accumulation)
    SUMMED = ("align_sum", "align_wsum")

    def fit_batch(self, data, P, **kw):
        nsub = int(data.shape[0])
        world = len(self.plans)
        results = [None] * world
        errors = [None] * world
        P = np.broadcast_to(np.asarray(P, dtype=np.float64), (nsub,))

        def slice_kw(a, b):
            out = {}
            for k, v in kw.items():
                if k in self.PER_SUBINT and v is not None and np.ndim(v) >= 1 and np.shape(v)[0] == nsub:
                    out[k] = v[a:b]
                else:
                    out[k] = v
            return out

        def work(i):
            a, b = shard_range(nsub, i, world)
            if b <= a:
                return
            bind_to_gpu_numa(self.devices[i])      # this thread's staging and copies stay on the GPU's node
            try:
                results[i] = self.plans[i].fit_batch(data[a:b], P[a:b], **slice_kw(a, b))
            except Exception as exc:  # noqa: BLE001
                errors[i] = exc

        threads = [threading.Thread(target=work, args=(i,)) for i in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        for e in errors:
            if e is not None:
                raise e
        parts = [r for r in results if r is not None]
        return merge_results(parts, self.SUMMED)


def merge_results(parts, summed=("align_sum", "align_wsum")):
    """Merge per-shard result dicts: per-subint arrays are concatenated in shard order, the fused
    ppalign sums (one array per shard) are added."""
    out = {}
    for k in parts[0]:
        if k in summed:
            out[k] = np.sum([np.asarray(p[k]) for p in parts], axis=0)
        else:
            out[k] = np.concatenate([np.asarray(p[k]) for p in parts], axis=0)
    return out
