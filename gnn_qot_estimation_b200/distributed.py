"""Data parallelism over the GPUs of one box (SURVEY.md 8e) -- NEW capability, the reference
has none (no torch.distributed anywhere, SURVEY.md 2.1).

Graphs are independent units, so the path shards by graph index with nothing exchanged on the
data path:

* inference: rank r owns the contiguous graph range ``shard_range(G, r, W)``; every rank writes
  its own outputs; no collective.
* training: per-rank disjoint batches, replicated parameters (5,291 floats = 21 KB for
  TopologicalGNN), and ONE all-reduce per step over a flat fp32 gradient buffer (one gather
  kernel in, ``p.grad`` re-pointed at its slices afterwards -- no copy back).  With equal per-rank
  batch sizes and a mean-reduction loss, the averaged gradient equals the gradient of the
  concatenated batch -- checked in tests/test_distributed_cpu.py (gloo, world 2) and
  tests/test_ddp_gpu.py (nccl).

The collective itself is ``torch.distributed.all_reduce`` (NCCL over NVLink/NVSwitch on the GPU
box, gloo in the CPU tests): 21 KB is latency-bound, there is no compute to overlap it with once
the last backward kernel has run, so a custom fused kernel has nothing to win here.
"""
from __future__ import annotations

from typing import Iterable, List, Optional

import torch
import torch.distributed as dist


def shard_range(num_items: int, rank: int, world: int) -> range:
    """Contiguous, balanced shard: the first ``num_items % world`` ranks get one extra item."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    base, extra = divmod(int(num_items), int(world))
    start = rank * base + min(rank, extra)
    return range(start, start + base + (1 if rank < extra else 0))


def world_info():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


class FlatGradBuffer:
    """One flat buffer (fp32 for the product modules) for every parameter gradient -- the buffer the
    collective reduces.  Autograd writes fresh ``p.grad`` tensors (no accumulate-adds, no zero
    fill); ``all_reduce_mean`` gathers them into the flat buffer with ONE concatenation kernel,
    reduces it once, and re-points every ``p.grad`` at its slice (views, no copy back) so the
    optimizer reads the averaged values."""

    def __init__(self, params: Iterable[torch.nn.Parameter]):
        self.params: List[torch.nn.Parameter] = [p for p in params if p.requires_grad]
        if not self.params:
            raise ValueError("no trainable parameters")
        dev = self.params[0].device
        dtype = self.params[0].dtype
        if any(p.device != dev or p.dtype != dtype for p in self.params):
            raise ValueError("FlatGradBuffer needs parameters of one dtype on one device")
        self.offsets, n = [], 0
        for p in self.params:
            self.offsets.append(n)
            n += p.numel()
        self.flat = torch.zeros(n, dtype=dtype, device=dev)

    def view_of(self, i: int) -> torch.Tensor:
        p = self.params[i]
        return self.flat[self.offsets[i]: self.offsets[i] + p.numel()].view_as(p)

    def zero(self) -> None:
        """Drops the gradients (``set_to_none``): the next backward writes them afresh."""
        for p in self.params:
            p.grad = None

    def gather(self) -> None:
        """Copies the current ``p.grad`` tensors into the flat buffer (one kernel) and re-points
        them at their slices.  Parameters without a gradient contribute zeros."""
        views = [self.view_of(i) for i in range(len(self.params))]
        if all(p.grad is not None and p.grad.data_ptr() == v.data_ptr() for p, v in zip(self.params, views)):
            return                                                 # already views of the flat buffer
        pieces = [(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in self.params]
        torch.cat(pieces, out=self.flat)
        for p, v in zip(self.params, views):
            p.grad = v

    def all_reduce_mean(self, group: Optional[dist.ProcessGroup] = None) -> None:
        rank, world = world_info()
        if world == 1:
            return                                                 # nothing to exchange: leave p.grad alone
        self.gather()                                              # no-op when p.grad already alias the buffer
        dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group)
        self.flat.mul_(1.0 / world)


class GraphDataParallel(torch.nn.Module):
    """Wraps a module for graph-sharded data-parallel training.

        ddp = GraphDataParallel(model)           # broadcasts rank 0's parameters and buffers
        for data in loader_of_this_rank:
            ddp.zero_grad()
            loss = criterion(ddp(data), y); loss.backward()
            ddp.sync_gradients()                 # one flat all-reduce, averaged
            optimizer.step()
    BatchNorm statistics stay per rank (the reference has no SyncBN)."""

    def __init__(self, module: torch.nn.Module, broadcast: bool = True):
        super().__init__()
        self.module = module
        _, world = world_info()
        if broadcast and world > 1:
            with torch.no_grad():
                for t in list(module.parameters()) + list(module.buffers()):
                    dist.broadcast(t, src=0)
        self.grads = FlatGradBuffer(module.parameters())

    def forward(self, *a, **k):
        return self.module(*a, **k)

    def zero_grad(self, set_to_none: bool = True) -> None:
        self.grads.zero()

    def sync_gradients(self) -> None:
        self.grads.all_reduce_mean()


class PeerExchange:
    """Exchange buffers for the one-shot gradient all-reduce of ``qot_ddp_sgd_step``: one buffer per rank in memory
    every peer of the box has mapped (``torch.distributed._symmetric_memory``: CUDA VMM handles exchanged through the
    process group's store, peer access over NVLink), plus the DEVICE array of the peers' addresses the kernel walks.
    Raises if the ranks cannot map each other's memory (callers fall back to the NCCL all-reduce)."""

    def __init__(self, numel: int, device, group=None, local: bool = False):
        import ctypes as C
        from . import _lib
        rank, world = (0, 1) if local else world_info()     # local: this trainer is not data-parallel (see FusedSGDStep)
        self.rank, self.world = rank, world
        nbytes = int(_lib.lib().qot_ddp_exchange_bytes(int(numel)))
        if world == 1:
            self.buf, self.peers, self.handle = None, None, None
            return
        import torch.distributed._symmetric_memory as symm_mem
        group = group or dist.group.WORLD
        self.buf = symm_mem.empty(nbytes // 4, dtype=torch.float32, device=device)
        self.buf.zero_()
        self.handle = symm_mem.rendezvous(self.buf, group)
        ptrs = [int(p) for p in self.handle.buffer_ptrs]
        if len(ptrs) != world or any(p == 0 for p in ptrs):
            raise RuntimeError("symmetric memory rendezvous did not return a mapping for every rank")
        self.peers = torch.tensor(ptrs, dtype=torch.int64, device=device)
        torch.cuda.synchronize(device)
        dist.barrier(group)                             # every rank's buffer is zeroed before anyone's first step


def pack_sgd_hyper(lr: float, momentum: float, dampening: float, weight_decay: float, nesterov: bool,
                   maximize: bool):
    """``qot_sgd_hyper_t`` of one SGD parameter group.  ``one_minus_dampening`` is ``1 - dampening`` in double, rounded
    to fp32 once: the ``alpha`` torch.optim.SGD hands its foreach kernels (``1.0f - float(dampening)`` is one ulp off
    for dampening 0.6, 0.8, 0.9, 0.99 or 1/3)."""
    from . import _lib
    return _lib.QotSgdHyper(lr, momentum, dampening, weight_decay, int(nesterov), int(maximize), 1.0 - float(dampening))


class FusedSGDStep:
    """``optimizer.step()`` of a plain ``torch.optim.SGD`` (one parameter group, fp32 CUDA parameters -- what
    topological_training/train.py:66 builds) fused with the data-parallel gradient exchange into ONE launch
    (``qot_ddp_sgd_step``, csrc/ddp_step.cu).  Reads the hyper-parameters from device memory: ``sync_hyper()`` uploads
    them when a scheduler changed ``param_groups`` (a few bytes, no re-capture).  The optimizer's ``momentum_buffer``
    state entries become views of one flat buffer, so ``optimizer.state_dict()`` keeps working."""

    @staticmethod
    def supports(optimizer) -> bool:
        if type(optimizer) is not torch.optim.SGD or len(optimizer.param_groups) != 1:
            return False
        g = optimizer.param_groups[0]
        if not all(isinstance(g[k], (int, float)) for k in ("lr", "momentum", "dampening", "weight_decay")):
            return False
        ps = [p for p in g["params"] if p.requires_grad]
        return bool(ps) and all(p.is_cuda and p.dtype == torch.float32 and p.is_contiguous() for p in ps)

    def __init__(self, optimizer, grads: FlatGradBuffer, group=None, distributed: bool = True):
        """``distributed=False``: the update only, no exchange, even when a process group exists -- a model trained by
        ONE rank of a multi-rank job (no ``GraphDataParallel`` around it) must not enter a collective its peers never
        reach (the rendezvous below would wait for them forever)."""
        import ctypes as C
        from . import _lib
        self.opt, self.grads = optimizer, grads
        params = grads.params
        if [id(p) for p in optimizer.param_groups[0]["params"] if p.requires_grad] != [id(p) for p in params]:
            raise RuntimeError("FusedSGDStep: the optimizer and the flat gradient buffer must hold the same parameters in the same order")
        dev = grads.flat.device
        self.dev, self.n = dev, int(grads.flat.numel())
        self.rank, self.world = world_info() if distributed else (0, 1)
        self.exchange = PeerExchange(self.n, dev, group, local=not distributed)
        segs = (_lib.QotParamSeg * len(params))()
        for i, p in enumerate(params):
            segs[i].param, segs[i].offset, segs[i].numel = p.data_ptr(), grads.offsets[i], p.numel()
        self.segs = torch.frombuffer(bytearray(bytes(segs)), dtype=torch.uint8).to(dev)
        self.nseg = len(params)
        self.momentum = torch.zeros(self.n, dtype=torch.float32, device=dev)
        self.state = torch.zeros(2, dtype=torch.int64, device=dev)
        self.status = torch.zeros(1, dtype=torch.int32, device=dev)
        had = False
        for i, p in enumerate(params):
            view = self.momentum[grads.offsets[i]: grads.offsets[i] + p.numel()].view_as(p)
            st = optimizer.state[p]
            if torch.is_tensor(st.get("momentum_buffer")):
                view.copy_(st["momentum_buffer"])
                had = True
            st["momentum_buffer"] = view
        self.had_state = had
        if had:
            self.state[1] = 1
        self._hyper_host = torch.zeros(C.sizeof(_lib.QotSgdHyper), dtype=torch.uint8).pin_memory()
        self.hyper = torch.zeros(C.sizeof(_lib.QotSgdHyper), dtype=torch.uint8, device=dev)
        self._hyper_key = None
        self.sync_hyper()

    def mark_fresh(self) -> None:
        """The next step clones the gradient into the momentum buffer (torch's rule for a fresh optimizer)."""
        self.momentum.zero_()
        self.state[1] = 0

    def sync_hyper(self) -> None:
        g = self.opt.param_groups[0]
        key = (float(g["lr"]), float(g["momentum"]), float(g["dampening"]), float(g["weight_decay"]),
               bool(g["nesterov"]), bool(g.get("maximize", False)))
        if key == self._hyper_key:
            return
        h = pack_sgd_hyper(*key)
        self._hyper_host.copy_(torch.frombuffer(bytearray(bytes(h)), dtype=torch.uint8))
        self.hyper.copy_(self._hyper_host, non_blocking=True)
        self._hyper_key = key

    def step(self) -> None:
        """Enqueues the exchange + update on the current stream (capturable).  ``p.grad`` must be the views of the flat
        gradient buffer (``FlatGradBuffer.gather()``)."""
        from . import _lib
        _lib.check(_lib.lib().qot_ddp_sgd_step(
            self.grads.flat.data_ptr(), None if self.exchange.peers is None else self.exchange.peers.data_ptr(),
            self.world, self.rank, self.n, self.segs.data_ptr(), self.nseg, self.momentum.data_ptr(),
            self.hyper.data_ptr(), self.state.data_ptr(), self.status.data_ptr(),
            torch.cuda.current_stream(self.dev).cuda_stream), "qot_ddp_sgd_step")


def bind_to_gpu_numa_node(device_index: int) -> str:
    """Pins the calling process to the CPU cores NVML reports as local to GPU `device_index`, so that
    the pinned host buffers it allocates afterwards (first-touch) and its copy-submitting threads sit on
    the GPU's own NUMA node.  With one process per GPU this keeps every rank's host->device traffic off
    the inter-socket link.  Returns a short description; never raises (no NVML / no affinity API: no-op).
    Disabled by QOT_NO_NUMA_BIND=1."""
    import os
    if os.environ.get("QOT_NO_NUMA_BIND") or not hasattr(os, "sched_setaffinity"):
        return "numa binding off"
    try:
        import pynvml
        pynvml.nvmlInit()
        # CUDA_VISIBLE_DEVICES re-numbering: resolve through the PCI bus id of the torch device
        import torch
        bus = torch.cuda.get_device_properties(device_index).pci_bus_id if hasattr(
            torch.cuda.get_device_properties(device_index), "pci_bus_id") else None
        h = None
        if bus is not None:
            for i in range(pynvml.nvmlDeviceGetCount()):
                hi = pynvml.nvmlDeviceGetHandleByIndex(i)
                if pynvml.nvmlDeviceGetPciInfo(hi).bus == bus:
                    h = hi
                    break
        if h is None:
            h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if not cpus:
            return "numa binding: empty affinity mask, unchanged"
        os.sched_setaffinity(0, cpus)
        return f"bound to {len(cpus)} cores local to GPU {device_index}"
    except Exception as e:                                  # noqa: BLE001 -- best effort by design
        return f"numa binding unavailable ({type(e).__name__})"
