"""Batch-sharded TQ inference: one process per GPU, weights replicated (term-revealed once per
rank, deterministic), each rank runs its own slice of the batch and the logits are gathered
with one NCCL all-gather over NVLink (SURVEY 8e).  Replaces the reference's
``nn.DataParallel(qmodel)`` (evaluate_cnn.py:33), which re-replicates the module on every
forward and calibrates on GPU 0's shard only; here calibration histograms are summed over
ranks before the scale-factor sweep.

PyTorch is plumbing (device memory, streams, torch.distributed); the TR kernels come from
libtq_b200.so.
"""
import torch
import torch.distributed as dist

from . import tr_layer


def bind_to_gpu_numa_node(device_index):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off (sysfs `local_cpulist` of the GPU's PCI
    function), so that pinned staging buffers are first-touched on that node and the H2D copies of the ranks do not
    cross the socket interconnect.  Returns the CPU set, or None when the topology cannot be read."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(device_index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bdf = bus.lower()[-12:]                                 # 0000:xx:yy.z
        with open(f"/sys/bus/pci/devices/{bdf}/local_cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:
        return None


IMAGENET_MEAN = (0.485, 0.456, 0.406)            # util.py:12-13
IMAGENET_STD = (0.229, 0.224, 0.225)


def normalize_u8(x_u8_nhwc, mean=IMAGENET_MEAN, std=IMAGENET_STD, out=None):
    """uint8 [N, H, W, 3] CUDA images -> bf16 [N, 3, H, W] view in channels_last memory holding
    ((u8 / 255) - mean) / std (the reference loader's ToTensor + Normalize, util.py:12-27, on the device)."""
    import ctypes
    from . import _lib
    if x_u8_nhwc.dtype != torch.uint8 or not x_u8_nhwc.is_cuda or not x_u8_nhwc.is_contiguous() or x_u8_nhwc.shape[-1] != 3:
        raise RuntimeError("normalize_u8 expects a contiguous uint8 CUDA [N, H, W, 3] tensor")
    if out is None:
        out = torch.empty(x_u8_nhwc.shape, dtype=torch.bfloat16, device=x_u8_nhwc.device)
    m = (ctypes.c_float * 3)(*mean)
    s = (ctypes.c_float * 3)(*std)
    with torch.cuda.device(x_u8_nhwc.device):
        rc = _lib.lib().tq_u8_normalize_bf16(x_u8_nhwc.data_ptr(), out.data_ptr(), x_u8_nhwc.numel() // 3,
                                             ctypes.cast(m, ctypes.c_void_p), ctypes.cast(s, ctypes.c_void_p),
                                             torch.cuda.current_stream(x_u8_nhwc.device).cuda_stream)
    _lib.check(rc)
    return out.permute(0, 3, 1, 2)


class U8Frontend(torch.nn.Module):
    """model(normalize_u8(images)): lets batches cross PCIe as uint8 (1 byte per value)."""

    def __init__(self, model, mean=IMAGENET_MEAN, std=IMAGENET_STD):
        super().__init__()
        self.model, self.mean, self.std = model, tuple(mean), tuple(std)

    def forward(self, x_u8_nhwc):
        if hasattr(self.model, "forward_u8"):       # fused engines that fold the normalisation into their first pass
            return self.model.forward_u8(x_u8_nhwc, self.mean, self.std)
        return self.model(normalize_u8(x_u8_nhwc, self.mean, self.std))


def shard_bounds(n_items, world_size, rank):
    """Contiguous [lo, hi) slice of rank `rank`; the first n % world ranks hold one extra."""
    base, extra = divmod(n_items, world_size)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def allreduce_histograms(model, group=None):
    """Sum every LinearQuantize histogram over ranks so that all ranks derive the same scale
    factors from the whole calibration set (works with gloo on CPU tensors and nccl on CUDA)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return model
    for m in model.modules():
        if isinstance(m, tr_layer.LinearQuantize):
            dist.all_reduce(m.hist_bins, op=dist.ReduceOp.SUM, group=group)
    return model


def gather_logits(logits, group=None):
    """Logits of the whole job on every rank, rank-major (the one collective of the path)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return logits
    world = dist.get_world_size(group)
    logits = logits.contiguous()
    if logits.is_cuda:
        out = torch.empty((world * logits.shape[0],) + tuple(logits.shape[1:]), dtype=logits.dtype,
                          device=logits.device)
        dist.all_gather_into_tensor(out, logits, group=group)
        return out
    parts = [torch.empty_like(logits) for _ in range(world)]
    dist.all_gather(parts, logits, group=group)
    return torch.cat(parts, dim=0)


def gather_steps(kept, group=None):
    """One all-gather for a whole run: `kept` = per-step local logits [batch, classes] -> [steps, world * batch,
    classes], rank-major within each step (the same order a per-step gather_logits gives)."""
    stacked = torch.stack(list(kept), dim=1).contiguous()      # [batch, steps, classes]
    return gather_logits(stacked, group).permute(1, 0, 2)


def calibrate(model, batches, group=None):
    """Reference protocol (evaluate_cnn.py:36-37): forward the calibration batches in tracking
    mode, then leave tracking, which runs the fused scale-factor sweep per layer."""
    tr_layer.set_tr_tracking(model, True)
    with torch.no_grad():
        for b in batches:
            model(b)
    allreduce_histograms(model, group)
    tr_layer.set_tr_tracking(model, False)
    return model


class ShardedInference:
    """Runs `model` on this rank's shard.  `forward(images_dev)` returns the logits of the
    whole job on every rank (all-gather) or just the local ones when world_size == 1.
    `stage(pinned)` + `run(slot)` add the host->device copy of the shard (double-buffered on a
    copy stream, overlapping the previous step's compute) and the device->host read of the
    gathered logits."""

    def __init__(self, model, device, group=None, cuda_graphs=False, gather="step", slots=3, d2h="local"):
        """gather: when the logits of the other ranks are collected.
        'step'  -- one all-gather per forward on the compute stream (every rank holds every step's logits before
                   the next forward starts; the ranks re-synchronise on every step);
        'async' -- the same all-gather on a side stream, off the compute stream's critical path (results of step i
                   are complete once `finish()` or the next-but-one forward has run);
        'end'   -- local logits are kept per step and ONE all-gather runs in `finish()` (the north star's "only a
                   final NCCL gather of logits")."""
        if gather not in ("step", "async", "end"):
            raise ValueError("gather must be 'step', 'async' or 'end'")
        if d2h not in ("local", "gathered"):
            raise ValueError("d2h must be 'local' or 'gathered'")
        # what `run()` reads back to the host: this rank's own logits (every rank returns its shard's results to its
        # caller; the gathered tensor stays on the device for whoever consumes all of them) or the gathered logits of
        # the whole job on EVERY rank (world x the bytes, all through the same host)
        self.d2h = d2h
        self._last_local = None
        self.gather = gather
        self._side = None
        self._gathered = [None, None]
        self._kept = []
        self._step = 0
        self.model = model.eval()
        self.cuda_graphs = bool(cuda_graphs)
        self._graphs = {}
        self.device = torch.device(device)
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.slots = max(2, int(slots))
        self._stage = [None] * self.slots
        self._stage_evt = [None] * self.slots
        self._done_evt = [None] * self.slots                    # recorded after the forward that read the slot
        self._slot = 0
        self._host_out = None

    @torch.no_grad()
    def _local_forward(self, images_dev):
        """The model on this rank's shard.  With cuda_graphs=True the forward is captured once per input
        buffer (address, shape, dtype) and replayed: ~25 kernel launches become one graph launch.  The
        returned logits are then a static buffer, overwritten by the next replay of the same graph."""
        if not self.cuda_graphs:
            return self.model(images_dev)
        key = (images_dev.data_ptr(), tuple(images_dev.shape), tuple(images_dev.stride()), images_dev.dtype)
        entry = self._graphs.get(key)
        if entry is None:
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):
                for _ in range(2):                      # allocator / lazy-init warm-up outside the capture
                    self.model(images_dev)
            torch.cuda.current_stream(self.device).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = self.model(images_dev)
            entry = self._graphs[key] = (graph, out, images_dev)    # keeps the input buffer alive
        entry[0].replay()
        return entry[1]

    @torch.no_grad()
    def forward(self, images_dev):
        local = self._local_forward(images_dev)
        self._last_local = local
        if self.world == 1 or self.gather == "step":
            return gather_logits(local, self.group)
        if self.gather == "end":
            self._kept.append(local.clone())                    # (the graph's static output is overwritten next step)
            return local
        # 'async': all-gather on a side stream into one of two rotating buffers
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.device)
        cur = torch.cuda.current_stream(self.device)
        slot = self._step & 1
        self._step += 1
        if self._gathered[slot] is None:
            self._gathered[slot] = torch.empty((self.world * local.shape[0],) + tuple(local.shape[1:]),
                                               dtype=local.dtype, device=self.device)
        snap = local.clone()
        self._side.wait_stream(cur)
        with torch.cuda.stream(self._side):
            dist.all_gather_into_tensor(self._gathered[slot], snap, group=self.group)
        snap.record_stream(self._side)
        return self._gathered[slot]

    @torch.no_grad()
    def finish(self):
        """Complete outstanding gathers.  Returns the gathered logits of what is still outstanding: of the last step
        ('async'), or of every step since the last finish(), shape [steps, world * batch, classes] ('end').  Returns
        None when nothing is outstanding: with 'step', with world size 1 (every forward already returned its logits)
        and when no step ran since the last finish()."""
        cur = torch.cuda.current_stream(self.device)
        if self.gather == "async" and self._side is not None:
            cur.wait_stream(self._side)
            return self._gathered[(self._step - 1) & 1]
        if self.gather == "end" and self.world > 1 and self._kept:
            kept, self._kept = self._kept, []
            return gather_steps(kept, self.group)
        self._kept = []
        return None

    def stage(self, pinned):
        """Start the host->device copy of a pinned shard on the copy stream; returns the slot.
        `slots` device buffers rotate: stage shards i+1 (and i+2), then run(shard i), and the copies overlap the
        compute; a slot is rewritten only after the forward that read it has been enqueued (staging more shards ahead
        than there are slots raises)."""
        s = self._slot
        if self._stage_evt[s] is not None and self._done_evt[s] is None:
            # the shard staged in this slot has not run yet: rewriting it would make that run read this shard
            raise RuntimeError(f"stage(): all {self.slots} slots hold shards that have not run; run() one first or "
                               "use more slots")
        self._slot = (s + 1) % self.slots
        if self._stage[s] is None or self._stage[s].shape != pinned.shape or \
                self._stage[s].stride() != pinned.stride():
            # same strides as the host tensor (e.g. channels_last): the copy is one plain DMA
            self._stage[s] = torch.empty_like(pinned, device=self.device)
        # the slot may still be read by the forward that last used it: wait for THAT forward only, so that the copy
        # of shard i+2 can run while forward i is still on the device
        if self._done_evt[s] is not None:
            self.copy_stream.wait_event(self._done_evt[s])
        with torch.cuda.stream(self.copy_stream):
            self._stage[s].copy_(pinned, non_blocking=True)
            evt = torch.cuda.Event()
            evt.record(self.copy_stream)
        self._stage_evt[s] = evt
        self._done_evt[s] = None
        return s

    @torch.no_grad()
    def run(self, slot):
        """Forward the staged shard and start the device->host read of the gathered logits;
        returns the pinned host tensor (valid after the current stream is synchronised)."""
        torch.cuda.current_stream(self.device).wait_event(self._stage_evt[slot])
        logits = self.forward(self._stage[slot])
        done = torch.cuda.Event()
        done.record(torch.cuda.current_stream(self.device))
        self._done_evt[slot] = done
        if self.d2h == "local":
            logits = self._last_local                            # this rank's shard; the gathered tensor stays on the device
        if self._host_out is None or self._host_out.shape != logits.shape:
            self._host_out = torch.empty(logits.shape, dtype=logits.dtype, pin_memory=True)
        if self.d2h == "gathered" and self.gather == "async" and self.world > 1:
            with torch.cuda.stream(self._side):                 # behind the gather it reads
                self._host_out.copy_(logits, non_blocking=True)
        else:
            self._host_out.copy_(logits, non_blocking=True)
        return self._host_out
