"""End-to-end driver over HOST buffers: a software pipeline of host->device copies, the model, and device->host copies.

The reference's callers hand the model host arrays and read host arrays back, one batch after the other
(pytorch/pytorch_utils.py:51-62: `.to(device)`, `model(...)`, `.data.cpu().numpy()` -- three serialised phases per
batch).  `HostPipeline` keeps `depth` batches in flight on three CUDA streams of the model's GPU:

    copy-in stream   batch k+1: pinned host waveform -> device staging (one cudaMemcpyAsync per micro-batch span)
    compute stream   batch k  : front-end + conv stack per span, temporal block, pooling head (chunked)
    copy-out stream  batch k-1 / k: clipwise + framewise of each finished head chunk -> pinned host buffers

so the PCIe traffic of a batch hides behind the kernels of its neighbours.  Nothing here touches the caller's
stream; results are host tensors, valid after `result()` returned.

    pipe = packed_model.host_pipeline()            # or HostPipeline(packed_model, depth=2)
    t0 = pipe.submit(wave0)                        # returns at once
    for wave in more:                              # keeps two batches in flight
        t1 = pipe.submit(wave)
        out = pipe.result(t0); consume(out); t0 = t1
    consume(pipe.result(t0))

or simply `for out in pipe.run(iterable_of_host_batches): ...`.
"""
import collections

import torch

from . import capi
from .engine import DEFAULT_MICRO_BATCH, clamp_micro_batch, plan_host_micro_batches


def plan_steady_spans(B, micro_batch, span):
    """Copy / launch spans of a batch submitted while another batch is still computing: its waveform has a whole
    batch time to arrive, so the spans are large (few launch groups = few drain / fill gaps of the persistent conv
    kernels) and uniform; multiples of 37 clips (whole waves of the 148-CTA grids), a short tail is folded in."""
    size = max(1, min(int(span), int(micro_batch)))
    spans, b0 = [], 0
    while b0 < B:
        b1 = B if B - b0 <= size + size // 2 and B - b0 <= micro_batch else b0 + size
        spans.append((b0, b1))
        b0 = b1
    return spans


class _Slot:
    """Buffers of one in-flight batch."""

    def __init__(self):
        self.key = None
        self.ticket = None       # ticket currently owning the slot (None = free)
        self.collected = True
        self.consumed = None     # event: the conv stacks of the owning batch have read the staging buffer
        self.done = None         # event: all result copies of the owning batch have landed in host memory


class HostPipeline:
    def __init__(self, pm, depth=2, micro_batch=DEFAULT_MICRO_BATCH, variant=4, head_chunk=256, steady_span=370):
        if depth < 1:
            raise ValueError("depth must be >= 1")
        self.pm = pm
        self.depth = int(depth)
        self.micro_batch = int(micro_batch)
        self.variant = variant
        self.head_chunk = int(head_chunk)
        self.steady_span = int(steady_span)
        dev = pm.device
        with torch.cuda.device(dev):
            self.copy_stream = torch.cuda.Stream(dev)
            self.compute = torch.cuda.Stream(dev)
            self.d2h_stream = torch.cuda.Stream(dev)
        self.slots = [_Slot() for _ in range(self.depth)]
        self._next = 0
        self._pending = collections.deque()  # tickets submitted and not yet collected, oldest first
        self.trace = None  # set to a list to collect (label, event) pairs (tools/e2e_ab.py)

    # ------------------------------------------------------------------ helpers
    def _mark(self, label, stream):
        if self.trace is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(stream)
            self.trace.append((label, ev))

    def _buffers(self, slot, B, L, dtype, frames, C):
        key = (B, L, dtype, frames, C)
        if slot.key != key:
            dev = self.pm.device
            slot.dev_wave = torch.empty((B, L), dtype=dtype, device=dev)
            slot.clip_dev = torch.empty((B, C), dtype=torch.float32, device=dev)
            slot.frame_dev = torch.empty((B, frames, C), dtype=torch.float32, device=dev)
            slot.clip = torch.empty((B, C), dtype=torch.float32).pin_memory()
            slot.frame = torch.empty((B, frames, C), dtype=torch.float32).pin_memory()
            slot.key = key
        return slot

    @property
    def in_flight(self):
        return len(self._pending)

    # ------------------------------------------------------------------ submit / result
    def submit(self, wave_host, result_parts=1):
        """Queue one batch: `wave_host` [B, L] float32 or int16 PCM (x = q / 32767, utils/utilities.py:78-79) CPU tensor,
        pinned for full speed.  Returns a ticket at once; the buffer must stay unmodified until `result(ticket)`."""
        pm = self.pm
        if wave_host.is_cuda or wave_host.dim() != 2 or wave_host.dtype not in (torch.float32, torch.int16):
            raise ValueError("expected a (batch_size, data_length) float32 or int16 CPU tensor")
        if len(self._pending) >= self.depth:
            raise RuntimeError("%d batches in flight: collect result(%d) before submitting another"
                               % (self.depth, self._pending[0]))
        B, L = wave_host.shape
        T = L // pm.front.hop + 1
        pm._check_frames(T)
        Tp = T // 8
        frames = pm.frames_for(Tp)
        C = pm.classes
        ticket = self._next
        self._next += 1
        slot = self.slots[ticket % self.depth]
        busy = len(self._pending) > 0
        with torch.cuda.device(pm.device), pm._lock:
            if slot.done is not None:
                slot.done.synchronize()  # the slot's previous owner was collected; its copies are long finished
            self._buffers(slot, B, L, wave_host.dtype, frames, C)
            slot.ticket, slot.collected = ticket, False
            slot.src = wave_host  # keeps a pinned source alive until its asynchronous copies have run
            cs, compute, ds = self.copy_stream, self.compute, self.d2h_stream
            pm._acquire_stream(compute)
            micro_batch = clamp_micro_batch(self.micro_batch, T)
            if busy and result_parts == 1:
                parts, plan = [(0, B)], [plan_steady_spans(B, micro_batch, self.steady_span)]
            else:
                parts, plan = plan_host_micro_batches(B, wave_host.dtype == torch.int16, micro_batch, result_parts)
            self._mark("submit %d" % ticket, compute)
            # ---- copy-in stream: the staging buffer is free once the conv stacks of its previous owner are done
            if slot.consumed is not None:
                cs.wait_event(slot.consumed)
            events = []
            with torch.cuda.stream(cs):
                for spans in plan:
                    for (b0, b1) in spans:
                        slot.dev_wave[b0:b1].copy_(wave_host[b0:b1], non_blocking=True)
                        ev = torch.cuda.Event()
                        ev.record(cs)
                        events.append(ev)
            events = iter(events)
            # ---- compute stream
            with torch.cuda.stream(compute):
                pm._workspace(max(b1 - b0 for spans in plan for b0, b1 in spans), T, need_a1=self.variant == 2)
                for (p0, p1), spans in zip(parts, plan):
                    n = p1 - p0
                    feat16, feat32, slot_kw = pm._alloc_features(n, Tp)
                    for (b0, b1) in spans:
                        compute.wait_event(next(events))
                        self._mark("conv %d:%d begin" % (b0, b1), compute)
                        pm.conv_stack(slot.dev_wave[b0:b1], variant=self.variant, **slot_kw(b0 - p0, b1 - p0))
                        self._mark("conv %d:%d end" % (b0, b1), compute)
                    if p1 == B:
                        slot.consumed = torch.cuda.Event()
                        slot.consumed.record(compute)
                    x = pm._temporal_or_features(feat16, feat32, n)
                    self._mark("temporal %d:%d end" % (p0, p1), compute)
                    out = (slot.clip_dev[p0:p1], slot.frame_dev[p0:p1])
                    # pooling head in chunks: the device->host copy of chunk i overlaps the head kernel of chunk i+1
                    blocks = x.dim() == 5 and pm.head_kind == "att"
                    if blocks:  # projections of the whole part once, then the per-clip pass chunk by chunk
                        scratch = torch.empty((capi.load().sed_attpool_blocks_scratch_bytes(n, Tp),), dtype=torch.uint8,
                                              device=pm.device)
                        pm._head_blocks(x, n, frames, False, False, out, stage=1, scratch=scratch)
                    elif x.dim() == 5:
                        from .engine import blocks_to_rows
                        x = blocks_to_rows(x, n, Tp)
                    for c0 in range(0, n, self.head_chunk):
                        c1 = min(n, c0 + self.head_chunk)
                        if blocks:
                            pm._head_blocks(x, n, frames, False, False, out, stage=2, clips=(c0, c1 - c0), scratch=scratch)
                        else:
                            pm.head(x[c0:c1], frames, want_cla=False, out=(out[0][c0:c1], out[1][c0:c1]))
                        done = torch.cuda.Event()
                        done.record(compute)
                        ds.wait_event(done)
                        with torch.cuda.stream(ds):
                            slot.clip[p0 + c0:p0 + c1].copy_(out[0][c0:c1], non_blocking=True)
                            slot.frame[p0 + c0:p0 + c1].copy_(out[1][c0:c1], non_blocking=True)
                        self._mark("head %d:%d end" % (p0 + c0, p0 + c1), compute)
                        self._mark("d2h %d:%d end" % (p0 + c0, p0 + c1), ds)
            slot.done = torch.cuda.Event()
            slot.done.record(ds)
        self._pending.append(ticket)
        return ticket

    def result(self, ticket=None, copy=False):
        """Host results of a submitted batch (oldest first when no ticket is given), blocking until its copies have
        landed: {'clipwise_output': [B, classes], 'framewise_output': [B, frames, classes]} float32 CPU tensors.
        copy=False returns views of the slot's pinned buffers, valid until `depth` further batches have been
        submitted; copy=True returns fresh tensors (what `.data.cpu()` gives the reference's callers)."""
        if not self._pending:
            raise RuntimeError("no batch in flight")
        if ticket is None:
            ticket = self._pending[0]
        if ticket != self._pending[0]:
            raise RuntimeError("results come back in submission order: next is %d, asked for %d" % (self._pending[0], ticket))
        slot = self.slots[ticket % self.depth]
        slot.done.synchronize()
        self._pending.popleft()
        slot.collected = True
        slot.src = None
        clip, frame = slot.clip, slot.frame
        if copy:
            clip, frame = clip.clone(), frame.clone()
        return {"clipwise_output": clip, "framewise_output": frame}

    def run(self, batches, copy=False):
        """Generator: results of every host batch of `batches`, in order, with up to `depth` batches in flight."""
        for wave in batches:
            if len(self._pending) >= self.depth:
                yield self.result(copy=copy)
            self.submit(wave)
        while self._pending:
            yield self.result(copy=copy)

    def drain(self):
        while self._pending:
            self.result()
