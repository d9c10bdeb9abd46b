"""Host-buffer front end of the rasterizer step: pinned host parameters in, pinned host gradients out.

The reference keeps everything on the device (ortho_gaussian_renderer/renderer.py:37 hard-codes
"cuda"), but a host integration (a CPU-side optimizer, a decoder that produces each frame's
Gaussians on the host — pipeline/stream_encode.py:42-110) feeds `render()` from host memory.  This
class is that call path and the one `bench.py` times as `e2e`:

    pipe = HostStepPipeline(P, device)
    pipe.prefetch(host_params)            # [14*P] fp32 pinned: means3D | colours | opacity | scales | rotation
    slot = pipe.step(rasterizer, dL)      # forward + backward of the oldest prefetched parameter set
    grads = pipe.grads(slot)              # [P,14] fp32 pinned (GRAD_LAYOUT), valid after this call returns

Copies run on their own streams and every buffer is ring-buffered over `slots` entries, so with one
`prefetch` issued ahead of each `step` the three engines (H2D copy, SMs, D2H copy) work on three
different steps at once and the step time is max(copy in, compute, copy out) instead of their sum.
The forward's only host wait (num_rendered, published by the tile scan) happens after the next
step's copy is already in flight.

Frame-sharded training on G GPUs (`sharded=True`, torch.distributed initialised): the Gaussians are
replicated on the devices but the HOST state is sharded by rows — rank r uploads only rows
[r·P/G, (r+1)·P/G) of each parameter segment and the devices all-gather the rest over NVLink; the
gradients are reduce-scattered and rank r reads back only its rows.  PCIe then carries 1/G of the bytes
per rank (the host link, not the GPUs, is what G replicated uploads would saturate).
Both exchanges are taken OFF THE SMs (`peer_copies=True`, the default when the ranks can map each other's memory):
the upload buffer and the gradient buffer of every slot live in symmetric memory (torch.distributed._symmetric_memory:
CUDA virtual-memory allocations every rank maps), each rank PULLS the other ranks' rows with plain device-to-device
copies — copy engines over NVLink, no CTA anywhere — between two signal-pad barriers, and sums the N row blocks it
pulled with one small kernel.  The blend kernels keep every SM full, so NCCL's all-gather / reduce-scatter kernels
(the fallback, `peer_copies=False` or when the mapping is refused) were only scheduled in the tails of the blend
grids while the peers' CTAs spun: 30-50 us exposed per step at 2-4 GPUs even on high-priority streams
(TORCH_NCCL_HIGH_PRIORITY=1, which bench.py and examples/fit_window.py still set for the fallback).
"""
from __future__ import annotations

from collections import deque
from typing import Callable, Dict, Optional

import torch

from .graphed import GraphedStep, _packed_step, _steps_fit
from .rasterizer import RasterizerError
from .sharding import GRAD_LAYOUT, GRAD_WIDTH


class HostStepPipeline:
    def __init__(self, P: int, device, slots: int = 2, use_graphs: bool = True, sharded: bool = False,
                 peer_copies: Optional[bool] = None):
        """`use_graphs`: on a slot's first step its forward + backward (8 kernels) is captured in a
        graphed.GraphedStep, whose eager warm-up sizes the binning buffer, and replayed from then on, so a step costs
        the host one graph launch instead of ~10 launches and the autograd bookkeeping; `capacity_ok()` reports
        whether the instance capacity fixed at capture time held (if not, call `recapture()`)."""
        if slots < 2:
            raise ValueError("need at least 2 slots to overlap copies with compute")
        self.P, self.slots = int(P), int(slots)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RasterizerError("HostStepPipeline needs a CUDA device: gsvc_b200 has no CPU fallback")
        f32 = dict(dtype=torch.float32, device=self.device)
        self.dev_flat = [torch.empty(GRAD_WIDTH * P, **f32) for _ in range(slots)]
        self.dev_grads = [torch.empty((P, GRAD_WIDTH), **f32) for _ in range(slots)]
        self.host_grads = [torch.empty((P, GRAD_WIDTH), dtype=torch.float32).pin_memory() for _ in range(slots)]
        # high priority: the few tiny kernels these streams launch between copies (signal-pad barriers, the sum of the
        # pulled gradient blocks) must not queue behind the 16 000-CTA blend grids of the step that is running
        self.s_h2d = torch.cuda.Stream(self.device, priority=-1)
        self.s_d2h = torch.cuda.Stream(self.device, priority=-1)
        self.in_ready = [None] * slots       # H2D of the slot finished
        self.compute_done = [None] * slots   # forward+backward that read the slot's parameters finished
        self.d2h_done = [None] * slots       # the slot's gradients are in host memory
        self.n_prefetched = 0
        self.n_stepped = 0
        self.ready = deque()
        self.use_graphs = bool(use_graphs)
        self.graphs = [None] * slots         # per slot: its GraphedStep once captured
        self.graph_keys = [None] * slots     # per slot: the (rasterizer, dL) its GraphedStep was captured with
        # host-side row sharding over the ranks of the default process group
        self.rank, self.world = 0, 1
        if sharded:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                self.rank, self.world = dist.get_rank(), dist.get_world_size()
                if P % self.world:
                    raise RasterizerError(f"sharded host state needs P ({P}) divisible by the world size ({self.world})")
        self.rows = P // self.world
        self.r0, self.r1 = self.rank * self.rows, (self.rank + 1) * self.rows
        self.peer = None
        if self.world > 1:
            self.dev_shard = [[torch.empty(self.rows * w, **f32) for _, w in GRAD_LAYOUT] for _ in range(slots)]
            self.dev_gshard = [torch.empty((self.rows, GRAD_WIDTH), **f32) for _ in range(slots)]
            # measured on one 8xB200 box (scripts/probe_hostpipe.py, 100 steps, ms per e2e step, peer / NCCL):
            #   2 GPUs 0.469 / 0.469, 4 GPUs 0.455 / 0.473, 8 GPUs 0.447 / 0.456  (compute alone: 0.449)
            # the three barriers of the peer path make its start-up and drain longer, which a 20-step window at 2 GPUs
            # sees: the default is the peer path from 4 ranks up
            if peer_copies if peer_copies is not None else self.world >= 4:
                self._setup_peer_copies(f32)
        self.h2d_bytes = GRAD_WIDTH * self.rows * 4     # per rank
        self.d2h_bytes = GRAD_WIDTH * self.rows * 4

    def _setup_peer_copies(self, f32) -> None:
        """Symmetric upload / gradient buffers + their handles; on any failure the NCCL path stays in place."""
        import torch.distributed as dist
        try:
            import torch.distributed._symmetric_memory as symm
            group = dist.group.WORLD
            P, rows, slots = self.P, self.rows, self.slots
            shard = [symm.empty(rows * GRAD_WIDTH, **f32) for _ in range(slots)]
            grads = [symm.empty(P * GRAD_WIDTH, **f32) for _ in range(slots)]
            h_shard = [symm.rendezvous(t, group) for t in shard]
            h_grads = [symm.rendezvous(t, group) for t in grads]
            self.peer = dict(shard=shard, grads=grads, h_shard=h_shard, h_grads=h_grads,
                             pulled=[torch.empty((self.world, rows, GRAD_WIDTH), **f32) for _ in range(slots)],
                             staged=[torch.empty((self.world, rows * GRAD_WIDTH), **f32) for _ in range(slots)])
            # every rank's buffers as this rank sees them (peer-mapped tensors, made once)
            self.peer["shard_of"] = [[h.get_buffer(q, (rows * GRAD_WIDTH,), torch.float32) for q in range(self.world)]
                                     for h in h_shard]
            self.peer["my_rows_of"] = [[h.get_buffer(q, (rows, GRAD_WIDTH), torch.float32, self.r0 * GRAD_WIDTH)
                                        for q in range(self.world)] for h in h_grads]
            # the backward writes its packed gradients straight into the symmetric buffer
            self.dev_grads = [g.view(P, GRAD_WIDTH) for g in grads]
            # segment offsets inside a rank's shard: [means3D rows | colours rows | opacity rows | scales rows | rotation rows]
            self.shard_off, o = [], 0
            for _, w in GRAD_LAYOUT:
                self.shard_off.append(o)
                o += rows * w
        except Exception as e:       # no peer mapping on this box / build: NCCL all-gather + reduce-scatter
            self.peer = None
            self.peer_error = f"{type(e).__name__}: {e}"

    def views(self, flat: torch.Tensor) -> Dict[str, torch.Tensor]:
        out, o, P = {}, 0, self.P
        for k, w in GRAD_LAYOUT:
            out[k] = flat[o:o + w * P].view(P, w)
            o += w * P
        return out

    def prefetch(self, host_flat: torch.Tensor) -> None:
        """Enqueue the host→device copy of one step's parameters ([14*P] fp32, pinned)."""
        if len(self.ready) >= self.slots:
            raise RasterizerError("all slots hold un-stepped parameters: call step() before prefetching more")
        if not host_flat.is_pinned():
            raise RasterizerError("host parameters must be in pinned memory (the copy has to be asynchronous)")
        b = self.n_prefetched % self.slots
        self.n_prefetched += 1
        with torch.cuda.stream(self.s_h2d):
            if self.compute_done[b] is not None:
                self.s_h2d.wait_event(self.compute_done[b])   # the step that read this slot has finished
            if self.world == 1:
                self.dev_flat[b].copy_(host_flat.view(-1), non_blocking=True)
            elif self.peer is not None:
                # this rank's rows of every segment over PCIe into ITS symmetric shard; then, between two barriers of
                # the copy stream, every rank pulls every rank's rows into place with device-to-device copies (copy
                # engines over NVLink).  The shard of a slot is rewritten two prefetches later, after the barrier of
                # the prefetch in between — which no rank passes before it has finished these pulls.
                pr, hf, off = self.peer, host_flat.view(-1), 0
                mine = pr["shard"][b]
                for i, (_, w) in enumerate(GRAD_LAYOUT):
                    mine[self.shard_off[i]:self.shard_off[i] + self.rows * w].copy_(
                        hf[off + self.r0 * w:off + self.r1 * w], non_blocking=True)
                    off += w * self.P
                h = pr["h_shard"][b]
                h.barrier(channel=0)
                # one contiguous pull per rank (copy engine), then five strided device copies put the segments in
                # place: N + 5 calls per step instead of 5 N (the host loop, not the link, is what 40 small copies per
                # step would saturate at 8 ranks)
                staged = pr["staged"][b]
                for step_ in range(self.world):
                    q = (self.rank - step_) % self.world
                    staged[q].copy_(pr["shard_of"][b][q], non_blocking=True)
                off = 0
                for i, (_, w) in enumerate(GRAD_LAYOUT):
                    n = self.rows * w
                    self.dev_flat[b][off:off + w * self.P].view(self.world, n).copy_(
                        staged[:, self.shard_off[i]:self.shard_off[i] + n], non_blocking=True)
                    off += w * self.P
            else:
                # this rank's rows of every segment over PCIe, everybody else's over NVLink
                import torch.distributed as dist
                hf, off = host_flat.view(-1), 0
                for i, (_, w) in enumerate(GRAD_LAYOUT):
                    self.dev_shard[b][i].copy_(hf[off + self.r0 * w:off + self.r1 * w], non_blocking=True)
                    off += w * self.P
                pairs, off = [], 0
                for i, (_, w) in enumerate(GRAD_LAYOUT):
                    pairs.append((self.dev_flat[b][off:off + w * self.P], self.dev_shard[b][i]))
                    off += w * self.P
                try:     # the five all-gathers as ONE NCCL group (one kernel launch)
                    from torch.distributed.distributed_c10d import _coalescing_manager
                    with _coalescing_manager(device=self.device, async_ops=False):
                        for out, inp in pairs:
                            dist.all_gather_into_tensor(out, inp)
                except ImportError:
                    for out, inp in pairs:
                        dist.all_gather_into_tensor(out, inp)
            self.in_ready[b] = self.s_h2d.record_event()
        self.ready.append(b)

    def step(self, rast, dL: torch.Tensor, reduce: Optional[Callable[[torch.Tensor], None]] = None) -> int:
        """Forward + backward of the oldest prefetched parameter set on the current stream, then the
        device→host copy of its packed gradients.  `rast`: a GaussianRasterizer (one view, dL [3,H,W]) or a
        views.ViewBatch (its views in one chain, dL [n_out,3,H,W], gradients summed over the views).
        `reduce(buf)` (frame-sharded training) is called on the [P,14] buffer after the backward; it either
        leaves the current stream ordered after its collective (returns None), or returns an asynchronous work
        handle (`dist.all_reduce(buf, async_op=True)`): then only the device→host copy waits for the collective
        and the next step's kernels run beside it."""
        if not self.ready:
            raise RasterizerError("step() without a prefetched parameter set")
        b = self.ready.popleft()
        main = torch.cuda.current_stream(self.device)
        main.wait_event(self.in_ready[b])
        if self.d2h_done[b] is not None:
            main.wait_event(self.d2h_done[b])                 # the slot's gradient buffer has been read out
        if self.use_graphs:
            key = (id(rast), dL.data_ptr(), tuple(dL.shape))
            if self.graphs[b] is None or self.graph_keys[b] != key:
                self.graphs[b] = GraphedStep(rast, self.views(self.dev_flat[b]), dL, packed=self.dev_grads[b],
                                             warmup=1)
                self.graph_keys[b] = key
            self.graphs[b]()
        else:
            _packed_step(rast, self.views(self.dev_flat[b]), dL, self.dev_grads[b])
        work = None
        if self.world > 1 and self.peer is not None:
            pass        # the gradients are exchanged on the copy-out stream below, without a collective kernel
        elif self.world > 1:
            # sum over ranks, each rank keeps (and reads back) its own rows
            import torch.distributed as dist
            work = dist.reduce_scatter_tensor(self.dev_gshard[b], self.dev_grads[b], op=dist.ReduceOp.SUM,
                                              async_op=True)
        elif reduce is not None:
            work = reduce(self.dev_grads[b])
        self.compute_done[b] = main.record_event()
        with torch.cuda.stream(self.s_d2h):
            self.s_d2h.wait_event(self.compute_done[b])
            if work is not None:
                work.wait()                                   # stream-level: the copy stream waits for the collective
            if self.world > 1 and self.peer is not None:
                # reduce-scatter without a collective kernel: barrier (every rank's backward of this step has landed in
                # its symmetric gradient buffer), pull this rank's rows of every rank's buffer with copy engines, sum
                # the N blocks with one small kernel, barrier again (nobody overwrites a buffer that is still being
                # read: the next compute on this slot waits for d2h_done, recorded after it)
                pr = self.peer
                h = pr["h_grads"][b]
                h.barrier(channel=0)
                for step_ in range(self.world):
                    q = (self.rank - step_) % self.world
                    pr["pulled"][b][q].copy_(pr["my_rows_of"][b][q], non_blocking=True)
                torch.sum(pr["pulled"][b], dim=0, out=self.dev_gshard[b])
                h.barrier(channel=1)
            src = self.dev_gshard[b] if self.world > 1 else self.dev_grads[b]
            self.host_grads[b][self.r0:self.r1].copy_(src, non_blocking=True)
            self.d2h_done[b] = self.s_d2h.record_event()
        self.n_stepped += 1
        return b

    def capacity_ok(self, rast=None) -> bool:
        """After a synchronisation: did the instance capacity of the slots' captured steps hold every replay since
        the last check?  (False: call `recapture()`; the gradients of those steps are invalid.)  `rast` is accepted
        for existing callers and not used: each slot's step knows its own capacity."""
        return _steps_fit(self.device, [g for g in self.graphs if g is not None])

    def recapture(self) -> None:
        """Drop the slots' captured steps: each slot captures a new one on its next step."""
        self.graphs = [None] * self.slots

    def grads(self, slot: int) -> torch.Tensor:
        """The [P,14] gradients of the step that returned `slot` (pinned host memory); blocks until they landed.
        With sharded host state only rows [r0, r1) of this rank are valid (summed over the ranks)."""
        ev = self.d2h_done[slot]
        if ev is None:
            raise RasterizerError(f"slot {slot} has no finished step")
        ev.synchronize()
        return self.host_grads[slot]
