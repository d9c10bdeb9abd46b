"""Frame-sharded rendering of a TSW window across the GPUs of one box (SURVEY.md §8e).

The reference is single-GPU (utils/general_utils.py:153) but already evaluates independent views
per step (/root/reference/pipeline/train.py:353-387: front/back view of two frames); views only
couple through gradient accumulation into the shared Gaussian parameters.  So: replicate the
Gaussians, give rank r the frames {f : f mod G == r} of the window, render both views of each
locally, and sum the [P,14] parameter-gradient buffer with ONE NCCL all-reduce per step.
There is no other exchange on this path (forward-only decode needs none at all).
"""
from __future__ import annotations

import contextlib
from typing import Callable, Dict, List, Optional, Sequence

import torch
import torch.distributed as dist

# layout of the packed per-Gaussian gradient buffer: 14 fp32 per Gaussian (56 B)
GRAD_LAYOUT = (("means3D", 3), ("colors_precomp", 3), ("opacities", 1), ("scales", 3), ("rotations", 4))
GRAD_WIDTH = sum(w for _, w in GRAD_LAYOUT)


def frames_for_rank(frames: Sequence[int], rank: int, world: int) -> List[int]:
    """Round-robin frame assignment (BASELINE config 3)."""
    return [f for i, f in enumerate(frames) if i % world == rank]


def pack_grads(grads: Dict[str, torch.Tensor], out: torch.Tensor = None) -> torch.Tensor:
    P = grads["means3D"].shape[0]
    if out is None:
        out = torch.empty((P, GRAD_WIDTH), dtype=torch.float32, device=grads["means3D"].device)
    c = 0
    for name, w in GRAD_LAYOUT:
        out[:, c:c + w] = grads[name].reshape(P, w)
        c += w
    return out


@contextlib.contextmanager
def packed_backward(buf: torch.Tensor, exchange=None):
    """While active, the FIRST rasterizer backward that fits writes the GRAD_LAYOUT gradients directly into `buf`
    ([P,14] fp32, contiguous, on the rasterizer's device) and returns views of it, so the all-reduce needs no pack
    pass.  One context serves one backward: a second rasterizer backward inside it (the reference loop's four
    render() calls under one loss.backward()) returns ordinary dense gradients — batch the views of a step into one
    call (views.rasterize_views) to get all of them into the buffer.

    `exchange`: the SwitchAllReduce that owns `buf` (buf = exchange.buffer().view(P, 14)).  The batched-view backward
    then CARRIES the all-reduce: the first CTAs of its per-Gaussian kernel sum the rows over the ranks chunk by chunk
    while the others still compute (gsvc_rast_backward_views_exchange), and the buffer holds the sum over the ranks
    when the backward's kernels have run — no separate collective launch.  Every rank must run the same backward;
    `exchange.fused_launches` counts the launches that carried it (a backward that does not — a GaussianRasterizer call —
    leaves the buffer un-reduced: call exchange.run())."""
    from . import rasterizer
    t = rasterizer._packed_target
    if exchange is not None and (buf.data_ptr() != exchange.buffer().data_ptr() or buf.numel() != exchange.numel):
        raise ValueError("packed_backward(buf, exchange): buf must be the exchange's whole buffer viewed as [P,14]")
    with t.lock:
        prev = (t.buf, t.taken, t.exchange)
        t.buf, t.taken, t.exchange = buf, False, exchange
    try:
        yield buf
    finally:
        with t.lock:
            t.buf, t.taken, t.exchange = prev


def unpack_grads(buf: torch.Tensor) -> Dict[str, torch.Tensor]:
    out, c = {}, 0
    for name, w in GRAD_LAYOUT:
        out[name] = buf[:, c:c + w]
        c += w
    return out


def allreduce_grads(buf: torch.Tensor, average: bool = False) -> torch.Tensor:
    """Sum (optionally average) the packed gradient buffer over all ranks: fp32, one collective."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(buf, op=dist.ReduceOp.SUM)
        if average:
            buf /= dist.get_world_size()
    return buf


class PeerAllReduce:
    """Sum all-reduce of the step's [P,14] gradient buffer WITHOUT a collective kernel.

    The blend kernels keep every SM of every GPU full, so NCCL's all-reduce CTAs — even on a high-priority stream —
    take SMs away from the next step's forward it is meant to overlap with (measured: every stage +7-9 % at 8 GPUs,
    96.8 % scaling).  Here the buffers live in symmetric memory (torch.distributed._symmetric_memory: allocations every
    rank of the box maps); on a high-priority side stream each rank, between two signal-pad barriers, PULLS its own
    row block of every rank's buffer with device-to-device copies (copy engines over NVLink / NVSwitch), sums the N
    blocks with one small kernel, and then pulls every rank's reduced block back into its buffer.  SM work per step:
    one elementwise sum over P*14/N floats times N.

        ar = PeerAllReduce(P * 14, device, slots=2)       # raises if the ranks cannot map each other's memory
        buf = ar.buffer(slot).view(P, 14)                  # the backward writes here (packed_backward / GraphedStep)
        done = ar.start(slot)                              # after the backward, on the current stream
        ...next step's forward...
        done.wait()                                        # current stream waits; buf now holds the sum over ranks
    """

    class _Done:
        def __init__(self, event, device):
            self.event, self.device = event, device

        def wait(self):
            torch.cuda.current_stream(self.device).wait_event(self.event)

    def __init__(self, numel: int, device, slots: int = 2, group=None):
        import torch.distributed._symmetric_memory as symm
        group = dist.group.WORLD if group is None else group
        self.device = torch.device(device)
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        if numel % self.world:
            raise ValueError(f"buffer of {numel} elements does not split over {self.world} ranks")
        self.n = numel // self.world
        f32 = dict(dtype=torch.float32, device=self.device)
        self.buf = [symm.empty(numel, **f32) for _ in range(slots)]
        self.red = [symm.empty(self.n, **f32) for _ in range(slots)]
        self.h_buf = [symm.rendezvous(t, group) for t in self.buf]
        self.h_red = [symm.rendezvous(t, group) for t in self.red]
        r = self.rank
        self.my_block_of = [[h.get_buffer(q, (self.n,), torch.float32, r * self.n) for q in range(self.world)]
                            for h in self.h_buf]
        self.red_of = [[h.get_buffer(q, (self.n,), torch.float32) for q in range(self.world)] for h in self.h_red]
        self.pulled = [torch.empty((self.world, self.n), **f32) for _ in range(slots)]
        self.stream = torch.cuda.Stream(self.device, priority=-1)

    def buffer(self, slot: int) -> torch.Tensor:
        return self.buf[slot]

    def start(self, slot: int) -> "PeerAllReduce._Done":
        cur = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            hb, hr, W, r = self.h_buf[slot], self.h_red[slot], self.world, self.rank
            hb.barrier(channel=0)                                   # every rank's backward has landed
            for step in range(W):
                q = (r - step) % W
                self.pulled[slot][q].copy_(self.my_block_of[slot][q], non_blocking=True)
            torch.sum(self.pulled[slot], dim=0, out=self.red[slot])
            hr.barrier(channel=0)                                   # every block is reduced; nobody reads buf any more
            out = self.buf[slot].view(W, self.n)
            for step in range(W):
                q = (r - step) % W
                out[q].copy_(self.red_of[slot][q], non_blocking=True)
            ev = self.stream.record_event()
        return PeerAllReduce._Done(ev, self.device)


class SwitchAllReduce:
    """Sum all-reduce of the step's gradient buffer THROUGH THE NVSWITCH, one kernel of this library per rank
    (csrc/collective.cu, `gsvc_rast_switch_allreduce`): rank r load-reduces its slice of the buffer through the
    multicast mapping (the switch sums the ranks' copies) and stores the sums back through it (the switch writes
    every rank).  For an all-reduce nothing overlaps — the window of BASELINE config 3 ends with it — this is the
    fastest path on an NVSwitch box: each GPU's links carry the buffer once out and once in.  All ranks end up with
    bit-identical sums.

        ar = SwitchAllReduce(P * 14, device)          # raises if the ranks cannot map a multicast object
        buf = ar.buffer().view(P, 14)                  # the backward writes here (packed_backward / GraphedStep)
        ar.run()                                       # on the current stream, after the backward; every rank calls it
    """

    def __init__(self, numel: int, device, group=None, n_ctas: int = 0, mode: str = "auto"):
        import torch.distributed._symmetric_memory as symm
        from . import _lib
        group = dist.group.WORLD if group is None else group
        self.device = torch.device(device)
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        if numel % 4:
            raise ValueError(f"buffer of {numel} floats is not a multiple of 4 (16-byte vector accesses)")
        self._group, self._mode_req, self._lib = group, mode, _lib
        if self.world * 4 > int(symm.get_signal_pad_size()):
            raise ValueError(f"{self.world} ranks do not fit the signal pad")
        self._allocate(numel)
        # measured at 28 MB: the switch path is fastest with FEW CTAs (8 GPUs: 82 / 85 / 91 / 99 us at 16 / 32 / 64 / 128
        # CTAs — more requests in flight only contend in the fabric), the peer path needs ~64 to cover the link latency
        self.n_ctas = int(n_ctas) if n_ctas else ((16 if self.world >= 8 else 32) if self.mode == "multicast" else 64)
        # where the CTAs of a launch meet: go, done, and the chunk counters of a backward that carries the exchange
        self.state = torch.zeros(_lib.EXCHANGE_STATE_WORDS, dtype=torch.int32, device=self.device)
        self.fused_launches = 0
        self._xstruct = None

    def _allocate(self, numel: int):
        """(Re)allocate the symmetric buffer: a collective — every rank calls it with the same size.  Addresses captured
        in a CUDA graph (GraphedStep(exchange=...)) die with the old buffer: `generation` tells them apart."""
        self.generation = getattr(self, "generation", -1) + 1
        import torch.distributed._symmetric_memory as symm
        _lib, mode = self._lib, self._mode_req
        self.numel = numel
        self.t = symm.empty(numel, dtype=torch.float32, device=self.device)
        self.h = symm.rendezvous(self.t, self._group)
        mc = int(getattr(self.h, "multicast_ptr", 0) or 0)
        # two ranks: a peer load of the other copy beats sending one's own copy through the switch and back
        if mode == "auto":
            mode = "multicast" if (mc and self.world > 2) else "peer"
        if mode == "multicast" and not mc:
            raise _lib.RasterizerError("the ranks of this group have no multicast mapping (no NVSwitch / fabric): "
                                       "use mode='peer', allreduce_grads (NCCL) or PeerAllReduce")
        if mode == "peer" and self.world not in (1, 2, 4, 8):
            raise _lib.RasterizerError(f"the peer-load path is built for 1, 2, 4 or 8 ranks, got {self.world}")
        self.mode = mode
        self.mc = mc if mode == "multicast" else 0
        self.bufs = int(self.h.buffer_ptrs_dev)
        self.pads = int(self.h.signal_pad_ptrs_dev)

    def buffer(self) -> torch.Tensor:
        return self.t

    def timeouts(self, reset: bool = False) -> int:
        """Waits of this exchange that gave up (every wait is bounded at ~20 s: a rank that never arrives leaves a wrong
        buffer and a count here instead of a spinning GPU).  Synchronises the device."""
        n = int(self.state[-1].item())
        if reset and n:
            self.state[-1].zero_()
        return n

    def exchange_struct(self, n_ctas: int = 0, chunk_rows: int = 0):
        """struct gsvc_rast_exchange for gsvc_rast_backward_views_exchange (kept alive by this object)."""
        import os
        # measured (profiles/r4_notes.md): the switch path wants few movers (8 GPUs, 28 MB: 33 CTAs beat 65), the peer path
        # many (2 GPUs: 129 beat 65; it still loses to the separate launch there, so bench.py does not use it for 2 ranks)
        n_ctas = int(n_ctas) or int(os.environ.get("GSVC_EXCHANGE_CTAS", "0")) or (33 if self.mode == "multicast" else 129)
        chunk_rows = int(chunk_rows) or int(os.environ.get("GSVC_EXCHANGE_CHUNK_ROWS", "0"))
        x = self._lib.Exchange(self.mc or None, self.bufs, self.pads, self.state.data_ptr(), self.rank, self.world,
                               n_ctas, chunk_rows)
        self._xstruct = x
        return x

    def run(self, numel: Optional[int] = None):
        """Sum the buffer (or its first `numel` floats, a multiple of 4 and the same on every rank) over the ranks."""
        n = self.numel if numel is None else int(numel)
        if n % 4 or not 0 <= n <= self.numel:
            raise ValueError(f"numel {n} must be a multiple of 4 within the buffer's {self.numel} floats")
        st = torch.cuda.current_stream(self.device).cuda_stream
        self._lib.check(self._lib.lib().gsvc_rast_switch_allreduce(self.mc or None, self.bufs, self.pads, self.state.data_ptr(), self.rank,
                                                                   self.world, n, self.n_ctas, st),
                        "gsvc_rast_switch_allreduce")
        return self.t

    def sum_(self, flat: torch.Tensor) -> torch.Tensor:
        """In-place sum over the ranks of any flat fp32 tensor that fits the buffer (a copy in, the exchange, a copy out:
        for buffers whose size changes from call to call, e.g. the anchor-level loop where anchors are grown and pruned —
        a caller with a fixed size writes into buffer() directly)."""
        n = flat.numel()
        n4 = (n + 3) // 4 * 4
        if n4 > self.numel:
            # every rank sums the same number of floats, so every rank gets here in the same call
            torch.cuda.current_stream(self.device).synchronize()
            self._allocate(2 * n4)
        self.t[:n].copy_(flat.reshape(-1))
        if n4 > n:
            self.t[n:n4].zero_()
        self.run(n4)
        flat.reshape(-1).copy_(self.t[:n])
        return flat


STATS_WIDTH = 2   # per Gaussian: (sum over views of |dL/dmeans2D[:2]| where drawn, number of views it was drawn in)


def step_buffer(P: int, device):
    """ONE flat fp32 buffer per step holding the packed gradients [P,14] followed by the densification statistic
    [P,2]: `allreduce_grads(flat)` then sums both over the ranks in a single collective.
    Returns (flat [P*16], packed [P,14] view, stats [P,2] view)."""
    flat = torch.zeros((P * (GRAD_WIDTH + STATS_WIDTH),), dtype=torch.float32, device=device)
    return flat, flat[:P * GRAD_WIDTH].view(P, GRAD_WIDTH), flat[P * GRAD_WIDTH:].view(P, STATS_WIDTH)


def densify_stats(means2D_grad: torch.Tensor, radii: torch.Tensor, out: torch.Tensor = None,
                  accumulate: bool = False) -> torch.Tensor:
    """The rasterizer-side half of GaussianModel.training_statis (scene/gaussian_model.py:1298-1314) for all views
    of a step in one kernel (C-ABI gsvc_rast_densify_stats): out[g] = (sum_v |means2D_grad[v,g,:2]| over the views
    with radii[v,g] > 0, the number of such views).  `means2D_grad` [n_views,P,3] or [P,3] (means2D.grad of
    rasterize_views / GaussianRasterizer), `radii` [n_views,P] or [P] int32; `out` [P,2] fp32 (rows may be strided,
    e.g. the stats view of `step_buffer`), overwritten unless `accumulate`.  The caller adds column 0 into
    offset_gradient_accum[combined_mask] and column 1 into offset_denom[combined_mask] once per iteration instead of
    once per view (pipeline/train.py:559-565); under frame sharding the all-reduced rows are the statistic of every
    rank's views, so all ranks take the same densification decisions."""
    from . import _lib
    from .rasterizer import RasterizerError, _stream_ptr
    if not means2D_grad.is_cuda:
        raise RasterizerError("densify_stats needs CUDA tensors: gsvc_b200 has no CPU fallback")
    device = means2D_grad.device
    g = means2D_grad if means2D_grad.dim() == 3 else means2D_grad.unsqueeze(0)
    r = radii if radii.dim() == 2 else radii.unsqueeze(0)
    V, P = int(g.shape[0]), int(g.shape[1])
    if g.shape[2] != 3 or tuple(r.shape) != (V, P) or r.dtype != torch.int32 or r.device != device:
        raise RasterizerError(f"densify_stats: means2D_grad {tuple(means2D_grad.shape)} / radii {tuple(radii.shape)} "
                              f"({radii.dtype}) do not match [n_views,P,3] fp32 / [n_views,P] int32")
    g = g if (g.dtype == torch.float32 and g.is_contiguous()) else g.float().contiguous()
    r = r if r.is_contiguous() else r.contiguous()
    if out is None:
        if accumulate:
            raise RasterizerError("densify_stats: accumulate needs `out`")
        out = torch.empty((P, STATS_WIDTH), dtype=torch.float32, device=device)
    if (tuple(out.shape) != (P, STATS_WIDTH) or out.dtype != torch.float32 or out.device != device or
            (P > 0 and out.stride(1) != 1)):
        raise RasterizerError(f"densify_stats: out must be [P,2] fp32 on {device} with unit column stride")
    with torch.cuda.device(device):
        _lib.check(_lib.lib().gsvc_rast_densify_stats(V, P, g.data_ptr(), r.data_ptr(), out.data_ptr(),
                                                      int(out.stride(0)) if P > 0 else STATS_WIDTH,
                                                      1 if accumulate else 0, _stream_ptr(device)),
                   "gsvc_rast_densify_stats")
    return out


ViewFn = Callable[[int, bool], Dict[str, torch.Tensor]]


def render_window_grads(frames: Sequence[int], view_grads: ViewFn, rank: int = 0, world: int = 1,
                        both_views: bool = True) -> torch.Tensor:
    """Accumulate this rank's frames (front and back view each), then all-reduce.

    `view_grads(frame_id, back)` renders one view forward+backward and returns the parameter
    gradients keyed like GRAD_LAYOUT.  Returns the summed [P,14] buffer, identical on every rank.
    """
    total = None
    for f in frames_for_rank(frames, rank, world):
        for back in ((False, True) if both_views else (False,)):
            g = pack_grads(view_grads(f, back))
            total = g if total is None else total.add_(g)
    if total is None:
        raise ValueError("rank has no frames; give every rank at least one frame of the window")
    return allreduce_grads(total)
