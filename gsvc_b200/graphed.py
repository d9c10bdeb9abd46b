"""CUDA-graph replay of a rasterizer step on static tensors.

The eager call has one unavoidable host wait per forward — `num_rendered` must come back as a Python
int (ortho_gaussian_renderer/renderer.py:90) — so the host can never run more than one step ahead of
the device, and with the blend kernels at ~0.1 ms the Python/autograd launch path between "count
published" and "backward enqueued" shows up as idle SM time.  A training loop whose tensors keep
their addresses (parameters updated in place by the optimizer, a fixed seed-gradient / loss buffer)
can instead capture forward + backward once and replay it: one graph launch per step, no host wait,
the 8 kernels back to back with their programmatic-dependent-launch edges preserved.

    step = GraphedStep(rasterizer, params, dL)        # params: dict of static CUDA tensors (GRAD_LAYOUT keys)
    color, radii, grads = step()                       # replay; outputs are static tensors, overwritten each call
    ...
    if not step.capacity_ok(): step.recapture()        # after a synchronisation, e.g. once per N steps

The step can also own its loss: with a static target tensor the captured graph renders, evaluates the fused
L1 + D-SSIM loss (gsvc_b200.loss) against it and back-propagates, so the whole step is one graph launch:

    step = GraphedStep(batch, params, None, loss_target=target, lambda_dssim=0.2)   # target [n_out,3,H,W]
    target.copy_(frames)                                # this iteration's target frames, in place
    color, radii, grads = step()                        # step.loss: the per-image losses of this replay

or against the video's 8-bit frames kept resident on the device (SPEC U12), picked per replay by a static index:

    idx = torch.zeros(n_out, dtype=torch.int32, device="cuda")
    step = GraphedStep(batch, params, None, loss_target=cube, loss_index=idx)     # cube [F,H,W,3] uint8
    idx.copy_(pair, non_blocking=True)                  # this iteration's frame numbers, 4 bytes per image, in place
    color, radii, grads = step()

The binning capacity is fixed at capture time from an eager warm-up (+50 % + 64 Ki instances) and recorded on the
step's own count slot; `capacity_ok()` compares it with the instance count the device published there for the last
replay.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import rasterizer as R
from .loss import _check_lambda, photometric_loss
from . import export as E
from . import quality as Q
from .rasterizer import RasterizerError
from .sharding import GRAD_LAYOUT, GRAD_WIDTH, packed_backward
from .views import ViewBatch, render_params


def _packed_step(rast, params, dL, packed, exchange=None, loss_target=None, lambda_dssim=0.2, loss_index=None):
    """Forward + backward of `rast` on the GRAD_LAYOUT dict `params`, the gradients written into `packed`
    (sharding.packed_backward); the backward is seeded with `dL`, or with the mean of photometric_loss(image,
    loss_target, index=loss_index) when a target is given.  Returns (color, radii, num_rendered, per-image loss or
    None)."""
    leaves = {k: params[k].detach().requires_grad_(True) for k, _ in GRAD_LAYOUT}
    color, radii, n = render_params(rast, leaves)
    loss = None if loss_target is None else photometric_loss(color, loss_target, lambda_dssim, index=loss_index)
    with packed_backward(packed, exchange=exchange):
        torch.autograd.grad(color if loss is None else loss.mean(), [leaves[k] for k, _ in GRAD_LAYOUT],
                            grad_outputs=dL)
    return color, radii, n, loss


def _check_rgb8_loss_target(target, index, device):
    """A uint8 loss target of a captured step: nothing that photometric_loss would convert (a copy baked into the
    graph would not see the caller's in-place writes).  Shapes are checked against the image by the warm-up."""
    if not target.is_contiguous():
        raise RasterizerError("a uint8 loss_target must be contiguous (the graph reads it in place)")
    if index is not None:
        if target.dim() != 4:
            raise RasterizerError(f"with loss_index, loss_target must be a [F,H,W,3] cube, got {tuple(target.shape)}")
        if (not isinstance(index, torch.Tensor) or index.device != device or index.dtype != torch.int32
                or index.dim() != 1 or not index.is_contiguous()):
            raise RasterizerError(f"loss_index must be a contiguous int32 [n_out] tensor on {device} (the graph reads "
                                  "it in place)")


def _steps_fit(device, steps) -> bool:
    """After a synchronisation: no rasterizer launch on `device` ran out of instance capacity since the last check
    (the sticky device counter, reset here once), and the last replay of every one of `steps` fits its slot."""
    if R.overflow_events(device) > 0:
        return False
    return all(step.slot.fits() for step in steps)


class GraphedStep:
    def __init__(self, rast, params: Dict[str, torch.Tensor], dL: Optional[torch.Tensor],
                 packed: Optional[torch.Tensor] = None, warmup: int = 2, exchange=None,
                 loss_target: Optional[torch.Tensor] = None, lambda_dssim: float = 0.2,
                 loss_index: Optional[torch.Tensor] = None):
        """`rast`: a GaussianRasterizer (one view, dL [3,H,W]) or a views.ViewBatch (all its views in one chain,
        dL [n_out,3,H,W], gradients summed over the views).  `dL` None: forward only.  `packed`: optional [P,14]
        buffer the backward writes (sharding.GRAD_LAYOUT); allocated here if omitted.  `exchange`: a
        sharding.SwitchAllReduce over P*14 floats — the backward then writes into ITS buffer and carries the sum over the
        ranks in its own launches (ViewBatch steps only; every rank builds and replays the same step).
        `loss_target`: a static CUDA tensor shaped like the rendered image ([3,H,W] / [n_out,3,H,W]) instead of `dL`:
        the step then evaluates photometric_loss(image, loss_target, lambda_dssim) into the static `self.loss` (0-dim /
        [n_out]) and back-propagates the MEAN of the per-image losses.  Write each iteration's targets into it in
        place.  8-bit targets (SPEC U12): `loss_target` a contiguous uint8 [H,W,3] / [n_out,H,W,3] tensor, or a
        contiguous uint8 [F,H,W,3] cube with `loss_index`, a contiguous int32 [n_out] CUDA tensor: the graph reads both
        in place, so an in-place write of the index picks the next replay's frames."""
        self.rast, self.params, self.dL = rast, params, dL
        m = params["means3D"]
        if not m.is_cuda:
            raise RasterizerError("GraphedStep needs CUDA tensors: gsvc_b200 has no CPU fallback")
        self.device, self.P = m.device, int(m.shape[0])
        self.loss_target, self.lambda_dssim, self.loss = loss_target, lambda_dssim, None
        self.loss_index = loss_index
        if loss_index is not None and (loss_target is None or loss_target.dtype != torch.uint8):
            raise RasterizerError("loss_index picks frames of a uint8 loss_target cube: pass both")
        if loss_target is not None:
            if dL is not None:
                raise RasterizerError("pass either dL (a fixed seed gradient) or loss_target (the step's own loss)")
            _check_lambda(lambda_dssim)
            if not isinstance(loss_target, torch.Tensor) or loss_target.device != self.device:
                raise RasterizerError(f"loss_target must be a tensor on {self.device}")
            if loss_target.dtype == torch.uint8:
                _check_rgb8_loss_target(loss_target, loss_index, self.device)
            elif loss_target.dtype != torch.float32 or not loss_target.is_contiguous():
                # a converted copy would be baked into the graph: in-place updates of the caller's tensor would be lost
                raise RasterizerError("loss_target must be a contiguous fp32 tensor (the graph reads it in place)")
        self.backward = dL is not None or loss_target is not None
        self.exchange = exchange
        if exchange is not None:
            if not isinstance(rast, ViewBatch) or not self.backward:
                raise RasterizerError("a step carries the exchange in its batched-view backward: pass a ViewBatch and dL")
            if packed is not None:
                raise RasterizerError("with `exchange` the packed buffer is the exchange's own")
            packed = exchange.buffer().view(self.P, GRAD_WIDTH)
            self._exchange_generation = exchange.generation
        if self.backward and packed is None:
            packed = torch.empty((self.P, GRAD_WIDTH), dtype=torch.float32, device=self.device)
        self.packed = packed
        self.warmup = max(int(warmup), 1)
        self.graph = None
        self.color = self.radii = None
        # the graph's own pinned count word: its scan kernel publishes num_rendered here on every replay, whatever
        # other graphs or eager calls of this thread do meanwhile; the capture records its capacity on it
        self.slot = R.CountSlot()
        self.capacity = None
        self.recapture()

    def _run(self):
        p = self.params
        if not self.backward:
            with torch.no_grad():
                return (*render_params(self.rast, p, means2D=p["means3D"]), None)   # no gradient: any tensor serves
        return _packed_step(self.rast, p, self.dL, self.packed, self.exchange, self.loss_target, self.lambda_dssim,
                            self.loss_index)

    def recapture(self) -> None:
        """(Re)build the graph: eager warm-up on a side stream (sets the capacity hint), then capture."""
        cur = torch.cuda.current_stream(self.device)
        side = torch.cuda.Stream(self.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(self.warmup):
                _, _, n, _ = self._run()
        cur.wait_stream(side)
        torch.cuda.synchronize(self.device)
        R.overflow_events(self.device)      # an eager warm-up call that outgrew its hint re-ran by itself: not ours
        self.num_rendered_at_capture = n
        self.graph = torch.cuda.CUDAGraph()
        with R.own_count_slot(self.slot), torch.cuda.graph(self.graph):
            self.color, self.radii, _, self.loss = self._run()
        self.capacity = self.slot.capacity

    def __call__(self):
        if self.exchange is not None and self.exchange.generation != self._exchange_generation:
            raise RasterizerError("the exchange's symmetric buffer was reallocated after this step was captured "
                                  "(SwitchAllReduce.sum_ outgrew it): build a new GraphedStep")
        self.graph.replay()
        return self.color, self.radii, self.packed

    def num_rendered(self) -> int:
        """Instance count of this graph's last replay (call after a synchronisation)."""
        return self.slot.value()

    def capacity_ok(self) -> bool:
        """After a synchronisation: no replay since the last check ran out of the instance capacity fixed at
        capture time (sticky device-side counter), and the last replay's published count fits too."""
        return _steps_fit(self.device, [self])


class FrameStreamer:
    """Throughput rendering of INDEPENDENT frames (video decode / evaluation: the Gaussians are fixed, only the
    frame's view matrices change — utils/report_utils.py:297-319 renders them one at a time with a synchronise
    around each).  `n_streams` forward-only graphs, each with private view-matrix tensors, are replayed round-robin
    on their own CUDA streams, so the latency-bound binning kernels of frame i+1 run under the issue-bound blend of
    frame i (measured: 170 -> 147 us per 1080p frame with 4 streams, config 2).

        streamer = FrameStreamer(front0, back0, params, n_streams=4)       # settings of any frame of the cube
        for i, (V_front, V_back) in enumerate(frames):                      # logical 4x4 view matrices (tensors)
            image = streamer.render(V_front, V_back)                        # [3,H,W], valid after streamer.wait(image)
        streamer.synchronize()

    `render` returns the stream's static output tensor: it is overwritten n_streams frames later, so consume it
    (on its stream, or after `wait`) before that.

    Decode-and-evaluate: with a `target` frame and a `quality` output (3 fp32 values on the device, typically a row
    of the caller's [F,3] tensor), the frame's PSNR / SSIM / MS-SSIM (gsvc_b200.quality) are computed on its stream
    right after the replay, before the output tensor can be reused; one synchronisation at the end of the loop:

        q = torch.empty(F, 3, device="cuda")
        for i, (V_front, V_back) in enumerate(frames):
            streamer.render(V_front, V_back, target=gt[i], quality=q[i])
        streamer.synchronize()                                              # q: [F,3] psnr, ssim, ms_ssim

    Decode-to-host: with `host_out`, a pinned contiguous uint8 CPU tensor shaped like the frame ([H,W,3] for a toast,
    [n_out,H,W,3] otherwise), the frame is converted to 8-bit RGB on its stream after the replay (and after the
    quality pass, if any) into one of 2 x n_streams device staging buffers, and copied from there into `host_out` on
    one device-to-host stream: the copy waits for the conversion, and a staging buffer is converted into again only
    after its previous copy.  The frame's own stream never waits for the link, so its next replay is not delayed by
    the ~0.11 ms a 1080p frame takes to cross it.  `last_event()` is recorded after the copy; a decode-to-disk loop
    keeps a ring of pinned buffers and waits on a buffer's event before it writes the frame out and reuses it:

        ring = [torch.empty(H, W, 3, dtype=torch.uint8).pin_memory() for _ in range(R)]
        done = [None] * R
        for i, (V_front, V_back) in enumerate(frames):
            j = i % R
            if done[j] is not None:
                done[j].synchronize(); write_png(ring[j])                   # frame i - R
            streamer.render(V_front, V_back, host_out=ring[j])
            done[j] = streamer.last_event()
        streamer.synchronize()                                              # then write the last R frames

    Evaluate against the source video's 8-bit frames (SPEC U12): `target` may be a uint8 frame ([H,W,3] for a toast,
    [n_out,H,W,3] otherwise, contiguous), on the device (e.g. `cube[i]` of a resident cube) or in pinned host memory.
    A host frame is copied on one host-to-device stream into one of 2 x n_streams device staging buffers, enqueued
    before the frame's replay so that the copy runs under the render; the frame's stream waits for it only before its
    quality pass, and a staging buffer is uploaded into again only after the quality pass that read it.  Pageable host
    memory is refused (the copy would block the host).  `last_event()` follows the quality pass, so it covers the
    upload: a caller streaming frames from disk refills its ring of pinned input buffers after a buffer's event:

        ring = [torch.empty(H, W, 3, dtype=torch.uint8).pin_memory() for _ in range(R)]
        done = [None] * R
        for i, (V_front, V_back) in enumerate(frames):
            j = i % R
            if done[j] is not None:
                done[j].synchronize()                                       # frame i - R has been read
            ring[j].copy_(source_frame(i))                                  # e.g. np.array(PIL.Image.open(...))
            streamer.render(V_front, V_back, target=ring[j], quality=q[i])
            done[j] = streamer.last_event()
        streamer.synchronize()

    A replay that overflowed its capacity (`capacity_ok()` false after a synchronisation) leaves invalid quality values
    and invalid host frames alike."""

    def __init__(self, front, back, params: Dict[str, torch.Tensor], n_streams: int = 4, toast: bool = True):
        m = params["means3D"]
        if not m.is_cuda:
            raise RasterizerError("FrameStreamer needs CUDA tensors: gsvc_b200 has no CPU fallback")
        self.device, self.n = m.device, int(n_streams)
        self.streams, self.steps, self.mats, self.events = [], [], [], []
        cur = torch.cuda.current_stream(self.device)
        for _ in range(self.n):
            s = torch.cuda.Stream(self.device)
            vf = front.viewmatrix.to(self.device, torch.float32).contiguous().clone()
            vb = back.viewmatrix.to(self.device, torch.float32).contiguous().clone()
            f, b = front._replace(viewmatrix=vf), back._replace(viewmatrix=vb)
            batch = ViewBatch.toast(f, b) if toast else ViewBatch([f, b])
            s.wait_stream(cur)
            with torch.cuda.stream(s):
                step = GraphedStep(batch, params, None)
            self.streams.append(s)
            self.steps.append(step)
            self.mats.append((vf, vb))
            self.events.append(None)
        self.scratch = [None] * self.n          # per-stream scratch of the quality metrics, allocated on first use
        self.staging = [None] * (2 * self.n)    # uint8 frames of the host copies, frame f in f % 2n (its stream's)
        self.copied = [None] * (2 * self.n)     # event after the last copy out of each staging buffer
        self.copy_stream = None                 # the device-to-host stream, created on first use
        self.t_staging = [None] * (2 * self.n)  # uint8 host targets uploaded for frame f in f % 2n
        self.t_read = [None] * (2 * self.n)     # event after the quality pass that last read each of them
        self.upload_stream = None               # the host-to-device stream, created on first use
        self._last_event = None
        self.i = 0

    def render(self, V_front: torch.Tensor, V_back: torch.Tensor, target: Optional[torch.Tensor] = None,
               quality: Optional[torch.Tensor] = None, host_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        k = self.i % self.n
        if (target is None) != (quality is None):
            raise RasterizerError("render: give both target and quality, or neither")
        rgb8 = isinstance(target, torch.Tensor) and target.dtype == torch.uint8
        if rgb8:
            self._check_rgb8_target(self.steps[k].color, target, quality)
        elif target is not None:
            self._check_quality_args(self.steps[k].color, target, quality)
        if host_out is not None:
            self._check_host_out(self.steps[k].color, host_out)
        j = self.i % (2 * self.n)
        self.i += 1
        s = self.streams[k]
        s.wait_stream(torch.cuda.current_stream(self.device))      # V_front / V_back may have just been produced
        uploaded = self._upload(j, target) if rgb8 and not target.is_cuda else None
        with torch.cuda.stream(s):
            self.mats[k][0].copy_(V_front, non_blocking=True)
            self.mats[k][1].copy_(V_back, non_blocking=True)
            color, _, _ = self.steps[k]()
            if rgb8:
                quality.record_stream(s)
                N, _, H, W = color.shape
                if self.scratch[k] is None:
                    self.scratch[k] = R._bytes(Q.scratch_bytes(N, H, W), self.device)
                if uploaded is not None:
                    s.wait_event(uploaded)
                    frames = self.t_staging[j]
                else:
                    target.record_stream(s)
                    frames = target
                Q.quality_rgb8_into(quality.view(N, 3), color, frames.view(N, H, W, 3), None, self.scratch[k])
            elif target is not None:
                target.record_stream(s)
                quality.record_stream(s)
                N, _, H, W = color.shape
                if self.scratch[k] is None:
                    self.scratch[k] = R._bytes(Q.scratch_bytes(N, H, W), self.device)
                y = R._dev_f32(target, self.device, "target").reshape(color.shape)
                Q.quality_into(quality, color, y, self.scratch[k])
            if host_out is not None:
                if self.copy_stream is None:
                    self.copy_stream = torch.cuda.Stream(self.device)
                if self.staging[j] is None:
                    self.staging[j] = torch.empty(host_out.shape, dtype=torch.uint8, device=self.device)
                if self.copied[j] is not None:
                    s.wait_event(self.copied[j])
                E.rgb8_into(self.staging[j], color)
            self.events[k] = s.record_event()
        if uploaded is not None:
            self.t_read[j] = self.events[k]
        self._last = k
        self._last_event = self.events[k]
        if host_out is not None:
            self.copy_stream.wait_event(self.events[k])
            with torch.cuda.stream(self.copy_stream):
                host_out.copy_(self.staging[j], non_blocking=True)
                self.copied[j] = self._last_event = self.copy_stream.record_event()
        return color[0] if color.shape[0] == 1 else color

    def _check_quality_args(self, color, target, quality):
        frame = color.shape[1:] if color.shape[0] == 1 else color.shape
        if not isinstance(target, torch.Tensor) or target.device != self.device or target.shape != frame:
            raise RasterizerError(f"render: target must be a tensor of shape {tuple(frame)} on {self.device}")
        self._check_quality_out(frame, quality)

    def _check_quality_out(self, frame, quality):
        want = frame[:-3] + (3,)
        if (not isinstance(quality, torch.Tensor) or quality.device != self.device or quality.shape != want
                or quality.dtype != torch.float32 or not quality.is_contiguous()):
            raise RasterizerError(f"render: quality must be a contiguous float32 tensor of shape {tuple(want)} "
                                  f"on {self.device}")

    def _check_rgb8_target(self, color, target, quality):
        frame = color.shape[1:] if color.shape[0] == 1 else color.shape
        want = tuple(frame[:-3]) + (frame[-2], frame[-1], 3)
        if tuple(target.shape) != want or not target.is_contiguous():
            raise RasterizerError(f"render: a uint8 target must be a contiguous tensor of shape {want}, got "
                                  f"{tuple(target.shape)}")
        if target.is_cuda:
            if target.device != self.device:
                raise RasterizerError(f"render: target is on {target.device}, expected {self.device} or pinned host memory")
        elif not target.is_pinned():
            raise RasterizerError("render: a host target must be pinned (a copy from pageable memory blocks the host)")
        self._check_quality_out(frame, quality)

    def _upload(self, j, target):
        """Enqueue the copy of pinned host frame `target` into staging buffer j; returns the event after it."""
        if self.upload_stream is None:
            self.upload_stream = torch.cuda.Stream(self.device)
        if self.t_staging[j] is None:
            self.t_staging[j] = torch.empty(target.shape, dtype=torch.uint8, device=self.device)
        u = self.upload_stream
        if self.t_read[j] is not None:
            u.wait_event(self.t_read[j])            # the quality pass that read this buffer last
        with torch.cuda.stream(u):
            self.t_staging[j].copy_(target, non_blocking=True)
            return u.record_event()

    def _check_host_out(self, color, host_out):
        frame = color.shape[1:] if color.shape[0] == 1 else color.shape
        want = tuple(frame[:-3]) + (frame[-2], frame[-1], 3)
        if not isinstance(host_out, torch.Tensor) or host_out.is_cuda:
            raise RasterizerError("render: host_out must be a CPU tensor (pinned), the frame's destination on the host")
        if not host_out.is_pinned():
            raise RasterizerError("render: host_out must be pinned (a copy into pageable memory blocks the host)")
        if host_out.dtype != torch.uint8 or tuple(host_out.shape) != want or not host_out.is_contiguous():
            raise RasterizerError(f"render: host_out must be a contiguous uint8 tensor of shape {want}")

    def last_event(self) -> torch.cuda.Event:
        """The event recorded after everything `render` enqueued for the most recent frame, its host copy and the
        upload of a host target included (the quality pass waits for the upload; this event follows both)."""
        if self._last_event is None:
            raise RasterizerError("last_event: no frame has been rendered yet")
        return self._last_event

    def wait(self, image: torch.Tensor = None) -> None:
        """Make the current stream wait for the most recently submitted frame."""
        torch.cuda.current_stream(self.device).wait_event(self.events[self._last])

    def synchronize(self) -> None:
        for s in self.streams + [t for t in (self.copy_stream, self.upload_stream) if t is not None]:
            s.synchronize()

    def capacity_ok(self) -> bool:
        """After `synchronize()`: every frame since the last check fitted the instance capacity of the graphs, and
        so did each stream's last frame."""
        return _steps_fit(self.device, self.steps)

    def recapture(self) -> None:
        for s, step in zip(self.streams, self.steps):
            with torch.cuda.stream(s):
                step.recapture()
