#!/usr/bin/env python
"""bench.py — headline benchmark of the rasterizer hot path (BASELINE.json metric, config 2).

    python bench.py --gpus N --steps K --warmup W            # product arm (CUDA, sm_100a)
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm: pure-PyTorch oracle on the host cores

A step = one pass of the hot path over one view of the synthetic UVG-shaped workload
(1920x1080, 200k Gaussians, BASELINE.json configs[1]): rasterizer forward + backward through the
reference-shaped GaussianRasterizer autograd surface.  Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

from gsvc_b200.frames import CONFIGS, CubeGeometry, synthetic_gaussians

WORKLOAD = "UVG-shaped synthetic 1920x1080 frame, 200k Gaussians, forward+backward (BASELINE.json configs[1])"
METRIC = "train_iters_per_s"
UNIT = "iters/s (1 iter = rasterizer fwd+bwd of one 1080p view, 200k Gaussians)"   # a step (one frame) is 2 iters
THRESHOLD = 0.05  # /root/reference/cfgs/cfg_20240919.yaml:13


def dist_stats(ms_list):
    """median / p10 / p90 / min / mean of a list of per-step times (ms)."""
    a = sorted(ms_list)
    n = len(a)
    q = lambda f: a[min(n - 1, int(f * n))]
    return {"n": n, "median_ms": q(0.5), "p10_ms": q(0.1), "p90_ms": q(0.9), "min_ms": a[0], "mean_ms": sum(a) / n}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(P, V, R, N, T, nv=1):
    """Compulsory HBM bytes per launch of each kernel (DESIGN.md §4; SURVEY.md §8d stages S1..S5
    restated for this design's buffers) for a batch of nv views: V = visible (view, Gaussian) pairs and
    R = instances over all views; P, N, T per view."""
    return {
        "preprocess": 56 * P + 4 * P * nv + 56 * V,      # inputs (once), radii, 3 float4 + rect per visible pair
        "tile_scan": (4 + 20) * T * nv,                   # counts in; offsets, cursors, ranges out
        "scatter": 24 * V + 8 * R,                        # rect + depth in; (depth_key|id) out
        "sort_tiles": 8 * R + 8 * R,                      # composites in; point_list + depth_keys out
        "render_forward": (8 * T + 20 * N) * nv + 40 * R,  # ranges, id + 36 B features per instance, colour+T+n_contrib
        "render_backward": (8 * T + 20 * N) * nv + 40 * R + 36 * V,  # + dL/dC, final_T, n_contrib in; 9 floats per visible out
        "preprocess_backward": 4 * P * nv + 76 * V + 56 * P + 12 * P * nv,   # radii, acc+geom+inputs; packed grads, means2D
        "visible_filter": 44 * P,
    }


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, sampled in-process through NVML
    (the same counters `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints; polling
    nvidia-smi itself stalls the driver for milliseconds at a time and would perturb the timing)."""

    def __init__(self, index, period=0.05):
        self.index, self.period, self.samples, self.stop_flag = index, period, [], False
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def _reasons(self):
        nv = self.nv
        try:
            return nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            return nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.samples.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), self._reasons()))
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.ok:
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()

    def stop(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self.stop_flag = True
        self.thread.join(timeout=2)
        nv = self.nv
        names = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4,
                 "hw_power_brake_slowdown": 0x80}
        sm = [c for c, _ in self.samples]
        bits = 0
        for _, r in self.samples:
            bits |= int(r)
        reasons = sorted(n for n, m in names.items() if bits & m)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_sm, "reasons": reasons,
                "samples": len(sm), "source": "nvml"}


def build_scene(n_frames: int, device):
    cfg = CONFIGS[2]
    geom = CubeGeometry(cfg["W"], cfg["H"], cfg["F"])
    f0 = cfg["F"] // 2
    g = synthetic_gaussians(cfg["P"], geom, f0, f0 + n_frames - 1, threshold=THRESHOLD, seed=2, device=device)
    return cfg, geom, f0, g


def settings_for(geom, frame_id, device, back=False):
    """GaussianRasterizationSettings exactly as renderer.py:63-83 builds them."""
    from gsvc_b200.rasterizer import GaussianRasterizationSettings
    fr = geom.frame(frame_id)
    vm = fr.view_matrix_s if back else fr.view_matrix
    return GaussianRasterizationSettings(
        image_height=int(fr.image_height), image_width=int(fr.image_width), x_min=fr.x_min, y_min=fr.y_min,
        scale=fr.scale, threshold=THRESHOLD, bg=torch.zeros(3, dtype=torch.float32, device=device),
        scale_modifier=1.0, viewmatrix=vm.permute(1, 0).to(device), sh_degree=0, campos=fr.cam_pos,
        prefiltered=False, debug=False)


# --------------------------------------------------------------------------------------------------
# CPU arm: the C oracle (oracle/splat_oracle.c, OpenMP over pixel rows / Gaussians) — there is no reference CPU
# implementation to run: renderer.py:37 is CUDA-only and the reference's CUDA rasterizer source is not in
# /root/reference.  The C port is the faster of the repo's two CPU restatements (the pure-PyTorch one does
# 0.4-0.6 view-iters/s on 16 cores), so it is the stronger baseline.
# --------------------------------------------------------------------------------------------------
def cpu_step(geom, f0, g_np, rows_div=1):
    """One view-iteration of the config-2 scene on the host cores: preprocess + binning + blend forward + blend
    backward + per-Gaussian backward, all Gaussians.  rows_div > 1 bounds the sample: only the top 1/rows_div of
    the image rows is rendered (the per-Gaussian stages still see every Gaussian) and the per-tile part of the time
    is scaled back by the row ratio.  Returns (seconds measured, seconds for the whole view, rows rendered)."""
    from oracle import c_oracle
    fr = geom.frame(f0)
    H = int(fr.image_height)
    h = H if rows_div == 1 else max(16, (H // rows_div) // 16 * 16)
    st = c_oracle.OracleSettings(image_height=h, image_width=int(fr.image_width), x_min=fr.x_min, y_min=fr.y_min,
                                 scale=fr.scale, threshold=THRESHOLD, bg=np.zeros(3, np.float32),
                                 viewmatrix=fr.view_matrix.permute(1, 0).numpy().copy(), campos=fr.cam_pos.numpy())
    dL = np.ones((3, h, int(fr.image_width)), np.float32)
    t0 = time.perf_counter()
    pre = c_oracle.preprocess(st, g_np["means3D"], g_np["scales"], g_np["rotations"], None, g_np["opacities"],
                              g_np["colors_precomp"])
    t1 = time.perf_counter()
    fwd = c_oracle.forward(st, g_np["means3D"], g_np["opacities"], g_np["scales"], g_np["rotations"],
                           colors_precomp=g_np["colors_precomp"])
    c_oracle.backward(fwd, dL)
    t2 = time.perf_counter()
    t_pre = t1 - t0                       # timed apart only to know the share that does not scale with the rows
    total = t2 - t1
    return total, t_pre + (total - t_pre) * (H / h), h


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    from oracle import c_oracle
    c_oracle.build()
    cores = c_oracle.set_threads(cores)                           # torchrun exports OMP_NUM_THREADS=1
    cfg, geom, f0, g = build_scene(1, "cpu")
    g_np = {k: v.numpy() for k, v in g.items()}
    H = int(geom.frame(f0).image_height)
    t_full, _, _ = cpu_step(geom, f0, g_np)                       # untimed: page in, size the sample
    budget = 170.0                                                # seconds for the whole --steps + --warmup run
    rows_div = max(1, int(np.ceil(t_full * (args.steps + args.warmup) / budget)))
    times, fulls = [], []
    for i in range(args.warmup + args.steps):
        total, full, h = cpu_step(geom, f0, g_np, rows_div)
        if i >= args.warmup:
            times.append(total)
            fulls.append(full)
    ms = 1000.0 * sum(times) / len(times)
    full_ms = 1000.0 * sum(fulls) / len(fulls)
    value = 1000.0 / full_ms
    sample = (f"C oracle (OpenMP, {cores} host threads) on the config 2 scene, one view forward+backward per step: all "
              f"{cfg['P']} Gaussians, " + ("every pixel" if h == H else
              f"the top {h} of {H} pixel rows (per-tile time scaled x{H / h:.1f} to the whole view; per-Gaussian "
              f"stages in full)"))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": full_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sampled_ms_per_step": ms},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# --------------------------------------------------------------------------------------------------
# product arm
# --------------------------------------------------------------------------------------------------
VIEWS_PER_STEP = 2   # a step renders one FRAME as the reference composes it: front + back view (train.py:353-375)


def run_product_arm(args, rank, local_rank, world):
    import torch.distributed as dist
    from gsvc_b200 import _lib
    from gsvc_b200.graphed import GraphedStep
    from gsvc_b200.hostpipe import HostStepPipeline
    from gsvc_b200.rasterizer import GaussianRasterizer
    from gsvc_b200.sharding import GRAD_LAYOUT, packed_backward
    from gsvc_b200.views import ViewBatch, rasterize_views
    from gsvc_b200.graphed import FrameStreamer

    if not torch.cuda.is_available():
        raise SystemExit("bench.py product arm needs a CUDA device (no CPU fallback exists)")
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
        # NCCL's kernels share the SMs with full-occupancy blend grids: on a normal-priority stream their CTAs are
        # only scheduled in a grid's tail while the peers' CTAs spin (measured at 2 GPUs: e2e 8 509 -> 8 873
        # view-iters/s with high-priority NCCL streams, `value` unchanged)
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")
        dist.init_process_group("nccl", device_id=device)
    L = _lib.lib()

    cfg, geom, f0, g = build_scene(world, device)
    frame_id = f0 + rank                     # frame-sharded window: rank r renders frame f0 + r of the shared set
    front, back = settings_for(geom, frame_id, device), settings_for(geom, frame_id, device, back=True)
    toast = ViewBatch.toast(front, back)     # image = (front + flip_x(back)) / 2, both views in ONE kernel chain
    rast = GaussianRasterizer(raster_settings=front)      # the single-view drop-in call, reported beside
    NV = VIEWS_PER_STEP
    P, W, H = cfg["P"], cfg["W"], cfg["H"]
    N, T = W * H, ((W + 15) // 16) * ((H + 15) // 16)
    params = {k: v.clone() for k, v in g.items()}         # static tensors: the graphs replay on them
    dL = torch.randn((1, 3, H, W), generator=torch.Generator().manual_seed(100 + rank)).to(device)
    # frame-sharded steps: the backward writes straight into one of two [P,14] buffers (no pack pass) and the
    # NCCL sum all-reduce of that buffer runs asynchronously, overlapping the next step's forward
    grad_bufs = [torch.empty((P, 14), dtype=torch.float32, device=device) for _ in range(2)]
    # multi-GPU: the all-reduce without a collective kernel (sharding.PeerAllReduce: symmetric-memory buffers,
    # copy-engine pulls, one small sum kernel) when the ranks can map each other's memory, NCCL otherwise
    peer_ar, allreduce_note = None, None
    if world > 1:
        from gsvc_b200.sharding import PeerAllReduce
        try:
            if os.environ.get("GSVC_BENCH_NCCL_ALLREDUCE") == "1" or (P * 14) % world:
                raise RuntimeError("disabled")
            peer_ar = PeerAllReduce(P * 14, device, slots=2)
            grad_bufs = [peer_ar.buffer(b).view(P, 14) for b in range(2)]
            allreduce_note = "sharding.PeerAllReduce: copy-engine pulls over symmetric memory + one sum kernel per rank"
        except Exception as e:
            allreduce_note = f"NCCL all_reduce (async, high-priority stream); peer path unavailable: {type(e).__name__}: {e}"

    def start_allreduce(b):
        if peer_ar is not None:
            return peer_ar.start(b)
        return dist.all_reduce(grad_bufs[b], op=dist.ReduceOp.SUM, async_op=True)

    pending = [None, None]
    step_no = [0]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=device)  # 256 MiB > 126 MB L2

    def leaves():
        return {k: params[k].detach().requires_grad_(True) for k, _ in GRAD_LAYOUT}

    def toast_eager(backward=True):
        """The step, launched eagerly (warm-up and the per-stage timing pass)."""
        if not backward:
            with torch.no_grad():
                return rasterize_views(toast, means3D=params["means3D"], opacities=params["opacities"],
                                       colors_precomp=params["colors_precomp"], scales=params["scales"],
                                       rotations=params["rotations"])
        p = leaves()
        images, radii, n = rasterize_views(toast, means3D=p["means3D"], opacities=p["opacities"],
                                           colors_precomp=p["colors_precomp"], scales=p["scales"],
                                           rotations=p["rotations"])
        b = step_no[0] & 1
        step_no[0] += 1
        if pending[b] is not None:
            pending[b].wait()                  # stream-level wait: the buffer's previous all-reduce has finished
        with packed_backward(grad_bufs[b]):
            torch.autograd.grad(images, [p[k] for k, _ in GRAD_LAYOUT], grad_outputs=dL)
        if world > 1:
            pending[b] = start_allreduce(b)
        return images, radii, n

    def toast_eager_fwd():
        return toast_eager(False)

    def single_eager():
        """One view through the reference-shaped drop-in call, eagerly, autograd and all."""
        p = leaves()
        means2D = torch.zeros_like(p["means3D"], requires_grad=True)
        color, radii, n = rast(means3D=p["means3D"], means2D=means2D, shs=None, colors_precomp=p["colors_precomp"],
                               opacities=p["opacities"], scales=p["scales"], rotations=p["rotations"],
                               cov3D_precomp=None)
        return torch.autograd.grad(color, [p[k] for k, _ in GRAD_LAYOUT], grad_outputs=dL[0])

    def single_eager_fwd():
        with torch.no_grad():
            return rast(means3D=params["means3D"], means2D=params["means3D"], shs=None,
                        colors_precomp=params["colors_precomp"], opacities=params["opacities"],
                        scales=params["scales"], rotations=params["rotations"], cov3D_precomp=None)

    def sync_all():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize(device)

    def timed(fn, steps):
        """EXACTLY `steps` steps between two barrier+synchronize brackets.  Each step is bracketed by its own
        CUDA events on the launching stream and the 256 MiB L2 flush runs between steps, outside the events;
        the host never synchronises inside the region, so it runs ahead of the device exactly as a training
        loop does.  Returns the max over ranks of the summed per-step device time."""
        sync_all()
        evs = []
        for _ in range(steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            evs.append((e0, e1))
        sync_all()
        per_step = [a.elapsed_time(b) for a, b in evs]
        total_ms = sum(per_step)
        if os.environ.get("GSVC_BENCH_DEBUG"):
            ps = sorted(per_step)
            sys.stderr.write(f"[bench debug] {fn.__name__}: mean {total_ms / steps:.4f} median {ps[len(ps) // 2]:.4f} "
                             f"p10 {ps[len(ps) // 10]:.4f} p90 {ps[9 * len(ps) // 10]:.4f} max {ps[-1]:.4f} ms\n")
        t = torch.tensor([total_ms], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        timed.last_per_step = per_step
        return float(t.item()), out

    # ---- warm-up (also sets the instance-capacity hints so no step re-sizes its buffers)
    for _ in range(max(args.warmup, 3)):
        flush.zero_()
        out = toast_eager()
        single_eager()
    torch.cuda.synchronize(device)
    num_rendered = out[2]                                   # instances of both views
    V = int((out[1] > 0).sum().item())                      # visible (view, Gaussian) pairs
    for w in pending:
        if w is not None:
            w.wait()

    # ---- the timed step: forward + backward of the frame replayed from a CUDA graph (gsvc_b200.graphed.GraphedStep),
    # one graph per gradient buffer.  An eager call must hand num_rendered back as a Python int, i.e. one host wait
    # per forward, which leaves the SMs idle for ~25 us per call now that the kernels are this short.
    L.gsvc_rast_launch_count(1)
    graph_note = None
    try:
        graphs = [GraphedStep(toast, params, dL, packed=grad_bufs[b]) for b in range(2)]
        kernels_per_step = int(L.gsvc_rast_launch_count(1)) // (2 * (graphs[0].warmup + 1))
        fwd_graph = GraphedStep(toast, params, None)
        single_graph = GraphedStep(rast, params, dL[0])
        single_fwd_graph = GraphedStep(rast, params, None)
    except Exception as e:   # a driver that cannot capture the chain: measure the eager launches instead, and say so
        graph_note = f"CUDA-graph capture failed ({type(e).__name__}: {e}); steps launched eagerly"
        sys.stderr.write("[bench] " + graph_note + "\n")
        torch.cuda.synchronize(device)
        graphs, kernels_per_step = None, 7
        fwd_graph, single_graph, single_fwd_graph = toast_eager_fwd, single_eager, single_eager_fwd

    def toast_graphed():
        if graphs is None:
            return toast_eager()
        b = step_no[0] & 1
        step_no[0] += 1
        if pending[b] is not None:
            pending[b].wait()
        out = graphs[b]()
        if world > 1:
            pending[b] = start_allreduce(b)
        return out

    for _ in range(4):
        toast_graphed()
        fwd_graph()
    torch.cuda.synchronize(device)

    clocks = ClockSampler(local_rank)
    clocks.start()
    # best of REPEATS measurements of exactly K steps each (a shared host occasionally stalls a step for
    # milliseconds; the minimum over repeats is the reproducible figure, as for MEASURED_PEAKS.json)
    REPEATS = 3
    per_step_all = []
    totals = []
    for _ in range(REPEATS):
        t_, last = timed(toast_graphed, args.steps)
        totals.append(t_)
        per_step_all += timed.last_per_step
    total_ms = min(totals)
    # distribution of the per-step device time over the REPEATS x K timed steps (this rank; SURVEY.md §8d asks for
    # median, p10, p90)
    step_stats = dist_stats(per_step_all)
    # what the caller of the timed step received from its last replay: the image, the radii and the packed [P,14]
    # gradients (summed over the ranks), copied to the host now, before other legs reuse the device buffers
    last_outputs = None
    if args.dump_outputs:
        b = (step_no[0] - 1) & 1
        if pending[b] is not None:
            pending[b].wait()
        torch.cuda.synchronize(device)
        n_last = graphs[b].num_rendered() if graphs is not None else last[2]
        last_outputs = {k: v.detach().float().cpu().numpy() for k, v in
                        (("image", last[0]), ("radii", last[1]), ("grads", grad_bufs[b]))}
        last_outputs["num_rendered"] = np.float64(n_last)
    if graphs is not None and not graphs[0].capacity_ok():
        raise SystemExit("the captured instance capacity was exceeded (cannot happen with a fixed scene)")
    launches = kernels_per_step * args.steps
    fwd_ms = min(timed(fwd_graph, args.steps)[0] for _ in range(REPEATS))
    for w in pending:
        if w is not None:
            w.wait()
    # single-view numbers (one rasterizer call = one view, no all-reduce): graph replay and the eager drop-in call
    single_ms = min(timed(single_graph, args.steps)[0] for _ in range(REPEATS))
    single_fwd_ms = min(timed(single_fwd_graph, args.steps)[0] for _ in range(REPEATS))
    eager_ms = min(timed(single_eager, args.steps)[0] for _ in range(REPEATS))
    eager_fwd_ms = min(timed(single_eager_fwd, args.steps)[0] for _ in range(REPEATS))
    # the same K steps again, launched eagerly with a CUDA-event pair around every kernel (events between kernels
    # defeat the programmatic-dependent-launch overlap, so this pass is slower: it only feeds the roofline)
    _lib.stage_timing(True)
    staged_ms, _ = timed(toast_eager, args.steps)
    stage_avg = _lib.stage_times()          # mean per stage over the timed steps (last 256)
    timed(toast_eager_fwd, args.steps)
    fwd_stage_avg = _lib.stage_times()
    _lib.stage_timing(False)
    for w in pending:
        if w is not None:
            w.wait()


    # ---- the reference's real call pattern (ortho_gaussian_renderer/renderer.py:28-98): a DIFFERENT P on every call
    # (the Gaussians of the anchors visible in that view), eager, through GaussianRasterizer and autograd.  Each step
    # takes a prefix of a 240k-Gaussian set with P uniform in 200k +- 20 %; the binning capacity comes from the
    # instances-per-Gaussian density hint, so scatter / sort / blend are launched before num_rendered is known.
    dropin = None
    if world == 1:
        from gsvc_b200 import rasterizer as R_
        gbig = synthetic_gaussians(int(cfg["P"] * 1.2), geom, f0, f0, threshold=THRESHOLD, seed=12, device=device)
        rng = np.random.default_rng(7)
        sizes = [int(cfg["P"] * (0.8 + 0.4 * rng.random())) for _ in range(64)]
        it = [0]

        def dropin_step():
            Pi = sizes[it[0] % len(sizes)]
            it[0] += 1
            p = {k: gbig[k][:Pi].detach().requires_grad_(True) for k, _ in GRAD_LAYOUT}
            means2D = torch.zeros_like(p["means3D"], requires_grad=True)
            color, radii, n = rast(means3D=p["means3D"], means2D=means2D, shs=None, colors_precomp=p["colors_precomp"],
                                   opacities=p["opacities"], scales=p["scales"], rotations=p["rotations"],
                                   cov3D_precomp=None)
            return torch.autograd.grad(color, [p[k] for k, _ in GRAD_LAYOUT], grad_outputs=dL[0])

        for _ in range(8):
            dropin_step()
        torch.cuda.synchronize(device)
        before = dict(R_.capacity_stats)
        ms = min(timed(dropin_step, args.steps)[0] for _ in range(REPEATS))
        st_ = dist_stats(timed.last_per_step)
        dropin = {"ms_per_view": ms / args.steps, "iters_per_s": 1000.0 * args.steps / ms, "median_ms": st_["median_ms"],
                  "p10_ms": st_["p10_ms"], "p90_ms": st_["p90_ms"], "P_min": min(sizes), "P_max": max(sizes),
                  "ratio_to_single_view_graph": (ms / args.steps) / (single_ms / args.steps),
                  "capacity_rerenders": R_.capacity_stats["rerendered"] - before["rerendered"],
                  "calls": R_.capacity_stats["calls"] - before["calls"],
                  "note": "eager GaussianRasterizer + autograd, P drawn per step from 200k +- 20 % (prefixes of one "
                          "240k set); mean P = 200k, so ms_per_view compares with single_view.graph at P = 200k"}
        del gbig

    # ---- GPU comparator (baseline/naive: the published 3DGS rasterizer structure on cub::DeviceScan /
    # cub::DeviceRadixSort, one pixel per thread, per-pixel-atomic backward, sm_100a build; test infrastructure):
    # the same config-2 view, forward + backward, eager with its one host synchronisation per forward
    gpu_baseline = None
    if world == 1 and not args.no_gpu_baseline:
        try:
            from baseline.naive import naive as NAIVE
            nv = NAIVE.NaiveRasterizer(front)
            a_ = [params[k] for k in ("means3D", "scales", "rotations", "opacities", "colors_precomp")]

            def naive_step():
                nv.forward(*a_)
                return nv.backward(dL[0])

            def naive_fwd():
                return nv.forward(*a_)

            for _ in range(3):
                naive_step()
            torch.cuda.synchronize(device)
            nb_ms = min(timed(naive_step, args.steps)[0] for _ in range(REPEATS))
            nf_ms = min(timed(naive_fwd, args.steps)[0] for _ in range(REPEATS))
            NAIVE.timing(True)
            naive_step()
            torch.cuda.synchronize(device)
            nstages = NAIVE.stage_times()
            NAIVE.timing(False)
            gpu_baseline = {"value": 1000.0 * args.steps / nb_ms, "unit": UNIT, "ms_per_view": nb_ms / args.steps,
                            "fwd_views_per_s": 1000.0 * args.steps / nf_ms, "stage_ms": {k: round(v, 5) for k, v in nstages.items()},
                            "num_rendered": nv.R, "kind": "upstream-design comparator (baseline/naive), same scene, same SPEC",
                            "speedup_single_view_graph": (nb_ms / args.steps) / (single_ms / args.steps),
                            "speedup_single_view_eager": (nb_ms / args.steps) / (eager_ms / args.steps)}
        except Exception as e:  # the comparator is optional infrastructure: say why it is absent
            gpu_baseline = {"unavailable": f"{type(e).__name__}: {e}"}

    # ---- BASELINE config 4: 1M Gaussians, 1080p, forward only (stream decode), both views
    config4 = None
    if world == 1:
        c4 = CONFIGS[4]
        g4 = synthetic_gaussians(c4["P"], geom, f0, f0, threshold=THRESHOLD, seed=4, device=device)
        rast_b = GaussianRasterizer(raster_settings=back)

        def c4_plain():
            with torch.no_grad():
                kw = dict(means2D=g4["means3D"], shs=None, colors_precomp=g4["colors_precomp"], opacities=g4["opacities"],
                          scales=g4["scales"], rotations=g4["rotations"], cov3D_precomp=None)
                a = rast(means3D=g4["means3D"], **kw)
                b = rast_b(means3D=g4["means3D"], **kw)
                return (a[0] + torch.flip(b[0], dims=(-1,))) * 0.5, a[2] + b[2]

        for _ in range(3):
            img4, R4 = c4_plain()
        torch.cuda.synchronize(device)
        plain_ms = min(timed(c4_plain, args.steps)[0] for _ in range(REPEATS))
        streamed4 = None
        if graphs is not None:
            st4 = FrameStreamer(front, back, g4, n_streams=4)
            for _ in range(8):
                st4.render(front.viewmatrix, back.viewmatrix)
            st4.synchronize()
            best = None
            for _ in range(REPEATS):
                sync_all()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    st4.render(front.viewmatrix, back.viewmatrix)
                st4.wait()
                for s_ in st4.streams:
                    torch.cuda.current_stream(device).wait_stream(s_)
                e1.record()
                sync_all()
                best = e0.elapsed_time(e1) if best is None else min(best, e0.elapsed_time(e1))
            streamed4 = best if st4.capacity_ok() else None
            del st4
        config4 = {"workload": "1M Gaussians, 1920x1080, forward only, front + back view per frame (BASELINE.json configs[3])",
                   "P": c4["P"], "R_frame": int(R4),
                   "plain_calls": {"frames_per_s": 1000.0 * args.steps / plain_ms, "views_per_s": 2000.0 * args.steps / plain_ms,
                                   "ms_per_frame": plain_ms / args.steps,
                                   "how": "two eager GaussianRasterizer calls + flip + average per frame"},
                   "streamed": None if streamed4 is None else {
                       "frames_per_s": 1000.0 * args.steps / streamed4, "views_per_s": 2000.0 * args.steps / streamed4,
                       "ms_per_frame": streamed4 / args.steps, "how": "gsvc_b200.graphed.FrameStreamer, 4 streams"}}
        del g4

    # ---- BASELINE config 5: 2M Gaussians, 3840x2160, forward + backward of one view (tile lists / sort stress)
    config5 = None
    if world == 1:
        c5 = CONFIGS[5]
        geom5 = CubeGeometry(c5["W"], c5["H"], c5["F"])
        f5 = c5["F"] // 2
        g5 = synthetic_gaussians(c5["P"], geom5, f5, f5, threshold=THRESHOLD, seed=5, device=device)
        rast5 = GaussianRasterizer(raster_settings=settings_for(geom5, f5, device))
        dL5 = torch.randn((3, c5["H"], c5["W"]), generator=torch.Generator().manual_seed(5)).to(device)
        step5 = GraphedStep(rast5, g5, dL5) if graphs is not None else None

        def c5_eager():
            p = {k: g5[k].detach().requires_grad_(True) for k, _ in GRAD_LAYOUT}
            m2 = torch.zeros_like(p["means3D"], requires_grad=True)
            color, radii, n = rast5(means3D=p["means3D"], means2D=m2, shs=None, colors_precomp=p["colors_precomp"],
                                    opacities=p["opacities"], scales=p["scales"], rotations=p["rotations"], cov3D_precomp=None)
            torch.autograd.grad(color, [p[k] for k, _ in GRAD_LAYOUT], grad_outputs=dL5)
            return n

        for _ in range(3):
            R5 = c5_eager()
        torch.cuda.synchronize(device)
        n5 = args.steps
        e5_ms = min(timed(c5_eager, n5)[0] for _ in range(2))
        g5_ms = min(timed(step5, n5)[0] for _ in range(2)) if step5 is not None else None
        config5 = {"workload": "2M Gaussians, 3840x2160, forward + backward of one view (BASELINE.json configs[4])",
                   "P": c5["P"], "R": int(R5), "T": ((c5["W"] + 15) // 16) * ((c5["H"] + 15) // 16),
                   "eager": {"iters_per_s": 1000.0 * n5 / e5_ms, "ms_per_view": e5_ms / n5},
                   "graph": None if g5_ms is None else {"iters_per_s": 1000.0 * n5 / g5_ms, "ms_per_view": g5_ms / n5}}
        del g5, step5, dL5

    # ---- BASELINE config 3: 500k Gaussians shared by an 8-frame TSW window, the 8 frames dealt round-robin to the N
    # ranks (STRONG scaling: 16 / N views per rank in one batched chain), then ONE fp32 sum all-reduce of the [P,14]
    # gradient buffer (28 MB) — issued after the backward and waited for INSIDE the timed events.
    config3 = None
    if 8 % world == 0:
        c3 = CONFIGS[3]
        frames3 = list(range(f0, f0 + c3["window"]))
        g3 = synthetic_gaussians(c3["P"], geom, frames3[0], frames3[-1], threshold=THRESHOLD, seed=3, device=device)
        mine = [f for i, f in enumerate(frames3) if i % world == rank]
        batch3 = ViewBatch.toasts([(settings_for(geom, f, device), settings_for(geom, f, device, back=True)) for f in mine])
        dL3 = torch.randn((len(mine), 3, H, W), generator=torch.Generator().manual_seed(300 + rank)).to(device)
        # This all-reduce is exposed by construction — the window ends with it, nothing overlaps it — so it should move the
        # 28 MB as fast as the links allow: gsvc_b200.sharding.SwitchAllReduce, ONE kernel of this library per rank
        # (csrc/collective.cu): multimem.ld_reduce / multimem.st through the NVSwitch from 4 ranks up, peer loads and
        # stores for 2 (measured at 28 MB, 2 / 8 GPUs: 61 / 86 us against 76 / 143 us for NCCL and 110 / 206 us for the
        # copy-engine PeerAllReduce, which is built for the OVERLAPPED all-reduce of the training step above).
        ar3, ar3_note = None, "NCCL all_reduce"
        buf3 = None
        if world > 1 and os.environ.get("GSVC_BENCH_C3_NCCL", "0") != "1":
            try:
                from gsvc_b200.sharding import SwitchAllReduce
                ar3 = SwitchAllReduce(c3["P"] * 14, device)
                buf3 = ar3.buffer().view(c3["P"], 14)
                ar3_note = (f"sharding.SwitchAllReduce ({ar3.mode}: " +
                            ("multimem.ld_reduce / multimem.st through the NVSwitch" if ar3.mode == "multicast"
                             else "peer loads + stores over NVLink") + f", one kernel, {ar3.n_ctas} CTAs)")
            except Exception as e:   # no symmetric memory on this box: NCCL
                ar3, ar3_note = None, f"NCCL all_reduce (switch path unavailable: {type(e).__name__}: {e})"
        if buf3 is None:
            buf3 = torch.empty((c3["P"], 14), dtype=torch.float32, device=device)
        for _ in range(2):
            rasterize_views(batch3, means3D=g3["means3D"], opacities=g3["opacities"], colors_precomp=g3["colors_precomp"],
                            scales=g3["scales"], rotations=g3["rotations"])
        step3 = GraphedStep(batch3, g3, dL3, packed=buf3) if graphs is not None else None
        # From 4 ranks up the backward CARRIES the exchange (gsvc_rast_backward_views_exchange): the first CTAs of the
        # per-Gaussian backward kernel sum the rows through the switch chunk by chunk while the others still compute
        # (8 GPUs: window 0.991 -> 0.964 ms; with 2 ranks and peer loads the separate launch is faster: 3.413 vs 3.451).
        step3x = None
        if ar3 is not None and ar3.mode == "multicast" and world >= 4 and graphs is not None and \
                os.environ.get("GSVC_BENCH_C3_FUSED", "1") == "1":
            try:
                step3x = GraphedStep(batch3, g3, dL3, exchange=ar3)
                ar3_note = ("sharding.SwitchAllReduce carried by the per-Gaussian backward's own launch "
                            "(gsvc_rast_backward_views_exchange: multimem.ld_reduce / multimem.st through the NVSwitch by "
                            "the kernel's first CTAs, chunk by chunk under the computation of the later rows)")
            except Exception as e:   # the separate launch below still works
                step3x = None
                ar3_note += f"; the carried exchange was unavailable: {type(e).__name__}: {e}"

        def c3_compute():
            if step3 is not None:
                return step3()
            p = {k: g3[k].detach().requires_grad_(True) for k, _ in GRAD_LAYOUT}
            img, _, _ = rasterize_views(batch3, means3D=p["means3D"], opacities=p["opacities"],
                                        colors_precomp=p["colors_precomp"], scales=p["scales"], rotations=p["rotations"])
            with packed_backward(buf3):
                torch.autograd.grad(img, [p[k] for k, _ in GRAD_LAYOUT], grad_outputs=dL3)

        def c3_step():
            if step3x is not None:
                step3x()                                         # forward + backward + exchange, one graph
                return
            c3_compute()
            if ar3 is not None:
                ar3.run()                                        # on the compute stream: the step ends when it has
            elif world > 1:
                dist.all_reduce(buf3, op=dist.ReduceOp.SUM)      # on the compute stream: the step ends when it has

        n3 = args.steps
        for _ in range(3):
            c3_step()
        torch.cuda.synchronize(device)
        w_ms = min(timed(c3_step, n3)[0] for _ in range(REPEATS))
        c_ms = min(timed(c3_compute, n3)[0] for _ in range(REPEATS)) if world > 1 else w_ms
        config3 = {"workload": "500k Gaussians, 8-frame TSW window (16 views) of a 600-frame 1080p video, frames dealt "
                               "round-robin to the ranks, fp32 sum all-reduce of [P,14] per window (BASELINE.json configs[2])",
                   "P": c3["P"], "scaling": "strong", "n_gpus": world, "views_per_rank": 2 * len(mine),
                   "window_ms": w_ms / n3, "windows_per_s": 1000.0 * n3 / w_ms, "view_iters_per_s": 16000.0 * n3 / w_ms,
                   "compute_only_window_ms": c_ms / n3, "exposed_collective_us": 1000.0 * (w_ms - c_ms) / n3,
                   "allreduce_bytes": c3["P"] * 14 * 4 if world > 1 else 0,
                   "allreduce": None if world == 1 else ar3_note,
                   # every wait of the exchange kernels is bounded; a non-zero count would mean a rank did not arrive in
                   # time and the timed windows are void
                   "exchange_waits_that_gave_up": None if ar3 is None else ar3.timeouts(),
                   "timing": "max over ranks; the all-reduce is issued on the compute stream after the backward and the "
                             "step's end event follows it"}
        del g3, step3, step3x, buf3, dL3, ar3


    # ---- row f2, second half: the generator's epilogue between the MLPs and the rasterizer call
    # (guassian.py:147-153, 251-293) fused (gsvc_b200.generate) against the PyTorch expression it replaces, forward and
    # forward + backward, 100k visible of 600k anchors x 10 offsets (reference scale: init_anchor_num x n_offsets)
    epilogue = None
    if world == 1:
        from gsvc_b200.generate import neural_gaussians_epilogue, reference_epilogue
        Na, Ka, nv_ = 600_000, 10, 100_000
        gg_ = torch.Generator().manual_seed(9)
        rr = lambda *s_: torch.randn(*s_, generator=gg_).to(device)
        ep_in = [torch.rand(Na, 3, generator=gg_).to(device), 0.3 * rr(Na, Ka, 3), torch.exp(0.3 * rr(Na, 6) - 3.0),
                 (torch.rand(Na, Ka, 1, generator=gg_) > 0.3).float().to(device)]
        ep_vis = torch.sort(torch.randperm(Na, generator=gg_)[:nv_])[0].to(torch.int32).to(device)
        ep_mlp = [torch.tanh(rr(nv_, Ka)), torch.sigmoid(rr(nv_, Ka * 3)), rr(nv_, Ka * 7), 0.1 * rr(nv_, Ka * 3)]
        lo_, hi_ = torch.zeros(1, 3, device=device), torch.ones(1, 3, device=device)
        for t_ in ep_in[:3] + ep_mlp:
            t_.requires_grad_(True)

        def ep_run(fn, backward, **kw):
            def step():
                o = fn(ep_in[0], ep_in[1], ep_in[2], ep_in[3], ep_vis, ep_mlp[0], ep_mlp[1], ep_mlp[2], ep_mlp[3], lo_, hi_, **kw)
                if backward:
                    torch.autograd.grad(o.xyz.sum() + o.color.sum() + o.opacity.sum() + o.scaling.sum() + o.rot.sum(),
                                        ep_in[:3] + ep_mlp)
                return o
            for _ in range(3):
                step()
            torch.cuda.synchronize(device)
            return min(timed(step, args.steps)[0] for _ in range(2)) / args.steps

        epilogue = {"anchors": Na, "visible": nv_, "n_offsets": Ka,
                    "fused_fwd_ms": ep_run(neural_gaussians_epilogue, False), "torch_fwd_ms": ep_run(reference_epilogue, False, K=Ka),
                    "fused_fwd_bwd_ms": ep_run(neural_gaussians_epilogue, True), "torch_fwd_bwd_ms": ep_run(reference_epilogue, True, K=Ka),
                    "note": "gsvc_b200.generate.neural_gaussians_epilogue (gather by visible index + mask + select + activate, "
                            "3 kernels, count through the pinned slot) vs the reference's PyTorch expression restated in "
                            "generate.reference_epilogue (boolean-mask gathers, repeat / cat / mask-index / split)"}
        del ep_in, ep_mlp

    # ---- forward frames as an independent stream (video decode / evaluation: fixed Gaussians, one frame after the
    # other): graphed.FrameStreamer replays them round-robin on 4 CUDA streams so the binning of frame i+1 runs
    # under the blend of frame i.  Device time for K frames between two synchronisations.
    from gsvc_b200.graphed import FrameStreamer
    streamed_ms = None
    if graphs is not None:
        streamer = FrameStreamer(front, back, params, n_streams=4)
        vf_, vb_ = front.viewmatrix, back.viewmatrix
        for _ in range(8):
            streamer.render(vf_, vb_)
        streamer.synchronize()
        best = None
        for _ in range(REPEATS):
            sync_all()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                streamer.render(vf_, vb_)
            streamer.wait()
            for s_ in streamer.streams:
                torch.cuda.current_stream(device).wait_stream(s_)
            e1.record()
            sync_all()
            t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            best = float(t.item()) if best is None else min(best, float(t.item()))
        if not streamer.capacity_ok():
            raise SystemExit("streamed frames: the captured instance capacity was exceeded")
        streamed_ms = best
        del streamer

    # ---- the reference's own FPS convention (utils/report_utils.py:297-319): per frame, synchronize, time.time(),
    # render front, render back, flip, average, clamp, synchronize — here the two renders are one render_toast call
    ref_style = []
    with torch.no_grad():
        for i in range(args.steps + 5):
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            img, _, _ = rasterize_views(toast, means3D=params["means3D"], opacities=params["opacities"],
                                        colors_precomp=params["colors_precomp"], scales=params["scales"],
                                        rotations=params["rotations"])
            img = torch.clamp(img[0], min=0, max=1.0)
            torch.cuda.synchronize(device)
            if i >= 5:
                ref_style.append(time.perf_counter() - t0)
    ref_style_fps = 1.0 / statistics.median(ref_style)

    # ---- end to end through the public API with HOST buffers (gsvc_b200.hostpipe.HostStepPipeline): every step
    # copies its inputs (all Gaussian parameters, one [14*P] pinned buffer) from host memory and reads its result
    # (the packed [P,14] parameter gradients a host optimizer consumes) back to pinned host memory, inside the
    # timed region.  Copies run on their own streams, ring-buffered over 2 slots, and the copy of step i+1 is
    # enqueued before step i runs.  (The rendered image stays on the device, where the reference computes its
    # loss: pipeline/train.py:407-444.)
    pipe = HostStepPipeline(P, device, slots=2,
                            use_graphs=graphs is not None and os.environ.get("GSVC_E2E_GRAPHS", "1") != "0",
                            sharded=world > 1 and P % world == 0,
                            peer_copies=False if os.environ.get("GSVC_BENCH_NCCL_ALLREDUCE") == "1" else None)
    host_flat = torch.empty(14 * P, dtype=torch.float32).pin_memory()
    off = 0
    for k, w in GRAD_LAYOUT:
        host_flat[off:off + w * P].copy_(g[k].detach().reshape(-1).cpu())
        off += w * P
    h2d, d2h = pipe.h2d_bytes * pipe.world, pipe.d2h_bytes * pipe.world      # all ranks together
    # replicated host state (P not divisible by the world size): every rank copies everything and all-reduces
    reduce = (lambda buf: dist.all_reduce(buf, op=dist.ReduceOp.SUM, async_op=True)) if world > 1 and pipe.world == 1 else None

    def e2e_steps(n):
        pipe.prefetch(host_flat)
        for i in range(n):
            if i + 1 < n:
                pipe.prefetch(host_flat)        # step i+1's copy is in flight while step i computes
            pipe.step(toast, dL, reduce)

    e2e_steps(6)      # per slot: one eager step (sizes the binning buffer), then the CUDA-graph capture

    # the pipeline's fill (first upload + exchange) and drain (last exchange + read-back) are inside the timed region:
    # about 1 % of 100 steps, 5 % of 20
    E2E_STEPS = args.steps

    def e2e_run():
        sync_all()
        e_start = torch.cuda.Event(enable_timing=True)
        e_end = torch.cuda.Event(enable_timing=True)
        e_start.record(pipe.s_h2d)
        e2e_steps(E2E_STEPS)
        e_end.record(pipe.s_d2h)
        sync_all()
        t = torch.tensor([e_start.elapsed_time(e_end)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def copy_gbs(dst, src, stream):
        """PCIe rate of one direction alone, same buffers as the e2e steps (explains the e2e number)."""
        with torch.cuda.stream(stream):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dst.copy_(src, non_blocking=True)
            a.record()
            for _ in range(10):
                dst.copy_(src, non_blocking=True)
            b.record()
        b.synchronize()
        return 10 * src.numel() * 4 / (a.elapsed_time(b) * 1e-3) / 1e9

    e2e_ms = min(e2e_run() for _ in range(REPEATS))
    torch.cuda.synchronize(device)
    if not pipe.capacity_ok(toast):
        raise SystemExit("e2e: the captured instance capacity was exceeded (cannot happen with a fixed scene)")
    pcie = {"h2d_GBs": round(copy_gbs(pipe.dev_flat[0], host_flat, pipe.s_h2d), 2),
            "d2h_GBs": round(copy_gbs(pipe.host_grads[0].view(-1), pipe.dev_grads[0].view(-1), pipe.s_d2h), 2),
            "note": "one direction alone, one rank"}
    # ---- the second native entry point, visible_filter over 1M anchors (prefilter_voxel, preprocess.py:99-104):
    # a pure stream kernel — the one stage whose HBM roofline fraction is meaningful as such
    vf = None
    if rank == 0:
        Pa = 1_000_000
        ga = synthetic_gaussians(Pa, geom, f0, f0, threshold=THRESHOLD, seed=4, device=device)
        _lib.stage_timing(True)
        for _ in range(3):
            rast.visible_filter(means3D=ga["means3D"], scales=ga["scales"], rotations=ga["rotations"], cov3D_precomp=None)
        torch.cuda.synchronize(device)
        _lib.stage_times()
        for _ in range(20):
            flush.zero_()
            rast.visible_filter(means3D=ga["means3D"], scales=ga["scales"], rotations=ga["rotations"], cov3D_precomp=None)
        torch.cuda.synchronize(device)
        vf_ms = _lib.stage_times()["visible_filter"]
        # row f2: the same filter fused with the compaction of the visible indices, against what the reference does
        # next with the mask (radii > 0 -> nonzero, guassian.py:147-153)
        for _ in range(3):     # warm-up: the first launch of a kernel loads it (lazy module loading), inside the timer
            rast.visible_filter_compact(means3D=ga["means3D"], scales=ga["scales"], rotations=ga["rotations"])
        torch.cuda.synchronize(device)
        _lib.stage_times()
        for _ in range(20):
            flush.zero_()
            idx, _r = rast.visible_filter_compact(means3D=ga["means3D"], scales=ga["scales"], rotations=ga["rotations"])
        torch.cuda.synchronize(device)
        vfc_ms = _lib.stage_times()["visible_filter"]
        _lib.stage_timing(False)
        radii_a = rast.visible_filter(means3D=ga["means3D"], scales=ga["scales"], rotations=ga["rotations"], cov3D_precomp=None)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(5):
            nz = torch.nonzero(radii_a > 0)
        torch.cuda.synchronize(device)
        e0.record()
        for _ in range(20):
            nz = torch.nonzero(radii_a > 0)
        e1.record()
        torch.cuda.synchronize(device)
        vf = {"P_anchors": Pa, "ms": vf_ms, "algorithmic_bytes": 44 * Pa, "achieved_GBs": 44 * Pa / (vf_ms * 1e-3) / 1e9,
              "fused_compaction_ms": vfc_ms, "visible": int(idx.numel()),
              "torch_mask_nonzero_ms": e0.elapsed_time(e1) / 20,
              "note": "fused_compaction_ms = filter + ascending visible indices + count in ONE kernel (visible_filter_compact); "
                      "torch_mask_nonzero_ms = what the mask costs the reference AFTER the filter (radii > 0, nonzero with its host sync)"}
        del ga
        # row f4: reference-scale anchors (1M over the WHOLE cube depth, as init_anchor_num x n_offsets gives), kept
        # z-sorted the way the stream codec stores them; the slab's index range comes from its interval table
        from gsvc_b200.frames import slab_index_range, z_interval_table
        gz = synthetic_gaussians(Pa, geom, 0, cfg["F"] - 1, threshold=THRESHOLD, seed=5, device=device)
        order = torch.argsort(gz["means3D"][:, 2], stable=True)
        gz = {k: v[order].contiguous() for k, v in gz.items() if k in ("means3D", "scales", "rotations")}
        table = z_interval_table(gz["means3D"][:, 2])
        rng_idx = slab_index_range(table, geom.z_of(frame_id), THRESHOLD)
        slab = {}
        for name, kw in (("full_scan_ms", {}), ("index_range_ms", {"index_range": rng_idx})):
            _lib.stage_timing(True)
            for _ in range(20):
                flush.zero_()
                rz = rast.visible_filter(means3D=gz["means3D"], scales=gz["scales"], rotations=gz["rotations"],
                                         cov3D_precomp=None, **kw)
            torch.cuda.synchronize(device)
            slab[name] = _lib.stage_times()["visible_filter"]
            _lib.stage_timing(False)
            slab["visible"] = int((rz > 0).sum().item())
        slab.update(P_anchors=Pa, index_range=list(rng_idx),
                    note="anchors over the whole cube depth, z-sorted; index_range = the codec-style interval table's "
                         "range for this frame's slab (the filter reads only those anchors)")
        vf["slab_ordered"] = slab
        del gz
    clk = clocks.stop()

    if rank == 0:
        ms_per_step = total_ms / args.steps
        value = world * NV * 1000.0 / ms_per_step
        peak, peak_src = load_peaks()
        alg = algorithmic_bytes(P, V, num_rendered, N, T, NV)
        # per-launch DRAM traffic and issue utilisation of each kernel from the committed ncu --set full capture of
        # this same command (profiles/traffic.json, made by scripts/ncu_traffic.py); None if it is absent
        prof, prof_note = {}, "profiles/traffic.json absent"
        try:
            from gsvc_b200.build import _digest
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                pj = json.load(f)
            if pj.get("csrc_digest") == _digest():
                prof, prof_note = pj["kernels"], "profiles/traffic.json (ncu --set full of scripts/prof_step.py; digest of the kernel sources matches)"
            else:
                prof_note = "profiles/traffic.json REFUSED: captured from other kernel sources than the library being timed"
        except Exception:
            pass
        dom = max(stage_avg, key=stage_avg.get)
        achieved = alg[dom] / (stage_avg[dom] * 1e-3) / 1e9
        pairs = 256.0 * num_rendered
        per_s = lambda ms, units: world * units * 1000.0 * args.steps / ms
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "P": P, "views_per_step": NV, "V": V, "R": num_rendered, "N": N, "T": T,
                       "frames": f"frame {f0}+rank of F=600, front + back view",
                       "step": "one frame = its front and back view (the reference's (front + flip(back)) / 2, "
                               "pipeline/train.py:353-375) forward + backward in ONE batched kernel chain "
                               "(gsvc_b200.views), replayed from a CUDA graph (gsvc_b200.graphed.GraphedStep); "
                               "V, R count both views; single-view and eager numbers under `single_view`",
                       "graph_fallback": graph_note,
                       "l2": "256 MiB flush between timed steps (outside the per-step events)",
                       "timing": "best of 3 repeats of exactly K steps; per-step CUDA events summed; max over ranks",
                       "step_ms_distribution": step_stats,
                       # the rest of BASELINE.json's table, in a key the driver's record keeps (full dicts below)
                       "baseline_table": {
                           "config2_fwd_frames_per_s": per_s(fwd_ms, 1), "config2_fwd_views_per_s": per_s(fwd_ms, NV),
                           "config2_train_view_iters_per_s": value,
                           "config2_single_view_graph_iters_per_s": per_s(single_ms, 1),
                           "config2_single_view_eager_iters_per_s": per_s(eager_ms, 1),
                           "config2_dropin_eager_variable_P_iters_per_s": None if dropin is None else dropin["iters_per_s"],
                           "config2_dropin_eager_vs_graph": None if dropin is None else dropin["ratio_to_single_view_graph"],
                           "config2_gpu_baseline_iters_per_s": (gpu_baseline or {}).get("value"),
                           "config3_window_ms": None if config3 is None else config3["window_ms"],
                           "config3_view_iters_per_s": None if config3 is None else config3["view_iters_per_s"],
                           "config3_exposed_collective_us": None if config3 is None else config3["exposed_collective_us"],
                           "config4_fwd_frames_per_s_plain": None if config4 is None else config4["plain_calls"]["frames_per_s"],
                           "config4_fwd_frames_per_s_streamed": None if not (config4 and config4["streamed"]) else config4["streamed"]["frames_per_s"],
                           "config5_train_iters_per_s_graph": None if not (config5 and config5["graph"]) else config5["graph"]["iters_per_s"],
                           "config5_train_iters_per_s_eager": None if config5 is None else config5["eager"]["iters_per_s"],
                           "config5_R": None if config5 is None else config5["R"],
                           "f2_epilogue_fused_vs_torch_fwd_bwd_ms": None if epilogue is None else
                           [epilogue["fused_fwd_bwd_ms"], epilogue["torch_fwd_bwd_ms"]]},
                       "parallelism": f"frame-sharded x{world}" + (f", fp32 sum all-reduce of [P,14] grads per step ({allreduce_note})" if world > 1 else "")},
            "fwd_views_per_s": per_s(fwd_ms, NV),
            "fwd_frames_per_s": per_s(fwd_ms, 1),
            "fwd_ms_per_frame": fwd_ms / args.steps,
            "fwd_streamed_frames_per_s": None if streamed_ms is None else {
                "value": per_s(streamed_ms, 1), "views_per_s": per_s(streamed_ms, NV),
                "note": "independent forward frames replayed round-robin on 4 CUDA streams (gsvc_b200.graphed.FrameStreamer): "
                        "the binning kernels of frame i+1 run under the blend of frame i; no L2 flush between frames"},
            "ref_iterations_per_s": per_s(total_ms, 1) / 2.0,
            "ref_style_eval_fps": {"value": ref_style_fps, "unit": "frames/s per GPU",
                                   "note": "the reference's evaluate() convention (utils/report_utils.py:297-319): wall "
                                           "clock around synchronize / 2 views + flip + average + clamp / synchronize, "
                                           "eager launches, median over K frames"},
            "single_view": {
                "graph": {"iters_per_s": per_s(single_ms, 1), "ms_per_step": single_ms / args.steps,
                          "fwd_views_per_s": per_s(single_fwd_ms, 1)},
                "eager": {"iters_per_s": per_s(eager_ms, 1), "ms_per_step": eager_ms / args.steps,
                          "fwd_views_per_s": per_s(eager_fwd_ms, 1)},
                "note": "one GaussianRasterizer call = one view (no all-reduce): replayed from a CUDA graph, and "
                        "called eagerly through autograd (one host wait per forward for num_rendered)"},
            "generator_epilogue": epilogue, "dropin_eager": dropin, "gpu_baseline": gpu_baseline, "config3": config3, "config4": config4, "config5": config5,
            "step_ms_distribution": step_stats,
            "ms_per_step_with_stage_events": staged_ms / args.steps,
            "stage_ms": {k: round(v, 5) for k, v in stage_avg.items()},
            "fwd_stage_ms": {k: round(v, 5) for k, v in fwd_stage_avg.items()},
            "pairs_per_s_fwd": pairs / (fwd_stage_avg["render_forward"] * 1e-3),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": prof.get(dom, {}).get("dram_bytes"), "traffic_source": prof_note,
                         "peak_source": peak_src,
                         "ncu_issue_active_pct": prof.get(dom, {}).get("issue_active_pct"),
                         "algorithmic_bytes": alg[dom],
                         "note": "blend kernels are FP32/issue-bound by construction (256 pixel-Gaussian pairs per 40 B "
                                 "instance; ncu: ~84 % issue-active, < 5 % DRAM); the HBM fraction of a stream kernel of "
                                 "this path is reported under visible_filter; see DESIGN.md §4"},
            # what actually bounds the dominant kernel: issued warp-instructions per second against the SMs' issue rate
            # (4 schedulers x 1 instruction per clock per SM); instruction count per launch from the committed ncu capture
            "issue_roofline": (lambda inst: None if not inst else {
                "kernel": dom, "warp_instructions_per_launch": inst, "source": "profiles/traffic.json (ncu smsp__inst_executed.sum)",
                "achieved_Ginstr_per_s": inst / (stage_avg[dom] * 1e-3) / 1e9,
                "peak_Ginstr_per_s": 148 * 4 * (clk.get("sm_mhz") or 1965.0) * 1e6 / 1e9,
                "frac": inst / (stage_avg[dom] * 1e-3) / (148 * 4 * (clk.get("sm_mhz") or 1965.0) * 1e6)})(
                    prof.get(dom, {}).get("inst_executed")),
            "e2e": {"value": world * NV * 1000.0 * E2E_STEPS / e2e_ms, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / E2E_STEPS, "steps": E2E_STEPS, "pcie_alone": pcie,
                    "host_state": ("sharded by rows over the ranks: each rank uploads 1/N of the parameters (the other rows "
                                   "come over NVLink) and reads back 1/N of the summed gradients; the byte counts are the N "
                                   "ranks together; exchange: " + ("copy-engine pulls over symmetric memory between signal-pad "
                                   "barriers (no collective kernel)" if pipe.peer is not None else "NCCL all-gather / reduce-scatter")
                                   ) if pipe.world > 1 else "one rank, everything",
                    "api": "gsvc_b200.hostpipe.HostStepPipeline (pinned host params in, pinned host [P,14] grads out; "
                           + ("the frame's forward+backward replayed from a CUDA graph per slot)" if pipe.use_graphs else "eager launches)")},
            "visible_filter": dict(vf, frac=vf["achieved_GBs"] / peak),
            "gpu_launches": launches,
            "clocks": clk,
        }
        if world == 1 and not args.no_cpu_baseline:
            from oracle import c_oracle
            cores = c_oracle.set_threads(os.cpu_count() or 1)
            g_np = {k: v.detach().cpu().numpy() for k, v in g.items()}
            cpu_step(geom, f0, g_np)                                        # warm-up (pages in, builds nothing)
            reps = [cpu_step(geom, f0, g_np) for _ in range(30)]
            best = min(r[1] for r in reps)
            line["cpu_baseline"] = {
                "value": 1.0 / best, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": (f"C oracle (oracle/splat_oracle.c, OpenMP, {cores} host threads), same scene, ONE view "
                           f"forward+backward over all {P} Gaussians and every pixel: best of 30 whole "
                           f"view-iterations, {best:.2f} s each ({sum(r[1] for r in reps):.0f} s of CPU-side work)")}
        if last_outputs is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in last_outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_JSON_OUT = None


def _claim_stdout():
    """stdout carries exactly ONE line, the JSON: everything else that writes to file descriptor 1 (NCCL's version
    banner, library chatter) is sent to stderr, and the JSON line goes to a private duplicate of the original fd."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="gsvc", choices=["gsvc", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed step returned in its last step (image, radii, packed [P,14] gradients, "
                         "instance count) as DIR/<name>.npy, float32 / float64, about 38 MB; the inputs are seeded")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "gsvc":
        ap.error("--dump-outputs writes the outputs of the product arm (--impl gsvc)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    run_product_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
