#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json: warp+loss fwd/bwd Mpixel/s and
HBM GB/s vs peak) on N GPUs of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload c2|c1|c3|c4|c5] [--batch B] [--no-sweep] [--dump-outputs DIR] ...
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic input; the timed region is exactly --steps steps.
`--dump-outputs DIR` writes what the last timed step computed (c4: the frames and label maps of the rollout; otherwise
the loss vector and the gradients to flow, src_rgb and src_layout) as DIR/<name>.npy.  Workloads = BASELINE.json configs:
  c2 (default)  16x256x512, K=20, fp32: flow-guided warp of RGB + layout, all loss terms, gradients to flow, src_rgb and
                src_layout (220 algorithmic B/px).  Weak scaling: every rank processes one such batch; the only exchange
                is one NCCL all-reduce of the 8-float loss vector.
  c1            2x128x256 (the reference's CPU-runnable case; L2-resident, launch-bound)
  c3            8x1024x2048 bf16 (122 B/px)
  c4            5-step autoregressive rollout at 512x1024, GLOBAL batch 32 split over the ranks (strong scaling),
                label layouts fed back (48 B/px per step)
  c5            Bx375x1242, sigma = 48 px + 5 % outliers (large displacement); --batch B, default 16

Prints ONE JSON line (rank 0).  `value` is device-resident throughput, `e2e` goes through the public module API from
pinned host buffers holding what the dataset holds (uint8 frames and class maps, fp32 flow), `roofline` is the
longest kernel of the step timed by CUDA events on its launch stream against MEASURED_PEAKS.json, `cpu_baseline` is
the oracle port on the host cores, `sweep` carries the other BASELINE configs (C3, C4, C5 batch sweep) in compact form.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: (N, H, W, K, flow sigma px, far fraction, dtype)
    "c1": (2, 128, 256, 20, 4.0, 0.0, "f32"),
    "c2": (16, 256, 512, 20, 4.0, 0.0, "f32"),
    "c2calm": (16, 256, 512, 20, 0.5, 0.0, "f32"),    # tuning: same shape, flow so small that no tap leaves the staged windows
    "c2q": (4, 256, 512, 20, 4.0, 0.0, "f32"),        # tuning: a quarter of c2 (pass 1's staging, 54 MB, stays in the L2 for pass 2)
    "c3": (8, 1024, 2048, 20, 4.0, 0.0, "bf16"),
    "c4": (32, 512, 1024, 20, 4.0, 0.0, "f32"),       # rollout: GLOBAL batch, 5 steps
    "c5": (16, 375, 1242, 20, 48.0, 0.05, "f32"),
}
ROLLOUT_STEPS = 5
# algorithmic bytes per output pixel (SURVEY.md 8d; DESIGN.md section 4): each input element read once, each required
# output written once.  Per kernel: rgb strip = coords 8 + src_rgb 12 + tgt_rgb 12; layout tile = src_layout 80 + label 8
# + d_flow 8; pass 2 = d_src_rgb 12 + d_src_layout 80 (bf16: activations and their gradients halve).
BYTES_PER_PX = {"f32": dict(step=220, pass1=128, rgb_strip=32, lay_tile=96, pass2=92),
                "bf16": dict(step=122, pass1=76, rgb_strip=20, lay_tile=56, pass2=46)}
ROLLOUT_BYTES_PER_PX = 48      # per rollout step: coords 8 + rgb 12 + label 8 read, rgb 12 + label 8 written
FALLBACK_HBM_GBS = 6650.0
WARM_MS = 250.0                # untimed passes right before every timed region
REF_SAMPLE_IMAGES = 2          # bounded sample of the CPU arms (cpu_baseline and --impl reference alike)
DUMP_LIMIT_BYTES = 64 * 10**6  # --dump-outputs: all files together
DUMP_SEED = 1024


def make_inputs(N, H, W, K, sigma, far, dtype, device, seed=1024):
    """Synthetic Cityscapes-shaped batch (SURVEY.md 8d): normalised RGB, block-constant one-hot
    layouts, block-constant int64 labels, box-smoothed Gaussian flow."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    mean = torch.tensor([0.485, 0.456, 0.406])[None, :, None, None]
    std = torch.tensor([0.229, 0.224, 0.225])[None, :, None, None]
    src_rgb = (torch.rand(N, 3, H, W, generator=g) - mean) / std
    tgt_rgb = (torch.rand(N, 3, H, W, generator=g) - mean) / std
    blk = 32

    def labels():
        l = torch.randint(0, K, (N, (H + blk - 1) // blk, (W + blk - 1) // blk), generator=g)
        return l.repeat_interleave(blk, 1).repeat_interleave(blk, 2)[:, :H, :W].contiguous()

    lab_src, lab_tgt = labels(), labels()
    src_layout = torch.zeros(N, K, H, W).scatter_(1, lab_src[:, None], 1.0)
    flow = torch.randn(N, 2, H, W, generator=g) * sigma
    flow = torch.nn.functional.avg_pool2d(torch.nn.functional.pad(flow, (4, 4, 4, 4), mode="replicate"), 9, 1)
    if far > 0:
        m = torch.rand(N, 1, H, W, generator=g) < far
        flow = torch.where(m, (torch.rand(N, 2, H, W, generator=g) - 0.5) * 2 * max(H, W), flow)
    flow = flow.permute(0, 2, 3, 1).contiguous()
    tdt = torch.float32 if dtype == "f32" else torch.bfloat16
    out = dict(src_rgb=src_rgb.to(tdt), src_layout=src_layout.to(tdt), flow=flow, tgt_rgb=tgt_rgb.to(tdt),
               tgt_label=lab_tgt)
    if device is not None:
        cl = lambda t: t.to(device).contiguous(memory_format=torch.channels_last)
        out = dict(src_rgb=cl(out["src_rgb"]), src_layout=cl(out["src_layout"]), flow=flow.to(device),
                   tgt_rgb=cl(out["tgt_rgb"]), tgt_label=lab_tgt.to(device))
    return out


def make_inputs_tiled(N, H, W, K, sigma, far, dtype, device, seed):
    """Batches larger than 16 are the 16-image synthetic batch repeated with rolled sample order (the host-side
    generator is the slow part; throughput does not depend on which samples repeat)."""
    base = make_inputs(min(N, 16), H, W, K, sigma, far, dtype, device, seed)
    if N <= 16:
        return base
    reps = (N + 15) // 16
    out = {}
    for k, v in base.items():
        t = torch.cat([v.roll(r, 0) for r in range(reps)], 0)[:N]
        out[k] = t.contiguous(memory_format=torch.channels_last) if k in ("src_rgb", "tgt_rgb", "src_layout") else t.contiguous()
    return out


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def wait_first(self, timeout=3.0):
        """nvidia-smi takes a moment to start: do not begin the timed region before its first sample."""
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.01)
        self.rows.clear()      # samples from before the timed region do not count

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arms
def cpu_oracle_run(wl, N, steps, warmup):
    """The reference's own CPU implementation of the path: it is pure Python / PyTorch with no compiled code of its
    own, so this is the oracle port (oracle/torch_oracle.py) on the host cores, all threads.  One step = fwd+bwd
    (rollout: 5 warps with argmax feedback) on a bounded sample of REF_SAMPLE_IMAGES images of the workload.
    Returns (Mpixel/s, mean seconds per step, description)."""
    from oracle import torch_oracle as TO
    _, H, W, K, sigma, far, dtype = WORKLOADS[wl]
    n_sample = min(N, REF_SAMPLE_IMAGES)
    d = make_inputs(n_sample, H, W, K, sigma, far, "f32", None)
    if wl == "c4":
        flows = [make_inputs(n_sample, H, W, K, sigma, 0.0, "f32", None, seed=78 + t)["flow"] for t in range(ROLLOUT_STEPS)]
        lab0 = d["src_layout"].argmax(1)

        def one():
            img, lab = d["src_rgb"], lab0
            with torch.no_grad():
                for t in range(ROLLOUT_STEPS):
                    grid = TO.flow_to_grid(flows[t])
                    img = TO.warp(img, grid)
                    lab = TO.warp(TO.one_hot_layout(lab, K), grid).argmax(1)     # src/trainer.py:461,467
            return lab
        px = n_sample * H * W * ROLLOUT_STEPS
        what = f"{n_sample}x{H}x{W} x{ROLLOUT_STEPS} rollout steps (dense one-hot feedback, src/trainer.py:460-469)"
    else:
        def one():
            return TO.warp_loss_fwd_bwd(d["src_rgb"], d["src_layout"], d["flow"], d["tgt_rgb"], d["tgt_label"], w_tv=0.5)
        px = n_sample * H * W
        what = f"{n_sample}x{H}x{W} slice of the batch, fwd+bwd (grads to flow, src_rgb, src_layout)"
    ts = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        one()
        if i >= warmup:
            ts.append(time.perf_counter() - t0)
    t = sum(ts) / len(ts)
    return px / t / 1e6, t, f"{what}; torch CPU oracle port, mean of {len(ts)} after {warmup} warm-up ({t * 1e3:.0f} ms/step)"


def workload_config(wl, N, world, dtype, with_src=True):
    _, H, W, K, _, _, _ = WORKLOADS[wl]
    if wl == "c4":
        return {"workload": f"c4: {ROLLOUT_STEPS}-step autoregressive rollout at {H}x{W}, global batch {N}, K={K} {dtype}, label layouts fed back",
                "global_batch": N, "parallelism": f"dp{world}"}
    return {"workload": f"{wl}: {N}x{H}x{W} K={K} {dtype} warp+loss fwd+bwd per GPU" + ("" if with_src else " (flow-grad only)"),
            "per_gpu_pixels": N * H * W, "grads": "flow,src_rgb,src_layout" if with_src else "flow", "parallelism": f"dp{world}"}


def run_reference(args, rank, world):
    """`--impl reference`: rank 0 alone runs the CPU arm on the same workload description as our arm."""
    if rank != 0:
        return
    try:   # torchrun exports OMP_NUM_THREADS=1; the reference arm uses every host thread it may
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except Exception:
        pass
    N0, H, W, K, sigma, far, dtype = WORKLOADS[args.workload]
    N = args.batch or N0
    val, t, sample = cpu_oracle_run(args.workload, N, args.steps, max(args.warmup, 1))
    print(json.dumps({
        "impl": "reference", "metric": "warp+loss fwd/bwd throughput", "value": val, "unit": "Mpixel/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": t * 1e3,
        "higher_is_better": True, "scaling": "strong" if args.workload == "c4" else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args.workload, N, world, dtype, not args.flow_grad_only),
        "cpu_baseline": {"value": val, "unit": "Mpixel/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ----------------------------------------------------------------------------------------------- GPU arm
class Ctx:
    """Process-wide handles of the GPU arm."""

    def __init__(self):
        import vlg_b200
        from vlg_b200 import _cabi, ops
        self.vlg, self.cabi, self.ops = vlg_b200, _cabi, ops
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group(backend="nccl", device_id=self.dev)
            self.dist = dist
        self.lib = _cabi.load()
        self.stream = torch.cuda.current_stream()

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        t = torch.tensor([ms], dtype=torch.float64, device=self.dev)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def timed(self, step, steps, min_ms=0.0):
        """EXACTLY `steps` step groups of `r` passes each, ending in a barrier + synchronize; `r` is 1 unless `min_ms` > 0,
        then it is chosen so that the region lasts >= min_ms.  Right before the region, WARM_MS of passes bring the clocks
        back up after whatever idle gap preceded the call, so that a short region is not timed at idle clocks.  Returns
        (ms per pass, max over ranks; r; ms of the whole region)."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record(self.stream)
        for i in range(4):
            step(i)
        e1.record(self.stream)
        self.barrier()
        est_ms = max(self.max_over_ranks(e0.elapsed_time(e1) / 4), 1e-6)
        r = max(1, int(math.ceil(min_ms / (est_ms * steps))))
        for i in range(int(math.ceil(WARM_MS / est_ms))):
            step(i)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # ranks start the region together; a single process leaves the warm-up queued ahead of e0 instead, so that the
        # GPU does not idle for a launch between e0 and the first timed pass (a visible share of a region of a few steps)
        if self.dist is not None:
            self.barrier()
        e0.record(self.stream)
        for i in range(steps * r):
            step(i)
        e1.record(self.stream)
        self.barrier()
        total = self.max_over_ranks(e0.elapsed_time(e1))
        return total / (steps * r), r, total


class Fused:
    """Device-resident fused warp+loss step of one workload: two alternating input sets (no step re-reads lines its
    predecessor left in L2), gradient buffers, workspace, CUDA graphs of the launch sequence."""

    def __init__(self, cx: Ctx, wl, N, with_src=True, use_graph=True, seed=1024):
        _, H, W, K, sigma, far, dtype = WORKLOADS[wl]
        self.cx, self.wl, self.N, self.H, self.W, self.K, self.dtype = cx, wl, N, H, W, K, dtype
        self.P = N * H * W
        self.with_src = with_src
        ops, cabi = cx.ops, cx.cabi
        tdt = torch.float32 if dtype == "f32" else torch.bfloat16
        self.tdt = tdt
        n_sets = 2 if self.P * 120 < 3e9 else 1       # large batches exceed the L2 many times over by themselves
        self.sets = [make_inputs_tiled(N, H, W, K, sigma, far, dtype, cx.dev, seed=seed + 7 * cx.rank + s) for s in range(n_sets)]
        cfg = ops.WarpLossConfig(w_tv=0.5)
        self.prob = ops._problem(N, H, W, K, tdt, cfg)
        self.ws = ops._workspace(self.prob, with_src, cx.dev, cached=False)
        self.loss = torch.zeros(cabi.LOSS_SLOTS, dtype=torch.float32, device=cx.dev)
        self.d_c = torch.empty(N, H, W, 2, dtype=torch.float32, device=cx.dev)
        self.d_a = ops.empty_nhwc((N, 3, H, W), tdt, cx.dev) if with_src else None
        self.d_b = ops.empty_nhwc((N, K, H, W), tdt, cx.dev) if with_src else None
        self.graphs = None
        self.launches_per_step = None
        for i in range(3):
            self.step(i)
        cx.barrier()
        if use_graph:
            self._capture()

    # ---- launch sequences through the C ABI
    def _sp(self):
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def launch_fused(self, s, sp):
        ptr, lib, ops = self.cx.ops._ptr, self.cx.lib, self.cx.ops
        ops.check(lib.vlg_warp_loss_fwd_bwd(C.byref(self.prob), ptr(s["src_rgb"]), ptr(s["src_layout"]), ptr(s["flow"]),
                                            ptr(s["tgt_rgb"]), ptr(s["tgt_label"]), ptr(self.loss), ptr(self.d_c), ptr(self.d_a),
                                            ptr(self.d_b), None, ptr(self.ws), self.ws.numel(), sp))

    def launch_pass1(self, s, sp):
        ptr, lib, ops = self.cx.ops._ptr, self.cx.lib, self.cx.ops
        ops.check(lib.vlg_warp_loss_pass1(C.byref(self.prob), ptr(s["src_rgb"]), ptr(s["src_layout"]), ptr(s["flow"]),
                                          ptr(s["tgt_rgb"]), ptr(s["tgt_label"]), ptr(self.loss), ptr(self.d_c), None,
                                          int(self.with_src), ptr(self.ws), self.ws.numel(), sp))

    def launch_pass2(self, s, sp):
        if self.with_src:
            ptr, lib, ops = self.cx.ops._ptr, self.cx.lib, self.cx.ops
            ops.check(lib.vlg_warp_bwd_src(C.byref(self.prob), ptr(s["flow"]), ptr(self.d_a), ptr(self.d_b), ptr(self.ws),
                                           self.ws.numel(), sp))

    def _capture(self):
        cx = self.cx
        try:
            n_before = cx.vlg.launch_count()
            gs = []
            for s in self.sets:
                if cx.dist is None:
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        self.launch_fused(s, self._sp())
                    gs.append(g)
                else:   # two graphs per input set: the all-reduce is issued between them
                    g1, g2 = torch.cuda.CUDAGraph(), None
                    with torch.cuda.graph(g1):
                        self.launch_pass1(s, self._sp())
                    if self.with_src:          # sources as data: there is no pass 2 (an empty capture only earns a warning)
                        g2 = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g2):
                            self.launch_pass2(s, self._sp())
                    gs.append((g1, g2))
            self.launches_per_step = (cx.vlg.launch_count() - n_before) // len(self.sets)
            self.graphs = gs
            for i in range(4):
                self.step(i)
            cx.barrier()
        except Exception as exc:   # capture unsupported: plain launches
            print(f"[bench] CUDA graph capture failed ({exc}); using plain launches", file=sys.stderr)
            self.graphs = None

    def step(self, i):
        """One pass of the hot path (the last pass-1 CTA reduces the loss vector).  Data parallel: the loss vector is
        complete after pass 1, so the path's only exchange -- one all-reduce of 8 floats -- is issued there and
        overlaps pass 2."""
        cx = self.cx
        k = i % len(self.sets)
        s = self.sets[k]
        sp = C.c_void_p(cx.stream.cuda_stream)
        if cx.dist is not None:
            if self.graphs is not None: self.graphs[k][0].replay()
            else: self.launch_pass1(s, sp)
            work = cx.dist.all_reduce(self.loss, async_op=True)
            if self.graphs is not None:
                if self.graphs[k][1] is not None: self.graphs[k][1].replay()
            else: self.launch_pass2(s, sp)
            work.wait()
        elif self.graphs is not None:
            self.graphs[k].replay()
        else:
            self.launch_fused(s, sp)

    def count_launches(self, n_steps):
        if self.graphs is not None:
            return self.launches_per_step * n_steps     # replayed from the graph: the host counter does not move
        n0 = self.cx.vlg.launch_count()
        self.step(0)
        torch.cuda.synchronize()
        return (self.cx.vlg.launch_count() - n0) * n_steps

    def kernel_times(self, reps=20):
        """Median device time of the three main kernels inside the real (direct) launch sequence: CUDA events recorded
        by the library on the launch stream right around each kernel (vlg_timeline_arm / vlg_timeline_read)."""
        cx = self.cx
        sp = C.c_void_p(cx.stream.cuda_stream)
        rows = []
        ms4 = (C.c_float * 4)()
        cx.barrier()
        for i in range(reps):
            cx.ops.check(cx.lib.vlg_timeline_arm(1))
            self.launch_fused(self.sets[i % len(self.sets)], sp)
            cx.ops.check(cx.lib.vlg_timeline_arm(0))
            cx.ops.check(cx.lib.vlg_timeline_read(ms4))
            rows.append(list(ms4))
        med = lambda j: sorted(r[j] for r in rows)[len(rows) // 2]
        return {"rgb_strip_kernel": med(0), "lay_tile_kernel": med(1), "pass2_rec_kernel": med(2), "span_first_to_last": med(3)}

    def cupti_table(self, n=10):
        try:
            from torch.profiler import profile, ProfilerActivity
            sp = C.c_void_p(self.cx.stream.cuda_stream)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for i in range(n):
                    self.launch_fused(self.sets[i % len(self.sets)], sp)
                torch.cuda.synchronize()
            return {e.key.split("(")[0].replace("void ", "").replace("vlg::", ""): round(e.device_time_total / n, 2)
                    for e in prof.key_averages() if e.device_time_total > 0}
        except Exception as exc:   # profiler unavailable: the event timings stand on their own
            return {"unavailable": str(exc)}

    def free(self):
        self.graphs = None
        self.sets = None
        self.ws = self.d_a = self.d_b = self.d_c = None
        torch.cuda.empty_cache()


def u8_host_inputs(d, K):
    """What the reference's dataset holds for one batch (src/folder.py:85-104): uint8 RGB frames [N,H,W,3], uint8
    class maps [N,H,W]; plus the fp32 flow the op consumes.  16 bytes per pixel."""
    mean = torch.tensor([0.485, 0.456, 0.406], device=d["src_rgb"].device)[None, :, None, None]
    std = torch.tensor([0.229, 0.224, 0.225], device=d["src_rgb"].device)[None, :, None, None]
    to_u8 = lambda x: ((x.float() * std + mean) * 255.0).round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()
    host = {
        "src_u8": to_u8(d["src_rgb"]), "tgt_u8": to_u8(d["tgt_rgb"]),
        "src_seg_u8": d["src_layout"].argmax(1).to(torch.uint8), "tgt_seg_u8": d["tgt_label"].to(torch.uint8),
        "flow": d["flow"],
    }
    return {k: v.cpu().pin_memory() for k, v in host.items()}


def e2e_fused(cx: Ctx, fz: Fused, steps, flow_from_host=False, captured=True):
    """End to end through the public API (vlg_b200.ingest + vlg_b200.WarpLoss + backward) from pinned host memory.
    Every step uploads one full input set -- what the dataset holds: uint8 frames and class maps -- and reads the
    step's loss vector back.  Double-buffered: the inputs of step i+1 travel on a copy stream while step i computes
    (what a DataLoader prefetcher does).  The flow is NOT part of the dataset: in the reference's step it is the
    network's output (src/trainer.py:183-210: frames and class maps are uploaded, the network computes its output from them) and never exists on the host, so it
    is device-resident here (two alternating flow fields); `flow_from_host=True` uploads it as well (the round-1/2
    figure, kept as `flow_uploaded` for comparison).

    `captured=True`: the step's device work -- the SAME public calls: ingest x2, WarpLoss, backward() -- is recorded once
    per input buffer set with `vlg_b200.CapturedStep` (torch.cuda.graph whole-step capture, the package's utility for
    static shapes) and replayed; uploads, the replay and the loss read-back still happen every step.  `captured=False`
    issues the calls eagerly every step (bound by ~0.45 ms of host time per step)."""
    vlg, dev, stream = cx.vlg, cx.dev, cx.stream
    host = u8_host_inputs(fz.sets[0], fz.K)
    if not flow_from_host:
        del host["flow"]
    dev_flow = [fz.sets[q % len(fz.sets)]["flow"] for q in range(2)]
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    crit = vlg.WarpLoss(weights=(40.0, 20.0, 10.0, 0.5))
    copy_stream = torch.cuda.Stream(device=dev)
    dbuf = [{k: torch.empty_like(v, device=dev) for k, v in host.items()} for _ in range(2)]
    up_done = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def upload(j):
        copy_stream.wait_event(consumed[j])      # the step that read this buffer set has finished with it
        with torch.cuda.stream(copy_stream):
            for k, v in host.items():
                dbuf[j][k].copy_(v, non_blocking=True)
            up_done[j].record(copy_stream)

    # results travel back the same way the inputs arrive: the loss vector of step i is copied into pinned host memory
    # right behind its kernels and the host looks at it while step i+1 runs (one step in flight in each direction)
    res_host = [torch.empty(cx.cabi.LOSS_SLOTS, dtype=torch.float32).pin_memory() for _ in range(2)]
    res_done = [torch.cuda.Event(), torch.cuda.Event()]
    seen = []

    def device_step(j):
        """The step's device work on buffer set j, through the public API; returns the loss vector."""
        cur = dbuf[j]
        src = vlg.ingest(cur["src_u8"], cur["src_seg_u8"], n_classes=fz.K, dtype=fz.tdt, want_label=False, want_one_hot=True)
        tgt = vlg.ingest(cur["tgt_u8"], cur["tgt_seg_u8"], n_classes=fz.K, dtype=fz.tdt, want_label=True)
        a = src["frames"].requires_grad_(fz.with_src)
        b = src["one_hot"].requires_grad_(fz.with_src)
        f = (cur["flow"] if flow_from_host else dev_flow[j]).detach().requires_grad_(True)
        total = crit(a, b, f, tgt["frames"], tgt["label"])
        total.backward()
        return crit.last_terms

    mode = "eager"
    run_step = device_step
    if captured:
        try:
            for j in range(2):                  # the buffers hold valid data before anything is recorded
                for k, v in host.items():
                    dbuf[j][k].copy_(v)
            torch.cuda.synchronize()
            graphs = [vlg.CapturedStep(lambda j=j: device_step(j)) for j in range(2)]
            run_step = lambda j: graphs[j]()
            mode = "captured"
        except Exception as exc:               # capture unsupported here: the eager call sequence
            print(f"[bench] whole-step capture failed ({exc}); e2e runs eagerly", file=sys.stderr)
            torch.cuda.synchronize()

    def e2e_step(i):
        j = i & 1
        upload(j ^ 1)                      # inputs of the NEXT step
        stream.wait_event(up_done[j])
        terms = run_step(j)
        consumed[j].record(stream)
        res_host[j].copy_(terms, non_blocking=True)               # device -> host read of the step's result
        res_done[j].record(stream)
        if i > 0:                          # the previous step's result has landed by now (or is waited for here)
            res_done[j ^ 1].synchronize()
            seen.append(float(res_host[j ^ 1][cx.cabi.LOSS_TOTAL]))

    def drain(i_last):
        res_done[i_last & 1].synchronize()
        seen.append(float(res_host[i_last & 1][cx.cabi.LOSS_TOTAL]))

    for j in range(2):
        consumed[j].record(stream)
    upload(0)
    for i in range(4):
        e2e_step(i)
    drain(3)
    cx.barrier()
    n = max(4, min(steps, 20)) & ~1
    seen.clear()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(n):
        e2e_step(i)
    drain(n - 1)
    e1.record(stream)
    cx.barrier()
    assert len(seen) == n and all(math.isfinite(v) for v in seen), "every step's result must have reached the host"
    ms = cx.max_over_ranks(e0.elapsed_time(e1) / n)
    return {"value": cx.world * fz.P / (ms * 1e-3) / 1e6, "unit": "Mpixel/s", "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": cx.cabi.LOSS_SLOTS * 4, "ms_per_step": ms, "steps": n,
            "launch": {"captured": "the step's public calls (vlg_b200.ingest x2, WarpLoss, backward) recorded once per buffer set with "
                                   "vlg_b200.CapturedStep and replayed every step",
                       "eager": "the step's public calls issued from Python every step"}[mode],
            "inputs": "pinned host, what the dataset holds (src/folder.py:85-104): uint8 RGB frames [N,H,W,3] x2, uint8 class maps "
                      "[N,H,W] x2" + (", and the fp32 flow = 16 B/px" if flow_from_host else " = 8 B/px; the flow is the network's output in "
                      "the reference's step (src/trainer.py:183-210) and stays on the device") + "; on the device vlg_ingest turns them into normalised NHWC frames, int64 "
                      "labels and the one-hot source layout (ToTensor + renorm + one_hot, bit-identical), then WarpLoss + "
                      "backward; the loss vector of every step is copied back to pinned host memory and read there one step later; "
                      "double-buffered uploads on a copy stream"}


class Rollout:
    """BASELINE config 4: 5 autoregressive steps with LABEL layout sources fed back (vlg_warp_fwd_labels),
    per-rank batch = global batch / world (the rollout of a sample is independent of every other sample)."""

    def __init__(self, cx: Ctx, n_rank, seed=77):
        _, H, W, K, sigma, _, _ = WORKLOADS["c4"]
        self.cx, self.n, self.H, self.W, self.K = cx, n_rank, H, W, K
        d = make_inputs_tiled(n_rank, H, W, K, sigma, 0.0, "f32", cx.dev, seed=seed + cx.rank)
        self.img = d["src_rgb"]
        self.lab = d["src_layout"].argmax(1)
        self.flows = [make_inputs_tiled(min(n_rank, 4), H, W, K, sigma, 0.0, "f32", cx.dev, seed=seed + 1 + t)["flow"] for t in range(ROLLOUT_STEPS)]
        if n_rank > 4:   # flows of larger per-rank batches: the 4-image flow set repeated (throughput does not depend on it)
            self.flows = [torch.cat([f.roll(r, 0) for r in range((n_rank + 3) // 4)], 0)[:n_rank].contiguous() for f in self.flows]
        self.px_steps = n_rank * H * W * ROLLOUT_STEPS
        del d

    def step(self, i=0):
        """One rollout; its (frames, label maps) stay in `self.out` until the next one."""
        self.out = self.cx.vlg.rollout(self.img, self.lab, lambda t, im, lb: self.flows[t], steps=ROLLOUT_STEPS)
        return self.out

    def e2e(self, steps):
        """Uploads the uint8 start frame + class map and the five fp32 flows, rolls out, reads the final class map back
        as uint8."""
        cx = self.cx
        mean = torch.tensor([0.485, 0.456, 0.406], device=cx.dev)[None, :, None, None]
        std = torch.tensor([0.229, 0.224, 0.225], device=cx.dev)[None, :, None, None]
        host = {"img_u8": ((self.img * std + mean) * 255).round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous().cpu().pin_memory(),
                "seg_u8": self.lab.to(torch.uint8).cpu().pin_memory()}
        for t in range(ROLLOUT_STEPS):
            host[f"flow{t}"] = self.flows[t].cpu().pin_memory()
        h2d = sum(v.numel() * v.element_size() for v in host.values())
        buf = {k: torch.empty_like(v, device=cx.dev) for k, v in host.items()}
        out_host = torch.empty(self.n, self.H, self.W, dtype=torch.uint8).pin_memory()

        def one():
            for k, v in host.items():
                buf[k].copy_(v, non_blocking=True)
            ing = cx.vlg.ingest(buf["img_u8"], buf["seg_u8"], n_classes=self.K, want_label=True)
            _, labs = cx.vlg.rollout(ing["frames"], ing["label"], lambda t, im, lb: buf[f"flow{t}"], steps=ROLLOUT_STEPS)
            out_host.copy_(labs[-1].to(torch.uint8), non_blocking=True)
            torch.cuda.synchronize()
        for _ in range(2):
            one()
        cx.barrier()
        n = max(2, min(steps, 6))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(cx.stream)
        for _ in range(n):
            one()
        e1.record(cx.stream)
        cx.barrier()
        ms = cx.max_over_ranks(e0.elapsed_time(e1) / n)
        return {"value": cx.world * self.px_steps / (ms * 1e-3) / 1e6, "unit": "Mpixel/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": out_host.numel(), "ms_per_step": ms, "steps": n,
                "inputs": "pinned host: uint8 start frame + class map, five fp32 flows; vlg_ingest + 5 x vlg_warp_fwd_labels; the final "
                          "class map is read back as uint8"}


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return json.load(open(path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth, burst)"
    return FALLBACK_HBM_GBS, "fallback 6.65 TB/s (B200_PROFILING.md)"


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel` on the c2 workload, from the committed
    `ncu --set full` capture (newest profiles/rNN_ncu_traffic.json)."""
    pdir = os.path.join(ROOT, "profiles")
    cands = sorted(f for f in os.listdir(pdir) if f.endswith("_ncu_traffic.json")) if os.path.isdir(pdir) else []
    for f in reversed(cands):
        k = json.load(open(os.path.join(pdir, f))).get("kernels", {}).get(kernel)
        if k:
            return k["dram_bytes_read"] + k["dram_bytes_write"], f
    return None, None


def sweep_entry(cx, wl, N, steps, peak, note=None):
    """Compact line of another BASELINE config: device-resident step time + fraction of its own HBM roofline."""
    _, H, W, K, _, _, dtype = WORKLOADS[wl]
    try:
        fz = Fused(cx, wl, N, with_src=True)
        ms, r, total = cx.timed(fz.step, steps, min_ms=120.0)
        kt = fz.kernel_times(reps=5) if cx.world == 1 else None
        bpp = BYTES_PER_PX[dtype]["step"]
        out = {"workload": f"{wl}: {N}x{H}x{W} {dtype} fwd+bwd per GPU", "batch": N, "ms_per_step": ms,
               "Mpixel_per_s": cx.world * fz.P / (ms * 1e-3) / 1e6, "algorithmic_bytes_per_px": bpp,
               "frac_of_hbm_roofline": fz.P * bpp / (ms * 1e-3) / 1e9 / peak, "timed_ms": total, "kernel_ms": kt}
        if note:
            out["note"] = note
        fz.free()
        return out
    except Exception as exc:   # a sweep entry never takes the headline down
        torch.cuda.empty_cache()
        return {"workload": wl, "batch": N, "error": str(exc)[:200]}


def sweep_variants_c2(cx, peak):
    """The two variants of the C2 step in which the sources are DATA, as in the reference's own data flow (the layout
    source is one_hot(label), src/trainer.py:461; no gradient is asked for the sources): no pass 2, no d_out staging.
      flow_grad_only : dense one-hot layout source, gradient to the flow only            128 algorithmic B/px
      label_source   : int64 class-id map as the layout source (vlg_warp_loss_labels_*)   56 algorithmic B/px
                       (coords 8 + rgb 12 + 12 + src label 8 + tgt label 8 read, d_flow 8 written)"""
    out = {}
    try:
        fz = Fused(cx, "c2", WORKLOADS["c2"][0], with_src=False)
        ms, r, total = cx.timed(fz.step, 5, min_ms=120.0)
        out["c2_flow_grad_only"] = {"ms_per_step": ms, "Mpixel_per_s": cx.world * fz.P / (ms * 1e-3) / 1e6, "algorithmic_bytes_per_px": 128,
                                    "frac_of_hbm_roofline": fz.P * 128 / (ms * 1e-3) / 1e9 / peak}
        # label source: same inputs, the layout source handed over as its class-id map
        ops, lib, ptr = cx.ops, cx.lib, cx.ops._ptr
        labs = [s["src_layout"].argmax(1).contiguous() for s in fz.sets]
        prob = ops._problem(fz.N, fz.H, fz.W, fz.K, fz.tdt, ops.WarpLossConfig(w_tv=0.5))
        ws = ops._workspace(prob, False, cx.dev, cached=False)
        sp = C.c_void_p(cx.stream.cuda_stream)

        def lab_step(i):
            s = fz.sets[i % len(fz.sets)]
            ops.check(lib.vlg_warp_loss_labels_fwd_bwd(C.byref(prob), ptr(s["src_rgb"]), ptr(labs[i % len(labs)]), ptr(s["flow"]), ptr(s["tgt_rgb"]),
                                                       ptr(s["tgt_label"]), ptr(fz.loss), ptr(fz.d_c), None, ptr(ws), ws.numel(), sp))
        for i in range(3):
            lab_step(i)
        ms, r, total = cx.timed(lab_step, 5, min_ms=120.0)
        out["c2_label_source"] = {"ms_per_step": ms, "Mpixel_per_s": cx.world * fz.P / (ms * 1e-3) / 1e6, "algorithmic_bytes_per_px": 56,
                                  "frac_of_hbm_roofline": fz.P * 56 / (ms * 1e-3) / 1e9 / peak, "launch": "direct launches"}
        fz.free()
    except Exception as exc:
        out["error"] = str(exc)[:200]
        torch.cuda.empty_cache()
    return out


def dump_outputs(outdir, arrays):
    """Writes every tensor of `arrays` as outdir/<name>.npy in float32.  Each array gets an equal share of
    DUMP_LIMIT_BYTES; a larger one is written as a fixed, seeded sample of its elements (sorted flat indices into its
    logical shape, e.g. NCHW whatever the memory format), so two runs with the same arguments compare element for
    element."""
    os.makedirs(outdir, exist_ok=True)
    share = (DUMP_LIMIT_BYTES // len(arrays) - 128) // 4      # elements per array; 128 bytes of .npy header
    g = torch.Generator().manual_seed(DUMP_SEED)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > share:
            idx = torch.randint(0, t.numel(), (share,), generator=g).sort().values.to(t.device)
            t = t[torch.unravel_index(idx, t.shape)]
        np.save(os.path.join(outdir, name + ".npy"), t.float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (c4: global batch); 0 = the workload's own")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the step's kernels directly instead of replaying a CUDA graph")
    ap.add_argument("--no-eager", action="store_true", help="skip timing the torch CUDA eager incumbent")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step (iters/s) measurement")
    ap.add_argument("--no-sweep", action="store_true", help="skip the compact lines of the other BASELINE configs")
    ap.add_argument("--no-aux", action="store_true", help="skip the boundary-fusion / forward-warp side measurements")
    ap.add_argument("--flow-grad-only", action="store_true", help="sources are data: no d_src (128 B/px variant)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (float32, "
                    "<= 64 MB in all; larger outputs as a fixed, seeded sample)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    cx = Ctx()
    vlg, dev, stream, dist = cx.vlg, cx.dev, cx.stream, cx.dist
    wl = args.workload
    N0, H, W, K, sigma, far, dtype = WORKLOADS[wl]
    N = args.batch or N0
    peak, peak_src = hbm_peak()
    warmup = max(args.warmup, 3)
    sampler = ClockSampler(cx.local_rank)

    # ------------------------------------------------------------------ rollout workload (c4)
    if wl == "c4":
        if N % world:
            raise SystemExit(f"global batch {N} is not divisible by {world} ranks")
        ro = Rollout(cx, N // world)
        for i in range(warmup):
            ro.step(i)
        cx.barrier()
        n0 = vlg.launch_count()
        ro.step(0)
        launches_per_step = vlg.launch_count() - n0
        if rank == 0:
            sampler.start(); sampler.wait_first()
        ms, r, total = cx.timed(ro.step, args.steps)
        clocks = sampler.stop() if rank == 0 else None
        if args.dump_outputs and rank == 0:
            imgs, labs = ro.out
            dump_outputs(args.dump_outputs, {**{f"frame{t + 1}": x for t, x in enumerate(imgs)},
                                             **{f"label{t + 1}": x for t, x in enumerate(labs)}})
        e2e = ro.e2e(args.steps)
        if rank != 0:
            if dist is not None: dist.destroy_process_group()
            return
        px_steps = world * ro.px_steps
        achieved = ro.px_steps * ROLLOUT_BYTES_PER_PX / (ms * 1e-3) / 1e9
        out = {"metric": "warp+loss fwd/bwd throughput", "value": px_steps / (ms * 1e-3) / 1e6, "unit": "Mpixel/s", "n_gpus": world,
               "steps": args.steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
               "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": {**workload_config(wl, N, world, dtype), "per_gpu_batch": N // world,
                          "unit_note": f"one step = one {ROLLOUT_STEPS}-frame rollout of the batch; Mpixel/s counts every warped frame",
                          "replays_per_step": r, "timed_region_ms": total,
                          "l2_policy": "inputs exceed the 126 MB L2 (%.0f MB of frames + flows per rollout)" % (ro.px_steps * 20 / 1e6)},
               "roofline": {"bound": "hbm", "kernel": "warp_fwd_labels_kernel (x5, including the Python wrapper's allocations)",
                            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                            "peak_source": peak_src, "algorithmic_bytes_per_px": ROLLOUT_BYTES_PER_PX,
                            "algorithmic_bytes": ro.px_steps * ROLLOUT_BYTES_PER_PX // ROLLOUT_STEPS, "kernel_ms": ms / ROLLOUT_STEPS},
               "e2e": e2e, "gpu_launches": launches_per_step * args.steps * r, "clocks": clocks}
        if world == 1 and not args.no_cpu_baseline:
            v, t, sample = cpu_oracle_run(wl, N, 3, 1)
            out["cpu_baseline"] = {"value": v, "unit": "Mpixel/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample}
        print(json.dumps(out))
        if dist is not None: dist.destroy_process_group()
        return

    # ------------------------------------------------------------------ fused warp + loss workloads
    with_src = not args.flow_grad_only
    fz = Fused(cx, wl, N, with_src=with_src, use_graph=not args.no_graph)
    for i in range(warmup):
        fz.step(i)
    cx.barrier()

    # ---- timed region 1: device-resident throughput (`value`) ----
    if rank == 0:
        sampler.start(); sampler.wait_first()
    ms_per_step, replays, timed_ms = cx.timed(fz.step, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:     # the buffers of the last timed step, before anything launches again
        outs = {"loss": fz.loss, "d_flow": fz.d_c, "d_src_rgb": fz.d_a, "d_src_layout": fz.d_b}
        dump_outputs(args.dump_outputs, {k: v for k, v in outs.items() if v is not None})
    launches = fz.count_launches(args.steps * replays)

    # ---- per-kernel device times inside the direct launch sequence (CUDA events on the launch stream) ----
    kt = fz.kernel_times(reps=20)
    kernels_us = fz.cupti_table() if rank == 0 else None

    # ---- timed region 2: end to end through the public module API from pinned host memory ----
    e2e = e2e_fused(cx, fz, args.steps)
    eg = e2e_fused(cx, fz, args.steps, captured=False)
    e2e["eager"] = {k: eg[k] for k in ("value", "unit", "ms_per_step", "launch")}
    up = e2e_fused(cx, fz, args.steps, flow_from_host=True)
    e2e["flow_uploaded"] = {k: up[k] for k in ("value", "unit", "h2d_bytes_per_step", "ms_per_step")}

    # ---- incumbent on the same GPU: the oracle composition run by torch CUDA eager (ATen kernels) ----
    eager = None
    if rank == 0 and dtype == "f32" and not args.no_eager and fz.P <= 4 * 1024 * 1024:
        from oracle import torch_oracle as TO
        s0 = fz.sets[0]

        def eager_step():
            a = s0["src_rgb"].detach().requires_grad_(with_src)
            b = s0["src_layout"].detach().requires_grad_(with_src)
            f = s0["flow"].detach().requires_grad_(True)
            o = TO.warp_loss(a, b, f, s0["tgt_rgb"], s0["tgt_label"], w_tv=0.5)
            o["total"].backward()
        for _ in range(2):
            eager_step()
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        for _ in range(5):
            eager_step()
        g1.record(stream)
        torch.cuda.synchronize()
        ms_eager = g0.elapsed_time(g1) / 5
        eager = {"ms_per_step": ms_eager, "value": fz.P / (ms_eager * 1e-3) / 1e6, "unit": "Mpixel/s",
                 "what": "oracle composition (F.grid_sample + losses + autograd) in torch CUDA eager, same inputs, checker only"}

    P = fz.P
    graph_used = fz.graphs is not None
    fz.free()

    # ---- side measurements on rank 0: boundary fusion, ingest, forward warp (HBM-bound passes) ----
    aux = None
    if rank == 0 and not args.no_aux:
        def timed(fn, reps):
            for _ in range(2):
                fn()
            t0_, t1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0_.record(stream)
            for _ in range(reps):
                fn()
            t1_.record(stream)
            torch.cuda.synchronize()
            return t0_.elapsed_time(t1_) / reps
        fr = torch.rand(8, 3, 1024, 2048, device=dev)          # 403 MB read+written per call: larger than the L2
        ms_fa = timed(lambda: vlg.prepare_frames(fr, flip=True), 10)
        aux = {"frame_affine": {"what": "vlg_frame_affine 8x3x1024x2048 fp32 NCHW -> normalised, flipped NHWC (24 B/px algorithmic; "
                                        "includes the output allocation of the Python wrapper)",
                                "ms": ms_fa, "achieved_GBs": fr.numel() * 4 * 2 / (ms_fa * 1e-3) / 1e9}}
        del fr
        u8 = torch.randint(0, 256, (8, 1024, 2048, 3), dtype=torch.uint8, device=dev)
        sg = torch.randint(0, K, (8, 1024, 2048), dtype=torch.uint8, device=dev)
        ms_in = timed(lambda: vlg.ingest(u8, sg, n_classes=K, want_label=True, want_one_hot=True), 5)
        in_px = 8 * 1024 * 2048
        aux["ingest"] = {"what": "vlg_ingest 8x1024x2048: uint8 frame + class map -> normalised fp32 NHWC frame, int64 label, one-hot "
                                 "layout (4 B/px read, 12 + 8 + 80 written; includes the Python wrapper's allocations)", "ms": ms_in,
                         "achieved_GBs": in_px * 104 / (ms_in * 1e-3) / 1e9}
        del u8, sg
        vn, vh, vw = 2, 1024, 2048
        vd = make_inputs(vn, vh, vw, K, 4.0, 0.0, dtype, dev, seed=79)
        ms_fw = timed(lambda: vlg.warp(vd["src_rgb"], vd["src_layout"], vd["flow"]), 5)
        fw_bpp = 200 if dtype == "f32" else 108
        aux["warp_fwd"] = {"what": f"vlg_warp_fwd {vn}x{vh}x{vw} {dtype}: warped rgb + layout + argmax written ({fw_bpp} B/px algorithmic)",
                           "ms": ms_fw, "Mpixel_per_s": vn * vh * vw / (ms_fw * 1e-3) / 1e6,
                           "achieved_GBs": vn * vh * vw * fw_bpp / (ms_fw * 1e-3) / 1e9}
        del vd
        for k_ in aux:
            aux[k_]["frac_of_hbm_peak"] = aux[k_]["achieved_GBs"] / peak
        torch.cuda.empty_cache()

    # ---- the other BASELINE configs, compact (every rank takes part: weak scaling / per-rank rollout shards) ----
    sweep = None
    if not args.no_sweep and wl == "c2":
        sweep = sweep_variants_c2(cx, peak)
        sweep["c3"] = sweep_entry(cx, "c3", WORKLOADS["c3"][0], 5, peak)
        for B in (1, 4, 16, 64):
            sweep[f"c5_b{B}"] = sweep_entry(cx, "c5", B, 5, peak)
        try:
            n_rank = WORKLOADS["c4"][0] // 8                      # the dp8 shard of BASELINE config 4
            ro = Rollout(cx, n_rank)
            ms_ro, r_, tot_ = cx.timed(ro.step, 3, min_ms=120.0)
            sweep["c4_dp8_shard"] = {"workload": f"c4: {ROLLOUT_STEPS}-step rollout, {n_rank}x512x1024 per GPU (global batch 32 over 8 GPUs)",
                                     "ms_per_rollout": ms_ro, "Mpixel_steps_per_s": world * ro.px_steps / (ms_ro * 1e-3) / 1e6,
                                     "algorithmic_bytes_per_px": ROLLOUT_BYTES_PER_PX,
                                     "frac_of_hbm_roofline": ro.px_steps * ROLLOUT_BYTES_PER_PX / (ms_ro * 1e-3) / 1e9 / peak,
                                     "note": "includes the Python wrapper's per-step allocations"}
            del ro
        except Exception as exc:
            sweep["c4_dp8_shard"] = {"error": str(exc)[:200]}
        torch.cuda.empty_cache()

    # ---- training step (SURVEY 8f-1): torch flow producer -> fused op -> DDP -> Adam, iters/s ----
    train = None
    if wl == "c2" and not args.no_train:
        from train import run_training
        train, _ = run_training(steps=max(3, min(args.steps, 10)), warmup=2, batch=N, height=H, width=W, classes=K)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    bpp = BYTES_PER_PX[dtype]
    step_bytes = bpp["step"] if with_src else bpp["pass1"]
    value = world * P / (ms_per_step * 1e-3) / 1e6
    # the longest kernel of the step, timed by CUDA events on its launch stream inside the direct launch sequence
    kb = {"rgb_strip_kernel": bpp["rgb_strip"], "lay_tile_kernel": bpp["lay_tile"], "pass2_rec_kernel": bpp["pass2"]}
    live = {k: v for k, v in kt.items() if k in kb and v > 0}
    dom = max(live, key=live.get)
    dom_ms = live[dom]
    achieved = P * kb[dom] / (dom_ms * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic(dom) if wl == "c2" and with_src else (None, None)
    out = {
        "metric": "warp+loss fwd/bwd throughput", "value": value, "unit": "Mpixel/s", "n_gpus": world,
        "steps": args.steps, "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
        "config": {**workload_config(wl, N, world, dtype, with_src),
                   "l2_policy": "inputs (%.0f MB/step) exceed the 126 MB L2; two input sets alternate" % (P * 120 / 1e6),
                   "launch": "cuda graph replay" if graph_used else "direct launches",
                   "replays_per_step": replays, "timed_region_ms": timed_ms,
                   "timing_note": f"the timed region is {args.steps} steps; ms_per_step is per step",
                   "exchange": ("one NCCL all-reduce of the 8-float loss vector per step, issued after pass 1 and overlapped with pass 2"
                                if world > 1 else "none (single GPU)")},
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes": P * kb[dom], "algorithmic_bytes_per_px": kb[dom], "kernel_ms": dom_ms},
        "roofline_kernels": {k: {"kernel_ms": v, "algorithmic_bytes_per_px": kb[k], "achieved": P * kb[k] / (v * 1e-3) / 1e9,
                                 "frac": P * kb[k] / (v * 1e-3) / 1e9 / peak} for k, v in live.items()},
        "roofline_step": {"algorithmic_bytes_per_px": step_bytes,
                          "achieved": P * step_bytes / (ms_per_step * 1e-3) / 1e9,
                          "frac": P * step_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                          "span_first_to_last_kernel_ms": kt["span_first_to_last"],
                          "kernels_us_cupti": kernels_us},
        "e2e": e2e,
        "gpu_launches": launches,
        "clocks": clocks,
        "sweep": sweep,
        "train": train,
        "torch_cuda_eager": eager,
        "aux": aux,
    }
    if world == 1 and not args.no_cpu_baseline:
        v, t, sample = cpu_oracle_run(wl, N, 5, 1)
        out["cpu_baseline"] = {"value": v, "unit": "Mpixel/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample}
    print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
