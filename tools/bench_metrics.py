#!/usr/bin/env python
"""Times vlg_confusion (the confusion-matrix kernel behind vlg_b200.confusion_matrix / LayoutIoU) on one GPU.

    python tools/bench_metrics.py [--out FILE]

For the C2 and C3 shapes of bench.py (bench.WORKLOADS, inputs from bench.make_inputs) it times the three modes --
int64 predicted labels, NHWC scores (channels_last), NCHW-contiguous scores -- and, on the same inputs, the torch
composition a user writes today (argmax -> mask -> t*K+p -> bincount), plus the single-class worst case (every pixel in
one bin) in label and NHWC mode.  Every figure is CUDA-event time over a region of at least 250 ms, right after 250 ms of
untimed passes; the passes cycle through two seeded input sets, and fresh copies of them until the working set of the
mode is at least twice the 126 MB L2, so every pass reads HBM.  Achieved GB/s counts the algorithmic bytes (every input
element read once; the K*K+1 counts are negligible).  Prints ONE JSON line with the card's name and power limit; --out also writes it there.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
import vlg_b200  # noqa: E402
from vlg_b200.ops import _confusion_into  # noqa: E402

REGION_MS = 250.0
MIN_WORKING_SET = 2 * 126 * 2 ** 20
IGNORE = -100


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else (torch.cuda.get_device_name(), "unknown")
    return name, power


def timed(fn, n_sets):
    """ms per call: CUDA events around >= REGION_MS of calls, after REGION_MS of untimed calls."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(2 * n_sets):
        fn(i)
    torch.cuda.synchronize()
    e0.record()
    for i in range(n_sets):
        fn(i)
    e1.record()
    e1.synchronize()
    est = max(e0.elapsed_time(e1) / n_sets, 1e-3)
    reps = max(n_sets, int(REGION_MS / est) + 1)
    for i in range(reps):
        fn(i)
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def torch_counts(pred, tgt, K):
    """What a user composes in torch today: argmax (scores) -> mask -> t*K + p -> bincount."""
    p = torch.argmax(pred, 1) if pred.dim() == 4 else pred
    m = tgt != IGNORE
    return torch.bincount((tgt * K + p)[m], minlength=K * K)


def measure(label, preds, tgts, K, P, bytes_px, peak, with_torch=True):
    """Times `preds` vs `tgts` (lists of equal length), cycled with fresh copies until the working set of this mode is
    >= MIN_WORKING_SET."""
    n0 = len(preds)
    n = max(n0, -(-MIN_WORKING_SET // (P * bytes_px)))
    preds = preds + [preds[i % n0].clone(memory_format=torch.preserve_format) for i in range(n0, n)]
    tgts = tgts + [tgts[i % n0].clone() for i in range(n0, n)]
    counts = torch.zeros(K * K + 1, dtype=torch.int64, device="cuda")
    ours = torch.zeros_like(counts)
    _confusion_into(ours, preds[0], tgts[0], K, ignore_index=IGNORE)
    ref = torch_counts(preds[0], tgts[0], K)
    agree = bool(torch.equal(ours[:K * K], ref)) and int(ours[K * K]) == 0
    ms = timed(lambda i: _confusion_into(counts, preds[i % n], tgts[i % n], K, ignore_index=IGNORE), n)
    gbs = P * bytes_px / (ms * 1e-3) / 1e9
    out = {"mode": label, "us": round(ms * 1e3, 2), "Gpx_per_s": round(P / (ms * 1e-3) / 1e9, 2),
           "algorithmic_bytes_per_px": bytes_px, "GB_per_s": round(gbs, 1), "frac_of_hbm_peak": round(gbs / peak, 3),
           "equals_torch": agree}
    if with_torch:
        ms_t = timed(lambda i: torch_counts(preds[i % n], tgts[i % n], K), n)
        out["torch_us"] = round(ms_t * 1e3, 2)
        out["speedup_vs_torch"] = round(ms_t / ms, 2)
    return out


def run_workload(wl, peak):
    N, H, W, K, sigma, far, dt = bench.WORKLOADS[wl]
    P = N * H * W
    esz = 4 if dt == "f32" else 2
    res = {"workload": f"{wl}: {N}x{H}x{W} K={K} {dt}"}

    def make(seed):
        x = bench.make_inputs(N, H, W, K, sigma, far, dt, "cuda", seed=seed)
        lay = x["src_layout"]                                # one-hot [N,K,H,W] in channels_last storage
        return lay, torch.argmax(lay, 1), x["tgt_label"]

    sets = [make(1024), make(1025)]
    tgts = [s[2] for s in sets]
    modes = [measure("labels", [s[1] for s in sets], tgts, K, P, 16, peak),
             measure("layout_nhwc", [s[0] for s in sets], tgts, K, P, K * esz + 8, peak),
             measure("layout_nchw", [s[0].contiguous() for s in sets], tgts, K, P, K * esz + 8, peak)]
    del sets
    torch.cuda.empty_cache()

    # worst case for the shared-memory histogram: every pixel of every warp in the same bin
    one_t = [torch.full((N, H, W), 3, dtype=torch.int64, device="cuda") for _ in range(2)]
    modes.append(measure("labels_single_class", [t.clone() for t in one_t], one_t, K, P, 16, peak, with_torch=False))
    tdt = torch.float32 if dt == "f32" else torch.bfloat16
    one_lay = torch.zeros(N, K, H, W, dtype=tdt, device="cuda").contiguous(memory_format=torch.channels_last)
    one_lay[:, 3] = 1
    modes.append(measure("layout_nhwc_single_class", [one_lay, one_lay.clone(memory_format=torch.channels_last)], one_t, K, P,
                         K * esz + 8, peak, with_torch=False))
    del one_lay, one_t
    torch.cuda.empty_cache()
    res["modes"] = modes
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON line to this file")
    ap.add_argument("--workloads", default="c2,c3")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_metrics.py needs a CUDA device")
    name, power = card()
    peak, peak_src = bench.hbm_peak()
    out = {"metric": "vlg_confusion", "card": name, "power_limit": power, "hbm_peak_GBs": peak, "hbm_peak_source": peak_src,
           "region_ms_min": REGION_MS, "workloads": [run_workload(wl, peak) for wl in args.workloads.split(",")]}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
