"""Segmentation quality at full size (160x384x384, OAI spacing 0.3646 x 0.3646 x 0.7 mm), FC + TC: oai_surface_metrics
against the scipy / numpy oracle (tests/surface_metrics_oracle.py) on the host.

  python scripts/bench_seg_quality.py [--iters 50] [--out FILE] [--profile DIR]

Prints one JSON line: card name and power limit (read in the same run), per-call times from CUDA events with the
distance maps off and on, the scipy time of the same two classes once on the host with its core count, and the bytes
the passes must move over the kernel time against 7.7 TB/s.  The working set (two 23.6 MB masks and a 189 MB
two-channel intermediate per class) exceeds the 126 MB L2, so nothing flushes L2 between calls.  --profile runs
torch.profiler in a separate pass and writes the per-kernel split to DIR."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import surface_metrics_oracle as so  # noqa: E402
from oai_analysis_2_b200 import ops  # noqa: E402

SHAPE = (160, 384, 384)
SPACING = (0.3646, 0.3646, 0.7)
HBM_BYTES_PER_S = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def pairs():
    """FC- and TC-like thin shells and a shifted copy of each (the same shapes as the GPU tests)."""
    fc = so.shell(SHAPE, (80, 150, 192), (110, 140, 150), 0.03, seed=1, cut=230)
    tc = so.shell(SHAPE, (80, 320, 192), (90, 120, 130), 0.04, seed=2) & (np.arange(SHAPE[1])[None, :, None] > 215)
    return [(fc, np.roll(fc, (1, 2, -1), axis=(0, 1, 2))), (tc, np.roll(tc, (0, 1, 2), axis=(0, 1, 2)))]


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_seg_quality: needs a CUDA device")
    host = pairs()
    dev = [(torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()) for a, b in host]

    def call(maps):
        return lambda: [ops.surface_metrics(a, b, SPACING, maps=maps) for a, b in dev]

    ms_off = timed(call(False), args.iters)
    ms_on = timed(call(True), args.iters)
    got = [ops.surface_metrics(a, b, SPACING) for a, b in dev]
    t0 = time.perf_counter()
    ref = [so.surface_metrics(a, b, SPACING) for a, b in host]
    scipy_s = time.perf_counter() - t0
    nvox = int(np.prod(SHAPE))
    # unavoidable traffic per class: both uint8 masks read once, the 8-byte two-channel intermediate written by pass 1,
    # read and written by pass 2 and read by pass 3
    bytes_per_class = nvox * (2 + 8 + 16 + 8)
    classes = []
    for (t, c), (rt, rc, _) in zip(got, ref):
        t, c = t.cpu().numpy(), c.cpu().numpy()
        classes.append({"dice": float(t[0]), "assd_mm": float(t[1]), "hd95_mm": float(t[2]), "hd_mm": float(t[3]),
                        "counts": [int(v) for v in c], "counts_equal_oracle": bool(np.array_equal(c, rc)),
                        "max_rel_err_vs_oracle": float(np.max(np.abs(t[1:] - rt[1:]) / np.abs(rt[1:])))})
    line = {"bench": "seg_quality", "card": card(), "shape": list(SHAPE), "spacing_xyz": list(SPACING),
            "classes": 2, "iters": args.iters, "ms_per_call_fc_tc_maps_off": round(ms_off, 4),
            "ms_per_call_fc_tc_maps_on": round(ms_on, 4), "scipy_s_fc_tc": round(scipy_s, 3),
            "host_cores": os.cpu_count(), "speedup_vs_scipy_maps_off": round(scipy_s * 1e3 / ms_off, 1),
            "bytes_moved_fc_tc": 2 * bytes_per_class,
            "hbm_floor_ms": round(2 * bytes_per_class / HBM_BYTES_PER_S * 1e3, 4),
            "achieved_tb_per_s_maps_off": round(2 * bytes_per_class / (ms_off * 1e-3) / 1e12, 3),
            "per_class": classes}
    if args.profile:
        os.makedirs(args.profile, exist_ok=True)
        from torch.profiler import ProfilerActivity, profile
        fn = call(False)
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(10):
                fn()
            torch.cuda.synchronize()
        table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=30)
        with open(os.path.join(args.profile, "seg_quality_kernels.txt"), "w") as f:
            f.write(table)
        print(table)
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
