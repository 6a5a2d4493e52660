"""Connected components at full size (160x384x384): ops.connected_components and ops.keep_components against
scipy.ndimage.label on the host, at connectivities 6 and 26, on three masks:
  * fc_segmenter : the segmenter's FC mask (> 0.5) of a synthetic knee, with the calibrated head of the full-size tests
                   (many small components);
  * shell_islands: an FC-like cartilage shell plus a few small islands (the post-processing case);
  * random_0.5   : uniform random at density 0.5 (about 216 k components at 6-connectivity, deep merges everywhere).

  python scripts/bench_components.py [--iters 50] [--out FILE] [--profile DIR]

Prints one JSON line: card name and power limit (read in the same run), per-call times from CUDA events after warm-up,
scipy's time on the host, whether labels equal scipy's, and bytes/s against the algorithmic floor of 1 B of mask read
plus 4 B of labels written per voxel (118 MB, about 15 us at 7.7 TB/s).  --profile runs torch.profiler in a separate
pass and writes the per-kernel split to DIR."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402
from scipy import ndimage as ndi  # noqa: E402

import surface_metrics_oracle as so  # noqa: E402
from oai_analysis_2_b200 import ops  # noqa: E402

SHAPE = (160, 384, 384)
HBM_BYTES_PER_S = 7.7e12
RANK = {6: 1, 26: 3}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def segmenter_fc():
    from helpers import write_seg_config
    from oai_analysis_2_b200 import synthetic
    from oai_analysis_2_b200.segmentation.segmenter import Segmenter3DInPatchClassWise
    from oracle import seg_oracle
    sd = seg_oracle.make_unet_state_dict(13, 1, 2, True, True, True, 88.16291826695385,
                                         [-4.068152692193752, -7.490846258792958])
    with tempfile.TemporaryDirectory() as tmp:
        seg = Segmenter3DInPatchClassWise(mode="pred", config=write_seg_config(tmp, sd, [128, 128, 32], True, True,
                                                                               (16, 16, 8)))
        out = seg.segment_device(torch.from_numpy(synthetic.synthetic_knee(SHAPE, seed=5)).cuda(), True)
    return (out[0] > 0.5).cpu().numpy()


def masks():
    shell = so.shell(SHAPE, (80, 150, 192), (110, 140, 150), 0.03, seed=1, cut=230)
    rng = np.random.default_rng(2)
    for _ in range(12):
        z, y, x = (int(rng.integers(4, s - 8)) for s in SHAPE)
        shell[z:z + 3, y:y + 4, x:x + 5] = True
    return {"fc_segmenter": segmenter_fc(), "shell_islands": shell,
            "random_0.5": np.random.default_rng(7).random(SHAPE) < 0.5}


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
        sys.exit("bench_components: needs a CUDA device")
    nvox = int(np.prod(SHAPE))
    floor_bytes = 5 * nvox
    cases = []
    for name, host in masks().items():
        dev = torch.from_numpy(host).cuda()
        for conn in (6, 26):
            ms_cc = timed(lambda: ops.connected_components(dev, conn), args.iters)
            ms_keep = timed(lambda: ops.keep_components(dev, conn), args.iters)
            labels, sizes, count = ops.connected_components(dev, conn)
            t0 = time.perf_counter()
            ref, n = ndi.label(host, ndi.generate_binary_structure(3, RANK[conn]))
            scipy_s = time.perf_counter() - t0
            cases.append({"mask": name, "connectivity": conn, "density": round(float(host.mean()), 5),
                          "components": int(count), "labels_equal_scipy": bool(int(count) == n and
                                                                               np.array_equal(labels.cpu().numpy(), ref)),
                          "ms_connected_components": round(ms_cc, 4), "ms_keep_largest": round(ms_keep, 4),
                          "scipy_label_s": round(scipy_s, 3), "speedup_vs_scipy": round(scipy_s * 1e3 / ms_cc, 1),
                          "achieved_tb_per_s_vs_floor": round(floor_bytes / (ms_cc * 1e-3) / 1e12, 3)})
    line = {"bench": "components", "card": card(), "shape": list(SHAPE), "iters": args.iters,
            "host_cores": os.cpu_count(), "floor_bytes": floor_bytes,
            "floor_us_at_7.7TBps": round(floor_bytes / HBM_BYTES_PER_S * 1e6, 2), "cases": cases}
    if args.profile:
        os.makedirs(args.profile, exist_ok=True)
        from torch.profiler import ProfilerActivity, profile
        tables = []
        for name, host in masks().items():
            if name == "fc_segmenter":
                continue
            dev = torch.from_numpy(host).cuda()
            for conn in (6, 26):
                ops.keep_components(dev, conn)
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(10):
                        ops.keep_components(dev, conn)
                    torch.cuda.synchronize()
                tables.append(f"== {name}, connectivity {conn}, 10 calls of keep_components\n" +
                              prof.key_averages().table(sort_by="cuda_time_total", row_limit=15))
        with open(os.path.join(args.profile, "components_kernels_profile.txt"), "w") as f:
            f.write("\n".join(tables))
        print("\n".join(tables))
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
