"""Registration-quality terms at the knee model's network shape: oai_reg_icon_loss against the torch restatement of the
same terms (tests/icon_loss_oracle.py) on the same GPU, after one registration of a synthetic pair.

  python scripts/bench_icon_loss.py [--shape 80 192 192] [--iters 50] [--out DIR]

Prints one JSON line: card name and power limit (read in the same run), per-call times from CUDA events for both
similarities, per-kernel times of the library call from torch.profiler (a separate run), the torch bar, and the bytes the
two LNCC passes move.  The working set (fields, maps, moments: ~0.2 GB at 80x192x192) exceeds the 126 MB L2, so the
passes stream from HBM; nothing flushes L2 between calls."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import icon_loss_oracle as lo  # noqa: E402
from oai_analysis_2_b200 import ops  # noqa: E402
from oracle import reg_oracle  # noqa: E402

SIMS = {"lncc": ops.SIM_LNCC, "ssd_only_interpolated": ops.SIM_SSD_ONLY_INTERPOLATED}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


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


def kernel_times(fn, iters, out_dir):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    if out_dir:
        prof.export_chrome_trace(os.path.join(out_dir, "icon_loss_trace.json"))
    per = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
        if t > 0 and ("kernel" in e.key or "Memset" in e.key):
            key = e.key.replace("(anonymous namespace)::", "").replace("void ", "")
            name = key.split("(")[0].split("<")[0].split("::")[-1].strip()
            per[name] = per.get(name, 0.0) + t / 1000.0 / iters
    return {k: round(v, 4) for k, v in sorted(per.items(), key=lambda kv: -kv[1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", type=int, nargs=3, default=[80, 192, 192])
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--torch-iters", type=int, default=5)
    ap.add_argument("--out", default=None, help="directory for the JSON line and the profiler trace")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_icon_loss needs a CUDA device")
    torch.backends.cudnn.allow_tf32 = False         # the torch bar computes in float32, as the library does
    torch.backends.cuda.matmul.allow_tf32 = False
    if args.out:
        os.makedirs(args.out, exist_ok=True)
    shape = tuple(args.shape)
    sd = reg_oracle.make_gradicon_state_dict(4321)
    stage = ops.RegHandle({"regis_net." + k: v for k, v in sd.items()}, shape)
    g = torch.Generator().manual_seed(0)
    A, B = [(F.interpolate(torch.randn(1, 1, *[max(2, s // 8) for s in shape], generator=g), size=shape,
                           mode="trilinear", align_corners=True)[0, 0] * 0.3 + 0.5).clamp(0, 1).contiguous().cuda()
            for _ in range(2)]
    stage.forward(A, B)
    reg_ms = timed(lambda: stage.forward(A, B, want_phi=False), 10)
    noise = torch.randn(1, 3, *shape, generator=g).cuda()
    n3 = noise[0].contiguous()
    fields = stage.fields()
    f_AB, f_BA = [f[0:1].contiguous() for f in fields], [f[1:2].contiguous() for f in fields]
    vol = shape[0] * shape[1] * shape[2]
    res = dict(bench="icon_loss", shape=list(shape), card=card(), registration_ms=round(reg_ms, 3),
               describe=stage.describe())
    for name, kind in SIMS.items():
        lib_ms = timed(lambda: stage.icon_loss(n3, kind, 5.0, 1.5), args.iters)
        terms = stage.icon_loss(n3, kind, 5.0, 1.5)[0].cpu().tolist()

        def bar():
            with torch.no_grad():
                return lo.icon_loss_from_fields(f_AB, f_BA, A[None, None], B[None, None], noise, similarity=name,
                                                sigma=5, lmbda=1.5)
        torch_ms = timed(bar, args.torch_iters, warmup=1)
        ref = [float(v) for v in bar()]
        res[name] = dict(lib_ms=round(lib_ms, 4), torch_ms=round(torch_ms, 3), speedup=round(torch_ms / lib_ms, 1),
                         terms=terms, torch_fp32_terms=ref,
                         kernels_ms=kernel_times(lambda: stage.icon_loss(n3, kind, 5.0, 1.5), 20, args.out))
    # LNCC passes, per direction: pass 1 reads I and J and writes five z-blurred moments; pass 2 reads the five back
    # (its halo re-reads come from L2).  A naive version writes and re-reads ten blurred volumes on top.
    res["lncc_bytes_per_direction"] = dict(zblur=4 * vol * (2 + 5), tile=4 * vol * 5, total=4 * vol * 12)
    k = res["lncc"]["kernels_ms"]
    t_lncc = (k.get("lncc_zblur_kernel", 0) + k.get("lncc_tile_kernel", 0)) / 2   # both directions are in the totals
    if t_lncc > 0:
        res["lncc_GBps_per_direction"] = round(4 * vol * 12 / (t_lncc * 1e-3) / 1e9, 1)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(os.path.join(args.out, "bench_icon_loss.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
