"""Per-launch times of conv_igemm_kernel over one full-size knee (CUDA events around every launch, oai_profile_*).

    python scripts/layer_times.py [precision ...]     # default: mixed fp16
Prints one JSON line per precision: [{layer, ms, algorithmic TFLOP/s, issued TFLOP/s}, ...] + totals."""
import ctypes
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NAMES = ["ec1", "ec2", "ec3", "ec4", "ec5", "ec6", "ec7", "dc9", "dc8", "dc7", "dc6", "dc5", "dc4", "dc3", "dc2", "dc1"]
# with the w halo skipped (the default at the production tile) dc2 runs as two launches: 32 x 4 tiles over 96 of its 98
# columns, then 8 x 16 tiles over the last 8
NAMES_STRIP = NAMES[:15] + ["dc2 strip", "dc1"]


def main():
    from oai_analysis_2_b200 import _lib, ops, synthetic
    from oracle import seg_oracle
    L = _lib.lib
    sd = seg_oracle.make_unet_state_dict(13, 1, 2, True, True, True)
    vol = torch.from_numpy(synthetic.synthetic_knee(synthetic.OAI_SHAPE, seed=5)).cuda()
    for prec in (sys.argv[1:] or ["mixed", "fp16"]):
        plan, fmt = {"fp16": (0, 0), "mixed": (1, 0), "fp16x2": (2, 0), "fp16x3": (3, 0), "bf16": (0, 1)}[prec]
        h = ops.SegHandle(sd, 1, 2, True, True, (128, 128, 32), (16, 16, 8), fmt, plan)
        nb = h.auto_tiles_per_batch(vol.shape)
        ws = torch.empty(h.workspace_bytes(vol.shape, nb), dtype=torch.uint8, device="cuda")
        for _ in range(2):
            h.forward(vol, 0, nb, workspace=ws)
        torch.cuda.synchronize()
        L.oai_profile_begin()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        h.forward(vol, 0, nb, workspace=ws)
        e1.record()
        torch.cuda.synchronize()
        rows = []
        i = 0
        while True:
            ms, fl, xfl = ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
            if L.oai_profile_entry(i, ctypes.byref(ms), ctypes.byref(fl), ctypes.byref(xfl)):
                break
            rows.append(dict(layer=i, ms=round(ms.value, 3), alg_tflops=round(fl.value / ms.value / 1e9, 1),
                             issued_tflops=round(xfl.value / ms.value / 1e9, 1), issued_tflop=round(xfl.value / 1e12, 3)))
            i += 1
        L.oai_profile_end(None, None, None, None)
        names = NAMES_STRIP if len(rows) % 17 == 0 else NAMES
        for r in rows:
            r["layer"] = names[r["layer"] % len(names)]
        tot = sum(r["ms"] for r in rows)
        print(json.dumps(dict(precision=prec, tiles_per_batch=nb, workspace_gb=round(ws.numel() / 2**30, 1),
                              seg_ms=round(e0.elapsed_time(e1), 2), conv_ms=round(tot, 2),
                              issued_tflops=round(sum(r["issued_tflop"] for r in rows) / tot * 1e3, 1), layers=rows)))
        del h, ws


if __name__ == "__main__":
    main()
