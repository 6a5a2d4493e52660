"""Dice / probability error of candidate per-layer precision plans on the golden fixtures (GPU)."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    from helpers import dice, load_golden
    from oai_analysis_2_b200 import ops
    from oracle import seg_oracle
    names = ["ec0", "ec1", "ec2", "ec3", "ec4", "ec5", "ec6", "ec7", "dc9", "dc8", "dc7", "dc6", "dc5", "dc4", "dc3",
             "dc2", "dc1"]
    plans = {"fp16": {}, "dc2 (mixed)": {"dc2": 2}, "dc1+dc2": {"dc1": 2, "dc2": 2},
             "dc2 skip only": {"dc2": 4}, "dc2 skip + dc1": {"dc2": 4, "dc1": 2}, "dc2 up only": {"dc2": 5},
             "dc2 skip + dc1 lo8 (mixed)": {"dc2": 6, "dc1": 7},
             "dc2 skip + dc1 x3": {"dc2": 4, "dc1": 3}, "dc2 skip + dc1 + ec1": {"dc2": 4, "dc1": 2, "ec1": 2},
             "dc2 skip + dc1 + dc5 skip": {"dc2": 4, "dc1": 2, "dc5": 4}, "dc2 up + dc1": {"dc2": 5, "dc1": 2},
             "dc2 skip + dc1 + ec2": {"dc2": 4, "dc1": 2, "ec2": 2},
             "dc1 only": {"dc1": 2}, "dc1 x3 only": {"dc1": 3},
             "fp16x2": {n: 2 for n in names[1:]}, "fp16x3": {n: 3 for n in names[1:]}}
    if len(sys.argv) > 1:
        plans = {k: v for k, v in plans.items() if any(a in k for a in sys.argv[1:])}
    for fx in ("seg_small_pertap", "seg_small_nobn", "seg_prod_tile"):
        z, m = load_golden(fx)
        sd = seg_oracle.make_unet_state_dict(m["seed"], 1, 2, m["bias"], m["BN"], True, m["head_gain"], m["head_bias"])
        vol = torch.from_numpy(seg_oracle.synthetic_knee(tuple(m["shape"]), m["seed"])).cuda()
        for pname, plan in plans.items():
            terms = [plan.get(n, 1) for n in names]
            h = ops.SegHandle(sd, 1, 2, m["bias"], m["BN"], m["patch"], m["overlap"], 0, 4, layer_terms=terms)
            out = h.forward(vol, 0).cpu().numpy()
            mask = h.forward(vol, 1).cpu().numpy()
            e = max(np.abs(out[0] - z["fc"]).max(), np.abs(out[1] - z["tc"]).max())
            print(json.dumps(dict(fixture=fx, plan=pname, prob_max_abs=float(e),
                                  dice_fc=dice(mask[0], z["fc_mask"]), dice_tc=dice(mask[1], z["tc_mask"]),
                                  flips=int((mask[0] != z["fc_mask"]).sum() + (mask[1] != z["tc_mask"]).sum()))))
            del h


if __name__ == "__main__":
    main()
