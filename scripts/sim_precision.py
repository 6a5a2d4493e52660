"""CPU simulation of the segmentation numerics: which operands must carry more than fp16's 11 bits for the
north-star Dice >= 0.999 bar?  (Design aid for the conv kernel's precision modes; not part of the product path.)

    python scripts/sim_precision.py seg_small_pertap

Each layer's (BN-folded) weights and stored activations are rounded the way a candidate kernel mode would round
them; products/accumulation are fp32 like the tensor pipe.  Modes per layer: w in {"h" fp16 error-feedback,
"hl" fp16 hi+lo}, a (the layer's INPUT activation) in {"h", "hl", "l8" fp16 hi + e4m3 lo plane (terms 6 / 7; the
e4m3 rounding of the weights the lo plane meets is left out: it scales a term already 2^-11 of the activation)}.
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import dice, load_golden  # noqa: E402
from oracle import seg_oracle as so  # noqa: E402


def fold(sd, name, kind, BN, bias):
    w = sd[f"{name}.0.weight"].double()
    if kind != "c":
        w = w.transpose(0, 1)
        if kind == "t3":
            w = w.flip(2, 3, 4)
    co = w.shape[0]
    b = sd[f"{name}.0.bias"].double() if bias else torch.zeros(co, dtype=torch.float64)
    if BN:
        g, beta = sd[f"{name}.1.weight"].double(), sd[f"{name}.1.bias"].double()
        mean, var = sd[f"{name}.1.running_mean"].double(), sd[f"{name}.1.running_var"].double()
        s = g / torch.sqrt(var + 1e-5)
        w = w * s.view(-1, 1, 1, 1, 1)
        b = (b - mean) * s + beta
    return w.contiguous(), b


def q16(x):
    return x.to(torch.float16).to(x.dtype)


def q_hl(x):
    hi = q16(x)
    return hi + q16(x - hi)


def q_l8(x):
    """fp16 hi + the e4m3 lo plane: satfinite(rn((x - hi) * 2^11)) * 2^-11"""
    hi = q16(x)
    lo = ((x - hi) * 2.0 ** 11).clamp(-448.0, 448.0).to(torch.float8_e4m3fn).to(x.dtype)
    return hi + lo * 2.0 ** -11


def q_w_ef(w):
    """error feedback along the taps of each (co, ci) filter, as oai_pack_conv_weights does"""
    co, ci = w.shape[:2]
    f = w.reshape(co * ci, -1).double()
    out = torch.empty_like(f)
    carry = torch.zeros(co * ci, dtype=torch.float64)
    for t in range(f.shape[1]):
        v = f[:, t] + carry
        h = v.float().to(torch.float16).double()
        out[:, t] = h
        carry = v - h
    return out.reshape(w.shape)


def run(name, plan, act_default="h", verbose=True):
    z, m = load_golden(name)
    sd = so.make_unet_state_dict(m["seed"], 1, 2, m["bias"], m["BN"], True, m["head_gain"], m["head_bias"])
    vol = so.synthetic_knee(tuple(m["shape"]), m["seed"])
    tiles, g = so.partition(vol, m["patch"], m["overlap"])
    kinds = {n: k for n, k, _, _ in so.UNET_LAYERS}
    W = {}
    for n, k, ci, co in so.unet_layer_table(1):
        w, b = fold(sd, n, k, m["BN"], m["bias"])
        wm = plan.get(n, ("h", act_default))[0]
        if n == "ec0":
            wq = w  # stem: split-fp16 operands, fp32-level
        elif wm == "h":
            wq = q_w_ef(w) if k != "t2" else q16(w)
        elif wm == "hl":
            wq = q_hl(w)
        else:
            wq = w
        W[n] = (wq.float(), b.float())

    def store(x, consumer_modes):
        """activation written by a layer; precision = the widest any consumer asks for"""
        if "f" in consumer_modes:
            return x
        if "hl" in consumer_modes:
            return q_hl(x)
        if "l8" in consumer_modes:
            return q_l8(x)
        return q16(x)

    am = lambda n: plan.get(n, ("h", act_default))[1]  # noqa: E731

    def blk(n, x):
        w, b = W[n]
        if kinds[n] == "t2":
            y = F.conv_transpose3d(x, w.transpose(0, 1).contiguous(), b, stride=2)
        else:
            y = F.conv3d(x, w, b, padding=1)
        return F.relu(y)

    outs = []
    with torch.no_grad():
        for i in range(0, tiles.shape[0], 4):
            x = tiles[i:i + 4]
            e0 = store(blk("ec0", x), [am("ec1")])
            syn0 = store(blk("ec1", e0), [am("ec2"), am("dc2"), am("dc2.skip")])
            e2 = store(blk("ec2", F.max_pool3d(syn0, 2)), [am("ec3")])
            syn1 = store(blk("ec3", e2), [am("ec4"), am("dc5")])
            e4 = store(blk("ec4", F.max_pool3d(syn1, 2)), [am("ec5")])
            syn2 = store(blk("ec5", e4), [am("ec6"), am("dc8")])
            e6 = store(blk("ec6", F.max_pool3d(syn2, 2)), [am("ec7")])
            e7 = store(blk("ec7", e6), [am("dc9")])
            d9 = store(blk("dc9", e7), [am("dc8")])
            d8 = store(blk("dc8", torch.cat((d9, syn2), 1)), [am("dc7")])
            d7 = store(blk("dc7", d8), [am("dc6")])
            d6 = store(blk("dc6", d7), [am("dc5")])
            d5 = store(blk("dc5", torch.cat((d6, syn1), 1)), [am("dc4")])
            d4 = store(blk("dc4", d5), [am("dc3")])
            d3 = store(blk("dc3", d4), [am("dc2"), am("dc2.up")])
            d2 = store(blk("dc2", torch.cat((d3, syn0), 1)), [am("dc1")])
            d1 = blk("dc1", d2)  # fp32 accumulators feed dc0 directly
            outs.append(F.conv3d(d1, sd["dc0.weight"], sd.get("dc0.bias")))
        pred = torch.sigmoid(torch.cat(outs, 0))
    fc = so.assemble(pred[:, 0].numpy(), g, m["overlap"])
    tc = so.assemble(pred[:, 1].numpy(), g, m["overlap"])
    e = max(np.abs(fc - z["fc"]).max(), np.abs(tc - z["tc"]).max())
    d_fc, d_tc = dice(fc, z["fc_mask"]), dice(tc, z["tc_mask"])
    flips = int(((fc > 0.5) != z["fc_mask"]).sum() + ((tc > 0.5) != z["tc_mask"]).sum())
    if verbose:
        print(f"{name}: max-abs {e:.2e}  Dice FC {d_fc:.5f} TC {d_tc:.5f}  mask flips {flips}")
    return e, d_fc, d_tc


LAYERS = [n for n, _, _, _ in so.UNET_LAYERS]

if __name__ == "__main__":
    name = sys.argv[1] if len(sys.argv) > 1 else "seg_small_pertap"
    torch.set_num_threads(os.cpu_count())
    print("all fp16 (shipped r01):")
    run(name, {})
    print("weights hi+lo everywhere, activations fp16:")
    run(name, {n: ("hl", "h") for n in LAYERS})
    print("activations hi+lo everywhere, weights fp16-EF:")
    run(name, {n: ("h", "hl") for n in LAYERS})
    print("both hi+lo (3-term):")
    run(name, {n: ("hl", "hl") for n in LAYERS})
    print("mixed with fp16 lo planes (dc2's skip input and dc1's input hi+lo, codes 4 / 2):")
    run(name, {"dc2.skip": ("h", "hl"), "dc1": ("h", "hl")})
    print("mixed with e4m3 lo planes (codes 6 / 7, the default):")
    run(name, {"dc2.skip": ("h", "l8"), "dc1": ("h", "l8")})
