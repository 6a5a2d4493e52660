"""CPU tier: UNet.weights_init (SURVEY row a6; reference oai_analysis/segmentation/networks.py:71-78, reached through
initialize_model(ckpoint_path=None), utils.py:42-44): xavier_normal_ on every conv weight, zero bias, BatchNorm left at
its defaults -- checked statistically, and draw for draw against the reference's nn.Module restated below."""
import math

import numpy as np
import pytest
import torch
from torch import nn

from helpers import load_golden
from oai_analysis_2_b200.segmentation.networks import UNet
from oai_analysis_2_b200.segmentation.utils import initialize_model
from oracle.seg_oracle import make_unet_state_dict


def test_weights_init_statistics():
    torch.manual_seed(7)
    net = UNet(1, 2, bias=True, BN=True)
    assert all(float(v.abs().max()) == 0 for k, v in net.state_dict().items() if k.endswith(".0.weight"))
    initialize_model(net, ckpoint_path=None)        # -> weights_init()
    sd = net.state_dict()
    for key, w in sd.items():
        if key.endswith(".0.weight") or key == "dc0.weight":
            k3 = int(np.prod(w.shape[2:]))
            # torch's fan computation on the STORED shape: fan_in = size(1) k^3, fan_out = size(0) k^3 (for a
            # ConvTranspose3d weight [cin, cout, ...] that swaps the roles, exactly as in the reference)
            std = math.sqrt(2.0 / ((w.shape[0] + w.shape[1]) * k3))
            n = w.numel()
            assert abs(float(w.std()) - std) < 5 * std / math.sqrt(2 * n) + 1e-3 * std, key
            assert abs(float(w.mean())) < 5 * std / math.sqrt(n), key
        elif key.endswith(".0.bias") or key == "dc0.bias":
            assert float(w.abs().max()) == 0, key
        elif key.endswith(".1.weight") or key.endswith(".1.running_var"):
            assert torch.equal(w, torch.ones_like(w)), key
        elif key.endswith(".1.bias") or key.endswith(".1.running_mean"):
            assert torch.equal(w, torch.zeros_like(w)), key


def test_weights_init_invalidates_packed_handles_and_keeps_keys():
    net = UNet(1, 3, bias=False, BN=False)
    keys = set(net.state_dict())
    assert "ec0.0.bias" not in keys and "ec0.1.weight" not in keys and net.state_dict()["dc0.weight"].shape == (3, 64, 1, 1, 1)
    net._handles["stale"] = object()
    net.weights_init()
    assert net._handles == {} and set(net.state_dict()) == keys


class RefUNet(nn.Module):
    """The reference UNet as an nn.Module (networks.py:39-66 constructor, encoder/decoder blocks :80-107, weights_init
    :71-78): submodules registered in the reference's order -- ec0..ec7 at :43-50, pool0..2 at :52-54, dc9..dc1 at
    :56-64, dc0 at :66 (SURVEY §2.2 and row a4) -- so self.modules() visits the conv layers, and weights_init draws, in
    the order the reference does.  Its state-dict keys and shapes are pinned to the reference's own by
    test_reference_module_takes_the_golden_fixture_state_dicts.  forward() is not needed here."""

    def __init__(self, in_channel, n_classes, bias=False, BN=False):
        super().__init__()
        for name, ci, co in (("ec0", in_channel, 32), ("ec1", 32, 64), ("ec2", 64, 64), ("ec3", 64, 128),
                             ("ec4", 128, 128), ("ec5", 128, 256), ("ec6", 256, 256), ("ec7", 256, 512)):
            setattr(self, name, self.block(nn.Conv3d(ci, co, 3, stride=1, padding=1, bias=bias), co, BN))
        self.pool0, self.pool1, self.pool2 = nn.MaxPool3d(2), nn.MaxPool3d(2), nn.MaxPool3d(2)
        for name, ci, co, k, s, p in (("dc9", 512, 512, 2, 2, 0), ("dc8", 256 + 512, 256, 3, 1, 1),
                                      ("dc7", 256, 256, 3, 1, 1), ("dc6", 256, 256, 2, 2, 0),
                                      ("dc5", 128 + 256, 128, 3, 1, 1), ("dc4", 128, 128, 3, 1, 1),
                                      ("dc3", 128, 128, 2, 2, 0), ("dc2", 64 + 128, 64, 3, 1, 1),
                                      ("dc1", 64, 64, 3, 1, 1)):
            setattr(self, name, self.block(nn.ConvTranspose3d(ci, co, k, stride=s, padding=p, bias=bias), co, BN))
        self.dc0 = nn.Conv3d(64, n_classes, 1, bias=bias)

    @staticmethod
    def block(conv, co, BN):
        return nn.Sequential(conv, nn.BatchNorm3d(co), nn.ReLU()) if BN else nn.Sequential(conv, nn.ReLU())

    def weights_init(self):
        for m in self.modules():
            if "Conv" in m.__class__.__name__:
                nn.init.xavier_normal_(m.weight.data)
                if m.bias is not None:
                    m.bias.data.zero_()


@pytest.mark.parametrize("name", ["seg_small_pertap", "seg_small_nobn"])
def test_reference_module_takes_the_golden_fixture_state_dicts(name):
    """The reference's own checkpoint loader (utils.py:20-41, strict) loaded exactly these state dicts into its UNet to
    produce tests/golden/<name>.npz (make_golden.py), so they carry the reference's keys and shapes: every transposed
    conv's [cin, cout, k, k, k] layout, dc0 as a 1x1x1 conv with its bias.  The restatement must take them the same
    way (a missing / unexpected key or a shape mismatch raises)."""
    _, m = load_golden(name)
    sd = make_unet_state_dict(m["seed"], 1, 2, m["bias"], m["BN"], True, m["head_gain"], m["head_bias"])
    ref = RefUNet(1, 2, bias=m["bias"], BN=m["BN"])
    ref.load_state_dict(sd, strict=True)


def test_weights_init_draws_match_the_reference_module():
    """Same seed, same draw order: the state dict equals the reference UNet's after its own weights_init()."""
    torch.manual_seed(1234)
    ref = RefUNet(1, 2, bias=True, BN=True)
    torch.manual_seed(99)
    ref.weights_init()
    torch.manual_seed(99)
    net = UNet(1, 2, bias=True, BN=True)
    net.weights_init()
    rsd, sd = ref.state_dict(), net.state_dict()
    assert set(rsd) == set(sd)
    for k in rsd:
        if rsd[k].is_floating_point() and not (k.endswith(".0.bias") or k == "dc0.bias"):
            assert torch.equal(rsd[k], sd[k]), k
        elif k.endswith(".0.bias") or k == "dc0.bias":
            assert float(sd[k].abs().max()) == 0 and float(rsd[k].abs().max()) == 0
