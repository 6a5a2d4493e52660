"""GPU tier: dc2 and dc1 in kh-shared mode compute only their needed (h, w) box at the production tile.

* every activation the segmenter leaves uncomputed is really dead: a workspace filled with NaN before the forward
  gives bit-identical probabilities to a zeroed one;
* against the row-shared plans (OAI_B200_SEG_W_HALO=0) the probabilities differ only by the reordered fp32
  accumulation of the taps."""
import numpy as np
import pytest
import torch

from oai_analysis_2_b200 import ops
from oracle import seg_oracle

pytestmark = pytest.mark.gpu

PATCH, OVERLAP = (128, 128, 32), (16, 16, 8)   # x, y, z: the production tile


@pytest.fixture(scope="module")
def knee():
    sd = seg_oracle.make_unet_state_dict(13, 1, 2, True, True, True)
    # two tiles along y, the second one cut by the volume edge (reflect padding)
    vol = torch.from_numpy(seg_oracle.synthetic_knee((20, 150, 96), 7)).float().cuda().contiguous()
    return sd, vol


def _forward(h, vol, fill):
    ws = torch.full((h.workspace_bytes(vol.shape),), fill, dtype=torch.uint8, device="cuda")
    out = h.forward(vol, 0, 0, workspace=ws)
    torch.cuda.synchronize()
    return out.cpu()


def test_dead_halo_of_every_layer_is_never_read(knee):
    sd, vol = knee
    h = ops.SegHandle(sd, 1, 2, True, True, PATCH, OVERLAP)
    clean = _forward(h, vol, 0)
    poisoned = _forward(h, vol, 0xFF)   # 0xFFFF is a NaN in fp16 and bf16
    assert torch.isfinite(clean).all()
    assert torch.equal(clean, poisoned)


def test_kh_shared_matches_row_shared_plans(knee, monkeypatch):
    sd, vol = knee
    new = _forward(ops.SegHandle(sd, 1, 2, True, True, PATCH, OVERLAP), vol, 0)
    monkeypatch.setenv("OAI_B200_SEG_W_HALO", "0")
    old = _forward(ops.SegHandle(sd, 1, 2, True, True, PATCH, OVERLAP), vol, 0)
    err = (new - old).abs().max().item()
    flips = ((new > 0.5) != (old > 0.5)).float().mean().item()
    assert err <= 1e-2, err
    assert flips <= 1e-4, flips
