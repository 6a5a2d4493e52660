"""GPU tier: the 8-bit lo terms (codes 6 / 7).

* layer level, through oai_conv3d_igemm_lo8: a source stored as fp16 hi + e4m3 lo plane, its lo chunks issued as
  block-scaled 8-bit MMAs into the same accumulators as the fp16 chunks, against torch fp64 and against the fp16 lo
  planes of codes 4 / 2 on the same inputs, in the row-shared, kh-shared and per-tap modes;
* the producer epilogue's e4m3 plane against the fp16 lo plane of the same launch;
* the production tile: the default mixed plan (6 / 7) against OAI_B200_SEG_LO8=0 (4 / 2)."""
import pytest
import torch
import torch.nn.functional as F

from oai_analysis_2_b200 import ops
from oracle import seg_oracle

pytestmark = pytest.mark.gpu

KH_SHARED = 256


def _ref(x, w, bias):
    out = F.conv3d(x.double().permute(0, 4, 1, 2, 3), w.double(), bias.double(), padding=1)
    return F.relu(out).permute(0, 2, 3, 4, 1)


@pytest.mark.parametrize("terms,c0,c1,dims,flags", [
    (7, 64, 0, (5, 8, 128), 0),             # dc1's shape, row-shared (whole 128-wide rows)
    (7, 64, 0, (5, 8, 128), KH_SHARED),     # kh-shared tiles
    (7, 128, 0, (4, 8, 16), 0),             # per-tap tiles, two lo8 chunks
    (6, 128, 64, (5, 8, 128), 0),           # dc2's shape: the skip source split
    (6, 128, 64, (9, 8, 128), KH_SHARED),   # d range in R = 5 + 4 accumulators
    (6, 64, 64, (4, 8, 16), 0),
])
def test_lo8_terms_match_fp64_and_fp16_lo(terms, c0, c1, dims, flags):
    D, H, W = dims
    cout = 64
    g = torch.Generator().manual_seed(terms * 100 + c0 + D)
    # the unsplit source (terms 6: source 0) is exact in fp16, so every difference below comes from the split source
    x0 = torch.randn(2, D, H, W, c0, generator=g) * 3
    x0 = x0.half().float() if terms == 6 else x0
    x1 = torch.randn(2, D, H, W, c1, generator=g) * 3 if c1 else None
    cin = c0 + c1
    w = (torch.randn(cout, cin, 3, 3, 3, generator=g) / (27 * cin) ** 0.5).half().float()
    bias = torch.randn(cout, generator=g)
    ref = _ref(x0 if x1 is None else torch.cat((x0, x1), -1), w, bias)

    def run(s0, s1, terms, **kw):
        wp = ops.pack_conv_weights_ex(w, c0, c1, D, H, W, 0, terms, flags=flags)
        out = ops.conv3d_igemm_ex(s0, s1, wp, bias.cuda(), cout, c0, c1, 0, True, 0, terms, flags=flags,
                                  out_split=True, **kw)
        return out[..., :cout].double().cpu() + out[..., cout:].double().cpu()   # hi + lo: fp32-level output

    split = x1 if terms == 6 else x0   # the source read with a lo term
    hi, lo8 = ops.split_lo8(split.cuda())
    both = ops.split16(split.cuda())
    if terms == 6:
        plain0 = x0.cuda().half()
        out8 = run(plain0, hi, 6, in_lo8=lo8)
        out16 = run(ops.split16(x0.cuda()), both, 4, in_split=True)   # in_split: both sources [hi | lo]
        out1 = run(plain0, hi, 1)
    else:
        out8 = run(hi, None, 7, in_lo8=lo8)
        out16 = run(both, None, 2, in_split=True)
        out1 = run(hi, None, 1)
    torch.cuda.synchronize()
    e8, e16, e1 = [(o - ref).abs().max().item() for o in (out8, out16, out1)]
    d = (out8 - out16).abs().max().item()
    print(f"terms {terms} {dims} flags {flags}: |ref| {ref.abs().max().item():.2f}  error lo8 {e8:.2e}  "
          f"lo16 {e16:.2e}  no lo term {e1:.2e}  lo8 vs lo16 {d:.2e}")
    # the e4m3 lo term keeps ~2^-16 of the activation against 2^-12 without it: 16x expected, 4x required
    assert e8 < e1 / 4 and d < e1 / 4
    assert e16 < e1 / 4


def test_lo8_output_plane_matches_fp16_lo():
    D, H, W, c0, cout = 4, 8, 128, 64, 64
    g = torch.Generator().manual_seed(3)
    x = torch.randn(1, D, H, W, c0, generator=g).cuda().half()
    w = torch.randn(cout, c0, 3, 3, 3, generator=g) / (27 * c0) ** 0.5
    bias = torch.randn(cout, generator=g).cuda()
    wp = ops.pack_conv_weights_ex(w, c0, 0, D, H, W, 0, 1)
    both = ops.conv3d_igemm_ex(x, None, wp, bias, cout, c0, 0, 0, True, 0, 1, out_split=True)
    hi, lo8 = ops.conv3d_igemm_ex(x, None, wp, bias, cout, c0, 0, 0, True, 0, 1, out_lo8=True)
    torch.cuda.synchronize()
    assert torch.equal(hi, both[..., :cout])
    lo16 = both[..., cout:].float()
    got = ops.lo8_value(lo8)
    # e4m3 keeps 4 significant bits: half an ulp of the value, or the subnormal step 2^-9 * 2^-11
    tol = lo16.abs() * 2.0 ** -4 + 2.0 ** -20
    assert ((got - lo16).abs() <= tol).all()
    assert (got != 0).float().mean().item() > 0.5


PATCH, OVERLAP = (128, 128, 32), (16, 16, 8)   # x, y, z: the production tile


def test_mixed_lo8_matches_fp16_lo_at_production_tile(monkeypatch):
    sd = seg_oracle.make_unet_state_dict(13, 1, 2, True, True, True)
    vol = torch.from_numpy(seg_oracle.synthetic_knee((20, 150, 96), 7)).float().cuda().contiguous()

    def run():
        h = ops.SegHandle(sd, 1, 2, True, True, PATCH, OVERLAP)
        ws = torch.zeros((h.workspace_bytes(vol.shape),), dtype=torch.uint8, device="cuda")
        out = h.forward(vol, 0, 0, workspace=ws)
        torch.cuda.synchronize()
        return out.cpu()

    assert list(ops.seg_layer_terms(1))[-2:] == [6, 7]
    new = run()
    monkeypatch.setenv("OAI_B200_SEG_LO8", "0")
    assert list(ops.seg_layer_terms(1))[-2:] == [4, 2]
    old = run()
    err = (new - old).abs().max().item()
    flips = ((new > 0.5) != (old > 0.5)).float().mean().item()
    print(f"mixed lo8 vs fp16 lo: probability max-abs {err:.3e}, mask voxels differing {flips:.3e}")
    assert torch.isfinite(new).all()
    assert err <= 1e-2, err
    assert flips <= 1e-4, flips
