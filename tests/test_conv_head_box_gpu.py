"""GPU tier: oai_conv3d_igemm_head (dc1 fused with the dc0 head, sigmoid / mask / logits and the assembler) against
fp64 conv -> bias -> relu -> 1x1 head -> sigmoid / mask / logit -> oracle.seg_oracle.assemble, for every head_dot
instantiation (ncls 1-4) and the runtime-ncls path (5-8), every out_mode, both formats, row-shared and kh-shared (the
interior (h, w) box as oai_conv3d_igemm_box runs it: 32 columns plus an overlapping 8-wide strip); and the bf16 forms of
the split maxpool and the stem."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import conv_cases as cc
from test_conv_conformance_gpu import _conv

pytestmark = pytest.mark.gpu

# name, volume (z, y, x), patch (x, y, z), overlap (x, y, z), flags; tiles are cut by the volume edge along every axis
HEAD_GEOMS = [
    ("row_shared", (9, 21, 150), (128, 8, 6), (16, 2, 1), 0),           # tile 6 x 8 x 128: whole 128-wide rows
    ("kh_shared", (9, 37, 80), (64, 16, 6), (15, 3, 1), cc.KH_SHARED),  # interior x 15..48: 32 columns + strip
]


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("geom_case", HEAD_GEOMS, ids=lambda g: g[0])
def test_fused_head_matches_fp64_assemble(geom_case, fmt):
    _cuda()
    from oai_analysis_2_b200 import ops
    from oracle.seg_oracle import assemble, tiling_geometry
    name, shape, patch, overlap, flags = geom_case
    g = tiling_geometry(shape, patch, overlap)
    T = int(np.prod(g["grid"]))
    D, H, W = (int(v) for v in g["tile"])
    gen = torch.Generator(device="cuda").manual_seed(17 + fmt)
    # exact activations of the 64 -> 64 layer (as in test_conv_conformance_gpu.py): integers, biases in 2^-4 steps
    x = torch.randint(-1, 2, (T, D, H, W, 64), generator=gen, device="cuda").double()
    w = torch.randint(-3, 4, (64, 64, 3, 3, 3), generator=gen, device="cuda").double()
    b = torch.randint(-64, 65, (64,), generator=gen, device="cuda").double() / 16
    y = torch.relu(_conv(x, w, 0) + b)                                  # exact in fp32: what the accumulators hold
    assert (_conv(x.abs(), w.abs(), 0) + b.abs()).max().item() < 2 ** 19
    hw = (torch.randn(8, 64, generator=gen, device="cuda") * 0.05).float()
    hb = torch.randn(8, generator=gen, device="cuda").float()
    wp = ops.pack_conv_weights_ex(w.float(), 64, 0, D, H, W, 0, 1, fmt, flags)
    src = x.to(ops._DT16[fmt]).contiguous()
    geom = ops.make_geom(g["tile"], g["effective"], g["overlap"], g["grid"])
    crop = (overlap[2], overlap[0], overlap[1])
    for ncls in (1, 2, 3, 4, 5, 8):
        logit = torch.einsum("tdhwc,kc->tkdhw", y, hw[:ncls].double()) + hb[:ncls].double().view(1, ncls, 1, 1, 1)
        # fp32 head: 64 fused multiply-adds and the bias, each rounded: 2^-17 of the sum of magnitudes covers them
        tol = 2.0 ** -17 * (torch.einsum("tdhwc,kc->tkdhw", y, hw[:ncls].double().abs())
                            + hb[:ncls].double().abs().view(1, ncls, 1, 1, 1))
        for mode in (0, 1, 2):
            out = torch.full((ncls,) + tuple(shape), float("nan"), device="cuda")
            ops.conv3d_igemm_head(src, wp, b.float(), hw[:ncls].contiguous(), hb[:ncls].contiguous(), out, geom, 0,
                                  crop, out_mode=mode, ab_format=fmt, flags=flags)
            torch.cuda.synchronize()
            got = out.cpu().numpy()
            assert np.isfinite(got).all(), f"{name} ncls {ncls} mode {mode}: voxels never written"
            worst = 0.0
            for k in range(ncls):
                lk, tk = logit[:, k].cpu().numpy(), tol[:, k].cpu().numpy()
                if mode == 0:
                    ref, bound = 1 / (1 + np.exp(-lk)), tk / 4 + 4e-6   # sigmoid' <= 1/4; __expf and the division
                elif mode == 1:
                    ref, bound = (lk > 0).astype(np.float64), np.where(np.abs(lk) <= tk, np.inf, 0.0)
                else:
                    ref, bound = lk, tk
                ref, bound = assemble(ref, g, overlap), assemble(bound, g, overlap)   # the shell: exactly 0
                err = np.abs(got[k] - ref)
                assert (err <= bound).all(), (f"{name} fmt {fmt} ncls {ncls} mode {mode} class {k}: "
                                              f"max error {err.max()} over the bound")
                worst = max(worst, float(np.max(np.where(np.isinf(bound), 0, err))))
            print(f"head {name} fmt {fmt} ncls {ncls} out_mode {mode}: max error {worst:.3g}")


def _bf16_ulp(v):
    a = v.abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - 7)


def test_split_maxpool_bf16_is_exact():
    _cuda()
    from oai_analysis_2_b200 import ops
    x = torch.randn(2, 4, 8, 16, 24, device="cuda") * 3
    s = ops.split16(x, 1)
    both = ops.maxpool2(s, 1, in_split=True, out_split=True)
    got = both[..., :24].float() + both[..., 24:].float()
    full = s[..., :24].float() + s[..., 24:].float()
    assert torch.equal(got, F.max_pool3d(full.permute(0, 4, 1, 2, 3), 2).permute(0, 2, 3, 4, 1))
    hi_only = ops.maxpool2(s, 1, in_split=True, out_split=False)
    assert torch.equal(hi_only, ops.maxpool2(s[..., :24].contiguous(), 1))
    plain = ops.maxpool2(x.bfloat16(), 1)
    assert torch.equal(plain, F.max_pool3d(x.bfloat16().float().permute(0, 4, 1, 2, 3), 2)
                       .permute(0, 2, 3, 4, 1).bfloat16())


@pytest.mark.parametrize("out_split", [False, True])
def test_stem_bf16_within_one_ulp_of_fp64(out_split):
    _cuda()
    from oai_analysis_2_b200 import ops
    from oracle.seg_oracle import partition
    rng = np.random.default_rng(1)
    vol = rng.standard_normal((11, 37, 29)).astype(np.float32)
    patch, overlap = [16, 24, 8], (4, 6, 2)
    tiles, g = partition(vol, patch, overlap)
    w = torch.randn(32, 1, 3, 3, 3) * 0.2
    b = torch.randn(32) * 0.1
    ref = F.relu(F.conv3d(tiles.double(), w.double(), b.double(), padding=1)).permute(0, 2, 3, 4, 1)
    geom = ops.make_geom(g["tile"], g["effective"], g["overlap"], g["grid"])
    got = ops.seg_stem(torch.from_numpy(vol).cuda(), geom, 0, tiles.shape[0], w.reshape(32, 27).t().contiguous().cuda(),
                       b.cuda(), ab_format=1, out_split=out_split).double().cpu()
    assert got.dtype == torch.float64 and got.shape[-1] == (64 if out_split else 32)
    hi = got[..., :32]
    # the fp32 accumulation of 27 products errs by at most 2^-18 of sum |x| |w| (far below a bf16 ulp unless the sum
    # cancels): the rounded output is within one ulp of fp64
    mag = F.conv3d(tiles.double().abs(), w.double().abs(), b.double().abs(), padding=1).permute(0, 2, 3, 4, 1)
    assert ((hi - ref).abs() <= _bf16_ulp(ref) + 2.0 ** -18 * mag).all()
    if out_split:
        # hi + lo: the lo rounding (2^-8 of an ulp) plus the fp32 accumulation
        both = hi + got[..., 32:]
        assert ((both - ref).abs() <= _bf16_ulp(ref) * 2.0 ** -8 + 2.0 ** -18 * mag).all()
