"""CPU tier: kh-shared mode of conv_igemm_kernel (conv_igemm.cuh kModeKhShared) through a software model of its
schedule, fed with the REAL packed weights: M tiles of TH x TW voxels placed from an arbitrary (h_lo, w_lo), one
(TH + 2) x TW TMA box per (chunk, kw), the three kh taps read TW rows apart in the swizzled stage, weight blocks
ordered (chunk, kw) with kh x kd inside.  Plus the tile plan seg_net.cu uses for dc2 / dc1 at the production tile."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conv_emulator import _box, _read_operand, _swizzled_store, build_chunks
from oai_analysis_2_b200 import ops

KH_SHARED = 256   # kConvFlagKhShared
MODE_KH_SHARED = 4


def tile_width(h_cnt, w_cnt, H, W):
    """conv_run's choice: the fewest M tiles over the box, the widest tile on a tie."""
    best = None
    for tw in (32, 16, 8):
        if tw > W or 128 // tw > H:
            continue
        n = -(-w_cnt // tw) * -(-h_cnt // (128 // tw))
        if best is None or n < best[0]:
            best = (n, tw)
    return best[1]


def tile_origins(h_lo, h_cnt, w_lo, w_cnt, H, W, tw):
    """decode_unit: origins from (h_lo, w_lo) in steps of the tile, the last one clamped inside the grid."""
    th = 128 // tw
    return [(min(h_lo + i * th, H - th), min(w_lo + j * tw, W - tw))
            for i in range(-(-h_cnt // th)) for j in range(-(-w_cnt // tw))]


def w_launches(w_lo, w_hi):
    """seg_net.cu conv_w_box: the largest multiple of 32 columns, then a strip of 8-multiples over the last columns."""
    w_cnt = w_hi - w_lo + 1
    main = w_cnt // 32 * 32
    out = [(w_lo, main)] if main else []
    rest = w_cnt - main
    if rest:
        n = min(-(-rest // 8) * 8, w_cnt)
        out.append((w_hi + 1 - n, n))
    return out


def emulate_kh_shared(x0, x1, wpack, bias, plan, cout, region, tw, out, relu=True):
    """x0 / x1: [NT, D, H, W, C] float16 (x1 may be None); writes the computed tiles into `out` (float32)."""
    NT, D, H, W, c0 = x0.shape
    c1 = 0 if x1 is None else x1.shape[-1]
    chunks = build_chunks(c0, c1, 1)
    R, nblk, wbytes, cph = plan["R"], plan["nblk"], plan["wblock_bytes"], plan["cout_per_half"]
    assert plan["mode"] == MODE_KH_SHARED and plan["nhalf"] == 1 and nblk == 3 * len(chunks)
    th, rb = 128 // tw, 128
    xs = (x0.view(np.uint16), None if x1 is None else x1.view(np.uint16))
    w16 = np.frombuffer(wpack.tobytes(), dtype=np.uint16)
    d_lo, d_cnt, h_lo, h_cnt, w_lo, w_cnt = region
    for n in range(NT):
        for d0 in range(d_lo, d_lo + d_cnt, R):
            rv = min(R, d_lo + d_cnt - d0)
            for h0, w0 in tile_origins(h_lo, h_cnt, w_lo, w_cnt, H, W, tw):
                acc = np.zeros((R, 128, cph), dtype=np.float32)
                for b in range(nblk):
                    c, kw = b // 3, b % 3
                    blk = w16[(b * wbytes) // 2:((b + 1) * wbytes) // 2]
                    src, cc = xs[chunks[c][0]], chunks[c][1]
                    for dp in range(max(0, d0 - 1), min(D - 1, d0 + rv) + 1):
                        # one box of TH + 2 rows x TW voxels at (w0 + kw - 1, h0 - 1), zero fill outside the grid
                        stage = _swizzled_store(_box(src, n, dp, h0 - 1, w0 + kw - 1, cc, th + 2, tw))
                        a_first = dp - 2 - d0 + 1
                        for kh in range(3):
                            # tap kh: the same stage, kh * TW rows (a whole number of 1024-byte atoms) further
                            assert (kh * tw * rb) % 1024 == 0
                            A = _read_operand(stage, kh * tw * rb, 128).view(np.float16).astype(np.float32)
                            for ti in range(3):   # kd = 2 - ti feeds accumulator a_first + ti
                                a = a_first + ti
                                if 0 <= a < rv:
                                    Bm = _read_operand(blk, (kh * 3 + ti) * cph * rb, cph)
                                    acc[a] += A @ Bm.view(np.float16).astype(np.float32).T
                for a in range(rv):
                    v = acc[a] + bias[None, :]
                    if relu:
                        v = np.maximum(v, 0)
                    out[n, d0 + a, h0:h0 + th, w0:w0 + tw] = v.reshape(th, tw, cph)


def _layer(D, H, W, c0, c1, cout, seed):
    g = torch.Generator().manual_seed(seed)
    x0 = torch.randn(1, D, H, W, c0, generator=g).half()
    x1 = torch.randn(1, D, H, W, c1, generator=g).half() if c1 else None
    w = (torch.randn(cout, c0 + c1, 3, 3, 3, generator=g) / (27 * (c0 + c1)) ** 0.5).half().float()
    bias = torch.randn(cout, generator=g)
    x = x0 if x1 is None else torch.cat((x0, x1), -1)
    ref = F.relu(F.conv3d(x.float().permute(0, 4, 1, 2, 3), w, bias, padding=1)).permute(0, 2, 3, 4, 1).numpy()
    return x0, x1, w, bias, ref


def test_packed_blocks_are_chunk_kw_major_with_kh_kd_inside():
    cout, cin, D, H, W = 64, 64, 4, 16, 128
    w = torch.randn(cout, cin, 3, 3, 3, generator=torch.Generator().manual_seed(1)) * 0.05
    plan = ops.conv_plan(D, H, W, cin, 0, cout, False, KH_SHARED)
    row = ops.conv_plan(D, H, W, cin, 0, cout, False, 0)
    assert plan["mode"] == MODE_KH_SHARED and row["mode"] == 0
    # same block size and count as a row-shared plan: only the order of the taps inside differs
    assert (plan["nblk"], plan["wblock_bytes"]) == (row["nblk"], row["wblock_bytes"])
    wp = ops.pack_conv_weights(w, cin, 0, D, H, W, False, 0, KH_SHARED, device="cpu").numpy()
    wr = ops.pack_conv_weights(w, cin, 0, D, H, W, False, 0, 0, device="cpu").numpy()
    w16, r16 = np.frombuffer(wp.tobytes(), np.uint16), np.frombuffer(wr.tobytes(), np.uint16)
    nb = plan["wblock_bytes"] // 2
    for kw in range(3):
        for kh in range(3):
            for ti in range(3):
                got = _read_operand(w16[kw * nb:(kw + 1) * nb], (kh * 3 + ti) * cout * 128, cout)
                want = _read_operand(r16[kh * nb:(kh + 1) * nb], (kw * 3 + ti) * cout * 128, cout)
                assert np.array_equal(got, want), (kw, kh, ti)


@pytest.mark.parametrize("tw", [32, 16, 8])
def test_emulated_kh_shared_tiles_match_conv3d_from_odd_origin(tw):
    """Region starting at odd h and w, last tile row clamped inside the grid, two sources (dc2's concatenation)."""
    D, H, W, c0, c1, cout = 5, 21, 45, 64, 64, 64
    x0, x1, w, bias, ref = _layer(D, H, W, c0, c1, cout, 2 + tw)
    region = (1, 3, 5, 13, 7, 33)
    plan = ops.conv_plan(region[1], H, W, c0, c1, cout, False, KH_SHARED)
    wp = ops.pack_conv_weights(w, c0, c1, D, H, W, False, 0, KH_SHARED, device="cpu").numpy()
    out = np.full((1, D, H, W, cout), np.nan, dtype=np.float32)
    emulate_kh_shared(x0.numpy(), x1.numpy(), wp, bias.numpy(), plan, cout, region, tw, out)
    covered = np.zeros((H, W), dtype=bool)
    th = 128 // tw
    for h0, w0 in tile_origins(*region[2:], H, W, tw):
        covered[h0:h0 + th, w0:w0 + tw] = True
    assert covered[5:18, 7:40].all()
    d = slice(1, 4)
    assert np.abs(out[:, d][:, :, covered] - ref[:, d][:, :, covered]).max() < 2e-3
    # nothing outside the computed tiles and d-slices is touched
    assert np.isnan(out[:, d][:, :, ~covered]).all()
    assert np.isnan(out[:, :1]).all() and np.isnan(out[:, 4:]).all()


def test_emulated_main_tiles_and_strip_cover_a_box_not_a_multiple_of_32():
    """dc2's split: 32-wide main tiles plus an 8-wide strip over the last columns, overlapping the main tiles."""
    D, H, W, c0, cout = 3, 24, 48, 64, 64
    x0, _, w, bias, ref = _layer(D, H, W, c0, 0, cout, 11)
    plan = ops.conv_plan(D, H, W, c0, 0, cout, False, KH_SHARED)
    wp = ops.pack_conv_weights(w, c0, 0, D, H, W, False, 0, KH_SHARED, device="cpu").numpy()
    h_lo, h_cnt, w_lo, w_hi = 3, 17, 5, 38   # 34 columns: 32 + a strip of 8 at [31, 38]
    launches = w_launches(w_lo, w_hi)
    assert launches == [(5, 32), (31, 8)]
    assert [tile_width(h_cnt, n, H, W) for _, n in launches] == [32, 8]
    out = np.full((1, D, H, W, cout), np.nan, dtype=np.float32)
    for lo, n in launches:
        emulate_kh_shared(x0.numpy(), None, wp, bias.numpy(), plan, cout, (0, D, h_lo, h_cnt, lo, n),
                          tile_width(h_cnt, n, H, W), out)
    box = (slice(None), slice(None), slice(h_lo, h_lo + h_cnt), slice(w_lo, w_hi + 1))
    assert np.abs(out[box] - ref[box]).max() < 2e-3
    assert np.isnan(out[:, :, :, :w_lo]).all() and np.isnan(out[:, :, :, w_hi + 1:]).all()


def test_production_plan_tiles_and_nan_poisoned_dc2_halo():
    """At the production tile (32 x 128 x 128, overlap 8 x 16 x 16) dc1 runs 72 tiles of 32 x 4 per d-slice and dc2
    75 + 7 (main + strip) instead of 96 / 98 row tiles; dc1's tiles read nothing of dc2's output outside the tiles dc2
    computes: poisoning the rest with NaN leaves dc1's needed box finite and unchanged."""
    from oai_analysis_2_b200.segmentation.networks import UNet
    B = UNet.needed_regions((32, 128, 128), (8, 16, 16))
    H = W = 128
    cover = {}
    for name, nexp in (("dc1", [72]), ("dc2", [75, 7])):
        lo, hi = B[name][0], B[name][1]
        h_lo, h_cnt = int(lo[1]), int(hi[1] - lo[1] + 1)
        m = np.zeros((H, W), dtype=bool)
        counts = []
        for w_lo, w_cnt in w_launches(int(lo[2]), int(hi[2])):
            tw = tile_width(h_cnt, w_cnt, H, W)
            tiles = tile_origins(h_lo, h_cnt, w_lo, w_cnt, H, W, tw)
            counts.append(len(tiles))
            for h0, w0 in tiles:
                m[h0:h0 + 128 // tw, w0:w0 + tw] = True
        assert counts == nexp, (name, counts)
        assert m[lo[1]:hi[1] + 1, lo[2]:hi[2] + 1].all()
        cover[name] = m
    # a stand-in for dc2's output over its d range (8 channels keep the CPU conv small), poisoned outside its tiles
    g = torch.Generator().manual_seed(4)
    d2 = torch.randn(1, 8, 18, H, W, generator=g)
    w1 = torch.randn(8, 8, 3, 3, 3, generator=g)
    ref = F.conv3d(d2, w1, padding=1)
    poisoned = d2.clone()
    poisoned[..., torch.from_numpy(~cover["dc2"])] = float("nan")
    got = F.conv3d(poisoned, w1, padding=1)
    keep = torch.from_numpy(cover["dc1"])
    inner = got[:, :, 1:17][..., keep]   # dc1's d range is dc2's without its first and last slice
    assert not torch.isnan(inner).any()
    assert torch.equal(inner, ref[:, :, 1:17][..., keep])
