"""CPU tier: the 8-bit lo terms (codes 6 / 7) replayed from the real packed weights.

The packer's blocks of a row-shared layer are unpacked chunk by chunk -- fp16 rows of the hi chunks, e4m3 rows of the
lo-plane chunks (64-byte rows, SWIZZLE_64B) and the two UE8M0 block-scale words after the blocks -- and the layer is
recomputed the way the kernel's MMAs do it: hi chunks as fp16 products, lo8 chunks as e4m3 x e4m3 products scaled by
2^-(S+T), all summed in fp32.  Against an fp64 convolution of the un-rounded activations the error stays below 2^-14
of sum |x| |w| per output, several times below the error of the fp16 hi term alone."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oai_analysis_2_b200 import ops


def _chunks(c0, c1, terms):
    """(source, first channel, lo8) of every K chunk, in the order api_conv.cu::build_chunks lists them."""
    out = []
    for src, c in ((0, c0), (1, c1)):
        if c == 0:
            continue
        out += [(src, j, False) for j in range(0, c, 64)]
        if (terms == 6 and src == 1) or (terms == 7 and src == 0):
            out += [(src, j, True) for j in range(0, c, 64)]
    return out


def _unswizzle(block, nrows, row_bytes):
    """[nrows, row_bytes] bytes of a K-major swizzled block: 16-byte chunk j of row r sits at chunk j ^ f(r)."""
    img = block[:nrows * row_bytes].reshape(nrows, row_bytes // 16, 16)
    r = np.arange(nrows)
    xor = r % 8 if row_bytes == 128 else (r // 2) % 4
    out = np.empty_like(img)
    for j in range(row_bytes // 16):
        out[:, j] = img[r, j ^ xor]
    return out.reshape(nrows, row_bytes)


def _unpack(wpack, plan, c0, c1, terms):
    """Row-shared layout -> per chunk the [cout, 64, 27] weights it multiplies (fp16 values, or e4m3 bytes), S, T."""
    cph, nblk, wbytes = plan["cout_per_half"], plan["nblk"], plan["wblock_bytes"]
    assert plan["mode"] == 0 and plan["nhalf"] == 1
    chunks = _chunks(c0, c1, terms)
    assert plan["nchunks"] == len(chunks) and nblk == 3 * len(chunks)
    w16 = [np.zeros((cph, 64, 27), np.float32) for _ in chunks]
    w8 = [np.zeros((cph, 64, 27), np.uint8) for _ in chunks]
    for b in range(nblk):
        c, kh = divmod(b, 3)
        lo8 = chunks[c][2]
        rb = 64 if lo8 else 128
        rows = _unswizzle(wpack[b * wbytes:(b + 1) * wbytes], 9 * cph, rb)
        vals = rows if lo8 else rows.view(np.float16).astype(np.float32)
        for kwi in range(3):
            for ti in range(3):
                tap = ((2 - ti) * 3 + kh) * 3 + kwi
                r = (kwi * 3 + ti) * cph
                (w8 if lo8 else w16)[c][:, :, tap] = vals[r:r + cph]
        if lo8:   # the lo8 rows fill the first half of the block
            assert not wpack[b * wbytes + wbytes // 2:(b + 1) * wbytes].any()
    sf = wpack[nblk * wbytes:nblk * wbytes + 8]
    assert wpack.size == nblk * wbytes + 16
    return chunks, w16, w8, 127 - int(sf[0]), 127 - int(sf[4])


@pytest.mark.parametrize("terms,c0,c1", [(7, 64, 0), (7, 128, 0), (6, 64, 64), (6, 128, 64)])
def test_lo8_chunks_reproduce_fp64_conv(terms, c0, c1):
    D, H, W, cout = 4, 2, 128, 64
    g = torch.Generator().manual_seed(terms + c0)
    cin = c0 + c1
    x = torch.randn(1, D, H, W, cin, generator=g) * 3
    w = (torch.randn(cout, cin, 3, 3, 3, generator=g) / (27 * cin) ** 0.5).half().float()   # exact fp16 weights
    split = slice(c0, cin) if terms == 6 else slice(0, c0)
    x[..., :c0] = x[..., :c0].half().float() if terms == 6 else x[..., :c0]   # the unsplit source is exact fp16
    plan = ops.conv_plan_ex(D, H, W, c0, c1, cout, 0, terms)
    wpack = ops.pack_conv_weights_ex(w, c0, c1, D, H, W, 0, terms, device=None)
    chunks, w16, w8, S, T = _unpack(wpack, plan, c0, c1, terms)
    assert S == 11 and 448 / 2 < w[:, split].abs().max().item() * 2.0 ** T <= 448
    hi, lo8 = ops.split_lo8(x[..., split])
    xs = x.clone()
    xs[..., split] = hi.float()
    lo_val = lo8.view(torch.float8_e4m3fn).float()      # (x - hi) * 2^S, as e4m3
    got = torch.zeros(1, cout, D, H, W)
    for (src, cc, lo8c), a16, a8 in zip(chunks, w16, w8):
        ch = (0 if src == 0 else c0) + cc
        if lo8c:
            a = lo_val[..., ch - split.start:ch - split.start + 64]
            wk = torch.from_numpy(a8).view(torch.float8_e4m3fn).float()
            part = F.conv3d(a.permute(0, 4, 1, 2, 3), wk.reshape(cout, 64, 3, 3, 3), padding=1) * 2.0 ** -(S + T)
        else:
            a = xs[..., ch:ch + 64]
            part = F.conv3d(a.permute(0, 4, 1, 2, 3), torch.from_numpy(a16).reshape(cout, 64, 3, 3, 3), padding=1)
        got += part
    xd, wd = x.double().permute(0, 4, 1, 2, 3), w.double()
    ref = F.conv3d(xd, wd, padding=1)
    mag = F.conv3d(xd.abs(), wd.abs(), padding=1)   # sum |x| |w| per output
    err = (got.double() - ref).abs()
    bound = mag * 2.0 ** -14 + mag * 27 * cin * 2.0 ** -24   # + fp32 accumulation
    assert (err <= bound).all(), (err / mag).max().item()
    # the lo term carries its weight: without it the error is several times larger (about 16x expected)
    no_lo = F.conv3d(xs.double().permute(0, 4, 1, 2, 3), wd, padding=1)
    assert (no_lo - ref).abs().max() > 4 * err.max()


def test_lo8_plans_leave_tmem_columns_for_the_block_scales(monkeypatch):
    from oai_analysis_2_b200 import _lib
    kh = 256
    # dc2 / dc1 at the production tile: the d range in equal groups of at most 7 accumulators (448 of 512 columns)
    assert ops.conv_plan_ex(18, 98, 128, 128, 64, 64, 0, 6, kh)["R"] == 6
    assert ops.conv_plan_ex(16, 96, 128, 64, 0, 64, 0, 7, kh)["R"] == 6
    assert ops.conv_plan_ex(16, 96, 128, 64, 0, 64, 0, 2, kh)["R"] == 8   # the 16-bit codes keep every column
    assert ops.conv_plan_ex(18, 98, 128, 128, 64, 64, 0, 6, kh)["nchunks"] == 4
    with pytest.raises(_lib.OaiError, match="one-source"):
        ops.conv_plan_ex(8, 8, 128, 64, 64, 64, 0, 7)
    with pytest.raises(_lib.OaiError, match="3x3x3"):
        ops.conv_plan_ex(8, 8, 16, 64, 0, 64, 2, 7)
    assert list(ops.seg_layer_terms(1))[-2:] == [6, 7]
    monkeypatch.setenv("OAI_B200_SEG_LO8", "0")
    assert list(ops.seg_layer_terms(1))[-2:] == [4, 2]
