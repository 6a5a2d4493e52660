"""GPU tier: the segmentation conv kernel layer by layer against exact answers -- every MMA issuer, mode, term code,
format and epilogue variant the case matrix in conv_cases.py lists (test_conv_conformance_cases.py checks on the host
that each case lands on the branch it names).

Exact operands.  Activations are small integers, weights integers (terms 3: a + b * 2^-12, so the packed hi / lo
weights are exactly a and b * 2^-12), e4m3 lo planes hold integers |l| <= 8 (worth l * 2^-S), and biases are multiples
of 2^-4.  Every product and every partial sum is then a multiple of 2^-f (f = 4, 12 or S) below 2^(23 - f) in
magnitude -- each case checks that bound before it runs -- so fp32 accumulates them exactly in any order and the answer
does not depend on how the tensor cores round.  The reference sums the taps as fp64 matmuls (exact on these values),
and every comparison is bitwise (signed zeros aside):
  * a plain 16-bit output equals rn16(y) of the exact y;
  * a [hi | lo] output has hi == rn16(y) and lo == rn16(y - hi) (hi + lo == y wherever y - hi fits the format, which
    the terms 3 cases in bf16, with their 2^-12 fractions, deliberately exceed);
  * an e4m3 lo plane equals ops.split_lo8(y) (those cases keep |y| < 512, so (y - hi) * 2^S is exact in e4m3).

Split sources are stored as two independent integer planes (they need not be a real rn16 split: the kernel only
multiplies planes), which pins the [hi | lo] channel mapping; the plane a term code must ignore (the lo half of the
unsplit source of terms 4 / 5) holds integers too.

Region launches (oai_conv3d_igemm_region's contract): into an output filled with a NaN sentinel, voxels inside the
region equal the full-layer launch, voxels outside are untouched or equal the full-layer launch, slices outside the d
range are untouched, and the written rows stay inside the region's whole M tiles."""
import math

import pytest
import torch

import conv_cases as cc
from oai_analysis_2_b200 import ops

pytestmark = pytest.mark.gpu

DT = {0: torch.float16, 1: torch.bfloat16}
DEVICE = "cuda"
SENTINEL = -1   # 0xFFFF: a NaN in both 16-bit formats (and 0xFF in the e4m3 plane)


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _ints(g, shape, lo, hi, density):
    x = torch.randint(lo, hi + 1, shape, generator=g, dtype=torch.int64, device=g.device).double()
    if density < 1.0:
        x = x * (torch.rand(shape, generator=g, dtype=torch.float64, device=g.device) < density)
    return x


def _conv(x, w, kind):
    """Exact fp64 reference: x [NT, D, H, W, cin], w conv orientation [cout, cin, taps...] -> [NT, D', H', W', cout].
    The taps are summed as matmuls; on the integer / dyadic operands here every partial sum is exact in fp64."""
    NT, D, H, W, _ = x.shape
    cout = w.shape[0]
    if kind == 1:
        return x @ w.T
    if kind == 2:
        y = x.new_zeros(NT, 2 * D, 2 * H, 2 * W, cout)
        for a in range(2):
            for b in range(2):
                for c in range(2):
                    y[:, a::2, b::2, c::2] = x @ w[:, :, a, b, c].T
        return y
    xp = torch.nn.functional.pad(x, (0, 0, 1, 1, 1, 1, 1, 1))
    y = x.new_zeros(NT, D, H, W, cout)
    for kd in range(3):
        for kh in range(3):
            for kw in range(3):
                y += xp[:, kd:kd + D, kh:kh + H, kw:kw + W] @ w[:, :, kd, kh, kw].T
    return y


def _rn16(w, fmt):
    return w.to(DT[fmt]).double()


class Layer:
    """Exact operands of one case, the tensors the kernel reads, and the exact fp64 answer."""

    def __init__(self, case, seed):
        self.case = c = case
        dev = DEVICE
        S = ops.LO8_SHIFT[c.fmt]
        lo8_src = {6: 1, 7: 0}.get(c.terms)
        self.in_split = any(cc.split_src(c.terms, s) for s in range(2))
        frac = 12 if c.terms == 3 else S if lo8_src is not None else 4
        limit = 2.0 ** (23 - frac)
        if c.out == "lo8":
            limit = min(limit, 511.0)   # |y| < 512: (y - hi) * 2^S is exact in e4m3
        taps = {0: (3, 3, 3), 1: (), 2: (2, 2, 2)}[c.kind]
        cin = c.c0 + c.c1
        density = 1.0
        # operands of the production-size layers are drawn on the device (host draws of 10^8 values take too long)
        gdev = "cuda" if c.NT * c.D * c.H * c.W * cin > 2 ** 24 else "cpu"
        for _ in range(12):
            g = torch.Generator(device=gdev).manual_seed(seed)
            xr = (-1, 1) if c.terms == 3 or lo8_src is not None or c.out == "lo8" else (-2, 2)
            hi = [_ints(g, (c.NT, c.D, c.H, c.W, ch), *xr, density) if ch else None for ch in (c.c0, c.c1)]
            lo = [_ints(g, (c.NT, c.D, c.H, c.W, ch), *xr, density) if ch else None for ch in (c.c0, c.c1)]
            l8 = _ints(g, (c.NT, c.D, c.H, c.W, (c.c0, c.c1)[lo8_src]), -8, 8, 1.0) if lo8_src is not None else None
            if c.terms == 3:
                a = torch.tensor([0.0, 2, -2, 3, -3], dtype=torch.float64, device=g.device)
                w = a[torch.randint(0, 5, (c.cout, cin) + taps, generator=g, device=g.device)]
                w = w + _ints(g, w.shape, -3, 3, 1.0) * 2.0 ** -12
            else:
                w = _ints(g, (c.cout, cin) + taps, -3, 3, 1.0)
            b_frac = torch.randint(0, 16, (c.cout,), generator=g, device=g.device).double() / 16
            b = _ints(g, (c.cout,), -8, 8, 1.0) + b_frac
            # the value of each source the kernel multiplies, and the sum of the magnitudes of the planes it multiplies
            # separately (hi * w and lo * w are separate products in the accumulation)
            vals, mags = [], []
            for s in range(2 if c.c1 else 1):
                v, m = hi[s], hi[s].abs()
                if cc.split_src(c.terms, s):
                    v, m = hi[s] + lo[s], hi[s].abs() + lo[s].abs()
                elif s == lo8_src:
                    v, m = hi[s] + l8 * 2.0 ** -S, hi[s].abs() + l8.abs() * 2.0 ** -S
                vals.append(v)
                mags.append(m)
            x = torch.cat(vals, -1).to(dev)
            xm = torch.cat(mags, -1).to(dev)
            wd = w.to(dev)
            if c.terms == 3:   # x_hi * w_hi + x_lo * w_hi + x_hi * w_lo (x_lo * w_lo is dropped by design)
                w_hi = _rn16(wd, c.fmt)
                w_lo = _rn16(wd - w_hi, c.fmt)
                xh = torch.cat([h for h in hi if h is not None], -1).to(dev)
                y = _conv(x, w_hi, c.kind) + _conv(xh, w_lo, c.kind)
                bound = _conv(xm, w_hi.abs(), c.kind) + _conv(xh.abs(), w_lo.abs(), c.kind)
                assert torch.equal(w_hi.cpu(), _rn16(w, c.fmt)) and (w_hi.cpu() - w.round()).abs().max() < 0.01
            else:
                y = _conv(x, wd, c.kind)
                bound = _conv(xm, wd.abs(), c.kind)
            y = y + b.to(dev)
            bound = bound + b.abs().to(dev)
            if bound.max().item() < limit:
                break
            density /= 2
        else:
            raise AssertionError(f"{c.name}: no operand density keeps the sums exact")
        self.bound = bound.max().item()
        self.y = torch.relu(y) if c.relu else y
        self.w, self.b = w, b.float().to(dev)
        # stored tensors
        dt = DT[c.fmt]
        self.src, self.lo8 = [], None
        for s, ch in enumerate((c.c0, c.c1)):
            if not ch:
                self.src.append(None)
                continue
            t = torch.cat((hi[s], lo[s]), -1) if self.in_split else hi[s]
            self.src.append(t.to(dt).to(dev).contiguous())
        if lo8_src is not None:
            self.lo8 = l8.float().to(torch.float8_e4m3fn).view(torch.uint8).to(dev).contiguous()
            assert torch.equal(self.lo8.view(torch.float8_e4m3fn).double(), l8.to(dev))

    def wpack(self):
        c = self.case
        if c.api == "convt2":
            return ops.pack_convt2_weights(self.w.float(), c.D, c.H, c.W, c.fmt)
        if c.api == "obase":
            return ops.pack_conv_weights(self.w.float(), c.c0, c.c1, c.D, c.H, c.W, c.kind, c.fmt, c.flags)
        return ops.pack_conv_weights_ex(self.w.float(), c.c0, c.c1, c.D, c.H, c.W, c.kind, c.terms, c.fmt, c.flags)

    def out_shape(self):
        c = self.case
        up = 2 if c.kind == 2 else 1
        return (c.NT, up * c.D, up * c.H, up * c.W, c.cout * (2 if c.out == "split" else 1))

    def sentinel_outputs(self):
        """Output tensors filled with NaN (0xFFFF; 0xFF in the e4m3 plane): a voxel no launch writes stays NaN."""
        out = torch.full(self.out_shape(), SENTINEL, dtype=torch.int16, device="cuda").view(DT[self.case.fmt])
        out8 = torch.full(self.out_shape(), 0xFF, dtype=torch.uint8, device="cuda") if self.case.out == "lo8" else None
        return out, out8

    def run(self, region=None, out=None, out_lo8=None):
        """One launch (region=None: the whole layer; api "box": its region through oai_conv3d_igemm_box); returns
        (16-bit output, e4m3 plane or None)."""
        c = self.case
        wp = self.wpack()
        if c.api == "convt2":
            return ops.convt2_igemm(self.src[0], wp, self.b, c.cout, c.relu, c.fmt, region=region, out=out), None
        if c.api == "obase":
            return self._run_obase(wp), None
        if c.api == "box" and region is not None:
            got = ops.conv3d_igemm_box(self.src[0], self.src[1], wp, self.b, c.cout, c.c0, c.c1, region, c.relu, c.fmt,
                                       c.terms, in_split=self.in_split, out_split=c.out == "split", flags=c.flags,
                                       in_lo8=self.lo8, out=out, out_lo8=out_lo8)
            return got, out_lo8
        got = ops.conv3d_igemm_ex(self.src[0], self.src[1], wp, self.b, c.cout, c.c0, c.c1, c.kind, c.relu, c.fmt,
                                  c.terms, in_split=self.in_split, out_split=c.out == "split", region=region,
                                  flags=c.flags, in_lo8=self.lo8,
                                  out_lo8=(out_lo8 if out_lo8 is not None else c.out == "lo8"), out=out)
        return got if c.out == "lo8" else (got, None)

    def _run_obase(self, wp):
        """oai_conv3d_igemm into channels [64, 64 + cout) of a wider tensor: the other channels must stay untouched."""
        c = self.case
        NT, D, H, W = c.NT, c.D, c.H, c.W
        CW, base = 192, 64
        big = torch.full((NT, D, H, W, CW), SENTINEL, dtype=torch.int16, device="cuda").view(DT[c.fmt])
        ops.conv3d_igemm(self.src[0], self.src[1], wp, self.b, c.cout, c.kind == 1, c.relu, c.fmt, out=big,
                         out_view=(base, D * H * W * CW, H * W * CW, W * CW, CW), flags=c.flags)
        torch.cuda.synchronize()
        bits = big.view(torch.int16)
        assert (bits[..., :base] == SENTINEL).all() and (bits[..., base + c.cout:] == SENTINEL).all(), \
            "channels outside the output slice were written"
        return big[..., base:base + c.cout].contiguous()

    def check(self, got, lo8):
        """Bitwise comparison with the exact answer; returns the largest difference (0 when it passes)."""
        c = self.case
        dt = DT[c.fmt]
        y = self.y
        hi_ref = y.to(dt)
        hi = got[..., :c.cout]
        diff = (hi.double() - hi_ref.double()).abs().nan_to_num(math.inf).max().item()
        if c.out == "split":
            lo_ref = (y - hi_ref.double()).to(dt)   # y - hi is exact in fp32, so the kernel rounds the same value
            lo = got[..., c.cout:]
            diff = max(diff, (lo.double() - lo_ref.double()).abs().nan_to_num(math.inf).max().item())
        if c.out == "lo8":
            ref8 = ops.split_lo8(y.float(), c.fmt)[1]
            if not torch.equal(lo8, ref8):
                d8 = (ops.lo8_value(lo8, c.fmt) - ops.lo8_value(ref8, c.fmt)).abs().nan_to_num(math.inf).max().item()
                diff = max(diff, d8 if d8 > 0 else math.inf)   # bits differ: never report 0
        assert torch.isfinite(y).all() and y.abs().max().item() < (65504 if c.fmt == 0 else 3e38)
        return diff


def _seed(case):
    return sum(ord(ch) * (i + 1) for i, ch in enumerate(case.name)) % 100003


@pytest.mark.parametrize("case", cc.CASES, ids=lambda c: c.id)
def test_layer_is_exact(case):
    _cuda()
    L = Layer(case, _seed(case))
    got, lo8 = L.run(None, *L.sentinel_outputs())
    torch.cuda.synchronize()
    diff = L.check(got, lo8)
    print(f"{case.name}: {case.why} -- max |diff| {diff:g} (|y| <= {L.y.abs().max().item():g}, "
          f"sum |x||w| <= {L.bound:g})")
    assert diff == 0, f"{case.name} ({case.why}): max difference {diff}"


def _check_region(case):
    """The region property: the full launch is exact; a region launch into NaN-filled outputs equals it inside the
    region, leaves every other voxel NaN or equal to it, never writes a slice outside the d range, and (region launches
    of oai_conv3d_igemm_region's kinds) writes exactly the rows of the region's whole M tiles."""
    L = Layer(case, _seed(case))
    full, full8 = L.run(None, *L.sentinel_outputs())
    torch.cuda.synchronize()
    diff = L.check(full, full8)
    assert diff == 0, f"{case.name}: full launch max difference {diff}"
    part, part8 = L.run(case.region, *L.sentinel_outputs())
    torch.cuda.synchronize()
    up = 2 if case.kind == 2 else 1
    d_lo, d_cnt, h_lo, h_cnt = (up * v for v in case.region[:4])
    w_lo, w_cnt = case.region[4:] if len(case.region) == 6 else (0, up * case.W)
    pairs = [(part.view(torch.int16), full.view(torch.int16), SENTINEL)]
    if part8 is not None:
        pairs.append((part8, full8, 0xFF))
    written_rows = set()
    for bits, ref, fill in pairs:
        box = (slice(None), slice(d_lo, d_lo + d_cnt), slice(h_lo, h_lo + h_cnt), slice(w_lo, w_lo + w_cnt))
        assert torch.equal(bits[box], ref[box]), f"{case.name}: region voxels differ from the full-layer launch"
        untouched = (bits == fill).all(-1)
        assert (untouched | (bits == ref).all(-1)).all(), \
            f"{case.name}: a voxel outside the region holds neither the sentinel nor its full-layer value"
        written = ~untouched
        ds = written.any(-1).any(-1).any(0).nonzero().flatten().tolist()
        assert all(d_lo <= d < d_lo + d_cnt for d in ds), f"{case.name}: slices {ds} outside the d range written"
        rows = written.any(-1).any(1).any(0).nonzero().flatten().tolist()
        if case.api != "box":
            r_lo, r_hi = cc.region_rows(case)
            assert rows == list(range(r_lo, r_hi)), \
                f"{case.name}: rows {rows} written, the region's whole M tiles are rows [{r_lo}, {r_hi})"
        written_rows |= set(rows)
    extra = sorted(r for r in written_rows if not h_lo <= r < h_lo + h_cnt)
    print(f"{case.name}: {case.why} -- region {case.region}: {len(written_rows)} rows written, outside the region "
          f"{extra}; max |diff| inside 0")
    if case.name == "reg_dc4":   # the rows the issue and the header's whole-M-tile rule name
        assert extra == [6, 57], extra
    if case.name == "reg_kh_shared":   # the second tile (9 + 4 = 13) is clamped to start at H - TH = 12
        assert sorted(written_rows) == list(range(9, 16)), sorted(written_rows)


@pytest.mark.parametrize("case", cc.REGION_CASES, ids=lambda c: c.id)
def test_region_launch_writes_full_layer_values_only(case):
    _cuda()
    _check_region(case)


@pytest.mark.parametrize("case", cc.BOX_CASES, ids=lambda c: c.id)
def test_w_box_launch_writes_full_layer_values_only(case):
    """oai_conv3d_igemm_box: the kh-shared main launch plus the overlapping 8-wide strip, as dc2 / dc1 run."""
    _cuda()
    _check_region(case)


def _production_cases():
    regions = ops.seg_needed_regions(cc.PROD_TILE, cc.PROD_OVERLAP)
    mixed = cc.production_cases(ops.seg_layer_terms(1), 0, regions)
    bf16 = cc.production_cases([1] * 17, 1, regions)
    return mixed + bf16


@pytest.mark.parametrize("case", _production_cases(), ids=lambda c: c.id)
def test_production_launch_replay(case):
    """Every tcgen05 conv launch oai_seg_forward makes at the production tile (32 x 128 x 128, overlap (8, 16, 16), two
    tiles per launch), one at a time, for the mixed plan and for all-terms-1 bf16: the layer's spec, storage, region
    (dc2 / dc1: their (h, w) box as kh-shared main launch + strip) with exact operands.  dc1's fused head is
    test_conv_head_box_gpu.py's."""
    _cuda()
    if case.region is None:
        L = Layer(case, _seed(case))
        got, lo8 = L.run(None, *L.sentinel_outputs())
        torch.cuda.synchronize()
        diff = L.check(got, lo8)
        print(f"{case.name}: whole layer -- max |diff| {diff:g}")
        assert diff == 0, f"{case.name}: max difference {diff}"
    else:
        _check_region(case)
