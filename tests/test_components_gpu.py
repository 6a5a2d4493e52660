"""GPU tier: connected-component labelling (oai_connected_components, csrc/components.cu) against scipy.ndimage.label
itself, bit for bit, and the keep policy (oai_keep_components) against numpy's rule, down to the segmenter's
keep_largest_component option.  Labels and sizes are integers, so every comparison is exact."""
import numpy as np
import pytest
import torch
from scipy import ndimage as ndi

from helpers import load_golden, write_seg_config

pytestmark = pytest.mark.gpu

RANK = {6: 1, 18: 2, 26: 3}
FULL = (160, 384, 384)


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _scipy(mask, conn):
    return ndi.label(mask, ndi.generate_binary_structure(3, RANK[conn]))


def _check(mask, conn):
    from oai_analysis_2_b200 import ops
    labels, sizes, count = ops.connected_components(torch.from_numpy(np.ascontiguousarray(mask)).cuda(), conn)
    ref, n = _scipy(mask, conn)
    got = labels.cpu().numpy()
    assert got.dtype == np.int32 and int(count) == n
    assert np.array_equal(got, ref), f"{int((got != ref).sum())} voxels differ at connectivity {conn}"
    s = sizes.cpu().numpy()
    assert np.array_equal(s[:n], np.bincount(ref.ravel(), minlength=n + 1)[1:]) and not s[n:].any()
    return labels, sizes, count


@pytest.mark.parametrize("conn", [6, 18, 26])
@pytest.mark.parametrize("shape", [(1, 1, 1), (1, 1, 37), (7, 33, 65), (5, 512, 3), (2, 3, 2000)])
def test_labels_equal_scipy_at_odd_shapes_and_densities(shape, conn):
    _cuda()
    rng = np.random.default_rng(sum(shape) + conn)
    for density in (0.0, 1.0, 0.05, 0.3, 0.7):
        _check(rng.random(shape) < density, conn)


def _serpentine(shape):
    """One component: full rows on even (z, y), joined at alternating row ends and at x = 0 between even slices."""
    D, H, W = shape
    m = np.zeros(shape, bool)
    m[::2, ::2, :] = True
    for y in range(0, H - 2, 2):
        m[::2, y + 1, W - 1 if (y // 2) % 2 == 0 else 0] = True
    m[1::2, 0, 0] = True
    return m[: D - (D + 1) % 2]    # an even D would end on an unjoined empty slice


@pytest.mark.parametrize("conn", [6, 18, 26])
def test_labels_equal_scipy_on_adversarial_masks(conn):
    _cuda()
    snake = _serpentine((13, 41, 97))
    assert _scipy(snake, conn)[1] == 1
    _check(snake, conn)
    z, y, x = np.indices((9, 35, 67))
    checker = (z + y + x) % 2 == 0
    _, n = _scipy(checker, conn)
    assert n == (checker.sum() if conn == 6 else 1)
    _check(checker, conn)


@pytest.mark.parametrize("conn", [6, 26])
def test_labels_equal_scipy_at_full_size_on_a_random_mask(conn):
    _cuda()
    mask = np.random.default_rng(7).random(FULL) < 0.5
    _check(mask, conn)


def _full_size_segmenter(tmp_path):
    from oai_analysis_2_b200.segmentation.segmenter import Segmenter3DInPatchClassWise
    from oracle import seg_oracle
    sd = seg_oracle.make_unet_state_dict(13, 1, 2, True, True, True, 88.16291826695385,
                                         [-4.068152692193752, -7.490846258792958])
    cfg = write_seg_config(tmp_path, sd, [128, 128, 32], True, True, (16, 16, 8))
    return Segmenter3DInPatchClassWise(mode="pred", config=cfg)


def test_labels_equal_scipy_on_the_segmenter_masks_of_a_full_size_knee(tmp_path):
    _cuda()
    from oai_analysis_2_b200 import synthetic
    seg = _full_size_segmenter(tmp_path)
    out = seg.segment_device(torch.from_numpy(synthetic.synthetic_knee(synthetic.OAI_SHAPE, seed=5)).cuda(), True)
    masks = (out > 0.5).cpu().numpy()
    for c in range(2):
        assert masks[c].any()
        for conn in (6, 18, 26):
            _check(masks[c], conn)


def test_labels_are_reproducible_and_replay_in_a_cuda_graph():
    _cuda()
    from oai_analysis_2_b200 import ops
    shape = (37, 70, 90)
    rng = np.random.default_rng(11)
    m1, m2 = rng.random(shape) < 0.3, rng.random(shape) < 0.31
    m = torch.from_numpy(m1).cuda()
    first = ops.connected_components(m, 26)
    for _ in range(3):
        again = ops.connected_components(m, 26)
        assert all(torch.equal(a, b) for a, b in zip(first, again))
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            captured = ops.connected_components(m, 26)
    torch.cuda.current_stream().wait_stream(s)
    for M in (m2, m1):
        m.copy_(torch.from_numpy(M))
        g.replay()
        eager = ops.connected_components(m, 26)
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(captured, eager))
        ref, n = _scipy(M, 26)
        assert int(captured[2]) == n and np.array_equal(captured[0].cpu().numpy(), ref)


def _numpy_keep(mask, conn, min_voxels):
    ref, n = _scipy(mask, conn)
    sizes = np.bincount(ref.ravel(), minlength=n + 1)
    if min_voxels is None:
        return ref == np.argmax(sizes[1:]) + 1 if n else np.zeros_like(mask)
    return (ref > 0) & (sizes >= min_voxels)[ref]


@pytest.mark.parametrize("conn", [6, 18, 26])
def test_keep_components_follows_the_numpy_rule(conn):
    _cuda()
    from oai_analysis_2_b200 import ops
    shape = (11, 40, 53)
    rng = np.random.default_rng(conn)
    mask = rng.random(shape) < 0.25
    for mv in (None, 0, 1, 3, 10, 10 ** 6):
        got = ops.keep_components(torch.from_numpy(mask).cuda(), conn, mv)
        assert got.dtype == torch.bool
        assert np.array_equal(got.cpu().numpy(), _numpy_keep(mask, conn, mv)), mv
    # a size tie: the lowest label wins, as numpy's argmax
    tie = np.zeros(shape, bool)
    tie[1:3, 30:33, 40:44] = True     # 24 voxels, label 1
    tie[5:7, 2:5, 1:5] = True         # 24 voxels, label 2
    tie[8, 0, 0] = True
    got = ops.keep_components(torch.from_numpy(tie).cuda(), conn).cpu().numpy()
    expect = np.zeros(shape, bool)
    expect[1:3, 30:33, 40:44] = True
    assert np.array_equal(got, expect) and np.array_equal(got, _numpy_keep(tie, conn, None))
    # an empty mask stays empty
    empty = torch.zeros(shape, dtype=torch.uint8, device="cuda")
    assert not ops.keep_components(empty, conn).any() and not ops.keep_components(empty, conn, 0).any()


def test_keep_components_zeroes_float_maps_outside_the_kept_components():
    _cuda()
    from oai_analysis_2_b200 import ops
    shape = (9, 47, 61)
    prob = np.random.default_rng(3).random(shape).astype(np.float32) * 0.9
    for conn, mv in [(6, None), (26, None), (18, 4)]:
        x = torch.from_numpy(prob.copy()).cuda()
        out = ops.keep_components(x, conn, mv)
        assert out.data_ptr() == x.data_ptr()
        keep = _numpy_keep(prob > 0.5, conn, mv)
        got = out.cpu().numpy()
        assert np.array_equal(got[keep], prob[keep])          # untouched inside
        assert not got[~keep].any()                           # exact zeros outside
    zero = torch.zeros(shape, device="cuda")
    assert not ops.keep_components(zero).any()


def test_component_summary_matches_scipy():
    _cuda()
    from oai_analysis_2_b200 import itk_compat, metrics
    shape = (20, 64, 72)
    rng = np.random.default_rng(5)
    probs = rng.random((2, *shape)).astype(np.float32) * 0.8
    spacing = (0.3646, 0.3646, 0.7)
    vox = spacing[0] * spacing[1] * spacing[2]
    for conn in (6, 26):
        got = metrics.component_summary(torch.from_numpy(probs).cuda(), spacing, connectivity=conn)
        imgs = tuple(itk_compat.Image(p, spacing=spacing) for p in probs)
        assert metrics.component_summary(imgs, connectivity=conn) == got
        for q, p in zip(got, probs):
            ref, n = _scipy(p > 0.5, conn)
            sizes = np.bincount(ref.ravel())[1:]
            assert q.n_components == n
            assert q.largest_mm3 == pytest.approx(sizes.max() * vox, rel=1e-12)
            assert q.total_mm3 == pytest.approx(sizes.sum() * vox, rel=1e-12)
    with pytest.raises(ValueError, match="spacing_xyz"):
        metrics.component_summary(probs)


def _small_segmenter(tmp_path, keep):
    from oai_analysis_2_b200.segmentation.segmenter import Segmenter3DInPatchClassWise
    from oracle.seg_oracle import make_unet_state_dict, synthetic_knee
    z, m = load_golden("seg_small_pertap")
    sd = make_unet_state_dict(m["seed"], 1, 2, m["bias"], m["BN"], True, m["head_gain"], m["head_bias"])
    tmp_path.mkdir(parents=True, exist_ok=True)
    cfg = write_seg_config(tmp_path, sd, m["patch"], m["bias"], m["BN"], m["overlap"])
    if keep is not None:
        cfg["keep_largest_component"] = keep
    vol = synthetic_knee(tuple(m["shape"]), m["seed"])
    return Segmenter3DInPatchClassWise(mode="pred", config=cfg), vol


def test_segmenter_keep_largest_component(tmp_path):
    _cuda()
    plain, vol = _small_segmenter(tmp_path / "a", None)
    v = torch.from_numpy(vol).cuda()
    base = plain.segment_device(v, True).clone()
    for off in (0, False):
        seg, _ = _small_segmenter(tmp_path / f"b{off!r}", off)
        assert torch.equal(seg.segment_device(v, True), base)      # absent or falsy: bitwise unchanged
    probs = base.cpu().numpy()
    for conn in (6, 26):
        seg, _ = _small_segmenter(tmp_path / f"c{conn}", conn)
        got = seg.segment_device(v, True).cpu().numpy()
        for c in range(2):
            keep = _numpy_keep(probs[c] > 0.5, conn, None)
            assert np.array_equal(got[c], np.where(keep, probs[c], 0).astype(np.float32))
        # the host entry point gets it too
        fc, tc = seg.segment(vol, if_output_prob_map=True, if_output_itk=False)
        assert np.array_equal(fc, got[0].astype(np.float64)) and np.array_equal(tc, got[1].astype(np.float64))


def test_segmenter_keep_largest_component_replays_in_a_cuda_graph(tmp_path):
    _cuda()
    seg, vol = _small_segmenter(tmp_path, 26)
    rng = np.random.default_rng(1)
    vols = [vol, np.clip(vol + rng.normal(0, 0.05, vol.shape), 0, None).astype(np.float32)]
    v = torch.from_numpy(vols[0]).cuda()
    out = torch.empty((2, *vol.shape), device="cuda")
    seg.segment_device(v, True, out=out)        # warm-up outside the capture
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            seg.segment_device(v, True, out=out)
    torch.cuda.current_stream().wait_stream(s)
    for V in (vols[1], vols[0]):
        v.copy_(torch.from_numpy(V))
        g.replay()
        eager = seg.segment_device(v, True)
        torch.cuda.synchronize()
        assert torch.equal(out, eager)
