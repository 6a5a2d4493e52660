"""GPU tier: the exact distance transform (oai_distance_transform) and the segmentation-quality terms
(oai_surface_metrics, csrc/seg_quality.cu) against scipy.ndimage / numpy (tests/surface_metrics_oracle.py).

Tolerances.  The transform keeps squared distances in float32 between its passes and returns float32, so a distance is
within a few float32 roundings of scipy's float64 value: |d - d_scipy| <= 1e-6 d_scipy + 1e-6 mm.  Counts and Dice are
integer arithmetic and must match exactly; the means are fp64 sums of those distances and HD / HD95 are order
statistics of them, within 1e-6 relative."""
import numpy as np
import pytest
import torch

import surface_metrics_oracle as so
from helpers import dice, load_golden, write_seg_config

pytestmark = pytest.mark.gpu

OAI = (0.3646, 0.3646, 0.7)
ISO = (1.0, 1.0, 1.0)
FULL = (160, 384, 384)


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _sparse(shape, seed, density):
    return np.random.default_rng(seed).random(shape) < density


def _check_edt(got, ref):
    got = got.cpu().numpy().astype(np.float64)
    inf = np.isinf(ref)
    assert np.array_equal(np.isinf(got), inf)
    err = np.abs(got[~inf] - ref[~inf])
    assert np.all(err <= 1e-6 * ref[~inf] + 1e-6), float(err.max())


@pytest.mark.parametrize("spacing", [OAI, ISO])
@pytest.mark.parametrize("shape,density", [((1, 1, 37), 0.05), ((7, 33, 65), 0.002), ((5, 512, 3), 0.01),
                                           ((512, 2, 9), 0.003), ((3, 4, 512), 0.0), ((1, 1, 1), 1.0),
                                           (FULL, 2e-6)])
def test_distance_transform_matches_scipy(shape, density, spacing):
    _cuda()
    from oai_analysis_2_b200 import ops
    f = _sparse(shape, hash((shape, density)) % 1000, density)
    got = ops.distance_transform(torch.from_numpy(f).cuda(), spacing)
    _check_edt(got, so.edt(f, spacing))


def test_distance_transform_of_a_dense_feature_set_and_a_single_voxel():
    _cuda()
    from oai_analysis_2_b200 import ops
    f = _sparse((40, 70, 90), 3, 0.6)           # long runs of features: deep envelope stacks
    _check_edt(ops.distance_transform(torch.from_numpy(f).cuda(), OAI), so.edt(f, OAI))
    f = np.zeros((9, 300, 500), bool)
    f[8, 0, 499] = True
    _check_edt(ops.distance_transform(torch.from_numpy(f).cuda(), OAI), so.edt(f, OAI))


def _full_pairs():
    D, H, W = FULL
    fc = so.shell(FULL, (80, 150, 192), (110, 140, 150), 0.03, seed=1, cut=230)
    tc = so.shell(FULL, (80, 320, 192), (90, 120, 130), 0.04, seed=2, cut=None) & (np.arange(H)[None, :, None] > 215)
    from scipy import ndimage as ndi
    fc_shift = np.roll(fc, (1, 2, -1), axis=(0, 1, 2))
    tc_eroded = ndi.binary_erosion(tc, so.CROSS) | (np.roll(tc, 3, axis=2) & tc)
    return [(fc, fc_shift), (tc, tc_eroded)]


def _compare(terms, counts, ref_terms, ref_counts):
    t, c = terms.cpu().numpy(), counts.cpu().numpy()
    assert np.array_equal(c, ref_counts), (c, ref_counts)
    assert t[0] == ref_terms[0] or (np.isnan(t[0]) and np.isnan(ref_terms[0]))
    for i in range(1, 8):
        if np.isnan(ref_terms[i]):
            assert np.isnan(t[i]), i
        else:
            assert abs(t[i] - ref_terms[i]) <= 1e-6 * abs(ref_terms[i]) + 1e-12, (i, t[i], ref_terms[i])


def test_surface_metrics_match_the_oracle_at_full_size():
    _cuda()
    from oai_analysis_2_b200 import ops
    for A, B in _full_pairs():
        ref_terms, ref_counts, _ = so.surface_metrics(A, B, OAI)
        assert ref_counts[3] > 1000 and ref_terms[1] > 0
        terms, counts = ops.surface_metrics(torch.from_numpy(A).cuda(), torch.from_numpy(B).cuda(), OAI)
        _compare(terms, counts, ref_terms, ref_counts)


def test_surface_metrics_maps_match_scipy_and_terms_are_reproducible():
    _cuda()
    from oai_analysis_2_b200 import ops
    A = so.shell((48, 96, 120), (24, 40, 60), (30, 50, 55), 0.08, seed=4, cut=70)
    B = np.roll(A, (2, -1, 3), axis=(0, 1, 2))
    ref_terms, ref_counts, (to_b, to_a) = so.surface_metrics(A, B, OAI)
    a, b = torch.from_numpy(A).cuda(), torch.from_numpy(B).cuda()
    terms, counts, got_b, got_a = ops.surface_metrics(a, b, OAI, maps=True)
    _compare(terms, counts, ref_terms, ref_counts)
    _check_edt(got_b, to_b)
    _check_edt(got_a, to_a)
    again, _ = ops.surface_metrics(a, b, OAI)
    assert torch.equal(again, terms)     # bitwise, NaN-free here
    # uint8 masks with values other than 1 count as inside
    t8, c8 = ops.surface_metrics(a.to(torch.uint8) * 7, b.to(torch.uint8) * 3, OAI)
    assert torch.equal(t8, terms) and torch.equal(c8, counts)


def test_surface_metrics_replays_in_a_cuda_graph_on_overwritten_inputs():
    _cuda()
    from oai_analysis_2_b200 import ops
    shape = (40, 80, 96)
    A1 = so.shell(shape, (20, 30, 48), (25, 40, 45), 0.1, seed=5, cut=60)
    B1 = np.roll(A1, 1, axis=1)
    A2 = so.shell(shape, (20, 35, 50), (22, 38, 40), 0.12, seed=6, cut=65)
    B2 = np.roll(A2, (1, 2), axis=(0, 2))
    a, b = torch.from_numpy(A1).cuda(), torch.from_numpy(B1).cuda()
    ops.surface_metrics(a, b, OAI)          # warm-up outside the capture
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            terms, counts = ops.surface_metrics(a, b, OAI)
    torch.cuda.current_stream().wait_stream(s)
    for A, B in [(A1, B1), (A2, B2)]:
        a.copy_(torch.from_numpy(A))
        b.copy_(torch.from_numpy(B))
        g.replay()
        eager_terms, eager_counts = ops.surface_metrics(a, b, OAI)
        torch.cuda.synchronize()
        assert torch.equal(terms, eager_terms) and torch.equal(counts, eager_counts)
        ref_terms, ref_counts, _ = so.surface_metrics(A, B, OAI)
        _compare(terms, counts, ref_terms, ref_counts)


def test_empty_masks_give_nans_without_a_fault():
    _cuda()
    from oai_analysis_2_b200 import ops
    shape = (6, 20, 33)
    E = np.zeros(shape, bool)
    A = np.zeros(shape, bool)
    A[2:4, 5:9, 10:20] = True
    for X, Y in [(E, E), (A, E), (E, A)]:
        ref_terms, ref_counts, (to_b, to_a) = so.surface_metrics(X, Y, OAI)
        terms, counts, got_b, got_a = ops.surface_metrics(torch.from_numpy(X).cuda(), torch.from_numpy(Y).cuda(),
                                                          OAI, maps=True)
        _compare(terms, counts, ref_terms, ref_counts)
        _check_edt(got_b, to_b)
        _check_edt(got_a, to_a)
    # the whole volume inside: every face voxel is surface, no background anywhere
    F = np.ones(shape, bool)
    ref_terms, ref_counts, _ = so.surface_metrics(F, A, OAI)
    terms, counts = ops.surface_metrics(torch.from_numpy(F).cuda(), torch.from_numpy(A).cuda(), OAI)
    _compare(terms, counts, ref_terms, ref_counts)


def test_segmenter_output_against_the_golden_masks(tmp_path):
    _cuda()
    from oai_analysis_2_b200 import itk_compat, metrics
    from oai_analysis_2_b200.segmentation.segmenter import Segmenter3DInPatchClassWise
    from oracle.seg_oracle import make_unet_state_dict, synthetic_knee
    z, m = load_golden("seg_small_pertap")
    sd = make_unet_state_dict(m["seed"], 1, 2, m["bias"], m["BN"], True, m["head_gain"], m["head_bias"])
    seg = Segmenter3DInPatchClassWise(mode="pred", config=write_seg_config(tmp_path, sd, m["patch"], m["bias"],
                                                                           m["BN"], m["overlap"]))
    spacing = (0.3646, 0.3646, 0.7)
    img = itk_compat.Image(synthetic_knee(tuple(m["shape"]), m["seed"]), spacing=spacing, origin=(1, 2, 3))
    fc, tc = seg.segment(img, if_output_prob_map=True, if_output_itk=True)
    ref = (itk_compat.Image(z["fc_mask"], spacing=spacing), itk_compat.Image(z["tc_mask"], spacing=spacing))
    got = metrics.segmentation_metrics((fc, tc), ref)
    for q, pred, mask in zip(got, (fc, tc), (z["fc_mask"], z["tc_mask"])):
        p = itk_compat.array_from_image(pred)
        assert np.asarray(mask).any() and q.dice == dice(p, mask)
        ref_terms, ref_counts, _ = so.surface_metrics(p > 0.5, np.asarray(mask) > 0.5, spacing)
        assert q.assd == pytest.approx(ref_terms[1], rel=1e-6, abs=1e-12)
        assert q.hd95 == pytest.approx(ref_terms[2], rel=1e-6, abs=1e-12)
        assert q.hd == pytest.approx(ref_terms[3], rel=1e-6, abs=1e-12)
        assert q.volume_pred_mm3 == pytest.approx(ref_counts[0] * spacing[0] * spacing[1] * spacing[2], rel=1e-12)
    with pytest.raises(ValueError, match="size"):
        metrics.segmentation_metrics(fc, itk_compat.Image(np.zeros((3, 4, 5)), spacing=spacing))
