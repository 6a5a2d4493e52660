"""CPU tier: the scipy / numpy oracle of the segmentation-quality terms (tests/surface_metrics_oracle.py) on cases with
known answers, and the argument checks of oai_distance_transform / oai_surface_metrics (they refuse bad input with a
message before any device work, so host buffers are enough here)."""
import ctypes
import math

import numpy as np
import pytest

import surface_metrics_oracle as so

SP = (0.3646, 0.3646, 0.7)


def test_identical_masks_give_dice_one_and_zero_distances():
    A = so.shell((20, 40, 40), (10, 20, 20), (8, 15, 15), 0.2)
    terms, counts, _ = so.surface_metrics(A, A, SP)
    assert terms[0] == 1.0 and np.all(terms[1:] == 0.0)
    assert counts[0] == counts[1] == counts[2] == A.sum() and counts[3] == counts[4] > 0


@pytest.mark.parametrize("p,q", [((2, 3, 4), (2, 3, 4)), ((1, 1, 1), (5, 7, 2)), ((0, 0, 0), (9, 10, 11))])
def test_single_voxels_are_apart_by_the_scaled_offset(p, q):
    A, B = np.zeros((10, 11, 12), bool), np.zeros((10, 11, 12), bool)
    A[p], B[q] = True, True
    d = math.sqrt(sum(((a - b) * s) ** 2 for a, b, s in zip(p, q, (SP[2], SP[1], SP[0]))))
    terms, counts, _ = so.surface_metrics(A, B, SP)
    assert terms[1] == pytest.approx(d) and terms[2] == pytest.approx(d) and terms[3] == pytest.approx(d)
    assert list(counts) == [1, 1, int(p == q), 1, 1]
    assert terms[0] == (1.0 if p == q else 0.0)


def test_solid_cube_has_26_surface_voxels_and_a_face_counts_as_surface():
    A = np.zeros((7, 7, 7), bool)
    A[2:5, 2:5, 2:5] = True
    assert so.surface(A).sum() == 26
    slab = np.zeros((4, 5, 6), bool)
    slab[0:3] = True                       # touches the z = 0 face and the four side faces
    s = so.surface(slab)
    assert s[0].all() and s[:3, 0].all() and s[:3, :, -1].all() and not s[3].any()
    assert not s[1, 1:-1, 1:-1].any()      # interior of the middle plane
    assert s[2].all()                       # the plane next to the background at z = 3


def test_empty_masks_give_the_specified_nans():
    E, A = np.zeros((5, 6, 7), bool), np.zeros((5, 6, 7), bool)
    A[2, 3, 4] = True
    t, c, (to_b, to_a) = so.surface_metrics(E, E, SP)
    assert np.all(np.isnan(t)) and list(c) == [0, 0, 0, 0, 0] and np.all(np.isinf(to_b))
    t, c, (to_b, to_a) = so.surface_metrics(A, E, SP)
    assert t[0] == 0.0 and np.all(np.isnan(t[1:])) and list(c) == [1, 0, 0, 1, 0]
    assert np.all(np.isinf(to_b)) and to_a[2, 3, 4] == 0.0
    assert so.edt(np.zeros((3, 3, 3), bool), SP).min() == np.inf


def test_edt_uses_the_spacing_per_axis():
    f = np.zeros((5, 6, 7), bool)
    f[0, 0, 0] = True
    d = so.edt(f, (0.5, 2.0, 3.0))
    assert d[0, 0, 6] == pytest.approx(3.0) and d[0, 5, 0] == pytest.approx(10.0) and d[4, 0, 0] == pytest.approx(12.0)


def _arrays(dims, spacing):
    from oai_analysis_2_b200 import _lib
    return _lib.ptr(np.asarray(dims, np.int32)), _lib.ptr(np.asarray(spacing, np.float64))


@pytest.mark.parametrize("dims,spacing,message", [
    ((0, 4, 4), SP, b"every axis"),
    ((4, 513, 4), SP, b"every axis"),
    ((4, 4, -3), SP, b"every axis"),
    ((4, 4, 4), (0.5, 0.0, 0.7), b"spacing"),
    ((4, 4, 4), (0.5, -1.0, 0.7), b"spacing"),
    ((4, 4, 4), (0.5, float("nan"), 0.7), b"spacing"),
    ((4, 4, 4), (float("inf"), 0.5, 0.7), b"spacing"),
])
def test_seg_quality_entry_points_reject_bad_grids_with_messages(dims, spacing, message):
    from oai_analysis_2_b200 import _lib
    L = _lib.lib
    buf, ws = np.zeros(64, np.uint8), np.zeros(1 << 12, np.uint8)
    out, terms, counts = np.zeros(64, np.float32), np.zeros(8), np.zeros(5, np.int64)
    d, s = _arrays(dims, spacing)
    rc = L.oai_distance_transform(_lib.ptr(buf), d, s, _lib.ptr(out), _lib.ptr(ws), ctypes.c_size_t(ws.size), None)
    assert rc != 0 and message in L.oai_last_error()
    rc = L.oai_surface_metrics(_lib.ptr(buf), _lib.ptr(buf), d, s, _lib.ptr(terms), _lib.ptr(counts), None, None,
                               _lib.ptr(ws), ctypes.c_size_t(ws.size), None)
    assert rc != 0 and message in L.oai_last_error()


def test_seg_quality_entry_points_reject_missing_arguments_and_short_workspaces():
    from oai_analysis_2_b200 import _lib
    L = _lib.lib
    n = 4 * 5 * 6
    a, out, terms, counts = np.zeros(n, np.uint8), np.zeros(n, np.float32), np.zeros(8), np.zeros(5, np.int64)
    d, s = _arrays((4, 5, 6), SP)
    need = L.oai_seg_quality_workspace_bytes(d)
    assert need >= 2 * 2 * n * 4
    assert L.oai_seg_quality_workspace_bytes(_arrays((4, 600, 6), SP)[0]) == 0
    assert L.oai_seg_quality_workspace_bytes(None) == 0
    ws = np.zeros(need + 256, np.uint8)
    wp = ctypes.c_void_p((ws.ctypes.data + 255) & ~255)     # 256-byte aligned view of the host buffer
    P = _lib.ptr
    cases = [
        (L.oai_distance_transform, (None, d, s, P(out), wp, ctypes.c_size_t(need), None), b"null pointer"),
        (L.oai_distance_transform, (P(a), None, s, P(out), wp, ctypes.c_size_t(need), None), b"null pointer"),
        (L.oai_distance_transform, (P(a), d, None, P(out), wp, ctypes.c_size_t(need), None), b"null pointer"),
        (L.oai_distance_transform, (P(a), d, s, None, wp, ctypes.c_size_t(need), None), b"null pointer"),
        (L.oai_distance_transform, (P(a), d, s, P(out), None, ctypes.c_size_t(need), None), b"null pointer"),
        (L.oai_distance_transform, (P(a), d, s, P(out), wp, ctypes.c_size_t(need - 1), None), b"workspace"),
        (L.oai_surface_metrics, (P(a), None, d, s, P(terms), P(counts), None, None, wp, ctypes.c_size_t(need), None),
         b"null pointer"),
        (L.oai_surface_metrics, (P(a), P(a), d, s, None, P(counts), None, None, wp, ctypes.c_size_t(need), None),
         b"null pointer"),
        (L.oai_surface_metrics, (P(a), P(a), d, s, P(terms), None, None, None, wp, ctypes.c_size_t(need), None),
         b"null pointer"),
        (L.oai_surface_metrics, (P(a), P(a), d, s, P(terms), P(counts), None, None, wp, ctypes.c_size_t(need - 1),
                                 None), b"workspace"),
    ]
    for fn, args, message in cases:
        assert fn(*args) != 0 and message in L.oai_last_error(), message


def test_metrics_module_validates_inputs_before_any_device_work():
    from oai_analysis_2_b200 import itk_compat, metrics
    assert metrics.SegmentationMetrics._fields == ("dice", "assd", "hd95", "hd", "volume_pred_mm3", "volume_ref_mm3")
    a = np.zeros((4, 5, 6), np.float32)
    with pytest.raises(ValueError, match="spacing_xyz is required"):
        metrics.segmentation_metrics(a, a)
    with pytest.raises(ValueError, match="spacing"):
        metrics.segmentation_metrics(itk_compat.Image(a, spacing=(0.36, 0.36, 0.7)),
                                     itk_compat.Image(a, spacing=(0.36, 0.36, 0.8)))
    with pytest.raises(ValueError, match="classes"):
        metrics.segmentation_metrics(np.zeros((2, 4, 5, 6)), a, spacing_xyz=SP)
