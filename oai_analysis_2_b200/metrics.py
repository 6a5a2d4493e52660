"""Segmentation quality: Dice, cartilage volume and surface distances (ASSD, HD95, HD) per class, on the GPU.

The definitions are medpy's ``dc`` / ``assd`` / ``hd95`` / ``hd`` (include/oai_b200.h, oai_surface_metrics): surface
voxels are mask voxels with a 6-neighbour outside the mask or off the volume, and distances are in mm between voxel
centres.  Dice is NaN when both masks are empty; the distances are NaN when either is empty.

Checking a segmentation against a manual labelling::

    fc, tc = segmenter.segment(image, if_output_prob_map=True, if_output_itk=True)
    fc_q, tc_q = segmentation_metrics((fc, tc), (manual_fc, manual_tc))

Checking a registration: warp knee A's segmentation onto knee B's grid, then compare it with B's::

    from oai_analysis_2_b200.dask_processing import deform_probmap
    warped = (deform_probmap(phi_AB, image_A, image_B, fc_A, "FC"),
              deform_probmap(phi_AB, image_A, image_B, tc_A, "TC"))
    fc_q, tc_q = segmentation_metrics(warped, (fc_B, tc_B))

How many pieces a mask falls into, and how much of its volume lies outside the main plate::

    fc_c, tc_c = component_summary((fc, tc))
    outside_mm3 = fc_c.total_mm3 - fc_c.largest_mm3
"""
import collections

import numpy as np
import torch

from . import itk_compat, ops

SegmentationMetrics = collections.namedtuple("SegmentationMetrics",
                                             ["dice", "assd", "hd95", "hd", "volume_pred_mm3", "volume_ref_mm3"])
ComponentSummary = collections.namedtuple("ComponentSummary", ["n_components", "largest_mm3", "total_mm3"])


def _is_image(x):
    return isinstance(x, itk_compat.Image) or hasattr(x, "GetLargestPossibleRegion")


def _classes(x):
    """-> list of per-class volumes [D,H,W] (images, arrays or tensors), and the spacing of images (None otherwise)."""
    if isinstance(x, (tuple, list)):
        items = list(x)
    elif _is_image(x):
        items = [x]
    else:
        items = [x] if x.ndim == 3 else [x[c] for c in range(x.shape[0])]
    spacing = None
    for it in items:
        if _is_image(it):
            sp = tuple(float(v) for v in itk_compat.image_metadata(it)[0])
            if spacing is not None and sp != spacing:
                raise ValueError(f"classes of one input have different spacings: {spacing} and {sp}")
            spacing = sp
    return items, spacing


def _mask(x, threshold):
    if _is_image(x):
        x = itk_compat.array_from_image(x)
    t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
    if t.dim() != 3:
        raise ValueError(f"expected a [D,H,W] volume per class, got shape {tuple(t.shape)}")
    if not t.is_cuda:
        t = t.cuda()
    return t.contiguous() if t.dtype == torch.bool else t > threshold


def _spacing(found, spacing_xyz):
    spacing = found
    if spacing is None:
        if spacing_xyz is None:
            raise ValueError("spacing_xyz is required for array or tensor inputs")
        spacing = spacing_xyz
    return tuple(float(v) for v in spacing)


def segmentation_metrics(pred, ref, spacing_xyz=None, threshold=0.5):
    """Per-class quality of `pred` against `ref`: a list of SegmentationMetrics(dice, assd, hd95, hd, volume_pred_mm3,
    volume_ref_mm3), distances in mm.

    pred / ref: the (FC, TC) tuple Segmenter3DInPatchClassWise.segment returns (itk or itk_compat images), or arrays /
    tensors [C,D,H,W] or [D,H,W], or lists of those per class.  Probabilities become masks by `> threshold` (the
    segmenter's own rule); bool inputs are taken as they are.  A label map is compared as ``ref == k``.  The spacing
    (x, y, z) comes from the images, which must share one grid; for arrays and tensors `spacing_xyz` is required.
    Synchronises once, to return Python floats."""
    p_items, p_sp = _classes(pred)
    r_items, r_sp = _classes(ref)
    if len(p_items) != len(r_items):
        raise ValueError(f"pred has {len(p_items)} classes and ref {len(r_items)}")
    if p_sp is not None and r_sp is not None and not np.allclose(p_sp, r_sp, rtol=1e-6, atol=0):
        raise ValueError(f"pred and ref grids differ in spacing: {p_sp} and {r_sp}")
    spacing = _spacing(p_sp or r_sp, spacing_xyz)
    voxel_mm3 = spacing[0] * spacing[1] * spacing[2]
    results = []
    for p, r in zip(p_items, r_items):
        a, b = _mask(p, threshold), _mask(r, threshold)
        if a.shape != b.shape:
            raise ValueError(f"pred and ref grids differ in size: {tuple(a.shape)} and {tuple(b.shape)}")
        results.append(ops.surface_metrics(a, b, spacing))
    # the one synchronisation; the counts are exact in float64 (below 2**53)
    host = torch.stack([torch.cat([t, c.to(torch.float64)]) for t, c in results]).cpu().numpy()
    return [SegmentationMetrics(float(h[0]), float(h[1]), float(h[2]), float(h[3]), float(h[8]) * voxel_mm3,
                                float(h[9]) * voxel_mm3) for h in host]


def component_summary(pred, spacing_xyz=None, threshold=0.5, connectivity=6):
    """Per-class connected components of `pred` (the inputs segmentation_metrics takes): a list of
    ComponentSummary(n_components, largest_mm3, total_mm3), components as scipy.ndimage.label counts them with
    connectivity 6, 18 or 26.  Synchronises once, to return Python numbers."""
    items, sp = _classes(pred)
    spacing = _spacing(sp, spacing_xyz)
    voxel_mm3 = spacing[0] * spacing[1] * spacing[2]
    rows = []
    for p in items:
        _, sizes, count = ops.connected_components(_mask(p, threshold), connectivity)
        rows.append(torch.stack([count, sizes.max().to(torch.int64), sizes.sum(dtype=torch.int64)]))
    host = torch.stack(rows).cpu().numpy()
    return [ComponentSummary(int(h[0]), float(h[1]) * voxel_mm3, float(h[2]) * voxel_mm3) for h in host]
