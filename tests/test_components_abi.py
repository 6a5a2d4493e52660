"""CPU tier: argument checks of the connected-component entry points (oai_connected_components, oai_keep_components,
csrc/components.cu), which refuse bad input with a message before any device work, and the bound oai_components_max
against scipy's count on the worst cases."""
import ctypes

import numpy as np
import pytest
from scipy import ndimage as ndi


def _dims(dims):
    return np.asarray(dims, np.int32)


def _call(L, P, mask, dims, conn, labels, sizes, count, ws, nbytes):
    return L.oai_connected_components(P(mask), P(dims), conn, P(labels), P(sizes), P(count), ws,
                                      ctypes.c_size_t(nbytes), None)


@pytest.mark.parametrize("dims,conn,message", [
    ((4, 5, 6), 8, b"connectivity must be 6, 18 or 26"),
    ((4, 5, 6), 0, b"connectivity must be 6, 18 or 26"),
    ((4, 0, 6), 6, b"at least 1 voxel"),
    ((-1, 5, 6), 26, b"at least 1 voxel"),
    ((2048, 1024, 1024), 6, b"below 2^31"),
    ((1, 46341, 46341), 18, b"below 2^31"),
])
def test_components_reject_bad_grids_and_connectivities(dims, conn, message):
    from oai_analysis_2_b200 import _lib
    L, P = _lib.lib, _lib.ptr
    buf = np.zeros(64, np.uint8)
    lab = np.zeros(64, np.int32)
    cnt = np.zeros(1, np.int64)
    ws = np.zeros(4096, np.uint8)
    d = _dims(dims)
    assert _call(L, P, buf, d, conn, lab, lab, cnt, P(ws), ws.size) != 0
    assert message in L.oai_last_error()
    if conn in (6, 18, 26):
        assert L.oai_keep_components(P(lab), P(lab), P(cnt), P(d), -1, P(buf), None, None) != 0
        assert message in L.oai_last_error()
        assert L.oai_components_workspace_bytes(P(d)) == 0
    assert L.oai_components_max(P(d), conn) == 0


def test_components_reject_missing_arguments_and_short_workspaces():
    from oai_analysis_2_b200 import _lib
    L, P = _lib.lib, _lib.ptr
    dims = (5, 9, 70)
    d = _dims(dims)
    n = int(np.prod(dims))
    need = L.oai_components_workspace_bytes(P(d))
    assert need >= 4 * n and L.oai_components_workspace_bytes(None) == 0
    mask = np.zeros(n, np.uint8)
    lab = np.zeros(n, np.int32)
    sizes = np.zeros(L.oai_components_max(P(d), 6), np.int32)
    cnt = np.zeros(1, np.int64)
    ws = np.zeros(need + 512, np.uint8)
    wp = ctypes.c_void_p((ws.ctypes.data + 255) & ~255)     # 256-byte aligned view of the host buffer
    for args, message in [
        ((None, d, 6, lab, sizes, cnt, wp, need), b"null pointer"),
        ((mask, None, 6, lab, sizes, cnt, wp, need), b"null pointer"),
        ((mask, d, 6, None, sizes, cnt, wp, need), b"null pointer"),
        ((mask, d, 6, lab, None, cnt, wp, need), b"null pointer"),
        ((mask, d, 6, lab, sizes, None, wp, need), b"null pointer"),
        ((mask, d, 6, lab, sizes, cnt, None, need), b"null pointer"),
        ((mask, d, 6, lab, sizes, cnt, wp, need - 1), b"workspace"),
        ((mask, d, 6, lab, sizes, cnt, ctypes.c_void_p(wp.value + 4), need), b"workspace"),
    ]:
        assert _call(L, P, *args) != 0 and message in L.oai_last_error(), message
    for args, message in [
        ((None, P(sizes), P(cnt), P(d), -1, P(mask), None, None), b"null pointer"),
        ((P(lab), None, P(cnt), P(d), -1, P(mask), None, None), b"null pointer"),
        ((P(lab), P(sizes), None, P(d), -1, P(mask), None, None), b"null pointer"),
        ((P(lab), P(sizes), P(cnt), None, -1, P(mask), None, None), b"null pointer"),
        ((P(lab), P(sizes), P(cnt), P(d), 5, None, None, None), b"neither a keep mask nor values"),
    ]:
        assert L.oai_keep_components(*args) != 0 and message in L.oai_last_error(), message


@pytest.mark.parametrize("shape", [(1, 1, 1), (1, 1, 37), (4, 4, 4), (5, 6, 7), (7, 33, 65), (3, 2, 9)])
def test_components_max_bounds_the_worst_cases(shape):
    from oai_analysis_2_b200 import _lib
    d = _dims(shape)
    z, y, x = np.indices(shape)
    checker = (z + y + x) % 2 == 0
    lattice = (z % 2 == 0) & (y % 2 == 0) & (x % 2 == 0)
    for conn, rank, worst in [(6, 1, checker), (18, 2, lattice), (26, 3, lattice)]:
        n = ndi.label(worst, ndi.generate_binary_structure(3, rank))[1]
        bound = _lib.lib.oai_components_max(_lib.ptr(d), conn)
        assert n <= bound
        if conn == 6:
            assert bound == n == (int(np.prod(shape)) + 1) // 2      # tight
        if conn == 26:
            assert bound == n                                         # tight


def test_keep_components_rejects_a_negative_min_voxels():
    from oai_analysis_2_b200 import ops
    with pytest.raises(ValueError, match="min_voxels"):
        ops.keep_components(np.zeros((2, 2, 2), bool), min_voxels=-3)


@pytest.mark.parametrize("value", [7, True, 2.5, "26"])
def test_segmenter_rejects_a_keep_largest_component_that_is_not_a_connectivity(value):
    from oai_analysis_2_b200.segmentation.segmenter import Segmenter3DInPatchClassWise
    seg = Segmenter3DInPatchClassWise(mode="pred", config={"keep_largest_component": value})
    with pytest.raises(ValueError, match="keep_largest_component"):
        seg.pred_setup()
