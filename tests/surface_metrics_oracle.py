"""Oracle of the segmentation-quality terms (oai_surface_metrics): medpy's dc / assd / hd / hd95 restated with
scipy.ndimage and numpy in float64.  The ground truth is scipy's own distance_transform_edt and numpy's own percentile.

A, B: bool [D, H, W] (z, y, x); spacing_xyz = (sx, sy, sz) in mm, so scipy's sampling is (sz, sy, sx)."""
import numpy as np
from scipy import ndimage as ndi

CROSS = ndi.generate_binary_structure(3, 1)


def surface(m):
    """M & ~binary_erosion(M, 6-connected cross, border_value=0): mask voxels on a volume face are surface."""
    m = np.asarray(m, dtype=bool)
    return m & ~ndi.binary_erosion(m, CROSS, border_value=0)


def edt(feature, spacing_xyz):
    """distance_transform_edt(~feature, sampling=(sz, sy, sx)); +inf everywhere for an empty feature set (scipy returns
    garbage for an input with no background)."""
    feature = np.asarray(feature, dtype=bool)
    if not feature.any():
        return np.full(feature.shape, np.inf)
    sx, sy, sz = spacing_xyz
    return ndi.distance_transform_edt(~feature, sampling=(sz, sy, sx))


def surface_metrics(A, B, spacing_xyz):
    """-> (terms float64[8] = dice, assd, hd95, hd, mean d_AB, mean d_BA, max d_AB, max d_BA;
    counts int64[5] = |A|, |B|, |A&B|, |dA|, |dB|;  (EDT to dB, EDT to dA))."""
    A, B = np.asarray(A, dtype=bool), np.asarray(B, dtype=bool)
    nA, nB, nAB = int(A.sum()), int(B.sum()), int((A & B).sum())
    sA, sB = surface(A), surface(B)
    to_B, to_A = edt(sB, spacing_xyz), edt(sA, spacing_xyz)
    counts = np.array([nA, nB, nAB, int(sA.sum()), int(sB.sum())], dtype=np.int64)
    dice = 2 * nAB / (nA + nB) if nA + nB else np.nan
    if nA == 0 or nB == 0:
        return np.array([dice] + [np.nan] * 7), counts, (to_B, to_A)
    d_ab, d_ba = to_B[sA], to_A[sB]
    assd = (d_ab.mean() + d_ba.mean()) / 2
    hd95 = np.percentile(np.hstack((d_ab, d_ba)), 95)
    hd = max(d_ab.max(), d_ba.max())
    terms = np.array([dice, assd, hd95, hd, d_ab.mean(), d_ba.mean(), d_ab.max(), d_ba.max()], dtype=np.float64)
    return terms, counts, (to_B, to_A)


def shell(shape, centre, radii, thickness, seed=0, cut=None):
    """A thin curved cartilage-like shell: voxels whose normalised ellipsoid radius lies in [1, 1 + thickness), with a
    gently perturbed surface, optionally cut by a plane y < cut."""
    D, H, W = shape
    z, y, x = np.ogrid[:D, :H, :W]
    r = np.sqrt(((z - centre[0]) / radii[0]) ** 2 + ((y - centre[1]) / radii[1]) ** 2 +
                ((x - centre[2]) / radii[2]) ** 2)
    rng = np.random.default_rng(seed)
    a, f = rng.uniform(0.005, 0.015, 2), rng.uniform(0.02, 0.06, 2)
    r = r + a[0] * np.sin(f[0] * x) * np.cos(f[1] * z) + a[1] * np.cos(f[0] * y)
    m = (r >= 1.0) & (r < 1.0 + thickness)
    if cut is not None:
        m &= y < cut
    return m
