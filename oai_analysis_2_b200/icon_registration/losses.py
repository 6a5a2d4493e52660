"""icon_registration.losses on B200: the ICONLoss tuple GradientICON.forward returns, the similarity measures that
configure it and the fold count.

The terms themselves are computed by the library (csrc/reg_loss.cu behind oai_reg_icon_loss, see
GradICONModel.icon_loss); LNCC and ssd_only_interpolated here select and parameterise that computation."""
from collections import namedtuple

from .. import ops

ICONLoss = namedtuple("ICONLoss", "all_loss inverse_consistency_loss similarity_loss transform_magnitude flips")


class LNCC:
    """Local normalised cross-correlation with a Gaussian window of 4*sigma (+1, odd) taps, sigma in voxels:
    mean(1 - (G(IJ) - G(I)G(J)) / sqrt((relu(G(I^2) - G(I)^2) + 1e-5) (relu(G(J^2) - G(J)^2) + 1e-5)))."""
    isInterpolated = False

    def __init__(self, sigma):
        if not sigma > 0:
            raise ValueError(f"LNCC sigma must be positive, got {sigma}")
        self.sigma = sigma

    def __repr__(self):
        return f"LNCC(sigma={self.sigma})"


class SSDOnlyInterpolated:
    """Mean squared difference over the voxels whose sample stayed inside the moving image: the images carry an
    in-bounds tag (1 on [1:-1]^3) warped with them, and the loss is sum(tag (A - B)^2) / sum(tag)."""
    isInterpolated = True

    def __repr__(self):
        return "ssd_only_interpolated"


ssd_only_interpolated = SSDOnlyInterpolated()


def similarity_config(similarity):
    """(oai_icon_loss_cfg.similarity, sigma) of a similarity object."""
    if isinstance(similarity, LNCC):
        return ops.SIM_LNCC, float(similarity.sigma)
    if isinstance(similarity, SSDOnlyInterpolated):
        return ops.SIM_SSD_ONLY_INTERPOLATED, 0.0
    raise ValueError(f"unsupported similarity {similarity!r}: use LNCC(sigma) or ssd_only_interpolated")


def flips(phi, in_percentage=False):
    """Number of cells where the map folds (dV < 0, forward differences at [1:, 1:, 1:]) per batch entry of phi
    [N, 3, D, H, W] (float32 CUDA), or their percentage of all cells.  Returns a 0-d float64 CUDA tensor."""
    if not phi.is_cuda:
        raise RuntimeError("flips runs on CUDA (sm_100a) only")
    if phi.dim() != 5 or phi.shape[1] != 3:
        raise ValueError(f"flips expects a map [N, 3, D, H, W], got {list(phi.shape)}")
    phi = phi.detach().float().contiguous()
    total = sum(ops.jacobian_flips(phi[n]).double() for n in range(phi.shape[0]))
    if in_percentage:
        cells = (phi.shape[2] - 1) * (phi.shape[3] - 1) * (phi.shape[4] - 1)
        return total / (phi.shape[0] * cells) * 100.0
    return total / phi.shape[0]


