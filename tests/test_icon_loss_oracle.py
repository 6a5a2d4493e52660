"""CPU tier: the torch oracle of GradientICON's loss terms (tests/icon_loss_oracle.py) on cases with known answers, and
the argument checks of the registration-quality entry points (they refuse bad input before any device call)."""
import ctypes

import numpy as np
import pytest
import torch

import icon_loss_oracle as lo
from oracle import reg_oracle


def test_flips_counts_a_mirrored_slab_exactly_and_nothing_on_the_identity():
    shape = (12, 9, 7)
    assert lo.flips(reg_oracle.identity_map(shape, torch.float64)).item() == 0
    for z0, z1 in [(3, 8), (1, 12), (5, 7)]:
        phi = lo.folded_map(shape, z0, z1)
        assert lo.flips(phi).item() == (z1 - z0 - 1) * (shape[1] - 1) * (shape[2] - 1)
        assert lo.jacobian_det(phi).shape == (1, 1, 11, 8, 6)
    pct = lo.flips(lo.folded_map(shape, 3, 8), in_percentage=True).item()
    assert pct == pytest.approx(100.0 * 4 * 8 * 6 / (11 * 8 * 6))


def _affine_pair(shape, scale, dtype=torch.float64):
    """Displacement fields of the contraction x -> c + s (x - c) toward the centre c = 0.5 and of its exact inverse."""
    ident = reg_oracle.identity_map(shape, dtype)
    fwd = (0.5 + scale * (ident - 0.5)) - ident
    inv = (0.5 + (ident - 0.5) / scale) - ident
    return fwd, inv


def test_gradient_icon_is_zero_for_an_affine_pair_and_its_inverse():
    shape = (9, 11, 10)
    fwd, inv = _affine_pair(shape, 0.8)
    # phi_BA contracts toward the centre, phi_AB expands back.  With zero noise the shifted starts Ie + delta e_d of the
    # upper faces lie outside [0, 1], where the border clamp breaks exactness; a "noise" that pulls every start 5%
    # toward the centre keeps all sample points inside
    phi_BA, phi_AB = lo.fields_closure([fwd]), lo.fields_closure([inv])
    ident = reg_oracle.identity_map(shape, torch.float64)
    inward = (0.5 + 0.95 * (ident - 0.5) - ident) * shape[-1]
    assert lo.gradient_icon_loss(phi_AB, phi_BA, inward).item() <= 1e-10
    zero = torch.zeros_like(inward)
    assert lo.gradient_icon_loss(phi_AB, phi_BA, zero).item() > 1e-3      # the clamp at the border
    g = torch.Generator().manual_seed(0)
    bump = torch.randn((1, 3) + shape, generator=g, dtype=torch.float64) * 0.01
    perturbed = lo.fields_closure([fwd + bump])
    assert lo.gradient_icon_loss(phi_AB, perturbed, inward).item() > 1e-3


def test_lncc_of_scaled_and_negated_images():
    g = torch.Generator().manual_seed(1)
    I = torch.nn.functional.interpolate(torch.rand(1, 1, 4, 5, 4, generator=g, dtype=torch.float64), size=(16, 20, 18),
                                        mode="trilinear", align_corners=True)
    assert lo.lncc(I, 2 * I, sigma=2).item() == pytest.approx(0.0, abs=2e-2)
    assert lo.lncc(I, -I, sigma=2).item() == pytest.approx(2.0, abs=2e-2)
    # the 1e-5 terms are what keeps the two away from exactly 0 and 2; without texture they dominate
    assert lo.lncc(I, 2 * I, sigma=2).item() >= 0.0
    assert lo.gaussian_taps(5).numel() == 21 and lo.gaussian_taps(5).sum().item() == pytest.approx(1.0)


def test_ssd_only_interpolated_counts_only_tagged_voxels():
    shape = (6, 7, 8)
    tag = lo.inbounds_tag(shape, torch.float64)
    A = torch.zeros((1, 1) + shape, dtype=torch.float64)
    B = torch.ones_like(A)
    B[:, :, 0] = 100.0                      # the untagged shell does not count
    assert lo.ssd_only_interpolated(torch.cat([A, tag], 1), torch.cat([B, tag], 1)).item() == pytest.approx(1.0)


def test_icon_terms_of_the_identity_registration():
    shape = (10, 12, 11)
    g = torch.Generator().manual_seed(2)
    A = torch.rand((1, 1) + shape, generator=g, dtype=torch.float64)
    zero = torch.zeros((1, 3) + shape, dtype=torch.float64)
    t = lo.icon_loss_from_fields([zero], [zero], A, A, torch.randn((1, 3) + shape, generator=g, dtype=torch.float64),
                                 similarity="ssd_only_interpolated")
    assert t.similarity_loss.item() <= 1e-20 and t.transform_magnitude.item() == 0 and t.flips.item() == 0
    assert t.inverse_consistency_loss.item() == 0 and t.all_loss.item() <= 1e-20


def _cfg(similarity, sigma=5.0, lmbda=1.5, delta=1e-3):
    from oai_analysis_2_b200 import ops
    return ops.icon_loss_cfg(similarity, sigma, lmbda, delta)


@pytest.mark.parametrize("cfg,message", [
    ((7, 5.0), b"unknown similarity 7"),
    ((0, 0.0), b"sigma"),
    ((0, -1.0), b"sigma"),
    ((0, 13.0), b"sigma"),
    ((1, 0.0, 1.5, 0.0), b"delta"),
])
def test_icon_loss_rejects_bad_configurations_with_messages(cfg, message):
    from oai_analysis_2_b200 import _lib
    L = _lib.lib
    c = _cfg(*cfg)
    rc = L.oai_reg_icon_loss(None, ctypes.byref(c), None, None, None, None, ctypes.c_size_t(0), None,
                             ctypes.c_size_t(0), None)
    assert rc != 0 and message in L.oai_last_error()
    assert L.oai_reg_loss_workspace_bytes(None, ctypes.byref(c)) == 0


def test_icon_loss_and_flips_reject_missing_arguments_with_messages():
    from oai_analysis_2_b200 import _lib
    L = _lib.lib
    c = _cfg(0)
    rc = L.oai_reg_icon_loss(None, ctypes.byref(c), None, None, None, None, ctypes.c_size_t(0), None,
                             ctypes.c_size_t(0), None)
    assert rc != 0 and b"null handle" in L.oai_last_error()
    assert L.oai_reg_icon_loss(None, None, None, None, None, None, ctypes.c_size_t(0), None, ctypes.c_size_t(0),
                               None) != 0 and b"configuration" in L.oai_last_error()
    phi, count = np.zeros(3 * 5 * 5, np.float32), np.zeros(1, np.int64)
    for dims in [(1, 5, 5), (5, 1, 5), (5, 5, 1)]:
        rc = L.oai_jacobian_flips(_lib.ptr(phi), _lib.ptr(np.asarray(dims, np.int32)), None, _lib.ptr(count), None)
        assert rc != 0 and b"at least 2" in L.oai_last_error()
    rc = L.oai_jacobian_flips(None, _lib.ptr(np.asarray((4, 4, 4), np.int32)), None, _lib.ptr(count), None)
    assert rc != 0 and b"null pointer" in L.oai_last_error()


def test_python_surface_of_the_losses_module():
    from oai_analysis_2_b200 import ops
    from oai_analysis_2_b200.icon_registration import losses
    assert losses.ICONLoss._fields == ("all_loss", "inverse_consistency_loss", "similarity_loss",
                                       "transform_magnitude", "flips")
    assert losses.similarity_config(losses.LNCC(sigma=5)) == (ops.SIM_LNCC, 5.0)
    assert losses.similarity_config(losses.ssd_only_interpolated) == (ops.SIM_SSD_ONLY_INTERPOLATED, 0.0)
    with pytest.raises(ValueError):
        losses.LNCC(sigma=0)
    with pytest.raises(ValueError):
        losses.similarity_config("ncc")
    with pytest.raises(RuntimeError, match="CUDA"):
        losses.flips(torch.zeros(1, 3, 4, 4, 4))
