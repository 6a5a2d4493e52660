"""Torch oracle of GradientICON.forward's loss terms (icon_registration==1.1.2, losses.py) -- TEST INFRASTRUCTURE
ONLY.  ** parity unpinned **: icon is not installable offline, so this RESTATES the recalled algorithm on the closures
oracle/reg_oracle.py already builds (tree_forward, sample).  Works in float32 and float64, on the CPU and, from tensors
that are already there, on a CUDA device (the torch bar of scripts/bench_icon_loss.py).

  ICONLoss(all_loss, inverse_consistency_loss, similarity_loss, transform_magnitude, flips)
    similarity_loss          = sim(S(A, phi_AB(id)), B) + sim(S(B, phi_BA(id)), A)
    inverse_consistency_loss = sum_d mean(((e(Ie) - e(Ie + delta e_d)) / delta)^2),  e(c) = c - phi_AB(phi_BA(c)),
                               Ie = identity + noise / W
    transform_magnitude      = mean((identity - phi_AB(id))^2)
    flips                    = #{dV < 0} of phi_BA(id)          (sic: GradientICON.forward counts phi_BA's folds)
    all_loss                 = lmbda * inverse_consistency_loss + similarity_loss
"""
from collections import namedtuple

import numpy as np
import torch
import torch.nn.functional as F

from oracle import reg_oracle

ICONLoss = namedtuple("ICONLoss", "all_loss inverse_consistency_loss similarity_loss transform_magnitude flips")


def gaussian_taps(sigma, dtype=torch.float64):
    """LNCC.blur's kernel: 4*sigma (+1 to make it odd) taps, exp(-x^2 / (2 sigma^2)) normalised to sum 1."""
    k = sigma * 4
    k = int(k + (1 - k % 2))
    x = torch.linspace(-(k - 1) / 2, (k - 1) / 2, k, dtype=torch.float64)
    w = torch.exp(-x ** 2 / (2 * sigma ** 2))
    return (w / w.sum()).to(dtype)


def blur(x, sigma):
    """Separable Gaussian along z, then y, then x as grouped conv3d(padding="same"): zero padding."""
    w = gaussian_taps(sigma, x.dtype).to(x.device)
    k = w.numel()
    C = x.shape[1]
    for shape in ((k, 1, 1), (1, k, 1), (1, 1, k)):
        x = F.conv3d(x, w.view(1, 1, *shape).repeat(C, 1, 1, 1, 1), padding="same", groups=C)
    return x


def lncc(I, J, sigma=5):
    """LNCC(sigma)(I, J) = mean(1 - (G(IJ) - G(I)G(J)) / sqrt((relu(G(I^2) - G(I)^2) + 1e-5)(relu(G(J^2) - G(J)^2) + 1e-5)))"""
    GI, GJ = blur(I, sigma), blur(J, sigma)
    num = blur(I * J, sigma) - GI * GJ
    den = torch.sqrt((torch.relu(blur(I * I, sigma) - GI ** 2) + 1e-5) * (torch.relu(blur(J * J, sigma) - GJ ** 2) + 1e-5))
    return torch.mean(1 - num / den)


def inbounds_tag(shape, dtype=torch.float32):
    t = torch.zeros((1, 1) + tuple(shape), dtype=dtype)
    t[:, :, 1:-1, 1:-1, 1:-1] = 1.0
    return t


def ssd_only_interpolated(image_A, image_B):
    """image_A / image_B carry the in-bounds tag as their last channel: sum(tag (A - B)^2) / sum(tag), batch mean."""
    mask = image_A[:, -1:]
    a, b = image_A[:, :-1], image_B[:, :-1]
    return torch.mean(torch.sum(mask * (a - b) ** 2, (2, 3, 4)) / torch.sum(mask, (2, 3, 4)))


def jacobian_det(phi):
    """losses.flips' dV: [N,1,D-1,H-1,W-1] from forward differences at [1:, 1:, 1:]."""
    a = phi[:, :, 1:, 1:, 1:] - phi[:, :, :-1, 1:, 1:]
    b = phi[:, :, 1:, 1:, 1:] - phi[:, :, 1:, :-1, 1:]
    c = phi[:, :, 1:, 1:, 1:] - phi[:, :, 1:, 1:, :-1]
    return torch.sum(torch.cross(a, b, dim=1) * c, dim=1, keepdim=True)


def flips(phi, in_percentage=False):
    dV = jacobian_det(phi)
    if in_percentage:
        return torch.mean((dV < 0).to(phi.dtype)) * 100.0
    return torch.sum(dV < 0) / phi.shape[0]


def gradient_icon_loss(phi_AB, phi_BA, noise, delta=1e-3):
    """phi_AB / phi_BA: closures c -> coordinates (called without the identity shortcut); noise [1,3,D,H,W] N(0,1)."""
    shape = noise.shape[2:]
    Ie = reg_oracle.identity_map(shape, noise.dtype).to(noise.device) + noise / shape[-1]
    err = Ie - phi_AB(phi_BA(Ie))
    loss = 0
    for d in range(3):
        step = torch.zeros((1, 3, 1, 1, 1), dtype=noise.dtype, device=noise.device)
        step[0, d] = delta
        err_d = Ie + step - phi_AB(phi_BA(Ie + step))
        loss = loss + torch.mean(((err - err_d) / delta) ** 2)
    return loss


def fields_closure(fields):
    """The cascade's transform from its displacement fields [1,3,d,h,w] in application order (first applied first):
    c -> c + S(u, c) per field; the first one is added without interpolation on the identity map of its own shape."""
    def t(c, ident=False):
        for i, u in enumerate(fields):
            c = c + u if (i == 0 and ident and c.shape == u.shape) else c + reg_oracle.sample(u, c)
        return c
    return t


def icon_terms(phi_AB, phi_BA, A, B, noise, similarity="lncc", sigma=5, lmbda=1.5, delta=1e-3):
    """GradientICON.forward's ICONLoss on transform closures t(c, is_identity_map) and the pair at the network shape."""
    ident = reg_oracle.identity_map(A.shape[2:], A.dtype).to(A.device)
    vf_AB, vf_BA = phi_AB(ident, True), phi_BA(ident, True)
    if similarity == "lncc":
        sim = lncc(reg_oracle.sample(A, vf_AB), B, sigma) + lncc(reg_oracle.sample(B, vf_BA), A, sigma)
    elif similarity == "ssd_only_interpolated":
        tag = inbounds_tag(A.shape[2:], A.dtype).to(A.device)
        At, Bt = torch.cat([A, tag], 1), torch.cat([B, tag], 1)
        sim = (ssd_only_interpolated(reg_oracle.sample(At, vf_AB), Bt) +
               ssd_only_interpolated(reg_oracle.sample(Bt, vf_BA), At))
    else:
        raise ValueError(similarity)
    ic = gradient_icon_loss(phi_AB, phi_BA, noise, delta)
    tm = torch.mean((ident - vf_AB) ** 2)
    return ICONLoss(lmbda * ic + sim, ic, sim, tm, flips(vf_BA))


def icon_loss_from_fields(fields_AB, fields_BA, A, B, noise, **kw):
    """icon_terms on the cascade's own displacement fields (application order), e.g. those of oai_reg_field."""
    return icon_terms(fields_closure(fields_AB), fields_closure(fields_BA), A, B, noise, **kw)


def icon_loss(sd, A, B, noise, dtype=torch.float64, **kw):
    """GradientICON.forward(A, B) from a regis_net state dict: A, B [1,1,*shape] at the network shape."""
    tree, nets = reg_oracle.tree_from_state_dict(sd)
    nets = {k: {n: (v.to(dtype) if v.is_floating_point() else v) for n, v in g.items()} for k, g in nets.items()}
    A, B, noise = A.to(dtype), B.to(dtype), noise.to(dtype)
    with torch.no_grad():
        return icon_terms(reg_oracle.tree_forward(tree, nets, A, B), reg_oracle.tree_forward(tree, nets, B, A), A, B,
                          noise, **kw)


def folded_map(shape, z0, z1):
    """Identity map whose z coordinate runs backwards on the slab z0 <= z < z1: every cell whose forward z difference
    lies inside the slab has dV < 0, i.e. (z1 - z0 - 1) * (H - 1) * (W - 1) folded cells when 1 <= z0 < z1 <= D."""
    phi = reg_oracle.identity_map(shape, torch.float64).clone()
    D = shape[0]
    z = np.arange(D, dtype=np.float64)
    zz = z.copy()
    zz[z0:z1] = (z0 + z1 - 1 - z[z0:z1])            # mirrored inside the slab
    phi[0, 0] = torch.from_numpy(zz / (D - 1)).view(D, 1, 1).expand(*shape)
    return phi
