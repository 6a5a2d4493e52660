"""icon_registration.pretrained_models.OAI_knees_gradICON_model on B200.

The reference builds GradientICON(TwoStep(TwoStep(Downsample(TwoStep(phi, psi)), xi), omega), similarity, lmbda) and
at inference only uses the four tallUNet2 and the closures composing them; the loss terms GradientICON.forward also
computes are discarded by register_pair, so model(A, B) does not evaluate them.  GradICONModel.icon_loss computes them
on request (similarity, inverse consistency, transform magnitude, folds) as a registration-quality check."""
import os

import numpy as np
import torch

from .. import ops
from ..segmentation.utils import load_checkpoint
from .losses import LNCC, ICONLoss, similarity_config
from .networks import TallUNet2

# Module tree of OAI_knees_gradICON_model().regis_net as SURVEY App. B.2 recalls it:
#   TwoStep(TwoStep(Downsample(TwoStep(FFVF(phi), FFVF(psi))), FFVF(xi)), FFVF(omega))
# The un-vendored package cannot be inspected offline, so this is only the DEFAULT (random-init) tree: loading a
# checkpoint re-derives the tree from the checkpoint's own key paths (parse_tree), e.g. icon's
# make_network(..., include_last_step=True) layout TwoStep(TwoStep(Down(TwoStep(Down(phi), psi)), xi), omega).
DEFAULT_PATHS = ("netPhi.netPhi.net.netPhi.net", "netPhi.netPhi.net.netPsi.net", "netPhi.netPsi.net", "netPsi.net")
INPUT_SHAPE = [1, 1, 80, 192, 192]
# GradientICON's similarity and lmbda of the knee model as recalled, not verified (SURVEY App. B.2, DESIGN.md §2)
DEFAULT_SIMILARITY_SIGMA = 5
DEFAULT_LMBDA = 1.5
WEIGHTS_ENV = "OAI_B200_GRADICON_WEIGHTS"
_UNET_PARAMS = ("downConvs.", "upConvs.", "batchNorms.", "lastConv.")


def split_checkpoint(sd):
    """{unet path: {unet key: tensor}} from a regis_net state dict (keys with or without the 'regis_net.' prefix).
    Every key must belong to a tallUNet2 somewhere in the tree; `identity_map` buffers (older icon versions saved
    them) are the only thing skipped.  Anything else raises: a checkpoint this loader does not understand must not
    "load" and leave random weights behind."""
    out, unknown = {}, []
    for k, v in sd.items():
        key = k[len("regis_net."):] if k.startswith("regis_net.") else k
        if key.endswith("identity_map"):
            continue
        cut = min((key.find(h) for h in _UNET_PARAMS if h in key), default=-1)
        path = key[:cut].rstrip(".") if cut > 0 else ""
        if cut <= 0 or not path or any(t not in ("netPhi", "netPsi", "net") for t in path.split(".")):
            unknown.append(k)
            continue
        out.setdefault(path, {})[key[cut:]] = v
    if unknown:
        raise RuntimeError(f"GradICON checkpoint has {len(unknown)} key(s) outside any tallUNet2 of the registration "
                           f"tree, e.g. {unknown[:3]}")
    if not out:
        raise RuntimeError("GradICON checkpoint holds no tallUNet2 weights")
    return out


def parse_tree(paths):
    """Registration module tree from the UNets' key paths.  'netPhi' / 'netPsi' are the children of a
    TwoStepRegistration; 'net' is FunctionFromVectorField.net when it ends a path and DownsampleRegistration.net
    otherwise.  Returns nested tuples ("twostep", phi, psi) | ("down", child) | ("ffvf", path)."""
    def build(prefix, rel):
        if rel == [("net",)]:
            return ("ffvf", ".".join(prefix + ("net",)))
        firsts = {r[0] for r in rel if r}
        if any(not r for r in rel) or not firsts:
            raise RuntimeError(f"GradICON checkpoint: malformed module path under {'.'.join(prefix) or '<root>'}")
        if firsts == {"net"}:
            return ("down", build(prefix + ("net",), [r[1:] for r in rel]))
        if firsts == {"netPhi", "netPsi"}:
            return ("twostep", build(prefix + ("netPhi",), [r[1:] for r in rel if r[0] == "netPhi"]),
                    build(prefix + ("netPsi",), [r[1:] for r in rel if r[0] == "netPsi"]))
        raise RuntimeError(f"GradICON checkpoint: cannot interpret children {sorted(firsts)} under "
                           f"{'.'.join(prefix) or '<root>'} (expected netPhi+netPsi, or net)")
    return build((), [tuple(p.split(".")) for p in sorted(paths)])


def tree_leaves(tree):
    if tree[0] == "ffvf":
        return [tree[1]]
    return [p for child in tree[1:] for p in tree_leaves(child)]


def describe_tree(tree):
    if tree[0] == "ffvf":
        return "FFVF"
    if tree[0] == "down":
        return f"Down({describe_tree(tree[1])})"
    return f"TwoStep({describe_tree(tree[1])}, {describe_tree(tree[2])})"


class GradICONModel:
    """Inference-side equivalent of the object OAI_knees_gradICON_model() returns: exposes .identity_map,
    .assign_identity_map, .to/.cuda/.eval, .regis_net state loading, __call__(A, B), .phi_AB / .phi_BA."""

    def __init__(self, paths=DEFAULT_PATHS):
        self.tree = parse_tree(paths)
        self.nets = {p: TallUNet2() for p in tree_leaves(self.tree)}
        self.device = torch.device("cpu")
        self.input_shape = list(INPUT_SHAPE)
        self._identity = None
        self._handle, self._handle_key = None, None
        self.phi_AB_vectorfield = None
        self.phi_BA_vectorfield = None
        self.similarity = LNCC(sigma=DEFAULT_SIMILARITY_SIGMA)
        self.lmbda = DEFAULT_LMBDA
        self.delta = 1e-3

    # -- module-like surface
    def assign_identity_map(self, input_shape):
        self.input_shape = [1, 1] + [int(v) for v in input_shape[2:]]
        self._identity = None

    @property
    def identity_map(self):
        if self._identity is None:
            D, H, W = self.input_shape[2:]
            axes = [torch.arange(n, dtype=torch.float64) * (1.0 / (n - 1)) for n in (D, H, W)]
            self._identity = torch.stack(torch.meshgrid(*axes, indexing="ij"), 0)[None].float().to(self.device)
        return self._identity

    def to(self, device):
        self.device = torch.device(device)
        for n in self.nets.values():
            n.to(self.device)
        self._identity = None
        return self

    def cuda(self):
        return self.to("cuda")

    def eval(self):
        return self

    def state_dict(self):
        sd = {}
        for path, net in self.nets.items():
            sd.update(net.state_dict(prefix=f"regis_net.{path}."))
        return sd

    def load_state_dict(self, sd, strict=True):
        """Loads a regis_net checkpoint (keys with or without the 'regis_net.' prefix) and REBUILDS the module tree
        from its key paths, so both the SURVEY tree and icon's two-level-downsample tree load.  Fails loudly: every
        tensor in the file must be consumed by exactly one tallUNet2 and every tallUNet2 must be complete -- strict
        is accepted for signature compatibility (icon calls regis_net.load_state_dict(..., strict=False)) but a
        partial load is never silently accepted."""
        groups = split_checkpoint(sd)
        tree = parse_tree(groups.keys())
        nets = {}
        for path in tree_leaves(tree):
            net = TallUNet2()
            net.load_state_dict(groups[path], strict=True)   # raises on missing / unexpected / mis-shaped keys
            nets[path] = net.to(self.device) if self.device.type == "cuda" else net
        self.tree, self.nets = tree, nets
        self.phi_AB_vectorfield = self.phi_BA_vectorfield = None
        return self

    # -- inference: the cascade runs behind the stage-level C ABI (csrc/reg_net.cu: oai_reg_create / oai_reg_forward)
    def _stage(self):
        """The library-side model (packed weights + workspace), rebuilt when the weights, the network shape or the
        device change (in-place edits of a UNet's tensors are seen through their version counters)."""
        key = (tuple(self.input_shape[2:]), str(self.device), tuple(self.nets),
               tuple((id(t), t._version) for net in self.nets.values() for t in net._sd.values()))
        if self._handle is None or self._handle_key != key:
            if self.device.type != "cuda":
                raise RuntimeError("oai_analysis_2_b200 registration runs on CUDA (sm_100a) only")
            self._handle = None   # release the old weights / workspace before allocating the new ones
            self._handle = ops.RegHandle(self.state_dict(), self.input_shape[2:], self.device)
            self._handle_key = key
        return self._handle

    def register_native(self, A, B):
        """A, B: float32 [D,H,W] cuda volumes of any size (register_pair resizes them to the network shape).  Runs both
        directions batched through the cascade and stores phi_AB / phi_BA evaluated on the identity map."""
        phi_AB, phi_BA, _, _ = self._stage().forward(A.contiguous().float(), B.contiguous().float())
        self.phi_AB_vectorfield, self.phi_BA_vectorfield = phi_AB[None], phi_BA[None]
        return self.phi_AB_vectorfield, self.phi_BA_vectorfield

    def forward(self, image_A, image_B):
        """image_A/B: [1,1,D,H,W] (or [D,H,W]) float32 cuda at the network resolution."""
        A = image_A.reshape(image_A.shape[-3:])
        B = image_B.reshape(image_B.shape[-3:])
        if list(A.shape) != self.input_shape[2:]:
            raise ValueError(f"images must be resized to the network shape {self.input_shape[2:]}, got {list(A.shape)}")
        return self.register_native(A, B)

    __call__ = forward

    @property
    def fields(self):
        """The cascade's displacement fields of the last pair, application order, [2 directions, 3, d, h, w] each
        (views into the stage workspace: the next pair overwrites them)."""
        return self._stage().fields()

    def warp_image(self, image, direction=0, out=None):
        """as_function(image)(phi(identity_map)) for the last registered pair: `image` [D,H,W] (any size) warped by
        phi_AB (direction 0) or phi_BA (1), fused with the composition (no map is materialised)."""
        if self.phi_AB_vectorfield is None:
            raise RuntimeError("call the model on an image pair first")
        shape = tuple(image.shape[-3:])
        return self._stage().warp_image(image.reshape(shape).contiguous(), direction, out)

    def icon_loss(self, image_A, image_B, noise=None):
        """GradientICON.forward(A, B)'s ICONLoss for the pair at the network shape ([1,1,D,H,W] or [D,H,W] float32
        cuda, as forward takes them): registers it (phi_AB / phi_BA are updated as by model(A, B)) and returns
        ICONLoss(all_loss, inverse_consistency_loss, similarity_loss, transform_magnitude, flips) of 0-d float64 CUDA
        tensors, with self.similarity and self.lmbda.  noise: N(0, 1) of the identity map's shape [1,3,D,H,W]; when
        None it is drawn as icon draws it (torch.randn on the CPU default generator), so torch.manual_seed reproduces
        icon's Iepsilon."""
        self.forward(image_A, image_B)
        if noise is None:
            noise = torch.randn(*self.identity_map.shape)
        noise = noise.to(device=self.device, dtype=torch.float32).reshape(3, *self.input_shape[2:]).contiguous()
        kind, sigma = similarity_config(self.similarity)
        terms, _ = self._stage().icon_loss(noise, kind, sigma, self.lmbda, self.delta)
        return ICONLoss(*terms.unbind())

    def _eval_on_identity(self, field, coords):
        if field is None:
            raise RuntimeError("call the model on an image pair first")
        if coords is not self.identity_map and tuple(coords.shape) != tuple(self.identity_map.shape):
            raise NotImplementedError("phi_AB / phi_BA are evaluated on the model's identity map (register_pair usage)")
        return field

    def phi_AB(self, coords):
        return self._eval_on_identity(self.phi_AB_vectorfield, coords)

    def phi_BA(self, coords):
        return self._eval_on_identity(self.phi_BA_vectorfield, coords)


def OAI_knees_gradICON_model(pretrained=True, weights_path=None, similarity=None, lmbda=None):
    """pretrained_models.OAI_knees_gradICON_model.  The reference downloads the checkpoint from a GitHub release;
    here `weights_path` (or $OAI_B200_GRADICON_WEIGHTS) must point at that file when pretrained=True.
    similarity (losses.LNCC(sigma) or losses.ssd_only_interpolated) and lmbda override the loss configuration that
    icon_loss uses; registration itself does not depend on them."""
    net = GradICONModel()
    net.assign_identity_map(INPUT_SHAPE)
    if similarity is not None:
        similarity_config(similarity)   # raises for anything the library cannot compute
        net.similarity = similarity
    if lmbda is not None:
        net.lmbda = float(lmbda)
    if pretrained:
        path = weights_path or os.environ.get(WEIGHTS_ENV)
        if not path or not os.path.isfile(path):
            raise FileNotFoundError(
                "pretrained GradICON knee weights not found: pass weights_path= or set $%s (no network access to the "
                "release the reference downloads from)" % WEIGHTS_ENV)
        net.load_state_dict(load_checkpoint(path), strict=False)
    if torch.cuda.is_available():
        net.to("cuda")
    net.eval()
    return net
