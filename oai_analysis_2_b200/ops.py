"""Thin Python wrappers over the C-ABI ops (torch tensors in, torch tensors out; torch is only the allocator)."""
import ctypes
import math

import numpy as np
import torch

from ._lib import c_double, c_float, c_int, c_ll, c_size, check, lib, ptr, stream_ptr

FLAG_FORCE_PER_TAP = 1
FLAG_BASE_OFF_FORMULA = 2
FLAG_FORCE_KD1 = 4
FLAG_NO_FAST_PATH = 8
FLAG_WIDE_N = 16

_DT16 = {0: torch.float16, 1: torch.bfloat16}


def conv_plan(D, H, W, c0, c1, cout, pointwise=False, flags=0):
    plan = (c_int * 9)()
    check(lib.oai_conv3d_igemm_plan(D, H, W, c0, c1, cout, int(pointwise), flags, plan), "conv plan")  # 2 = up2
    keys = ("mode", "kd_per_block", "R", "nhalf", "cout_per_half", "nblk", "wblock_bytes", "nchunks", "row_bytes")
    return dict(zip(keys, list(plan)))


def pack_conv_weights(w, c0, c1, D, H, W, pointwise=False, ab_format=0, flags=0, device="cuda"):
    """w: float32 [cout, c0+c1, 3,3,3] (conv orientation) or [cout, c0+c1] when pointwise.  Returns a uint8 tensor."""
    w = np.ascontiguousarray(w.detach().cpu().numpy() if hasattr(w, "detach") else w, dtype=np.float32)
    cout = w.shape[0]
    assert w.shape[1] == c0 + c1
    pl = conv_plan(D, H, W, c0, c1, cout, pointwise, flags)
    nbytes = pl["nhalf"] * pl["nblk"] * pl["wblock_bytes"]
    dst = np.zeros(nbytes, dtype=np.uint8)
    check(lib.oai_pack_conv_weights(ptr(w), cout, c0, c1, D, H, W, int(pointwise), ab_format, flags, ptr(dst),
                                    c_size(nbytes)), "pack weights")
    return torch.from_numpy(dst).to(device)


def conv3d_igemm(src0, src1, wpack, bias, cout, pointwise=False, relu=True, ab_format=0, out=None, out_view=None,
                 flags=0, region=None):
    """src*: [NT, D, H, W, C] 16-bit channels-last.  Returns [NT, D, H, W, cout] unless `out`/`out_view` given.

    out_view = (obase, osN, osD, osH, osW) in elements addresses into `out` (k2s2 transposed-conv scatter).
    """
    NT, D, H, W, c0 = src0.shape
    c1 = 0 if src1 is None else src1.shape[-1]
    assert src0.is_contiguous() and (src1 is None or src1.is_contiguous())
    if out is None:
        out = torch.empty((NT, D, H, W, cout), dtype=_DT16[ab_format], device=src0.device)
    if out_view is None:
        out_view = (0, D * H * W * cout, H * W * cout, W * cout, cout)
    ob, sn, sd, sh, sw = out_view
    if region is None:
        check(lib.oai_conv3d_igemm(ptr(src0), c0, ptr(src1), c1, NT, D, H, W, ptr(wpack), c_size(wpack.numel()),
                                   ptr(bias), cout, int(pointwise), int(relu), ab_format, ptr(out), c_ll(ob), c_ll(sn),
                                   c_ll(sd), c_ll(sh), c_ll(sw), flags, stream_ptr()), "conv3d_igemm")
    else:
        reg = np.asarray(region, dtype=np.int32)  # d_lo, d_cnt, h_lo, h_cnt: dead halo outside is not computed
        check(lib.oai_conv3d_igemm_region(ptr(src0), c0, ptr(src1), c1, NT, D, H, W, ptr(wpack),
                                          c_size(wpack.numel()), ptr(bias), cout, int(pointwise), int(relu), ab_format,
                                          ptr(out), c_ll(ob), c_ll(sn), c_ll(sd), c_ll(sh), c_ll(sw), flags, ptr(reg),
                                          stream_ptr()), "conv3d_igemm_region")
    return out


# ------------------------------------------------------------------------------------------------ stage-level segmentation
class _SegConfig(ctypes.Structure):
    _fields_ = [("in_channels", c_int), ("n_classes", c_int), ("bias", c_int), ("BN", c_int),
                ("patch_xyz", c_int * 3), ("overlap_xyz", c_int * 3), ("ab_format", c_int), ("precision", c_int),
                ("layer_terms", c_int * 17)]


class _Tensor(ctypes.Structure):
    _fields_ = [("name", ctypes.c_char_p), ("data", ctypes.c_void_p), ("ndim", c_int), ("shape", c_ll * 5)]


def seg_layer_terms(precision):
    t = (c_int * 17)()
    check(lib.oai_seg_layer_terms(int(precision), t), "seg_layer_terms")
    return list(t)


def seg_needed_regions(tile_zyx, overlap_zyx):
    """[17, 6] int array: inclusive lo(z,y,x), hi(z,y,x) per layer ec0..dc1 (host arithmetic in the library)."""
    boxes = np.zeros((17, 6), dtype=np.int32)
    check(lib.oai_seg_needed_regions(ptr(np.asarray(tile_zyx, dtype=np.int32)),
                                     ptr(np.asarray(overlap_zyx, dtype=np.int32)), ptr(boxes)), "seg_needed_regions")
    return boxes


class SegHandle:
    """oai_seg_create / oai_seg_forward / oai_seg_destroy: the whole segmentation stage behind one handle."""

    def __init__(self, state_dict, in_channels, n_classes, bias, BN, patch_xyz, overlap_xyz, ab_format=0, precision=1,
                 layer_terms=None):
        cfg = _SegConfig(int(in_channels), int(n_classes), int(bool(bias)), int(bool(BN)),
                         (c_int * 3)(*[int(v) for v in patch_xyz]), (c_int * 3)(*[int(v) for v in overlap_xyz]),
                         int(ab_format), 4 if layer_terms is not None else int(precision),
                         (c_int * 17)(*([int(v) for v in layer_terms] if layer_terms is not None else [1] * 17)))
        keep, arr = [], (_Tensor * len(state_dict))()
        for i, (k, v) in enumerate(state_dict.items()):
            a = np.ascontiguousarray(torch.as_tensor(v).detach().cpu().numpy(), dtype=np.float32)
            keep.append(a)
            shape = list(a.shape) + [0] * (5 - a.ndim)
            arr[i] = _Tensor(k.encode(), a.ctypes.data, a.ndim, (c_ll * 5)(*shape))
        self._h = ctypes.c_void_p()
        self._auto = {}
        self._ws = None
        self.n_classes = int(n_classes)
        self.device = torch.device("cuda", torch.cuda.current_device())
        check(lib.oai_seg_create(ctypes.byref(cfg), arr, len(state_dict), ctypes.byref(self._h)), "seg_create")

    def __del__(self, _destroy=lib.oai_seg_destroy):   # bound at class creation: module globals are gone at shutdown
        h, self._h = getattr(self, "_h", None), None
        if h:
            _destroy(h)

    def num_tiles(self, vol_shape):
        return int(lib.oai_seg_num_tiles(self._h, ptr(np.asarray(vol_shape, dtype=np.int32))))

    def workspace_bytes(self, vol_shape, tiles_per_batch=0):
        return int(lib.oai_seg_workspace_bytes(self._h, ptr(np.asarray(vol_shape, dtype=np.int32)),
                                               int(tiles_per_batch or 0)))

    def auto_tiles_per_batch(self, vol_shape, fraction=0.5):
        """All tiles in one batch when the activation workspace fits `fraction` of the free device memory (plus what
        torch's caching allocator already holds), otherwise the largest even split that does.  (On a 180 GB B200 the
        default "mixed" plan runs a 160-tile knee as one batch, 75 GB: measured 1.7 ms per knee faster than 2 x 80 tiles
        and 3 ms faster than 4 x 40 -- fewer launches and shorter tails; pass tiles_per_batch to override.)"""
        key = tuple(int(v) for v in vol_shape)
        if key in self._auto:   # decided once per shape (also keeps CUDA-graph capture free of memory queries)
            return self._auto[key]
        T = self.num_tiles(vol_shape)
        free, _ = torch.cuda.mem_get_info(self.device)
        budget = fraction * (free + torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device))
        for parts in range(1, T + 1):
            nb = -(-T // parts)
            if self.workspace_bytes(vol_shape, nb) <= budget:
                self._auto[key] = nb
                return nb
        raise OaiErrorNoMemory(f"not even one tile's activations fit the free device memory ({free} bytes)")

    def forward(self, vol, out_mode=0, tiles_per_batch=0, out=None, workspace=None):
        """vol: float32 [D,H,W] cuda -> float32 [ncls, D, H, W] (0 probabilities, 1 masks, 2 logits)."""
        assert vol.dtype == torch.float32 and vol.is_contiguous() and vol.is_cuda
        dims = np.asarray(vol.shape, dtype=np.int32)
        if out is None:
            out = torch.empty((self.n_classes,) + tuple(vol.shape), dtype=torch.float32, device=vol.device)
        need = self.workspace_bytes(vol.shape, tiles_per_batch)
        if workspace is None or workspace.numel() < need:
            # The activation workspace (tens of GB) is kept on the handle and reused by later calls: allocating and
            # freeing it per call leaves one cached block per stream / graph pool behind, and three of those do not fit
            # a 180 GB device.  A handle therefore serves one stream at a time (the reference's segmenter is not
            # thread-safe either, SURVEY 8b); a CUDA graph captured over it keeps using this buffer.
            if self._ws is None or self._ws.numel() < need or self._ws.device != vol.device:
                self._ws = None
                self._ws = torch.empty(need, dtype=torch.uint8, device=vol.device)
            workspace = self._ws
        check(lib.oai_seg_forward(self._h, ptr(vol), ptr(dims), ptr(out), int(out_mode), int(tiles_per_batch or 0),
                                  ptr(workspace), c_size(workspace.numel()), stream_ptr()), "seg_forward")
        return out


def conv_overflow_count(reset=True):
    """fp16 saturation guard of the conv epilogue (synchronises the current stream)."""
    n = c_ll(0)
    check(lib.oai_conv_overflow_count(ctypes.byref(n), int(reset), stream_ptr()), "conv_overflow_count")
    return int(n.value)


class OaiErrorNoMemory(RuntimeError):
    pass


# ------------------------------------------------------------------------------------------------ segmentation misc
def make_geom(tile_zyx, effective_zyx, overlap_zyx, grid_zyx):
    """geom[12] = tile, effective, overlap, grid (all z,y,x) as the C ABI expects."""
    return np.asarray(list(tile_zyx) + list(effective_zyx) + list(overlap_zyx) + list(grid_zyx), dtype=np.int32)


def seg_stem(vol, geom, tile0, ntiles, w27c, bias, ab_format=0, out_split=False):
    """vol: float32 [D,H,W] cuda.  Returns act16 [ntiles, td, th, tw, c0] ([.., 2*c0] = [hi | lo] when out_split)."""
    assert vol.dtype == torch.float32 and vol.is_contiguous()
    dims = np.asarray(vol.shape, dtype=np.int32)
    c0 = w27c.shape[1]
    td, th, tw = (int(v) for v in geom[:3])
    out = torch.empty((ntiles, td, th, tw, c0 * (2 if out_split else 1)), dtype=_DT16[ab_format], device=vol.device)
    check(lib.oai_seg_stem_ex(ptr(vol), ptr(dims), ptr(geom), tile0, ntiles, ptr(w27c), ptr(bias), c0, ptr(out),
                              ab_format, int(out_split), stream_ptr()), "seg_stem")
    return out


def maxpool2(x, ab_format=0, in_split=False, out_split=False):
    """x: act16 [N,D,H,W,C] ([.., 2C] = [hi | lo] when in_split)."""
    N, D, H, W, CP = x.shape
    C = CP // 2 if in_split else CP
    out = torch.empty((N, D // 2, H // 2, W // 2, C * (2 if out_split else 1)), dtype=x.dtype, device=x.device)
    check(lib.oai_maxpool3d_2_ex(ptr(x), ptr(out), N, D, H, W, C, int(in_split), int(out_split), ab_format,
                                 stream_ptr()), "maxpool3d_2")
    return out


def split16(x, ab_format=0):
    """float32 [..., C] -> act16 [..., 2C] = [hi | lo] (hi = rn16(x), lo = rn16(x - hi)): the split-tensor layout."""
    hi = x.to(_DT16[ab_format])
    lo = (x - hi.float()).to(_DT16[ab_format])
    return torch.cat((hi, lo), dim=-1).contiguous()


def conv_plan_ex(D, H, W, c0, c1, cout, pointwise=0, terms=1, flags=0):
    plan = (c_int * 10)()
    check(lib.oai_conv3d_igemm_plan_ex(D, H, W, c0, c1, cout, int(pointwise), int(terms), flags, plan), "conv plan")
    keys = ("mode", "kd_per_block", "R", "nhalf", "cout_per_half", "nblk", "wblock_bytes", "nchunks", "row_bytes",
            "packed_16B")
    return dict(zip(keys, list(plan)))


def pack_conv_weights_ex(w, c0, c1, D, H, W, pointwise=0, terms=1, ab_format=0, flags=0, device="cuda"):
    """w: float32 conv orientation [cout, c0+c1, taps...] (27 taps, none, or 2x2x2 for pointwise 0 / 1 / 2)."""
    w = np.ascontiguousarray(w.detach().cpu().numpy() if hasattr(w, "detach") else w, dtype=np.float32)
    cout = w.shape[0]
    assert w.shape[1] == c0 + c1
    nbytes = conv_plan_ex(D, H, W, c0, c1, cout, pointwise, terms, flags)["packed_16B"] * 16
    dst = np.zeros(nbytes, dtype=np.uint8)
    check(lib.oai_pack_conv_weights_ex(ptr(w), cout, c0, c1, D, H, W, int(pointwise), int(terms), ab_format, flags,
                                       ptr(dst), c_size(nbytes)), "pack weights")
    return dst if device is None else torch.from_numpy(dst).to(device)


def conv3d_igemm_ex(src0, src1, wpack, bias, cout, c0, c1=0, pointwise=0, relu=True, ab_format=0, terms=1,
                    in_split=False, out_split=False, region=None, flags=0):
    """Split-precision form of conv3d_igemm: src* are [NT,D,H,W,C] (or [.., 2C] = [hi | lo] when in_split)."""
    NT, D, H, W, _ = src0.shape
    assert src0.is_contiguous() and (src1 is None or src1.is_contiguous())
    up = 2 if pointwise == 2 else 1
    out = torch.empty((NT, up * D, up * H, up * W, cout * (2 if out_split else 1)), dtype=_DT16[ab_format],
                      device=src0.device)
    reg = None if region is None else np.asarray(region, dtype=np.int32)
    check(lib.oai_conv3d_igemm_ex(ptr(src0), c0, ptr(src1), c1, int(in_split), NT, D, H, W, ptr(wpack),
                                  c_size(wpack.numel()), ptr(bias), cout, int(pointwise), int(relu), ab_format,
                                  int(terms), ptr(out), int(out_split), flags, ptr(reg), stream_ptr()),
          "conv3d_igemm_ex")
    return out


def seg_head(act, w, b, out, geom, tile0, crop_zyx, out_mode=0, ab_format=0):
    """act: act16 [ntiles, td, th, tw, C]; out: float32 [ncls, VD, VH, VW] (written in place)."""
    ntiles, C = act.shape[0], act.shape[-1]
    ncls = w.shape[0]
    dims = np.asarray(out.shape[1:], dtype=np.int32)
    crop = np.asarray(crop_zyx, dtype=np.int32)
    check(lib.oai_seg_head(ptr(act), C, ncls, ptr(w), ptr(b), ptr(out), ptr(dims), ptr(geom), tile0, ntiles,
                           ptr(crop), out_mode, ab_format, stream_ptr()), "seg_head")
    return out


# ------------------------------------------------------------------------------------------------ stage-level registration
def _tensor_array(state_dict):
    keep, arr = [], (_Tensor * len(state_dict))()
    for i, (k, v) in enumerate(state_dict.items()):
        a = np.ascontiguousarray(torch.as_tensor(v).detach().cpu().numpy(), dtype=np.float32)
        keep.append(a)
        shape = list(a.shape)[:5] + [0] * max(0, 5 - a.ndim)
        arr[i] = _Tensor(k.encode(), a.ctypes.data, a.ndim, (c_ll * 5)(*shape))
    return keep, arr


def reg_parse_tree(state_dict):
    """Host-only: the module tree a regis_net state dict encodes, e.g. 'TwoStep(Down(FFVF), FFVF)'; raises OaiError
    for anything oai_reg_create would refuse."""
    keep, arr = _tensor_array(state_dict)
    buf = ctypes.create_string_buffer(1024)
    check(lib.oai_reg_parse_tree(arr, len(state_dict), buf, c_size(1024)), "reg_parse_tree")
    return buf.value.decode()


SIM_LNCC, SIM_SSD_ONLY_INTERPOLATED = 0, 1   # oai_icon_loss_cfg.similarity


class RegHandle:
    """oai_reg_create / oai_reg_forward / oai_reg_destroy: register_pair on the GradICON cascade behind one handle.
    The workspace (concatenation buffers, intermediate images, the cascade's displacement fields) is owned here and
    reused by every call, so a CUDA graph captured over the handle keeps valid pointers; one stream at a time."""

    def __init__(self, state_dict, net_dims, device=None):
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.net_dims = tuple(int(v) for v in net_dims)
        keep, arr = _tensor_array(state_dict)
        self._h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            check(lib.oai_reg_create(arr, len(state_dict), ptr(_dims(*self.net_dims)), ctypes.byref(self._h)),
                  "reg_create")
        self._ws = torch.empty(int(lib.oai_reg_workspace_bytes(self._h)), dtype=torch.uint8, device=self.device)

    def __del__(self, _destroy=lib.oai_reg_destroy):
        h, self._h = getattr(self, "_h", None), None
        if h:
            _destroy(h)

    def describe(self):
        buf = ctypes.create_string_buffer(1024)
        check(lib.oai_reg_describe(self._h, buf, c_size(1024)), "reg_describe")
        return buf.value.decode()

    def forward(self, A, B, want_phi=True, want_disp=False):
        """A, B: float32 contiguous cuda volumes [D,H,W] (any size).  Returns (phi_AB, phi_BA, disp_AB, disp_BA) with
        phi [3,d,h,w] and disp [d,h,w,3] on the network grid (None for what was not asked for)."""
        for t in (A, B):
            assert t.dtype == torch.float32 and t.is_contiguous() and t.is_cuda and t.dim() == 3
        d = self.net_dims
        phi = [torch.empty((3,) + d, dtype=torch.float32, device=A.device) if want_phi else None for _ in range(2)]
        disp = [torch.empty(d + (3,), dtype=torch.float32, device=A.device) if want_disp else None for _ in range(2)]
        check(lib.oai_reg_forward(self._h, ptr(A), ptr(_dims(*A.shape)), ptr(B), ptr(_dims(*B.shape)), ptr(phi[0]),
                                  ptr(phi[1]), ptr(disp[0]), ptr(disp[1]), ptr(self._ws), c_size(self._ws.numel()),
                                  stream_ptr()), "reg_forward")
        return phi[0], phi[1], disp[0], disp[1]

    def fields(self):
        """The cascade's displacement fields of the last forward, application order: views [2, 3, d, h, w] into the
        workspace (overwritten by the next forward)."""
        out = []
        for i in range(int(lib.oai_reg_num_fields(self._h))):
            off, dims = c_size(0), (c_int * 3)()
            check(lib.oai_reg_field(self._h, i, ctypes.byref(off), dims), "reg_field")
            n = 2 * 3 * dims[0] * dims[1] * dims[2] * 4
            out.append(self._ws[off.value:off.value + n].view(torch.float32).view(2, 3, dims[0], dims[1], dims[2]))
        return out

    def warp_image(self, image, direction=0, out=None):
        assert image.dtype == torch.float32 and image.is_contiguous() and image.is_cuda
        shape = tuple(image.shape[-3:])
        if out is None:
            out = torch.empty(shape, dtype=torch.float32, device=image.device)
        check(lib.oai_reg_warp_image(self._h, ptr(image), ptr(_dims(*shape)), int(direction), ptr(out), ptr(self._ws),
                                     c_size(self._ws.numel()), stream_ptr()), "reg_warp_image")
        return out

    def loss_workspace_bytes(self, similarity=SIM_LNCC, sigma=5.0, lmbda=1.5, delta=1e-3):
        cfg = icon_loss_cfg(similarity, sigma, lmbda, delta)
        n = int(lib.oai_reg_loss_workspace_bytes(self._h, ctypes.byref(cfg)))
        if n == 0:   # a refused configuration: the call reports why before touching anything
            check(lib.oai_reg_icon_loss(self._h, ctypes.byref(cfg), None, None, None, None, c_size(0), None,
                                        c_size(0), None), "reg_icon_loss")
        return n

    def icon_loss(self, noise, similarity=SIM_LNCC, sigma=5.0, lmbda=1.5, delta=1e-3, want_det=False, terms=None,
                  det=None):
        """GradientICON.forward's loss terms for the last forward (oai_reg_icon_loss).  noise: float32 cuda
        [3, *net_dims] (or [1, 3, *net_dims]) of N(0, 1) values.  Returns (terms, det): terms float64 [5] in ICONLoss
        order (all, inverse consistency, similarity, transform magnitude, flips), det the dV map of phi_BA
        [D-1, H-1, W-1] when want_det (else None).  The loss workspace is owned by the handle and only grows, so a
        CUDA graph captured over this call keeps valid pointers."""
        d = self.net_dims
        assert noise.dtype == torch.float32 and noise.is_cuda and noise.is_contiguous() and noise.numel() == 3 * math.prod(d)
        need = self.loss_workspace_bytes(similarity, sigma, lmbda, delta)
        if getattr(self, "_loss_ws", None) is None or self._loss_ws.numel() < need:
            self._loss_ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        if terms is None:
            terms = torch.empty(5, dtype=torch.float64, device=self.device)
        if want_det and det is None:
            det = torch.empty(tuple(v - 1 for v in d), dtype=torch.float32, device=self.device)
        cfg = icon_loss_cfg(similarity, sigma, lmbda, delta)
        check(lib.oai_reg_icon_loss(self._h, ctypes.byref(cfg), ptr(noise), ptr(terms), ptr(det if want_det else None),
                                    ptr(self._loss_ws), c_size(self._loss_ws.numel()), ptr(self._ws),
                                    c_size(self._ws.numel()), stream_ptr()), "reg_icon_loss")
        return terms, (det if want_det else None)


class _IconLossCfg(ctypes.Structure):
    _fields_ = [("similarity", c_int), ("sigma", c_double), ("lmbda", c_double), ("delta", c_double)]


def icon_loss_cfg(similarity=SIM_LNCC, sigma=5.0, lmbda=1.5, delta=1e-3):
    """oai_icon_loss_cfg: similarity SIM_LNCC (with sigma) or SIM_SSD_ONLY_INTERPOLATED, lmbda, delta."""
    return _IconLossCfg(int(similarity), float(sigma), float(lmbda), float(delta))


def jacobian_flips(phi, det=False):
    """losses.flips' fold count of one map phi [3, D, H, W] (or [1, 3, D, H, W]) float32 cuda: returns the number of
    cells with dV < 0 as a 0-d int64 cuda tensor, and with det=True also the dV map [D-1, H-1, W-1]."""
    assert phi.dtype == torch.float32 and phi.is_cuda and phi.is_contiguous() and phi.shape[-4] == 3
    shape = tuple(int(v) for v in phi.shape[-3:])
    count = torch.empty((), dtype=torch.int64, device=phi.device)
    dv = torch.empty(tuple(max(v - 1, 0) for v in shape), dtype=torch.float32, device=phi.device) if det else None
    check(lib.oai_jacobian_flips(ptr(phi), ptr(_dims(*shape)), ptr(dv), ptr(count), stream_ptr()), "jacobian_flips")
    return (count, dv) if det else count


# ------------------------------------------------------------------------------------------------ segmentation quality
def _mask_u8(m):
    assert m.is_cuda and m.dim() == 3 and m.dtype in (torch.bool, torch.uint8), "expected a bool/uint8 cuda [D,H,W]"
    return (m.view(torch.uint8) if m.dtype == torch.bool else m).contiguous()


def _seg_quality_ws(device, shape):
    dims = _dims(*shape)
    nbytes = int(lib.oai_seg_quality_workspace_bytes(ptr(dims)))
    return dims, _scratch_buf(device, "seg_quality", nbytes), nbytes


def distance_transform(feature, spacing_xyz):
    """scipy.ndimage.distance_transform_edt(~feature, sampling=(sz, sy, sx)) on the device, exact: feature bool/uint8
    cuda [D,H,W] -> float32 [D,H,W], the distance in mm to the nearest non-zero voxel (+inf when there is none)."""
    f = _mask_u8(feature)
    out = torch.empty(f.shape, dtype=torch.float32, device=f.device)
    dims, ws, nbytes = _seg_quality_ws(f.device, f.shape)
    sp = np.asarray(spacing_xyz, dtype=np.float64)
    check(lib.oai_distance_transform(ptr(f), ptr(dims), ptr(sp), ptr(out), ptr(ws), c_size(nbytes), stream_ptr()),
          "distance_transform")
    return out


def surface_metrics(mask_a, mask_b, spacing_xyz, maps=False):
    """Overlap and surface distances of two bool/uint8 cuda masks [D,H,W] (medpy's dc / assd / hd95 / hd): returns
    (terms float64[8] = dice, assd, hd95, hd, mean d_AB, mean d_BA, max d_AB, max d_BA;  counts int64[5] = |A|, |B|,
    |A&B|, |dA|, |dB|), and with maps=True also the EDT maps (dist_to_B, dist_to_A) float32 [D,H,W] in mm.  Everything
    stays on the device; nothing synchronises."""
    a, b = _mask_u8(mask_a), _mask_u8(mask_b)
    assert a.shape == b.shape and a.device == b.device, "masks must share one grid"
    terms = torch.empty(8, dtype=torch.float64, device=a.device)
    counts = torch.empty(5, dtype=torch.int64, device=a.device)
    to_b = torch.empty(a.shape, dtype=torch.float32, device=a.device) if maps else None
    to_a = torch.empty(a.shape, dtype=torch.float32, device=a.device) if maps else None
    dims, ws, nbytes = _seg_quality_ws(a.device, a.shape)
    sp = np.asarray(spacing_xyz, dtype=np.float64)
    check(lib.oai_surface_metrics(ptr(a), ptr(b), ptr(dims), ptr(sp), ptr(terms), ptr(counts), ptr(to_b), ptr(to_a),
                                  ptr(ws), c_size(nbytes), stream_ptr()), "surface_metrics")
    return (terms, counts, to_b, to_a) if maps else (terms, counts)


# ------------------------------------------------------------------------------------------------ connected components
def connected_components(mask, connectivity=6):
    """scipy.ndimage.label(mask, generate_binary_structure(3, 1 / 2 / 3)) for connectivity 6 / 18 / 26, bit for bit:
    mask bool/uint8 cuda [D,H,W] -> (labels int32 [D,H,W], sizes int32 [oai_components_max], count int64 scalar).
    sizes[k - 1] is the voxel count of label k; entries past count are zero.  Everything stays on the device; nothing
    synchronises."""
    m = _mask_u8(mask)
    dims = _dims(*m.shape)
    labels = torch.empty(m.shape, dtype=torch.int32, device=m.device)
    sizes = torch.empty(max(int(lib.oai_components_max(ptr(dims), int(connectivity))), 1), dtype=torch.int32,
                        device=m.device)
    count = torch.empty((), dtype=torch.int64, device=m.device)
    nbytes = int(lib.oai_components_workspace_bytes(ptr(dims)))
    ws = _scratch_buf(m.device, "components", nbytes)
    check(lib.oai_connected_components(ptr(m), ptr(dims), int(connectivity), ptr(labels), ptr(sizes), ptr(count),
                                       ptr(ws), c_size(nbytes), stream_ptr()), "connected_components")
    return labels, sizes, count


def keep_components(x, connectivity=6, min_voxels=None):
    """Keep the largest connected component (min_voxels None; the lowest label on a size tie) or every component of at
    least min_voxels voxels.  x: bool/uint8 cuda mask [D,H,W] -> bool mask of the kept voxels; or a float32 cuda
    probability map [D,H,W], whose `> 0.5` mask is labelled -> x itself, zeroed in place outside the kept components.
    No synchronisation."""
    if min_voxels is not None and int(min_voxels) < 0:
        raise ValueError(f"min_voxels must be >= 0 or None, got {min_voxels}")
    mv = -1 if min_voxels is None else int(min_voxels)
    if x.dtype == torch.float32:
        assert x.is_cuda and x.dim() == 3 and x.is_contiguous(), "expected a contiguous float32 cuda [D,H,W]"
        mask, values, keep = x > 0.5, x, None
    else:
        mask, values = x, None
        keep = torch.empty(x.shape, dtype=torch.bool, device=x.device)
    labels, sizes, count = connected_components(mask, connectivity)
    dims = _dims(*labels.shape)
    check(lib.oai_keep_components(ptr(labels), ptr(sizes), ptr(count), ptr(dims), mv,
                                  ptr(None if keep is None else keep.view(torch.uint8)), ptr(values), stream_ptr()),
          "keep_components")
    return x if keep is None else keep


# ------------------------------------------------------------------------------------------------ registration
def _dims(*v):
    return np.asarray(v, dtype=np.int32)


_scratch = {}


def _scratch_buf(device, tag, nbytes):
    """Device scratch for the kernels that need a workspace.  Eager calls share one growing buffer per (device, tag,
    stream); while a CUDA graph is being captured the buffer comes from the graph's own memory pool instead, so replays never
    depend on the shared buffer (which a later, larger eager call may reallocate)."""
    if torch.cuda.is_current_stream_capturing():
        return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)
    key = (device, tag, torch.cuda.current_stream(device).cuda_stream)   # one buffer per stream: no cross-stream reuse
    if key not in _scratch or _scratch[key].numel() < nbytes:
        _scratch[key] = torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)
    return _scratch[key]


def reg_conv3(x, cin, w, bias, out, cout, stride, leaky_in, residual, out_scale=1.0):
    """x / out: views [N, C, D, H, W] float32 whose channel slice may be part of a larger buffer."""
    N, _, D, H, W = x.shape
    dims = _dims(D, H, W)
    need = int(lib.oai_reg_conv3_workspace(cin, cout, ptr(dims), N, stride, int(leaky_in)))
    ws = _scratch_buf(x.device, "conv3", need) if need else None
    check(lib.oai_reg_conv3(ptr(x), c_ll(x.stride(0)), c_ll(x.stride(1)), cin, ptr(dims), ptr(w), ptr(bias),
                            ptr(out), c_ll(out.stride(0)), c_ll(out.stride(1)), cout, w.shape[-1], N, stride,
                            int(leaky_in), int(residual), c_float(out_scale), ptr(ws), c_size(need), stream_ptr()),
          "reg_conv3")
    return out


def reg_convt4(x, cin, w, bias, bn_scale, bn_shift, out, cout, wpk=None, wexp=0, workspace=None):
    N, _, D, H, W = x.shape
    od = _dims(*out.shape[2:])
    if wpk is not None:
        need = int(lib.oai_reg_convt4_mma_workspace(cin, cout, ptr(_dims(D, H, W)), N))
        if workspace is None or workspace.numel() < need:
            workspace = _scratch_buf(x.device, "convt4", need)
        check(lib.oai_reg_convt4_mma(ptr(x), c_ll(x.stride(0)), c_ll(x.stride(1)), cin, ptr(_dims(D, H, W)), ptr(w),
                                     ptr(wpk), wexp, ptr(bias), ptr(bn_scale), ptr(bn_shift), ptr(out),
                                     c_ll(out.stride(0)), c_ll(out.stride(1)), cout, ptr(od), N, ptr(workspace),
                                     c_size(workspace.numel()), stream_ptr()), "reg_convt4_mma")
        return out
    check(lib.oai_reg_convt4(ptr(x), c_ll(x.stride(0)), c_ll(x.stride(1)), cin, ptr(_dims(D, H, W)), ptr(w),
                             ptr(bias), ptr(bn_scale), ptr(bn_shift), ptr(out), c_ll(out.stride(0)),
                             c_ll(out.stride(1)), cout, ptr(od), N, stream_ptr()), "reg_convt4")
    return out


def reg_pack_conv3_umma(w, cin, cout):
    """w: [cin, 27, cout] float32 cuda -> (pre-swizzled weight blocks of the tcgen05 down step, wexp)."""
    wmax = float(w.abs().max())
    wexp = 0 if wmax == 0.0 else max(-14, min(30, int(13 - math.floor(math.log2(wmax)))))
    dst = torch.empty(int(lib.oai_reg_conv3_umma_wbytes(cin, cout)), dtype=torch.uint8, device=w.device)
    check(lib.oai_reg_pack_conv3_umma(ptr(w), cin, cout, w.shape[-1], wexp, ptr(dst), stream_ptr()),
          "reg_pack_conv3_umma")
    return dst, wexp


def reg_conv3_umma(x, cin, wumma, wexp, bias, out, cout):
    """The strided down step (leaky input, avg-pool residual) on tcgen05; x / out are views [N, C, D, H, W]."""
    N, _, D, H, W = x.shape
    need = int(lib.oai_reg_conv3_umma_workspace(cin, ptr(_dims(D, H, W)), N))
    ws = _scratch_buf(x.device, "conv3u", need)
    check(lib.oai_reg_conv3_umma(ptr(x), c_ll(x.stride(0)), c_ll(x.stride(1)), cin, ptr(_dims(D, H, W)), ptr(wumma),
                                 int(wexp), ptr(bias), ptr(out), c_ll(out.stride(0)), c_ll(out.stride(1)), cout, N,
                                 ptr(ws), c_size(ws.numel()), stream_ptr()), "reg_conv3_umma")
    return out


def reg_pack_convt4_umma(w, cin, cout, wexp):
    """w: [cin, 64, cout] float32 cuda -> pre-swizzled weight blocks of the tcgen05 up step (uint8 tensor)."""
    n = int(lib.oai_reg_convt4_umma_wbytes(cin, cout))
    dst = torch.empty(n, dtype=torch.uint8, device=w.device)
    check(lib.oai_reg_pack_convt4_umma(ptr(w), cin, cout, int(wexp), ptr(dst), stream_ptr()), "reg_pack_convt4_umma")
    return dst


def reg_convt4_umma(x, cin, wumma, wexp, bias, bn_scale, bn_shift, out, cout):
    """The up step on tcgen05 (cout in {16, 32, 64}); x / out are views [N, C, D, H, W] as for reg_convt4."""
    N, _, D, H, W = x.shape
    need = N * cin * D * H * W * 4
    ws = _scratch_buf(x.device, "convt4", need)
    check(lib.oai_reg_convt4_umma(ptr(x), c_ll(x.stride(0)), c_ll(x.stride(1)), cin, ptr(_dims(D, H, W)), ptr(wumma),
                                  int(wexp), ptr(bias), ptr(bn_scale), ptr(bn_shift), ptr(out), c_ll(out.stride(0)),
                                  c_ll(out.stride(1)), cout, ptr(_dims(*out.shape[2:])), N, ptr(ws),
                                  c_size(ws.numel()), stream_ptr()), "reg_convt4_umma")
    return out


def reg_pack_convt4(w, cin, cout):
    """w: [cin, 64, cout] float32 cuda -> (wpk uint8 tensor, wexp) for reg_convt4(..., wpk=...)."""
    wmax = float(w.abs().max())
    wexp = 0 if wmax == 0.0 else int(13 - math.floor(math.log2(wmax)))
    wexp = max(-14, min(30, wexp))
    wpk = torch.empty(cin * 64 * cout * 4, dtype=torch.uint8, device=w.device)
    check(lib.oai_reg_pack_convt4(ptr(w), cin, cout, wexp, ptr(wpk), stream_ptr()), "reg_pack_convt4")
    return wpk, wexp


def compose(grid_dims, fields, shortcut_first=False, img=None, want_phi=True, phi_out=None, img_out=None):
    """fields: list of [3,d,h,w] float32 tensors applied in order.  Returns (phi [3,D,H,W] | None, warped | None)."""
    dev = fields[0].device if fields else img.device
    D, H, W = (int(v) for v in grid_dims)
    arr = (ctypes.c_void_p * 4)(*[f.data_ptr() for f in fields] + [0] * (4 - len(fields)))
    fd = np.asarray([s for f in fields for s in f.shape[1:]] + [0] * (12 - 3 * len(fields)), dtype=np.int32)
    for f in fields:
        assert f.is_contiguous() and f.dtype == torch.float32
    if want_phi and phi_out is None:
        phi_out = torch.empty((3, D, H, W), dtype=torch.float32, device=dev)
    if img is not None and img_out is None:
        img_out = torch.empty((D, H, W), dtype=torch.float32, device=dev)
    if img is not None:
        assert img.is_contiguous() and img_out.is_contiguous()
    idims = _dims(*img.shape[-3:]) if img is not None else None
    check(lib.oai_compose(ptr(_dims(D, H, W)), len(fields), arr, ptr(fd), int(shortcut_first), ptr(img), ptr(idims),
                          ptr(phi_out if want_phi else None), ptr(img_out if img is not None else None),
                          stream_ptr()), "compose")
    return (phi_out if want_phi else None), (img_out if img is not None else None)


def resize_trilinear(x, out_dims, out=None):
    if out is None:
        out = torch.empty(tuple(int(v) for v in out_dims), dtype=torch.float32, device=x.device)
    assert x.is_contiguous() and out.is_contiguous()
    check(lib.oai_resize_trilinear(ptr(x), ptr(_dims(*x.shape[-3:])), ptr(out), ptr(_dims(*out.shape[-3:])),
                                   stream_ptr()), "resize_trilinear")
    return out


def avgpool2_ceil(x):
    """x: [C, D, H, W] float32 contiguous."""
    C, D, H, W = x.shape
    out = torch.empty((C, (D + 1) // 2, (H + 1) // 2, (W + 1) // 2), dtype=torch.float32, device=x.device)
    check(lib.oai_avgpool3d_2_ceil(ptr(x), C, ptr(_dims(D, H, W)), ptr(out), stream_ptr()), "avgpool3d_2_ceil")
    return out


def displacement_field(phi):
    _, D, H, W = phi.shape
    out = torch.empty((D, H, W, 3), dtype=torch.float32, device=phi.device)
    check(lib.oai_displacement_field(ptr(phi), ptr(_dims(D, H, W)), ptr(out), stream_ptr()), "displacement_field")
    return out


def _affine(M, t):
    a = np.zeros((3, 4), dtype=np.float64)
    a[:, :3] = M
    a[:, 3] = t
    return np.ascontiguousarray(a)


def warp_volume(src, disp, out_index_to_net, net_to_src_index, out_dims, default_value=0.0, out=None):
    """src: [C, SD, SH, SW] float32; disp: [FD, FH, FW, 3]; affines: (M, t) float64 on x,y,z.  Returns [C, *out_dims]."""
    C = src.shape[0]
    if out is None:
        out = torch.empty((C,) + tuple(int(v) for v in out_dims), dtype=torch.float32, device=src.device)
    assert src.is_contiguous() and disp.is_contiguous() and out.is_contiguous()
    a, b = _affine(*out_index_to_net), _affine(*net_to_src_index)
    check(lib.oai_warp_volume(ptr(src), C, ptr(_dims(*src.shape[1:])), ptr(disp), ptr(_dims(*disp.shape[:3])), ptr(a),
                              ptr(b), ptr(out), ptr(_dims(*out.shape[1:])), c_float(default_value), stream_ptr()),
          "warp_volume")
    return out


def warp_points(pts, disp, phys_to_net, net_to_phys):
    """pts: [n,3] float64 cuda tensor (x,y,z physical).  Returns [n,3] float64."""
    assert pts.dtype == torch.float64 and pts.is_contiguous()
    out = torch.empty_like(pts)
    a, b = _affine(*phys_to_net), _affine(*net_to_phys)
    check(lib.oai_warp_points(ptr(pts), c_ll(pts.shape[0]), ptr(disp), ptr(_dims(*disp.shape[:3])), ptr(a), ptr(b),
                              ptr(out), stream_ptr()), "warp_points")
    return out


def conv3d_igemm_head(src0, wpack, bias, head_w, head_b, out, geom, tile0, crop_zyx, out_mode=0, ab_format=0,
                      flags=0):
    """Last decoder layer (64->64, k3) fused with dc0 + sigmoid + crop-and-place into out [ncls, VD, VH, VW]."""
    NT, D, H, W, c0 = src0.shape
    ncls = head_w.shape[0]
    dims = np.asarray(out.shape[1:], dtype=np.int32)
    crop = np.asarray(crop_zyx, dtype=np.int32)
    check(lib.oai_conv3d_igemm_head(ptr(src0), c0, None, 0, NT, D, H, W, ptr(wpack), c_size(wpack.numel()), ptr(bias),
                                    ab_format, ncls, ptr(head_w), ptr(head_b), ptr(out), ptr(dims), ptr(geom), tile0,
                                    ptr(crop), out_mode, flags, stream_ptr()), "conv3d_igemm_head")
    return out


def pack_convt2_weights(w, D, H, W, ab_format=0, device="cuda"):
    """w: float32 [cout, cin, 2, 2, 2] (conv orientation) of a ConvTranspose3d(k=2, s=2)."""
    w = np.ascontiguousarray(w.detach().cpu().numpy() if hasattr(w, "detach") else w, dtype=np.float32)
    cout, cin = w.shape[:2]
    pl = conv_plan(D, H, W, cin, 0, cout, 2)
    nbytes = pl["nhalf"] * pl["kd_per_block"] * pl["nblk"] * pl["wblock_bytes"]
    dst = np.zeros(nbytes, dtype=np.uint8)
    check(lib.oai_pack_convt2_weights(ptr(w), cout, cin, D, H, W, ab_format, ptr(dst), c_size(nbytes)),
          "pack convt2 weights")
    return torch.from_numpy(dst).to(device)


def convt2_igemm(src, wpack, bias, cout, relu=True, ab_format=0, region=None, out=None):
    """ConvTranspose3d(k=2,s=2): src [NT,D,H,W,cin] act16 -> [NT,2D,2H,2W,cout]; region on the input grid."""
    NT, D, H, W, cin = src.shape
    assert src.is_contiguous()
    if out is None:
        out = torch.empty((NT, 2 * D, 2 * H, 2 * W, cout), dtype=_DT16[ab_format], device=src.device)
    reg = None if region is None else np.asarray(region, dtype=np.int32)
    check(lib.oai_convt2_igemm(ptr(src), cin, NT, D, H, W, ptr(wpack), c_size(wpack.numel()), ptr(bias), cout,
                               int(relu), ab_format, ptr(out), ptr(reg), stream_ptr()), "convt2_igemm")
    return out


def intensity_window(vol, perc_lo=0.1, perc_hi=99.9, out_min=0.0, out_max=1.0, out=None, return_window=False):
    """dask_processing.image_normalize on the device: vol float32 cuda tensor (any shape, contiguous) -> windowed copy
    (or in place with out=vol).  return_window=True also returns (window_min, window_max) (synchronises)."""
    assert vol.dtype == torch.float32 and vol.is_contiguous()
    if out is None:
        out = torch.empty_like(vol)
    nbytes = int(lib.oai_intensity_window_workspace())
    ws = _scratch_buf(vol.device, "window", nbytes)
    check(lib.oai_intensity_window(ptr(vol), c_ll(vol.numel()), ctypes.c_double(perc_lo), ctypes.c_double(perc_hi),
                                   c_float(out_min), c_float(out_max), ptr(out), ptr(ws), c_size(nbytes),
                                   stream_ptr()), "intensity_window")
    if return_window:
        w = (ctypes.c_double * 2)()
        check(lib.oai_intensity_window_result(ptr(ws), w, stream_ptr()), "intensity_window_result")
        return out, (w[0], w[1])
    return out


# ------------------------------------------------------------------------------------------------ iso-surface extraction
def mc_table():
    """The generated marching-cubes polygon table [256, 64, 32] uint8 (host arithmetic in the library)."""
    t = np.zeros((256, 64, 32), dtype=np.uint8)
    check(lib.oai_mc_table(ptr(t), c_size(t.size)), "mc_table")
    return t


def marching_cubes(vol, level=0.5, spacing_xyz=(1.0, 1.0, 1.0), gradient_direction="ascent"):
    """vol: float32 [D,H,W] cuda (z,y,x).  Returns (verts float32 [n,3] (x,y,z) * spacing, faces int32 [m,3]) on the
    device: skimage.measure.marching_cubes(np.swapaxes(vol, 0, 2), level, spacing=spacing_xyz, step_size=1,
    gradient_direction=...)[:2] with one vertex per crossed lattice edge."""
    assert vol.dtype == torch.float32 and vol.is_contiguous() and vol.is_cuda and vol.dim() == 3
    dims = np.asarray(vol.shape, dtype=np.int32)
    nbytes = int(lib.oai_mc_workspace_bytes(ptr(dims)))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=vol.device)
    counts = (c_ll * 2)()
    check(lib.oai_mc_count(ptr(vol), ptr(dims), c_float(level), ptr(ws), c_size(nbytes), counts, stream_ptr()),
          "mc_count")
    nv, nf = int(counts[0]), int(counts[1])
    verts = torch.empty((nv, 3), dtype=torch.float32, device=vol.device)
    faces = torch.empty((nf, 3), dtype=torch.int32, device=vol.device)
    if nv and nf:
        sp = np.asarray(spacing_xyz, dtype=np.float64)
        check(lib.oai_mc_emit(ptr(vol), ptr(dims), c_float(level), ptr(sp), int(gradient_direction == "ascent"),
                              ptr(ws), c_size(nbytes), ptr(verts), ptr(faces), stream_ptr()), "mc_emit")
    return verts, faces


def keep_large_regions(verts, faces, min_cells=3000):
    """get_vtk_mesh's region filter on the device: (verts, faces) of the connected regions with > min_cells faces."""
    nv, nf = int(verts.shape[0]), int(faces.shape[0])
    if nv == 0 or nf == 0:
        return verts[:0], faces[:0]
    assert verts.dtype == torch.float32 and faces.dtype == torch.int32 and verts.is_contiguous() and faces.is_contiguous()
    nbytes = int(lib.oai_mesh_regions_workspace_bytes(c_ll(nv), c_ll(nf)))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=verts.device)
    ov, of = torch.empty_like(verts), torch.empty_like(faces)
    counts = (c_ll * 2)()
    check(lib.oai_mesh_keep_large_regions(ptr(verts), c_ll(nv), ptr(faces), c_ll(nf), int(min_cells), ptr(ws),
                                          c_size(nbytes), ptr(ov), ptr(of), counts, stream_ptr()), "keep_large_regions")
    return ov[:int(counts[0])], of[:int(counts[1])]


# ------------------------------------------------------------------------------------------------ mesh post-processing
def smooth_mesh(verts, faces, iterations=150, relaxation=0.01):
    nv, nf = int(verts.shape[0]), int(faces.shape[0])
    out = torch.empty_like(verts)
    if nv == 0:
        return out
    assert verts.dtype == torch.float32 and faces.dtype == torch.int32 and verts.is_contiguous() and faces.is_contiguous()
    nbytes = int(lib.oai_mesh_smooth_workspace_bytes(c_ll(nv), c_ll(nf)))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=verts.device)
    check(lib.oai_mesh_smooth(ptr(verts), c_ll(nv), ptr(faces), c_ll(nf), int(iterations), c_float(relaxation), ptr(ws),
                              c_size(nbytes), ptr(out), stream_ptr()), "mesh_smooth")
    return out


def face_features(verts, faces):
    nf = int(faces.shape[0])
    normals = torch.empty((nf, 3), dtype=torch.float32, device=verts.device)
    cent = torch.empty((nf, 3), dtype=torch.float32, device=verts.device)
    check(lib.oai_mesh_face_features(ptr(verts), ptr(faces), c_ll(nf), ptr(normals), ptr(cent), stream_ptr()),
          "mesh_face_features")
    return normals, cent


def mesh_distance(points, verts, faces):
    """Unsigned distance of every point [n,3] float32 to the closest point on the triangles of (verts, faces)."""
    n = int(points.shape[0])
    out = torch.empty(n, dtype=torch.float32, device=points.device)
    assert points.is_contiguous() and verts.is_contiguous() and faces.is_contiguous()
    check(lib.oai_mesh_distance(ptr(points), c_ll(n), ptr(verts), ptr(faces), c_ll(int(faces.shape[0])), ptr(out),
                                stream_ptr()), "mesh_distance")
    return out


def kmeans2(features, max_iter=300):
    """labels int32 [n] of a 2-cluster Lloyd KMeans on float32 features [n, dim <= 16]; returns (labels, sweeps)."""
    x = features.contiguous().float()
    n, dim = x.shape
    labels = torch.empty(n, dtype=torch.int32, device=x.device)
    nbytes = int(lib.oai_kmeans2_workspace_bytes(int(dim)))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    it = c_int(0)
    check(lib.oai_kmeans2(ptr(x), c_ll(n), int(dim), int(max_iter), ptr(labels), ptr(ws), c_size(nbytes),
                          ctypes.byref(it), stream_ptr()), "kmeans2")
    return labels, int(it.value)


def map_attributes(source_points, source_attr, target_points, radius=1.0):
    """vtkPointInterpolator(linear kernel, radius) + closest-point null strategy: float32 [n_target(, k)]."""
    sp, tp = source_points.contiguous().float(), target_points.contiguous().float()
    a = source_attr.contiguous().float()
    k = 1 if a.dim() == 1 else int(a.shape[1])
    out = torch.empty((tp.shape[0],) + tuple(a.shape[1:]), dtype=torch.float32, device=tp.device)
    check(lib.oai_mesh_map_attributes(ptr(sp), ptr(a), c_ll(int(sp.shape[0])), k, ptr(tp), c_ll(int(tp.shape[0])),
                                      c_float(float(radius)), ptr(out), stream_ptr()), "mesh_map_attributes")
    return out


def _project_ws(device):
    return torch.empty(int(lib.oai_mesh_project_workspace_bytes()), dtype=torch.uint8, device=device)


def circle_fit(points, coord_x, coord_y, index=None):
    """Least-squares circle through coordinates (coord_x, coord_y) of points [n,3]: ((xc, yc), radius, iterations)."""
    p = points.contiguous().float()
    idx = None if index is None else index.contiguous().to(torch.int32)
    n = int(p.shape[0] if idx is None else idx.shape[0])
    center = (c_double * 2)()
    radius, it = c_double(0.0), c_int(0)
    ws = _project_ws(p.device)
    check(lib.oai_circle_fit(ptr(p), ptr(idx), c_ll(n), int(coord_x), int(coord_y), center, ctypes.byref(radius),
                             ctypes.byref(it), ptr(ws), c_size(ws.numel()), stream_ptr()), "circle_fit")
    return (float(center[0]), float(center[1])), float(radius.value), int(it.value)


def cylinder_project(points, coord_x, coord_y, coord_z, center):
    """(angle, height) float64 [n]: polar angle of (p[coord_x], p[coord_y]) around center, and p[coord_z]."""
    p = points.contiguous().float()
    n = int(p.shape[0])
    angle = torch.empty(n, dtype=torch.float64, device=p.device)
    height = torch.empty(n, dtype=torch.float64, device=p.device)
    check(lib.oai_cylinder_project(ptr(p), c_ll(n), int(coord_x), int(coord_y), int(coord_z), c_double(center[0]),
                                   c_double(center[1]), ptr(angle), ptr(height), stream_ptr()), "cylinder_project")
    return angle, height


def pca2_project(points, index=None, rotate_deg=0.0, mirror_x=False, offset=(0.0, 0.0)):
    """Linear KernelPCA(2) scores of the selected points, rotated / mirrored / offset: (x, y) float64 [n]."""
    p = points.contiguous().float()
    idx = None if index is None else index.contiguous().to(torch.int32)
    n = int(p.shape[0] if idx is None else idx.shape[0])
    ox = torch.empty(n, dtype=torch.float64, device=p.device)
    oy = torch.empty(n, dtype=torch.float64, device=p.device)
    ws = _project_ws(p.device)
    check(lib.oai_pca2_project(ptr(p), ptr(idx), c_ll(n), c_double(float(rotate_deg)), int(bool(mirror_x)),
                               c_double(float(offset[0])), c_double(float(offset[1])), ptr(ox), ptr(oy), ptr(ws),
                               c_size(ws.numel()), stream_ptr()), "pca2_project")
    return ox, oy
