"""Drop-in for oai_analysis/segmentation/segmenter.py on B200.

Same class names, constructor (`mode`, `config` dict with the keys of analysis_object.py:18-26) and
`segment(image, if_output_prob_map=False, if_output_itk=True) -> (FC, TC)` contract.  The whole prediction
(tile gather, 18 conv layers, sigmoid, assembly) runs on the GPU through the C ABI; the host only moves the input
volume in and the two class maps out.
"""
import json
from abc import ABC, abstractmethod

import numpy as np
import torch

from .. import itk_compat, ops
from .image_transforms import Partition
from .networks import get_network
from .utils import initialize_model


def load_json_to_dict(json_file):
    """segmenter.py:14-17 (ParameterDict.load_JSON(...).ext): the training config is a plain JSON object."""
    with open(json_file) as f:
        return json.load(f)


class Segmenter(ABC):
    @abstractmethod
    def __init__(self, *args, **kwargs):
        self.model = None
        self.config = None

    @abstractmethod
    def segment(self, *args, **kwargs):
        pass


class Segmenter3DInPatch(Segmenter):
    def __init__(self, mode=None, config=None):
        super().__init__()
        self.config = config
        self.ready = False

    def pred_setup(self):
        """segmenter.py:51-62.  Optional config key "keep_largest_component": 6, 18 or 26 makes segment_device zero
        each class map outside the largest connected component (with that connectivity) of its > 0.5 mask; absent or
        falsy leaves the output as the reference computes it."""
        keep = self.config.get("keep_largest_component")
        if keep and (isinstance(keep, bool) or keep not in (6, 18, 26)):
            raise ValueError(f"keep_largest_component must be 6, 18 or 26 (a connectivity), got {keep!r}")
        self.keep_largest = int(keep) if keep else None
        training_config = load_json_to_dict(self.config["training_config_file"])
        self.partition = Partition(training_config["patch_size"], self.config["overlap_size"],
                                   padding_mode="reflect", mode="pred")
        self.model = get_network(training_config["model"])(**training_config["model_setting"])
        self.device = torch.device(self.config["device"])
        initialize_model(self.model, ckpoint_path=self.config["ckpoint_path"])
        self.model.to(self.device)
        self.model.eval()
        self.ready = True

    def segment(self, image):
        pass


class Segmenter3DInPatchClassWise(Segmenter3DInPatch):
    def __init__(self, mode=None, config=None):
        super().__init__(mode, config)

    def segment_device(self, volume, if_output_prob_map=False, tiles_per_batch=None, out=None):
        """volume: float32 [D,H,W] tensor already on the device.  Returns float32 [n_classes, D, H, W] on the device
        (class 0 = FC, class 1 = TC), i.e. segmenter.py:105-129 without the host round trips: one oai_seg_forward."""
        if not self.ready:
            self.pred_setup()
        part = self.partition.plan(volume.shape)   # validates the geometry exactly like the reference's Partition
        handle = self.model.seg_handle(self.partition.tile_size[::-1], self.config["overlap_size"])
        # the reference batches config['batch_size'] tiles per forward (results do not depend on it: BN is in eval
        # mode); here the whole tile set is one batch unless the workspace would not fit the free device memory
        if tiles_per_batch is None:
            tiles_per_batch = self.config.get("tiles_per_batch") or handle.auto_tiles_per_batch(volume.shape)
        out = handle.forward(volume, out_mode=0 if if_output_prob_map else 1, tiles_per_batch=tiles_per_batch,
                             out=out)
        if self.keep_largest:
            for c in range(out.shape[0]):
                ops.keep_components(out[c], self.keep_largest)
        return out

    def segment(self, image, if_output_prob_map=False, if_output_itk=True):
        if not self.ready:
            self.pred_setup()
        vol = itk_compat.to_device_f32(image, self.device, "seg_in")
        out = self.segment_device(vol, if_output_prob_map, self.config.get("tiles_per_batch"))
        # D2H through a cached pinned buffer, then the float64 the reference assembles into (np.zeros default, :493)
        # with torch's multi-threaded cast (a pageable .cpu() plus numpy's astype cost ~4x more per knee)
        key = (tuple(out.shape), out.dtype)
        if getattr(self, "_pin_key", None) != key:
            self._pin, self._pin_key = torch.empty(out.shape, dtype=out.dtype, pin_memory=True), key
        self._pin.copy_(out, non_blocking=True)
        torch.cuda.current_stream(out.device).synchronize()
        host = self._pin.to(torch.float64).numpy()
        if self.model._fmt() == 0 and ops.conv_overflow_count(reset=True):
            raise FloatingPointError("segmentation activations left the fp16 range (|x| > 65504) with this checkpoint; "
                                     "set model.precision = 'bf16' (UNet.precision / OAI_B200_SEG_PRECISION)")
        fc, tc = host[0], host[1]
        if if_output_itk:
            return itk_compat.image_from_array(fc, like=image), itk_compat.image_from_array(tc, like=image)
        return fc, tc
