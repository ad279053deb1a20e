"""torch.ops.bpc_b200.* -- the hot path as dispatcher-registered PyTorch operators (the thin C++ extension ``_C``).

``_C.so`` (csrc/torch_ext.cpp) wraps the C ABI of include/bpc_b200.h: each operator validates its tensors with
TORCH_CHECK, allocates outputs and scratch with the caching allocator, takes the current CUDA stream and calls one
``extern "C"`` launcher of libbpc_b200.so.  Registered CUDA + Meta kernels make the operators capturable in CUDA graphs
and visible to FakeTensor / torch.compile tracing.  ``batched`` (ctypes over the same C ABI) and this module are two
doors to the same launchers; there is no CPU kernel behind either (a CPU tensor raises).

    from bpc_baseline_b200 import ops
    idx, n, cost, X, reproj, F = ops.match_triangulate(Ks, RTs, centers, counts, 30.0)
    rois, offs = ops.build_rois(boxes, idx, n, image_of_scene)
    crops, status = ops.roi_crop(images, rois, 224, lut=ops.normalise_lut(images.device), n_rois=offs[-1:])
"""
from __future__ import annotations

import os
from typing import Optional, Sequence

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
EXT_PATH = os.path.join(HERE, '_C.so')
MEAN = (0.485, 0.456, 0.406)
STD = (0.229, 0.224, 0.225)
_loaded = False


def load():
    """Load ``_C.so`` (built in-tree by ``python -m bpc_baseline_b200.build``) and return ``torch.ops.bpc_b200``."""
    global _loaded
    if not _loaded:
        if not os.path.exists(EXT_PATH):
            raise RuntimeError(f'{EXT_PATH} is missing: run `python -m bpc_baseline_b200.build` (there is no fallback)')
        torch.ops.load_library(EXT_PATH)
        if int(torch.ops.bpc_b200.abi_version()) != 2:
            raise RuntimeError('_C.so was built against another ABI version of libbpc_b200.so')
        _loaded = True
    return torch.ops.bpc_b200


def match_triangulate(Ks, RTs, centers, counts, threshold=30.0, reproj_thresh: Optional[float] = None, want_F: bool = False):
    """(idx, n, cost, X, reproj, F) -- PoseEstimator._match for S scenes (process_pose.py:144-188)."""
    import numpy as np
    return load().match_triangulate(Ks, RTs, centers, counts, float(np.float32(threshold)), reproj_thresh, want_F)


def box_centers(boxes):
    return load().box_centers(boxes)


def build_rois(boxes, idx, n, image_of_scene):
    return load().build_rois(boxes, idx, n, image_of_scene)


_LUT: dict = {}


def normalise_lut(device, mean: Sequence[float] = MEAN, std: Sequence[float] = STD):
    import numpy as np
    device = torch.device(device)
    key = (device.index if device.index is not None else torch.cuda.current_device(), tuple(mean), tuple(std))
    if key not in _LUT:
        _LUT[key] = load().normalise_lut([float(np.float32(v)) for v in mean], [float(np.float32(v)) for v in std],
                                         torch.device('cuda', key[0]))
    return _LUT[key]


def roi_crop(images, rois, T: int = 256, fill=(255, 255, 255), swap_rb: bool = True, lut=None, n_rois=None, roi_first: int = 0, out=None):
    """(crops f32 [R,3,T,T], status i32 [R]) -- data_utils.py:34-44 + process_pose.py:199-209."""
    if lut is None:
        lut = normalise_lut(images.device)
    return load().roi_crop(images, rois, int(T), [int(v) for v in fill], bool(swap_rb), lut, n_rois, int(roi_first), out)


def roi_crop_u8(images, rois, T: int = 256, fill=(255, 255, 255), n_rois=None, roi_first: int = 0):
    return load().roi_crop_u8(images, rois, int(T), [int(v) for v in fill], n_rois, int(roi_first))


def roi_crop_bf16(images, rois, T: int = 256, fill=(255, 255, 255), swap_rb: bool = True, lut=None, n_rois=None, roi_first: int = 0):
    """(bfloat16 [R,3,T,T] in channels_last memory format, status): roi_crop's values rounded to bfloat16 (bpc_roi_crop_bf16)."""
    if lut is None:
        lut = normalise_lut(images.device)
    return load().roi_crop_bf16(images, rois, int(T), [int(v) for v in fill], bool(swap_rb), lut, n_rois, int(roi_first))


def color_jitter(canvases, order, factors, swap_rb: bool = False, lut=None):
    """f32 [n,3,T,T]: torchvision ColorJitter (draws of utils.data_utils.draw_color_jitter) + to_tensor + normalize on uint8
    canvases [n,T,T,3], bit-exact (bpc_color_jitter)."""
    if lut is None:
        lut = normalise_lut(canvases.device)
    return load().color_jitter(canvases, order, factors, bool(swap_rb), lut)


def pack_records(idx, n, cost, X, reproj, scene_offset, offset_div: int = 3):
    return load().pack_records(idx, n, cost, X, reproj, scene_offset, int(offset_div))


def fundamental(Ks, RTs):
    return load().fundamental(Ks, RTs)
