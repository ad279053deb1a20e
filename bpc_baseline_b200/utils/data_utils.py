"""CUDA counterpart of the hot-path helpers of bpc/utils/data_utils.py (same names and arguments)."""
from __future__ import annotations

import glob
import json
import os

import numpy as np

from .. import _host, batched
from ..inference.utils.camera_utils import load_camera_params


def _resize_error(msg):
    try:
        import cv2
        return cv2.error(msg)
    except Exception:                                    # cv2 is not a dependency of this package
        return ValueError(msg)


def letterbox_preserving_aspect_ratio(img, target_size=256, fill_color=(255, 255, 255)):
    """Aspect-preserving INTER_AREA resize onto a fill_color canvas -- reference data_utils.py:34-44.

    Returns (canvas uint8 [T, T, 3], scale, dx, dy) exactly as the reference; the resize runs on the GPU
    and is bit-identical to cv2.resize(..., interpolation=cv2.INTER_AREA).
    """
    img = np.asarray(img)
    h, w = img.shape[:2]
    scale = float(target_size) / max(h, w)                # ZeroDivisionError on an empty crop, as the reference
    new_w = int(round(w * scale))
    new_h = int(round(h * scale))
    dx = (target_size - new_w) // 2
    dy = (target_size - new_h) // 2
    if img.ndim != 3 or img.shape[2] != 3 or img.dtype != np.uint8:
        raise TypeError('img must be an H x W x 3 uint8 array')
    if new_w < 1 or new_h < 1:
        raise _resize_error("OpenCV(-215:Assertion failed) !dsize.empty() in function 'resize'")
    if not 1 <= int(target_size) <= batched.MAX_TARGET:
        raise NotImplementedError(f'target_size above {batched.MAX_TARGET} is not supported by the CUDA crop kernels')
    images = _host.to_dev(img[None], np.uint8)
    rois = _host.to_dev([[0, 0, 0, w, h]], np.int32)
    import torch
    status = torch.zeros(1, dtype=torch.int32, device=images.device)
    canvas = batched.roi_crop_u8(images, rois, T=int(target_size), fill=fill_color, status=status)
    if int(status.item()):                                  # e.g. wider than BPC_MAX_ROI_WIDTH: an error, never a blank canvas
        raise _resize_error(f'crop of {w} x {h} pixels was rejected by the CUDA crop kernels (wider than {batched.MAX_ROI_WIDTH}?)')
    return _host.to_host(canvas)[0].copy(), scale, dx, dy


def calc_pose_matrix(R_mat, t):
    """4x4 float64 pose from R, t -- reference data_utils.py:383-387 (a container, no arithmetic)."""
    pose = np.eye(4)
    pose[:3, :3] = R_mat
    pose[:3, 3] = t
    return pose


def _read_json(path):
    with open(path) as fh:
        return json.load(fh)


def load_gt_poses(scene_dir, scene_id, cam_ids, image_id, obj_id):
    """4x4 ground-truth poses of object ``obj_id`` in image ``image_id`` of the FIRST camera only, or [] when the
    scene_gt / scene_gt_info files or the image entry are missing -- behaviour of reference data_utils.py:355-380."""
    cam = list(cam_ids)[0] if len(cam_ids) else None
    if cam is None:
        return []
    base = os.path.join(scene_dir, scene_id)
    gt_file, info_file = (os.path.join(base, f"{stem}_{cam}.json") for stem in ("scene_gt", "scene_gt_info"))
    if not (os.path.exists(gt_file) and os.path.exists(info_file)):
        return []
    gt, info = _read_json(gt_file), _read_json(info_file)
    key = str(image_id)
    if key not in gt or key not in info:
        return []
    entries = gt[key][:len(info[key])]                      # the reference zips the two lists
    return [calc_pose_matrix(np.asarray(e["cam_R_m2c"], dtype=np.float32).reshape(3, 3),
                             np.asarray(e["cam_t_m2c"], dtype=np.float32))
            for e in entries if e["obj_id"] == obj_id]


class Capture:
    """Images + intrinsics + extrinsics of one multi-camera capture -- reference data_utils.py:390-409."""

    def __init__(self, images, Ks, RTs, obj_id, gt_poses=None):
        self.images = images
        self.Ks = Ks
        self.RTs = RTs
        self.obj_id = obj_id
        if gt_poses:
            self.gt_poses = np.linalg.inv(RTs[0]) @ gt_poses

    @classmethod
    def from_dir(cls, scene_dir, cam_ids, image_id, obj_id):
        """Read one capture from a BOP scene directory (reference data_utils.py:399-409): intrinsics / extrinsics from
        scene_camera_<cam>.json, the image ``rgb_<cam>/<image_id:06d>.{png,jpg}`` per camera, RT as float64 4x4."""
        import cv2                                        # image decoding only (host I/O)
        cams = load_camera_params(scene_dir, cam_ids)
        Ks = [cams[c]['K'][image_id] for c in cam_ids]
        RTs = [calc_pose_matrix(cams[c]['R'][image_id], cams[c]['t'][image_id]) for c in cam_ids]
        images = []
        for c in cam_ids:
            hits = glob.glob(os.path.join(scene_dir, f"rgb_{c}", f"{image_id:06d}.*g"))
            images.append(cv2.imread(hits[0]))
        return cls(images, Ks, RTs, obj_id, load_gt_poses(scene_dir, '', cam_ids, image_id, obj_id))


class SceneBatch:
    """Device-resident captures of S scenes x C cameras -- the matcher's and the crop kernels' input layout.

    ``Ks`` float32 [S, C, 3, 3], ``RTs`` float64 [S, C, 4, 4], ``images`` uint8 [S * C, H, W, 3] BGR (image of scene s, camera
    c at index s * C + c), all CUDA tensors; ``decoders`` names what decoded each image file."""

    def __init__(self, Ks, RTs, images, decoders):
        self.Ks, self.RTs, self.images, self.decoders = Ks, RTs, images, decoders

    def capture(self, s, obj_id=None):
        """Scene ``s`` as a host-side :class:`Capture` (a device -> host copy; for the single-scene drop-ins and tests)."""
        C = self.Ks.shape[1]
        return Capture([im for im in _host.to_host(self.images[s * C:(s + 1) * C])], [k for k in _host.to_host(self.Ks[s])],
                       [rt for rt in _host.to_host(self.RTs[s])], obj_id)


def load_scene_batch(scene_dirs, cam_ids, image_ids, decode='cv2'):
    """Batched BOP loader: ``Capture.from_dir`` (reference data_utils.py:399-409) and ``load_camera_params``
    (camera_utils.py:6-20) for S (scene_dir, image_id) pairs at once, landing in HBM as the tensors the batched API takes.

    * intrinsics / extrinsics: ``scene_camera_<cam>.json`` is parsed once per directory; K, R, t are float32 as the reference
      loads them, and RT is the float64 4x4 of ``calc_pose_matrix`` (:383-387) holding those float32-rounded values;
      both are assembled in pinned host memory and copied with one asynchronous H2D each;
    * images ``rgb_<cam>/<image_id:06d>.{png,jpg}``: ``decode='cv2'`` (default) decodes on the host exactly as the reference
      does (``cv2.imread``, BGR) into a two-slot pinned staging buffer and overlaps each slot's asynchronous H2D with the next
      file's decode; ``decode='nvjpeg'`` sends JPEG files through nvJPEG (``torchvision.io.decode_jpeg(device='cuda')``, library
      code) straight to HBM and reorders RGB planes to BGR pixels on the device -- its IDCT is not bit-identical to libjpeg's,
      so the pixels can differ from ``cv2.imread`` by one grey level; PNG (lossless) always takes the cv2 path.

    Returns a :class:`SceneBatch`.  All images must share one size (one camera model per batch, as in BOP)."""
    import cv2
    import torch
    scene_dirs, image_ids, cam_ids = list(scene_dirs), [int(i) for i in image_ids], list(cam_ids)
    if len(scene_dirs) != len(image_ids):
        raise ValueError('scene_dirs and image_ids must have one entry per scene')
    if decode not in ('cv2', 'nvjpeg'):
        raise ValueError("decode must be 'cv2' or 'nvjpeg'")
    dev = _host.device()
    S, C = len(scene_dirs), len(cam_ids)
    Ks_h = torch.empty((S, C, 3, 3), dtype=torch.float32).pin_memory()
    RTs_h = torch.empty((S, C, 4, 4), dtype=torch.float64).pin_memory()
    Ks_n, RTs_n = Ks_h.numpy(), RTs_h.numpy()
    params = {}
    for s, (d, i) in enumerate(zip(scene_dirs, image_ids)):
        if d not in params:
            params[d] = load_camera_params(d, cam_ids)
        for c, cam in enumerate(cam_ids):
            Ks_n[s, c] = params[d][cam]['K'][i]
            RTs_n[s, c] = calc_pose_matrix(params[d][cam]['R'][i], params[d][cam]['t'][i])      # float32 -> float64 widening
    Ks = Ks_h.to(dev, non_blocking=True)
    RTs = RTs_h.to(dev, non_blocking=True)

    files = []
    for d, i in zip(scene_dirs, image_ids):
        for cam in cam_ids:
            hits = sorted(glob.glob(os.path.join(d, f"rgb_{cam}", f"{i:06d}.*g")))
            if not hits:
                raise FileNotFoundError(os.path.join(d, f"rgb_{cam}", f"{i:06d}.*g"))
            files.append(hits[0])
    images, stage, events, decoders = None, None, [None, None], []
    for n, path in enumerate(files):
        if decode == 'nvjpeg' and path.lower().endswith(('.jpg', '.jpeg')):
            from torchvision.io import ImageReadMode, decode_jpeg, read_file
            rgb = decode_jpeg(read_file(path), mode=ImageReadMode.RGB, device=dev)              # [3, H, W] in HBM
            if images is None:
                images = torch.empty((len(files), rgb.shape[1], rgb.shape[2], 3), dtype=torch.uint8, device=dev)
            if tuple(rgb.shape[1:]) != tuple(images.shape[1:3]):
                raise ValueError(f'{path}: image size differs from the first image of the batch')
            images[n].copy_(rgb.flip(0).permute(1, 2, 0))
            decoders.append('nvjpeg')
            continue
        img = cv2.imread(path)
        if img is None:
            raise IOError(f'cannot decode {path}')
        if images is None:
            images = torch.empty((len(files),) + img.shape, dtype=torch.uint8, device=dev)
        if img.shape != tuple(images.shape[1:]):
            raise ValueError(f'{path}: image size differs from the first image of the batch')
        if stage is None:
            stage = torch.empty((2,) + img.shape, dtype=torch.uint8).pin_memory()
        k = n & 1
        if events[k] is not None:
            events[k].synchronize()                         # the slot's previous upload has left pinned memory
        np.copyto(stage[k].numpy(), img)
        images[n].copy_(stage[k], non_blocking=True)
        events[k] = torch.cuda.Event()
        events[k].record()
        decoders.append('cv2+pinned')
    torch.cuda.current_stream().synchronize()               # pinned staging goes out of scope below
    return SceneBatch(Ks, RTs, images, decoders)


def draw_crop_jitter(bbox_visib, rnd=None):
    """The three draws BOPSingleObjDataset.__getitem__ makes per sample, in its order (data_utils.py:257-263):
    ``scale_factor = 1.0 + 0.2 * random.random()``, then ``randint`` for shift_x and shift_y within +-int(0.1 * side).
    ``rnd`` defaults to Python's global ``random`` module, so seeding it reproduces the reference's boxes.
    Returns (scale float64 [n], shift int32 [n, 2])."""
    import random
    rnd = random if rnd is None else rnd
    boxes = np.asarray(bbox_visib).reshape(-1, 4)
    scale = np.empty(len(boxes), np.float64)
    shift = np.empty((len(boxes), 2), np.int32)
    for r, (_, _, w, h) in enumerate(boxes):
        scale[r] = 1.0 + 0.2 * rnd.random()
        max_x, max_y = int(0.1 * int(w)), int(0.1 * int(h))
        shift[r] = (rnd.randint(-max_x, max_x), rnd.randint(-max_y, max_y))
    return scale, shift


def draw_color_jitter(n, brightness=None, contrast=None, saturation=None, hue=None):
    """The draws ``torchvision.transforms.ColorJitter(brightness, contrast, saturation, hue)`` makes for n samples, in its
    order: per sample ``ColorJitter.get_params`` (``torch.randperm(4)``, then one float32 ``uniform_`` per enabled op), so
    seeding torch's global RNG reproduces the per-sample transform.  The ranges are normalised by ColorJitter's own
    argument checks (None = the op is off).  Returns (order int32 [n, 4] = op ids in application order with disabled ops
    as -1, factors float32 [n, 4] = (brightness, contrast, saturation, hue), NaN where an op is off) for
    :func:`batched.color_jitter` or ``dataset_crops(color_jitter=...)``."""
    from torchvision.transforms import ColorJitter
    cj = ColorJitter(brightness=0 if brightness is None else brightness, contrast=0 if contrast is None else contrast,
                     saturation=0 if saturation is None else saturation, hue=0 if hue is None else hue)
    order = np.empty((int(n), 4), np.int32)
    factors = np.empty((int(n), 4), np.float32)
    for r in range(int(n)):
        fn_idx, *fac = ColorJitter.get_params(cj.brightness, cj.contrast, cj.saturation, cj.hue)
        order[r] = [int(k) if fac[int(k)] is not None else -1 for k in fn_idx]
        factors[r] = [np.nan if f is None else f for f in fac]
    return order, factors


def dataset_crops(images, bbox_visib, image_index=None, target_size=256, jitter=None, as_uint8=False, color_jitter=None):
    """Batched crop transform of BOPSingleObjDataset.__getitem__ (data_utils.py:243-252, 282; jittered window :257-271).

    ``images`` uint8 [B, H, W, 3] BGR (NumPy or CUDA tensor), ``bbox_visib`` int [n, 4] = (x, y, w, h), ``jitter`` =
    None for the original crop or the (scale, shift) pair of :func:`draw_crop_jitter` for the augmented window.
    Returns the normalised float32 [n, 3, T, T] CUDA tensor in the dataset's channel order (BGR kept, no swap), or the
    uint8 letterboxed images [n, T, T, 3] with ``as_uint8``.  ``color_jitter`` = the (order, factors) pair of
    :func:`draw_color_jitter` (NumPy arrays, or int32 / float32 CUDA tensors taken as they are): the canvases go through
    torchvision's ColorJitter (on ``Image.fromarray(canvas)``, bit-exact) before to_tensor + normalize; it cannot be
    combined with ``as_uint8``.  Raises RuntimeError on an empty crop, as the reference (:247-248, :269-270).
    """
    import torch
    if color_jitter is not None and as_uint8:
        raise ValueError('color_jitter produces the normalised float32 tensor; it cannot be combined with as_uint8')
    imgs = images if isinstance(images, torch.Tensor) else _host.to_dev(images, np.uint8)
    _, H, W, _ = imgs.shape
    xywh = _host.to_dev(np.asarray(bbox_visib).reshape(-1, 4), np.int32)
    idx = None if image_index is None else _host.to_dev(image_index, np.int32)
    scale = shift = None
    if jitter is not None:
        scale, shift = _host.to_dev(jitter[0], np.float64), _host.to_dev(jitter[1], np.int32)
    rois = batched.train_rois(xywh, W, H, image=idx, scale=scale, shift=shift)
    status = torch.zeros(rois.shape[0], dtype=torch.int32, device=rois.device)
    if as_uint8 or color_jitter is not None:
        out = batched.roi_crop_u8(imgs, rois, T=int(target_size), status=status)
    else:
        out = batched.roi_crop(imgs, rois, T=int(target_size), swap_rb=False, status=status)
    if int(status.sum().item()):
        raise RuntimeError('Empty crop for %s image' % ('augmented' if jitter is not None else 'original'))
    if color_jitter is not None:
        order, factors = (d if isinstance(d, torch.Tensor) and d.is_cuda else _host.to_dev(d, dt)
                          for d, dt in zip(color_jitter, (np.int32, np.float32)))
        out = batched.color_jitter(out, order, factors, swap_rb=False)
    return out
