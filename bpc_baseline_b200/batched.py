"""Batched, device-resident API over the C ABI (include/bpc_b200.h).

torch is used for device memory and streams only; every computation is a kernel of
libbpc_b200.so launched on torch's current stream.  All inputs must be contiguous CUDA tensors of
the documented dtype; nothing here falls back to the CPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib

MEAN = (0.485, 0.456, 0.406)   # process_pose.py:208
STD = (0.229, 0.224, 0.225)    # process_pose.py:209


def _chk(t: torch.Tensor, dtype, name: str, ndim: Optional[int] = None):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f'{name}: expected a torch.Tensor, got {type(t).__name__}')
    if not t.is_cuda:
        raise RuntimeError(f'{name}: must be a CUDA tensor (no CPU fallback)')
    if t.dtype != dtype:
        raise RuntimeError(f'{name}: dtype {t.dtype}, expected {dtype}')
    if not t.is_contiguous():
        raise RuntimeError(f'{name}: must be contiguous')
    if ndim is not None and t.dim() != ndim:
        raise RuntimeError(f'{name}: {t.dim()} dims, expected {ndim}')
    return t


def _chk_device(t: torch.Tensor, dev: torch.device, name: str):
    if t.device != dev:
        raise RuntimeError(f'{name}: on {t.device}, but the kernel runs on {dev}')
    return t


def _chk_lut(lut: torch.Tensor, dev: torch.device):
    """The kernels read all 3 x 256 entries of the table from the device they run on."""
    _chk(lut, torch.float32, 'lut', 2)
    if tuple(lut.shape) != (3, 256):
        raise RuntimeError(f'lut: shape {tuple(lut.shape)}, expected (3, 256)')
    return _chk_device(lut, dev, 'lut')


def _p(t: Optional[torch.Tensor]):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream(dev) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


@dataclass
class MatchResult:
    """Output of match_triangulate; rows of a scene are sorted by (cost, r) as process_pose.py:183."""
    idx: torch.Tensor      # i32 [S, Kmax, 3]  (i, j, k), -1 padded
    n: torch.Tensor        # i32 [S]           matches per scene (-1: infeasible costs, SciPy would raise)
    cost: torch.Tensor     # f32 [S, Kmax]
    X: torch.Tensor        # f64 [S, Kmax, 3]
    reproj: Optional[torch.Tensor]   # f64 [S, Kmax, 3]
    F: Optional[torch.Tensor]        # f64 [S, 3, 3, 3]


def fundamental(Ks: torch.Tensor, RTs: torch.Tensor) -> torch.Tensor:
    """F12, F13, F23 per scene: f64 [S,3,3,3] (camera_utils.py:23-46 via process_pose.py:154-159)."""
    _chk(Ks, torch.float32, 'Ks', 4); _chk(RTs, torch.float64, 'RTs', 4)
    S = Ks.shape[0]
    if tuple(Ks.shape[1:]) != (3, 3, 3) or tuple(RTs.shape) != (S, 3, 4, 4):
        raise RuntimeError('Ks must be [S,3,3,3] and RTs [S,3,4,4]')
    F = torch.empty((S, 3, 3, 3), dtype=torch.float64, device=Ks.device)
    with torch.cuda.device(Ks.device):
        _lib.check(_lib.load().bpc_fundamental(_p(Ks), _p(RTs), S, _p(F), _stream(Ks.device)), 'bpc_fundamental')
    return F


def detections_from_yolo(xyxy: torch.Tensor, conf: torch.Tensor, cls: torch.Tensor, nraw: torch.Tensor,
                         conf_thresh: float, Dmax: int):
    """Detector outputs -> the matcher's detection tensors (process_pose.py:123-141), all on the device.

    xyxy f32 [S,3,Nraw,4], conf / cls f32 [S,3,Nraw], nraw i32 [S,3] -> (boxes i32 [S,3,Dmax,4],
    centers f64 [S,3,Dmax,2], counts i32 [S,3]); counts above Dmax mean detections were dropped.
    """
    _chk(xyxy, torch.float32, 'xyxy', 4); _chk(conf, torch.float32, 'conf', 3); _chk(cls, torch.float32, 'cls', 3)
    _chk(nraw, torch.int32, 'nraw', 2)
    S, C, N, _ = xyxy.shape
    if xyxy.shape[3] != 4 or tuple(conf.shape) != (S, C, N) or tuple(cls.shape) != (S, C, N) or tuple(nraw.shape) != (S, C):
        raise RuntimeError('expected xyxy [S,C,Nraw,4], conf / cls [S,C,Nraw], nraw [S,C]')
    dev = xyxy.device
    boxes = torch.zeros((S, C, Dmax, 4), dtype=torch.int32, device=dev)
    centers = torch.zeros((S, C, Dmax, 2), dtype=torch.float64, device=dev)
    counts = torch.empty((S, C), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().bpc_detections_from_yolo(_p(xyxy), _p(conf), _p(cls), _p(nraw), S * C, N,
                                                        float(np.float32(conf_thresh)), int(Dmax), _p(boxes), _p(centers),
                                                        _p(counts), _stream(dev)), 'bpc_detections_from_yolo')
    return boxes, centers, counts


def box_centers(boxes: torch.Tensor) -> torch.Tensor:
    """centres f64 [..., 2] from int32 boxes [..., 4] (process_pose.py:134-136)."""
    _chk(boxes, torch.int32, 'boxes')
    if boxes.shape[-1] != 4:
        raise RuntimeError('boxes must end in a dimension of 4')
    out = torch.empty((*boxes.shape[:-1], 2), dtype=torch.float64, device=boxes.device)
    with torch.cuda.device(boxes.device):
        _lib.check(_lib.load().bpc_box_centers(_p(boxes), boxes.numel() // 4, _p(out), _stream(boxes.device)), 'bpc_box_centers')
    return out


def cost_tensor(F: torch.Tensor, centers: torch.Tensor, counts: torch.Tensor) -> torch.Tensor:
    """Materialised cost f32 [S,Dmax,Dmax,Dmax] (epipolar_matching.py:83-98); entries beyond (N,M,P) are NaN."""
    _chk(F, torch.float64, 'F', 4); _chk(centers, torch.float64, 'centers', 4); _chk(counts, torch.int32, 'counts', 2)
    S, _, D, _ = centers.shape
    if tuple(F.shape) != (S, 3, 3, 3) or tuple(centers.shape) != (S, 3, D, 2) or tuple(counts.shape) != (S, 3):
        raise RuntimeError('shape mismatch between F, centers and counts')
    cost = torch.full((S, D, D, D), float('nan'), dtype=torch.float32, device=F.device)
    with torch.cuda.device(F.device):
        _lib.check(_lib.load().bpc_cost_tensor(_p(F), _p(centers), _p(counts), S, D, _p(cost), _stream(F.device)), 'bpc_cost_tensor')
    return cost


def match_objects(cost: torch.Tensor, threshold) -> tuple[torch.Tensor, torch.Tensor]:
    """LSAP + threshold on explicit cost f32 [S,N,M,P] -> (idx i32 [S,Kmax,3] ascending r, n i32 [S])."""
    _chk(cost, torch.float32, 'cost', 4)
    S, N, M, P = cost.shape
    if N == 0 or M == 0 or P == 0:
        raise RuntimeError('cost tensor has an empty dimension')
    kmax = min(N * M, P)
    idx = torch.empty((S, kmax, 3), dtype=torch.int32, device=cost.device)
    n = torch.empty((S,), dtype=torch.int32, device=cost.device)
    with torch.cuda.device(cost.device):
        _lib.check(_lib.load().bpc_match_objects(_p(cost), S, N, M, P, float(np.float32(threshold)), _p(idx), _p(n),
                                                 _stream(cost.device)), 'bpc_match_objects')
    return idx, n


_MATCH_WS: dict = {}


def _match_workspace(dev, S: int, D: int) -> Optional[torch.Tensor]:
    """Scratch for scenes too large for shared memory (Dmax above ~450); None below that.  Cached per (device, stream)."""
    need = int(_lib.load().bpc_match_workspace_bytes(int(S), int(D)))
    if need == 0:
        return None
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), int(torch.cuda.current_stream(dev).cuda_stream))
    ws = _MATCH_WS.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.empty((need,), dtype=torch.uint8, device=dev)
        _MATCH_WS[key] = ws
    return ws


def match_triangulate(Ks: torch.Tensor, RTs: torch.Tensor, centers: torch.Tensor, counts: torch.Tensor,
                      threshold=30, want_reproj: bool = True, want_F: bool = False,
                      reproj_thresh: Optional[float] = None) -> MatchResult:
    """PoseEstimator._match (process_pose.py:144-188) for S scenes in one launch.

    ``reproj_thresh`` (pixels, default None = the reference's behaviour): drop every match whose reprojection error
    (utils/triangulation.py:14-18) exceeds it in any view; the survivors keep their order.  The test is ``error >
    reproj_thresh``: an error equal to the threshold is kept, and so is a NaN error (NaN never exceeds it), e.g. a view
    whose projection of X has w = 0 and a zero numerator.  ``n`` is negative for a
    scene SciPy would reject (-1) or whose counts exceed Dmax (-2): see :func:`check_match_status`."""
    _chk(Ks, torch.float32, 'Ks', 4); _chk(RTs, torch.float64, 'RTs', 4)
    _chk(centers, torch.float64, 'centers', 4); _chk(counts, torch.int32, 'counts', 2)
    S, _, D, _ = centers.shape
    if tuple(Ks.shape) != (S, 3, 3, 3) or tuple(RTs.shape) != (S, 3, 4, 4) or tuple(centers.shape) != (S, 3, D, 2) \
            or tuple(counts.shape) != (S, 3):
        raise RuntimeError('expected Ks [S,3,3,3], RTs [S,3,4,4], centers [S,3,Dmax,2], counts [S,3]')
    dev = Ks.device
    idx = torch.empty((S, D, 3), dtype=torch.int32, device=dev)
    n = torch.empty((S,), dtype=torch.int32, device=dev)
    cost = torch.empty((S, D), dtype=torch.float32, device=dev)
    X = torch.empty((S, D, 3), dtype=torch.float64, device=dev)
    reproj = torch.empty((S, D, 3), dtype=torch.float64, device=dev) if (want_reproj or reproj_thresh is not None) else None
    F = torch.empty((S, 3, 3, 3), dtype=torch.float64, device=dev) if want_F else None
    with torch.cuda.device(dev):
        ws = _match_workspace(dev, S, D)
        _lib.check(_lib.load().bpc_match_triangulate(
            _p(Ks), _p(RTs), _p(centers), _p(counts), S, D, float(np.float32(threshold)),
            int(reproj_thresh is not None), float(reproj_thresh) if reproj_thresh is not None else 0.0,
            _p(idx), _p(n), _p(cost), _p(X), _p(reproj), _p(F), _p(ws), ws.numel() if ws is not None else 0, _stream(dev)),
            'bpc_match_triangulate')
    return MatchResult(idx, n, cost, X, reproj, F)


N_INFEASIBLE, N_OVERFLOW = -1, -2        # BPC_N_INFEASIBLE, BPC_N_OVERFLOW


def check_match_status(n: torch.Tensor) -> None:
    """Raise for the per-scene status values of ``MatchResult.n`` (synchronises): ValueError where SciPy raises, RuntimeError
    where a camera's count exceeds Dmax (e.g. the overflow count of :func:`detections_from_yolo`)."""
    lo = int(n.min().item()) if n.numel() else 0
    if lo == N_OVERFLOW:
        bad = torch.nonzero(n == N_OVERFLOW).flatten()[:8].tolist()
        raise RuntimeError(f'detection counts exceed Dmax in scenes {bad}: raise Dmax (detections were truncated)')
    if lo < 0:
        raise ValueError('matrix contains invalid numeric entries')


def pack_records(res: MatchResult, scene_offset: Optional[torch.Tensor] = None, offset_div: int = 3,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The valid matches of every scene as compact 64-byte pose records in one uint8 buffer (see bpc_pack_records in
    bpc_b200.h): header | n[S] | records (idx i32 x3, cost f32, X f64 x3, reproj f64 x3).  ``scene_offset`` = the
    exclusive prefix sum from :func:`build_rois` (``offset_div`` 3); computed here if absent."""
    S, K, _ = res.idx.shape
    dev = res.idx.device
    if scene_offset is None:
        scene_offset = torch.zeros((S + 1,), dtype=torch.int32, device=dev)
        scene_offset[1:] = torch.cumsum(res.n.clamp(min=0), 0).to(torch.int32)
        offset_div = 1
    _chk(scene_offset, torch.int32, 'scene_offset', 1)
    nbytes = int(_lib.load().bpc_pack_records_bytes(S, K))
    if out is None:
        out = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    else:
        _chk(out, torch.uint8, 'out', 1)
        if out.numel() < nbytes:
            raise RuntimeError(f'out must hold {nbytes} bytes')
    with torch.cuda.device(dev):
        _lib.check(_lib.load().bpc_pack_records(_p(res.idx), _p(res.n), _p(res.cost), _p(res.X), _p(res.reproj), _p(scene_offset),
                                                int(offset_div), S, K, _p(out), _stream(dev)), 'bpc_pack_records')
    return out


def triangulate(P: torch.Tensor, pts: torch.Tensor) -> torch.Tensor:
    """DLT for n matches: P f64 [n,3,3,4], pts f64 [n,3,2] -> X f64 [n,3] (epipolar_matching.py:118-127)."""
    _chk(P, torch.float64, 'P', 4); _chk(pts, torch.float64, 'pts', 3)
    n = P.shape[0]
    if tuple(P.shape) != (n, 3, 3, 4) or tuple(pts.shape) != (n, 3, 2):
        raise RuntimeError('expected P [n,3,3,4] and pts [n,3,2]')
    X = torch.empty((n, 3), dtype=torch.float64, device=P.device)
    with torch.cuda.device(P.device):
        _lib.check(_lib.load().bpc_triangulate(_p(P), _p(pts), n, _p(X), _stream(P.device)), 'bpc_triangulate')
    return X


def reprojection_error(P: torch.Tensor, X: torch.Tensor, pts: torch.Tensor) -> torch.Tensor:
    """Per-view pixel error f64 [n,3] (utils/triangulation.py:14-18)."""
    _chk(P, torch.float64, 'P', 4); _chk(X, torch.float64, 'X', 2); _chk(pts, torch.float64, 'pts', 3)
    n = P.shape[0]
    if tuple(P.shape) != (n, 3, 3, 4) or tuple(X.shape) != (n, 3) or tuple(pts.shape) != (n, 3, 2):
        raise RuntimeError('expected P [n,3,3,4], X [n,3] and pts [n,3,2]')
    err = torch.empty((n, 3), dtype=torch.float64, device=P.device)
    with torch.cuda.device(P.device):
        _lib.check(_lib.load().bpc_reprojection_error(_p(P), _p(X), _p(pts), n, _p(err), _stream(P.device)), 'bpc_reprojection_error')
    return err


def projection(K: torch.Tensor, RT: torch.Tensor) -> torch.Tensor:
    """P = K (f32 [n,3,3]) @ RT[:3] (f64 [n,4,4]) -> f64 [n,3,4] (process_pose.py:88-92)."""
    _chk(K, torch.float32, 'K', 3); _chk(RT, torch.float64, 'RT', 3)
    n = K.shape[0]
    if tuple(K.shape) != (n, 3, 3) or tuple(RT.shape) != (n, 4, 4):
        raise RuntimeError('expected K [n,3,3] and RT [n,4,4]')
    P = torch.empty((n, 3, 4), dtype=torch.float64, device=K.device)
    with torch.cuda.device(K.device):
        _lib.check(_lib.load().bpc_projection(_p(K), _p(RT), n, _p(P), _stream(K.device)), 'bpc_projection')
    return P


def epipolar_error(F: torch.Tensor, pt1: torch.Tensor, pt2: torch.Tensor) -> torch.Tensor:
    """epipolar_error for n (pt1, pt2, F) triples: F f64 [n,3,3], pt f64 [n,2] -> f64 [n] (epipolar_matching.py:5-28)."""
    _chk(F, torch.float64, 'F', 3); _chk(pt1, torch.float64, 'pt1', 2); _chk(pt2, torch.float64, 'pt2', 2)
    n = F.shape[0]
    if tuple(F.shape) != (n, 3, 3) or tuple(pt1.shape) != (n, 2) or tuple(pt2.shape) != (n, 2):
        raise RuntimeError('expected F [n,3,3], pt1 [n,2], pt2 [n,2]')
    e = torch.empty((n,), dtype=torch.float64, device=F.device)
    with torch.cuda.device(F.device):
        _lib.check(_lib.load().bpc_epipolar_error(_p(F), _p(pt1), _p(pt2), n, _p(e), _stream(F.device)), 'bpc_epipolar_error')
    return e


def epipolar_error_full(F: torch.Tensor, pts: torch.Tensor) -> torch.Tensor:
    """(e12 + e13 + e23) / 3 for n triples: F f64 [n,3,3,3], pts f64 [n,3,2] -> f64 [n] (epipolar_matching.py:73-81)."""
    _chk(F, torch.float64, 'F', 4); _chk(pts, torch.float64, 'pts', 3)
    n = F.shape[0]
    if tuple(F.shape) != (n, 3, 3, 3) or tuple(pts.shape) != (n, 3, 2):
        raise RuntimeError('expected F [n,3,3,3] and pts [n,3,2]')
    e = torch.empty((n,), dtype=torch.float64, device=F.device)
    with torch.cuda.device(F.device):
        _lib.check(_lib.load().bpc_epipolar_error_full(_p(F), _p(pts), n, _p(e), _stream(F.device)), 'bpc_epipolar_error_full')
    return e


def triangulate_views(P: torch.Tensor, pts: torch.Tensor) -> torch.Tensor:
    """DLT with V views (2..8): P f64 [n,V,3,4], pts f64 [n,V,2] -> X f64 [n,3] (epipolar_matching.py:118-127)."""
    _chk(P, torch.float64, 'P', 4); _chk(pts, torch.float64, 'pts', 3)
    n, V = P.shape[0], P.shape[1]
    if tuple(P.shape) != (n, V, 3, 4) or tuple(pts.shape) != (n, V, 2) or not 2 <= V <= 8:
        raise RuntimeError('expected P [n,V,3,4] and pts [n,V,2] with 2 <= V <= 8')
    X = torch.empty((n, 3), dtype=torch.float64, device=P.device)
    with torch.cuda.device(P.device):
        _lib.check(_lib.load().bpc_triangulate_views(_p(P), _p(pts), n, V, _p(X), _stream(P.device)), 'bpc_triangulate_views')
    return X


def build_rois(boxes: torch.Tensor, idx: torch.Tensor, n: torch.Tensor, image_of_scene: torch.Tensor,
               rois: Optional[torch.Tensor] = None) -> tuple[torch.Tensor, torch.Tensor]:
    """(rois i32 [S*Kmax*3, 5], scene_offset i32 [S+1]); 3 ROIs per match in (scene, match, view) order.

    scene_offset[S] (device) is the number of valid ROIs; rows beyond it are unspecified.
    """
    _chk(boxes, torch.int32, 'boxes', 4); _chk(idx, torch.int32, 'idx', 3); _chk(n, torch.int32, 'n', 1)
    _chk(image_of_scene, torch.int32, 'image_of_scene', 2)
    S, _, D, _ = boxes.shape
    K = idx.shape[1]
    dev = boxes.device
    if rois is None:
        rois = torch.empty((S * K * 3, 5), dtype=torch.int32, device=dev)
    else:
        _chk(rois, torch.int32, 'rois', 2)
        if rois.shape[0] < S * K * 3 or rois.shape[1] != 5:
            raise RuntimeError('rois must be int32 [>= S*Kmax*3, 5]')
    offs = torch.empty((S + 1,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().bpc_build_rois(_p(boxes), _p(idx), _p(n), _p(image_of_scene), S, D, K, _p(offs), _p(rois),
                                              _stream(dev)), 'bpc_build_rois')
    return rois, offs


_LUT_CACHE: dict = {}


def normalise_lut(device, mean: Sequence[float] = MEAN, std: Sequence[float] = STD) -> torch.Tensor:
    """f32 [3,256] table: lut[c][v] = (v/255 - mean[c]) / std[c] in float32 (process_pose.py:207-209)."""
    device = torch.device(device)
    key = (device.index if device.index is not None else torch.cuda.current_device(), tuple(mean), tuple(std))
    if key not in _LUT_CACHE:
        lut = torch.empty((3, 256), dtype=torch.float32, device=device)
        m = (C.c_float * 3)(*[float(np.float32(v)) for v in mean])
        s = (C.c_float * 3)(*[float(np.float32(v)) for v in std])
        with torch.cuda.device(device):
            _lib.check(_lib.load().bpc_normalise_lut(m, s, _p(lut), _stream(device)), 'bpc_normalise_lut')
        _LUT_CACHE[key] = lut
    return _LUT_CACHE[key]


_WS_CACHE: dict = {}
MAX_ROIS_PER_LAUNCH = 32768
MAX_TARGET = 1024              # BPC_MAX_TARGET
MAX_ROI_WIDTH = 8192           # BPC_MAX_ROI_WIDTH


def _crop_workspace(dev, R: int, T: int) -> torch.Tensor:
    """Device scratch for the crop kernels, cached per (device, stream) and grown on demand.

    Keyed by the current stream as well: two streams cropping concurrently must not share tap descriptors."""
    need = int(_lib.load().bpc_roi_crop_workspace_bytes(int(R), int(T)))
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), int(torch.cuda.current_stream(dev).cuda_stream))
    ws = _WS_CACHE.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.empty((max(need, 1 << 16),), dtype=torch.uint8, device=dev)
        _WS_CACHE[key] = ws
    return ws


def _chk_status(status, R: int) -> None:
    if status is not None:
        _chk(status, torch.int32, 'status', 1)
        if status.shape[0] < R:
            raise RuntimeError('status must hold one int32 per ROI')


def _crop_args(images, rois, T, fill):
    _chk(images, torch.uint8, 'images', 4); _chk(rois, torch.int32, 'rois', 2)
    B, H, W, ch = images.shape
    if ch != 3 or rois.shape[1] != 5:
        raise RuntimeError('images must be [B,H,W,3] and rois [R,5]')
    if not 1 <= int(T) <= MAX_TARGET:
        raise RuntimeError(f'target size must be in 1..{MAX_TARGET}')
    f = (C.c_uint8 * 3)(*[int(v) for v in fill])
    return B, H, W, rois.shape[0], f


def roi_crop(images: torch.Tensor, rois: torch.Tensor, T: int = 256, fill=(255, 255, 255), swap_rb: bool = True,
             lut: Optional[torch.Tensor] = None, n_rois: Optional[torch.Tensor] = None, roi_first: int = 0,
             out: Optional[torch.Tensor] = None, status: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Network inputs f32 [R,3,T,T] for R ROIs (data_utils.py:34-44 + process_pose.py:199-209).

    ``n_rois``: optional device int32 scalar tensor holding the number of valid ROIs of the whole batch;
    record r is processed iff ``roi_first + r < n_rois`` (skipped rows of ``out`` are left untouched), so
    a long ROI list can be processed chunk by chunk into one reusable ``out`` buffer.  ``status``: optional int32 [R], 1 where an ROI was rejected.
    """
    B, H, W, R, f = _crop_args(images, rois, T, fill)
    dev = images.device
    if lut is None:
        lut = normalise_lut(dev)
    _chk_lut(lut, dev)
    if out is None:
        out = torch.empty((R, 3, T, T), dtype=torch.float32, device=dev)
    else:
        _chk(out, torch.float32, 'out', 4)
        if out.shape[0] < R or tuple(out.shape[1:]) != (3, T, T):
            raise RuntimeError('out must be [>=R,3,T,T]')
        _chk_device(out, dev, 'out')
    _chk_status(status, R)
    if n_rois is not None:
        _chk(n_rois, torch.int32, 'n_rois')
    ws = _crop_workspace(dev, min(R, MAX_ROIS_PER_LAUNCH), T)
    with torch.cuda.device(dev):
        for lo in range(0, R, MAX_ROIS_PER_LAUNCH):          # bounds the scratch (8.3 KB of tap descriptors per ROI)
            r = min(MAX_ROIS_PER_LAUNCH, R - lo)
            _lib.check(_lib.load().bpc_roi_crop(_p(images), B, H, W, _p(rois[lo:lo + r]), r, _p(n_rois), int(roi_first) + lo, int(T),
                                                f, int(bool(swap_rb)), _p(lut), _p(out[lo:lo + r]),
                                                _p(status[lo:lo + r]) if status is not None else None,
                                                _p(ws), ws.numel(), _stream(dev)), 'bpc_roi_crop')
    return out


def roi_crop_bf16(images: torch.Tensor, rois: torch.Tensor, T: int = 256, fill=(255, 255, 255), swap_rb: bool = True,
                  lut: Optional[torch.Tensor] = None, n_rois: Optional[torch.Tensor] = None, roi_first: int = 0,
                  out: Optional[torch.Tensor] = None, status: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Network inputs as a bfloat16 tensor of logical shape [R,3,T,T] in ``torch.channels_last`` memory format (memory
    [R,T,T,3]): :func:`roi_crop`'s float32 values rounded to bfloat16 -- what a bf16 tensor-core pose head reads, at half the
    output bytes and without a layout pass.  ``out``: a bfloat16 [>=R,3,T,T] tensor that is channels_last-contiguous.
    Raises for image pools the 2-D TMA path cannot take (row pitch not a multiple of 16 bytes, T > 256): use roi_crop there."""
    B, H, W, R, f = _crop_args(images, rois, T, fill)
    dev = images.device
    if lut is None:
        lut = normalise_lut(dev)
    _chk_lut(lut, dev)
    if out is None:
        out = torch.empty((R, 3, T, T), dtype=torch.bfloat16, device=dev, memory_format=torch.channels_last)
    else:
        if out.dtype != torch.bfloat16 or not out.is_cuda or out.dim() != 4 or out.shape[0] < R or tuple(out.shape[1:]) != (3, T, T) \
                or not out.is_contiguous(memory_format=torch.channels_last):
            raise RuntimeError('out must be a channels_last bfloat16 CUDA tensor [>=R,3,T,T]')
        _chk_device(out, dev, 'out')
    _chk_status(status, R)
    if n_rois is not None:
        _chk(n_rois, torch.int32, 'n_rois')
    ws = _crop_workspace(dev, min(R, MAX_ROIS_PER_LAUNCH), T)
    with torch.cuda.device(dev):
        for lo in range(0, R, MAX_ROIS_PER_LAUNCH):
            r = min(MAX_ROIS_PER_LAUNCH, R - lo)
            _lib.check(_lib.load().bpc_roi_crop_bf16(_p(images), B, H, W, _p(rois[lo:lo + r]), r, _p(n_rois), int(roi_first) + lo, int(T),
                                                     f, int(bool(swap_rb)), _p(lut), out[lo:lo + r].data_ptr(),
                                                     _p(status[lo:lo + r]) if status is not None else None,
                                                     _p(ws), ws.numel(), _stream(dev)), 'bpc_roi_crop_bf16')
    return out


def roi_crop_u8(images: torch.Tensor, rois: torch.Tensor, T: int = 256, fill=(255, 255, 255),
                   n_rois: Optional[torch.Tensor] = None, roi_first: int = 0, out: Optional[torch.Tensor] = None,
                status: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Letterboxed uint8 crops [R,T,T,3] in source channel order (data_utils.py:34-44)."""
    B, H, W, R, f = _crop_args(images, rois, T, fill)
    dev = images.device
    if out is None:
        out = torch.empty((R, T, T, 3), dtype=torch.uint8, device=dev)
    else:
        _chk(out, torch.uint8, 'out', 4)
        if out.shape[0] < R or tuple(out.shape[1:]) != (T, T, 3):
            raise RuntimeError('out must be uint8 [>=R,T,T,3]')
        _chk_device(out, dev, 'out')
    _chk_status(status, R)
    if n_rois is not None:
        _chk(n_rois, torch.int32, 'n_rois')
    ws = _crop_workspace(dev, min(R, MAX_ROIS_PER_LAUNCH), T)
    with torch.cuda.device(dev):
        for lo in range(0, R, MAX_ROIS_PER_LAUNCH):
            r = min(MAX_ROIS_PER_LAUNCH, R - lo)
            _lib.check(_lib.load().bpc_roi_crop_u8(_p(images), B, H, W, _p(rois[lo:lo + r]), r, _p(n_rois), int(roi_first) + lo, int(T),
                                                   f, _p(out[lo:lo + r]), _p(status[lo:lo + r]) if status is not None else None,
                                                   _p(ws), ws.numel(), _stream(dev)), 'bpc_roi_crop_u8')
    return out


def crops_normalise(sources: Sequence[torch.Tensor], T: int, swap_rb: bool = True, lut: Optional[torch.Tensor] = None,
                    out: Optional[torch.Tensor] = None, device=None) -> torch.Tensor:
    """uint8 letterboxed crops -> f32 [sum(n_s),3,T,T]: BGR2RGB + to_tensor + normalize (process_pose.py:206-209).

    ``sources`` are uint8 [n_s,T,T,3] tensors (the output of :func:`roi_crop_u8`), concatenated in order.  They may
    alias PEER memory (another rank's buffer obtained through ``distributed.PeerBuffers``); the kernel then pulls
    the bytes over NVLink while it converts.  Bit-identical to :func:`roi_crop` on the same ROIs.
    """
    if not 1 <= len(sources) <= 16:
        raise RuntimeError('1..16 sources')
    for s in sources:
        _chk(s, torch.uint8, 'sources[*]', 4)
        if tuple(s.shape[1:]) != (T, T, 3):
            raise RuntimeError('every source must be uint8 [n,T,T,3]')
    dev = torch.device(device) if device is not None else sources[0].device
    if dev.type == 'cuda' and dev.index is None:
        dev = torch.device('cuda', torch.cuda.current_device())
    if lut is None:
        lut = normalise_lut(dev)
    _chk_lut(lut, dev)
    total = sum(int(s.shape[0]) for s in sources)
    if out is None:
        out = torch.empty((total, 3, T, T), dtype=torch.float32, device=dev)
    else:
        _chk(out, torch.float32, 'out', 4)
        if out.shape[0] < total or tuple(out.shape[1:]) != (3, T, T):
            raise RuntimeError('out must be [>=sum(n_s),3,T,T]')
        _chk_device(out, dev, 'out')
    ptrs = (C.c_void_p * len(sources))(*[s.data_ptr() if s.shape[0] else None for s in sources])
    counts = (C.c_int32 * len(sources))(*[int(s.shape[0]) for s in sources])
    with torch.cuda.device(dev):
        _lib.check(_lib.load().bpc_crops_normalise(ptrs, counts, len(sources), int(T), int(bool(swap_rb)), _p(lut), _p(out),
                                                   _stream(dev)), 'bpc_crops_normalise')
    return out


def color_jitter(canvases: torch.Tensor, order: torch.Tensor, factors: torch.Tensor, swap_rb: bool = False,
                 lut: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """torchvision ColorJitter on ``Image.fromarray(canvas)`` + to_tensor + normalize, bit-exact, for n canvases at once.

    ``canvases`` uint8 [n,T,T,3] (e.g. :func:`roi_crop_u8`; channel 0 is treated as PIL's R), ``order`` i32 [n,4] and
    ``factors`` f32 [n,4] as drawn by ``utils.data_utils.draw_color_jitter``.  Returns f32 [n,3,T,T]; ``swap_rb`` and
    ``lut`` as :func:`roi_crop` (the training dataset keeps the stored order: ``swap_rb=False``)."""
    _chk(canvases, torch.uint8, 'canvases', 4); _chk(order, torch.int32, 'order', 2); _chk(factors, torch.float32, 'factors', 2)
    n, T = canvases.shape[0], canvases.shape[1]
    if tuple(canvases.shape[1:]) != (T, T, 3) or tuple(order.shape) != (n, 4) or tuple(factors.shape) != (n, 4):
        raise RuntimeError('expected canvases [n,T,T,3], order [n,4] and factors [n,4]')
    if not 1 <= T <= MAX_TARGET:
        raise RuntimeError(f'target size must be in 1..{MAX_TARGET}')
    dev = canvases.device
    if order.device != dev or factors.device != dev:
        raise RuntimeError('canvases, order and factors must be on the same device')
    if lut is None:
        lut = normalise_lut(dev)
    _chk_lut(lut, dev)
    if out is None:
        out = torch.empty((n, 3, T, T), dtype=torch.float32, device=dev)
    else:
        _chk(out, torch.float32, 'out', 4)
        if out.shape[0] < n or tuple(out.shape[1:]) != (3, T, T):
            raise RuntimeError('out must be [>=n,3,T,T]')
        _chk_device(out, dev, 'out')
    with torch.cuda.device(dev):
        _lib.check(_lib.load().bpc_color_jitter(_p(canvases), n, T, _p(order), _p(factors), int(bool(swap_rb)), _p(lut), _p(out),
                                                _stream(dev)), 'bpc_color_jitter')
    return out


def train_rois(xywh: torch.Tensor, W: int, H: int, image: Optional[torch.Tensor] = None, scale: Optional[torch.Tensor] = None,
               shift: Optional[torch.Tensor] = None) -> torch.Tensor:
    """ROI records i32 [n,5] of the dataset's crops (data_utils.py:243-271): the original window, or with ``scale``
    (f64 [n]) / ``shift`` (i32 [n,2]) the jittered one.  Feed to :func:`roi_crop` with ``swap_rb=False``."""
    _chk(xywh, torch.int32, 'xywh', 2)
    n = xywh.shape[0]
    if xywh.shape[1] != 4:
        raise RuntimeError('xywh must be [n,4]')
    if image is not None:
        _chk(image, torch.int32, 'image', 1)
    if scale is not None:
        _chk(scale, torch.float64, 'scale', 1)
    if shift is not None:
        _chk(shift, torch.int32, 'shift', 2)
        if scale is None:
            raise RuntimeError('shift needs scale (the reference draws both, data_utils.py:257-263)')
    for t, name in ((image, 'image'), (scale, 'scale'), (shift, 'shift')):
        if t is not None and t.shape[0] != n:
            raise RuntimeError(f'{name}: first dimension must be {n}')
    dev = xywh.device
    rois = torch.empty((n, 5), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().bpc_train_rois(_p(xywh), _p(image), _p(scale), _p(shift), n, int(W), int(H), _p(rois),
                                              _stream(dev)), 'bpc_train_rois')
    return rois
