"""Every compiled variant of the ROI-crop kernels against cv2, with non-white fills, arbitrary LUTs and odd target sizes.

Which kernel and which template instantiation crops a ROI is decided at run time (``launch_crop`` in csrc/crop.cu,
``crop_cta_launch`` in csrc/crop_cta.cu) from the pool width W, the target size T, the output type and ``swap_rb``:

    aligned = 3 W % 16 == 0 and 3 W >= 576                      (2-D tensor-map staging possible)
    use_cta = aligned and T <= 256 and 3 W >= cta_pitch_max(T)   (cta_pitch_max(224) = 1408, (256) = 1600)
    TT      = T if T in (224, 256) else 0                        (compile-time target size of the float kernels)

    classes 0 / 1 / 3 / 4 (rejected, area < 2, grow, area 2..5)   class 2 (integer ratio >= 2, or scale > 5)
    use_cta: bpc_crop_cta_kernel                                  bpc_crop_generic_kernel<NTH>,
      f32   <TT, swap>         TT in {224, 256, 0}                  NTH = 256 if 32 ceil(T / 32) <= 256 else 1024,
      bf16  <0, swap>                                               for u8, f32 and (NTH = 256 only) bf16
      u8    <0>
    else:    bpc_crop_warp_kernel
      f32   <TT, aligned, swap>
      u8    <0, aligned>
      bf16  refused (BPC_EUNSUPPORTED)

That is 9 CTA, 14 warp and 5 generic instantiations (``generic<bf16, 1024>`` is compiled but cannot run: bf16 needs
T <= 256).  ``TABLE`` lists the cells (kernel, instantiation, class) they make: 4 classes on the CTA and warp kernels,
class 2 on the generic one.  ``crop_plan`` / ``roi_class`` restate the dispatch and the prep kernel's classification
(``bpc_crop_prep_kernel``) in Python.  After every launch the tests read what the prep kernel actually did from the crop
workspace (class of every ROI, list lengths and work counters of the kernels that ran) and check it against the
restatement; ``test_every_cell_of_the_table_is_reached`` then asserts that the matrix reached every cell, so a change
of the dispatch fails here instead of quietly dropping coverage.

Outputs are compared bit for bit: uint8 with cv2 on a ``np.full(fill)`` canvas (``oracle.crop.letterbox_ref``), float32
with ``lut[p][canvas[..., 2 - p if swap else p]]`` of that canvas, bfloat16 with the same rounded by torch.  Fills are
asymmetric as well as white, and a random LUT of 768 distinct finite values (one +0.0, one -0.0) makes every output value
name its plane, source channel and byte.
"""
import functools
import math

import numpy as np
import pytest
import torch

from oracle import crop as ocrop
from tests.gpu_util import to_dev

TMAP_MAX_PITCH = 576
CTA_MAX_T = 256
MAX_ROI_WIDTH = 8192
GEOM_BYTES = 88                  # sizeof(RoiGeom); cls is the int32 at byte 68
FILLS = ((255, 255, 255), (0, 128, 255), (7, 200, 31))


# ----------------------------------------------------------------------------------------------------------------------
# restatement of the dispatch (csrc/crop.cu launch_crop, csrc/crop_cta.cu crop_cta_launch) and of the prep rules
# ----------------------------------------------------------------------------------------------------------------------
def desc_stride(T):
    return (T + 31) & ~31


def ydesc_stride(T):
    base, rows4 = desc_stride(T) + 8, (5 * T + 33) // 2
    return rows4 if (T <= 256 and rows4 > base) else base


def cta_pitch_max(T):
    return ((15 + 3 * (2 * T - 1) + 12 + 63) >> 6) << 6


def ws_off_count(R, T):
    """Byte offset of the 16 launch counters in the crop workspace (geom | xdesc | ydesc | counters | lists)."""
    off_x = (R * GEOM_BYTES + 15) & ~15
    return off_x + R * desc_stride(T) * 16 + R * ydesc_stride(T) * 16


def pool_flags(W, T):
    aligned = (3 * W) % 16 == 0 and 3 * W >= TMAP_MAX_PITCH
    return aligned, aligned and T <= CTA_MAX_T and 3 * W >= cta_pitch_max(T)


def crop_plan(W, T, out_type, swap):
    """{class: (kernel, instantiation)} of one launch, or None where the call is refused (bf16 off the CTA path)."""
    aligned, use_cta = pool_flags(W, T)
    sw = 'swap' if swap else 'keep'
    tt = T if T in (224, 256) else 0
    if out_type == 'bf16' and not use_cta:
        return None
    if use_cta:
        fast = ('cta', {'f32': f'f32<{tt},{sw}>', 'bf16': f'bf16<0,{sw}>', 'u8': 'u8<0>'}[out_type])
    else:
        al = 'aligned' if aligned else 'unaligned'
        fast = ('warp', f'f32<{tt},{al},{sw}>' if out_type == 'f32' else f'u8<0,{al}>')
    nth = 256 if (T + 31) // 32 * 32 <= 256 else 1024
    return {0: fast, 1: fast, 3: fast, 4: fast, 2: ('generic', f'{out_type}<{nth}>')}


def _table():
    cells = set()
    for sw in ('swap', 'keep'):
        for tt in (224, 256, 0):
            cells |= {('cta', f'f32<{tt},{sw}>', c) for c in (0, 1, 3, 4)}
            for al in ('aligned', 'unaligned'):
                cells |= {('warp', f'f32<{tt},{al},{sw}>', c) for c in (0, 1, 3, 4)}
        cells |= {('cta', f'bf16<0,{sw}>', c) for c in (0, 1, 3, 4)}
    cells |= {('cta', 'u8<0>', c) for c in (0, 1, 3, 4)}
    cells |= {('warp', f'u8<0,{al}>', c) for al in ('aligned', 'unaligned') for c in (0, 1, 3, 4)}
    cells |= {('generic', f'{o}<{n}>', 2) for o, n in (('u8', 256), ('f32', 256), ('bf16', 256), ('u8', 1024), ('f32', 1024))}
    return frozenset(cells)


TABLE = _table()


def _area_taps(d, scale, ssize):
    """(start, n) of computeResizeAreaTab for destination index d (area_taps in crop_common.cuh, float64)."""
    fsx1 = d * scale
    fsx2 = fsx1 + scale
    sx1, sx2 = math.ceil(fsx1), min(math.floor(fsx2), ssize - 1)
    sx1 = min(sx1, sx2)
    start, n = sx1, sx2 - sx1
    if sx1 - fsx1 > 1e-3:
        start, n = sx1 - 1, n + 1
    if fsx2 - sx2 > 1e-3:
        n += 1
    return start, n


def _records_bad(h, new_h, scale_y, cap, maxtaps):
    """src_row_records refuses the per-source-row form (the ROI then takes the generic kernel)."""
    if h + 8 > cap:
        return True
    prev_last = -1
    for d in range(new_h):
        ys, yn = _area_taps(d, scale_y, h)
        if yn < 1 or yn > maxtaps or ys < prev_last or ys + yn > h or (ys == prev_last and yn == 1):
            return True
        prev_last = ys + yn - 1
    return False


def roi_class(w, h, T, use_cta, aligned):
    """Class bpc_crop_prep_kernel gives a w x h box (crop.cu:103-137 plus the record check of classes 1 and 4):
    0 rejected, 1 area with scale < 2 (or exactly 1), 3 grow, 4 area with 4..6 taps, 2 the generic kernel."""
    if w <= 0 or h <= 0 or w > MAX_ROI_WIDTH:
        return 0
    scale = T / max(h, w)
    new_w, new_h = round(w * scale), round(h * scale)           # Python round: half to even, as the reference
    if not (1 <= new_w <= T and 1 <= new_h <= T):
        return 0
    sx, sy = 1.0 / (new_w / w), 1.0 / (new_h / h)
    if sx >= 1.0 and sy >= 1.0:
        isx, isy = round(sx), round(sy)
        regime = 2 if abs(sx - isx) < 2.220446049250313e-16 and abs(sy - isy) < 2.220446049250313e-16 else 1
    else:
        regime = 3
    if (regime == 1 and sx < 2.0 and sy < 2.0) or (regime == 2 and isx == 1 and isy == 1):
        cls = 1
    elif regime == 3:
        cls = 3
    elif regime == 1:
        seg_px = int(31.0 * sx) + math.ceil(sx) + 3
        pitch_max = ((3 * seg_px + 46) >> 4) << 4
        taps6 = math.ceil(sx) + 1 <= 6 and math.ceil(sy) + 1 <= 6
        cls = 4 if taps6 and (use_cta or pitch_max <= TMAP_MAX_PITCH) else 2
    else:
        cls = 2
    if cls == 4 and use_cta and _records_bad(h, new_h, sy, 2 * ydesc_stride(T), 6):
        cls = 2
    if cls == 1 and aligned and _records_bad(h, new_h, sy, 2 * desc_stride(T) + 16, 3):
        cls = 2
    return cls


def box_class(box, B, H, W, T):
    img, x1, y1, x2, y2 = (int(v) for v in box)
    if not (0 <= img < B and x1 >= 0 and y1 >= 0 and x2 <= W and y2 <= H):
        return 0
    aligned, use_cta = pool_flags(W, T)
    return roi_class(x2 - x1, y2 - y1, T, use_cta, aligned)


# ----------------------------------------------------------------------------------------------------------------------
# the matrix: pools whose width selects each instantiation, boxes of every class
# ----------------------------------------------------------------------------------------------------------------------
TS = (1, 2, 3, 31, 33, 97, 100, 224, 255, 256, 257)
MATRIX = (
    [(1920, T) for T in TS]                                         # CTA (T <= 256), aligned warp at T = 257
    + [(1918, T) for T in TS]                                       # unaligned warp (pitch 5754)
    + [(448, 224), (448, 256), (512, 256), (320, 160), (192, 97)]   # aligned warp: 16-byte pitch below cta_pitch_max(T)
    + [(1913, 224), (1913, 33)]                                     # unaligned warp, another misalignment step
    + [(176, 3), (176, 33), (176, 224), (176, 256)]                 # 528-byte pitch: a multiple of 16, below 576
)
POOL_H, POOL_B = 1400, 2


def matrix_boxes(W, H, B, T, seed):
    """ROIs of classes 0..4 for a pool: landscape and portrait (borders on all four sides), scale exactly 1, squares and
    the whole image (no border), letterbox rounding ties (k + 0.5: Python rounds them half to even, some reject the
    crop), the bottom-right corner of the last image, and rejected boxes."""
    rng = np.random.default_rng(seed)
    sizes = []
    for lo, hi in ((0.3, 0.95), (1.05, 1.95), (2.1, 2.9), (3.1, 4.9), (5.2, 6.0)):     # 3, 1, 4, 4, 2
        for _ in range(2):
            L = max(1, int(rng.uniform(lo, hi) * T))
            s = int(rng.integers(max(1, L // 4), L + 1))
            sizes += [(L, s), (s, L)]
    sizes += [(T, max(1, T // 2)), (max(1, T // 3), T), (2 * T, 2 * T), (3 * T, T), (T, 2 * T), (max(1, T - 1), max(1, T - 1))]
    sizes += [(2, 1), (1, 2), (6, 3), (3, 6), (14, 7), (5, 10), (1, 1), (3, 1)]
    rois = []
    for w, h in sizes:
        w, h = min(w, W), min(h, H)
        x1, y1 = int(rng.integers(0, W - w + 1)), int(rng.integers(0, H - h + 1))
        rois.append((int(rng.integers(0, B)), x1, y1, x1 + w, y1 + h))
    rois += [(B - 1, 0, 0, W, H), (B - 1, W - min(W, T + 5), H - min(H, 2 * T + 3), W, H),
             (B - 1, W - min(W, 3 * T // 2 + 1), H - min(H, T + 1), W, H)]
    rois += [(0, 5, 5, 5, 40), (0, W - 3, 0, W + 1, 10), (B, 0, 0, 8, 8), (0, 0, 0, W, 1), (-1, 0, 0, 4, 4)]
    return np.asarray(rois, np.int32)


def random_lut(seed=1234):
    """768 distinct finite float32 values, +0.0 and -0.0 among them (at entries the fills below look up)."""
    rng = np.random.default_rng(seed)
    v = rng.uniform(-60.0, 60.0, 4096).astype(np.float32)
    v = v[v != 0]
    _, first = np.unique(v.view(np.uint32), return_index=True)
    v = v[np.sort(first)][:768].reshape(3, 256).copy()
    v[1, 128] = 0.0
    v[2, 255] = -0.0
    assert len(np.unique(v.view(np.uint32))) == 768
    return v


# ----------------------------------------------------------------------------------------------------------------------
# CPU part
# ----------------------------------------------------------------------------------------------------------------------
def test_workspace_layout_matches_the_library():
    """The offsets used to read the prep kernel's records are those of the library's workspace."""
    from bpc_baseline_b200 import _lib
    lib = _lib.load()
    for R in (1, 7, 45, 1000):
        for T in (1, 2, 3, 31, 33, 97, 100, 160, 224, 255, 256, 257, 1000, 1024):
            assert ws_off_count(R, T) + 64 + 8 * R + 64 == lib.bpc_roi_crop_workspace_bytes(R, T), (R, T)


def test_dispatch_restatement_table_and_boundaries():
    reached = set()
    for W in list(range(16, 2000, 16)) + [1913, 1918, 8208]:
        for T in list(range(1, 300)) + [320, 512, 1000, 1024]:
            for out in ('u8', 'f32', 'bf16'):
                for swap in (False, True):
                    plan = crop_plan(W, T, out, swap)
                    if plan is not None:
                        reached |= {(*plan[c], c) for c in plan}
    assert reached == TABLE and len(TABLE) == 36 + 56 + 5
    assert cta_pitch_max(224) == 1408 and cta_pitch_max(256) == 1600
    kern = lambda W, T: crop_plan(W, T, 'f32', True)[1][0]
    assert [kern(W, 224) for W in (176, 192, 464, 480, 601)] == ['warp', 'warp', 'warp', 'cta', 'warp']
    assert [kern(W, 256) for W in (528, 544)] == ['warp', 'cta']
    assert [kern(1920, T) for T in (256, 257)] == ['cta', 'warp']
    assert pool_flags(176, 64) == (False, False) and pool_flags(192, 64) == (True, True)


def test_matrix_plan_reaches_every_cell():
    """The boxes of the matrix reach every cell of the table by the restated rules (the GPU test checks the kernel)."""
    reached = set()
    for W, T in MATRIX:
        rois = matrix_boxes(W, POOL_H, POOL_B, T, seed=(W, T))
        classes = {box_class(b, POOL_B, POOL_H, W, T) for b in rois}
        for out in ('u8', 'f32', 'bf16'):
            for swap in (False, True):
                plan = crop_plan(W, T, out, swap)
                if plan is not None:
                    reached |= {(*plan[c], c) for c in classes}
    assert reached == TABLE, sorted(TABLE - reached)


def test_roi_class_rounding_ties():
    # 6 x 3 and 2 x 1 at T = 1: the short side is 0.5 -> 0 (rejected); at T = 3: 1.5 -> 2; 2 x 1 at T = 7: 3.5 -> 4
    assert [roi_class(6, 3, 1, False, False), roi_class(2, 1, 1, False, False)] == [0, 0]
    assert ocrop.letterbox_geometry(3, 6, 3)[1:3] == (3, 2) and ocrop.letterbox_geometry(1, 2, 7)[1:3] == (7, 4)
    assert roi_class(6, 3, 3, False, False) == 4 and roi_class(2, 1, 3, False, False) == 3
    assert roi_class(8192, 600, 224, True, True) == 2 and roi_class(8193, 600, 224, True, True) == 0


# ----------------------------------------------------------------------------------------------------------------------
# GPU part
# ----------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _pool(W, H, B, seed):
    from bpc_baseline_b200 import synth
    return synth.make_images(B, seed=seed, width=W, height=H)


@functools.lru_cache(maxsize=None)
def _luts():
    from bpc_baseline_b200 import batched
    return {'norm': batched.normalise_lut('cuda').cpu().numpy(), 'rand': random_lut()}


def _launch_record(R, T):
    """(class per ROI, the 16 launch counters) that the last crop launch of R ROIs left in the cached workspace."""
    from bpc_baseline_b200 import batched
    ws = batched._crop_workspace(torch.device('cuda'), R, T)
    cls = ws[:R * GEOM_BYTES].cpu().numpy().view(np.int32).reshape(R, GEOM_BYTES // 4)[:, 17]
    off = ws_off_count(R, T)
    return cls, ws[off:off + 64].cpu().numpy().view(np.int32)


def _check_launch(W, T, out_type, swap, rois, want_cls, n_valid=None):
    """The prep kernel's classes and the kernels that ran, against the restatement; returns the cells reached."""
    R = len(rois)
    cls, cnt = _launch_record(R, T)
    assert np.array_equal(cls, want_cls), (W, T, out_type, [(tuple(rois[i]), int(cls[i]), int(want_cls[i]))
                                                            for i in np.nonzero(cls != want_cls)[0][:8]])
    plan = crop_plan(W, T, out_type, swap)
    fast = np.isin(cls, (0, 1, 3, 4))
    assert cnt[0] == int((cls == 2).sum())                                  # generic list length
    if plan[0][0] == 'cta':
        assert cnt[8] == int(fast.sum()) and cnt[12] > 0 and cnt[4] == 0    # CTA list filled and walked, no warp launch
    else:
        assert cnt[8] == 0 and cnt[12] == 0 and cnt[4] >= R * ((T + 31) // 32 + 1)
    return {(*plan[int(c)], int(c)) for c in np.unique(cls) if c != -1}


def _reference(imgs, rois, T, fill):
    """uint8 canvases [R,T,T,3] (cv2 through oracle.crop.letterbox_ref on a np.full(fill) canvas) and the status."""
    B, H, W = imgs.shape[:3]
    out = np.empty((len(rois), T, T, 3), np.uint8)
    status = np.zeros(len(rois), np.int32)
    for r, (b, x1, y1, x2, y2) in enumerate(rois):
        w, h = x2 - x1, y2 - y1
        ok = 0 <= b < B and x1 >= 0 and y1 >= 0 and x2 <= W and y2 <= H and 0 < w <= MAX_ROI_WIDTH and h > 0
        if ok:
            _, nw, nh, _, _ = ocrop.letterbox_geometry(h, w, T)
            ok = nw >= 1 and nh >= 1
        if ok:
            out[r] = ocrop.letterbox_ref(imgs[b, y1:y2, x1:x2], T, fill_color=fill)[0]
        else:
            out[r] = np.asarray(fill, np.uint8)
            status[r] = 1
    return out, status


def _planes(canvas, lut, swap):
    return np.stack([lut[p][canvas[..., 2 - p if swap else p]] for p in range(3)], axis=1)


def _bf16_hwc_bits(f32_nchw):
    return torch.as_tensor(f32_nchw).to(torch.bfloat16).permute(0, 2, 3, 1).contiguous().view(torch.int16)


def _u32(a):
    return np.ascontiguousarray(a).view(np.uint32)


@functools.lru_cache(maxsize=None)
def _matrix_case(W, T):
    """Run and check one matrix case; returns the cells it reached (cached: the coverage test reuses the results)."""
    from bpc_baseline_b200 import batched
    imgs = _pool(W, POOL_H, POOL_B, 40 + W % 97)
    rois = matrix_boxes(W, POOL_H, POOL_B, T, seed=(W, T))
    R = len(rois)
    want_cls = np.array([box_class(b, POOL_B, POOL_H, W, T) for b in rois], np.int32)
    dimgs, drois = to_dev(imgs), to_dev(rois)
    luts = _luts()
    dluts = {k: to_dev(v) for k, v in luts.items()}
    ref = {fill: _reference(imgs, rois, T, fill) for fill in FILLS}
    cells = set()
    status = torch.full((R,), -1, dtype=torch.int32, device='cuda')
    for fill in FILLS:
        canvas, st_want = ref[fill]
        out = batched.roi_crop_u8(dimgs, drois, T=T, fill=fill, status=status).cpu().numpy()
        cells |= _check_launch(W, T, 'u8', False, rois, want_cls)
        assert np.array_equal(status.cpu().numpy(), st_want)
        bad = [r for r in range(R) if not np.array_equal(out[r], canvas[r])]
        assert not bad, ('u8', fill, [tuple(rois[r]) for r in bad[:6]])
    aligned, use_cta = pool_flags(W, T)
    for swap in (False, True):
        for fill, lk in (((0, 128, 255), 'rand'), ((7, 200, 31), 'norm'), ((255, 255, 255), 'rand')):
            canvas, st_want = ref[fill]
            want = _planes(canvas, luts[lk], swap)
            f32 = batched.roi_crop(dimgs, drois, T=T, fill=fill, swap_rb=swap, lut=dluts[lk], status=status)
            cells |= _check_launch(W, T, 'f32', swap, rois, want_cls)
            assert np.array_equal(status.cpu().numpy(), st_want)
            got = f32.cpu().numpy()
            bad = [r for r in range(R) if not np.array_equal(_u32(got[r]), _u32(want[r]))]
            assert not bad, ('f32', swap, fill, lk, [tuple(rois[r]) for r in bad[:6]])
            if not use_cta:
                with pytest.raises(RuntimeError, match='BPC_EUNSUPPORTED|code -5'):
                    batched.roi_crop_bf16(dimgs, drois, T=T, fill=fill, swap_rb=swap, lut=dluts[lk])
                continue
            b16 = batched.roi_crop_bf16(dimgs, drois, T=T, fill=fill, swap_rb=swap, lut=dluts[lk], status=status)
            cells |= _check_launch(W, T, 'bf16', swap, rois, want_cls)
            assert np.array_equal(status.cpu().numpy(), st_want)
            got16 = b16.permute(0, 2, 3, 1).contiguous().view(torch.int16).cpu()
            assert torch.equal(got16, _bf16_hwc_bits(want)), ('bf16', swap, fill, lk)
            assert torch.equal(got16, _bf16_hwc_bits(got))
    return frozenset(cells)



@pytest.mark.gpu
@pytest.mark.parametrize('W,T', MATRIX, ids=[f'W{W}-T{T}' for W, T in MATRIX])
def test_crop_matrix(W, T):
    """uint8 (three fills), float32 (both channel orders, white / asymmetric fills, default / random LUT) and, where the
    CTA kernel runs, bfloat16: bit-equal to cv2 + the LUT, status 1 exactly for rejected boxes."""
    _matrix_case(W, T)


@pytest.mark.gpu
@pytest.mark.parametrize('W,T', [(176, 224), (192, 224), (176, 64), (192, 64), (464, 224), (480, 224), (528, 256),
                                 (544, 256), (601, 224), (1918, 64), (1920, 256), (1920, 257)])
def test_bf16_refused_exactly_off_the_cta_path(W, T):
    """roi_crop_bf16 succeeds exactly where the restated dispatch says CTA kernel; the float launch on the same pool runs
    the kernel the restatement names (workspace counters)."""
    from bpc_baseline_b200 import batched
    H = 300
    imgs = _pool(W, H, 1, 3)
    rois = np.asarray([(0, 0, 0, min(W, 150), 100), (0, 1, 2, min(W, 2 * T + 3), 3), (0, 0, 0, W, H)], np.int32)
    want_cls = np.array([box_class(b, 1, H, W, T) for b in rois], np.int32)
    dimgs, drois = to_dev(imgs), to_dev(rois)
    f32 = batched.roi_crop(dimgs, drois, T=T, fill=(0, 128, 255), swap_rb=False)
    _check_launch(W, T, 'f32', False, rois, want_cls)
    if crop_plan(W, T, 'bf16', False) is None:
        with pytest.raises(RuntimeError):
            batched.roi_crop_bf16(dimgs, drois, T=T, fill=(0, 128, 255), swap_rb=False)
    else:
        b16 = batched.roi_crop_bf16(dimgs, drois, T=T, fill=(0, 128, 255), swap_rb=False)
        _check_launch(W, T, 'bf16', False, rois, want_cls)
        assert torch.equal(b16.view(torch.int16), f32.to(torch.bfloat16).contiguous(memory_format=torch.channels_last).view(torch.int16))


@pytest.mark.gpu
@pytest.mark.parametrize('W,T', [(1918, 100), (448, 224), (176, 33), (1920, 300), (1920, 97)])
def test_device_count_on_every_kernel(W, T):
    """n_rois with a nonzero roi_first falling inside one launch: rows at or beyond the count keep the sentinel (output
    and status), their class is -1, and the rows below it are correct -- on the warp kernel (aligned / unaligned, rejected
    boxes among the skipped rows), the generic kernel (class-2 boxes on both sides of the count) and the CTA kernel."""
    from bpc_baseline_b200 import batched
    imgs = _pool(W, POOL_H, POOL_B, 40 + W % 97)
    rois = matrix_boxes(W, POOL_H, POOL_B, T, seed=(W, T, 1))
    R, first, count = len(rois), 5, 5 + len(rois) // 2
    keep = count - first                                            # rows [0, keep) are processed
    all_cls = np.array([box_class(b, POOL_B, POOL_H, W, T) for b in rois], np.int32)
    assert 2 in all_cls[:keep] and {0, 2} <= set(all_cls[keep:].tolist())     # class-2 and rejected boxes beyond the count
    want_cls = np.where(np.arange(R) < keep, all_cls, -1).astype(np.int32)
    dimgs, drois = to_dev(imgs), to_dev(rois)
    nro = torch.tensor([count], dtype=torch.int32, device='cuda')
    fill, lut = (0, 128, 255), _luts()['rand']
    canvas, st_want = _reference(imgs, rois, T, fill)
    for swap in (False, True):
        out = torch.full((R, 3, T, T), 7.0, device='cuda')
        status = torch.full((R,), -7, dtype=torch.int32, device='cuda')
        batched.roi_crop(dimgs, drois, T=T, fill=fill, swap_rb=swap, lut=to_dev(lut), n_rois=nro, roi_first=first, out=out,
                         status=status)
        _check_launch(W, T, 'f32', swap, rois, want_cls)
        got, st = out.cpu().numpy(), status.cpu().numpy()
        assert bool((got[keep:] == 7.0).all()) and bool((st[keep:] == -7).all())
        assert np.array_equal(st[:keep], st_want[:keep])
        assert np.array_equal(_u32(got[:keep]), _u32(_planes(canvas[:keep], lut, swap)))
    out8 = torch.full((R, T, T, 3), 7, dtype=torch.uint8, device='cuda')
    batched.roi_crop_u8(dimgs, drois, T=T, fill=fill, n_rois=nro, roi_first=first, out=out8)
    _check_launch(W, T, 'u8', False, rois, want_cls)
    got8 = out8.cpu().numpy()
    assert bool((got8[keep:] == 7).all()) and np.array_equal(got8[:keep], canvas[:keep])


@pytest.mark.gpu
@pytest.mark.parametrize('T', [224, 257])
def test_roi_width_limit(T):
    """BPC_MAX_ROI_WIDTH on a 8208-px pool: 8192-wide boxes match cv2, 8193-wide ones are rejected (status 1, all fill)."""
    from bpc_baseline_b200 import batched
    W, H = 8208, 700
    imgs = _pool(W, H, 1, 11)
    rois = np.asarray([(0, 0, 0, 8192, H), (0, 16, 100, 8208, 400), (0, 0, 0, 8193, H), (0, 15, 3, 8208, 40),
                       (0, 5000, 0, 8208, H)], np.int32)
    want_cls = np.array([box_class(b, 1, H, W, T) for b in rois], np.int32)
    assert list(want_cls[:4]) == [2, 2, 0, 0]
    dimgs, drois = to_dev(imgs), to_dev(rois)
    fill, lut = (7, 200, 31), _luts()['rand']
    canvas, st_want = _reference(imgs, rois, T, fill)
    assert list(st_want) == [0, 0, 1, 1, 0]
    status = torch.full((5,), -1, dtype=torch.int32, device='cuda')
    out8 = batched.roi_crop_u8(dimgs, drois, T=T, fill=fill, status=status).cpu().numpy()
    _check_launch(W, T, 'u8', False, rois, want_cls)
    assert np.array_equal(out8, canvas) and np.array_equal(status.cpu().numpy(), st_want)
    f32 = batched.roi_crop(dimgs, drois, T=T, fill=fill, swap_rb=True, lut=to_dev(lut), status=status).cpu().numpy()
    _check_launch(W, T, 'f32', True, rois, want_cls)
    assert np.array_equal(_u32(f32), _u32(_planes(canvas, lut, True))) and np.array_equal(status.cpu().numpy(), st_want)


@pytest.mark.gpu
@pytest.mark.parametrize('w,h,T,kernel', [(480, 300, 224, 'cta'), (480, 700, 224, 'cta'), (301, 250, 224, 'warp'),
                                          (176, 100, 224, 'warp'), (464, 200, 224, 'warp'), (2000, 150, 224, 'generic'),
                                          (448, 448, 224, 'generic'), (208, 120, 91, 'cta')])
def test_letterbox_dropin_on_each_kernel(w, h, T, kernel):
    """utils.data_utils.letterbox_preserving_aspect_ratio uploads the crop as a pool of its own width: crop widths that
    send it to each kernel, non-white fill, against the reference's cv2 call."""
    from bpc_baseline_b200.utils import data_utils
    img = np.random.default_rng([w, h]).integers(0, 256, (h, w, 3), dtype=np.uint8)
    cls = box_class((0, 0, 0, w, h), 1, h, w, T)
    plan = crop_plan(w, T, 'u8', False)
    assert plan[cls][0] == kernel
    fill = (7, 200, 31)
    got = data_utils.letterbox_preserving_aspect_ratio(img, T, fill_color=fill)
    want = ocrop.letterbox_ref(img, T, fill_color=fill)
    _check_launch(w, T, 'u8', False, np.asarray([(0, 0, 0, w, h)], np.int32), np.array([cls], np.int32))
    assert np.array_equal(got[0], want[0]) and got[1:] == want[1:]


@pytest.mark.gpu
def test_torch_ops_with_fill_and_lut_match_batched():
    """torch.ops.bpc_b200.roi_crop / roi_crop_bf16 / roi_crop_u8 pass the fill and the LUT through unchanged."""
    from bpc_baseline_b200 import batched, ops
    W, T = 1920, 224
    imgs = _pool(W, POOL_H, POOL_B, 40 + W % 97)
    rois = matrix_boxes(W, POOL_H, POOL_B, T, seed=(W, T))
    dimgs, drois, dlut = to_dev(imgs), to_dev(rois), to_dev(_luts()['rand'])
    fill = (0, 128, 255)
    for swap in (False, True):
        crops, st = ops.roi_crop(dimgs, drois, T, fill=fill, swap_rb=swap, lut=dlut)
        want_st = torch.zeros(len(rois), dtype=torch.int32, device='cuda')
        want = batched.roi_crop(dimgs, drois, T=T, fill=fill, swap_rb=swap, lut=dlut, status=want_st)
        assert torch.equal(crops.view(torch.int32), want.view(torch.int32)) and torch.equal(st, want_st)
        b16, st16 = ops.roi_crop_bf16(dimgs, drois, T, fill=fill, swap_rb=swap, lut=dlut)
        want16 = batched.roi_crop_bf16(dimgs, drois, T=T, fill=fill, swap_rb=swap, lut=dlut)
        assert torch.equal(b16.view(torch.int16), want16.view(torch.int16)) and torch.equal(st16, want_st)
    u8, st8 = ops.roi_crop_u8(dimgs, drois, T, fill=fill)
    assert torch.equal(u8, batched.roi_crop_u8(dimgs, drois, T=T, fill=fill)) and torch.equal(st8, want_st)


@pytest.mark.gpu
def test_every_cell_of_the_table_is_reached():
    """Union of the (kernel, instantiation, class) cells the matrix launches reached, read back from the workspace."""
    reached = set()
    for W, T in MATRIX:
        reached |= _matrix_case(W, T)
    assert reached == TABLE, ('missing', sorted(TABLE - reached), 'unexpected', sorted(reached - TABLE))
