"""Order of the CTA kernel's crop list: after a launch on the CTA path, the list in the crop workspace holds every crop of
classes 0 / 1 / 3 / 4 exactly once and, where the crops must share source lines, is sorted by the bucket of the crop's
first source row in the pool.

The crops are reordered so that those in flight together read a narrow band of the image pool and share its lines in L2
(``bpc_crop_order_kernel`` in csrc/crop.cu).  The key of a crop is its first source row ``image * H + y1``; buckets are
2^shift rows, shift the least that leaves at most ORDER_BUCKETS of them in ``[0, B H)``; a rejected box (class 0) has no
source rows and goes to bucket 0.  A list is reordered only when it has two or more entries and the source areas of its
crops add up to more than the pool's pixels; counter 9 is then 1.  The list (``list1``) sits behind the counters and the
generic list: ``ws_off_count + 64 + 4 R``, its length is counter 8.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from tests.test_gpu_crop_matrix import GEOM_BYTES, box_class, pool_flags, ws_off_count

ORDER_BUCKETS = 4096


def bucket_of(rois, cls, B, H):
    """Bucket of each ROI's first source row (0 for rejected boxes)."""
    rois = np.asarray(rois, np.int64)
    shift = max(0, (B * H - 1).bit_length() - ORDER_BUCKETS.bit_length() + 1)
    return np.where(np.asarray(cls) == 0, 0, (rois[:, 0] * H + rois[:, 2]) >> shift)


def reordered(rois, cls, B, H, W):
    """Whether the kernel reorders the list: two or more entries whose crops read more source pixels than the pool holds."""
    cls = np.asarray(cls)
    r = np.asarray(rois, np.int64)[np.isin(cls, (1, 3, 4))]
    return int(np.isin(cls, (0, 1, 3, 4)).sum()) >= 2 and int(((r[:, 3] - r[:, 1]) * (r[:, 4] - r[:, 2])).sum()) > B * H * W


def check_order(order, flag, rois, cls, B, H, W):
    """``order``: the list read back, ``flag``: counter 9; ``cls``: the class of every ROI (-1 beyond the device count)."""
    fast = np.flatnonzero(np.isin(cls, (0, 1, 3, 4)))
    assert np.array_equal(np.sort(order), fast), 'not a permutation of the fast-class ROIs'
    want = reordered(rois, cls, B, H, W)
    assert flag == int(want), (flag, want)
    if want:
        b = bucket_of(np.asarray(rois)[order], np.asarray(cls)[order], B, H)
        assert bool((np.diff(b) >= 0).all()), f'bucket decreases at list positions {np.flatnonzero(np.diff(b) < 0)[:8]}'


def test_bucket_and_gate_restatement():
    B, H, W = 24, 2160, 3840                              # 51840 rows: buckets of 16 rows
    rois = np.array([(0, 0, 0, 5, 5), (23, 9, H - 1, 10, H), (1, 0, 0, 4, 4), (1, 0, 7, 4, 9), (0, 0, 0, 0, 0)], np.int32)
    cls = np.array([1, 1, 3, 4, 0])
    assert list(bucket_of(rois, cls, B, H)) == [0, 3239, 135, 135, 0]
    assert list(bucket_of(rois, cls, 2, 2048)) == [0, 23 * 2048 + 2159, 2048, 2055, 0]         # 4096 rows: one each
    assert list(bucket_of(rois, cls, 2, 2049)) == [0, (23 * 2049 + 2159) >> 1, 1024, 1028, 0]  # 4098 rows: two each
    assert not reordered(rois, cls, B, H, W) and reordered(rois, cls, 1, 1, 49) and not reordered(rois, cls, 1, 1, 50)   # 50 px
    assert not reordered(rois[:1], cls[:1], 1, 1, 1)
    with pytest.raises(AssertionError, match='bucket decreases'):
        check_order(np.array([1, 0]), 1, rois[:2], cls[:2], 1, 1, 25)
    with pytest.raises(AssertionError, match='permutation'):
        check_order(np.array([0]), 0, rois[:2], cls[:2], B, H, W)
    check_order(np.array([4, 0, 2, 3, 1]), 1, rois, cls, 1, 1, 49)
    check_order(np.array([1, 0, 2, 3, 4]), 0, rois, cls, B, H, W)


def _rois(rng, R, B, H, W, T):
    """Boxes of every class in random list order: area (class 1 / 4), growing (3), integer ratio and very large (2),
    boxes outside the pool (0)."""
    kind = rng.integers(0, 10, R)
    side = np.where(kind < 5, rng.integers(T + 1, 2 * T, R), np.where(kind < 7, rng.integers(2 * T, 5 * T, R),
                    rng.integers(8, T, R)))
    w = np.minimum(side, W)
    h = np.minimum(np.maximum(8, (side * rng.uniform(0.3, 1.0, R)).astype(np.int64)), H)
    x1 = (rng.random(R) * (W - w + 1)).astype(np.int64)
    y1 = (rng.random(R) * (H - h + 1)).astype(np.int64)
    img = rng.integers(0, B, R)
    rois = np.stack([img, x1, y1, x1 + w, y1 + h], axis=1)
    sq = kind == 8                                        # 2T x 2T: integer ratio 2, the generic kernel
    rois[sq, 3] = rois[sq, 1] + min(2 * T, W)
    rois[sq, 4] = rois[sq, 2] + min(2 * T, H)
    rois[sq, 1:5:2] -= np.maximum(0, rois[sq, 3:4] - W)
    rois[sq, 2:5:2] -= np.maximum(0, rois[sq, 4:5] - H)
    rois[kind == 9, 0] = B                                # no such image: rejected
    return rois.astype(np.int32)


def _launch(images, rois, T, n_rois=None, roi_first=0):
    """One bpc_roi_crop call over all of ``rois`` with a workspace of its own; returns (list1, counter 9, class per ROI)."""
    from bpc_baseline_b200 import _lib, batched
    B, H, W, _ = images.shape
    R = len(rois)
    lib = _lib.load()
    drois = torch.as_tensor(rois).cuda()
    ws = torch.empty((int(lib.bpc_roi_crop_workspace_bytes(R, T)),), dtype=torch.uint8, device='cuda')
    out = torch.empty((R, 3, T, T), dtype=torch.float32, device='cuda')
    nro = torch.tensor([n_rois], dtype=torch.int32, device='cuda') if n_rois is not None else None
    lut = batched.normalise_lut('cuda')
    fill = (C.c_uint8 * 3)(255, 255, 255)
    _lib.check(lib.bpc_roi_crop(batched._p(images), B, H, W, batched._p(drois), R, batched._p(nro), roi_first, T, fill, 1,
                                batched._p(lut), batched._p(out), None, batched._p(ws), ws.numel(), batched._stream(images.device)),
               'bpc_roi_crop')
    off = ws_off_count(R, T)
    cnt = ws[off:off + 64].cpu().numpy().view(np.int32)
    list1 = ws[off + 64 + 4 * R:off + 64 + 8 * R].cpu().numpy().view(np.int32)[:cnt[8]]
    cls = ws[:R * GEOM_BYTES].cpu().numpy().view(np.int32).reshape(R, GEOM_BYTES // 4)[:, 17]
    assert cnt[8] == 0 or cnt[12] > 0
    return list1, int(cnt[9]), cls


@pytest.fixture(scope='module')
def pools():
    """Pools of one and of three 1920 x 1080 images (noise)."""
    gen = torch.Generator(device='cuda').manual_seed(5)
    three = torch.randint(0, 256, (3, 1080, 1920, 3), dtype=torch.uint8, device='cuda', generator=gen)
    return {1: three[:1], 3: three}


# (R, T, images in the pool, list reordered): R = 37 reads more pixels than one image holds and fewer than three
CASES = [(1, 224, 3, False), (37, 224, 1, True), (37, 224, 3, False), (16384, 224, 3, True), (70000, 64, 3, True)]


@pytest.mark.gpu
@pytest.mark.parametrize('R,T,nimg,sorted_', CASES, ids=[f'R{c[0]}-T{c[1]}-B{c[2]}' for c in CASES])
def test_list_sorted_by_first_source_row(pools, R, T, nimg, sorted_):
    pool = pools[nimg]
    B, H, W, _ = pool.shape
    assert pool_flags(W, T)[1]
    rois = _rois(np.random.default_rng([R, T]), R, B, H, W, T)
    order, flag, cls = _launch(pool, rois, T)
    assert np.array_equal(cls, np.array([box_class(b, B, H, W, T) for b in rois], np.int32))
    if R > 1:
        assert {0, 1, 2, 3, 4} <= set(cls.tolist())
    assert reordered(rois, cls, B, H, W) == sorted_
    check_order(order, flag, rois, cls, B, H, W)


@pytest.mark.gpu
@pytest.mark.parametrize('R,nimg', [(37, 1), (16384, 3)])
def test_device_count_truncates_the_list(pools, R, nimg):
    """Rows at or beyond n_rois - roi_first are not on the list; an empty list (nothing below the count) launches fine."""
    pool = pools[nimg]
    B, H, W, _ = pool.shape
    T = 224
    rois = _rois(np.random.default_rng([R, 1]), R, B, H, W, T)
    for first, count in ((5, 5 + R // 2), (7, 7), (3, 2)):
        order, flag, cls = _launch(pool, rois, T, n_rois=count, roi_first=first)
        keep = max(0, count - first)
        assert bool((cls[keep:] == -1).all()) and bool((cls[:keep] != -1).all())
        check_order(order, flag, rois, cls, B, H, W)
        assert len(order) > 0 or keep == 0


@pytest.mark.gpu
def test_all_rejected_and_all_generic(pools):
    pool = pools[1]
    B, H, W, _ = pool.shape
    T = 224
    rej = np.array([(B, 0, 0, 50, 50), (0, 0, 0, 0, 5), (-1, 0, 0, 4, 4), (0, W - 3, 0, W + 1, 10)] * 10, np.int32)
    order, flag, cls = _launch(pool, rej, T)
    assert bool((cls == 0).all()) and len(order) == len(rej)
    check_order(order, flag, rej, cls, B, H, W)
    gen = np.array([(0, 16 * i, 3 * i, 16 * i + 2 * T, 3 * i + 2 * T) for i in range(40)], np.int32)
    order, flag, cls = _launch(pool, gen, T)
    assert bool((cls == 2).all()) and len(order) == 0 and flag == 0
