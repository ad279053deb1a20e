"""CUDA ROI-crop path (through the C ABI) against the reference's own letterbox outputs and cv2.

Bar: crops within 1e-3 absolute in normalised units; 1 uint8 LSB is 0.017 there, so the uint8 resize
must be, and is asserted to be, bit-exact; the float tensor is asserted bit-equal to torchvision's.
"""
import numpy as np
import pytest
import torch

from oracle import crop as ocrop
from tests.gpu_util import to_dev

pytestmark = pytest.mark.gpu


def _rois(boxes, img=0):
    return np.concatenate([np.full((len(boxes), 1), img, np.int32), np.asarray(boxes, np.int32)], axis=1)


@pytest.mark.parametrize('T', [224, 256, 64])
def test_letterbox_u8_golden(golden_crops, T):
    from bpc_baseline_b200 import batched
    g = golden_crops
    boxes = g['boxes'] if T != 256 else g['boxes'][::2]
    images = to_dev(g['image'][None])
    status = torch.zeros(len(boxes), dtype=torch.int32, device='cuda')
    out = batched.roi_crop_u8(images, to_dev(_rois(boxes)), T=T, status=status).cpu().numpy()
    assert int(status.sum()) == 0
    for r, b in enumerate(boxes):
        diff = out[r].astype(int) - g[f'canvas_T{T}'][r]
        assert not diff.any(), (T, tuple(b), int(np.abs(diff).max()), int((diff != 0).sum()))


def test_tensor_golden_and_lut(golden_crops):
    from bpc_baseline_b200 import batched
    g = golden_crops
    lut = batched.normalise_lut('cuda').cpu().numpy()
    assert np.array_equal(lut.view(np.uint32), g['lut'].view(np.uint32))
    images = to_dev(g['image'][None])
    out = batched.roi_crop(images, to_dev(_rois(g['boxes'][:4])), T=64, swap_rb=True).cpu().numpy()
    assert np.array_equal(out.view(np.uint32), g['tensor_T64'].view(np.uint32))


@pytest.mark.parametrize('T,swap', [(224, True), (256, True), (224, False)])
def test_tensor_vs_reference_calls(golden_crops, T, swap):
    """f32 [R,3,T,T] against the reference's four library calls (cv2.resize, cvtColor, to_tensor, normalize)."""
    from bpc_baseline_b200 import batched
    g = golden_crops
    boxes = g['boxes']
    out = batched.roi_crop(to_dev(g['image'][None]), to_dev(_rois(boxes)), T=T, swap_rb=swap).cpu().numpy()
    for r, b in enumerate(boxes):
        want = ocrop.crop_tensor_ref(g['image'], b, target_size=T, swap_rb=swap)
        assert np.abs(out[r] - want).max() <= 1e-3                       # the north-star tolerance
        assert np.array_equal(out[r].view(np.uint32), want.view(np.uint32)), tuple(b)


@pytest.mark.parametrize('T', [224, 256, 160])
def test_random_boxes_all_regimes_full_res(T):
    """Full-resolution image pool, random boxes U{8..900}: bit-exact uint8 vs cv2 through the oracle (T = 224 / 256: the
    compile-time instantiations of the CTA kernel, 160: its run-time-T one with five consumer warps)."""
    from bpc_baseline_b200 import batched, synth
    from oracle.area_spec import regime
    imgs = synth.make_images(2, seed=5, width=1920, height=1080)
    rng = np.random.default_rng(17)
    rois = []
    for _ in range(160):
        w, h = rng.integers(8, 900, 2)
        x1 = int(rng.integers(0, 1920 - w + 1)); y1 = int(rng.integers(0, 1080 - h + 1))
        rois.append((int(rng.integers(0, 2)), x1, y1, x1 + int(w), y1 + int(h)))
    # bottom-right corner of the LAST image of the pool: the staging code must not read past the allocation
    rois += [(1, 1700, 900, 1920, 1080), (1, 1500, 700, 1920, 1080), (1, 1000, 300, 1920, 1080), (1, 1912, 1000, 1920, 1080)]
    rois += [(1, 0, 0, 1920, 1080), (0, 1919 - 8, 1080 - 9, 1919, 1080), (1, 0, 0, 2 * T, 2 * T), (0, 5, 5, 5 + 3 * T, 5 + 2 * T),
             (0, 0, 0, T, T), (1, 100, 100, 100 + T, 100 + T // 2)]                 # integer ratios (regime 2) and scale exactly 1
    rois = np.asarray(rois, np.int32)
    out = batched.roi_crop_u8(to_dev(imgs), to_dev(rois), T=T).cpu().numpy()
    outf = batched.roi_crop(to_dev(imgs), to_dev(rois), T=T, swap_rb=True).cpu().numpy()
    lut = batched.normalise_lut('cuda').cpu().numpy()
    seen = set()
    for r, (b, x1, y1, x2, y2) in enumerate(rois):
        want = ocrop.crop_u8_ref(imgs[b], (x1, y1, x2, y2), T)
        _, nw, nh, _, _ = ocrop.letterbox_geometry(y2 - y1, x2 - x1, T)
        seen.add(regime(x2 - x1, y2 - y1, nw, nh))
        assert np.array_equal(out[r], want), (r, tuple(rois[r]))
        assert np.array_equal(outf[r], np.stack([lut[p][want[..., 2 - p]] for p in range(3)])), (r, tuple(rois[r]))
    assert seen == {1, 2, 3}


@pytest.mark.parametrize('T,width', [(224, 1920), (64, 1920), (256, 1920), (128, 3840), (256, 1918), (100, 1913)])
def test_large_boxes_four_to_six_taps(T, width):
    """Boxes of 2T .. 5.3T: the 4 / 5 / 6-tap class (source-row records in the CTA kernel, wide rows by 1-D bulk copies; the
    row-streaming ring of the per-strip kernel on the pools the CTA kernel does not take) and, beyond scale 5, the generic kernel.  width 1920 / 3840:
    image pitch a multiple of 16 bytes (CTA kernel, 2-D TMA staging); 1918 / 1913: the per-strip kernel's 1-D bulk-copy path."""
    from bpc_baseline_b200 import batched, synth
    imgs = synth.make_images(2, seed=9, width=width, height=1080)
    rng = np.random.default_rng([23, T, width])
    rois = []
    for lo, hi in ((2.0, 3.0), (3.0, 4.0), (4.0, 5.0), (5.0, 5.3)):
        for _ in range(10):
            long_side = min(int(rng.uniform(lo, hi) * T), 1080)
            short = int(rng.integers(max(8, long_side // 6), long_side + 1))
            w, h = (long_side, short) if rng.random() < 0.5 else (short, long_side)
            w = min(w, width)
            x1 = int(rng.integers(0, width - w + 1)); y1 = int(rng.integers(0, 1080 - h + 1))
            rois.append((int(rng.integers(0, 2)), x1, y1, x1 + w, y1 + h))
    # exact integer-ish ratios next to the class boundaries, and the bottom-right corner of the last image
    rois += [(1, width - 4 * T - 1 if width > 4 * T + 1 else 0, 0, width, min(1080, 4 * T + 1)),
             (1, max(0, width - 5 * T), 1080 - min(1080, 3 * T), width, 1080), (0, 0, 0, min(width, 4 * T + 3), min(1080, 2 * T + 1))]
    rois = np.asarray(rois, np.int32)
    out = batched.roi_crop_u8(to_dev(imgs), to_dev(rois), T=T).cpu().numpy()
    outf = batched.roi_crop(to_dev(imgs), to_dev(rois), T=T, swap_rb=True).cpu().numpy()
    lut = batched.normalise_lut('cuda').cpu().numpy()
    for r, (b, x1, y1, x2, y2) in enumerate(rois):
        want = ocrop.crop_u8_ref(imgs[b], (x1, y1, x2, y2), T)
        assert np.array_equal(out[r], want), (r, tuple(rois[r]))
        wantf = np.stack([lut[p][want[..., 2 - p]] for p in range(3)])
        assert np.array_equal(outf[r], wantf), (r, tuple(rois[r]))


@pytest.mark.parametrize('T', [320, 512, 1000])
def test_target_sizes_above_256(T):
    """The reference's target_size is a free parameter (data_utils.py:34): T up to BPC_MAX_TARGET, every regime and class."""
    from bpc_baseline_b200 import batched, synth
    imgs = synth.make_images(2, seed=21, width=1920, height=1080)
    rng = np.random.default_rng([41, T])
    rois = [(1, 0, 0, 1920, 1080), (0, 0, 0, min(T, 1080), min(T, 1080)), (1, 1920 - 2 * min(T, 540), 0, 1920, 2 * min(T, 540))]
    for lo, hi in ((0.1, 0.6), (0.6, 1.0), (1.0, 1.5), (1.5, 2.0), (2.0, 3.3)):
        for _ in range(5):
            long_side = max(8, min(int(rng.uniform(lo, hi) * T), 1080))
            short = int(rng.integers(max(4, long_side // 5), long_side + 1))
            w, h = (long_side, short) if rng.random() < 0.5 else (short, long_side)
            x1 = int(rng.integers(0, 1920 - w + 1)); y1 = int(rng.integers(0, 1080 - h + 1))
            rois.append((int(rng.integers(0, 2)), x1, y1, x1 + w, y1 + h))
    rois = np.asarray(rois, np.int32)
    out = batched.roi_crop_u8(to_dev(imgs), to_dev(rois), T=T).cpu().numpy()
    outf = batched.roi_crop(to_dev(imgs), to_dev(rois), T=T, swap_rb=True).cpu().numpy()
    lut = batched.normalise_lut('cuda').cpu().numpy()
    for r, (b, x1, y1, x2, y2) in enumerate(rois):
        want = ocrop.crop_u8_ref(imgs[b], (x1, y1, x2, y2), T)
        assert np.array_equal(out[r], want), (r, tuple(rois[r]))
        wantf = np.stack([lut[p][want[..., 2 - p]] for p in range(3)])
        assert np.array_equal(outf[r], wantf), (r, tuple(rois[r]))


@pytest.mark.parametrize('width', [16, 64, 176, 192, 208, 256])
def test_small_images_with_16_byte_pitch(width):
    """Image rows of 48 .. 768 bytes, all multiples of 16: the per-strip kernel's 1-D copies at T = 224 and below 576 bytes
    (WARP_MAX_PITCH); from 192 px on at T = 64 the CTA kernel, whose 2-D tensor-map boxes may then be as wide as, or wider
    than, what is left of a row."""
    from bpc_baseline_b200 import batched, synth
    H = 120
    imgs = synth.make_images(3, seed=12, width=width, height=H)
    rng = np.random.default_rng([31, width])
    rois = [(2, 0, 0, width, H), (2, width - min(width, 9), H - 7, width, H), (0, 0, 0, min(width, 8), 8)]
    for _ in range(40):
        w = int(rng.integers(2, width + 1)); h = int(rng.integers(2, H + 1))
        x1 = int(rng.integers(0, width - w + 1)); y1 = int(rng.integers(0, H - h + 1))
        rois.append((int(rng.integers(0, 3)), x1, y1, x1 + w, y1 + h))
    rois = np.asarray(rois, np.int32)
    for T in (64, 224):
        status = torch.zeros(len(rois), dtype=torch.int32, device='cuda')
        out = batched.roi_crop_u8(to_dev(imgs), to_dev(rois), T=T, status=status).cpu().numpy()
        st = status.cpu().numpy()
        for r, (b, x1, y1, x2, y2) in enumerate(rois):
            _, nw, nh, _, _ = ocrop.letterbox_geometry(y2 - y1, x2 - x1, T)
            if nw < 1 or nh < 1:
                assert st[r] == 1
                continue
            assert st[r] == 0
            assert np.array_equal(out[r], ocrop.crop_u8_ref(imgs[b], (x1, y1, x2, y2), T)), (T, r, tuple(rois[r]))


def test_rejected_rois_and_device_count():
    from bpc_baseline_b200 import batched, synth
    imgs = to_dev(synth.make_images(1, seed=6, width=640, height=480))
    rois = np.array([[0, 10, 10, 200, 150], [0, 50, 50, 50, 90], [0, 600, 400, 700, 470], [3, 0, 0, 10, 10],
                     [0, 0, 0, 640, 1], [0, 20, 30, 120, 140]], np.int32)
    status = torch.full((6,), -1, dtype=torch.int32, device='cuda')
    out = batched.roi_crop(imgs, to_dev(rois), T=64, status=status)
    st = status.cpu().numpy()
    # empty box, out of image, bad image index, and a box whose short side rounds to 0 (640x1 -> 64x0)
    assert list(st) == [0, 1, 1, 1, 1, 0]
    white = batched.normalise_lut('cuda')[:, 255].cpu().numpy()
    for r in (1, 2, 3, 4):
        assert np.array_equal(out[r].cpu().numpy(), np.broadcast_to(white[:, None, None], (3, 64, 64)))
    # device-side ROI count: rows beyond it are not written
    out2 = torch.full((6, 3, 64, 64), 7.0, device='cuda')
    batched.roi_crop(imgs, to_dev(rois), T=64, n_rois=torch.tensor([1], dtype=torch.int32, device='cuda'), out=out2)
    assert torch.equal(out2[0], out[0]) and bool((out2[1:] == 7.0).all())


def test_build_rois_matches_host_mirror():
    from bpc_baseline_b200 import batched, synth
    from tests.gpu_util import batch_to_dev
    batch = synth.make_scenes(32, 7, seed=synth.SEED + 21, p_drop=0.2)
    Ks, RTs, centers, boxes, counts = batch_to_dev(batch)
    res = batched.match_triangulate(Ks, RTs, centers, counts, 30)
    ios = np.arange(32 * 3, dtype=np.int32).reshape(32, 3) % 5
    rois, offs = batched.build_rois(boxes, res.idx, res.n, to_dev(ios))
    offs = offs.cpu().numpy()
    want = synth.rois_for_matches(batch.boxes, res.idx.cpu().numpy(), res.n.cpu().numpy(), ios)
    assert offs[-1] == len(want)
    assert np.array_equal(rois.cpu().numpy()[:offs[-1]], want)
    assert np.array_equal(offs[:-1], np.concatenate([[0], np.cumsum(3 * res.n.cpu().numpy())[:-1]]))


def test_long_roi_lists_are_split_into_launches(monkeypatch):
    """More ROIs than one launch's scratch covers: the wrapper splits the list; roi_first / n_rois keep working."""
    from bpc_baseline_b200 import batched, synth
    imgs = synth.make_images(1, seed=8, width=800, height=600)
    rng = np.random.default_rng(8)
    rois = []
    for _ in range(23):
        w, h = rng.integers(16, 500, 2)
        x1 = int(rng.integers(0, 800 - w + 1)); y1 = int(rng.integers(0, 600 - h + 1))
        rois.append((0, x1, y1, x1 + int(w), y1 + int(h)))
    rois = np.asarray(rois, np.int32)
    whole = batched.roi_crop_u8(to_dev(imgs), to_dev(rois), T=96).cpu().numpy()
    monkeypatch.setattr(batched, 'MAX_ROIS_PER_LAUNCH', 5)
    status = torch.full((23,), -1, dtype=torch.int32, device='cuda')
    split = batched.roi_crop_u8(to_dev(imgs), to_dev(rois), T=96, status=status).cpu().numpy()
    assert np.array_equal(whole, split) and int(status.sum()) == 0
    out = torch.full((23, 3, 96, 96), 7.0, device='cuda')
    batched.roi_crop(to_dev(imgs), to_dev(rois), T=96, n_rois=torch.tensor([13], dtype=torch.int32, device='cuda'), out=out)
    assert bool((out[13:] == 7.0).all()) and not bool((out[:13] == 7.0).all(dim=(1, 2, 3)).any())
    for r in (0, 7, 12):
        want = ocrop.crop_tensor_ref(imgs[0], rois[r, 1:], target_size=96)
        assert np.array_equal(out[r].cpu().numpy().view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize('T,swap', [(224, True), (256, False), (96, True), (97, True), (100, False), (255, False)])
def test_bf16_channels_last_variant_equals_rounded_float_tensor(T, swap):
    """bpc_roi_crop_bf16 (the pose head's input, process_pose.py:210-212): every value of the float32 tensor rounded to
    bfloat16 (round-to-nearest-even, what torch's .to(bfloat16) does), stored channels-last -- all regimes and classes,
    a rejected box included; bit-equal to the float path's output after that rounding.  Odd T (97, 255) alternates the
    crops' base between 4- and 2-byte alignment, T = 100 leaves a partial last strip."""
    from bpc_baseline_b200 import batched, synth
    images = to_dev(synth.make_images(3, seed=9))
    rng = np.random.default_rng([77, T])
    R = 256
    w = rng.integers(8, 1500, R); h = rng.integers(8, 1200, R)
    w[:8] = [T, 2 * T, 3 * T, 40, 5 * T, 6 * T, 100, 17]; h[:8] = [T, T, 3 * T, 90, 2 * T, 6 * T, 100, 1100]
    x1 = (rng.random(R) * (synth.IMG_W - w)).astype(np.int64); y1 = (rng.random(R) * (synth.IMG_H - h)).astype(np.int64)
    rois = np.stack([rng.integers(0, 3, R), x1, y1, x1 + w, y1 + h], axis=1).astype(np.int32)
    rois[9] = [0, 10, 10, 10, 50]                                   # empty box -> rejected -> all fill
    drois = to_dev(rois)
    st_f = torch.zeros(R, dtype=torch.int32, device='cuda'); st_b = torch.zeros_like(st_f)
    f32 = batched.roi_crop(images, drois, T=T, swap_rb=swap, status=st_f)
    b16 = batched.roi_crop_bf16(images, drois, T=T, swap_rb=swap, status=st_b)
    assert b16.dtype == torch.bfloat16 and tuple(b16.shape) == (R, 3, T, T) and b16.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(st_f, st_b) and int(st_b[9]) == 1 and int(st_b.sum()) == 1
    want = f32.to(torch.bfloat16)
    assert torch.equal(b16.view(torch.int16), want.contiguous(memory_format=torch.channels_last).view(torch.int16))
    # device-side ROI count: rows beyond it are left untouched
    sentinel = torch.full((R, 3, T, T), 7.0, dtype=torch.bfloat16, device='cuda').contiguous(memory_format=torch.channels_last)
    nro = torch.tensor([100], dtype=torch.int32, device='cuda')
    batched.roi_crop_bf16(images, drois, T=T, swap_rb=swap, n_rois=nro, out=sentinel)
    assert torch.equal(sentinel[:100].view(torch.int16), b16[:100].view(torch.int16)) and bool((sentinel[100:] == 7.0).all())


def test_bf16_variant_refuses_unaligned_pools():
    """The bfloat16 output exists on the 2-D TMA path only (include/bpc_b200.h): an image pitch that is not a multiple of 16
    bytes is an error, never a silent fallback."""
    from bpc_baseline_b200 import batched
    images = torch.zeros((1, 600, 601, 3), dtype=torch.uint8, device='cuda')
    rois = to_dev(np.array([[0, 5, 5, 300, 200]], np.int32))
    with pytest.raises(RuntimeError):
        batched.roi_crop_bf16(images, rois, T=224)
    assert tuple(batched.roi_crop(images, rois, T=224).shape) == (1, 3, 224, 224)


# ----------------------------------------------------------------------------------------------------------------------
# argument checks of the batched crop API: a table or an output the kernels cannot use is refused before any launch
# ----------------------------------------------------------------------------------------------------------------------
class _NoLaunch:
    """Stands in for libbpc_b200.so: reaching any entry point fails the test, so a wrapper that lets a bad argument
    through fails here without a kernel ever reading or writing past a buffer."""

    def __getattr__(self, name):
        def entry(*args):
            pytest.fail(f'{name} was called with arguments the wrapper must refuse')
        return entry


LUT_WRAPPERS = ('roi_crop', 'roi_crop_bf16', 'crops_normalise', 'color_jitter')
OUT_WRAPPERS = LUT_WRAPPERS + ('roi_crop_u8',)


def _call(name, lut_device='cuda:0', lut_shape=(3, 256), out_device='cuda:0', T=32):
    from bpc_baseline_b200 import batched
    images = torch.zeros((1, 64, 96, 3), dtype=torch.uint8, device='cuda:0')
    rois = torch.tensor([[0, 4, 4, 60, 40]], dtype=torch.int32, device='cuda:0')
    crops = torch.zeros((1, T, T, 3), dtype=torch.uint8, device='cuda:0')
    lut = torch.zeros(lut_shape, dtype=torch.float32, device=lut_device)
    out = torch.empty((1, 3, T, T), dtype=torch.float32, device=out_device)
    if name == 'roi_crop':
        return batched.roi_crop(images, rois, T=T, lut=lut, out=out)
    if name == 'roi_crop_bf16':
        out = out.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        return batched.roi_crop_bf16(images, rois, T=T, lut=lut, out=out)
    if name == 'roi_crop_u8':
        return batched.roi_crop_u8(images, rois, T=T, out=torch.empty((1, T, T, 3), dtype=torch.uint8, device=out_device))
    if name == 'crops_normalise':
        return batched.crops_normalise([crops], T, lut=lut, out=out)
    order = torch.tensor([[0, 1, 2, 3]], dtype=torch.int32, device='cuda:0')
    factors = torch.ones((1, 4), dtype=torch.float32, device='cuda:0')
    return batched.color_jitter(crops, order, factors, lut=lut, out=out)


@pytest.mark.parametrize('shape', [(3, 128), (256, 3)])
@pytest.mark.parametrize('name', LUT_WRAPPERS)
def test_lut_of_another_shape_is_refused(monkeypatch, name, shape):
    """A [3,128] table would be read 768 floats deep; a transposed [256,3] one would be read with the wrong layout."""
    from bpc_baseline_b200 import _lib
    monkeypatch.setattr(_lib, 'load', _NoLaunch)
    with pytest.raises(RuntimeError, match=r'lut: shape'):
        _call(name, lut_shape=shape)


def test_crops_normalise_refuses_a_lut_off_its_device(monkeypatch):
    """``device`` names where the kernel runs (its sources may be peer mappings); the table must be there."""
    from bpc_baseline_b200 import _lib, batched
    monkeypatch.setattr(_lib, 'load', _NoLaunch)
    crops = torch.zeros((1, 32, 32, 3), dtype=torch.uint8, device='cuda:0')
    lut = torch.zeros((3, 256), dtype=torch.float32, device='cuda:0')
    with pytest.raises(RuntimeError, match=r'lut: on cuda:0, but the kernel runs on cuda:1'):
        batched.crops_normalise([crops], 32, lut=lut, device='cuda:1')


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
@pytest.mark.parametrize('name', OUT_WRAPPERS)
def test_lut_and_out_off_the_launch_device_are_refused(monkeypatch, name):
    from bpc_baseline_b200 import _lib
    monkeypatch.setattr(_lib, 'load', _NoLaunch)
    with pytest.raises(RuntimeError, match=r'out: on cuda:1, but the kernel runs on cuda:0'):
        _call(name, out_device='cuda:1')
    if name in LUT_WRAPPERS:
        with pytest.raises(RuntimeError, match=r'lut: on cuda:1, but the kernel runs on cuda:0'):
            _call(name, lut_device='cuda:1')
