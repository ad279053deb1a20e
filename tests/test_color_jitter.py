"""Training-side ColorJitter (bpc_color_jitter): torchvision.transforms.ColorJitter on Image.fromarray(canvas), then
to_tensor + normalize, as BOPSingleObjDataset.__getitem__ does with the jittered canvas.

CPU: the NumPy restatement (oracle/jitter_spec.py) against Pillow and torchvision on every input of each op, the torch-RNG
draws of draw_color_jitter, argument errors of the C entry point.  GPU: the kernel's float32 output bit-equal to torchvision.
"""
import ctypes
import itertools
import os

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import jitter_spec as js

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MEAN = [0.485, 0.456, 0.406]
STD = [0.229, 0.224, 0.225]
PERMS = list(itertools.permutations(range(4)))


def all_colours():
    """uint8 [2^24, 3], colour k = (k >> 16, (k >> 8) & 255, k & 255)."""
    k = np.arange(1 << 24, dtype=np.uint32)
    return np.stack([(k >> 16) & 255, (k >> 8) & 255, k & 255], -1).astype(np.uint8)


# ---- the spec against Pillow / torchvision (CPU) -------------------------------------------------------------------

def test_rgb_to_hsv_matches_pillow_on_every_colour():
    rgb = all_colours().reshape(16, 1 << 20, 3)
    for part in rgb:                                         # 16 chunks of 2^20 colours keep the temporaries small
        want = np.asarray(Image.fromarray(part.reshape(1024, 1024, 3)).convert('HSV')).reshape(-1, 3)
        assert np.array_equal(js.rgb2hsv(part), want)


def test_hsv_to_rgb_matches_pillow_on_every_triple():
    hsv = all_colours().reshape(16, 1 << 20, 3)
    for part in hsv:
        want = np.asarray(Image.fromarray(part.reshape(1024, 1024, 3), 'HSV').convert('RGB')).reshape(-1, 3)
        assert np.array_equal(js.hsv2rgb(part), want)


def test_hue_reciprocal_form_gives_pillows_byte_on_every_colour():
    """The kernel forms h / 6.0 of Pillow's rgb2hsv as h * (1.0 / 6.0): the double can differ in its last bit, but the
    hue byte (int)(float32(fmod(. + 1.0, 1.0)) * 255.0) is the same for every colour."""
    rgb = all_colours()
    R, G, B = [rgb[:, i].astype(np.int32) for i in range(3)]
    mx, mn = np.maximum(R, np.maximum(G, B)), np.minimum(R, np.minimum(G, B))
    keep = mx != mn
    R, G, B, mx, mn = R[keep], G[keep], B[keep], mx[keep], mn[keep]
    cr = (mx - mn).astype(np.float32)
    rc, gc, bc = [((mx - c).astype(np.float32) / cr).astype(np.float64) for c in (R, G, B)]
    h = np.float32(np.where(R == mx, bc - gc, np.where(G == mx, 2.0 + rc - bc, 4.0 + gc - rc))).astype(np.float64)

    def byte(x):
        x = np.where(x >= 1.0, x - 1.0, x)
        return (np.float32(x).astype(np.float64) * 255.0).astype(np.int64)
    assert np.array_equal(byte(h / 6.0 + 1.0), byte(h * (1.0 / 6.0) + 1.0))


def test_luma_matches_pillow_on_every_colour():
    rgb = all_colours().reshape(4096, 4096, 3)
    assert np.array_equal(js.luma(rgb), np.asarray(Image.fromarray(rgb).convert('L')))


def test_blend_matches_pillow_on_every_pair():
    a = np.repeat(np.arange(256, dtype=np.uint8)[:, None], 256, 1)
    b = a.T.copy()
    rng = np.random.default_rng(0)
    alphas = np.concatenate([[0.0, 1.0, 0.5, 1.0 - 2 ** -24, 1.0 + 2 ** -23, 2.0, 1.7], np.linspace(0, 1, 101)[1:-1],
                             rng.uniform(0, 2, 100), rng.uniform(1, 1.7, 20)]).astype(np.float32)
    assert len(alphas) >= 200
    ia, ib = Image.fromarray(a), Image.fromarray(b)
    for al in alphas:
        assert np.array_equal(js.blend(a, b, al), np.asarray(Image.blend(ia, ib, float(al)))), al


def _cj(**kw):
    import torchvision.transforms as T
    return T.ColorJitter(**kw)


CHAIN_CONFIGS = [                                            # (ColorJitter arguments, number of seeded images)
    (dict(brightness=0.4, contrast=0.6, saturation=0.7, hue=0.5), 120),
    (dict(brightness=0.4), 25), (dict(contrast=0.6), 25), (dict(saturation=0.7), 25), (dict(hue=0.5), 25),
    (dict(brightness=(0, 0), contrast=(0, 0), saturation=(0, 0), hue=0.2), 20),
    (dict(hue=(0.5, 0.5), saturation=(1.5, 2.0)), 20), (dict(hue=(-0.5, -0.5), contrast=(1.2, 1.9)), 20),
    (dict(brightness=(1.0, 1.9), contrast=(0.0, 2.0), saturation=(0.0, 2.0), hue=(-0.5, 0.5)), 30),
]


def test_spec_chain_matches_colorjitter():
    import torchvision.transforms as T
    rng = np.random.default_rng(1)
    n = 0
    for kw, count in CHAIN_CONFIGS:
        cj = _cj(**kw)
        for _ in range(count):
            img = rng.integers(0, 256, (int(rng.integers(8, 48)), int(rng.integers(8, 48)), 3), dtype=np.uint8)
            if n % 3 == 0:                                   # smooth gradients as well as noise
                img = (img // 4 + np.arange(img.shape[1], dtype=np.uint8)[None, :, None] * 4).astype(np.uint8)
            torch.manual_seed(n)
            want = np.asarray(cj(Image.fromarray(img)))
            torch.manual_seed(n)
            fn_idx, *fac = T.ColorJitter.get_params(cj.brightness, cj.contrast, cj.saturation, cj.hue)
            order = [int(k) if fac[int(k)] is not None else -1 for k in fn_idx]
            got = js.color_jitter(img, order, [np.float32(np.nan if f is None else f) for f in fac])
            assert np.array_equal(got, want), (kw, n)
            n += 1
    assert n >= 300


def test_draw_color_jitter_consumes_the_rng_like_colorjitter():
    import torchvision.transforms as T
    from bpc_baseline_b200.utils.data_utils import draw_color_jitter
    kw = dict(brightness=0.4, contrast=0.6, saturation=0.7, hue=0.5)
    cj = T.ColorJitter(**kw)
    img = Image.fromarray(np.random.default_rng(0).integers(0, 256, (16, 16, 3), dtype=np.uint8))
    for partial in (kw, dict(contrast=0.6), dict(hue=0.3, brightness=(0.5, 0.5)), {}):
        torch.manual_seed(11)
        for _ in range(3):
            T.ColorJitter(**partial)(img)
        after_forward = torch.get_rng_state()
        torch.manual_seed(11)
        order, factors = draw_color_jitter(3, **partial)
        assert torch.equal(torch.get_rng_state(), after_forward), partial
        assert order.dtype == np.int32 and factors.dtype == np.float32 and order.shape == factors.shape == (3, 4)
        for op, name in enumerate(('brightness', 'contrast', 'saturation', 'hue')):
            on = getattr(T.ColorJitter(**partial), name) is not None
            assert (order == op).any(axis=1).all() == on and np.isnan(factors[:, op]).all() == (not on)
    torch.manual_seed(3)
    a = draw_color_jitter(20, **kw)
    torch.manual_seed(3)
    b = [draw_color_jitter(1, **kw) for _ in range(20)]
    assert np.array_equal(a[0], np.concatenate([x[0] for x in b])) and np.array_equal(a[1], np.concatenate([x[1] for x in b]))
    torch.manual_seed(3)
    for r in range(20):                                      # the draws are ColorJitter.get_params', in its order
        fn_idx, *fac = T.ColorJitter.get_params(cj.brightness, cj.contrast, cj.saturation, cj.hue)
        assert a[0][r].tolist() == fn_idx.tolist() and a[1][r].tolist() == fac


def test_color_jitter_argument_errors_without_a_gpu():
    from bpc_baseline_b200 import _lib, batched, build
    from bpc_baseline_b200.utils.data_utils import dataset_crops
    build.build()
    lib = _lib.load()
    buf = ctypes.c_void_p(16)                                 # never dereferenced: every call below fails or does nothing first
    assert lib.bpc_color_jitter(buf, 1, 0, buf, buf, 0, buf, buf, None) == -1              # T < 1
    assert lib.bpc_color_jitter(buf, 1, 1025, buf, buf, 0, buf, buf, None) == -1           # T > BPC_MAX_TARGET
    assert lib.bpc_color_jitter(buf, -1, 64, buf, buf, 0, buf, buf, None) == -1            # n < 0
    assert lib.bpc_color_jitter(None, 0, 64, None, None, 0, None, None, None) == 0         # nothing to do
    for k in range(5):                                                                      # each null pointer
        ptrs = [buf] * 5
        ptrs[k] = None
        assert lib.bpc_color_jitter(ptrs[0], 1, 64, ptrs[1], ptrs[2], 0, ptrs[3], ptrs[4], None) == -1, k
    with pytest.raises(RuntimeError, match='CUDA tensor'):
        batched.color_jitter(torch.zeros(1, 8, 8, 3, dtype=torch.uint8), torch.zeros(1, 4, dtype=torch.int32), torch.zeros(1, 4))
    with pytest.raises(ValueError, match='as_uint8'):
        dataset_crops(np.zeros((1, 8, 8, 3), np.uint8), [[0, 0, 4, 4]], target_size=8, as_uint8=True,
                      color_jitter=(np.zeros((1, 4), np.int32), np.zeros((1, 4), np.float32)))


def test_torch_op_is_registered_with_a_meta_kernel():
    from bpc_baseline_b200 import build, ops
    build.build_torch_ext()
    meta = lambda shape, dt: torch.empty(shape, dtype=dt, device='meta')
    out = ops.load().color_jitter(meta((5, 101, 101, 3), torch.uint8), meta((5, 4), torch.int32), meta((5, 4), torch.float32), False,
                                  meta((3, 256), torch.float32))
    assert tuple(out.shape) == (5, 3, 101, 101) and out.dtype == torch.float32


# ---- the kernel against torchvision (GPU) ----------------------------------------------------------------------------

def pil_jitter(canvas, order, factors):
    """uint8 [T,T,3]: what ColorJitter.forward does with these draws (the _functional_pil ops in fn_idx order)."""
    import torchvision.transforms.functional as TF
    img = Image.fromarray(canvas)
    fns = (TF.adjust_brightness, TF.adjust_contrast, TF.adjust_saturation, TF.adjust_hue)
    for op in order:
        if op >= 0:
            img = fns[op](img, float(factors[op]))
    return np.asarray(img)


def tv_tensor(canvas, order, factors, swap_rb=False):
    """pil_jitter, then to_tensor + normalize; swap_rb reverses the channels of the jittered image before to_tensor, as
    bpc_roi_crop's swap_rb."""
    import torchvision.transforms.functional as TF
    arr = pil_jitter(canvas, order, factors)
    if swap_rb:
        arr = arr[..., ::-1].copy()
    return TF.normalize(TF.to_tensor(arr), MEAN, STD).numpy()


def random_canvases(rng, n, T):
    """Letterbox-like canvases: white fill, a noisy gradient object, some flat and grey regions."""
    c = np.full((n, T, T, 3), 255, np.uint8)
    for i in range(n):
        y0, x0 = rng.integers(0, T // 4, 2)
        y1, x1 = T - rng.integers(0, T // 4, 2)
        grad = np.linspace(0, 255, x1 - x0)[None, :, None] * rng.uniform(0.2, 1.0, 3)[None, None, :]
        noise = rng.integers(-40, 41, (y1 - y0, x1 - x0, 3))
        c[i, y0:y1, x0:x1] = np.clip(grad + noise + rng.integers(0, 80, 3), 0, 255).astype(np.uint8)
        c[i, y0:y0 + 3, x0:x1] = rng.integers(0, 256)                       # a grey band (max == min)
    return c


def order_cases(rng):
    """Every order of the four ops, then every subset (disabled ops as -1 at a random place); random float32 factors
    including 0 and values above 1, hue in [-0.5, 0.5]."""
    cases = [list(p) for p in PERMS]
    for mask in range(16):
        perm = list(PERMS[int(rng.integers(24))])
        cases.append([op if mask >> op & 1 else -1 for op in perm])
    order = np.array(cases, np.int32)
    n = len(order)
    factors = np.stack([rng.uniform(0, 2, n), rng.uniform(0, 2, n), rng.uniform(0, 2, n), rng.uniform(-0.5, 0.5, n)], 1).astype(np.float32)
    factors[::7, :3] = 0.0
    factors[3::11, 3] = 0.5
    factors[5::11, 3] = -0.5
    return order, factors


@pytest.mark.gpu
@pytest.mark.parametrize('T', [64, 100, 101, 224, 256])
def test_kernel_bit_equal_to_torchvision_every_order(T):
    from bpc_baseline_b200 import batched
    rng = np.random.default_rng(T)
    order, factors = order_cases(rng)
    # contrast after hue and after saturation are among the cases
    pos = {op: np.argmax(order == op, axis=1) for op in range(4)}
    assert ((pos[1] > pos[3]) & (order == 3).any(1) & (order == 1).any(1)).any()
    assert ((pos[1] > pos[2]) & (order == 2).any(1) & (order == 1).any(1)).any()
    canv = random_canvases(rng, len(order), T)
    d = lambda a: torch.as_tensor(np.ascontiguousarray(a)).cuda()
    for swap in (False, True):
        got = batched.color_jitter(d(canv), d(order), d(factors), swap_rb=swap).cpu().numpy()
        for i in range(len(order)):
            want = tv_tensor(canv[i], order[i], factors[i], swap)
            assert np.array_equal(got[i].view(np.uint32), want.view(np.uint32)), (T, swap, i, order[i].tolist(), factors[i].tolist())


@pytest.mark.gpu
def test_unaligned_buffers_take_the_scalar_loop_with_the_same_result():
    """T % 4 == 0 but canvases at a 1-byte offset, or out at a 1-float offset: the scalar loop, bit-equal to the
    vectorised one, which the order test pins to torchvision."""
    from bpc_baseline_b200 import batched
    rng = np.random.default_rng(5)
    order, factors = order_cases(rng)
    n, T = len(order), 68
    host = random_canvases(rng, n, T)
    o, f = torch.as_tensor(order).cuda(), torch.as_tensor(factors).cuda()
    want = batched.color_jitter(torch.as_tensor(host).cuda(), o, f)
    raw = torch.empty(host.size + 1, dtype=torch.uint8, device='cuda')
    canv = raw[1:].view(n, T, T, 3)
    canv.copy_(torch.as_tensor(host))
    assert canv.data_ptr() % 16 == 1
    got = batched.color_jitter(canv, o, f)
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    raw_out = torch.empty(n * 3 * T * T + 1, dtype=torch.float32, device='cuda')
    out = raw_out[1:].view(n, 3, T, T)
    batched.color_jitter(torch.as_tensor(host).cuda(), o, f, out=out)
    assert torch.equal(out.view(torch.int32), want.view(torch.int32))
    for i in range(0, n, 9):
        assert np.array_equal(want[i].cpu().numpy().view(np.uint32), tv_tensor(host[i], order[i], factors[i]).view(np.uint32)), i


@pytest.mark.gpu
def test_kernel_on_every_colour():
    """256 canvases of 256 x 256 holding all 2^24 colours, through hue shifts and saturation factors.  Both ops are per
    pixel, so Pillow's reference runs on the whole set as one image."""
    import torchvision.transforms.functional as TF
    from bpc_baseline_b200 import batched
    from oracle.crop import normalise_lut
    rgb = all_colours().reshape(256, 256, 256, 3)
    canv = torch.as_tensor(rgb).cuda()
    lut = torch.as_tensor(normalise_lut()).cuda()
    whole = Image.fromarray(rgb.reshape(256 * 256, 256, 3))
    cases = [([3, -1, -1, -1], (np.nan, np.nan, np.nan, h)) for h in (0.0, 0.1, -0.25, 0.5, -0.5, 1 / 255)]
    cases += [([2, -1, -1, -1], (np.nan, np.nan, s, np.nan)) for s in (0.0, 0.3, 1.0, 1.7)]
    cases += [([2, 3, -1, -1], (np.nan, np.nan, 1.3, 0.37)), ([3, 2, -1, -1], (np.nan, np.nan, 0.6, -0.2))]
    for order, fac in cases:
        fac = np.float32(fac)
        img = whole
        for op in order:
            if op == 2:
                img = TF.adjust_saturation(img, float(fac[2]))
            elif op == 3:
                img = TF.adjust_hue(img, float(fac[3]))
        want_u8 = torch.as_tensor(np.asarray(img).reshape(256, 256, 256, 3).copy()).cuda().long()
        o = torch.tensor([order] * 256, dtype=torch.int32, device='cuda')
        f = torch.tensor(np.tile(fac, (256, 1)), device='cuda')
        got = batched.color_jitter(canv, o, f, lut=lut)
        for c in range(3):
            want = lut[c][want_u8[..., c]]
            assert torch.equal(got[:, c].view(torch.int32), want.view(torch.int32)), (order, fac.tolist(), c)


@pytest.mark.gpu
def test_dataset_crops_with_color_jitter_match_colorjitter(golden_train):
    """dataset_crops(..., jitter, color_jitter) == torchvision's ColorJitter, seeded per sample, on the golden aug_canvas."""
    import torchvision.transforms as T
    import torchvision.transforms.functional as TF
    from bpc_baseline_b200.utils.data_utils import dataset_crops, draw_color_jitter
    g = golden_train
    image, Tsz = g['image'], int(g['T'])
    kw = dict(brightness=0.4, contrast=0.6, saturation=0.7, hue=0.5)
    cj = T.ColorJitter(**kw)
    torch.manual_seed(2024)
    want = np.stack([TF.normalize(TF.to_tensor(np.asarray(cj(Image.fromarray(c)))), MEAN, STD).numpy() for c in g['aug_canvas']])
    torch.manual_seed(2024)
    draws = draw_color_jitter(len(g['bbox']), **kw)
    got = dataset_crops(image[None], g['bbox'], target_size=Tsz, jitter=(g['scale'], g['shift']), color_jitter=draws).cpu().numpy()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    on_dev = tuple(torch.as_tensor(d).cuda() for d in draws)                  # draws already on the device are taken as they are
    got = dataset_crops(image[None], g['bbox'], target_size=Tsz, jitter=(g['scale'], g['shift']), color_jitter=on_dev).cpu().numpy()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


@pytest.mark.gpu
def test_torch_op_equals_batched_and_captures_into_a_graph():
    from bpc_baseline_b200 import batched, ops
    rng = np.random.default_rng(9)
    order, factors = order_cases(rng)
    n = len(order)
    canv = torch.as_tensor(random_canvases(rng, n, 96)).cuda()
    o, f = torch.as_tensor(order).cuda(), torch.as_tensor(factors).cuda()
    want = batched.color_jitter(canv, o, f)
    got = ops.color_jitter(canv, o, f)
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    lut = ops.normalise_lut(canv.device)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.color_jitter(canv, o, f, lut=lut)                  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = ops.color_jitter(canv, o, f, lut=lut)
    canv.copy_(torch.flip(canv, [0]))
    o.copy_(torch.flip(o, [0]))
    f.copy_(torch.flip(f, [0]))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out.view(torch.int32), torch.flip(want, [0]).view(torch.int32))
