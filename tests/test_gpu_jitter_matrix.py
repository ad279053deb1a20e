"""The ColorJitter kernel (``bpc_color_jitter``, csrc/jitter.cu) in every launch regime and at its rounding edges, bit for
bit against Pillow (torchvision's ``ColorJitter`` functional ops on ``Image.fromarray(canvas)``, then to_tensor + normalize).

Launch.  One CTA of 16 warps per crop.  The host code picks the path, the kernel tiles the crop (P = T^2 pixels):

    vec      T % 4 == 0 and both pointers 16-byte aligned: warp w takes tiles w, w + 16, ... of 512 pixels, loading the
             next tile while it converts the current one; tiles = ceil(P / 512) per crop
    scalar   otherwise: one pixel per thread, 512 threads striding over P

``jitter_plan`` restates this.  The regime cells (each with swap_rb = false and true) and the sizes that reach them:

    path     regime                                  last tile   T
    vec      tiles <= 16 (each warp one at most)     partial     4, 8, 20, 88
                                                     whole       64
             16 < tiles < 32 (some warps take two)   partial     92, 124
                                                     whole       96
             tiles >= 32 (every warp two or more)    partial     260, 1020
                                                     whole       128, 224, 256, 512, 1024
    scalar   T % 4 != 0, P < 512 (idle threads)                  1, 2, 3, 5, 22
             T % 4 != 0, P >= 512                                23, 101, 255, 257, 1023
             input misaligned by 1 byte                          64, 224
             out misaligned by 1 float                           64, 224

Program.  Per crop the kernel compiles the order: phase 1 (only with contrast) streams the crop through the ops before
contrast and sums L; phase 2 composes each run of adjacent table ops (brightness, contrast) into one byte table and folds
a run at the end of the chain into the output LUT.  ``jitter_program`` restates this.  The shape cells:

    identity         no op at all (must equal to_tensor + normalize of the canvas)
    fold-all         only table ops: phase 2 is a pure LUT lookup
    lead-table       phase 2 starts with a composed table
    trail-fold       a table run after saturation / hue folded into the LUT
    mid-table        a table step between saturation and hue
    contrast@0       phase 1 with no op before contrast
    contrast@k/op    contrast in slot k = 1, 2, 3 with op (brightness, saturation, hue) before it in phase 1
    none@k           a disabled op (-1, NaN factor) in slot k = 0..3

Every matrix case runs all 40 programs of ``PROGRAMS`` (the 24 orders and the 16 subsets of the four ops) at T <= 260 and
a few of them at T >= 512, with both ``swap_rb`` values, through the default LUT (compared with torchvision's to_tensor +
normalize) and through a random LUT of 768 distinct values with +-0.0, infinities and NaN payloads (compared with
``lut[c][byte]`` of Pillow's bytes).  ``test_matrix_reaches_every_cell`` checks that the cases reach every cell of both
tables; each GPU case asserts its regime from its real pointers.

Arithmetic edges: canvases whose L sum over T^2 sits exactly on a contrast-mean tie k + 0.5 or one unit either side of
it (also above 2^24, where float32 cannot hold the sum, and after brightness, saturation or hue have moved it there);
the blend factors either side of the truncate / clip boundary on every byte and every reachable (L, x) pair; every hue
shift byte a factor in [-0.5, 0.5] gives, from k/255 and its float32 neighbours, on 2^16 colours with greys and near-greys.
"""
import functools
import itertools
import random
from dataclasses import dataclass

import numpy as np
import pytest
import torch

from oracle import jitter_spec as js
from tests.test_color_jitter import MEAN, STD, pil_jitter, random_canvases
from tests.test_gpu_gather_matrix import SENTINEL, random_lut

TILE_PIX = 512
WARPS = 16
THREADS = WARPS * 32
NAMES = ('brightness', 'contrast', 'saturation', 'hue')


# ----------------------------------------------------------------------------------------------------------------------
# restatement of bpc_color_jitter's dispatch and of the kernel's per-crop compilation
# ----------------------------------------------------------------------------------------------------------------------
def jitter_plan(T, in_ptr, out_ptr):
    """The path bpc_color_jitter takes and how the kernel splits one crop."""
    P = T * T
    if T % 4 or in_ptr % 16 or out_ptr % 16:
        reason = 'T % 4' if T % 4 else 'in' if in_ptr % 16 else 'out'
        return {'path': 'scalar', 'reason': reason, 'idle': P < THREADS}
    tiles = -(-P // TILE_PIX)
    regime = 'le16' if tiles <= WARPS else 'lt32' if tiles < 2 * WARPS else 'ge32'
    return {'path': 'vec', 'tiles': tiles, 'regime': regime, 'partial': P % TILE_PIX != 0}


def plan_cell(plan, swap):
    if plan['path'] == 'vec':
        return f'vec<{swap}>', plan['regime'], 'partial' if plan['partial'] else 'whole'
    return f'scalar<{swap}>', plan['reason'], 'idle' if plan['idle'] else 'busy'


REGIME_CELLS = frozenset(
    {(f'vec<{s}>', r, e) for s in (False, True) for r in ('le16', 'lt32', 'ge32') for e in ('partial', 'whole')}
    | {(f'scalar<{s}>', r, e) for s in (False, True) for r, e in (('T % 4', 'idle'), ('T % 4', 'busy'), ('in', 'busy'),
                                                                   ('out', 'busy'))})


def jitter_program(order):
    """What the kernel does for one order: phase 1 (contrast's slot and the ops before it), phase 2's steps after adjacent
    tables are merged, and whether a trailing table run is folded into the LUT."""
    ops = [int(o) if 0 <= o <= 3 else -1 for o in order]
    real = [k for k, o in enumerate(ops) if o >= 0]
    hi = real[-1] + 1 if real else 0
    cpos = ops.index(1) if 1 in ops else -1
    steps, run = [], False
    for o in ops[:hi]:
        if o < 0:
            continue
        if o in (0, 1):
            run = True
            continue
        if run:
            steps.append('table')
            run = False
        steps.append(NAMES[o])
    return {'phase1': cpos >= 0, 'cpos': cpos, 'prefix': tuple(NAMES[o] for o in ops[:max(cpos, 0)] if o >= 0),
            'steps': tuple(steps), 'fold': run}


def shape_cells(order):
    p = jitter_program(order)
    cells = {('none', k) for k, o in enumerate(order) if o < 0}
    if all(o < 0 for o in order):
        cells.add(('identity',))
    if p['fold'] and not p['steps']:
        cells.add(('fold-all',))
    if p['steps'][:1] == ('table',):
        cells.add(('lead-table',))
    if p['fold'] and p['steps']:
        cells.add(('trail-fold',))
    if 'table' in p['steps'][1:-1]:
        cells.add(('mid-table',))
    if p['phase1']:
        cells.add(('contrast', 0) if p['cpos'] == 0 else ('contrast', p['cpos'], None))
        cells |= {('contrast', p['cpos'], op) for op in p['prefix']}
    return cells


SHAPE_CELLS = frozenset({('identity',), ('fold-all',), ('lead-table',), ('trail-fold',), ('mid-table',), ('contrast', 0)}
                        | {('contrast', k, op) for k in (1, 2, 3) for op in ('brightness', 'saturation', 'hue')}
                        | {('contrast', k, None) for k in (1, 2, 3)} | {('none', k) for k in range(4)})

PERMS = list(itertools.permutations(range(4)))
# the 24 orders, then each subset of the ops (mask bit = op) in one of the orders with the disabled ops as -1
PROGRAMS = [list(p) for p in PERMS] + [[o if m >> o & 1 else -1 for o in PERMS[(7 * m + 3) % 24]] for m in range(16)]
# T >= 512: contrast after hue and saturation, a leading, a middle and a trailing table run, -1 slots, contrast alone,
# no op at all
BIG_PROGRAMS = [[3, 2, 1, 0], [0, 1, 2, 3], [2, 0, 1, 3], [-1, 3, -1, 1], [1, -1, -1, -1], [-1, -1, -1, -1]]


# ----------------------------------------------------------------------------------------------------------------------
# the matrix
# ----------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    name: str
    T: int
    cell: tuple          # (path, regime or reason, edge) without the swap
    in_off: int = 0      # byte offset of the canvases inside their buffer
    out_off: int = 0     # float offset of out inside its buffer


VEC_TS = (4, 8, 20, 64, 88, 92, 96, 124, 128, 224, 256, 260, 512, 1020, 1024)
SCALAR_TS = (1, 2, 3, 5, 22, 23, 101, 255, 257, 1023)
CASES = (
    [Case(f'vec-T{T}', T, ('vec',) + plan_cell(jitter_plan(T, 0, 0), 0)[1:]) for T in VEC_TS]
    + [Case(f'scalar-T{T}', T, ('scalar', 'T % 4', 'idle' if T * T < THREADS else 'busy')) for T in SCALAR_TS]
    + [Case(f'scalar-T{T}-in+1', T, ('scalar', 'in', 'busy'), in_off=1) for T in (64, 224)]
    + [Case(f'scalar-T{T}-out+1', T, ('scalar', 'out', 'busy'), out_off=1) for T in (64, 224)]
)


def case_programs(case):
    return BIG_PROGRAMS if case.T >= 512 else PROGRAMS


def draw_factors(rng, order):
    """float32 [n,4]: brightness, contrast, saturation in [0, 2], hue in [-0.5, 0.5]; NaN for the ops an order leaves out."""
    order = np.asarray(order)
    n = len(order)
    f = np.concatenate([rng.uniform(0, 2, (n, 3)), rng.uniform(-0.5, 0.5, (n, 1))], 1).astype(np.float32)
    for op in range(4):
        f[~(order == op).any(1), op] = np.nan
    return f


def canvases(rng, n, T):
    """uint8 [n,T,T,3]: letterbox-like canvases and byte noise alternately (noise only below T = 8)."""
    c = rng.integers(0, 256, (n, T, T, 3), dtype=np.uint8)
    if T >= 8:
        c[::2] = random_canvases(rng, len(c[::2]), T)
    return c


@functools.lru_cache(maxsize=None)
def case_data(case):
    """(canvases, order, factors, Pillow's jittered bytes) of a case, shared by its four runs."""
    rng = np.random.default_rng([case.T, case.in_off, case.out_off])
    order = np.array(case_programs(case), np.int32)
    factors = draw_factors(rng, order)
    canv = canvases(rng, len(order), case.T)
    return canv, order, factors, np.stack([pil_jitter(c, o, f) for c, o, f in zip(canv, order, factors)])


def expected(pil, lut, swap):
    """float32 [n,3,T,T] from Pillow's bytes: to_tensor + normalize for the default LUT (lut None), else lut[c][byte]."""
    import torchvision.transforms.functional as TF
    if swap:
        pil = pil[..., ::-1]
    if lut is None:
        return np.stack([TF.normalize(TF.to_tensor(np.ascontiguousarray(a)), MEAN, STD).numpy() for a in pil])
    return np.stack([lut[c][pil[..., c]] for c in range(3)], axis=1)


# ----------------------------------------------------------------------------------------------------------------------
# CPU part
# ----------------------------------------------------------------------------------------------------------------------
def test_plan_restatement():
    vec = {T: jitter_plan(T, 0, 0) for T in VEC_TS}
    assert {T: p['tiles'] for T, p in vec.items()} == {4: 1, 8: 1, 20: 1, 64: 8, 88: 16, 92: 17, 96: 18, 124: 31, 128: 32,
                                                       224: 98, 256: 128, 260: 133, 512: 512, 1020: 2033, 1024: 2048}
    assert sorted(T for T, p in vec.items() if p['partial']) == [4, 8, 20, 88, 92, 124, 260, 1020]
    assert {T: jitter_plan(T, 0, 0)['idle'] for T in SCALAR_TS} == {T: T <= 22 for T in SCALAR_TS}
    assert jitter_plan(64, 1, 0)['reason'] == 'in' and jitter_plan(64, 0, 4)['reason'] == 'out'
    assert jitter_plan(64, 16, 32)['path'] == 'vec' and jitter_plan(66, 0, 0)['reason'] == 'T % 4'


def test_program_restatement():
    p = jitter_program
    assert p([-1] * 4) == {'phase1': False, 'cpos': -1, 'prefix': (), 'steps': (), 'fold': False}
    assert p([0, -1, 1, -1]) == {'phase1': True, 'cpos': 2, 'prefix': ('brightness',), 'steps': (), 'fold': True}
    assert p([0, 1, 2, 3])['steps'] == ('table', 'saturation', 'hue') and not p([0, 1, 2, 3])['fold']
    assert p([2, 3, 0, 1])['steps'] == ('saturation', 'hue') and p([2, 3, 0, 1])['fold']
    assert p([2, 0, 1, 3])['steps'] == ('saturation', 'table', 'hue')
    assert p([3, 2, 1, 0])['prefix'] == ('hue', 'saturation') and p([3, 2, 1, 0])['cpos'] == 2
    assert p([2, -1, 3, -1])['steps'] == ('saturation', 'hue') and not p([2, -1, 3, -1])['fold']


def test_matrix_reaches_every_cell():
    """Each case claims the regime the restated plan gives its pointers, and the cases reach every regime cell with both
    channel orders and every program-shape cell."""
    regimes, shapes = set(), set()
    for case in CASES:
        for swap in (False, True):
            plan = jitter_plan(case.T, 256 + case.in_off, 1 << 20 | 4 * case.out_off)
            cell = plan_cell(plan, swap)
            assert (cell[0].split('<')[0],) + cell[1:] == case.cell, (case.name, plan)
            regimes.add(cell)
        for order in case_programs(case):
            shapes |= shape_cells(order)
    assert regimes == REGIME_CELLS, sorted(REGIME_CELLS ^ regimes)
    assert shapes == SHAPE_CELLS, sorted(SHAPE_CELLS ^ shapes, key=str)
    assert all(shape_cells(o) <= SHAPE_CELLS for o in BIG_PROGRAMS)


# ---- contrast-mean ties ----------------------------------------------------------------------------------------------
TIE_KS = {2: (100, 101), 64: (40, 41), 256: (126, 127), 1024: (16, 17)}
PREFIX_FACTOR = {None: None, 0: np.float32(0.77), 2: np.float32(1.6), 3: np.float32(0.23)}
TIE_CONTRAST = np.float32(0.6)


def _prefix(img, op):
    return img if op is None else js.apply_op(img, op, PREFIX_FACTOR[op])


def tie_canvas(T, k, delta, op):
    """uint8 [T,T,3] whose L sum, after the prefix op, is (k + 0.5) T^2 + delta.  Half the pixels are colours near level k
    (before brightness, near k / 0.77), half are greys: every prefix op maps a grey to a grey, so the greys make up the
    exact remainder."""
    rng = np.random.default_rng([T, k, delta + 1, 4 if op is None else op])
    P = T * T
    m = P // 2
    target = (2 * k + 1) * P // 2 + delta
    level = k / PREFIX_FACTOR[0] if op == 0 else k
    colour = np.clip(round(level) + rng.integers(-8, 9, (P - m, 3)), 0, 255).astype(np.uint8)
    grey = np.repeat(np.arange(256, dtype=np.uint8)[:, None], 3, 1)
    gmap = js.luma(_prefix(grey[None], op))[0].astype(np.int64)           # grey g -> its L after the prefix
    rest = target - int(js.luma(_prefix(colour[None], op)).astype(np.int64).sum())
    base, extra = divmod(rest, m)
    inv = {int(v): g for g, v in reversed(list(enumerate(gmap)))}        # the smallest grey giving each L
    assert base in inv and base + 1 in inv, (T, k, delta, op, base)
    greys = np.array([inv[base]] * (m - extra) + [inv[base + 1]] * extra, np.uint8)
    px = np.concatenate([colour, np.repeat(greys[:, None], 3, 1)])
    return px[rng.permutation(P)].reshape(T, T, 3)


@functools.lru_cache(maxsize=None)
def tie_cases(T):
    """(canvases, order, factors, the mean Pillow must take) for every k of TIE_KS[T], delta and prefix op."""
    canv, order, factors, means = [], [], [], []
    for k, delta, op in itertools.product(TIE_KS[T], (-1, 0, 1), PREFIX_FACTOR):
        canv.append(tie_canvas(T, k, delta, op))
        order.append([1, -1, -1, -1] if op is None else [op, 1, -1, -1])
        f = np.full(4, np.nan, np.float32)
        f[1] = TIE_CONTRAST
        if op is not None:
            f[op] = PREFIX_FACTOR[op]
        factors.append(f)
        means.append((k, delta, op, k + (delta >= 0)))
    return np.stack(canv), np.array(order, np.int32), np.stack(factors), means


@pytest.mark.parametrize('T', sorted(TIE_KS))
def test_tie_canvases_hit_their_ties(T):
    """The spec's image after the prefix op sums to (k + 0.5) T^2 + delta exactly, and ImageStat's mean rounds as intended."""
    canv, _, _, means = tie_cases(T)
    P = T * T
    for c, (k, delta, op, mean) in zip(canv, means):
        img = _prefix(c, op)
        total = int(js.luma(img).astype(np.int64).sum())
        assert total == (2 * k + 1) * P // 2 + delta, (k, delta, op)
        assert js.contrast_mean(img) == mean, (k, delta, op)
        if T == 1024:
            assert total > 1 << 24
            # a float32 mean, int(float(total) / float(P) + 0.5f), rounds the sum below the tie up onto it
            f32 = int(np.float32(total) / np.float32(P) + np.float32(0.5))
            assert f32 == (k + 1 if delta == -1 else mean), (k, delta, f32)


# ---- blend boundary --------------------------------------------------------------------------------------------------
ALPHAS = np.float32([0, 2 ** -24, 0.5, 1 - 2 ** -24, 1, 1 + 2 ** -23, 1.7, 2, 10])
RAMP_FILLS = (0, 37, 90, 128, 200, 255)


def ramp_canvas(fill):
    """uint8 [32,32,3]: 256 pixels holding every byte in every channel, then 768 pixels of grey ``fill`` to move the mean."""
    i = np.arange(256)
    ramp = np.stack([i, (97 * i + 13) % 256, (181 * i + 7) % 256], -1)
    return np.concatenate([ramp, np.full((768, 3), fill)]).astype(np.uint8).reshape(32, 32, 3)


def _luma_all():
    k = np.arange(1 << 24, dtype=np.int32)
    ch = [(k >> 16) & 255, (k >> 8) & 255, k & 255]
    return k, ch, (ch[0] * 19595 + ch[1] * 38470 + ch[2] * 7471 + 0x8000) >> 16


@functools.lru_cache(maxsize=None)
def saturation_canvases():
    """uint8 [m,256,256,3]: for every channel c and every (L, x) such that some colour has luma L and channel c equal to x,
    one such colour (131 328 pairs, 103 891 colours), padded by repetition."""
    k, ch, L = _luma_all()
    wit = []
    for c in range(3):
        w = np.full(1 << 16, -1, np.int32)
        w[L * 256 + ch[c]] = k                       # one colour per (L, x); which one does not matter
        wit.append(w[w >= 0])
    cols = np.unique(np.concatenate(wit))
    rgb = np.stack([(cols >> 16) & 255, (cols >> 8) & 255, cols & 255], -1).astype(np.uint8)
    m = -(-len(rgb) // 65536)
    return np.resize(rgb, (m * 65536, 3)).reshape(m, 256, 256, 3)


def test_saturation_canvases_hold_every_reachable_pair():
    _, ch, L = _luma_all()
    px = saturation_canvases().reshape(-1, 3).astype(np.int64)
    Lc = js.luma(px).astype(np.int64)
    for c in range(3):
        assert np.array_equal(np.unique(Lc * 256 + px[:, c]), np.unique(L * 256 + ch[c])), c
    for fill in RAMP_FILLS:
        assert all(len(np.unique(ramp_canvas(fill)[..., c])) == 256 for c in range(3))


def blend_cases():
    """(canvases, order, factors): brightness and contrast on the ramp canvases, folded into the LUT ([op]) and as a phase-2
    table ([op, saturation 1]); saturation on the witness colours, alone and before an identity brightness table."""
    canv, order, factors = [], [], []
    for op, a, fill in itertools.product((0, 1), ALPHAS, RAMP_FILLS):
        for o in ([op, -1, -1, -1], [op, 2, -1, -1]):
            canv.append(ramp_canvas(fill))
            order.append(o)
            f = np.full(4, np.nan, np.float32)
            f[op] = a
            if 2 in o:
                f[2] = 1.0
            factors.append(f)
    small = (np.stack(canv), np.array(order, np.int32), np.stack(factors))
    sat = saturation_canvases()
    canv, order, factors = [], [], []
    for a in ALPHAS:
        for o in ([2, -1, -1, -1], [-1, 2, 0, -1]):
            for c in sat:
                canv.append(c)
                order.append(o)
                factors.append(np.float32([1.0 if 0 in o else np.nan, np.nan, a, np.nan]))
    return small, (np.stack(canv), np.array(order, np.int32), np.stack(factors))


# ---- hue shift bytes -------------------------------------------------------------------------------------------------
def hue_factors():
    """float32: k/255 for k = -127..127 and its float32 neighbours on both sides, and +-0.5."""
    f = []
    for k in range(-127, 128):
        f0 = np.float32(k / 255)
        f += [np.nextafter(f0, np.float32(-1)), f0, np.nextafter(f0, np.float32(1))]
    return np.float32(f + [0.5, -0.5])


@functools.lru_cache(maxsize=None)
def hue_colours():
    """uint8 [256,256,3]: the 256 greys, every near-grey (channels v and v +- 1) and random colours, 2^16 in all."""
    v = np.arange(256)
    near = [np.stack([v, v, v], -1)]
    for d in itertools.product((-1, 0, 1), repeat=3):
        if any(d):
            near.append(np.stack([v + d[0], v + d[1], v + d[2]], -1))
    near = np.concatenate(near)
    near = near[(near >= 0).all(1) & (near <= 255).all(1)]
    rnd = np.random.default_rng(31).integers(0, 256, (65536 - len(near), 3))
    return np.concatenate([near, rnd]).astype(np.uint8).reshape(256, 256, 3)


def test_hue_factors_reach_every_shift_byte():
    """Every byte but 128, which no factor in [-0.5, 0.5] gives (|int32(f * 255)| <= 127)."""
    f = hue_factors()
    assert ((f >= -0.5) & (f <= 0.5)).all()
    assert {js.hue_shift(x) for x in f} == set(range(256)) - {128}
    below = [js.hue_shift(x) for x in f[0:-2:3]]
    assert below != [js.hue_shift(x) for x in f[1:-2:3]]      # the lower neighbours change the byte for some k
    c = hue_colours().reshape(-1, 3).astype(np.int64)
    assert len(c) == 65536 and (np.ptp(c, 1) == 0).sum() >= 256 and (np.ptp(c, 1) == 1).sum() >= 1500


# ----------------------------------------------------------------------------------------------------------------------
# GPU part
# ----------------------------------------------------------------------------------------------------------------------
_LUT = {}


def _lut(kind):
    """(device LUT or None for the default one, host LUT or None)."""
    if kind == 'default':
        return None, None
    if 'dev' not in _LUT:
        _LUT['host'] = random_lut()
        _LUT['dev'] = torch.as_tensor(_LUT['host']).cuda()
    return _LUT['dev'], _LUT['host']


def _dev(a, off=0):
    """A contiguous device copy of ``a`` that starts ``off`` bytes into its own buffer."""
    a = np.ascontiguousarray(a)
    raw = torch.empty(a.nbytes + off, dtype=torch.uint8, device='cuda')
    t = raw[off:].view(torch.from_numpy(a).dtype).view(a.shape)
    t.copy_(torch.from_numpy(a))
    return t


def _sentinel_rows(rows, T, off=0):
    buf = torch.full((rows * 3 * T * T + off,), SENTINEL, dtype=torch.int32, device='cuda')
    return buf[off:].view(torch.float32).view(rows, 3, T, T), buf


def _assert_bits_equal(got, want, order, factors, what):
    a, b = np.ascontiguousarray(got).view(np.uint32), np.ascontiguousarray(want).view(np.uint32)
    bad = [i for i in range(len(a)) if not np.array_equal(a[i], b[i])]
    if bad:
        i = bad[0]
        pytest.fail(f'{what}: crops {bad[:8]} differ from Pillow, first order {order[i].tolist()} factors {factors[i].tolist()}')


def _jitter(canv, order, factors, swap=False, lut=None, out=None):
    from bpc_baseline_b200 import batched
    return batched.color_jitter(canv, _dev(order), _dev(factors), swap_rb=swap, lut=lut, out=out)


@pytest.mark.gpu
@pytest.mark.parametrize('lut_kind', ['default', 'random'])
@pytest.mark.parametrize('swap', [False, True])
@pytest.mark.parametrize('case', CASES, ids=[c.name for c in CASES])
def test_matrix_case(case, swap, lut_kind):
    host, order, factors, pil = case_data(case)
    n, T = len(order), case.T
    canv = _dev(host, case.in_off)
    out, buf = _sentinel_rows(n, T, case.out_off)
    plan = jitter_plan(T, canv.data_ptr(), out.data_ptr())
    assert plan_cell(plan, swap) == (f'{case.cell[0]}<{swap}>',) + case.cell[1:], (case.name, plan)
    lut_d, lut_h = _lut(lut_kind)
    got = _jitter(canv, order, factors, swap, lut_d, out)
    assert got.data_ptr() == out.data_ptr()
    _assert_bits_equal(out.cpu().numpy(), expected(pil, lut_h, swap), order, factors, f'{case.name} swap={swap} {lut_kind}')
    assert bool((buf[:case.out_off] == SENTINEL).all())


@pytest.mark.gpu
@pytest.mark.parametrize('T', sorted(TIE_KS))
def test_contrast_mean_ties(T):
    """The kernel takes the mean Pillow takes on every tie canvas: half away from zero on the tie, the exact double
    quotient one unit either side of it, with the sum above 2^24 at T = 1024."""
    canv, order, factors, means = tie_cases(T)
    pil = np.stack([pil_jitter(c, o, f) for c, o, f in zip(canv, order, factors)])
    got = _jitter(_dev(canv), order, factors).cpu().numpy()
    want = expected(pil, None, False)
    bad = [means[i][:3] for i in range(len(canv)) if not np.array_equal(got[i].view(np.uint32), want[i].view(np.uint32))]
    assert not bad, f'(k, delta, prefix op) of the canvases that differ: {bad}'


@pytest.mark.gpu
def test_blend_boundary():
    """Brightness, contrast and saturation at alpha in {0, 2^-24, 0.5, 1 - 2^-24, 1, 1 + 2^-23, 1.7, 2, 10} on every byte
    (for contrast at six means) and every reachable (L, x) pair of saturation."""
    lut_d, lut_h = _lut('random')
    for canv, order, factors in blend_cases():
        pil = np.stack([pil_jitter(c, o, f) for c, o, f in zip(canv, order, factors)])
        got = _jitter(_dev(canv), order, factors, lut=lut_d).cpu().numpy()
        _assert_bits_equal(got, expected(pil, lut_h, False), order, factors, f'T={canv.shape[1]}')


@pytest.mark.gpu
def test_hue_every_shift_byte():
    """[hue] with each factor of hue_factors() on the same 2^16 colours, in launches of 128 crops."""
    import torchvision.transforms.functional as TF
    from PIL import Image
    lut_d, lut_h = _lut('random')
    colours = hue_colours()
    img = Image.fromarray(colours)
    fac = hue_factors()
    canv = _dev(np.broadcast_to(colours, (128, 256, 256, 3)))
    for lo in range(0, len(fac), 128):
        f = fac[lo:lo + 128]
        factors = np.full((len(f), 4), np.nan, np.float32)
        factors[:, 3] = f
        order = np.tile(np.int32([3, -1, -1, -1]), (len(f), 1))
        got = _jitter(canv[:len(f)], order, factors, lut=lut_d).cpu().numpy()
        pil = np.stack([np.asarray(TF.adjust_hue(img, float(x))) for x in f])
        _assert_bits_equal(got, expected(pil, lut_h, False), order, factors, f'hue factors from {lo}')


@pytest.mark.gpu
def test_no_crops_launches_nothing():
    from bpc_baseline_b200 import _lib
    T = 64
    empty = torch.empty((0, T, T, 3), dtype=torch.uint8, device='cuda')
    order, factors = np.zeros((0, 4), np.int32), np.zeros((0, 4), np.float32)
    before = _lib.launch_count()
    got = _jitter(empty, order, factors)
    assert tuple(got.shape) == (0, 3, T, T)
    out, buf = _sentinel_rows(2, T)
    assert _jitter(empty, order, factors, out=out).data_ptr() == out.data_ptr()
    torch.cuda.synchronize()
    assert _lib.launch_count() == before and bool((buf == SENTINEL).all())


@pytest.mark.gpu
@pytest.mark.parametrize('T', [100, 101])
def test_one_crop(T):
    rng = np.random.default_rng(T)
    order = np.int32([[3, 2, 1, 0]])
    factors = draw_factors(rng, order)
    canv = canvases(rng, 1, T)
    lut_d, lut_h = _lut('random')
    got = _jitter(_dev(canv), order, factors, lut=lut_d).cpu().numpy()
    _assert_bits_equal(got, expected(pil_jitter(canv[0], order[0], factors[0])[None], lut_h, False), order, factors, f'T={T}')


@pytest.mark.gpu
@pytest.mark.parametrize('T', [100, 37])
def test_out_row_offset_with_spare_rows(T):
    """``out`` is a view starting two rows into a sentinel buffer with three rows to spare: those five rows keep the
    sentinel (T = 100 keeps the vectorised path, T = 37 takes the scalar one)."""
    rng = np.random.default_rng(T + 1)
    order = np.array(PROGRAMS[::5], np.int32)
    factors = draw_factors(rng, order)
    canv = canvases(rng, len(order), T)
    n = len(order)
    big, buf = _sentinel_rows(2 + n + 3, T)
    out = big[2:]
    assert jitter_plan(T, 0, out.data_ptr())['path'] == ('vec' if T % 4 == 0 else 'scalar')
    _jitter(_dev(canv), order, factors, swap=True, out=out)
    pil = np.stack([pil_jitter(c, o, f) for c, o, f in zip(canv, order, factors)])
    _assert_bits_equal(out[:n].cpu().numpy(), expected(pil, None, True), order, factors, f'T={T}')
    assert bool((big[:2].view(torch.int32) == SENTINEL).all()) and bool((big[2 + n:].view(torch.int32) == SENTINEL).all())


@pytest.mark.gpu
def test_large_launch_past_2_31_bytes():
    """700 distinct crops at T = 1024: the input offset crop * 3 T^2 passes 2^31 from crop 683 on (the output offset from
    crop 171 on).  Crops on both sides of that line and the last three match Pillow; no crop equals its neighbour."""
    T, n = 1024, 700
    assert 682 * 3 * T * T < 1 << 31 <= 683 * 3 * T * T
    rng = np.random.default_rng(700)
    order = np.array([PROGRAMS[i % len(PROGRAMS)] for i in range(n)], np.int32)
    factors = draw_factors(rng, order)
    g = torch.Generator(device='cuda').manual_seed(700)
    canv = out = None
    try:
        canv = torch.randint(0, 256, (n, T, T, 3), dtype=torch.uint8, device='cuda', generator=g)
        out = _jitter(canv, order, factors)
        check = [0, 682, 683, n - 3, n - 2, n - 1]
        host = canv[check].cpu().numpy()
        got = out[check].cpu().numpy()
        same = [i for i in range(n - 1) if torch.equal(out[i], out[i + 1])]
    finally:
        del canv, out
        torch.cuda.empty_cache()
    pil = np.stack([pil_jitter(c, order[i], factors[i]) for c, i in zip(host, check)])
    _assert_bits_equal(got, expected(pil, None, False), order[check], factors[check], 'T=1024 n=700')
    assert not same, f'crops equal to the next one: {same[:8]}'


@pytest.mark.gpu
@pytest.mark.parametrize('jittered', [False, True])
@pytest.mark.parametrize('T', [1, 37, 100, 256, 512])
def test_dataset_crops_against_colorjitter(T, jittered):
    """dataset_crops(images, boxes, image_index, jitter, color_jitter) == cv2 letterbox canvas (oracle.crop), then
    torchvision's ColorJitter seeded as the draws, then to_tensor + normalize."""
    import torchvision.transforms as TT
    import torchvision.transforms.functional as TF
    from PIL import Image

    from bpc_baseline_b200 import synth
    from bpc_baseline_b200.utils.data_utils import dataset_crops, draw_color_jitter, draw_crop_jitter
    from oracle import crop as ocrop
    images = synth.make_images(3, seed=T, width=320, height=240)
    B, H, W, _ = images.shape
    rng = np.random.default_rng([T, jittered])
    n = 4 if T >= 256 else 8
    w = rng.integers(12, 160, n)
    h = np.clip((w * rng.uniform(0.8, 1.25, n)).astype(int), 10, H - 1)    # letterboxed to T = 1, no side rounds to 0
    bbox = np.stack([rng.integers(0, W - w), rng.integers(0, H - h), w, h], 1).astype(np.int32)
    idx = rng.integers(0, B, n).astype(np.int32)
    jitter = draw_crop_jitter(bbox, rnd=random.Random(T)) if jittered else None
    kw = dict(brightness=0.4, contrast=0.6, saturation=0.7, hue=0.5)
    torch.manual_seed(T)
    draws = draw_color_jitter(n, **kw)
    got = dataset_crops(images, bbox, image_index=idx, target_size=T, jitter=jitter, color_jitter=draws).cpu().numpy()
    cj = TT.ColorJitter(**kw)
    torch.manual_seed(T)
    for r in range(n):
        win = ocrop.dataset_window(bbox[r], W, H, *((jitter[0][r], jitter[1][r]) if jittered else ()))
        canvas = ocrop.crop_u8_ref(images[idx[r]], win, T)
        want = TF.normalize(TF.to_tensor(np.asarray(cj(Image.fromarray(canvas)))), MEAN, STD).numpy()
        assert np.array_equal(got[r].view(np.uint32), want.view(np.uint32)), (T, jittered, r, draws[0][r].tolist())


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['scalar-T3', 'vec-T92', 'scalar-T64-in+1', 'vec-T1020'])
def test_torch_op_equals_batched(name):
    from bpc_baseline_b200 import batched, ops
    case = next(c for c in CASES if c.name == name)
    host, order, factors, _ = case_data(case)
    canv, o, f = _dev(host, case.in_off), _dev(order), _dev(factors)
    for swap, kind in ((False, 'default'), (True, 'random')):
        lut = _lut(kind)[0]
        want = batched.color_jitter(canv, o, f, swap_rb=swap, lut=lut)
        got = ops.color_jitter(canv, o, f, swap_rb=swap, lut=lut)
        assert torch.equal(got.view(torch.int32), want.view(torch.int32)), (name, swap, kind)
