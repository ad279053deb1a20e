"""The receiver kernel of the crop gather (``bpc_crops_normalise``, csrc/gather.cu) in every launch regime on one GPU.

The host code of ``bpc_crops_normalise`` picks the kernel and the order in which it walks the crops:

    n_src > 16 or T outside 1..256: BPC_EINVAL     total > 2^24: BPC_ETOOBIG     total == 0: no launch
    fast = T % 4 == 0 and out and every source pointer are 16-byte aligned
    fast:  bpc_crops_normalise_kernel<swap_rb>  ("tiled")  one warp per 512-pixel tile, tiles = ceil(T^2 / 512) per crop,
           items = total x tiles, grid = min(ceil(items / 8), SMs x occupancy) CTAs of 8 warps, item stride 8 x grid.
           walk = round_robin (crop k of source 0, of source 1, ...) if n_src > 1 and all counts are equal, else concat
    else:  bpc_crops_normalise_any_kernel       ("scalar") one thread per output float, items = total x 3 T^2,
           SMs x 8 CTAs of 256 threads, walk = concat

A CTA of 256 threads fits at most 8 times on an SM, so the number of tiled warps lies between min(items, 8 x SMs) and
64 x SMs whatever the occupancy: every warp takes one tile at most when items <= 8 x SMs ("one" pass), and every warp
takes at least two when items >= 128 x SMs ("several" passes; the loop's look-ahead and the reuse of the per-warp stage
only run there).  ``gather_plan`` restates this; ``REGIMES`` is the table of (kernel, walk, passes) cells, 10 in all:

    kernel, walk               one pass                                  several passes
    tiled<swap>, concat        T = 4, 8, 12, 100, 224, 252, 256;         the same T; 16 sources with empty ones
                               3 and 16 sources with empty ones;
                               out as a row offset with rows to spare
    tiled<swap>, round_robin   2, 3, 8, 16 equal sources                 the same; 2 x 4 096 and 8 x 1 024 crops at
                                                                         T = 224; 16 x 2^20 crops at T = 4
    scalar, concat             T = 1, 2, 3, 6; T = 64 with a source      T = 37, 97, 255; T = 224 misaligned as at
                               misaligned by 1, 4 or 8 bytes, or out     T = 64; 2^24 crops at T = 1
                               by one float

(swap = false and true, as ``swap_rb`` throughout).  Every case asserts the cell it claims against the plan computed from its actual
pointers and the device's SM count; ``test_matrix_reaches_every_regime`` checks that the cases cover the table, and
``test_kernel_names_under_the_profiler`` that the plan's kernel is the one launched.

Reference: ``out[c, p] = lut[p][u8[c, ..., 2 - p if swap else p]]`` by torch indexing on the device (NumPy for a few
small cases), compared bit for bit.  The LUT holds 768 distinct bit patterns including +0.0, -0.0, +-inf, a quiet NaN
and a signalling NaN with payloads, so a wrong plane, channel or LUT row, or a copy that goes through float arithmetic,
shows.  Every source has its own random bytes, so a crop written to the wrong slot shows too.  ``out`` starts as a
NaN sentinel that no LUT entry has; rows the kernel must not write keep it.
"""
import ctypes as C
from dataclasses import dataclass

import numpy as np
import pytest
import torch

TILE_PIX = 512
GATHER_WARPS = 8
MAX_CTAS_PER_SM = 2048 // (GATHER_WARPS * 32)       # 8 CTAs of 256 threads
SCALAR_THREADS_PER_SM = 8 * 256
MAX_SRC = 16
MAX_TOTAL = 1 << 24
SENTINEL = 0x7F80DEAD                               # a signalling-NaN pattern absent from the LUT
BPC_EINVAL, BPC_ETOOBIG = -1, -4


# ----------------------------------------------------------------------------------------------------------------------
# restatement of the host code of bpc_crops_normalise
# ----------------------------------------------------------------------------------------------------------------------
def gather_plan(T, src_ptrs, counts, out_ptr, sms, swap=True):
    """What bpc_crops_normalise launches: {'status'} for a refused call or one without a launch, else the kernel
    ('tiled<false>', 'tiled<true>' or 'scalar'), the walk, tiles per crop, items, and whether every warp (thread) of the
    grid takes at most one item ('one_pass') or some warp must take more than one ('multi_pass')."""
    n_src = len(counts)
    if n_src > MAX_SRC or not 1 <= T <= 256:
        return {'status': 'EINVAL'}
    if n_src == 0:
        return {'status': 'no launch'}
    if any(c < 0 or (c > 0 and not src_ptrs[s]) for s, c in enumerate(counts)):
        return {'status': 'EINVAL'}
    total = sum(counts)
    if total > MAX_TOTAL:
        return {'status': 'ETOOBIG'}
    if total == 0:
        return {'status': 'no launch'}
    fast = T % 4 == 0 and out_ptr % 16 == 0 and all((p or 0) % 16 == 0 for p in src_ptrs)
    if fast:
        tiles = -(-T * T // TILE_PIX)
        items = total * tiles
        equal = n_src > 1 and all(c == counts[0] for c in counts)
        return {'status': 'ok', 'kernel': f'tiled<{str(bool(swap)).lower()}>', 'walk': 'round_robin' if equal else 'concat',
                'tiles': tiles, 'items': items, 'one_pass': items <= GATHER_WARPS * sms,
                'multi_pass': items > GATHER_WARPS * MAX_CTAS_PER_SM * sms}
    items = total * 3 * T * T
    threads = SCALAR_THREADS_PER_SM * sms
    return {'status': 'ok', 'kernel': 'scalar', 'walk': 'concat', 'tiles': None, 'items': items,
            'one_pass': items <= threads, 'multi_pass': items > threads}


def plan_cell(plan):
    return plan['kernel'], plan['walk'], 'one' if plan['one_pass'] else 'several' if plan['multi_pass'] else 'either'


REGIMES = frozenset({(f'tiled<{sw}>', walk, passes) for sw in ('false', 'true') for walk in ('concat', 'round_robin')
                     for passes in ('one', 'several')} | {('scalar', 'concat', 'one'), ('scalar', 'concat', 'several')})


def kernel_symbol(kernel):
    return 'bpc_crops_normalise_any_kernel' if kernel == 'scalar' else kernel.replace('tiled', 'bpc_crops_normalise_kernel')


# ----------------------------------------------------------------------------------------------------------------------
# the matrix
# ----------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    name: str
    T: int
    counts: tuple            # crops per source ('several' cases with scale=True multiply them up to the regime)
    kernel: str              # 'tiled' or 'scalar'
    walk: str
    passes: str              # 'one' or 'several'
    scale: bool = True
    src_off: tuple = ()      # byte offset of each source inside its own buffer
    out_off: int = 0         # float offset of out inside its buffer
    lead: int = 0            # sentinel rows in front of out
    tail: int = 1            # rows of out beyond the crops


TILED_TS = (4, 8, 12, 100, 224, 252, 256)
SCALAR_TS = (1, 2, 3, 6, 37, 97, 255)
CONCAT16 = (0, 3, 1, 0, 2, 5, 0, 1, 4, 2, 0, 3, 1, 1, 2, 0)
CASES = (
    [Case(f'tiled-T{T}-one', T, (37,) if T <= 12 else (5,), 'tiled', 'concat', 'one') for T in TILED_TS]
    + [Case(f'tiled-T{T}-several', T, (3,), 'tiled', 'concat', 'several') for T in TILED_TS]
    + [Case('concat3-empty-first', 100, (0, 5, 4), 'tiled', 'concat', 'one'),
       Case('concat3-empty-middle', 100, (5, 0, 4), 'tiled', 'concat', 'one'),
       Case('concat3-empty-last', 100, (5, 4, 0), 'tiled', 'concat', 'one'),
       Case('concat16-one', 100, CONCAT16, 'tiled', 'concat', 'one'),
       Case('concat16-several', 100, CONCAT16, 'tiled', 'concat', 'several')]
    + [Case(f'rr{n}-one', 100, (c,) * n, 'tiled', 'round_robin', 'one') for n, c in ((2, 3), (3, 2), (8, 2), (16, 2))]
    + [Case(f'rr{n}-several', 100, (1,) * n, 'tiled', 'round_robin', 'several') for n in (2, 3, 8, 16)]
    + [Case('rr2x4096-T224', 224, (4096,) * 2, 'tiled', 'round_robin', 'several', scale=False),
       Case('rr8x1024-T224', 224, (1024,) * 8, 'tiled', 'round_robin', 'several', scale=False)]
    + [Case(f'scalar-T{T}', T, (2, 0, 3), 'scalar', 'concat', 'one' if T <= 6 else 'several') for T in SCALAR_TS]
    + [Case(f'scalar-T{T}-src+{off}', T, (3, 3), 'scalar', 'concat', 'one' if T == 64 else 'several', scale=False,
            src_off=(0, off)) for T in (64, 224) for off in (1, 4, 8)]
    + [Case(f'scalar-T{T}-out+1', T, (1, 2), 'scalar', 'concat', 'one' if T == 64 else 'several', scale=False, out_off=1)
       for T in (64, 224)]
    + [Case('tiled-T100-out-rows', 100, (2, 3), 'tiled', 'concat', 'one', lead=2, tail=3),
       Case('rr3-T64-out-rows', 64, (3, 3, 3), 'tiled', 'round_robin', 'one', lead=1, tail=4),
       Case('scalar-T37-out-rows', 37, (2, 3), 'scalar', 'concat', 'one', lead=2, tail=3)]
)


def case_counts(case, sms):
    """Per-source counts at this SM count.  'several' cases are scaled until every warp (thread) takes at least two items,
    with an item count that is not a multiple of any possible warp count."""
    counts = list(case.counts)
    if case.passes != 'several' or not case.scale:
        return counts
    per = -(-case.T * case.T // TILE_PIX) if case.kernel == 'tiled' else 3 * case.T * case.T
    units = GATHER_WARPS * MAX_CTAS_PER_SM * sms if case.kernel == 'tiled' else SCALAR_THREADS_PER_SM * sms
    m = -(-(2 * units) // (sum(counts) * per))
    counts = [c * m for c in counts]
    if case.kernel == 'tiled':
        while any(sum(counts) * per % (GATHER_WARPS * k * sms) == 0 for k in range(1, MAX_CTAS_PER_SM + 1)):
            counts = [c + 1 if c else 0 for c in counts]
    return counts


def fake_ptrs(case, counts):
    base = 1 << 20
    src = [base * (s + 1) + (case.src_off[s] if s < len(case.src_off) else 0) if c else None for s, c in enumerate(counts)]
    return src, base * 64 + case.lead * 12 * case.T * case.T + 4 * case.out_off


def check_claim(case, plan, sms):
    assert plan['status'] == 'ok', (case.name, plan)
    assert plan['kernel'].startswith(case.kernel) and plan['walk'] == case.walk, (case.name, plan)
    if case.passes == 'one':
        assert plan['one_pass'], (case.name, plan)
    else:
        assert plan['multi_pass'], (case.name, plan)
        if case.scale:
            units = GATHER_WARPS * MAX_CTAS_PER_SM * sms if case.kernel == 'tiled' else SCALAR_THREADS_PER_SM * sms
            assert plan['items'] >= 2 * units, (case.name, plan)


def random_lut(seed=2024):
    """float32 [3,256]: 768 distinct bit patterns, with +0.0, -0.0, +inf, -inf and two NaNs with payloads."""
    rng = np.random.default_rng(seed)
    v = rng.uniform(-60.0, 60.0, 4096).astype(np.float32)
    v = v[v != 0]
    _, first = np.unique(v.view(np.uint32), return_index=True)
    v = v[np.sort(first)][:768].reshape(3, 256).copy()
    bits = v.view(np.uint32)
    bits[0, 255] = 0x80000000            # -0.0
    bits[1, 200] = 0x00000000            # +0.0
    bits[0, 17] = 0x7F800000             # +inf
    bits[1, 0] = 0xFF800000              # -inf
    bits[2, 128] = 0x7FC01234            # quiet NaN, payload 0x1234
    bits[2, 3] = 0xFF800ABC              # signalling NaN, payload 0xABC
    assert len(np.unique(bits)) == 768 and SENTINEL not in bits
    return v


# ----------------------------------------------------------------------------------------------------------------------
# CPU part
# ----------------------------------------------------------------------------------------------------------------------
def test_plan_restatement():
    tiles = {T: gather_plan(T, [16], [1], 0, 148)['tiles'] for T in TILED_TS + (64,)}
    assert tiles == {4: 1, 8: 1, 12: 1, 64: 8, 100: 20, 224: 98, 252: 125, 256: 128}
    assert [T * T % TILE_PIX for T in (100, 224, 252, 256)] == [272, 0, 16, 0]          # ragged last tile at 100 and 252
    p = gather_plan(224, [16], [20], 0, 148)                                            # 1 960 items: one tile per warp only
    assert (p['items'], p['one_pass'], p['multi_pass']) == (1960, False, False)         # if occupancy >= 2 CTAs per SM
    assert not gather_plan(4, [16], [9472], 0, 148)['multi_pass'] and gather_plan(4, [16], [9473], 0, 148)['multi_pass']
    assert gather_plan(64, [16, 32], [3, 3], 0, 148)['walk'] == 'round_robin'
    assert gather_plan(64, [16, 32], [3, 4], 0, 148)['walk'] == 'concat'
    assert gather_plan(64, [16], [3], 0, 148, swap=False)['kernel'] == 'tiled<false>'
    assert gather_plan(64, [16, 33], [3, 3], 0, 148)['kernel'] == 'scalar'
    assert gather_plan(64, [16, None], [3, 0], 4, 148)['kernel'] == 'scalar'
    assert gather_plan(63, [16], [3], 0, 148)['kernel'] == 'scalar'
    assert gather_plan(64, [16] * 17, [1] * 17, 0, 148)['status'] == 'EINVAL'
    assert gather_plan(257, [16], [1], 0, 148)['status'] == 'EINVAL'
    assert gather_plan(1, [16], [MAX_TOTAL + 1], 0, 148)['status'] == 'ETOOBIG'
    assert gather_plan(4, [16] * 16, [1 << 20] * 16, 0, 148)['status'] == 'ok'
    assert gather_plan(64, [None] * 4, [0] * 4, 0, 148)['status'] == 'no launch'


@pytest.mark.parametrize('sms', [148, 132, 160])
def test_matrix_reaches_every_regime(sms):
    """Every case claims the cell the restated plan gives it, and the cases reach every cell of the table."""
    reached = set()
    for case in CASES:
        counts = case_counts(case, sms)
        for swap in (False, True):
            src, out = fake_ptrs(case, counts)
            plan = gather_plan(case.T, src, counts, out, sms, swap)
            check_claim(case, plan, sms)
            reached.add(plan_cell(plan))
    for T, n in ((1, [MAX_TOTAL]), (4, [1 << 20] * 16)):
        reached.add(plan_cell(gather_plan(T, [16] * len(n), n, 0, sms)))
    assert reached == REGIMES, sorted(REGIMES ^ reached)


# ----------------------------------------------------------------------------------------------------------------------
# GPU part
# ----------------------------------------------------------------------------------------------------------------------
def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


_LUT = {}


def _lut():
    if 'dev' not in _LUT:
        _LUT['host'] = random_lut()
        _LUT['dev'] = torch.as_tensor(_LUT['host']).cuda()
    return _LUT['dev']


def _source(n, T, seed, off=0):
    """uint8 [n,T,T,3] of random bytes, starting ``off`` bytes into its own buffer."""
    g = torch.Generator(device='cuda').manual_seed(seed)
    flat = torch.randint(0, 256, (n * T * T * 3 + off,), dtype=torch.uint8, device='cuda', generator=g)
    return flat[off:].view(n, T, T, 3)


def _sentinel_rows(rows, T, off=0):
    """(float32 [rows,3,T,T] starting ``off`` floats into its buffer, the whole buffer), filled with SENTINEL."""
    buf = torch.full((rows * 3 * T * T + off,), SENTINEL, dtype=torch.int32, device='cuda')
    return buf[off:].view(torch.float32).view(rows, 3, T, T), buf


def _reference(src, lut, swap):
    """float32 [n,3,T,T]: the table lookup by torch indexing."""
    return torch.stack([lut[p][src[..., 2 - p if swap else p].long()] for p in range(3)], dim=1)


def _assert_bits_equal(got, want, what):
    a, b = got.view(torch.int32), want.view(torch.int32)
    if not torch.equal(a, b):
        bad = (a != b).flatten(1).any(1).nonzero().flatten()[:8].tolist()
        pytest.fail(f'{what}: crops {bad} differ from the reference')


def _run(case, swap):
    from bpc_baseline_b200 import batched
    sms = _sms()
    counts = case_counts(case, sms)
    T, total = case.T, sum(counts)
    seed0 = sum(map(ord, case.name)) * 1000 + 17 * swap
    srcs = [_source(c, T, seed0 + s, case.src_off[s] if s < len(case.src_off) else 0) for s, c in enumerate(counts)]
    big, buf = _sentinel_rows(case.lead + total + case.tail, T, case.out_off)
    out = big[case.lead:]
    plan = gather_plan(T, [s.data_ptr() if c else None for s, c in zip(srcs, counts)], counts, out.data_ptr(), sms, swap)
    check_claim(case, plan, sms)
    got = batched.crops_normalise(srcs, T, swap_rb=swap, lut=_lut(), out=out)
    assert got.data_ptr() == out.data_ptr()
    row = 0
    for s, (src, c) in enumerate(zip(srcs, counts)):
        _assert_bits_equal(out[row:row + c], _reference(src, _lut(), swap), f'{case.name} swap={swap} source {s}')
        row += c
    rest = torch.cat([big[:case.lead].reshape(-1), big[case.lead + total:].reshape(-1)]).view(torch.int32)
    assert bool((rest == SENTINEL).all()), f'{case.name}: a row outside the crops was written'
    assert bool((buf[:case.out_off] == SENTINEL).all())
    return plan


@pytest.mark.gpu
@pytest.mark.parametrize('swap', [False, True])
@pytest.mark.parametrize('case', CASES, ids=[c.name for c in CASES])
def test_matrix_case(case, swap):
    _run(case, swap)


@pytest.mark.gpu
@pytest.mark.parametrize('swap', [False, True])
@pytest.mark.parametrize('T,counts', [(12, (2, 0, 3)), (100, (2, 2)), (6, (1, 0, 2)), (37, (3,))])
def test_small_cases_against_numpy(T, counts, swap):
    """The same lookup written in NumPy on the host, for a tiled concat, a tiled round-robin and two scalar launches."""
    from bpc_baseline_b200 import batched
    rng = np.random.default_rng([T, len(counts), int(swap)])
    host = [rng.integers(0, 256, (c, T, T, 3), dtype=np.uint8) for c in counts]
    got = batched.crops_normalise([torch.as_tensor(h).cuda() for h in host], T, swap_rb=swap, lut=_lut()).cpu().numpy()
    lut = random_lut()
    want = np.concatenate([np.stack([lut[p][h[..., 2 - p if swap else p]] for p in range(3)], axis=1) for h in host])
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


@pytest.mark.gpu
def test_equal_zero_counts_leave_out_untouched():
    from bpc_baseline_b200 import batched
    T = 64
    srcs = [torch.empty((0, T, T, 3), dtype=torch.uint8, device='cuda') for _ in range(4)]
    assert gather_plan(T, [None] * 4, [0] * 4, 0, _sms())['status'] == 'no launch'
    out, buf = _sentinel_rows(3, T)
    got = batched.crops_normalise(srcs, T, lut=_lut(), out=out)
    torch.cuda.synchronize()
    assert got.shape[0] == 3 and bool((buf == SENTINEL).all())


@pytest.mark.gpu
def test_kernel_names_under_the_profiler():
    """Each compiled kernel (tiled<false>, tiled<true>, and the scalar one for both of its reasons) is the one the plan
    names."""
    from torch.profiler import ProfilerActivity, profile

    from bpc_baseline_b200 import batched
    runs = [(64, False, 0), (64, True, 0), (37, False, 0), (64, True, 4)]     # T, swap, misalignment of source 1
    inputs, want = [], []
    for T, swap, off in runs:
        srcs = [_source(3, T, 1), _source(3, T, 2, off)]
        out = torch.empty((6, 3, T, T), dtype=torch.float32, device='cuda')
        plan = gather_plan(T, [s.data_ptr() for s in srcs], [3, 3], out.data_ptr(), _sms(), swap)
        inputs.append((srcs, T, swap, out))
        want.append(kernel_symbol(plan['kernel']))
    assert want == ['bpc_crops_normalise_kernel<false>', 'bpc_crops_normalise_kernel<true>',
                    'bpc_crops_normalise_any_kernel', 'bpc_crops_normalise_any_kernel']
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        torch.zeros(1, device='cuda').add_(1)
        for srcs, T, swap, out in inputs:
            batched.crops_normalise(srcs, T, swap_rb=swap, lut=_lut(), out=out)
        torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                     key=lambda e: e.time_range.start)
    if not kernels:
        pytest.skip('the profiler recorded no CUDA kernels on this machine')
    names = [e.name for e in kernels if 'crops_normalise' in e.name]
    assert len(names) == len(want) and all(w in n for w, n in zip(want, names)), names


@pytest.mark.gpu
def test_sixteen_sources_accepted_seventeen_refused():
    from bpc_baseline_b200 import _lib, batched
    T = 4
    srcs = [_source(1, T, 100 + s) for s in range(17)]
    out, buf = _sentinel_rows(17, T)
    batched.crops_normalise(srcs[:16], T, lut=_lut(), out=out)
    for s in range(16):
        _assert_bits_equal(out[s:s + 1], _reference(srcs[s], _lut(), True), f'source {s}')
    with pytest.raises(RuntimeError, match='1..16 sources'):
        batched.crops_normalise(srcs, T, lut=_lut(), out=out)
    out.view(torch.int32).fill_(SENTINEL)
    ptrs = (C.c_void_p * 17)(*[s.data_ptr() for s in srcs])
    counts = (C.c_int32 * 17)(*[1] * 17)
    code = _lib.load().bpc_crops_normalise(ptrs, counts, 17, T, 1, C.c_void_p(_lut().data_ptr()), C.c_void_p(out.data_ptr()),
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert code == BPC_EINVAL and bool((buf == SENTINEL).all())


@pytest.mark.gpu
def test_largest_total_on_the_scalar_kernel():
    """Exactly 2^24 crops at T = 1: 50 MB in, 201 MB out, every thread of the grid takes several elements."""
    from bpc_baseline_b200 import batched
    src = _source(MAX_TOTAL, 1, 7)
    out, _ = _sentinel_rows(MAX_TOTAL + 1, 1)
    plan = gather_plan(1, [src.data_ptr()], [MAX_TOTAL], out.data_ptr(), _sms())
    assert plan_cell(plan) == ('scalar', 'concat', 'several')
    batched.crops_normalise([src], 1, lut=_lut(), out=out)
    _assert_bits_equal(out[:MAX_TOTAL], _reference(src, _lut(), True), 'T=1')
    assert int(out[MAX_TOTAL:].view(torch.int32).flatten()[0]) == SENTINEL


@pytest.mark.gpu
def test_largest_total_on_the_tiled_kernel():
    """Exactly 2^24 crops at T = 4 walked round robin over 16 sources of 2^20: 805 MB in, 3.2 GB out."""
    from bpc_baseline_b200 import batched
    n = MAX_TOTAL // 16
    srcs = [_source(n, 4, 300 + s) for s in range(16)]
    out, _ = _sentinel_rows(MAX_TOTAL + 1, 4)
    plan = gather_plan(4, [s.data_ptr() for s in srcs], [n] * 16, out.data_ptr(), _sms(), swap=False)
    assert plan_cell(plan) == ('tiled<false>', 'round_robin', 'several')
    batched.crops_normalise(srcs, 4, swap_rb=False, lut=_lut(), out=out)
    for s in range(16):
        _assert_bits_equal(out[s * n:(s + 1) * n], _reference(srcs[s], _lut(), False), f'T=4 source {s}')
    assert bool((out[MAX_TOTAL:].view(torch.int32) == SENTINEL).all())


@pytest.mark.gpu
def test_one_crop_too_many_is_refused():
    from bpc_baseline_b200 import _lib, batched
    src = _source(MAX_TOTAL + 1, 1, 9)
    out, buf = _sentinel_rows(MAX_TOTAL + 1, 1)
    assert gather_plan(1, [src.data_ptr()], [MAX_TOTAL + 1], out.data_ptr(), _sms())['status'] == 'ETOOBIG'
    with pytest.raises(_lib.BpcError, match=f'code {BPC_ETOOBIG}:'):
        batched.crops_normalise([src], 1, lut=_lut(), out=out)
    torch.cuda.synchronize()
    assert bool((buf == SENTINEL).all())
