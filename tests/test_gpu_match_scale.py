"""The matcher in every launch regime up to Dmax = 2048, and the explicit-cost LSAP at each of its block sizes, against
the oracle (reference restatement + SciPy).

Launch regimes of bpc_match_kernel (match_plan / match_smem_bytes / lsap_state_bytes in csrc/match.cu and
csrc/lsap.cuh; restated in _plan below and anchored to the library by test_regime_edges):

    Dmax       threads  scene state
    1-32         32     shared memory
    33-64       128     shared memory
    65-451      256     shared memory
    452-524     128     shared memory (halved to fit 227 KB)
    525-568      64     shared memory (halved)
    569-593      32     shared memory (halved)
    594-2048    256     per-CTA block of the caller's workspace; grid = min(S, 2 x 148), the CTAs walk the scenes

bpc_match_objects picks 32 threads for nc <= 1024 columns, 128 for nc <= 8192, 256 beyond, and returns BPC_ETOOBIG
when the state of the (nr x nc) problem exceeds shared memory.

Bars as in the rest of the suite: indices identical including order, n identical, float32 costs bit-equal, X within
1e-9 relative (norm-wise), F within 1e-12, reprojection errors within 1e-6 relative.
"""
import numpy as np
import pytest

from oracle import geometry as og
from tests.gpu_util import check_match_properties, oracle_map, oracle_match, rel_err, to_dev

SMEM_MAX = 227 * 1024
GRID_CAP = 2 * 148
WORKERS = 4                 # the oracle of a D = 600 scene peaks at several GB: at most 4 at once


# ---------------------------------------------------------------------------------------------------------------------
# A. regime edges (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def _lsap_state_bytes(nr, nc):
    # u, vcol | cm, cu, sspc, newv | 32 Cand of 24 bytes | col4row | crow, scol, spath, ovpos, ovcol | asg | ctl | inchain
    b = nr * 8 * 2 + (nr + 1) * 8 * 4 + 24 * 32 + nr * 4 + (nr + 1) * 4 * 5 + (nc + 31) // 32 * 4 + 16 + (nr + 7) // 8 * 8
    return (b + 15) & ~15


def _match_smem_bytes(D, nwarps):
    b = (27 + 36) * 8 + 3 * D * 2 * 8 + 6 * D * 3 * 8 + nwarps * D * 8 * 2 + _lsap_state_bytes(D, D * D)
    b += D * 4 * 6 + nwarps * D * 2 * 2 + 6 * D
    return (b + 64 + 15) & ~15


def _plan(D):
    """(threads, spill bytes per CTA) of bpc_match_kernel for Dmax = D."""
    th = 32 if D <= 32 else (128 if D <= 64 else 256)
    while _match_smem_bytes(D, th // 32) > SMEM_MAX and th > 32:
        th //= 2
    if _match_smem_bytes(D, th // 32) <= SMEM_MAX:
        return th, 0
    return 256, (_match_smem_bytes(D, 8) + 255) & ~255


REGIMES = [((1, 32), 32, False), ((33, 64), 128, False), ((65, 451), 256, False), ((452, 524), 128, False),
           ((525, 568), 64, False), ((569, 593), 32, False), ((594, 2048), 256, True)]


def test_regime_edges():
    """The restated plan agrees with bpc_match_workspace_bytes at every Dmax, so the table above (and the Dmax values the
    GPU tests below use) provably reach the regime they claim."""
    from bpc_baseline_b200 import _lib
    lib = _lib.load()
    assert lib.bpc_match_workspace_bytes(1, 593) == 0 and lib.bpc_match_workspace_bytes(1, 594) == 315904
    for D in range(1, 2049):
        th, spill = _plan(D)
        assert lib.bpc_match_workspace_bytes(1, D) == spill, D
        (lo, hi), want_th, want_spill = next(r for r in REGIMES if r[0][0] <= D <= r[0][1])
        assert (th, spill > 0) == (want_th, want_spill), D
    # the grid of the workspace kernel is capped at 296 CTAs: the workspace stops growing there
    assert lib.bpc_match_workspace_bytes(295, 640) == 295 * _plan(640)[1]
    assert lib.bpc_match_workspace_bytes(296, 640) == lib.bpc_match_workspace_bytes(297, 640) \
        == lib.bpc_match_workspace_bytes(5000, 640) == GRID_CAP * _plan(640)[1]
    assert lib.bpc_match_workspace_bytes(1, 2049) == 0                                   # beyond BPC_MAX_DET


# the largest column count of bpc_match_objects at nr = 24 rows: its state + keep[nr] + 32 bytes must fit 227 KB
OBJ_NC_MAX = 1837856


def test_match_objects_shared_memory_edge_restated():
    assert _lsap_state_bytes(24, OBJ_NC_MAX) + 24 * 4 + 32 == SMEM_MAX
    assert _lsap_state_bytes(24, OBJ_NC_MAX + 1) + 24 * 4 + 32 > SMEM_MAX
    assert 32 * 57433 == OBJ_NC_MAX and 3 * 612619 == OBJ_NC_MAX + 1


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def _pack(parts, Dmax):
    """SceneBatch of the given (batch, scene) pairs, padded to Dmax detections per camera."""
    from bpc_baseline_b200 import synth
    S = len(parts)
    Ks = np.stack([b.Ks[s] for b, s in parts])
    RTs = np.stack([b.RTs[s] for b, s in parts])
    boxes = np.zeros((S, 3, Dmax, 4), np.int32)
    centers = np.zeros((S, 3, Dmax, 2), np.float64)
    truth = np.full((S, 3, Dmax), -1, np.int32)
    counts = np.zeros((S, 3), np.int32)
    for t, (b, s) in enumerate(parts):
        d = min(Dmax, b.centers.shape[2])
        boxes[t, :, :d], centers[t, :, :d], truth[t, :, :d] = b.boxes[s, :, :d], b.centers[s, :, :d], b.truth[s, :, :d]
        counts[t] = b.counts[s]
    assert counts.max() <= Dmax
    return synth.SceneBatch(Ks, RTs, boxes, centers, counts, truth)


def _run(batch):
    import torch
    from bpc_baseline_b200 import batched
    res = batched.match_triangulate(to_dev(batch.Ks), to_dev(batch.RTs), to_dev(batch.centers), to_dev(batch.counts), 30,
                                    want_reproj=True, want_F=True)
    torch.cuda.synchronize()
    return {k: getattr(res, k).cpu().numpy() for k in ('idx', 'n', 'cost', 'X', 'reproj', 'F')}


def _job(batch, s):
    Ks, RTs = batch.capture_arrays(s)
    return Ks, RTs, [batch.centers[s, c, :batch.counts[s, c]].copy() for c in range(3)]


def _check_scene(out, s, want):
    """Scene s of a match_triangulate result against og.match_scene (or the ValueError it raised)."""
    from bpc_baseline_b200 import batched
    n = int(out['n'][s])
    if isinstance(want, Exception):
        assert n == batched.N_INFEASIBLE, (s, n, want)
        return
    assert n == len(want['idx']) and np.array_equal(out['idx'][s, :n], want['idx']), (s, n, len(want['idx']))
    assert np.all(out['idx'][s, n:] == -1), s
    for p in range(3):
        if np.all(np.isfinite(want['F'][p])):
            np.testing.assert_allclose(out['F'][s, p], want['F'][p], rtol=1e-12, atol=0, err_msg=str((s, p)))
        else:   # a NaN intrinsic: which entries np.linalg.inv makes NaN depends on the LAPACK build; NaN on both sides
            assert np.isnan(out['F'][s, p]).any(), (s, p)
    if n:
        assert np.array_equal(out['cost'][s, :n].view(np.uint32), want['cost'].view(np.uint32)), s
        assert rel_err(out['X'][s, :n], want['X']).max() < 1e-9, s
        np.testing.assert_allclose(out['reproj'][s, :n], want['reproj'], rtol=1e-6, atol=1e-7, err_msg=str(s))


def _check_against_oracle(batch, out, scenes):
    scenes = list(scenes)
    wants = oracle_map([_job(batch, s) for s in scenes], WORKERS)
    for s, want in zip(scenes, wants):
        _check_scene(out, s, want)
    return wants


def _same_scene(a, sa, b, sb):
    """Bit-equality of scene sa of result a and scene sb of result b (Dmax may differ: the padding is not compared)."""
    n = int(a['n'][sa])
    assert n == int(b['n'][sb]), (sa, sb)
    if n <= 0:
        return
    for k, dt in (('idx', np.int32), ('cost', np.uint32), ('X', np.uint64), ('reproj', np.uint64)):
        assert np.array_equal(a[k][sa, :n].view(dt), b[k][sb, :n].view(dt)), (k, sa, sb)


def _conflict_heavy(D, seed):
    """One scene whose counts are at most D: dropped (p 0.1), 2 px noise, duplicated and false detections."""
    from bpc_baseline_b200 import synth
    extra = max(1, D // 16)
    return synth.make_scenes(1, D - 2 * extra, seed=seed, p_drop=0.1, sigma=2.0, n_dup=extra, n_false=extra)


# ---------------------------------------------------------------------------------------------------------------------
# B. real scenes in every regime
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('Dmax', [32, 33, 64, 65, 451, 452, 524, 525, 568, 569, 593, 594, 700])
def test_every_regime_matches_scipy(Dmax):
    """Per Dmax: a clean scene whose counts fill the buffer (the immediate sinks), a conflict-heavy scene (the full
    shortest-augmenting-path search with the pruned scan) and a ragged scene with N*M <= P (the exhaustive scan of the
    untransposed problem)."""
    from bpc_baseline_b200 import synth
    clean = synth.make_scenes(1, Dmax, seed=synth.SEED + 300 + Dmax)
    heavy = _conflict_heavy(Dmax, synth.SEED + 400 + Dmax)
    batch = _pack([(clean, 0), (heavy, 0), (clean, 0)], Dmax)
    batch.counts[2] = (2, Dmax // 2, Dmax)
    assert batch.counts[0].tolist() == [Dmax] * 3 and batch.counts[1].max() <= Dmax
    # the conflict-heavy scene has exact duplicates among its third-camera detections (the rows of the transposed
    # problem): two rows with the same argmin, so at least one full augmenting-path search
    P = batch.counts[1, 2]
    assert len(np.unique(batch.centers[1, 2, :P], axis=0)) < P
    out = _run(batch)
    check_match_properties(batch, out)
    assert out['n'][0] >= 0.9 * Dmax
    _check_against_oracle(batch, out, range(3))


# ---------------------------------------------------------------------------------------------------------------------
# C. the largest scenes the matcher accepts (Dmax = 2048)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_rectangular_scenes_at_dmax_2048():
    """(2048, 3, 2048) and (3, 2048, 2048): transposed, 2048 rows; (20, 30, 2048): untransposed, the exhaustive scan on
    600 rows; (900, 900, 30): 810 000 columns, r = i*M + j up to 809 999 for the division by M.  All four against the
    oracle.  (2048, 2048, 2048) is beyond the oracle (a 34 GB cost tensor): its properties, every cost against
    epipolar_error_full of its own triple, and X against triangulate_multi_view of the matched centres."""
    from bpc_baseline_b200 import synth
    D = 2048
    src = synth.make_scenes(5, D, seed=synth.SEED + 500)
    batch = _pack([(src, s) for s in range(5)], D)
    batch.counts[:] = [(2048, 3, 2048), (3, 2048, 2048), (20, 30, 2048), (900, 900, 30), (2048, 2048, 2048)]
    out = _run(batch)
    check_match_properties(batch, out)
    assert out['n'][4] >= 0.9 * D
    _check_against_oracle(batch, out, range(4))
    s = 4
    n = int(out['n'][s])
    Ks, RTs, cen = _job(batch, s)
    F12, F13, F23 = og.scene_fundamentals(Ks, RTs)
    np.testing.assert_allclose(out['F'][s], np.stack([F12, F13, F23]), rtol=1e-12, atol=0)
    Ps = og.projection_matrices(Ks, RTs)
    for m in range(n):
        i, j, k = (int(v) for v in out['idx'][s, m])
        want = np.float32(og.epipolar_error_full(cen[0][i], cen[1][j], cen[2][k], F12, F13, F23))
        assert out['cost'][s, m].view(np.uint32) == want.view(np.uint32), m
        X = og.triangulate_multi_view(Ps, np.array([cen[0][i], cen[1][j], cen[2][k]]))
        assert rel_err(out['X'][s, m][None], X[None])[0] < 1e-9, m


# ---------------------------------------------------------------------------------------------------------------------
# D. the scene walk of the workspace kernel
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_workspace_scene_walk():
    """Dmax 640, S = 2*296 + 9: CTA b takes scenes b, b + 296 (and b + 592 for b < 9).  Real 600+-detection scenes share
    CTAs with small conflict-heavy ones in both orders, next to an empty scene and an overflowing one.  Every scene
    must equal the oracle, the small ones must be bit-equal to the same scenes run alone through the shared-memory
    kernel, and the result must not depend on what the (torch.empty) workspace held before the launch."""
    import torch
    from bpc_baseline_b200 import batched, synth
    D, S = 640, 2 * GRID_CAP + 9
    small = synth.make_scenes(S, 16, seed=synth.SEED + 600, p_drop=0.15, sigma=2.0, n_dup=4, n_false=4)
    rng = np.random.default_rng(600)
    small.counts = np.minimum(small.counts, rng.integers(6, 25, (S, 3))).astype(np.int32)
    big = synth.make_scenes(4, 620, seed=synth.SEED + 601, p_drop=0.02, sigma=2.0, n_dup=10, n_false=10)
    assert big.counts.min() > 593                        # each of them needs the workspace on its own
    # CTA 0: big -> small -> big; CTA 1: small -> big -> small; CTA 10: big -> small
    at_big = {0: 0, GRID_CAP + GRID_CAP: 1, 1 + GRID_CAP: 2, 10: 3}
    parts = [(big, at_big[s]) if s in at_big else (small, s) for s in range(S)]
    batch = _pack(parts, D)
    zero, over = 2, 3 + GRID_CAP                          # CTA 2: empty -> small -> small; CTA 3: small -> overflow -> small
    batch.counts[zero, 1] = 0
    batch.counts[over, 0] = D + 1
    out = _run(batch)
    assert out['n'][zero] == 0 and out['n'][over] == batched.N_OVERFLOW
    assert np.all(out['idx'][[zero, over]] == -1) and np.all(np.isnan(out['cost'][[zero, over]]))
    _check_against_oracle(batch, out, [s for s in range(S) if s != over])
    # the small scenes alone, at their own Dmax (shared-memory kernel)
    alone_batch = _pack([(small, s) for s in range(S)], 24)
    alone_batch.counts[zero, 1] = 0
    assert batched._match_workspace(torch.device('cuda'), S, 24) is None
    alone = _run(alone_batch)
    checked = 0
    for s in range(S):
        if s in at_big or s == over:
            continue
        _same_scene(out, s, alone, s)
        checked += 1
    assert checked == S - 5
    # the same launch after the cached workspace was filled with 0x00, 0xFF and NaN doubles: bit-identical outputs
    ws = batched._match_workspace(torch.device('cuda'), S, D)
    assert ws is not None and ws.numel() == batched._lib.load().bpc_match_workspace_bytes(S, D)
    for fill in (lambda w: w.fill_(0x00), lambda w: w.fill_(0xFF), lambda w: w.view(torch.float64).fill_(float('nan'))):
        fill(ws)
        torch.cuda.synchronize()
        again = _run(batch)
        for k, dt in (('idx', np.int32), ('n', np.int32), ('cost', np.uint32), ('X', np.uint64), ('reproj', np.uint64),
                      ('F', np.uint64)):
            assert np.array_equal(again[k].view(dt), out[k].view(dt)), k


# ---------------------------------------------------------------------------------------------------------------------
# E. bpc_match_objects at scale
# ---------------------------------------------------------------------------------------------------------------------
def _explicit_costs(shape, seed):
    """Four problems of one shape, the modes of test_match_objects_any_shape: uniform random, integer costs with heavy
    exact ties, 9999 sentinels, duplicated first-camera rows."""
    N, M, P = shape
    rng = np.random.default_rng([seed, N, M, P])
    out = np.empty((4, N, M, P), np.float32)
    out[0] = rng.random((N, M, P)) * 60
    out[1] = rng.integers(0, 3, (N, M, P)).astype(np.float32) * 10
    out[2] = rng.integers(0, 4, (N, M, P))
    out[2][rng.random((N, M, P)) < 0.4] = 9999
    out[3] = np.tile(rng.random((1, M, P)) * 40, (N, 1, 1))
    return out


def _shape_id(shape):
    return 'x'.join(str(v) for v in shape)


def _objects_vs_scipy(costs):
    from bpc_baseline_b200 import batched
    idx, n = batched.match_objects(to_dev(costs), 30)
    idx, n = idx.cpu().numpy(), n.cpu().numpy()
    for s in range(len(costs)):
        try:
            want = og.match_objects(costs[s], 30)
        except ValueError:
            assert n[s] == batched.N_INFEASIBLE, s
            continue
        assert n[s] == len(want) and [tuple(r) for r in idx[s, :n[s]]] == want, s
        assert np.all(idx[s, n[s]:] == -1)


@pytest.mark.gpu
@pytest.mark.parametrize('shape', [(32, 32, 5), (32, 33, 5), (64, 128, 9), (91, 91, 40), (10, 10, 9000)], ids=_shape_id)
def test_match_objects_thread_switches(shape):
    """nc = 1024 | 1056 | 8192 | 8281 columns: 32 | 128 | 128 | 256 threads, and (10, 10, 9000): 100 untransposed rows
    over 9000 columns (256 threads).  Four problems per launch."""
    _objects_vs_scipy(_explicit_costs(shape, 7))


@pytest.mark.gpu
@pytest.mark.parametrize('shape', [(91, 91, 40), (10, 10, 9000)], ids=_shape_id)
def test_match_objects_non_finite_at_scale(shape):
    """+inf entries that leave the problem feasible; a row of the assignment that is all +inf (no feasible
    assignment), a NaN and a -inf: n = -1 where SciPy raises, the other problems of the launch unaffected."""
    N, M, P = shape
    rng = np.random.default_rng([8, N, M, P])
    base = (rng.random((N, M, P)) * 60).astype(np.float32)
    costs = np.repeat(base[None], 6, axis=0)
    costs[0][rng.random((N, M, P)) < 0.05] = np.inf
    if N * M > P:                                               # SciPy transposes: rows are k, columns (i, j)
        costs[0][1, 2, :] = np.inf                              # a whole column
        costs[1][:, :, 7] = np.inf                              # a whole row: no feasible assignment
    else:                                                       # rows are (i, j), columns k
        costs[0][:, :, 5] = np.inf
        costs[1][3, 4, :] = np.inf
    costs[2][N - 1, M - 1, P - 1] = np.nan
    costs[3][N // 2, 0, P // 3] = -np.inf
    costs[4][0, 0, 0] = np.nan
    assert len(og.match_objects(costs[0], 30)) > 0
    for s in (1, 2, 3, 4):
        with pytest.raises(ValueError):
            og.match_objects(costs[s], 30)
    _objects_vs_scipy(costs)


@pytest.mark.gpu
def test_match_objects_shared_memory_limit():
    """nr = 24 rows over the widest column count whose state fits shared memory (32 x 57433 = 1 837 856 columns): equal
    to SciPy; one column more (3 x 612619) is refused with BPC_ETOOBIG, not computed wrongly."""
    import torch
    from bpc_baseline_b200 import batched
    rng = np.random.default_rng(9)
    cost = (rng.random((1, 32, 57433, 24)) * 60).astype(np.float32)        # unique minima: short augmenting paths
    _objects_vs_scipy(cost)
    del cost
    big = torch.zeros((1, 3, 612619, 24), dtype=torch.float32, device='cuda')
    with pytest.raises(RuntimeError, match='code -4'):
        batched.match_objects(big, 30)


# ---------------------------------------------------------------------------------------------------------------------
# F. non-finite inputs to the geometry path
# ---------------------------------------------------------------------------------------------------------------------
# (what, camera, value, whether SciPy raises): a NaN / infinite centre makes NaN costs ("invalid numeric entries");
# a 1e300 centre makes +inf float32 costs, infeasible only when the third camera (the rows of the transposed problem)
# has it; a NaN intrinsic turns every line into the 9999 sentinel: a valid problem without matches
VARIANTS = [('centre', 0, np.nan, True), ('centre', 1, np.nan, True), ('centre', 2, np.nan, True),
            ('centre', 0, np.inf, True), ('centre', 1, -np.inf, True), ('centre', 2, np.inf, True),
            ('centre', 0, 1e300, False), ('centre', 1, -1e300, False), ('centre', 2, 1e300, True),
            ('K', 0, np.nan, False), ('K', 2, np.nan, False)]


def _spoil(batch, s, variant, d=3):
    what, cam, value, _ = variant
    if what == 'centre':
        batch.centers[s, cam, d, cam % 2] = value
    else:
        batch.Ks[s, cam, 0, 0] = value


@pytest.mark.parametrize('variant', VARIANTS, ids=lambda v: f'{v[0]}{v[1]}={v[2]}')
def test_oracle_on_non_finite_inputs(variant):
    """The expectations of test_non_finite_inputs, on the CPU: where the oracle raises ValueError."""
    from bpc_baseline_b200 import synth
    what, cam, _, raises = variant
    batch = synth.make_scenes(1, 20, seed=synth.SEED + 700)
    _spoil(batch, 0, variant)
    with np.errstate(all='ignore'):
        want = oracle_match(_job(batch, 0))
    assert isinstance(want, ValueError) == raises
    if raises:
        return
    if what == 'K':                     # every pair distance through that camera is the sentinel: no cost below 30
        assert len(want['idx']) == 0
    else:                               # matches, none through the spoiled detection (its costs are +inf)
        assert len(want['idx']) > 0 and not np.any(want['idx'][:, cam] == 3)


@pytest.mark.gpu
@pytest.mark.parametrize('Dmax', [20, 640])
def test_non_finite_inputs(Dmax):
    """Each bad scene sits between two clean ones, in a shared-memory batch (Dmax 20) and a workspace batch (Dmax 640):
    n = -1 and PoseEstimator._match raises ValueError where the oracle raises, the oracle's result otherwise, and the
    clean scenes bit-equal to the same batch without the bad scenes."""
    from types import SimpleNamespace

    from bpc_baseline_b200 import synth
    from bpc_baseline_b200.inference.process_pose import PoseEstimator, PoseEstimatorParams
    V = len(VARIANTS)
    src = synth.make_scenes(2 * V + 1, 20, seed=synth.SEED + 700)
    clean = _pack([(src, s) for s in range(2 * V + 1)], Dmax)
    bad = _pack([(src, s) for s in range(2 * V + 1)], Dmax)
    for v, variant in enumerate(VARIANTS):
        _spoil(bad, 2 * v + 1, variant)
    ref, out = _run(clean), _run(bad)
    for s in range(0, 2 * V + 1, 2):
        _same_scene(out, s, ref, s)
        assert np.array_equal(out['F'][s].view(np.uint64), ref['F'][s].view(np.uint64))
    with np.errstate(all='ignore'):
        wants = _check_against_oracle(bad, out, range(1, 2 * V + 1, 2))
    est = PoseEstimator(PoseEstimatorParams())
    for v, (variant, want) in enumerate(zip(VARIANTS, wants)):
        s = 2 * v + 1
        assert isinstance(want, Exception) == variant[3], variant
        Ks, RTs, cen = _job(bad, s)
        capture = SimpleNamespace(images=[None] * 3, Ks=Ks, RTs=RTs)
        dets = {c: [{'bbox': tuple(int(x) for x in bad.boxes[s, c, d]), 'bb_center': (float(p[0]), float(p[1]))}
                    for d, p in enumerate(cen[c])] for c in range(3)}
        if variant[3]:
            with pytest.raises(ValueError):
                est._match(capture, dets)
        else:
            assert [p.match for p in est._match(capture, dets)] == [tuple(int(x) for x in r) for r in want['idx']]
