"""The small geometry kernels of csrc/match.cu against high-precision references, on ill-conditioned inputs and at scale.

1. DLT triangulation (bpc_triangulate, bpc_triangulate_views for V = 2..8, bpc_match_tri_kernel through
   match_triangulate).  Reference: an mpmath SVD at 60 digits of the float64 A the kernels build
   (oracle/hp_geometry.py), its singular values s1 >= s2 >= s3 >= s4 and the unit right singular vector v* of s4.
   With v = (X, 1) / ||(X, 1)|| of the computed X, every case must satisfy

       residual   ||A v|| <= s4 + C_DLT eps s1                        (backward stability; every case)
       forward    sin angle(v, v*) <= C_DLT eps s1 / (s3 - s4)        (where s3 - s4 >= GAP_MIN eps s1)
       point      ||X - X*|| <= C_DLT eps s1 / (s3 - s4) (1 + ||X*||^2) + C_DLT eps ||X*||   (also |v*_3| >= 1e-8)

   C_DLT = 64.  One-sided Jacobi applies plane rotations to the columns of A: each rotation perturbs the two columns it
   touches by a few eps (relative), the Gram sums over 2V <= 16 rows are accurate to 16 eps, and the kernels converge in
   at most ~8 sweeps of 6 rotations; the errors of successive rotations add in norm.  That gives a few tens of eps s1,
   and 64 = 4 rows x 16 rows, the size of the largest A, leaves headroom without hiding a kernel that stops early (with a
   sweep cap of 2 the views kernel fails these bounds in 8 of the 10 regimes).  LAPACK's SVD is backward stable with a
   constant of the same order, and the CPU part applies the same bounds to np.linalg.svd on every case.

   Worst ratios observed over V = 2..8 (residual / forward / point, each in units of its bound's eps term, so the
   assertion is ratio <= C_DLT; the tests print them per kernel, regime and V).  GPU: the worst of the three kernels,
   one B200 run.  In no regime is NumPy the more accurate of the two:

       regime         GPU kernels         NumPy (np.linalg.svd)
       clean          0.9 / 1.1 / 0.8     1.7 /  1.8 /  1.4
       noisy 0.5 px   0.0 / 0.8 / 0.6     0.0 / 11.1 /  9.1
       noisy 2 px     0.0 / 0.9 / 0.7     0.0 / 32.5 / 23.0
       far            0.0 / 0.0 / 0.0     1.3 /  1.2 /  1.2
       tiny baseline  0.0 / 0.1 / 0.1     0.0 /  0.1 /  0.1
       telephoto      0.0 / 0.0 / 0.0     0.0 /  1.0 /  0.0
       behind         0.0 / 0.9 / 0.7     0.0 / 29.7 / 20.6
       exact          0.6 / 0.4 / 0.2     16.3 / 16.2 /  4.4
       duplicate      0.0 / 0.9 / 0.6     0.0 / 32.9 / 22.0
       collinear      0.7 /  -  /  -      2.0 /   -  /   -

   Regimes, seeded: clean; noisy (0.5 and 2 px); far (depth 1e2..1e5 x baseline); tiny baseline (1e-4); telephoto
   (f = 1e5 on 3840 x 2160, the translation column 1e8 times the rotation columns); the point behind one camera; exact
   data (integer cameras, dyadic projections: A v* = 0 exactly); a duplicated view; collinear centres and point
   (s3 = s4: residual only).

2. Reprojection error (bpc_reprojection_error, the reproj output of match_triangulate) against mpmath on the same
   float64 P, X and point.  The result is a difference of nearly equal numbers, so the bound is absolute: per component
   c eps (|q| + |pt| + (sum |P_0||X~| + |q| sum |P_2||X~|) / |w|), q = proj / w, plus 3 eps err for the norm, c = 8 (a
   4-term row sum, one division, one subtraction).  Worst observed on one B200: 0.036 of that bound.

3. Epipolar distances, bit-exact where operation order shows: next to an epipole l = F p cancels, and near the
   1e-8 norm threshold a one-ulp difference flips the 9999 sentinel.  The CPU part checks that the oracle (NumPy)
   equals an exact restatement with a correctly rounded FMA on every input, so a GPU failure here is the kernel's.

4. Fundamental matrix on general intrinsics (every Gauss-Jordan pivot pattern, K[8] != 1, nearly singular K) and both
   sides of the |F22| <= 1e-8 branch.

5. The post-match kernels at scale: the reprojection filter (300 scenes, thresholds 0 / +inf / equal to a stored
   error, a NaN error), bpc_build_rois beyond one scan thread per scene and beyond one grid-stride pass,
   bpc_pack_records in every count-padding case, bpc_train_rois at rounding ties and clamps.
"""
from __future__ import annotations

import functools
import math

import mpmath  # noqa: F401  (the references below are mpmath: a missing module must fail, not skip)
import numpy as np
import pytest

from oracle import crop as ocrop
from oracle import geometry as og
from oracle import hp_geometry as hp
from tests.gpu_util import to_dev

C_DLT = 64.0
GAP_MIN = 1e3            # forward / point checks only where (s3 - s4) >= GAP_MIN eps s1
C_REPROJ = 8.0
EPS = hp.EPS


# ---------------------------------------------------------------------------------------------------------------------
# triangulation cases
# ---------------------------------------------------------------------------------------------------------------------
def _lookat(C, T, rng):
    z = T - C
    z = z / np.linalg.norm(z)
    up = rng.normal(size=3)
    x = np.cross(up, z)
    x /= np.linalg.norm(x)
    y = np.cross(z, x)
    R = np.stack([x, y, z])
    RT = np.eye(4)
    RT[:3, :3] = R
    RT[:3, 3] = -R @ C
    return RT


def _K(f, cx, cy):
    return np.array([[f, 0, cx], [0, f, cy], [0, 0, 1]], np.float32)


def _project(K, RT, X):
    p = (K.astype(np.float64) @ RT[:3]) @ np.append(X, 1.0)
    return p[:2] / p[2]


REGIMES = ['clean', 'noisy0.5', 'noisy2', 'far', 'tinybase', 'telephoto', 'behind', 'exact', 'duplicate', 'collinear']
RESIDUAL_ONLY = {'collinear'}


def _tri_case(regime, V, rng):
    """(Ks f32 [V,3,3], RTs f64 [V,4,4], pts f64 [V,2]) of one seeded case of the regime."""
    K = _K(1400.0, 960.0, 540.0)
    Ks = [K] * V
    noise = {'noisy0.5': 0.5, 'noisy2': 2.0, 'tinybase': 0.5, 'telephoto': 0.5, 'behind': 0.5, 'duplicate': 0.5}.get(regime, 0.0)
    if regime == 'exact':
        X = rng.integers(-8, 9, 3).astype(np.float64)
        RTs = []
        for v in range(V):
            perm = rng.permutation(3)
            R = np.eye(3)[perm] * rng.choice([-1.0, 1.0], 3)[:, None]
            if np.linalg.det(R) < 0:
                R[0] = -R[0]
            t = rng.integers(-6, 7, 3).astype(np.float64)
            t[2] = 2.0 ** int(rng.integers(3, 7)) - (R @ X)[2]          # depth a power of two: x / z is exact
            RT = np.eye(4)
            RT[:3, :3], RT[:3, 3] = R, t
            RTs.append(RT)
        Ks = [np.eye(3, dtype=np.float32)] * V
        pts = np.array([_project(Ks[v], RTs[v], X) for v in range(V)])
        return np.stack(Ks), np.stack(RTs), pts
    if regime == 'far':
        b = 0.5
        X = np.array([rng.normal() * 2, rng.normal() * 2, b * 10 ** rng.uniform(2, 5)])
        X[:2] *= X[2] * 1e-3
        RTs = [_lookat(rng.normal(size=3) * b, X + rng.normal(size=3) * X[2] * 1e-3, rng) for _ in range(V)]
    elif regime == 'tinybase':
        X = rng.normal(size=3) * 0.2 + np.array([0, 0, 1.5])
        RTs = [_lookat(rng.normal(size=3) * 1e-4, X + rng.normal(size=3) * 0.05, rng) for _ in range(V)]
    elif regime == 'telephoto':
        Ks = [_K(1e5, 1920.0, 1080.0)] * V
        D = 1e10                                  # |P[:, 3]| ~ cx D: 1e8 times the rotation columns (~f)
        X = rng.normal(size=3) * D * 1e-3
        RTs = []
        for _ in range(V):
            d = rng.normal(size=3)
            RTs.append(_lookat(d / np.linalg.norm(d) * D * rng.uniform(0.8, 1.2), X + rng.normal(size=3) * D * 2e-4, rng))
    elif regime == 'collinear':
        X = rng.normal(size=3) * 0.3
        d = rng.normal(size=3)
        d /= np.linalg.norm(d)
        s = rng.uniform(1.5, 4.0, V) * rng.choice([-1.0, 1.0], V)
        RTs = [_lookat(X + s[v] * d, X, rng) for v in range(V)]
    else:
        X = rng.normal(size=3) * 0.3
        RTs = []
        for _ in range(V):
            c = rng.normal(size=3)
            RTs.append(_lookat(c / np.linalg.norm(c) * rng.uniform(2.0, 3.0), X + rng.normal(size=3) * 0.1, rng))
        if regime == 'behind':                       # camera 0 looks away from the point: negative depth
            RTs[0] = RTs[0].copy()
            RTs[0][:3] = np.diag([-1.0, 1.0, -1.0]) @ RTs[0][:3]
    pts = np.array([_project(Ks[v], RTs[v], X) for v in range(V)]) + rng.normal(size=(V, 2)) * noise
    if regime == 'duplicate':
        RTs[-1], pts[-1], Ks[-1] = RTs[0].copy(), pts[0].copy(), Ks[0]
    return np.stack(Ks), np.stack(RTs), pts


N_V3 = 200          # cases per regime at V = 3 (bpc_triangulate, the matcher's triangulation, triangulate_views)
N_VX = 40           # cases per regime at every other V


@functools.lru_cache(maxsize=None)
def tri_cases(regime, V):
    """Seeded cases with their float64 P, A and the 60-digit reference."""
    rng = np.random.default_rng([REGIMES.index(regime), V, 7])
    n = N_V3 if V == 3 else N_VX
    Ks, RTs, P, pts, refs = [], [], [], [], []
    for _ in range(n):
        k, rt, p = _tri_case(regime, V, rng)
        Pv = np.stack([k[v].astype(np.float64) @ rt[v, :3] for v in range(V)])
        Ks.append(k); RTs.append(rt); P.append(Pv); pts.append(p)
        refs.append(hp.DltRef(hp.dlt_matrix(Pv, p)))
    return dict(Ks=np.stack(Ks), RTs=np.stack(RTs), P=np.stack(P), pts=np.stack(pts), refs=refs)


def _dlt_ratios(regime, refs, X):
    """Per case (residual, forward, point) ratios to C_DLT's eps terms; forward / point NaN where not checked."""
    out = np.full((len(refs), 3), np.nan)
    for i, (ref, x) in enumerate(zip(refs, X)):
        out[i, 0] = ref.residual_ratio(x)
        if regime in RESIDUAL_ONLY or ref.gap < GAP_MIN * EPS * ref.s1:
            continue
        out[i, 1] = ref.angle_ratio(x)
        if abs(float(ref.v[3])) >= 1e-8:
            out[i, 2] = ref.X_ratio(x)
    return out


def _check_dlt(regime, refs, X, what):
    r = _dlt_ratios(regime, refs, X)
    worst = np.nanmax(np.where(np.isnan(r), -np.inf, r), axis=0)
    print(f'{what} {regime}: worst residual {worst[0]:.2f} forward {worst[1]:.2f} point {worst[2]:.2f} (x eps s1)')
    bad = np.argwhere(~(r <= C_DLT) & ~np.isnan(r))
    assert len(bad) == 0, f'{what} {regime}: case {bad[0][0]} ratios {r[bad[0][0]]}'
    if regime not in RESIDUAL_ONLY:
        assert np.isfinite(r[:, 1]).sum() > 0 or regime in ('tinybase', 'duplicate'), 'no forward check ran'
    return worst


@pytest.mark.parametrize('regime', REGIMES)
def test_dlt_bounds_hold_for_numpy(regime):
    """Fairness: the bounds are met by np.linalg.svd on every case, so they are not tuned to the kernels."""
    for V in range(2, 9):
        c = tri_cases(regime, V)
        X = np.stack([hp.numpy_dlt(hp.dlt_matrix(P, p)) for P, p in zip(c['P'], c['pts'])])
        _check_dlt(regime, c['refs'], X, f'numpy V={V}')


def test_regimes_reach_their_conditioning():
    """The regimes produce what they claim: exact data has s4 = 0, collinear s3 = s4, far / tiny-baseline a small gap,
    telephoto columns 1e8 apart, the behind case a negative depth."""
    c = tri_cases('exact', 3)
    assert all(float(r.sigma[3]) == 0.0 or float(r.sigma[3]) < 1e-40 * r.s1 for r in c['refs'])
    c = tri_cases('collinear', 3)
    assert all(float(r.sigma[2] - r.sigma[3]) < 1e-6 * r.s1 for r in c['refs'])
    assert np.median([abs(float(r.v[3])) for r in tri_cases('far', 3)['refs']]) < 1e-2        # near infinity
    clean_gap = np.median([r.gap / r.s1 for r in tri_cases('clean', 3)['refs']])
    assert np.median([r.gap / r.s1 for r in tri_cases('tinybase', 3)['refs']]) < 1e-2 * clean_gap
    P = tri_cases('telephoto', 3)['P']
    assert np.median(np.abs(P[..., 3]).max(-1) / np.abs(P[..., :3]).max((-1, -2))) > 1e7
    c = tri_cases('behind', 3)
    Xs = [np.array([float(x) for x in r.X_star()]) for r in c['refs']]
    assert all((c['RTs'][i, 0, 2, :3] @ Xs[i] + c['RTs'][i, 0, 2, 3]) < 0 for i in range(len(Xs)))


@pytest.mark.gpu
@pytest.mark.parametrize('regime', REGIMES)
def test_triangulate_views_every_v(regime):
    from bpc_baseline_b200 import batched
    for V in range(2, 9):
        c = tri_cases(regime, V)
        X = batched.triangulate_views(to_dev(c['P']), to_dev(c['pts'])).cpu().numpy()
        _check_dlt(regime, c['refs'], X, f'triangulate_views V={V}')


@pytest.mark.gpu
@pytest.mark.parametrize('regime', REGIMES)
def test_triangulate3_and_views_agree(regime):
    """bpc_triangulate (triangulate3) and bpc_triangulate_views at V = 3 are separate code paths: both meet the bounds,
    and the angle between their answers is within twice the forward bound."""
    from bpc_baseline_b200 import batched
    c = tri_cases(regime, 3)
    X3 = batched.triangulate(to_dev(c['P']), to_dev(c['pts'])).cpu().numpy()
    Xv = batched.triangulate_views(to_dev(c['P']), to_dev(c['pts'])).cpu().numpy()
    _check_dlt(regime, c['refs'], X3, 'triangulate')
    import mpmath as mp
    for i, ref in enumerate(c['refs']):
        if regime in RESIDUAL_ONLY or ref.gap < GAP_MIN * EPS * ref.s1:
            continue
        a, b = ref.unit_from_X(X3[i]), ref.unit_from_X(Xv[i])
        with mp.workdps(hp.DPS):
            cs = mp.fsum(x * y for x, y in zip(a, b))
            s = float(mp.sqrt(max(mp.mpf(0), 1 - cs * cs)))
        assert s <= 2 * C_DLT * EPS * ref.s1 / ref.gap, (regime, i)


def _match_one_detection(c):
    """match_triangulate on S scenes of one detection per camera (threshold +inf: every case is a match)."""
    import torch
    from bpc_baseline_b200 import batched
    S = len(c['pts'])
    centers = c['pts'][:, :, None, :].copy()
    counts = np.ones((S, 3), np.int32)
    res = batched.match_triangulate(to_dev(c['Ks']), to_dev(c['RTs']), to_dev(centers), to_dev(counts), float('inf'),
                                    want_reproj=True)
    torch.cuda.synchronize()
    n = res.n.cpu().numpy()
    assert np.all(n == 1), np.unique(n)
    assert np.all(res.idx.cpu().numpy() == 0)
    return res.X.cpu().numpy()[:, 0], res.reproj.cpu().numpy()[:, 0]


@pytest.mark.gpu
@pytest.mark.parametrize('regime', REGIMES)
def test_match_triangulate_point_and_reprojection(regime):
    """bpc_match_tri_kernel (200 scenes: two blocks, not a multiple of 64) meets the DLT bounds, and its reproj output
    the absolute reprojection bound at the X it returned."""
    c = tri_cases(regime, 3)
    X, rep = _match_one_detection(c)
    _check_dlt(regime, c['refs'], X, 'match_triangulate')
    P = c['P']
    for v in range(3):
        _check_reproj(P[:, v], X, c['pts'][:, v], rep[:, v], f'match_triangulate {regime} view {v}')


# ---------------------------------------------------------------------------------------------------------------------
# reprojection error
# ---------------------------------------------------------------------------------------------------------------------
def _reproj_ref(P, X, pt):
    """(err*, bound) for one view at 60 digits."""
    import mpmath as mp
    with mp.workdps(hp.DPS):
        Xh = [mp.mpf(float(x)) for x in X] + [mp.mpf(1)]
        pr = [mp.fsum(mp.mpf(float(P[r, c])) * Xh[c] for c in range(4)) for r in range(3)]
        w = pr[2]
        if w == 0:
            return math.nan, math.nan
        q = [pr[0] / w, pr[1] / w]
        d = [q[0] - float(pt[0]), q[1] - float(pt[1])]
        err = mp.sqrt(d[0] ** 2 + d[1] ** 2)
        s2 = mp.fsum(abs(mp.mpf(float(P[2, c])) * Xh[c]) for c in range(4))
        b = 0
        for r in range(2):
            sr = mp.fsum(abs(mp.mpf(float(P[r, c])) * Xh[c]) for c in range(4))
            b += C_REPROJ * EPS * (abs(q[r]) + abs(float(pt[r])) + (sr + abs(q[r]) * s2) / abs(w))
        return float(err), float(b + 3 * EPS * err)


def _check_reproj(P, X, pts, got, what):
    worst = 0.0
    for i in range(len(got)):
        if not np.all(np.isfinite(X[i])):
            continue
        want, bound = _reproj_ref(P[i], X[i], pts[i])
        if math.isnan(want):
            continue
        r = abs(got[i] - want) / bound
        assert r <= 1.0, (what, i, got[i], want, bound)
        worst = max(worst, r)
    print(f'{what}: worst reprojection error / bound {worst:.3f}')


def _reproj_cases():
    """Near-perfect matches (errors of ~1e-9 px), coordinates of ~1e5 px, and points next to a camera's principal
    plane (|w| small)."""
    rng = np.random.default_rng(31)
    P, X, pts = [], [], []
    for kind in range(3):
        for _ in range(100):
            K = _K(1400.0, 960.0, 540.0)
            Xw = rng.normal(size=3) * 0.3
            RTs = []
            for _v in range(3):
                c = rng.normal(size=3)
                RTs.append(_lookat(c / np.linalg.norm(c) * 2.5, Xw, rng))
            if kind == 1:
                Xw = Xw + rng.normal(size=3) * 1e3
                K = _K(1e5, 1920.0, 1080.0)
            Pv = np.stack([K.astype(np.float64) @ rt[:3] for rt in RTs])
            if kind == 2:                          # move X onto camera 0's principal plane, up to ~1e-9
                n3 = Pv[0, 2, :3]
                Xw = Xw - (n3 @ Xw + Pv[0, 2, 3]) / (n3 @ n3) * n3 + n3 * rng.normal() * 1e-9
            p = np.array([(Pv[v] @ np.append(Xw, 1.0))[:2] / (Pv[v] @ np.append(Xw, 1.0))[2] for v in range(3)])
            p += rng.normal(size=p.shape) * (1e-9 if kind == 0 else 1.0)
            P.append(Pv); X.append(Xw); pts.append(p)
    return np.stack(P), np.stack(X), np.stack(pts)


@pytest.mark.gpu
def test_reprojection_error_absolute_bound():
    from bpc_baseline_b200 import batched
    P, X, pts = _reproj_cases()
    err = batched.reprojection_error(to_dev(P), to_dev(X), to_dev(pts)).cpu().numpy()
    assert np.median(err[:100]) < 1e-7                                   # the near-perfect cases are near perfect
    assert np.median(np.abs([(P[i, 0] @ np.append(X[i], 1))[2] for i in range(200, 300)])) < 1e-5
    for v in range(3):
        _check_reproj(P[:, v], X, pts[:, v], err[:, v], f'reprojection_error view {v}')


@pytest.mark.gpu
@pytest.mark.parametrize('views', [(2, 2), (4, 4), (8, 8), (5, 3), (2, 4)])
def test_triangulate_multi_view_drop_in(views):
    """inference.utils.triangulation.triangulate_multi_view with 2, 4 and 8 views, and with more matrices than points
    or more points than matrices (zip truncates): the answer of triangulate_views on the common prefix, within the
    DLT bounds."""
    import torch
    from bpc_baseline_b200 import batched
    from bpc_baseline_b200.inference.utils.triangulation import triangulate_multi_view
    nP, npt = views
    V = min(nP, npt)
    c = tri_cases('noisy0.5', max(nP, npt))
    for i in range(8):
        X = triangulate_multi_view(list(c['P'][i, :nP]), [tuple(p) for p in c['pts'][i, :npt]])
        want = batched.triangulate_views(to_dev(c['P'][i:i + 1, :V]), to_dev(c['pts'][i:i + 1, :V])).cpu().numpy()[0]
        assert np.array_equal(X, want)
        ref = hp.DltRef(hp.dlt_matrix(c['P'][i, :V], c['pts'][i, :V]))
        assert ref.residual_ratio(X) <= C_DLT
        if ref.gap >= GAP_MIN * EPS * ref.s1:
            assert ref.angle_ratio(X) <= C_DLT
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------------
# epipolar distances at the epipoles
# ---------------------------------------------------------------------------------------------------------------------
def _rot(rng):
    q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    return q * np.sign(np.linalg.det(q))


EPI_KINDS = ['pinhole', 'skewed', 'small_focal']
N_EPI_SCENES = 6            # per kind


def _epi_K(kind, rng):
    if kind == 'pinhole':
        return _K(1400.0, 960.0, 540.0)
    if kind == 'skewed':
        K = _K(1400.0, 960.0, 540.0)
        K[0, 1] = np.float32(3.5)
        K[1, 1] = np.float32(1380.25)
        return K
    return _K(np.float32(rng.uniform(2.0, 12.0)), 960.0, 540.0)


def _oracle_norm(F, transpose, x, y):
    l = (F.T if transpose else F) @ np.array([x, y, 1.0])
    return np.linalg.norm(l[:2])


def _null(F, transpose):
    """The epipole of F (transpose 0: F e = 0, camera of the first point) as a float64 point, from a 60-digit SVD."""
    import mpmath as mp
    with mp.workdps(hp.DPS):
        M = mp.matrix((F.T if transpose else F).tolist())
        _, S, Vt = mp.svd_r(M)
        k = min(range(3), key=lambda i: S[i])
        return np.array([float(Vt[k, 0] / Vt[k, 2]), float(Vt[k, 1] / Vt[k, 2])])


def _crossing_points(F, transpose, e):
    """The rounded epipole, and the 64 consecutive float64 x on each side of where the oracle's norm of the line crosses
    1e-8 (y fixed at the epipole's): the last bits of l decide the sentinel and the distances there."""
    x0, y = float(e[0]), float(e[1])
    lo, step = x0, 1e-12 * max(1.0, abs(x0))
    assert _oracle_norm(F, transpose, lo, y) <= 1e-8
    while _oracle_norm(F, transpose, x0 + step, y) <= 1e-8:
        step *= 2
    hi = x0 + step
    while np.nextafter(lo, hi) != hi:
        mid = lo + (hi - lo) / 2
        if mid == lo or mid == hi:
            break
        if _oracle_norm(F, transpose, mid, y) <= 1e-8:
            lo = mid
        else:
            hi = mid
    xs = [lo]
    for _ in range(63):
        xs.append(np.nextafter(xs[-1], -np.inf))
    xs.append(hi)
    for _ in range(63):
        xs.append(np.nextafter(xs[-1], np.inf))
    return [(x0, y)] + [(float(x), y) for x in xs]


@functools.lru_cache(maxsize=None)
def epi_scenes():
    """Per scene: Ks, RTs, (F12, F13, F23) and per camera a list of detections next to the epipoles of its two pairs,
    at 1e5 px, and inside the image."""
    rng = np.random.default_rng(77)
    out = []
    for kind in EPI_KINDS:
        for _ in range(N_EPI_SCENES):
            Ks = np.stack([_epi_K(kind, rng) for _ in range(3)])
            RTs = np.stack([og.calc_pose_matrix(_rot(rng), rng.normal(size=3)) for _ in range(3)])
            Fs = og.scene_fundamentals(list(Ks), list(RTs))
            pts = [[], [], []]
            for f, (a, b) in enumerate(((0, 1), (0, 2), (1, 2))):
                pts[a] += _crossing_points(Fs[f], 0, _null(Fs[f], 0))
                pts[b] += _crossing_points(Fs[f], 1, _null(Fs[f], 1))
            for c in range(3):
                pts[c] += [tuple(p) for p in rng.uniform(-1e5, 1e5, (4, 2))] + [(1e5, -1e5), (-1e5, 1e5)]
                pts[c] += [tuple(p) for p in rng.uniform(0, 1920, (8, 2))]
            out.append(dict(kind=kind, Ks=Ks, RTs=RTs, F=np.stack(Fs), pts=[np.array(p) for p in pts]))
    return out


@functools.lru_cache(maxsize=None)
def epi_pairs():
    """(F [n,3,3], pt1 [n,2], pt2 [n,2]) over every scene and pair: each point of camera a against a point of camera b
    (a cyclic shift, so points next to both epipoles meet), and the oracle's epipolar_error of each."""
    F, p1, p2 = [], [], []
    for sc in epi_scenes():
        for f, (a, b) in enumerate(((0, 1), (0, 2), (1, 2))):
            A, B = sc['pts'][a], sc['pts'][b]
            m = max(len(A), len(B))
            for i in range(m):
                F.append(sc['F'][f]); p1.append(A[i % len(A)]); p2.append(B[(i * 7 + 3) % len(B)])
    F, p1, p2 = np.stack(F), np.stack(p1), np.stack(p2)
    want = np.array([og.epipolar_error(a, b, f) for f, a, b in zip(F, p1, p2)], np.float64)
    return F, p1, p2, want


def test_oracle_epipolar_order_is_the_exact_restatement():
    """NumPy's F @ p, F.T @ p, norm and dot on this host round exactly as the spelled-out FMA orders the kernels use,
    on every input below (so the GPU tests compare against the kernels' own arithmetic), and the inputs reach both sides
    of the sentinel."""
    F, p1, p2, want = epi_pairs()
    exact = np.array([hp.epipolar_error_exact(f, a, b) for f, a, b in zip(F, p1, p2)])
    assert np.array_equal(want.view(np.int64), exact.view(np.int64))
    ok = np.array([hp.epiline_exact(f, 0, *a)[1] for f, a in zip(F, p1)])
    assert ok.sum() > 1000 and (~ok).sum() > 1000
    for f, a in list(zip(F, p1))[:2000]:               # the lines themselves, not only the distances
        for tr in (0, 1):
            l = (f.T if tr else f) @ np.array([a[0], a[1], 1.0])
            l_ex, _ = hp.epiline_exact(f, tr, *a)
            n = np.linalg.norm(l[:2])
            if n > 1e-8:
                l = l / n
            assert np.array_equal(l, np.array(l_ex))


@pytest.mark.gpu
def test_epipolar_error_bit_exact_at_epipoles():
    from bpc_baseline_b200 import batched
    F, p1, p2, want = epi_pairs()
    got = batched.epipolar_error(to_dev(F), to_dev(p1), to_dev(p2)).cpu().numpy()
    bad = np.flatnonzero(got.view(np.int64) != want.view(np.int64))
    assert len(bad) == 0, f'{len(bad)} of {len(want)} differ, first {bad[:4]}: {got[bad[:4]]} vs {want[bad[:4]]}'
    assert (want >= 4999.5).sum() > 100 and (want < 4999.5).sum() > 100       # both sides of the sentinel


@pytest.mark.gpu
def test_epipolar_error_full_bit_exact_at_epipoles():
    from bpc_baseline_b200 import batched
    F, pts, want = [], [], []
    for sc in epi_scenes():
        A, B, C = sc['pts']
        m = max(len(A), len(B), len(C))
        for i in range(m):
            p = np.stack([A[i % len(A)], B[(i * 5 + 1) % len(B)], C[(i * 11 + 2) % len(C)]])
            F.append(sc['F']); pts.append(p)
            want.append(og.epipolar_error_full(p[0], p[1], p[2], *sc['F']))
    F, pts, want = np.stack(F), np.stack(pts), np.array(want, np.float64)
    got = batched.epipolar_error_full(to_dev(F), to_dev(pts)).cpu().numpy()
    assert np.array_equal(got.view(np.int64), want.view(np.int64))


def _epi_match_batch(D):
    """The epipole scenes as a batch of D detections per camera: points next to the epipoles (every 9th of each camera's
    list, so the crossings and the rounded epipoles are among them) and in the image."""
    scenes = epi_scenes()
    S = len(scenes)
    centers = np.zeros((S, 3, D, 2))
    counts = np.zeros((S, 3), np.int32)
    for s, sc in enumerate(scenes):
        for c in range(3):
            p = sc['pts'][c]
            sel = np.concatenate([[0, 1, 64, 65, 129, 130, 193, 194], np.arange(3, len(p), 9)])[:20]
            counts[s, c] = len(sel)
            centers[s, c, :len(sel)] = p[sel]
    Ks = np.stack([sc['Ks'] for sc in scenes])
    RTs = np.stack([sc['RTs'] for sc in scenes])
    return Ks, RTs, centers, counts


@pytest.mark.gpu
def test_cost_tensor_bit_exact_with_detections_at_epipoles():
    from bpc_baseline_b200 import batched
    Ks, RTs, centers, counts = _epi_match_batch(20)
    F = batched.fundamental(to_dev(Ks), to_dev(RTs))
    cost = batched.cost_tensor(F, to_dev(centers), to_dev(counts)).cpu().numpy()
    nsent = 0
    for s, sc in enumerate(epi_scenes()):
        N, M, P = counts[s]
        want = og.cost_tensor(centers[s, 0, :N], centers[s, 1, :M], centers[s, 2, :P], *sc['F'])
        assert np.array_equal(cost[s, :N, :M, :P].view(np.uint32), want.view(np.uint32)), s
        nsent += int((want > 1666).sum())
    assert nsent > 0                                      # the sentinel-line path (0, 0, 9999) is taken


@pytest.mark.gpu
@pytest.mark.parametrize('Dmax', [20, 640])
def test_match_triangulate_bit_exact_with_detections_at_epipoles(Dmax):
    """The full matcher on those scenes, in shared memory (Dmax 20) and in the workspace (Dmax 640): the oracle's idx in
    order and bit-equal costs (threshold 1e6, so the assignment itself is compared, sentinel costs included)."""
    from bpc_baseline_b200 import batched
    Ks, RTs, centers, counts = _epi_match_batch(Dmax)
    res = batched.match_triangulate(to_dev(Ks), to_dev(RTs), to_dev(centers), to_dev(counts), 1e6)
    idx, n, cost = res.idx.cpu().numpy(), res.n.cpu().numpy(), res.cost.cpu().numpy()
    for s in range(len(Ks)):
        cen = [centers[s, c, :counts[s, c]] for c in range(3)]
        want = og.match_scene(list(Ks[s]), list(RTs[s]), cen, 1e6)
        assert int(n[s]) == len(want['idx']), s
        assert np.array_equal(idx[s, :n[s]], want['idx']), s
        assert np.array_equal(cost[s, :n[s]].view(np.uint32), want['cost'].view(np.uint32)), s


# ---------------------------------------------------------------------------------------------------------------------
# fundamental matrix
# ---------------------------------------------------------------------------------------------------------------------
def _pivots(K):
    """Row swaps of the kernel's Gauss-Jordan (inv3_f32, csrc/geometry.cuh) on the float64 copy of K."""
    a = np.asarray(K, np.float64).copy()
    piv = []
    for col in range(3):
        p = col
        for r in range(col + 1, 3):
            if abs(a[r, col]) > abs(a[p, col]):
                p = r
        piv.append(p)
        a[[col, p]] = a[[p, col]]
        a[col] /= a[col, col]
        for r in range(3):
            if r != col:
                a[r] -= a[r, col] * a[col]
    return tuple(piv[:2])


@functools.lru_cache(maxsize=None)
def general_K_batch():
    """Scenes with general float32 K: every pivot pattern of the 3x3 inverse, K[8] != 1, nearly singular K."""
    rng = np.random.default_rng(91)
    Ks, RTs, kinds = [], [], []
    for t in range(240):
        K = rng.normal(size=(3, 3)) * np.array([1000.0, 1000.0, 1.0])[:, None] + np.diag([1400.0, 1400.0, 0.0])
        K[2] = rng.normal(size=3) * [1e-3, 1e-3, 1.0] + [0, 0, 1.5]
        K = K[rng.permutation(3)]
        if t % 4 == 3:                                     # nearly singular: row 2 close to a combination of 0 and 1
            K[2] = 0.3 * K[0] - 0.7 * K[1] + rng.normal(size=3) * 1e-5 * np.abs(K[0]).max()
        Ks.append(np.stack([K.astype(np.float32)] + [(K[rng.permutation(3)] * rng.uniform(0.5, 2)).astype(np.float32)
                                                     for _ in range(2)]))
        RTs.append(np.stack([og.calc_pose_matrix(_rot(rng), rng.normal(size=3)) for _ in range(3)]))
        kinds.append(t % 4 == 3)
    return np.stack(Ks), np.stack(RTs), np.array(kinds)


def test_general_K_cases_reach_every_pivot_pattern():
    Ks, _, sing = general_K_batch()
    pats = {_pivots(K) for K in Ks.reshape(-1, 3, 3)}
    assert pats == {(a, b) for a in range(3) for b in range(1, 3)}, pats
    assert np.all(Ks[..., 2, 2] != 1.0)
    assert np.median(np.linalg.cond(Ks[sing].reshape(-1, 3, 3).astype(np.float64))) > 1e4


@pytest.mark.gpu
def test_fundamental_general_intrinsics():
    """Within 1e-12 of the oracle for every well-conditioned general K.  For the nearly singular K neither the kernel's
    Gauss-Jordan nor LAPACK's LU gives the float64 inverse to better than ~cond(K) eps, so the two float32 inverses may
    round one float32 ulp apart; F, a product with cancellation, then differs by up to ~cond(K) 2^-24 relative (norm-wise),
    and that is the bound asserted there."""
    from bpc_baseline_b200 import batched
    Ks, RTs, sing = general_K_batch()
    F = batched.fundamental(to_dev(Ks), to_dev(RTs)).cpu().numpy()
    loose = 0
    for s in range(len(Ks)):
        want = np.stack(og.scene_fundamentals(list(Ks[s]), list(RTs[s])))
        if not sing[s]:
            np.testing.assert_allclose(F[s], want, rtol=1e-12, atol=0, err_msg=str(s))
            continue
        cond = np.linalg.cond(Ks[s].astype(np.float64)).max()
        for f in range(3):
            d = np.abs(F[s, f] - want[f]).max() / np.abs(want[f]).max()
            assert d <= cond * 2.0 ** -24, (s, f, d, cond)
            loose += d > 1e-12
    print(f'nearly singular K: {loose} of {3 * int(sing.sum())} F beyond 1e-12 of the oracle')


def _f22_scene(f22, rng):
    """Three cameras with principal point (0, 0): camera 1 at the origin with R = I, cameras 2 and 3 translated along x
    and rotated about x so that F12[2,2] and F13[2,2] (before normalisation) are ~f22 (0: exactly 0)."""
    Ks = np.stack([_K(np.float32(rng.uniform(800, 2000)), 0.0, 0.0) for _ in range(3)])
    RTs = [np.eye(4)]
    for _ in range(2):
        tx = float(np.float32(rng.uniform(0.2, 2.0) * rng.choice([-1, 1])))
        s = -f22 / tx if f22 else 0.0           # F[2,2] = E[2,2] = tx * R[1,2] = -tx * s
        c = math.sqrt(1 - s * s)
        R = np.array([[1, 0, 0], [0, c, -s], [0, s, c]])
        RTs.append(og.calc_pose_matrix(R, np.array([tx, 0.0, 0.0])))
    return Ks, np.stack(RTs)


def _raw_F22(K1, RT1, K2, RT2):
    """F[2,2] of fundamental_matrix before the normalisation (camera_utils.py:23-42)."""
    R1, R2, t1, t2 = RT1[:3, :3], RT2[:3, :3], RT1[:3, 3], RT2[:3, 3]
    R_rel = R2 @ R1.T
    t = t2 - R_rel @ t1
    tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]], dtype=np.float32)
    return (np.linalg.inv(K2).T @ (tx @ R_rel) @ np.linalg.inv(K1))[2, 2]


F22_VALUES = [0.0, 1e-9, -1e-9, 1e-7, -1e-7, 1e-8 * (1 + 1e-9), 1e-8 * (1 - 1e-9), -1e-8 * (1 + 1e-9)]


@functools.lru_cache(maxsize=None)
def f22_batch():
    rng = np.random.default_rng(5)
    Ks, RTs = zip(*[_f22_scene(v, rng) for v in F22_VALUES for _ in range(4)])
    return np.stack(Ks), np.stack(RTs)


def test_f22_cases_sit_where_they_claim():
    Ks, RTs = f22_batch()
    for s, v in enumerate(np.repeat(F22_VALUES, 4)):
        for a, b in ((0, 1), (0, 2)):
            raw = _raw_F22(Ks[s, a], RTs[s, a], Ks[s, b], RTs[s, b])
            if v == 0:
                assert raw == 0.0
            else:
                assert abs(raw - v) < 1e-3 * abs(v) and abs(abs(raw) - 1e-8) > 1e-12 * 1e-8


@pytest.mark.gpu
def test_fundamental_f22_branch():
    """Both sides of |F22| <= 1e-8 (no normalisation) against the oracle, and the same branch."""
    from bpc_baseline_b200 import batched
    Ks, RTs = f22_batch()
    F = batched.fundamental(to_dev(Ks), to_dev(RTs)).cpu().numpy()
    for s in range(len(Ks)):
        want = np.stack(og.scene_fundamentals(list(Ks[s]), list(RTs[s])))
        np.testing.assert_allclose(F[s], want, rtol=1e-12, atol=0, err_msg=str(s))
        assert np.array_equal(F[s, :, 2, 2] == 1.0, want[:, 2, 2] == 1.0), s


@pytest.mark.gpu
def test_match_triangulate_on_unnormalised_F():
    """F22 = 0 scenes (F12 and F13 not normalised) through the matcher, against the oracle."""
    from bpc_baseline_b200 import batched
    Ks, RTs = f22_batch()
    Ks, RTs = Ks[:4], RTs[:4]
    rng = np.random.default_rng(6)
    D = 8
    centers = np.zeros((4, 3, D, 2))
    for s in range(4):
        X = rng.normal(size=(D, 3)) * 0.3 + [0, 0, 4.0]
        for c in range(3):
            centers[s, c] = [_project(Ks[s, c], RTs[s, c], x) for x in X]
        centers[s] += rng.normal(size=centers[s].shape) * 0.5
    counts = np.full((4, 3), D, np.int32)
    res = batched.match_triangulate(to_dev(Ks), to_dev(RTs), to_dev(centers), to_dev(counts), 30, want_F=True)
    idx, n, cost = res.idx.cpu().numpy(), res.n.cpu().numpy(), res.cost.cpu().numpy()
    for s in range(4):
        want = og.match_scene(list(Ks[s]), list(RTs[s]), [centers[s, c] for c in range(3)], 30)
        assert want['F'][0, 2, 2] == 0.0 and int(n[s]) == len(want['idx']) > 0
        assert np.array_equal(idx[s, :n[s]], want['idx'])
        assert np.array_equal(cost[s, :n[s]].view(np.uint32), want['cost'].view(np.uint32))


# ---------------------------------------------------------------------------------------------------------------------
# post-match kernels at scale
# ---------------------------------------------------------------------------------------------------------------------
def _nan_view_scene(rng):
    """A scene whose third camera has the rows 0 and 2 of [R | t] zero: its P has rows 0 and 2 zero, so the
    reprojection error of that view is 0 / 0 = NaN, while F13 = F23 = 0 and every cost stays finite."""
    K = _K(1400.0, 960.0, 540.0)
    X = np.array([0.1, -0.2, 0.05])
    RT1 = _lookat(np.array([2.5, 0, 0.5]), X, rng)
    RT2 = _lookat(np.array([0, 2.5, 0.5]), X, rng)
    r = rng.normal(size=3)
    r /= np.linalg.norm(r)
    RT3 = np.zeros((4, 4))
    RT3[1, :3], RT3[1, 3], RT3[3, 3] = r, -r @ X, 1.0                  # X on the plane of row 1: views 1, 2 stay exact
    Ks = np.stack([K, K, K])
    RTs = np.stack([RT1, RT2, RT3])
    cen = np.array([_project(K, RT1, X), _project(K, RT2, X), [960.0, 700.0]])
    return Ks, RTs, cen


@functools.lru_cache(maxsize=None)
def _filter_batch():
    import torch
    from bpc_baseline_b200 import batched, synth
    b = synth.make_scenes(300, 6, seed=synth.SEED + 71, p_drop=0.2, sigma=3.0, n_false=1)
    Ks, RTs, centers, counts = b.Ks.copy(), b.RTs.copy(), b.centers.copy(), b.counts.copy()
    rng = np.random.default_rng(8)
    for s in (5, 150, 299):
        Ks[s], RTs[s], c = _nan_view_scene(rng)
        centers[s] = 0.0
        centers[s, :, 0] = c
        counts[s] = 1
    dev = tuple(to_dev(a) for a in (Ks, RTs, centers, counts))
    base = batched.match_triangulate(*dev, 1e4, want_reproj=True)
    torch.cuda.synchronize()
    return dev, {k: getattr(base, k).cpu().numpy() for k in ('idx', 'n', 'cost', 'X', 'reproj')}


def _filtered(base, t):
    """NumPy restatement of bpc_match_filter_kernel: keep a match unless some view's error is > t."""
    S, K, _ = base['idx'].shape
    out = {'idx': np.full((S, K, 3), -1, np.int32), 'n': base['n'].copy(), 'cost': np.full((S, K), np.nan, np.float32),
           'X': np.full((S, K, 3), np.nan), 'reproj': np.full((S, K, 3), np.nan)}
    for s in range(S):
        n = int(base['n'][s])
        if n <= 0:
            for k in out:
                if k != 'n':
                    out[k][s] = base[k][s]
            continue
        keep = np.flatnonzero(~(base['reproj'][s, :n] > t).any(axis=1))
        out['n'][s] = len(keep)
        for k in ('idx', 'cost', 'X', 'reproj'):
            out[k][s, :len(keep)] = base[k][s, keep]
    return out


@pytest.mark.gpu
def test_reprojection_filter_at_scale():
    """300 scenes (three blocks).  Thresholds 0 (every match with a positive error dropped), +inf, and exactly a stored
    error (kept: the test is `>`); the NaN scenes keep their match, since NaN never exceeds the threshold."""
    from bpc_baseline_b200 import batched
    dev, base = _filter_batch()
    n = base['n']
    for s in (5, 150, 299):
        assert n[s] == 1 and np.isnan(base['reproj'][s, 0, 2]) and np.isfinite(base['reproj'][s, 0, :2]).all()
    valid = np.arange(base['idx'].shape[1])[None] < n[:, None]
    worst = np.where(valid, np.nanmax(np.where(valid[..., None], base['reproj'], 0.0), axis=-1), np.nan)
    errs = np.sort(worst[valid & np.isfinite(base['reproj']).all(-1)])
    ties = [float(errs[len(errs) // 3]), float(errs[len(errs) // 2]), float(errs[-2])]
    for t in [0.0, float('inf')] + ties:
        res = batched.match_triangulate(*dev, 1e4, reproj_thresh=t)
        got = {k: getattr(res, k).cpu().numpy() for k in ('idx', 'n', 'cost', 'X', 'reproj')}
        want = _filtered(base, t)
        assert np.array_equal(got['n'], want['n']), t
        for k in ('idx', 'cost', 'X', 'reproj'):
            assert np.array_equal(got[k], want[k], equal_nan=True), (t, k)
        for s in (5, 150, 299):                             # a NaN error is kept: only the finite views decide
            assert got['n'][s] == int(t >= np.nanmax(base['reproj'][s, 0])), t
        if t in ties:                                       # the match holding exactly t as its largest error is kept
            hit = np.argwhere(worst == t)
            assert len(hit)
            for s, m in hit:
                assert any(np.array_equal(got['idx'][s, q], base['idx'][s, m]) for q in range(got['n'][s])), (t, s, m)
        if t == 0.0:
            assert ((got['n'] == 0) & (n > 0)).sum() > 200  # whole scenes dropped and re-padded


@pytest.mark.gpu
@pytest.mark.parametrize('S', [1, 1023, 1024, 1025, 3000])
def test_build_rois_at_scale(S):
    """bpc_build_rois against a NumPy restatement: S > 1024 gives a scan thread several scenes, S = 3000 x 40 x 3 ROI
    slots (360 000 > 148 x 8 x 256) sends the fill kernel round its grid-stride loop; n takes 0, -1 and -2."""
    from bpc_baseline_b200 import batched
    K, D = 40, 7
    rng = np.random.default_rng(S)
    n = rng.integers(-2, K + 1, S).astype(np.int32)
    n[: min(S, 3)] = [-2, -1, 0][: min(S, 3)]
    if S > 10:
        n[-1] = K
    idx = rng.integers(0, D, (S, K, 3)).astype(np.int32)
    boxes = rng.integers(-2**31, 2**31 - 1, (S, 3, D, 4), dtype=np.int64).astype(np.int32)
    ios = rng.integers(-2**31, 2**31 - 1, (S, 3), dtype=np.int64).astype(np.int32)
    rois, offs = batched.build_rois(to_dev(boxes), to_dev(idx), to_dev(n), to_dev(ios))
    rois, offs = rois.cpu().numpy(), offs.cpu().numpy()
    cnt = 3 * np.maximum(n, 0).astype(np.int64)
    want_offs = np.concatenate([[0], np.cumsum(cnt)])
    assert np.array_equal(offs, want_offs)
    want = np.zeros((int(want_offs[-1]), 5), np.int32)
    for s in range(S):
        for m in range(max(int(n[s]), 0)):
            for v in range(3):
                r = want_offs[s] + 3 * m + v
                want[r, 0] = ios[s, v]
                want[r, 1:] = boxes[s, v, idx[s, m, v]]
    assert np.array_equal(rois[: len(want)], want)


@pytest.mark.gpu
@pytest.mark.parametrize('S', [1, 2, 3, 5, 1025])
@pytest.mark.parametrize('with_reproj', [True, False])
@pytest.mark.parametrize('offset_div', [1, 3])
def test_pack_records_every_count_padding(S, with_reproj, offset_div):
    """bpc_pack_records byte for byte against pack_records_torch over the used bytes, on a buffer that starts as 0xFF;
    S mod 4 = 1, 2, 3, 1 (and 0 records) covers every padding of the counts; negative n; reproj=None gives NaN."""
    import torch
    from bpc_baseline_b200 import batched, distributed
    K = 6
    rng = np.random.default_rng([S, offset_div, with_reproj])
    n = rng.integers(-2, K + 1, S).astype(np.int32)
    n[0] = -1 if S > 1 else n[0]
    idx = rng.integers(-5, 100, (S, K, 3)).astype(np.int32)
    cost = rng.normal(size=(S, K)).astype(np.float32)
    X = rng.normal(size=(S, K, 3))
    rep = rng.normal(size=(S, K, 3)) if with_reproj else None
    res = batched.MatchResult(to_dev(idx), to_dev(n), to_dev(cost), to_dev(X), to_dev(rep) if with_reproj else None, None)
    off = np.concatenate([[0], np.cumsum(np.maximum(n, 0))]).astype(np.int32) * offset_div
    nbytes = distributed.records_bytes(S, K)
    out = torch.full((nbytes,), 0xFF, dtype=torch.uint8, device='cuda')
    buf = batched.pack_records(res, to_dev(off), offset_div, out=out).cpu().numpy()
    want = distributed.pack_records_torch(res.idx, res.n, res.cost, res.X, res.reproj).cpu().numpy()
    total = int(np.maximum(n, 0).sum())
    used = nbytes - (S * K - total) * 64
    assert np.array_equal(buf[:used], want[:used])
    head = buf[:16].view(np.int32)
    assert list(head) == [total, S, K, 0]
    base = 16 + ((S * 4 + 15) & ~15)
    assert np.array_equal(buf[16:16 + 4 * S].view(np.int32), n) and not buf[16 + 4 * S:base].any()
    if not with_reproj and total:
        recs = buf[base:base + 64 * total].view(np.float64).reshape(total, 8)
        assert np.isnan(recs[:, 5:]).all()


def _tie_scales():
    """(w, s) with w * s exactly k + 0.5 in float64, and the float64 neighbours of s."""
    from fractions import Fraction
    out = []
    for w in range(1, 1200):
        for q in range(2 * w + 1, int(2.4 * w), 2):           # w * s = q / 2, s in [1, 1.2]
            s = q / (2 * w)
            if Fraction(w) * Fraction(s) == Fraction(q, 2):
                out += [(w, s), (w, float(np.nextafter(s, 0))), (w, float(np.nextafter(s, 2)))]
    return out


@pytest.mark.gpu
def test_train_rois_ties_and_clamps():
    """bpc_train_rois against oracle.crop.dataset_window: round-half-even at exact ties of w * s (and either side),
    shifts past both image edges, windows clamped to width 1 at x1 = W - 1, image=None, n not a multiple of 256."""
    from bpc_baseline_b200 import batched
    W, H = 1920, 1080
    rng = np.random.default_rng(12)
    ties = _tie_scales()
    assert sum(1 for w, s in ties if (w * s) % 1 == 0.5) > 300
    n = len(ties) + 1000
    n += (-n) % 256 + 77                                    # not a multiple of 256
    xywh = np.zeros((n, 4), np.int64)
    scale = rng.uniform(1.0, 1.2, n)
    shift = rng.integers(-300, 300, (n, 2))
    xywh[:, 0] = rng.integers(0, W, n); xywh[:, 1] = rng.integers(0, H, n)
    xywh[:, 2] = rng.integers(1, 500, n); xywh[:, 3] = rng.integers(1, 500, n)
    for r, (w, s) in enumerate(ties):                       # at x = y = 0 and no shift, no clamp hides the rounding
        xywh[r], scale[r], shift[r] = (0, 0, w, w), s, 0
    m = len(ties)
    shift[m:m + 200, 0] = xywh[m:m + 200, 0] + rng.integers(1, 400, 200)          # x - sx < 0
    shift[m + 200:m + 400, 0] = xywh[m + 200:m + 400, 0] - W - rng.integers(0, 400, 200)   # x - sx > W - 1
    shift[m + 400:m + 600, 1] = xywh[m + 400:m + 600, 1] - H - rng.integers(0, 400, 200)   # y1 = H - 1
    xywh = xywh.astype(np.int32); shift = shift.astype(np.int32)
    for image in (None, rng.integers(0, 1000, n).astype(np.int32)):
        got = batched.train_rois(to_dev(xywh), W, H, image=None if image is None else to_dev(image), scale=to_dev(scale),
                                 shift=to_dev(shift)).cpu().numpy()
        want = np.array([(0 if image is None else image[r],) + ocrop.dataset_window(xywh[r], W, H, scale[r], shift[r])
                         for r in range(n)], np.int32)
        assert np.array_equal(got, want)
    assert (want[:, 1] == W - 1).sum() >= 200 and ((want[:, 3] - want[:, 1]) == 1).sum() >= 200
    assert (want[:, 1] == 0).sum() >= 200
