"""Helpers shared by the -m gpu parity tests."""
import numpy as np
import torch


def to_dev(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def pack_scenes(scenes):
    """List of golden scene dicts (tests/conftest.py) -> batched arrays padded to a common Dmax."""
    D = max(int(sc['centers_arr'].shape[1]) for sc in scenes)
    S = len(scenes)
    Ks = np.zeros((S, 3, 3, 3), np.float32)
    RTs = np.zeros((S, 3, 4, 4), np.float64)
    centers = np.zeros((S, 3, D, 2), np.float64)
    boxes = np.zeros((S, 3, D, 4), np.int32)
    counts = np.zeros((S, 3), np.int32)
    for s, sc in enumerate(scenes):
        d = sc['centers_arr'].shape[1]
        Ks[s], RTs[s], counts[s] = sc['Ks_arr'], sc['RTs_arr'], sc['counts']
        centers[s, :, :d] = sc['centers_arr']
        boxes[s, :, :d] = sc['boxes']
    return Ks, RTs, centers, boxes, counts


def batch_to_dev(batch):
    return (to_dev(batch.Ks), to_dev(batch.RTs), to_dev(batch.centers), to_dev(batch.boxes), to_dev(batch.counts))


def rel_err(a, b):
    """Norm-wise relative error per row (SURVEY.md a8: ||dX|| / ||X_ref||)."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.linalg.norm(a - b, axis=-1) / np.maximum(np.linalg.norm(b, axis=-1), 1e-300)


def check_match_properties(batch, out, threshold=30.0, min_recovery=None):
    """Size-independent properties of match_triangulate's outputs (every scene must have n >= 0)."""
    idx, n, cost, X, reproj = out['idx'], out['n'], out['cost'], out['X'], out['reproj']
    S, K, _ = idx.shape
    cnt = batch.counts.astype(np.int64)
    assert np.all(n >= 0) and np.all(n <= np.minimum(cnt[:, 0] * cnt[:, 1], cnt[:, 2]))   # min(N*M, P) assignments (F2)
    slot = np.arange(K)[None, :]
    valid = slot < n[:, None]
    # padding / validity
    assert np.all(idx[~valid] == -1) and np.all(np.isnan(cost[~valid]))
    assert np.all(idx[valid] >= 0)
    for c in range(3):
        assert np.all(idx[..., c][valid] < np.broadcast_to(batch.counts[:, c:c + 1], (S, K))[valid])
    # threshold and order: costs < threshold, non-decreasing; ties in ascending r = i*M + j (process_pose.py:183)
    assert np.all(cost[valid] < np.float32(threshold))
    c0, c1 = cost[:, :-1], cost[:, 1:]
    both = valid[:, 1:]
    assert np.all(c0[both] <= c1[both])
    r = idx[..., 0].astype(np.int64) * batch.counts[:, 1:2] + idx[..., 1]
    tie = both & (c0 == c1)
    assert np.all(r[:, :-1][tie] < r[:, 1:][tie])
    # a rectangular assignment: third-camera detections are used at most once, (i, j) pairs at most once
    big = 1 << 40
    kk = np.where(valid, idx[..., 2], -1 - slot).astype(np.int64)
    assert all(len(np.unique(row)) == K for row in kk[:: max(1, S // 512)])
    rr = np.where(valid, r, -big - slot)
    assert all(len(np.unique(row)) == K for row in rr[:: max(1, S // 512)])
    # triangulation: finite, and consistent with the detections (reprojection error of a 3-view DLT)
    assert np.all(np.isfinite(X[valid])) and np.all(np.isfinite(reproj[valid]))
    assert np.median(reproj[valid]) < 5.0
    if min_recovery is not None:
        s_ix = np.repeat(np.arange(S), K).reshape(S, K)
        t0 = batch.truth[s_ix, 0, idx[..., 0].clip(min=0)]
        t1 = batch.truth[s_ix, 1, idx[..., 1].clip(min=0)]
        t2 = batch.truth[s_ix, 2, idx[..., 2].clip(min=0)]
        same = (t0 == t1) & (t1 == t2) & (t0 >= 0)
        assert same[valid].mean() >= min_recovery, same[valid].mean()


def oracle_match(job):
    """og.match_scene on one (Ks, RTs, centers) job; the ValueError SciPy raises is returned, not raised."""
    from oracle import geometry as og
    Ks, RTs, cen = job
    try:
        return og.match_scene(Ks, RTs, cen, 30, cost_fn=og.cost_tensor_fast)
    except ValueError as e:
        return e


def oracle_map(jobs, workers):
    """oracle_match over the jobs, fanned out over at most ``workers`` spawned processes (one at a time if 1)."""
    jobs = list(jobs)
    if workers <= 1 or len(jobs) <= 1:
        return [oracle_match(j) for j in jobs]
    import concurrent.futures as cf
    import multiprocessing as mp
    import os
    nproc = min(workers, len(jobs), len(os.sched_getaffinity(0)))
    with cf.ProcessPoolExecutor(nproc, mp_context=mp.get_context('spawn')) as pool:
        return list(pool.map(oracle_match, jobs))
