"""BASELINE.json configurations at their full sizes, checked through size-independent properties (plus the
oracle on a sample of scenes / ROIs): config 2 (4 096 x D=20), config 3 (dense bin, 16 384 x D=200), config 4
(crop-only sweep, 64 matches per scene, three side ranges) and config 5 (131 072 scenes)."""
import numpy as np
import pytest
import torch

from oracle import crop as ocrop
from tests.gpu_util import batch_to_dev, check_match_properties, oracle_map, rel_err, to_dev

pytestmark = pytest.mark.gpu


def _match(batch, threshold=30):
    from bpc_baseline_b200 import batched
    Ks, RTs, centers, boxes, counts = batch_to_dev(batch)
    res = batched.match_triangulate(Ks, RTs, centers, counts, threshold)
    torch.cuda.synchronize()
    return {k: getattr(res, k).cpu().numpy() for k in ('idx', 'n', 'cost', 'X', 'reproj')}


def _check_against_oracle(batch, out, scenes):
    scenes = list(scenes)
    jobs = []
    for s in scenes:
        Ks, RTs = batch.capture_arrays(s)
        jobs.append((Ks, RTs, [batch.centers[s, c, :batch.counts[s, c]] for c in range(3)]))
    # a D = 200 scene costs the oracle ~0.3 s: fan a large sample out over the host cores
    wants = oracle_map(jobs, 16 if len(scenes) > 16 else 1)
    for s, want in zip(scenes, wants):
        assert not isinstance(want, Exception), (s, want)
        widx, wcost, wX = want['idx'], want['cost'], want['X']
        n = int(out['n'][s])
        assert n == len(widx) and np.array_equal(out['idx'][s, :n], widx), s
        if n:
            assert np.array_equal(out['cost'][s, :n].view(np.uint32), wcost.view(np.uint32)), s
            assert rel_err(out['X'][s, :n], wX).max() < 1e-9, s


def test_config2_batch_4096x20():
    from bpc_baseline_b200 import synth
    batch = synth.make_scenes(4096, 20)
    out = _match(batch)
    assert int(out['n'].sum()) == 4096 * 20                      # clean scenes: every object matched
    check_match_properties(batch, out, min_recovery=0.99)
    _check_against_oracle(batch, out, range(0, 4096, 256))


def test_config3_dense_bin_16384x200():
    from bpc_baseline_b200 import synth
    batch = synth.make_scenes(16384, 200)
    out = _match(batch)
    check_match_properties(batch, out, min_recovery=0.9)
    assert out['n'].mean() > 190
    _check_against_oracle(batch, out, [0, 9999])


def test_config3_dense_bin_with_dropped_detections():
    """Robustness variant of config 3 (p_drop 0.1, sigma 2 px): every scene has argmin conflicts, so the full
    shortest-augmenting-path search runs on 40 000-column problems."""
    from bpc_baseline_b200 import synth
    batch = synth.make_scenes(512, 200, p_drop=0.1, sigma=2.0, seed=synth.SEED + 31)
    out = _match(batch)
    check_match_properties(batch, out)
    _check_against_oracle(batch, out, [0, 300])


@pytest.mark.parametrize('D,p_drop,sigma,n_dup,n_false,nscenes', [(48, 0.25, 3.0, 3, 3, 96), (96, 0.15, 2.0, 5, 4, 32),
                                                                 (200, 0.1, 2.0, 0, 0, 128), (200, 0.3, 3.0, 6, 6, 128),
                                                                 (200, 0.0, 1.0, 0, 0, 128)])
def test_conflict_heavy_scenes_match_scipy(D, p_drop, sigma, n_dup, n_false, nscenes):
    """Every scene here runs the full shortest-augmenting-path search several times (dropped, duplicated and false
    detections): the pruned column scan of the Dijkstra step must reproduce SciPy's choice of optimum, scene by scene."""
    from bpc_baseline_b200 import synth
    batch = synth.make_scenes(nscenes, D, p_drop=p_drop, sigma=sigma, n_dup=n_dup, n_false=n_false, seed=synth.SEED + 57)
    out = _match(batch)
    check_match_properties(batch, out)
    _check_against_oracle(batch, out, range(nscenes))


def test_config5_131072_scenes_in_shards():
    """Config 5 on one GPU: the 131 072-scene stream in 8 shards of 16 384 (what 8 ranks would each take)."""
    from bpc_baseline_b200 import distributed, synth
    total = 0
    for rank in range(8):
        lo, hi = distributed.shard_range(131072, rank, 8, synth.CHUNK)
        batch = synth.make_scenes(hi - lo, 20, first=lo)
        out = _match(batch)
        total += int(out['n'].sum())
        if rank in (0, 7):
            check_match_properties(batch, out, min_recovery=0.99)
            _check_against_oracle(batch, out, [0, hi - lo - 1])
    assert total == 131072 * 20


@pytest.mark.parametrize('lo,hi', [(32, 96), (60, 400), (300, 900)])
def test_config4_crop_sweep(lo, hi):
    """64 matches per scene (192 ROIs), full-resolution 3-view images, T=224, through the chunked pipeline
    buffers; a sample of ROIs is compared bit-for-bit with the reference's four library calls."""
    from bpc_baseline_b200 import batched, synth
    B, scenes = 6, 96
    images = synth.make_images(B, seed=44)
    rng = np.random.default_rng([44, lo, hi])
    R = scenes * 192
    w = rng.integers(lo, hi, R); h = rng.integers(lo, hi, R)
    x1 = (rng.random(R) * (synth.IMG_W - w)).astype(np.int64); y1 = (rng.random(R) * (synth.IMG_H - h)).astype(np.int64)
    rois = np.stack([rng.integers(0, B, R), x1, y1, x1 + w, y1 + h], axis=1).astype(np.int32)
    dimg = to_dev(images)
    chunk = 4096
    out = torch.empty((chunk, 3, 224, 224), dtype=torch.float32, device='cuda')
    status = torch.zeros(R, dtype=torch.int32, device='cuda')
    drois = to_dev(rois)
    sample = set(int(v) for v in rng.choice(R, 48, replace=False))
    white = batched.normalise_lut('cuda')[:, 255].cpu().numpy()
    checked = 0
    for first in range(0, R, chunk):
        r = min(chunk, R - first)
        batched.roi_crop(dimg, drois[first:first + r], T=224, out=out, status=status[first:first + r])
        for g in sorted(s for s in sample if first <= s < first + r):
            got = out[g - first].cpu().numpy()
            b, bx1, by1, bx2, by2 = rois[g]
            want = ocrop.crop_tensor_ref(images[b], (bx1, by1, bx2, by2), target_size=224, swap_rb=True)
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (g, tuple(rois[g]))
            # letterbox padding is the normalised white constant
            _, nw, nh, dx, dy = ocrop.letterbox_geometry(by2 - by1, bx2 - bx1, 224)
            pad = np.ones((224, 224), bool); pad[dy:dy + nh, dx:dx + nw] = False
            assert np.all(got[:, pad] == white[:, None])
            checked += 1
    assert checked == 48 and int(status.sum()) == 0
    assert bool(torch.isfinite(out).all())
