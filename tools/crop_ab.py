#!/usr/bin/env python
"""A/B of crop-kernel builds on one GPU: the config-4 side ranges timed per library, with a checksum of the float32 output
so that a faster variant whose bytes differ is caught in the same run.

    python tools/crop_ab.py [--reps N] libA.so libB.so ...      # paths relative to the repo root; each runs in its own process

Environment: RANGES (box side ranges in px), T (target size, default 224), POOL_W (pool width in px, default 3840; boxes are
clipped to it).  The crop count scales as 1 / T^2, so every T writes about the output bytes of 16384 crops at T = 224.
LAYOUT: `random` (default) places the boxes anywhere in a pool of 24 images, so crops overlap as the detections of a
shared pool do; `disjoint` gives every box a grid cell of its own (hi x hi px, cells in random list order) in a pool of
as many noise images as that takes (9 GB for 60-400 px, 51 GB for 300-900 px), so no source pixel is read by two crops.

Build variants here first (nvcc cross-compiles):  python -c "from bpc_baseline_b200 import build; build.build(True, defines=['X'], out='...')"
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RANGES = tuple(tuple(int(v) for v in r.split('-')) for r in os.environ.get('RANGES', '60-400,300-900,32-96').split(','))
T = int(os.environ.get('T', 224))
POOL_W = int(os.environ.get('POOL_W', 3840))
LAYOUT = os.environ.get('LAYOUT', 'random')


def one(reps):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import numpy as np
    import torch
    import bench_configs as bc
    from bpc_baseline_b200 import batched, pipeline, synth
    if LAYOUT not in ('random', 'disjoint'):
        raise SystemExit(f'LAYOUT must be random or disjoint, not {LAYOUT!r}')
    out = {}
    R, B = 16384 * 224 * 224 // (T * T), 8
    images = bc.dev(synth.make_images(B * 3, seed=44, width=POOL_W)) if LAYOUT == 'random' else None
    buf = torch.empty((R, 3, T, T), dtype=torch.float32, device='cuda')
    for lo, hi in RANGES:
        rng = np.random.default_rng([44, lo, hi, T])
        w = np.minimum(rng.integers(lo, hi, R), POOL_W); h = rng.integers(lo, hi, R)
        if LAYOUT == 'random':
            x1 = (rng.random(R) * (POOL_W - w)).astype(np.int64); y1 = (rng.random(R) * (synth.IMG_H - h)).astype(np.int64)
            img = rng.integers(0, B * 3, R)
            pool = images
        else:
            nx, ny = POOL_W // hi, synth.IMG_H // hi
            cell = rng.permutation(R)
            img, cx, cy = cell // (nx * ny), cell % nx, (cell // nx) % ny
            x1 = cx * hi + (rng.random(R) * (hi - w + 1)).astype(np.int64)
            y1 = cy * hi + (rng.random(R) * (hi - h + 1)).astype(np.int64)
            gen = torch.Generator(device='cuda').manual_seed(44)
            pool = torch.randint(0, 256, (int(img.max()) + 1, synth.IMG_H, POOL_W, 3), dtype=torch.uint8, device='cuda',
                                 generator=gen)
        rois = np.stack([img, x1, y1, x1 + w, y1 + h], axis=1).astype(np.int32)
        drois = bc.dev(rois)
        buf.zero_()
        ms = bc.timed(lambda: batched.roi_crop(pool, drois, T=T, out=buf), warm=3, reps=reps)
        nbytes = pipeline.algorithmic_crop_bytes(rois, T)
        chk = int(buf.view(torch.int32).to(torch.int64).sum().item())
        out[f'{lo}-{hi}'] = {'ms': round(ms, 4), 'frac': round(nbytes / ms / 1e6 / bc.PEAK, 4), 'chk': chk}
        del pool
    print(json.dumps(out))


if __name__ == '__main__':
    args = sys.argv[1:]
    reps = 10
    if '--reps' in args:
        i = args.index('--reps'); reps = int(args[i + 1]); del args[i:i + 2]
    if args and args[0] == '--one':
        one(reps)
        sys.exit(0)
    ref = None
    for lib in args:
        env = dict(os.environ, BPC_LIB=os.path.join(ROOT, lib))
        r = subprocess.run([sys.executable, os.path.abspath(__file__), '--one', '--reps', str(reps)], env=env, capture_output=True, text=True)
        if r.returncode != 0:
            print(f'{lib}: FAILED\n{r.stderr[-2000:]}')
            continue
        res = json.loads(r.stdout.strip().splitlines()[-1])
        if ref is None:
            ref = res
        line = f'{lib:40s}'
        for k, v in res.items():
            same = 'ok ' if v['chk'] == ref[k]['chk'] else 'DIFF'
            line += f'  {k}: {v["ms"]:7.3f} ms {v["frac"]:.3f} {same}'
        print(line, flush=True)
