#!/usr/bin/env python
"""A/B of crop-kernel builds on one GPU: the config-4 side ranges timed per library, with a checksum of the float32 output
so that a faster variant whose bytes differ is caught in the same run.

    python tools/crop_ab.py [--reps N] libA.so libB.so ...      # paths relative to the repo root; each runs in its own process

Environment: RANGES (box side ranges in px), T (target size, default 224), POOL_W (pool width in px, default 3840; boxes are
clipped to it).  The crop count scales as 1 / T^2, so every T writes about the output bytes of 16384 crops at T = 224.

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


def one(reps):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import numpy as np
    import torch
    import bench_configs as bc
    from bpc_baseline_b200 import batched, pipeline, synth
    out = {}
    R, B = 16384 * 224 * 224 // (T * T), 8
    images = bc.dev(synth.make_images(B * 3, seed=44, width=POOL_W))
    buf = torch.empty((R, 3, T, T), dtype=torch.float32, device='cuda')
    for lo, hi in RANGES:
        rng = np.random.default_rng([44, lo, hi, T])
        w = np.minimum(rng.integers(lo, hi, R), POOL_W); h = rng.integers(lo, hi, R)
        x1 = (rng.random(R) * (POOL_W - w)).astype(np.int64); y1 = (rng.random(R) * (synth.IMG_H - h)).astype(np.int64)
        rois = np.stack([rng.integers(0, B * 3, R), x1, y1, x1 + w, y1 + h], axis=1).astype(np.int32)
        drois = bc.dev(rois)
        buf.zero_()
        ms = bc.timed(lambda: batched.roi_crop(images, drois, T=T, out=buf), warm=3, reps=reps)
        nbytes = pipeline.algorithmic_crop_bytes(rois, T)
        chk = int(buf.view(torch.int32).to(torch.int64).sum().item())
        out[f'{lo}-{hi}'] = {'ms': round(ms, 4), 'frac': round(nbytes / ms / 1e6 / bc.PEAK, 4), 'chk': chk}
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
