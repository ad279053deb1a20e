#!/usr/bin/env python
"""Training-side ColorJitter (bpc_color_jitter) on one GPU: uint8 canvases [n,T,T,3] -> jittered, normalised f32 [n,3,T,T].

For each T: 16 384 resident canvases (3.2 GB at T = 256, larger than the 126 MB L2, so every pass reads HBM), timed with
CUDA events for all four ops, each op alone, brightness + contrast + saturation (hue off) and no op, next to
bpc_crops_normalise on the same canvases, which reads and writes the same bytes without the jitter.  Achieved GB/s counts
the algorithmic bytes, 3 T^2 read + 12 T^2 written per crop (phase 1's second read of a crop comes from L2).  The CPU
column is the per-sample path of a DataLoader worker: PIL ColorJitter + to_tensor + normalize on one core.

    python tools/bench_color_jitter.py [--crops 16384] [--reps 10] [--cpu-samples 200]      -> one JSON object
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# torchvision ColorJitter arguments per case; the reference's own ranges cannot be read from this repository
CASES = {
    'all_four': dict(brightness=0.4, contrast=0.4, saturation=0.4, hue=0.1),
    'hue_off': dict(brightness=0.4, contrast=0.4, saturation=0.4),
    'brightness': dict(brightness=0.4),
    'contrast': dict(contrast=0.4),
    'saturation': dict(saturation=0.4),
    'hue': dict(hue=0.1),
    'none': dict(),
}


def gpu_info():
    import torch
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = q.stdout.strip()
    except Exception as e:                                        # informative only
        info['power_limit_and_max_sm_clock'] = f'unavailable ({type(e).__name__})'
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--crops', type=int, default=16384)
    ap.add_argument('--targets', default='256,224')
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--cpu-samples', type=int, default=200)
    args = ap.parse_args()
    import numpy as np
    import torch
    from bpc_baseline_b200 import batched
    from bpc_baseline_b200.utils.data_utils import draw_color_jitter
    if not torch.cuda.is_available():
        raise SystemExit('bench_color_jitter needs a CUDA device')
    try:
        peak = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))['hbm_gbs']
    except Exception:
        peak = 6562.9
    dev = torch.device('cuda')
    n = args.crops

    def timed(fn, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.reps

    out = {'gpu': gpu_info(), 'crops': n, 'peak_GBps': peak, 'cases': {k: v for k, v in CASES.items()},
           'canvases': 'uniform random bytes (every pixel a random colour: the hue step never takes its grey shortcut)'}
    gen = torch.Generator(device=dev).manual_seed(0)
    for T in [int(t) for t in args.targets.split(',')]:
        canv = torch.randint(0, 256, (n, T, T, 3), dtype=torch.uint8, device=dev, generator=gen)
        dst = torch.empty((n, 3, T, T), dtype=torch.float32, device=dev)
        nbytes = 15 * T * T * n
        rate = lambda ms: {'ms': ms, 'crops_per_s': n / ms * 1e3, 'GBps': nbytes / ms / 1e6, 'frac_of_peak': nbytes / ms / 1e6 / peak}
        res = {'algorithmic_bytes': nbytes, 'canvas_bytes': 3 * T * T * n}
        ms_norm = timed(lambda: batched.crops_normalise([canv], T, swap_rb=False, out=dst))
        res['crops_normalise'] = rate(ms_norm)
        for name, kw in CASES.items():
            torch.manual_seed(1)
            order, factors = draw_color_jitter(n, **kw)
            o, f = torch.as_tensor(order).to(dev), torch.as_tensor(factors).to(dev)
            ms = timed(lambda: batched.color_jitter(canv, o, f, out=dst))
            res['color_jitter_' + name] = dict(rate(ms), vs_crops_normalise=ms_norm / ms)
        ms_norm2 = timed(lambda: batched.crops_normalise([canv], T, swap_rb=False, out=dst))   # drift check, same command
        res['crops_normalise_again'] = rate(ms_norm2)
        out[f'T{T}'] = res
        if T == 256 and args.cpu_samples > 0:
            out['cpu_per_sample_T256'] = cpu_path(canv[:args.cpu_samples].cpu().numpy())
        del canv, dst
        torch.cuda.empty_cache()
    print(json.dumps(out))


def cpu_path(canvases):
    """DataLoader-worker path on one core: Image.fromarray -> ColorJitter -> to_tensor -> normalize."""
    import torch
    import torchvision.transforms as T
    import torchvision.transforms.functional as TF
    from PIL import Image
    torch.set_num_threads(1)
    cj = T.ColorJitter(**CASES['all_four'])
    mean, std = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
    for c in canvases[:5]:
        TF.normalize(TF.to_tensor(cj(Image.fromarray(c))), mean, std)
    t0 = time.perf_counter()
    for c in canvases:
        TF.normalize(TF.to_tensor(cj(Image.fromarray(c))), mean, std)
    s = time.perf_counter() - t0
    return {'samples': len(canvases), 'threads': 1, 's': s, 'crops_per_s': len(canvases) / s, 'ops': 'all_four'}


if __name__ == '__main__':
    main()
