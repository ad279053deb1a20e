#!/usr/bin/env python
"""bench.py -- throughput of the match + triangulate + ROI-crop hot path on B200s of one node.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 2 --warmup 1       # CPU arm (oracle port, all host cores)

A step = one pass of the hot path over one batch of synthetic scenes: fundamental matrices, virtual epipolar cost
tensor, SciPy-exact assignment, DLT triangulation + reprojection error, and the 224x224 float32 network input of
EVERY matched detection in all three views, produced chunk-wise into a reusable buffer.

  N = 1   BASELINE.json config 2: 4,096 3-camera scenes x 20 detections (245,760 crops, 148 GB of output per step).
          The line also carries `configs`: config 1 (single-scene latency through the CUDA-graphed SceneSession and
          through the reference's Python call surface), config 3 (dense bin, 16,384 x 200, clean and stress), config 4
          (crop-only sweep over three side ranges, a roofline fraction each) and config 5 on this one GPU.
  N > 1   BASELINE.json config 5: 131,072 scenes sharded over the ranks (strong scaling: distributed.shard_range), the
          64-byte pose records (idx, cost, X, reproj) packed by one kernel and all-gathered over NCCL every step;
          crops stay on the GPU that made them (their consumer, the pose network, is data-parallel too).  Rank 0
          recomputes a sample of every other rank's scenes and compares the gathered records bit for bit
          (`multi_rank_parity`).  `weak_config2` = config 2 per rank (the round-1 workload), `crop_gather` = the
          separate crops-to-rank-0 stage.

One JSON line is printed by rank 0; see the keys in main().
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'matched+triangulated scenes/s with the ROI crops of every match (crops/s alongside)'
UNIT = 'scenes/s'


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--scenes', type=int, default=4096, help='scenes per step at N = 1 (config 2), and per GPU in weak_config2')
    ap.add_argument('--total-scenes', type=int, default=131072, help='scenes per step over ALL ranks at N > 1 (config 5, strong scaling)')
    ap.add_argument('--no-configs', action='store_true', help='skip the `configs` object (configs 1, 3, 4, 5) at N = 1')
    ap.add_argument('--cpu-scenes-as-written', type=int, default=64, help='scenes in the as-written (Python triple loop) CPU sample')
    ap.add_argument('--dets', type=int, default=20, help='detections per camera')
    ap.add_argument('--target', type=int, default=224, help='crop side T')
    ap.add_argument('--pool', type=int, default=8, help='image pool: number of 3-view full-resolution triplets')
    ap.add_argument('--chunk-rois', type=int, default=16384, help='ROIs per crop launch (16384 x 602 KB = 9.9 GB chunk buffer)')
    ap.add_argument('--p-drop', type=float, default=0.0)
    ap.add_argument('--sigma', type=float, default=1.0)
    ap.add_argument('--no-crops', action='store_true', help='geometry only (dense-bin experiments)')
    ap.add_argument('--cpu-scenes', type=int, default=256, help='scenes in the bounded CPU-baseline sample (~12 s on one core)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-crop-gather', action='store_true', help='skip the separate crop-gather stage at N > 1')
    ap.add_argument('--gather-chunk', type=int, default=4096, help='uint8 crops per rank and chunk in the crop-gather stage')
    ap.add_argument('--gather-steps', type=int, default=8)
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write what the last one computed to '
                    'DIR/<name>.npy (float32 / float64, at most 64 MB; see OutputDump), e.g. DIR = bench_outputs')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


def workload_config(args, world=1, scenes_rank=None):
    if world > 1:
        name = f'config 5: {args.total_scenes} synthetic 3-camera scenes x {args.dets} detections per step, sharded over {world} ranks'
    else:
        name = ('config 2' if (args.scenes, args.dets) == (4096, 20) and not args.no_crops
                else 'config 3 (dense bin)' if args.dets == 200 else 'custom')
        name += f': {args.scenes} synthetic 3-camera scenes x {args.dets} detections per step'
    path = ('geometry only (no crops)' if args.no_crops else
            f'full path incl. {args.target}x{args.target} float32 crops of every matched detection in 3 views')
    return {
        'workload': f'{name} (sigma={args.sigma}px, p_drop={args.p_drop}); {path}',
        'scenes_per_gpu': scenes_rank if scenes_rank is not None else args.scenes,
        'scenes_per_step': args.total_scenes if world > 1 else args.scenes,
        'detections_per_camera': args.dets, 'target_size': args.target,
        'image_pool': f'{args.pool} triplets of 3840x2160 BGR uint8 ({args.pool * 3 * 3840 * 2160 * 3 / 1e6:.0f} MB), '
                      'scene s uses triplet s % pool',
        'crop_chunk_rois': args.chunk_rois,
        'l2': 'inputs (image pool) and outputs (crop chunk buffer) are both larger than the 126 MB L2; no explicit flush',
        'threshold': 30,
    }


# ---------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--query-gpu={self.FIELDS}', '--format=csv,noheader,nounits', '-lms', '100', '-i', str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.rows.append((time.time(), line.strip()))
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self, t0=None, t1=None):
        """Summary of the samples that arrived inside the timed region [t0, t1] (host clock); if the region was
        shorter than the sampling period, of the samples taken under load since warm-up began."""
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smmax, power, reasons = [], [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        rows = [r for (ts, r) in self.rows if t0 is None or t0 <= ts <= t1 + 0.12]
        scope = 'timed region'
        if not rows:
            rows = [r for (ts, r) in self.rows[1:]]
            scope = 'warm-up + timed region (timed region shorter than the 100 ms sampling period)'
        for row in rows:
            parts = [p.strip() for p in row.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); smmax.append(float(parts[1])); power.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(smmax)), 'power_w_max': float(max(power)),
                'samples': len(sm), 'scope': scope, 'reasons': sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (NumPy + the reference's own SciPy / OpenCV / torchvision calls)
# ---------------------------------------------------------------------------------------------------------
def _cpu_scene(batch, images, s, T, pool, as_written=False):
    """One scene through the oracle: _match restatement + the crop of every match in 3 views.

    ``as_written``: the cost tensor by the reference's Python triple loop (epipolar_matching.py:90-96, three
    epipolar_error calls per element) instead of the bit-identical vectorised restatement."""
    from oracle import crop as ocrop
    from oracle import geometry as og
    Ks, RTs = batch.capture_arrays(s)
    cen = [batch.centers[s, c, :batch.counts[s, c]] for c in range(3)]
    res = og.match_scene(Ks, RTs, cen, 30, cost_fn=og.cost_tensor_loop if as_written else og.cost_tensor_fast)
    crops = 0
    for (i, j, k) in res['idx']:
        for v, d in enumerate((i, j, k)):
            ocrop.crop_tensor_ref(images[(s % pool) * 3 + v], batch.boxes[s, v, d], target_size=T, swap_rb=True)
            crops += 1
    return len(res['idx']), crops


_W = {}


def _cpu_worker_init(scenes, dets, sigma, p_drop, pool, T):
    import cv2
    import torch
    from bpc_baseline_b200 import synth
    cv2.setNumThreads(1)
    torch.set_num_threads(1)
    _W['batch'] = synth.make_scenes(scenes, dets, sigma=sigma, p_drop=p_drop)
    _W['images'] = synth.make_images(pool * 3).reshape(pool * 3, synth.IMG_H, synth.IMG_W, 3)
    _W['T'], _W['pool'] = T, pool


def _cpu_worker_run(s):
    return _cpu_scene(_W['batch'], _W['images'], s, _W['T'], _W['pool'])


def _cpu_worker_run_as_written(s):
    return _cpu_scene(_W['batch'], _W['images'], s, _W['T'], _W['pool'], as_written=True)


def _cpu_model():
    try:
        with open('/proc/cpuinfo') as f:
            for line in f:
                if line.startswith('model name'):
                    return line.split(':', 1)[1].strip()
    except Exception:
        pass
    return 'unknown'


def cpu_baseline_single(args, batch, images):
    """Bounded single-thread samples of the same workload on this host: the `cpu_baseline` object is the reference AS
    WRITTEN (restated: Python triple loop over the cost tensor, SURVEY.md 8d-i); `cpu_baseline_vectorised` the stronger
    comparator (bit-identical vectorised cost tensor, 8d-ii).  Both run SciPy's LSAP, NumPy's SVD, cv2's INTER_AREA resize
    and torchvision's to_tensor / normalize -- the reference's own library calls."""
    import cv2
    import torch
    cv2.setNumThreads(1)
    nthreads = torch.get_num_threads()
    torch.set_num_threads(1)
    cores = len(os.sched_getaffinity(0))
    out = {}
    _cpu_scene(batch, images, 0, args.target, args.pool)          # warm caches / imports
    for key, n, aw in (('cpu_baseline', min(args.cpu_scenes_as_written, len(batch)), True),
                       ('cpu_baseline_vectorised', min(args.cpu_scenes, len(batch)), False)):
        t0 = time.perf_counter()
        crops = 0
        for s in range(n):
            crops += _cpu_scene(batch, images, s, args.target, args.pool, as_written=aw)[1]
        dt = time.perf_counter() - t0
        what = ('the reference as written, restated in oracle/: compute_cost_matrix as the Python triple loop '
                '(epipolar_matching.py:90-96) + scipy LSAP + numpy SVD' if aw else
                'oracle.geometry.match_scene with the vectorised bit-identical cost tensor + scipy LSAP + numpy SVD')
        out[key] = {'value': n / dt, 'unit': UNIT, 'cores': 1, 'kind': 'port',
                    'variant': 'as-written restatement' if aw else 'vectorised restatement',
                    'crops_per_s': crops / dt, 'cpu_model': _cpu_model(), 'host_cores': cores, 'cv2_threads': 1,
                    'sample': f'{n} of the {len(batch)} scenes ({crops} crops): {what}; crops through oracle.crop.crop_tensor_ref '
                              f'(cv2.resize INTER_AREA + cvtColor + torchvision to_tensor/normalize); 1 thread, {dt:.1f} s; '
                              f'throughput of the full workload is extrapolated from this sample'}
    torch.set_num_threads(nthreads)
    return out


def run_reference(args):
    """--impl reference: the oracle port on all host cores (the reference is pure Python: there is no
    oracle/_ref binary; /root/reference does not exist on the GPU box).  `value` times the vectorised restatement (the
    stronger CPU comparator); `as_written` in the same line times the reference's own triple loop on a smaller sample."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0))
    per_step = max(cores * 4, 16)
    pool_imgs = min(args.pool, 2)                                   # image content does not change the CPU cost
    total = per_step * (args.steps + args.warmup)
    ctx = mp.get_context('fork')
    t_setup = time.perf_counter()
    with ctx.Pool(cores, initializer=_cpu_worker_init,
                  initargs=(min(total, 1024), args.dets, args.sigma, args.p_drop, pool_imgs, args.target)) as pool:
        nscn = min(total, 1024)
        pool.map(_cpu_worker_run, range(cores))                     # every worker initialised and warm
        for w in range(args.warmup):
            pool.map(_cpu_worker_run, [(w * per_step + i) % nscn for i in range(per_step)], chunksize=1)
        t0 = time.perf_counter()
        crops = 0
        for k in range(args.steps):
            res = pool.map(_cpu_worker_run, [((args.warmup + k) * per_step + i) % nscn for i in range(per_step)], chunksize=1)
            crops += sum(c for _, c in res)
        dt = time.perf_counter() - t0
        # the reference as written (Python triple loop): one scene per core, once
        ta = time.perf_counter()
        pool.map(_cpu_worker_run_as_written, range(cores), chunksize=1)
        dta = time.perf_counter() - ta
    value = per_step * args.steps / dt
    sample = (f'{per_step} scenes per step ({crops // max(args.steps, 1)} crops) of the config-2 workload, fanned out over '
              f'{cores} processes (oracle port: NumPy restatement + scipy LSAP + cv2 INTER_AREA + torchvision normalize)')
    cfg = workload_config(args)
    cfg['scenes_per_step_sampled'] = per_step
    cfg['sampling'] = (f'each step is a bounded sample of {per_step} scenes of the {cfg["scenes_per_step"]}-scene workload; '
                       'scenes are independent, so scenes/s of the sample is scenes/s of the workload')
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': dt / max(args.steps, 1) * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64 geometry / u8+f32 crops', 'data': 'synthetic', 'config': cfg,
        'crops_per_s': crops / dt,
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'variant': 'vectorised restatement',
                         'cpu_model': _cpu_model(), 'sample': sample},
        'as_written': {'value': cores / dta, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'variant': 'as-written restatement',
                       'sample': f'{cores} scenes (one per process) with compute_cost_matrix as the Python triple loop of '
                                 f'epipolar_matching.py:90-96, {dta:.1f} s'},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0, 'setup_s': t0 - t_setup,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
def _peak():
    peaks = {}
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    src = 'measured (MEASURED_PEAKS.json hbm_gbs)' if 'hbm_gbs' in peaks else 'fallback 6650 GB/s (B200_PROFILING.md)'
    return peak, src


_REAL_STDOUT = None


def _guard_stdout():
    """Libraries (the NCCL version banner, torch's c10d logs) write to file descriptor 1; stdout must carry exactly one JSON line.
    From here on fd 1 points at stderr and the line goes out through a saved copy of the original descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(text):
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        print(text, flush=True)
    else:
        os.write(_REAL_STDOUT, (text + '\n').encode())


def _measured_traffic(workload_key):
    """DRAM bytes of one crop launch from the committed ncu capture of the CURRENT kernel (profiles/crop_traffic.json,
    written by tools/ncu_summary.py --traffic): {workload key: {"dram_bytes": ..., "source": ...}}."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'crop_traffic.json')) as f:
            t = json.load(f).get(workload_key)
        return (float(t['dram_bytes']), t.get('source')) if t else (None, None)
    except Exception:
        return None, None


def _timed(torch, fn, warm=3, reps=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def extra_configs(args, torch, dev, images, images_h, peak, crops_buf):
    """BASELINE.json configs 1, 3, 4 and 5 on this one GPU (config 2 is the line's main workload)."""
    from types import SimpleNamespace
    from bpc_baseline_b200 import batched, pipeline, scene, synth
    from bpc_baseline_b200.inference.process_pose import PoseEstimator, PoseEstimatorParams
    todev = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(dev)
    T = args.target
    out = {}

    # ---- config 1: one IPD-style scene, 3 cameras x 10 detections -------------------------------------------
    b1 = synth.make_scenes(1, 10, seed=synth.SEED + 2)
    Ks1, RTs1 = b1.capture_arrays(0)
    boxes1 = [b1.boxes[0, c, :b1.counts[0, c]] for c in range(3)]
    sess = scene.SceneSession(Dmax=10, T=T, image_shape=(3, synth.IMG_H, synth.IMG_W, 3), device=dev)
    t0 = time.perf_counter(); sess.set_images(images_h[:3]); sess.stream.synchronize(); up_ms = (time.perf_counter() - t0) * 1e3
    r1 = sess.run(Ks1, RTs1, boxes1)
    lat = []
    for _ in range(200):
        t0 = time.perf_counter(); sess.run(Ks1, RTs1, boxes1); lat.append((time.perf_counter() - t0) * 1e3)
    with torch.cuda.stream(sess.stream):
        g_ms = _timed(torch, sess.graph.replay, warm=3, reps=50)          # back-to-back replays, CUDA events on the session's stream
    est = PoseEstimator(PoseEstimatorParams(target_size=T))
    cap = SimpleNamespace(images=[images_h[0], images_h[1], images_h[2]], Ks=Ks1, RTs=RTs1)
    dets = b1.detections(0)
    for _ in range(2):
        preds = est._match(cap, dets); torch.cuda.synchronize()
    t0 = time.perf_counter(); preds = est._match(cap, dets); torch.cuda.synchronize(); api_match_ms = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter(); tens = est.crop_inputs(preds); torch.cuda.synchronize(); api_crop_ms = (time.perf_counter() - t0) * 1e3
    same = (len(preds) == r1['n'] and all(tuple(int(v) for v in r1['idx'][m]) == preds[m].match for m in range(r1['n']))
            and bool(torch.equal(tens, r1['crops'])))
    out['config1'] = {'what': 'single IPD-style scene, 3 cameras x 10 detections, match + triangulate + 224x224 crops',
                      'matches': r1['n'], 'crops': 3 * r1['n'],
                      'session_latency_ms_median': float(np.median(lat)), 'session_latency_ms_p90': float(np.percentile(lat, 90)),
                      'session_note': 'SceneSession.run: pinned staging fill + ONE CUDA-graph replay (H2D of K/RT/boxes, match, '
                                      'triangulate, ROI list, crops, D2H of the pose records) + stream synchronise; images resident',
                      'graph_replay_gpu_ms': g_ms, 'image_upload_ms': up_ms, 'image_upload_bytes': int(images_h[:3].nbytes),
                      'python_surface_match_ms': api_match_ms, 'python_surface_crop_ms_incl_image_upload': api_crop_ms,
                      'session_equals_python_surface': bool(same)}
    del sess

    # ---- config 3: dense bin, 3 x 200 detections, 16,384 scenes (geometry path; crops of D=200 scenes are config 4's job) ----
    def geometry(S, D, **kw):
        b = synth.make_scenes(S, D, **kw)
        Ks, RTs, cen, cnt = todev(b.Ks), todev(b.RTs), todev(b.centers), todev(b.counts)
        ms = _timed(torch, lambda: batched.match_triangulate(Ks, RTs, cen, cnt, 30), warm=2, reps=3)
        res = batched.match_triangulate(Ks, RTs, cen, cnt, 30)
        elems = float(b.counts.astype(np.float64).prod(axis=1).sum())
        return {'scenes': S, 'detections_per_camera': D, **kw, 'ms': ms, 'scenes_per_s': S / ms * 1e3,
                'matches': int(res.n.clamp(min=0).sum()), 'virtual_cost_elements_per_s': elems / ms * 1e3}
    out['config3'] = {'clean': geometry(16384, 200), 'stress': geometry(2048, 200, p_drop=0.1, sigma=2.0),
                      'bound': 'fp64 issue / latency (no DRAM traffic to speak of); see profiles/ for the ncu summary'}

    # ---- config 4: crop-only sweep, 64 matches x 3 views per scene = 192 ROIs / scene, three side ranges ----
    c4 = []
    R4 = 65536
    for (lo, hi, TT) in ((32, 96, T), (60, 400, T), (300, 900, T), (60, 400, 256)):
        rng = np.random.default_rng([44, lo, hi, TT])
        w = rng.integers(lo, hi, R4); h = rng.integers(lo, hi, R4)
        x1 = (rng.random(R4) * (synth.IMG_W - w)).astype(np.int64); y1 = (rng.random(R4) * (synth.IMG_H - h)).astype(np.int64)
        rois = np.stack([rng.integers(0, images.shape[0], R4), x1, y1, x1 + w, y1 + h], axis=1).astype(np.int32)
        drois = todev(rois)
        chunk = args.chunk_rois if TT == T else (args.chunk_rois * T * T) // (TT * TT)
        buf = crops_buf.view(-1)[:chunk * 3 * TT * TT].view(chunk, 3, TT, TT)

        def run():
            for first in range(0, R4, chunk):
                r = min(chunk, R4 - first)
                batched.roi_crop(images, drois[first:first + r], T=TT, out=buf)
        ms = _timed(torch, run, warm=2, reps=3)
        nbytes = pipeline.algorithmic_crop_bytes(rois, TT)
        c4.append({'sides': [lo, hi], 'T': TT, 'rois': R4, 'scenes_equiv': R4 // 192, 'ms': ms, 'crops_per_s': R4 / ms * 1e3,
                   'roofline': {'bound': 'hbm', 'achieved': nbytes / ms / 1e6, 'peak': peak, 'unit': 'GB/s',
                                'frac': nbytes / ms / 1e6 / peak}})
    out['config4'] = c4

    # ---- config 5 on this one GPU: 131,072 scenes, full path, crops chunk-wise ----
    S5 = args.total_scenes
    b5 = synth.make_scenes(S5, args.dets, sigma=args.sigma, p_drop=args.p_drop)
    ios5 = todev(((np.arange(S5)[:, None] % args.pool) * 3 + np.arange(3)[None, :]).astype(np.int32))
    t5 = [todev(a) for a in (b5.Ks, b5.RTs, b5.centers, b5.counts, b5.boxes)]
    pipe5 = pipeline.MatchCropPipeline(S5, b5.boxes.shape[2], T=T, chunk_rois=args.chunk_rois, device=dev, crops=crops_buf)
    res5, offs5 = pipe5.run_device(*t5, images, ios5)
    n5 = int(offs5[-1])
    ms5 = _timed(torch, lambda: pipe5.run_device(*t5, images, ios5, n_rois_host=n5), warm=1, reps=2)
    out['config5_one_gpu'] = {'scenes': S5, 'detections_per_camera': args.dets, 'rois': n5, 'ms_per_step': ms5,
                              'scenes_per_s': S5 / ms5 * 1e3, 'crops_per_s': n5 / ms5 * 1e3}
    return out


class OutputDump:
    """--dump-outputs: what the timed path hands its caller in the last timed step, so that two builds run with the same
    arguments can be compared file by file.

    Per scene (all scenes while they fit in 14 MB, else a fixed seeded sample): the matcher's outputs idx, n, cost, X,
    reproj and the scene's first ROI (scene_offset).  Per ROI (a fixed seeded sample that fits in 48 MB): the ROI
    record, its status and its float32 crop.  The crops of a step never exist all at once (the pipeline reuses one
    chunk buffer), so the sampled ones are copied out of each chunk as the pipeline hands it to its consumer.  Integer
    arrays are written as float64 (exact); scene_index / roi_index say which rows were sampled."""

    SCENE_BYTES, CROP_BYTES = 14_000_000, 48_000_000                    # + n_rois and the .npy headers: < 64 MB in all
    SEED = 20251020

    def __init__(self, torch, dev, S, Dmax, T, n_rois, chunk, crops):
        def sample(n, k, stream):
            if k >= n:
                return np.arange(n)
            return np.sort(np.random.default_rng([self.SEED, stream]).choice(n, k, replace=False))

        self.torch, self.S = torch, S
        per_scene = Dmax * 3 * 8 * 3 + Dmax * 4 + 3 * 8                  # idx, X, reproj; cost; n, scene_offset, scene_index
        self.scenes = sample(S, self.SCENE_BYTES // per_scene, 0)
        per_roi = 5 * 8 + 8 + (8 + 3 * T * T * 4 if crops else 0)       # ROI record, roi_index; status, crop
        self.rois = sample(n_rois, self.CROP_BYTES // per_roi, 1)
        self.crops = torch.empty((len(self.rois), 3, T, T), dtype=torch.float32, device=dev) if crops else None
        self.parts = {}                                                  # chunk start -> (rows of self.crops, rows of the chunk)
        for first in range(0, n_rois if crops else 0, chunk):
            pos = np.flatnonzero((self.rois >= first) & (self.rois < first + chunk))
            if len(pos):
                self.parts[first] = (torch.as_tensor(pos, device=dev), torch.as_tensor(self.rois[pos] - first, device=dev))

    def consumer(self, out, first):
        part = self.parts.get(first)
        if part is not None:
            self.crops.index_copy_(0, part[0], out.index_select(0, part[1]))

    def write(self, path, res, offs, rois, status):
        torch = self.torch
        sel = torch.as_tensor(self.scenes, device=offs.device)
        ridx = torch.as_tensor(self.rois, device=offs.device)
        arrays = {'scene_index': self.scenes, 'idx': res.idx[sel], 'n': res.n[sel], 'cost': res.cost[sel], 'X': res.X[sel],
                  'reproj': res.reproj[sel], 'scene_offset': offs[sel], 'n_rois': offs[self.S:],
                  'roi_index': self.rois, 'rois': rois[ridx]}
        if self.crops is not None:
            arrays.update(status=status[ridx], crops=self.crops)
        os.makedirs(path, exist_ok=True)
        for name, a in arrays.items():
            a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
            np.save(os.path.join(path, f'{name}.npy'), a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))


def multi_rank_parity(args, torch, dist, dev, gathered, shards, Dmax, sample=64):
    """Rank 0: regenerate the first and the last `sample` scenes of every other rank's shard, run them locally and compare
    with the records that came through the all-gather, bit for bit (idx, n, cost, X, reproj)."""
    from bpc_baseline_b200 import batched, distributed, synth
    todev = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(dev)
    got = distributed.unpack_records(gathered)
    S = shards[0][1] - shards[0][0]
    checked, equal = 0, True
    for r, (lo, hi) in enumerate(shards):
        if r == 0:
            continue
        for (first, a, b) in ((lo, 0, min(sample, hi - lo)), (max(lo, hi - synth.CHUNK), max(0, hi - lo - sample) - (max(lo, hi - synth.CHUNK) - lo), None)):
            blk = synth.make_scenes(min(synth.CHUNK, hi - first), args.dets, first=first, sigma=args.sigma, p_drop=args.p_drop)
            b = len(blk) if b is None else b
            sub = blk.slice(a, b)
            if len(sub) == 0:
                continue
            c = np.zeros((len(sub), 3, Dmax, 2)); c[:, :, :sub.centers.shape[2]] = sub.centers
            res = batched.match_triangulate(todev(sub.Ks), todev(sub.RTs), todev(c), todev(sub.counts), 30)
            g0 = r * S + (first - lo) + a
            for k, t in (('idx', res.idx), ('n', res.n), ('cost', res.cost), ('X', res.X), ('reproj', res.reproj)):
                gv = got[k][g0:g0 + len(sub)]
                bits = (lambda x: x.view(torch.int64) if x.dtype == torch.float64 else (x.view(torch.int32) if x.dtype == torch.float32 else x))
                equal = equal and bool(torch.equal(bits(gv.contiguous()), bits(t.contiguous())))
            checked += len(sub)
    return {'checked_scenes': checked, 'ranks_checked': len(shards) - 1, 'equal': bool(equal),
            'what': 'gathered pose records (idx, n, cost, X, reproj) of the first and last scenes of every other rank vs a '
                    'local recomputation on rank 0, bit for bit'}


def main():
    args = parse_args()
    if args.impl == 'reference':
        run_reference(args)
        return
    import torch
    import torch.distributed as dist

    from bpc_baseline_b200 import _lib, batched, distributed, pipeline, synth

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    _guard_stdout()
    if args.dump_outputs and world > 1:
        raise SystemExit('--dump-outputs is supported at N = 1 only')
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        # NCCL writes its version banner / log lines to stdout (the level may come from /etc/nccl.conf, not the
        # environment); stdout carries the one JSON line, so send them to stderr
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')
        dist.init_process_group('nccl', device_id=dev)
    _lib.load()

    D, T = args.dets, args.target
    if world > 1:                        # config 5: a fixed total, contiguous CHUNK-aligned shards (strong scaling)
        shards = [distributed.shard_range(args.total_scenes, r, world, align=synth.CHUNK) for r in range(world)]
        if len({hi - lo for lo, hi in shards}) != 1:
            raise SystemExit(f'--total-scenes must split into {world} equal multiples of {synth.CHUNK}')
        first, S = shards[rank][0], shards[rank][1] - shards[rank][0]
    else:
        shards, first, S = [(0, args.scenes)], 0, args.scenes
    batch = synth.make_scenes(S, D, first=first, sigma=args.sigma, p_drop=args.p_drop)
    Dmax = batch.boxes.shape[2]
    nimg = args.pool * 3
    # image pool: generated on the host once (also the e2e source), resident in HBM for the device-timed run
    images_h = synth.make_images(nimg)
    ios = (((first + np.arange(S))[:, None] % args.pool) * 3 + np.arange(3)[None, :]).astype(np.int32)
    todev = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(dev)
    Ks, RTs, centers, counts, boxes = (todev(batch.Ks), todev(batch.RTs), todev(batch.centers), todev(batch.counts), todev(batch.boxes))
    images = todev(images_h)
    ios_d = todev(ios)

    pipe = pipeline.MatchCropPipeline(S, Dmax, T=T, chunk_rois=args.chunk_rois, device=dev)

    # one untimed pass to learn the ROI count and the algorithmic bytes (identical inputs every step)
    res, offs = pipe.run_device(Ks, RTs, centers, counts, boxes, images, ios_d)
    torch.cuda.synchronize()
    n_rois = int(offs[-1].item())
    n_matches = int(res.n.clamp(min=0).sum().item())
    rois_h = pipe.rois[:n_rois].cpu().numpy()
    rejected = int(pipe.status[:n_rois].sum().item())
    crop_bytes = pipeline.algorithmic_crop_bytes(rois_h, T)
    n_rois_arg = 0 if args.no_crops else n_rois

    def make_step(pipe, tensors, n_rois_arg, S):
        recbuf = torch.empty((distributed.records_bytes(S, Dmax),), dtype=torch.uint8, device=dev) if world > 1 else None
        gathered = torch.empty((world, recbuf.numel()), dtype=torch.uint8, device=dev) if world > 1 else None

        def step(e=None, consumer=None):
            if e is not None:
                e[3].record()
            r, o = pipe.run_device(*tensors, n_rois_host=n_rois_arg, events=(e[0], e[1], e[2]) if e is not None else None,
                                   consumer=consumer)
            if world > 1:                 # final gather of the pose records over NVLink (SURVEY.md 8e): one pack kernel + one all-gather
                distributed.gather_records(distributed.pack_records(r, o, 3, out=recbuf), out=gathered)
            return r, o
        return step, gathered

    def timed_loop(step, steps, warmup, last_consumer=None):
        """(ms, crop_ms, match_ms, wall0, wall1, (MatchResult, scene_offset) of the last step); ``last_consumer`` receives
        the crop chunks of the last step."""
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(steps)]
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t_start, t_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        wall0 = time.time()
        t_start.record()
        for k in range(steps):
            last = step(ev[k], consumer=last_consumer if k == steps - 1 else None)
        t_stop.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        wall1 = time.time()
        ms = t_start.elapsed_time(t_stop)
        crop_ms = sum(e[1].elapsed_time(e[2]) for e in ev)
        match_ms = sum(e[3].elapsed_time(e[0]) for e in ev)
        if world > 1:
            t = torch.tensor([ms, crop_ms, match_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, crop_ms, match_ms = [float(v) for v in t.cpu()]
        return ms, crop_ms, match_ms, wall0, wall1, last

    step, gathered = make_step(pipe, (Ks, RTs, centers, counts, boxes, images, ios_d), n_rois_arg, S)
    dump = (OutputDump(torch, dev, S, Dmax, T, n_rois, pipe.chunk, crops=not args.no_crops)
            if args.dump_outputs else None)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = None
    warm = max(args.warmup, 3)
    for _ in range(warm):
        step(consumer=dump.consumer if dump else None)      # the dump's copy kernels load here, not in the timed window
    launches0 = _lib.launch_count()
    ms, crop_ms, match_ms, wall0, wall1, last = timed_loop(step, args.steps, 0, dump.consumer if dump else None)
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    launches = _lib.launch_count() - launches0
    crop_launches = pipe.last_crop_launches * args.steps
    if dump is not None:
        dump.write(args.dump_outputs, *last, pipe.rois, pipe.status)

    # ---- N > 1: bit equality of what came through the gather, and the round-1 weak-scaling workload next to it ----
    parity = None
    weak = None
    if world > 1:
        if rank == 0:
            parity = multi_rank_parity(args, torch, dist, dev, gathered, shards, Dmax)
        dist.barrier()
        if not args.no_crops:
            Sw = args.scenes
            firstw = ((rank * Sw + synth.CHUNK - 1) // synth.CHUNK) * synth.CHUNK
            bw = synth.make_scenes(Sw, D, first=firstw, sigma=args.sigma, p_drop=args.p_drop)
            iosw = todev(((np.arange(Sw)[:, None] % args.pool) * 3 + np.arange(3)[None, :]).astype(np.int32))
            tw = (todev(bw.Ks), todev(bw.RTs), todev(bw.centers), todev(bw.counts), todev(bw.boxes), images, iosw)
            pipew = pipeline.MatchCropPipeline(Sw, bw.boxes.shape[2], T=T, chunk_rois=args.chunk_rois, device=dev, crops=pipe.crops)
            _, offw = pipew.run_device(*tw)
            nw = int(offw[-1].item())
            stepw, _ = make_step(pipew, tw, nw, Sw)
            msw, _, _, _, _, _ = timed_loop(stepw, 5, 3)
            weak = {'workload': f'config 2 per rank: {Sw} scenes x {D} detections per GPU per step (weak scaling, the round-1 line)',
                    'value': world * Sw * 5 / (msw * 1e-3), 'unit': UNIT, 'ms_per_step': msw / 5, 'steps': 5, 'warmup': 3,
                    'crops_per_s': world * nw * 5 / (msw * 1e-3)}
            del pipew

    # ---- end-to-end from pinned host buffers (H2D of all inputs incl. the image pool, D2H of pose records) ----
    e2e = None
    if not args.no_e2e and not args.no_crops:
        hb = pipe.host_buffers(images_h.shape)
        hb['Ks'].copy_(torch.from_numpy(batch.Ks)); hb['RTs'].copy_(torch.from_numpy(batch.RTs))
        hb['boxes'].copy_(torch.from_numpy(batch.boxes)); hb['counts'].copy_(torch.from_numpy(batch.counts))
        hb['image_of_scene'].copy_(torch.from_numpy(ios)); hb['images'].copy_(torch.from_numpy(images_h))
        out = pipe.run_host(n_rois_host=None)                       # serial variant: warm-up + check
        assert int(out['n_rois'][0]) == n_rois and bool((out['idx'] == res.idx.cpu()).all())
        pipe.run_host_stream(2)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        # K steps, uploads double buffered behind the previous step's kernels (MatchCropPipeline.run_host_stream);
        # the wall clock brackets everything incl. the first upload and the last read-back
        t0 = time.perf_counter()
        out = pipe.run_host_stream(args.steps)
        torch.cuda.synchronize()
        e2e_ms = (time.perf_counter() - t0) * 1e3
        if world > 1:
            t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_ms = float(t.item())
        assert int(out['n_rois'][0]) == n_rois and bool((out['idx'] == res.idx.cpu()).all())
        e2e = {'value': world * S * args.steps / (e2e_ms * 1e-3), 'unit': UNIT,
               'h2d_bytes_per_step': pipe.h2d_bytes(), 'd2h_bytes_per_step': pipe.d2h_bytes(),
               'ms_per_step': e2e_ms / args.steps,
               'note': 'host wall clock over K steps; inputs (K, RT, boxes, counts, image pool) copied from pinned host memory '
                       'every step (double buffered behind the previous step), centres derived on device; pose records '
                       '(idx, n, cost, X, reproj) read back; crops stay in HBM for the on-device pose network '
                       '(the reference moves them H2D at process_pose.py:210); per rank at N > 1'}

    # ---- crop gather to rank 0 (SURVEY.md 8e options 2/3), its own stage with its own bound: uint8 crops pulled
    #      over NVLink by the receiver's normalise kernel; NOT part of `value` (crops stay sharded there) ----
    crop_gather = None
    if world > 1 and not args.no_crops and not args.no_crop_gather:
        try:
            gchunk = min(args.gather_chunk, n_rois)
            cg = distributed.CropGather(gchunk, T=T, root=0, transport='p2p', device=dev)
            g_rois = pipe.rois[:gchunk]
            outg = None
            for i in range(3):
                cg.produce(i, lambda slot: batched.roi_crop_u8(images, g_rois, T=T, out=slot))
                outg = cg.collect(i)
            torch.cuda.synchronize()
            # parity of the gathered crops: rank 0 regenerates the head of every rank's ROI list and crops it directly
            gpar = None
            if rank == 0:
                ncheck, eq = 256, True
                for r, (lo, hi) in enumerate(shards):
                    blk = synth.make_scenes(min(synth.CHUNK, hi - lo), D, first=lo, sigma=args.sigma, p_drop=args.p_drop)
                    rr = batched.match_triangulate(todev(blk.Ks), todev(blk.RTs), todev(blk.centers), todev(blk.counts), 30)
                    iosr = todev((((lo + np.arange(len(blk)))[:, None] % args.pool) * 3 + np.arange(3)[None, :]).astype(np.int32))
                    rois_r, offs_r = batched.build_rois(todev(blk.boxes), rr.idx, rr.n, iosr)
                    k = min(ncheck, gchunk, int(offs_r[-1]))
                    direct = batched.roi_crop(images, rois_r[:k].contiguous(), T=T)
                    eq = eq and bool(torch.equal(direct.view(torch.int32), outg[r * gchunk:r * gchunk + k].view(torch.int32)))
                gpar = {'checked_crops_per_rank': ncheck, 'equal': bool(eq)}
            dist.barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for i in range(args.gather_steps):
                cg.produce(i, lambda slot: batched.roi_crop_u8(images, g_rois, T=T, out=slot))
                cg.collect(i)
            g1.record()
            torch.cuda.synchronize()
            t = torch.tensor([g0.elapsed_time(g1)], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t.item()) * 1e-3 / args.gather_steps
            ingest = cg.wire_bytes() / sec / 1e9
            crop_gather = {'transport': 'uint8 crops pulled over NVLink peer memory by the receiver kernel (bpc_crops_normalise)',
                           'root': 0, 'chunk_rois_per_rank': gchunk, 'chunks': args.gather_steps,
                           'crops_per_s': world * gchunk / sec, 'ms_per_chunk': sec * 1e3,
                           'roofline': {'bound': 'nvlink ingest of rank 0', 'achieved': ingest, 'peak': 900.0, 'unit': 'GB/s',
                                        'frac': ingest / 900.0, 'peak_source': 'NVLink 5 per direction (nominal)'},
                           'root_hbm_write_GBps': world * gchunk * 3 * T * T * 4 / sec / 1e9,
                           'parity': gpar,
                           'note': 'every rank produces a chunk of uint8 crops, rank 0 converts all of them to the float32 '
                                   'network input; separate from `value`, where crops stay on the GPU that produced them'}
            cg.close()
        except Exception as exc:              # noqa: BLE001 -- the headline numbers do not depend on this stage
            crop_gather = {'unavailable': f'{type(exc).__name__}: {exc}'[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = _peak()
    roofline = None
    if crop_launches and crop_ms > 0:
        per_launch_bytes = crop_bytes / pipe.last_crop_launches
        avg_launch_s = crop_ms * 1e-3 / crop_launches
        achieved = per_launch_bytes / avg_launch_s / 1e9
        default_wl = (D, T, args.chunk_rois, args.pool, args.p_drop, args.sigma) == (20, 224, 16384, 8, 0.0, 1.0)
        traffic, traffic_src = _measured_traffic('config2_chunk16384_T224') if default_wl else (None, None)
        roofline = {'bound': 'hbm', 'kernel': 'bpc_crop_cta_kernel<false,224,true> (+ bpc_crop_prep_kernel and the empty per-strip / generic launches)', 'achieved': achieved,
                    'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic,
                    'traffic_source': traffic_src, 'peak_source': peak_src,
                    'algorithmic_bytes_per_launch': per_launch_bytes, 'avg_launch_ms': avg_launch_s * 1e3,
                    'launches_per_step': pipe.last_crop_launches, 'share_of_step': crop_ms / ms}

    cpu = {}
    if not args.no_cpu_baseline and world == 1:
        cpu = cpu_baseline_single(args, batch, images_h)

    configs = None
    if world == 1 and not args.no_configs and not args.no_crops:
        configs = extra_configs(args, torch, dev, images, images_h, peak, pipe.crops)

    total = world * S
    value = total * args.steps / (ms * 1e-3)
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': warm,
        'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'strong' if world > 1 else 'weak', 'vs_baseline': None,
        'dtype': 'f64 geometry / u8+f32 crops', 'data': 'synthetic', 'config': workload_config(args, world, S),
        'crops_per_s': world * n_rois * args.steps / (ms * 1e-3) if not args.no_crops else 0.0,
        'matches_per_step_per_gpu': n_matches, 'rois_per_step_per_gpu': n_rois, 'rois_rejected': rejected,
        'geometry_ms_per_step': match_ms / args.steps, 'crop_ms_per_step': crop_ms / args.steps,
        'non_crop_share_of_step': 1.0 - crop_ms / ms if ms > 0 else None,
        'roofline': roofline, 'cpu_baseline': cpu.get('cpu_baseline'), 'e2e': e2e, 'gpu_launches': int(launches), 'clocks': clocks,
    }
    if cpu.get('cpu_baseline_vectorised') is not None:
        line['cpu_baseline_vectorised'] = cpu['cpu_baseline_vectorised']
    if configs is not None:
        line['configs'] = configs
    if parity is not None:
        line['multi_rank_parity'] = parity
    if weak is not None:
        line['weak_config2'] = weak
    if crop_gather is not None:
        line['crop_gather'] = crop_gather
    _emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
