"""Crop gather over NVLink, run under torchrun with one rank per GPU (2, 4 or 8):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 \
        tools/gather_check.py --transport p2p --check --bench

--check  root rebuilds every rank's ROIs locally, crops them directly (bpc_roi_crop) and compares bit for bit
         with the tensor gathered from the ranks' uint8 crops, over five chunks: both slots are reused (on the root
         after waiting for the conversion that last read them) and the last chunk is ragged.  Prints GATHER_OK.
--bench  times (a) produce + gather: every rank runs the uint8 crop kernel per chunk and the root collects;
         (b) gather only: the root collects chunks that are already in the ranks' buffers.  Device time
         (CUDA events on the root), one JSON line.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from bpc_baseline_b200 import batched, synth                      # noqa: E402
from bpc_baseline_b200.distributed import CropGather             # noqa: E402


def rank_rois(rank, n, B, H, W, lo=60, hi=400):
    rng = np.random.default_rng([synth.SEED, 991, rank])
    w = rng.integers(lo, hi + 1, n); h = rng.integers(lo, hi + 1, n)
    x1 = rng.integers(0, W - w + 1); y1 = rng.integers(0, H - h + 1)
    return np.stack([rng.integers(0, B, n), x1, y1, x1 + w, y1 + h], axis=1).astype(np.int32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--transport', default='p2p', choices=['p2p', 'nccl'])
    ap.add_argument('--chunk', type=int, default=4096)
    ap.add_argument('--target', type=int, default=224)
    ap.add_argument('--pool', type=int, default=2)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--check', action='store_true')
    ap.add_argument('--bench', action='store_true')
    a = ap.parse_args()

    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    T, chunk = a.target, a.chunk
    images_h = synth.make_images(a.pool, width=1920, height=1080)
    B, H, W, _ = images_h.shape
    images = torch.as_tensor(images_h).to(dev)
    cg = CropGather(chunk, T=T, root=0, transport=a.transport, device=dev)
    if rank == 0:
        print(f'transport {a.transport} peer mapping {cg.peers.method if cg.peers else None} world {world}', flush=True)

    if a.check:
        ck = min(chunk, 400)
        n_check = 4 * ck + max(1, ck // 3)                          # five chunks, the last one ragged
        mine = torch.as_tensor(rank_rois(rank, n_check, B, H, W)).to(dev)
        ok = True
        for i, first in enumerate(range(0, n_check, ck)):
            r = min(ck, n_check - first)
            cg.produce(i, lambda slot: batched.roi_crop_u8(images, mine[first:first + r], T=T, out=slot))
            got = cg.collect(i, [r] * world)
            if rank == 0:
                for src in range(world):
                    rois = torch.as_tensor(rank_rois(src, n_check, B, H, W)[first:first + r]).to(dev)
                    want = batched.roi_crop(images, rois, T=T, swap_rb=True)
                    same = torch.equal(got[src * r:(src + 1) * r].view(torch.int32), want.view(torch.int32))
                    ok = ok and same
                    if not same:
                        print(f'MISMATCH chunk {i} source rank {src}', flush=True)
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.broadcast(flag, 0)
        if rank == 0:
            print(f'GATHER_OK chunks {i + 1}' if ok else 'GATHER_FAILED', flush=True)
        if not int(flag.item()):
            cg.close()
            dist.destroy_process_group()
            sys.exit(1)

    if a.bench:
        rois = torch.as_tensor(rank_rois(rank, chunk, B, H, W)).to(dev)
        res = {}
        for name, produce in (('produce_and_gather', True), ('gather_only', False), ('remote_only', False)):
            for b in range(2):                                         # both slots hold valid crops
                batched.roi_crop_u8(images, rois, T=T, out=cg.slot(b))
            for i in range(3):
                if produce:
                    cg.produce(i, lambda slot: batched.roi_crop_u8(images, rois, T=T, out=slot))
                cg.collect(i)
            torch.cuda.synchronize(); dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            cnt = [0 if r == 0 else chunk for r in range(world)] if name == 'remote_only' else None     # only crops that cross NVLink
            for i in range(a.steps):
                if produce:
                    cg.produce(i, lambda slot: batched.roi_crop_u8(images, rois, T=T, out=slot))
                cg.collect(i, cnt)
            e1.record()
            torch.cuda.synchronize()
            ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            sec = float(ms.item()) * 1e-3 / a.steps
            ncrops = (world - 1) * chunk if name == 'remote_only' else world * chunk
            res[name] = {'ms_per_chunk': sec * 1e3, 'crops_per_s': ncrops / sec,
                         'nvlink_ingest_GBps': cg.wire_bytes() / sec / 1e9,
                         'root_hbm_write_GBps': ncrops * 3 * T * T * 4 / sec / 1e9}
        if rank == 0:
            print(json.dumps({'what': 'crop gather to rank 0', 'transport': a.transport,
                              'peer_mapping': cg.peers.method if cg.peers else None, 'n_gpus': world,
                              'chunk_rois_per_rank': chunk, 'T': T, 'steps': a.steps, **res}), flush=True)
    cg.close()
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
