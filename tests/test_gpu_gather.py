"""Receiver side of the crop gather (bpc_crops_normalise) and the two-rank gather itself.

Bar: the float32 tensor rebuilt from gathered uint8 crops is bit-equal to what bpc_roi_crop writes directly,
which tests/test_gpu_crop.py pins bit-equal to the reference's cv2 + torchvision calls.
"""
import os
import re
import signal
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import crop as ocrop
from tests.gpu_util import to_dev

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rois(boxes, img=0):
    return np.concatenate([np.full((len(boxes), 1), img, np.int32), np.asarray(boxes, np.int32)], axis=1)


@pytest.mark.parametrize('T,swap', [(224, True), (224, False), (256, True), (100, True), (50, True), (37, False)])
def test_normalise_matches_direct_crop(golden_crops, T, swap):
    """T % 4 == 0 takes the tiled kernel (T=100: ragged last tile), other T the scalar one."""
    from bpc_baseline_b200 import batched
    g = golden_crops
    images, rois = to_dev(g['image'][None]), to_dev(_rois(g['boxes']))
    direct = batched.roi_crop(images, rois, T=T, swap_rb=swap)
    u8 = batched.roi_crop_u8(images, rois, T=T)
    out = batched.crops_normalise([u8], T, swap_rb=swap)
    assert torch.equal(out.view(torch.int32), direct.view(torch.int32))


def test_normalise_against_reference_calls(golden_crops):
    from bpc_baseline_b200 import batched
    g = golden_crops
    boxes = g['boxes'][:6]
    u8 = batched.roi_crop_u8(to_dev(g['image'][None]), to_dev(_rois(boxes)), T=224)
    out = batched.crops_normalise([u8], 224, swap_rb=True).cpu().numpy()
    for r, b in enumerate(boxes):
        want = ocrop.crop_tensor_ref(g['image'], b, target_size=224, swap_rb=True)
        assert np.array_equal(out[r].view(np.uint32), want.view(np.uint32)), tuple(b)


def test_normalise_several_sources_and_empty_ones():
    """Concatenation order, empty sources, a source count that does not divide anything."""
    from bpc_baseline_b200 import batched
    rng = np.random.default_rng(5)
    T = 64
    u8 = to_dev(rng.integers(0, 256, (23, T, T, 3), dtype=np.uint8))
    whole = batched.crops_normalise([u8], T, swap_rb=True)
    parts = [u8[:5], u8[5:5], u8[5:6], u8[6:23], u8[:0]]
    out = torch.full((30, 3, T, T), -7.0, dtype=torch.float32, device='cuda')
    got = batched.crops_normalise([p.contiguous() for p in parts], T, swap_rb=True, out=out)
    assert got.data_ptr() == out.data_ptr()
    assert torch.equal(out[:23], whole)
    assert bool((out[23:] == -7.0).all())
    lut = batched.normalise_lut('cuda').cpu().numpy()
    h = u8.cpu().numpy()
    want = np.stack([lut[p][h[..., 2 - p]] for p in range(3)], axis=1)
    assert np.array_equal(whole.cpu().numpy(), want)


def test_normalise_rejects_bad_arguments():
    from bpc_baseline_b200 import batched
    u8 = torch.zeros((2, 32, 32, 3), dtype=torch.uint8, device='cuda')
    with pytest.raises(RuntimeError):
        batched.crops_normalise([u8], 64)
    with pytest.raises(RuntimeError):
        batched.crops_normalise([u8.cpu()], 32)
    with pytest.raises(RuntimeError):
        batched.crops_normalise([u8] * 17, 32)
    with pytest.raises(RuntimeError):
        batched.crops_normalise([u8], 32, out=torch.empty((1, 3, 32, 32), device='cuda'))


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _gather_check(nproc, transport, timeout=600):
    """tools/gather_check.py --check under torchrun: (exit code, stdout, stderr).  torchrun and its workers run in a
    session of their own, and the whole process group is killed when the run ends, so no worker outlives the test."""
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', f'--nproc-per-node={nproc}', '--master-addr',
           '127.0.0.1', '--master-port', str(_free_port()), os.path.join(ROOT, 'tools', 'gather_check.py'),
           '--transport', transport, '--check']
    proc = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, cwd=ROOT,
                            start_new_session=True)
    try:
        out, err = proc.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        os.killpg(proc.pid, signal.SIGKILL)
        out, err = proc.communicate()
        pytest.fail(f'gather_check did not finish in {timeout} s\n' + out[-2000:] + err[-4000:])
    finally:
        try:
            os.killpg(proc.pid, signal.SIGKILL)
        except ProcessLookupError:
            pass
    return proc.returncode, out, err


def _assert_gathered(res):
    code, out, err = res
    assert code == 0, out[-2000:] + err[-4000:]
    m = re.search(r'GATHER_OK chunks (\d+)', out)
    assert m and int(m.group(1)) >= 5, out[-2000:]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
@pytest.mark.parametrize('transport', ['p2p', 'nccl'])
def test_two_rank_crop_gather(transport):
    """tools/gather_check.py under torchrun: root's gathered tensor is bit-equal to direct crops of both shards."""
    _assert_gathered(_gather_check(2, transport))


@pytest.mark.parametrize('transport', ['nccl', 'p2p'])
def test_one_rank_crop_gather(transport):
    """The root's side of the gather on one GPU: its own chunks produced on the side stream, each slot reused at chunk
    i + 2 after the conversion that read it (five chunks, the last ragged), against direct crops."""
    _assert_gathered(_gather_check(1, transport))
