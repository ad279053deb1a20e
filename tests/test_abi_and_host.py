"""CPU-side checks: the C-ABI library loads and exports every symbol include/bpc_b200.h declares, argument
validation that needs no GPU, and the host-side logic (scene generator, ROI mirror, install() rebinding)."""
import ctypes
import os
import re
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def lib():
    from bpc_baseline_b200 import _lib, build
    build.build()                                        # nvcc cross-compiles for sm_100a without a GPU
    return _lib.load()


def test_library_exports_every_declared_symbol(lib):
    from bpc_baseline_b200 import _lib
    header = open(os.path.join(ROOT, 'include', 'bpc_b200.h')).read()
    header = re.sub(r'/\*.*?\*/', '', header, flags=re.S)
    declared = set(re.findall(r'\b(bpc_[a-z0-9_]+)\s*\(', header))
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in bpc_b200.h but not exported'
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert lib.bpc_abi_version() == 2


def test_error_strings_and_argument_validation(lib):
    assert lib.bpc_error_string(0) == b'ok'
    assert b'invalid argument' in lib.bpc_error_string(-1)
    # argument errors are detected before any CUDA call, so they can be exercised without a GPU
    assert lib.bpc_fundamental(None, None, -1, None, None) == -1
    assert lib.bpc_fundamental(None, None, 4, None, None) == -1
    assert lib.bpc_fundamental(None, None, 0, None, None) == 0
    assert lib.bpc_match_triangulate(None, None, None, None, 0, 0, 30.0, 0, 0.0, None, None, None, None, None, None, None, 0, None) == -1
    assert lib.bpc_match_triangulate(None, None, None, None, 0, 20, 30.0, 0, 0.0, None, None, None, None, None, None, None, 0, None) == 0
    assert lib.bpc_match_triangulate(None, None, None, None, 0, 4096, 30.0, 0, 0.0, None, None, None, None, None, None, None, 0, None) == -4
    # a scene stays in shared memory up to Dmax ~ 450; beyond that the caller supplies a workspace
    assert lib.bpc_match_workspace_bytes(4096, 200) == 0 and lib.bpc_match_workspace_bytes(4096, 384) == 0
    assert lib.bpc_match_workspace_bytes(4, 1024) > 4 * 1024 * 1024 // 8
    assert lib.bpc_pack_records_bytes(4096, 20) == 16 + 4096 * 4 + 4096 * 20 * 64
    fill = (ctypes.c_uint8 * 3)(255, 255, 255)
    assert lib.bpc_roi_crop(None, 1, 8, 8, None, 0, None, 0, 1025, fill, 1, None, None, None, None, 0, None) == -1  # T > BPC_MAX_TARGET
    assert lib.bpc_roi_crop(None, 1, 8, 8, None, 0, None, 0, 224, fill, 1, None, None, None, None, 0, None) == 0    # R == 0
    assert lib.bpc_roi_crop_workspace_bytes(8192, 256) > 8192 * 8192
    assert lib.bpc_roi_crop_workspace_bytes(8192, 512) > lib.bpc_roi_crop_workspace_bytes(8192, 256)
    assert lib.bpc_roi_crop_workspace_bytes(8192, 1025) == 0
    assert lib.bpc_triangulate_views(None, None, 1, 9, None, None) == -1
    assert lib.bpc_launch_count() == 0


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from bpc_baseline_b200 import _lib
    monkeypatch.setattr(_lib, '_lib', None)
    monkeypatch.setattr(_lib, 'LIB_PATH', str(tmp_path / 'nope.so'))
    with pytest.raises(_lib.BpcError, match='no CPU fallback'):
        _lib.load()


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'bpc_baseline_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh')):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle\b', src, flags=re.M), f


def test_batched_api_rejects_cpu_tensors():
    import torch
    from bpc_baseline_b200 import batched
    with pytest.raises(RuntimeError, match='CUDA tensor'):
        batched.fundamental(torch.zeros(1, 3, 3, 3), torch.zeros(1, 3, 4, 4, dtype=torch.float64))
    with pytest.raises(RuntimeError, match='CUDA tensor'):
        batched.roi_crop(torch.zeros(1, 8, 8, 3, dtype=torch.uint8), torch.zeros(1, 5, dtype=torch.int32))


def test_scene_generator_is_chunk_reproducible_and_valid():
    from bpc_baseline_b200 import synth
    a = synth.make_scenes(600, 7, p_drop=0.2, n_dup=1, n_false=1)
    b = synth.make_scenes(88, 7, first=512, p_drop=0.2, n_dup=1, n_false=1)
    for k in ('Ks', 'RTs', 'boxes', 'centers', 'counts'):
        assert np.array_equal(getattr(a, k)[512:600], getattr(b, k))
    assert a.Ks.dtype == np.float32 and a.RTs.dtype == np.float64 and a.boxes.dtype == np.int32
    # RT carries float32-rounded values (data_utils.py:383-387); rotations are orthonormal to float32 accuracy
    assert np.array_equal(a.RTs, a.RTs.astype(np.float32).astype(np.float64))
    R = a.RTs[:, :, :3, :3]
    np.testing.assert_allclose(R @ R.transpose(0, 1, 3, 2), np.broadcast_to(np.eye(3), R.shape), atol=1e-6)
    for s in range(0, 600, 97):
        for c in range(3):
            n = a.counts[s, c]
            bx = a.boxes[s, c, :n]
            assert np.all(bx[:, 0] >= 0) and np.all(bx[:, 1] >= 0) and np.all(bx[:, 2] <= synth.IMG_W) and np.all(bx[:, 3] <= synth.IMG_H)
            assert np.all(bx[:, 2] - bx[:, 0] >= 8) and np.all(bx[:, 3] - bx[:, 1] >= 8)
            assert np.array_equal(a.centers[s, c, :n, 0], 0.5 * (bx[:, 0] + bx[:, 2]))


def test_rois_host_mirror_and_algorithmic_bytes():
    from bpc_baseline_b200 import pipeline, synth
    boxes = np.zeros((2, 3, 4, 4), np.int32)
    boxes[..., 2] = 100; boxes[..., 3] = 50
    boxes[1, 2, 3] = (5, 6, 25, 36)
    idx = np.full((2, 4, 3), -1, np.int32)
    idx[0, 0] = (0, 1, 2); idx[1, 0] = (1, 1, 3); idx[1, 1] = (0, 0, 0)
    rois = synth.rois_for_matches(boxes, idx, np.array([1, 2]), np.arange(6, dtype=np.int32).reshape(2, 3))
    assert rois.shape == (9, 5) and list(rois[5]) == [5, 5, 6, 25, 36] and list(rois[:, 0]) == [0, 1, 2, 3, 4, 5, 3, 4, 5]
    want = 8 * (3 * 100 * 50) + 3 * 20 * 30 + 9 * (3 * 224 * 224 * 4 + 20)
    assert pipeline.algorithmic_crop_bytes(rois, 224) == want


def test_install_only_touches_imported_modules(lib):
    import sys
    import bpc_baseline_b200 as pkg
    mod = types.ModuleType('fakeref.inference.epipolar_matching')
    sentinel = object()
    mod.match_objects = sentinel
    sys.modules['fakeref.inference.epipolar_matching'] = mod
    try:
        done = pkg.install('fakeref')
        assert done == ['fakeref.inference.epipolar_matching.match_objects']
        assert mod.match_objects is not sentinel
        pkg.uninstall()
        assert mod.match_objects is sentinel
    finally:
        pkg.uninstall()
        sys.modules.pop('fakeref.inference.epipolar_matching', None)


def test_header_is_plain_c(tmp_path):
    """include/bpc_b200.h must be consumable from C (the boundary is a C ABI, not C++)."""
    import shutil
    import subprocess
    gcc = shutil.which('gcc')
    if gcc is None:
        pytest.skip('gcc not available')
    src = tmp_path / 'use_header.c'
    src.write_text('#include "bpc_b200.h"\n'
                   'int probe(void) { return bpc_abi_version() == BPC_ABI_VERSION && BPC_OK == 0 ? (int)sizeof(size_t) : -1; }\n')
    res = subprocess.run([gcc, '-std=c99', '-Wall', '-Werror', '-pedantic', '-I', os.path.join(ROOT, 'include'), '-c', str(src),
                          '-o', str(tmp_path / 'use_header.o')], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr


def test_bop_directory_io(tmp_path):
    """load_camera_params / load_gt_poses / Capture.from_dir: structure and dtypes of the reference loaders
    (camera_utils.py:6-20, data_utils.py:355-409) -- float32 K / R / t, float64 4x4 RT, first camera's GT only."""
    import json
    import cv2
    from bpc_baseline_b200.inference.utils.camera_utils import load_camera_params
    from bpc_baseline_b200.utils.data_utils import Capture, load_gt_poses
    d = str(tmp_path)
    cams = ['cam1', 'cam2', 'cam3']
    for c, cid in enumerate(cams):
        entry = lambda f, t: {'cam_K': [f, 0, 2, 0, f, 3, 0, 0, 1], 'cam_R_w2c': list(np.eye(3).ravel()), 'cam_t_w2c': t}
        with open(os.path.join(d, f'scene_camera_{cid}.json'), 'w') as fh:
            json.dump({'0': entry(1.5, [1, 2, 3]), '7': entry(4.25 + c, [4, 5, 6.125])}, fh)
        os.makedirs(os.path.join(d, f'rgb_{cid}'))
        cv2.imwrite(os.path.join(d, f'rgb_{cid}', '000007.png'), np.full((8, 9, 3), 10 * c, np.uint8))
    eye = list(np.eye(3).ravel())
    with open(os.path.join(d, 'scene_gt_cam1.json'), 'w') as fh:
        json.dump({'7': [{'obj_id': 8, 'cam_R_m2c': eye, 'cam_t_m2c': [1, 1, 1]}, {'obj_id': 9, 'cam_R_m2c': eye, 'cam_t_m2c': [2, 2, 2]}]}, fh)
    with open(os.path.join(d, 'scene_gt_info_cam1.json'), 'w') as fh:
        json.dump({'7': [{}, {}]}, fh)
    p = load_camera_params(d, cams)
    assert p['cam2']['K'][7].dtype == np.float32 and p['cam2']['K'][7].shape == (3, 3) and p['cam2']['K'][7][0, 0] == 5.25
    assert p['cam3']['t'][0].shape == (3,) and p['cam1']['R'][0].dtype == np.float32
    gt = load_gt_poses(d, '', cams, 7, 8)
    assert len(gt) == 1 and gt[0].dtype == np.float64 and gt[0][0, 3] == 1
    assert load_gt_poses(d, '', ['cam2'], 7, 8) == [] and load_gt_poses(d, '', cams, 3, 8) == []
    cap = Capture.from_dir(d, cams, 7, 8)
    assert [im.shape for im in cap.images] == [(8, 9, 3)] * 3 and int(cap.images[2][0, 0, 0]) == 20
    assert all(k.dtype == np.float32 for k in cap.Ks) and all(rt.dtype == np.float64 and rt.shape == (4, 4) for rt in cap.RTs)
    assert cap.RTs[1][2, 3] == 6.125 and cap.gt_poses.shape == (1, 4, 4)


def test_rotation_decode_and_pose_assembly_match_reference():
    """Tail of _estimate_rotation (process_pose.py:211-239) against tests/golden/rotation.npz, which was produced with
    the reference's own decoders (bpc/pose/models/losses.py) and calc_pose_matrix: host code, no GPU involved."""
    import torch
    from bpc_baseline_b200.inference.process_pose import decode_rotations
    from bpc_baseline_b200.utils.data_utils import calc_pose_matrix
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'rotation.npz'))
    for mode in ('euler', 'quat', '6d'):
        raw = torch.from_numpy(g[f'raw_{mode}'])
        rot = decode_rotations(raw, mode)
        assert np.array_equal(decode_rotations(raw, None), rot)            # head inferred from the output width
        for r in range(len(rot)):
            final = g['cam_R'][r].T @ rot[r]                                   # :233
            assert np.allclose(final, g[f'final_{mode}'][r], rtol=0, atol=2e-6), (mode, r)
            assert np.allclose(calc_pose_matrix(final, g['t'][r]), g[f'pose_{mode}'][r], rtol=0, atol=1e-3)
        # batched decode == the reference's one-at-a-time decode, to float32 rounding of the batched torch ops
        assert np.abs(np.stack([g['cam_R'][r].T @ rot[r] for r in range(len(rot))]) - g[f'final_{mode}']).max() < 2e-6


def test_torch_extension_loads_and_registers_its_operators():
    """bpc_baseline_b200/_C.so (csrc/torch_ext.cpp): loads without a GPU, links the same ABI version, registers every
    operator with a schema, and its Meta kernels give shapes / dtypes without running anything."""
    import torch
    from bpc_baseline_b200 import build, ops
    build.build_torch_ext()
    o = ops.load()
    assert int(o.abi_version()) == 2
    for name in ('match_triangulate', 'box_centers', 'build_rois', 'normalise_lut', 'roi_crop', 'roi_crop_u8', 'roi_crop_bf16', 'pack_records', 'fundamental'):
        assert hasattr(o, name), name
    meta = lambda shape, dt: torch.empty(shape, dtype=dt, device='meta')
    r = o.match_triangulate(meta((4, 3, 3, 3), torch.float32), meta((4, 3, 4, 4), torch.float64), meta((4, 3, 9, 2), torch.float64),
                            meta((4, 3), torch.int32), 30.0, None, True)
    assert [tuple(t.shape) for t in r] == [(4, 9, 3), (4,), (4, 9), (4, 9, 3), (4, 9, 3), (4, 3, 3, 3)]
    rois, offs = o.build_rois(meta((4, 3, 9, 4), torch.int32), r[0], r[1], meta((4, 3), torch.int32))
    assert tuple(rois.shape) == (4 * 9 * 3, 5) and tuple(offs.shape) == (5,)
    crops, status = o.roi_crop(meta((2, 64, 64, 3), torch.uint8), rois, 32, [255, 255, 255], True, meta((3, 256), torch.float32), None, 0, None)
    assert tuple(crops.shape) == (108, 3, 32, 32) and crops.dtype == torch.float32 and tuple(status.shape) == (108,)
    with pytest.raises(NotImplementedError):            # no CPU kernel: a CPU tensor cannot fall back to anything
        o.box_centers(torch.zeros((3, 4), dtype=torch.int32))


def _stubs(*names):
    return ''.join(f'def {name}(*args, **kwargs):\n    return "reference"\n\n\n' for name in names)


# The reference package's layout (INTEGRATION.md): the modules that define the hot-path names, and the
# `from ... import` lines of bpc/inference/process_pose.py:23-26.  The bodies are placeholders; install() only rebinds names.
REFERENCE_TREE = {
    'bpc/__init__.py': '',
    'bpc/inference/__init__.py': '',
    'bpc/inference/utils/__init__.py': '',
    'bpc/utils/__init__.py': '',
    'bpc/inference/utils/camera_utils.py': _stubs('compute_fundamental_matrix'),
    'bpc/inference/utils/triangulation.py': _stubs('triangulate_multi_view', 'compute_reprojection_error'),
    'bpc/inference/epipolar_matching.py': _stubs('epipolar_error', 'epipolar_error_full', 'compute_cost_matrix', 'match_objects',
                                                 'triangulate_multi_view'),
    'bpc/utils/data_utils.py': _stubs('letterbox_preserving_aspect_ratio'),
    'bpc/inference/process_pose.py': (
        'from bpc.utils.data_utils import letterbox_preserving_aspect_ratio\n'
        'from bpc.inference.epipolar_matching import compute_cost_matrix, match_objects, triangulate_multi_view\n'
        'from bpc.inference.utils.camera_utils import compute_fundamental_matrix\n\n\n'
        'class PosePrediction:\n    pass\n\n\n'
        'class PoseEstimator:\n    def _match(self, capture, detections):\n        return "reference"\n'),
}


def test_install_rebinds_every_hot_path_name_of_a_reference_tree(lib, tmp_path, monkeypatch):
    """install() against a `bpc` package imported from disk with the reference's layout (REFERENCE_TREE): every hot-path
    name that bpc/inference/process_pose.py:23-26 bound with `from ... import`, the defining modules' own names, and
    PoseEstimator._match must point at this package afterwards; uninstall() restores them."""
    import importlib
    import sys
    import bpc_baseline_b200 as pkg
    for rel, text in REFERENCE_TREE.items():
        (tmp_path / rel).parent.mkdir(parents=True, exist_ok=True)
        (tmp_path / rel).write_text(text)
    monkeypatch.syspath_prepend(str(tmp_path))
    mod = lambda name: importlib.import_module(f'bpc.{name}')
    ref = types.SimpleNamespace(pp=mod('inference.process_pose'), em=mod('inference.epipolar_matching'),
                                cu=mod('inference.utils.camera_utils'), tri=mod('inference.utils.triangulation'),
                                du=mod('utils.data_utils'))
    before = {name: getattr(ref.pp, name) for name in ('compute_cost_matrix', 'match_objects', 'triangulate_multi_view',
                                                      'compute_fundamental_matrix', 'letterbox_preserving_aspect_ratio', 'PosePrediction')}
    ref_match = ref.pp.PoseEstimator._match
    try:
        done = pkg.install('bpc')
        for name in before:                                     # process_pose.py:23-26 (+ its own PosePrediction)
            assert f'bpc.inference.process_pose.{name}' in done
            assert getattr(ref.pp, name).__module__.startswith('bpc_baseline_b200.'), name
        for mod, names in ((ref.em, ('epipolar_error', 'epipolar_error_full', 'compute_cost_matrix', 'match_objects', 'triangulate_multi_view')),
                           (ref.cu, ('compute_fundamental_matrix',)), (ref.tri, ('triangulate_multi_view', 'compute_reprojection_error')),
                           (ref.du, ('letterbox_preserving_aspect_ratio',))):
            for name in names:
                assert getattr(mod, name).__module__.startswith('bpc_baseline_b200.'), (mod.__name__, name)
        assert 'bpc.inference.process_pose.PoseEstimator._match' in done and ref.pp.PoseEstimator._match is not ref_match
        # every name the reference's process_pose imports from the hot-path modules is covered by the patch list
        import ast
        src = REFERENCE_TREE['bpc/inference/process_pose.py']
        hot = {'bpc.utils.data_utils': {'letterbox_preserving_aspect_ratio'}, 'bpc.inference.epipolar_matching': None,
               'bpc.inference.utils.camera_utils': {'compute_fundamental_matrix'}}
        for node in ast.walk(ast.parse(src)):
            if isinstance(node, ast.ImportFrom) and node.module in hot:
                for alias in node.names:
                    if hot[node.module] is None or alias.name in hot[node.module]:
                        assert f'bpc.inference.process_pose.{alias.asname or alias.name}' in done, alias.name
        pkg.uninstall()
        for name, fn in before.items():
            assert getattr(ref.pp, name) is fn
        assert ref.pp.PoseEstimator._match is ref_match
    finally:
        pkg.uninstall()
        for m in [k for k in sys.modules if k == 'bpc' or k.startswith('bpc.')]:
            sys.modules.pop(m, None)
