"""ctypes binding of libbpc_b200.so (include/bpc_b200.h).  No CPU fallback: if the library is
missing or a call fails, this raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('BPC_LIB') or os.path.join(HERE, 'libbpc_b200.so')      # BPC_LIB: experiment builds

_p = C.c_void_p
_i = C.c_int
_f = C.c_float
_sz = C.c_size_t

# name -> (restype, argtypes); mirrors include/bpc_b200.h one to one
SIGNATURES = {
    'bpc_abi_version': (_i, []),
    'bpc_error_string': (C.c_char_p, [_i]),
    'bpc_launch_count': (C.c_ulonglong, []),
    'bpc_fundamental': (_i, [_p, _p, _i, _p, _p]),
    'bpc_cost_tensor': (_i, [_p, _p, _p, _i, _i, _p, _p]),
    'bpc_match_objects': (_i, [_p, _i, _i, _i, _i, _f, _p, _p, _p]),
    'bpc_match_workspace_bytes': (_sz, [_i, _i]),
    'bpc_match_triangulate': (_i, [_p, _p, _p, _p, _i, _i, _f, _i, C.c_double, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    'bpc_pack_records_bytes': (_sz, [_i, _i]),
    'bpc_pack_records': (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _p, _p]),
    'bpc_triangulate': (_i, [_p, _p, _i, _p, _p]),
    'bpc_projection': (_i, [_p, _p, _i, _p, _p]),
    'bpc_reprojection_error': (_i, [_p, _p, _p, _i, _p, _p]),
    'bpc_epipolar_error': (_i, [_p, _p, _p, _i, _p, _p]),
    'bpc_epipolar_error_full': (_i, [_p, _p, _i, _p, _p]),
    'bpc_triangulate_views': (_i, [_p, _p, _i, _i, _p, _p]),
    'bpc_box_centers': (_i, [_p, _i, _p, _p]),
    'bpc_detections_from_yolo': (_i, [_p, _p, _p, _p, _i, _i, _f, _i, _p, _p, _p, _p]),
    'bpc_build_rois': (_i, [_p, _p, _p, _p, _i, _i, _i, _p, _p, _p]),
    'bpc_train_rois': (_i, [_p, _p, _p, _p, _i, _i, _i, _p, _p]),
    'bpc_roi_crop_workspace_bytes': (_sz, [_i, _i]),
    'bpc_roi_crop': (_i, [_p, _i, _i, _i, _p, _i, _p, _i, _i, _p, _i, _p, _p, _p, _p, _sz, _p]),
    'bpc_roi_crop_u8': (_i, [_p, _i, _i, _i, _p, _i, _p, _i, _i, _p, _p, _p, _p, _sz, _p]),
    'bpc_roi_crop_bf16': (_i, [_p, _i, _i, _i, _p, _i, _p, _i, _i, _p, _i, _p, _p, _p, _p, _sz, _p]),
    'bpc_normalise_lut': (_i, [_p, _p, _p, _p]),
    'bpc_crops_normalise': (_i, [_p, _p, _i, _i, _i, _p, _p, _p]),
    'bpc_color_jitter': (_i, [_p, _i, _i, _p, _p, _i, _p, _p, _p]),
}

_lib = None
ABI_VERSION = 2


class BpcError(RuntimeError):
    pass


def load():
    """Load the shared library once.  Raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BpcError(f'{LIB_PATH} not found: build it with `python -m bpc_baseline_b200.build` '
                       '(or __graft_entry__.build()); there is no CPU fallback')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)            # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.bpc_abi_version() != ABI_VERSION:
        raise BpcError(f'ABI version mismatch: library {lib.bpc_abi_version()}, binding {ABI_VERSION}')
    _lib = lib
    return lib


def check(code: int, what: str):
    if code != 0:
        msg = load().bpc_error_string(code).decode()
        raise BpcError(f'{what} failed with code {code}: {msg}')


def launch_count() -> int:
    return int(load().bpc_launch_count())
