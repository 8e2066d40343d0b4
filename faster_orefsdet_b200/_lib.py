"""Loader for the C-ABI CUDA library (``libfod_b200.so``, see include/fod_b200.h).

There is no fallback: if the library is missing or a call fails the error is
raised.  ``build()`` compiles it in-tree with nvcc for sm_100a.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FOD_B200_LIB_DEV") or os.path.join(_HERE, "libfod_b200.so")  # env: kernel A/B experiments only
CSRC = os.path.join(_HERE, "csrc")

FOD_STATUS_CAND_OVERFLOW = 1
FOD_STATUS_PROPOSAL_OVERFLOW = 2
FOD_STATUS_DET_OVERFLOW = 4
FOD_NMS_MAX_BOXES = 8192


class fod_level_t(ctypes.Structure):
    _fields_ = [("height", ctypes.c_int), ("width", ctypes.c_int), ("stride", ctypes.c_int)]


class FodError(RuntimeError):
    pass


_lock = threading.Lock()
_lib = None

_vp, _i, _f, _d = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_double
_PROTOTYPES = {
    "fod_version": ([], _i),
    "fod_last_error": ([ctypes.c_char_p, ctypes.c_size_t], _i),
    "fod_support_taps": ([_vp, _i, _i, _i, _vp, _vp], _i),
    "fod_correlate_levels": ([ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.POINTER(fod_level_t), _i, _vp, _vp,
                              ctypes.POINTER(_vp), ctypes.POINTER(_vp), _i, _i, _vp], _i),
    "fod_decode_topk": ([ctypes.POINTER(_vp), ctypes.POINTER(_vp), ctypes.POINTER(fod_level_t), _i, _i, _i, _i,
                         ctypes.POINTER(_i), ctypes.POINTER(_i), ctypes.POINTER(_f), _f, _i,
                         _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp], _i),
    "fod_decode_topk_taps": ([ctypes.POINTER(_vp), ctypes.POINTER(_i), ctypes.POINTER(_f), ctypes.POINTER(fod_level_t), _i, _i,
                              ctypes.POINTER(_f), _f, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp], _i),
    "fod_decode_topk_taps_workspace_bytes": ([ctypes.POINTER(fod_level_t), _i, _i], ctypes.c_size_t),
    "fod_nms_proposals": ([_vp, _vp, _vp, _i, _i, _d, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp], _i),
    "fod_rpn_proposals_workspace_bytes": ([ctypes.POINTER(fod_level_t), _i, _i, _i, _i], ctypes.c_size_t),
    "fod_rpn_proposals": ([ctypes.POINTER(_vp), ctypes.POINTER(_i), ctypes.POINTER(_vp), ctypes.POINTER(fod_level_t), _i, _i, _i,
                           _vp, _i, ctypes.POINTER(_f), _f, _d, _i, _vp, _vp, _vp, _vp, _vp], _i),
    "fod_roi_align_workspace_bytes": ([_i, _i, _i], ctypes.c_size_t),
    "fod_roi_align": ([ctypes.POINTER(_vp), ctypes.POINTER(fod_level_t), _i, _i, _i, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp],
                      _i),
    "fod_roi_align_wide": ([ctypes.POINTER(_vp), ctypes.POINTER(fod_level_t), _i, _i, _i, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp,
                            _vp], _i),
    "fod_roi_align_per_roi": ([ctypes.POINTER(_vp), ctypes.POINTER(fod_level_t), _i, _i, _i, _vp, _vp, _i, _i, _i, _i, _vp, _vp,
                               _vp, _vp], _i),
    "fod_relation_head": ([_vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, ctypes.POINTER(_f), _vp, _vp, _vp, _vp,
                           _vp], _i),
    "fod_final_detect": ([_vp, _vp, _vp, _i, _i, _i, _f, _d, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp], _i),
    "fod_batched_nms": ([_vp, _vp, _vp, _i, _d, _vp, _vp, _vp], _i),
    "fod_group_norm_workspace_bytes": ([_i, _i], ctypes.c_size_t),
    "fod_group_norm_nhwc": ([_vp, _i, ctypes.c_long, _i, _i, _vp, _vp, _f, _i, _vp, _vp, _i, _vp, _vp], _i),
    "fod_absmax": ([_vp, ctypes.c_size_t, _vp, _vp], _i),
    "fod_absmax_rows": ([_vp, _i, ctypes.c_size_t, _vp, _vp], _i),
    "fod_stem_patches": ([_vp, _i, _i, _i, _vp, _vp], _i),
    "fod_stem_patches_u8": ([_vp, _i, _i, _i, ctypes.POINTER(_f), ctypes.POINTER(_f), _vp, _vp], _i),
    "fod_stem1_u8_tc": ([_vp, _i, _i, _i, ctypes.POINTER(_f), ctypes.POINTER(_f), _vp, _vp, _vp, ctypes.c_long, _vp, _i, _vp], _i),
    "fod_conv2d_nhwc_split": ([_vp, _i, _i, _i, _i, ctypes.c_long, _vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _vp, ctypes.c_long, _vp, _vp,
                               _vp, _vp, _f, _f, _i, ctypes.POINTER(_i), _vp], _i),
    "fod_stem1_u8_tc_split": ([_vp, _i, _i, _i, ctypes.POINTER(_f), ctypes.POINTER(_f), _vp, _vp, _vp, ctypes.c_long, _vp, _i, _vp,
                               _vp], _i),
    "fod_stem1_u8": ([_vp, _i, _i, _i, ctypes.POINTER(_f), ctypes.POINTER(_f), _vp, _vp, _vp, _vp, _i, _vp], _i),
    "fod_maxpool3x3s2_nhwc": ([_vp, _i, _i, _i, _i, ctypes.c_long, _vp, _vp, ctypes.c_long, _vp], _i),
    "fod_maxpool3x3s2_nhwc_split": ([_vp, _i, _i, _i, _i, ctypes.c_long, _vp, _vp, ctypes.c_long, _vp, _vp], _i),
    "fod_conv2d_packed_floats": ([_i, _i, _i], ctypes.c_size_t),
    "fod_conv2d_pack_weights": ([_vp, _i, _i, _i, _vp, _vp], _i),
    "fod_conv2d_nhwc": ([_vp, _i, _i, _i, _i, ctypes.c_long, _vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _vp, ctypes.c_long, _vp, _vp,
                         _i, _vp, _vp, _i, _vp, _vp, _vp], _i),
    "fod_group_norm_affine": ([_vp, _vp, _i, _i, _i, _i, ctypes.c_long, _vp, _vp, _f, _vp, _vp, _vp, _vp, _i, _vp], _i),
    "fod_conv2d_tiles_per_image": ([_i, _i], _i),
    "fod_ese_gate": ([_vp, _i, _i, _i, ctypes.c_long, _vp, _vp, _vp, _vp], _i),
}

EXPORTED_SYMBOLS = tuple(_PROTOTYPES)


def build(verbose: bool = False) -> str:
    """Compile csrc/*.cu into libfod_b200.so (nvcc, sm_100a, -lineinfo)."""
    res = subprocess.run(["make", "-C", CSRC, "-j8"], capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
        print(res.stderr)
    if res.returncode != 0:
        raise FodError("building libfod_b200.so failed:\n" + res.stderr[-4000:])
    return LIB_PATH


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise FodError(
                        f"{LIB_PATH} not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(or `make -C faster_orefsdet_b200/csrc`). There is no CPU / PyTorch fallback for the head.")
                handle = ctypes.CDLL(LIB_PATH)
                for name, (argtypes, restype) in _PROTOTYPES.items():
                    fn = getattr(handle, name)
                    fn.argtypes, fn.restype = argtypes, restype
                _lib = handle
    return _lib


def last_error() -> str:
    buf = ctypes.create_string_buffer(512)
    lib().fod_last_error(buf, 512)
    return buf.value.decode(errors="replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise FodError(f"{what} failed (code {rc}): {last_error()}")
