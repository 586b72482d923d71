"""ctypes binding of ``libaz_stereo.so`` (the C ABI declared in
``include/az_stereo.h``).

The signatures carry plain pointers and sizes only -- PyTorch is used by the
callers for device memory and streams, exactly like the reference drives its
NVRTC kernel with ``data_ptr()``s and the current stream
(``/root/reference/utils/warp_ops.py:79-93``).

There is NO fallback: if the library is missing or a call fails, an exception
is raised.
"""
from __future__ import annotations

import ctypes
import os
import re

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libaz_stereo.so")
HEADER_PATH = os.path.join(os.path.dirname(_PKG_DIR), "include", "az_stereo.h")

_P = ctypes.c_void_p
_I = ctypes.c_int64
_F = ctypes.c_float
_D = ctypes.c_double

# name -> (restype, argtypes); mirrors include/az_stereo.h one to one
SIGNATURES = {
    "az_version": (ctypes.c_char_p, []),
    "az_error_string": (ctypes.c_char_p, [ctypes.c_int]),
    "az_concat_volume_fwd": (ctypes.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "az_concat_volume_bwd": (ctypes.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "az_concat_volume_fwd_ndhwc": (ctypes.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "az_concat_volume_bwd_ndhwc": (ctypes.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "az_concat_volume_fwd_16": (ctypes.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, ctypes.c_int, _P]),
    "az_concat_volume_bwd_16": (ctypes.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, ctypes.c_int, ctypes.c_int, _P]),
    "az_volume_conv0_pack": (ctypes.c_int, [_P, _P, _P]),
    "az_volume_conv0_fwd": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, ctypes.c_int, _P]),
    "az_volume_conv0_pack_16": (ctypes.c_int, [_P, _P, ctypes.c_int, _P]),
    "az_volume_conv0_fwd_16": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, ctypes.c_int, ctypes.c_int, _P]),
    "az_volume_conv0_bwd_workspace_bytes": (_I, [_I, _I, _I, _I]),
    "az_volume_conv0_bwd": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "az_volume_conv0_bwd_16": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, ctypes.c_int, ctypes.c_int, _P]),
    "az_gwc_volume_fwd": (ctypes.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "az_gwc_volume_bwd": (ctypes.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "az_soft_argmin_fwd": (ctypes.c_int, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "az_soft_argmin_bwd": (ctypes.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "az_soft_argmin_fwd_16": (ctypes.c_int, [_P, _P, _P, _I, _I, _I, _I, ctypes.c_int, _P]),
    "az_soft_argmin_bwd_16": (ctypes.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, ctypes.c_int, _P]),
    "az_upsample_soft_argmin_fwd": (ctypes.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "az_upsample_soft_argmin_workspace_bytes": (_I, [_I, _I, _I, _I, _I]),
    "az_upsample_soft_argmin_bwd": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "az_upsample_soft_argmin_fwd_16": (ctypes.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, ctypes.c_int, _P]),
    "az_upsample_soft_argmin_bwd_16": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, ctypes.c_int, _P]),
    "az_warp_fwd": (ctypes.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "az_warp_bwd": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "az_reproj_workspace_bytes": (_I, [_I, _I]),
    "az_reproj_loss_fwd": (ctypes.c_int, [_P, _P, _P, _F, _P, _P, _P, _I, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "az_reproj_loss_bwd": (ctypes.c_int, [_P, _P, _P, _F, _P, _I, _I, _I, _I, _I, _P]),
    "az_reproj_loss_img_bwd": (ctypes.c_int, [_P, _P, _P, _F, _P, _P, _P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "az_patch_fold": (ctypes.c_int, [_P, _P, _F, _P, _P, _I, _P, _I, _I, _I, _I, _P]),
    "az_bilinear_rescale_fwd": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _F, _F, _P]),
    "az_bilinear_rescale_bwd": (ctypes.c_int, [_P, _P, _I, _I, _I, _I, _I, _F, _F, _F, _P]),
    "az_scatter_warp": (ctypes.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "az_scatter_warp_gt": (ctypes.c_int, [_P, _P, _P, _P, _F, _I, _I, _I, _P]),
    "az_temporal_ir_workspace_bytes": (_I, [_I, _I, _I]),
    "az_temporal_ir": (ctypes.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _D, _P]),
    "az_sim_ir_pattern_workspace_bytes": (_I, [_I, _I, _I, _I]),
    "az_sim_ir_pattern": (ctypes.c_int, [_P, _P, ctypes.c_int, _P, _P, _I, _I, _I, _I, _D, _P]),
    "az_error_metrics_workspace_bytes": (_I, [_I, _I, _I]),
    "az_error_metrics": (ctypes.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "az_local_contrast_norm": (ctypes.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _F, _P]),
}

# CUDA kernels enqueued by one successful call of each compute entry point
KERNELS_PER_CALL = {"az_reproj_loss_fwd": 2, "az_warp_bwd": 2, "az_bilinear_rescale_fwd": 1, "az_temporal_ir": 3, "az_upsample_soft_argmin_bwd": 3, "az_upsample_soft_argmin_bwd_16": 3, "az_error_metrics": 2, "az_sim_ir_pattern": 4, "az_volume_conv0_bwd": 4, "az_volume_conv0_bwd_16": 4}

_lib = None
launch_count = 0    # C-ABI compute calls issued
kernel_launches = 0  # CUDA kernels those calls enqueued (bench.py reports it as gpu_launches)


def header_symbols() -> list[str]:
    """Function names declared in include/az_stereo.h."""
    text = open(HEADER_PATH).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(az_[a-z0-9_]+)\s*\(", text)))


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m activezero_b200.build` "
            "(or __graft_entry__.build()). activezero_b200 has no CPU or PyTorch fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the build is stale: loud by design
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def call(name: str, *args, batch=None):
    """Invoke a compute entry point; raise on any non-zero status.  ``batch=0`` (an empty batch: the reference's
    torch code returns empty tensors there) enqueues nothing -- there is no element to compute and a zero-sized
    grid is not launchable; the C ABI itself rejects non-positive sizes."""
    global launch_count, kernel_launches
    lib = load()
    if batch is not None and int(batch) == 0:
        return
    rc = getattr(lib, name)(*args)
    launch_count += 1
    kernel_launches += KERNELS_PER_CALL.get(name, 1)
    if rc != 0:
        msg = lib.az_error_string(rc).decode()
        raise RuntimeError(f"{name} failed with status {rc}: {msg}")


def query(name: str, *args) -> int:
    """Workspace-size queries; never negative (an empty batch needs no workspace)."""
    return max(0, int(getattr(load(), name)(*args)))
