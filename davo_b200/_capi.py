"""ctypes binding of libdavo_b200.so (the C ABI in ``include/davo_b200.h``).

There is no CPU fallback: if the shared library is missing or a symbol is
absent, importing callers get an ImportError; if there is no sm_100a device,
``davo_create`` fails and the wrapper raises RuntimeError with the library's
message.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_LIB = None

SYMBOLS = (
    "davo_create", "davo_set_weight", "davo_finalize_weights", "davo_forward",
    "davo_forward_host", "davo_get_intermediate", "davo_last_launch_count",
    "davo_last_host_copy_bytes",
    "davo_profile_layers", "davo_debug_set_conv_impl", "davo_forward_pairs", "davo_forward_host_pairs",
    "davo_forward_features", "davo_debug_flows_to_half", "davo_debug_labels_to_bytes", "davo_forward_host_compact", "davo_bind_host_numa",
    "davo_compose_trajectory", "davo_kitti_errors", "davo_decode_jpeg_batch",
    "davo_forward_host_pairs_async", "davo_forward_host_compact_async", "davo_host_wait",
    "davo_comm_unique_id", "davo_comm_create", "davo_comm_world", "davo_allgather_poses",
    "davo_forward_sequence", "davo_forward_sequence_host",
    "davo_odometry_create", "davo_odometry_push", "davo_odometry_reset", "davo_odometry_frames",
    "davo_odometry_push_many", "davo_odometry_push_many_host", "davo_odometry_move",
    "davo_last_error",
    "davo_destroy", "davo_build_info", "davo_config_bytes", "davo_odometry_destroy",
)


class DavoConfigC(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "H", "W", "max_batch", "posenn", "cnv6_out", "in_mode", "att_src", "att_tgt_ones",
        "mask_mode", "se_act", "flow_abs", "flow_norm", "posenn_se", "micro_batch", "depth_norm", "se_pool", "se_hidden",
        "pixel_map", "depth_split", "flow_f16", "batch_norm")]


class DavoFeaturesC(C.Structure):
    """include/davo_b200.h: davo_features (device pointers, NULL skips the output)."""
    _fields_ = [(n, C.c_void_p) for n in (
        "image", "attention", "masked_image", "seg_19", "seg_color", "flow_color", "cnv6_rot", "cnv6_trans")]


def lib_path() -> str:
    return _build.LIB


def load() -> C.CDLL:
    """Load (building first if the sources are newer and nvcc exists)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if _build.is_stale():
        try:
            _build.build()
        except Exception as e:  # no nvcc on this box: use the shipped .so if any
            if not os.path.exists(path):
                raise ImportError("libdavo_b200.so is not built and cannot be built here: %s" % e)
    try:
        lib = C.CDLL(path)
    except OSError as e:
        raise ImportError("cannot load %s: %s (there is no CPU fallback)" % (path, e))
    for s in SYMBOLS:
        if not hasattr(lib, s):
            raise ImportError("%s does not export %s" % (path, s))
    vp, ip, fp = C.c_void_p, C.c_int, C.POINTER(C.c_float)
    lib.davo_create.argtypes = [C.POINTER(DavoConfigC), ip, C.POINTER(vp)]
    lib.davo_set_weight.argtypes = [vp, C.c_char_p, vp, C.POINTER(C.c_int64), ip]
    lib.davo_finalize_weights.argtypes = [vp]
    lib.davo_forward.argtypes = [vp, ip, vp, vp, vp, vp, vp, vp]
    lib.davo_forward_host.argtypes = [vp, ip, vp, vp, vp, vp, vp, vp]
    lib.davo_forward_pairs.argtypes = [vp, ip, ip, vp, vp, vp, vp, vp, vp]
    lib.davo_forward_host_pairs.argtypes = [vp, ip, ip, vp, vp, vp, vp, vp, vp]
    lib.davo_forward_host_compact.argtypes = [vp, ip, ip, vp, vp, vp, vp, vp, vp]
    lib.davo_bind_host_numa.argtypes = [vp]
    lib.davo_compose_trajectory.argtypes = [vp, vp, ip, vp, vp]
    lib.davo_kitti_errors.argtypes = [vp, vp, vp, ip, vp, fp, vp]
    lib.davo_decode_jpeg_batch.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_int64), ip, vp, vp]
    lib.davo_forward_host_pairs_async.argtypes = [vp, ip, ip, vp, vp, vp, vp, vp, vp, C.POINTER(C.c_longlong)]
    lib.davo_forward_host_compact_async.argtypes = [vp, ip, ip, vp, vp, vp, vp, vp, vp, C.POINTER(C.c_longlong)]
    lib.davo_host_wait.argtypes = [vp, C.c_longlong]
    lib.davo_forward_sequence.argtypes = [vp, ip, ip, vp, vp, vp, vp, vp, vp, vp]
    lib.davo_forward_sequence_host.argtypes = [vp, ip, ip, vp, vp, vp, vp, vp, vp, vp, C.POINTER(C.c_longlong)]
    lib.davo_odometry_create.argtypes = [vp, ip, ip, ip, C.POINTER(vp)]
    lib.davo_odometry_push.argtypes = [vp, ip, vp, vp, vp, vp, vp, vp, vp, C.POINTER(ip), C.POINTER(ip), vp,
                                       C.POINTER(C.c_longlong)]
    lib.davo_odometry_push_many.argtypes = [ip, C.POINTER(vp), C.POINTER(ip)] + [C.POINTER(vp)] * 7 + [
        C.POINTER(ip), C.POINTER(ip), vp]
    lib.davo_odometry_push_many_host.argtypes = [ip, C.POINTER(vp), C.POINTER(ip)] + [C.POINTER(vp)] * 7 + [
        C.POINTER(ip), C.POINTER(ip), vp, C.POINTER(C.c_longlong)]
    lib.davo_odometry_move.argtypes = [vp, vp]
    lib.davo_odometry_reset.argtypes = [vp]
    lib.davo_odometry_frames.argtypes = [vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    lib.davo_odometry_destroy.argtypes = [vp]
    lib.davo_odometry_destroy.restype = None
    lib.davo_get_intermediate.argtypes = [vp, C.c_char_p, ip, vp, C.c_int64, C.POINTER(C.c_int64)]
    lib.davo_last_launch_count.argtypes = [vp]
    lib.davo_last_host_copy_bytes.argtypes = [vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    lib.davo_profile_layers.argtypes = [vp, ip, fp, C.POINTER(ip), vp]
    lib.davo_debug_set_conv_impl.argtypes = [vp, ip]
    lib.davo_forward_features.argtypes = [vp, ip, vp, vp, vp, vp, vp, C.POINTER(DavoFeaturesC), vp]
    lib.davo_debug_flows_to_half.argtypes = [vp, vp, C.c_longlong, ip]
    lib.davo_debug_labels_to_bytes.argtypes = [vp, vp, C.c_longlong, ip]
    lib.davo_comm_unique_id.argtypes = [vp]
    lib.davo_comm_create.argtypes = [vp, vp, ip, ip]
    lib.davo_comm_world.argtypes = [vp, C.POINTER(ip), C.POINTER(ip)]
    lib.davo_allgather_poses.argtypes = [vp, vp, vp, ip, vp, vp]
    lib.davo_last_error.argtypes = [vp]
    lib.davo_last_error.restype = C.c_char_p
    lib.davo_destroy.argtypes = [vp]
    lib.davo_destroy.restype = None
    lib.davo_build_info.restype = C.c_char_p
    lib.davo_config_bytes.restype = ip
    if lib.davo_config_bytes() != C.sizeof(DavoConfigC):
        raise ImportError("%s: davo_config is %d bytes in the library, %d in this binding (rebuild: python davo_b200/build.py --force)"
                          % (path, lib.davo_config_bytes(), C.sizeof(DavoConfigC)))
    for s in SYMBOLS[:SYMBOLS.index("davo_last_error")]:
        getattr(lib, s).restype = ip
    _LIB = lib
    return lib


PAIRS = {"all": 0, "trajectory": 1, "trajectory_first": 2}     # include/davo_b200.h DAVO_PAIRS_*


def last_error(lib, handle) -> str:
    msg = lib.davo_last_error(handle)
    return msg.decode() if msg else ""
