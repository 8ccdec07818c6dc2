"""ctypes binding of libp2m_b200.so (C ABI declared in include/p2m_b200.h).

There is deliberately NO fallback: if the shared library is missing or a call fails, a
RuntimeError is raised (the product has no CPU / eager path — north_star, SURVEY.md §7).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libp2m_b200.so")

P2M_PREC_FP32_SIMT = 0
P2M_PREC_FP16X3_TC = 1
PRECISIONS = {"fp32": P2M_PREC_FP32_SIMT, "fp16x3": P2M_PREC_FP16X3_TC}


def default_precision() -> int:
    """Precision of new modules / graph handles: the tcgen05 path (fp16x3: error-compensated split, fp32
    accumulate, 1e-4 parity like the fp32 path) unless the environment says ``P2M_PRECISION=fp32`` (the CUDA-core
    escape hatch for activations beyond fp16's range).  A drop-in user (install.py) therefore gets the fast path
    without touching the module; ``Pose2Mesh.set_precision`` / ``set_default_precision`` still override it."""
    name = os.environ.get("P2M_PRECISION", "fp16x3").strip().lower()
    if name not in PRECISIONS:
        raise RuntimeError(f"P2M_PRECISION={name!r}: expected one of {sorted(PRECISIONS)}")
    return PRECISIONS[name]

c_float_p = C.POINTER(C.c_float)
c_int32_p = C.POINTER(C.c_int32)
c_int64_p = C.POINTER(C.c_int64)


class ModelDesc(C.Structure):
    _fields_ = [
        ("n_levels", C.c_int32),
        ("level_size", c_int32_p),
        ("rowptr", C.POINTER(c_int32_p)),
        ("colidx", C.POINTER(c_int32_p)),
        ("values", C.POINTER(c_float_p)),
        ("n_blocks", C.c_int32),
        ("block_len", c_int32_p),
        ("block_chans", c_int32_p),
        ("device", C.c_int32),
    ]


class Params(C.Structure):
    _fields_ = [
        ("fc_w", C.c_void_p),
        ("fc_b", C.c_void_p),
        ("cl_w", C.POINTER(C.c_void_p)),
        ("cl_b", C.POINTER(C.c_void_p)),
        ("bn_w", C.POINTER(C.c_void_p)),
        ("bn_b", C.POINTER(C.c_void_p)),
        ("bn_rm", C.POINTER(C.c_void_p)),
        ("bn_rv", C.POINTER(C.c_void_p)),
        ("bn_nbt", C.POINTER(C.c_void_p)),
    ]


class ConvFwdArgs(C.Structure):
    _fields_ = [
        ("level", C.c_int32), ("batch", C.c_int32), ("fin", C.c_int32), ("fout", C.c_int32),
        ("x", C.c_void_p), ("weight", C.c_void_p), ("bias", C.c_void_p),
        ("bn_mode", C.c_int32),
        ("bn_weight", C.c_void_p), ("bn_bias", C.c_void_p),
        ("bn_running_mean", C.c_void_p), ("bn_running_var", C.c_void_p),
        ("bn_num_batches_tracked", C.c_void_p),
        ("save_mean", C.c_void_p), ("save_invstd", C.c_void_p),
        ("relu", C.c_int32),
        ("y", C.c_void_p),
    ]


class ConvBwdArgs(C.Structure):
    _fields_ = [
        ("level", C.c_int32), ("batch", C.c_int32), ("fin", C.c_int32), ("fout", C.c_int32),
        ("x", C.c_void_p), ("weight", C.c_void_p), ("dz", C.c_void_p),
        ("dx", C.c_void_p), ("dweight", C.c_void_p), ("dbias", C.c_void_p),
    ]


class PoseNetStage(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("w1_w", "w1_b", "w2_w", "w2_b", "bn1_w", "bn1_b", "bn1_rm", "bn1_rv",
                                          "bn2_w", "bn2_b", "bn2_rm", "bn2_rv")]


class PoseNetParams(C.Structure):
    _fields_ = [("num_joint", C.c_int32), ("hidden", C.c_int32), ("num_stage", C.c_int32),
                ("w1_w", C.c_void_p), ("w1_b", C.c_void_p), ("w2_w", C.c_void_p), ("w2_b", C.c_void_p),
                ("stages", C.POINTER(PoseNetStage))]


EXPORTS = [
    "p2m_model_create", "p2m_model_destroy", "p2m_model_num_layers", "p2m_model_layer_info",
    "p2m_model_set_precision", "p2m_debug_kernel_status", "p2m_debug_set_trace", "p2m_debug_set_split_t1", "p2m_debug_set_fuse_head", "p2m_debug_set_elide_padding", "p2m_debug_set_dedup_padding", "p2m_debug_set_dw_swap", "p2m_model_set_profiling", "p2m_model_layer_times_ms", "p2m_meshnet_workspace_bytes", "p2m_meshnet_backward_scratch_bytes",
    "p2m_meshnet_forward", "p2m_meshnet_backward", "p2m_model_set_output_gather", "p2m_meshnet_forward_vertices", "p2m_meshnet_host_io_bytes", "p2m_meshnet_forward_host", "p2m_meshnet_forward_vertices_host",
    "p2m_cheb_conv_workspace_bytes", "p2m_cheb_conv_fwd", "p2m_cheb_conv_bwd", "p2m_graph_match_level", "p2m_posenet_workspace_bytes", "p2m_posenet_forward", "p2m_regress_joints", "p2m_normalize_pose2d", "p2m_crop_pose2d", "p2m_fit_camera", "p2m_mesh_losses", "p2m_coord_loss",
    "p2m_last_error", "p2m_version", "p2m_launch_count", "p2m_launch_count_reset",
]

_lib = None
_lock = threading.Lock()


def load() -> C.CDLL:
    """Load (once) and type the shared library.  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -m pose2mesh_release_b200.build` "
                "(or __graft_entry__.build()).  pose2mesh_release_b200 has no CPU / eager fallback.")
        lib = C.CDLL(LIB_PATH)
        vp, i32, i64, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t
        lib.p2m_model_create.argtypes = [C.POINTER(ModelDesc), C.POINTER(vp)]
        lib.p2m_model_create.restype = C.c_int
        lib.p2m_model_destroy.argtypes = [vp]
        lib.p2m_model_destroy.restype = None
        lib.p2m_model_num_layers.argtypes = [vp]
        lib.p2m_model_num_layers.restype = C.c_int
        lib.p2m_model_layer_info.argtypes = [vp, C.c_int, c_int32_p]
        lib.p2m_model_layer_info.restype = C.c_int
        lib.p2m_model_set_precision.argtypes = [vp, C.c_int]
        lib.p2m_model_set_precision.restype = C.c_int
        lib.p2m_model_set_profiling.argtypes = [vp, C.c_int]
        lib.p2m_model_set_profiling.restype = C.c_int
        lib.p2m_model_layer_times_ms.argtypes = [vp, c_float_p, C.c_int]
        lib.p2m_model_layer_times_ms.restype = C.c_int
        lib.p2m_debug_set_split_t1.argtypes = [vp, C.c_int]
        lib.p2m_debug_set_split_t1.restype = C.c_int
        lib.p2m_debug_set_fuse_head.argtypes = [vp, C.c_int]
        lib.p2m_debug_set_fuse_head.restype = C.c_int
        lib.p2m_debug_set_elide_padding.argtypes = [vp, C.c_int]
        lib.p2m_debug_set_elide_padding.restype = C.c_int
        lib.p2m_debug_set_dedup_padding.argtypes = [vp, C.c_int]
        lib.p2m_debug_set_dedup_padding.restype = C.c_int
        lib.p2m_debug_set_dw_swap.argtypes = [vp, C.c_int]
        lib.p2m_debug_set_dw_swap.restype = C.c_int
        lib.p2m_debug_set_trace.argtypes = [vp, vp]
        lib.p2m_debug_set_trace.restype = C.c_int
        lib.p2m_debug_kernel_status.argtypes = [vp, c_int32_p]
        lib.p2m_debug_kernel_status.restype = C.c_int
        lib.p2m_meshnet_workspace_bytes.argtypes = [vp, C.c_int, C.c_int]
        lib.p2m_meshnet_workspace_bytes.restype = sz
        lib.p2m_meshnet_backward_scratch_bytes.argtypes = [vp, C.c_int]
        lib.p2m_meshnet_backward_scratch_bytes.restype = sz
        lib.p2m_meshnet_host_io_bytes.argtypes = [vp, C.c_int]
        lib.p2m_meshnet_host_io_bytes.restype = sz
        lib.p2m_meshnet_forward.argtypes = [vp, C.POINTER(Params), vp, vp, C.c_int, C.c_int, vp, sz, vp]
        lib.p2m_meshnet_forward.restype = C.c_int
        lib.p2m_model_set_output_gather.argtypes = [vp, c_int32_p, C.c_int]
        lib.p2m_model_set_output_gather.restype = C.c_int
        lib.p2m_meshnet_forward_vertices.argtypes = [vp, C.POINTER(Params), vp, vp, C.c_int, vp, sz, vp]
        lib.p2m_meshnet_forward_vertices.restype = C.c_int
        lib.p2m_meshnet_forward_host.argtypes = [vp, C.POINTER(Params), vp, vp, C.c_int, vp, sz, vp]
        lib.p2m_meshnet_forward_host.restype = C.c_int
        lib.p2m_meshnet_forward_vertices_host.argtypes = [vp, C.POINTER(Params), vp, vp, C.c_int, vp, sz, vp]
        lib.p2m_meshnet_forward_vertices_host.restype = C.c_int
        lib.p2m_meshnet_backward.argtypes = [vp, C.POINTER(Params), C.POINTER(Params), vp, vp, vp, C.c_int, vp, sz,
                                             vp, sz, vp]
        lib.p2m_meshnet_backward.restype = C.c_int
        lib.p2m_cheb_conv_workspace_bytes.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int]
        lib.p2m_cheb_conv_workspace_bytes.restype = sz
        lib.p2m_cheb_conv_fwd.argtypes = [vp, C.POINTER(ConvFwdArgs), vp, sz, vp]
        lib.p2m_cheb_conv_fwd.restype = C.c_int
        lib.p2m_cheb_conv_bwd.argtypes = [vp, C.POINTER(ConvBwdArgs), vp, sz, vp]
        lib.p2m_cheb_conv_bwd.restype = C.c_int
        lib.p2m_posenet_workspace_bytes.argtypes = [C.c_int, C.c_int]
        lib.p2m_posenet_workspace_bytes.restype = sz
        lib.p2m_posenet_forward.argtypes = [C.POINTER(PoseNetParams), vp, vp, vp, C.c_int, vp, sz, vp]
        lib.p2m_posenet_forward.restype = C.c_int
        lib.p2m_regress_joints.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]
        lib.p2m_regress_joints.restype = C.c_int
        lib.p2m_normalize_pose2d.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]
        lib.p2m_normalize_pose2d.restype = C.c_int
        lib.p2m_crop_pose2d.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int,
                                        vp]
        lib.p2m_crop_pose2d.restype = C.c_int
        lib.p2m_fit_camera.argtypes = [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, vp]
        lib.p2m_fit_camera.restype = C.c_int
        lib.p2m_mesh_losses.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]
        lib.p2m_mesh_losses.restype = C.c_int
        lib.p2m_coord_loss.argtypes = [vp, vp, vp, i64, vp, vp, vp, vp]
        lib.p2m_coord_loss.restype = C.c_int
        lib.p2m_graph_match_level.argtypes = [i64, c_int32_p, c_int32_p, C.POINTER(C.c_double), c_int64_p,
                                              C.POINTER(C.c_double), c_int32_p]
        lib.p2m_graph_match_level.restype = i32
        lib.p2m_last_error.argtypes = []
        lib.p2m_last_error.restype = C.c_char_p
        lib.p2m_version.argtypes = []
        lib.p2m_version.restype = C.c_char_p
        lib.p2m_launch_count.argtypes = []
        lib.p2m_launch_count.restype = i64
        lib.p2m_launch_count_reset.argtypes = []
        lib.p2m_launch_count_reset.restype = None
        _lib = lib
    return _lib


def check(status: int, what: str = "p2m call"):
    if status != 0:
        msg = load().p2m_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (status {status}): {msg}")
