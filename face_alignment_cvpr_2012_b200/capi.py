"""ctypes binding of the C ABI declared in include/crf_b200.h (libcrf_b200.so).

This is plumbing only: every compute call below runs CUDA kernels inside the shared library.  There
is no CPU fallback — if the library is missing or no CUDA device is present the calls raise.
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "_lib" / "libcrf_b200.so"
CSRC = _PKG / "csrc"

NUM_PARTS = 10
NUM_POSE_FORESTS = 5
NUM_STAGES = 8
STAGE_NAMES = ["resize", "plain_channels", "gabor", "hp_traverse", "hp_reduce", "ffd_traverse", "votes", "meanshift"]
MAX_SCALED_H = 521
FACE_NOT_ANALYSED = 8   # crf_face_t::flags of a detected box the analysis path cannot take (crf_analyze_images)


class CrfError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"crf_b200 error {code}: {msg}")
        self.code = code


class Rect(C.Structure):
    _fields_ = [("x", C.c_int), ("y", C.c_int), ("width", C.c_int), ("height", C.c_int)]


class Image(C.Structure):
    """crf_image_t: one BGR frame of any size (rows x cols pixels, step bytes per row)."""
    _fields_ = [("bgr", C.c_void_p), ("rows", C.c_int), ("cols", C.c_int), ("step", C.c_size_t)]


def images(frames) -> "C.Array":
    """crf_image_t descriptors of C-contiguous [rows, cols, 3] u8 frames (at least one element, so an empty list still passes a pointer)."""
    return (Image * max(len(frames), 1))(*[Image(f.ctypes.data, f.shape[0], f.shape[1], f.strides[0]) for f in frames])


class Options(C.Structure):
    _fields_ = [("hp_stride", C.c_int), ("hp_min_foreground", C.c_float), ("ffd_stride", C.c_int), ("ffd_min_samples", C.c_int),
                ("ffd_min_foreground", C.c_float), ("ffd_min_pf", C.c_float), ("ffd_max_variance", C.c_float),
                ("ms_kernel_size", C.c_int), ("ms_max_iterations", C.c_int), ("ms_stopping_criteria", C.c_float),
                ("max_chunk", C.c_int), ("max_scaled_h", C.c_int), ("ms_mode", C.c_int)]


class ModelInfo(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("hp_trees", "hp_nodes", "hp_leaves", "hp_max_depth", "mp_forests", "mp_trees", "mp_nodes",
                                       "mp_leaves", "mp_max_depth", "patch_size", "face_size", "num_channels", "hp_ntrees_cfg", "mp_ntrees_cfg")]


class Counters(C.Structure):
    _fields_ = [(n, C.c_ulonglong) for n in ("faces", "hp_node_tests", "ffd_node_tests", "hp_traversals", "ffd_traversals", "votes",
                                             "vote_passes", "kernel_launches", "h2d_bytes", "d2h_bytes")]


FACE_DTYPE = np.dtype([
    ("headpose", "<f4"), ("variance", "<f4"), ("tree_counts", "<i4", (5,)), ("dominant", "<i4"),
    ("scaled_w", "<i4"), ("scaled_h", "<i4"), ("scale", "<f4"),
    ("ffd_f", "<f4", (10, 2)), ("ffd_scaled", "<i4", (10, 2)), ("ffd", "<i4", (10, 2)),
    ("ms_iters", "<i4", (10,)), ("n_votes", "<i4", (10,)), ("flags", "<i4"),
])

# every symbol include/crf_b200.h declares
EXPORTS = [
    "crf_last_error", "crf_version", "crf_options_default", "crf_model_load", "crf_model_save_packed", "crf_model_load_packed",
    "crf_model_info", "crf_model_tree_dump", "crf_model_check_packing", "crf_model_free", "crf_device_count", "crf_ctx_create", "crf_ctx_destroy",
    "crf_ctx_set_profiling", "crf_ctx_stage_ms", "crf_ctx_counters", "crf_ctx_reset_counters", "crf_ctx_stream", "crf_host_alloc",
    "crf_host_free", "crf_analyze_faces", "crf_analyze_batch", "crf_analyze_crops", "crf_headpose_crops", "crf_analyze_crops_device",
    "crf_stage_gray_resize", "crf_stage_channels", "crf_stage_minmax", "crf_stage_norm", "crf_stage_canny", "crf_stage_eval_forest", "crf_stage_headpose",
    "crf_stage_compose", "crf_stage_compose_batch", "crf_stage_votes_meanshift", "crf_stage_meanshift",
    "crf_model_load_forest", "crf_model_set_features", "crf_model_get_features", "crf_model_leaf_dump", "crf_stage_feature_channels",
    "crf_stage_eval_patches", "crf_stage_eval_tests", "crf_stage_eval_tests_sum", "crf_model_load_tree", "crf_stage_meanshift_opt", "crf_stage_area_under_curve",
    "crf_cascade_load", "crf_cascade_free", "crf_cascade_info", "crf_detect_faces", "crf_detect_faces_batch", "crf_analyze_images",
    "crf_multi_create", "crf_multi_destroy", "crf_multi_device_count", "crf_multi_ctx", "crf_multi_analyze_batch", "crf_multi_analyze_crops",
    "crf_analyze_batch_mixed", "crf_detect_faces_batch_mixed", "crf_analyze_images_mixed", "crf_multi_analyze_batch_mixed",
]

_lib = None


def build(force: bool = False) -> Path:
    """Compile libcrf_b200.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    srcs = [CSRC / n for n in ("engine.cu", "kernels.cuh", "haar.cuh", "device_forest.h", "model.h", "model.cc", "pack.cc", "Makefile")] + \
           [_PKG.parent / "include" / "crf_b200.h"]
    if not force and LIB_PATH.exists() and all(LIB_PATH.stat().st_mtime >= s.stat().st_mtime for s in srcs):
        return LIB_PATH
    r = subprocess.run(["make", "-C", str(CSRC), "-B"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("building libcrf_b200.so failed:\n" + r.stdout + r.stderr)
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (there is no CPU fallback)")
    L = C.CDLL(str(LIB_PATH))
    vp, u8p, i32p, f32p = C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_int32), C.POINTER(C.c_float)
    L.crf_last_error.restype = C.c_char_p
    L.crf_version.restype = C.c_char_p
    L.crf_options_default.argtypes = [C.POINTER(Options)]
    L.crf_model_load.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.POINTER(vp)]
    L.crf_model_save_packed.argtypes = [vp, C.c_char_p]
    L.crf_model_load_packed.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.crf_model_info.argtypes = [vp, C.POINTER(ModelInfo)]
    L.crf_model_tree_dump.argtypes = [vp, C.c_int, C.c_int, i32p, C.c_int]
    L.crf_model_check_packing.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.crf_model_free.argtypes = [vp]
    L.crf_model_free.restype = None
    L.crf_ctx_create.argtypes = [vp, C.c_int, C.POINTER(Options), C.POINTER(vp)]
    L.crf_ctx_destroy.argtypes = [vp]
    L.crf_ctx_destroy.restype = None
    L.crf_ctx_set_profiling.argtypes = [vp, C.c_int]
    L.crf_ctx_stage_ms.argtypes = [vp, f32p, i32p]
    L.crf_ctx_counters.argtypes = [vp, C.POINTER(Counters)]
    L.crf_ctx_reset_counters.argtypes = [vp]
    L.crf_ctx_stream.argtypes = [vp]
    L.crf_ctx_stream.restype = vp
    L.crf_host_alloc.argtypes = [C.POINTER(vp), C.c_size_t]
    L.crf_host_free.argtypes = [vp]
    L.crf_host_free.restype = None
    L.crf_analyze_faces.argtypes = [vp, vp, C.c_int, C.c_int, C.c_size_t, C.POINTER(Rect), C.c_int, vp]
    L.crf_analyze_batch.argtypes = [vp, C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_size_t, C.POINTER(Rect), i32p, C.c_int, vp]
    L.crf_analyze_batch_mixed.argtypes = [vp, C.POINTER(Image), C.c_int, C.POINTER(Rect), i32p, C.c_int, vp]
    L.crf_analyze_crops.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, vp]
    L.crf_headpose_crops.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, vp]
    L.crf_analyze_crops_device.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, vp, C.c_int]
    L.crf_stage_gray_resize.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_size_t, Rect, u8p, i32p, i32p]
    L.crf_stage_channels.argtypes = [vp, u8p, C.c_int, C.c_int, u8p, C.POINTER(C.c_uint32)]
    L.crf_stage_minmax.argtypes = [vp, u8p, C.c_int, C.c_int, u8p, C.POINTER(C.c_uint32)]
    L.crf_stage_norm.argtypes = [vp, u8p, C.c_int, C.c_int, u8p, C.POINTER(C.c_uint32)]
    L.crf_stage_canny.argtypes = [vp, u8p, C.c_int, C.c_int, u8p, C.POINTER(C.c_uint32)]
    L.crf_stage_eval_forest.argtypes = [vp, C.c_int, i32p, i32p, C.c_int, u8p, C.c_int, C.c_int, C.c_int, C.c_int, i32p]
    L.crf_stage_headpose.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_int, C.c_int, f32p, f32p, i32p, i32p, i32p, i32p, i32p, i32p]
    L.crf_stage_compose.argtypes = [vp, C.c_float, C.c_float, i32p, i32p, i32p, i32p, i32p, i32p]
    L.crf_stage_compose_batch.argtypes = [vp, f32p, f32p, C.c_int, i32p, i32p, i32p, i32p, i32p, i32p, C.c_int]
    L.crf_stage_votes_meanshift.argtypes = [vp, i32p, i32p, C.c_int, u8p, C.c_int, C.c_int, C.c_int, C.c_int, i32p, f32p, C.c_int, f32p, i32p, i32p]
    L.crf_stage_meanshift.argtypes = [vp, f32p, C.c_int, f32p, i32p, i32p]
    L.crf_model_load_forest.argtypes = [C.c_char_p, C.c_int, C.c_int, C.POINTER(vp)]
    L.crf_model_set_features.argtypes = [vp, i32p, C.c_int]
    L.crf_model_get_features.argtypes = [vp, i32p, C.c_int]
    L.crf_model_leaf_dump.argtypes = [vp, C.c_int, C.c_int, f32p, C.c_int]
    L.crf_stage_feature_channels.argtypes = [vp, u8p, C.c_int, C.c_int, i32p, C.c_int, u8p, C.POINTER(C.c_uint32)]
    L.crf_stage_eval_patches.argtypes = [vp, C.c_int, i32p, i32p, C.c_int, u8p, C.c_int, C.c_int, C.c_int, i32p, C.c_int, i32p]
    L.crf_stage_eval_tests.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_int, i32p, C.c_int, i32p]
    L.crf_stage_eval_tests_sum.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_int, i32p, C.c_int, i32p]
    L.crf_model_load_tree.argtypes = [C.c_char_p, C.c_int, C.POINTER(vp)]
    L.crf_stage_meanshift_opt.argtypes = [vp, f32p, C.c_int, C.c_int, C.c_int, C.c_float, f32p, i32p, i32p]
    L.crf_stage_area_under_curve.argtypes = [vp, C.c_float, C.c_float, C.c_double, C.c_double, f32p]
    L.crf_cascade_load.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.crf_cascade_free.argtypes = [vp]
    L.crf_cascade_free.restype = None
    L.crf_cascade_info.argtypes = [vp, i32p, i32p, i32p, i32p]
    L.crf_detect_faces.argtypes = [vp, vp, u8p, C.c_int, C.c_int, C.c_size_t, C.c_double, C.c_int, C.c_int, C.POINTER(Rect), C.c_int]
    L.crf_detect_faces_batch.argtypes = [vp, vp, C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_double, C.c_int, C.c_int,
                                         C.POINTER(Rect), i32p, C.c_int]
    L.crf_analyze_images.argtypes = [vp, vp, C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_double, C.c_int, C.c_int,
                                     C.POINTER(Rect), i32p, vp, C.c_int]
    L.crf_detect_faces_batch_mixed.argtypes = [vp, vp, C.POINTER(Image), C.c_int, C.c_double, C.c_int, C.c_int, C.POINTER(Rect), i32p, C.c_int]
    L.crf_analyze_images_mixed.argtypes = [vp, vp, C.POINTER(Image), C.c_int, C.c_double, C.c_int, C.c_int, C.POINTER(Rect), i32p, vp, C.c_int]
    L.crf_multi_create.argtypes = [vp, i32p, C.c_int, C.POINTER(Options), C.POINTER(vp)]
    L.crf_multi_destroy.argtypes = [vp]
    L.crf_multi_destroy.restype = None
    L.crf_multi_device_count.argtypes = [vp]
    L.crf_multi_ctx.argtypes = [vp, C.c_int]
    L.crf_multi_ctx.restype = vp
    L.crf_multi_analyze_batch.argtypes = [vp, C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_size_t, C.POINTER(Rect), i32p, C.c_int, vp]
    L.crf_multi_analyze_batch_mixed.argtypes = [vp, C.POINTER(Image), C.c_int, C.POINTER(Rect), i32p, C.c_int, vp]
    L.crf_multi_analyze_crops.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, vp, C.c_int]
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != 0:
        raise CrfError(rc, lib().crf_last_error().decode(errors="replace"))


def ptr(a: np.ndarray, t):
    return a.ctypes.data_as(C.POINTER(t))
