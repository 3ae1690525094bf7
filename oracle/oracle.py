"""ctypes binding of the CPU oracle (oracle/crf_oracle.cc).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package never imports this module.
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_BUILD = _HERE / "_build"


class OrcFace(C.Structure):
    _fields_ = [
        ("headpose", C.c_float), ("variance", C.c_float),
        ("tree_counts", C.c_int * 5), ("dominant", C.c_int),
        ("scaled_w", C.c_int), ("scaled_h", C.c_int), ("scale", C.c_float),
        ("ffd_f", (C.c_float * 2) * 10), ("ffd_scaled", (C.c_int * 2) * 10), ("ffd", (C.c_int * 2) * 10),
        ("ms_iters", C.c_int * 10), ("n_votes", C.c_int * 10), ("flags", C.c_int),
    ]


class OrcOptions(C.Structure):
    _fields_ = [("hp_stride", C.c_int), ("ffd_stride", C.c_int), ("threads", C.c_int),
                ("features_mask", C.c_int), ("headpose_only", C.c_int)]


FACE_DTYPE = np.dtype([
    ("headpose", "<f4"), ("variance", "<f4"), ("tree_counts", "<i4", (5,)), ("dominant", "<i4"),
    ("scaled_w", "<i4"), ("scaled_h", "<i4"), ("scale", "<f4"),
    ("ffd_f", "<f4", (10, 2)), ("ffd_scaled", "<i4", (10, 2)), ("ffd", "<i4", (10, 2)),
    ("ms_iters", "<i4", (10,)), ("n_votes", "<i4", (10,)), ("flags", "<i4"),
])
assert FACE_DTYPE.itemsize == C.sizeof(OrcFace)


def build(force: bool = False) -> None:
    src = _HERE / "crf_oracle.cc"
    outs = [_BUILD / "libcrf_oracle.so", _BUILD / "libcrf_oracle_v3.so"]
    if not force and all(o.exists() and o.stat().st_mtime >= src.stat().st_mtime for o in outs):
        return
    subprocess.run(["make", "-C", str(_HERE), "-B"], check=True, capture_output=True)


def _has_avx2_fma() -> bool:
    try:
        flags = open("/proc/cpuinfo").read()
        return " avx2" in flags and " fma" in flags
    except OSError:
        return False


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    name = "libcrf_oracle_v3.so" if _has_avx2_fma() else "libcrf_oracle.so"
    path = _BUILD / name
    if not path.exists():
        build()
    L = C.CDLL(str(path))
    u8p, i32p, f32p, i64p = (C.POINTER(C.c_uint8), C.POINTER(C.c_int32), C.POINTER(C.c_float), C.POINTER(C.c_longlong))
    L.orc_last_error.restype = C.c_char_p
    L.orc_model_load.restype = C.c_void_p
    L.orc_model_load.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int]
    L.orc_model_free.argtypes = [C.c_void_p]
    L.orc_model_load_packed.restype = C.c_void_p
    L.orc_model_load_packed.argtypes = [C.c_char_p]
    L.orc_leaf_dump.argtypes = [C.c_void_p, C.c_int, C.c_int, f32p, C.c_int]
    L.orc_model_info.argtypes = [C.c_void_p, i32p]
    L.orc_tree_dump.argtypes = [C.c_void_p, C.c_int, C.c_int, i32p, C.c_int]
    L.orc_bgr2gray.argtypes = [u8p, C.c_int, C.c_int, C.c_size_t, u8p]
    L.orc_scaled_size.argtypes = [C.c_int, C.c_int, C.c_int, i32p, i32p, f32p]
    L.orc_resize.argtypes = [u8p, C.c_int, C.c_int, C.c_size_t, u8p, C.c_int, C.c_int]
    L.orc_num_planes.argtypes = [C.c_int]
    L.orc_channels.argtypes = [u8p, C.c_int, C.c_int, C.c_int, C.c_int, u8p, f32p]
    L.orc_gabor_bank.argtypes = [i32p, f32p, f32p, C.c_int]
    L.orc_gabor_response.argtypes = [u8p, C.c_int, C.c_int, C.c_int, f32p, f32p]
    L.orc_num_patches.argtypes = [C.c_int] * 4
    L.orc_sample_create.restype = C.c_void_p
    L.orc_sample_create.argtypes = [u8p, C.c_int, C.c_int, C.c_int, C.c_int]
    L.orc_sample_from_planes.restype = C.c_void_p
    L.orc_sample_from_planes.argtypes = [u8p, C.c_int, C.c_int, C.c_int]
    L.orc_sample_free.argtypes = [C.c_void_p]
    L.orc_eval_hp.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, i32p, f32p, f32p, i64p]
    L.orc_compose.argtypes = [C.c_void_p, C.c_float, C.c_float, i32p, i32p, i32p, i32p, C.c_int, i32p]
    L.orc_area_under_curve.restype = C.c_float
    L.orc_area_under_curve.argtypes = [C.c_float, C.c_float, C.c_double, C.c_double]
    L.orc_eval_ffd.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, i32p, i32p, C.c_int,
                               i32p, i32p, f32p, C.c_int, f32p, i32p, i32p, i64p]
    L.orc_meanshift.argtypes = [f32p, C.c_int, f32p, i32p, i32p]
    L.orc_analyze_face.argtypes = [C.c_void_p, u8p, C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.POINTER(OrcOptions), C.POINTER(OrcFace), i64p]
    L.orc_analyze_crops_timed.restype = C.c_double
    L.orc_analyze_crops_timed.argtypes = [C.c_void_p, u8p, C.c_int, C.c_int, C.c_int, C.POINTER(OrcOptions),
                                          C.POINTER(OrcFace), C.POINTER(C.c_double)]
    _lib = L
    return L


def _p(a: np.ndarray, t):
    return a.ctypes.data_as(C.POINTER(t))


def _u8(a):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    return a, _p(a, C.c_uint8)


class OracleError(RuntimeError):
    pass


class Model:
    """What FaceForest's constructor loads (src/FaceForest.cpp:15-58)."""

    def __init__(self, hp_dir: str | None = None, ffd_dir: str | None = None, hp_ntrees: int = 15, ffd_ntrees: int = 20, packed: str | None = None):
        L = lib()
        if packed:
            self.h = L.orc_model_load_packed(str(packed).encode())
        else:
            self.h = L.orc_model_load((hp_dir or "").encode(), hp_ntrees, (ffd_dir or "").encode(), ffd_ntrees)
        if not self.h:
            raise OracleError(L.orc_last_error().decode())
        info = np.zeros(11, np.int32)
        L.orc_model_info(self.h, _p(info, C.c_int32))
        self.info = dict(zip(["hp_trees", "hp_nodes", "hp_leaves", "mp_forests", "mp_trees", "mp_nodes", "mp_leaves",
                              "hp_max_depth", "mp_max_depth", "patch_size", "face_size"], info.tolist()))

    def close(self):
        if self.h:
            lib().orc_model_free(self.h)
            self.h = None

    def tree_dump(self, which: int, tree: int) -> np.ndarray:
        L = lib()
        n = L.orc_tree_dump(self.h, which, tree, None, 0)
        out = np.zeros((n, 16), np.int32)
        L.orc_tree_dump(self.h, which, tree, _p(out, C.c_int32), n)
        return out

    def leaf_dump(self, which: int, tree: int) -> np.ndarray:
        L = lib()
        n = L.orc_leaf_dump(self.h, which, tree, None, 0)
        out = np.zeros((n, 44), np.float32)
        L.orc_leaf_dump(self.h, which, tree, _p(out, C.c_float), n)
        return out

    def compose(self, headpose: float, variance: float):
        L = lib()
        counts = np.zeros(5, np.int32); dom = C.c_int(0); flags = C.c_int(0)
        fi = np.zeros(128, np.int32); ti = np.zeros(128, np.int32)
        n = L.orc_compose(self.h, headpose, variance, _p(counts, C.c_int32), C.byref(dom), _p(fi, C.c_int32), _p(ti, C.c_int32), 128, C.byref(flags))
        if n < 0:
            raise OracleError(L.orc_last_error().decode())
        return counts, dom.value, fi[:n].copy(), ti[:n].copy(), flags.value

    def eval_hp(self, sample: "Sample", stride: int = 4, threads: int = 1):
        L = lib()
        n = L.orc_num_patches(sample.W, sample.H, self.info["patch_size"], stride) * self.info["hp_trees"]
        ids = np.zeros(n, np.int32); hp = C.c_float(); var = C.c_float(); vis = C.c_longlong()
        L.orc_eval_hp(self.h, sample.h, sample.H, sample.W, stride, threads, _p(ids, C.c_int32), C.byref(hp), C.byref(var), C.byref(vis))
        return ids.reshape(-1, self.info["hp_trees"]), np.float32(hp.value), np.float32(var.value), vis.value

    def eval_ffd(self, sample: "Sample", forest_idx, tree_idx, stride: int = 3, threads: int = 1, vote_cap: int = 0):
        L = lib()
        fi = np.ascontiguousarray(forest_idx, np.int32); ti = np.ascontiguousarray(tree_idx, np.int32)
        nt = len(fi)
        n = L.orc_num_patches(sample.W, sample.H, self.info["patch_size"], stride) * nt
        ids = np.zeros(n, np.int32); nv = np.zeros(10, np.int32)
        votes = np.zeros((10, max(vote_cap, 1), 3), np.float32)
        mean = np.zeros((10, 2), np.float32); rnd = np.zeros((10, 2), np.int32); it = np.zeros(10, np.int32); vis = C.c_longlong()
        r = L.orc_eval_ffd(self.h, sample.h, sample.H, sample.W, stride, threads, _p(fi, C.c_int32), _p(ti, C.c_int32), nt,
                           _p(ids, C.c_int32), _p(nv, C.c_int32), _p(votes, C.c_float) if vote_cap else None, vote_cap,
                           _p(mean, C.c_float), _p(rnd, C.c_int32), _p(it, C.c_int32), C.byref(vis))
        if r < 0:
            raise OracleError(L.orc_last_error().decode())
        return dict(leaf_ids=ids.reshape(-1, nt), n_votes=nv, votes=votes if vote_cap else None, mean=mean, rounded=rnd,
                    iters=it, visits=vis.value)

    def analyze_face(self, bgr: np.ndarray, box, hp_stride=4, ffd_stride=3, threads=1, headpose_only=False, want_stats=False, features_mask=7):
        L = lib()
        bgr = np.ascontiguousarray(bgr, np.uint8)
        rows, cols = bgr.shape[:2]
        opt = OrcOptions(hp_stride, ffd_stride, threads, features_mask, int(headpose_only))
        out = OrcFace(); stats = np.zeros(4, np.int64)
        r = L.orc_analyze_face(self.h, _p(bgr, C.c_uint8), rows, cols, cols * 3, int(box[0]), int(box[1]), int(box[2]), int(box[3]),
                               C.byref(opt), C.byref(out), _p(stats, C.c_longlong) if want_stats else None)
        if r != 0:
            raise OracleError(L.orc_last_error().decode())
        rec = np.frombuffer(bytes(out), dtype=FACE_DTYPE)[0]
        return (rec, stats) if want_stats else rec

    def analyze_crops_timed(self, crops: np.ndarray, hp_stride=4, ffd_stride=3, threads=1, headpose_only=False):
        """crops: n x rows x cols x 3 u8.  Returns (faces recarray, seconds, per-face ms)."""
        L = lib()
        crops = np.ascontiguousarray(crops, np.uint8)
        n, rows, cols = crops.shape[:3]
        opt = OrcOptions(hp_stride, ffd_stride, threads, 7, int(headpose_only))
        out = np.zeros(n, FACE_DTYPE); ms = np.zeros(n, np.float64)
        sec = L.orc_analyze_crops_timed(self.h, _p(crops, C.c_uint8), n, rows, cols, C.byref(opt),
                                        out.ctypes.data_as(C.POINTER(OrcFace)), _p(ms, C.c_double))
        return out, sec, ms


class Sample:
    """ImageSample (include/ImageSample.hpp:146-199) built from a scaled gray face."""

    def __init__(self, gray: np.ndarray | None = None, features_mask: int = 7, threads: int = 1, planes: np.ndarray | None = None):
        L = lib()
        if planes is not None:
            planes = np.ascontiguousarray(planes, np.uint8)
            self.C, self.H, self.W = planes.shape
            self.h = L.orc_sample_from_planes(_p(planes, C.c_uint8), self.C, self.H, self.W)
        else:
            gray = np.ascontiguousarray(gray, np.uint8)
            self.H, self.W = gray.shape
            self.C = L.orc_num_planes(features_mask)
            self.h = L.orc_sample_create(_p(gray, C.c_uint8), self.H, self.W, features_mask, threads)

    def close(self):
        if self.h:
            lib().orc_sample_free(self.h)
            self.h = None


def bgr2gray(bgr: np.ndarray) -> np.ndarray:
    bgr = np.ascontiguousarray(bgr, np.uint8)
    rows, cols = bgr.shape[:2]
    out = np.zeros((rows, cols), np.uint8)
    lib().orc_bgr2gray(_p(bgr, C.c_uint8), rows, cols, cols * 3, _p(out, C.c_uint8))
    return out


def scaled_size(roi_cols: int, roi_rows: int, face_size: int = 125):
    w = C.c_int(); h = C.c_int(); s = C.c_float()
    lib().orc_scaled_size(roi_cols, roi_rows, face_size, C.byref(w), C.byref(h), C.byref(s))
    return w.value, h.value, np.float32(s.value)


def resize(src: np.ndarray, dh: int, dw: int) -> np.ndarray:
    src = np.ascontiguousarray(src, np.uint8)
    out = np.zeros((dh, dw), np.uint8)
    lib().orc_resize(_p(src, C.c_uint8), src.shape[0], src.shape[1], src.shape[1], _p(out, C.c_uint8), dh, dw)
    return out


def channels(gray: np.ndarray, features_mask: int = 7, threads: int = 1):
    """Returns (planes u8 [C,H,W], integrals f32 [C,H+1,W+1])."""
    gray = np.ascontiguousarray(gray, np.uint8)
    H, W = gray.shape
    Cn = lib().orc_num_planes(features_mask)
    planes = np.zeros((Cn, H, W), np.uint8)
    integ = np.zeros((Cn, H + 1, W + 1), np.float32)
    lib().orc_channels(_p(gray, C.c_uint8), H, W, features_mask, threads, _p(planes, C.c_uint8), _p(integ, C.c_float))
    return planes, integ


def gabor_bank():
    widths = np.zeros(35, np.int32)
    n = lib().orc_gabor_bank(_p(widths, C.c_int32), None, None, 0)
    re = np.zeros(n, np.float32); im = np.zeros(n, np.float32)
    lib().orc_gabor_bank(_p(widths, C.c_int32), _p(re, C.c_float), _p(im, C.c_float), n)
    out, o = [], 0
    for w in widths:
        out.append((re[o:o + w * w].reshape(w, w).copy(), im[o:o + w * w].reshape(w, w).copy()))
        o += w * w
    return out


def gabor_response(gray: np.ndarray, index: int):
    gray = np.ascontiguousarray(gray, np.uint8)
    H, W = gray.shape
    re = np.zeros((H, W), np.float32); im = np.zeros((H, W), np.float32)
    lib().orc_gabor_response(_p(gray, C.c_uint8), H, W, index, _p(re, C.c_float), _p(im, C.c_float))
    return re, im


def meanshift(votes_xyw: np.ndarray):
    v = np.ascontiguousarray(votes_xyw, np.float32).reshape(-1, 3)
    mean = np.zeros(2, np.float32); rnd = np.zeros(2, np.int32); it = C.c_int()
    lib().orc_meanshift(_p(v, C.c_float), len(v), _p(mean, C.c_float), _p(rnd, C.c_int32), C.byref(it))
    return mean, rnd, it.value


def area_under_curve(x1, x2, mean, std) -> np.float32:
    return np.float32(lib().orc_area_under_curve(x1, x2, mean, std))


def hardware_concurrency() -> int:
    return int(lib().orc_hardware_concurrency())
