"""ctypes binding of oracle/_ref/libcrf_ref.so: the REAL reference sources (unmodified, compiled where they lie in a
checkout of the reference project by oracle/Makefile `ref`) behind the C entry points of oracle/ref_driver.cc.

TEST INFRASTRUCTURE ONLY.  The reference project is not part of this repository: the library is built only when
CRF_REFERENCE names a checkout of it (src/, include/, data/).  Without it the tests use the golden vectors this module
produced (tests/golden/make_ref_golden.py -> tests/golden/ref_*.npz).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "_ref" / "libcrf_ref.so"
REFERENCE = Path(os.environ["CRF_REFERENCE"]) if os.environ.get("CRF_REFERENCE") else None
REF_DATA = REFERENCE / "data" if REFERENCE else None   # the shipped forests (trees_*), LFW fixtures (imgs/) and config files


def can_build() -> bool:
    return REFERENCE is not None and (REFERENCE / "src" / "FaceForest.cpp").exists()


def available() -> bool:
    return LIB_PATH.exists() or can_build()


def build(force: bool = False) -> None:
    if not can_build():
        return
    srcs = [_HERE / "ref_driver.cc", _HERE / "crf_oracle.cc", _HERE / "shim" / "cvshim.cc", _HERE / "shim" / "boost" / "crf_boost_shim.hpp",
            _HERE / "shim" / "opencv2" / "core" / "core.hpp"]
    if not force and LIB_PATH.exists() and all(LIB_PATH.stat().st_mtime >= s.stat().st_mtime for s in srcs):
        return
    subprocess.run(["make", "-C", str(_HERE), "-B", "ref"], check=True, capture_output=True)


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(str(LIB_PATH))
    u8p, i32p, f32p = C.POINTER(C.c_uint8), C.POINTER(C.c_int32), C.POINTER(C.c_float)
    L.ref_last_error.restype = C.c_char_p
    L.ref_create.restype = C.c_void_p
    L.ref_create.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int]
    L.ref_free.argtypes = [C.c_void_p]
    L.ref_set_strides.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.ref_num_trees.argtypes = [C.c_void_p, C.c_int]
    L.ref_analyze_face.argtypes = [C.c_void_p, u8p, C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, f32p, i32p, i32p, i32p, C.c_int]
    L.ref_sample_from_planes.restype = C.c_void_p
    L.ref_sample_from_planes.argtypes = [u8p, C.c_int, C.c_int, C.c_int]
    L.ref_sample_create.restype = C.c_void_p
    L.ref_sample_create.argtypes = [u8p, C.c_int, C.c_int, i32p, C.c_int]
    L.ref_sample_channels.argtypes = [C.c_void_p]
    L.ref_sample_plane.argtypes = [C.c_void_p, C.c_int, f32p]
    L.ref_sample_free.argtypes = [C.c_void_p]
    L.ref_eval_test.argtypes = [C.c_void_p, C.c_int, i32p, i32p, C.c_int, C.c_int, C.c_int]
    L.ref_eval_hp.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, i32p, f32p, f32p]
    L.ref_area_under_curve.restype = C.c_float
    L.ref_area_under_curve.argtypes = [C.c_float, C.c_float, C.c_double, C.c_double]
    L.ref_eval_ffd.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, i32p, i32p, C.c_int, i32p, i32p, f32p, C.c_int, i32p]
    L.ref_meanshift.argtypes = [f32p, C.c_int, i32p, f32p, i32p]
    L.crf_ref_set_gabor_mode.argtypes = [C.c_int]
    L.crf_ref_set_threads.argtypes = [C.c_int]
    _lib = L
    return L


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


class RefError(RuntimeError):
    pass


def set_gabor_mode(mode: int) -> None:
    """0 = canonical separable arithmetic for the bank's >= 9x9 kernels (default), 1 = double-accumulated direct sum."""
    lib().crf_ref_set_gabor_mode(mode)


def set_threads(n: int) -> None:
    """boost::thread::hardware_concurrency() as the reference sees it (0 = the host's)."""
    lib().crf_ref_set_threads(n)


class Sample:
    """The reference's ImageSample (include/ImageSample.hpp:146-199)."""

    def __init__(self, gray: np.ndarray | None = None, features=(0, 1, 2), planes: np.ndarray | None = None):
        L = lib()
        if planes is not None:
            planes = np.ascontiguousarray(planes, np.uint8)
            self.C, self.H, self.W = planes.shape
            self.h = L.ref_sample_from_planes(_p(planes, C.c_uint8), self.C, self.H, self.W)
        else:
            gray = np.ascontiguousarray(gray, np.uint8)
            self.H, self.W = gray.shape
            f = np.ascontiguousarray(features, np.int32)
            self.h = L.ref_sample_create(_p(gray, C.c_uint8), self.H, self.W, _p(f, C.c_int32), len(f))
            self.C = L.ref_sample_channels(self.h)

    def integrals(self) -> np.ndarray:
        out = np.zeros((self.C, self.H + 1, self.W + 1), np.float32)
        for c in range(self.C):
            lib().ref_sample_plane(self.h, c, _p(out[c], C.c_float))
        return out

    def eval_test(self, channel, r1, r2, px, py, patch=31) -> int:
        a = np.ascontiguousarray(r1, np.int32); b = np.ascontiguousarray(r2, np.int32)
        return int(lib().ref_eval_test(self.h, channel, _p(a, C.c_int32), _p(b, C.c_int32), px, py, patch))

    def close(self):
        if self.h:
            lib().ref_sample_free(self.h)
            self.h = None


class FaceForest:
    """The reference's FaceForest (include/FaceForest.hpp:81-157), loaded from the shipped text archives."""

    def __init__(self, hp_dir: str, ffd_dir: str, hp_ntrees: int = 15, ffd_ntrees: int = 20):
        L = lib()
        self.h = L.ref_create(str(hp_dir).encode(), hp_ntrees, str(ffd_dir).encode(), ffd_ntrees)
        if not self.h:
            raise RefError(L.ref_last_error().decode())
        self.hp_trees = L.ref_num_trees(self.h, -1)

    def close(self):
        if self.h:
            lib().ref_free(self.h)
            self.h = None

    def set_strides(self, hp_stride: int, ffd_stride: int) -> None:
        lib().ref_set_strides(self.h, hp_stride, ffd_stride)

    def analyze_face(self, bgr: np.ndarray, box):
        """FaceForest::analyzeFace.  Returns dict(headpose f32, ffd int32 [10,2], list_forest, list_tree)."""
        L = lib()
        bgr = np.ascontiguousarray(bgr, np.uint8)
        rows, cols = bgr.shape[:2]
        hp = C.c_float(); ffd = np.zeros((10, 2), np.int32); lf = np.zeros(128, np.int32); lt = np.zeros(128, np.int32)
        n = L.ref_analyze_face(self.h, _p(bgr, C.c_uint8), rows, cols, cols * 3, int(box[0]), int(box[1]), int(box[2]), int(box[3]), C.byref(hp),
                               _p(ffd, C.c_int32), _p(lf, C.c_int32), _p(lt, C.c_int32), 128)
        if n < 0:
            raise RefError(L.ref_last_error().decode())
        return dict(headpose=np.float32(hp.value), ffd=ffd, list_forest=lf[:n].copy(), list_tree=lt[:n].copy())

    def eval_hp(self, sample: Sample, stride: int = 4, want_leaves: bool = True):
        L = lib()
        nx = len(range(0, sample.W - 31, stride)); ny = len(range(0, sample.H - 31, stride))
        ids = np.zeros((nx * ny, self.hp_trees), np.int32)
        hp = C.c_float(); var = C.c_float()
        n = L.ref_eval_hp(self.h, sample.h, sample.W, sample.H, stride, _p(ids, C.c_int32) if want_leaves else None, C.byref(hp), C.byref(var))
        if n < 0:
            raise RefError(L.ref_last_error().decode())
        return ids, np.float32(hp.value), np.float32(var.value)

    def eval_ffd(self, sample: Sample, forest_idx, tree_idx, stride: int = 3, vote_cap: int = 0, want_leaves: bool = True):
        L = lib()
        fi = np.ascontiguousarray(forest_idx, np.int32); ti = np.ascontiguousarray(tree_idx, np.int32)
        nt = len(fi)
        nx = len(range(0, sample.W - 31, stride)); ny = len(range(0, sample.H - 31, stride))
        ids = np.zeros((nx * ny, nt), np.int32); nv = np.zeros(10, np.int32); rnd = np.zeros((10, 2), np.int32)
        votes = np.zeros((10, max(vote_cap, 1), 3), np.float32)
        n = L.ref_eval_ffd(self.h, sample.h, sample.W, sample.H, stride, _p(fi, C.c_int32), _p(ti, C.c_int32), nt, _p(ids, C.c_int32) if want_leaves else None,
                           _p(nv, C.c_int32), _p(votes, C.c_float) if vote_cap else None, vote_cap, _p(rnd, C.c_int32))
        if n < 0:
            raise RefError(L.ref_last_error().decode())
        return dict(leaf_ids=ids, n_votes=nv, votes=votes if vote_cap else None, rounded=rnd)


def area_under_curve(x1, x2, mean, std) -> np.float32:
    return np.float32(lib().ref_area_under_curve(x1, x2, mean, std))


def meanshift(votes_xyw: np.ndarray):
    """MeanShift::shift.  Returns (rounded int32[2], mean f32[2] traced through the class's own statics, iterations)."""
    v = np.ascontiguousarray(votes_xyw, np.float32).reshape(-1, 3)
    rnd = np.zeros(2, np.int32); mean = np.zeros(2, np.float32); it = C.c_int()
    lib().ref_meanshift(_p(v, C.c_float), len(v), _p(rnd, C.c_int32), _p(mean, C.c_float), C.byref(it))
    return rnd, mean, it.value
