"""Host-side mirror of the reference's C++ interface for the inference path, on top of the C ABI.

Same names, argument meaning and error behaviour as the reference (citations: /root/reference):
FaceForest / FaceForestOptions / Face (include/FaceForest.hpp:21-159), Forest<S>::load / evaluateMT
(include/Forest.hpp:81-129), ImageSample (include/ImageSample.hpp:146-199), MeanShift::shift
(include/MeanShift.hpp:41-50).  cv::Mat becomes a numpy uint8 array, cv::Rect a 4-tuple (x, y, w, h),
cv::Point a length-2 int array.  Everything computes on the GPU through libcrf_b200.so.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from pathlib import Path

import numpy as np

from . import capi
from .capi import FACE_DTYPE, CrfError, Options, Rect


@dataclass
class ForestParam:
    """include/Constants.hpp:24-60 — the fields the inference path reads."""
    tree_path: str = ""
    image_path: str = ""
    ntrees: int = 0
    max_depth: int = 0
    face_size: int = 125
    patch_size_ratio: float = 0.25
    features: list = field(default_factory=lambda: [0, 1, 2])

    def getPatchSize(self) -> int:
        return int(round(self.face_size * self.patch_size_ratio))


def loadConfigFile(path: str) -> ForestParam:
    """src/face_utils.cpp:50-140: label line then value line, 11 entries."""
    p = ForestParam()
    try:
        lines = Path(path).read_text().split("\n")
    except OSError:
        raise FileNotFoundError(f"file not found {path}")
    vals = [lines[i].strip() for i in range(1, len(lines), 2)]
    # order of data/config_*.txt: image index, tree path, ntrees, ntests, max depth, min patches, images, patches, face size, ratio, features
    p.image_path = vals[0]; p.tree_path = vals[1]; p.ntrees = int(vals[2]); p.max_depth = int(vals[4])
    p.face_size = int(vals[8]); p.patch_size_ratio = float(vals[9]); p.features = [int(v) for v in vals[10].split()]
    return p


@dataclass
class HeadPoseEstimatorOption:  # include/FaceForest.hpp:33-43
    num_head_pose_labels: int = 5
    step_size: int = 4
    min_foreground_probability: float = 0.5


@dataclass
class MultiPartEstimatorOption:  # include/FaceForest.hpp:45-58
    num_parts: int = 10
    step_size: int = 3
    min_samples: int = 2
    min_forground: float = 0.5
    min_pf: float = 0.25
    max_variance: float = 25.0


@dataclass
class MeanShiftOption:  # include/MeanShift.hpp:16-25
    kernel_size: int = 10
    max_iterations: int = 7
    stopping_criteria: float = 0.05


@dataclass
class FaceDetectionOption:  # include/FaceForest.hpp:21-31
    min_feature_size: int = 30
    min_neighbors: int = 1
    search_scale_factor: float = 1.3
    path_face_cascade: str = ""


def intersect(r1, r2):
    """src/face_utils.cpp:325-347."""
    x = r2[0] if r1[0] < r2[0] else r1[0]
    y = r2[1] if r1[1] < r2[1] else r1[1]
    w = (r1[0] + r1[2] if r1[0] + r1[2] < r2[0] + r2[2] else r2[0] + r2[2]) - x
    h = (r1[1] + r1[3] if r1[1] + r1[3] < r2[1] + r2[3] else r2[1] + r2[3]) - y
    return (0, 0, 0, 0) if w <= 0 or h <= 0 else (x, y, w, h)


def enlarge_detections(boxes, rows: int, cols: int) -> list:
    """The box post-processing of FaceForest::detectFace (src/FaceForest.cpp:147-157): Haar boxes are too tight, so each
    grows by 5 % of its width on both sides and by 2 x 15 % of its width downwards, clipped to the image."""
    out = []
    for (x, y, w, h) in boxes:
        offset_x = int(w * 0.05)
        offset_y = int(w * 0.15)
        out.append(intersect((int(x) - offset_x, int(y), int(w) + offset_x * 2, int(h) + offset_y * 2), (0, 0, cols, rows)))
    return out


@dataclass
class FaceForestOptions:  # include/FaceForest.hpp:60-68
    hp_forest_param: ForestParam = field(default_factory=ForestParam)
    mp_forest_param: ForestParam = field(default_factory=ForestParam)
    fd_option: FaceDetectionOption = field(default_factory=FaceDetectionOption)
    hp_option: HeadPoseEstimatorOption = field(default_factory=HeadPoseEstimatorOption)
    mp_option: MultiPartEstimatorOption = field(default_factory=MultiPartEstimatorOption)
    mp_forest_paths: list = field(default_factory=list)
    # extensions (not in the reference's struct)
    mean_shift_option: MeanShiftOption = field(default_factory=MeanShiftOption)   # default-constructed inside estimateFacialFeatures there
    packed_model: str = ""   # "next" row f1: pre-packed binary image instead of the two tree directories
    device: int = 0
    max_chunk: int = 0
    ms_mode: str = "default"   # crf_b200.h: MeanShift evaluation mode ("default" | "exact" | "fast")


@dataclass
class Face:  # include/FaceForest.hpp:70-75
    headpose: float = 0.0
    bbox: tuple = (0, 0, 0, 0)
    ffd_cordinates: np.ndarray = field(default_factory=lambda: np.zeros((10, 2), np.int32))
    record: np.void | None = None  # the full crf_face_t (pre-rounding means, composition, vote counts)


class Model:
    """What FaceForest's constructor loads (src/FaceForest.cpp:15-58): the head-pose forest + the jungle."""

    def __init__(self, hp_dir: str | None = None, ffd_dir: str | None = None, hp_ntrees: int = 15, ffd_ntrees: int = 20, packed: str | None = None,
                 forest_dir: str | None = None, kind: str = "hp", ntrees: int | None = None, features=None):
        L = capi.lib()
        h = C.c_void_p()
        if packed:
            capi.check(L.crf_model_load_packed(str(packed).encode(), C.byref(h)))
        elif forest_dir is not None:   # Forest<S>::load on its own: one forest, no composition
            capi.check(L.crf_model_load_forest(str(forest_dir).encode(), ntrees if ntrees is not None else (hp_ntrees if kind == "hp" else ffd_ntrees),
                                               0 if kind == "hp" else 1, C.byref(h)))
        else:
            capi.check(L.crf_model_load(str(hp_dir).encode(), hp_ntrees, str(ffd_dir).encode(), ffd_ntrees, C.byref(h)))
        self.h = h
        if features is not None:
            self.set_features(features)
        self._refresh()

    def _refresh(self) -> None:
        info = capi.ModelInfo()
        capi.check(capi.lib().crf_model_info(self.h, C.byref(info)))
        self.info = {n: getattr(info, n) for n, _ in info._fields_}

    def set_features(self, features) -> None:
        """ForestParam::features of the run-time configuration (any subset of 0..5)."""
        f = np.ascontiguousarray(features, np.int32)
        capi.check(capi.lib().crf_model_set_features(self.h, capi.ptr(f, C.c_int32), len(f)))
        self._refresh()

    @property
    def features(self) -> list:
        f = np.zeros(8, np.int32)
        n = capi.lib().crf_model_get_features(self.h, capi.ptr(f, C.c_int32), 8)
        return f[:n].tolist()

    def leaf_dump(self, which: int, tree: int) -> np.ndarray:
        L = capi.lib()
        n = L.crf_model_leaf_dump(self.h, which, tree, None, 0)
        if n < 0:
            capi.check(n)
        out = np.zeros((n, 44), np.float32)
        L.crf_model_leaf_dump(self.h, which, tree, capi.ptr(out, C.c_float), n)
        return out

    def save_packed(self, path: str) -> None:
        capi.check(capi.lib().crf_model_save_packed(self.h, str(path).encode()))

    def tree_dump(self, which: int, tree: int) -> np.ndarray:
        L = capi.lib()
        n = L.crf_model_tree_dump(self.h, which, tree, None, 0)
        if n < 0:
            capi.check(n)
        out = np.zeros((n, 16), np.int32)
        L.crf_model_tree_dump(self.h, which, tree, capi.ptr(out, C.c_int32), n)
        return out

    def close(self) -> None:
        if getattr(self, "h", None):
            capi.lib().crf_model_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


MS_MODES = {None: 0, "default": 0, "exact": 1, "fast": 2}   # crf_b200.h: CRF_MS_DEFAULT / CRF_MS_EXACT / CRF_MS_FAST


def _options(o: FaceForestOptions | None, hp_stride=None, ffd_stride=None, max_chunk=None, ms_mode=None) -> Options:
    opt = Options()
    capi.lib().crf_options_default(C.byref(opt))
    if o is not None:
        opt.hp_stride = o.hp_option.step_size
        opt.hp_min_foreground = o.hp_option.min_foreground_probability
        opt.ffd_stride = o.mp_option.step_size
        opt.ffd_min_samples = o.mp_option.min_samples
        opt.ffd_min_foreground = o.mp_option.min_forground
        opt.ffd_min_pf = o.mp_option.min_pf
        opt.ffd_max_variance = o.mp_option.max_variance
        opt.ms_kernel_size = o.mean_shift_option.kernel_size
        opt.ms_max_iterations = o.mean_shift_option.max_iterations
        opt.ms_stopping_criteria = o.mean_shift_option.stopping_criteria
        opt.max_chunk = o.max_chunk
        opt.ms_mode = MS_MODES[o.ms_mode]
    if hp_stride is not None:
        opt.hp_stride = hp_stride
    if ffd_stride is not None:
        opt.ffd_stride = ffd_stride
    if max_chunk is not None:
        opt.max_chunk = max_chunk
    if ms_mode is not None:
        opt.ms_mode = MS_MODES[ms_mode]
    return opt


def _frame_list(frames) -> list:
    """C-contiguous u8 copies (where needed) of the BGR frames of a list or an [n, rows, cols, 3] array.  An array's frames stay back to
    back in memory, so that they go up in one copy."""
    if isinstance(frames, np.ndarray):
        frames = np.ascontiguousarray(frames, np.uint8)
    return [np.ascontiguousarray(f, np.uint8) for f in frames]


class Context:
    """One GPU's packed forests + work buffers (crf_ctx)."""

    def __init__(self, model: Model, device: int = 0, options: Options | None = None):
        self.model = model
        h = C.c_void_p()
        # model may be None: a context without forests (feature channels, evalTest, MeanShift)
        capi.check(capi.lib().crf_ctx_create(model.h if model is not None else None, device, C.byref(options) if options is not None else None, C.byref(h)))
        self.h = h
        self.device = device

    def close(self) -> None:
        if getattr(self, "h", None):
            capi.lib().crf_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- profiling / counters
    def set_profiling(self, stage_events: bool = False, count_work: bool = False) -> None:
        capi.check(capi.lib().crf_ctx_set_profiling(self.h, (1 if stage_events else 0) | (2 if count_work else 0)))

    def stage_ms(self):
        ms = np.zeros(capi.NUM_STAGES, np.float32); ln = np.zeros(capi.NUM_STAGES, np.int32)
        capi.check(capi.lib().crf_ctx_stage_ms(self.h, capi.ptr(ms, C.c_float), capi.ptr(ln, C.c_int32)))
        return dict(zip(capi.STAGE_NAMES, ms.tolist())), dict(zip(capi.STAGE_NAMES, ln.tolist()))

    def counters(self) -> dict:
        c = capi.Counters()
        capi.check(capi.lib().crf_ctx_counters(self.h, C.byref(c)))
        return {n: int(getattr(c, n)) for n, _ in c._fields_}

    def reset_counters(self) -> None:
        capi.check(capi.lib().crf_ctx_reset_counters(self.h))

    @property
    def stream(self) -> int:
        return int(capi.lib().crf_ctx_stream(self.h) or 0)

    # ---- whole path
    def analyze_crops(self, crops: np.ndarray, headpose_only: bool = False) -> np.ndarray:
        crops = np.ascontiguousarray(crops, np.uint8)
        n, rows, cols = crops.shape[:3]
        out = np.zeros(n, FACE_DTYPE)
        fn = capi.lib().crf_headpose_crops if headpose_only else capi.lib().crf_analyze_crops
        capi.check(fn(self.h, crops.ctypes.data, n, rows, cols, out.ctypes.data))
        return out

    def analyze_crops_ptr(self, host_ptr: int, n: int, rows: int, cols: int, out: np.ndarray, headpose_only: bool = False) -> None:
        fn = capi.lib().crf_headpose_crops if headpose_only else capi.lib().crf_analyze_crops
        capi.check(fn(self.h, host_ptr, n, rows, cols, out.ctypes.data))

    def analyze_crops_device(self, d_bgr: int, n: int, rows: int, cols: int, d_out: int, headpose_only: bool = False) -> None:
        capi.check(capi.lib().crf_analyze_crops_device(self.h, d_bgr, n, rows, cols, d_out, int(headpose_only)))

    def analyze_faces(self, bgr: np.ndarray, boxes) -> np.ndarray:
        bgr = np.ascontiguousarray(bgr, np.uint8)
        rows, cols = bgr.shape[:2]
        n = len(boxes)
        rects = (Rect * max(n, 1))(*[Rect(int(b[0]), int(b[1]), int(b[2]), int(b[3])) for b in boxes])
        out = np.zeros(n, FACE_DTYPE)
        capi.check(capi.lib().crf_analyze_faces(self.h, bgr.ctypes.data, rows, cols, cols * 3, rects, n, out.ctypes.data))
        return out

    def analyze_batch(self, frames, boxes, image_of_box) -> np.ndarray:
        """frames: [n_images, rows, cols, 3] u8, or a list of BGR frames of any sizes; box i lies in frame image_of_box[i]."""
        frames = _frame_list(frames)
        n = len(boxes)
        rects = (Rect * max(n, 1))(*[Rect(int(b[0]), int(b[1]), int(b[2]), int(b[3])) for b in boxes])
        iob = np.ascontiguousarray(image_of_box, np.int32)
        out = np.zeros(n, FACE_DTYPE)
        capi.check(capi.lib().crf_analyze_batch_mixed(self.h, capi.images(frames), len(frames), rects, capi.ptr(iob, C.c_int32), n, out.ctypes.data))
        return out

    # ---- stages (parity tests)
    def stage_gray_resize(self, bgr: np.ndarray, box) -> np.ndarray:
        bgr = np.ascontiguousarray(bgr, np.uint8)
        rows, cols = bgr.shape[:2]
        buf = np.zeros(capi.MAX_SCALED_H * 125, np.uint8)
        W = C.c_int(); H = C.c_int()
        capi.check(capi.lib().crf_stage_gray_resize(self.h, capi.ptr(bgr, C.c_uint8), rows, cols, cols * 3, Rect(*[int(v) for v in box]),
                                                    capi.ptr(buf, C.c_uint8), C.byref(W), C.byref(H)))
        return buf[: W.value * H.value].reshape(H.value, W.value).copy()

    def stage_channels(self, scaled: np.ndarray, minmax: bool = False, norm: bool = False, canny: bool = False):
        """features {0,1,2} (38 planes), or FC_MIN_MAX (2 planes), or FC_NORM (1 plane), or FC_CANNY (1 plane)."""
        scaled = np.ascontiguousarray(scaled, np.uint8)
        H, W = scaled.shape
        n = 1 if (norm or canny) else 2 if minmax else 38
        planes = np.zeros((n, H, W), np.uint8); integ = np.zeros((n, H + 1, W + 1), np.uint32)
        L = capi.lib()
        fn = L.crf_stage_canny if canny else L.crf_stage_norm if norm else L.crf_stage_minmax if minmax else L.crf_stage_channels
        capi.check(fn(self.h, capi.ptr(scaled, C.c_uint8), W, H, capi.ptr(planes, C.c_uint8), capi.ptr(integ, C.c_uint32)))
        return planes, integ

    def stage_feature_channels(self, scaled: np.ndarray, features):
        """ImageSample::extractFeatureChannels for an explicit feature list: (planes u8 [C,H,W], integrals u32 [C,H+1,W+1])."""
        scaled = np.ascontiguousarray(scaled, np.uint8)
        H, W = scaled.shape
        f = np.ascontiguousarray(features, np.int32)
        n = sum({0: 1, 1: 35, 2: 2, 3: 2, 4: 1, 5: 1}.get(int(v), 0) for v in set(f.tolist()))
        planes = np.zeros((max(n, 1), H, W), np.uint8); integ = np.zeros((max(n, 1), H + 1, W + 1), np.uint32)
        rc = capi.lib().crf_stage_feature_channels(self.h, capi.ptr(scaled, C.c_uint8), W, H, capi.ptr(f, C.c_int32), len(f), capi.ptr(planes, C.c_uint8),
                                                   capi.ptr(integ, C.c_uint32))
        if rc < 0:
            capi.check(rc)
        assert rc == n
        return planes, integ

    def stage_eval_patches(self, planes: np.ndarray, patch_xy, forest_idx=None, tree_idx=None) -> np.ndarray:
        """Forest<S>::evaluateMT for explicit patch origins: leaf ids [patch][tree]."""
        planes = np.ascontiguousarray(planes, np.uint8)
        Cn, H, W = planes.shape
        xy = np.ascontiguousarray(patch_xy, np.int32).reshape(-1, 2)
        if forest_idx is None:
            ids = np.zeros((len(xy), self.model.info["hp_trees"]), np.int32)
            capi.check(capi.lib().crf_stage_eval_patches(self.h, -1, None, None, 0, capi.ptr(planes, C.c_uint8), Cn, W, H, capi.ptr(xy, C.c_int32), len(xy),
                                                         capi.ptr(ids, C.c_int32)))
            return ids
        fi = np.ascontiguousarray(forest_idx, np.int32); ti = np.ascontiguousarray(tree_idx, np.int32)
        ids = np.zeros((len(xy), len(fi)), np.int32)
        capi.check(capi.lib().crf_stage_eval_patches(self.h, 0, capi.ptr(fi, C.c_int32), capi.ptr(ti, C.c_int32), len(fi), capi.ptr(planes, C.c_uint8), Cn, W, H,
                                                     capi.ptr(xy, C.c_int32), len(xy), capi.ptr(ids, C.c_int32)))
        return ids

    def stage_eval_tests(self, planes: np.ndarray, tests, use_integral: bool = True) -> np.ndarray:
        """ImageSample::evalTest for n tests {channel, r1(x,y,w,h), r2(x,y,w,h), patch_x, patch_y}; use_integral selects the branch of
        src/ImageSample.cpp:40-63 (integral corners, or cv::sum over the 8-bit rectangles)."""
        planes = np.ascontiguousarray(planes, np.uint8)
        Cn, H, W = planes.shape
        t = np.ascontiguousarray(tests, np.int32).reshape(-1, 11)
        out = np.zeros(len(t), np.int32)
        fn = capi.lib().crf_stage_eval_tests if use_integral else capi.lib().crf_stage_eval_tests_sum
        capi.check(fn(self.h, capi.ptr(planes, C.c_uint8), Cn, W, H, capi.ptr(t, C.c_int32), len(t), capi.ptr(out, C.c_int32)))
        return out

    def stage_eval_forest(self, planes: np.ndarray, stride: int, forest_idx=None, tree_idx=None) -> np.ndarray:
        planes = np.ascontiguousarray(planes, np.uint8)
        Cn, H, W = planes.shape
        ps = self.model.info["patch_size"]
        npatch = max(0, -(-(W - ps) // stride)) * max(0, -(-(H - ps) // stride))
        if forest_idx is None:
            nt = self.model.info["hp_trees"]
            ids = np.zeros((npatch, nt), np.int32)
            capi.check(capi.lib().crf_stage_eval_forest(self.h, -1, None, None, 0, capi.ptr(planes, C.c_uint8), Cn, W, H, stride, capi.ptr(ids, C.c_int32)))
            return ids
        fi = np.ascontiguousarray(forest_idx, np.int32); ti = np.ascontiguousarray(tree_idx, np.int32)
        ids = np.zeros((npatch, len(fi)), np.int32)
        capi.check(capi.lib().crf_stage_eval_forest(self.h, 0, capi.ptr(fi, C.c_int32), capi.ptr(ti, C.c_int32), len(fi), capi.ptr(planes, C.c_uint8),
                                                    Cn, W, H, stride, capi.ptr(ids, C.c_int32)))
        return ids

    def _compose_out(self):
        return (np.zeros(5, np.int32), C.c_int(), np.zeros(128, np.int32), np.zeros(128, np.int32), C.c_int(), C.c_int())

    def stage_headpose(self, planes: np.ndarray, stride: int) -> dict:
        planes = np.ascontiguousarray(planes, np.uint8)
        Cn, H, W = planes.shape
        hp = C.c_float(); var = C.c_float()
        counts, dom, fi, ti, nt, flags = self._compose_out()
        capi.check(capi.lib().crf_stage_headpose(self.h, capi.ptr(planes, C.c_uint8), Cn, W, H, stride, C.byref(hp), C.byref(var), capi.ptr(counts, C.c_int32),
                                                 C.byref(dom), capi.ptr(fi, C.c_int32), capi.ptr(ti, C.c_int32), C.byref(nt), C.byref(flags)))
        return dict(headpose=np.float32(hp.value), variance=np.float32(var.value), tree_counts=counts, dominant=dom.value,
                    forest_idx=fi[: nt.value].copy(), tree_idx=ti[: nt.value].copy(), flags=flags.value)

    def stage_compose(self, headpose: float, variance: float) -> dict:
        counts, dom, fi, ti, nt, flags = self._compose_out()
        capi.check(capi.lib().crf_stage_compose(self.h, headpose, variance, capi.ptr(counts, C.c_int32), C.byref(dom), capi.ptr(fi, C.c_int32),
                                                capi.ptr(ti, C.c_int32), C.byref(nt), C.byref(flags)))
        return dict(tree_counts=counts, dominant=dom.value, forest_idx=fi[: nt.value].copy(), tree_idx=ti[: nt.value].copy(), flags=flags.value)

    def stage_compose_batch(self, headpose, variance, list_cap: int = 24) -> dict:
        hp = np.ascontiguousarray(headpose, np.float32); var = np.ascontiguousarray(variance, np.float32)
        n = len(hp)
        counts = np.zeros((n, 5), np.int32); dom = np.zeros(n, np.int32); nt = np.zeros(n, np.int32); flags = np.zeros(n, np.int32)
        fi = np.zeros((n, list_cap), np.int32); ti = np.zeros((n, list_cap), np.int32)
        capi.check(capi.lib().crf_stage_compose_batch(self.h, capi.ptr(hp, C.c_float), capi.ptr(var, C.c_float), n, capi.ptr(counts, C.c_int32), capi.ptr(dom, C.c_int32),
                                                      capi.ptr(nt, C.c_int32), capi.ptr(flags, C.c_int32), capi.ptr(fi, C.c_int32), capi.ptr(ti, C.c_int32), list_cap))
        return dict(tree_counts=counts, dominant=dom, ntrees=nt, flags=flags, forest_idx=fi, tree_idx=ti)

    def stage_votes_meanshift(self, planes: np.ndarray, stride: int, forest_idx, tree_idx, vote_cap: int = 0) -> dict:
        planes = np.ascontiguousarray(planes, np.uint8)
        Cn, H, W = planes.shape
        fi = np.ascontiguousarray(forest_idx, np.int32); ti = np.ascontiguousarray(tree_idx, np.int32)
        nv = np.zeros(10, np.int32); votes = np.zeros((10, max(vote_cap, 1), 3), np.float32)
        mean = np.zeros((10, 2), np.float32); rnd = np.zeros((10, 2), np.int32); it = np.zeros(10, np.int32)
        capi.check(capi.lib().crf_stage_votes_meanshift(self.h, capi.ptr(fi, C.c_int32), capi.ptr(ti, C.c_int32), len(fi), capi.ptr(planes, C.c_uint8),
                                                        Cn, W, H, stride, capi.ptr(nv, C.c_int32), capi.ptr(votes, C.c_float) if vote_cap else None, vote_cap,
                                                        capi.ptr(mean, C.c_float), capi.ptr(rnd, C.c_int32), capi.ptr(it, C.c_int32)))
        return dict(n_votes=nv, votes=votes if vote_cap else None, mean=mean, rounded=rnd, iters=it)

    def stage_meanshift(self, votes_xyw: np.ndarray):
        v = np.ascontiguousarray(votes_xyw, np.float32).reshape(-1, 3)
        mean = np.zeros(2, np.float32); rnd = np.zeros(2, np.int32); it = C.c_int()
        capi.check(capi.lib().crf_stage_meanshift(self.h, capi.ptr(v, C.c_float), len(v), capi.ptr(mean, C.c_float), capi.ptr(rnd, C.c_int32), C.byref(it)))
        return mean, rnd, it.value


class CascadeClassifier:
    """cv::CascadeClassifier (src/FaceForest.cpp:23) for OpenCV's HAAR cascades: the reference's face cascade or any other that
    cv::CascadeClassifier loads (stump or tree weak classifiers, upright or tilted features, new or old XML format; not LBP / HOG).
    load() parses the XML on the host, detectMultiScale evaluates it on the GPU (crf_detect_faces)."""

    def __init__(self, path: str | None = None):
        self.h = None
        if path:
            self.load(path)

    def load(self, path: str) -> bool:
        h = C.c_void_p()
        if capi.lib().crf_cascade_load(str(path).encode(), C.byref(h)) != 0:
            return False
        self.close()
        self.h = h
        return True

    def empty(self) -> bool:
        return self.h is None

    def close(self) -> None:
        if getattr(self, "h", None):
            capi.lib().crf_cascade_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def detectMultiScale(self, ctx: "Context", img: np.ndarray, scaleFactor: float = 1.1, minNeighbors: int = 3, minSize=(0, 0)) -> list:
        img = np.ascontiguousarray(img, np.uint8)
        rows, cols = img.shape[:2]
        cap = 1024
        out = (Rect * cap)()
        n = capi.lib().crf_detect_faces(ctx.h, self.h, capi.ptr(img, C.c_uint8), rows, cols, cols * 3, float(scaleFactor), int(minNeighbors), int(max(minSize)), out, cap)
        if n < 0:
            capi.check(n)
        return [(r.x, r.y, r.width, r.height) for r in out[: min(n, cap)]]

    def detectMultiScaleBatch(self, ctx: "Context", frames, scaleFactor: float = 1.1, minNeighbors: int = 3, minSize=(0, 0)) -> list:
        """detectMultiScale on every frame of `frames` (BGR frames of any sizes: a list or an [n, rows, cols, 3] array) in one call
        (crf_detect_faces_batch_mixed): one list of (x, y, w, h) per frame, each equal to detectMultiScale on that frame."""
        frames = _frame_list(frames)
        if not frames:
            return []
        L = capi.lib()
        args = (ctx.h, self.h, capi.images(frames), len(frames), float(scaleFactor), int(minNeighbors), int(max(minSize)))
        cap = 64 * len(frames)
        while True:
            out, iob = (Rect * cap)(), np.zeros(cap, np.int32)
            n = L.crf_detect_faces_batch_mixed(*args, out, capi.ptr(iob, C.c_int32), cap)
            if n < 0:
                capi.check(n)
            if n <= cap:
                break
            cap = n
        per = [[] for _ in frames]
        for r, i in zip(out[:n], iob[:n]):
            per[i].append((r.x, r.y, r.width, r.height))
        return per


class MultiContext:
    """Several GPUs behind one caller (crf_multi_*): one context and one host thread per GPU inside the library, contiguous
    shards of the faces, records written straight into one array.  devices=None: every visible GPU."""

    def __init__(self, model: Model, devices=None, options: Options | None = None):
        self.model = model
        h = C.c_void_p()
        d = None if devices is None else np.ascontiguousarray(devices, np.int32)
        capi.check(capi.lib().crf_multi_create(model.h, None if d is None else capi.ptr(d, C.c_int32), 0 if d is None else len(d),
                                               C.byref(options) if options is not None else None, C.byref(h)))
        self.h = h
        self.n_devices = capi.lib().crf_multi_device_count(self.h)

    def close(self) -> None:
        if getattr(self, "h", None):
            capi.lib().crf_multi_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def analyze_crops(self, crops: np.ndarray, headpose_only: bool = False) -> np.ndarray:
        crops = np.ascontiguousarray(crops, np.uint8)
        n, rows, cols = crops.shape[:3]
        out = np.zeros(n, FACE_DTYPE)
        capi.check(capi.lib().crf_multi_analyze_crops(self.h, crops.ctypes.data, n, rows, cols, out.ctypes.data, int(headpose_only)))
        return out

    def analyze_crops_ptr(self, host_ptr: int, n: int, rows: int, cols: int, out: np.ndarray, headpose_only: bool = False) -> None:
        capi.check(capi.lib().crf_multi_analyze_crops(self.h, host_ptr, n, rows, cols, out.ctypes.data, int(headpose_only)))

    def analyze_batch(self, frames, boxes, image_of_box) -> np.ndarray:
        """Context.analyze_batch sharded over the GPUs: frames of any sizes."""
        frames = _frame_list(frames)
        n = len(boxes)
        rects = (Rect * max(n, 1))(*[Rect(int(b[0]), int(b[1]), int(b[2]), int(b[3])) for b in boxes])
        iob = np.ascontiguousarray(image_of_box, np.int32)
        out = np.zeros(n, FACE_DTYPE)
        capi.check(capi.lib().crf_multi_analyze_batch_mixed(self.h, capi.images(frames), len(frames), rects, capi.ptr(iob, C.c_int32), n,
                                                            out.ctypes.data))
        return out


class FaceForest:
    """FaceForest (include/FaceForest.hpp:77-159, src/FaceForest.cpp).  Face boxes are supplied by the caller."""

    def __init__(self, option: FaceForestOptions | None = None, model: Model | None = None):
        self.is_inizialized = False
        self.option = option or FaceForestOptions()
        try:
            if model is None:
                o = self.option
                if o.packed_model:
                    model = Model(packed=o.packed_model)
                else:
                    model = Model(o.hp_forest_param.tree_path, o.mp_forest_param.tree_path, o.hp_forest_param.ntrees or 15,
                                  o.mp_forest_param.ntrees or 20)
            self.model = model
            self.ctx = Context(model, self.option.device, _options(self.option))
            self.m_face_cascade = None
            if self.option.fd_option.path_face_cascade:   # src/FaceForest.cpp:23-28
                self.m_face_cascade = CascadeClassifier(self.option.fd_option.path_face_cascade)
                if self.m_face_cascade.empty():
                    import sys
                    print(f"(!) Error loading face detection model: {self.option.fd_option.path_face_cascade}", file=sys.stderr)
                    self.model = None; self.ctx = None
                    return
        except CrfError as e:  # src/FaceForest.cpp:31-36: ERROR(...) and leave is_inizialized false
            import sys
            print(f"(!) Error loading forest: {e}", file=sys.stderr)
            self.model = None; self.ctx = None
            return
        self.is_inizialized = True

    def _to_faces(self, recs: np.ndarray, boxes) -> list:
        return [Face(float(r["headpose"]), tuple(int(v) for v in b), r["ffd"].copy(), r) for r, b in zip(recs, boxes)]

    def analyzeFace(self, img: np.ndarray, face_bbox, face: Face | None = None, normalize: bool = True) -> Face:
        """src/FaceForest.cpp:183-258."""
        if not self.is_inizialized:
            raise AssertionError("CV_Assert(is_inizialized)")  # src/FaceForest.cpp:191
        f = self._to_faces(self.ctx.analyze_faces(img, [face_bbox]), [face_bbox])[0]
        if face is not None:
            face.headpose, face.bbox, face.ffd_cordinates, face.record = f.headpose, f.bbox, f.ffd_cordinates, f.record
            return face
        return f

    def detectFace(self, img: np.ndarray, face_cascade: CascadeClassifier, fd_option: FaceDetectionOption) -> list:
        """src/FaceForest.cpp:136-159: detectMultiScale(img, boxes, search_scale_factor, min_neighbors, 0, Size(min_feature_size))
        with the cascade evaluated on the GPU (SURVEY 8 f2) + the reference's box enlargement."""
        mfs = (fd_option.min_feature_size, fd_option.min_feature_size)
        det = face_cascade.detectMultiScale(self.ctx, img, scaleFactor=fd_option.search_scale_factor, minNeighbors=fd_option.min_neighbors, minSize=mfs)
        return enlarge_detections(det, img.shape[0], img.shape[1])

    def analyzeImage(self, img: np.ndarray, faces_bboxes=None, faces: list | None = None) -> list:
        """src/FaceForest.cpp:161-181.  With faces_bboxes=None the Haar cascade of fd_option runs first (on the GPU), as in the
        reference; otherwise the caller's boxes are used.  All faces of the frame go through the GPU in one launch."""
        if not self.is_inizialized:
            raise AssertionError("CV_Assert(is_inizialized)")  # src/FaceForest.cpp:167
        if faces_bboxes is None:
            if self.m_face_cascade is None:
                raise AssertionError("no face cascade loaded: pass boxes or set fd_option.path_face_cascade")
            faces_bboxes = self.detectFace(img, self.m_face_cascade, self.option.fd_option)
        out = self._to_faces(self.ctx.analyze_faces(img, list(faces_bboxes)), faces_bboxes)
        if faces is not None:
            faces.clear(); faces.extend(out)
        return out

    def analyzeImages(self, frames) -> list:
        """analyzeImage(img) with the Haar cascade of fd_option for every frame of `frames` (BGR frames of any sizes) in one call
        (crf_analyze_images_mixed): the frames cross PCIe once, for detection and analysis.  One list of Face per frame, in
        detectMultiScale's order.  A detection whose enlarged box the analysis path cannot take (a face cut by the bottom border) comes
        back with a zero record whose flags carry capi.FACE_NOT_ANALYSED, where analyzeImage would raise."""
        if not self.is_inizialized:
            raise AssertionError("CV_Assert(is_inizialized)")
        if self.m_face_cascade is None:
            raise AssertionError("no face cascade loaded: set fd_option.path_face_cascade")
        fd = self.option.fd_option
        frames = _frame_list(frames)
        if not frames:
            return []
        L = capi.lib()
        args = (self.ctx.h, self.m_face_cascade.h, capi.images(frames), len(frames), float(fd.search_scale_factor), int(fd.min_neighbors),
                int(fd.min_feature_size))
        cap = 64 * len(frames)
        while True:   # a second call only when the frames hold more than 64 faces each on average
            boxes, iob, recs = (Rect * cap)(), np.zeros(cap, np.int32), np.zeros(cap, FACE_DTYPE)
            n = L.crf_analyze_images_mixed(*args, boxes, capi.ptr(iob, C.c_int32), recs.ctypes.data, cap)
            if n < 0:
                capi.check(n)
            if n <= cap:
                break
            cap = n
        per = [[] for _ in frames]
        for k in range(n):
            b = boxes[k]
            per[iob[k]].extend(self._to_faces(recs[k:k + 1], [(b.x, b.y, b.width, b.height)]))
        return per


class MeanShift:
    """include/MeanShift.hpp:27-50."""

    @staticmethod
    def shift(ctx: Context, votes_xyw: np.ndarray):
        return ctx.stage_meanshift(votes_xyw)
