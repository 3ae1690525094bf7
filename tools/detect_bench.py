"""Detection + alignment of whole frames (FaceForest::analyzeImage without boxes): the per-frame route against the batched calls.

  (a) per frame: crf_detect_faces, detectFace's enlargement on the host, crf_analyze_faces on the boxes the analysis path takes
  (b) crf_detect_faces_batch on all frames of a resolution in one call
  (c) crf_analyze_images on the same frames in one call
  (d) crf_detect_faces_batch_mixed and crf_analyze_images_mixed on all frames of the set in one call, whatever their sizes
plus the latency of crf_detect_faces on one frame, and (b) for a few cascade stage-group splits (CRF_HAAR_SPLIT).  Frames: the C3 set
(workloads.make_frames, 64 x 1080p), the C5 mixed-resolution set (workloads.make_mixed: 5 sizes, so (b) and (c) make one call per
resolution) and the R64 set (workloads.make_ragged: 64 distinct sizes, so (b) and (c) go frame by frame); whether their faces are
LFW-based or procedural is in the output's `data`.  C5 with its boxes given: one crf_analyze_faces call per image against one
crf_analyze_batch_mixed call.  Every call ends in a device synchronise, so host clocks time the whole call.
With --lib pointing at the library of an earlier build, entry points that build lacks are skipped, to give the "before" numbers on the
same frames.

--cascade names another cascade file (default: the face cascade); --sets C3,R64 limits the run to those frame sets (the extras: boxes
given, single-frame latency, split sweep, only run with the default sets).  --cv2 also times cv2.CascadeClassifier.detectMultiScale with
the same cascade and parameters on the first 16 frames of each set, one host call per frame on the host's cores, for scale.  With a library that has
the counters, `launches_per_group` is the kernel launches of crf_detect_faces_batch on one group (one C3 frame).

  python tools/detect_bench.py [--lib path/to/libcrf_b200.so] [--reps 3] [--cascade file.xml] [--sets C3,R64] [--cv2] [--out detect_bench.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


class Rect(C.Structure):
    _fields_ = [("x", C.c_int), ("y", C.c_int), ("width", C.c_int), ("height", C.c_int)]


class Image(C.Structure):
    _fields_ = [("bgr", C.c_void_p), ("rows", C.c_int), ("cols", C.c_int), ("step", C.c_size_t)]


def images(frames):
    return (Image * len(frames))(*[Image(f.ctypes.data, f.shape[0], f.shape[1], f.strides[0]) for f in frames])


def load(path: str):
    L = C.CDLL(path)
    vp = C.c_void_p
    L.crf_last_error.restype = C.c_char_p
    L.crf_model_load.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.POINTER(vp)]
    L.crf_model_load_packed.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.crf_ctx_create.argtypes = [vp, C.c_int, vp, C.POINTER(vp)]
    L.crf_ctx_destroy.argtypes = [vp]
    L.crf_cascade_load.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.crf_detect_faces.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_size_t, C.c_double, C.c_int, C.c_int, C.POINTER(Rect), C.c_int]
    L.crf_analyze_faces.argtypes = [vp, vp, C.c_int, C.c_int, C.c_size_t, C.POINTER(Rect), C.c_int, vp]
    if hasattr(L, "crf_detect_faces_batch"):
        L.crf_detect_faces_batch.argtypes = [vp, vp, C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_double, C.c_int, C.c_int,
                                             C.POINTER(Rect), vp, C.c_int]
        L.crf_analyze_images.argtypes = [vp, vp, C.POINTER(vp), C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_double, C.c_int, C.c_int,
                                         C.POINTER(Rect), vp, vp, C.c_int]
    if hasattr(L, "crf_detect_faces_batch_mixed"):
        L.crf_detect_faces_batch_mixed.argtypes = [vp, vp, C.POINTER(Image), C.c_int, C.c_double, C.c_int, C.c_int, C.POINTER(Rect), vp, C.c_int]
        L.crf_analyze_images_mixed.argtypes = [vp, vp, C.POINTER(Image), C.c_int, C.c_double, C.c_int, C.c_int, C.POINTER(Rect), vp, vp, C.c_int]
        L.crf_analyze_batch_mixed.argtypes = [vp, C.POINTER(Image), C.c_int, C.POINTER(Rect), vp, C.c_int, vp]
    return L


def check(L, rc):
    if rc < 0:
        raise RuntimeError(f"crf error {rc}: {L.crf_last_error().decode()}")
    return rc


# FaceForest's defaults (fd_option): scale factor 1.3, min_neighbors 1, min_feature_size 30
SF, MN, MS = 1.3, 1, 30
RECORD = 640   # sizeof(crf_face_t) is smaller; a generous buffer per face


def analysable(b):
    if b[2] <= 0 or b[3] <= 0:
        return False
    s = np.float32(125) / np.float32(b[2])
    return 31 < int(np.float32(b[2]) * s) <= 125 and 31 < int(np.float32(b[3]) * s) <= 521


def per_frame_route(L, ctx, cas, frames):
    """(a): returns (faces analysed, boxes found, detection seconds, total seconds)"""
    from face_alignment_cvpr_2012_b200.face_forest import enlarge_detections
    rows, cols = frames[0].shape[:2]
    out = (Rect * 4096)()
    rec = np.zeros(4096 * RECORD, np.uint8)
    faces = found = 0
    t_det = 0.0
    t0 = time.perf_counter()
    for f in frames:
        t1 = time.perf_counter()
        n = check(L, L.crf_detect_faces(ctx, cas, f.ctypes.data, rows, cols, cols * 3, SF, MN, MS, out, 4096))
        t_det += time.perf_counter() - t1
        found += n
        boxes = [b for b in enlarge_detections([(r.x, r.y, r.width, r.height) for r in out[:n]], rows, cols) if analysable(b)]
        if boxes:
            rb = (Rect * len(boxes))(*[Rect(*b) for b in boxes])
            check(L, L.crf_analyze_faces(ctx, f.ctypes.data, rows, cols, cols * 3, rb, len(boxes), rec.ctypes.data))
            faces += len(boxes)
    return faces, found, t_det, time.perf_counter() - t0


def batch_detect(L, ctx, cas, frames):
    rows, cols = frames[0].shape[:2]
    ptrs = (C.c_void_p * len(frames))(*[f.ctypes.data for f in frames])
    t0 = time.perf_counter()
    n = check(L, L.crf_detect_faces_batch(ctx, cas, ptrs, len(frames), rows, cols, cols * 3, SF, MN, MS, None, None, 0))
    return n, time.perf_counter() - t0


def batch_analyze(L, ctx, cas, frames):
    rows, cols = frames[0].shape[:2]
    ptrs = (C.c_void_p * len(frames))(*[f.ctypes.data for f in frames])
    cap = 64 * len(frames)
    boxes, iob, rec = (Rect * cap)(), np.zeros(cap, np.int32), np.zeros(cap * RECORD, np.uint8)
    t0 = time.perf_counter()
    n = check(L, L.crf_analyze_images(ctx, cas, ptrs, len(frames), rows, cols, cols * 3, SF, MN, MS, boxes, iob.ctypes.data, rec.ctypes.data, cap))
    return n, time.perf_counter() - t0


def mixed_detect(L, ctx, cas, frames):
    im = images(frames)
    t0 = time.perf_counter()
    n = check(L, L.crf_detect_faces_batch_mixed(ctx, cas, im, len(frames), SF, MN, MS, None, None, 0))
    return n, time.perf_counter() - t0


def mixed_analyze(L, ctx, cas, frames):
    im = images(frames)
    cap = 64 * len(frames)
    boxes, iob, rec = (Rect * cap)(), np.zeros(cap, np.int32), np.zeros(cap * RECORD, np.uint8)
    t0 = time.perf_counter()
    n = check(L, L.crf_analyze_images_mixed(ctx, cas, im, len(frames), SF, MN, MS, boxes, iob.ctypes.data, rec.ctypes.data, cap))
    return n, time.perf_counter() - t0


def boxes_per_image(L, ctx, data):
    """C5 with boxes given, one crf_analyze_faces call per image: (faces, seconds)"""
    rec = np.zeros(64 * RECORD, np.uint8)
    t0 = time.perf_counter()
    for f, b in data:
        rb = (Rect * len(b))(*[Rect(*map(int, x)) for x in b])
        check(L, L.crf_analyze_faces(ctx, f.ctypes.data, f.shape[0], f.shape[1], f.strides[0], rb, len(b), rec.ctypes.data))
    return sum(len(b) for _, b in data), time.perf_counter() - t0


def boxes_one_call(L, ctx, data):
    """C5 with boxes given, all images in one crf_analyze_batch_mixed call: (faces, seconds)"""
    frames = [f for f, _ in data]
    rb = [Rect(*map(int, x)) for _, b in data for x in b]
    iob = np.array([k for k, (_, b) in enumerate(data) for _ in b], np.int32)
    rects, rec = (Rect * len(rb))(*rb), np.zeros(len(rb) * RECORD, np.uint8)
    im = images(frames)
    t0 = time.perf_counter()
    check(L, L.crf_analyze_batch_mixed(ctx, im, len(frames), rects, iob.ctypes.data, len(rb), rec.ctypes.data))
    return len(rb), time.perf_counter() - t0


def med(fn, reps):
    """fn() -> (value..., seconds); median of the seconds over reps runs after one warm-up run"""
    fn()
    runs = [fn() for _ in range(reps)]
    return runs[len(runs) // 2][:-1] + (statistics.median(r[-1] for r in runs),)


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=str(ROOT / "face_alignment_cvpr_2012_b200" / "_lib" / "libcrf_b200.so"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--splits", default="0;1;1,3;2,5;3,8;1,2,4,8", help="CRF_HAAR_SPLIT values for the split sweep of (b) ('0' = one stage group)")
    ap.add_argument("--out", default="detect_bench.json", help="where the JSON result goes")
    ap.add_argument("--cascade", default=None, help="cascade XML (default: the face cascade, staged or cv2's haarcascade_frontalface_alt.xml)")
    ap.add_argument("--sets", default="C3,C5,R64", help="frame sets to run, of C3, C5, R64; the extras run only with all three")
    ap.add_argument("--cv2", action="store_true", help="also time cv2's detectMultiScale on the same frames (host cores)")
    a = ap.parse_args()
    import cv2
    from face_alignment_cvpr_2012_b200 import synthetic_model as sm
    from face_alignment_cvpr_2012_b200 import workloads as wl

    L = load(a.lib)
    batched = hasattr(L, "crf_detect_faces_batch")
    ragged = hasattr(L, "crf_detect_faces_batch_mixed")
    vp = C.c_void_p
    model = vp()
    packed = wl.staged_model_path()
    if packed:
        check(L, L.crf_model_load_packed(str(packed).encode(), C.byref(model)))
        model_tag = "staged (shipped forests)"
    else:
        hp, ffd = sm.write_model(tempfile.mkdtemp(prefix="crf_detect_bench_"), seed=5)
        check(L, L.crf_model_load(str(hp).encode(), 15, str(ffd).encode(), 20, C.byref(model)))
        model_tag = "synthetic forests (seed 5)"
    xml = wl.STAGED / "haarcascade_frontalface_alt.xml"
    if not xml.exists():
        xml = Path(cv2.data.haarcascades) / "haarcascade_frontalface_alt.xml"
    if a.cascade:
        xml = Path(a.cascade)
    sets = set(a.sets.split(","))
    cas = vp()
    check(L, L.crf_cascade_load(str(xml).encode(), C.byref(cas)))

    def new_ctx():
        c = vp()
        check(L, L.crf_ctx_create(model, 0, None, C.byref(c)))
        return c

    ctx = new_ctx()
    c3, _, _, tag = wl.make_frames(a.frames, 1080, 1920, 16)
    c3 = [np.ascontiguousarray(f) for f in c3]
    mixed, _ = wl.make_mixed(64)
    mixed = [(np.ascontiguousarray(f), b) for f, b in mixed]
    by_res = {}
    for fr, _ in mixed:
        by_res.setdefault(fr.shape[:2], []).append(fr)
    r64 = [(np.ascontiguousarray(f), b) for f, b in wl.make_ragged(64)]
    this_build = Path(a.lib).resolve() == (ROOT / "face_alignment_cvpr_2012_b200" / "_lib" / "libcrf_b200.so").resolve()
    res = {"gpu": gpu_info(), "library": "this build" if this_build else "earlier build (--lib)", "data": tag, "model": model_tag, "cascade": xml.name, "reps": a.reps,
           "params": {"scale_factor": SF, "min_neighbors": MN, "min_size": MS}, "sets": {}}

    def run_set(name, groups):
        nfr = sum(len(g) for g in groups)
        row = {"frames": nfr}
        fa = [med(lambda g=g: per_frame_route(L, ctx, cas, g), a.reps) for g in groups]
        faces, found, t_det, t_all = (sum(v[i] for v in fa) for i in range(4))
        row["a_per_frame"] = {"faces_found": found, "faces_analysed": faces, "frames_per_s": nfr / t_all, "ms_per_frame": 1e3 * t_all / nfr,
                              "detect_ms_per_frame": 1e3 * t_det / nfr}
        if batched:
            fb = [med(lambda g=g: batch_detect(L, ctx, cas, g), a.reps) for g in groups]
            n, t = sum(v[0] for v in fb), sum(v[1] for v in fb)
            row["b_detect_batch"] = {"faces_found": n, "frames_per_s": nfr / t, "detect_ms_per_frame": 1e3 * t / nfr}
            fc = [med(lambda g=g: batch_analyze(L, ctx, cas, g), a.reps) for g in groups]
            n, t = sum(v[0] for v in fc), sum(v[1] for v in fc)
            row["c_analyze_images"] = {"faces_found": n, "frames_per_s": nfr / t, "ms_per_frame": 1e3 * t / nfr}
        if ragged:
            frames = [f for g in groups for f in g]
            n, t = med(lambda: mixed_detect(L, ctx, cas, frames), a.reps)
            row["d_detect_mixed_one_call"] = {"faces_found": n, "frames_per_s": nfr / t, "detect_ms_per_frame": 1e3 * t / nfr}
            n, t = med(lambda: mixed_analyze(L, ctx, cas, frames), a.reps)
            row["d_analyze_images_mixed_one_call"] = {"faces_found": n, "frames_per_s": nfr / t, "ms_per_frame": 1e3 * t / nfr}
        if a.cv2:
            cc = cv2.CascadeClassifier(str(xml))
            frames = [cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for g in groups for f in g][:16]   # the first 16 frames, once: it is slow
            cc.detectMultiScale(frames[0], SF, MN, minSize=(MS, MS))
            t0 = time.perf_counter()
            n = sum(len(cc.detectMultiScale(f, SF, MN, minSize=(MS, MS))) for f in frames)
            t = time.perf_counter() - t0
            row["cv2_detect_host"] = {"frames": len(frames), "faces_found": n, "threads": cv2.getNumThreads(), "cpus": os.cpu_count(),
                                      "detect_ms_per_frame": 1e3 * t / len(frames)}
        res["sets"][name] = row
        print(name, json.dumps(row), flush=True)

    if hasattr(L, "crf_ctx_counters") and batched:
        from face_alignment_cvpr_2012_b200 import capi
        cnt = capi.Counters()
        L.crf_ctx_counters.argtypes = [vp, C.c_void_p]
        L.crf_ctx_reset_counters.argtypes = [vp]
        L.crf_ctx_reset_counters(ctx)
        batch_detect(L, ctx, cas, c3[:1])   # one frame: one group
        L.crf_ctx_counters(ctx, C.byref(cnt))
        res["launches_per_group"] = int(cnt.kernel_launches)
    if "C3" in sets:
        run_set(f"C3_{a.frames}x1080p", [c3])
    if "C5" in sets:
        run_set("C5_mixed_64", list(by_res.values()))
    if "R64" in sets:
        run_set("R64_ragged_64", [[f] for f, _ in r64])
    if sets != {"C3", "C5", "R64"}:
        L.crf_ctx_destroy(ctx)
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))
        print(json.dumps(res))
        return
    given = {}
    n, t = med(lambda: boxes_per_image(L, ctx, mixed), a.reps)
    given["per_image_analyze_faces"] = {"faces": n, "faces_per_s": n / t, "ms_per_call_set": 1e3 * t}
    if ragged:
        n, t = med(lambda: boxes_one_call(L, ctx, mixed), a.reps)
        given["one_call_analyze_batch_mixed"] = {"faces": n, "faces_per_s": n / t, "ms_per_call_set": 1e3 * t}
    res["C5_boxes_given"] = given
    print("C5 boxes given", json.dumps(given), flush=True)
    out = (Rect * 4096)()
    f0 = c3[0]
    lat = []
    for k in range(25):
        t0 = time.perf_counter()
        check(L, L.crf_detect_faces(ctx, cas, f0.ctypes.data, 1080, 1920, 1920 * 3, SF, MN, MS, out, 4096))
        if k >= 5:
            lat.append(time.perf_counter() - t0)
    res["single_frame_detect_ms_1080p"] = {"median": 1e3 * statistics.median(lat), "min": 1e3 * min(lat)}
    print("single frame", res["single_frame_detect_ms_1080p"], flush=True)
    if batched:
        sweep = {}
        for sp in a.splits.split(";"):
            os.environ["CRF_HAAR_SPLIT"] = sp
            c = new_ctx()
            n, t = med(lambda c=c: batch_detect(L, c, cas, c3), a.reps)
            sweep[sp] = {"faces_found": n, "detect_ms_per_frame": 1e3 * t / len(c3)}
            L.crf_ctx_destroy(c)
            print("split", sp, sweep[sp], flush=True)
        os.environ.pop("CRF_HAAR_SPLIT", None)
        res["split_sweep_C3"] = sweep
    L.crf_ctx_destroy(ctx)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
