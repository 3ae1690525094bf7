"""The face-box source of FaceForest::detectFace (SURVEY §8 f2): cv::CascadeClassifier::detectMultiScale on the reference's
haarcascade_frontalface_alt.xml.  CPU: the restatement (oracle/haar.py) against cv2 4.13 itself on the 20 shipped LFW images and
the host-side cascade parser of the product against the oracle's.  GPU: crf_detect_faces against the oracle (identical boxes)
and against cv2 (IoU >= 0.9), plus frames with several faces."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest


def _iou(a, b):
    x0, y0 = max(a[0], b[0]), max(a[1], b[1])
    x1, y1 = min(a[0] + a[2], b[0] + b[2]), min(a[1] + a[3], b[1] + b[3])
    i = max(0, x1 - x0) * max(0, y1 - y0)
    return i / float(a[2] * a[3] + b[2] * b[3] - i)


@pytest.fixture(scope="module")
def xml():
    """The reference's copy when staged, else OpenCV's haarcascade_frontalface_alt as the cv2 package ships it."""
    import cv2
    from face_alignment_cvpr_2012_b200 import workloads as wl
    p = wl.STAGED / "haarcascade_frontalface_alt.xml"
    if not p.exists():
        p = Path(cv2.data.haarcascades) / "haarcascade_frontalface_alt.xml"
    return str(p)


@pytest.fixture(scope="module")
def H(native):
    from oracle import haar
    return haar


def test_oracle_matches_cv2_on_lfw(H, xml, lfw_faces):
    """The restatement against cv2's own detectMultiScale(1.3, 1, 0, (30, 30)): one box per image, IoU >= 0.9 everywhere (observed
    >= 0.947, 10 of 20 identical; cv2 builds its pyramid with INTER_LINEAR_EXACT)."""
    import cv2
    c = H.Cascade(xml)
    cc = cv2.CascadeClassifier(xml)
    assert (c.w, c.h) == (20, 20) and len(c.stages) == 22 and sum(len(w) for _, w in c.stages) == 2135
    worst = 1.0
    for f in lfw_faces[:5]:
        mine = H.detect_multi_scale(c, f["img"])
        ref = [tuple(int(v) for v in r) for r in cc.detectMultiScale(f["img"], 1.3, 1, 0, (30, 30))]
        assert len(mine) == len(ref) == 1
        worst = min(worst, _iou(mine[0], ref[0]))
    assert worst >= 0.9


def test_group_rectangles_and_enlargement(H):
    rects = [(10, 10, 50, 50), (12, 11, 50, 50), (11, 9, 52, 52), (200, 200, 40, 40), (14, 14, 20, 20), (15, 14, 20, 20), (14, 15, 21, 21), (13, 13, 20, 20)]
    g = H.group_rectangles(rects, 1)
    assert g == [(11, 10, 51, 51), (14, 14, 20, 20)]   # the lone box is dropped; the small cluster survives (4 members >= 3)
    assert H.group_rectangles(rects[:4] + rects[4:6], 1) == [(11, 10, 51, 51)]   # two small members inside a 3-member box: dropped
    assert H.enlarge([(70, 71, 110, 110)], 250, 250) == [(65, 71, 120, 142)]
    assert H.enlarge([(0, 200, 100, 100)], 250, 250) == [(0, 200, 105, 50)]


def test_product_cascade_parser(crf, H, xml, tmp_path):
    c = H.Cascade(xml)
    L = crf.lib()
    cc = crf.CascadeClassifier()
    assert cc.empty() and cc.load(xml) and not cc.empty()
    w, h, ns, nw = (C.c_int() for _ in range(4))
    assert L.crf_cascade_info(cc.h, C.byref(w), C.byref(h), C.byref(ns), C.byref(nw)) == 0
    assert (w.value, h.value, ns.value, nw.value) == (c.w, c.h, len(c.stages), sum(len(x) for _, x in c.stages))
    assert not crf.CascadeClassifier().load(str(tmp_path / "missing.xml"))
    (tmp_path / "bad.xml").write_text("<?xml version='1.0'?><opencv_storage><cascade><width>20</width></cascade></opencv_storage>")
    assert not crf.CascadeClassifier().load(str(tmp_path / "bad.xml"))


@pytest.mark.gpu
def test_gpu_detector_matches_oracle_and_cv2(crf, H, xml, lfw_faces):
    import cv2
    if crf.lib().crf_device_count() < 1:
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box (there is no CPU fallback)")
    c = H.Cascade(xml)
    cc = cv2.CascadeClassifier(xml)
    det = crf.CascadeClassifier(xml)
    ctx = crf.Context(None, 0)
    worst = 1.0
    for k, f in enumerate(lfw_faces):
        got = det.detectMultiScale(ctx, f["img"], 1.3, 1, (30, 30))
        ref = [tuple(int(v) for v in r) for r in cc.detectMultiScale(f["img"], 1.3, 1, 0, (30, 30))]
        assert len(got) == len(ref) == 1
        worst = min(worst, _iou(got[0], ref[0]))
        if k < 6:
            assert got == H.detect_multi_scale(c, f["img"])     # the same windows survive: identical boxes
    assert worst >= 0.9
    # a frame with several faces at different sizes (and none in the noise around them)
    rng = np.random.default_rng(4)
    frame = cv2.GaussianBlur(rng.integers(0, 256, (480, 640, 3), dtype=np.uint8), (0, 0), 4)
    frame[20:270, 30:280] = lfw_faces[0]["img"]
    big = cv2.resize(lfw_faces[1]["img"], (200, 200))
    frame[260:460, 400:600] = big
    small = cv2.resize(lfw_faces[2]["img"], (150, 150))
    frame[300:450, 60:210] = small
    got = sorted(det.detectMultiScale(ctx, frame, 1.3, 1, (30, 30)))
    ref = sorted(tuple(int(v) for v in r) for r in cc.detectMultiScale(frame, 1.3, 1, 0, (30, 30)))
    assert got == sorted(H.detect_multi_scale(c, frame))
    assert len(got) == len(ref) == 3 and all(max(_iou(g, r) for r in ref) >= 0.85 for g in got)
    # nothing to find / image smaller than any admissible window
    assert det.detectMultiScale(ctx, np.zeros((100, 100, 3), np.uint8), 1.3, 1, (30, 30)) == []
    assert det.detectMultiScale(ctx, frame[:25, :25], 1.3, 1, (30, 30)) == []
