"""Every OpenCV HAAR cascade on the GPU detector: tree weak classifiers, tilted features and the old XML format.

For each of the 17 cascades of the cv2 package and for seeded synthetic ones (trees of 1 to 3 nodes, tilted and upright features, each
written in both XML formats), crf_detect_faces returns exactly the boxes of the CPU oracle (tests/haar_cascade_oracle.py), whose pyramid
arithmetic is the GPU's.  The batched and analysing entry points give frame-by-frame results with these cascades too, a tilted cascade
costs one launch more per group than an upright one, and switching cascades in one context gives what a fresh context gives."""
from pathlib import Path

import numpy as np
import pytest

import haar_cascade_oracle as G
from test_gpu_detect_batch import _analysable, _textured, detect_one
from test_gpu_detect_mixed import _recs_equal, analyze_images_mixed, detect_mixed, padded, per_frame

cv2 = pytest.importorskip("cv2")
CV2_DIR = Path(cv2.data.haarcascades)
CV2_CASCADES = sorted(p.name for p in CV2_DIR.glob("haarcascade_*.xml"))
FACE = CV2_DIR / "haarcascade_frontalface_alt.xml"
ALT2 = CV2_DIR / "haarcascade_frontalface_alt2.xml"
EYEGLASSES = CV2_DIR / "haarcascade_eye_tree_eyeglasses.xml"


@pytest.fixture(scope="module")
def gpu_ctx(crf):
    if crf.lib().crf_device_count() < 1:
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box (there is no CPU fallback)")
    return crf.Context(None, 0)


@pytest.fixture(scope="module")
def synth(tmp_path_factory):
    """{name: (new-format path, old-format path)} of seeded synthetic cascades."""
    d = tmp_path_factory.mktemp("cascades")
    out = {}
    for name, kw in {"trees_tilted": dict(seed=3), "trees": dict(seed=4, p_tilted=0.0), "tilted_stumps": dict(seed=5, max_nodes=1, p_tilted=0.6),
                     "flat_24x12": dict(seed=6, w=24, h=12, stage_sizes=(3, 5, 5))}.items():
        out[name] = tuple(G.write_cascade(d / f"{name}_{fmt}.xml", fmt=fmt, **kw) for fmt in ("new", "old"))
    return out


@pytest.fixture(scope="module")
def frames():
    """Procedural faces (workloads.procedural_lfw, 250 x 250) and textured frames of odd sizes."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    lfw = [f["img"] for f in wl.procedural_lfw()]
    return [lfw[0], lfw[7], lfw[13], _textured(1, 161, 203, 3)[0], _textured(1, 97, 131, 4)[0]]


def _oracle(path, frame, mn, ms):
    from oracle import oracle as O
    c = G.Cascade(path)
    gray = O.bgr2gray(np.ascontiguousarray(frame))
    ref = G.detect_candidates(c, gray, 1.3, ms) if mn == 0 else G.detect_multi_scale(c, gray, 1.3, mn, ms)
    return [tuple(int(v) for v in r) for r in ref]


# ---- every cascade against the oracle ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", CV2_CASCADES)
def test_cv2_cascade_equals_oracle(crf, gpu_ctx, frames, name, tmp_path):
    """The whole cascade, and its first 3 stages: the body, plate and profile cascades find nothing in these frames, the truncated copies
    of every cascade find windows, so each cascade's own features, trees and tilted rects are compared on real candidates."""
    for path in (CV2_DIR / name, G.truncate_cascade(CV2_DIR / name, tmp_path / name, 3)):
        cas = crf.CascadeClassifier(str(path))
        assert not cas.empty(), crf.lib().crf_last_error()
        found = 0
        for mn in (0, 1):
            for i, f in enumerate(frames):
                got = detect_one(crf, gpu_ctx, cas, f, mn=mn, ms=0)
                assert got == _oracle(path, f, mn, 0), (name, path, mn, i)
                found += len(got)
        if path != CV2_DIR / name:
            assert found > 0, name


@pytest.mark.gpu
def test_synthetic_cascades_equal_oracle_in_both_formats(crf, gpu_ctx, frames, synth):
    found = 0
    for name, (new, old) in synth.items():
        a, b = crf.CascadeClassifier(new), crf.CascadeClassifier(old)
        for mn in (0, 1):
            for i, f in enumerate(frames):
                got = detect_one(crf, gpu_ctx, a, f, mn=mn, ms=0)
                assert got == detect_one(crf, gpu_ctx, b, f, mn=mn, ms=0) == _oracle(new, f, mn, 0), (name, mn, i)
                found += len(got)
    assert found > 0


# ---- batched entry points -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("which", ["eye_tree_eyeglasses", "trees_tilted"])
def test_mixed_batch_equals_frame_by_frame(crf, gpu_ctx, synth, which):
    from face_alignment_cvpr_2012_b200 import workloads as wl
    cas = crf.CascadeClassifier(str(EYEGLASSES) if which == "eye_tree_eyeglasses" else synth["trees_tilted"][0])
    fr = [wl.make_frames(1, 480, 640, 6, seed=21)[0][0], _textured(1, 240, 320, 5)[0], _textured(1, 15, 15, 1)[0], padded(_textured(1, 130, 170, 7)[0]),
          wl.procedural_lfw()[3]["img"], _textured(1, 97, 131, 6)[0], wl.make_frames(1, 1080, 1920, 12, seed=22)[0][0]]
    for mn in (0, 1):
        want_boxes, want_iob = per_frame(crf, gpu_ctx, cas, fr, mn=mn, ms=0)
        n, boxes, iob = detect_mixed(crf, gpu_ctx, cas, fr, mn=mn, ms=0)
        assert n == len(want_boxes) > 0 and boxes == want_boxes and iob == want_iob, mn


@pytest.mark.gpu
def test_analyze_images_mixed_equals_analyze_faces(crf, synth_models, tmp_path):
    """crf_analyze_images_mixed with tree cascades: records bitwise equal to crf_analyze_faces on the enlarged boxes, and the boxes that
    fail the analysis path's checks flagged CRF_FACE_NOT_ANALYSED.  frontalface_alt2 on faces; a synthetic tree + tilted cascade with a
    flat 24 x 5 window on texture, because a square window never leaves a clipped box shorter than a patch."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    from oracle import haar as H
    gm, _ = synth_models
    ctx = crf.Context(gm, 0)
    lfw = wl.procedural_lfw()
    flat = G.write_cascade(tmp_path / "flat_24x5.xml", w=24, h=5, stage_sizes=(3, 5), seed=8)
    cases = [(str(ALT2), [wl.make_frames(1, 480, 640, 6, seed=31)[0][0], lfw[2]["img"], padded(lfw[5]["img"]), lfw[11]["img"][:, :140],
                          lfw[17]["img"][200:]]),
             (flat, [_textured(1, 90, 160, 12)[0], _textured(1, 70, 120, 13)[0], padded(_textured(1, 100, 140, 14)[0])])]
    analysed = rejected = 0
    for path, fr in cases:
        cas = crf.CascadeClassifier(path)
        got, iob, recs = analyze_images_mixed(crf, ctx, cas, fr, 0, 0)
        k = 0
        for i, f in enumerate(fr):
            rows, cols = f.shape[:2]
            want = H.enlarge(detect_one(crf, ctx, cas, np.ascontiguousarray(f), mn=0, ms=0), rows, cols)
            assert got[k:k + len(want)] == want and iob[k:k + len(want)] == [i] * len(want)
            ok = [j for j, b in enumerate(want) if _analysable(b)]
            ref = ctx.analyze_faces(f, [want[j] for j in ok]) if ok else np.zeros(0, crf.FACE_DTYPE)
            for j, b in enumerate(want):
                r = recs[k + j]
                if j in ok:
                    assert r["flags"] & crf.capi.FACE_NOT_ANALYSED == 0 and _recs_equal(r, ref[ok.index(j)]), (path, i, j)
                    analysed += 1
                else:
                    zero = np.zeros(1, crf.FACE_DTYPE)[0]
                    zero["flags"] = crf.capi.FACE_NOT_ANALYSED
                    assert _recs_equal(r, zero), (path, i, j, b)
                    rejected += 1
            k += len(want)
        assert k == len(got) > 0, path
    assert analysed > 0 and rejected > 0


# ---- launches per group ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_launches_per_group(crf, gpu_ctx, synth):
    """Per group: 3 pyramid passes (+1, the tilted integral, when the cascade has tilted features), one per later stage group, 3 for the
    scan rule and the candidate compaction; trees cost no launch.  The count does not depend on the frame count."""
    fr = [_textured(1, r, c, 50 + k)[0] for k, (r, c) in enumerate([(240, 320), (120, 160), (97, 131), (200, 300), (240, 320)])]

    def launches(path, n):
        cas = crf.CascadeClassifier(str(path))
        gpu_ctx.reset_counters()
        detect_mixed(crf, gpu_ctx, cas, fr[:n], mn=1, ms=0, cap=0)
        return gpu_ctx.counters()["kernel_launches"]

    for path, want in ((FACE, 8), (ALT2, 8), (EYEGLASSES, 9), (CV2_DIR / "haarcascade_smile.xml", 9), (CV2_DIR / "haarcascade_license_plate_rus_16stages.xml", 8),
                       (synth["trees"][0], 7), (synth["trees_tilted"][0], 8), (synth["tilted_stumps"][1], 8)):
        assert launches(path, 1) == launches(path, 5) == want, Path(path).name


# ---- the device cache ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_switching_cascades_in_one_context(crf, gpu_ctx, synth):
    """stump -> tree -> tilted -> tree + tilted -> stump in one context, every cascade's boxes equal to a fresh context's: the device
    tables (weak classifiers, nodes, leaves, tilted flags) follow the cascade id."""
    fr = [_textured(1, 161, 203, 3)[0], _textured(1, 120, 160, 8)[0]]
    order = [FACE, synth["trees"][0], synth["tilted_stumps"][0], ALT2, synth["trees_tilted"][1], EYEGLASSES, FACE, synth["trees"][1], FACE]
    for path in order:
        cas = crf.CascadeClassifier(str(path))
        fresh = crf.Context(None, 0)
        for f in fr:
            assert detect_one(crf, gpu_ctx, cas, f, mn=0, ms=0) == detect_one(crf, fresh, cas, f, mn=0, ms=0), Path(path).name
        del fresh
