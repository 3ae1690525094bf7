"""Detection and alignment across a batch of frames in one call: crf_detect_faces_batch and crf_analyze_images.

The batched path must give, frame by frame, exactly what crf_detect_faces / crf_analyze_faces give: the same candidate windows in the
same order, hence the same grouped boxes and records.  Besides the real face cascade, a synthetic stump cascade written here makes many
windows pass some stages and some pass all on textured frames, so the stage-group compaction, the stage-0 skip rule and the border cases
are exercised without real faces (from a clean checkout)."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

ERR_ARG = -1


def write_stump_cascade(path, w=20, h=20, stage_sizes=(3, 5, 7, 5, 9), seed=7):
    """An OpenCV new-format stump cascade: random two-rectangle features (a rect and its right or lower half, weights -1 and 2), stump
    thresholds 0 and leaves near -1 / +1.  Each stage has an odd number of stumps and threshold 0, so on texture about half of the windows
    pass each stage: stage 0 rejects about half, and a few per cent pass all five."""
    rng = np.random.default_rng(seed)
    feats, stages = [], []
    for n in stage_sizes:
        weak = []
        for _ in range(n):
            horizontal = rng.random() < 0.5
            a = int(rng.integers(1, (w if horizontal else h) // 2 + 1))   # half the feature's extent along its axis
            b = int(rng.integers(1, (h if horizontal else w) + 1))
            if horizontal:
                x, y = int(rng.integers(0, w - 2 * a + 1)), int(rng.integers(0, h - b + 1))
                rects = [(x, y, 2 * a, b, -1.0), (x + a, y, a, b, 2.0)]
            else:
                x, y = int(rng.integers(0, w - b + 1)), int(rng.integers(0, h - 2 * a + 1))
                rects = [(x, y, b, 2 * a, -1.0), (x, y + a, b, a, 2.0)]
            feats.append(rects)
            left, right = -float(rng.uniform(0.8, 1.2)), float(rng.uniform(0.8, 1.2))
            if rng.random() < 0.5:
                left, right = right, left
            weak.append((len(feats) - 1, left, right))
        stages.append(weak)
    out = ['<?xml version="1.0"?>', "<opencv_storage>", '<cascade type_id="opencv-cascade-classifier">', "  <stageType>BOOST</stageType>",
           "  <featureType>HAAR</featureType>", f"  <height>{h}</height>", f"  <width>{w}</width>", f"  <stageNum>{len(stages)}</stageNum>",
           "  <stages>"]
    for weak in stages:
        out += ["    <_>", f"      <maxWeakCount>{len(weak)}</maxWeakCount>", "      <stageThreshold>0.</stageThreshold>", "      <weakClassifiers>"]
        for fi, left, right in weak:
            out += ["        <_>", f"          <internalNodes>0 -1 {fi} 0.</internalNodes>", f"          <leafValues>{left:.6f} {right:.6f}</leafValues></_>"]
        out += ["      </weakClassifiers></_>"]
    out += ["  </stages>", "  <features>"]
    for rects in feats:
        out += ["    <_>", "      <rects>"] + [f"        <_>{x} {y} {rw} {rh} {wt:.1f}</_>" for x, y, rw, rh, wt in rects] + ["      </rects></_>"]
    out += ["  </features>", "</cascade>", "</opencv_storage>", ""]
    Path(path).write_text("\n".join(out))
    return str(path)


@pytest.fixture(scope="module")
def xml():
    """The reference's face cascade when staged, else OpenCV's haarcascade_frontalface_alt as the cv2 package ships it."""
    import cv2
    from face_alignment_cvpr_2012_b200 import workloads as wl
    p = wl.STAGED / "haarcascade_frontalface_alt.xml"
    if not p.exists():
        p = Path(cv2.data.haarcascades) / "haarcascade_frontalface_alt.xml"
    return str(p)


@pytest.fixture(scope="module")
def synth_xml(tmp_path_factory):
    return write_stump_cascade(tmp_path_factory.mktemp("cascade") / "stumps_20x20.xml")


@pytest.fixture(scope="module")
def flat_xml(tmp_path_factory):
    """A 20 x 4 window: clipped at the bottom border, its enlarged box scales to a face shorter than a 31-px patch (a square window
    never does: its enlarged box is at least as tall as the window)."""
    return write_stump_cascade(tmp_path_factory.mktemp("cascade") / "stumps_20x4.xml", 20, 4, (3, 5), seed=3)


def _textured(n, rows, cols, seed):
    import cv2
    rng = np.random.default_rng(seed)
    return np.stack([cv2.GaussianBlur(rng.integers(0, 256, (rows, cols, 3), dtype=np.uint8), (0, 0), 1.5) for _ in range(n)])


@pytest.fixture(scope="module")
def gpu_ctx(crf):
    if crf.lib().crf_device_count() < 1:
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box (there is no CPU fallback)")
    return crf.Context(None, 0)


def _ptrs(frames):
    return (C.c_void_p * max(len(frames), 1))(*[f.ctypes.data for f in frames])


def detect_one(crf, ctx, cas, frame, sf=1.3, mn=1, ms=30):
    L = crf.lib()
    rows, cols = frame.shape[:2]
    args = (ctx.h, cas.h, crf.capi.ptr(frame, C.c_uint8), rows, cols, cols * 3, sf, mn, ms)
    n = L.crf_detect_faces(*args, None, 0)
    assert n >= 0, crf.lib().crf_last_error()
    out = (crf.Rect * max(n, 1))()
    assert L.crf_detect_faces(*args, out, n) == n
    return [(r.x, r.y, r.width, r.height) for r in out[:n]]


def detect_batch(crf, ctx, cas, frames, sf=1.3, mn=1, ms=30, cap=None, ptrs=None, step=None):
    """(total, boxes of the first min(total, cap), their frames)"""
    L = crf.lib()
    rows, cols = frames[0].shape[:2] if len(frames) else (1, 1)
    ptrs = _ptrs(frames) if ptrs is None else ptrs
    args = (ctx.h, cas.h, ptrs, len(frames), rows, cols, step or cols * 3, sf, mn, ms)
    if cap is None:
        cap = L.crf_detect_faces_batch(*args, None, None, 0)
        assert cap >= 0, L.crf_last_error()
    out, iob = (crf.Rect * max(cap, 1))(), np.full(max(cap, 1), -1, np.int32)
    n = L.crf_detect_faces_batch(*args, out, crf.capi.ptr(iob, C.c_int32), cap)
    assert n >= 0, L.crf_last_error()
    k = min(n, cap)
    return n, [(r.x, r.y, r.width, r.height) for r in out[:k]], iob[:k].tolist()


def per_frame(crf, ctx, cas, frames, **kw):
    boxes, iob = [], []
    for i, f in enumerate(frames):
        b = detect_one(crf, ctx, cas, np.ascontiguousarray(f), **kw)
        boxes += b; iob += [i] * len(b)
    return boxes, iob


# ---- CPU -----------------------------------------------------------------------------------------------------------------------------
def test_synthetic_cascade_parses_and_finds_candidates(crf, synth_xml, flat_xml):
    """The writer's XML reads to the same sizes in the product's parser and the oracle's, and the oracle finds candidates with it on the
    textured test frames (so the GPU comparisons below cannot pass on empty lists)."""
    from oracle import haar as H
    from oracle import oracle as O
    for path, sizes in ((synth_xml, [20, 20, 5, 29]), (flat_xml, [20, 4, 2, 8])):
        c = H.Cascade(path)
        cc = crf.CascadeClassifier(path)
        assert not cc.empty()
        vals = [C.c_int() for _ in range(4)]
        assert crf.lib().crf_cascade_info(cc.h, *[C.byref(v) for v in vals]) == 0
        assert [v.value for v in vals] == [c.w, c.h, len(c.stages), sum(len(x) for _, x in c.stages)] == sizes
    c = H.Cascade(synth_xml)
    gray = O.bgr2gray(_textured(1, 240, 320, 5)[0])
    cand = H.detect_candidates(c, gray, 1.3, 0)
    assert len(cand) > 20
    assert len(H.detect_multi_scale(c, gray, 1.3, 1, 0)) > 0


# ---- GPU -----------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("which", ["face", "synthetic"])
@pytest.mark.parametrize("min_neighbors", [0, 1])
def test_batch_equals_frame_by_frame(crf, gpu_ctx, xml, synth_xml, which, min_neighbors):
    from face_alignment_cvpr_2012_b200 import workloads as wl
    cas = crf.CascadeClassifier(xml if which == "face" else synth_xml)
    ms = 30
    sets = [wl.make_frames(3, 480, 640, 6, seed=21)[0], wl.make_frames(2, 1080, 1920, 12, seed=22)[0],
            _textured(3, 240, 320, 5), np.zeros((2, 200, 300, 3), np.uint8)]
    rng = np.random.default_rng(9)
    sets.append(rng.integers(0, 256, (2, 300, 400, 3), dtype=np.uint8))
    found = 0
    for frames in sets:
        want_boxes, want_iob = per_frame(crf, gpu_ctx, cas, frames, mn=min_neighbors, ms=ms)
        n, boxes, iob = detect_batch(crf, gpu_ctx, cas, frames, mn=min_neighbors, ms=ms)
        assert n == len(want_boxes) and boxes == want_boxes and iob == want_iob, frames.shape
        found += n
    if which == "synthetic":
        assert found > 0
        # the oracle is independent of the CUDA code: raw candidates and grouped boxes of the textured frames
        from oracle import haar as H
        from oracle import oracle as O
        c = H.Cascade(synth_xml)
        frames = sets[2]
        _, boxes, iob = detect_batch(crf, gpu_ctx, cas, frames, mn=min_neighbors, ms=ms)
        for i, f in enumerate(frames):
            gray = O.bgr2gray(f)
            ref = H.detect_candidates(c, gray, 1.3, ms) if min_neighbors == 0 else H.detect_multi_scale(c, gray, 1.3, min_neighbors, ms)
            assert [b for b, k in zip(boxes, iob) if k == i] == [tuple(int(v) for v in r) for r in ref]


@pytest.mark.gpu
def test_staged_faces_in_one_call(crf, gpu_ctx, xml, lfw_faces):
    """The 20 LFW images (250 x 250) in one call give the boxes crf_detect_faces gives and test_haar pins: one face each."""
    frames = np.stack([f["img"] for f in lfw_faces])
    cas = crf.CascadeClassifier(xml)
    per = cas.detectMultiScaleBatch(gpu_ctx, frames, 1.3, 1, (30, 30))
    assert len(per) == 20 and all(len(p) == 1 for p in per)
    assert per == [cas.detectMultiScale(gpu_ctx, f, 1.3, 1, (30, 30)) for f in frames]


def _analysable(box):
    """The analysis path's box checks (crf_analyze_faces fails the whole call on a box that fails them)."""
    x, y, w, h = box
    if w <= 0 or h <= 0:
        return False
    scale = np.float32(125) / np.float32(w)
    sw, sh = int(np.float32(w) * scale), int(np.float32(h) * scale)
    return 31 < sw <= 125 and 31 < sh <= 521


def _recs_equal(a, b):
    return a.tobytes() == b.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("ms_mode", ["exact", "fast"])
def test_analyze_images_equals_analyze_faces(crf, synth_models, xml, synth_xml, flat_xml, ms_mode):
    """Records of crf_analyze_images equal crf_analyze_faces on the enlarged detections of each frame, every field bitwise.  Boxes the
    analysis path rejects come back with CRF_FACE_NOT_ANALYSED, a zero record and the expected box; the flat synthetic cascade with
    min_neighbors 0 puts windows on the bottom border, so such boxes do occur."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    from oracle import haar as H
    gm, _ = synth_models
    ctx = crf.Context(gm, 0, crf._options(None, ms_mode=ms_mode))
    L = crf.lib()
    cases = [(xml, wl.make_frames(3, 480, 640, 6, seed=31)[0], 1, 30), (synth_xml, _textured(2, 160, 200, 8), 1, 0),
             (flat_xml, _textured(3, 90, 160, 12), 0, 0)]
    rejected = analysed = 0
    for path, frames, mn, ms in cases:
        cas = crf.CascadeClassifier(path)
        rows, cols = frames.shape[1:3]
        args = (ctx.h, cas.h, _ptrs(frames), len(frames), rows, cols, cols * 3, 1.3, mn, ms)
        n = L.crf_detect_faces_batch(*args, None, None, 0)
        boxes, iob, recs = (crf.Rect * max(n, 1))(), np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1), crf.FACE_DTYPE)
        assert L.crf_analyze_images(*args, boxes, crf.capi.ptr(iob, C.c_int32), recs.ctypes.data, n) == n, L.crf_last_error()
        got = [(b.x, b.y, b.width, b.height) for b in boxes[:n]]
        k = 0
        for i, f in enumerate(frames):
            want = H.enlarge(detect_one(crf, ctx, cas, f, mn=mn, ms=ms), rows, cols)
            assert got[k:k + len(want)] == want and iob[k:k + len(want)].tolist() == [i] * len(want)
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
        assert k == n
    assert analysed > 0 and rejected > 0


@pytest.mark.gpu
def test_batching_is_real(crf, synth_models, gpu_ctx, synth_xml):
    """Eight frames cost the launches of one, and crf_analyze_images uploads each frame once plus the face descriptors."""
    L = crf.lib()
    cas = crf.CascadeClassifier(synth_xml)
    frames = _textured(8, 240, 320, 14)

    def launches(fr):
        gpu_ctx.reset_counters()
        detect_batch(crf, gpu_ctx, cas, fr, mn=1, ms=0, cap=0)
        return gpu_ctx.counters()["kernel_launches"]

    one, eight = launches(frames[:1]), launches(frames)
    assert one == eight and one > 0
    gm, _ = synth_models
    ctx = crf.Context(gm, 0)
    rows, cols = frames.shape[1:3]
    # sizeof(FaceDesc), from crf_analyze_faces on a pageable frame: one descriptor + the box's pixels packed to 16 bytes
    ctx.reset_counters()
    ctx.analyze_faces(frames[0], [(10, 10, 100, 120)])
    desc = ctx.counters()["h2d_bytes"] - ((100 * 120 * 3 + 15) & ~15)
    args = (ctx.h, cas.h, _ptrs(frames), len(frames), rows, cols, cols * 3, 1.3, 1, 0)
    n = L.crf_detect_faces_batch(*args, None, None, 0)
    boxes, iob, recs = (crf.Rect * max(n, 1))(), np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1), crf.FACE_DTYPE)
    ctx.reset_counters()
    assert L.crf_analyze_images(*args, boxes, crf.capi.ptr(iob, C.c_int32), recs.ctypes.data, n) == n > 0
    n_analysed = int((recs[:n]["flags"] & crf.capi.FACE_NOT_ANALYSED == 0).sum())
    assert ctx.counters()["h2d_bytes"] == len(frames) * rows * cols * 3 + n_analysed * desc


@pytest.mark.gpu
def test_edge_cases_and_switching(crf, gpu_ctx, xml, synth_xml):
    L = crf.lib()
    syn, face = crf.CascadeClassifier(synth_xml), crf.CascadeClassifier(xml)
    frames = _textured(5, 120, 160, 17)
    want_boxes, want_iob = per_frame(crf, gpu_ctx, syn, frames, mn=0, ms=0)
    assert len(want_boxes) > 10
    # no frames; frames smaller than any window; min_size above the frame
    assert detect_batch(crf, gpu_ctx, syn, [], mn=0, ms=0)[0] == 0
    assert detect_batch(crf, gpu_ctx, syn, _textured(3, 15, 15, 1), mn=0, ms=0)[0] == 0
    assert detect_batch(crf, gpu_ctx, syn, frames, mn=0, ms=200)[0] == 0
    # cap = 0 counts; a smaller cap writes the first cap boxes and still returns the total
    assert detect_batch(crf, gpu_ctx, syn, frames, mn=0, ms=0, cap=0)[0] == len(want_boxes)
    n, boxes, iob = detect_batch(crf, gpu_ctx, syn, frames, mn=0, ms=0, cap=7)
    assert n == len(want_boxes) and boxes == want_boxes[:7] and iob == want_iob[:7]
    # pinned and pageable frames mixed
    p = C.c_void_p()
    crf.capi.check(L.crf_host_alloc(C.byref(p), frames[0].nbytes * 3))
    try:
        ptrs = _ptrs(frames)
        for k in (0, 1, 3):   # frames 0 and 1 adjacent in pinned memory, 3 on its own
            dst = p.value + frames[0].nbytes * (k if k < 2 else 2)
            C.memmove(dst, frames[k].ctypes.data, frames[k].nbytes)
            ptrs[k] = dst
        n, boxes, iob = detect_batch(crf, gpu_ctx, syn, frames, mn=0, ms=0, ptrs=ptrs)
        assert (boxes, iob) == (want_boxes, want_iob)
    finally:
        L.crf_host_free(p)
    # two cascades alternating on one context (the device cascade cache follows the cascade of the call)
    want_face = per_frame(crf, gpu_ctx, face, frames, mn=0, ms=0)
    for _ in range(2):
        assert detect_batch(crf, gpu_ctx, face, frames, mn=0, ms=0)[1:] == want_face
        assert detect_batch(crf, gpu_ctx, syn, frames, mn=0, ms=0)[1:] == (want_boxes, want_iob)
    # more frames than one group holds: equal to calling them a group at a time
    many = _textured(150, 120, 160, 23)
    n, boxes, iob = detect_batch(crf, gpu_ctx, syn, many, mn=1, ms=0)
    parts_b, parts_i = [], []
    for g0 in range(0, 150, 50):
        _, b, i = detect_batch(crf, gpu_ctx, syn, many[g0:g0 + 50], mn=1, ms=0)
        parts_b += b; parts_i += [g0 + v for v in i]
    assert n > 0 and (boxes, iob) == (parts_b, parts_i)
    # bad arguments
    rows, cols = frames.shape[1:3]
    out, iobuf = (crf.Rect * 4)(), np.zeros(4, np.int32)
    good = dict(images=_ptrs(frames), n=len(frames), step=cols * 3, sf=1.3)

    def call(images=good["images"], n=good["n"], step=good["step"], sf=good["sf"], cascade=syn.h, o=out, i=crf.capi.ptr(iobuf, C.c_int32)):
        return L.crf_detect_faces_batch(gpu_ctx.h, cascade, images, n, rows, cols, step, sf, 1, 0, o, i, 4)

    assert call() >= 0
    assert call(images=None) == ERR_ARG
    assert call(cascade=None) == ERR_ARG
    assert call(step=cols * 3 - 1) == ERR_ARG
    assert call(sf=1.0) == ERR_ARG and call(sf=0.5) == ERR_ARG
    assert call(o=None) == ERR_ARG and call(i=None) == ERR_ARG
    null_frame = _ptrs(frames)
    null_frame[2] = None
    assert call(images=null_frame) == ERR_ARG
    assert L.crf_analyze_images(gpu_ctx.h, syn.h, None, 1, rows, cols, cols * 3, 1.3, 1, 0, out, crf.capi.ptr(iobuf, C.c_int32), None, 4) == ERR_ARG


@pytest.mark.gpu
def test_face_forest_analyze_images(crf, synth_models, xml, synth_xml):
    """FaceForest.analyzeImages equals analyzeImage frame by frame (the cascade and options of fd_option)."""
    opt = crf.FaceForestOptions()
    opt.fd_option.path_face_cascade = synth_xml
    opt.fd_option.min_feature_size = 0
    ff = crf.FaceForest(opt, model=synth_models[0])
    assert ff.is_inizialized
    frames = _textured(3, 240, 320, 29)
    per = ff.analyzeImages(frames)
    assert len(per) == 3 and sum(len(p) for p in per) > 0
    for f, faces in zip(frames, per):
        ref = ff.analyzeImage(f)
        assert [x.bbox for x in faces] == [x.bbox for x in ref]
        assert all(_recs_equal(a.record, b.record) for a, b in zip(faces, ref))
    cas = crf.CascadeClassifier(xml)
    assert cas.detectMultiScaleBatch(ff.ctx, frames, 1.3, 1, (30, 30)) == [cas.detectMultiScale(ff.ctx, f, 1.3, 1, (30, 30)) for f in frames]
