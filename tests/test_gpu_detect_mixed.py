"""Detection and alignment across frames of different sizes in one call: crf_detect_faces_batch_mixed, crf_analyze_images_mixed,
crf_analyze_batch_mixed and crf_multi_analyze_batch_mixed.

Each frame is described by its own (bgr, rows, cols, step).  Frame by frame, the mixed calls must give exactly what crf_detect_faces /
crf_analyze_faces give on that frame alone, and on equal-size frames exactly what the equal-size batch calls give."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_detect_batch import _analysable, _recs_equal, _textured, detect_one, write_stump_cascade

ERR_ARG = -1


@pytest.fixture(scope="module")
def xml():
    """The reference's face cascade when staged, else OpenCV's haarcascade_frontalface_alt as the cv2 package ships it."""
    from pathlib import Path

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
    """20 x 4 window: boxes on the bottom border that the analysis path rejects (see test_gpu_detect_batch.flat_xml)."""
    return write_stump_cascade(tmp_path_factory.mktemp("cascade") / "stumps_20x4.xml", 20, 4, (3, 5), seed=3)


@pytest.fixture(scope="module")
def gpu_ctx(crf):
    if crf.lib().crf_device_count() < 1:
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box (there is no CPU fallback)")
    return crf.Context(None, 0)


def padded(frame, pad=23):
    """frame as a view into rows of (cols + pad) pixels: step > cols * 3"""
    rows, cols = frame.shape[:2]
    buf = np.full((rows, cols + pad, 3), 77, np.uint8)
    buf[:, :cols] = frame
    return buf[:, :cols]


def images(crf, frames):
    """crf_image_t descriptors (each frame's own rows, cols and row step)"""
    return (crf.capi.Image * max(len(frames), 1))(*[crf.capi.Image(f.ctypes.data, f.shape[0], f.shape[1], f.strides[0]) for f in frames])


@pytest.fixture(scope="module")
def mixed():
    """Frames of the mixed lists: video frames with faces, textured frames, a zero and a noise frame, a frame smaller than any window
    and a frame with padded rows."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    rng = np.random.default_rng(9)
    return {"480p": wl.make_frames(1, 480, 640, 6, seed=21)[0][0], "1080p": wl.make_frames(1, 1080, 1920, 12, seed=22)[0][0],
            "tex240": _textured(1, 240, 320, 5)[0], "tex97": _textured(1, 97, 131, 6)[0], "zero": np.zeros((200, 300, 3), np.uint8),
            "noise": rng.integers(0, 256, (300, 400, 3), dtype=np.uint8), "tiny": _textured(1, 15, 15, 1)[0],
            "padded": padded(_textured(1, 130, 170, 7)[0])}


ORDER = ["tex240", "480p", "tiny", "tex97", "padded", "1080p", "zero", "tex97", "noise", "tex240"]


def detect_mixed(crf, ctx, cas, frames, sf=1.3, mn=1, ms=30, cap=None):
    """(total, boxes of the first min(total, cap), their frames)"""
    L = crf.lib()
    args = (ctx.h, cas.h, images(crf, frames), len(frames), sf, mn, ms)
    if cap is None:
        cap = L.crf_detect_faces_batch_mixed(*args, None, None, 0)
        assert cap >= 0, L.crf_last_error()
    out, iob = (crf.Rect * max(cap, 1))(), np.full(max(cap, 1), -1, np.int32)
    n = L.crf_detect_faces_batch_mixed(*args, out, crf.capi.ptr(iob, C.c_int32), cap)
    assert n >= 0, L.crf_last_error()
    k = min(n, cap)
    return n, [(r.x, r.y, r.width, r.height) for r in out[:k]], iob[:k].tolist()


def per_frame(crf, ctx, cas, frames, **kw):
    boxes, iob = [], []
    for i, f in enumerate(frames):
        b = detect_one(crf, ctx, cas, np.ascontiguousarray(f), **kw)
        boxes += b; iob += [i] * len(b)
    return boxes, iob


def analyze_images_mixed(crf, ctx, cas, frames, mn, ms):
    L = crf.lib()
    args = (ctx.h, cas.h, images(crf, frames), len(frames), 1.3, mn, ms)
    n = L.crf_detect_faces_batch_mixed(*args, None, None, 0)
    assert n >= 0, L.crf_last_error()
    boxes, iob, recs = (crf.Rect * max(n, 1))(), np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1), crf.FACE_DTYPE)
    assert L.crf_analyze_images_mixed(*args, boxes, crf.capi.ptr(iob, C.c_int32), recs.ctypes.data, n) == n, L.crf_last_error()
    return [(b.x, b.y, b.width, b.height) for b in boxes[:n]], iob[:n].tolist(), recs[:n]


def analyze_batch_mixed(crf, ctx, frames, boxes, iob):
    L = crf.lib()
    n = len(boxes)
    rects = (crf.Rect * max(n, 1))(*[crf.Rect(*map(int, b)) for b in boxes])
    iob = np.ascontiguousarray(iob, np.int32)
    out = np.zeros(max(n, 1), crf.FACE_DTYPE)
    assert L.crf_analyze_batch_mixed(ctx.h, images(crf, frames), len(frames), rects, crf.capi.ptr(iob, C.c_int32), n, out.ctypes.data) == 0, \
        L.crf_last_error()
    return out[:n]


# ---- 1. detection equals frame by frame ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("which", ["face", "synthetic"])
@pytest.mark.parametrize("min_neighbors", [0, 1])
def test_mixed_detection_equals_frame_by_frame(crf, gpu_ctx, xml, synth_xml, mixed, which, min_neighbors):
    cas = crf.CascadeClassifier(xml if which == "face" else synth_xml)
    ms = 30
    frames = [mixed[k] for k in ORDER]
    want_boxes, want_iob = per_frame(crf, gpu_ctx, cas, frames, mn=min_neighbors, ms=ms)
    n, boxes, iob = detect_mixed(crf, gpu_ctx, cas, frames, mn=min_neighbors, ms=ms)
    assert n == len(want_boxes) and boxes == want_boxes and iob == want_iob
    assert ORDER.index("tiny") not in iob
    if which == "synthetic":
        assert n > 0
        # the oracle is independent of the CUDA code: raw candidates and grouped boxes of the textured frames
        from oracle import haar as H
        from oracle import oracle as O
        c = H.Cascade(synth_xml)
        for i, k in enumerate(ORDER):
            if not k.startswith("tex") and k != "padded":
                continue
            gray = O.bgr2gray(np.ascontiguousarray(frames[i]))
            ref = H.detect_candidates(c, gray, 1.3, ms) if min_neighbors == 0 else H.detect_multi_scale(c, gray, 1.3, min_neighbors, ms)
            assert [b for b, f in zip(boxes, iob) if f == i] == [tuple(int(v) for v in r) for r in ref], k


# ---- 2. equal sizes through the mixed calls ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_equal_sizes_through_mixed(crf, synth_models, synth_xml):
    from face_alignment_cvpr_2012_b200 import workloads as wl
    L = crf.lib()
    gm, _ = synth_models
    ctx = crf.Context(gm, 0)
    cas = crf.CascadeClassifier(synth_xml)
    frames = _textured(4, 120, 160, 31)
    rows, cols = frames.shape[1:3]
    ptrs = (C.c_void_p * len(frames))(*[f.ctypes.data for f in frames])
    eq = (ctx.h, cas.h, ptrs, len(frames), rows, cols, cols * 3, 1.3, 1, 0)
    n = L.crf_detect_faces_batch(*eq, None, None, 0)
    assert n > 0
    out, iob = (crf.Rect * n)(), np.zeros(n, np.int32)
    assert L.crf_detect_faces_batch(*eq, out, crf.capi.ptr(iob, C.c_int32), n) == n
    assert detect_mixed(crf, ctx, cas, list(frames), mn=1, ms=0) == (n, [(r.x, r.y, r.width, r.height) for r in out], iob.tolist())
    boxes, iob2, recs = (crf.Rect * n)(), np.zeros(n, np.int32), np.zeros(n, crf.FACE_DTYPE)
    assert L.crf_analyze_images(*eq, boxes, crf.capi.ptr(iob2, C.c_int32), recs.ctypes.data, n) == n
    got_b, got_i, got_r = analyze_images_mixed(crf, ctx, cas, list(frames), 1, 0)
    assert got_b == [(b.x, b.y, b.width, b.height) for b in boxes] and got_i == iob2.tolist() and _recs_equal(got_r, recs)
    vf, vboxes, viob, _ = wl.make_frames(3, 480, 640, 6, seed=33)
    want = ctx.analyze_batch(vf, vboxes, viob)   # equal-size frames of an array go through crf_analyze_batch_mixed too
    vptrs = (C.c_void_p * 3)(*[f.ctypes.data for f in vf])
    rects = (crf.Rect * len(vboxes))(*[crf.Rect(*map(int, b)) for b in vboxes])
    recs = np.zeros(len(vboxes), crf.FACE_DTYPE)
    assert L.crf_analyze_batch(ctx.h, vptrs, 3, 480, 640, 640 * 3, rects, crf.capi.ptr(np.ascontiguousarray(viob, np.int32), C.c_int32),
                               len(vboxes), recs.ctypes.data) == 0
    assert _recs_equal(recs, want) and _recs_equal(analyze_batch_mixed(crf, ctx, list(vf), vboxes, viob), want)


# ---- 3. crf_analyze_images_mixed against crf_analyze_faces ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("ms_mode", ["exact", "fast"])
def test_analyze_images_mixed_equals_analyze_faces(crf, synth_models, xml, synth_xml, flat_xml, ms_mode):
    from face_alignment_cvpr_2012_b200 import workloads as wl
    from oracle import haar as H
    gm, _ = synth_models
    ctx = crf.Context(gm, 0, crf._options(None, ms_mode=ms_mode))
    cases = [(xml, [wl.make_frames(1, 480, 640, 6, seed=31)[0][0], wl.make_frames(1, 720, 1280, 8, seed=32)[0][0]], 1, 30),
             (synth_xml, [_textured(1, 160, 200, 8)[0], padded(_textured(1, 120, 250, 9)[0]), _textured(1, 15, 15, 2)[0]], 1, 0),
             (flat_xml, [_textured(1, 90, 160, 12)[0], _textured(1, 70, 120, 13)[0], padded(_textured(1, 100, 140, 14)[0])], 0, 0)]
    rejected = analysed = 0
    for path, frames, mn, ms in cases:
        cas = crf.CascadeClassifier(path)
        got, iob, recs = analyze_images_mixed(crf, ctx, cas, frames, mn, ms)
        k = 0
        for i, f in enumerate(frames):
            rows, cols = f.shape[:2]
            want = H.enlarge(detect_one(crf, ctx, cas, np.ascontiguousarray(f), mn=mn, ms=ms), rows, cols)
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
        assert k == len(got)
    assert analysed > 0 and rejected > 0


# ---- 4. crf_analyze_batch_mixed against crf_analyze_faces ----------------------------------------------------------------------------
def _pinned_copies(crf, frames, which):
    """frames with those in `which` moved into one pinned host block (adjacent when consecutive); returns (frames, free)"""
    L = crf.lib()
    total = sum(frames[k].nbytes for k in which)
    p = C.c_void_p()
    crf.capi.check(L.crf_host_alloc(C.byref(p), max(total, 1)))
    out, off = list(frames), 0
    for k in which:
        a = np.ctypeslib.as_array((C.c_uint8 * frames[k].nbytes).from_address(p.value + off)).reshape(frames[k].shape)
        a[...] = frames[k]
        out[k] = a
        off += frames[k].nbytes
    return out, lambda: L.crf_host_free(p)


@pytest.mark.gpu
def test_analyze_batch_mixed_equals_analyze_faces(crf, synth_models):
    from face_alignment_cvpr_2012_b200 import workloads as wl
    gm, _ = synth_models
    ctx = crf.Context(gm, 0)
    small = crf.Context(gm, 0, crf._options(None, max_chunk=7))
    data, _ = wl.make_mixed(10)
    frames = [np.ascontiguousarray(f) for f, _ in data]
    per_image = [ctx.analyze_faces(f, b) for f, b in data]
    flat, first = np.concatenate(per_image), np.cumsum([0] + [len(r) for r in per_image])
    # boxes interleaved across frames; frame 3 is named twice (entries 3 and 10 describe the same pixels)
    frames.append(frames[3])
    items = [(i, j) for i, (_, b) in enumerate(data) for j in range(len(b))] + [(10, j) for j in range(len(data[3][1]))]
    rng = np.random.default_rng(4)
    items = [items[k] for k in rng.permutation(len(items))]
    boxes = [data[3 if i == 10 else i][1][j] for i, j in items]
    want = flat[[first[3 if i == 10 else i] + j for i, j in items]]
    for c in (ctx, small):
        assert _recs_equal(analyze_batch_mixed(crf, c, frames, boxes, [i for i, _ in items]), want)
    # dense boxes on the small frames (frame mode once every frame is pinned) ahead of the sparse 4K boxes (ROI mode)
    dense = [(i, (x, y, 260, 300)) for i in (0, 5) for x in range(0, 380, 60) for y in (0, 90, 180)]
    sparse = [(i, tuple(b)) for i in (4, 9) for b in data[i][1]]
    both = dense + sparse
    d_want = np.concatenate([ctx.analyze_faces(frames[i], [b]) for i, b in both])
    d_boxes, d_iob = [b for _, b in both], [i for i, _ in both]
    pinned, free = _pinned_copies(crf, frames, range(len(data)))
    try:
        for c in (ctx, small):
            assert _recs_equal(analyze_batch_mixed(crf, c, pinned[:len(data)], d_boxes, d_iob), d_want)
    finally:
        free()
    # pinned and pageable frames mixed
    half, free = _pinned_copies(crf, frames, [0, 1, 2, 4])
    try:
        for c in (ctx, small):
            assert _recs_equal(analyze_batch_mixed(crf, c, half, boxes, [i for i, _ in items]), want)
            assert _recs_equal(analyze_batch_mixed(crf, c, half[:len(data)], d_boxes, d_iob), d_want)
    finally:
        free()
    mc = crf.MultiContext(gm, [0, 0])
    assert _recs_equal(mc.analyze_batch(frames, boxes, [i for i, _ in items]), want)
    assert _recs_equal(mc.analyze_batch(frames[:len(data)], d_boxes, d_iob), d_want)


@pytest.mark.gpu
def test_analyze_batch_mixed_frame_mode(crf, synth_models):
    """Dense boxes on pinned frames of three sizes in one chunk: the frames go up whole (frame mode), each at its own slot offset.  Frames
    adjacent in one pinned block (one copy) and in separate blocks; records bitwise equal to crf_analyze_faces per frame."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    gm, _ = synth_models
    ctx = crf.Context(gm, 0)
    chunked = crf.Context(gm, 0, crf._options(None, max_chunk=40))
    data, _ = wl.make_mixed(3)   # 480 x 640, 720 x 1280, 1080 x 1920
    frames = [np.ascontiguousarray(f) for f, _ in data]
    per = [[(i, (x, y, 260, 300)) for x in range(0, f.shape[1] - 259, 120) for y in range(0, f.shape[0] - 299, 120)] for i, f in enumerate(frames)]
    both = [b for k in range(max(map(len, per))) for p in per if k < len(p) for b in [p[k]]]   # interleaved across the frames
    assert len({i for i, _ in both[:40]}) == 3
    want = np.concatenate([ctx.analyze_faces(frames[i], [b]) for i, b in both])
    boxes, iob = [b for _, b in both], [i for i, _ in both]
    ctx.reset_counters()
    ctx.analyze_faces(frames[0], [(10, 10, 100, 120)])
    desc = ctx.counters()["h2d_bytes"] - ((100 * 120 * 3 + 15) & ~15)
    block, free = _pinned_copies(crf, frames, [0, 1, 2])
    try:
        ctx.reset_counters()
        assert _recs_equal(analyze_batch_mixed(crf, ctx, block, boxes, iob), want)
        # the whole frames went up, not the boxes' pixels
        assert ctx.counters()["h2d_bytes"] == sum(f.nbytes for f in frames) + len(boxes) * desc
        assert _recs_equal(analyze_batch_mixed(crf, chunked, block, boxes, iob), want)
    finally:
        free()
    sep = list(frames)
    frees = []
    try:
        for k in (2, 0, 1):
            one, fr = _pinned_copies(crf, frames, [k])
            sep[k] = one[k]; frees.append(fr)
        ctx.reset_counters()
        assert _recs_equal(analyze_batch_mixed(crf, ctx, sep, boxes, iob), want)
        assert ctx.counters()["h2d_bytes"] == sum(f.nbytes for f in frames) + len(boxes) * desc
        assert _recs_equal(analyze_batch_mixed(crf, chunked, sep, boxes, iob), want)
    finally:
        for fr in frees:
            fr()


# ---- 5. batching is real -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_mixed_batching_is_real(crf, synth_models, gpu_ctx, synth_xml):
    """A group of 8 frames of 5 sizes costs the launches of one frame, and crf_analyze_images_mixed uploads each frame once plus the
    descriptors of the analysed faces."""
    L = crf.lib()
    cas = crf.CascadeClassifier(synth_xml)
    sizes = [(240, 320), (120, 160), (97, 131), (200, 300), (64, 80), (240, 320), (97, 131), (120, 160)]
    frames = [_textured(1, r, c, 40 + k)[0] for k, (r, c) in enumerate(sizes)]
    frames[3] = padded(frames[3], 5)

    def launches(fr):
        gpu_ctx.reset_counters()
        detect_mixed(crf, gpu_ctx, cas, fr, mn=1, ms=0, cap=0)
        return gpu_ctx.counters()["kernel_launches"]

    one, eight = launches(frames[:1]), launches(frames)
    assert one == eight and one > 0
    gm, _ = synth_models
    ctx = crf.Context(gm, 0)
    ctx.reset_counters()
    ctx.analyze_faces(frames[0], [(10, 10, 100, 120)])
    desc = ctx.counters()["h2d_bytes"] - ((100 * 120 * 3 + 15) & ~15)
    args = (ctx.h, cas.h, images(crf, frames), len(frames), 1.3, 1, 0)
    n = L.crf_detect_faces_batch_mixed(*args, None, None, 0)
    boxes, iob, recs = (crf.Rect * max(n, 1))(), np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1), crf.FACE_DTYPE)
    ctx.reset_counters()
    assert L.crf_analyze_images_mixed(*args, boxes, crf.capi.ptr(iob, C.c_int32), recs.ctypes.data, n) == n > 0
    recs = recs[:n]
    n_analysed = int((recs["flags"] & crf.capi.FACE_NOT_ANALYSED == 0).sum())
    assert n_analysed > 0
    assert ctx.counters()["h2d_bytes"] == sum(f.shape[0] * f.strides[0] for f in frames) + n_analysed * desc


# ---- 6. groups -----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_mixed_groups(crf, gpu_ctx, synth_xml):
    cas = crf.CascadeClassifier(synth_xml)
    sizes = [(120, 160), (100, 140), (90, 130), (110, 120), (64, 100)]
    many = [_textured(1, *sizes[k % len(sizes)], 100 + k)[0] for k in range(150)]
    n, boxes, iob = detect_mixed(crf, gpu_ctx, cas, many, mn=1, ms=0)
    parts_b, parts_i = [], []
    for g0 in range(0, 150, 50):
        _, b, i = detect_mixed(crf, gpu_ctx, cas, many[g0:g0 + 50], mn=1, ms=0)
        parts_b += b; parts_i += [g0 + v for v in i]
    assert n > 0 and (boxes, iob) == (parts_b, parts_i)


# ---- 7. bad arguments ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_mixed_bad_arguments(crf, synth_models, synth_xml):
    L = crf.lib()
    gm, _ = synth_models
    ctx = crf.Context(gm, 0)
    cas = crf.CascadeClassifier(synth_xml)
    frames = [_textured(1, 120, 160, 51)[0], _textured(1, 60, 80, 52)[0], _textured(1, 90, 100, 53)[0]]
    cap = 4
    out, iob, recs = (crf.Rect * cap)(), np.full(cap, -7, np.int32), np.zeros(cap, crf.FACE_DTYPE)

    def untouched():
        return all((r.x, r.y, r.width, r.height) == (-5, -5, -5, -5) for r in out) and (iob == -7).all() and (recs["flags"] == 99).all()

    def reset():
        for r in out:
            r.x = r.y = r.width = r.height = -5
        iob[:] = -7
        recs[:] = np.zeros(1, crf.FACE_DTYPE)[0]
        recs["flags"] = 99

    def detect(im, n=3, sf=1.3):
        return L.crf_detect_faces_batch_mixed(ctx.h, cas.h, im, n, sf, 0, 0, out, crf.capi.ptr(iob, C.c_int32), cap)

    def analyze(im, n=3, sf=1.3):
        return L.crf_analyze_images_mixed(ctx.h, cas.h, im, n, sf, 0, 0, out, crf.capi.ptr(iob, C.c_int32), recs.ctypes.data, cap)

    def batch(im, bxs, which, n=3):
        rects = (crf.Rect * len(bxs))(*[crf.Rect(*b) for b in bxs])
        w = np.ascontiguousarray(which, np.int32)
        return L.crf_analyze_batch_mixed(ctx.h, im, n, rects, crf.capi.ptr(w, C.c_int32), len(bxs), recs.ctypes.data)

    def multi(im, bxs, which, n=3):
        rects = (crf.Rect * len(bxs))(*[crf.Rect(*b) for b in bxs])
        w = np.ascontiguousarray(which, np.int32)
        return L.crf_multi_analyze_batch_mixed(mc.h, im, n, rects, crf.capi.ptr(w, C.c_int32), len(bxs), recs.ctypes.data)

    mc = crf.MultiContext(gm, [0, 0])   # two shards: a bad box in the second must stop the first from writing
    good_boxes, good_iob = [(0, 0, 60, 60), (10, 5, 50, 50)], [0, 1]
    reset()
    assert batch(images(crf, frames), good_boxes, good_iob) == 0 and not (recs["flags"][:2] == 99).any()
    bad = []
    for field, value in (("bgr", None), ("rows", 0), ("cols", 0), ("step", 80 * 3 - 1)):
        im = images(crf, frames)
        setattr(im[1], field, value)
        bad.append(im)
    for im in bad:
        for call in (lambda: detect(im), lambda: analyze(im), lambda: batch(im, good_boxes, good_iob), lambda: multi(im, good_boxes, good_iob)):
            reset()
            assert call() == ERR_ARG and untouched()
    for call in (lambda: detect(None), lambda: analyze(None), lambda: batch(None, good_boxes, good_iob), lambda: multi(None, good_boxes, good_iob)):
        reset()
        assert call() == ERR_ARG and untouched()
    for sf in (1.0, 0.5):
        for call in (detect, analyze):
            reset()
            assert call(images(crf, frames), sf=sf) == ERR_ARG and untouched()
    for which in ([0, 3], [0, -1]):
        for call in (batch, multi):
            reset()
            assert call(images(crf, frames), good_boxes, which) == ERR_ARG and untouched()
    # (70, 0, 60, 60) fits frame 0 (160 wide) but not frame 1 (80 wide)
    for call in (batch, multi):
        reset()
        assert call(images(crf, frames), [(70, 0, 60, 60)], [0]) == 0
        reset()
        assert call(images(crf, frames), good_boxes + [(70, 0, 60, 60)], good_iob + [1]) == ERR_ARG and untouched()
    # the mixed calls reject a null frame that no box names; the equal-size calls keep accepting one, and keep checking their one
    # geometry when there are no frames
    unnamed = images(crf, frames)
    unnamed[2].bgr = None
    for call in (batch, multi):
        reset()
        assert call(unnamed, good_boxes, good_iob) == ERR_ARG and untouched()
    eq = [frames[0], frames[0], frames[0]]
    ptrs = (C.c_void_p * 3)(*[f.ctypes.data for f in eq])
    ptrs[2] = None
    rects = (crf.Rect * 2)(*[crf.Rect(*b) for b in good_boxes])
    w = np.ascontiguousarray([0, 1], np.int32)
    assert L.crf_analyze_batch(ctx.h, ptrs, 3, 120, 160, 480, rects, crf.capi.ptr(w, C.c_int32), 2, recs.ctypes.data) == 0
    assert L.crf_multi_analyze_batch(mc.h, ptrs, 3, 120, 160, 480, rects, crf.capi.ptr(w, C.c_int32), 2, recs.ctypes.data) == 0
    for rows, cols, step in ((0, 160, 480), (120, 0, 480), (120, 160, 479)):
        assert L.crf_detect_faces_batch(ctx.h, cas.h, ptrs, 0, rows, cols, step, 1.3, 1, 0, out, crf.capi.ptr(iob, C.c_int32), cap) == ERR_ARG
        assert L.crf_analyze_images(ctx.h, cas.h, ptrs, 0, rows, cols, step, 1.3, 1, 0, out, crf.capi.ptr(iob, C.c_int32), recs.ctypes.data,
                                    cap) == ERR_ARG
    # no frames; a small cap
    reset()
    assert detect(images(crf, []), n=0) == 0 and analyze(images(crf, []), n=0) == 0 and untouched()
    n, want_b, want_i = detect_mixed(crf, ctx, cas, frames, mn=0, ms=0)
    assert n > cap
    reset()
    assert detect(images(crf, frames)) == n
    assert [(r.x, r.y, r.width, r.height) for r in out] == want_b[:cap] and iob.tolist() == want_i[:cap]
    reset()
    assert analyze(images(crf, frames)) == n and (iob.tolist() == want_i[:cap]) and not (recs["flags"] == 99).any()


# ---- 8. Python ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_python_mixed_lists(crf, synth_models, xml, synth_xml):
    from face_alignment_cvpr_2012_b200 import workloads as wl
    opt = crf.FaceForestOptions()
    opt.fd_option.path_face_cascade = synth_xml
    opt.fd_option.min_feature_size = 0
    ff = crf.FaceForest(opt, model=synth_models[0])
    assert ff.is_inizialized
    frames = [_textured(1, 240, 320, 61)[0], _textured(1, 130, 150, 62)[0], _textured(1, 15, 15, 63)[0], _textured(1, 180, 200, 64)[0]]
    per = ff.analyzeImages(frames)
    assert len(per) == 4 and sum(len(p) for p in per) > 0 and per[2] == []
    for f, faces in zip(frames, per):
        ref = ff.analyzeImage(f)
        assert [x.bbox for x in faces] == [x.bbox for x in ref]
        assert all(_recs_equal(a.record, b.record) for a, b in zip(faces, ref))
    cas = crf.CascadeClassifier(xml)
    video = [wl.make_frames(1, 480, 640, 6, seed=65)[0][0], wl.make_frames(1, 720, 1280, 8, seed=66)[0][0]]
    assert cas.detectMultiScaleBatch(ff.ctx, video + frames, 1.3, 1, (30, 30)) == [cas.detectMultiScale(ff.ctx, f, 1.3, 1, (30, 30)) for f in video + frames]
    # boxes given: Context / MultiContext.analyze_batch read each frame with its own shape
    data, _ = wl.make_mixed(5)
    fr = [f for f, _ in data][::-1]   # the smallest frame last: frame 0's geometry would misread it
    boxes = [tuple(b) for f, bs in data[::-1] for b in bs]
    iob = [k for k, (f, bs) in enumerate(data[::-1]) for _ in bs]
    want = np.concatenate([ff.ctx.analyze_faces(f, bs) for f, bs in data[::-1]])
    assert _recs_equal(ff.ctx.analyze_batch(fr, boxes, iob), want)
    assert _recs_equal(crf.MultiContext(synth_models[0], [0, 0]).analyze_batch(fr, boxes, iob), want)


@pytest.mark.gpu
def test_cascade_loaded_after_a_free(crf, gpu_ctx, xml, synth_xml, mixed):
    """A context caches the device tables of the last cascade it ran; a cascade loaded after another was freed (typically at the same
    address) must not run with the freed cascade's tables."""
    frame = mixed["tex240"]
    fresh = crf.Context(None, 0)
    want = detect_one(crf, fresh, crf.CascadeClassifier(synth_xml), frame, mn=0, ms=0)
    for _ in range(4):
        face = crf.CascadeClassifier(xml)
        detect_one(crf, gpu_ctx, face, frame, mn=0, ms=0)
        face.close()
        assert detect_one(crf, gpu_ctx, crf.CascadeClassifier(synth_xml), frame, mn=0, ms=0) == want
