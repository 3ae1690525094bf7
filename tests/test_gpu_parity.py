"""GPU: the CUDA path (through the C ABI) against the CPU oracle on the same inputs, stage by stage and end to end.
Bit-exact for every integer / byte / index result (scaled pixels, 8-bit planes, integrals, leaf ids, vote lists,
head pose and its variance, forest composition); MeanShift means within the 0.5 px of the north star (observed: 0.0 px in the
exact mode, <= 0.024 px in the default tolerance mode on a 3543-face campaign)."""
import zlib
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
TOL_PX = 0.5


@pytest.fixture(scope="module")
def gpu(crf):
    if crf.lib().crf_device_count() < 1:
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box (there is no CPU fallback)")
    return True


@pytest.fixture(scope="module")
def sctx(crf, gpu, synth_models):
    return crf.Context(synth_models[0], 0)


@pytest.fixture(scope="module")
def rctx(crf, gpu, staged_models):
    return crf.Context(staged_models[0], 0)


def _planes(rng, C=38, H=125, W=125, smooth=True):
    import cv2
    p = rng.integers(0, 256, (C, H, W), dtype=np.uint8)
    if smooth:
        p = np.stack([cv2.GaussianBlur(q, (0, 0), 2.0) for q in p])
        p = np.clip((p.astype(np.float32) - 128) * 6 + 128, 0, 255).astype(np.uint8)
    return p


# ------------------------------------------------------------------ stages
@pytest.mark.parametrize("shape,box", [((250, 250), (61, 72, 130, 130)), ((97, 143), (3, 5, 100, 90)), ((300, 400), (10, 20, 333, 250)),
                                       ((480, 640), (100, 50, 211, 300)), ((1080, 1920), (700, 200, 507, 611)), ((64, 64), (0, 0, 64, 64))])
def test_gray_resize(O, sctx, shape, box):
    rng = np.random.default_rng(shape[0] * 7 + box[2])
    img = rng.integers(0, 256, shape + (3,), dtype=np.uint8)
    got = sctx.stage_gray_resize(img, box)
    x, y, w, h = box
    sw, sh, _ = O.scaled_size(w, h)
    want = O.resize(O.bgr2gray(img)[y:y + h, x:x + w], sh, sw)
    assert got.shape == want.shape and np.array_equal(got, want)


def test_gray_resize_matches_cv2(sctx, cv2_golden):
    """Directly against cv2 (same image on the GPU box): cvtColor + crop + resize."""
    import cv2
    bgr = cv2_golden["bgr"]
    for box in [(0, 0, 143, 97), (10, 5, 100, 80), (40, 30, 60, 60)]:
        x, y, w, h = box
        g = sctx.stage_gray_resize(bgr, box)
        ref = cv2.resize(cv2_golden["gray"][y:y + h, x:x + w], (g.shape[1], g.shape[0]), interpolation=cv2.INTER_LINEAR)
        assert np.array_equal(g, ref), box


@pytest.mark.parametrize("H,W", [(125, 125), (141, 125), (148, 124), (32, 125), (200, 125)])
def test_channels_bit_exact(O, sctx, H, W):
    import cv2
    rng = np.random.default_rng(H * 1000 + W)
    img = cv2.GaussianBlur(rng.integers(0, 256, (H, W), dtype=np.uint8), (0, 0), 1.2)
    planes, integ = sctx.stage_channels(img)
    op, oi = O.channels(img)
    assert np.array_equal(planes, op)
    assert np.array_equal(integ, oi.astype(np.uint32))
    mm, mi = sctx.stage_channels(img, minmax=True)
    omm, omi = O.channels(img, features_mask=0b1000)
    assert np.array_equal(mm, omm) and np.array_equal(mi, omi.astype(np.uint32))


def test_channels_golden_plane(sctx, cv2_golden):
    """Against cv2 itself: gray integral, Sobel planes and the 7x7 Gabor planes are bit-exact; larger kernels +-1 LSB."""
    img = cv2_golden["plane"]
    planes, integ = sctx.stage_channels(img)
    assert np.array_equal(integ[0], cv2_golden["integral"].astype(np.uint32))
    assert np.array_equal(planes[36], cv2_golden["sobel_dy"]) and np.array_equal(planes[37], cv2_golden["sobel_dx"])
    ref = cv2_golden["gabor_u8_cv2"]
    assert np.array_equal(planes[1:8], ref[:7])
    d = planes[1:36].astype(int) - ref.astype(int)
    assert np.abs(d).max() <= 1 and (d != 0).mean() <= 2e-4


def test_norm_channel(O, sctx, cv2_golden):
    """FC_NORM (cv::equalizeHist + integral) against cv2's own output and the oracle, incl. a constant image."""
    for src, ref in ((cv2_golden["plane"], cv2_golden["equalize"]), (cv2_golden["equalize_src2"], cv2_golden["equalize2"])):
        p, integ = sctx.stage_channels(src, norm=True)
        assert np.array_equal(p[0], ref)
        assert np.array_equal(integ[0], O.channels(src, features_mask=0b100000)[1][0].astype(np.uint32))
    p, _ = sctx.stage_channels(np.full((64, 125), 200, np.uint8), norm=True)
    assert (p[0] == 200).all()


@pytest.mark.parametrize("H,W", [(125, 125), (148, 124), (40, 125), (521, 125)])
def test_canny_channel(O, sctx, cv2_golden, H, W):
    """FC_CANNY as a stage (crf_stage_canny): bit-exact vs the oracle, and vs cv2 on the golden plane."""
    import cv2
    rng = np.random.default_rng(H + W)
    for img in (cv2.GaussianBlur(rng.integers(0, 256, (H, W), dtype=np.uint8), (0, 0), 2.0), rng.integers(0, 256, (H, W), dtype=np.uint8),
                np.zeros((H, W), np.uint8), np.tile(np.arange(W, dtype=np.uint8), (H, 1))):
        planes, integ = sctx.stage_channels(img, canny=True)
        op, oi = O.channels(img, features_mask=16)
        assert np.array_equal(planes, op) and np.array_equal(integ, oi.astype(np.uint32))
    planes, _ = sctx.stage_channels(cv2_golden["plane"], canny=True)
    assert np.array_equal(planes[0], cv2_golden["canny"])


def test_channels_degenerate_images(O, sctx):
    for img in (np.zeros((125, 125), np.uint8), np.full((125, 125), 255, np.uint8), np.tile(np.arange(125, dtype=np.uint8), (125, 1))):
        planes, integ = sctx.stage_channels(img)
        op, oi = O.channels(img)
        assert np.array_equal(planes, op) and np.array_equal(integ, oi.astype(np.uint32))


@pytest.mark.parametrize("stride,H,W", [(4, 125, 125), (3, 125, 125), (1, 125, 125), (4, 148, 124), (3, 33, 125), (2, 190, 125), (7, 125, 125)])
def test_forest_leaf_ids_synthetic_model(O, sctx, synth_models, stride, H, W):
    _, om = synth_models
    rng = np.random.default_rng(stride * 100 + H)
    planes = _planes(rng, 38, H, W)
    s = O.Sample(planes=planes)
    ids_o, hp_o, var_o, _ = om.eval_hp(s, stride)
    assert np.array_equal(sctx.stage_eval_forest(planes, stride), ids_o)
    fi = rng.integers(0, 5, 20); ti = rng.integers(0, 20, 20)
    e = om.eval_ffd(s, fi, ti, stride)
    assert np.array_equal(sctx.stage_eval_forest(planes, stride, fi, ti), e["leaf_ids"])
    s.close()


@pytest.mark.parametrize("win", ["default", "rows", "pairx", "fmt1", "win2_15x2"])
@pytest.mark.parametrize("H,W,nt", [(125, 125, 20), (148, 124, 20), (33, 125, 7), (40, 125, 23), (200, 125, 20), (32, 125, 20), (70, 124, 41)])
def test_window_traversal_forced(O, crf, gpu, synth_models, monkeypatch, H, W, nt, win):
    """k_traverse_win (shared-memory window, ring rows, two walks per lane) on one ragged face: partial tiles right and
    below, heights that need 1..22 tile steps, tree lists shorter / longer than the warps of a CTA, and the counters.
    win: the launch shapes in use — library defaults, two walks per lane on rows ly / ly + 4 (and one walk per lane for
    the head-pose forest), two walks per lane on horizontal neighbours with the shared record fetch (PAIRX)."""
    gm, om = synth_models
    monkeypatch.setenv("CRF_TRAVERSE_VARIANT", "0x100001")
    if win == "rows":
        monkeypatch.setenv("CRF_WIN_HP", str(32 | 1 << 8)); monkeypatch.setenv("CRF_WIN_FFD", str(20 | 2 << 8))
    elif win == "pairx":
        monkeypatch.setenv("CRF_WIN_HP", str(15 | 2 << 8 | 1 << 12)); monkeypatch.setenv("CRF_WIN_FFD", str(20 | 2 << 8 | 1 << 12))
    elif win == "fmt1":   # k_traverse_win on the records that keep leaf slots (the default is k_traverse_win2 on DevSlotN)
        monkeypatch.setenv("CRF_WIN_FMT", "1")
    elif win == "win2_15x2":   # k_traverse_win2 with the pipelined two-walk loop for both forests
        monkeypatch.setenv("CRF_WIN_HP", str(15 | 2 << 8)); monkeypatch.setenv("CRF_WIN_FFD", str(24 | 2 << 8))
    ctx = crf.Context(gm, 0)
    ctx.set_profiling(False, True)
    rng = np.random.default_rng(H * 7 + nt)
    for smooth in (True, False):
        planes = _planes(rng, 38, H, W, smooth=smooth)
        s = O.Sample(planes=planes)
        ctx.reset_counters()
        ids_o, _, _, vis_hp = om.eval_hp(s, 1)
        assert np.array_equal(ctx.stage_eval_forest(planes, 1), ids_o)
        fi = rng.integers(0, 5, nt); ti = rng.integers(0, 20, nt)
        e = om.eval_ffd(s, fi, ti, 1)
        assert np.array_equal(ctx.stage_eval_forest(planes, 1, fi, ti), e["leaf_ids"])
        c = ctx.counters()
        assert c["hp_traversals"] == ids_o.size and c["ffd_traversals"] == e["leaf_ids"].size
        assert c["hp_node_tests"] == vis_hp - ids_o.size and c["ffd_node_tests"] == e["visits"] - e["leaf_ids"].size
        s.close()
    ctx.close()


@pytest.mark.parametrize("depth", [0, 1, 2])
def test_degenerate_forests_through_every_traversal(O, crf, gpu, tmp_path, monkeypatch, depth):
    """Forests of one-leaf trees (depth 0: the root is a leaf, so the internal-nodes-only record array of k_traverse_win2 is empty and the
    root tag is ~leaf), of three-node trees and of depth-2 trees: leaf ids and whole records against the oracle through the window kernels
    (both record formats) and the global-gather kernels."""
    from face_alignment_cvpr_2012_b200 import synthetic_model as sm, workloads as wl
    hp, ffd = sm.write_model(tmp_path / f"d{depth}", seed=40 + depth, hp_depth=depth, ffd_depth=depth)
    gm, om = crf.Model(hp, ffd, 15, 20), O.Model(hp, ffd, 15, 20)
    rng = np.random.default_rng(depth)
    planes = _planes(rng, 38, 125, 125, smooth=True)
    s = O.Sample(planes=planes)
    ids_o, _, _, _ = om.eval_hp(s, 1)
    fi = rng.integers(0, 5, 20); ti = rng.integers(0, 20, 20)
    e = om.eval_ffd(s, fi, ti, 1)
    crops, _ = wl.make_crops(48, seed=5)
    want = [om.analyze_face(c, (0, 0, 100, 100), 1, 1) for c in crops[:3]]
    for env in ({"CRF_TRAVERSE_VARIANT": "0x100001"}, {"CRF_TRAVERSE_VARIANT": "0x100001", "CRF_WIN_FMT": "1"}, {"CRF_TRAVERSE_VARIANT": hex(32 | (4 << 8) | (10 << 16))}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        ctx = crf.Context(gm, 0, crf._options(None, hp_stride=1, ffd_stride=1))
        assert np.array_equal(ctx.stage_eval_forest(planes, 1), ids_o), env
        assert np.array_equal(ctx.stage_eval_forest(planes, 1, fi, ti), e["leaf_ids"]), env
        got = ctx.analyze_crops(crops)
        for i, w in enumerate(want):
            assert got[i]["headpose"] == w["headpose"] and (got[i]["n_votes"] == w["n_votes"]).all() and (got[i]["tree_counts"] == w["tree_counts"]).all(), (env, i)
            assert float(np.nanmax(np.abs(got[i]["ffd_f"] - w["ffd_f"]))) <= 0.5 or not np.isfinite(w["ffd_f"]).all(), (env, i)
        ctx.close()
        for k in env:
            monkeypatch.delenv(k)
    s.close()


def test_window_and_gather_traversals_agree_in_batches(crf, gpu, synth_models, monkeypatch):
    """Whole pipeline at stride 1 on 80 crops: the default (window kernel, persistent CTAs over (face, column) items) against
    the global-gather kernels forced through CRF_TRAVERSE_VARIANT; records must be byte-identical."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    gm, _ = synth_models
    crops, _ = wl.make_crops(80, seed=77)
    got = crf.Context(gm, 0, crf._options(None, hp_stride=1, ffd_stride=1)).analyze_crops(crops)
    monkeypatch.setenv("CRF_TRAVERSE_VARIANT", hex(32 | (4 << 8) | (10 << 16)))
    ref = crf.Context(gm, 0, crf._options(None, hp_stride=1, ffd_stride=1)).analyze_crops(crops)
    assert got.tobytes() == ref.tobytes()


def test_forest_large_rectangles(crf, O, gpu, tmp_path):
    """Rectangles up to 30x30 (area 900): the modulo-2^16 integral layout needs up to 4 strips per rectangle."""
    from face_alignment_cvpr_2012_b200 import synthetic_model as sm
    hp, ffd = sm.write_model(tmp_path / "bigrect", seed=9, hp_depth=9, ffd_depth=9, max_rect=30)
    gm, om = crf.Model(hp, ffd, 15, 20), O.Model(hp, ffd, 15, 20)
    ctx = crf.Context(gm, 0)
    rng = np.random.default_rng(12)
    for planes in (_planes(rng, 38, 125, 125), np.full((38, 125, 125), 255, np.uint8), _planes(rng, 38, 140, 124, smooth=False)):
        s = O.Sample(planes=planes)
        ids_o, _, _, _ = om.eval_hp(s, 2)
        assert np.array_equal(ctx.stage_eval_forest(planes, 2), ids_o)
        fi = rng.integers(0, 5, 20); ti = rng.integers(0, 20, 20)
        assert np.array_equal(ctx.stage_eval_forest(planes, 3, fi, ti), om.eval_ffd(s, fi, ti, 3)["leaf_ids"])
        s.close()


def test_forest_errors(crf, sctx):
    planes = np.zeros((10, 125, 125), np.uint8)
    with pytest.raises(crf.CrfError):  # forests read channels up to 37
        sctx.stage_eval_forest(planes, 4)
    with pytest.raises(crf.CrfError):
        sctx.stage_eval_forest(np.zeros((38, 125, 125), np.uint8), 3, [9], [0])
    # a face no larger than a patch has an empty grid in the reference (face_utils.cpp:200-202): argument error here
    with pytest.raises(crf.CrfError):
        sctx.stage_eval_forest(np.zeros((38, 31, 125), np.uint8), 4)


@pytest.mark.parametrize("stride", [4, 1])
def test_headpose_reduce_and_composition(O, sctx, synth_models, stride):
    _, om = synth_models
    rng = np.random.default_rng(77 + stride)
    for k in range(3):
        planes = _planes(rng, 38, 125 + 10 * k, 125)
        s = O.Sample(planes=planes)
        _, hp_o, var_o, _ = om.eval_hp(s, stride)
        r = sctx.stage_headpose(planes, stride)
        assert r["headpose"] == hp_o and r["variance"] == var_o  # same sequential f32 order
        counts, dom, fi, ti, fl = om.compose(hp_o, var_o)
        assert np.array_equal(r["tree_counts"], counts) and r["dominant"] == dom and r["flags"] == fl
        assert np.array_equal(r["forest_idx"], fi) and np.array_equal(r["tree_idx"], ti)
        s.close()


def test_composition_grid_including_pathological(O, sctx, synth_models):
    """Composition on a grid of (headpose, variance), incl. zero / tiny / negative / NaN variance (SURVEY A.9, E.6, E.7)."""
    _, om = synth_models
    hps = [-2.0, -0.6, -0.35, -0.2, -0.05, 0.0, 0.13, 0.2, 0.35, 0.9, 2.0, float("nan")]
    vars_ = [0.0, 1e-9, 1e-6, 2.5e-5, 1e-4, 0.003, 0.02, 0.05, 0.3, 2.0, -0.01, float("nan"), float("inf")]
    for hp in hps:
        for v in vars_:
            counts, dom, fi, ti, fl = om.compose(np.float32(hp), np.float32(v))
            r = sctx.stage_compose(float(np.float32(hp)), float(np.float32(v)))
            assert np.array_equal(r["tree_counts"], counts), (hp, v, r["tree_counts"], counts)
            assert r["dominant"] == dom and r["flags"] == fl, (hp, v)
            assert np.array_equal(r["forest_idx"], fi) and np.array_equal(r["tree_idx"], ti), (hp, v)


@pytest.mark.parametrize("stride", [3, 1])
def test_votes_and_meanshift(O, sctx, synth_models, stride):
    _, om = synth_models
    rng = np.random.default_rng(5 + stride)
    planes = _planes(rng, 38, 130, 125)
    fi = rng.integers(0, 5, 20); ti = rng.integers(0, 20, 20)
    s = O.Sample(planes=planes)
    cap = 40000 if stride == 1 else 8000
    e = om.eval_ffd(s, fi, ti, stride, vote_cap=cap)
    v = sctx.stage_votes_meanshift(planes, stride, fi, ti, vote_cap=cap)
    assert np.array_equal(v["n_votes"], e["n_votes"]) and e["n_votes"].max() <= cap and e["n_votes"].sum() > 0
    assert np.array_equal(v["votes"], e["votes"])  # same votes in the same order
    assert np.array_equal(v["iters"], e["iters"])
    assert np.abs(v["mean"] - e["mean"]).max() <= TOL_PX
    assert np.abs(v["mean"] - e["mean"]).max() <= 1e-3  # what the exp() difference actually allows
    assert np.abs(v["rounded"] - e["rounded"]).max() <= 1
    s.close()


def test_meanshift_lists(O, sctx):
    rng = np.random.default_rng(3)
    for n in (0, 1, 2, 31, 32, 33, 1000, 20000):
        v = np.zeros((n, 3), np.float32)
        v[:, 0] = rng.integers(-30, 160, n); v[:, 1] = rng.integers(-30, 160, n); v[:, 2] = rng.choice([0.55, 0.6, 0.75, 1.0], n)
        mo, ro, io = O.meanshift(v)
        mg, rg, ig = sctx.stage_meanshift(v)
        assert ig == io and np.abs(mg - mo).max() <= 1e-3, n
    # two tight clusters: converges to the heavier one
    v = np.array([[10, 10, 1.0]] * 50 + [[100, 100, 1.0]] * 30, np.float32)
    mo, ro, io = O.meanshift(v)
    mg, rg, ig = sctx.stage_meanshift(v)
    assert ig == io and np.array_equal(rg, ro)


# ------------------------------------------------------------------ whole path
def _check_faces(got, want, exact_counts=True):
    assert got["headpose"].tobytes() == want["headpose"].tobytes()  # bit-exact incl. NaN
    assert got["variance"].tobytes() == want["variance"].tobytes()
    for k in ("tree_counts", "dominant", "scaled_w", "scaled_h", "n_votes", "ms_iters", "flags"):
        assert np.array_equal(got[k], want[k]), k
    assert got["scale"].tobytes() == want["scale"].tobytes()
    d = np.abs(got["ffd_f"] - want["ffd_f"])
    assert np.nanmax(d) <= TOL_PX
    return float(np.nanmax(d)), float((got["ffd"] == want["ffd"]).mean())


def test_analyze_crops_synthetic_model(O, crf, sctx, synth_models):
    from face_alignment_cvpr_2012_b200 import workloads as wl
    _, om = synth_models
    crops, _ = wl.make_crops(24, seed=31)
    got = sctx.analyze_crops(crops)
    want = np.array([om.analyze_face(c, (0, 0, 100, 100)) for c in crops])
    dmax, int_eq = _check_faces(got, want)
    assert dmax <= 1e-3 and int_eq >= 0.99
    hp_only = sctx.analyze_crops(crops, headpose_only=True)
    assert hp_only["headpose"].tobytes() == want["headpose"].tobytes() and (hp_only["n_votes"] == 0).all()


def test_analyze_faces_ragged_boxes(O, sctx, synth_models):
    """One frame, boxes of many sizes and aspect ratios (W = 124 and 125, H from 60 to 230), incl. image borders."""
    _, om = synth_models
    import cv2
    rng = np.random.default_rng(8)
    img = cv2.GaussianBlur(rng.integers(0, 256, (600, 800, 3), dtype=np.uint8), (0, 0), 2)
    boxes = [(0, 0, 100, 100), (700, 480, 100, 120), (50, 60, 212, 180), (300, 100, 131, 240), (10, 300, 400, 200), (500, 10, 90, 133),
             (123, 77, 250, 250), (600, 300, 64, 64), (400, 350, 334, 170), (20, 20, 120, 160)]
    got = sctx.analyze_faces(img, boxes)
    want = np.array([om.analyze_face(img, b) for b in boxes])
    assert set(want["scaled_w"].tolist()) == {124, 125}
    _check_faces(got, want)


def test_vote_budget_overflow_is_rerun(crf, O, gpu, tmp_path):
    """A forest whose every leaf votes for every part needs 10 votes per leaf; the batched path budgets 3 and must
    re-run such faces with the worst-case capacity, giving the oracle's result all the same."""
    from face_alignment_cvpr_2012_b200 import synthetic_model as sm, workloads as wl
    hp, ffd = sm.write_model(tmp_path / "allvote", seed=21, hp_depth=6, ffd_depth=6, always_vote=True)
    gm, om = crf.Model(hp, ffd, 15, 20), O.Model(hp, ffd, 15, 20)
    crops, _ = wl.make_crops(5, seed=77)
    got = crf.Context(gm, 0).analyze_crops(crops)
    want = np.array([om.analyze_face(c, (0, 0, 100, 100)) for c in crops])
    assert (want["n_votes"].sum(axis=1) > 3 * 1024 * 20).all()
    _check_faces(got, want)


def test_argument_errors(crf, sctx):
    img = np.zeros((100, 100, 3), np.uint8)
    for box in [(-1, 0, 50, 50), (60, 60, 50, 50), (0, 0, 0, 10), (0, 0, 100, 20), (0, 0, 20, 100)]:  # outside / empty / flatter than a patch / taller than 521
        with pytest.raises(crf.CrfError) as e:
            sctx.analyze_faces(img, [box])
        assert e.value.code == -1
    assert len(sctx.analyze_faces(img, [])) == 0
    assert len(sctx.analyze_crops(np.zeros((0, 100, 100, 3), np.uint8))) == 0


def test_batch_api_and_chunk_independence(crf, O, synth_models, gpu):
    """Results do not depend on how faces are chunked or which frame buffer they came through."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    gm, om = synth_models
    frames, boxes, iob, _ = wl.make_frames(5, 360, 640, 4, seed=4, wmin=60, wmax=150)
    a = crf.Context(gm, 0, crf._options(None, max_chunk=3)).analyze_batch(frames, boxes, iob)
    b = crf.Context(gm, 0, crf._options(None, max_chunk=64)).analyze_batch(frames, boxes, iob)
    assert a.tobytes() == b.tobytes()
    want = np.array([om.analyze_face(frames[i], bx) for bx, i in zip(boxes, iob)])
    _check_faces(a, want)


def test_video_batch_is_cut_in_two_and_stays_identical(crf, O, synth_models, gpu):
    """A batch that fits one launch but moves >= 64 KB of box pixels per face (faces in video frames) runs as two chunks so that the second
    half's pack + copy overlaps the first half's kernels (analyze_host): 36 frames 1080p x 16 faces of 150..220 px, against the same call with an
    explicit max_chunk (which switches the automatic cut off), pinned and pageable sources, and the oracle on a few faces."""
    import torch
    from face_alignment_cvpr_2012_b200 import workloads as wl
    gm, om = synth_models
    frames, boxes, iob, _ = wl.make_frames(36, 1080, 1920, 16, seed=12, wmin=150, wmax=220)
    assert len(boxes) >= 512 and int((boxes[:, 2].astype(np.int64) * boxes[:, 3] * 3).mean()) >= 64 * 1024
    auto_ctx = crf.Context(gm, 0)
    auto = auto_ctx.analyze_batch(frames, boxes, iob)
    one = crf.Context(gm, 0, crf._options(None, max_chunk=4096)).analyze_batch(frames, boxes, iob)
    assert auto.tobytes() == one.tobytes()
    pinned = torch.from_numpy(frames).pin_memory().numpy()
    assert auto_ctx.analyze_batch(pinned, boxes, iob).tobytes() == one.tobytes()
    idx = [0, len(boxes) // 2 - 1, len(boxes) // 2, len(boxes) - 1]
    want = np.array([om.analyze_face(frames[iob[i]], boxes[i]) for i in idx])
    _check_faces(auto[idx], want)


def test_mixed_resolution_images(crf, O, synth_models, gpu):
    """BASELINE config 5 shape: images from 480p to 4K, 1-8 boxes each, face boxes from 64 px to >1000 px wide
    (heavy down-scaling in cv::resize, tall scaled faces), each image through crf_analyze_faces."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    gm, om = synth_models
    ctx = crf.Context(gm, 0)
    imgs, _ = wl.make_mixed(10, seed=2015)
    widths = []
    for frame, boxes in imgs:
        got = ctx.analyze_faces(frame, boxes)
        want = np.array([om.analyze_face(frame, b) for b in boxes])
        _check_faces(got, want)
        widths += [int(b[2]) for b in boxes]
    assert min(widths) < 100 and max(widths) > 900


def test_headpose_only_many_crops(crf, O, synth_models, gpu):
    """BASELINE config 4 shape (head-pose forest only, stride 4) on a few hundred crops incl. pure-noise ones."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    gm, om = synth_models
    crops, _ = wl.make_crops(300, seed=2014)
    got = crf.Context(gm, 0, crf._options(None, max_chunk=128)).analyze_crops(crops, headpose_only=True)
    idx = list(range(0, 300, 23)) + [7, 15]
    want = np.array([om.analyze_face(crops[i], (0, 0, 100, 100), headpose_only=True) for i in idx])
    assert got["headpose"][idx].tobytes() == want["headpose"].tobytes() and got["variance"][idx].tobytes() == want["variance"].tobytes()


def test_counters_match_oracle_visits(O, crf, synth_models, gpu):
    from face_alignment_cvpr_2012_b200 import workloads as wl
    gm, om = synth_models
    crops, _ = wl.make_crops(3, seed=2)
    ctx = crf.Context(gm, 0)
    ctx.set_profiling(True, True)
    ctx.reset_counters()
    ctx.analyze_crops(crops)
    c = ctx.counters()
    hp = ffd = votes = 0
    for cr in crops:
        rec, st = om.analyze_face(cr, (0, 0, 100, 100), want_stats=True)
        hp += st[0]; ffd += st[1]; votes += st[2]
    # the oracle counts node visits incl. the leaf; the device counts node tests (internal nodes only)
    assert c["hp_node_tests"] == hp - c["hp_traversals"] and c["ffd_node_tests"] == ffd - c["ffd_traversals"]
    assert c["votes"] == votes and c["faces"] == 3 and c["kernel_launches"] > 0


# ------------------------------------------------------------------ shipped forests (staged packed image)
def test_lfw_golden_end_to_end(rctx, lfw_faces, lfw_golden):
    """The 20 shipped LFW faces with the shipped forests against the committed oracle records (made from the
    reference's own text archives) and their ground truth."""
    names = lfw_golden["names"].tolist()
    recs = lfw_golden["recs"]
    errs = []
    for f in lfw_faces:
        k = names.index(f["name"])
        got = rctx.analyze_faces(f["img"], [f["box"]])[0]
        want = recs[k]
        assert got["headpose"] == want["headpose"] and got["variance"] == want["variance"]
        assert np.array_equal(got["tree_counts"], want["tree_counts"]) and np.array_equal(got["n_votes"], want["n_votes"])
        assert np.abs(got["ffd_f"] - want["ffd_f"]).max() <= 1e-3
        assert np.array_equal(got["ffd"], want["ffd"])
        gt = lfw_golden["gt"][k].astype(np.float64)
        iod = np.linalg.norm((gt[0] + gt[1]) / 2 - (gt[6] + gt[7]) / 2)
        errs.append(np.linalg.norm(gt - got["ffd"], axis=1) / iod)
    assert abs(float(np.mean(errs)) - 0.0747) < 0.01  # SURVEY §4 / Appendix D


def test_lfw_leaf_id_checksums(O, rctx, staged_models, faces, lfw_golden):
    _, om = staged_models
    names = lfw_golden["names"].tolist()
    for f in faces[:6]:
        k = names.index(f["name"])
        sc = rctx.stage_gray_resize(f["img"], f["box"])
        planes, _ = rctx.stage_channels(sc)
        ids = rctx.stage_eval_forest(planes, 4)
        assert zlib.crc32(ids.tobytes()) == int(lfw_golden["hp_crc"][k])
        r = rctx.stage_headpose(planes, 4)
        ids = rctx.stage_eval_forest(planes, 3, r["forest_idx"], r["tree_idx"])
        assert zlib.crc32(ids.tobytes()) == int(lfw_golden["ffd_crc"][k])


def test_stride1_shipped_forests(O, crf, staged_models, gpu):
    """BASELINE config 2 shape at a size the oracle finishes in seconds: dense stride-1 grids, incl. a pure-noise crop."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    gm, om = staged_models
    crops, _ = wl.make_crops(8, seed=2012)
    ctx = crf.Context(gm, 0, crf._options(None, hp_stride=1, ffd_stride=1))
    got = ctx.analyze_crops(crops)
    idx = [0, 5, 7]
    want = np.array([om.analyze_face(crops[i], (0, 0, 100, 100), 1, 1) for i in idx])
    dmax, _ = _check_faces(got[idx], want)
    assert dmax <= 1e-3
    assert want["ms_iters"][2].max() == 7  # the noise crop runs MeanShift to its iteration cap


def test_full_size_properties(crf, staged_models, gpu):
    """BASELINE config 2 at full size (4096 crops, stride 1): size-independent properties instead of the oracle —
    identical crops give identical records wherever they sit in the batch, chunking does not matter, and the
    host-buffer and device-buffer entry points agree bit for bit."""
    import torch
    from face_alignment_cvpr_2012_b200 import workloads as wl
    gm, _ = staged_models
    base, _ = wl.make_crops(64, seed=2012)
    rng = np.random.default_rng(0)
    perm = rng.integers(0, 64, 4096)
    crops = base[perm]
    ctx = crf.Context(gm, 0, crf._options(None, hp_stride=1, ffd_stride=1, max_chunk=256))
    got = ctx.analyze_crops(crops)
    # chunks of 16 faces stay below the window kernel's batch threshold: the reference records come from the global-gather traversal
    ref = crf.Context(gm, 0, crf._options(None, hp_stride=1, ffd_stride=1, max_chunk=16)).analyze_crops(base)
    assert got.tobytes() == ref[perm].tobytes()
    d_crops = torch.from_numpy(crops).cuda()
    d_out = torch.empty(4096 * crf.FACE_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.analyze_crops_device(d_crops.data_ptr(), 4096, 100, 100, d_out.data_ptr())
    assert d_out.cpu().numpy().tobytes() == got.tobytes()


def test_face_forest_class_mirror(crf, staged_models, faces, lfw_golden, gpu):
    gm, _ = staged_models
    ff = crf.FaceForest(model=gm)
    assert ff.is_inizialized
    f = faces[0]
    face = ff.analyzeFace(f["img"], f["box"])
    k = lfw_golden["names"].tolist().index(f["name"])
    assert np.array_equal(face.ffd_cordinates, lfw_golden["recs"][k]["ffd"]) and face.bbox == tuple(f["box"])
    faces = ff.analyzeImage(f["img"], [f["box"], f["box"]])
    assert len(faces) == 2 and np.array_equal(faces[1].ffd_cordinates, face.ffd_cordinates)


def test_cpp_compat_header_on_gpu(crf, synth_dirs, synth_models, O, gpu, tmp_path):
    """The C++ binding end to end: reference-shaped FaceForest::analyzeImage through libcrf_b200.so vs the oracle."""
    import subprocess
    from face_alignment_cvpr_2012_b200 import capi
    exe = tmp_path / "compat_smoke"
    subprocess.run(["g++", "-std=c++17", "-O1", "-I", str(capi.LIB_PATH.parents[2] / "include"), str(capi.LIB_PATH.parents[2] / "tests" / "cpp" / "compat_smoke.cc"),
                    "-o", str(exe), "-L", str(capi.LIB_PATH.parent), "-lcrf_b200", f"-Wl,-rpath,{capi.LIB_PATH.parent}"], check=True)
    hp, ffd = synth_dirs
    r = subprocess.run([str(exe), hp, ffd, "run"], capture_output=True, text=True)
    assert r.returncode == 0 and "compat_smoke ok" in r.stdout, r.stdout + r.stderr
    _, om = synth_models
    px = ((np.arange(120 * 160 * 3, dtype=np.uint64) * 2654435761 % (1 << 32)) >> 24).astype(np.uint8).reshape(120, 160, 3)
    want = [om.analyze_face(px, b) for b in [(10, 5, 100, 100), (40, 10, 90, 105)]]
    line = [l for l in r.stdout.split("\n") if l.startswith("headpose")][0].split()
    assert abs(float(line[1]) - float(want[0]["headpose"])) < 1e-5 and abs(float(line[2]) - float(want[1]["headpose"])) < 1e-5
    assert line[-1] == f"({want[0]['ffd'][0][0]},{want[0]['ffd'][0][1]})"


def test_eval_ffd_driver(crf, staged_models, lfw_faces, lfw_golden, gpu, tmp_path):
    """SURVEY 8 f3: the reference's eval_ffd workflow (config files -> annotations -> analyzeFace -> output/errors.txt)
    on the 20 shipped LFW faces; errors equal the ones derived from the committed oracle records."""
    from face_alignment_cvpr_2012_b200 import eval as ev, workloads as wl
    idx = wl.STAGED / "imgs" / "index_random_subset.txt"
    ann = ev.loadAnnotations(str(idx))
    assert len(ann) == 20 and ann[0].parts.shape == (10, 2)
    test10 = ev.split_test(ann)            # 90/10 split per pose class, as src/eval_ffd.cpp:155-169
    assert 0 < len(test10) <= 5 and len(ev.split_test(ann, everything=True)) == 20
    ff = crf.FaceForest(model=staged_models[0])
    out = tmp_path / "output" / "errors.txt"
    err = ev.evalForest_ffd(ff, ev.split_test(ann, everything=True), str(idx), str(out))
    assert err.shape == (20, 10) and abs(float(err.mean()) - 0.0747) < 0.01
    rows = [l.split() for l in out.read_text().strip().split("\n")]
    assert len(rows) == 20 and all(len(r) == 10 for r in rows)
    names = lfw_golden["names"].tolist()
    order = [a for cls in range(-2, 3) for a in ann if a.pose == cls]
    for a, e in zip(order, err):
        k = names.index(a.url)
        gt = lfw_golden["gt"][k].astype(np.float64)
        iod = np.linalg.norm((gt[0] + gt[1]) / 2 - (gt[6] + gt[7]) / 2)
        want = np.linalg.norm(gt - lfw_golden["recs"][k]["ffd"], axis=1) / iod
        assert np.allclose(e, want, rtol=1e-5, atol=1e-6)


def test_cpp_eval_ffd_driver(crf, staged_models, lfw_faces, lfw_golden, gpu, tmp_path):
    """SURVEY 8 f3 in the reference's language: examples/eval_ffd.cpp (config files -> annotations -> FaceForest::analyzeFace through
    include/crf_b200_compat.hpp -> errors.txt) on the 20 shipped LFW faces; its errors equal the committed oracle records'."""
    import subprocess
    import cv2
    from face_alignment_cvpr_2012_b200 import capi, workloads as wl
    root = capi.LIB_PATH.parents[2]
    exe = tmp_path / "eval_ffd"
    subprocess.run(["g++", "-std=c++17", "-O1", "-I", str(root / "include"), str(root / "examples" / "eval_ffd.cpp"), "-o", str(exe),
                    f"-L{capi.LIB_PATH.parent}", "-lcrf_b200", f"-Wl,-rpath,{capi.LIB_PATH.parent}"], check=True)
    data = tmp_path / "data"; data.mkdir()
    for f in lfw_faces:
        cv2.imwrite(str(data / (Path(f["name"]).stem + ".ppm")), f["img"])
    idx = data / "index_random_subset.txt"
    idx.write_text((wl.STAGED / "imgs" / "index_random_subset.txt").read_text())
    def cfg(name, ntrees):
        p = tmp_path / name
        p.write_text("\n".join(["____Path to images index file", str(idx), "____Path to trees", str(wl.staged_model_path()), "____Number of trees", str(ntrees),
                                "____Number of tests", "2500", "____Max depth", "20", "____Min patches per node", "20", "____Images per class", "600",
                                "____Patches per image", "150", "____Face size", "125", "____Patch size ratio", "0.250000", "____Features", "0 1 2"]) + "\n")
        return str(p)
    out = tmp_path / "errors.txt"
    r = subprocess.run([str(exe), "--all", "--out", str(out), cfg("config_ffd.txt", 20), cfg("config_headpose.txt", 15)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "20 faces" in r.stdout, r.stdout + r.stderr
    err = np.array([[float(v) for v in l.split()] for l in out.read_text().strip().split("\n")])
    assert err.shape == (20, 10) and abs(float(err.mean()) - 0.0747) < 0.01
    names = lfw_golden["names"].tolist()
    order = [f for cls in range(-2, 3) for f in lfw_faces if f["pose"] == cls]
    for f, e in zip(order, err):
        k = names.index(f["name"])
        gt = lfw_golden["gt"][k].astype(np.float64)
        iod = np.linalg.norm((gt[0] + gt[1]) / 2 - (gt[6] + gt[7]) / 2)
        want = np.linalg.norm(gt - lfw_golden["recs"][k]["ffd"], axis=1) / iod
        assert np.allclose(e, want, rtol=1e-4, atol=1e-5)   # errors.txt holds 6 significant digits
    # the reference's eval_headpose main (src/eval_headpose.cpp): "Real:<pose> Predict:<headpose>" per image
    r = subprocess.run([str(exe), "--all", "--headpose", cfg("config_ffd.txt", 20), cfg("config_headpose.txt", 15)], capture_output=True, text=True, timeout=300)
    lines = [l for l in r.stdout.split("\n") if l.startswith("Real:")]
    assert r.returncode == 0 and len(lines) == 20, r.stdout + r.stderr
    for f, l in zip(order, lines):
        real, pred = l.split(" Predict:")
        assert int(real[5:]) == f["pose"]
        assert abs(float(pred) - float(lfw_golden["recs"][names.index(f["name"])]["headpose"])) < 1e-5


def test_analyze_image_with_the_cascade_detector(crf, staged_models, lfw_faces, gpu):
    """FaceForest::analyzeImage as the reference runs it: Haar cascade (evaluated on the GPU), enlarged boxes, GPU pipeline."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    xml = wl.STAGED / "haarcascade_frontalface_alt.xml"
    if not xml.exists():
        pytest.skip("Haar cascade not staged")
    opt = crf.FaceForestOptions()
    opt.fd_option.path_face_cascade = str(xml)
    ff = crf.FaceForest(opt, model=staged_models[0])
    assert ff.is_inizialized
    found = 0
    for f in lfw_faces[:8]:
        faces = ff.analyzeImage(f["img"])
        for face in faces:
            x, y, w, h = face.bbox
            ax, ay, aw, ah = f["box"]
            inter = max(0, min(x + w, ax + aw) - max(x, ax)) * max(0, min(y + h, ay + ah) - max(y, ay))
            if inter > 0.5 * aw * ah:   # the detection that matches the annotated face: landmarks must land near the annotation
                found += 1
                pred = face.ffd_cordinates + np.array([x, y])
                gt = f["parts"] + np.array([ax, ay])
                iod = np.linalg.norm((gt[0] + gt[1]) / 2.0 - (gt[6] + gt[7]) / 2.0)
                assert np.mean(np.linalg.norm(pred - gt, axis=1)) / iod < 0.25
    assert found >= 6


def test_pinned_and_pageable_sources_agree(crf, synth_models, gpu):
    """The host entry point takes two upload routes: whole frames straight from pinned memory, or box pixels packed into the
    library's pinned staging (pageable callers, sparse boxes).  Same records either way."""
    import ctypes as C
    from face_alignment_cvpr_2012_b200 import workloads as wl
    gm, _ = synth_models
    crops, _ = wl.make_crops(70, seed=5)
    ctx = crf.Context(gm, 0, crf._options(None, max_chunk=32))
    pageable = ctx.analyze_crops(crops)
    p = C.c_void_p()
    crf.capi.check(crf.lib().crf_host_alloc(C.byref(p), crops.nbytes))
    try:
        C.memmove(p, crops.ctypes.data, crops.nbytes)
        out = np.zeros(len(crops), crf.FACE_DTYPE)
        ctx.analyze_crops_ptr(p.value, len(crops), 100, 100, out)
        assert out.tobytes() == pageable.tobytes()
        h2d = ctx.counters()["h2d_bytes"]
        assert h2d >= 2 * crops.nbytes
    finally:
        crf.lib().crf_host_free(p)
