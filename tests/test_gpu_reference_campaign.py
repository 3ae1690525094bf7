"""GPU: the CUDA path with the SHIPPED forests against (a) golden vectors produced by the real reference code
(tests/golden/ref_campaign.npz, made by tests/golden/make_ref_golden.py from oracle/_ref = the reference's own sources)
and (b) the oracle run live on the same inputs (all record fields).  Shapes follow BASELINE.json's configurations:
stride-1 crops through the shared-memory window kernel (config 2), default-stride crops incl. noise, 1080p frames with
ragged boxes (config 3), head pose only (config 4), mixed resolutions up to 4K with a > 1000 px box (config 5).
Bit-exact: head pose / variance bits, forest composition, vote counts, MeanShift iterations (exact mode), final integer
landmarks; pre-rounding MeanShift means within TOL_PX.
Without the shipped forests and LFW fixtures staged, the same checks run on the synthetic forests and procedural faces
against tests/golden/synth_campaign.npz (tests/golden/make_synth_golden.py: the reference library's results on those inputs
where it is available, else the CPU oracle's; its `source` entry says which)."""
import importlib.util
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
TOL_PX = 0.5
GOLDEN = Path(__file__).resolve().parent / "golden"


def _load_sets(faces):
    spec = importlib.util.spec_from_file_location("make_ref_golden", GOLDEN / "make_ref_golden.py")
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m.campaign_sets(faces)


@pytest.fixture(scope="module")
def gpu(crf):
    if crf.lib().crf_device_count() < 1:
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box (there is no CPU fallback)")
    return True


@pytest.fixture(scope="module")
def sets(faces):
    return _load_sets(faces)


@pytest.fixture(scope="module")
def ref_golden(shipped):
    """The reference's own results on the shipped forests; on the synthetic forests, synth_campaign.npz (see its `source`)."""
    return np.load(GOLDEN / ("ref_campaign.npz" if shipped else "synth_campaign.npz"))


def _list_from_record(rec, ntrees=20):
    """The composed forest implied by (tree_counts, dominant): src/FaceForest.cpp:239-250."""
    lst = [(i, j) for i in range(5) for j in range(int(rec["tree_counts"][i]))]
    lst += [(int(rec["dominant"]), t) for t in range(len(lst), ntrees)]
    return lst


def _check_against_reference(got, g, name, exact_landmarks=True):
    hp = g[f"{name}_headpose"]; ffd = g[f"{name}_ffd"]; lf = g[f"{name}_list_forest"]; lt = g[f"{name}_list_tree"]
    assert len(got) == len(hp)
    assert got["headpose"].tobytes() == hp.tobytes()                       # the reference's own f32 sums, bit for bit
    for i in range(len(got)):
        n = int((lf[i] >= 0).sum())
        assert _list_from_record(got[i]) == list(zip(lf[i, :n].tolist(), lt[i, :n].tolist())), (name, i)
    d = np.abs(got["ffd"].astype(np.int64) - ffd)
    if exact_landmarks:
        assert d.max() == 0, (name, int(d.max()), float((d != 0).mean()))
    else:   # tolerance-mode MeanShift: a mean within 0.5 px of the reference's may round to the neighbouring integer
        scale = np.maximum(1.0 / got["scale"], 1.0)
        assert (d <= np.ceil(scale)[:, None, None] + 1).all() and (d != 0).mean() < 0.02, (name, int(d.max()), float((d != 0).mean()))


def _check_against_oracle(got, want, exact=True):
    assert got["headpose"].tobytes() == want["headpose"].tobytes() and got["variance"].tobytes() == want["variance"].tobytes()
    for k in ("tree_counts", "dominant", "scaled_w", "scaled_h", "n_votes", "flags"):
        assert np.array_equal(got[k], want[k]), k
    d = np.abs(got["ffd_f"] - want["ffd_f"])
    assert np.nanmax(d) <= TOL_PX
    if exact:
        assert np.array_equal(got["ms_iters"], want["ms_iters"]) and np.nanmax(d) <= 1e-3 and np.array_equal(got["ffd"], want["ffd"])
    return float(np.nanmax(d))


@pytest.mark.parametrize("ms_mode", ["exact", "fast"])
def test_stride1_crops_window_kernel(crf, O, gpu, staged_models, sets, ref_golden, monkeypatch, ms_mode):
    """Config 2 shape: 48 stride-1 crops in ONE call so the persistent shared-memory window kernel runs (forced, so a fallback
    to the global-gather kernels would fail the call instead of silently passing)."""
    gm, om = staged_models
    items, hs, fs = sets["s1"]
    crops = np.stack([c for c, _ in items])
    monkeypatch.setenv("CRF_TRAVERSE_VARIANT", "0x100001")
    ctx = crf.Context(gm, 0, crf._options(None, hp_stride=hs, ffd_stride=fs, ms_mode=ms_mode))
    got = ctx.analyze_crops(crops)
    _check_against_reference(got, ref_golden, "s1", exact_landmarks=ms_mode == "exact")
    idx = list(range(0, 48, 3)) + [7, 47]
    want = np.array([om.analyze_face(crops[i], (0, 0, 100, 100), hs, fs, threads=O.hardware_concurrency()) for i in idx])
    _check_against_oracle(got[idx], want, exact=ms_mode == "exact")
    assert want["ms_iters"][idx.index(7)].max() == 7   # the noise crop runs MeanShift to its cap


@pytest.mark.parametrize("ms_mode", ["exact", "fast"])
def test_default_stride_crops(crf, O, gpu, staged_models, sets, ref_golden, ms_mode):
    gm, om = staged_models
    items, hs, fs = sets["dflt"]
    crops = np.stack([c for c, _ in items])
    ctx = crf.Context(gm, 0, crf._options(None, hp_stride=hs, ffd_stride=fs, ms_mode=ms_mode))
    got = ctx.analyze_crops(crops)
    _check_against_reference(got, ref_golden, "dflt", exact_landmarks=ms_mode == "exact")
    want = np.array([om.analyze_face(c, (0, 0, 100, 100), hs, fs, threads=O.hardware_concurrency()) for c in crops])
    dmax = _check_against_oracle(got, want, exact=ms_mode == "exact")
    print(f"default strides, 256 crops, MeanShift {ms_mode}: max |ffd_f - oracle| = {dmax:.2e} px")


def test_headpose_only_matches_reference(crf, gpu, staged_models, sets, ref_golden):
    """Config 4 shape: stop after getHeadPoseVotesMT."""
    gm, _ = staged_models
    items, hs, fs = sets["dflt"]
    crops = np.stack([c for c, _ in items])
    got = crf.Context(gm, 0, crf._options(None, hp_stride=hs, ffd_stride=fs)).analyze_crops(crops, headpose_only=True)
    assert got["headpose"].tobytes() == ref_golden["dflt_headpose"].tobytes() and (got["n_votes"] == 0).all()


def test_1080p_frames_ragged_boxes(crf, O, gpu, staged_models, ref_golden):
    """Config 3 shape: 4 frames x 16 boxes through crf_analyze_batch (gray conversion + crop + resize on the GPU)."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    gm, om = staged_models
    frames, boxes, iob, _ = wl.make_frames(4, seed=4803)
    ctx = crf.Context(gm, 0)
    got = ctx.analyze_batch(frames, boxes, iob)
    _check_against_reference(got, ref_golden, "c3")
    want = np.array([om.analyze_face(frames[i], tuple(int(v) for v in b), threads=O.hardware_concurrency()) for b, i in zip(boxes, iob)])
    _check_against_oracle(got, want)
    assert len(set(got["scaled_h"].tolist())) > 1


def test_mixed_resolution_up_to_4k(crf, O, gpu, staged_models, sets, ref_golden):
    """Config 5 shape: one call per image, sizes 480p .. 4K, incl. a 1400-px-wide box."""
    gm, om = staged_models
    items, hs, fs = sets["c5"]
    ctx = crf.Context(gm, 0)
    got = np.concatenate([ctx.analyze_faces(img, [box]) for img, box in items])
    _check_against_reference(got, ref_golden, "c5")
    want = np.array([om.analyze_face(img, box, threads=O.hardware_concurrency()) for img, box in items])
    _check_against_oracle(got, want)
    assert max(b[2] for _, b in items) > 1000 and max(img.shape[0] for img, _ in items) == 2160


def test_lfw_matches_reference(crf, gpu, staged_models, sets, ref_golden):
    gm, _ = staged_models
    items, _, _ = sets["lfw"]
    ctx = crf.Context(gm, 0)
    got = np.concatenate([ctx.analyze_faces(img, [box]) for img, box in items])
    _check_against_reference(got, ref_golden, "lfw")


def test_compose_knife_edges(crf, O, gpu, staged_models):
    """floor(areaUnderCurve * 20) picks the trees (src/FaceForest.cpp:243): >= 1e5 (mean, variance) pairs, most of them placed
    where area * 20 sits next to an integer (found by bisection on the oracle's own areaUnderCurve, then the +-8 neighbouring
    floats of the variance), the rest random incl. degenerate variances.  The oracle's areaUnderCurve is pinned bit for bit to
    the reference's (tests/test_reference_pin.py); the device evaluates exp() itself."""
    gm, om = staged_models
    rng = np.random.default_rng(2012)
    T = np.array([-2.5, -0.35, -0.20, 0.20, 0.35, 2.5], np.float32)
    hp, var = [], []
    n_edges = 0
    while n_edges < 4500:
        mean = np.float32(rng.uniform(-1.2, 1.2)); j = int(rng.integers(0, 5)); k = int(rng.integers(1, 20))
        f = lambda v: float(O.area_under_curve(float(T[j]), float(T[j + 1]), float(mean), float(np.sqrt(np.float64(np.float32(v)))))) * 20 - k
        lo, hi = 1e-5, 2.0
        if (f(lo) > 0) == (f(hi) > 0):
            continue
        for _ in range(40):
            mid = 0.5 * (lo + hi)
            if (f(mid) > 0) == (f(lo) > 0): lo = mid
            else: hi = mid
        v0 = np.float32(lo)
        v = v0
        for _ in range(8): v = np.nextafter(v, np.float32(0))
        for _ in range(17):
            hp.append(mean); var.append(v); v = np.nextafter(v, np.float32(4))
        n_edges += 1
    n_rand = 30000
    hp += list(rng.uniform(-2.2, 2.2, n_rand).astype(np.float32)); var += list((10.0 ** rng.uniform(-7, 0.7, n_rand)).astype(np.float32))
    for h in (-2.0, -0.35, -0.2, 0.0, 0.2, 0.35, 2.0, float("nan")):
        for v in (0.0, 1e-12, -1e-3, float("nan"), float("inf"), 1e-38):
            hp.append(np.float32(h)); var.append(np.float32(v))
    hp = np.array(hp, np.float32); var = np.array(var, np.float32)
    assert len(hp) >= 100000
    ctx = crf.Context(gm, 0)
    g = ctx.stage_compose_batch(hp, var, list_cap=24)
    bad = 0
    for i in range(len(hp)):
        counts, dom, fi, ti, fl = om.compose(hp[i], var[i])
        ok = np.array_equal(g["tree_counts"][i], counts) and g["dominant"][i] == dom and g["flags"][i] == fl
        n = min(len(fi), 24)
        ok = ok and np.array_equal(g["forest_idx"][i, :n], fi[:n]) and np.array_equal(g["tree_idx"][i, :n], ti[:n])
        bad += not ok
    assert bad == 0, f"{bad} of {len(hp)} compositions differ"


def test_cv2_gabor_planes_downstream(crf, O, gpu, staged_models, faces):
    """The canonical (separable) Gabor arithmetic against cv2's own filter2D (DFT path for kernels >= 9x9) on the 20 LFW faces
    + 64 synthetic crops: the 8-bit planes differ by +-1 LSB at a rate <= 2e-4, and pushing BOTH sets of planes through the
    shipped forests on the GPU moves no landmark by more than 0.5 px."""
    import cv2
    from face_alignment_cvpr_2012_b200 import workloads as wl
    gm, _ = staged_models
    ctx = crf.Context(gm, 0)
    bank = O.gabor_bank()
    crops, _ = wl.make_crops(64, seed=4806)
    items = [(f["img"], f["box"]) for f in faces] + [(c, (0, 0, 100, 100)) for c in crops]
    n_px = n_diff = n_leaf = n_leaf_diff = 0
    worst = 0.0
    for img, box in items:
        g = ctx.stage_gray_resize(img, box)
        planes, _ = ctx.stage_channels(g)
        cvp = planes.copy()
        for k, (re, im) in enumerate(bank):
            r = cv2.filter2D(g, cv2.CV_32F, re); i = cv2.filter2D(g, cv2.CV_32F, im)
            m = cv2.pow(cv2.add(cv2.pow(i, 2), cv2.pow(r, 2)), 0.5)
            cvp[1 + k] = cv2.convertScaleAbs(cv2.normalize(m, None, 0, 1, cv2.NORM_MINMAX), alpha=255)
        assert np.array_equal(cvp[0], planes[0]) and np.array_equal(cvp[36:], planes[36:])
        d = cvp.astype(np.int16) - planes
        assert np.abs(d).max() <= 1
        n_px += d.size - 3 * d[0].size; n_diff += int((d != 0).sum())
        a = ctx.stage_headpose(planes, 4); b = ctx.stage_headpose(cvp, 4)
        la = ctx.stage_eval_forest(planes, 3, a["forest_idx"], a["tree_idx"]); lb = ctx.stage_eval_forest(cvp, 3, a["forest_idx"], a["tree_idx"])
        n_leaf += la.size; n_leaf_diff += int((la != lb).sum())
        va = ctx.stage_votes_meanshift(planes, 3, a["forest_idx"], a["tree_idx"]); vb = ctx.stage_votes_meanshift(cvp, 3, a["forest_idx"], a["tree_idx"])
        worst = max(worst, float(np.abs(va["mean"] - vb["mean"]).max()), abs(float(a["headpose"]) - float(b["headpose"])))
    print(f"cv2 vs canonical Gabor: {n_diff}/{n_px} u8 samples differ ({n_diff / n_px:.2e}), {n_leaf_diff}/{n_leaf} FFD leaf ids differ, worst landmark / head-pose shift {worst:.3e}")
    assert n_diff / n_px <= 2e-4
    assert n_leaf_diff / n_leaf <= 1e-3
    assert worst <= TOL_PX
