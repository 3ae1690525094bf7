"""CPU: the oracle against the committed cv2 4.13 golden vectors (tests/golden/make_golden.py) — this is what pins
the oracle, since the reference ships no tests or vectors for the path and cannot be built here (SURVEY §8c)."""
import numpy as np


def test_bgr2gray(O, cv2_golden):
    assert np.array_equal(O.bgr2gray(cv2_golden["bgr"]), cv2_golden["gray"])


def test_resize_bit_exact(O, cv2_golden):
    k = 0
    while f"resize_src_{k}" in cv2_golden:
        dst = cv2_golden[f"resize_dst_{k}"]
        got = O.resize(cv2_golden[f"resize_src_{k}"], dst.shape[0], dst.shape[1])
        assert np.array_equal(got, dst), k
        k += 1
    assert k >= 7


def test_scaled_size_follows_float_math(O):
    assert O.scaled_size(130, 130)[:2] == (125, 125)
    assert O.scaled_size(100, 100)[:2] == (125, 125)
    for w in range(40, 700):
        sw, sh, s = O.scaled_size(w, w + 7)
        sc = np.float32(125) / np.float32(w)
        assert sw == int(np.float32(w) * sc) and sh == int(np.float32(w + 7) * sc) and sw in (124, 125)


def test_plain_channels(O, cv2_golden):
    img = cv2_golden["plane"]
    planes, integ = O.channels(img, features_mask=0b0101)  # gray + sobel
    assert np.array_equal(planes[0], img)
    assert np.array_equal(integ[0], cv2_golden["integral"])
    assert np.array_equal(planes[1], cv2_golden["sobel_dy"])  # plane 36 of the full stack = d/dy (reference misnames it sob_x)
    assert np.array_equal(planes[2], cv2_golden["sobel_dx"])
    mm, _ = O.channels(img, features_mask=0b1000)
    assert np.array_equal(mm[0], cv2_golden["erode"]) and np.array_equal(mm[1], cv2_golden["dilate"])


def test_equalize_hist(O, cv2_golden):
    """FC_NORM = cv::equalizeHist (include/FeatureChannelFactory.hpp:58-70)."""
    p, _ = O.channels(cv2_golden["plane"], features_mask=0b100000)
    assert np.array_equal(p[0], cv2_golden["equalize"])
    p, _ = O.channels(cv2_golden["equalize_src2"], features_mask=0b100000)
    assert np.array_equal(p[0], cv2_golden["equalize2"])
    const = np.full((40, 125), 77, np.uint8)
    p, _ = O.channels(const, features_mask=0b100000)
    assert (p[0] == 77).all()


def test_gabor_7x7_filter2d_bit_exact(O, cv2_golden):
    img = cv2_golden["plane"]
    for idx in range(7):
        re, im = O.gabor_response(img, idx)
        assert np.array_equal(re, cv2_golden[f"f2d_re_{idx}"]), idx
        assert np.array_equal(im, cv2_golden[f"f2d_im_{idx}"]), idx


def test_gabor_planes_vs_cv2(O, cv2_golden):
    """nu = 0 planes are bit-exact; for >= 9x9 kernels cv2 switches to a DFT path, so the pin is statistical:
    every difference is +-1 LSB and rarer than 2e-4 (observed ~6e-5)."""
    img = cv2_golden["plane"]
    planes, _ = O.channels(img, features_mask=0b0010)
    ref = cv2_golden["gabor_u8_cv2"]
    assert planes.shape == ref.shape == (35,) + img.shape
    assert np.array_equal(planes[:7], ref[:7])
    d = planes.astype(int) - ref.astype(int)
    assert np.abs(d).max() <= 1
    assert (d != 0).mean() <= 2e-4


def test_gabor_bank_geometry(O):
    bank = O.gabor_bank()
    assert [b[0].shape[0] for b in bank] == [7] * 7 + [9] * 7 + [13] * 7 + [19] * 7 + [25] * 7


def test_node_test_integer_division_equivalence():
    """(int)((float)s / (float)(w*h)) == s / (w*h) == umulhi(s << 1, floor(2^31 / area) + 1) for every area the patch
    admits and every sum a u8 plane can produce (SURVEY A.6; device_forest.h magic_for_area)."""
    for area in list(range(1, 485)) + [529, 600, 900, 961]:
        s = np.arange(0, 255 * area + 1, dtype=np.int64)
        q = s // area
        fl = (s.astype(np.float32) / np.float32(area)).astype(np.int64)
        m = (1 << 31) // area + 1
        mg = ((s << 1) * m) >> 32
        assert np.array_equal(q, fl) and np.array_equal(q, mg), area
        # k_traverse16's reciprocal-free form: float estimate + one exact fix-up step
        est = (s.astype(np.float32) * (np.float32(1) / np.float32(area))).astype(np.int64)
        r = s - est * area
        est = est + (r >= area) - (r < 0)
        assert np.array_equal(q, est), area


def test_canny_matches_cv2(O, cv2_golden):
    """FC_CANNY: the restated cv::Canny(img, out, -1, 5) against cv2 4.13, bit for bit (planes are 0 / 255)."""
    for src, want in ((cv2_golden["plane"], cv2_golden["canny"]), (cv2_golden["canny_src2"], cv2_golden["canny2"])):
        planes, integ = O.channels(src, features_mask=16)
        assert planes.shape[0] == 1 and np.array_equal(planes[0], want)
        assert np.array_equal(integ[0][1:, 1:], np.cumsum(np.cumsum(want.astype(np.float64), 0), 1).astype(np.float32))
    # sorted feature order: gray (0), canny (4), norm (5)
    planes, _ = O.channels(cv2_golden["plane"], features_mask=1 | 16 | 32)
    assert planes.shape[0] == 3 and np.array_equal(planes[1], cv2_golden["canny"]) and np.array_equal(planes[2], cv2_golden["equalize"])


def test_index_division_by_multiplication():
    """k_votes_emit turns the flat leaf index into (patch, tree) and (ix, iy) with umulhi(k, 0xffffffff / d + 1), exact for
    k < 2^32 / d: trees per face d <= 128 with k < 94 * 490 * 128 < 2^23, patch rows d <= 490 with patch < 94 * 490 < 2^16."""
    full = np.arange(0, 1 << 23, dtype=np.uint64)
    sparse = np.concatenate([full[::13], full[-8192:]])
    for d in range(2, 129):
        k = full if d in (15, 20, 128) else sparse   # the shipped forests (15 / 20 trees) and the cap exhaustively
        m = np.uint64(0xffffffff // d + 1)
        assert np.array_equal((k * m) >> np.uint64(32), k // np.uint64(d)), d
    k = np.arange(0, 1 << 17, dtype=np.uint64)
    for d in range(2, 491):
        m = np.uint64(0xffffffff // d + 1)
        assert np.array_equal((k * m) >> np.uint64(32), k // np.uint64(d)), d


def test_meanshift_empty_and_single(O):
    mean, rnd, it = O.meanshift(np.zeros((0, 3), np.float32))
    assert mean.tolist() == [0, 0] and it == 1
    mean, rnd, it = O.meanshift(np.array([[10, 20, 0.75]], np.float32))
    assert rnd.tolist() == [10, 20] and it == 1


def test_area_under_curve_sums_to_one(O):
    edges = [-2.5, -0.35, -0.2, 0.2, 0.35, 2.5]
    tot = sum(float(O.area_under_curve(edges[i], edges[i + 1], 0.1, 0.15)) for i in range(5))
    assert abs(tot - 1.0) < 0.06


def test_cv2_gabor_planes_downstream(O, staged_models, faces):
    """What the +-1-LSB distance between the canonical Gabor arithmetic and cv2's filter2D (DFT path for kernels >= 9x9) does
    downstream: cv2-made planes and the oracle's planes through the shipped forests on LFW faces + synthetic crops.  Observed on
    the full set (20 faces + 64 crops, tests/test_gpu_reference_campaign.py runs it on the GPU): 2.8e-5 of the u8 samples differ,
    1e-5 of the leaf ids, landmarks move by <= 0.02 px."""
    import cv2
    from face_alignment_cvpr_2012_b200 import workloads as wl
    _, om = staged_models
    bank = O.gabor_bank()
    crops, _ = wl.make_crops(6, seed=4806)
    items = [(f["img"], f["box"]) for f in faces[:6]] + [(c, (0, 0, 100, 100)) for c in crops]
    n_px = n_diff = n_leaf = n_leaf_diff = 0
    worst = 0.0
    for img, box in items:
        x, y, w, h = box
        sw, sh, _ = O.scaled_size(w, h)
        g = O.resize(O.bgr2gray(img)[y:y + h, x:x + w], sh, sw)
        planes, _ = O.channels(g, threads=4)
        cvp = planes.copy()
        for k, (re, im) in enumerate(bank):
            r = cv2.filter2D(g, cv2.CV_32F, re); i = cv2.filter2D(g, cv2.CV_32F, im)
            m = cv2.pow(cv2.add(cv2.pow(i, 2), cv2.pow(r, 2)), 0.5)
            cvp[1 + k] = cv2.convertScaleAbs(cv2.normalize(m, None, 0, 1, cv2.NORM_MINMAX), alpha=255)
        d = cvp.astype(np.int16) - planes
        assert np.abs(d).max() <= 1 and not d[0].any() and not d[36:].any()
        n_px += d[1:36].size; n_diff += int((d != 0).sum())
        sa, sb = O.Sample(planes=planes), O.Sample(planes=cvp)
        _, hpa, va, _ = om.eval_hp(sa, 4); _, hpb, vb, _ = om.eval_hp(sb, 4)
        _, _, fi, ti, _ = om.compose(hpa, va)
        ea, eb = om.eval_ffd(sa, fi, ti, 3), om.eval_ffd(sb, fi, ti, 3)
        n_leaf += ea["leaf_ids"].size; n_leaf_diff += int((ea["leaf_ids"] != eb["leaf_ids"]).sum())
        worst = max(worst, float(np.abs(ea["mean"] - eb["mean"]).max()), abs(float(hpa) - float(hpb)))
        sa.close(); sb.close()
    assert n_diff / n_px <= 2e-4 and n_leaf_diff / n_leaf <= 1e-3 and worst <= 0.5
