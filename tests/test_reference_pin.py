"""CPU: the oracle against the REAL reference (oracle/_ref/libcrf_ref.so = the reference's own sources compiled
unmodified against type stand-ins for OpenCV / Boost, see oracle/ref_driver.cc).

What this pins, bit for bit, to code the reference's authors wrote: the Boost text-archive reading of all 115 shipped
trees through the reference's serialize() methods, Forest/Tree::evaluateMT + TreeNode::eval + ImageSample::evalTest
(leaf ids), getHeadPoseVotesMT (f32 mean / variance), areaUnderCurve, the forest composition and final rescale of
FaceForest::analyzeFace, getFacialFeaturesVotesMT (vote lists, in order) and MeanShift::shift.  The OpenCV arithmetic
under the reference comes from the stand-in, i.e. from the oracle's cv2-pinned stages (tests/test_oracle_golden.py).

Needs the reference's library: built from a checkout of the reference project named by CRF_REFERENCE, or a prebuilt
oracle/_ref/libcrf_ref.so.  The forests are the shipped text archives of that checkout when present, else the synthetic
ones (synthetic_model.py writes the reference's own archive format); the faces are the LFW fixtures of that checkout,
else workloads.procedural_lfw().  Without the library the GPU tests use the golden vectors made from it
(tests/golden/make_ref_golden.py, tests/golden/ref_*.npz)."""
import numpy as np
import pytest

from conftest import REF_DATA

HP_DIR, FFD_DIR = (REF_DATA / "trees_headpose", REF_DATA / "trees_ffd") if REF_DATA else (None, None)


@pytest.fixture(scope="module")
def R():
    from oracle import ref
    if not ref.available():
        pytest.skip("no reference library: oracle/_ref/libcrf_ref.so is absent and CRF_REFERENCE names no checkout to build it from")
    ref.build()
    return ref


@pytest.fixture(scope="module")
def archives(synth_dirs):
    return (str(HP_DIR), str(FFD_DIR)) if HP_DIR is not None and HP_DIR.exists() else synth_dirs


@pytest.fixture(scope="module")
def ff(R, archives):
    return R.FaceForest(*archives)


@pytest.fixture(scope="module")
def om(O, R, archives):
    return O.Model(*archives)


def _planes(rng, C=38, H=125, W=125):
    import cv2
    p = rng.integers(0, 256, (C, H, W), dtype=np.uint8)
    p = np.stack([cv2.GaussianBlur(q, (0, 0), 2.0) for q in p])
    return np.clip((p.astype(np.float32) - 128) * 6 + 128, 0, 255).astype(np.uint8)


def _lfw():
    import cv2
    if REF_DATA is None or not (REF_DATA / "imgs" / "index_random_subset.txt").exists():
        from face_alignment_cvpr_2012_b200 import workloads as wl
        return [(f["img"], f["box"]) for f in wl.procedural_lfw()]
    out = []
    for line in (REF_DATA / "imgs" / "index_random_subset.txt").read_text().split("\n"):
        t = line.split()
        if len(t) >= 27:
            out.append((cv2.imread(str(REF_DATA / "imgs" / t[0])), tuple(int(v) for v in t[1:5])))
    return out


def test_reference_loads_every_shipped_tree(ff, R):
    """Forest::load / Tree::load through the reference's own serialize() (the archive reader of the stand-in only supplies
    tokens): 15 + 5 x 20 finished trees."""
    L = R.lib()
    assert L.ref_num_trees(ff.h, -1) == 15
    assert [L.ref_num_trees(ff.h, k) for k in range(5)] == [20] * 5


@pytest.mark.parametrize("stride,H,W", [(4, 125, 125), (3, 148, 124), (1, 64, 125)])
def test_leaf_ids_and_headpose_match_reference(O, R, ff, om, stride, H, W):
    rng = np.random.default_rng(stride * 10 + H)
    planes = _planes(rng, 38, H, W)
    rs, os_ = R.Sample(planes=planes), O.Sample(planes=planes)
    ids_r, hp_r, var_r = ff.eval_hp(rs, stride)
    ids_o, hp_o, var_o, _ = om.eval_hp(os_, stride)
    assert np.array_equal(ids_r, ids_o)                                  # Boost object ids, [patch][tree]
    assert hp_r.tobytes() == hp_o.tobytes() and var_r.tobytes() == var_o.tobytes()
    fi = rng.integers(0, 5, 20); ti = rng.integers(0, 20, 20)
    cap = 60000 if stride == 1 else 12000
    er = ff.eval_ffd(rs, fi, ti, stride, vote_cap=cap)
    eo = om.eval_ffd(os_, fi, ti, stride, vote_cap=cap)
    assert np.array_equal(er["leaf_ids"], eo["leaf_ids"])
    assert np.array_equal(er["n_votes"], eo["n_votes"]) and er["n_votes"].max() <= cap and er["n_votes"].sum() > 0
    assert np.array_equal(er["votes"], eo["votes"])                      # same votes, same order, same weights
    assert np.array_equal(er["rounded"], eo["rounded"])                  # MeanShift::shift's integer result
    rs.close(); os_.close()


def test_eval_test_matches_reference(O, R):
    """ImageSample::evalTest on random rectangles (the integer mean-difference of SURVEY A.6) against the stage the oracle's
    leaf ids are built on — checked indirectly above; here directly against the integer formula."""
    rng = np.random.default_rng(7)
    planes = rng.integers(0, 256, (3, 80, 125), dtype=np.uint8)
    rs = R.Sample(planes=planes)
    integ = np.zeros((3, 81, 126), np.int64)
    integ[:, 1:, 1:] = planes.astype(np.int64).cumsum(1).cumsum(2)
    for _ in range(2000):
        c = int(rng.integers(0, 3)); px = int(rng.integers(0, 125 - 31)); py = int(rng.integers(0, 80 - 31))
        r = []
        for _k in range(2):
            w, h = int(rng.integers(1, 23)), int(rng.integers(1, 23))
            r.append((int(rng.integers(0, 31 - w)), int(rng.integers(0, 31 - h)), w, h))
        means = []
        for (x, y, w, h) in r:
            s = integ[c, py + y + h, px + x + w] - integ[c, py + y, px + x + w] - integ[c, py + y + h, px + x] + integ[c, py + y, px + x]
            means.append(int(s) // (w * h))
        assert rs.eval_test(c, r[0], r[1], px, py) == means[0] - means[1]
    rs.close()


def test_area_under_curve_matches_reference(O, R):
    rng = np.random.default_rng(11)
    T = np.array([-2.5, -0.35, -0.20, 0.20, 0.35, 2.5], np.float32)
    for _ in range(400):
        mean = float(np.float32(rng.uniform(-2, 2))); var = np.float32(10.0 ** rng.uniform(-6, 0.5))
        sd = float(np.sqrt(np.float64(var)))
        for j in range(5):
            a = R.area_under_curve(float(T[j]), float(T[j + 1]), mean, sd); b = O.area_under_curve(float(T[j]), float(T[j + 1]), mean, sd)
            assert a.tobytes() == b.tobytes()


def test_meanshift_matches_reference(O, R):
    rng = np.random.default_rng(3)
    for n in (0, 1, 2, 33, 1000, 20000):
        v = np.zeros((n, 3), np.float32)
        v[:, 0] = rng.integers(-30, 160, n); v[:, 1] = rng.integers(-30, 160, n); v[:, 2] = rng.choice([0.55, 0.6, 0.75, 1.0], n)
        rr, mr, ir = R.meanshift(v)
        mo, ro, io = O.meanshift(v)
        assert np.array_equal(rr, ro) and ir == io and mr.tobytes() == mo.tobytes(), n


def test_analyze_face_matches_reference_on_lfw(O, R, ff, om):
    """FaceForest::analyzeFace end to end on the shipped images: head pose bit-exact, the composed forest tree by tree, and
    the final landmarks (after both roundings)."""
    ff.set_strides(4, 3)
    for img, box in _lfw()[:10]:
        a = ff.analyze_face(img, box)
        b = om.analyze_face(img, box, threads=4)
        assert a["headpose"].tobytes() == b["headpose"].tobytes()
        counts, dom, fi, ti, _ = om.compose(b["headpose"], b["variance"])
        assert np.array_equal(a["list_forest"], fi) and np.array_equal(a["list_tree"], ti)
        assert np.array_equal(a["ffd"], b["ffd"])


def test_analyze_face_matches_reference_on_crops(O, R, ff, om):
    """Synthetic crops incl. pure noise (MeanShift runs to its cap) and a stride-1 face (BASELINE config 2)."""
    import cv2
    rng = np.random.default_rng(5)
    base = _lfw()[3]
    x, y, w, h = base[1]
    face = cv2.resize(base[0][y:y + h, x:x + w], (100, 100))
    crops = [face, rng.integers(0, 256, (100, 100, 3), dtype=np.uint8), cv2.GaussianBlur(rng.integers(0, 256, (120, 100, 3), dtype=np.uint8), (0, 0), 3)]
    ff.set_strides(4, 3)
    for c in crops:
        a = ff.analyze_face(c, (0, 0, c.shape[1], c.shape[0])); b = om.analyze_face(c, (0, 0, c.shape[1], c.shape[0]))
        assert a["headpose"].tobytes() == b["headpose"].tobytes() and np.array_equal(a["ffd"], b["ffd"])
    ff.set_strides(1, 1)
    a = ff.analyze_face(crops[0], (0, 0, 100, 100)); b = om.analyze_face(crops[0], (0, 0, 100, 100), 1, 1, threads=4)
    ff.set_strides(4, 3)
    assert a["headpose"].tobytes() == b["headpose"].tobytes() and np.array_equal(a["ffd"], b["ffd"])


def test_canonical_gabor_vs_neutral_direct_sum(O, R, ff, om):
    """How far is the canonical (separable) Gabor arithmetic from a neutral evaluation of cv::filter2D for the >= 9x9 kernels
    (double-accumulated direct sum, the closest f32 to the exact response)?  Planes: +-1 LSB only, at a rate < 2e-4; downstream on
    real faces: leaf ids of the head-pose forest differ in < 1e-3 of the traversals and the landmarks move by <= 1 px."""
    planes_c, planes_d = [], []
    faces = _lfw()[:4]
    for img, box in faces:
        x, y, w, h = box
        sw, sh, _ = O.scaled_size(w, h)
        g = O.resize(O.bgr2gray(img)[y:y + h, x:x + w], sh, sw)
        R.set_gabor_mode(0); sc = R.Sample(gray=g)
        R.set_gabor_mode(1); sd = R.Sample(gray=g)
        R.set_gabor_mode(0)
        ic, id_ = sc.integrals(), sd.integrals()
        pc = np.diff(np.diff(ic, axis=1), axis=2); pd = np.diff(np.diff(id_, axis=1), axis=2)   # back to the 8-bit planes
        planes_c.append(pc); planes_d.append(pd)
        assert np.array_equal(pc.astype(np.uint8), O.channels(g)[0])     # canonical mode == the oracle's planes
        lc, hc, vc = ff.eval_hp(sc, 4); ld, hd, vd = ff.eval_hp(sd, 4)
        assert (lc != ld).mean() < 1e-3 and abs(float(hc) - float(hd)) < 1e-3
        sc.close(); sd.close()
    d = np.concatenate([(a - b).ravel() for a, b in zip(planes_c, planes_d)])
    assert np.abs(d).max() <= 1 and (d != 0).mean() < 2e-4
    R.set_gabor_mode(1)
    try:
        for img, box in faces:
            a = ff.analyze_face(img, box); b = om.analyze_face(img, box)
            assert np.abs(a["ffd"] - b["ffd"]).max() <= 1 and abs(float(a["headpose"]) - float(b["headpose"])) < 1e-3
    finally:
        R.set_gabor_mode(0)
