"""Every OpenCV HAAR cascade on the detector: tree weak classifiers, tilted features and the old XML format (CPU side).

The loader (crf_cascade_load) and the oracle (tests/haar_cascade_oracle.py) read the 17 cascades of the cv2 package and the seeded
synthetic ones in both XML formats; the oracle is pinned against cv2 itself, window for window, on one pyramid level; malformed trees
and unsupported layouts fail at load time."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

import haar_cascade_oracle as G

cv2 = pytest.importorskip("cv2")
CV2_DIR = Path(cv2.data.haarcascades)
CV2_CASCADES = sorted(p.name for p in CV2_DIR.glob("haarcascade_*.xml"))
ERR_FORMAT, ERR_UNSUPPORTED = -3, -6


def load(crf, path):
    """(rc, (win_w, win_h, nstages, nweak) or None)"""
    L = crf.lib()
    h = C.c_void_p()
    rc = L.crf_cascade_load(str(path).encode(), C.byref(h))
    if rc:
        return rc, None
    v = [C.c_int() for _ in range(4)]
    assert L.crf_cascade_info(h, *[C.byref(x) for x in v]) == 0
    L.crf_cascade_free(h)
    return rc, tuple(x.value for x in v)


def xml_counts(path):
    """(stages, weak classifiers, nodes, tilted features used) counted from the XML text directly."""
    s = Path(path).read_text()
    if "opencv-haar-classifier" in s:
        stages = len(re.findall(r"<stage_threshold>", s))
        nodes = len(re.findall(r"<threshold>", s))
        weak = len(re.findall(r"<!-- tree \d+ -->", s)) or None
        tilted = len(re.findall(r"<tilted>\s*1\s*</tilted>", s))
        return stages, weak, nodes, tilted
    stages = len(re.findall(r"<stageThreshold>", s))
    internal = re.findall(r"<internalNodes>([^<]*)</internalNodes>", s)
    nodes = sum(len(t.split()) // 4 for t in internal)
    used = {int(t.split()[k + 2]) for t in internal for k in range(0, len(t.split()), 4)}
    feats = re.search(r"<features>(.*)</features>", s, re.S).group(1)
    flags = [int(m) for m in re.findall(r"<tilted>\s*(\d)\s*</tilted>", feats)]
    tilted = sum(1 for f in used if f < len(flags) and flags[f]) if flags else 0
    return stages, len(internal), nodes, tilted


@pytest.fixture(scope="module")
def synth(tmp_path_factory):
    """Seeded synthetic cascades, each in both formats: {name: (new-format path, old-format path)}."""
    d = tmp_path_factory.mktemp("cascades")
    out = {}
    for name, kw in {"trees_tilted": dict(seed=3), "trees": dict(seed=4, p_tilted=0.0), "tilted_stumps": dict(seed=5, max_nodes=1, p_tilted=0.6),
                     "flat_24x12": dict(seed=6, w=24, h=12, stage_sizes=(3, 5, 5))}.items():
        out[name] = tuple(G.write_cascade(d / f"{name}_{fmt}.xml", fmt=fmt, **kw) for fmt in ("new", "old"))
    return out


def _textured(rows, cols, seed):
    rng = np.random.default_rng(seed)
    return cv2.GaussianBlur(rng.integers(0, 256, (rows, cols), dtype=np.uint8), (0, 0), 1.5)


# ---- tilted integral ----------------------------------------------------------------------------------------------------------------
def test_tilted_integral_equals_cv2():
    rng = np.random.default_rng(1)
    for shape in [(1, 1), (1, 9), (9, 1), (2, 2), (7, 13), (30, 41), (41, 30), (33, 1), (1, 33), (64, 63)]:
        img = rng.integers(0, 256, shape, dtype=np.uint8)
        assert np.array_equal(G.tilted_integral(img), cv2.integral3(img, sdepth=cv2.CV_32S)[2]), shape
    img = np.full((17, 23), 255, np.uint8)
    assert np.array_equal(G.tilted_integral(img), cv2.integral3(img, sdepth=cv2.CV_32S)[2])


# ---- loading ------------------------------------------------------------------------------------------------------------------------
def test_cv2_cascades_all_load(crf):
    assert len(CV2_CASCADES) == 17
    for name in CV2_CASCADES:
        path = CV2_DIR / name
        rc, info = load(crf, path)
        assert rc == 0, (name, crf.lib().crf_last_error())
        c = G.Cascade(path)
        stages, weak, nodes, tilted = c.counts()
        want = xml_counts(path)
        assert (stages, nodes, tilted) == (want[0], want[2], want[3]), name
        if want[1] is not None:
            assert weak == want[1], name
        assert info == (c.w, c.h, stages, weak), name
    # what makes each one new: trees, tilted features, the old format
    kinds = {n: G.Cascade(CV2_DIR / n) for n in ("haarcascade_frontalface_alt2.xml", "haarcascade_eye_tree_eyeglasses.xml", "haarcascade_smile.xml",
                                                 "haarcascade_license_plate_rus_16stages.xml")}
    assert kinds["haarcascade_frontalface_alt2.xml"].counts()[2] > kinds["haarcascade_frontalface_alt2.xml"].counts()[1]
    assert kinds["haarcascade_eye_tree_eyeglasses.xml"].counts()[3] > 0 and kinds["haarcascade_smile.xml"].counts()[3] > 0
    assert kinds["haarcascade_license_plate_rus_16stages.xml"].format == "old"


def test_synthetic_cascades_both_formats(crf, synth):
    """The product's parse and the oracle's agree for both formats; cv2 loads both and finds the same candidates in each."""
    img = _textured(121, 161, 2)
    for name, (new, old) in synth.items():
        cn, co = G.Cascade(new), G.Cascade(old)
        assert (cn.w, cn.h, cn.counts()) == (co.w, co.h, co.counts()), name
        assert cn.stages == co.stages and np.array_equal(cn.features, co.features) and np.array_equal(cn.tilted, co.tilted), name
        assert load(crf, new) == load(crf, old) == (0, (cn.w, cn.h, len(cn.stages), cn.counts()[1])), name
        a, b = cv2.CascadeClassifier(new), cv2.CascadeClassifier(old)
        assert not a.empty() and not b.empty()
        ra = sorted(map(tuple, np.asarray(a.detectMultiScale(img, 1.2, 0)).reshape(-1, 4).tolist()))
        rb = sorted(map(tuple, np.asarray(b.detectMultiScale(img, 1.2, 0)).reshape(-1, 4).tolist()))
        assert ra == rb and len(ra) > 10, name
    assert G.Cascade(synth["trees_tilted"][0]).counts()[3] > 0 and G.Cascade(synth["trees"][0]).counts()[2] > G.Cascade(synth["trees"][0]).counts()[1]


# ---- the oracle against cv2, one pyramid level -------------------------------------------------------------------------------------
def _level0(cascade_path, c, gray):
    """cv2's and the oracle's raw candidates on level 0 only (minNeighbors 0, a scale factor past the frame), and the oracle's stage sums.
    cv2 4.13 splits a level's window rows into stripes of (rows / ystep) windows rounded down, which can leave out the last window row
    when H - h is even: the frames here have H - h odd, so both scan the same grid."""
    Hh, W = gray.shape
    assert (Hh - c.h) % 2 == 1
    sf = 1.01 + max(W / c.w, Hh / c.h)
    got = sorted(map(tuple, np.asarray(cv2.CascadeClassifier(str(cascade_path)).detectMultiScale(gray, sf, 0)).reshape(-1, 4).tolist()))
    want = sorted(G.detect_candidates(c, gray, sf, 0))
    return got, want


def _deciding_stage_is_a_knife_edge(c, gray, box):
    """A window on which the oracle and cv2 disagree must be decided by rounding.  The oracle sums a stage in f32 and passes it when
    sum >= threshold (the GPU's arithmetic); cv2 sums it in double and passes it when sum >= float(threshold) - 1e-5.  The feature values
    and tree walks are the same f32 arithmetic in both.  With both restated, the first stage whose decisions differ must exist, and the
    oracle's f32 sum there must lie within cv2's 1e-5 margin plus the f32 rounding of its sum of that stage's leaves."""
    s32 = G.stage_sums(c, gray)[0][:, box[1] // 2, box[0] // 2]
    s64 = G.stage_sums(c, gray, cv2_arith=True)[0][:, box[1] // 2, box[0] // 2]
    for si, (thr, trees) in enumerate(c.stages):
        if np.isnan(s32[si]) or np.isnan(s64[si]):
            return False   # both decided the same way on every stage they reached: the difference is not in the stage sums
        if bool(s32[si] >= thr) != bool(s64[si] >= G.cv2_stage_threshold(thr)):
            ulp = np.spacing(np.float32(max(abs(float(s64[si])), abs(float(thr)), 1.0)))
            return abs(float(s32[si]) - float(thr)) <= 1e-5 + len(trees) * float(ulp)
    return False


def _compare_level0(path, c, frames):
    """The raw level-0 candidates of cv2 and of the oracle; every window in only one of them is a knife edge.  Returns cv2's count."""
    found = 0
    for gray in frames:
        gray = gray[: gray.shape[0] - (1 - (gray.shape[0] - c.h) % 2)]
        got, want = _level0(path, c, gray)
        for box in set(got) ^ set(want):
            assert _deciding_stage_is_a_knife_edge(c, gray, box), (Path(path).name, box, box in want)
        found += len(got)
    return found


def test_oracle_equals_cv2_on_synthetic_cascades(synth):
    for name, (new, old) in synth.items():
        c = G.Cascade(new)
        frames = [_textured(121, 161, 5), _textured(97, 130, 6)]
        assert _compare_level0(new, c, frames) > 0, name
        assert _compare_level0(old, c, frames) > 0, name


@pytest.mark.parametrize("name", ["haarcascade_eye_tree_eyeglasses.xml", "haarcascade_lefteye_2splits.xml", "haarcascade_smile.xml",
                                  "haarcascade_frontalface_alt2.xml", "haarcascade_license_plate_rus_16stages.xml"])
def test_oracle_equals_cv2_on_shipped_cascades(O, name, tmp_path):
    """The shipped tree / tilted / old-format cascades on the procedural faces at their own size and downscaled (faces of about 20-60 px),
    and their first 4 and 8 stages (2 and 4 for the plates), which pass many more windows through the same trees and tilted rects.  Minimum counts keep every
    comparison from being empty."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    grays = [O.bgr2gray(f["img"]) for f in wl.procedural_lfw()]
    scaled = grays + [cv2.resize(g, (s, s), interpolation=cv2.INTER_AREA) for g in grays for s in (70, 90, 130, 170)]
    full = G.Cascade(CV2_DIR / name)
    n_full = _compare_level0(CV2_DIR / name, full, scaled)
    if "license_plate" not in name:   # no plates in these frames: only its truncated copies find windows
        assert n_full >= 2, (name, n_full)
    for k in ((2, 4) if "license_plate" in name else (4, 8)):
        path = G.truncate_cascade(CV2_DIR / name, tmp_path / f"{k}_{name}", k)
        n = _compare_level0(path, G.Cascade(path), grays[:8])
        assert n >= 20, (name, k, n)


# ---- malformed cascades ----------------------------------------------------------------------------------------------------------
def _edit(src, dst, pattern, repl, count=1):
    s = Path(src).read_text()
    t = re.sub(pattern, repl, s, count=count)
    assert t != s
    Path(dst).write_text(t)
    return str(dst)


def test_malformed_cascades_fail_cleanly(crf, synth, tmp_path):
    new, old = synth["trees"]
    s = Path(new).read_text()
    # the first tree with more than one node: its first child node index
    m = re.search(r"<internalNodes>((?:\s*-?\d+\s+-?\d+\s+\d+\s+\S+){2,})\s*</internalNodes>", s)
    assert m
    v = m.group(1).split()
    cases = []
    k = 0 if int(v[0]) > 0 else 1   # the side of node 0 that names node 1
    # node 1 points back at node 1 (itself): not after its parent
    selfloop = list(v); selfloop[4] = "1"
    cases.append(("self", selfloop, "does not follow"))
    # node 0's child points at a node past the tree
    past = list(v); past[k] = str(len(v) // 4)
    cases.append(("past", past, "does not follow"))
    # a leaf index out of range
    leaf = list(v); leaf[5] = str(-(len(v) // 4 + 1))
    cases.append(("leaf", leaf, "leaf index out of range"))
    # node 1 unreachable: node 0 has two leaves
    unreach = list(v); unreach[0], unreach[1] = "0", "-1"
    cases.append(("unreachable", unreach, "unreachable"))
    for tag, vals, msg in cases:
        p = tmp_path / f"bad_{tag}.xml"
        p.write_text(s.replace(m.group(0), "<internalNodes>" + " ".join(vals) + "</internalNodes>", 1))
        assert load(crf, p)[0] == ERR_FORMAT, tag
        assert msg in crf.lib().crf_last_error().decode(), (tag, crf.lib().crf_last_error())
    # a backward child in the old format, the leaf count kept: node 1 of a tree whose node 1 has a child node names itself (a cycle)
    import xml.etree.ElementTree as ET
    top = ET.parse(old).getroot()
    nodes1 = [tree[1] for st in top.find("synthetic_cascade").find("stages") for tree in st.find("trees") if len(tree) >= 3]
    node1 = next(n for n in nodes1 if n.find("left_node") is not None or n.find("right_node") is not None)
    (node1.find("left_node") if node1.find("left_node") is not None else node1.find("right_node")).text = "1"
    (tmp_path / "bad_cycle_old.xml").write_text('<?xml version="1.0"?>\n' + ET.tostring(top, encoding="unicode"))
    assert load(crf, tmp_path / "bad_cycle_old.xml")[0] == ERR_FORMAT
    assert "does not follow" in crf.lib().crf_last_error().decode()
    # a tilted rect outside the window (x - h < 0)
    tn = synth["tilted_stumps"][0]
    st = Path(tn).read_text()
    i = st.index("<tilted>1</tilted>")
    r0 = st.rindex("<rects>", 0, i)
    mt = re.compile(r"<_>(\d+) (\d+) (\d+) (\d+) (\S+)</_>").search(st, r0)
    x, y, w, h = (int(mt.group(k)) for k in range(1, 5))
    bad = st[:mt.start()] + f"<_>{h - 1} {y} {w} {h} {mt.group(5)}</_>" + st[mt.end():]
    (tmp_path / "bad_tilt.xml").write_text(bad)
    assert load(crf, tmp_path / "bad_tilt.xml")[0] == ERR_FORMAT
    # old format with branching stages
    assert load(crf, _edit(old, tmp_path / "branch.xml", r"<parent>1</parent>", "<parent>0</parent>"))[0] == ERR_UNSUPPORTED
    assert load(crf, _edit(old, tmp_path / "next.xml", r"<next>-1</next>", "<next>2</next>"))[0] == ERR_UNSUPPORTED
    # LBP features, categorical splits
    assert load(crf, _edit(new, tmp_path / "lbp.xml", r"<featureType>HAAR</featureType>", "<featureType>LBP</featureType>"))[0] == ERR_UNSUPPORTED
    assert load(crf, _edit(new, tmp_path / "cat.xml", r"<maxCatCount>0</maxCatCount>", "<maxCatCount>256</maxCatCount>"))[0] == ERR_UNSUPPORTED
    # an unknown layout
    p = tmp_path / "other.xml"
    p.write_text('<?xml version="1.0"?>\n<opencv_storage>\n<thing type_id="opencv-matrix"><rows>1</rows></thing>\n</opencv_storage>\n')
    assert load(crf, p)[0] == ERR_FORMAT


# ---- the level reference of the detector's device passes (crf_stage_haar_levels) -------------------------------------------------------
def test_level_integrals_equal_cv2():
    """S equals cv2.integral, Q cv2.integral2's square sums modulo 2^32 and T the closed-form tilted integral, on levels whose square sums
    pass 2^32 (so Q wraps): a bright textured frame, an all-255 frame and a 0/255 checkerboard."""
    from oracle import oracle as O
    rng = np.random.default_rng(3)
    bright = cv2.GaussianBlur(rng.integers(128, 256, (330, 420, 3), dtype=np.uint8), (0, 0), 1.0)
    white = np.full((300, 330, 3), 255, np.uint8)
    check = np.repeat(((np.indices((320, 420)).sum(0) % 2) * 255).astype(np.uint8)[..., None], 3, 2)
    for frame in (bright, white, check):
        gray = O.bgr2gray(frame)
        plan = G.level_plan(20, 20, *gray.shape, 1.3)
        assert len(plan) >= 3
        wrapped = False
        for L in plan[:3]:
            img = G.level_image(gray, L)
            assert img.shape == (L["sh"], L["sw"])
            S, Q, T = G.level_integrals(img)
            assert np.array_equal(S, cv2.integral(img, sdepth=cv2.CV_32S).view(np.uint32))
            q = cv2.integral2(img, sdepth=cv2.CV_32S, sqdepth=cv2.CV_64F)[1]
            assert np.array_equal(Q, (q.astype(np.uint64) & np.uint64(0xffffffff)).astype(np.uint32))
            assert np.array_equal(T, G.tilted_integral(img).view(np.uint32))
            wrapped |= q[-1, -1] >= 2.0 ** 32
        assert wrapped


def test_level_plan_equals_oracle_scale_loop(monkeypatch):
    """level_plan gives the levels of oracle.haar.detect_candidates' scale loop: the level sizes it resizes to, its window grids (count
    and ystep) and the levels it skips below min_size or stops at, for scale factors 1.05 to 2.5 and frames from 1 x 1 to 1080p."""
    from oracle import haar as H
    c = H.Cascade(CV2_DIR / "haarcascade_frontalface_alt.xml")
    seen = []
    real_meshgrid = np.meshgrid
    # the oracle's scale loop on zero frames: every window fails the variance test, so only the loop itself runs
    monkeypatch.setattr(H, "_resize", lambda gray, dh, dw: (seen.append(("resize", dh, dw)), np.zeros((dh, dw), np.uint8))[1])

    class RecordingNumpy:
        def __getattr__(self, name):
            return getattr(np, name)

        @staticmethod
        def meshgrid(ys, xs, **kw):
            seen.append(("grid", len(ys), len(xs), int(xs[1] - xs[0]) if len(xs) > 1 else None))
            return real_meshgrid(ys, xs, **kw)

    monkeypatch.setattr(H, "np", RecordingNumpy())
    ystep1 = ystep2 = skipped = 0
    for rows, cols in [(250, 250), (480, 640), (97, 131), (20, 20), (21, 21), (19, 19), (1, 1), (48, 4000), (4000, 48), (1080, 1920)]:
        for sf in (1.05, 1.1, 1.3, 2.5):
            for ms in (0, 30, 50, 100):
                seen.clear()
                assert H.detect_candidates(c, np.zeros((rows, cols), np.uint8), sf, ms) == []
                plan = G.level_plan(c.w, c.h, rows, cols, sf, ms)
                want = []
                for L in plan:
                    if L["factor"] != 1.0:
                        want.append(("resize", L["sh"], L["sw"]))
                    want.append(("grid", L["ny"], L["nx"], L["ystep"] if L["nx"] > 1 else None))
                    assert (L["win_w"], L["win_h"]) == (int(round(20 * L["factor"])), int(round(20 * L["factor"]))) and min(L["win_w"], L["win_h"]) >= ms
                    ystep1 += L["ystep"] == 1
                    ystep2 += L["ystep"] == 2
                assert seen == want, (rows, cols, sf, ms)
                skipped += len(plan) < len(G.level_plan(c.w, c.h, rows, cols, sf, 0))
    assert ystep1 and ystep2 and skipped


def test_level_candidates_equal_oracle(tmp_path):
    """detect_candidates through level_plan, window_flags and the scan of scan_candidates gives oracle.haar.detect_candidates' raw
    candidates for a stump cascade (the face cascade's first stages and a synthetic one)."""
    from oracle import haar as H
    from oracle import oracle as O
    from test_gpu_detect_batch import write_stump_cascade
    paths = [G.truncate_cascade(CV2_DIR / "haarcascade_frontalface_alt.xml", tmp_path / "face3.xml", 3), write_stump_cascade(tmp_path / "stumps.xml")]
    found = 0
    for path in paths:
        for k, (rows, cols) in enumerate([(161, 203), (240, 320)]):
            gray = O.bgr2gray(cv2.cvtColor(_textured(rows, cols, 40 + k), cv2.COLOR_GRAY2BGR))
            for sf, ms in ((1.1, 0), (1.3, 30), (2.5, 0)):
                want = H.detect_candidates(H.Cascade(path), gray, sf, ms)
                assert G.detect_candidates(G.Cascade(path), gray, sf, ms) == want, (path, rows, sf, ms)
                found += len(want)
    assert found > 0
