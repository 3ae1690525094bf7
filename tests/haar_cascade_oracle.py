"""CPU restatement of cv::CascadeClassifier for every HAAR cascade OpenCV ships: tree weak classifiers, 45-degree (tilted) features and
the old opencv-haar-classifier XML format.  TEST INFRASTRUCTURE ONLY: the oracle for the GPU evaluator in csrc/haar.cuh.

It extends oracle/haar.py (stump cascades, upright features, new format), whose scales, pyramid, scan rule and grouping it reuses:
  tree     OpenCV's predictOrdered: from node 0, go left while value * (1 / nf) < threshold, until the child is <= 0, then add leaf -child
  tilted   a rect (x, y, w, h) sums T[y][x] - T[y+h][x-h] - T[y+w][x+w] + T[y+w+h][x+w-h] of the tilted integral T (CV_TILTED_OFS),
           T = cv2.integral3(img)[2], restated here from the row prefixes R(y, x) = sum_{x' < x} I(y, x'):
           T(Y, X) = sum_{y < Y} R(y, clamp(X + Y - 1 - y)) - R(y, clamp(X - Y + y))
  old XML  <size>, stages of <trees> of nodes (<feature>, <threshold>, left_val | left_node, right_val | right_node), <stage_threshold>;
           one feature per node, a tree's leaves numbered in node order, left before right
The arithmetic per window is the GPU's: f32 feature values and stage sums in the cascade's order.

Also here: the detector's device passes level by level (level_plan, level_image, level_integrals, window_flags), the reference of
crf_stage_haar_levels; and write_cascade, a seeded writer of synthetic cascades (trees of 1 to 3 nodes, tilted and upright features) in
either format.
"""
from __future__ import annotations

import xml.etree.ElementTree as ET
from pathlib import Path

import numpy as np

from oracle import haar as H


class Cascade:
    """Same attributes as oracle.haar.Cascade, generalised: features [nfeat][3][x, y, w, h, weight], tilted [nfeat] (bool), stages a
    list of (threshold f32, [tree, ...]) with tree = (nodes, leaves), nodes a list of (feature, threshold, left, right)."""

    def __init__(self, path: str | Path):
        top = ET.parse(str(path)).getroot()
        root = top.find("cascade")
        feats, tilted, self.stages = [], [], []

        def feature(f):
            rects = [[float(v) for v in r.text.split()] for r in f.find("rects")]
            while len(rects) < 3:
                rects.append([0, 0, 0, 0, 0.0])
            feats.append(rects)
            tilted.append(f.find("tilted") is not None and int(f.find("tilted").text) != 0)
            return len(feats) - 1

        if root is not None:
            self.format = "new"
            self.w, self.h = int(root.find("width").text), int(root.find("height").text)
            for f in root.find("features"):
                feature(f)
            for st in root.find("stages"):
                trees = []
                for wc in st.find("weakClassifiers"):
                    v = wc.find("internalNodes").text.split()
                    nodes = [(int(v[k + 2]), float(v[k + 3]), int(v[k]), int(v[k + 1])) for k in range(0, len(v), 4)]
                    trees.append((nodes, [float(x) for x in wc.find("leafValues").text.split()]))
                self.stages.append((np.float32(float(st.find("stageThreshold").text)), trees))
        else:
            root = next(k for k in top if k.get("type_id") == "opencv-haar-classifier")
            self.format = "old"
            self.w, self.h = (int(v) for v in root.find("size").text.split())
            for i, st in enumerate(root.find("stages")):
                assert int(st.find("parent").text) == i - 1 and int(st.find("next").text) == -1
                trees = []
                for tr in st.find("trees"):
                    nodes, leaves = [], []
                    for nd in tr:
                        fi = feature(nd.find("feature"))
                        kids = []
                        for side in ("left", "right"):
                            val = nd.find(side + "_val")
                            if val is not None:
                                kids.append(-len(leaves))
                                leaves.append(float(val.text))
                            else:
                                kids.append(int(nd.find(side + "_node").text))
                        nodes.append((fi, float(nd.find("threshold").text), kids[0], kids[1]))
                    trees.append((nodes, leaves))
                self.stages.append((np.float32(float(st.find("stage_threshold").text)), trees))
        self.features = np.array(feats, np.float64)
        self.tilted = np.array(tilted, bool)

    def counts(self):
        """(stages, weak classifiers, nodes, tilted features used by a node)"""
        trees = [t for _, ts in self.stages for t in ts]
        used = {n[0] for nodes, _ in trees for n in nodes}
        return len(self.stages), len(trees), sum(len(n) for n, _ in trees), int(sum(self.tilted[f] for f in used))


def tilted_integral(img: np.ndarray) -> np.ndarray:
    """cv2.integral3(img, sdepth=CV_32S)[2] for a u8 image, from the closed form above (u32 modulo 2^32, as cv2's int32)."""
    H_, W = img.shape
    R = np.zeros((H_, W + 1), np.uint32)
    R[:, 1:] = np.cumsum(img.astype(np.uint32), 1, dtype=np.uint32)
    T = np.zeros((H_ + 1, W + 1), np.uint32)
    X = np.arange(W + 1)
    for Y in range(1, H_ + 1):
        y = np.arange(Y)[:, None]
        a = R[y, np.clip(X[None, :] + Y - 1 - y, 0, W)]
        b = R[y, np.clip(X[None, :] - Y + y, 0, W)]
        T[Y] = (a.sum(0, dtype=np.uint32) - b.sum(0, dtype=np.uint32)).astype(np.uint32)
    return T.view(np.int32)


def cv2_stage_threshold(thr) -> np.float64:
    """The threshold cv2 compares a stage sum with: the file's value as float, minus THRESHOLD_EPS = 1e-5, stored as float."""
    return np.float64(np.float32(np.float64(np.float32(thr)) - 1e-5))


def stage_sums(c: Cascade, gray: np.ndarray, factor: float = 1.0, cv2_arith: bool = False):
    """Level `factor` of the pyramid: per window of its ystep grid, the stage sums ([nstages][ny][nx], NaN after the first failed
    stage), the window's validity (nf > 0 and area / nf < 0.1) and its top-left corner in the level.  The sums are the GPU's (f32 sum,
    passed when sum >= threshold) or, with cv2_arith, cv2's (double sum of the f32 leaves, passed when sum >= cv2_stage_threshold); the
    feature values and tree walks are the same f32 arithmetic in both."""
    Hh, W = gray.shape
    sw, sh = int(round(W / factor)), int(round(Hh / factor))
    img = H._resize(gray, sh, sw).astype(np.int64) if factor != 1.0 else gray.astype(np.int64)
    S = np.zeros((sh + 1, sw + 1), np.int64); S[1:, 1:] = img.cumsum(0).cumsum(1)
    Q = np.zeros((sh + 1, sw + 1), np.int64); Q[1:, 1:] = (img * img).cumsum(0).cumsum(1)
    T = cv2_tilted_integral(img.astype(np.uint8)).astype(np.int64) if c.tilted.any() else None
    ystep = 1 if factor > 2.0 else 2
    ys, xs = np.arange(0, sh - c.h + 1, ystep), np.arange(0, sw - c.w + 1, ystep)
    yy, xx = np.meshgrid(ys, xs, indexing="ij")

    def rs(A, x, y, w, h):
        return A[yy + y + h, xx + x + w] - A[yy + y, xx + x + w] - A[yy + y + h, xx + x] + A[yy + y, xx + x]

    def ts(x, y, w, h):
        return T[yy + y, xx + x] - T[yy + y + h, xx + x - h] - T[yy + y + w, xx + x + w] + T[yy + y + w + h, xx + x + w - h]

    area = float((c.w - 2) * (c.h - 2))
    vs = rs(S, 1, 1, c.w - 2, c.h - 2).astype(np.float64)
    vq = (rs(Q, 1, 1, c.w - 2, c.h - 2) & 0xffffffff).astype(np.float64)
    nf = area * vq - vs * vs
    ok = nf > 0
    inv = np.where(ok, 1.0 / np.sqrt(np.where(ok, nf, 1.0)), 1.0).astype(np.float32)
    ok &= (np.float32(area) * inv) < np.float32(0.1)
    cache = {}

    def value(fi):   # feature value x inv, f32, rects in order (u32 sums wrap as in the GPU's)
        if fi not in cache:
            v = np.zeros(ok.shape, np.float32)
            for x, y, w, h, wt in c.features[fi]:
                if wt != 0:
                    r = ts(int(x), int(y), int(w), int(h)) if c.tilted[fi] else rs(S, int(x), int(y), int(w), int(h))
                    v = v + np.float32(wt) * (r & 0xffffffff).astype(np.uint32).astype(np.float32)
            cache[fi] = v * inv
        return cache[fi]

    acc = np.float64 if cv2_arith else np.float32
    sums = np.full((len(c.stages),) + ok.shape, np.nan, acc)
    alive = ok.copy()
    for si, (thr, trees) in enumerate(c.stages):
        if not alive.any():
            break
        ssum = np.zeros(ok.shape, acc)
        for nodes, leaves in trees:
            idx = np.zeros(ok.shape, np.int64)
            done = np.zeros(ok.shape, bool)
            for _ in range(len(nodes)):
                nxt = idx.copy()
                for k, (fi, t, left, right) in enumerate(nodes):
                    at = ~done & (idx == k)
                    if at.any():
                        nxt[at] = np.where(value(fi)[at] < np.float32(t), left, right)
                done |= nxt <= 0
                idx = nxt
                if done.all():
                    break
            assert done.all()
            ssum = ssum + np.asarray(leaves, np.float32)[-idx].astype(acc)
        sums[si][alive] = ssum[alive]
        alive &= ssum >= (cv2_stage_threshold(thr) if cv2_arith else thr)
        cache.clear()
    return sums, ok, ys, xs


def window_flags(c: Cascade, sums, ok) -> np.ndarray:
    """The detector's flag byte of each window of a level from stage_sums' (sums, ok): 1 passed every stage, 2 rejected by stage 0, 0
    otherwise (rejected by a later stage, or skipped by the variance test: nf <= 0 or area / nf >= 0.1)."""
    passed = np.stack([sums[si] >= thr for si, (thr, _) in enumerate(c.stages)])
    return np.where(ok & passed.all(0), 1, np.where(ok & ~passed[0], 2, 0)).astype(np.uint8)


def scan_candidates(flags, ys, xs, factor, win):
    """OpenCV's scan of one level: windows in (iy, ix) order, one extra step after a stage-0 reject; the visited windows that passed every
    stage, as frame rectangles."""
    rej0 = (flags & 2) != 0
    pos = np.arange(flags.shape[1])
    # a window is visited when an even number of stage-0 rejects precede it in its row (each visited reject skips the next window)
    last = np.maximum.accumulate(np.where(rej0, -1, pos), axis=1)   # last position at or before ix that stage 0 did not reject
    run = np.zeros(flags.shape, np.int64)
    run[:, 1:] = pos[:-1] - last[:, :-1]
    iy, ix = np.nonzero(((flags & 1) != 0) & (run % 2 == 0))
    x, y = np.rint(xs[ix] * factor).astype(np.int64), np.rint(ys[iy] * factor).astype(np.int64)
    return [(int(a), int(b), win[0], win[1]) for a, b in zip(x, y)]


def detect_levels(c: Cascade, gray: np.ndarray, scale_factor: float = 1.3, min_size: int = 30):
    """Per level of level_plan: (level, window flags [ny][nx], ys, xs)."""
    for L in level_plan(c.w, c.h, *gray.shape, scale_factor, min_size):
        sums, ok, ys, xs = stage_sums(c, gray, L["factor"])
        yield L, window_flags(c, sums, ok), ys, xs


def level_candidates(levels):
    """The raw candidates of detect_levels' levels, in (level, iy, ix) order."""
    return [r for L, flags, ys, xs in levels for r in scan_candidates(flags, ys, xs, L["factor"], (L["win_w"], L["win_h"]))]


def detect_candidates(c: Cascade, gray: np.ndarray, scale_factor: float = 1.3, min_size: int = 30):
    """oracle.haar.detect_candidates for any cascade: raw candidates in (level, iy, ix) order."""
    return level_candidates(detect_levels(c, gray, scale_factor, min_size))


# ---- the detector's device passes, level by level ----------------------------------------------------------------------------------
def level_plan(win_w: int, win_h: int, rows: int, cols: int, scale_factor: float, min_size: int = 0) -> list:
    """The pyramid levels of one rows x cols frame, as detect_plan (csrc/engine.cu) and oracle.haar's scale loop build them: factor = 1,
    scale_factor, scale_factor^2, ...; the level is round(cols / factor) x round(rows / factor) and the window round(win * factor); the
    loop stops when the window exceeds the frame or the level is smaller than the cascade's window, and skips levels whose window is
    below min_size.  Windows lie ystep level pixels apart (2 while factor <= 2, then 1).  One dict per level with the fields of
    crf_haar_level_t."""
    out = []
    factor = 1.0
    while True:
        ww, wh = int(round(win_w * factor)), int(round(win_h * factor))
        sw, sh = int(round(cols / factor)), int(round(rows / factor))
        if ww > cols or wh > rows or sw < win_w or sh < win_h:
            return out
        if ww >= min_size and wh >= min_size:
            ystep = 1 if factor > 2.0 else 2
            out.append(dict(factor=factor, sw=sw, sh=sh, ystep=ystep, nx=(sw - win_w + ystep) // ystep, ny=(sh - win_h + ystep) // ystep,
                            win_w=ww, win_h=wh))
        factor *= scale_factor


def level_image(gray: np.ndarray, level: dict) -> np.ndarray:
    """The level's u8 pixels: oracle.haar's bilinear resize of the gray frame (the frame itself at factor 1)."""
    return H._resize(gray, level["sh"], level["sw"]) if level["factor"] != 1.0 else gray


def cv2_tilted_integral(img: np.ndarray) -> np.ndarray:
    """cv2.integral3(img)[2] as u32: the tilted integral tilted_integral restates (test_tilted_integral_equals_cv2), at cv2's speed."""
    import cv2
    return cv2.integral3(np.ascontiguousarray(img, np.uint8), sdepth=cv2.CV_32S)[2].view(np.uint32)


def level_integrals(img: np.ndarray, tilted: bool = True):
    """(S, Q, T) of a u8 level image, each [(h + 1) x (w + 1)] u32: the integrals of the values and of their squares (np.cumsum in u64,
    reduced modulo 2^32 as the detector's u32 sums are) and the tilted integral (None unless tilted)."""
    h, w = img.shape
    v = img.astype(np.uint64)
    S = np.zeros((h + 1, w + 1), np.uint64)
    Q = np.zeros((h + 1, w + 1), np.uint64)
    S[1:, 1:] = np.cumsum(np.cumsum(v, 0), 1)
    Q[1:, 1:] = np.cumsum(np.cumsum(v * v, 0), 1)
    m = np.uint64(0xffffffff)
    return (S & m).astype(np.uint32), (Q & m).astype(np.uint32), cv2_tilted_integral(img) if tilted else None


def detect_multi_scale(c: Cascade, bgr_or_gray: np.ndarray, scale_factor: float = 1.3, min_neighbors: int = 1, min_size: int = 30):
    from oracle import oracle as O
    gray = O.bgr2gray(bgr_or_gray) if bgr_or_gray.ndim == 3 else bgr_or_gray
    return H.group_rectangles(detect_candidates(c, gray, scale_factor, min_size), min_neighbors)


# ---- synthetic cascades ---------------------------------------------------------------------------------------------------------------
def _random_feature(rng, w, h, tilted):
    """Two rects, a rect and half of it, weights -1 and 2: upright, or tilted inside the window (x - h >= 0, x + w <= W, y + w + h <= H)."""
    if not tilted:
        horizontal = rng.random() < 0.5
        a = int(rng.integers(1, (w if horizontal else h) // 2 + 1))
        b = int(rng.integers(1, (h if horizontal else w) + 1))
        if horizontal:
            x, y = int(rng.integers(0, w - 2 * a + 1)), int(rng.integers(0, h - b + 1))
            return [(x, y, 2 * a, b, -1.0), (x + a, y, a, b, 2.0)]
        x, y = int(rng.integers(0, w - b + 1)), int(rng.integers(0, h - 2 * a + 1))
        return [(x, y, b, 2 * a, -1.0), (x, y + a, b, a, 2.0)]
    lim = min(w, h)
    while True:
        rw, rh = 2 * int(rng.integers(1, lim // 4 + 1)), int(rng.integers(1, lim // 2 + 1))
        if rw + rh <= h and rw + rh <= w:
            break
    x, y = int(rng.integers(rh, w - rw + 1)), int(rng.integers(0, h - rw - rh + 1))
    return [(x, y, rw, rh, -1.0), (x, y, rw // 2, rh, 2.0)]


def _random_tree(rng, nodes):
    """(left, right) children of `nodes` nodes (1 to 3), each child node after its parent, leaves numbered in node order, left before
    right (leaf k is the child -k, so leaf 0 is the child 0)."""
    shapes = {1: [((0, -1),)], 2: [((1, 0), (-1, -2)), ((0, 1), (-1, -2))],
              3: [((1, 2), (0, -1), (-2, -3)), ((1, 0), (2, -1), (-2, -3)), ((0, 1), (-1, 2), (-2, -3))]}
    return list(shapes[nodes][int(rng.integers(len(shapes[nodes])))])


def write_cascade(path, w=20, h=20, stage_sizes=(3, 5, 7, 5, 9), seed=7, max_nodes=3, p_tilted=0.5, fmt="new"):
    """write_stump_cascade of test_gpu_detect_batch.py generalised: weak classifiers are random trees of 1 to max_nodes nodes, features
    tilted with probability p_tilted, node thresholds within 1e-3 of 0 and leaves near -1 / +1 of alternating sign, stage thresholds 0, so that on texture many windows
    survive each stage.  fmt "new" (opencv-cascade-classifier) or "old" (opencv-haar-classifier); the same seed gives the same cascade
    in both, with one feature per node in node order."""
    rng = np.random.default_rng(seed)
    stages = []
    for n in stage_sizes:
        trees = []
        for _ in range(n):
            kids = _random_tree(rng, int(rng.integers(1, max_nodes + 1)))
            nodes = []
            for l, r in kids:
                tilt = bool(rng.random() < p_tilted)
                nodes.append((_random_feature(rng, w, h, tilt), tilt, float(rng.uniform(-1e-3, 1e-3)), l, r))
            sign = 1 if rng.random() < 0.5 else -1   # leaves alternate in sign, so every tree splits the windows
            leaves = [float(rng.uniform(0.8, 1.2)) * sign * (-1) ** k for k in range(len(nodes) + 1)]
            trees.append((nodes, leaves))
        stages.append(trees)
    rects_xml = lambda rects, ind: [ind + "<rects>"] + [f"{ind}  <_>{x} {y} {rw} {rh} {wt:.1f}</_>" for x, y, rw, rh, wt in rects] + [ind + "</rects>"]
    if fmt == "new":
        feats = []
        out = ['<?xml version="1.0"?>', "<opencv_storage>", '<cascade type_id="opencv-cascade-classifier">', "  <stageType>BOOST</stageType>",
               "  <featureType>HAAR</featureType>", f"  <height>{h}</height>", f"  <width>{w}</width>",
               "  <stageParams><boostType>GAB</boostType><minHitRate>0.995</minHitRate><maxFalseAlarm>0.5</maxFalseAlarm>"
               f"<weightTrimRate>0.95</weightTrimRate><maxDepth>{max_nodes}</maxDepth><maxWeakCount>100</maxWeakCount></stageParams>",
               "  <featureParams><maxCatCount>0</maxCatCount><featSize>1</featSize><mode>ALL</mode></featureParams>",
               f"  <stageNum>{len(stages)}</stageNum>", "  <stages>"]
        for trees in stages:
            out += ["    <_>", f"      <maxWeakCount>{len(trees)}</maxWeakCount>", "      <stageThreshold>0.</stageThreshold>", "      <weakClassifiers>"]
            for nodes, leaves in trees:
                internal = []
                for rects, tilt, t, l, r in nodes:
                    feats.append((rects, tilt))
                    internal += [str(l), str(r), str(len(feats) - 1), repr(t)]
                out += ["        <_>", f"          <internalNodes>{' '.join(internal)}</internalNodes>",
                        f"          <leafValues>{' '.join(repr(v) for v in leaves)}</leafValues></_>"]
            out += ["      </weakClassifiers></_>"]
        out += ["  </stages>", "  <features>"]
        for rects, tilt in feats:
            out += ["    <_>"] + rects_xml(rects, "      ") + [f"      <tilted>{int(tilt)}</tilted></_>"]
        out += ["  </features>", "</cascade>", "</opencv_storage>", ""]
    else:
        out = ['<?xml version="1.0"?>', "<opencv_storage>", '<synthetic_cascade type_id="opencv-haar-classifier">', f"  <size>{w} {h}</size>", "  <stages>"]
        for si, trees in enumerate(stages):
            out += ["    <_>", "      <trees>"]
            for nodes, leaves in trees:
                out += ["        <_>"]
                li = 0
                for rects, tilt, t, l, r in nodes:
                    out += ["          <_>", "            <feature>"] + rects_xml(rects, "              ") + \
                           [f"              <tilted>{int(tilt)}</tilted></feature>", f"            <threshold>{t!r}</threshold>"]
                    for side, ch in (("left", l), ("right", r)):
                        if ch > 0:
                            out += [f"            <{side}_node>{ch}</{side}_node>"]
                        else:
                            assert -ch == li
                            out += [f"            <{side}_val>{leaves[li]!r}</{side}_val>"]
                            li += 1
                    out += ["          </_>"]
                out += ["        </_>"]
            out += ["      </trees>", "      <stage_threshold>0.</stage_threshold>", f"      <parent>{si - 1}</parent>", "      <next>-1</next></_>"]
        out += ["  </stages>", "</synthetic_cascade>", "</opencv_storage>", ""]
    Path(path).write_text("\n".join(out))
    return str(path)



def truncate_cascade(src, dst, nstages):
    """A copy of the cascade at src (either format) with its first nstages stages only: the same features, trees and tilted rects, but
    windows on texture pass, so comparisons on cascades that find nothing in test frames (bodies, plates, profiles) are not empty."""
    tree = ET.parse(str(src))
    top = tree.getroot()
    root = top.find("cascade")
    if root is None:
        root = next(k for k in top if k.get("type_id") == "opencv-haar-classifier")
    stages = root.find("stages")
    for st in list(stages)[nstages:]:
        stages.remove(st)
    if root.find("stageNum") is not None:
        root.find("stageNum").text = str(nstages)
    Path(dst).write_text('<?xml version="1.0"?>\n' + ET.tostring(top, encoding="unicode") + "\n")
    return str(dst)
