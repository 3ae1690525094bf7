"""Synthetic inputs of the benchmark configurations (SURVEY.md §8d; BASELINE.json `configs`).

Deterministic from fixed seeds so the CPU baseline and the GPU read identical bytes.  The LFW
fixtures (20 jpgs + index_random_subset.txt of the reference's data/imgs) are looked up under
staged/imgs (tools/stage_data.py); without them the generators fall back to procedural blobs and
say so in the returned `data` tag.
"""
from __future__ import annotations

import os
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
STAGED = ROOT / "staged"


def staged_model_path() -> Path | None:
    if os.environ.get("CRF_NO_STAGED"):   # exercise the fallbacks (seeded random forests, procedural faces)
        return None
    p = STAGED / "model.crfb200"
    return p if p.exists() else None


def load_lfw(dir_: Path | None = None):
    """Parses index_random_subset.txt (src/face_utils.cpp:142-181): name x y w h pose n (x y)*n.
    Returns a list of dicts(img BGR u8, box (x,y,w,h), pose, parts [10,2] bbox-relative)."""
    import cv2
    dir_ = Path(dir_) if dir_ else STAGED / "imgs"
    idx = dir_ / "index_random_subset.txt"
    if not idx.exists() or os.environ.get("CRF_NO_STAGED"):
        return []
    out = []
    for line in idx.read_text().split("\n"):
        t = line.split()
        if len(t) < 7:
            continue
        img = cv2.imread(str(dir_ / t[0]), cv2.IMREAD_COLOR)
        if img is None:
            continue
        x, y, w, h, pose, n = (int(v) for v in t[1:7])
        parts = np.array([int(v) for v in t[7:7 + 2 * n]], np.int32).reshape(n, 2)
        out.append(dict(name=t[0], img=img, box=(x, y, w, h), pose=pose, parts=parts))
    return out


def _procedural_face(rng: np.random.Generator, size: int = 130) -> np.ndarray:
    """Smooth blobs standing in for a face when the LFW fixtures are not staged."""
    import cv2
    g = rng.uniform(60, 200, (size // 8 + 2, size // 8 + 2, 3)).astype(np.float32)
    img = cv2.resize(g, (size, size), interpolation=cv2.INTER_CUBIC)
    yy, xx = np.mgrid[0:size, 0:size]
    for cx, cy, r, v in [(0.33, 0.4, 0.07, -80), (0.67, 0.4, 0.07, -80), (0.5, 0.72, 0.12, -50), (0.5, 0.55, 0.05, 30)]:
        img += v * np.exp(-(((xx - cx * size) ** 2 + (yy - cy * size) ** 2) / (2 * (r * size) ** 2)))[..., None]
    return np.clip(img, 0, 255).astype(np.uint8)


def procedural_lfw(n: int = 20, seed: int = 2016):
    """Stand-ins for the LFW fixtures in load_lfw's format: a procedural face pasted into a 250x250 frame, its box, a pose class and
    no landmark annotation (parts are zeros).  The tests run on these when the fixtures are not staged."""
    import cv2
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n):
        frame = cv2.GaussianBlur(rng.integers(0, 256, (250, 250, 3), dtype=np.uint8), (0, 0), 3)
        s = int(rng.integers(100, 161))
        x, y = (int(v) for v in rng.integers(0, 250 - s, 2))
        frame[y:y + s, x:x + s] = _procedural_face(rng, s)
        out.append(dict(name=f"procedural_{k:02d}", img=frame, box=(x, y, s, s), pose=int(rng.integers(-2, 3)), parts=np.zeros((10, 2), np.int32)))
    return out


def _bases(rng: np.random.Generator):
    faces = load_lfw()
    if faces:
        bases = []
        for f in faces:
            x, y, w, h = f["box"]
            bases.append(np.ascontiguousarray(f["img"][y:y + h, x:x + w]))
        return bases, "synthetic (jittered LFW fixtures, seeded)"
    return [_procedural_face(rng) for _ in range(20)], "synthetic (procedural blobs, seeded; LFW fixtures not staged)"


def make_crops(n: int, seed: int = 2012, size: int = 100):
    """C2 / C4: n crops size x size x 3 (box = whole crop).  Every 8th crop is pure uniform noise
    (MeanShift worst case)."""
    import cv2
    rng = np.random.default_rng(seed)
    bases, tag = _bases(rng)
    out = np.empty((n, size, size, 3), np.uint8)
    for i in range(n):
        if i % 8 == 7:
            out[i] = rng.integers(0, 256, (size, size, 3), dtype=np.uint8)
            continue
        b = bases[i % len(bases)]
        s = rng.uniform(0.9, 1.1) * size / b.shape[1]
        tx, ty = rng.integers(-6, 7, 2)
        M = np.array([[s, 0, (size - s * b.shape[1]) / 2 + tx], [0, s, (size - s * b.shape[0]) / 2 + ty]], np.float64)
        w = cv2.warpAffine(b, M, (size, size), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_REFLECT_101).astype(np.float32)
        w = w * rng.uniform(0.8, 1.2) + rng.uniform(-20, 20) + rng.normal(0, 4, w.shape).astype(np.float32)
        out[i] = np.clip(np.rint(w), 0, 255).astype(np.uint8)
    return out, tag


def _haar_like_box(rng, rows, cols, wmin, wmax, taken):
    """Boxes shaped like FaceForest::detectFace's enlarged output (src/FaceForest.cpp:152-154)."""
    for _ in range(200):
        w0 = int(rng.integers(wmin, wmax + 1))
        w = w0 + 2 * int(0.05 * w0)
        h = w0 + 2 * int(0.15 * w0)
        if w >= cols or h >= rows:
            continue
        x = int(rng.integers(0, cols - w)); y = int(rng.integers(0, rows - h))
        if all(x + w <= bx or bx + bw <= x or y + h <= by or by + bh <= y for bx, by, bw, bh in taken):
            return (x, y, w, h)
    return None


def make_frames(n_frames: int, rows: int = 1080, cols: int = 1920, faces_per_frame: int = 16, seed: int = 2013, wmin: int = 96, wmax: int = 320):
    """C3: frames with pasted faces and given boxes.  Returns frames [n,rows,cols,3], boxes [m,4], image_of_box [m]."""
    import cv2
    rng = np.random.default_rng(seed)
    bases, tag = _bases(rng)
    frames = np.empty((n_frames, rows, cols, 3), np.uint8)
    boxes, iob = [], []
    for f in range(n_frames):
        bg = rng.integers(0, 256, (rows // 8, cols // 8, 3), dtype=np.uint8)
        frames[f] = cv2.GaussianBlur(cv2.resize(bg, (cols, rows), interpolation=cv2.INTER_LINEAR), (0, 0), 3)
        taken = []
        for k in range(faces_per_frame):
            b = _haar_like_box(rng, rows, cols, wmin, wmax, taken)
            if b is None:
                continue
            taken.append(b)
            x, y, w, h = b
            face = cv2.resize(bases[(f * faces_per_frame + k) % len(bases)], (w, h), interpolation=cv2.INTER_LINEAR).astype(np.float32)
            face = face * rng.uniform(0.8, 1.2) + rng.uniform(-20, 20)
            frames[f, y:y + h, x:x + w] = np.clip(np.rint(face), 0, 255).astype(np.uint8)
            boxes.append(b); iob.append(f)
    return frames, np.array(boxes, np.int32), np.array(iob, np.int32), tag


def make_mixed(n_images: int = 64, seed: int = 2015):
    """C5: mixed-resolution images (up to 4K), 1-8 boxes each, widths 64..1500 with scaled H <= 521.
    Returns a list of (frame, boxes[k,4])."""
    rng = np.random.default_rng(seed)
    sizes = [(480, 640), (720, 1280), (1080, 1920), (1440, 2560), (2160, 3840)]
    out, tag = [], ""
    for i in range(n_images):
        rows, cols = sizes[i % len(sizes)]
        fr, boxes, _, tag = make_frames(1, rows, cols, int(rng.integers(1, 9)), seed=seed * 1000 + i, wmin=64, wmax=min(1500, rows * 2 // 3))
        out.append((fr[0], boxes))
    return out, tag
