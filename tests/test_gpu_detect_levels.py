"""The detector's device passes against the CPU reference, level by level (crf_stage_haar_levels, Context.stage_haar_levels).

- Integrals: S, Q and the tilted T of every (frame, level) instance equal tests/haar_cascade_oracle.py's level reference bit for bit, and
  the pixels recovered from S equal the reference level image.  The frames reach what the small frames of the other detector tests do
  not: 1080p and 4K levels whose square sums wrap modulo 2^32, 4000-pixel strips whose diagonals span more than 1024 rows and columns,
  sizes at the edges of the row, column and diagonal tiles, frames of exactly the window's size, and up to 64 frames in one group.
- Window flags: the flag byte of every window equals the one the oracle's stage sums give, with whole cascades on small frames and
  their first stages at 1080p and 4K, including the windows the variance test skips; raw candidates at those sizes equal the oracle's.
- Stage groups: CRF_HAAR_SPLIT changes the launches per group and nothing else."""
from pathlib import Path

import numpy as np
import pytest

import haar_cascade_oracle as G
from test_gpu_detect_batch import _textured, detect_one, write_stump_cascade
from test_gpu_detect_mixed import detect_mixed

cv2 = pytest.importorskip("cv2")
CV2_DIR = Path(cv2.data.haarcascades)
FACE = CV2_DIR / "haarcascade_frontalface_alt.xml"
ALT2 = CV2_DIR / "haarcascade_frontalface_alt2.xml"
EYE = CV2_DIR / "haarcascade_eye_tree_eyeglasses.xml"


@pytest.fixture(scope="module")
def gpu_ctx(crf):
    if crf.lib().crf_device_count() < 1:
        pytest.fail("no CUDA device: the gpu-marked tests must run on the B200 box (there is no CPU fallback)")
    return crf.Context(None, 0)


@pytest.fixture(scope="module")
def cascades(tmp_path_factory):
    """{name: path}: the face cascade (stumps), alt2 (trees), eye_tree_eyeglasses (trees + tilted features), a synthetic stump cascade,
    and copies of the first three truncated to their first stages."""
    d = tmp_path_factory.mktemp("level_cascades")
    out = {"face": str(FACE), "alt2": str(ALT2), "eye": str(EYE), "stumps": write_stump_cascade(d / "stumps.xml")}
    for name, n in (("face", 3), ("face", 1), ("alt2", 2), ("alt2", 1), ("eye", 2), ("eye", 1)):
        out[f"{name}{n}"] = G.truncate_cascade(out[name], d / f"{name}{n}.xml", n)
    return out


def _gray3(gray):
    return np.repeat(np.ascontiguousarray(gray, np.uint8)[..., None], 3, 2)


def _checker(rows, cols):
    return _gray3((np.indices((rows, cols)).sum(0) % 2) * 255)


def _contrast(rows=240, cols=320, seed=5):
    """A flat band (every window there has nf = 0), a low-contrast band (nf > 0 but area / sqrt(nf) >= 0.1) and a textured band."""
    rng = np.random.default_rng(seed)
    g = np.full((rows, cols), 100, np.uint8)
    b = cols // 3
    g[:, b:2 * b] = 128 + rng.integers(-3, 4, (rows, b))
    out = _gray3(g)
    out[:, 2 * b:] = _textured(1, rows, cols - 2 * b, seed)[0]
    return out


@pytest.fixture(scope="module")
def frames():
    """name -> BGR frame.  The edge sizes are level 0 of a 20 x 20 window: sw + 1 = 320 / 321 / 319 (0, 1, 31 mod 32); sh = 96 / 97 / 103
    (0, 1, 7 mod 8); sw + sh = 256 / 257 (0, 1 mod 32); the window itself, one pixel more and one less (no level), and 1 x 1."""
    from face_alignment_cvpr_2012_b200 import workloads as wl
    out = {}
    for tag, (rows, cols) in (("1080", (1080, 1920)), ("4k", (2160, 3840))):
        out["tex" + tag] = _textured(1, rows, cols, 11 + len(tag))[0]
        out["white" + tag] = np.full((rows, cols, 3), 255, np.uint8)
        out["black" + tag] = np.zeros((rows, cols, 3), np.uint8)
        out["check" + tag] = _checker(rows, cols)
    out["video1080"] = wl.make_frames(1, 1080, 1920, 12, seed=22)[0][0]
    out["wide"] = _textured(1, 48, 4000, 21)[0]
    out["tall"] = _textured(1, 4000, 48, 22)[0]
    for k, (rows, cols) in enumerate([(101, 319), (101, 320), (101, 318), (96, 150), (97, 150), (103, 150), (100, 156), (100, 157),
                                      (20, 20), (21, 21), (19, 19), (1, 1)]):
        out[f"{rows}x{cols}"] = _textured(1, rows, cols, 30 + k)[0]
    out["face250"] = wl.procedural_lfw()[0]["img"]
    out["contrast"] = _contrast()
    out["tex240"] = _textured(1, 240, 320, 5)[0]
    return out


BIG = ["tex1080", "white1080", "black1080", "check1080", "tex4k", "white4k", "black4k", "check4k"]
EDGE = ["101x319", "101x320", "101x318", "96x150", "97x150", "103x150", "100x156", "100x157", "20x20", "21x21", "19x19", "1x1"]
PLAN_KEYS = ("frame", "factor", "sw", "sh", "ystep", "nx", "ny", "win_w", "win_h")


def _gray(frame):
    from oracle import oracle as O
    return O.bgr2gray(np.ascontiguousarray(frame))


def _check_integrals(results, fr, sf, what):
    """results: stage_haar_levels of the frames fr, one list per cascade (the same plan: every cascade here has a 20 x 20 window); compares
    every instance with the level reference.  Returns the number of levels whose square sum passes 2^32."""
    k = wrapped = 0
    for i, f in enumerate(fr):
        gray = _gray(f)
        for L in G.level_plan(20, 20, *gray.shape, sf):
            img = G.level_image(gray, L)
            S, Q, T = G.level_integrals(img, any(got[k]["T"] is not None for got in results))
            wrapped += int((img.astype(np.uint64) ** 2).sum()) >= 2 ** 32
            where = (what, i, L["factor"], L["sw"], L["sh"])
            for got in results:
                g = got[k]
                assert tuple(g[n] for n in PLAN_KEYS) == (i,) + tuple(L[n] for n in PLAN_KEYS[1:]), where
                assert np.array_equal(g["S"], S), where
                assert np.array_equal(g["Q"], Q), where
                s = g["S"]
                assert np.array_equal(s[1:, 1:] - s[:-1, 1:] - s[1:, :-1] + s[:-1, :-1], img), where   # u32 arithmetic, modulo 2^32
                if g["T"] is not None:
                    assert np.array_equal(g["T"], T), where
            k += 1
    assert all(k == len(got) for got in results), what
    return wrapped


def _integrals(gpu_ctx, face, eye, fr, sf):
    """stage_haar_levels of an upright cascade (T None) and of the tilted one (T given) on the frames fr"""
    a, b = gpu_ctx.stage_haar_levels(face, fr, sf), gpu_ctx.stage_haar_levels(eye, fr, sf)
    assert all(g["T"] is None for g in a) and all(g["T"] is not None for g in b)
    return [a, b]


# ---- integrals, every level -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("sf", [1.05, 1.1, 1.3, 2.5])
def test_integrals_every_level(crf, gpu_ctx, cascades, frames, sf):
    """Frame by frame, with an upright cascade (S, Q) and the tilted one (S, Q, T).  1.05 and 1.1 leave out the 4K frames (90 and 50
    levels each, for kernels that 1.3 and 2.5 exercise on the same frames)."""
    names = (BIG if sf >= 1.3 else BIG[:4]) + ["video1080", "wide", "tall"] + EDGE
    face, eye = crf.CascadeClassifier(cascades["face"]), crf.CascadeClassifier(cascades["eye"])
    wrapped = 0
    for name in names:
        f = frames[name]
        res = _integrals(gpu_ctx, face, eye, [f], sf)
        assert (len(res[0]) == 0) == (name in ("19x19", "1x1")), name
        wrapped += _check_integrals(res, [f], sf, name)
    assert wrapped >= 4


@pytest.mark.gpu
def test_integrals_one_group(crf, gpu_ctx, cascades, frames):
    """64 frames of different sizes in one call and one group (the launches of a one-frame call): every instance's integrals, so the
    blocks of each pass find their instance among several hundred."""
    rng = np.random.default_rng(17)
    fr = [frames[n] for n in BIG + ["video1080", "wide", "tall"] + EDGE]
    while len(fr) < 64:
        fr.append(_textured(1, int(rng.integers(20, 400)), int(rng.integers(20, 600)), 100 + len(fr))[0])
    face, eye = crf.CascadeClassifier(cascades["face"]), crf.CascadeClassifier(cascades["eye"])
    for cas in (face, eye):
        gpu_ctx.reset_counters()
        gpu_ctx.stage_haar_levels(cas, fr[-1:], 1.3, integrals=False)
        one = gpu_ctx.counters()["kernel_launches"]
        gpu_ctx.reset_counters()
        gpu_ctx.stage_haar_levels(cas, fr, 1.3, integrals=False)
        assert gpu_ctx.counters()["kernel_launches"] == one > 0
    res = _integrals(gpu_ctx, face, eye, fr, 1.3)
    assert len(res[0]) > 300
    assert _check_integrals(res, fr, 1.3, "group") > 0


# ---- window flags and raw candidates --------------------------------------------------------------------------------------------------
FLAG_CASES = [
    # whole cascades on small frames
    ("face", ["face250", "contrast"], 1.3), ("alt2", ["face250", "contrast"], 1.3), ("eye", ["face250", "contrast"], 1.1),
    ("stumps", ["tex240", "contrast", "101x319"], 1.1),
    # their first stages at full size
    ("face3", ["video1080", "tex1080", "white1080", "black1080"], 1.3), ("face1", ["tex4k", "check4k"], 1.3),
    ("alt2", ["white4k"], 1.3), ("alt21", ["check1080"], 2.5), ("alt21", ["video1080", "tall", "wide"], 1.1),
    ("eye2", ["tex1080"], 1.3), ("eye1", ["tex4k"], 1.3), ("eye2", ["tall", "wide"], 1.05),
    ("stumps", ["tex1080"], 1.3),
]


def _skipped_windows(gray, L, c):
    """(nf <= 0, nf > 0 and area / sqrt(nf) >= 0.1) over the level's windows: the two cases the variance test decides alone."""
    img = G.level_image(gray, L).astype(np.int64)
    S = np.zeros((img.shape[0] + 1, img.shape[1] + 1), np.int64)
    Q = S.copy()
    S[1:, 1:], Q[1:, 1:] = img.cumsum(0).cumsum(1), (img * img).cumsum(0).cumsum(1)
    ys, xs = np.arange(L["ny"]) * L["ystep"], np.arange(L["nx"]) * L["ystep"]
    yy, xx = np.meshgrid(ys, xs, indexing="ij")
    w, h = c.w - 2, c.h - 2

    def rs(A):
        return A[yy + 1 + h, xx + 1 + w] - A[yy + 1, xx + 1 + w] - A[yy + 1 + h, xx + 1] + A[yy + 1, xx + 1]

    area = float(w * h)
    nf = area * (rs(Q) & 0xffffffff).astype(np.float64) - rs(S).astype(np.float64) ** 2
    inv = (1.0 / np.sqrt(np.where(nf > 0, nf, 1.0))).astype(np.float32)
    return nf <= 0, (nf > 0) & (np.float32(area) * inv >= np.float32(0.1))


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(FLAG_CASES)), ids=[f"{c}-{'+'.join(f)}-{sf}" for c, f, sf in FLAG_CASES])
def test_window_flags_and_candidates(crf, gpu_ctx, cascades, frames, case):
    """Every window's flag byte equals the oracle's, and crf_detect_faces with min_neighbors 0 returns the oracle's raw candidates."""
    name, names, sf = FLAG_CASES[case]
    c = G.Cascade(cascades[name])
    cas = crf.CascadeClassifier(cascades[name])
    for fname in names:
        f = frames[fname]
        gray = _gray(f)
        got = gpu_ctx.stage_haar_levels(cas, [f], sf, integrals=False)
        levels = list(G.detect_levels(c, gray, sf, 0))
        assert len(got) == len(levels) > 0, fname
        flat = weak = 0
        for g, (L, flags, ys, xs) in zip(got, levels):
            where = (name, fname, L["factor"])
            assert tuple(g[n] for n in PLAN_KEYS[1:]) == tuple(L[n] for n in PLAN_KEYS[1:]), where
            assert np.array_equal(g["flags"], flags), (where, int((g["flags"] != flags).sum()))
            if fname in ("contrast", "white1080", "black1080", "white4k"):
                nf0, small = _skipped_windows(gray, L, c)
                assert (flags[nf0 | small] == 0).all(), where
                flat += int(nf0.sum()); weak += int(small.sum())
        if fname == "contrast":
            assert flat > 0 and weak > 0
        if fname.startswith(("white", "black")):
            assert flat > 0 and all((g["flags"] == 0).all() for g in got)
        assert detect_one(crf, gpu_ctx, cas, f, sf=sf, mn=0, ms=0) == G.level_candidates(levels), (name, fname)


# ---- stage groups ---------------------------------------------------------------------------------------------------------------------
def _groups(split, nstages):
    """Stage groups the engine runs for a CRF_HAAR_SPLIT list: bounds that are not above the previous one or not below the stage count are
    dropped."""
    bounds = []
    for b in split:
        if b > (bounds[-1] if bounds else 0) and b < nstages:
            bounds.append(b)
    return len(bounds) + 1


@pytest.mark.gpu
def test_split_does_not_change_results(crf, cascades, frames, monkeypatch):
    """For each CRF_HAAR_SPLIT value (read when a context is created): raw candidates, grouped boxes and window flags of a mixed batch
    with a 1080p frame equal the default split's, and a group costs 3 + (stage groups - 1) + 3 launches, plus 1 with tilted features."""
    import ctypes as C
    fr = [frames["video1080"], frames["face250"], frames["tex240"], frames["contrast"], frames["21x21"], frames["19x19"]]
    names = ["face", "alt2", "eye", "stumps"]
    cas = {n: crf.CascadeClassifier(cascades[n]) for n in names}
    nst = {}
    for n in names:
        v = C.c_int()
        assert crf.lib().crf_cascade_info(cas[n].h, None, None, C.byref(v), None) == 0
        nst[n] = v.value

    def run(ctx, n):
        ctx.reset_counters()
        detect_mixed(crf, ctx, cas[n], fr, mn=1, ms=0, cap=0)
        launches = ctx.counters()["kernel_launches"]
        flags = [g["flags"] for g in ctx.stage_haar_levels(cas[n], fr, 1.3, integrals=False)]
        return launches, detect_mixed(crf, ctx, cas[n], fr, mn=0, ms=0), detect_mixed(crf, ctx, cas[n], fr, mn=1, ms=0), flags

    monkeypatch.delenv("CRF_HAAR_SPLIT", raising=False)
    ctx = crf.Context(None, 0)
    want = {n: run(ctx, n) for n in names}
    ctx.close()
    for n in names:
        assert want[n][0] == 3 + (_groups([3, 8], nst[n]) - 1) + 3 + (n == "eye"), n
        assert want[n][1][0] > 0, n
    for n in names:
        for value in ["0", "1", ",".join(str(k) for k in range(1, nst[n])), "3,8", "8,3", "20", "100", "-1"]:
            monkeypatch.setenv("CRF_HAAR_SPLIT", value)
            ctx = crf.Context(None, 0)
            launches, raw, grouped, flags = run(ctx, n)
            ctx.close()
            split = [int(v) for v in value.split(",")]
            assert launches == 3 + (_groups(split, nst[n]) - 1) + 3 + (n == "eye"), (n, value)
            assert raw == want[n][1] and grouped == want[n][2], (n, value)
            assert len(flags) == len(want[n][3]) and all(np.array_equal(a, b) for a, b in zip(flags, want[n][3])), (n, value)
