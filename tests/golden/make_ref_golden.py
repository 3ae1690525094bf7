#!/usr/bin/env python
"""Golden vectors from the REAL reference (oracle/_ref/libcrf_ref.so: the reference's own sources, unmodified, see
oracle/ref_driver.cc), for machines without a checkout of the reference project.  Run with one:

    CRF_REFERENCE=<checkout> python tests/golden/make_ref_golden.py        ->  tests/golden/ref_campaign.npz

Every set is regenerated on the GPU box from its seed by face_alignment_cvpr_2012_b200/workloads.py (same image, same
cv2), so only the reference's RESULTS are stored: FaceForest::analyzeFace's head pose (f32 bits), the final landmarks
(Face::ffd_cordinates after both roundings) and the composed forest (which trees of which pose forest ran).

  s1      48 crops 100x100, strides 1/1   (BASELINE config 2 shape; every 8th crop pure noise)
  dflt    256 crops 100x100, strides 4/3  (reference defaults)
  c3      4 frames 1080p x 16 ragged Haar-like boxes, strides 4/3 (config 3 shape)
  c5      5 mixed-resolution images up to 4K, 1-8 boxes each + one 1400-px box, strides 4/3 (config 5 shape)
  lfw     the 20 shipped LFW faces, strides 4/3 (config 1)
"""
import sys
import time
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parents[1]
sys.path.insert(0, str(ROOT))
from face_alignment_cvpr_2012_b200 import workloads as wl  # noqa: E402
from oracle import ref as R  # noqa: E402

REF = R.REF_DATA
BIG_BOX = (100, 50, 1400, 1800)   # > 1000 px wide, inside the 4K frame of the c5 set


def campaign_sets(faces=None):
    """name -> (list of (image, box), hp_stride, ffd_stride); shared with tests/test_gpu_reference_campaign.py and
    make_synth_golden.py.  faces: the "lfw" set in load_lfw's format (default: the staged LFW fixtures)."""
    sets = {}
    crops, _ = wl.make_crops(48, seed=4801)
    sets["s1"] = ([(c, (0, 0, 100, 100)) for c in crops], 1, 1)
    crops, _ = wl.make_crops(256, seed=4802)
    sets["dflt"] = ([(c, (0, 0, 100, 100)) for c in crops], 4, 3)
    frames, boxes, iob, _ = wl.make_frames(4, seed=4803)
    sets["c3"] = ([(frames[i], tuple(int(v) for v in b)) for b, i in zip(boxes, iob)], 4, 3)
    mixed, _ = wl.make_mixed(5, seed=4805)
    items = [(fr, tuple(int(v) for v in b)) for fr, bs in mixed for b in bs]
    items.append((mixed[4][0], BIG_BOX))
    sets["c5"] = (items, 4, 3)
    sets["lfw"] = ([(f["img"], f["box"]) for f in (wl.load_lfw() if faces is None else faces)], 4, 3)
    return sets


def campaign_results(analyze, sets, who):
    """The arrays of ref_campaign.npz: analyze(image, box, hp_stride, ffd_stride) -> (headpose, ffd, list_forest, list_tree) on every set."""
    out = {}
    for name, (items, hs, fs) in sets.items():
        t0 = time.time()
        hp = np.zeros(len(items), np.float32); ffd = np.zeros((len(items), 10, 2), np.int32)
        lf = np.full((len(items), 32), -1, np.int32); lt = np.full((len(items), 32), -1, np.int32)
        for i, (img, box) in enumerate(items):
            hp[i], ffd[i], fi, ti = analyze(img, box, hs, fs)
            n = len(fi)
            assert n <= 32
            lf[i, :n] = fi; lt[i, :n] = ti
        out[f"{name}_headpose"] = hp; out[f"{name}_ffd"] = ffd; out[f"{name}_list_forest"] = lf; out[f"{name}_list_tree"] = lt
        print(f"{name}: {len(items)} faces in {time.time() - t0:.1f} s ({who}, strides {hs}/{fs})")
    return out


def reference_analyze(ff):
    """FaceForest::analyzeFace of the reference library (ff: oracle.ref.FaceForest) in campaign_results' form."""
    def analyze(img, box, hs, fs):
        ff.set_strides(hs, fs)
        r = ff.analyze_face(img, box)
        return r["headpose"], r["ffd"], r["list_forest"], r["list_tree"]
    return analyze


def main():
    ff = R.FaceForest(str(REF / "trees_headpose"), str(REF / "trees_ffd"))
    np.savez_compressed(HERE / "ref_campaign.npz", **campaign_results(reference_analyze(ff), campaign_sets(), "reference code"))


if __name__ == "__main__":
    main()
