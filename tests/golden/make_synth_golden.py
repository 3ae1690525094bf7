#!/usr/bin/env python
"""Golden vectors for the tests that use the shipped forests and LFW fixtures, for checkouts where neither is staged:
the same sets run on the seeded synthetic forests (tests/conftest.py synth_dirs, seed 5) and, in place of the LFW
images, on workloads.procedural_lfw().

    python tests/golden/make_synth_golden.py   ->  tests/golden/synth_campaign.npz  (layout of ref_campaign.npz)
                                                   tests/golden/synth_lfw.npz       (layout of lfw_e2e.npz, without ground truth)

synth_campaign.npz comes from the reference's own code (oracle/ref.py: oracle/_ref/libcrf_ref.so, built from a checkout of
the reference project named by CRF_REFERENCE) whenever that library is available, and from the CPU oracle otherwise; its
`source` entry says which.  synth_lfw.npz holds whole oracle records and leaf-id checksums, as lfw_e2e.npz does.
"""
import importlib.util
import sys
import tempfile
import zlib
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parents[1]
sys.path.insert(0, str(ROOT))
from face_alignment_cvpr_2012_b200 import synthetic_model as sm, workloads as wl  # noqa: E402
from oracle import oracle as O, ref as R  # noqa: E402

SYNTH_SEED = 5   # tests/conftest.py synth_dirs


def main():
    O.build()
    hp_dir, ffd_dir = sm.write_model(tempfile.mkdtemp(prefix="crf_synth_golden_"), seed=SYNTH_SEED)
    om = O.Model(hp_dir, ffd_dir, 15, 20)
    threads = O.hardware_concurrency()
    spec = importlib.util.spec_from_file_location("make_ref_golden", HERE / "make_ref_golden.py")
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    faces = wl.procedural_lfw()

    if R.available():
        analyze, source = m.reference_analyze(R.FaceForest(hp_dir, ffd_dir)), "reference code (oracle/_ref/libcrf_ref.so)"
    else:
        def analyze(img, box, hs, fs):
            r = om.analyze_face(img, box, hs, fs, threads=threads)
            _, _, fi, ti, _ = om.compose(r["headpose"], r["variance"])
            return r["headpose"], r["ffd"], fi, ti
        source = "CPU oracle (oracle/oracle.py); no reference library was available"
    out = m.campaign_results(analyze, m.campaign_sets(faces), source)
    np.savez_compressed(HERE / "synth_campaign.npz", source=np.array(source), **out)

    recs, hp_crc, ffd_crc = [], [], []
    for f in faces:
        recs.append(om.analyze_face(f["img"], f["box"], threads=threads))
        x, y, w, h = f["box"]
        sw, sh, _ = O.scaled_size(w, h)
        s = O.Sample(O.resize(O.bgr2gray(f["img"])[y:y + h, x:x + w], sh, sw))
        ids, hp, var, _ = om.eval_hp(s, 4)
        hp_crc.append(zlib.crc32(ids.tobytes()))
        _, _, fi, ti, _ = om.compose(hp, var)
        ffd_crc.append(zlib.crc32(om.eval_ffd(s, fi, ti, 3)["leaf_ids"].tobytes()))
        s.close()
    np.savez_compressed(HERE / "synth_lfw.npz", names=np.array([f["name"] for f in faces]), boxes=np.array([f["box"] for f in faces], np.int32),
                        recs=np.array(recs), hp_crc=np.array(hp_crc, np.uint32), ffd_crc=np.array(ffd_crc, np.uint32))


if __name__ == "__main__":
    main()
