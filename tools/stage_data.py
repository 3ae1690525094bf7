#!/usr/bin/env python
"""Stage what the tests and the benchmark use from the reference project's data/ (checkout named by CRF_REFERENCE) into
staged/ (git-ignored):

  staged/model.crfb200   packed binary image of data/trees_headpose + data/trees_ffd (crf_model_save_packed)
  staged/imgs/           the 20 LFW jpgs + index_random_subset.txt (fixtures for C1 and the synthetic generators)
  staged/trees_headpose, staged/trees_ffd   the 115 Boost text archives themselves (282 MB): what the REAL reference code
                         (oracle/_ref/libcrf_ref.so, bench.py's cpu_baseline kind "reference") loads on the GPU box

Nothing at run time reads the reference checkout itself.
"""
import shutil
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from oracle.ref import REF_DATA as REF  # noqa: E402


def main() -> int:
    if REF is None:
        raise SystemExit("set CRF_REFERENCE to a checkout of the reference project")
    import face_alignment_cvpr_2012_b200 as crf
    crf.build()
    out = ROOT / "staged"
    (out / "imgs").mkdir(parents=True, exist_ok=True)
    t = time.time()
    m = crf.Model(str(REF / "trees_headpose"), str(REF / "trees_ffd"), 15, 20)
    print(f"parsed 115 Boost text archives in {time.time() - t:.1f}s: {m.info}")
    m.save_packed(str(out / "model.crfb200"))
    t = time.time()
    m2 = crf.Model(packed=str(out / "model.crfb200"))
    assert m2.info == m.info
    print(f"packed image: {(out / 'model.crfb200').stat().st_size / 1e6:.1f} MB, reloads in {time.time() - t:.2f}s")
    for p in sorted((REF / "imgs").iterdir()):
        shutil.copy(p, out / "imgs" / p.name)
    shutil.copy(REF / "haarcascade_frontalface_alt.xml", out / "haarcascade_frontalface_alt.xml")
    for d in ("trees_headpose", "trees_ffd"):
        if not (out / d).exists():
            shutil.copytree(REF / d, out / d)
    print("staged", len(list((out / "imgs").iterdir())), "files under staged/imgs + the Haar cascade (host-side detectFace)")
    return 0


if __name__ == "__main__":
    sys.exit(main())
