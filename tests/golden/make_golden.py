#!/usr/bin/env python
"""Generates the committed golden fixtures (needs cv2 4.13 and CRF_REFERENCE naming a checkout of the reference project).

  cv2_stages.npz   inputs + cv2 4.13 outputs of the OpenCV-defined stages of the path (SURVEY Appendix A):
                   cvtColor(BGR2GRAY), resize(INTER_LINEAR), integral, Sobel(8U), erode/dilate 3x3, equalizeHist, Canny(-1, 5),
                   filter2D with the 7x7 Gabor kernels (bit-exact by construction of the canonical arithmetic),
                   and the whole Gabor plane (magnitude -> normalize -> x255 -> u8) of cv2 for all 35 kernels
                   (+-1 LSB statistical pin for kernels >= 9x9, where cv2 takes its DFT path).
  lfw_e2e.npz      oracle results on the 20 shipped LFW faces (data/imgs/index_random_subset.txt) with the shipped
                   forests at the reference's default strides, plus ground-truth landmarks: the end-to-end pin
                   (mean normalised error must stay ~0.075) and the cross-box regression vector for the GPU path.
"""
import sys
import zlib
from pathlib import Path

import cv2
import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parents[1]
sys.path.insert(0, str(ROOT))
from oracle import oracle as O  # noqa: E402
from oracle.ref import REF_DATA as REF  # noqa: E402  (CRF_REFERENCE: a checkout of the reference project)


def gabor_planes_cv2(gray):
    out = []
    for re, im in O.gabor_bank():
        r = cv2.filter2D(gray, cv2.CV_32F, re); i = cv2.filter2D(gray, cv2.CV_32F, im)
        r = cv2.pow(r, 2); i = cv2.pow(i, 2)
        m = cv2.pow(cv2.add(i, r), 0.5)
        m = cv2.normalize(m, None, 0, 1, cv2.NORM_MINMAX)
        out.append(cv2.convertScaleAbs(m, alpha=255))  # == convertTo(CV_8UC1, 255) for m >= 0
    return np.stack(out)


def main():
    rng = np.random.default_rng(20121)
    d = {}
    bgr = rng.integers(0, 256, (97, 143, 3), dtype=np.uint8)
    d["bgr"] = bgr
    d["gray"] = cv2.cvtColor(bgr, cv2.COLOR_BGR2GRAY)
    sizes = [(130, 130, 125, 125), (100, 100, 125, 125), (250, 250, 125, 125), (118, 139, 147, 125), (211, 180, 146, 124), (61, 53, 143, 125), (400, 300, 166, 125)]
    for k, (sh, sw, dh, dw) in enumerate(sizes):
        src = rng.integers(0, 256, (sh, sw), dtype=np.uint8)
        d[f"resize_src_{k}"] = src
        d[f"resize_dst_{k}"] = cv2.resize(src, (dw, dh), interpolation=cv2.INTER_LINEAR)
    img = cv2.GaussianBlur(rng.integers(0, 256, (141, 125), dtype=np.uint8), (0, 0), 1.5)
    d["plane"] = img
    d["integral"] = cv2.integral(img, sdepth=cv2.CV_32F)
    d["sobel_dy"] = cv2.Sobel(img, cv2.CV_8U, 0, 1)
    d["sobel_dx"] = cv2.Sobel(img, cv2.CV_8U, 1, 0)
    k3 = np.ones((3, 3), np.uint8)
    d["erode"] = cv2.erode(img, k3); d["dilate"] = cv2.dilate(img, k3)
    d["equalize"] = cv2.equalizeHist(img)
    lowc = (img // 4 + 90).astype(np.uint8)
    d["equalize_src2"] = lowc; d["equalize2"] = cv2.equalizeHist(lowc)
    # FC_CANNY (include/FeatureChannelFactory.hpp:169): cv::Canny(img, out, -1, 5) on a blurred and on a raw noise plane
    d["canny"] = cv2.Canny(img, -1, 5)
    raw = np.random.default_rng(4).integers(0, 256, (64, 124), dtype=np.uint8)
    d["canny_src2"] = raw; d["canny2"] = cv2.Canny(raw, -1, 5)
    bank = O.gabor_bank()
    for idx in range(7):
        d[f"f2d_re_{idx}"] = cv2.filter2D(img, cv2.CV_32F, bank[idx][0]); d[f"f2d_im_{idx}"] = cv2.filter2D(img, cv2.CV_32F, bank[idx][1])
    d["gabor_u8_cv2"] = gabor_planes_cv2(img)
    np.savez_compressed(HERE / "cv2_stages.npz", **d)

    om = O.Model(str(REF / "trees_headpose"), str(REF / "trees_ffd"))
    names, boxes, poses, gts, recs, hp_crc, ffd_crc = [], [], [], [], [], [], []
    for line in (REF / "imgs" / "index_random_subset.txt").read_text().split("\n"):
        t = line.split()
        if len(t) < 27:
            continue
        im = cv2.imread(str(REF / "imgs" / t[0]))
        box = tuple(int(v) for v in t[1:5])
        rec = om.analyze_face(im, box)
        names.append(t[0]); boxes.append(box); poses.append(int(t[5])); gts.append(np.array(t[7:27], np.int32).reshape(10, 2)); recs.append(rec)
        # leaf-id checksums of both forests on this face
        x, y, w, h = box
        sw, sh, _ = O.scaled_size(w, h)
        sc = O.resize(O.bgr2gray(im)[y:y + h, x:x + w], sh, sw)
        s = O.Sample(sc)
        ids, hp, var, _ = om.eval_hp(s, 4)
        hp_crc.append(zlib.crc32(ids.tobytes()))
        _, _, fi, ti, _ = om.compose(hp, var)
        ffd_crc.append(zlib.crc32(om.eval_ffd(s, fi, ti, 3)["leaf_ids"].tobytes()))
        s.close()
    np.savez_compressed(HERE / "lfw_e2e.npz", names=np.array(names), boxes=np.array(boxes, np.int32), poses=np.array(poses, np.int32),
                        gt=np.stack(gts), recs=np.array(recs), hp_crc=np.array(hp_crc, np.uint32), ffd_crc=np.array(ffd_crc, np.uint32))
    gt = np.stack(gts).astype(np.float64); pr = np.stack([r["ffd"] for r in recs]).astype(np.float64)
    iod = np.linalg.norm((gt[:, 0] + gt[:, 1]) / 2 - (gt[:, 6] + gt[:, 7]) / 2, axis=1)
    print("mean normalised error on the 20 LFW faces:", float((np.linalg.norm(gt - pr, axis=2) / iod[:, None]).mean()))


if __name__ == "__main__":
    main()
