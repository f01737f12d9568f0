#!/usr/bin/env python
"""cv2's answers for the pins of tests/test_oracle_pins.py that compare the oracle with OpenCV itself on fresh inputs: the
reference's ORB + BFMatcher call sequence on a seed of its own, the OpenCV primitives src/surf.cpp delegates to, cornerSubPix /
getRectSubPix, ORB Harris scores, INTER_LINEAR_EXACT resizing and BFMatcher on 64-byte rows (cv2 4.13).  The inputs come from
the test module's own builders, so the stored answers belong to exactly the inputs the tests construct.
Run: python tests/golden/make_golden_cv2_pins.py"""
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(os.path.dirname(HERE)), os.path.dirname(HERE)]
import test_oracle_pins as t  # noqa: E402
from conftest import golden  # noqa: E402
from oracle import match  # noqa: E402


def knn_rows(d, p, rows):
    """knnMatch(k=2) rows as per-row counts + (n, 2) train indices / distances (-1 / inf past the count)."""
    d[p + "_knn_cnt"] = np.array([len(r) for r in rows], np.int32)
    idx, dist = np.full((len(rows), 2), -1, np.int32), np.full((len(rows), 2), np.inf, np.float32)
    for i, r in enumerate(rows):
        for j, m in enumerate(r):
            idx[i, j], dist[i, j] = m.trainIdx, m.distance
    d[p + "_knn_idx"], d[p + "_knn_dist"] = idx, dist


def cross_check(d, p, mc):
    d[p + "_cc_q"] = np.array([m.queryIdx for m in mc], np.int32)
    d[p + "_cc_t"] = np.array([m.trainIdx for m in mc], np.int32)
    d[p + "_cc_d"] = np.array([m.distance for m in mc], np.float32)


def main():
    d = {}
    o = cv2.ORB_create(nfeatures=800, scaleFactor=1.2, nlevels=1, edgeThreshold=31, firstLevel=0, WTA_K=2,
                       scoreType=cv2.ORB_FAST_SCORE, patchSize=31, fastThreshold=15)
    for eye, img in zip("lr", t.fresh_seed_pair()):
        kps, desc = o.detectAndCompute(img, None)
        x = np.array([k.pt[0] for k in kps], np.float32)
        y = np.array([k.pt[1] for k in kps], np.float32)
        order = np.lexsort((x, y))
        p = "fresh_%s_" % eye
        d[p + "x"], d[p + "y"], d[p + "desc"] = x[order], y[order], desc[order]
        d[p + "angle"] = np.array([k.angle for k in kps], np.float32)[order]
    ld, rd = d["fresh_l_desc"], d["fresh_r_desc"]
    mask = match.epipolar_mask(d["fresh_l_y"], d["fresh_r_y"], 2.0).astype(np.uint8)
    knn_rows(d, "fresh", cv2.BFMatcher(cv2.NORM_HAMMING, False).knnMatch(ld, rd, 2, mask))
    cross_check(d, "fresh", cv2.BFMatcher(cv2.NORM_HAMMING, True).match(ld, rd))

    img, windows, y, x = t.surf_primitive_inputs()
    d["surf_integral"] = cv2.integral(img, sdepth=cv2.CV_32S)
    d["surf_gauss13"] = cv2.getGaussianKernel(13, 2.5, cv2.CV_32F).ravel()
    d["surf_resize21"] = np.stack([cv2.resize(w, (21, 21), interpolation=cv2.INTER_AREA) for w in windows])
    d["surf_atan2"] = np.array([cv2.fastAtan2(float(a), float(b)) for a, b in zip(y, x)], np.float32)

    small, pts, centres = t.subpix_inputs(golden("grid_subpix_480x360")["img_f0_l"])
    d["subpix_small_out"] = cv2.cornerSubPix(small, pts.copy().reshape(-1, 1, 2), (5, 5), (-1, -1),
                                             (cv2.TERM_CRITERIA_EPS | cv2.TERM_CRITERIA_COUNT, 40, 0.001)).reshape(-1, 2)
    d["subpix_rect"] = np.stack([cv2.getRectSubPix(small, (13, 13), c, patchType=cv2.CV_32F) for c in centres])

    kps = cv2.ORB_create(nfeatures=150, nlevels=1, scoreType=cv2.ORB_HARRIS_SCORE, fastThreshold=12).detect(t.harris_fresh_image(), None)
    d["harris_x"] = np.array([int(k.pt[0]) for k in kps], np.int32)
    d["harris_y"] = np.array([int(k.pt[1]) for k in kps], np.int32)
    d["harris_response"] = np.array([k.response for k in kps], np.float32)

    for i, (img, dw, dh) in enumerate(t.resize_inputs()):
        d["resize_linear_exact_%d" % i] = cv2.resize(img, (dw, dh), interpolation=cv2.INTER_LINEAR_EXACT)

    ql, tr, masks = t.wide_row_inputs()
    for i, m in enumerate(masks):
        knn_rows(d, "wide%d" % i, cv2.BFMatcher(cv2.NORM_HAMMING, False).knnMatch(ql, tr, 2, None if m is None else m.astype(np.uint8)))
    cross_check(d, "wide", cv2.BFMatcher(cv2.NORM_HAMMING, True).match(ql, tr))

    np.savez_compressed(os.path.join(HERE, "cv2_pins.npz"), **d)
    print({k: v.shape for k, v in d.items()})


if __name__ == "__main__":
    main()
