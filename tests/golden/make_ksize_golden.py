"""Generates tests/golden/kat_ksize.npz: what the cv2 wheel (opencv-python-headless 4.13.0.92) returns for the Sobel apertures
other than 3 -- cv2.cornerMinEigenVal(img, blockSize, ksize=g), cv2.cornerHarris(img, blockSize, g, 0.04) and
cv2.goodFeaturesToTrack(..., gradientSize=g), min-eig and Harris, with and without the scene's mask -- for g = -1 (Scharr), 1,
5, 7 on the two golden scenes stored in kat_texture.npz / kat_iceberg.npz (their f0 frame and mask).  The maps cover a crop of
each scene (MAP_CROP in tests/ksize_cases.py) to keep the file small; the corner lists are of the whole scene.

Run:  python tests/golden/make_ksize_golden.py      (needs cv2; not needed to RUN the tests)
"""
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from ksize_cases import KSIZE_SETS, MAP_BLOCKS, MAP_CROP, OTHER_APERTURES  # noqa: E402


def main():
    out = {}
    for scene in ("texture", "iceberg"):
        g = np.load(os.path.join(HERE, "kat_%s.npz" % scene))
        f0, mask = g["f0"], g["mask"]
        crop = np.ascontiguousarray(f0[MAP_CROP])
        for ks in OTHER_APERTURES:
            for bs in MAP_BLOCKS:
                out["%s_mineig_g%d_bs%d" % (scene, ks, bs)] = cv2.cornerMinEigenVal(crop, bs, ksize=ks)
                out["%s_harris_g%d_bs%d" % (scene, ks, bs)] = cv2.cornerHarris(crop, bs, ks, 0.04)
            for si, gp in enumerate(KSIZE_SETS):
                for harris in (0, 1):
                    for mi, m in enumerate((None, mask)):
                        p = cv2.goodFeaturesToTrack(f0, mask=m, useHarrisDetector=bool(harris), k=0.04, gradientSize=ks, **gp)
                        out["%s_gftt%d_g%d_h%d_m%d" % (scene, si, ks, harris, mi)] = (
                            np.zeros((0, 1, 2), np.float32) if p is None else p)
    out["cv2_version"] = np.array(cv2.__version__)
    np.savez_compressed(os.path.join(HERE, "kat_ksize.npz"), **out)
    print("kat_ksize.npz:", len(out), "arrays")


if __name__ == "__main__":
    main()
