"""Generates tests/golden/kat_f32.npz: what the cv2 wheel (opencv-python-headless 4.13.0.92) returns on float32 images --
cv2.cornerMinEigenVal / cv2.cornerHarris maps (a crop of the texture scene under each non-integer transform of
tests/f32_cases.py, every aperture, blockSize 3 / 10 / 31; tiny random images, blockSize 2 and wider than the image) and
cv2.goodFeaturesToTrack lists (both golden scenes under each transform, every aperture, min-eig and Harris, with and without
the scene's mask).  The scenes are the f0 frame and mask of kat_texture.npz / kat_iceberg.npz.

Run:  python tests/golden/make_f32_golden.py      (needs cv2; not needed to RUN the tests)
"""
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import f32_cases as FC  # noqa: E402


def main():
    out = {}
    for ti, (tname, T) in enumerate(FC.TRANSFORMS.items()):
        for scene in ("texture", "iceberg"):
            g = np.load(os.path.join(HERE, "kat_%s.npz" % scene))
            f, mask = T(g["f0"]), g["mask"]
            crop = np.ascontiguousarray(f[FC.MAP_CROP])
            for ks in FC.APERTURES:
                if scene == "texture":
                    for bs in FC.MAP_BLOCKS:
                        out["map_%s_mineig_g%d_bs%d" % (tname, ks, bs)] = cv2.cornerMinEigenVal(crop, bs, ksize=ks)
                        out["map_%s_harris_g%d_bs%d" % (tname, ks, bs)] = cv2.cornerHarris(crop, bs, ks, 0.04)
                gp = FC.F32_SETS[FC.set_index(ti, ks)]
                for key, (harris, m) in zip(FC.golden_keys(scene, tname, ks), [(h, m) for h in (0, 1) for m in (None, mask)]):
                    p = cv2.goodFeaturesToTrack(f, mask=m, useHarrisDetector=bool(harris), k=0.04, gradientSize=ks, **gp)
                    out["gftt_" + key] = np.zeros((0, 1, 2), np.float32) if p is None else p
    for i, (h, w) in enumerate(FC.TINY_SIZES):
        img = FC.tiny_image(h, w, 100 + i)
        out["tiny_img_%dx%d" % (h, w)] = img
        for ks in FC.APERTURES:
            for bs in (2, min(h, w) + 1):
                out["tiny_mineig_%dx%d_g%d_bs%d" % (h, w, ks, bs)] = cv2.cornerMinEigenVal(img, bs, ksize=ks)
                out["tiny_harris_%dx%d_g%d_bs%d" % (h, w, ks, bs)] = cv2.cornerHarris(img, bs, ks, 0.04)
    out["cv2_version"] = np.array(cv2.__version__)
    np.savez_compressed(os.path.join(HERE, "kat_f32.npz"), **out)
    print("kat_f32.npz:", len(out), "arrays")


if __name__ == "__main__":
    main()
