"""Generates tests/golden/opencv/pad.npz: OpenCV's own texture post-process (the calls of the
reference's src/pointsTransfer.cpp:593-611) on seeded sparse BGRA images, so that
tests/test_texture.py checks the oracle's restatement against it without OpenCV installed.
Needs the cv2 wheel.  Re-run: `python tools/make_golden_opencv.py`.
"""
import os

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "opencv")


def opencv_pad(img):
    kern = cv2.getStructuringElement(cv2.MORPH_RECT, (25, 25))      # :595
    dilated = cv2.dilate(img, kern)                                 # :598
    bgra = cv2.split(img)                                           # :601
    alpha_mask = cv2.bitwise_not(cv2.merge([bgra[3]] * 4))          # :603-607
    return cv2.add(img, cv2.bitwise_and(dilated, alpha_mask))       # :609-612


def main():
    rng = np.random.default_rng(1)
    out = {}
    for res, fill in ((256, 0.3), (200, 0.02), (64, 1.0)):
        img = np.zeros((res, res, 4), np.uint8)
        m = rng.random((res, res)) < fill
        img[m, :3] = rng.integers(0, 256, (int(m.sum()), 3))
        img[m, 3] = 255
        out[f"in_{res}"], out[f"padded_{res}"] = img, opencv_pad(img)
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, "pad.npz"), opencv_version=cv2.__version__, **out)


if __name__ == "__main__":
    main()
