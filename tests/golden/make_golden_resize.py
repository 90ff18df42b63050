"""Generates tests/golden/resize_cases.npz and tests/golden/resize_images.npz with the REAL cv2.resize(...,
interpolation=cv2.INTER_LINEAR) / cv2.imread calls of the reference (utils/datasets.py:106-111, test.py:34-37).  Needs OpenCV
and a checkout of the reference (for its bundled img/*.jpg); the tests need neither.

resize_cases.npz: sources are seeded noise (oracle.resize.noise_image) and are not stored; `cases` holds (seed, h, w, H, W) per
row.  The cv2 output of row i (HWC, as cv2 returns it) is stored as `out_<i>` when it is at most STORE_BYTES bytes, otherwise as
`sha256_<i>`, the SHA-256 of its bytes (oracle.resize.digest): noise does not compress, and the digest pins it just as exactly.
resize_images.npz: `img_000139` / `img_000004`, cv2.imread of the reference's bundled img/*.jpg (decoded arrays, the input
test.py resizes).  Both record the OpenCV that produced them in `cv2_version`.

    python tests/golden/make_golden_resize.py <reference checkout>
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

STORE_BYTES = 32 * 1024

# (h, w, H, W): source -> destination
CASES = [
    (480, 640, 352, 352), (640, 480, 192, 352),          # COCO-like downscales to the network input
    (853, 1280, 640, 640),                               # ... and to 640
    (427, 640, 61, 97), (375, 500, 37, 50),              # COCO-like sizes to small destinations
    (24, 31, 352, 352),                                  # upscale
    (1, 1, 352, 352), (1, 500, 352, 352), (500, 1, 352, 352),
    (122, 194, 61, 97), (183, 291, 61, 97), (244, 388, 61, 97),   # exact 2x, 3x, 4x downscales (OpenCV: INTER_AREA path)
    (61, 97, 61, 97),                                    # identity
    (97, 61, 61, 97), (50, 40, 3, 2), (33, 17, 1, 1), (1, 1, 1, 1),   # odd destinations
    (2000, 300, 45, 200), (7, 900, 300, 13), (300, 5, 17, 400),        # skipped source rows, thin sources
]


def main(ref):
    import cv2
    from oracle.resize import digest, noise_image
    version = np.array(cv2.__version__)
    out = {"cases": np.array([(100 + i,) + c for i, c in enumerate(CASES)], np.int64), "cv2_version": version}
    for i, (h, w, H, W) in enumerate(CASES):
        r = cv2.resize(noise_image(100 + i, h, w), (W, H), interpolation=cv2.INTER_LINEAR)
        if r.nbytes <= STORE_BYTES:
            out["out_%d" % i] = r
        else:
            out["sha256_%d" % i] = digest(r)
    np.savez_compressed(os.path.join(HERE, "resize_cases.npz"), **out)
    imgs = {"img_" + name: cv2.imread(os.path.join(ref, "img", name + ".jpg")) for name in ("000139", "000004")}
    np.savez_compressed(os.path.join(HERE, "resize_images.npz"), cv2_version=version, **imgs)
    print("wrote resize_cases.npz, resize_images.npz (cv2 %s, %d cases)" % (cv2.__version__, len(CASES)))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
