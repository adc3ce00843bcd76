"""Generates tests/golden/clahe_golden.npz with cv2 (the OpenCV the reference links): `cv::createCLAHE(3.0, Size(21, 21))->apply(img, img)`
exactly as ic_gvins/ic_gvins/tracking/tracking.cc:62,141 calls it, plus parameter / size variations.  Needs cv2 (the stored file
was made with 4.13.0); the parity tests never import it.  Each case keeps its input image and the SHA-256 of cv2's uint8 output:
the textured images barely compress, and the full outputs would more than double the file."""
import hashlib
import os

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def texture(rng, W, H, sigma):
    img = cv2.GaussianBlur(rng.integers(0, 256, (H, W), dtype=np.uint8), (0, 0), sigma)
    return cv2.normalize(img, None, 0, 255, cv2.NORM_MINMAX).astype(np.uint8)


def main():
    rng = np.random.default_rng(20240923)
    cases = {}
    # name: (W, H, tiles_x, tiles_y, clip)
    spec = {
        "ref_1280x560": (1280, 560, 21, 21, 3.0),   # the reference's configuration: padded to 1281 x 567, tiles 61 x 27
        "divisible_640x480": (640, 480, 8, 8, 2.0),
        "odd_333x217": (333, 217, 21, 21, 3.0),
        "small_highclip": (100, 60, 4, 3, 40.0),
        "noclip_320x200": (320, 200, 5, 4, 0.0),
    }
    out = {}
    for name, (W, H, tx, ty, clip) in spec.items():
        img = texture(rng, W, H, 2.0 if "ref" in name else 1.2)
        if name == "small_highclip":
            img[:30] = 17  # a flat half: exercises clipping + residual redistribution
        ref = cv2.createCLAHE(clip, (tx, ty)).apply(img)
        out[name + "_in"] = img
        out[name + "_out_sha256"] = hashlib.sha256(ref.tobytes()).hexdigest()
        out[name + "_par"] = np.array([tx, ty, clip], np.float64)
    np.savez_compressed(os.path.join(HERE, "clahe_golden.npz"), cv2_version=cv2.__version__, **out)
    print("wrote clahe_golden.npz:", list(spec))


if __name__ == "__main__":
    main()
