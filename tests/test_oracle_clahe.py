"""The CLAHE oracle (oracle/clahe_ref.c) against the cv2 golden vectors: bit-exact.  CPU only."""
import hashlib
import os

import numpy as np
import pytest

from tests import oracle_api as oa

GOLD = os.path.join(os.path.dirname(__file__), "golden", "clahe_golden.npz")


def cases():
    g = np.load(GOLD)
    return sorted(k[:-3] for k in g.files if k.endswith("_in"))


def assert_cv2_golden(out, g, name):
    """bit-exact with cv2: the fixture holds the SHA-256 of cv2's uint8 output (tests/golden/make_clahe_golden.py)"""
    assert out.dtype == np.uint8 and out.shape == g[name + "_in"].shape
    assert hashlib.sha256(np.ascontiguousarray(out).tobytes()).hexdigest() == str(g[name + "_out_sha256"]), f"{name}: output differs from cv2"


@pytest.mark.parametrize("name", cases())
def test_clahe_oracle_matches_cv2_golden(oracle, name):
    g = np.load(GOLD)
    img = g[name + "_in"]
    tx, ty, clip = g[name + "_par"]
    out = oa.clahe_apply(oracle, img, clip, int(tx), int(ty))
    assert_cv2_golden(out, g, name)


def test_clahe_oracle_in_place(oracle):
    g = np.load(GOLD)
    img = g["ref_1280x560_in"].copy()
    oa.clahe_apply(oracle, img, 3.0, 21, 21, in_place=True)
    assert_cv2_golden(img, g, "ref_1280x560")


def test_clahe_oracle_flat_and_extremes(oracle):
    """edge cases the golden set does not hold: a constant image (every histogram is one spike that the clip limit spreads out), pure
    black / white, and a 1-tile grid (global histogram equalisation with a clip)"""
    cv2 = pytest.importorskip("cv2")  # live comparison (the build container has cv2 4.13.0; fixtures cover the rest)
    for img, clip, grid in ((np.full((64, 96), 77, np.uint8), 3.0, (4, 4)), (np.zeros((48, 48), np.uint8), 2.0, (3, 3)),
                            (np.full((40, 56), 255, np.uint8), 40.0, (7, 5)), (np.arange(60 * 80, dtype=np.uint32).reshape(60, 80).astype(np.uint8), 4.0, (1, 1))):
        ref = cv2.createCLAHE(clip, grid).apply(img)
        assert np.array_equal(oa.clahe_apply(oracle, img, clip, grid[0], grid[1]), ref)
