"""GPU parity tests for CLAHE (icg_clahe_apply / _apply_dev) through the C ABI: bit-exact against the cv2 golden vectors and the oracle."""
import os

import numpy as np
import pytest

from tests import oracle_api as oa
from tests.test_oracle_clahe import assert_cv2_golden

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "clahe_golden.npz")


def cases():
    g = np.load(GOLD)
    return sorted(k[:-3] for k in g.files if k.endswith("_in"))


@pytest.mark.parametrize("name", cases())
def test_clahe_matches_cv2_golden(name):
    from ic_gvins_b200.clahe import Clahe
    g = np.load(GOLD)
    img = g[name + "_in"]
    tx, ty, clip = g[name + "_par"]
    c = Clahe(img.shape[1], img.shape[0], clip, (int(tx), int(ty)))
    out = c.apply(img)
    assert_cv2_golden(out, g, name)
    inplace = img.copy()
    c.apply(inplace, inplace)  # clahe_->apply(image, image) as the reference calls it (tracking.cc:141)
    assert_cv2_golden(inplace, g, name)
    c.close()


def test_clahe_matches_oracle_on_stream_frames(oracle):
    """the bench's synthetic frames, at the reference's size and parameters (1280 x 560, clip 3.0, 21 x 21 tiles)"""
    from datagen import synth_klt
    from ic_gvins_b200.clahe import Clahe
    st = synth_klt.KltStream(1280, 560, 10, 77)
    c = Clahe(1280, 560, 3.0, (21, 21))
    for t in range(3):
        img = st.frame(t)
        assert np.array_equal(c.apply(img), oa.clahe_apply(oracle, img, 3.0, 21, 21))
    c.close()


def test_clahe_device_resident_into_klt_slot(oracle):
    """upload a raw frame into a KLT slot, equalise it in place on the device, build the pyramid: level 0 must equal the oracle's CLAHE"""
    import ctypes as C
    from ic_gvins_b200._lib import check, lib, vp
    from ic_gvins_b200.clahe import Clahe
    from ic_gvins_b200.klt import KltTracker
    rng = np.random.default_rng(5)
    W, H = 640, 480
    img = rng.integers(0, 256, (H, W), dtype=np.uint8)
    img[100:200, 50:300] //= 4
    trk = KltTracker(W, H, n_slots=2, max_points=16)
    trk.upload(0, img, build=False)
    ptr, pitch = vp(), C.c_int()
    check(lib().icg_klt_slot_level0(trk._h, 0, C.byref(ptr), C.byref(pitch)), "icg_klt_slot_level0")
    trk.sync()
    c = Clahe(W, H, 3.0, (21, 21))
    c.apply_dev(ptr.value, pitch.value, ptr.value, pitch.value)
    c.sync()
    trk.build_pyramids(0, 1)
    got = trk.download_level(0, 0)
    assert np.array_equal(got, oa.clahe_apply(oracle, img, 3.0, 21, 21))
    c.close()
    trk.close()


def test_batched_device_clahe_and_fused_histogram_gate(oracle):
    """icg_clahe_apply_batch_dev on the level-0 planes of consecutive KLT slots: every frame bit-exact with the oracle (== cv2), and the
    histogram-gate statistic of the RAW frames (Tracking::calculateHistigram) equal to the host function / the cv2.calcHist restatement."""
    import ctypes as C
    from datagen import synth_klt as synth
    from ic_gvins_b200._lib import lib, vp
    from ic_gvins_b200.camera import calculate_histogram
    from ic_gvins_b200.clahe import Clahe
    from ic_gvins_b200.klt import KltTracker
    from tests import oracle_api as oa
    W, H, NF = 1280, 560, 4
    st = synth.KltStream(W, H, 300, 91)
    frames = [st.frame(t) for t in range(NF)]
    frames[2] = (frames[2].astype(np.int32) * 3 // 4).astype(np.uint8)  # a darker frame: the gate statistic must move
    trk = KltTracker(W, H, n_slots=NF, max_points=64)
    for k, f in enumerate(frames):
        trk.upload(k, f, build=False)
    trk.sync()
    p0, p1, pitch = vp(), vp(), C.c_int()
    lib().icg_klt_slot_level0(trk._h, 0, C.byref(p0), C.byref(pitch))
    lib().icg_klt_slot_level0(trk._h, 1, C.byref(p1), C.byref(pitch))
    stride = p1.value - p0.value
    cl = Clahe(W, H, 3.0, (21, 21))
    hist = cl.apply_batch_dev(NF, p0.value, pitch.value, stride, p0.value, pitch.value, stride, want_hist=True)
    for k, f in enumerate(frames):
        assert np.array_equal(trk.download_level(k, 0), oa.clahe_apply(oracle, f, 3.0, 21, 21)), k
        assert hist[k] == calculate_histogram(f), k
    assert abs(hist[2] - hist[1]) / hist[1] > 0.1  # the darker frame would be skipped by the gate (tracking.cc:121-131)
    # without the statistic the call is asynchronous and gives the same pixels
    for k, f in enumerate(frames):
        trk.upload(k, f, build=False)
    assert cl.apply_batch_dev(NF, p0.value, pitch.value, stride, p0.value, pitch.value, stride) is None
    cl.sync()
    for k, f in enumerate(frames):
        assert np.array_equal(trk.download_level(k, 0), oa.clahe_apply(oracle, f, 3.0, 21, 21)), k
    cl.close()
    trk.close()
