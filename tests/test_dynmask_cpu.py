"""Dynamic-mask stages (perfect/src/Flow.cc:24-47, perfect/src/Frame.cc:356-377): the oracle against OpenCV's own outputs
(fixtures written from cv2 by tools/make_dynmask_golden.py, and cv2 live where it is importable), CPU only."""
import os

import numpy as np
import pytest

from oracle import dynmask_py as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = ["a", "b", "c", "d", "e"]   # e: odd-sized gray image (33 x 47 over a 16 x 23 flow field)


def _load(name):
    g = np.load(os.path.join(GOLD, "dynmask_%s.npz" % name))
    return g, g["flow"], float(g["thr"])


@pytest.mark.parametrize("name", CASES)
def test_oracle_equals_cv2_golden(name):
    g, flow, thr = _load(name)
    f2 = O.pyr_up(flow)
    assert f2.shape == (2 * flow.shape[0], 2 * flow.shape[1], 2)
    assert (f2[::7, ::5] == g["flow2_sample"]).all()                                         # bit-exact floats
    border = np.concatenate([f2[0].ravel(), f2[-1].ravel(), f2[:, 0].ravel(), f2[:, -1].ravel()])
    assert (border == g["flow2_border"]).all()
    shape = tuple(int(v) for v in g["shape"])
    m0 = np.ones(shape, np.uint8)
    m0[:f2.shape[0], :f2.shape[1]] = O.flow_mask(f2, thr)
    assert (np.packbits(m0) == g["mask0"]).all()
    assert (np.packbits(O.mask_from_flow(flow, thr, shape)) == g["mask"]).all()
    assert (O.ellipse(21) == g["element"]).all()


def test_oracle_equals_cv2_live():
    cv2 = pytest.importorskip("cv2")
    from orb_slam2_ssd_semantic_b200.synth import flow_field
    flow = flow_field(21, 57, 91)
    up = cv2.pyrUp(flow, dstsize=(2 * 91, 2 * 57))
    assert (O.pyr_up(flow) == up).all()
    k = cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (21, 21), (10, 10))
    assert (O.ellipse(21) == k).all()
    m0 = O.flow_mask(up, 40.0)
    ref = cv2.dilate(cv2.erode(cv2.erode(m0, k), k), k)
    assert (O.mask_from_flow(flow, 40.0) == ref).all()
    m1 = np.ones((115, 183), np.uint8)            # odd-sized gray image: the extra row / column starts as 1
    m1[:114, :182] = m0
    ref = cv2.dilate(cv2.erode(cv2.erode(m1, k), k), k)
    assert (O.mask_from_flow(flow, 40.0, (115, 183)) == ref).all()


def test_threshold_floor_and_nan():
    f2 = np.zeros((4, 4, 2), np.float32)
    f2[0, 0] = (6.0, 2.0)          # 40 -> not below 40 -> dynamic
    f2[0, 1] = (6.0, 1.9)          # 39.61 -> static
    f2[0, 2] = (np.nan, 0.0)       # NaN compares false -> dynamic
    m = O.flow_mask(f2, 1.0)       # thresholds below 40 are raised to 40 (Flow.cc:24)
    assert m[0, 0] == 0 and m[0, 1] == 1 and m[0, 2] == 0 and m[1:].all()


def test_filter_keypoints_rule():
    from orb_slam2_ssd_semantic_b200.extractor import KP_DTYPE
    rng = np.random.Generator(np.random.PCG64(5))
    mask = np.ones((48, 64), np.uint8)
    mask[10:20, 10:30] = 0
    mask[30, 40] = 2                                     # "val == 1" only
    kps = np.zeros(200, KP_DTYPE)
    kps["x"] = rng.uniform(0, 63.99, 200).astype(np.float32)
    kps["y"] = rng.uniform(0, 47.99, 200).astype(np.float32)
    kps["x"][0], kps["y"][0] = 40.7, 30.2                # lands on the 2
    desc = rng.integers(0, 256, (200, 32)).astype(np.uint8)
    k2, d2 = O.filter_keypoints(mask, kps, desc)
    keep = mask[kps["y"].astype(int), kps["x"].astype(int)] == 1
    assert not keep[0] and len(k2) == keep.sum() and (d2 == desc[keep]).all() and k2.tobytes() == kps[keep].tobytes()
    # at most 65 % ones: nothing is dropped
    mask2 = np.zeros((48, 64), np.uint8)
    mask2[:31] = 1                                       # 31/48 = 64.6 %
    k3, d3 = O.filter_keypoints(mask2, kps, desc)
    assert len(k3) == 200 and (d3 == desc).all()


def test_filter_oracle_equals_the_reference_masked_constructor():
    """oracle == the `perfect` tree's OWN code: perfect/src/Frame.cc compiled unmodified (oracle/_ref/librefperfect.so).
    filter_keypoints(mask, what the plain RGB-D constructor keeps) must be what the masked constructor keeps (:328-427),
    bit for bit -- with a real dynamic mask (filter on), with a mask at 64.6 % (filter off, :358) and with stray values.
    The reference's outputs are recorded (tests/reference_outputs.py); live where the library exists."""
    from oracle import ref
    from orb_slam2_ssd_semantic_b200 import synth
    from tests.reference_outputs import Reference
    R = Reference("test_filter_oracle_equals_the_reference_masked_constructor", ref.refperfect_available())
    ws = synth.WallStream(seed=1234, n=2)
    gray, depth, _, _ = ws.frame(1)
    real = O.mask_from_flow(synth.flow_field(11, 240, 320), 40.0)
    assert 0.65 < real.mean() < 0.9
    off = np.zeros((480, 640), np.uint8)
    off[:310] = 1                                          # 64.6 % ones: not above 65 %, nothing may be dropped
    stray = np.ones((480, 640), np.uint8)
    stray[:, 200:330] = 2                                  # "val == 1" only: a 2 is outside
    stray[100:140] = 0
    # what the plain constructor keeps is the extractor's output (zero distortion), which tests/test_refsrc_cpu.py pins
    kp, dp = ref.RefExtractor(1000, 1.2, 8, 20, 7)(gray)
    assert len(kp) > 900
    for name, mask in (("real", real), ("off", off), ("stray", stray)):
        ko, do = O.filter_keypoints(mask, kp, dp)
        R.same(name, ((kp, dp), (ko, do)), lambda: ref.perfect_frames(gray, depth, mask))
        if name == "off":
            assert len(ko) == len(kp)
        else:
            assert 0 < len(ko) < len(kp)


@pytest.mark.parametrize("rows,cols,gray_shape,thr,seed", [(2, 2, (4, 4), 40.0, 1), (2, 9, (5, 19), 40.0, 2), (31, 17, (63, 34), 55.5, 3),
                                                           (64, 48, (128, 97), 200.0, 4), (100, 3, (201, 7), 0.0, 5)])
def test_mask_oracle_equals_cv2_live_shapes(rows, cols, gray_shape, thr, seed):
    """Random shapes incl. 2-pixel-wide fields and odd-sized gray images, against cv2 run here (skipped without cv2)."""
    cv2 = pytest.importorskip("cv2")
    from orb_slam2_ssd_semantic_b200.synth import flow_field
    flow = flow_field(100 + seed, rows, cols, blobs=3)
    up = cv2.pyrUp(flow, dstsize=(2 * cols, 2 * rows))
    assert (O.pyr_up(flow) == up).all()
    m0 = np.ones(gray_shape, np.uint8)
    t2 = up[..., 0] * up[..., 0] + up[..., 1] * up[..., 1]
    m0[:2 * rows, :2 * cols] = (t2 < max(np.float32(thr), np.float32(40.0))).astype(np.uint8)
    k = cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (21, 21), (10, 10))
    ref = cv2.dilate(cv2.erode(cv2.erode(m0, k), k), k)
    assert (O.mask_from_flow(flow, thr, gray_shape) == ref).all()
