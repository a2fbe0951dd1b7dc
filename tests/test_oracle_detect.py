"""CPU tests: the detector oracle (oracle/detect_oracle.c) against (a) golden vectors dumped from the reference's own
FeatureExtractor (tools/make_golden_detect.py) and (b) the reference, live or recorded.  Bit-exact, floats included."""
import ctypes as C

import numpy as np
import pytest

from conftest import P, golden
from alvaar_b200 import synth
from detect_util import oracle_detect, random_cur


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_detect_golden(oracle, tag):
    g = golden("detect")
    img, cs = np.ascontiguousarray(g[f"{tag}_img"]), int(g[f"{tag}_cell"])
    pts, _, q = oracle_detect(oracle, img, cs, g[f"{tag}_cur"], g[f"{tag}_roi"])
    want = g[f"{tag}_pts"]
    assert len(pts) == len(want) > 5
    assert (bits(pts) == bits(want)).all()
    h, w = img.shape
    hm = np.zeros((cs, cs), np.float32)
    bl = np.zeros((cs, cs), np.uint8)
    oracle.orc_blur3_cell(P(img), w, h, cs, cs, cs, P(bl))
    oracle.orc_min_eig_cell(P(img), w, h, cs, cs, cs, P(hm))
    assert (bl == g[f"{tag}_blur11"]).all()
    assert (bits(hm) == bits(g[f"{tag}_hmap11"])).all()


@pytest.mark.parametrize("w,h,cs,seed,ncur", [(640, 480, 40, 5, 0), (640, 480, 40, 6, 80), (1280, 720, 40, 7, 250), (400, 300, 30, 8, 20)])
def test_detect_live_reference(oracle, ref_results, w, h, cs, seed, ncur):
    fr, _ = synth.make_frames(1, w, h, seed=seed, rgba=False)
    img = np.ascontiguousarray(fr[0])
    cur = random_cur(w, h, ncur, seed)
    roi = np.array([20, 20, w - 40, h - 40], np.int32)
    for q0 in (0.001, 0.00002):
        def detect():
            ref = ref_results.lib
            ref.ref_detect_points.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_void_p, C.c_int]
            want = np.zeros((4096, 2), np.float32)
            n = ref.ref_detect_points(P(img), w, h, cs, P(cur), ncur, P(roi), q0, P(want), 4096)
            return (n, want[:n])
        n, want = ref_results.get(f"detect/{w}x{h}/{cs}/{seed}/{ncur}/{q0}", detect)
        pts, _, _ = oracle_detect(oracle, img, cs, cur, roi, q0)
        assert len(pts) == n
        assert (bits(pts) == bits(want[:n])).all()


def test_quality_adaptation(oracle):
    """feature_extractor.cpp:138-145: many detections -> x1.5; a flat image -> x0.5."""
    fr, _ = synth.make_frames(1, 320, 240, seed=1, rgba=False)
    roi = [20, 20, 280, 200]
    _, _, q = oracle_detect(oracle, np.ascontiguousarray(fr[0]), 40, np.zeros((0, 2)), roi, 0.001)
    assert q == 0.001 * 1.5
    flat = np.full((240, 320), 77, np.uint8)
    pts, _, q = oracle_detect(oracle, flat, 40, np.zeros((0, 2)), roi, 0.001)
    assert len(pts) == 0 and q == 0.0005


def test_occupied_cells_are_skipped(oracle):
    fr, _ = synth.make_frames(1, 320, 240, seed=2, rgba=False)
    img = np.ascontiguousarray(fr[0])
    cur = np.array([[60.5, 60.5], [100.0, 60.0], [140.2, 100.9]], np.float32)   # cells (1,1), (1,2), (2,3)
    pts, ints, _ = oracle_detect(oracle, img, 40, cur, [20, 20, 280, 200])
    cells = set((int(y) // 40, int(x) // 40) for x, y in ints)
    assert not cells & {(1, 1), (1, 2), (2, 3)}
    d = np.sqrt(((ints[:, None, :].astype(np.float32) - cur[None]) ** 2).sum(-1)).min(1)
    assert d.min() > 9.0   # nothing inside the radius-10 discs


def test_corner_subpix_live_reference_with_border_points(oracle, ref_results):
    """cv::cornerSubPix incl. the replicate-border sampling path (points within 5 px of the frame)."""
    w, h, n = 320, 240, 600
    fr, _ = synth.make_frames(1, w, h, seed=4, rgba=False)
    img = np.ascontiguousarray(fr[0])
    rng = np.random.default_rng(2)
    pts = np.stack([rng.uniform(0, w - 1, n), rng.uniform(0, h - 1, n)], 1).astype(np.float32)
    pts[:50, 0] = rng.uniform(0, 5, 50); pts[50:100, 1] = rng.uniform(h - 6, h - 1, 50); pts[100:150, 0] = rng.uniform(w - 6, w - 1, 50)
    args = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double]

    def subpix():
        a = pts.copy()
        ref_results.lib.ref_corner_subpix.argtypes = args
        ref_results.lib.ref_corner_subpix(P(img), w, h, P(a), n, 3, 30, 0.01)
        return (a,)
    a, = ref_results.get("corner_subpix", subpix)
    b = pts.copy()
    oracle.orc_corner_subpix.argtypes = args
    oracle.orc_corner_subpix(P(img), w, h, P(b), n, 3, 30, 0.01)
    assert (bits(a) == bits(b)).all()
