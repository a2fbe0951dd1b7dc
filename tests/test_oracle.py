"""CPU tests: the plain-C oracle against (a) the committed golden vectors dumped from the reference's own
vendored OpenCV 4.5.5 (tools/make_golden.py) and (b) the reference library itself, live when it is built in this tree,
else its recorded results (tests/golden/reference)."""
import ctypes as C

import numpy as np
import pytest

from conftest import P, digest, golden
from alvaar_b200 import synth


def test_gray_golden(oracle):
    g = golden("gray")
    out = np.empty_like(g["gray"])
    oracle.orc_gray(P(np.ascontiguousarray(g["rgba"])), 64, 48, P(out))
    assert (out == g["gray"]).all()


def test_pyramid_golden(oracle):
    g = golden("pyramid")
    img = np.ascontiguousarray(g["img"])
    h, w = img.shape
    assert oracle.orc_pyramid_levels(w, h, 9, 3) == int(g["levels"])
    cur = img
    for k in (1, 2, 3):
        hh, ww = cur.shape
        nxt = np.empty(((hh + 1) // 2, (ww + 1) // 2), np.uint8)
        oracle.orc_pyrdown(P(cur), ww, hh, P(nxt))
        assert (nxt == g[f"l{k}"]).all(), k
        cur = nxt


def test_pyramid_level_rule(oracle):
    # buildOpticalFlowPyramid stops when a level is not larger than the window (lkpyramid.cpp:811-816)
    assert oracle.orc_pyramid_levels(1280, 720, 9, 3) == 3
    assert oracle.orc_pyramid_levels(40, 30, 9, 3) == 1
    assert oracle.orc_pyramid_levels(16, 16, 9, 3) == 0


@pytest.mark.parametrize("thr,nms", [(20, 1), (20, 0), (7, 1), (7, 0)])
def test_fast_golden(oracle, thr, nms):
    g = golden("fast")
    img = np.ascontiguousarray(g["img"])
    h, w = img.shape
    want = g[f"kp_t{thr}_n{nms}"]
    got = np.zeros((w * h, 3), np.int32)
    n = oracle.orc_fast9(P(img), w, h, thr, nms, P(got), w * h)
    assert n == len(want)
    assert (got[:n] == want).all()


def test_orb_golden(oracle):
    g = golden("orb")
    img = np.ascontiguousarray(g["img"])
    h, w = img.shape
    k7 = np.zeros(7, np.float32)
    oracle.orc_gauss7_kernel(P(k7))
    assert (k7.view(np.uint32) == g["gauss7"].view(np.uint32)).all()
    for fused, key in ((0, "blur"), (1, "blur_fma")):
        b = np.empty_like(img)
        oracle.orc_orb_blur(P(img), w, h, fused, P(b))
        assert (b == g[key]).all(), key
    blur = np.ascontiguousarray(g["blur"])
    pts = np.ascontiguousarray(g["pts"])
    n = len(pts)
    for ang_key, d_key, k_key in ((None, "desc", "kept"), ("angles", "desc_angles", "kept_angles")):
        desc = np.zeros((n, 32), np.uint8)
        kept = np.zeros(n, np.uint8)
        ang = np.ascontiguousarray(g[ang_key]) if ang_key else None
        oracle.orc_orb_describe(P(blur), w, h, P(pts), P(ang) if ang is not None else None, n, P(desc), P(kept))
        assert (kept == g[k_key]).all()
        m = kept == 1
        assert m.sum() > 100
        assert (desc[m] == g[d_key][m]).all()


def test_orb_detect_golden(oracle):
    """ORB::detectAndCompute (nlevels 1): Harris response, IC angle and descriptors of the reference's keypoints."""
    g = golden("orb")
    img = np.ascontiguousarray(g["img"])
    h, w = img.shape
    kp = g["det_kp"]
    n = len(kp)
    assert n > 100
    pts = np.ascontiguousarray(kp[:, :2])
    ang = np.zeros(n, np.float32)
    oracle.orc_ic_angles(P(img), w, h, P(pts), n, P(ang))
    assert (ang.view(np.uint32) == kp[:, 3].copy().view(np.uint32)).all()
    hr = np.zeros(n, np.float32)
    oracle.orc_harris(P(img), w, h, P(pts), n, P(hr))
    assert (hr.view(np.uint32) == kp[:, 2].copy().view(np.uint32)).all()
    blur = np.ascontiguousarray(g["blur"])
    desc = np.zeros((n, 32), np.uint8)
    kept = np.zeros(n, np.uint8)
    oracle.orc_orb_describe(P(blur), w, h, P(pts), P(ang), n, P(desc), P(kept))
    assert kept.all() and (desc == g["det_desc"]).all()


def test_knn_golden(oracle):
    g = golden("knn")
    q, t = np.ascontiguousarray(g["q"]), np.ascontiguousarray(g["t"])
    out = np.zeros((len(q), 4), np.int32)
    oracle.orc_knn2(P(q), len(q), P(t), len(t), P(out))
    assert (out == g["out"]).all()
    # tie rule: duplicates of the same train row -> the LOWEST index wins, the duplicate is second
    assert (out[150:160, 0] == np.arange(10)).all() and (out[150:160, 1] == 0).all()
    assert (out[150:160, 2] == 400 + np.arange(10)).all()


def test_retain_best_threshold(oracle):
    xs = np.zeros((10, 3), np.int32)
    xs[:, 2] = [50, 40, 40, 40, 30, 30, 20, 20, 20, 20]
    assert oracle.orc_retain_best_threshold(P(xs), 10, 3) == 40     # ties at the boundary are all kept
    assert oracle.orc_retain_best_threshold(P(xs), 10, 10) == 0
    assert oracle.orc_retain_best_threshold(P(xs), 10, 1) == 50


# ---------------------------------------------------------------- the reference library (live, or its recorded results)
def test_live_reference_frontend(oracle, ref_results):
    ref = ref_results.lib
    for (w, h, seed) in [(640, 480, 1), (333, 217, 2), (1280, 720, 3)]:
        rgba = synth.random_rgba(w, h, 1, seed)[0]
        img = synth.crop(w, h, 17 * seed, 29 * seed)
        dw, dh = (w + 1) // 2, (h + 1) // 2

        def gray():
            a = np.empty((h, w), np.uint8)
            ref.ref_gray(P(rgba), w, h, P(a))
            return (digest(a),)

        def pyrdown():
            a = np.empty((dh, dw), np.uint8)
            ref.ref_pyrdown(P(img), w, h, P(a))
            return (digest(a),)

        def fast():
            xa = np.zeros((w * h, 3), np.int32)
            na = ref.ref_fast(P(img), w, h, 20, 1, P(xa), w * h)
            return (na, digest(xa[:na]))
        a, = ref_results.get(f"frontend/{w}x{h}/gray", gray)
        b = np.empty((h, w), np.uint8)
        oracle.orc_gray(P(rgba), w, h, P(b))
        assert (digest(b) == a).all()
        a, = ref_results.get(f"frontend/{w}x{h}/pyrdown", pyrdown)
        b = np.empty((dh, dw), np.uint8)
        oracle.orc_pyrdown(P(img), w, h, P(b))
        assert (digest(b) == a).all()
        xb = np.zeros((w * h, 3), np.int32)
        na, xa = ref_results.get(f"frontend/{w}x{h}/fast", fast)
        nb = oracle.orc_fast9(P(img), w, h, 20, 1, P(xb), w * h)
        assert na == nb and (digest(xb[:nb]) == xa).all()


def test_live_reference_orb(oracle, ref_results):
    ref = ref_results.lib
    w, h = 640, 480
    img = synth.crop(w, h, 100, 900)
    rng = np.random.default_rng(8)
    n = 4000
    pts = np.stack([rng.uniform(0, w, n), rng.uniform(0, h, n)], 1).astype(np.float32)
    ang = rng.uniform(0, 360, n).astype(np.float32)
    blur = np.empty_like(img)
    oracle.orc_orb_blur(P(img), w, h, 0, P(blur))
    for angles in (None, ang):
        db, kb = np.zeros((n, 32), np.uint8), np.zeros(n, np.uint8)

        def compute():
            da, ka = np.zeros((n, 32), np.uint8), np.zeros(n, np.uint8)
            ref.ref_orb_compute(P(img), w, h, P(pts), P(angles) if angles is not None else None, n, P(da), P(ka))
            return (digest(da[ka == 1]), ka)
        da, ka = ref_results.get(f"orb/{'angles' if angles is not None else 'upright'}", compute)
        oracle.orc_orb_describe(P(blur), w, h, P(pts), P(angles) if angles is not None else None, n, P(db), P(kb))
        assert (ka == kb).all() and (digest(db[kb == 1]) == da).all()


def _sorted_kp(kp, desc):
    o = np.lexsort((kp[:, 0], kp[:, 1]))
    return kp[o], desc[o]


def test_orb_detect_composition_golden(oracle):
    """orc_orb_detect (FAST -> border -> retainBest(2n) -> Harris -> retainBest(n) -> IC angle -> blur -> rBRIEF) equals the
    reference's ORB::detectAndCompute keypoint SET bit for bit (x, y, response, angle, descriptor)."""
    g = golden("orb")
    img = np.ascontiguousarray(g["img"])
    h, w = img.shape
    kp, d = np.zeros((2000, 4), np.float32), np.zeros((2000, 32), np.uint8)
    n = oracle.orc_orb_detect(P(img), w, h, 300, 20, 0, P(kp), P(d), 2000)
    gk, gd = _sorted_kp(g["det_kp"], g["det_desc"])
    assert n == len(gk)
    assert (kp[:n].view(np.uint32) == np.ascontiguousarray(gk[:, :4]).view(np.uint32)).all()
    assert (d[:n] == gd).all()


@pytest.mark.parametrize("w,h,nfeat,thr", [(640, 480, 500, 20), (320, 240, 100, 30), (200, 150, 1000, 10)])
def test_orb_detect_composition_vs_reference(oracle, ref_results, w, h, nfeat, thr):
    img = synth.crop(w, h, 100 + w, 50 + h // 2)
    assert img.shape == (h, w)
    kp, d = np.zeros((8000, 4), np.float32), np.zeros((8000, 32), np.uint8)
    n = oracle.orc_orb_detect(P(img), w, h, nfeat, thr, 0, P(kp), P(d), 8000)

    def detect():
        rk, rd = np.zeros((8000, 5), np.float32), np.zeros((8000, 32), np.uint8)
        nr = ref_results.lib.ref_orb_detect(P(img), w, h, nfeat, thr, P(rk), P(rd), 8000)
        return (nr, rk[:nr], rd[:nr])
    nr, rk, rd = ref_results.get(f"orb_detect/{w}x{h}/{nfeat}/{thr}", detect)
    assert n == nr and n > 20
    gk, gd = _sorted_kp(rk[:nr], rd[:nr])
    assert (kp[:n].view(np.uint32) == np.ascontiguousarray(gk[:, :4]).view(np.uint32)).all()
    assert (d[:n] == gd).all()


def test_scharr_golden(oracle):
    """Derivative pyramid of buildOpticalFlowPyramid(withDerivatives): int16 (dx, dy) per level, bit-exact."""
    g = golden("scharr")
    for k in range(4):
        lv = np.ascontiguousarray(g[f"l{k}"])
        h, w = lv.shape
        out = np.zeros((h, w, 2), np.int16)
        oracle.orc_scharr(P(lv), w, h, P(out))
        assert (out == g[f"d{k}"]).all()


@pytest.mark.parametrize("w,h", [(640, 480), (33, 17), (7, 5), (1, 9), (9, 1), (2, 2)])
def test_scharr_vs_reference(oracle, ref_results, w, h):
    img = np.ascontiguousarray(synth.crop(max(w, 16), max(h, 16), 40, 60)[:h, :w])

    def pyramid():
        lv, dv = np.zeros((h, w), np.uint8), np.zeros((h, w, 2), np.int16)
        LP, DP = (C.c_void_p * 4)(lv.ctypes.data, None, None, None), (C.c_void_p * 4)(dv.ctypes.data, None, None, None)
        ref_results.lib.ref_build_pyramid(P(img), w, h, 3, 0, LP, DP)
        return (digest(lv), digest(dv))
    lv, dv = ref_results.get(f"scharr/{w}x{h}", pyramid)
    out = np.zeros((h, w, 2), np.int16)
    oracle.orc_scharr(P(img), w, h, P(out))
    assert (digest(img) == lv).all() and (digest(out) == dv).all()
