"""CPU tests: the KLT oracle (oracle/klt_oracle.c) against (a) golden vectors dumped from the reference's own
FeatureTracker + vendored OpenCV 4.5.5 (tools/make_golden_klt.py) and (b) the reference, live or recorded.
Bit-exact: positions are compared as float bit patterns."""
import ctypes as C

import numpy as np
import pytest

from conftest import P, golden
from alvaar_b200 import synth
from klt_util import build_pyramid, klt_points, oracle_fb_klt, oracle_klt_lk


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("levels", [1, 3])
def test_fb_klt_golden(oracle, levels):
    g = golden("klt")
    a, b = g["prev"], g["cur"]
    h, w = a.shape
    L = int(g["pyr_levels"])
    pa, da = build_pyramid(oracle, a, L)
    pb, db = build_pyramid(oracle, b, L)
    q, good = oracle_fb_klt(oracle, pa, da, pb, db, w, h, levels, g["pts"], g["priors"])
    assert good.sum() > 100
    assert (good == g[f"fb{levels}_good"]).all()
    assert (bits(q) == bits(g[f"fb{levels}_pos"])).all()


@pytest.mark.parametrize("levels,ui", [(1, 0), (1, 1), (3, 0), (3, 1)])
def test_klt_lk_golden(oracle, levels, ui):
    g = golden("klt")
    a, b = g["prev"], g["cur"]
    h, w = a.shape
    L = int(g["pyr_levels"])
    pa, da = build_pyramid(oracle, a, L)
    pb, _ = build_pyramid(oracle, b, L)
    q, st, er = oracle_klt_lk(oracle, pa, da, pb, w, h, levels, g["pts"], g["priors"], use_initial=ui)
    assert (st == g[f"lk{levels}_{ui}_status"]).all()
    assert (bits(q) == bits(g[f"lk{levels}_{ui}_pos"])).all()
    assert (bits(er) == bits(g[f"lk{levels}_{ui}_err"])).all()   # level 0 always defines err (min-eig, or 0 when out of range)


@pytest.mark.parametrize("w,h,seed", [(161, 91, 2), (320, 240, 7)])
def test_fb_klt_live_reference(oracle, ref_results, w, h, seed):
    ref = ref_results.lib
    fr, _ = synth.make_frames(2, w, h, seed=seed, rgba=False)
    a, b = np.ascontiguousarray(fr[0]), np.ascontiguousarray(fr[1])
    n = 250
    pts, pri = klt_points(w, h, n, seed)
    L = int(ref_results.get(f"pyramid_levels/{w}x{h}/{seed}", lambda: (ref.ref_build_pyramid(P(a), w, h, 9, 3, None, None),))[0])
    pa, da = build_pyramid(oracle, a, L)
    pb, db = build_pyramid(oracle, b, L)
    for levels in (1, 3):
        def fb_klt():
            ref.ref_fb_klt.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
            q1, g1 = pri.copy(), np.zeros(n, np.uint8)
            ref.ref_fb_klt(P(a), P(b), w, h, 9, 3, levels, 30.0, 0.5, P(pts), P(q1), P(g1), n)
            return (q1, g1)
        q1, g1 = ref_results.get(f"fb_klt/{w}x{h}/{seed}/{levels}", fb_klt)
        q2, g2 = oracle_fb_klt(oracle, pa, da, pb, db, w, h, levels, pts, pri)
        assert (g1 == g2).all() and g1.sum() > 50
        assert (bits(q1) == bits(q2)).all()


def test_klt_identity(oracle):
    """Tracking a frame onto itself from exact priors: every textured point stays put (delta = 0; the reference's
    (p - 4) + 4 round trip may move the float by an ulp)."""
    w, h = 160, 120
    a = synth.crop(w, h, 40, 60)
    pa, da = build_pyramid(oracle, a, 3)
    rng = np.random.default_rng(3)
    pts = np.stack([rng.uniform(12, w - 12, 100), rng.uniform(12, h - 12, 100)], 1).astype(np.float32)
    q, good = oracle_fb_klt(oracle, pa, da, pa, da, w, h, 3, pts, pts)
    assert good.sum() > 80
    assert np.abs(q[good == 1] - pts[good == 1]).max() <= 2e-5
