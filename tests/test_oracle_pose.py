"""CPU tests: the pose oracle (oracle/pose_oracle.c) against (a) golden vectors dumped from the reference's own
MultiViewGeometry + vendored OpenGV / Ceres (tools/make_golden_pose.py) and (b) the reference, live or recorded.
fp64: poses within 1e-9 (far inside the 1e-4 relative bar), inlier / outlier sets exact."""
import ctypes as C

import numpy as np
import pytest

from conftest import P, golden
from pose_util import make_pose_problem

f32 = C.c_float
HUBER = float(np.sqrt(np.float32(5.9915)))   # ceresPnP: std::sqrt(float chi2th) (multi_view_geometry.cpp:147)
CHI2 = float(np.float32(5.9915))


def orc_p3p(oracle, bv, X, K, seed=12345, max_iter=100, err=3.0):
    n = len(bv)
    oracle.orc_p3p_lmeds.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, f32, f32, f32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
    T, o, info = np.zeros(12), np.zeros(n, np.uint8), np.zeros(3)
    ok = oracle.orc_p3p_lmeds(P(np.ascontiguousarray(bv)), P(np.ascontiguousarray(X)), n, max_iter, err, K[0], K[1], seed, P(T), P(o), P(info))
    return ok, T, o, info


def orc_pnp(oracle, uv, X, K, pose0, rob=1, l2=1, max_iter=5):
    n = len(uv)
    oracle.orc_pnp.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int,
                               C.c_void_p, C.c_void_p]
    p, o, s = np.array(pose0, np.float64).copy(), np.zeros(n, np.uint8), np.zeros(10)
    Kd = np.ascontiguousarray(K, np.float64)
    ok = oracle.orc_pnp(P(Kd), P(np.ascontiguousarray(uv)), P(np.ascontiguousarray(X)), n, P(p), HUBER, CHI2, max_iter, rob, l2, P(o), P(s))
    return ok, p, o, s


@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_p3p_lmeds_golden(oracle, tag):
    g = golden("pose")
    ok, T, o, _ = orc_p3p(oracle, g[f"{tag}_bv"], g[f"{tag}_X"], g[f"{tag}_K"])
    assert ok == int(g[f"{tag}_p3p_ok"]) == 1
    assert (o == g[f"{tag}_p3p_outlier"]).all()
    assert np.abs(T - g[f"{tag}_p3p_T"]).max() < 1e-9


@pytest.mark.parametrize("tag", ["a", "b", "c"])
@pytest.mark.parametrize("rob,l2", [(1, 1), (1, 0), (0, 0)])
def test_pnp_golden(oracle, tag, rob, l2):
    g = golden("pose")
    ok, p, o, _ = orc_pnp(oracle, g[f"{tag}_uv"], g[f"{tag}_X"], g[f"{tag}_K"].astype(np.float64), g[f"{tag}_pose0"], rob, l2)
    assert ok == int(g[f"{tag}_pnp{rob}{l2}_ok"]) == 1
    assert (o == g[f"{tag}_pnp{rob}{l2}_outlier"]).all()
    assert np.abs(p - g[f"{tag}_pnp{rob}{l2}_pose"]).max() < 1e-9


def test_sampler_sequence_is_mt19937_shift(oracle):
    """SampleConsensusProblem::rnd(): uniform_int_distribution<int>(0, INT_MAX) over mt19937(12345) == x >> 1 (libstdc++)."""
    out = np.zeros(8, np.int32)
    oracle.orc_sac_rnd(12345, 8, P(out))
    # first outputs of std::mt19937(12345): 3992670690, 3823185381, ... (checked against numpy's MT19937 below)
    bg = np.random.MT19937()
    st = bg.state
    key = np.zeros(624, np.uint32)
    key[0] = 12345
    for i in range(1, 624):
        key[i] = (1812433253 * (int(key[i - 1]) ^ (int(key[i - 1]) >> 30)) + i) & 0xFFFFFFFF
    st["state"]["key"], st["state"]["pos"] = key, 624
    bg.state = st
    want = (bg.random_raw(8) >> 1).astype(np.int32)
    assert (out == want).all()


@pytest.mark.parametrize("n,seed,of", [(120, 11, 0.2), (700, 12, 0.35), (9, 13, 0.0)])
def test_pose_live_reference(oracle, ref_results, n, seed, of):
    ref = ref_results.lib
    pr = make_pose_problem(n, seed, outlier_frac=of)
    K32 = pr["K"].astype(np.float32)

    def p3p():
        ref.ref_p3p_lmeds.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, f32, f32, f32, C.c_void_p, C.c_void_p]
        T1, o1 = np.zeros(12), np.zeros(n, np.uint8)
        ok1 = ref.ref_p3p_lmeds(P(pr["bv"]), P(pr["X"]), n, 100, 3.0, K32[0], K32[1], P(T1), P(o1))
        return (ok1, T1, o1)
    ok1, T1, o1 = ref_results.get(f"p3p/{n}/{seed}/{of}", p3p)
    ok2, T2, o2, _ = orc_p3p(oracle, pr["bv"], pr["X"], K32)
    assert ok1 == ok2 == 1 and (o1 == o2).all() and np.abs(T1 - T2).max() < 1e-9
    for rob, l2 in ((1, 1), (0, 0)):
        def pnp():
            ref.ref_pnp.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, f32, C.c_int, C.c_int, f32, f32, f32, f32, C.c_void_p]
            p1, oo1 = pr["pose0"].copy(), np.zeros(n, np.uint8)
            k1 = ref.ref_pnp(P(pr["uv"]), P(pr["X"]), n, P(p1), 5, 5.9915, rob, l2, K32[0], K32[1], K32[2], K32[3], P(oo1))
            return (k1, p1, oo1)
        k1, p1, oo1 = ref_results.get(f"pnp/{n}/{seed}/{of}/{rob}{l2}", pnp)
        k2, p2, oo2, _ = orc_pnp(oracle, pr["uv"], pr["X"], K32.astype(np.float64), pr["pose0"], rob, l2)
        assert k1 == k2 == 1 and (oo1 == oo2).all() and np.abs(p1 - p2).max() < 1e-9


def test_p3p_too_few_points(oracle):
    pr = make_pose_problem(3, 1, outlier_frac=0.0)
    ok, _, _, _ = orc_p3p(oracle, pr["bv"], pr["X"], pr["K"].astype(np.float32))
    assert ok == 0   # multi_view_geometry.cpp:40-43


def test_pnp_recovers_true_pose(oracle):
    """Property: with clean data the refinement lands on the generating pose (3 LM iterations from a 5 cm / 1 deg offset)."""
    pr = make_pose_problem(400, 5, noise_px=0.0, outlier_frac=0.0)
    ok, p, o, _ = orc_pnp(oracle, pr["uv"], pr["X"], pr["K"], pr["pose0"], 1, 1, max_iter=20)
    assert ok == 1 and o.sum() == 0
    q = p[3:] * np.sign(p[6]) * np.sign(pr["pose_true"][6])
    assert np.abs(p[:3] - pr["pose_true"][:3]).max() < 1e-5 and np.abs(q - pr["pose_true"][3:]).max() < 1e-5
