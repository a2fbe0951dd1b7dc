"""CPU tests of the map initialisation (5-point essential matrix RANSAC + refinement, mid-point triangulation):
the oracle (oracle/init_oracle.c) and the HOST build of the device arithmetic (alvaar_b200/csrc/init_core.h, the code the CUDA
kernels in init.cu run) against (a) golden vectors dumped from the reference's own MultiViewGeometry + vendored OpenGV
(tools/make_golden_init.py) and (b) the reference, live or recorded.

Tolerances, and why.  RANSAC (sampler, hypotheses, inlier counts, adaptive stop): the selected model agrees to 1e-9 and the
outlier set exactly.  The refinement (relative_pose::optimize_nonlinear) is NOISE-LIMITED in the reference itself: it runs
Eigen's LM on forward differences of a (1 - cos) cost whose values are ~1e-7, down to ftol = xtol = 10 eps, so its end point
moves by 1e-6 .. 1e-3 when the INPUT changes by one ulp (test_reference_refinement_is_noise_limited, and the `_ulp` golden).
Parity of that stage therefore means: within the reference's own 1-ulp spread (floored at 1e-4), and a cost no worse than the
reference's."""
import ctypes as C

import numpy as np
import pytest

from conftest import P, golden
from init_util import TAGS, host_core, orc_essential, pose_error, ransac_threshold, ref_essential, refine_cost
from alvaar_b200 import synth


def spread(g, tag):
    dR, dt = pose_error(g[f"{tag}_refined_Rt"], g[f"{tag}_refined_Rt_ulp"])
    return max(10 * dR, 1e-4), max(10 * dt, 1e-4)


@pytest.mark.parametrize("tag", TAGS)
def test_ransac_model_golden(oracle, tag):
    g = golden("init")
    ok, Rt, o, info = orc_essential(oracle, g[f"{tag}_bv1"], g[f"{tag}_bv2"], g[f"{tag}_K"], 0)
    assert ok == int(g[f"{tag}_ok"]) == 1
    assert (o == g[f"{tag}_outlier"]).all()
    assert np.abs(Rt - g[f"{tag}_ransac_Rt"]).max() < 1e-9
    assert info[0] == (o == 0).sum()


@pytest.mark.parametrize("tag", TAGS)
def test_refined_model_golden(oracle, tag):
    g = golden("init")
    bv1, bv2 = g[f"{tag}_bv1"], g[f"{tag}_bv2"]
    ok, Rt, o, _ = orc_essential(oracle, bv1, bv2, g[f"{tag}_K"], 1)
    assert ok == 1 and (o == g[f"{tag}_outlier"]).all()
    tolR, tolt = spread(g, tag)
    dR, dt = pose_error(Rt, g[f"{tag}_refined_Rt"])
    assert dR < tolR and dt < tolt, (dR, dt, tolR, tolt)
    inl = o == 0
    assert refine_cost(Rt, bv1, bv2, inl) <= refine_cost(g[f"{tag}_refined_Rt"], bv1, bv2, inl) * (1 + 1e-4)


@pytest.mark.parametrize("tag", TAGS)
@pytest.mark.parametrize("opt", [0, 1, 2])
def test_device_arithmetic_on_host_golden(oracle, tag, opt):
    """init_core.h compiled for the host == the oracle == the reference (same bars).  opt = 2: the refinement by the reference's
    own minimiser restated (lmdif_core.h: MINPACK LM on forward differences) -- same bar on the pose; its cost may sit a little
    above the reference's (both stall in the rounding noise of the forward differences, at different points)."""
    g = golden("init")
    H = host_core()
    bv1, bv2, K = np.ascontiguousarray(g[f"{tag}_bv1"]), np.ascontiguousarray(g[f"{tag}_bv2"]), g[f"{tag}_K"]
    n = len(bv1)
    tab = np.zeros(8 * 1200, np.int32)
    oracle.orc_sac_rnd(12345, len(tab), P(tab))
    Rt, o, info = np.zeros(12), np.zeros(n, np.uint8), np.zeros(4)
    ok = H.host_essential_5pt(P(bv1), P(bv2), n, 100, ransac_threshold(K), opt, P(tab), len(tab), P(Rt), P(o), P(info))
    assert ok == 1 and info[0] == 1 and (o == g[f"{tag}_outlier"]).all()
    _, _, _, oinfo = orc_essential(oracle, bv1, bv2, K, min(opt, 1))
    assert info[1] == oinfo[0] and info[2] == oinfo[1] and info[3] == oinfo[2]          # inliers, iterations, draws
    if opt == 0:
        assert np.abs(Rt - g[f"{tag}_ransac_Rt"]).max() < 1e-9
    else:
        tolR, tolt = spread(g, tag)
        dR, dt = pose_error(Rt, g[f"{tag}_refined_Rt"])
        assert dR < tolR and dt < tolt
        assert refine_cost(Rt, bv1, bv2, o == 0) <= refine_cost(g[f"{tag}_refined_Rt"], bv1, bv2, o == 0) * (1 + (1e-4 if opt == 1 else 0.5))


def test_fivept_recovers_the_true_essential_matrix(oracle):
    pr = synth.make_twoview_problem(n=40, seed=3, noise_px=0, outlier_frac=0)
    t, R = pr["t12"], pr["R12"]
    E = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]]) @ R
    E /= np.linalg.norm(E)
    H = host_core()
    for lib, fn in ((oracle, "orc_fivept_nister"), (H, "host_fivept_nister")):
        for s in range(4):
            Es = np.zeros((10, 9))
            ne = getattr(lib, fn)(P(np.ascontiguousarray(pr["bv1"][5 * s:5 * s + 5])), P(np.ascontiguousarray(pr["bv2"][5 * s:5 * s + 5])), P(Es))
            assert 1 <= ne <= 10
            assert min(min(np.abs(Es[k].reshape(3, 3) - E).max(), np.abs(Es[k].reshape(3, 3) + E).max()) for k in range(ne)) < 1e-10


def test_degenerate_inputs(oracle):
    pr = synth.make_twoview_problem(n=7, seed=1)
    ok, _, _, _ = orc_essential(oracle, pr["bv1"], pr["bv2"], pr["K"].astype(np.float32), 1)
    assert ok == 0                                                                           # fewer than 8 correspondences
    pr = synth.make_twoview_problem(n=40, seed=2, outlier_frac=0.9)
    ok, _, o, info = orc_essential(oracle, pr["bv1"], pr["bv2"], pr["K"].astype(np.float32), 1)
    assert ok == 0 or info[0] >= 10                                                          # < 10 inliers -> false


def test_triangulation_golden(oracle):
    g = golden("init")
    out = np.zeros_like(g["tri_points"])
    oracle.orc_triangulate(P(g["tri_Tlr"]), P(np.ascontiguousarray(g["a_bv1"])), P(np.ascontiguousarray(g["a_bv2"])), len(out), P(out))
    assert np.abs(out - g["tri_points"]).max() < 1e-11 * np.abs(g["tri_points"]).max()
    H = host_core()
    q = g["tri_Tlr"][3:]
    R = synth.quat_to_R(q)
    p = np.zeros(3)
    for i in (0, 17, 100):
        H.host_triangulate2(P(np.ascontiguousarray(R)), P(np.ascontiguousarray(g["tri_Tlr"][:3])), P(np.ascontiguousarray(g["a_bv1"][i])), P(np.ascontiguousarray(g["a_bv2"][i])), P(p))
        assert np.abs(p - g["tri_points"][i]).max() < 1e-11 * np.abs(g["tri_points"]).max()


def test_live_reference_agreement(oracle, ref_results):
    """30 seeded problems against the reference.  The draws, the iteration count and (29 of 30) the outlier set are the
    reference's; the RANSAC-only model is the reference's to 1e-9 in 26 of 30 -- the rest are hypotheses for which the
    reference's OWN root finder stopped short (5 Newton steps from a coarse Sturm bracket + one LM polishing step,
    Sturm.cpp:296-330, fivept_nister/modules.cpp:518-545) or picked a neighbouring hypothesis with the same inlier count; its
    null-space basis comes out of a Jacobi SVD of a rank-deficient matrix and cannot be reproduced, so those stay.  After the
    refinement the poses agree whenever the outlier sets do (same band as the goldens)."""
    bad_set = bad_model = 0
    for seed in range(30):
        n = [60, 150, 192, 400][seed % 4]
        pr = synth.make_twoview_problem(n=n, seed=100 + seed, noise_px=[0.1, 0.3, 0.6][seed % 3], outlier_frac=[0.05, 0.15, 0.3][(seed // 3) % 3])
        K = pr["K"].astype(np.float32)
        ok_r, Rt_r, o_r = ref_results.get(f"agreement/{seed}/0", lambda: ref_essential(ref_results.lib, pr["bv1"], pr["bv2"], K, 0))
        ok_o, Rt_o, o_o, _ = orc_essential(oracle, pr["bv1"], pr["bv2"], K, 0)
        assert ok_r == ok_o
        if (o_r != o_o).any():
            bad_set += 1
            continue
        bad_model += np.abs(Rt_r - Rt_o).max() > 1e-9
        ok_r, Rt_r, o_r = ref_results.get(f"agreement/{seed}/1", lambda: ref_essential(ref_results.lib, pr["bv1"], pr["bv2"], K, 1))
        ok_o, Rt_o, o_o, _ = orc_essential(oracle, pr["bv1"], pr["bv2"], K, 1)
        dR, dt = pose_error(Rt_o, Rt_r)
        assert dR < 2e-3 and dt < 5e-3, (seed, dR, dt)
        assert refine_cost(Rt_o, pr["bv1"], pr["bv2"], o_o == 0) <= refine_cost(Rt_r, pr["bv1"], pr["bv2"], o_r == 0) * (1 + 1e-4)
    assert bad_set <= 2 and bad_model <= 5, (bad_set, bad_model)


def test_reference_refinement_is_noise_limited(ref_results):
    """The finding that sets the tolerance of the refined pose: a 1-ulp change of the bearing vectors moves the REFERENCE's own
    refined rotation by > 1e-7 (up to 1e-3) -- far more than the 1e-16 an exact minimiser would move."""
    rng = np.random.default_rng(0)
    moved = []
    for seed in range(6):
        pr = synth.make_twoview_problem(n=150, seed=seed)
        K = pr["K"].astype(np.float32)
        _, A, _ = ref_results.get(f"noise/{seed}/exact", lambda: ref_essential(ref_results.lib, pr["bv1"], pr["bv2"], K, 1))
        b1 = pr["bv1"] * (1 + rng.choice([-1, 0, 1], pr["bv1"].shape) * 2.2e-16)
        b2 = pr["bv2"] * (1 + rng.choice([-1, 0, 1], pr["bv2"].shape) * 2.2e-16)
        _, B, _ = ref_results.get(f"noise/{seed}/ulp", lambda: ref_essential(ref_results.lib, b1, b2, K, 1))
        moved.append(max(pose_error(A, B)))
    assert max(moved) > 1e-7
