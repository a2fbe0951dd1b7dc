"""CPU tests: the BA oracle (oracle/ba_oracle.c) against ceres::Solve + AlvaAR's cost functor (live reference when
built in this tree, else its recorded results) and the committed golden solution."""
import ctypes as C

import numpy as np
import pytest

from conftest import P, golden
from alvaar_b200 import synth


def solve_with(L, prefix, pb, max_iter=5, huber=None):
    poses = pb["poses"].copy()
    invd = pb["invd"].copy()
    summary = np.zeros(8)
    costs = np.zeros(64)
    fn = getattr(L, prefix + "_ba_solve")
    fn.restype = C.c_int
    ok = fn(P(pb["calib"]), P(poses), P(pb["pose_const"]), len(poses), P(invd), P(pb["anch_kf"]), P(pb["anch_uv"]),
            len(invd), P(pb["obs_kf"]), P(pb["obs_lm"]), P(pb["obs_uv"]), len(pb["obs_kf"]),
            C.c_double(pb["huber"] if huber is None else huber), max_iter, P(summary), P(costs))
    return ok, poses, invd, summary, costs


def test_se3_plus_and_functor_vs_reference(oracle, ref_results):
    ref = ref_results.lib
    rng = np.random.default_rng(0)
    pb = synth.make_ba_problem(6, 50, 3, seed=1)
    xs, ds = [], []
    for _ in range(200):
        xs.append(pb["poses"][rng.integers(0, 6)].copy())
        ds.append(rng.normal(0, 0.05, 6) * (rng.random() < 0.9))

    def plus():
        a = np.zeros((len(xs), 7))
        for x, d, ai in zip(xs, ds, a):
            ref.ref_se3_plus(P(x), P(d), P(ai))
        return (a,)
    a_all, = ref_results.get("se3_plus", plus)
    for x, d, a in zip(xs, ds, a_all):
        b = np.zeros(7)
        oracle.orc_se3_plus(P(x), P(d), P(b))
        assert np.allclose(a, b, rtol=0, atol=1e-14)
    oracle.orc_ba_evaluate.restype = C.c_int
    nobs = len(pb["obs_kf"])

    def inputs(o):
        l = pb["obs_lm"][o]
        obs = np.array([*pb["obs_uv"][o], *pb["anch_uv"][l]])
        return l, obs, pb["poses"][pb["anch_kf"][l]].copy(), pb["poses"][pb["obs_kf"][o]].copy()

    def evaluate():
        ref.ref_ba_evaluate.restype = C.c_int
        fa, ra, Ja7, Jp7, Jda, c2a = np.zeros(nobs, np.int32), np.zeros((nobs, 2)), np.zeros((nobs, 14)), np.zeros((nobs, 14)), np.zeros((nobs, 2)), np.zeros((nobs, 1))
        for o in range(nobs):
            l, obs, anch, pose = inputs(o)
            fa[o] = ref.ref_ba_evaluate(P(pb["calib"]), P(anch), P(pose), C.c_double(pb["invd"][l]), P(obs), P(ra[o]), P(Ja7[o]), P(Jp7[o]), P(Jda[o]), P(c2a[o]))
        return (fa, ra, Ja7, Jp7, Jda, c2a)
    ref_eval = ref_results.get("evaluate", evaluate)
    for o in range(nobs):
        l, obs, anch, pose = inputs(o)
        fa, ra, Ja7, Jp7, Jda, c2a = (v[o] for v in ref_eval)
        rb, Ja6, Jp6, Jdb, c2b = np.zeros(2), np.zeros(12), np.zeros(12), np.zeros(2), np.zeros(1)
        fb = oracle.orc_ba_evaluate(P(pb["calib"]), P(anch), P(pose), C.c_double(pb["invd"][l]), P(obs), P(rb), P(Ja6), P(Jp6), P(Jdb), P(c2b))
        assert fa == fb
        assert np.allclose(ra, rb, rtol=1e-12, atol=1e-10)
        assert np.allclose(Ja7.reshape(2, 7)[:, :6], Ja6.reshape(2, 6), rtol=1e-11, atol=1e-9)
        assert np.allclose(Jp7.reshape(2, 7)[:, :6], Jp6.reshape(2, 6), rtol=1e-11, atol=1e-9)
        assert (Ja7.reshape(2, 7)[:, 6] == 0).all()
        assert np.allclose(Jda, Jdb, rtol=1e-11, atol=1e-9) and np.isclose(c2a[0], c2b[0], rtol=1e-12)


@pytest.mark.parametrize("nkf,nlm,k,seed,huber", [(20, 3000, 4, 42, None), (8, 300, 3, 7, None), (6, 120, 4, 9, 0.0),
                                                  (20, 3000, 4, 43, None)])
def test_solve_vs_ceres(oracle, ref_results, nkf, nlm, k, seed, huber):
    """Same iteration count, termination, and poses / inverse depths within 1e-4 relative (north_star tolerance;
    observed agreement is ~1e-9) of ceres::Solve(SPARSE_SCHUR, LM, <=5 it, Huber)."""
    pb = synth.make_ba_problem(nkf, nlm, k, seed=seed)
    ok_a, pa, da, sa, ca = ref_results.get(f"solve/{nkf}/{nlm}/{k}/{seed}/{huber}", lambda: solve_with(ref_results.lib, "ref", pb, huber=huber),
                                           sample=(2,))
    ok_b, pb_, db, sb, cb = solve_with(oracle, "orc", pb, huber=huber)
    m = ~np.isnan(da)                                     # inverse depths: all of them, or the recorded sample
    assert ok_a == ok_b == 1
    assert sa[3] == sb[3] and sa[2] == sb[2] and sa[4] == sb[4], (sa, sb)
    assert np.allclose(sa[:2], sb[:2], rtol=1e-9)
    n = int(sa[3])
    assert np.allclose(ca[:n], cb[:n], rtol=1e-9)
    assert sb[1] < 0.9 * sb[0]                            # it actually optimised something
    assert np.allclose(pa, pb_, rtol=1e-4, atol=1e-9) and np.allclose(da[m], db[m], rtol=1e-4, atol=1e-9)
    assert np.abs(pa - pb_).max() < 1e-8 and np.abs(da[m] - db[m]).max() < 1e-7


def test_solve_golden(oracle):
    g = golden("ba")
    pb = {k: np.ascontiguousarray(g[k]) for k in ("calib", "poses", "pose_const", "invd", "anch_kf", "anch_uv", "obs_kf",
                                                   "obs_lm", "obs_uv")}
    pb["huber"] = float(g["huber"])
    ok, poses, invd, summary, costs = solve_with(oracle, "orc", pb)
    assert ok == 1
    assert (summary[2:5] == g["summary"][2:5]).all()
    assert np.allclose(summary[:2], g["summary"][:2], rtol=1e-9)
    assert np.allclose(poses, g["poses_out"], rtol=1e-4, atol=1e-9)
    assert np.allclose(invd, g["invd_out"], rtol=1e-4, atol=1e-9)


def local_with(L, prefix, pb, max_iter=5, thr=5.9915):
    poses, invd = pb["poses"].copy(), pb["invd"].copy()
    summary, flags = np.zeros(10), np.zeros(len(pb["obs_kf"]), np.int32)
    fn = getattr(L, prefix + "_ba_local")
    fn.restype = C.c_int
    nbad = fn(P(pb["calib"]), P(poses), P(pb["pose_const"]), len(poses), P(invd), P(pb["anch_kf"]), P(pb["anch_uv"]), len(invd),
              P(pb["obs_kf"]), P(pb["obs_lm"]), P(pb["obs_uv"]), len(pb["obs_kf"]), C.c_double(pb["huber"]), C.c_double(thr),
              max_iter, P(flags), P(summary))
    return nbad, poses, invd, flags, summary


@pytest.mark.parametrize("nkf,nlm,k,seed", [(20, 3000, 4, 42), (8, 300, 3, 7), (12, 800, 5, 3), (10, 400, 3, 11)])
def test_local_ba_vs_ceres(oracle, ref_results, nkf, nlm, k, seed):
    """Optimizer::localBA steps 2-4 (solve, drop chi2 / negative-depth outliers at the functors' last evaluation,
    conditional second solve, second flagging): identical outlier sets and iteration counts, solution to 1e-12."""
    pb = synth.make_ba_problem(nkf, nlm, k, seed=seed)
    ra, pa, da, fa, sa = ref_results.get(f"local/{nkf}/{nlm}/{k}/{seed}", lambda: local_with(ref_results.lib, "ref", pb), sample=(2,))
    rb, pb_, db, fb, sb = local_with(oracle, "orc", pb)
    m = ~np.isnan(da)                                     # inverse depths: all of them, or the recorded sample
    assert ra == rb and ra > 0 and (fa == fb).all()
    assert (sa[[2, 3, 4, 7, 8, 9]] == sb[[2, 3, 4, 7, 8, 9]]).all()
    assert np.allclose(sa, sb, rtol=1e-9)
    assert np.abs(pa - pb_).max() < 1e-11 and np.abs(da[m] - db[m]).max() < 1e-11


def test_local_ba_no_outliers_skips_second_solve(oracle, ref_results):
    """Without outliers the refinement must not run (optimizer.cpp:305): result == plain first solve."""
    pb = synth.make_ba_problem(8, 300, 3, seed=7, outlier_frac=0.0, noise_px=0.2)
    nb, p1, d1, f1, s1 = local_with(oracle, "orc", pb, thr=1e9)
    ok, p0, d0, s0, _ = solve_with(oracle, "orc", pb)
    assert nb == 0 and (f1 == 0).all() and (s1[5:] == 0).all()
    assert (p1 == p0).all() and (d1 == d0).all()
    nr, pr, dr, fr, sr = ref_results.get("local_no_outliers", lambda: local_with(ref_results.lib, "ref", pb, thr=1e9))
    assert nr == 0 and np.abs(pr - p1).max() < 1e-11


def test_local_ba_golden_ceres(oracle):
    g = golden("ba_local")
    pb = {k: np.ascontiguousarray(g[k]) for k in ("calib", "poses", "pose_const", "invd", "anch_kf", "anch_uv", "obs_kf",
                                                   "obs_lm", "obs_uv")}
    pb["huber"] = float(g["huber"])
    nb, p, d, f, s = local_with(oracle, "orc", pb)
    assert (f == g["flags"]).all() and nb == (g["flags"] == 1).sum() and (g["flags"] == 2).sum() >= 1
    assert (s[[2, 3, 4, 7, 8, 9]] == g["summary"][[2, 3, 4, 7, 8, 9]]).all()
    assert np.abs(p - g["poses_out"]).max() < 1e-11 and np.abs(d - g["invd_out"]).max() < 1e-11
