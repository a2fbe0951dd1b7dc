"""CPU tests of the host-side System state machine (alvaar_b200/csrc/system_core.h) -- the code that, in the product, drives
the CUDA kernels -- instantiated over the CPU oracle backend (test infrastructure) and compared with a 100-frame trace of the
reference's own System (tests/golden/system.npz, dumped by tools/make_golden_system.py: initialisation at frame 13, eight keyframes,
the first local BA at frame 27).

What is exact over all 100 frames: status codes, track ids IN THE REFERENCE'S ITERATION ORDER (it decides RANSAC sample indices
and Ceres residual order), 3-D flags, keyframe events, frame / map counters -- and, before the initialisation, every pixel
position bit for bit.
What is toleranced: after the initialisation, poses / world points carry the reference's own noise-limited 5-point refinement
(tests/test_oracle_init.py: a 1-ulp input change moves ITS result by 1e-6 .. 1e-3).  The bar is data-driven (system_util.
pose_deviation): 1e-4 relative (north_star), or 4 x the reference's OWN spread on this trace under a 1-ulp change of one intrinsic
(stored in the golden) where that spread is larger; the worst observed deviation is printed.
With the reference's OWN initialisation stage plugged in (live, or its recorded results) everything downstream -- KLT with projected
priors, P3P-LMedS, PnP, keyframe decisions, triangulation, local-map matching, local BA, culling -- is in lockstep: poses and
world points 1e-9, pixel positions bit-identical, over the whole trace (tools/compare_system_cpu.py shows the same over 140
frames / 11 keyframes / 9 local BAs)."""
import ctypes as C

import numpy as np

from conftest import P, digest
from system_util import (CAP, PoseReport, ReferenceEssential, cpu_system_lib, frame_slice, frames_and_golden, quat_dist,
                         reference_system_trace)


def run(S, frames, K, hook=None):
    w, h = frames.shape[2], frames.shape[1]
    s = S.cpu_system_create(w, h, K[0], K[1], K[2], K[3])
    if hook is not None:
        S.cpu_system_set_essential_hook(s, hook)
    out = []
    for k in range(len(frames)):
        T = np.zeros(7)
        st = S.cpu_system_process(s, P(np.ascontiguousarray(frames[k])), k * 33.333, P(T))
        ids = np.zeros(CAP, np.int32); px = np.zeros((CAP, 2), np.float32); d3 = np.zeros(CAP, np.uint8); wp = np.zeros((CAP, 3)); info = np.zeros(8, np.int32)
        n = S.cpu_system_keypoints(s, P(ids), P(px), P(d3), P(wp), CAP)
        S.cpu_system_info(s, P(info))
        out.append((st, T, info, ids[:n].copy(), px[:n].copy(), d3[:n].copy(), wp[:n].copy()))
    S.cpu_system_destroy(s)
    return out


def test_state_machine_follows_the_reference(oracle):
    g, frames = frames_and_golden()
    tr = run(cpu_system_lib(), frames, g["K"])
    fb = int(g["first_ba_frame"])
    init = int(np.argmax(g["ref_status"] == 1))
    assert 10 <= init < fb < len(frames)
    rep = PoseReport("state machine over the CPU oracle vs the reference System, free-running")
    for k, (st, T, info, ids, px, d3, wp) in enumerate(tr):
        rids, rpx, rd3, rwp = frame_slice(g, "ref_", k)
        assert st == g["ref_status"][k], k
        assert (info == g["ref_info"][k]).all(), (k, info, g["ref_info"][k])
        assert (ids == rids).all() and (d3 == rd3).all(), k                 # ids in the reference's iteration order, 3-D flags
        if k < init:
            assert (px.view(np.uint32) == rpx.view(np.uint32)).all()        # bit-identical tracks before the initialisation
            assert (T == g["ref_Twc"][k]).all()
        else:
            assert np.abs(px - rpx).max() < 0.02
            rep.check(g, k, T)                                               # 1e-4, or SPREAD_K x the reference's own 1-ulp spread where that is larger
        # the committed cpu_* trace (what the GPU build is compared with) is this very run
        cids, cpx, cd3, cwp = frame_slice(g, "cpu_", k)
        assert (ids == cids).all() and (px.view(np.uint32) == cpx.view(np.uint32)).all() and np.abs(T - g["cpu_Twc"][k]).max() < 1e-12
    rep.summary(g)


def test_lockstep_given_the_reference_initialisation(oracle, ref_results):
    g, frames = frames_and_golden()
    hook = ReferenceEssential(ref_results, "lockstep/essential")
    tr = run(cpu_system_lib(), frames, g["K"], hook.ptr)
    hook.finish()
    assert int(g["first_ba_frame"]) < len(frames) - 5                        # the trace does contain a local BA
    for k in range(len(frames)):
        st, T, info, ids, px, d3, wp = tr[k]
        rids, rpx, rd3, rwp = frame_slice(g, "ref_", k)
        assert st == g["ref_status"][k] and (ids == rids).all() and (d3 == rd3).all()
        assert (px.view(np.uint32) == rpx.view(np.uint32)).all()
        assert np.abs(T - g["ref_Twc"][k]).max() < 1e-9
        assert np.abs(wp - rwp).max() < 1e-9 * max(1.0, np.abs(rwp).max())


def test_reset_when_tracks_are_lost(oracle):
    """visual_frontend.cpp:54-58: fewer than 50 tracked keypoints before initialisation -> reset, status 2, a fresh first frame"""
    from alvaar_b200 import synth
    w, h = 640, 480
    frames, _ = synth.make_frames(1, w, h, seed=3, rgba=True)
    other = synth.random_rgba(w, h, 1, seed=5)[0]
    K = synth.intrinsics(w, h)
    S = cpu_system_lib()
    s = S.cpu_system_create(w, h, K[0], K[1], K[2], K[3])
    T = np.zeros(7)
    assert S.cpu_system_process(s, P(np.ascontiguousarray(frames[0])), 0.0, P(T)) == 3
    assert S.cpu_system_process(s, P(np.ascontiguousarray(other)), 33.3, P(T)) == 2
    info = np.zeros(8, np.int32)
    S.cpu_system_info(s, P(info))
    assert info[0] == -1 and info[2] == 0 and info[5] == 0
    assert S.cpu_system_process(s, P(np.ascontiguousarray(frames[0])), 66.6, P(T)) == 3
    S.cpu_system_info(s, P(info))
    assert info[0] == 0 and info[2] > 100 and info[5] == 1
    S.cpu_system_destroy(s)


def lockstep_with_reference_system(ref_results, key, seq, K, pose_tol, wpt_tol=None):
    """The state machine over the CPU oracle, the reference's own initialisation stage plugged in, frame by frame against the
    reference's own System: every discrete quantity equal, pixel positions bit-identical, poses (and world points) to the
    given bars.  Returns the reference's trace."""
    h, w = seq[0].shape[:2]
    want = reference_system_trace(ref_results, key + "/system", seq, K, world_points=wpt_tol is not None)
    S = cpu_system_lib()
    s = S.cpu_system_create(w, h, K[0], K[1], K[2], K[3])
    hook = ReferenceEssential(ref_results, key + "/essential")
    S.cpu_system_set_essential_hook(s, hook.ptr)
    for k, f in enumerate(seq):
        T_s = np.zeros(7)
        st_s = S.cpu_system_process(s, P(np.ascontiguousarray(f)), k * 33.333, P(T_s))
        ids_s = np.zeros(CAP, np.int32); px_s = np.zeros((CAP, 2), np.float32); d3_s = np.zeros(CAP, np.uint8); w_s = np.zeros((CAP, 3))
        n_s = S.cpu_system_keypoints(s, P(ids_s), P(px_s), P(d3_s), P(w_s), CAP)
        i_s = np.zeros(8, np.int32)
        S.cpu_system_info(s, P(i_s))
        st_r, i_r, T_r, ids_r, d3_r, px_r, w_r = want[k]
        n_r = len(ids_r)
        assert st_r == st_s and n_r == n_s and (i_r == i_s).all(), (k, st_r, st_s, i_r, i_s)
        assert (ids_r == ids_s[:n_s]).all() and (d3_r == d3_s[:n_s]).all(), k
        assert (digest(px_s[:n_s]) == px_r).all(), k                       # bit-identical pixel positions
        assert np.abs(T_r - T_s).max() < pose_tol, k
        if wpt_tol is not None:
            assert np.abs(w_r - w_s[:n_s]).max() < wpt_tol * max(1.0, np.abs(w_r).max()), k
    S.cpu_system_destroy(s)
    hook.finish()
    return want


def test_failure_paths_in_lockstep_with_the_live_reference(oracle, ref_results):
    """Blackout frame, a jump to an unrelated sequence, a jump back: lost tracks, P3P / PnP outlier removal, failed poses,
    resets (status 2) with a stale motion model, re-initialisations -- against the reference System frame by frame
    (its own initialisation stage plugged in): every discrete quantity equal, poses 1e-6."""
    from alvaar_b200 import synth
    w, h = 640, 480
    K = synth.intrinsics(w, h)
    A, _ = synth.make_frames(40, w, h, seed=7, rgba=True)
    B, _ = synth.make_frames(26, w, h, seed=33, rgba=True)
    black = np.zeros_like(A[0]); black[..., 3] = 255
    seq = [A[k] for k in range(24)] + [black] + [B[k] for k in range(26)] + [A[k] for k in range(20, 40)]
    want = lockstep_with_reference_system(ref_results, "failure_paths", seq, K, 1e-6)
    assert {f[0] for f in want} == {1, 2, 3}                              # the sequence did exercise resets and re-initialisation


def test_lockstep_at_720p_with_the_live_reference(oracle, ref_results):
    """BASELINE's frame size (1280x720, 784 keypoints / frame): 36 frames through initialisation (frame 12), two more keyframes
    and the first local BA against the reference System, its own initialisation stage plugged in: lockstep as at 640x480."""
    from alvaar_b200 import synth
    w, h, nf = 1280, 720, 36
    K = synth.intrinsics(w, h)
    frames, _ = synth.make_frames(nf, w, h, seed=7, rgba=True)
    last = lockstep_with_reference_system(ref_results, "720p", [frames[k] for k in range(nf)], K, 1e-9, 1e-9)[-1][1]
    assert last[4] == 1 and last[1] >= 2 and last[2] > 500          # initialised, at least keyframe 2 (a local BA ran), 720p-sized


def test_find_plane_on_the_planar_scene(oracle):
    """System::findPlane as intended (system_core.h lists the defects of the reference's own processPlane, which make it
    unpinnable): 0 before the initialisation; afterwards the synthetic scene -- a textured plane facing the first camera -- is
    found: unit rotation whose first column (the image of `up` = (1, 0, 0) under R1) is the plane normal ~ +-z, origin at the
    inliers' centroid, normal pointing away from the camera; repeatable call to call."""
    g, frames = frames_and_golden()
    S = cpu_system_lib()
    S.cpu_system_find_plane.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    K = g["K"]
    s = S.cpu_system_create(frames.shape[2], frames.shape[1], K[0], K[1], K[2], K[3])
    out = np.zeros(16, np.float32)
    T = np.zeros(7)
    for k in range(40):
        S.cpu_system_process(s, P(np.ascontiguousarray(frames[k])), k * 33.333, P(T))
        if k == 5:
            assert S.cpu_system_find_plane(s, P(out), 250) == 0          # fewer than 32 map points: no plane
    assert S.cpu_system_find_plane(s, P(out), 250) == 1
    M = out.reshape(4, 4).T                                              # Utils::toPoseArray(Mat) writes column-major
    R, t = M[:3, :3].astype(np.float64), M[:3, 3]
    assert np.abs(R.T @ R - np.eye(3)).max() < 1e-5 and abs(np.linalg.det(R) - 1) < 1e-5 and M[3, 3] == 1
    n = R[:, 0]
    assert abs(n[2]) > 0.999                                             # the plane z = const of the first camera
    ids = np.zeros(CAP, np.int32); px = np.zeros((CAP, 2), np.float32); d3 = np.zeros(CAP, np.uint8); wp = np.zeros((CAP, 3))
    m = S.cpu_system_keypoints(s, P(ids), P(px), P(d3), P(wp), CAP)
    pts = wp[:m][d3[:m] == 1]
    assert np.abs(t - pts.mean(0)).max() < 0.5 and np.abs((pts - t) @ n).mean() < 0.2   # on the plane of the map points
    cam = T[:3]
    assert (cam - t) @ n < 0                                             # turned away from the camera
    S.cpu_system_destroy(s)
