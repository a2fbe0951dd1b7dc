#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200-native per-frame visual-SLAM hot path.

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA, sm_100a)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU code on the host cores

Metric (BASELINE.json): frames/sec @1280x720, 1000 ORB features/frame, 20-keyframe local BA; plus the achieved HBM
bandwidth of the fused pyramid+FAST kernel against the measured copy peak (MEASURED_PEAKS.json).

One "step" = one pass of the whole hot path over a batch of BATCH synthetic frames:
  RGBA -> gray + 4-level Gaussian pyramid + FAST-9/NMS (level 0) -> retainBest(1000) -> ORB (7x7 blur, IC angle,
  rBRIEF-256) -> brute-force Hamming 2-NN against a 10 000-descriptor local map -> one local BA
  (20 KF x 3000 landmarks x 12 000 observations, LM <= 5 it, Huber, Schur) per KF_INTERVAL frames.
`value`  : inputs already resident in HBM when the timed region starts (CUDA events, max over ranks).
`e2e`    : the same step through the host-buffer C-ABI call (alva_pipeline_step_host): pinned host RGBA in,
           per-frame feature counts + matches + BA poses back out, copies inside the timed region.
Multi-GPU: independent camera streams shard one-per-GPU (weak scaling, no data-path collective).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# workloads (BASELINE.json configs): c2 = the headline (1280x720, 1000 features; `metric` is quoted on it), c3 = 1920x1080 with
# 2000 features through the same pipeline.  --config selects; the module constants below are the selected workload's.
CONFIGS = {"c2": dict(w=1280, h=720, nfeat=1000, batch=64, name="c2_720p_stream+c4_local_ba"),
           "c3": dict(w=1920, h=1080, nfeat=2000, batch=32, name="c3_1080p_stream+c4_local_ba")}
W, H = 1280, 720
BATCH = 64            # frames per step: 64 x 3.69 MB RGBA = 236 MB per step, larger than the 126 MB L2
NFEAT = 1000
WORKLOAD = "c2_720p_stream+c4_local_ba"
MAP_SIZE = 10000
KF_INTERVAL = 5
BA_NKF, BA_NLM, BA_OBS_PER_LM, BA_ITERS = 20, 3000, 4, 5
FAST_THR = 20
# algorithmic bytes of the fused front-end kernel per frame (SURVEY 8d): RGBA read once + gray + L1 written once
ALGO_BYTES_FRONTEND = 4 * W * H + W * H + ((W + 1) // 2) * ((H + 1) // 2)


METRIC = {"c2": "frames_per_sec_720p_1000orb_20kf_ba", "c3": "frames_per_sec_1080p_2000orb_20kf_ba"}


def select_config(name):
    global W, H, BATCH, NFEAT, WORKLOAD, ALGO_BYTES_FRONTEND
    c = CONFIGS[name]
    W, H, BATCH, NFEAT, WORKLOAD = c["w"], c["h"], c["batch"], c["nfeat"], c["name"]
    ALGO_BYTES_FRONTEND = 4 * W * H + W * H + ((W + 1) // 2) * ((H + 1) // 2)
# dram__bytes_read.sum + dram__bytes_write.sum of one 64-frame front-end launch, from the committed `ncu --set full`
# capture (profiles/r02_frontend_v2_full.txt).  Static by nature: a profiler cannot run inside bench.
FRONTEND_DRAM_TRAFFIC_BYTES_B64 = 294_047_488   # dram__bytes_read.sum 235.976 MB + dram__bytes_write.sum 58.072 MB


# sha256[:16] of the step's integer outputs (selected-feature counts + 2-NN match lists of all 64 frames) for the stream seeds
# 99 + rank, rank 0..7: every run checks its own outputs against these (bit-exact stages: any change of a kernel's results, a
# race, or a skipped stage shows here, inside the timed configuration).  Printed by `bench.py --print-checksums`.
EXPECTED_OUTPUT_SHA = {99: "204d42bd422277ed", 100: "e04ea0ed49e3f800", 101: "acde5d4ba6701be4", 102: "f54044662430e0e4",
                       103: "31071a9894265b65", 104: "75e995f22e29f387", 105: "d98331275913f47e", 106: "0e082756b2905b60"}


def stream_frames(rank):
    """Synthetic camera stream of a rank: its own path (seed 99 + rank) over a scene it shares with ONE other stream (ranks 2k and
    2k + 1 watch the same plane, other pairs other planes) -- so that at any N every stream has exactly one remote stream to close
    loops with, and the cross-stream detector's work per rank does not grow with N."""
    from alvaar_b200 import synth
    return synth.make_frames(BATCH, W, H, seed=99 + rank, texture_seed=1234 + rank // 2)[0]


def output_checksum(nfeat, matches):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(nfeat).tobytes() + np.ascontiguousarray(matches).tobytes()).hexdigest()[:16]


def gpu_local_cpus(index):
    """CPUs of the NUMA node the GPU hangs off (sysfs local_cpulist of its PCI function), or None"""
    try:
        import pynvml as nv
        nv.nvmlInit()
        bus = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(":", 1)
        path = f"/sys/bus/pci/devices/{int(dom, 16):04x}:{rest.lower()}/local_cpulist"
        cpus = []
        for part in open(path).read().strip().split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus += list(range(int(a), int(b) + 1))
            elif part:
                cpus.append(int(part))
        return cpus or None
    except Exception:
        return None


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.maxclk = index, [], set(), False, None

    def run(self):
        try:
            self._run_nvml()
        except Exception:
            self._run_smi()

    def _run_nvml(self):
        """NVML directly (a query is ~0.1 ms, so even a 40 ms timed region gets several samples)."""
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        self.maxclk = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        bits = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4}
        while not self.stop_flag:
            self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            for n, b in bits.items():
                if r & b:
                    self.reasons.add(n)
            time.sleep(0.004)

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.maxclk = float(out[1])
                for n, v in zip(names, out[2:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.maxclk,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ reference arm
def load_cpu_impl():
    """oracle/_ref (the reference's own vendored OpenCV 4.5.5 + Ceres 2.0 build) if it travelled here, else the
    plain-C port.  Returns (lib, kind)."""
    ref = os.path.join(ROOT, "oracle", "_ref", "libalva_ref.so")
    if os.path.exists(ref):
        try:
            return C.CDLL(ref), "reference"
        except OSError:
            pass
    so = os.path.join(ROOT, "oracle", "_build", "libalva_oracle.so")
    if not os.path.exists(so):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
    return C.CDLL(so), "port"


def cpu_pipeline_frames(L, kind, frames_rgba, map_desc, ba, nthreads):
    """The reference's CPU path for the same step on `frames_rgba` ([n, H, W, 4]); returns seconds.
    reference kind: cv::cvtColor + buildOpticalFlowPyramid(win 9, 3 levels) + ORB::detectAndCompute(1000, 1 level:
    FAST + Harris + retainBest + IC angle + blur + rBRIEF) + BFMatcher.knnMatch(k=2) with cv::setNumThreads(nthreads),
    and ceres::Solve once per KF_INTERVAL frames (single-threaded, as the product is)."""
    P = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    n = len(frames_rgba)
    gray = np.empty((H, W), np.uint8)
    t0 = time.perf_counter()
    if kind == "reference":
        L.ref_config(1, nthreads)
        lv = [np.empty((H, W), np.uint8), np.empty(((H + 1) // 2, (W + 1) // 2), np.uint8)]
        lv.append(np.empty(((lv[1].shape[0] + 1) // 2, (lv[1].shape[1] + 1) // 2), np.uint8))
        lv.append(np.empty(((lv[2].shape[0] + 1) // 2, (lv[2].shape[1] + 1) // 2), np.uint8))
        ptrs = (C.c_void_p * 4)(*[a.ctypes.data for a in lv])
        kp = np.empty((4096, 5), np.float32)
        desc = np.empty((4096, 32), np.uint8)
        out = np.empty((4096, 4), np.int32)
        for f in range(n):
            L.ref_gray(P(frames_rgba[f]), W, H, P(gray))
            L.ref_build_pyramid(P(gray), W, H, 9, 3, ptrs, None)
            nd = L.ref_orb_detect(P(gray), W, H, NFEAT, FAST_THR, P(kp), P(desc), 4096)
            L.ref_knn2(P(desc), min(nd, 4096), P(map_desc), len(map_desc), P(out))
            if f % KF_INTERVAL == 0:
                run_cpu_ba(L, "ref", ba)
    else:
        xs = np.empty((W * H // 4, 3), np.int32)
        blur = np.empty((H, W), np.uint8)
        for f in range(n):
            L.orc_gray(P(frames_rgba[f]), W, H, P(gray))
            cur, cw, ch = gray, W, H
            for _ in range(3):
                nxt = np.empty(((ch + 1) // 2, (cw + 1) // 2), np.uint8)
                L.orc_pyrdown(P(cur), cw, ch, P(nxt))
                cur, cw, ch = nxt, nxt.shape[1], nxt.shape[0]
            nk = L.orc_fast9(P(gray), W, H, FAST_THR, 1, P(xs), len(xs))
            k = xs[:nk]
            k = k[(k[:, 0] >= 31) & (k[:, 0] < W - 31) & (k[:, 1] >= 31) & (k[:, 1] < H - 31)]
            thr = L.orc_retain_best_threshold(P(np.ascontiguousarray(k)), len(k), NFEAT)
            k = k[k[:, 2] >= thr]
            pts = np.ascontiguousarray(k[:, :2].astype(np.float32))
            ang = np.empty(len(pts), np.float32)
            L.orc_ic_angles(P(gray), W, H, P(pts), len(pts), P(ang))
            L.orc_orb_blur(P(gray), W, H, 0, P(blur))
            desc = np.empty((len(pts), 32), np.uint8)
            kept = np.empty(len(pts), np.uint8)
            L.orc_orb_describe(P(blur), W, H, P(pts), P(ang), len(pts), P(desc), P(kept))
            out = np.empty((len(pts), 4), np.int32)
            L.orc_knn2(P(desc), len(pts), P(map_desc), len(map_desc), P(out))
            if f % KF_INTERVAL == 0:
                run_cpu_ba(L, "orc", ba)
    return time.perf_counter() - t0


def run_cpu_ba(L, prefix, pb):
    P = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    poses, invd = pb["poses"].copy(), pb["invd"].copy()
    summary = np.zeros(8)
    getattr(L, prefix + "_ba_solve")(P(pb["calib"]), P(poses), P(pb["pose_const"]), len(poses), P(invd), P(pb["anch_kf"]),
                                    P(pb["anch_uv"]), len(invd), P(pb["obs_kf"]), P(pb["obs_lm"]), P(pb["obs_uv"]),
                                    len(pb["obs_kf"]), C.c_double(pb["huber"]), BA_ITERS, P(summary), None)


REF_SAMPLE = 8   # frames per CPU step: a bounded sample of the 64-frame step (the CPU needs ~0.2 s for it on 128 cores)


def local_cpus():
    try:
        return sorted(os.sched_getaffinity(0))
    except AttributeError:
        return list(range(os.cpu_count() or 1))


def reference_worker(args):
    """one independent reference stream on the cores in args.cores (comma list): prints {"frames": n, "seconds": t}"""
    from alvaar_b200 import synth
    cores = [int(c) for c in args.cores.split(",")]
    try:
        os.sched_setaffinity(0, cores)
    except Exception:
        pass
    L, kind = load_cpu_impl()
    sample = REF_SAMPLE if kind == "reference" else 2
    frames = synth.make_frames(sample, W, H, seed=99 + args.stream, texture_seed=1234 + args.stream // 2)[0]
    _, map_desc = synth.make_descriptors(8, MAP_SIZE, seed=7)
    ba = synth.make_ba_problem(BA_NKF, BA_NLM, BA_OBS_PER_LM, seed=42)
    for _ in range(max(1, min(args.warmup, 2))):
        cpu_pipeline_frames(L, kind, frames[:2], map_desc, ba, len(cores))
    t = sum(cpu_pipeline_frames(L, kind, frames, map_desc, ba, len(cores)) for _ in range(args.steps))
    print(json.dumps({"frames": sample * args.steps, "seconds": t, "kind": kind, "cores": len(cores) if kind == "reference" else 1, "sample": sample}))


def bench_reference(args, rank, world):
    """The reference's own CPU implementation of the step on the host cores.  N = 1: one stream on all cores.  N > 1 (rank 0
    only): N independent streams, one process each, pinned to N disjoint core sets (BASELINE.md row S8: one System per core
    set) -- the CPU counterpart of N streams on N GPUs; the aggregate is reported."""
    if rank != 0:
        return
    cpus = local_cpus()
    nstream = max(1, args.gpus)
    per = max(1, len(cpus) // nstream)
    steps = max(1, args.steps)
    procs = []
    for i in range(nstream):
        cs = cpus[i * per:(i + 1) * per] if i < nstream - 1 or nstream == 1 else cpus[i * per:]
        if nstream == 1:
            cs = cpus
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference-worker", "--cores", ",".join(map(str, cs)), "--stream", str(i),
               "--steps", str(steps), "--warmup", str(args.warmup), "--config", args.config]
        procs.append(subprocess.Popen(cmd, stdout=subprocess.PIPE, text=True))
    res = []
    for pr in procs:
        out, _ = pr.communicate()
        res.append(json.loads(out.strip().splitlines()[-1]))
    # streams run side by side: the aggregate rate is the sum of the per-stream rates
    fps = sum(r["frames"] / r["seconds"] for r in res)
    t_step = max(r["seconds"] for r in res) / steps
    kind, sample = res[0]["kind"], res[0]["sample"]
    cores_used = sum(r["cores"] for r in res)
    line = {"impl": "reference", "metric": METRIC[args.config], "value": fps, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/f64", "data": "synthetic",
            "config": workload_config(BATCH, nstream, nstream > 1 and not args.no_loop_closure),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores_used, "kind": kind,
                             "sample": f"{nstream} stream(s) x {steps} steps x {sample} frames of the {BATCH}-frame 720p step (each incl. "
                                       f"{(sample + KF_INTERVAL - 1) // KF_INTERVAL} local BA solves); per stream: OpenCV stages on its "
                                       f"{per if nstream > 1 else len(cpus)} cores (cv::setNumThreads), Ceres single-threaded as shipped"},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config(batch, world=1, loop_closure=False):
    cfg = _workload_config(batch)
    cfg["parallelism"] = f"{world} independent camera-stream batch(es), one per GPU" + (
        "; NCCL all-gather of the step's keyframe blocks + cross-stream loop-closure detection on a side stream" if loop_closure else "")
    return cfg


BA_SCHEDULE = ["own high-priority stream, forked at the start of the step and joined at its end"]


def _workload_config(batch):
    return {"workload": WORKLOAD, "frame": f"{W}x{H} RGBA", "batch_frames_per_step": batch,
            "pyramid": "4 levels + Scharr derivative levels (buildOpticalFlowPyramid withDerivatives, as the reference)",
            "features_per_frame": NFEAT, "fast_threshold": FAST_THR, "orb": "ORB::detectAndCompute semantics, 1 level: FAST-9 -> retainBest(2n) -> Harris -> retainBest(n) -> IC angle -> 7x7 blur -> rBRIEF-256",
            "map_descriptors": MAP_SIZE, "ba": f"{BA_NKF} KF x {BA_NLM} landmarks x {BA_NLM * BA_OBS_PER_LM} obs, LM<={BA_ITERS}",
            "ba_every_n_frames": KF_INTERVAL,
            "ba_schedule": BA_SCHEDULE[0],
            "l2_policy": f"inputs ({4 * W * H * batch / 1e6:.0f} MB/step) larger than L2 (126 MB)",
            "parallelism": "1 stream batch per GPU"}


# ------------------------------------------------------------------------------------------------ our arm
def bench_b200(args, rank, world, local_rank):
    import torch
    import alvaar_b200
    from alvaar_b200 import synth
    from alvaar_b200.pipeline import Pipeline

    torch.cuda.set_device(local_rank)
    # page-locked buffers are first-touched by this process: run it on the CPUs of the GPU's own NUMA node while they are
    # allocated and while the copies are issued, so that the e2e leg does not depend on where the scheduler put the process
    all_cpus = local_cpus()
    numa = gpu_local_cpus(local_rank)
    if numa:
        try:
            os.sched_setaffinity(0, [c for c in numa if c in all_cpus] or all_cpus)
        except Exception:
            numa = None
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's banner ("NCCL version ...") must not share stdout with the JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    frames = stream_frames(rank)
    _, map_desc = synth.make_descriptors(8, MAP_SIZE, seed=7)
    ba = synth.make_ba_problem(BA_NKF, BA_NLM, BA_OBS_PER_LM, seed=42)
    stream = torch.cuda.Stream()
    ctx = alvaar_b200.Context(local_rank, stream.cuda_stream)
    ctx.L.alva_set_option(b"pipeline_ba_overlap", 0 if args.no_ba_overlap else 1)
    lag = args.ba_lag and not args.no_ba_overlap
    ctx.L.alva_set_option(b"pipeline_ba_lag", 1 if lag else 0)
    if args.no_ba_overlap:
        BA_SCHEDULE[0] = "after the frame stages, same stream (A/B measurement)"
    elif lag:
        BA_SCHEDULE[0] = ("own high-priority streams; the chain of step s is joined at the end of step s+1 (two chains in flight, results "
                          "delivered one step later as the reference's mapper thread does); the timed region starts drained and ends with "
                          "alva_pipeline_drain, so it holds exactly K frame batches and K x 13 BA solves")
    ctx.L.alva_set_option(b"pipeline_graphs", 0 if args.no_graphs else 1)
    if args.frontend_ctas:
        assert ctx.L.alva_set_option(b"frontend_ctas", args.frontend_ctas) == 0
    if args.ba_ctl_threads:
        assert ctx.L.alva_set_option(b"ba_ctl_threads", args.ba_ctl_threads) == 0
    pipe = Pipeline(ctx, W, H, BATCH, fast_thr=FAST_THR, nfeatures=NFEAT, orb_flags=alvaar_b200.ORB_IC_ANGLE | alvaar_b200.ORB_HARRIS,
                    map_size=MAP_SIZE, kf_interval=KF_INTERVAL, ba_nkf=BA_NKF, ba_nlm=BA_NLM, ba_nobs=len(ba["obs_kf"]),
                    ba_max_iter=BA_ITERS, ba_huber=ba["huber"], derivatives=True)
    pipe.set_map(map_desc)
    for s in range(pipe.nprob):
        pipe.set_ba(s, ba)
    host_in = torch.from_numpy(frames).pin_memory()
    d_in = host_in.to(f"cuda:{local_rank}")
    nfeat_host = torch.zeros(BATCH, dtype=torch.int32).pin_memory()
    matches_host = torch.zeros((BATCH, pipe.fcap, 4), dtype=torch.int32).pin_memory()
    poses_host = torch.zeros((max(pipe.nprob, 1), BA_NKF, 7), dtype=torch.float64).pin_memory()
    summ_host = torch.zeros((max(pipe.nprob, 1), 8), dtype=torch.float64).pin_memory()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    # Optional cross-stream loop-closure exchange (SURVEY 8e, config C5): every rank contributes the descriptor blocks of
    # this step's keyframes (fixed shape [nprob, fcap, 32] + counts), NCCL all-gathers them over NVLink, and the newest
    # local keyframe is matched (brute-force Hamming 2-NN) against every gathered block.  No reference behaviour to
    # match (the reference is single-stream); validated as "gather == concatenation of the per-rank inputs".
    lc = None
    lc_events, det = [], None
    if dist is not None and not args.no_loop_closure:
        from alvaar_b200.loopclosure import LoopClosure, block_bytes
        dev_s = f"cuda:{local_rank}"
        # One communication stream (the NCCL all-gather of every step, never behind a detection) and ND detectors, each with its own
        # stream and buffers.  A geometric check (one round of the five-point RANSAC) takes 2.8 ms alone and ~6 ms beside the frame
        # stages -- several steps -- so a step's gathered blocks go to a detector only if one is idle; otherwise the step is exchanged
        # but not examined (counted in loop_closure.steps_not_examined).  Skipping is a local decision: the collective runs every step.
        LC_RING, ND = 8, 3
        comm = torch.cuda.Stream()
        sides = [torch.cuda.Stream() for _ in range(ND)]
        lc_ctxs = [alvaar_b200.Context(local_rank, sd.cuda_stream) for sd in sides]
        dets = [LoopClosure(c, pipe.fcap, pipe.nprob, world, rank, synth.intrinsics(W, H), min_matches=max(30, NFEAT // 10)) for c in lc_ctxs]
        det = dets[0]
        for d in dets:
            d.L.alva_lc_inflight.argtypes = [C.c_void_p]
        kf_idx = torch.arange(0, BATCH, KF_INTERVAL, dtype=torch.int32, device=dev_s)[:pipe.nprob].contiguous()
        desc_all = pipe.buffer("desc", (BATCH, pipe.fcap, 32), torch.uint8)
        pts_all = pipe.buffer("pts", (BATCH, pipe.fcap, 2), torch.float32)
        cnt_all = pipe.buffer("selcounts", (BATCH,), torch.int32)
        bb = block_bytes(pipe.fcap)
        send = [torch.zeros(pipe.nprob * bb, dtype=torch.uint8, device=dev_s) for _ in range(LC_RING)]
        gathered_buf = [torch.zeros(world * pipe.nprob * bb, dtype=torch.uint8, device=dev_s) for _ in range(LC_RING)]
        ev_packed = [torch.cuda.Event() for _ in range(LC_RING)]
        ev_gathered = [torch.cuda.Event() for _ in range(LC_RING)]
        ev_examined = [torch.cuda.Event() for _ in range(LC_RING)]
        slot_examined = [False] * LC_RING
        lc_state = {"step": 0, "examined": 0, "skipped": 0}

        def lc():
            # Off the per-frame path.  The step's keyframe blocks are packed on the MAIN stream (microseconds, right behind the
            # kernels that produced the descriptors) into a ring of send buffers; the all-gather runs on the communication stream;
            # the detection (Hamming 2-NN of the live descriptors, ratio test, five-point RANSAC) on an idle detector's stream.  The
            # main stream never waits for a detection: only, LC_RING steps later, for the all-gather that read the ring slot it is
            # about to refill.  Results are polled without blocking.
            st_ = lc_state["step"]
            i = st_ % LC_RING
            for d in dets:
                lc_events.extend(d.poll())
            idle = [j for j in range(ND) if dets[j].L.alva_lc_inflight(dets[j].h) == 0]
            d = dets[idle[0]] if idle else dets[0]
            if st_ >= LC_RING:
                stream.wait_event(ev_gathered[i])
            d.seq = st_ * pipe.nprob          # keyframe sequence numbers run on across the detectors
            d.pack(desc_all, pts_all, cnt_all, kf_idx, send[i], on=ctx)
            ev_packed[i].record(stream)
            with torch.cuda.stream(comm):
                comm.wait_event(ev_packed[i])
                if slot_examined[i]:
                    comm.wait_event(ev_examined[i])   # the detection that read this slot LC_RING steps ago
                    slot_examined[i] = False
                dist.all_gather_into_tensor(gathered_buf[i], send[i])
                ev_gathered[i].record(comm)
            if idle:
                side = sides[idle[0]]
                with torch.cuda.stream(side):
                    side.wait_event(ev_gathered[i])
                    d.detect(gathered_buf[i])
                    ev_examined[i].record(side)
                slot_examined[i] = True
                lc_state["examined"] += 1
            else:
                lc_state["skipped"] += 1
            lc_state["step"] += 1
            return gathered_buf[i]

    sampler = ClockSampler(local_rank)
    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            pipe.step_dev(d_in)
            if lc:
                lc()
        pipe.drain()
        if lc:
            for sd in sides + [comm]:
                stream.wait_stream(sd)
            lc_state["examined"] = lc_state["skipped"] = 0
        barrier()
        l0 = ctx.launches
        sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(args.steps):
            pipe.step_dev(d_in)
            if lc:
                gathered = lc()
        pipe.drain()   # the last step's BA chain belongs to the timed region
        if lc:
            for sd in sides + [comm]:
                stream.wait_stream(sd)   # ... and so do the exchanges + detections still in flight
        ev1.record(stream)
        barrier()
        launches = ctx.launches - l0
        ms = ev0.elapsed_time(ev1)
        graphs = pipe.graph_stats()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, pipe)
        # The dominant kernel's launch duration (roofline.achieved): CUDA events around the fused front-end launch of every
        # step of a SECOND pass of the same K steps, launched kernel by kernel -- the timed pass above replays CUDA graphs,
        # which cannot carry per-launch event pairs.  Same kernel, same inputs, same stream, right after the timed pass.
        pipe.profile(True)
        for _ in range(args.steps):
            pipe.step_dev(d_in)
        pipe.drain()
        barrier()
        fe = pipe.frontend_ms(args.steps)
        pipe.profile(False)
        # e2e: host buffers through the C-ABI call, copies inside the timed region.  The throughput form of the call is used:
        # submit (returns at once) / wait, two submissions in flight, so the upload of one batch overlaps the compute of the
        # previous one -- every step still uploads its own 236 MB from pinned host memory and reads its results back.
        res = [(nfeat_host, matches_host, poses_host, summ_host),
               (torch.zeros_like(nfeat_host).pin_memory(), torch.zeros_like(matches_host).pin_memory(),
                torch.zeros_like(poses_host).pin_memory(), torch.zeros_like(summ_host).pin_memory())]
        for _ in range(min(args.warmup, 2)):
            pipe.step_host(host_in, *res[0])
        pipe.drain()
        barrier()
        e2e_steps = max(2, min(args.steps, 10))
        t0 = time.perf_counter()
        ev0.record(stream)
        for i in range(e2e_steps):
            pipe.submit_host(host_in, *res[i % 2])
            if i >= 1:
                pipe.wait()
        pipe.wait()
        pipe.drain()
        ev1.record(stream)
        barrier()
        e2e_ms = ev0.elapsed_time(ev1)
        _ = time.perf_counter() - t0
        assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])   # both slots deliver the same results
    out_sha = output_checksum(res[0][0].numpy(), res[0][1].numpy())
    want_sha = EXPECTED_OUTPUT_SHA.get(99 + rank) if args.config == "c2" else None
    if want_sha is not None and out_sha != want_sha:
        raise SystemExit(f"bench: the step's outputs changed: sha {out_sha}, expected {want_sha} (stream seed {99 + rank})")
    try:
        os.sched_setaffinity(0, all_cpus)   # the CPU legs below use every host core again
    except Exception:
        pass
    sampler.stop_flag = True
    sampler.join(timeout=2)
    tracking = None
    if rank == 0 and not args.no_stage_stats:
        try:
            tracking = tracking_stage_times(ctx, pipe, stream, local_rank)
        except Exception as e:   # explanatory numbers only: never let them take the headline line down
            tracking = {"error": repr(e)}
        try:
            tracking["system_api"] = system_api_times(not args.no_cpu_baseline)
        except Exception as e:
            tracking["system_api"] = {"error": repr(e)}

    lc_report = None
    if det is not None:
        torch.cuda.synchronize()
        for d in dets:
            lc_events.extend(d.poll(wait=True))
        sc = det.last_scores()
        lc_report = {"keyframe_blocks_per_step": int(world * pipe.nprob), "block_bytes": int(block_bytes(pipe.fcap)),
                     "steps_examined": lc_state["examined"], "steps_not_examined": lc_state["skipped"],
                     "events": len(lc_events), "remote_ranks_with_events": sorted({int(e["remote_rank"]) for e in lc_events}),
                     "last_step_pairs_checked": int((sc[:, :, 0] >= max(30, NFEAT // 10)).sum()),
                     "last_step_pairs_verified": int((sc[:, :, 1] == 1).sum()),
                     "schedule": "pack on the main stream -> ncclAllGather on a communication stream (every step) -> an idle detector (3, own "
                                 "streams): Hamming 2-NN (live descriptors) -> ratio test -> 5-point RANSAC on the newest keyframe; polled; "
                                 "streams 2k and 2k+1 watch the same scene"}
    t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=f"cuda:{local_rank}")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = t.tolist()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    fps = world * BATCH * args.steps / (ms * 1e-3)
    e2e_fps = world * BATCH * e2e_steps / (e2e_ms * 1e-3)
    peak, peak_src = read_peaks()
    fe_avg_ms = float(np.mean(fe))
    achieved = ALGO_BYTES_FRONTEND * BATCH / (fe_avg_ms * 1e-3) / 1e9
    nf = nfeat_host.numpy()
    summ = summ_host.numpy()
    h2d = int(host_in.numel())
    d2h = int(nfeat_host.numel() * 4 + matches_host.numel() * 4 + poses_host.numel() * 8 + summ_host.numel() * 8)

    # CPU baseline on a bounded sample (rank 0, N = 1 only)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        L, kind = load_cpu_impl()
        cores = len(all_cpus)
        sample = REF_SAMPLE if kind == "reference" else 2
        cpu_pipeline_frames(L, kind, frames[:2], map_desc, ba, cores)
        t1 = cpu_pipeline_frames(L, kind, frames[:sample], map_desc, ba, cores)
        passes = int(max(1, min(8, 10.0 / max(t1, 1e-3))))          # about 10 s of CPU work, at most the whole 64-frame step
        tcpu = t1 + sum(cpu_pipeline_frames(L, kind, frames[sample * (i % (BATCH // sample)):sample * (i % (BATCH // sample)) + sample], map_desc, ba, cores)
                        for i in range(1, passes))
        cpu = {"value": sample * passes / tcpu, "unit": "frames/s", "cores": cores if kind == "reference" else 1, "kind": kind,
               "sample": f"{sample * passes} frames of the same 720p step (incl. {passes * ((sample + KF_INTERVAL - 1) // KF_INTERVAL)} local BA solves), "
                         "OpenCV stages on all host cores, Ceres single-threaded as shipped"}

    line = {"metric": METRIC[args.config], "value": fps, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/f64", "data": "synthetic",
            "config": workload_config(BATCH, world, lc is not None),
            "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "api": "alva_pipeline_submit_host + alva_pipeline_wait, two batches in flight (pinned host RGBA in, counts+matches+BA poses out per step)"},
            "gpu_launches": int(launches),
            "loop_closure": lc_report,
            "cuda_graphs": {"captured": graphs[0], "graph_launches": graphs[1], "capture_failed": graphs[2],
                            "note": "gpu_launches counts the kernels inside the replayed graphs"},
            "output_sha": out_sha, "output_check": "matches the stored checksum" if want_sha else "no stored checksum for this stream seed",
            "host_numa_cpus": (f"{min(numa)}-{max(numa)} ({len(numa)} CPUs local to the GPU)" if numa else None),
            "clocks": sampler.summary(),
            "roofline": {"kernel": "frontend_tile_kernel_v2<RGBA> (gray + pyramid L1 + FAST-9/NMS, fused)", "bound": "hbm",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": FRONTEND_DRAM_TRAFFIC_BYTES_B64 if (BATCH, W, H) == (64, 1280, 720) else None,
                         "traffic_source": "ncu --set full of frontend_tile_kernel_v2, profiles/r02_frontend_v2_full.txt (bytes per launch)",
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": ALGO_BYTES_FRONTEND * BATCH,
                         "launch_ms": fe_avg_ms,
                         "launch_ms_source": f"CUDA events around the launch in each of {len(fe)} steps of a second, kernel-by-kernel pass "
                                             "(the timed pass replays CUDA graphs)"},
            "cpu_baseline": cpu,
            "stats": {"features_per_frame_mean": float(nf.mean()), "features_per_frame_min": int(nf.min()),
                      "ba_final_over_initial_cost": float((summ[:, 1] / np.maximum(summ[:, 0], 1e-300)).mean()),
                      "ba_iterations_mean": float(summ[:, 3].mean()),
                      "tracking_stages_us": tracking}}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(out_dir, pipe):
    """What the last timed step left for its caller -- the arrays alva_pipeline_step_host copies out: selected-feature counts
    per frame, the 2-NN match lists, the local-BA poses and solver summaries -- as out_dir/<name>.npy (float64: exact for the
    int32 arrays).  The inputs are seeded, so two builds run with the same arguments can be compared array by array."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"nfeat": pipe.buffer("selcounts", (BATCH,), torch.int32),
              "matches": pipe.buffer("matches", (BATCH, pipe.fcap, 4), torch.int32),
              "ba_poses": pipe.buffer("ba_poses", (pipe.nprob, BA_NKF, 7), torch.float64),
              "ba_summary": pipe.buffer("ba_summary", (pipe.nprob, 8), torch.float64)}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float64))


def print_checksums():
    """the integer outputs of one step for the stream seeds 99..106, on one GPU: paste the dict into EXPECTED_OUTPUT_SHA"""
    import torch
    import alvaar_b200
    from alvaar_b200 import synth
    from alvaar_b200.pipeline import Pipeline
    _, map_desc = synth.make_descriptors(8, MAP_SIZE, seed=7)
    ba = synth.make_ba_problem(BA_NKF, BA_NLM, BA_OBS_PER_LM, seed=42)
    stream = torch.cuda.Stream()
    ctx = alvaar_b200.Context(0, stream.cuda_stream)
    pipe = Pipeline(ctx, W, H, BATCH, fast_thr=FAST_THR, nfeatures=NFEAT, orb_flags=alvaar_b200.ORB_IC_ANGLE | alvaar_b200.ORB_HARRIS,
                    map_size=MAP_SIZE, kf_interval=KF_INTERVAL, ba_nkf=BA_NKF, ba_nlm=BA_NLM, ba_nobs=len(ba["obs_kf"]),
                    ba_max_iter=BA_ITERS, ba_huber=ba["huber"], derivatives=True)
    pipe.set_map(map_desc)
    for s in range(pipe.nprob):
        pipe.set_ba(s, ba)
    out = {}
    for seed in range(99, 107):
        frames = stream_frames(seed - 99)
        host_in = torch.from_numpy(frames).pin_memory()
        nf = torch.zeros(BATCH, dtype=torch.int32).pin_memory()
        mt = torch.zeros((BATCH, pipe.fcap, 4), dtype=torch.int32).pin_memory()
        with torch.cuda.stream(stream):
            pipe.step_host(host_in, nf, mt, None, None)
        torch.cuda.synchronize()
        out[seed] = output_checksum(nf.numpy(), mt.numpy())
    print("EXPECTED_OUTPUT_SHA =", json.dumps(out).replace('"', ""))


def tracking_stage_times(ctx, pipe, stream, local_rank):
    """The reference's own per-frame association / pose stages (SURVEY 8a rows a6, a17, a18) on the same batch, timed one by
    one with CUDA events AFTER the headline measurement (they are reported, not part of `value`): forward-backward KLT of
    every frame's 1000 selected features into the next frame (63 frame pairs out of the step's pyramids), P3P-LMedS and
    PnP on 64 synthetic 1000-point problems, the grid Shi-Tomasi detector + cornerSubPix on the step's 13 keyframes."""
    import torch
    from alvaar_b200 import synth
    dev = f"cuda:{local_rank}"
    ws, hs = [W], [H]
    for _ in range(3):
        ws.append((ws[-1] + 1) // 2); hs.append((hs[-1] + 1) // 2)
    lv = [pipe.buffer(f"l{k}", (BATCH, hs[k], ws[k]), torch.uint8) for k in range(4)]
    dv = [pipe.buffer(f"d{k}", (BATCH, hs[k], ws[k], 2), torch.int16) for k in range(4)]
    pts = pipe.buffer("pts", (BATCH, pipe.fcap, 2), torch.float32)
    cnt = pipe.buffer("selcounts", (BATCH,), torch.int32)
    nf = BATCH - 1
    good = torch.zeros((nf, pipe.fcap), dtype=torch.uint8, device=dev)

    def timed(fn, reps=5):
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream); fn(); e1.record(stream); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        return float(np.median(ts[1:]))

    out = {}
    with torch.cuda.stream(stream):
        pri = torch.empty((nf, pipe.fcap, 2), dtype=torch.float32, device=dev)

        def klt():
            pri.copy_(pts[:nf])
            ctx.klt_fb([t[:nf] for t in lv], [t[:nf] for t in dv], [t[1:] for t in lv], [t[1:] for t in dv], W, H, nf, 3,
                       pts[:nf], pri, pipe.fcap, good, npts_per_frame=cnt[:nf])
        out[f"klt_fb_{nf}x{NFEAT}"] = timed(klt)
        out["klt_tracked_fraction"] = float(good.sum().item()) / float(cnt[:nf].sum().item())
        prs = [synth.make_pose_problem(NFEAT, i, w=W, h=H, outlier_frac=0.1) for i in range(8)]
        t = lambda key: torch.from_numpy(np.stack([prs[i % 8][key] for i in range(BATCH)])).to(dev)  # noqa: E731
        bv, X, uv, pose0 = t("bv"), t("X"), t("uv"), t("pose0")
        K = torch.from_numpy(np.tile(prs[0]["K"], (BATCH, 1))).to(dev)
        T = torch.zeros((BATCH, 12), dtype=torch.float64, device=dev)
        outl = torch.zeros((BATCH, NFEAT), dtype=torch.uint8, device=dev)
        info = torch.zeros((BATCH, 4), dtype=torch.float64, device=dev)
        summ = torch.zeros((BATCH, 12), dtype=torch.float64, device=dev)
        out[f"p3p_lmeds_{BATCH}x{NFEAT}"] = timed(lambda: ctx.p3p_lmeds(BATCH, NFEAT, bv, X, None, T, outl, info, fx=float(prs[0]["K"][0]),
                                                                       fy=float(prs[0]["K"][1])))

        def pnp():
            p = pose0.clone()
            ctx.pnp(BATCH, NFEAT, K, uv, X, None, p, outl, summ, float(np.sqrt(np.float32(5.9915))), float(np.float32(5.9915)))
        out[f"pnp_{BATCH}x{NFEAT}"] = timed(pnp)
        assert int(info[:, 0].sum().item()) == BATCH and int(summ[:, 10].sum().item()) == BATCH
        kf = torch.arange(0, BATCH, KF_INTERVAL, device=dev)
        kimg = lv[0].index_select(0, kf).contiguous()
        kcur = pts.index_select(0, kf)[:, ::2].contiguous()      # half of the tracked points: about half the cells stay free
        kn = torch.clamp(cnt.index_select(0, kf) // 2, max=kcur.shape[1]).to(torch.int32).contiguous()
        dout = torch.zeros((len(kf), 2048, 2), dtype=torch.float32, device=dev)
        dcnt = torch.zeros(len(kf), dtype=torch.int32, device=dev)

        def det():
            q = torch.full((len(kf),), 0.001, dtype=torch.float64, device=dev)
            ctx.detect_grid(kimg, W, H, len(kf), 40, kcur, kn, kcur.shape[1], [20, 20, W - 40, H - 40], q, dout, None, dcnt, 2048)
        out[f"detect_grid_{len(kf)}kf"] = timed(det)
        out["detect_corners_per_kf"] = float(dcnt.float().mean().item())
    return out


def system_api_times(with_reference):
    """findCameraPose timings at 640x480 (40 frames), at the headline frame size 1280x720 (30 frames) and at 1920x1080 (24 frames)."""
    out = system_api_times_at(640, 480, 40, with_reference)
    try:
        out["at_1280x720"] = system_api_times_at(1280, 720, 30, with_reference)
    except Exception as e:
        out["at_1280x720"] = {"error": repr(e)}
    try:
        out["at_1920x1080"] = system_api_times_at(1920, 1080, 24, with_reference)
    except Exception as e:
        out["at_1920x1080"] = {"error": repr(e)}
    try:
        out["concurrent_streams"] = system_concurrent_streams(8, 640, 480, 40)
    except Exception as e:
        out["concurrent_streams"] = {"error": repr(e)}
    return out


def system_concurrent_streams(nstreams, w, h, nf):
    """nstreams independent System handles (one camera stream each, own CUDA stream) on ONE GPU, driven through the batched entry
    point (alva_system_find_camera_pose_batch: one call per frame step, host RGBA in): aggregate frames/s, and a determinism
    check -- all streams see the same frames, so they must report bit-identical poses."""
    import ctypes as C
    import alvaar_b200
    from alvaar_b200 import synth
    K = synth.intrinsics(w, h)
    frames, _ = synth.make_frames(nf, w, h, seed=7, rgba=True)
    frames = [np.ascontiguousarray(f) for f in frames]
    L = alvaar_b200.lib()
    L.alva_system_create.restype = C.c_void_p
    L.alva_system_configure.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_double] * 8
    L.alva_system_find_camera_pose_ts.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
    L.alva_system_destroy.argtypes = [C.c_void_p]
    handles = []
    for _ in range(nstreams):
        s = C.c_void_p(L.alva_system_create(0))
        assert L.alva_system_configure(s, w, h, K[0], K[1], K[2], K[3], 0, 0, 0, 0) == 0
        handles.append(s)
    L.alva_system_pin_buffer.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    fr_all = np.ascontiguousarray(np.stack(frames))      # one page-locked block for the sequence (registration is process-wide)
    frames = [fr_all[k] for k in range(nf)]
    pinned = L.alva_system_pin_buffer(handles[0], fr_all.ctypes.data_as(C.c_void_p), fr_all.nbytes) == 0
    poses = [np.zeros((nf, 16), np.float32) for _ in range(nstreams)]
    status = [np.zeros(nf, np.int32) for _ in range(nstreams)]
    # all streams through ONE call per frame step (alva_system_find_camera_pose_batch: one host thread per stream inside the library)
    L.alva_system_find_camera_pose_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    harr = (C.c_void_p * nstreams)(*[s.value for s in handles])
    bp = np.zeros((nstreams, 16), np.float32)
    bs = np.zeros(nstreams, np.int32)
    t0 = time.perf_counter()
    for k in range(nf):
        parr = (C.c_void_p * nstreams)(*[frames[k].ctypes.data] * nstreams)
        ts = np.full(nstreams, k * 33.333)
        L.alva_system_find_camera_pose_batch(harr, parr, ts.ctypes.data_as(C.c_void_p), nstreams, bp.ctypes.data_as(C.c_void_p), bs.ctypes.data_as(C.c_void_p))
        for i in range(nstreams):
            poses[i][k] = bp[i]
            status[i][k] = bs[i]
    dt = time.perf_counter() - t0
    for s in handles:
        L.alva_system_destroy(s)
    same = all(np.array_equal(poses[0], p) and np.array_equal(status[0], st) for p, st in zip(poses, status))
    return {"streams": nstreams, "frame": f"{w}x{h}", "frames_per_stream": nf, "aggregate_frames_per_sec": float(nstreams * nf / dt),
            "all_streams_bit_identical": bool(same), "final_status": int(status[0][-1]), "input_pinned": bool(pinned),
            "api": "alva_system_find_camera_pose_batch"}


def system_api_times_at(w, h, nf, with_reference):
    """The reference's public API itself -- System::findCameraPose, one frame per call, host RGBA in, pose out
    (alva_system_*: upload + pyramid + KLT + P3P/PnP every frame; detector, ORB, triangulation, local-map matching and local BA
    on keyframes) -- over a synthetic sequence, wall clock per call, AFTER the headline measurement.  With the
    reference built in the tree (oracle/_ref), its own System is timed on the same frames (one host thread, as shipped)."""
    import ctypes as C
    import alvaar_b200
    from alvaar_b200 import synth
    K = synth.intrinsics(w, h)
    frames, _ = synth.make_frames(nf, w, h, seed=7, rgba=True)
    P = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    L = alvaar_b200.lib()
    L.alva_system_create.restype = C.c_void_p
    L.alva_system_configure.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_double] * 8
    L.alva_system_find_camera_pose_ts.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
    L.alva_system_get_info.argtypes = [C.c_void_p, C.c_void_p]
    L.alva_system_destroy.argtypes = [C.c_void_p]
    L.alva_system_pin_buffer.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    out = {}
    for rep in range(2):   # the second pass is the warm one
        s = C.c_void_p(L.alva_system_create(0))
        assert L.alva_system_configure(s, w, h, K[0], K[1], K[2], K[3], 0, 0, 0, 0) == 0
        # the caller-owned frame memory is page-locked once, as a host that reuses its image buffer would do (e2e: pinned host RGBA in)
        out["input_pinned"] = L.alva_system_pin_buffer(s, P(frames), frames.nbytes) == 0
        pose = np.zeros(16, np.float32)
        ms, status, kf = [], [], []
        info = np.zeros(8, np.int32)
        last_kf = 0
        for k in range(nf):
            f = np.ascontiguousarray(frames[k])
            t0 = time.perf_counter()
            st = L.alva_system_find_camera_pose_ts(s, P(f), k * 33.333, P(pose))
            ms.append((time.perf_counter() - t0) * 1e3)
            L.alva_system_get_info(s, P(info))
            status.append(int(st)); kf.append(int(info[5]) != last_kf); last_kf = int(info[5])
        L.alva_system_destroy(s)
    ms, kf, status = np.array(ms), np.array(kf), np.array(status)
    out.update({"frames": nf, "frame": f"{w}x{h}", "ms_per_tracked_frame_median": float(np.median(ms[~kf & (status == 1)])),
                "ms_per_keyframe_median": float(np.median(ms[kf])), "frames_per_sec_whole_sequence": float(nf / (ms.sum() * 1e-3)),
                "status_counts": {str(v): int((status == v).sum()) for v in (1, 2, 3)}, "keyframes": int(kf.sum())})
    ref_so = os.path.join(ROOT, "oracle", "_ref", "libalva_ref.so")
    if with_reference and os.path.exists(ref_so):
        R = C.CDLL(ref_so)
        R.ref_config(1, 1)
        R.ref_system_create.restype = C.c_void_p
        R.ref_system_create.argtypes = [C.c_int, C.c_int] + [C.c_double] * 8
        R.ref_system_find_camera_pose.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
        R.ref_system_destroy.argtypes = [C.c_void_p]
        r = R.ref_system_create(w, h, K[0], K[1], K[2], K[3], 0, 0, 0, 0)
        pose = np.zeros(16, np.float32)
        t0 = time.perf_counter()
        for k in range(nf):
            R.ref_system_find_camera_pose(r, P(np.ascontiguousarray(frames[k])), k * 33.333, P(pose))
        out["reference_system_frames_per_sec"] = float(nf / (time.perf_counter() - t0))
        R.ref_system_destroy(r)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-worker"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="c2: 1280x720 / 1000 features (headline); c3: 1920x1080 / 2000 features")
    ap.add_argument("--cores", default="", help=argparse.SUPPRESS)
    ap.add_argument("--stream", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--print-checksums", action="store_true", help="print the output checksums of the step for the stream seeds 99..106 and exit")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stage-stats", action="store_true",
                    help="skip the explanatory per-stage / System-API timings after the timed region (profiling aid: ncu's "
                         "serialisation of the 8 concurrent System threads corrupted its own heap at visit 9)")
    ap.add_argument("--no-ba-overlap", action="store_true", help="run the local BA after the frame stages instead of beside them")
    ap.add_argument("--no-loop-closure", action="store_true", help="N > 1: skip the NCCL keyframe-descriptor all-gather")
    ap.add_argument("--ba-lag", action="store_true",
                    help="join a step's BA chain at the end of the NEXT step (pipeline_ba_lag = 1; measured +6 %% frames/s, but the chain "
                         "then shares the GPU with the next step's front end, whose launch the roofline figure times)")
    ap.add_argument("--frontend-ctas", type=int, default=0, help="A/B: resident front-end CTAs per SM (4 | 5)")
    ap.add_argument("--ba-ctl-threads", type=int, default=0, help="A/B: CTA size of the BA control kernels (256 | 512 | 1024)")
    ap.add_argument("--no-graphs", action="store_true", help="launch kernel by kernel instead of replaying CUDA graphs (profiling aid)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    select_config(args.config)
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.print_checksums:
        print_checksums()
    elif args.impl == "reference-worker":
        reference_worker(args)
    elif args.impl == "reference":
        bench_reference(args, rank, world)
    else:
        bench_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
