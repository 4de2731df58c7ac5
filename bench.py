#!/usr/bin/env python
"""bench.py — frames/sec of the PL-SLAM front-end hot path (extract + match + pose-LM) on B200.

One "step" = one batch of synthetic frames per GPU through the whole per-frame hot path (ORB extract, undistort, LSD+LBD
extract, point matching frame k-1 -> k, line matching, 2 x Optimizer::PoseOptimization on the frame's pose problem).
BASELINE.json metric: "frames/sec (extract+match+pose-LM) 640x480".  Configurations (BASELINE.json `configs`):

  --config tum    (default, the headline)  640x480, TUM1 camera, ORB 1000, B = 4736 frames per GPU, WEAK scaling
  --config kitti  configs[3]: 1241x376, ORB 2000, no distortion, 256 frames sharded over the ranks (contiguous blocks with a
                  1-frame halo, pl-slam_b200/sharding.py), + one LocalBundleAdjustmentWithLine window (20+40 KFs, 3000 points,
                  400 lines) per rank and step; STRONG scaling
  --config euroc  configs[4]: 752x480, EuRoC camera, ORB 1000, 512 frames sharded over the ranks; STRONG scaling

  value     frames/s with the frames already resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e       the same through the C ABI's streaming host-buffer entry points pl_frontend_submit()/wait(): pinned host frames AND
            the step's pose problems -> H2D -> kernels -> D2H of every per-frame result, inside the timed region
  latency   (N=1) ms per frame through the synchronous host-buffer call pl_frontend_run at B = 1 and B = 64: what a Tracking
            thread that hands over one frame (or one second of video) at a time sees
  roofline  the dominant kernel (k_lsd_grow_ordered) timed with CUDA events on its own stream, algorithmic bytes / time
  cpu_baseline  the CPU oracle (a port: the reference cannot be built here, DESIGN.md) on one thread: median of >= 50 frames
  extra_configs  (default run only) a short run of the kitti and euroc configurations on the same GPUs

`--impl reference` times the CPU oracle of the same path on the host threads this process may use.
`--steps K` is the number of timed steps of every timed loop (the headline, e2e and extra_configs).
`--dump-outputs DIR` writes what the last timed step of the headline configuration computed to DIR/<name>.npy (see dump_outputs).
Nothing is written inside the tree: the -march=native oracle of the CPU legs is built in a temporary directory.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

sys.dont_write_bytecode = True

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "frames/sec (extract+match+pose-LM) 640x480"
N_PTS, N_LINES = 300, 80             # SURVEY.md §8d config 3
LINES = (200, 0.0)
KITTI_K = (718.856, 718.856, 607.1928, 185.2157)      # Examples/Monocular/KITTI00-02.yaml:8-11
CONFIGS = {
    "tum": dict(W=640, H=480, orb=(1000, 1.2, 8, 20, 7), camera="tum", scaling="weak", batch=4736, lba=False,
                workload="640x480 synthetic sequence, TUM1 camera: ORB(1000) + undistort + LSD/LBD(200) extract, frame-to-frame point+line "
                         "matching, the 4 projection searches of steady-state tracking (points: last frame 15/30 px + local map; lines: last frame + local map), "
                         "2x PoseOptimization(300 pts + 80 lines)"),
    "kitti": dict(W=1241, H=376, orb=(2000, 1.2, 8, 20, 7), camera="kitti", scaling="strong", total=256, lba=True,
                  workload="KITTI-shaped 1241x376 mono (BASELINE configs[3]): ORB(2000) + LSD/LBD(200) extract, frame-to-frame point+line matching, "
                           "4 tracking projection searches, 2x PoseOptimization, + one LocalBundleAdjustmentWithLine window (20+40 KFs, 3000 pts, 400 lines) per rank and step; "
                           "256 frames sharded over the ranks with a 1-frame halo"),
    "euroc": dict(W=752, H=480, orb=(1000, 1.2, 8, 20, 7), camera="euroc", scaling="strong", total=512, lba=False,
                  workload="EuRoC-shaped 752x480 mono (BASELINE configs[4]): EuRoC camera, ORB(1000) + undistort + LSD/LBD(200) extract, matching, "
                           "4 tracking projection searches, 2x PoseOptimization; 512 frames sharded over the ranks with a 1-frame halo, all-gather of the pose records"),
}
W, H = CONFIGS["tum"]["W"], CONFIGS["tum"]["H"]
ORB = CONFIGS["tum"]["orb"]
BASE_FRAMES = 64     # distinct host-generated frames; larger batches add per-replica sensor noise (deterministic)


def camera_of(cfg):
    from plslam_b200 import synth
    if cfg["camera"] == "tum":
        return synth.TUM1_K, synth.TUM1_DIST
    if cfg["camera"] == "euroc":
        return synth.EUROC_K, synth.EUROC_DIST
    return KITTI_K, (0.0, 0.0, 0.0, 0.0, 0.0)


def make_inputs(B, seed, w=W, h=H, K=None):
    """B synthetic frames + B pose problems.  The first min(B, 64) frames are a warped sequence (synth.synth_sequence);
    frames beyond that repeat the sequence with fresh additive sensor noise (sigma 2 grey levels, PCG64 seeded), so every
    frame of the batch has different content."""
    from plslam_b200 import synth
    nb = min(B, BASE_FRAMES)
    base = synth.synth_sequence(nb, w, h, seed=seed)
    if B > nb:
        rng = np.random.Generator(np.random.PCG64(77 + seed))
        frames = np.empty((B, h, w), np.uint8)
        frames[:nb] = base
        for r in range(nb, B, nb):
            k = min(nb, B - r)
            noise = rng.normal(0, 2.0, (k, h, w)).astype(np.float32)
            frames[r:r + k] = np.clip(np.rint(base[:k].astype(np.float32) + noise), 0, 255).astype(np.uint8)
    else:
        frames = base
    kw = {} if K is None else dict(K=K, w=w, h=h)
    problems = [synth.synth_pose_problem(1000 * seed + k, n_points=N_PTS, n_lines=N_LINES, **kw) for k in range(B)]
    return frames, problems


# ------------------------------------------------------------------------------------------------ CPU oracle arm
_NATIVE_DIR = None


def use_native_oracle():
    """The CPU legs time the -march=native build of the oracle (BASELINE.md §3: -O3 -march=native), compiled on the box that
    does the timing; the portable build that travels with the repo stays the checker of the tests."""
    global _NATIVE_DIR
    if _NATIVE_DIR is None:
        _NATIVE_DIR = tempfile.TemporaryDirectory(prefix="plslam-bench-")
    lib = os.path.join(_NATIVE_DIR.name, "liboracle_native.so")
    try:
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s", "native", f"NATIVE_LIB={lib}"],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        os.environ["PLSLAM_ORACLE_LIB"] = lib
        return "-O3 -march=native"
    except Exception:
        return "-O3 -march=x86-64-v3 (native build failed)"


def oracle_features(o_orb, img, cfg):
    import oracle
    K, D = camera_of(cfg)
    kps, desc = o_orb.extract(img)                                   # Frame.cc:224 (raw image)
    und = oracle.undistort_remap(img, K, D) if D[0] != 0.0 else img  # Frame.cc:220-222
    kl, ldesc, lf = oracle.line_extract(und, nfeatures=LINES[0], min_line_length=LINES[1])   # Frame.cc:225
    kps = oracle.undistort_keypoints(kps, K, D)                      # Frame.cc:233
    return kps, desc, ldesc, kl, lf


def oracle_frame_pipeline(o_orb, prev, img, prob, cfg, bounds):
    """The same per-frame work on the CPU oracle; returns the frame's features (to serve as `prev`)."""
    import oracle
    kps, desc, ldesc, kl, lf = oracle_features(o_orb, img, cfg)
    if prev is not None:
        pk, pd, pl_, pkl, _ = prev
        pm = np.stack([pk["x"], pk["y"]], 1).astype(np.float32)
        oracle.search_for_initialization(pk, pd, kps, desc, bounds, pm, 100, 0.9, True)
        oracle.search_double(pl_, ldesc, 0.7)
        # steady-state tracking searches on the previous frame's features as the map (the GPU step's tracking stage, frontend.cu)
        T = np.asarray(prob["Tcw0"], np.float32).reshape(4, 4); Kc = np.asarray(prob["K"], np.float32)
        sf = np.cumprod(np.r_[np.float32(1), np.full(cfg["orb"][2] - 1, np.float32(cfg["orb"][1]))]).astype(np.float32)
        z = (np.float32(1.5) + np.float32(0.25) * (np.arange(len(pk)) & 15).astype(np.float32)).astype(np.float32)
        Xc = np.stack([(pk["x"] - Kc[2]) / Kc[0] * z, (pk["y"] - Kc[3]) / Kc[1] * z, z], 1).astype(np.float32)
        pos = ((Xc - T[:3, 3]) @ T[:3, :3]).astype(np.float32)
        valid = np.ones(len(pk), np.uint8)
        nm, m = oracle.search_by_projection_last(kps, desc, bounds, T, Kc, sf, valid, pos, pd, pk["octave"], pk["angle"], 15.0, True)
        if nm < 20:
            nm, m = oracle.search_by_projection_last(kps, desc, bounds, T, Kc, sf, valid, pos, pd, pk["octave"], pk["angle"], 30.0, True)
        view = valid.copy(); view[m[m >= 0]] = 0
        oracle.search_by_projection_points(kps, desc, bounds, sf, view, pm, pk["octave"], np.ones(len(pk), np.float32), pd, 1.0, 0.8,
                                           (m >= 0).astype(np.uint8))
        proj = np.stack([pkl["startPointX"], pkl["startPointY"], pkl["endPointX"], pkl["endPointY"]], 1).astype(np.float32)
        lvalid = np.ones(len(pkl), np.uint8)
        lnm, lm = oracle.line_search_by_projection_last(kl, lf, ldesc, bounds, lvalid, proj, pl_, pkl["lineLength"], 15.0)
        lview = lvalid.copy(); lview[lm[lm >= 0]] = 0
        oracle.line_search_by_projection_lines(kl, lf, ldesc, bounds, lview, proj, np.ones(len(pkl), np.float32), pl_, 1.0, 0.7,
                                               (lm >= 0).astype(np.uint8))
    for _ in range(2):
        oracle.pose_optimization(0, prob["Tcw0"], prob["K"], prob["pt_obs"], prob["pt_inv_sigma2"], prob["pt_Xw"],
                                 prob["line_func"], prob["line_Xw"])
    return kps, desc, ldesc, kl, lf


def cpu_sample(frames, problems, n_frames, threads, cfg=None, per_frame=False):
    """Time n_frames frames of the oracle pipeline on `threads` host threads; returns (frames/s, n_frames, seconds) or, with
    per_frame, the list of per-frame seconds.  Frame i+1 is matched against frame i; the predecessor's features are prepared
    outside the timed region (a frame's extraction is counted once, as in the GPU batch)."""
    import oracle
    from concurrent.futures import ThreadPoolExecutor
    cfg = cfg or CONFIGS["tum"]
    K, D = camera_of(cfg)
    bounds = oracle.image_bounds(K, D, cfg["W"], cfg["H"])
    n_frames = min(n_frames, len(frames) - 1)

    def features(idx):
        return oracle_features(oracle.OrbOracle(*cfg["orb"]), frames[idx], cfg)

    def one(i):
        t = time.perf_counter()
        oracle_frame_pipeline(oracle.OrbOracle(*cfg["orb"]), prevs[i], frames[i + 1], problems[i + 1], cfg, bounds)
        return time.perf_counter() - t

    with ThreadPoolExecutor(max(threads, 1)) as ex:
        prevs = list(ex.map(features, range(n_frames)))
        t0 = time.perf_counter()
        per = [one(i) for i in range(n_frames)] if threads == 1 else list(ex.map(one, range(n_frames)))
        dt = time.perf_counter() - t0
    return per if per_frame else (n_frames / dt, n_frames, dt)


def host_threads():
    try:
        return max(len(os.sched_getaffinity(0)), 1)
    except Exception:
        return os.cpu_count() or 1


def run_reference(args):
    """CPU arm: the oracle (a port of the reference's CPU path) on the host threads this process may use, bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    flags = use_native_oracle()
    import oracle
    oracle.build()
    cfg = CONFIGS[args.config]
    threads = host_threads()
    per_step = max(2 * threads, 8)
    K, _ = camera_of(cfg)
    frames, problems = make_inputs(per_step + 1, 1, cfg["W"], cfg["H"], K)
    for _ in range(max(args.warmup, 1)):
        cpu_sample(frames, problems, threads, threads, cfg)
    tot_n, tot_t = 0, 0.0
    for _ in range(args.steps):
        _, n, dt = cpu_sample(frames, problems, per_step, threads, cfg)
        tot_n += n; tot_t += dt
    value = tot_n / tot_t
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": max(args.warmup, 1), "ms_per_step": 1000.0 * tot_t / args.steps, "higher_is_better": True,
            "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "u8/i32 front-end, f32 descriptors, f64 LM", "data": "synthetic",
            "config": {"workload": cfg["workload"], "frames_per_step": per_step, "name": args.config},
            "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "port",
                             "sample": f"{per_step} frames per step x {args.steps} steps on {threads} threads (sched_getaffinity); CPU oracle built {flags} "
                                       "(restatement: the reference needs OpenCV/Eigen headers that are not installed)"},
            "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ------------------------------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([c.strip() for c in ln.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ GPU arm
class Ctx:
    """Process-wide state of the GPU arm: rank layout, the launching stream, and (N > 1) the library's own NCCL communicator
    for the one exchange step (pl_allgather_poses, include/plslam_b200.h)."""

    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0")); self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: plslam_b200 has no CPU fallback (use --impl reference for the CPU oracle)")
        torch.cuda.set_device(self.local)
        self.dist = None
        self.comm = None
        if self.world > 1:
            import ctypes as C
            import torch.distributed as dist
            import plslam_b200 as pl
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
            L = pl.binding.lib()
            uid = np.zeros(128, np.uint8)
            if self.rank == 0:
                pl.binding.check(L.pl_comm_unique_id(uid.ctypes.data_as(C.c_void_p)))
            box = [uid.tobytes()]
            dist.broadcast_object_list(box, src=0)
            uid = np.frombuffer(box[0], np.uint8).copy()
            h = C.c_void_p()
            L.pl_comm_create.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
            pl.binding.check(L.pl_comm_create(uid.ctypes.data_as(C.c_void_p), self.world, self.rank, C.byref(h)))
            L.pl_allgather_poses.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
            self.comm = h
            self._L = L
        self.stream = torch.cuda.Stream()      # a real (non-NULL) stream: the C ABI treats NULL as "the handle's own stream"
        torch.cuda.set_stream(self.stream)
        self.sptr = self.stream.cuda_stream
        assert self.sptr != 0

    def allgather(self, send, recv, floats_per_rank):
        import plslam_b200 as pl
        pl.binding.check(self._L.pl_allgather_poses(self.comm, send.data_ptr(), recv.data_ptr(), floats_per_rank, self.sptr))

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()


DUMP_FRAMES = 64           # frames of the batch whose per-feature outputs --dump-outputs writes (fixed seed, sorted)


def dump_outputs(fe, B, out_dir):
    """What the last timed step computed, as a caller of the device-resident path fetches it (Frontend.fetch and fetch_tracking),
    written as out_dir/<name>.npy in float32 / float64.  Per-frame counts and poses cover the whole batch; per-feature arrays
    (keypoints, descriptors, keylines, matches) cover DUMP_FRAMES frames drawn with a fixed seed, with the entries past each
    frame's count zeroed (they are unused buffer space).  Integers are stored as float64, exactly."""
    os.makedirs(out_dir, exist_ok=True)
    o = fe.fetch(B)
    t = [fe.fetch_tracking(B, which) for which in (0, 1)]
    frames = np.sort(np.random.default_rng(0).choice(B, min(B, DUMP_FRAMES), replace=False))

    def valid(a, n):              # a[frames] with entries at or past the frame's count zeroed
        a = a[frames].copy()
        a[np.arange(a.shape[1])[None, :] >= n[frames][:, None]] = 0
        return a

    def fields(a):                # structured records -> [..., n_fields]
        return np.stack([a[f].astype(np.float64) for f in a.dtype.names], -1)

    arrays = {"frames": frames, "n_keypoints": o["n"], "n_keylines": o["nl"], "n_point_matches": o["n_pt_matches"],
              "n_line_matches": o["n_line_matches"], "poses": o["poses"], "inliers": o["inliers"],
              "keypoints": fields(valid(o["kps"], o["n"])), "descriptors": valid(o["desc"], o["n"]),
              "keylines": fields(valid(o["keylines"], o["nl"])), "line_descriptors": valid(o["ldesc"], o["nl"]),
              "point_matches": valid(o["pt_matches"], o["n"]), "line_matches": valid(o["line_matches"], o["nl"])}
    for k, tk in enumerate(t):
        arrays[f"tracking{k}_n_point"] = tk["n_pt"]
        arrays[f"tracking{k}_n_line"] = tk["n_line"]
        arrays[f"tracking{k}_point_match"] = valid(tk["pt_match"], o["n"])
        arrays[f"tracking{k}_line_match"] = valid(tk["line_match"], o["nl"])
    total = 0
    for k, a in arrays.items():
        a = np.ascontiguousarray(a, np.float32 if a.dtype in (np.float32, np.uint8) else np.float64)
        total += a.nbytes
        np.save(os.path.join(out_dir, k + ".npy"), a)
    assert total <= 64 << 20, total


def run_config(ctx, name, steps, warmup, batch=None, full=True, dump_dir=None):
    """One configuration on this process's GPU; returns the measurements (rank-local python values, timings max over ranks)."""
    import plslam_b200 as pl
    from plslam_b200 import synth, sharding
    torch = ctx.torch
    cfg = CONFIGS[name]
    w, h = cfg["W"], cfg["H"]
    K, D = camera_of(cfg)
    if cfg["scaling"] == "weak":
        B = batch or cfg["batch"]
        halo, count, first, total = 0, B, ctx.rank * B, ctx.world * B
        frames, problems = make_inputs(B, 1 + ctx.rank, w, h, K)      # weak scaling: every rank gets its own B frames
    else:
        total = batch or cfg["total"]
        first, count, halo = sharding.shard_frames(total, ctx.world, ctx.rank)
        allf, allp = make_inputs(total, 1, w, h, K)                     # one sequence, a contiguous block (+1-frame halo) per rank
        frames = np.ascontiguousarray(allf[first - halo:first + count]); problems = allp[first - halo:first + count]
        B = count + halo
    fe = pl.Frontend(w, h, max_batch=B, orb=cfg["orb"], lines=LINES, lm_caps=(N_PTS + 20, N_LINES + 8))
    fe.set_camera(K, D)             # TUM1 / EuRoC: frames and keypoints are undistorted on the device; KITTI: bounds only
    fe.pack_pose_problems(problems, pinned=True)
    prob_bytes = fe.upload_pose_problems(None)
    fe.set_tracking(True)           # the four projection searches of steady-state tracking (Tracking.cc:1345-1357, :1799, :1855)
    torch.cuda.synchronize()
    d_frames = torch.from_numpy(frames).cuda()
    max_count = -(-total // ctx.world)
    poses = torch.zeros((B, 16), dtype=torch.float32, device="cuda")
    send = torch.zeros((max_count, 16), dtype=torch.float32, device="cuda")
    gathered = torch.empty((ctx.world * max_count, 16), dtype=torch.float32, device="cuda") if ctx.world > 1 else None
    ba = None
    if cfg["lba"]:
        ba = synth.synth_ba_problem(seed=4 + ctx.rank, K=KITTI_K, w=w, h=h)

    def step():
        fe.run_dev(d_frames.data_ptr(), w, w * h, B, ctx.sptr)
        if ctx.world > 1:      # SURVEY.md §8e: the one exchange — all-gather of the per-frame pose records (halo frame excluded)
            fe.copy_poses_dev(B, poses.data_ptr(), ctx.sptr)
            send[:count].copy_(poses[halo:halo + count])
            ctx.allgather(send, gathered, max_count * 16)
        if ba is not None:     # LocalMapping's window of this rank (replicas only, SURVEY.md §8e); runs beside the front-end kernels
            pl.LocalBundleAdjustmentWithLine(ba)

    for _ in range(max(warmup, 3)):
        step()
    torch.cuda.synchronize()
    sampler = None
    if ctx.rank == 0 and full:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        idx = int(vis.split(",")[ctx.local]) if vis and vis.split(",")[0].isdigit() else torch.cuda.current_device()
        sampler = ClockSampler(idx)
        sampler.start()
    ctx.barrier()
    torch.cuda.synchronize()
    launches0 = pl.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(ctx.stream)
    for _ in range(steps):
        step()
    ev1.record(ctx.stream)
    torch.cuda.synchronize()
    ctx.barrier()
    ms = ctx.max_over_ranks(ev0.elapsed_time(ev1))
    launches = pl.launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    if dump_dir and ctx.rank == 0:
        dump_outputs(fe, B, dump_dir)
    res = dict(name=name, B=B, total=total, halo=halo, ms=ms, steps=steps, value=total * steps / (ms / 1000.0), launches=int(launches),
               clocks=clocks, frame=[w, h], orb=list(cfg["orb"]))
    if ba is not None:
        t = []
        for _ in range(3):
            torch.cuda.synchronize(); t0 = time.perf_counter(); pl.LocalBundleAdjustmentWithLine(ba); t.append(1000 * (time.perf_counter() - t0))
        res["lba_ms"] = float(np.median(t))
        res["lba_window"] = "20 free + 40 fixed KFs, 3000 points, 400 lines"
    if not full:
        del fe, d_frames
        torch.cuda.empty_cache()
        return res

    # ---- dominant kernel, timed on its launching stream (roofline)
    fe.set_timing(True)
    grow = []
    for _ in range(3):
        fe.run_dev(d_frames.data_ptr(), w, w * h, B, ctx.sptr)
        torch.cuda.synchronize()
        grow.append(fe.grow_ms())
    fe.set_timing(False)
    res["grow_ms"] = float(np.mean(grow))
    res["grow_bytes"] = fe.grow_bytes_per_frame() * B

    # ---- e2e through the host-buffer C ABI (pinned host memory; frames AND pose problems H2D, every result D2H, all timed)
    pin = torch.empty((B, h, w), dtype=torch.uint8, pin_memory=True)
    pin.numpy()[:] = frames
    # streaming entry points: submit(i+1) is enqueued while step i computes, so its H2D copy and the D2H copy of step i-1
    # overlap the kernels; two alternating sets of pinned output buffers, every step's results land on the host.
    outs = [fe.alloc_outputs(B, pinned=True) for _ in range(2)]
    for k in range(2):
        fe.upload_pose_problems(None); fe.submit(pin.numpy(), outs[k])
    fe.wait(0)
    torch.cuda.synchronize()
    ctx.barrier()
    e2e_steps = steps
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        fe.upload_pose_problems(None)      # the step's LM problems travel with the step (14 KB per frame)
        fe.submit(pin.numpy(), outs[k & 1])
        fe.wait(1)                 # results of step k-1 are on the host here
    fe.wait(0)
    torch.cuda.synchronize()
    e2e_s = ctx.max_over_ranks(time.perf_counter() - t0)
    h2d, d2h = fe.io_bytes()
    res["e2e"] = {"value": total * e2e_steps / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": int(h2d * B + prob_bytes),
                  "d2h_bytes_per_step": int(d2h * B), "steps": e2e_steps}
    res["frames"], res["problems"] = frames, problems
    del fe, d_frames
    torch.cuda.empty_cache()
    return res


def measure_latency(ctx, frames, problems):
    """ms per frame of the synchronous host-buffer call (pl_frontend_run) at B = 1 and B = 64: H2D, all kernels, D2H, sync."""
    import plslam_b200 as pl
    from plslam_b200 import synth
    out = {}
    fe = pl.Frontend(W, H, max_batch=64, orb=ORB, lines=LINES, lm_caps=(N_PTS + 20, N_LINES + 8))
    fe.set_camera(synth.TUM1_K, synth.TUM1_DIST)
    for B, reps in ((1, 30), (64, 7)):
        fr = np.ascontiguousarray(frames[:B])
        fe.set_pose_problems(problems[:B])
        fe.set_tracking(True)
        o = fe.alloc_outputs(B)
        t = []
        for r in range(reps + 3):
            t0 = time.perf_counter(); fe.run(fr, o); t.append(time.perf_counter() - t0)
        med = float(np.median(t[3:]))
        out[f"b{B}"] = {"ms_per_call": 1000 * med, "ms_per_frame": 1000 * med / B, "fps": B / med, "calls": reps}
    out["api"] = "pl_frontend_run (host buffers in, host buffers out, synchronous)"
    del fe
    ctx.torch.cuda.empty_cache()
    return out


def cpu_baseline_single_thread(frames, problems):
    """The oracle on ONE thread: median per-frame time of >= 50 frames after 5 warm-up frames (BASELINE.md §3)."""
    flags = use_native_oracle()
    import oracle
    oracle.build()
    n = min(55, len(frames) - 1)
    per = cpu_sample(frames, problems, n, 1, CONFIGS["tum"], per_frame=True)
    per = per[5:] if len(per) > 10 else per
    med = float(np.median(per))
    cpu = {"value": 1.0 / med, "unit": "frames/s", "cores": 1, "kind": "port",
           "sample": f"median of {len(per)} frames after 5 warm-up frames, one thread, CPU oracle built {flags} (restatement)",
           "ms_per_frame_median": 1000 * med, "ms_per_frame_mean": 1000 * float(np.mean(per))}
    try:   # cv2 single-thread cross-check recorded in the build container (the GPU box has no cv2): tools/cv2_crosscheck.py
        cpu["cv2_check"] = json.load(open(os.path.join(ROOT, "profiles", "r02_cpu_crosscheck.json")))
    except Exception:
        pass
    return cpu


def run_ours(args):
    ctx = Ctx()
    name = args.config
    res = run_config(ctx, name, args.steps, args.warmup, args.batch, full=True, dump_dir=args.dump_outputs)
    cfg = CONFIGS[name]
    latency, extra, cpu = None, None, None
    if ctx.world == 1 and name == "tum":
        latency = measure_latency(ctx, res["frames"], res["problems"])
    if name == "tum" and not args.no_extra:
        extra = {}
        for other in ("kitti", "euroc"):
            r = run_config(ctx, other, args.steps, 3, None, full=False)
            extra[other] = {"value": r["value"], "unit": "frames/s", "ms_per_step": r["ms"] / r["steps"], "frames_per_step_total": r["total"],
                            "frames_this_rank": r["B"], "halo": r["halo"], "scaling": "strong", "frame": r["frame"], "orb": r["orb"],
                            **({"lba_ms": r["lba_ms"], "lba_window": r["lba_window"]} if "lba_ms" in r else {})}
    if ctx.rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = res["grow_bytes"] / (res["grow_ms"] / 1000.0) / 1e9
        if ctx.world == 1 and name == "tum":      # CPU baseline: the oracle, one thread, bounded sample (rank 0, N=1 only)
            cpu = cpu_baseline_single_thread(res["frames"], res["problems"])
        B = res["B"]
        line = {
            "metric": METRIC, "value": res["value"], "unit": "frames/s", "n_gpus": ctx.world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": res["ms"] / args.steps, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": "u8/i32 front-end, f32 descriptors, f64 LM", "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": name, "batch_per_gpu": B, "frames_per_step_total": res["total"], "halo_frames": res["halo"],
                       "frame": res["frame"], "orb": res["orb"], "lines": list(LINES),
                       "l2": f"inputs {B * res['frame'][0] * res['frame'][1] / 1e6:.0f} MB per step vs the 126 MB L2; every kernel streams a different frame",
                       "predecessor": "frame 0 of a step is matched against the last frame of the previous step (one sequence)",
                       "exchange": "none at 1 GPU; pl_allgather_poses (NCCL) of the [frames][16] pose records per step at N>1",
                       **({"lba_ms": res["lba_ms"], "lba_window": res["lba_window"]} if "lba_ms" in res else {})},
            "clocks": res["clocks"], "gpu_launches": res["launches"],
            "e2e": res["e2e"],
            "roofline": {"kernel": "k_lsd_grow_ordered", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": None, "ms_per_launch": res["grow_ms"],
                         "peak_source": "MEASURED_PEAKS.json (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                         "share_of_step": res["grow_ms"] / (res["ms"] / args.steps)},
            "cpu_baseline": cpu,
        }
        if latency:
            line["latency"] = latency
        if extra:
            line["extra_configs"] = extra
        traffic_file = os.path.join(ROOT, "profiles", "traffic_k_lsd_grow.json")
        if os.path.exists(traffic_file):
            try:
                tj = json.load(open(traffic_file))     # one `ncu --set full` capture: DRAM bytes per frame of the launch
                if tj.get("kernel") == "k_lsd_grow_ordered":
                    line["roofline"]["traffic"] = float(tj["dram_bytes_per_frame"]) * B
                    line["roofline"]["traffic_source"] = tj.get("source")
            except Exception:
                pass
        emit(line)
    if ctx.world > 1:
        ctx.dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """The one JSON line of the contract, written to the process's ORIGINAL stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # Native libraries write to fd 1 on their own (NCCL prints "NCCL version ..." there when NCCL_DEBUG=VERSION, a setting
    # that ignores NCCL_DEBUG_FILE).  stdout must carry exactly one JSON line, so fd 1 is pointed at stderr for the whole run
    # and the JSON line goes to the saved descriptor.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=None, help="tum: frames per GPU per step (default 4736 = 148 SMs x 32 resident region-growing "
                                                            "warps); kitti / euroc: total frames per step over all ranks (default 256 / 512)")
    ap.add_argument("--config", default="tum", choices=sorted(CONFIGS), help="BASELINE.json configuration (tum = the headline metric)")
    ap.add_argument("--no-extra", action="store_true", help="default run: skip the short kitti / euroc runs")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
