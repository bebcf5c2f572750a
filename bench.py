#!/usr/bin/env python
"""bench.py -- stereo frames/sec of the circularMatching() hot path on B200 (+ the CPU reference arm).

  python bench.py --gpus N --steps K --warmup W            this library (one process per GPU)
  python bench.py --impl reference --gpus N --steps K ...  the reference's OpenCV CPU path on the host cores

One "step" = one pass of the whole path (FAST -> select 2000 -> pyramids -> LK ring -> filters ->
triangulation -> PnP/RANSAC) over `--units` independent KITTI-shaped synthetic stereo pairs per GPU.
Prints ONE JSON line (see README "bench contract"):
  value      frames/s, inputs resident in HBM when the timed region starts (vo_batch_submit(units = NULL) / vo_batch_wait,
             two submissions in flight, L2 flushed before every submission)
  e2e        frames/s through the C-ABI with pinned HOST buffers: H2D of the 4 images per unit + run + D2H of the result
             records AND of every unit's point lists inside the timed region (vo_batch_submit / vo_batch_wait /
             vo_batch_outputs, three submissions in flight; with N GPUs the record gather vo_dist_* is inside too)
  roofline   LK ring kernel: algorithmic bytes (SURVEY.md 8d: 17044 B per feature-ring) / its own
             CUDA-event time on the launching stream, vs the measured HBM copy bandwidth; + the feature sweep
  cpu_baseline  cv2 (the OpenCV the reference links) through the reference glue, timed on this host
  parity     one unit per rank checked against the cv2 oracle outside the timed region
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True        # the tree the bench runs from may be read-only: nothing is written there
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W_IMG, H_IMG, N_FEAT = 1241, 376, 2000
E2E_DEPTH = int(os.environ.get("VO_BENCH_DEPTH", "3"))     # submissions in flight on the end-to-end path (the library has 3 lanes)
LK_BYTES_PER_FEATURE = 4 * (4 * ((21 + 3) ** 2 + (21 + 1) ** 2) + 21)      # 17044, SURVEY.md 8(d)
METRIC = "stereo frames/sec at 1241x376, 2000 feats; LK kernel HBM GB/s vs roofline"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200,
                    help="steps in a timed block; each path's block is timed 5 times and the median block reported")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--units", type=int, default=8, help="independent stereo pairs per step per GPU")
    ap.add_argument("--features", type=int, default=N_FEAT)
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="timed host work per CPU mode (sequential / process pool), in 3 repetitions")
    ap.add_argument("--cpu-sample", type=int, default=0, help="(ignored; kept for old command lines)")
    ap.add_argument("--sweep", type=int, default=1, help="N = 1: also run the feature sweep / 1080p / single-pair / sequence points (0 = headline only)")
    ap.add_argument("--sequence", type=int, default=48,
                    help="frames of the streaming-mode (vo_seq_push) side measurement at N=1; 0 = skip")
    ap.add_argument("--width", type=int, default=W_IMG)
    ap.add_argument("--height", type=int, default=H_IMG)
    ap.add_argument("--calib", default="kitti", choices=["kitti", "zed"], help="intrinsics of the synthetic rig")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last resident and the last end-to-end step returned as "
                         "DIR/<name>.npy (rank 0's units, at most 64 MB)")
    return ap.parse_args()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t_end = time.perf_counter() + 0.5          # a very short timed region: wait for the first sample (clocks are still up)
        while not self.lines and time.perf_counter() < t_end:
            time.sleep(0.01)
        self.proc.terminate()          # exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[2 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
def _cpu_one_frame(u, n_feat):
    """One work unit through the reference's CPU path: cv2 (the OpenCV the reference's calls resolve to) behind the
    verbatim glue of oracle/ref_path.py -- FAST, stride selection, 4-call LK ring, filters, triangulation, PnP."""
    from oracle import ref_path
    from visual_odom_b200 import synth
    corners = ref_path.fast_cv2(u["l0"])
    pts = synth.select_features(corners, n_feat)
    fs = ref_path.FeatureSet(); fs.points = pts; fs.ages = np.zeros(len(pts), np.int32)
    cm = ref_path.circular_matching(u["l0"], u["r0"], u["l1"], u["r1"], pts, fs, "cv2")
    ok = ref_path.check_valid_match(cm["l0"], cm["l0_ret"], 0)
    pL0, pR0, pL1 = (ref_path.remove_invalid_points(cm[k], ok) for k in ("l0", "r0", "l1"))
    X = ref_path.triangulate(u["P_l"], u["P_r"], pL0, pR0, "cv2")
    return ref_path.tracking_frame2frame(u["P_l"], pL0, pL1, X, np.array([0.0, 0.0, -0.8]), "cv2")


def cpu_reference_frames(units, n_feat, frames, threads=None):
    """Sequential frames, OpenCV's own thread pool inside each call (how the reference program runs)."""
    import cv2
    if threads is not None:
        cv2.setNumThreads(threads)
    for i in range(min(3, len(units))):
        _cpu_one_frame(units[i], n_feat)                      # warm-up
    t0 = time.perf_counter()
    for i in range(frames):
        _cpu_one_frame(units[i % len(units)], n_feat)
    dt = time.perf_counter() - t0
    return frames / dt, dt, cv2.getNumThreads()


_POOL_STATE = {}


def _pool_init(w, h, calib, n_feat, threads):
    """Runs once in every worker process: its own work unit + OpenCV thread count + one warm-up frame."""
    import cv2
    from visual_odom_b200 import synth
    cv2.setNumThreads(threads)
    cal = synth.KITTI00 if calib == "kitti" else synth.ZED
    _POOL_STATE["unit"] = synth.stereo_unit(w, h, os.getpid() % 64, cal=cal)
    _POOL_STATE["n_feat"] = n_feat
    _cpu_one_frame(_POOL_STATE["unit"], n_feat)


def _pool_run(reps):
    for _ in range(reps):
        _cpu_one_frame(_POOL_STATE["unit"], _POOL_STATE["n_feat"])
    return reps


def cpu_reference_parallel(n_proc, w, h, calib, n_feat, frames, threads_per_proc):
    """Independent work units on `n_proc` host processes at once (each with `threads_per_proc` OpenCV threads): what a
    CPU deployment of the batched workload would do with all the cores.  Returns (frames/s, wall seconds, frames)."""
    import multiprocessing as mp
    ctxm = mp.get_context("spawn")                 # no fork: OpenCV's thread pool does not survive one
    with ctxm.Pool(n_proc, initializer=_pool_init, initargs=(w, h, calib, n_feat, threads_per_proc)) as pool:
        pool.map(_pool_run, [1] * (2 * n_proc), chunksize=1)          # every worker initialised and warm
        chunk = 2
        tasks = max(n_proc, int(round(frames / chunk)))
        tasks = ((tasks + n_proc - 1) // n_proc) * n_proc               # whole waves
        t0 = time.perf_counter()
        done = sum(pool.map(_pool_run, [chunk] * tasks, chunksize=1))
        dt = time.perf_counter() - t0
    return done / dt, dt, done


def _median(xs):
    return float(np.median(np.asarray(xs, np.float64)))


def cpu_reference_measure(units, args, seconds_per_mode=10.0, reps=3):
    """The reference's CPU path on this host, both ways, each for >= `seconds_per_mode` of timed work in `reps`
    repetitions (median / min / max reported):
      sequential -- one frame after the other, OpenCV's own thread pool inside every call: how the reference's ./run
                    executes (src/main.cpp:123-224 is a serial loop);
      pool       -- independent work units on a process pool, one OpenCV thread per process; the number of busy
                    workers is chosen from a measured scaling curve (quarter / half / all of the affinity cores), not fixed.
    The headline CPU figure is the better median of the two."""
    import cv2
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    out = {"affinity_cores": cores, "cv2": cv2.__version__}
    # ---- sequential -------------------------------------------------------------------------------------------
    cv2.setNumThreads(-1)
    for i in range(min(3, len(units))):
        _cpu_one_frame(units[i], args.features)
    fps, frames_seq = [], 0
    t_seq = 0.0
    for r in range(reps):                       # time-based repetitions: whole frames until the repetition's share has passed
        n, t0 = 0, time.perf_counter()
        while True:
            _cpu_one_frame(units[n % len(units)], args.features)
            n += 1
            dt = time.perf_counter() - t0
            if dt >= seconds_per_mode / reps and n >= 2:
                break
        t_seq += dt
        frames_seq += n
        fps.append(n / dt)
    per_rep = frames_seq // reps
    out["sequential"] = {"median": _median(fps), "min": min(fps), "max": max(fps), "opencv_threads": cv2.getNumThreads(),
                         "frames_per_rep": per_rep, "reps": reps, "seconds": t_seq}
    # ---- process pool -----------------------------------------------------------------------------------------
    try:
        import multiprocessing as mp
        n_proc = max(1, min(cores, 128))
        ctxm = mp.get_context("spawn")                 # no fork: OpenCV's thread pool does not survive one
        with ctxm.Pool(n_proc, initializer=_pool_init, initargs=(W_IMG, H_IMG, args.calib, args.features, 1)) as pool:
            pool.map(_pool_run, [1] * (2 * n_proc), chunksize=1)          # every worker initialised and warm
            curve = {}
            for k in sorted({max(1, n_proc // 4), max(1, n_proc // 2), n_proc}):
                best = 0.0
                for _ in range(2):                                            # best of two: the first pass can still see workers finishing their initialiser
                    t0 = time.perf_counter()
                    done = sum(pool.map(_pool_run, [2] * k, chunksize=1))     # k tasks -> k busy workers
                    best = max(best, done / (time.perf_counter() - t0))
                curve[k] = best
            k_best = max(curve, key=curve.get)
            chunk = max(2, int(np.ceil(curve[k_best] * seconds_per_mode / reps / k_best)))
            fps = []
            t_pool = 0.0
            for r in range(reps):
                t0 = time.perf_counter()
                done = sum(pool.map(_pool_run, [chunk] * k_best, chunksize=1))
                dt = time.perf_counter() - t0
                t_pool += dt
                fps.append(done / dt)
        out["pool"] = {"median": _median(fps), "min": min(fps), "max": max(fps), "busy_workers": k_best, "opencv_threads_per_worker": 1,
                       "frames_per_rep": chunk * k_best, "reps": reps, "seconds": t_pool,
                       "scaling_curve_fps": {str(k): round(v, 1) for k, v in curve.items()}}
    except Exception as e:                       # never lose the line to the pool
        out["pool"] = {"error": str(e)[:160]}
    seq_med = out["sequential"]["median"]
    pool_med = out["pool"].get("median", 0.0)
    if pool_med > seq_med:
        out["best"] = {"value": pool_med, "mode": "pool", "cores": out["pool"]["busy_workers"], "seconds": out["pool"]["seconds"],
                       "frames": out["pool"]["frames_per_rep"] * reps, "spread": [out["pool"]["min"], out["pool"]["max"]]}
    else:
        out["best"] = {"value": seq_med, "mode": "sequential", "cores": out["sequential"]["opencv_threads"], "seconds": t_seq,
                       "frames": frames_seq, "spread": [out["sequential"]["min"], out["sequential"]["max"]]}
    return out


def cpu_sample_text(m):
    b = m["best"]
    return (f"{b['frames']} frames of the same workload in {b['seconds']:.1f} s ({b['mode']}: median of {m['sequential']['reps']} repetitions, "
            f"min {b['spread'][0]:.1f} / max {b['spread'][1]:.1f} frames/s); sequential (how the reference's ./run executes, OpenCV "
            f"x{m['sequential']['opencv_threads']} threads): {m['sequential']['median']:.1f} frames/s; process pool: "
            f"{m['pool'].get('median', float('nan')):.1f} frames/s on {m['pool'].get('busy_workers', 0)} single-thread workers "
            f"(scaling curve {m['pool'].get('scaling_curve_fps')}); cv2 {m['cv2']} (the OpenCV build the reference's calls resolve to) "
            f"through the oracle/ref_path.py glue restatement; affinity cores={m['affinity_cores']}")


def sequence_mode(ctx, torch, cal, n_frames):
    """SURVEY.md 8f row N1, reported beside the headline: the reference's actual usage pattern -- one stereo pair
    at a time through vo_seq_push (pinned host images in, pose out, main-loop state resident on the GPU) -- against
    the same loop on the CPU (cv2 through oracle/ref_path.matching_features).  Latency-bound: ~300 bucketed
    features per frame, one frame in flight."""
    from oracle import ref_path
    from visual_odom_b200 import synth
    step_r = np.array([0.001, -0.004, 0.0005]); step_t = np.array([0.01, -0.003, -0.2])
    base = synth.stereo_unit(W_IMG, H_IMG, 31, cal=cal)
    frames = [(base["l0"], base["r0"])]
    for k in range(1, n_frames + 1):
        u = synth.stereo_unit(W_IMG, H_IMG, 31, rvec=step_r * k, tvec=step_t * k, cal=cal)
        frames.append((u["l1"], u["r1"]))
    pin = []
    for l, r in frames:
        a = torch.empty((2, H_IMG, W_IMG), dtype=torch.uint8, pin_memory=True)
        a.numpy()[0] = l; a.numpy()[1] = r
        pin.append(a.numpy())
    lat = []
    for rep in range(2):                      # rep 0 warms up (graph capture), rep 1 is timed
        ctx.seq_begin(pin[0][0], pin[0][1], base["P_l"], base["P_r"])
        lat = []
        t0 = time.perf_counter()
        for k in range(1, n_frames + 1):
            t1 = time.perf_counter()
            got = ctx.seq_push(pin[k][0], pin[k][1], want_points=False)
            lat.append(time.perf_counter() - t1)
        dt_sync = time.perf_counter() - t0
    # pipelined: frame k+1 submitted before frame k is waited for (one frame of result lag)
    for rep in range(2):
        ctx.seq_begin(pin[0][0], pin[0][1], base["P_l"], base["P_r"])
        t0 = time.perf_counter()
        ctx.seq_submit(pin[1][0], pin[1][1])
        for k in range(1, n_frames + 1):
            if k + 1 <= n_frames:
                ctx.seq_submit(pin[k + 1][0], pin[k + 1][1])
            got_p = ctx.seq_wait(want_points=False)
        dt = time.perf_counter() - t0
    assert got_p["n_inliers"] == got["n_inliers"] and np.array_equal(got_p["tvec"], got["tvec"])
    gpu_fps = n_frames / dt
    # row N3: the same frames from a KITTI-layout PNG directory: vo_reader (worker threads decode ahead into a pinned
    # ring) -> vo_seq_submit / vo_seq_wait, against cv2.imread + cvtColor + the cv2 loop below
    png = None
    try:
        import cv2, shutil, tempfile
        from visual_odom_b200 import capi
        d = tempfile.mkdtemp(prefix="vo_png_")
        os.makedirs(os.path.join(d, "image_0")); os.makedirs(os.path.join(d, "image_1"))
        for i, (l, r) in enumerate(frames):
            cv2.imwrite(os.path.join(d, "image_0", "%06d.png" % i), l)
            cv2.imwrite(os.path.join(d, "image_1", "%06d.png" % i), r)
        threads = max(2, min(16, len(os.sched_getaffinity(0)) // 2))
        for rep in range(2):
            rd = capi.SequenceReader(d, 0, n_frames + 1, threads=threads, depth=threads + 3)
            t0 = time.perf_counter()
            lp, rp, rw, rh, rpitch, ch, fid = rd.next_ptr()
            ctx.seq_begin_ptr(rw, rh, lp, rp, rpitch, base["P_l"], base["P_r"], ch)
            lp, rp, rw, rh, rpitch, ch, fid = rd.next_ptr()
            ctx.seq_submit_ptr(lp, rp, rpitch, ch)
            for k in range(1, n_frames + 1):
                if k + 1 <= n_frames:
                    lp, rp, rw, rh, rpitch, ch, fid = rd.next_ptr()
                    ctx.seq_submit_ptr(lp, rp, rpitch, ch)
                got_f = ctx.seq_wait(want_points=False)
            dt_png = time.perf_counter() - t0
            rd.close()
        t0 = time.perf_counter()
        for i in range(min(n_frames + 1, 13)):
            for cam in (0, 1):
                cv2.cvtColor(cv2.imread(os.path.join(d, "image_%d" % cam, "%06d.png" % i), cv2.IMREAD_COLOR), cv2.COLOR_BGR2GRAY)
        cpu_load_ms = 1e3 * (time.perf_counter() - t0) / min(n_frames + 1, 13)
        shutil.rmtree(d, ignore_errors=True)
        png = {"value": n_frames / dt_png, "unit": "frames/s", "decode_threads": threads, "ring_depth": threads + 3,
               "same_result_as_memory_path": bool(got_f["n_inliers"] == got["n_inliers"] and np.array_equal(got_f["tvec"], got["tvec"])),
               "cpu_imread_cvtcolor_ms_per_frame_pair": cpu_load_ms,
               "note": "PNG files -> vo_reader (decode ahead, pinned ring) -> vo_seq_submit / vo_seq_wait; includes vo_seq_begin"}
    except Exception as e:
        png = {"error": str(e)[:200]}
    pose = ctx.seq_pose()
    # CPU: same loop, bounded sample
    fs = ref_path.FeatureSet(); translation = np.zeros(3)
    ncpu = min(n_frames, 12)
    t0 = time.perf_counter()
    for k in range(1, ncpu + 1):
        l0, r0 = frames[k - 1]; l1, r1 = frames[k]
        pL0, pR0, pL1, pR1, info = ref_path.matching_features(l0, r0, l1, r1, fs, backend="cv2")
        X = ref_path.triangulate(base["P_l"], base["P_r"], pL0, pR0, "cv2")
        R, translation, inl, rvec = ref_path.tracking_frame2frame(base["P_l"], pL0, pL1, X, translation, "cv2")
    cpu_fps = ncpu / (time.perf_counter() - t0)
    return {"value": gpu_fps, "unit": "frames/s", "frames": n_frames, "synchronous_fps": n_frames / dt_sync,
            "median_latency_ms": 1e3 * float(np.median(lat)),
            "max_latency_ms": 1e3 * float(np.max(lat)), "cpu_reference": cpu_fps, "cpu_frames": ncpu,
            "features_last_frame": int(got["n_features"]), "inliers_last_frame": int(got["n_inliers"]),
            "pose_translation": [float(x) for x in pose[:3, 3]], "from_png": png,
            "note": "value: vo_seq_submit / vo_seq_wait with two frames in flight (wall clock incl. H2D of every new pair and "
                    "the pose read-back); synchronous_fps / latency: one vo_seq_push at a time"}


def run_reference(args, rank, world):
    """--impl reference: the reference's own OpenCV CPU implementation on the host cores (rank 0 only)."""
    if rank != 0:
        return
    from visual_odom_b200 import synth
    global W_IMG, H_IMG
    W_IMG, H_IMG = args.width, args.height
    cal = synth.KITTI00 if args.calib == "kitti" else synth.ZED
    units = [synth.stereo_unit(W_IMG, H_IMG, s, cal=cal) for s in range(args.units)]
    m = cpu_reference_measure(units, args, seconds_per_mode=args.cpu_seconds, reps=3)
    value = m["best"]["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * args.units / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8/i32 fixed point + f32 (LK), f64 (pose)", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": m["best"]["cores"], "kind": "port", "sample": cpu_sample_text(m),
                         "sequential": m["sequential"], "pool": m["pool"],
                         "timing": f"time-based: >= {args.cpu_seconds:.0f} s of timed work per mode in 3 repetitions, median reported "
                                   f"(--steps / --warmup do not shorten it); one step = {args.units} frames"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(args, world):
    return {"workload": f"{args.calib}-calibrated synthetic stereo {W_IMG}x{H_IMG}, {args.features} FAST features (thr 20, even-stride "
                        f"selection), LK 21x21 maxLevel=3 (4 images) 30 it / 0.01, PnP RANSAC 500/0.5/0.999; "
                        f"{args.units} independent stereo pairs per step per GPU",
            "units_per_gpu": args.units, "global_units": args.units * world, "features": args.features,
            "l2": "flushed before every step's submission by a 256 MiB write (inside the timed region)", "parallelism": f"units sharded over {world} GPU(s), no data-path collective"}


# ------------------------------------------------------------------------------------------------
def reference_unit_outputs(u, n_feat, t_prev=(0.0, 0.0, -0.8)):
    """Everything the reference hands back for one work unit, from cv2 through the verbatim glue (the parity oracle)."""
    from oracle import ref_path
    from visual_odom_b200 import synth
    corners = ref_path.fast_cv2(u["l0"])
    pts = synth.select_features(corners, n_feat)
    fs = ref_path.FeatureSet(); fs.points = pts; fs.ages = np.zeros(len(pts), np.int32)
    cm = ref_path.circular_matching(u["l0"], u["r0"], u["l1"], u["r1"], pts, fs, "cv2")
    ok = ref_path.check_valid_match(cm["l0"], cm["l0_ret"], 0)
    pL0, pR0, pL1, pR1 = (ref_path.remove_invalid_points(cm[k], ok) for k in ("l0", "r0", "l1", "r1"))
    X = ref_path.triangulate(u["P_l"], u["P_r"], pL0, pR0, "cv2")
    R, t, inl, rvec = ref_path.tracking_frame2frame(u["P_l"], pL0, pL1, X, np.array(t_prev, np.float64), "cv2")
    return dict(kept_idx=cm["kept_idx"][ok], l0=pL0, r0=pR0, l1=pL1, r1=pR1, X=X, inliers=np.asarray(inl).ravel(), R=R, t=np.asarray(t).ravel())


def check_against_oracle(got, res, ref):
    """north_star gates: tracked-feature indices and RANSAC inlier list bit-exact, positions / [R|t] within 1e-4 relative
    (the positions are in fact compared bit for bit)."""
    bad = []
    if not np.array_equal(got["kept_idx"], ref["kept_idx"]):
        bad.append("kept_idx")
    for k in ("l0", "r0", "l1", "r1"):
        if got[k].shape != ref[k].shape or not np.array_equal(got[k], ref[k]):
            bad.append(k)
    if got["X"].shape != ref["X"].shape or not np.array_equal(got["X"], ref["X"]):
        bad.append("X")
    if not np.array_equal(got["inliers"], ref["inliers"]):
        bad.append("inliers")
    if np.linalg.norm(res["R"] - ref["R"]) > 1e-4 * np.linalg.norm(ref["R"]):
        bad.append("R")
    if np.linalg.norm(res["tvec"] - ref["t"]) > 1e-4 * max(np.linalg.norm(ref["t"]), 1e-12):
        bad.append("t")
    return bad


DUMP_BYTES = 64 << 20
RECORD_COUNTS = ("n_features", "n_detected", "n_tracked", "n_valid", "n_inliers", "ransac_iters", "pnp_status")
POINT_LISTS = (("l0", np.float32), ("r0", np.float32), ("l1", np.float32), ("r1", np.float32), ("X", np.float32),
               ("kept_idx", np.float64), ("inliers", np.float64))


def dump_outputs(out_dir, res, res_e2e, outputs, features):
    """What the last step of the timed paths returned, one DIR/<name>.npy per array (float64; point lists float32):
      units                  the units written (indices into the step's units)
      resident_*, e2e_*      their result records: counts (columns as RECORD_COUNTS), rvec, tvec, R
      e2e_l0 ... e2e_inliers their point lists from the end-to-end path, concatenated in unit order (a unit has
                             e2e_counts[:, 3] = n_valid rows of each list but inliers, and e2e_counts[:, 4] of those)
    When the worst case of all units exceeds DUMP_BYTES, a fixed seeded sample of the units is written."""
    per_unit = 60 * features + 360        # n_valid <= features rows of all lists (60 B), two records, the unit index
    units = np.arange(len(res))
    if len(units) * per_unit > DUMP_BYTES:
        units = np.sort(np.random.default_rng(0).choice(len(units), DUMP_BYTES // per_unit, replace=False))
    arrays = {"units": units.astype(np.float64)}
    for prefix, recs in (("resident", res), ("e2e", res_e2e)):
        recs = [recs[u] for u in units]
        arrays[prefix + "_counts"] = np.array([[r[k] for k in RECORD_COUNTS] for r in recs], np.float64).reshape(-1, len(RECORD_COUNTS))
        for k, shape in (("rvec", (3,)), ("tvec", (3,)), ("R", (3, 3))):
            arrays[f"{prefix}_{k}"] = np.array([r[k] for r in recs], np.float64).reshape((-1,) + shape)
    for k, dt in POINT_LISTS:
        arrays["e2e_" + k] = np.concatenate([np.asarray(outputs[u][k], dt) for u in units])
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class Point:
    """One workload point (image size, features, units per step) measured on a context: the pipelined resident pass
    (`value`), the LK kernel alone on one stream (roofline) and the pipelined end-to-end pass with pinned host images in
    and the full per-unit outputs back (`e2e`)."""

    def __init__(self, ctx, torch, stream, flush, pinned, feats, B, w, h, P_l, P_r, barrier, world, gather=None, my_units=None):
        self.ctx, self.torch, self.stream, self.flush, self.B, self.feats = ctx, torch, stream, flush, B, feats
        self.w, self.h, self.barrier, self.world, self.gather, self.my_units = w, h, barrier, world, gather, my_units
        self.depth = E2E_DEPTH
        ctx.batch_configure(w, h, self.depth * B, P_l, P_r)         # slot ranges of B units: `depth` submissions in flight end to end, two resident
        spec = [dict(p, n_select=feats, t_prev=(0.0, 0.0, -0.8)) for p in pinned]
        self.arr, self.keep, self.pitch = ctx.make_units(spec)
        self.arr2, self.keep2, _ = ctx.make_units(spec + spec)
        self.into = [[dict(pts4=np.zeros((4, feats, 2), np.float32), kept_idx=np.zeros(feats, np.int32),
                           X=np.zeros((feats, 3), np.float32), inliers=np.zeros(feats, np.int32)) for _ in range(B)] for _ in range(self.depth)]
        self.last_outputs = None
        self.d2h_outputs = 0

    def _timed(self, fn, steps):
        torch = self.torch
        ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        self.barrier()
        t0 = time.perf_counter()
        out = fn(steps, ev)
        self.barrier()
        wall = time.perf_counter() - t0
        return ev[0].elapsed_time(ev[1]), wall, out

    # ---- resident inputs: both ranges uploaded once, a step re-runs one range (units = NULL) -----------------
    def resident_steps(self, n, ev=None):
        ctx, B, flush = self.ctx, self.B, self.flush
        out = None
        if ev:
            ev[0].record(self.stream)
        flush.fill_(1)
        ctx.batch_submit(None, 0, self.pitch, n_units=B)
        for s in range(n):
            if s + 1 < n:
                flush.fill_(s & 0xFF)
                ctx.batch_submit(None, ((s + 1) & 1) * B, self.pitch, n_units=B)
            out = ctx.batch_wait((s & 1) * B, B)
        if ev:
            ev[1].record(self.stream)
        return out

    def measure_resident(self, steps, warmup, blocks=1):
        self.ctx.set_option("batch_outputs", 0)
        self.ctx.batch_upload(self.arr2, self.pitch)
        self.resident_steps(max(2, warmup))
        self.torch.cuda.synchronize()
        l0 = self.ctx.kernel_launches()
        ms, res = [], None
        for _ in range(blocks):
            t, _w, res = self._timed(self.resident_steps, steps)
            ms.append(t)
        launches = (self.ctx.kernel_launches() - l0) // blocks
        return ms, res, launches

    # ---- the LK kernel alone: one stream, plain launches, bracketed by its own CUDA events --------------------
    def measure_lk_alone(self, steps, warmup):
        ctx, torch = self.ctx, self.torch
        ctx.batch_upload(self.arr, self.pitch)
        ctx.set_option("batch_streams", 1)
        ctx.set_option("graphs", 0)
        for _ in range(max(3, warmup)):
            ctx.batch_run()
        torch.cuda.synchronize()
        ctx.lk_kernel_time(reset=True)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for s in range(steps):
            self.flush.fill_(s & 0xFF)
            evs[s][0].record(self.stream)
            ctx.batch_run()
            evs[s][1].record(self.stream)
        torch.cuda.synchronize()
        t_single = sum(a.elapsed_time(b) for a, b in evs)
        lk_ms, lk_n = ctx.lk_kernel_time(reset=True)
        res = ctx.batch_download(self.B)
        ctx.set_option("batch_streams", 2)
        ctx.set_option("graphs", 1)
        return lk_ms / max(lk_n, 1), lk_ms, t_single, sum(r["n_features"] for r in res)

    # ---- end to end: pinned host images in, records + all point lists out, every step -------------------------
    def e2e_steps(self, n, ev=None):
        ctx, B = self.ctx, self.B
        out = None
        if ev:
            ev[0].record(self.stream)
        D = self.depth                                         # submissions in flight: the upload of step s + D - 1 is queued
        for k in range(min(D - 1, n)):                         # before the host waits for step s, so neither the host's enqueue
            ctx.batch_submit(self.arr, (k % D) * B, self.pitch)  # time nor the H2D copy sits between two steps of the GPU
        for s in range(n):
            if s + D - 1 < n:
                ctx.batch_submit(self.arr, ((s + D - 1) % D) * B, self.pitch)
            slot = (s % D) * B
            out = ctx.batch_wait(slot, B, raw=True)            # the records as one structured array (no per-record Python objects)
            if self.full_outputs:                              # what matchingFeatures / trackingFrame2Frame hand back
                self.last_outputs = [ctx.batch_outputs(slot + u, out[u], into=self.into[s % D][u]) for u in range(B)]
            if self.gather is not None:                        # result gather: fixed-size records over NCCL, non-blocking
                self.gather.post_step(slot, out, self.my_units)
        if self.gather is not None:
            self.tables = self.gather.drain()                  # the last tables arrive inside the timed region
        if ev:
            ev[1].record(self.stream)
        return ctx.records_to_dicts(out)

    def measure_e2e(self, steps, warmup, full_outputs=True, blocks=1):
        self.full_outputs = full_outputs
        self.ctx.set_option("batch_outputs", 1 if full_outputs else 0)
        self.e2e_steps(max(2, warmup))
        self.torch.cuda.synchronize()
        ms, walls, res = [], [], None
        for _ in range(blocks):
            t, w, res = self._timed(self.e2e_steps, steps)
            ms.append(t); walls.append(w)
        if full_outputs and self.last_outputs:
            self.d2h_outputs = self.B * self.last_outputs[0]["d2h_bytes"]
        return ms, walls, res


class NativeGather:
    """Record gather through the library's own C-ABI (vo_dist_*: every step posts a device snapshot of the waited submission's
    records; one in-place ncclAllGather + one D2H into pinned memory per 4 posts; nothing blocks until VO_DIST_DEPTH posts are
    outstanding, and a submission that refills the slots never waits for another rank)."""
    kind = "C-ABI vo_dist_gather_post / vo_dist_gather_wait (NCCL resolved with dlopen inside libvo_b200.so): per-step device snapshot, one all-gather per 4 steps, up to 8 posts outstanding"
    DEPTH = 8                                   # VO_DIST_DEPTH, include/vo_b200.h

    def __init__(self, ctx, B):
        self.ctx, self.B, self.outstanding, self.tables = ctx, B, 0, []

    def _harvest(self):
        self.tables.append(self.ctx.dist_gather_wait(self.B, raw=True))     # one array, not world x B dicts
        self.outstanding -= 1

    def post_step(self, slot, out, my_units):
        if self.outstanding == self.DEPTH:
            self._harvest()
        self.ctx.dist_gather_post(slot, self.B)
        self.outstanding += 1

    def drain(self):
        while self.outstanding:
            self._harvest()
        out, self.tables = self.tables, []
        return out


class TorchGather:
    """Fallback when the host has no loadable NCCL for the C-ABI path: torch.distributed all_gather on a side stream."""
    kind = "torch.distributed all_gather_into_tensor on a side stream (visual_odom_b200/dist.py AsyncRecordGather)"

    def __init__(self, n_units):
        from visual_odom_b200 import dist as vd
        self.vd, self.g = vd, vd.AsyncRecordGather(n_units, device="cuda")

    def post_step(self, slot, out, my_units):
        self.g.post([self.vd.result_to_record(r) for r in out], my_units)

    def drain(self):
        return self.g.drain()


def bind_to_gpu_numa_node(torch, index):
    """Multi-rank runs: keep this rank's host threads -- and therefore the pinned staging it allocates next, which the kernel
    places on the allocating thread's node -- on the NUMA node its GPU hangs off, so the per-step H2D / D2H copies do not cross
    the socket interconnect.  Pure host plumbing (sysfs + sched_setaffinity); returns what was done for the JSON line."""
    try:
        pr = torch.cuda.get_device_properties(index)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return {"node": None, "why": "sysfs reports no NUMA node for " + bdf}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"node": node, "why": "no allowed CPU on that node"}
        os.sched_setaffinity(0, cpus)
        return {"node": node, "cpus": len(cpus), "pci": bdf}
    except Exception as e:
        return {"node": None, "why": str(e)[:100]}


def lk_profile_constants():
    """ncu-derived constants of the LK kernel (committed under profiles/, refreshed per round): DRAM traffic per launch,
    issue-slot utilisation and warp instructions per feature-ring."""
    tp = os.path.join(ROOT, "profiles", "lk_traffic.json")
    try:
        return json.load(open(tp))
    except Exception:
        return {}


# ------------------------------------------------------------------------------------------------
def main():
    global W_IMG, H_IMG
    args = parse()
    W_IMG, H_IMG = args.width, args.height
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from visual_odom_b200 import synth
    from visual_odom_b200.capi import Context

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: this library has no CPU fallback")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(torch, local_rank) if world > 1 and os.environ.get("VO_BENCH_NUMA", "1") != "0" else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from visual_odom_b200 import dist as vd
    B = args.units
    # work-queue scatter: rank 0 owns the unit table (seeds), broadcast over NCCL; unit u -> rank u mod world
    table = vd.broadcast_unit_table(np.arange(world * B) if rank == 0 else np.zeros(world * B, np.int64), device="cuda")
    my_units = vd.unit_assignment(world * B, world)[rank]
    seeds = [int(table[u]) for u in my_units]
    cal = synth.KITTI00 if args.calib == "kitti" else synth.ZED
    units = [synth.stereo_unit(W_IMG, H_IMG, s, cal=cal) for s in seeds]

    def pin_units(us, w, h):
        out = []
        for u in us:                    # pinned host copies of the images (what a capture / decode thread would hand over)
            d = {}
            for k in ("l0", "r0", "l1", "r1"):
                t = torch.empty((h, w), dtype=torch.uint8, pin_memory=True)
                t.numpy()[:] = u[k]
                d[k] = t.numpy()
            d["_keep"] = None
            out.append(d)
        return out

    pinned = pin_units(units, W_IMG, H_IMG)
    ctx = Context(local_rank, max_features=max(2048, args.features), max_units=E2E_DEPTH * B)
    stream = torch.cuda.Stream()          # a real (non-default) stream shared by torch's events and the library's kernels
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    for opt in ("graphs", "priorities", "batch_graphs", "lk_span", "lk_ctas_per_sm", "lk_quota", "sm_partition"):   # A/B switches, e.g. VO_OPT_LK_SPAN=16
        if os.environ.get("VO_OPT_" + opt.upper()) is not None:
            ctx.set_option(opt, float(os.environ["VO_OPT_" + opt.upper()]))
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    gather = None
    if world > 1 and os.environ.get("VO_BENCH_GATHER", "1") != "0":       # =0: diagnostic only (how much the collective costs)
        try:                               # NCCL unique id: made by rank 0 inside the library, broadcast out of band
            uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                uid.copy_(torch.from_numpy(ctx.dist_unique_id()))
            dist.broadcast(uid, src=0)
            ctx.dist_init(uid.cpu().numpy(), rank, world)
            gather = NativeGather(ctx, B)
        except Exception as e:
            if rank == 0:
                print(f"bench: C-ABI gather unavailable ({str(e)[:120]}), using torch.distributed", file=sys.stderr)
            gather = TorchGather(world * B)
    P = units[0]
    pt = Point(ctx, torch, stream, flush, pinned, args.features, B, W_IMG, H_IMG, P["P_l"], P["P_r"], barrier, world, gather, my_units)
    BLOCKS = 5                            # the K-step timed region is repeated and the median block reported (a block is ~40 ms)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms_res, res, launches = pt.measure_resident(args.steps, args.warmup, BLOCKS)
    lk_avg_ms, lk_ms, t_single_ms, feats_per_launch = pt.measure_lk_alone(args.steps, args.warmup)
    ms_e2e, wall_e2e, res_e2e = pt.measure_e2e(args.steps, args.warmup, True, BLOCKS)
    clocks = sampler.stop() if sampler else None
    ms_sum, _w, res_sum = pt.measure_e2e(args.steps, args.warmup, False, 1)       # records only (round-1 definition of e2e)

    # ---- parity on hardware: one unit of THIS rank against cv2 through the reference glue (outside the timed region) ----
    t_or = time.perf_counter()
    last_slot_unit = 0                                         # unit 0 of the rank's range, outputs of the last e2e step
    ref = reference_unit_outputs(units[last_slot_unit], args.features)
    bad = check_against_oracle(pt.last_outputs[last_slot_unit], res_e2e[last_slot_unit], ref)
    oracle_s = time.perf_counter() - t_or
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, res_e2e, pt.last_outputs, args.features)
    gather_ok = True
    if world > 1 and getattr(pt, "tables", None):          # the gathered table holds this rank's records where they belong
        last = pt.tables[-1]
        if isinstance(gather, NativeGather):
            mine = last[rank * B:(rank + 1) * B]
            gather_ok = len(last) == world * B and all(a["n_inliers"] == b["n_inliers"] and np.array_equal(a["tvec"], b["tvec"])
                                                       for a, b in zip(mine, res_e2e))
        else:
            gather_ok = all(int(last[u][4]) == res_e2e[i]["n_inliers"] for i, u in enumerate(my_units))
    ok_t = torch.tensor([0.0 if (bad or not gather_ok) else 1.0], dtype=torch.float64, device="cuda")

    # max over ranks (device-timed), block by block
    tt = torch.tensor(ms_res + ms_e2e + ms_sum + [lk_ms, float(feats_per_launch)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(ok_t, op=dist.ReduceOp.MIN)
    tt = tt.cpu().numpy()
    ms_res, ms_e2e, ms_sum = list(tt[:BLOCKS]), list(tt[BLOCKS:2 * BLOCKS]), float(tt[2 * BLOCKS])
    parity_ok = bool(ok_t.item() >= 1.0)
    t_dev_ms, t_e2e_ms = _median(ms_res), _median(ms_e2e)

    if rank == 0:
        frames = world * B * args.steps
        value = frames / (t_dev_ms * 1e-3)
        e2e_value = frames / (t_e2e_ms * 1e-3)
        peak, peak_src = peaks()
        prof = lk_profile_constants()

        def roofline_of(lk_avg, nfeat):
            alg = LK_BYTES_PER_FEATURE * nfeat
            ach = alg / (lk_avg * 1e-3) / 1e9 if lk_avg > 0 else 0.0
            return alg, ach

        alg_bytes, achieved = roofline_of(lk_avg_ms, feats_per_launch)
        # ---- the other BASELINE.json configs on the same box, N = 1: feature sweep, 1080p / 4000, a single pair, a sequence ----
        sweep, single_pair, seq = [], None, None
        if world == 1 and args.sweep:
            try:
                ctx.close()
                ctx = Context(local_rank, max_features=8192, max_units=E2E_DEPTH * B)
                ctx.set_stream(stream.cuda_stream)

                def run_point(us_pinned, feats, b, w, h, Pm, steps=10):
                    q = Point(ctx, torch, stream, flush, us_pinned[:b], feats, b, w, h, Pm["P_l"], Pm["P_r"], barrier, 1)
                    r_ms, r_res, _l = q.measure_resident(steps, 3, 3)
                    lk_a, _lm, t_s, nf = q.measure_lk_alone(steps, 3)
                    e_ms, _ww, _er = q.measure_e2e(steps, 3, True, 3)
                    alg, ach = roofline_of(lk_a, nf)
                    return {"width": w, "height": h, "features": feats, "units_per_step": b, "steps": steps,
                            "value_fps": b * steps / (_median(r_ms) * 1e-3), "e2e_fps": b * steps / (_median(e_ms) * 1e-3),
                            "lk_avg_launch_ms": lk_a, "lk_algorithmic_GBps": ach, "lk_frac": ach / peak,
                            "lk_us_per_feature_ring": 1e3 * lk_a / max(nf, 1), "n_valid": [r["n_valid"] for r in r_res][:4]}

                for nf in (500, 1000, 2000, 4000, 8000):        # BASELINE.json configs[4]
                    sweep.append(run_point(pinned, nf, B, W_IMG, H_IMG, P))
                single_pair = run_point(pinned, args.features, 1, W_IMG, H_IMG, P, steps=20)     # configs[1]: one pair per step
                zu = [synth.stereo_unit(1920, 1080, 50 + i, cal=synth.ZED) for i in range(4)]     # configs[2]
                sweep.append(dict(run_point(pin_units(zu, 1920, 1080), 4000, 4, 1920, 1080, zu[0]), calib="zed"))
                if args.sequence > 0:
                    W0, H0 = W_IMG, H_IMG
                    seq = sequence_mode(ctx, torch, cal, args.sequence)
            except Exception as e:           # a side measurement must never cost the headline line
                sweep.append({"error": str(e)[:300]})
        if world == 1:
            m = cpu_reference_measure(units, args, seconds_per_mode=args.cpu_seconds, reps=3)
            cpu = {"value": m["best"]["value"], "unit": "frames/s", "cores": m["best"]["cores"], "kind": "port",
                   "sample": cpu_sample_text(m), "sequential": m["sequential"], "pool": m["pool"]}
        else:                                    # the host baseline is an N = 1 measurement (see --impl reference)
            cpu = {"value": None, "unit": "frames/s", "cores": 0, "kind": "port", "sample": "not measured at N > 1 (rank 0 at N = 1 only)"}
        d2h_records = B * 152
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t_dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8/i32 fixed point + f32 (LK), f64 (pose)", "data": "synthetic",
            "config": workload_config(args, world),
            "timed_blocks_ms": {"resident": [round(x, 3) for x in ms_res], "e2e": [round(x, 3) for x in ms_e2e],
                                "note": f"the {args.steps}-step timed region is run {BLOCKS} times (barrier + synchronize on both sides "
                                        "of every block, max over ranks per block); value / e2e use the median block"},
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": B * 4 * W_IMG * H_IMG + B * 32,
                    "d2h_bytes_per_step": d2h_records + pt.d2h_outputs, "ms_per_step": t_e2e_ms / args.steps,
                    "wall_ms_per_step": 1e3 * _median(wall_e2e) / args.steps,
                    "mode": f"vo_batch_submit / vo_batch_wait / vo_batch_outputs, {E2E_DEPTH} submissions of units_per_gpu in flight; every step's H2D "
                            "(4 images per unit from pinned host memory), kernels, and D2H of the result records AND of every unit's point "
                            "lists (4 x n_valid points, tracked-feature indices, points3D, inlier list: one packed copy per submission) "
                            "are inside the timed region" + ("; the NCCL all-gather of the records runs non-blocking on a side stream and "
                                                             "is drained inside the timed region (" + gather.kind + ")" if gather is not None else
                                                            ("; record gather DISABLED by VO_BENCH_GATHER=0 (diagnostic run)" if world > 1 else "")),
                    "l2": "no flush on this path: every step's inputs are new bytes arriving over PCIe (the resident path flushes instead)",
                    "host_numa_binding": numa,
                    "summary_only": {"value": frames / (ms_sum * 1e-3), "d2h_bytes_per_step": d2h_records,
                                     "note": "round-1 definition: result records only"},
                    "equals_resident_results": all(a["n_inliers"] == b["n_inliers"] and np.array_equal(a["tvec"], b["tvec"])
                                                   for a, b in zip(res_e2e, res)),
                    "single_pair": single_pair, "sequence": seq},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "k_lk_ring", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": prof.get("dram_bytes_per_launch"), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "features_per_launch": feats_per_launch,
                         "avg_launch_ms": lk_avg_ms, "lk_share_of_step": lk_ms / t_single_ms if t_single_ms else None,
                         "single_stream_ms_per_step": t_single_ms / args.steps,
                         "issue_frac": prof.get("issue_active_frac"),
                         "warp_inst_per_feature_ring": prof.get("warp_inst_per_feature_ring"),
                         "profile_source": prof.get("source"),
                         "sweep": sweep,
                         "note": "algorithmic bytes per SURVEY.md 8(d); the kernel is issue bound (pyramids are L2 resident), see DESIGN.md; "
                                 "issue_frac / warp_inst_per_feature_ring come from the committed ncu capture named in profile_source"},
            "cpu_baseline": cpu,
            "clocks": clocks,
            "parity": {"vs_oracle": parity_ok, "units_checked": world, "mismatches_rank0": bad, "gathered_records_ok_rank0": gather_ok,
                       "oracle": "cv2 4.13.0 through oracle/ref_path.py (the reference's glue), one unit per rank, outside the timed region",
                       "oracle_seconds_rank0": oracle_s,
                       "n_valid": [r["n_valid"] for r in res], "n_inliers": [r["n_inliers"] for r in res]},
        }
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    if not parity_ok:
        raise SystemExit(3)


if __name__ == "__main__":
    main()
