#!/usr/bin/env python
"""bench.py — front-end frames/s of the B200-native PL-VIWO visual front end (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload at every N: BASELINE.json configs[4] — 64 independent camera streams, each the configs[1] front end
(synthetic KAIST-shaped 1280x560 mono, point + line front end, 400 points, 5x5 grid, maxLevel 4, 15x15 window),
stream s on rank s mod N (pl-viwo_b200/shard.py).  Streams never exchange data: no collective on the data path; NCCL
only carries the barrier and the SUM(frames) / MAX(ms) reduction.

A STEP is a block of FRAMES_PER_STEP frames of EVERY stream through the whole point + line front end.  Before the timed
region the pipeline is filled AND DRAINED (every submitted frame collected, device synchronised); the timed region then
submits and collects exactly steps x FRAMES_PER_STEP frames per stream between two CUDA events, so every counted
frame's copies, kernels and result read-back happen inside it (pipeline fill and drain included).

  value  : frames/s, frames already resident in HBM (device pointers handed to the library; the resident sequences
           are far larger than L2, every frame is read from HBM)
  e2e    : the same from pinned HOST frames through the C ABI: H2D of every frame and D2H of every result row inside
           the timed region
  roofline / cpu_baseline / clocks : see DESIGN.md "Measurement"
--dump-outputs DIR writes, after the timed steps, the rows the resident pass returned for the last frame of every stream
(engine_rows / dump_outputs below).  The inputs are seeded, so two builds run with the same arguments can be compared
file by file.
--impl reference times the reference's CPU path on the host cores: the oracle's restatement of TrackKLT / TrackLSD
driving the real OpenCV kernels (cv2), one process per core group over independent streams (the reference itself needs
OpenCV C++ / Eigen / ROS headers and cannot be compiled in this image).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before the CUDA context exists (INTEGRATION.md)

WORKLOAD = dict(width=1280, height=560, num_features=400, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10,
                pyr_levels=4, win_size=15)
N_STREAMS = int(os.environ.get("PLVIWO_BENCH_STREAMS", "64"))   # 64 = BASELINE.json configs[4]; the override is for experiments
SEQ_FRAMES = 64          # distinct frames per stream, played forwards and backwards (ping-pong: no jump at the wrap)
FRAMES_PER_STEP = 32
METRIC = "front-end frames/sec @1280x560"
WORKLOAD_NAME = ("BASELINE.json configs[4]: 64 independent camera streams sharded s mod N, each the configs[1] front end "
                 "(synthetic KAIST-shaped 1280x560 mono, point+line, 400 pts, 5x5 grid, maxLevel 4, win 15)")
CACHE_DIR = os.environ.get("PLVIWO_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "plviwo_bench_cache"))
KERNEL_OF_STAGE = {"hist": "k_hist", "eq_pyr1": "k_eq_pyr1", "pyr_rest": "k_pyr_down", "fast": "k_fast", "subpix": "k_corner_subpix",
                   "lk": "k_lk15", "canny": "k_canny", "fld_walk": "k_fld_walk_cc", "fld_ccl": "k_ccl_merge", "fld_seg": "k_fld_segments"}


def bench_config(world: int) -> dict:
    """The workload description: IDENTICAL in both arms (the driver compares the dicts)."""
    return {"workload": WORKLOAD_NAME, "streams": N_STREAMS, "gpus": world, "frames_per_step": FRAMES_PER_STEP,
            "frames_per_step_note": "a step = %d frames of every stream" % FRAMES_PER_STEP,
            "stream_to_gpu": "stream s -> rank s mod N, seed 1000 + s", "sequence_frames": SEQ_FRAMES,
            "sequence_order": "ping-pong",
            "cache": "inputs larger than L2: %d streams x %d distinct frames x 0.72 MB (2.9 GB per job) are cycled, every frame is read "
                     "from HBM (GPU arm) / DRAM (reference arm); no L2 flush between steps" % (N_STREAMS, SEQ_FRAMES),
            **{k: v for k, v in WORKLOAD.items()}}


def frame_index(i: int, n: int = SEQ_FRAMES) -> int:
    """Ping-pong order over the n stored frames: 0 .. n-1, n-2 .. 1, 0 .. (continuous motion, no jump)."""
    if n <= 1:
        return 0
    period = 2 * (n - 1)
    k = i % period
    return k if k < n else period - k


def algorithmic_bytes(n_lk_pts: float, cfg=WORKLOAD) -> dict:
    """SURVEY.md 8(d): every stage reads its input once and writes its output once (per frame)."""
    N = cfg["width"] * cfg["height"]
    L, w = cfg["pyr_levels"], cfg["win_size"]
    sizes, ww, hh = [], cfg["width"], cfg["height"]
    for _ in range(L + 1):
        sizes.append(ww * hh)
        ww, hh = (ww + 1) // 2, (hh + 1) // 2
    b = {
        "hist": N,                                            # read the frame
        "eq_pyr1": N + N + sizes[1] + N // 4,                 # read frame, write level 0, level 1, half-res image
        "pyr_rest": sum(sizes[l - 1] + sizes[l] for l in range(2, L + 1)),
        "fast": N,                                            # worst case: every cell valid
        "canny": N // 4 + N // 4,                             # Canny read + write (one byte per half-res pixel, SURVEY 8d)
        "fld_walk": N // 4,                                   # chain walk: every half-res pixel read once
        "fld_ccl": 0, "fld_seg": 0,                           # implementation artefacts of the parallel walk: no SURVEY bytes
        "lk": n_lk_pts * (L + 1) * ((w + 3) ** 2 + (w + 1) ** 2),
        "subpix": 0,
    }
    b["frame_total"] = 3 * N + sum(sizes[l - 1] + sizes[l] for l in range(1, L + 1)) + N + (N + 4 * (N // 4)) + b["lk"]
    return b


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index: int):
        self.path = tempfile.mktemp(suffix=".csv")
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.f = open(self.path, "w")
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                       "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1]))
                    mx.append(float(c[2]))
                except ValueError:
                    continue
                for nme, v in zip(names, c[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


# --------------------------------------------------------------------------------------------- synthetic sequences
def _gen_stream(args):
    """(seed, n) -> uint8 array (n, H, W); cached on disk so the four scaling runs and the reference arm of one round
    generate each stream once.  Runs in worker processes (no CUDA there)."""
    seed, n = args
    path = os.path.join(CACHE_DIR, "seq_%d_%dx%d_%d.npy" % (seed, WORKLOAD["width"], WORKLOAD["height"], n))
    try:
        a = np.load(path)
        if a.shape == (n, WORKLOAD["height"], WORKLOAD["width"]):
            return a
    except Exception:
        pass
    import plviwo_b200  # noqa: F401
    from plviwo_b200 import synth
    seq = synth.SynthSequence(seed=seed, width=WORKLOAD["width"], height=WORKLOAD["height"], n_frames=300)
    a = np.stack([seq.frame(t) for t in range(n)])
    try:
        os.makedirs(CACHE_DIR, exist_ok=True)
        tmp = path + ".%d.tmp" % os.getpid()
        with open(tmp, "wb") as f:
            np.save(f, a)
        os.replace(tmp, path)
    except Exception:
        pass
    return a


def stream_meta(seed: int):
    """Calibration / timestamps / vanishing points of a stream (the generator's, without building its canvas)."""
    import plviwo_b200  # noqa: F401
    from plviwo_b200 import synth
    sc = WORKLOAD["width"] / 1280.0
    K = tuple(v * sc for v in synth.KAIST_K)
    vps = [(1.0e5, 263.0 * sc), (608.0 * sc, -1.0e5), (608.0 * sc, 263.0 * sc)]
    return K, synth.KAIST_D, vps


def timestamp(i: int) -> float:
    return 1.0 + 0.1 * i


def generate_streams(seeds, n, workers):
    """Frames of several streams, generated in parallel worker processes."""
    import multiprocessing as mp
    if len(seeds) == 1 or workers <= 1:
        return [_gen_stream((s, n)) for s in seeds]
    with mp.get_context("spawn").Pool(min(workers, len(seeds))) as pool:
        return pool.map(_gen_stream, [(s, n) for s in seeds])


# ----------------------------------------------------------------------------------------------- CPU arm
def _cpu_worker(args):
    """One process = one core group: the oracle front end (reference glue restated, real OpenCV kernels) over one stream.
    Returns timing of `frames` frames after `warm` warm-up frames."""
    seed, threads, warm, frames, want_rows, barrier_file = args
    import cv2
    cv2.setNumThreads(threads)
    from oracle import frontend as ofe
    from oracle import cvops
    data = _gen_stream((seed, SEQ_FRAMES))
    K, D, vps = stream_meta(seed)
    in_kernels = [0.0]

    class TimedOps:
        """oracle.cvops with the time spent INSIDE the OpenCV calls (and the FastLineDetector / std::sort shim) added up:
        the rest of a frame is the Python restatement of the reference's glue, which the C++ reference does much faster."""

        def __getattr__(self, name):
            f = getattr(cvops, name)
            if not callable(f):
                return f

            def timed(*a, **k):
                t = time.perf_counter()
                r = f(*a, **k)
                in_kernels[0] += time.perf_counter() - t
                return r
            return timed

    kw = {k: v for k, v in WORKLOAD.items() if k not in ("width", "height")}
    fe = ofe.FrontEnd(ofe.FeConfig(K=K, D=D, **kw), ops=TimedOps())
    rows = []
    for i in range(warm):
        p, _ = fe.feed(timestamp(i), data[frame_index(i)], None, vps)
        if want_rows:
            rows.append(np.array([(r.id, r.u, r.v) for r in p], np.float64).reshape(-1, 3))
    # all workers of a mode start their timed part together (file-system barrier: a spawn pool has no shared objects)
    if barrier_file:
        open(barrier_file + ".%d" % os.getpid(), "w").close()
        n_expected = int(barrier_file.rsplit("_", 1)[1])
        d, b = os.path.split(barrier_file)
        t_end = time.time() + 120
        while sum(1 for f in os.listdir(d) if f.startswith(b + ".")) < n_expected and time.time() < t_end:
            time.sleep(0.002)
    in_kernels[0] = 0.0
    per = []
    t0 = time.perf_counter()
    for k in range(frames):
        i = warm + k
        a = time.perf_counter()
        p, _ = fe.feed(timestamp(i), data[frame_index(i)], None, vps)
        per.append(time.perf_counter() - a)
        if want_rows:
            rows.append(np.array([(r.id, r.u, r.v) for r in p], np.float64).reshape(-1, 3))
    t1 = time.perf_counter()
    # what the port does differently from the C++ reference inside OpenCV: cv2.calcOpticalFlowPyrLK (image form) builds
    # both pyramids per call where the reference builds ONE per frame (TrackKLT.cpp:71) — one build too many; and the
    # port equalises once where the reference equalises twice (TrackKLT.cpp:59 and TrackLSD.cpp:83) — one too few
    eq = cv2.equalizeHist(data[0])
    t = time.perf_counter()
    for _ in range(10):
        cv2.buildOpticalFlowPyramid(eq, (WORKLOAD["win_size"],) * 2, WORKLOAD["pyr_levels"], withDerivatives=False)
    t_pyr = (time.perf_counter() - t) / 10
    t = time.perf_counter()
    for _ in range(10):
        cv2.equalizeHist(data[1])
    t_eq = (time.perf_counter() - t) / 10
    return dict(t0=t0, t1=t1, frames=frames, kernel_s=in_kernels[0], p50_ms=1e3 * float(np.median(per)), t_pyr=t_pyr, t_eq=t_eq,
                rows=rows if want_rows else None)


def run_cpu_mode(procs: int, threads: int, warm: int, frames: int, want_rows=False):
    """`procs` worker processes (independent streams, seeds 1000 ..), `threads` OpenCV threads each."""
    import multiprocessing as mp
    bdir = tempfile.mkdtemp(prefix="plviwo_bar_")
    bfile = os.path.join(bdir, "go_%d" % procs)
    jobs = [(1000 + p, threads, warm, frames, want_rows and p == 0, bfile) for p in range(procs)]
    if procs == 1:
        res = [_cpu_worker(jobs[0][:5] + (None,))]
    else:
        with mp.get_context("spawn").Pool(procs) as pool:
            res = pool.map(_cpu_worker, jobs)
    try:
        for f in os.listdir(bdir):
            os.unlink(os.path.join(bdir, f))
        os.rmdir(bdir)
    except Exception:
        pass
    # perf_counter is CLOCK_MONOTONIC: comparable across the processes of one box
    elapsed = max(r["t1"] for r in res) - min(r["t0"] for r in res)
    tot = sum(r["frames"] for r in res)
    busy = sum(r["t1"] - r["t0"] for r in res)
    kern = sum(r["kernel_s"] for r in res)
    corr = sum((r["t1"] - r["t0"]) - r["frames"] * (r["t_pyr"] - r["t_eq"]) for r in res)
    return dict(procs=procs, threads=threads, fps=tot / elapsed, elapsed_s=elapsed, frames=tot,
                p50_ms=float(np.median([r["p50_ms"] for r in res])),
                kernel_ms=1e3 * kern / tot, glue_ms=1e3 * (busy - kern) / tot,
                kernels_only_fps=tot / elapsed * busy / kern if kern > 0 else None,
                corrected_fps=tot / elapsed * busy / corr if corr > 0 else None,
                rows=res[0]["rows"])


def cpu_modes(cores: int):
    """OpenCV thread counts 1, 4 (the reference's own choice, test_tracking.cpp:115) and all, processes filling the box."""
    modes = [(max(cores, 1), 1)]
    if cores >= 4:
        modes.append((cores // 4, 4))
    modes.append((1, cores))
    return modes


def run_cpu_arm(frames_per_proc: int, warm: int, sweep_frames: int, want_rows=False):
    """Thread sweep on a short sample, then the timed run in the best mode."""
    cores = len(os.sched_getaffinity(0))
    _gen_stream((1000, SEQ_FRAMES))
    sweep = []
    for procs, threads in cpu_modes(cores):
        generate_streams([1000 + p for p in range(procs)], SEQ_FRAMES, min(procs, cores))
        r = run_cpu_mode(procs, threads, 8, sweep_frames)
        sweep.append({k: r[k] for k in ("procs", "threads", "fps", "p50_ms", "kernel_ms", "glue_ms", "kernels_only_fps", "corrected_fps")})
    best = max(sweep, key=lambda r: r["fps"])
    r = run_cpu_mode(best["procs"], best["threads"], warm, frames_per_proc, want_rows)
    return r, sweep, cores


def cpu_baseline_dict(r, sweep, cores, label):
    return {"value": r["fps"], "unit": "frames/s", "cores": r["procs"] * r["threads"], "kind": "port",
            "host_cores": cores, "processes": r["procs"], "opencv_threads_per_process": r["threads"],
            "sample": "%s: %d frames on each of %d independent streams (seeds 1000..), one process per stream with %d OpenCV "
                      "thread(s); oracle/frontend.py (reference glue restated in Python) driving the real OpenCV kernels via "
                      "cv2; per frame %.2f ms inside OpenCV / the FLD shim + %.2f ms Python glue"
                      % (label, r["frames"] // r["procs"], r["procs"], r["threads"], r["kernel_ms"], r["glue_ms"]),
            "kernels_only_value": r["kernels_only_fps"],
            "kernels_only_note": "frames/s if the reference's glue cost nothing: the upper bound for any CPU implementation "
                                 "built on these OpenCV kernels, and the denominator README / DESIGN quote",
            "pyramid_corrected_value": r["corrected_fps"],
            "pyramid_corrected_note": "per frame minus one cv::buildOpticalFlowPyramid (the image form of calcOpticalFlowPyrLK "
                                      "builds two per call, the reference one per frame, TrackKLT.cpp:71) plus one "
                                      "cv::equalizeHist (the reference equalises twice, TrackLSD.cpp:83), both timed in the run",
            "thread_sweep": sweep, "p50_ms_per_frame": r["p50_ms"]}


# ----------------------------------------------------------------------------------------------- GPU arm
class HandleEngine:
    """One FeHandle per stream (plviwo_fe_create), each driven by its own host thread through plviwo_fe_play — the
    submit / collect loop inside the library, so the Python GIL is not part of the measurement."""
    name = "handles"

    def __init__(self, fe_mod, dev, metas, lookahead):
        self.fe = fe_mod
        self.h = [fe_mod.FrontEnd(fe_mod.default_config(K=K, D=D, lookahead=lookahead, **WORKLOAD), device=dev) for K, D, _ in metas]
        self.metas = metas
        self.lookahead = lookahead

    def run(self, first, n_frames, ptrs, pitch, on_device, frame_index=None):
        """Frames first .. first + n_frames - 1 of every stream; returns when every frame has been collected."""
        done = [0] * len(self.h)
        errs = []

        fi = frame_index or globals()["frame_index"]

        def drive(k):
            try:
                idx = [fi(first + i) for i in range(n_frames)]
                ts = [timestamp(first + i) for i in range(n_frames)]
                vps = [self.metas[k][2]] * n_frames
                st = self.h[k].play(ts, [ptrs[k][t] for t in idx], stride=pitch, on_device=on_device, vanishing_points=vps)
                done[k] = int(st.frames)
            except Exception as e:   # noqa: BLE001
                errs.append(e)
        th = [threading.Thread(target=drive, args=(k,)) for k in range(len(self.h))]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errs:
            raise errs[0]
        return sum(done)

    def counters(self, reset=False):
        tot = {"kernel_launches_total": 0, "h2d_bytes": 0, "d2h_bytes": 0, "frames": 0}
        for h in self.h:
            st = h.stage_times(reset=reset)
            for k in tot:
                tot[k] += st[k]
        return tot

    def stage_times(self, reset=False):
        return [h.stage_times(reset=reset) for h in self.h]

    def enable_timing(self, on):
        for h in self.h:
            h.enable_timing(on)

    def close(self):
        for h in self.h:
            h.close()


def make_engine(kind, fe_mod, dev, metas):
    if kind == "group":
        return fe_mod.GroupEngine(fe_mod, dev, metas, WORKLOAD)
    la = int(os.environ.get("PLVIWO_BENCH_LA", "16" if len(metas) > 2 else "48"))
    return HandleEngine(fe_mod, dev, metas, la)


def timed_pass(torch, dist, eng, first, n_frames, ptrs, pitch, on_device):
    """The timed region: barrier + synchronise, event, submit and collect n_frames of every stream, synchronise, event."""
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    eng.counters(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    t0 = time.perf_counter()
    frames = eng.run(first, n_frames, ptrs, pitch, on_device, frame_index=frame_index)
    torch.cuda.synchronize()
    ev1.record()
    ev1.synchronize()
    wall = time.perf_counter() - t0
    c = eng.counters(reset=False)
    if dist is not None:
        dist.barrier()
    return dict(ms=float(ev0.elapsed_time(ev1)), wall_ms=1e3 * wall, frames=frames, counters=c)


def engine_rows(eng):
    """Per stream (point rows, line rows, points on lines) of the last frame the engine played: what a caller of
    plviwo_fe_play / plviwo_fe_group_play reads once the call returns."""
    if eng.name == "group":
        return [(eng.g.point_rows(s),) + eng.g.line_rows(s) for s in range(eng.g.n)]
    return [(h.point_rows(),) + h.line_rows() for h in eng.h]


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, streams, rows, suffix=""):
    """Writes `rows` (engine_rows) as out_dir/<name><suffix>.npy.  Ids and counts go to float64 arrays (exact below 2^53) whose
    column 0 is the stream index, coordinates to float32 arrays with the same row order, so that ids can be compared exactly
    and coordinates with a tolerance."""
    def stream_col(parts):
        return np.concatenate([np.full(len(p), s, np.float64) for s, p in zip(streams, parts)])

    pts, lines, lpts = ([r[k] for r in rows] for k in range(3))
    P, L, Q = np.concatenate(pts), np.concatenate(lines), np.concatenate(lpts)
    out = {
        "point_ids": np.stack([stream_col(pts), P["id"].astype(np.float64)], 1),
        "point_uv": np.stack([P["u"], P["v"], P["un"], P["vn"]], 1).astype(np.float32),
        "line_ids": np.stack([stream_col(lines)] + [L[k].astype(np.float64) for k in ("id", "D", "n_pts", "pt_offset", "matched")], 1),
        "line_endpoints": np.concatenate([L["line"], L["line_n"]], 1).astype(np.float32),
        "line_point_ids": np.stack([stream_col(lpts), Q["pid"].astype(np.float64)], 1),
        "line_point_uv": np.stack([Q["dist"], Q["u"], Q["v"]], 1).astype(np.float32),
    }
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("bench.py: --dump-outputs would write %d bytes, more than %d" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def parity_against(fe_mod, dev, data, meta, rows_cpu):
    """BASELINE.json's third metric ("KLT px err").  The oracle is the checker here, nothing of it is timed.
    (a) teacher forced over 40 frames: the GPU tracker is loaded with the oracle's state before every frame, so each frame
        is compared on identical inputs (what tests/test_frontend_gpu.py asserts);
    (b) free running: the frames the CPU baseline has just processed through the synchronous drop-in call from the same
        initial state; one flipped status flag changes every later feature id (SURVEY.md 7.3), so id equality is reported
        up to the first frame where the row sets differ."""
    from oracle import frontend as ofe
    K, D, vps = meta
    kw = dict(WORKLOAD)
    okw = {k: v for k, v in kw.items() if k not in ("width", "height")}
    W, H = kw["width"], kw["height"]
    o = ofe.FrontEnd(ofe.FeConfig(K=K, D=D, **okw))
    h = fe_mod.FrontEnd(fe_mod.default_config(K=K, D=D, lookahead=0, **kw), device=dev)
    tf_duv, tf_rows, tf_sym, tf_equal = [], 0, 0, 0
    for t in range(40):
        img = data[frame_index(t)]
        if t > 0:
            k, l = o.klt.get_state(), o.lsd.get_state()
            h.set_state(fe_mod.pack_state(W, H, k["currid"], k["pts_last"], k["ids_last"], k["img_last"], k["mask_last"], l["currid"],
                                          l["lines_last"], l["ids_last"], l["pol_last"]))
        prow, _ = o.feed(timestamp(t), img, None, vps)
        h.feed_new_camera(timestamp(t), img, None, vps, update_db=False)
        got = h.point_rows()
        ids_g = {int(i): k2 for k2, i in enumerate(got["id"])}
        ids_c = {r.id: r for r in prow}
        d = set(ids_g) ^ set(ids_c)
        tf_rows += len(ids_c)
        tf_sym += len(d)
        tf_equal += int(not d and [r.id for r in prow] == [int(i) for i in got["id"]])
        for i in set(ids_g) & set(ids_c):
            a, b = got[ids_g[i]], ids_c[i]
            tf_duv.append(max(abs(float(a["u"]) - b.u), abs(float(a["v"]) - b.v)))
    h.close()
    tf_duv = np.array(tf_duv) if tf_duv else np.zeros(1)
    teacher = {"frames": 40, "frames_rows_identical_ids_and_order": tf_equal, "rows": tf_rows,
               "rows_with_flipped_status": tf_sym, "status_agreement": 1.0 - tf_sym / max(tf_rows, 1),
               "max_duv_px": float(tf_duv.max()), "p99_duv_px": float(np.percentile(tf_duv, 99)),
               "rows_over_0.05px": int((tf_duv > 0.05).sum()),
               "rows_over_0.05px_note": "rows on which cv2's own LK is unstable (tests/test_frontend_gpu.py carve-out: each "
                                        "must match the scalar restatement or be shown chaotic)"}
    out = {"teacher_forced": teacher}
    if rows_cpu:
        h = fe_mod.FrontEnd(fe_mod.default_config(K=K, D=D, lookahead=0, **kw), device=dev)
        first_div, eq_frames, duv, sym = None, 0, [], 0
        for t, want in enumerate(rows_cpu):
            h.feed_new_camera(timestamp(t), data[frame_index(t)], None, vps, update_db=False)
            got = h.point_rows()
            ids_g = {int(i): k for k, i in enumerate(got["id"])}
            ids_c = {int(i): k for k, i in enumerate(want[:, 0])}
            d = set(ids_g) ^ set(ids_c)
            if first_div is None:
                if d:
                    first_div = t
                else:
                    eq_frames += 1
            if first_div is None or t == first_div:
                sym += len(d)
                for i in set(ids_g) & set(ids_c):
                    a, b = got[ids_g[i]], want[ids_c[i]]
                    duv.append(max(abs(float(a["u"]) - b[1]), abs(float(a["v"]) - b[2])))
        h.close()
        duv = np.array(duv) if duv else np.zeros(1)
        out.update({"frames": len(rows_cpu), "frames_ids_identical": eq_frames, "first_frame_with_different_rows": first_div,
                    "rows_compared": int(len(duv)), "max_duv_px": float(duv.max()), "p99_duv_px": float(np.percentile(duv, 99)),
                    "rows_only_on_one_side_at_divergence": sym})
    return out


def pin_to_gpu_numa_node(torch, dev):
    """Keep the rank on the cores of the NUMA node its GPU hangs off, when the platform says which that is."""
    try:
        pr = torch.cuda.get_device_properties(dev)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if len(cpus) >= 4:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--engine", default=os.environ.get("PLVIWO_BENCH_ENGINE", "auto"), choices=["auto", "group", "handles"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the single-stream / synchronous / stereo extras")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the rows of the last frame of every stream as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path, not of --impl reference")
    args.warmup = max(args.warmup, 3)
    # exactly ONE line on stdout: libraries that print banners there (NCCL's version line) are sent to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        if rank != 0:
            return 0
        steps = args.steps
        warm = min(args.warmup, 4) * 4
        # a step of the reference arm = FRAMES_PER_STEP frames on each stream of its bounded sample (one stream per process)
        r, sweep, cores = run_cpu_arm(steps * FRAMES_PER_STEP, warm, 24)
        cb = cpu_baseline_dict(r, sweep, cores, "bounded sample of the 64-stream workload")
        line = {"metric": METRIC, "value": r["fps"], "unit": "frames/s", "n_gpus": args.gpus, "steps": steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * r["elapsed_s"] / steps, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "u8/int32 fixed-point + f32/f64 (OpenCV)", "data": "synthetic", "impl": "reference",
                "config": bench_config(args.gpus),
                "sample_streams": r["procs"], "cpu_baseline": cb,
                "e2e": {"value": r["fps"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "p50_ms_per_frame": r["p50_ms"]}
        emit(line)
        return 0

    import torch
    import plviwo_b200 as fe_mod
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the front end has no CPU fallback (use --impl reference for the CPU arm)")
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        torch.cuda.set_device(local_rank)
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist = dist_mod
    dev = local_rank if world > 1 else 0
    torch.cuda.set_device(dev)
    numa = pin_to_gpu_numa_node(torch, dev)

    # ---- this rank's streams (config 5): s -> rank s mod N, seed 1000 + s
    streams = fe_mod.shard.streams_of_rank(N_STREAMS, rank, world)
    S = len(streams)
    seeds = [fe_mod.shard.seed_of_stream(s) for s in streams]
    cores = len(os.sched_getaffinity(0))
    t_gen = time.perf_counter()
    data = generate_streams(seeds, SEQ_FRAMES, max(1, cores // max(world, 1)))
    t_gen = time.perf_counter() - t_gen
    metas = [stream_meta(s) for s in seeds]
    H, W = WORKLOAD["height"], WORKLOAD["width"]
    # device-resident copy (S x 64 frames x 0.72 MB: 2.9 GB at S = 64, far larger than the 126 MB L2) and a pinned host copy
    d_seq = torch.empty((S, SEQ_FRAMES, H, W), dtype=torch.uint8, device="cuda")
    h_seq = torch.empty((S, SEQ_FRAMES, H, W), dtype=torch.uint8).pin_memory()
    for k in range(S):
        h_seq[k].copy_(torch.from_numpy(data[k]))
    d_seq.copy_(h_seq)
    torch.cuda.synchronize()
    # what the host link gives this process (pinned -> device), for reading the e2e number: every frame crosses it once
    nb = min(S, 8)
    t0 = time.perf_counter()
    d_seq[:nb].copy_(h_seq[:nb], non_blocking=True)
    torch.cuda.synchronize()
    h2d_gbps = nb * SEQ_FRAMES * H * W / (time.perf_counter() - t0) / 1e9
    d_ptrs = [[d_seq[k, t].data_ptr() for t in range(SEQ_FRAMES)] for k in range(S)]
    h_ptrs = [[h_seq[k, t].numpy() for t in range(SEQ_FRAMES)] for k in range(S)]

    kind = args.engine
    if kind == "auto":
        kind = "group" if hasattr(fe_mod, "GroupEngine") else "handles"
    n_timed = args.steps * FRAMES_PER_STEP
    n_warm = max(args.warmup * FRAMES_PER_STEP, 64)

    # ---- resident pass
    eng = make_engine(kind, fe_mod, dev, metas)
    eng.run(0, n_warm, d_ptrs, W, True, frame_index=frame_index)                       # untimed: graph capture, clocks, then DRAINED (run returns when
    torch.cuda.synchronize()                                   # every frame is collected)
    sampler = ClockSampler(dev) if rank == 0 else None
    try:
        res = timed_pass(torch, dist, eng, n_warm, n_timed, d_ptrs, W, True)
    finally:   # the sampler is a child process: never leave it running
        clocks = sampler.stop() if sampler else {}
    if res["counters"]["kernel_launches_total"] == 0 or res["frames"] != n_timed * S:
        raise SystemExit("bench.py: the timed region launched no kernel or lost frames (%r)" % (res,))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, streams, engine_rows(eng), "" if world == 1 else "_rank%d" % rank)
    # ---- per-kernel durations: a short pass with CUDA-event stage timing on
    stage = None
    try:
        eng.enable_timing(True)
        eng.run(n_warm + n_timed, 8, d_ptrs, W, True, frame_index=frame_index)          # timing on: direct launches, first frames
        eng.stage_times(reset=True)
        eng.run(n_warm + n_timed + 8, min(n_timed, 96), d_ptrs, W, True, frame_index=frame_index)
        stage = eng.stage_times(reset=False)
        eng.enable_timing(False)
    except Exception as e:   # noqa: BLE001
        stage = {"error": str(e)}
    eng.close()
    # ---- end to end: the same through the C ABI from pinned HOST frames
    eng = make_engine(kind, fe_mod, dev, metas)
    eng.run(0, n_warm, h_ptrs, W, False, frame_index=frame_index)
    torch.cuda.synchronize()
    res_e2e = timed_pass(torch, dist, eng, n_warm, n_timed, h_ptrs, W, False)
    eng.close()

    extras = {}
    if world == 1 and not args.no_extras:
        try:   # one pipelined stream (configs[1] alone on the GPU)
            e1 = make_engine("handles", fe_mod, dev, metas[:1])
            e1.run(0, 128, d_ptrs[:1], W, True, frame_index=frame_index)
            r1 = timed_pass(torch, None, e1, 128, 600, d_ptrs[:1], W, True)
            extras["single_stream"] = {"value": r1["frames"] / (r1["ms"] * 1e-3), "unit": "frames/s", "frames": r1["frames"],
                                       "api": "plviwo_fe_play on one handle, lookahead %d, frames resident in HBM" % e1.lookahead}
            e1.close()
        except Exception as e:   # noqa: BLE001
            extras["single_stream"] = {"error": str(e)}
        try:   # strict drop-in: synchronous plviwo_fe_feed per frame from host memory
            K, D, vps = metas[0]
            h = fe_mod.FrontEnd(fe_mod.default_config(K=K, D=D, lookahead=0, **WORKLOAD), device=dev)
            for t in range(16):
                h.feed_new_camera(timestamp(t), h_ptrs[0][frame_index(t)], None, vps, update_db=False)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for t in range(16, 216):
                h.feed_new_camera(timestamp(t), h_ptrs[0][frame_index(t)], None, vps, update_db=False)
            extras["sync_feed_fps"] = 200 / (time.perf_counter() - t0)
            h.close()
        except Exception as e:   # noqa: BLE001
            extras["sync_feed_fps"] = {"error": str(e)}

    ms, ms_e2e = res["ms"], res_e2e["ms"]
    frames_rank = res["frames"]
    per_rank = [[ms, ms_e2e, float(frames_rank)]]
    total_frames, total_frames_e2e = frames_rank, res_e2e["frames"]
    launches = res["counters"]["kernel_launches_total"]
    if dist is not None:
        # whole-job numbers: SUM of frames, MAX of elapsed time over the ranks (pl-viwo_b200/shard.py)
        tt = torch.tensor([ms, ms_e2e, float(frames_rank)], device="cuda", dtype=torch.float64)
        allv = [torch.zeros_like(tt) for _ in range(world)]
        dist.all_gather(allv, tt)
        per_rank = [[float(v[0]), float(v[1]), float(v[2])] for v in allv]
        ms, ms_e2e = max(v[0] for v in per_rank), max(v[1] for v in per_rank)
        total_frames = int(round(fe_mod.shard.distributed_throughput(dist, torch, frames_rank, res["ms"], device="cuda") * ms * 1e-3))
        total_frames_e2e = int(sum(v[2] for v in per_rank))
        lt = torch.tensor([float(launches)], device="cuda", dtype=torch.float64)
        dist.all_reduce(lt)
        launches = int(lt[0])
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel (largest cost per frame), live CUDA-event durations
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    roofline = build_roofline(stage, peak, peak_src, total_frames / (ms * 1e-3) / world, res)
    try:   # what the image-domain kernels reach when ONE launch carries a batch of frames' worth of pixels
        AW, AH = 16384, 8192
        t = fe_mod.op_image_kernels_time(AW, AH, 5, device=dev)
        NA = AW * AH
        bytes_ = {"hist": NA, "eq_pyr1": NA + NA + NA // 4 + NA // 4, "fast": NA, "canny": NA // 4 + NA // 4}
        roofline["at_scale"] = {"image": "%dx%d (= %.0f frames of 1280x560 per launch)" % (AW, AH, NA / (1280 * 560.0)),
                                "kernels": {k: {"ms": t[k], "algorithmic_bytes": bytes_[k], "GBps": bytes_[k] / (t[k] * 1e-3) / 1e9,
                                                "frac": bytes_[k] / (t[k] * 1e-3) / 1e9 / peak} for k in t if t[k] > 0}}
    except Exception as e:   # never fatal for the bench line
        roofline["at_scale"] = {"error": str(e)}

    cpu = parity = None
    if not args.no_cpu_baseline and world == 1:
        r, sweep, ncores = run_cpu_arm(160, 8, 16, want_rows=True)
        cpu = cpu_baseline_dict(r, sweep, ncores, "bounded sample of the 64-stream workload")
        try:
            parity = parity_against(fe_mod, dev, data[0], metas[0], r["rows"][:120] if r["rows"] else None)
        except Exception as e:   # an extra, never fatal for the bench line
            parity = {"error": str(e)}

    cfg = bench_config(world)
    line = {
        "metric": METRIC, "value": total_frames / (ms * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8/int32 fixed-point + f32 (LK), f64 (sub-pixel, undistort, RANSAC)", "data": "synthetic",
        "config": cfg,
        "engine": {"kind": eng.name, "streams_per_gpu": S, "frames_timed_per_stream": n_timed, "untimed_frames_per_stream": n_warm,
                   "timed_region": "pipeline drained before the first event; steps x frames_per_step frames of every stream "
                                   "submitted AND collected between the events",
                   "host": {"cores": os.cpu_count(), "rank0_numa_node": numa, "rank0_cpus": len(os.sched_getaffinity(0))},
                   "per_rank_ms": {"resident": [round(v[0], 2) for v in per_rank], "e2e": [round(v[1], 2) for v in per_rank]},
                   "synthesis_s": round(t_gen, 1),
                   "cache": "inputs larger than L2 (%.1f GB of device-resident frames per GPU, every frame read from HBM)"
                            % (S * SEQ_FRAMES * H * W / 1e9)},
        "p50_ms_per_frame": 1e3 / (total_frames / (ms * 1e-3)) if total_frames else None,
        "p50_note": "reciprocal of the whole-job throughput (the batched engine completes frames a tick at a time); the strictly "
                    "synchronous per-frame latency is 1000 / extras.sync_feed_fps ms",
        "klt_parity": parity,
        "e2e": {"value": total_frames_e2e / (ms_e2e * 1e-3), "unit": "frames/s",
                "h2d_bytes_per_step": res_e2e["counters"]["h2d_bytes"] / args.steps,
                "d2h_bytes_per_step": res_e2e["counters"]["d2h_bytes"] / args.steps,
                "api": "pinned host frames through the C ABI (%s), H2D of every frame and D2H of every row inside the timed region" % eng.name,
                "h2d_link_GBps_measured": round(h2d_gbps, 1),
                "h2d_GBps_used": round(total_frames_e2e / world / (ms_e2e * 1e-3) * H * W / 1e9, 1)},
        "gpu_launches": launches,
        "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "extras": extras,
    }
    emit(line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


def build_roofline(stage, peak, peak_src, fps_per_gpu, res):
    """roofline{} of the bench line from the library's CUDA-event stage times (per LAUNCH) of the timing pass."""
    out = {"bound": "hbm", "peak": peak, "unit": "GB/s", "peak_source": peak_src, "traffic": None}
    ab1 = algorithmic_bytes(300.0)
    out["whole_frame"] = {"algorithmic_bytes": ab1["frame_total"], "achieved_GBps": ab1["frame_total"] * fps_per_gpu / 1e9,
                          "frac": ab1["frame_total"] * fps_per_gpu / 1e9 / peak}
    if not stage or isinstance(stage, dict) and "error" in stage:
        out.update(kernel=None, achieved=0.0, frac=0.0, error=(stage or {}).get("error", "no stage times"))
        return out
    if isinstance(stage, dict) and "group" in stage:    # stream group: per-kernel CUDA-event times from the library
        t = stage["group"]
        ab = algorithmic_bytes(300.0)
        # FAST runs on the valid cells of the detection only, as the reference does (Grider_GRID.h:108-125): its algorithmic
        # bytes are the pixels of the cells it ran on (counted by the library), not the whole frame
        n_cells = WORKLOAD["grid_x"] * WORKLOAD["grid_y"]
        fast_frames = t["frames_of"].get("fast", 0)
        fast_frac = min(1.0, t.get("fast_cells", 0) / max(fast_frames * n_cells, 1)) if fast_frames else 1.0
        out["fast_cells_per_frame"] = round(fast_frac * n_cells, 3)
        out["whole_frame"]["algorithmic_bytes"] = ab1["frame_total"] - ab1["fast"] * (1.0 - fast_frac)
        out["whole_frame"]["achieved_GBps"] = out["whole_frame"]["algorithmic_bytes"] * fps_per_gpu / 1e9
        out["whole_frame"]["frac"] = out["whole_frame"]["achieved_GBps"] / peak
        out["whole_frame"]["note"] = ("SURVEY 8(d) bytes of a frame with FAST counted on the %.2f of %d grid cells per frame it ran on "
                                      "(the all-cells figure is %d B)" % (fast_frac * n_cells, n_cells, ab1["frame_total"]))
        bytes_of = {"hist": ab["hist"], "eq_pyr1": ab["eq_pyr1"], "pyr_rest": ab["pyr_rest"], "fast": ab["fast"] * fast_frac,
                    "canny": ab["canny"], "walk": ab["fld_walk"], "lk": ab["lk"]}
        ks = {}
        for k, msv in t["ms"].items():
            n, fr = t["launches"][k], t["frames_of"][k]
            if not n or not fr:
                continue
            fpl = fr / n
            a = msv / n
            ks[k] = {"avg_ms": a, "frames_per_launch": round(fpl, 2), "algorithmic_bytes": bytes_of.get(k, 0) * fpl,
                     "ms_per_frame": msv / fr, "GBps": bytes_of.get(k, 0) * fpl / (a * 1e-3) / 1e9 if a > 0 else 0.0}
            ks[k]["frac"] = ks[k]["GBps"] / peak
        dom = max(ks, key=lambda k: ks[k]["ms_per_frame"]) if ks else None
        if dom:
            k = ks[dom]
            out.update(kernel=dom, achieved=k["GBps"], frac=k["GBps"] / peak, avg_launch_ms=k["avg_ms"],
                       algorithmic_bytes_per_launch=k["algorithmic_bytes"], frames_per_launch=k["frames_per_launch"])
        out["per_kernel"] = ks
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["group_kernels"]
            if dom and tr.get(dom) is not None:
                out["traffic"] = tr[dom]["dram_bytes_per_frame"] * ks[dom]["frames_per_launch"]
                out["traffic_note"] = tr[dom].get("note")
        except Exception:
            pass
        return out
    # handle engine: merge the per-handle FeStageTimes
    ms, launches, frames = {}, {}, 0
    for st in stage:
        frames += st["frames"]
        for k, v in st["ms"].items():
            ms[k] = ms.get(k, 0.0) + v
        for k, v in st["launches"].items():
            launches[k] = launches.get(k, 0) + v
    nfr = max(frames, 1)
    lk_pts = 300.0
    ab = algorithmic_bytes(lk_pts)
    LINE = ("canny", "fld", "fld_ccl", "fld_walk", "fld_seg")
    line_frames = launches.get("line_frames", 0)
    stage_ms = {k: v for k, v in ms.items() if k not in ("h2d", "fld", "line_frames") and launches.get(k)}
    fpl = {k: (line_frames / max(launches[k], 1) if k in LINE and line_frames else 1.0) for k in stage_ms}
    frames_of = {k: (line_frames if k in LINE and line_frames else nfr) for k in stage_ms}
    per_kernel = {}
    for k, v in stage_ms.items():
        a = v / max(launches[k], 1)
        per_kernel[k] = {"avg_ms": a, "frames_per_launch": round(fpl[k], 2), "algorithmic_bytes": ab.get(k, 0) * fpl[k],
                         "ms_per_frame": v / max(frames_of[k], 1),
                         "GBps": (ab.get(k, 0) * fpl[k] / (a * 1e-3)) / 1e9 if a > 0 else 0.0}
        per_kernel[k]["frac"] = per_kernel[k]["GBps"] / peak
    dom = max(per_kernel, key=lambda k: per_kernel[k]["ms_per_frame"]) if per_kernel else None
    if dom:
        k = per_kernel[dom]
        out.update(kernel=dom, achieved=k["GBps"], frac=k["frac"], avg_launch_ms=k["avg_ms"],
                   algorithmic_bytes_per_launch=k["algorithmic_bytes"], frames_per_launch=k["frames_per_launch"])
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["kernels"].get(KERNEL_OF_STAGE.get(dom, dom))
            out["traffic"] = tr * fpl[dom] if tr is not None else None
        except Exception:
            pass
    else:
        out.update(kernel=None, achieved=0.0, frac=0.0)
    out["per_kernel"] = per_kernel
    return out


if __name__ == "__main__":
    sys.exit(main())
