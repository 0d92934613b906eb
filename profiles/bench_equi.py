"""Throughput of the equidistant (fisheye) camera model against radtan on BASELINE.json configs[4] (64 independent 1280x560
streams, each the configs[1] front end: 400 points, 5x5 grid, maxLevel 4, win 15, lines on): one stream group per model,
timed alternately in one process through plviwo_fe_group_play on frames resident in HBM.

    python profiles/bench_equi.py [--streams 64] [--ticks 192] [--reps 3] [--out result.json]

The frames: --seqs sequences of --seq-frames distinct frames each (16 x 24 = 384 frames, 275 MB, more than the 126 MB of L2),
played ping-pong; stream s plays sequence s mod seqs from its own offset.  The radtan group runs the sequences' own
calibration, the equidistant group the same K with EuRoC-like fisheye coefficients.  A rep = one play of --ticks ticks per
group (groups keep their tracker state from rep to rep); frames/s = streams x ticks / wall time of the play call, which
returns once every tick is collected.  Prints one JSON line, with the GPU's name and power limit (nvidia-smi, read only).
"""
import argparse
import ctypes as C
import json
import multiprocessing as mp
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

from bench_group_line_samples import gpu_card, ping_pong  # noqa: E402

W, H = 1280, 560
CONFIG1 = dict(num_features=400, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10, pyr_levels=4, win_size=15)
EQUI_D = (-0.0348, 0.0123, -0.0071, 0.0021)


def _gen(args):
    seed, n = args
    import plviwo_b200  # noqa: F401
    from plviwo_b200 import synth
    q = synth.SynthSequence(seed=seed, width=W, height=H, n_frames=n)
    return np.stack([q.frame(t) for t in range(n)]), tuple(q.K), tuple(q.D), q.vanishing_points(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--seqs", type=int, default=16)
    ap.add_argument("--seq-frames", type=int, default=24)
    ap.add_argument("--ticks", type=int, default=192)
    ap.add_argument("--warmup-ticks", type=int, default=48)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--lookahead", type=int, default=24)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import plviwo_b200 as fe
    S, F = a.streams, a.seq_frames
    with mp.get_context("spawn").Pool(min(a.seqs, os.cpu_count() or 1)) as pool:
        seqs = pool.map(_gen, [(4000 + i, F) for i in range(a.seqs)])
    frames = torch.from_numpy(np.stack([q[0] for q in seqs])).cuda()   # (seqs, F, H, W), resident for the whole run
    torch.cuda.synchronize()
    vps = [seqs[s % a.seqs][3] for s in range(S)]
    offset = [(s // a.seqs) * 5 for s in range(S)]

    def table(first, n):
        ptrs = [frames[s % a.seqs, ping_pong(first + t + offset[s], F)].data_ptr() for t in range(n) for s in range(S)]
        return (C.c_void_p * len(ptrs))(*ptrs)

    cfg = lambda: fe.default_config(width=W, height=H, lookahead=a.lookahead, **CONFIG1)
    groups = {
        "radtan": fe.GroupFrontEnd(cfg(), S, calibs=[(seqs[s % a.seqs][1], seqs[s % a.seqs][2]) for s in range(S)]),
        "equidistant": fe.GroupFrontEnd(cfg(), S, calibs=[(seqs[s % a.seqs][1], EQUI_D) for s in range(S)],
                                        camera_model=fe.CAM_EQUI),
    }
    tick = {m: 0 for m in groups}

    def play(m, n):
        st = groups[m].play([0.1 * (tick[m] + t) for t in range(n)], table(tick[m], n), W, True, vanishing_points=vps)
        tick[m] += n
        return st

    for m in groups:
        play(m, a.warmup_ticks)
    wall = {m: [] for m in groups}
    rows = {m: 0 for m in groups}
    for _ in range(a.reps):
        for m in groups:
            t0 = time.perf_counter()
            st = play(m, a.ticks)
            wall[m].append(time.perf_counter() - t0)
            assert all(x.frames == a.ticks for x in st)
            rows[m] += sum(x.point_rows for x in st)
    for grp in groups.values():
        grp.close()
    res = {"workload": "BASELINE.json configs[4]: %d streams of one GPU, each the configs[1] front end (1280x560, 400 pts, 5x5 "
                       "grid, maxLevel 4, win 15, lines on), plviwo_fe_group_play, lookahead %d, frames resident in HBM (%d "
                       "distinct, %.0f MB)" % (S, a.lookahead, a.seqs * F, a.seqs * F * W * H / 1e6),
           "gpu": gpu_card(), "ticks_per_rep": a.ticks, "reps": a.reps}
    for m, ws in wall.items():
        fps = [S * a.ticks / w for w in ws]
        res[m] = {"frames_per_s": fps, "frames_per_s_median": float(np.median(fps)),
                  "point_rows_per_frame": rows[m] / (S * a.ticks * a.reps)}
    res["equidistant_over_radtan"] = res["equidistant"]["frames_per_s_median"] / res["radtan"]["frames_per_s_median"]
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
