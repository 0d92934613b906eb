"""Throughput of BASELINE.json configs[2] (line-heavy 1280x560 scene, 200 points, maxLevel 5, win 15, 10 LK samples per
segment) on many streams of one GPU: one stream group with cfg.line_samples = 10 and one with 0, timed alternately in one
process through plviwo_fe_group_play on frames resident in HBM.

    python profiles/bench_group_line_samples.py [--streams 64] [--ticks 192] [--reps 3] [--out result.json]

The frames: --seqs line-heavy sequences of --seq-frames distinct frames each (16 x 24 x 0.72 MB = 275 MB, more than the
126 MB of L2), played ping-pong; stream s plays sequence s mod seqs from its own offset, so streams that share a sequence
do not read the same frame in the same tick.  A rep = one play of --ticks ticks per group (groups keep their tracker state
from rep to rep); frames/s = streams x ticks / wall time of the play call, which returns once every tick is collected.
Samples per frame are counted afterwards in an untimed submit / collect pass of the line_samples group over the same frames;
samples/s = frames/s x that mean.  Prints one JSON line, with the GPU's name and power limit (nvidia-smi, read only).
"""
import argparse
import ctypes as C
import json
import multiprocessing as mp
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

W, H = 1280, 560
CONFIG3 = dict(num_features=200, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10, pyr_levels=5, win_size=15)


def _gen(args):
    seed, n = args
    import plviwo_b200  # noqa: F401
    from plviwo_b200 import synth
    q = synth.SynthSequence(seed=seed, width=W, height=H, n_frames=n, line_heavy=True)
    return np.stack([q.frame(t) for t in range(n)]), tuple(q.K), tuple(q.D), q.vanishing_points(0)


def ping_pong(i, n):
    p = 2 * (n - 1)
    k = i % p
    return k if k < n else p - k


def gpu_card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=64)
    ap.add_argument("--seqs", type=int, default=16)
    ap.add_argument("--seq-frames", type=int, default=24)
    ap.add_argument("--ticks", type=int, default=192)
    ap.add_argument("--warmup-ticks", type=int, default=48)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--lookahead", type=int, default=24)
    ap.add_argument("--count-ticks", type=int, default=24)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import plviwo_b200 as fe
    S, F = a.streams, a.seq_frames
    with mp.get_context("spawn").Pool(min(a.seqs, os.cpu_count() or 1)) as pool:
        seqs = pool.map(_gen, [(3000 + i, F) for i in range(a.seqs)])
    frames = torch.from_numpy(np.stack([q[0] for q in seqs])).cuda()   # (seqs, F, H, W), resident for the whole run
    torch.cuda.synchronize()
    calibs = [(seqs[s % a.seqs][1], seqs[s % a.seqs][2]) for s in range(S)]
    vps = [seqs[s % a.seqs][3] for s in range(S)]
    offset = [(s // a.seqs) * 5 for s in range(S)]

    def table(first, n):
        ptrs = [frames[s % a.seqs, ping_pong(first + t + offset[s], F)].data_ptr() for t in range(n) for s in range(S)]
        return (C.c_void_p * len(ptrs))(*ptrs)

    groups = {ls: fe.GroupFrontEnd(fe.default_config(width=W, height=H, lookahead=a.lookahead, line_samples=ls, **CONFIG3), S,
                                   calibs=calibs) for ls in (10, 0)}
    tick = {ls: 0 for ls in groups}

    def play(ls, n):
        st = groups[ls].play([0.1 * (tick[ls] + t) for t in range(n)], table(tick[ls], n), W, True, vanishing_points=vps)
        tick[ls] += n
        return st

    for ls in groups:
        play(ls, a.warmup_ticks)
    wall = {ls: [] for ls in groups}
    for _ in range(a.reps):
        for ls in groups:
            t0 = time.perf_counter()
            st = play(ls, a.ticks)
            wall[ls].append(time.perf_counter() - t0)
            assert all(x.frames == a.ticks for x in st)
    # samples per frame (untimed): submit / collect the line_samples group tick by tick over the same frames
    g = groups[10]
    n = C.c_int(0)
    n_samples = n_frames = 0
    for t in range(a.count_ticks):
        tab = table(tick[10], 1)
        g.submit([0.1 * tick[10]] * S, [tab[s] for s in range(S)], stride=W, on_device=True, vanishing_points=vps)
        g.collect()
        tick[10] += 1
        for s in range(S):
            assert g._lib.plviwo_fe_group_get_line_samples(g._h, s, None, None, 0, C.byref(n)) == fe.FE_OK
            n_samples += n.value
            n_frames += 1
    for grp in groups.values():
        grp.close()
    per_frame = n_samples / max(n_frames, 1)
    res = {"workload": "BASELINE.json configs[2] on %d streams of one GPU (line-heavy 1280x560, 200 pts, maxLevel 5, win 15), "
                       "plviwo_fe_group_play, lookahead %d, frames resident in HBM (%d distinct, %.0f MB)" %
                       (S, a.lookahead, a.seqs * F, a.seqs * F * W * H / 1e6),
           "gpu": gpu_card(), "ticks_per_rep": a.ticks, "reps": a.reps, "samples_per_frame": per_frame}
    for ls, ws in wall.items():
        fps = [S * a.ticks / w for w in ws]
        res["line_samples_%d" % ls] = {"frames_per_s": fps, "frames_per_s_median": float(np.median(fps))}
    res["line_samples_10"]["samples_per_s_median"] = res["line_samples_10"]["frames_per_s_median"] * per_frame
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
