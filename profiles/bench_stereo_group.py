"""Stereo pairs per second on one GPU: the stereo group (plviwo_fe_stereo_group_*) against R stereo handles, with the
monocular stream group on the same images as the ceiling.

    python profiles/bench_stereo_group.py [--rigs 8 16 32] [--ticks 96] [--reps 3] [--out result.json]

Workload: BASELINE.json configs[1]'s knobs (1280x560, 400 points, 5 x 5 grid, 4-level pyramid, 15 x 15 window) with the
line tracker fed (vanishing points given, left image only on the stereo paths).  The pairs: --seqs synthetic stereo
sequences of --seq-frames pairs each (16 x 24 x 2 x 0.72 MB = 550 MB, more than the 126 MB of L2), played ping-pong; rig r
plays sequence r mod seqs from its own offset.  Per R, four arms, timed alternately --reps times (medians reported):
  group_resident   the stereo group's play() on pairs resident in HBM
  group_host       the stereo group's play() on the same pairs in pinned host memory (end to end: the copies included)
  handles          R FeStereoHandles on the resident pairs, pipelined: submit() up to --lookahead pairs ahead, collect()
  mono_group       the monocular stream group on 2R streams of the same resident images (every image one frame)
pairs/s = R x ticks / wall time of the arm (mono_group: images/s / 2); every arm returns once every pair is collected.
All arms use the same lookahead.  Prints one JSON line with the GPU's name and power limit (nvidia-smi, read only).
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
CONFIG1 = dict(num_features=400, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10, pyr_levels=4, win_size=15)


def _gen(args):
    seed, n = args
    import plviwo_b200  # noqa: F401
    from plviwo_b200 import synth
    q = synth.SynthSequence(seed=seed, width=W, height=H, n_frames=n)
    return np.stack([np.stack([q.frame(t, 0), q.frame(t, 1)]) for t in range(n)]), tuple(q.K), tuple(q.D), q.vanishing_points(0)


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
    ap.add_argument("--rigs", type=int, nargs="+", default=[8, 16, 32])
    ap.add_argument("--seqs", type=int, default=16)
    ap.add_argument("--seq-frames", type=int, default=24)
    ap.add_argument("--ticks", type=int, default=96)
    ap.add_argument("--warmup-ticks", type=int, default=24)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--lookahead", type=int, default=12)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import plviwo_b200 as fe
    F, NS = a.seq_frames, a.seqs
    with mp.get_context("spawn").Pool(min(NS, os.cpu_count() or 1)) as pool:
        seqs = pool.map(_gen, [(4000 + i, F) for i in range(NS)])
    host = torch.from_numpy(np.stack([q[0] for q in seqs])).pin_memory()   # (seqs, F, 2, H, W)
    dev = host.cuda()
    torch.cuda.synchronize()
    res = {"workload": "BASELINE.json configs[1] knobs (1280x560, 400 pts, 5x5 grid, pyr_levels 4, win 15), lines fed; %d distinct "
                       "pairs (%.0f MB), lookahead %d, %d ticks per rep" % (NS * F, NS * F * 2 * W * H / 1e6, a.lookahead, a.ticks),
           "gpu": gpu_card(), "reps": a.reps}

    for R in a.rigs:
        calib = [(seqs[r % NS][1], seqs[r % NS][2]) for r in range(R)]
        vps = [seqs[r % NS][3] for r in range(R)]
        offset = [(r // NS) * 5 for r in range(R)]

        def frame(src, r, t, cam):
            return src[r % NS, ping_pong(t + offset[r], F), cam]

        def stereo_table(src, first, n):
            ptrs = [frame(src, r, first + t, cam).data_ptr() for t in range(n) for r in range(R) for cam in (0, 1)]
            return (C.c_void_p * len(ptrs))(*ptrs)

        def mono_table(first, n):   # stream 2r + cam = camera cam of rig r
            return stereo_table(dev, first, n)

        cfg = dict(width=W, height=H, lookahead=a.lookahead, use_lines=1, **CONFIG1)
        sg = fe.StereoGroupFrontEnd(fe.default_config(**cfg), R, calibs=[(c, c) for c in calib])
        mg = fe.GroupFrontEnd(fe.default_config(**cfg), 2 * R, calibs=[c for c in calib for _ in (0, 1)])
        hs = [fe.StereoFrontEnd(fe.default_config(K=calib[r][0], D=calib[r][1], **cfg), K_right=calib[r][0], D_right=calib[r][1])
              for r in range(R)]
        tick = dict(group_resident=0, group_host=0, handles=0, mono_group=0)

        def run(arm, n):
            t0 = tick[arm]
            ts = [1.0 + 0.1 * (t0 + t) for t in range(n)]
            if arm in ("group_resident", "group_host"):
                src = dev if arm == "group_resident" else host
                st = sg.play(ts, stereo_table(src, t0, n), W, arm == "group_resident", vanishing_points=vps)
                assert all(x.frames == n for x in st)
            elif arm == "mono_group":
                st = mg.play(ts, mono_table(t0, n), W, True, vanishing_points=[v for v in vps for _ in (0, 1)])
                assert all(x.frames == n for x in st)
            else:
                sub = 0
                for i in range(n):
                    while sub < n and sub <= i + a.lookahead:
                        for r, h in enumerate(hs):
                            h.submit(ts[sub], frame(dev, r, t0 + sub, 0).data_ptr(), frame(dev, r, t0 + sub, 1).data_ptr(), stride=W,
                                     on_device=True, vanishing_points=vps[r])
                        sub += 1
                    for h in hs:
                        h.collect()
            tick[arm] += n

        for arm in tick:
            run(arm, a.warmup_ticks)
        torch.cuda.synchronize()
        wall = {arm: [] for arm in tick}
        for _ in range(a.reps):
            for arm in tick:
                t0 = time.perf_counter()
                run(arm, a.ticks)
                wall[arm].append(time.perf_counter() - t0)
        sg.close()
        mg.close()
        for h in hs:
            h.close()
        out = {}
        for arm, ws in wall.items():
            pps = [R * a.ticks / w for w in ws]
            out[arm] = {"pairs_per_s": pps, "pairs_per_s_median": float(np.median(pps))}
        out["group_resident_over_handles"] = out["group_resident"]["pairs_per_s_median"] / out["handles"]["pairs_per_s_median"]
        res["rigs_%d" % R] = out
        print(json.dumps({"rigs": R, **{k: (v["pairs_per_s_median"] if isinstance(v, dict) else v) for k, v in out.items()}}),
              file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
