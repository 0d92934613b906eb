"""cfg.line_samples in a stream group (plviwo_fe_group_get_line_samples, BASELINE.json configs[2] on many streams).

The bar: after every collect, stream s returns EXACTLY the samples a single FeHandle returns from
plviwo_fe_get_line_samples when fed the same frames, masks and vanishing points — count, order, u0 v0 u1 v1 bytes and
status bytes — and every other output of the group stays what a handle gives (point rows, last obs, line rows, point-on-line
entries, frame info).
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W, H = 1280, 560
CFG1 = dict(num_features=200, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10, pyr_levels=3, win_size=15)
CFG3 = dict(CFG1, pyr_levels=5)   # BASELINE.json configs[2]


def _info(info):
    return (info.reset, info.first_frame, info.n_detected, info.detection_ran, info.n_lk_in, info.n_klt_ok, info.n_ransac_ok,
            info.n_lines_detected, info.n_line_matches)


def _handle_frames(fe, q, cfg_kw, frames, vps, masks=None):
    """Outputs of one FeHandle (lookahead 0) fed frames[t] (None: skipped) with vps[t] (None: line tracker not fed) and
    masks[t], recorded after every frame: the usual rows plus line_samples()."""
    h = fe.FrontEnd(fe.default_config(width=W, height=H, K=q.K, D=q.D, lookahead=0, **cfg_kw))
    out = {}
    for t, im in enumerate(frames):
        if im is None:
            continue
        info = h.feed_new_camera(q.timestamp(t), im, masks[t] if masks else None, vps[t], update_db=False)
        lr, lp = h.line_rows()
        ids, uv = h._last()
        su, ss = h.line_samples()
        out[t] = dict(rows=h.point_rows(), lrows=lr, lpts=lp, ids=ids, uv=uv, su=su, ss=ss, info=_info(info))
    h.close()
    return out


def _group_frames(fe, seqs, cfg_kw, frames, vps, lookahead, masks=None):
    """The same through one group: frames[s][t] (None: stream s has no frame in tick t), vps[t] = per-stream vanishing
    points or None for the whole tick, masks[s][t]."""
    S, n = len(seqs), len(frames[0])
    g = fe.GroupFrontEnd(fe.default_config(width=W, height=H, lookahead=lookahead, **cfg_kw), S, calibs=[(q.K, q.D) for q in seqs])
    out = [{} for _ in range(S)]
    sub = 0
    for t in range(n):
        while sub < n and sub <= t + lookahead:
            g.submit([q.timestamp(sub) for q in seqs], [frames[s][sub] for s in range(S)], vanishing_points=vps[sub],
                     masks=[masks[s][sub] if frames[s][sub] is not None else None for s in range(S)] if masks else None)
            sub += 1
        g.collect()
        for s in range(S):
            if frames[s][t] is None:
                assert g.infos[s].timestamp == -1.0
                assert len(g.line_samples(s)[0]) == 0
                continue
            lr, lp = g.line_rows(s)
            ids, uv = g.last_obs(s)
            su, ss = g.line_samples(s)
            out[s][t] = dict(rows=g.point_rows(s), lrows=lr, lpts=lp, ids=ids, uv=uv, su=su, ss=ss, info=_info(g.infos[s]))
    g.close()
    return out


def _assert_same(a, b, where):
    assert len(a["su"]) == len(b["su"]), ("sample count differs " + where, len(a["su"]), len(b["su"]))
    assert a["su"].tobytes() == b["su"].tobytes(), "sample positions differ " + where
    assert a["ss"].tobytes() == b["ss"].tobytes(), "sample status differs " + where
    assert a["rows"].tobytes() == b["rows"].tobytes(), "point rows differ " + where
    assert np.array_equal(a["ids"], b["ids"]) and a["uv"].tobytes() == b["uv"].tobytes(), "last obs differ " + where
    assert a["info"] == b["info"], ("frame info differs " + where, a["info"], b["info"])
    assert a["lrows"].tobytes() == b["lrows"].tobytes(), "line rows differ " + where
    assert a["lpts"].tobytes() == b["lpts"].tobytes(), "line points differ " + where


def _run(fe, seqs, cfg_kw, frames, vps_tick, lookahead, masks=None):
    """Group vs one handle per stream; returns the handles' outputs (stream -> frame -> dict)."""
    S = len(seqs)
    ref = [_handle_frames(fe, q, cfg_kw, frames[s], [None if v is None else v[s] for v in vps_tick],
                          masks[s] if masks else None) for s, q in enumerate(seqs)]
    got = _group_frames(fe, seqs, cfg_kw, frames, vps_tick, lookahead, masks)
    for s in range(S):
        assert sorted(ref[s]) == sorted(got[s])
        for t in ref[s]:
            _assert_same(ref[s][t], got[s][t], "stream %d frame %d" % (s, t))
    return ref


@pytest.mark.parametrize("lookahead,n_streams", [(0, 3), (4, 2)])
def test_group_line_samples_equal_handles_config3(fe, synth, lookahead, n_streams):
    """configs[2]: the line-heavy scene, maxLevel 5, 10 samples per segment (> 3000 samples per frame)."""
    n = 12
    seqs = [synth.SynthSequence(seed=1004 + s, width=W, height=H, n_frames=n, line_heavy=True) for s in range(n_streams)]
    frames = [[q.frame(t) for t in range(n)] for q in seqs]
    vps = [[q.vanishing_points(t) for q in seqs] for t in range(n)]
    ref = _run(fe, seqs, dict(CFG3, line_samples=10), frames, vps, lookahead)
    for s in range(n_streams):
        assert len(ref[s][0]["su"]) == 0   # detection-only first frame
        counts = [len(ref[s][t]["su"]) for t in range(2, n)]
        assert min(counts) > 3000, (s, counts)
        assert len(ref[s][1]["su"]) == 10 * ref[s][0]["info"][7]   # the segments of frame 0, 10 each
        st = np.concatenate([ref[s][t]["ss"] for t in range(1, n)])
        assert 0 < st.sum() < len(st)   # statuses of both kinds: the comparison is not vacuous


def test_group_line_samples_cut_at_the_lk_buffer(fe, synth):
    """200 samples per segment: more than a handle's LK buffer holds after the points, both stop at max_pts - n."""
    n = 4
    seqs = [synth.SynthSequence(seed=1004, width=W, height=H, n_frames=n, line_heavy=True)]
    frames = [[seqs[0].frame(t) for t in range(n)]]
    vps = [[seqs[0].vanishing_points(t)] for t in range(n)]
    ref = _run(fe, seqs, dict(CFG3, line_samples=200), frames, vps, 1)[0]
    max_pts = max(4096, 8 * CFG3["num_features"]) + 32768   # fe_context.cu: the handle's LK buffer with line_samples > 0
    for t in range(1, n):
        n_pts, n_seg = ref[t]["info"][4], ref[t - 1]["info"][7]
        assert 200 * n_seg > max_pts - n_pts and len(ref[t]["su"]) == max_pts - n_pts, (t, n_pts, n_seg, len(ref[t]["su"]))


@pytest.mark.parametrize("line_samples,win", [(1, 15), (2, 15), (3, 21)])
def test_group_line_samples_per_segment_and_window(fe, synth, line_samples, win):
    """S = 1 (a = 0.5), S = 2 (the end points) and a 21 x 21 window (the generic LK kernel), 2 streams, 2 ticks ahead."""
    n = 8
    seqs = [synth.SynthSequence(seed=1050 + s, width=W, height=H, n_frames=n) for s in range(2)]
    frames = [[q.frame(t) for t in range(n)] for q in seqs]
    vps = [[q.vanishing_points(t) for q in seqs] for t in range(n)]
    ref = _run(fe, seqs, dict(CFG1, win_size=win, line_samples=line_samples), frames, vps, 2)
    assert all(len(ref[s][t]["su"]) > 0 for s in range(2) for t in range(1, n))


def test_group_line_samples_tick_without_vanishing_points(fe, synth):
    """A tick fed without vanishing points does not update the segments: the next frame samples the older ones."""
    n, gap = 9, 4
    seqs = [synth.SynthSequence(seed=1060 + s, width=W, height=H, n_frames=n) for s in range(2)]
    frames = [[q.frame(t) for t in range(n)] for q in seqs]
    vps = [None if t == gap else [q.vanishing_points(t) for q in seqs] for t in range(n)]
    ref = _run(fe, seqs, dict(CFG1, line_samples=4), frames, vps, 2)
    for s in range(2):
        a, b = ref[s][gap]["su"], ref[s][gap + 1]["su"]
        assert len(a) > 0 and len(a) == len(b) and np.array_equal(a[:, :2], b[:, :2])   # both on the segments of frame gap - 1
        assert ref[s][gap]["info"][7] == 0 and len(ref[s][gap]["lrows"]) == 0


def test_group_line_samples_partial_ticks_black_frame_masks_clahe(fe, synth):
    """Stream 1 skips every second tick, stream 2 sees a black frame (tracker reset), moving masks with CLAHE."""
    n, black = 12, 5
    seqs = [synth.SynthSequence(seed=1070 + s, width=W, height=H, n_frames=n, moving_mask=True) for s in range(3)]
    frames = [[q.frame(t) if not (s == 1 and t % 2 == 1) else None for t in range(n)] for s, q in enumerate(seqs)]
    frames[2][black] = np.zeros((H, W), np.uint8)
    masks = [[q.mask(t) for t in range(n)] for q in seqs]
    vps = [[q.vanishing_points(t) for q in seqs] for t in range(n)]
    ref = _run(fe, seqs, dict(CFG1, line_samples=5, histogram_method=fe.HIST_CLAHE), frames, vps, 1, masks=masks)
    r = ref[2]
    assert r[black]["info"][4] >= 10 and len(r[black]["su"]) > 0   # the black frame still runs LK, with samples
    after = [t for t in range(black + 1, n) if r[t]["info"][1]]
    assert after and len(r[after[0]]["su"]) == 0                    # the detection-only frame after the reset has none
    assert all(len(ref[1][t]["su"]) > 0 for t in range(2, n, 2))   # stream 1: its previous frame is two ticks back


def test_group_line_samples_without_line_tracker(fe, synth):
    """use_lines = 0: no segments, no samples; the point rows are those of a group without line_samples."""
    n, S = 6, 2
    seqs = [synth.SynthSequence(seed=1080 + s, width=W, height=H, n_frames=n) for s in range(S)]
    frames = [[q.frame(t) for t in range(n)] for q in seqs]
    vps = [[q.vanishing_points(t) for q in seqs] for t in range(n)]
    runs = [_group_frames(fe, seqs, dict(CFG1, use_lines=0, line_samples=ls), frames, vps, 1) for ls in (10, 0)]
    for s in range(S):
        for t in range(n):
            a, b = runs[0][s][t], runs[1][s][t]
            assert len(a["su"]) == 0
            assert a["rows"].tobytes() == b["rows"].tobytes() and a["uv"].tobytes() == b["uv"].tobytes() and a["info"] == b["info"]


def test_group_line_samples_getter(fe, synth):
    """Bad stream: FE_BAD_ARG; cap below the count: FE_OVERFLOW with n_out set."""
    seqs = [synth.SynthSequence(seed=1090 + s, width=W, height=H, n_frames=3) for s in range(2)]
    g = fe.GroupFrontEnd(fe.default_config(width=W, height=H, lookahead=0, line_samples=10, **CFG1), 2,
                         calibs=[(q.K, q.D) for q in seqs])
    L = g._lib
    n = C.c_int(-1)
    assert L.plviwo_fe_group_get_line_samples(g._h, 0, None, None, 0, C.byref(n)) == fe.FE_BAD_ARG   # nothing collected yet
    for t in range(3):
        g.feed([q.timestamp(t) for q in seqs], [q.frame(t) for q in seqs], vanishing_points=[q.vanishing_points(t) for q in seqs])
    for bad in (-1, 2):
        assert L.plviwo_fe_group_get_line_samples(g._h, bad, None, None, 0, C.byref(n)) == fe.FE_BAD_ARG
    assert L.plviwo_fe_group_get_line_samples(None, 0, None, None, 0, C.byref(n)) == fe.FE_BAD_ARG
    assert L.plviwo_fe_group_get_line_samples(g._h, 0, None, None, 0, C.byref(n)) == fe.FE_OK
    count = n.value
    assert count > 1
    uv = np.zeros((count, 4), np.float32)
    st = np.zeros((count,), np.uint8)
    n.value = -1
    assert L.plviwo_fe_group_get_line_samples(g._h, 0, uv.ctypes.data, st.ctypes.data, count - 1, C.byref(n)) == fe.FE_OVERFLOW
    assert n.value == count
    assert L.plviwo_fe_group_get_line_samples(g._h, 0, uv.ctypes.data, None, count, C.byref(n)) == fe.FE_OK
    uv2, st2 = g.line_samples(0)
    assert uv.tobytes() == uv2.tobytes() and len(st2) == count
    g.close()
