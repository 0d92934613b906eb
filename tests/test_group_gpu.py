"""Stream group (plviwo_fe_group_*, BASELINE.json configs[4]) through the C ABI.

The bar: stream s of a group produces, frame by frame, EXACTLY the rows a single FeHandle produces on the same frames
(point rows, pts_last / ids_last, line rows, point-on-line entries) — the group batches the kernels of all streams and
runs the state machine on the device, which must not change a bit — and, teacher-forced against the oracle, the same
bars as tests/test_frontend_gpu.py (ids bit-exact, 0.05 px, status >= 99.5 %).
"""
import numpy as np
import pytest

from oracle import frontend as ofe

pytestmark = pytest.mark.gpu

CFG1 = dict(num_features=200, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10, pyr_levels=3, win_size=15)
CFG2 = dict(num_features=400, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10, pyr_levels=4, win_size=15)
CFG_KAIST = dict(num_features=1500, fast_threshold=30, grid_x=15, grid_y=15, min_px_dist=15, pyr_levels=5, win_size=15)
CFG4 = dict(num_features=1000, fast_threshold=20, grid_x=10, grid_y=6, min_px_dist=15, pyr_levels=5, win_size=21)
CFG_DEEP = dict(CFG_KAIST, pyr_levels=6)   # at 1280 x 560 the pyramid stops at 6 images (40 x 18): the 15 x 15 bodies


def _single_rows(fe, seq, kw, n_frames, W, H, lines=True, masks=False, hist=1):
    """Rows of one FeHandle fed frame by frame (the synchronous drop-in)."""
    h = fe.FrontEnd(fe.default_config(width=W, height=H, K=seq.K, D=seq.D, lookahead=0, histogram_method=hist, **kw))
    out = []
    for t in range(n_frames):
        info = h.feed_new_camera(seq.timestamp(t), seq.frame(t), seq.mask(t) if masks else None,
                                 seq.vanishing_points(t) if lines else None, update_db=False)
        lr, lp = h.line_rows()
        ids, uv = h._last()
        out.append(dict(rows=h.point_rows(), lrows=lr, lpts=lp, ids=ids, uv=uv,
                        info=(info.reset, info.first_frame, info.n_detected, info.detection_ran, info.n_lk_in, info.n_klt_ok,
                              info.n_ransac_ok, info.n_lines_detected, info.n_line_matches)))
    h.close()
    return out


def _assert_same(a, got, where):
    rows, lr, lp, ids, uv, info = got
    assert a["rows"].tobytes() == rows.tobytes(), "point rows differ " + where
    assert np.array_equal(a["ids"], ids) and a["uv"].tobytes() == uv.tobytes(), "last obs differ " + where
    assert a["info"] == info, ("frame info differs " + where, a["info"], info)
    assert len(a["lrows"]) == len(lr), ("line row count differs " + where, len(a["lrows"]), len(lr))
    assert a["lrows"].tobytes() == lr.tobytes(), "line rows differ " + where
    assert a["lpts"].tobytes() == lp.tobytes(), "line points differ " + where


def _group_frame(g, s):
    info = g.infos[s]
    lr, lp = g.line_rows(s)
    ids, uv = g.last_obs(s)
    return (g.point_rows(s), lr, lp, ids, uv,
            (info.reset, info.first_frame, info.n_detected, info.detection_ran, info.n_lk_in, info.n_klt_ok, info.n_ransac_ok,
             info.n_lines_detected, info.n_line_matches))


@pytest.mark.parametrize("kw,lookahead,n_streams", [(CFG2, 0, 3), (CFG2, 4, 5), (CFG1, 2, 2)])
def test_group_equals_single_handles(fe, synth, kw, lookahead, n_streams):
    W, H, n_frames = 1280, 560, 14
    seqs = [synth.SynthSequence(seed=1000 + s, width=W, height=H, n_frames=n_frames) for s in range(n_streams)]
    ref = [_single_rows(fe, q, kw, n_frames, W, H) for q in seqs]
    cfg = fe.default_config(width=W, height=H, lookahead=lookahead, **kw)
    g = fe.GroupFrontEnd(cfg, n_streams, calibs=[(q.K, q.D) for q in seqs])
    frames = [[q.frame(t) for t in range(n_frames)] for q in seqs]
    sub = 0
    for t in range(n_frames):
        while sub < n_frames and sub <= t + lookahead:
            g.submit([q.timestamp(sub) for q in seqs], [frames[s][sub] for s in range(n_streams)],
                     vanishing_points=[q.vanishing_points(sub) for q in seqs])
            sub += 1
        g.collect()
        for s in range(n_streams):
            _assert_same(ref[s][t], _group_frame(g, s), "stream %d frame %d" % (s, t))
    g.close()


def test_group_kaist_yaml_and_wide_window(fe, synth):
    """KAIST yaml (1500 points, 15 x 15 grid), config 4 (1920 x 1080, 21 x 21 window: the generic LK kernel) and pyr_levels
    6 at 1280 x 560 (a pyramid of 6 images: the 15 x 15 kernels, as in a handle)."""
    for kw, W, H, n_frames in ((CFG_KAIST, 1280, 560, 8), (CFG4, 1920, 1080, 6), (CFG_DEEP, 1280, 560, 8)):
        seqs = [synth.SynthSequence(seed=1010 + s, width=W, height=H, n_frames=n_frames) for s in range(2)]
        ref = [_single_rows(fe, q, kw, n_frames, W, H) for q in seqs]
        g = fe.GroupFrontEnd(fe.default_config(width=W, height=H, lookahead=2, **kw), 2, calibs=[(q.K, q.D) for q in seqs])
        frames = [[q.frame(t) for t in range(n_frames)] for q in seqs]
        sub = 0
        for t in range(n_frames):
            while sub < n_frames and sub <= t + 2:
                g.submit([q.timestamp(sub) for q in seqs], [frames[s][sub] for s in range(2)],
                         vanishing_points=[q.vanishing_points(sub) for q in seqs])
                sub += 1
            g.collect()
            for s in range(2):
                _assert_same(ref[s][t], _group_frame(g, s), "%dx%d stream %d frame %d" % (W, H, s, t))
        g.close()


def test_group_masks_clahe_partial_ticks_and_reset(fe, synth):
    """Moving masks, CLAHE, a stream that skips ticks, a black frame (tracker reset), no line tracker."""
    W, H, n_frames = 1280, 560, 12
    seqs = [synth.SynthSequence(seed=1020 + s, width=W, height=H, n_frames=n_frames, moving_mask=True) for s in range(3)]
    # stream 1 only has a frame every second tick; stream 2 sees a black frame at t = 5
    frames = [[q.frame(t) for t in range(n_frames)] for q in seqs]
    frames[2][5] = np.zeros((H, W), np.uint8)
    active = lambda s, t: not (s == 1 and t % 2 == 1)
    ref = []
    for s, q in enumerate(seqs):
        h = fe.FrontEnd(fe.default_config(width=W, height=H, K=q.K, D=q.D, lookahead=0, histogram_method=fe.HIST_CLAHE, **CFG1))
        out = {}
        for t in range(n_frames):
            if not active(s, t):
                continue
            info = h.feed_new_camera(q.timestamp(t), frames[s][t], q.mask(t), q.vanishing_points(t), update_db=False)
            lr, lp = h.line_rows()
            ids, uv = h._last()
            out[t] = dict(rows=h.point_rows(), lrows=lr, lpts=lp, ids=ids, uv=uv,
                          info=(info.reset, info.first_frame, info.n_detected, info.detection_ran, info.n_lk_in, info.n_klt_ok,
                                info.n_ransac_ok, info.n_lines_detected, info.n_line_matches))
        h.close()
        ref.append(out)
    g = fe.GroupFrontEnd(fe.default_config(width=W, height=H, lookahead=1, histogram_method=fe.HIST_CLAHE, **CFG1), 3,
                         calibs=[(q.K, q.D) for q in seqs])
    lost = 0
    for t in range(n_frames):
        g.submit([q.timestamp(t) for q in seqs], [frames[s][t] if active(s, t) else None for s in range(3)],
                 vanishing_points=[q.vanishing_points(t) for q in seqs],
                 masks=[seqs[s].mask(t) if active(s, t) else None for s in range(3)])
        g.collect()
        for s in range(3):
            if not active(s, t):
                assert g.infos[s].timestamp == -1.0
                continue
            _assert_same(ref[s][t], _group_frame(g, s), "stream %d frame %d" % (s, t))
            lost += int(s == 2 and t > 5 and (g.infos[s].reset or g.infos[s].first_frame))
    assert lost >= 1   # the black frame really made the tracker of stream 2 lose everything and start over
    g.close()


@pytest.mark.parametrize("thread_walk", [False, True])
def test_group_teacher_forced_against_oracle(fe, synth, thread_walk, monkeypatch):
    """Every frame of every stream on the oracle's state (plviwo_fe_group_set_state): ids and row order bit-exact, UVs
    within 0.05 px, status flags >= 99.5 %, line ids / point-on-line sets identical.  thread_walk: the chain walk's
    thread-per-component class, which a group otherwise uses from 16 frames per launch on (the 64-stream bench)."""
    if thread_walk:
        monkeypatch.setenv("PLVIWO_WALK_THREAD_MIN", "1")
    else:
        monkeypatch.delenv("PLVIWO_WALK_THREAD_MIN", raising=False)
    W, H, n_frames, S = 1280, 560, 12, 2
    seqs = [synth.SynthSequence(seed=1030 + s, width=W, height=H, n_frames=n_frames) for s in range(S)]
    oracles = [ofe.FrontEnd(ofe.FeConfig(K=q.K, D=q.D, **CFG2)) for q in seqs]
    g = fe.GroupFrontEnd(fe.default_config(width=W, height=H, lookahead=0, **CFG2), S, calibs=[(q.K, q.D) for q in seqs])
    rows_total = flipped = 0
    duv = [0.0]
    for t in range(n_frames):
        if t > 0:
            for s, o in enumerate(oracles):
                k, l = o.klt.get_state(), o.lsd.get_state()
                g.set_state(s, fe.pack_state(W, H, k["currid"], k["pts_last"], k["ids_last"], k["img_last"], k["mask_last"],
                                             l["currid"], l["lines_last"], l["ids_last"], l["pol_last"]))
        imgs = [q.frame(t) for q in seqs]
        want = [o.feed(q.timestamp(t), im, None, q.vanishing_points(t)) for o, q, im in zip(oracles, seqs, imgs)]
        g.feed([q.timestamp(t) for q in seqs], imgs, vanishing_points=[q.vanishing_points(t) for q in seqs])
        for s in range(S):
            prow_o, lrow_o = want[s]
            rows = g.point_rows(s)
            ids_o = {r.id: r for r in prow_o}
            ids_g = {int(r["id"]): r for r in rows}
            sym = set(ids_o) ^ set(ids_g)
            rows_total += len(ids_o)
            flipped += len(sym)
            if not sym:
                assert [r.id for r in prow_o] == [int(v) for v in rows["id"]], "row order differs at frame %d" % t
                lr, lp = g.line_rows(s)
                assert len(lr) == len(lrow_o), (t, s)
                for a, b in zip(lr, lrow_o):
                    assert int(a["id"]) == b.id and int(a["D"]) == b.D and int(a["n_pts"]) == len(b.pids), (t, s)
                    assert np.abs(a["line"] - b.line).max() <= 2e-3
                    assert list(lp[a["pt_offset"]:a["pt_offset"] + a["n_pts"]]["pid"]) == list(b.pids)
            for fid in set(ids_o) & set(ids_g):
                a, b = ids_g[fid], ids_o[fid]
                duv.append(max(abs(float(a["u"]) - b.u), abs(float(a["v"]) - b.v)))
    g.close()
    duv = np.array(duv)
    print(dict(rows=rows_total, flipped=flipped, max_duv=float(duv.max()), p99=float(np.percentile(duv, 99))))
    assert flipped <= 0.005 * rows_total
    assert np.percentile(duv, 99) < 0.01 and (duv > 0.05).sum() <= max(1, int(0.001 * len(duv)))


def test_group_state_roundtrip_and_play(fe, synth):
    """get_state / set_state per stream resumes bit-identically; plviwo_fe_group_play equals tick-by-tick feeding; device
    resident frames equal host frames."""
    import ctypes as C
    torch = pytest.importorskip("torch")
    W, H, n_frames, S = 1280, 560, 12, 3
    seqs = [synth.SynthSequence(seed=1040 + s, width=W, height=H, n_frames=n_frames) for s in range(S)]
    frames = [[q.frame(t) for t in range(n_frames)] for q in seqs]
    cfg = fe.default_config(width=W, height=H, lookahead=3, **CFG2)
    calibs = [(q.K, q.D) for q in seqs]
    vps = [q.vanishing_points(0) for q in seqs]
    # reference: tick by tick, checksums as plviwo_fe_play computes them
    g = fe.GroupFrontEnd(cfg, S, calibs=calibs)
    chk = [0.0] * S
    snap = None
    mid = n_frames // 2
    tail = []
    for t in range(n_frames):
        if t == mid:
            snap = [g.get_state(s) for s in range(S)]
        g.feed([q.timestamp(t) for q in seqs], [frames[s][t] for s in range(S)], vanishing_points=vps)
        for s in range(S):
            r = g.point_rows(s)
            lr, _ = g.line_rows(s)
            chk[s] += float(np.sum(r["id"].astype(np.float64) + r["u"] + r["v"]))
            chk[s] += float(np.sum(lr["id"].astype(np.float64) + lr["line"].astype(np.float64).sum(1))) if len(lr) else 0.0
        if t >= mid:
            tail.append([_group_frame(g, s) for s in range(S)])
    g.close()
    # resume from the snapshot in a fresh group
    g = fe.GroupFrontEnd(cfg, S, calibs=calibs)
    for s in range(S):
        g.set_state(s, snap[s])
        assert g.get_state(s) == snap[s]
    for t in range(mid, n_frames):
        g.feed([q.timestamp(t) for q in seqs], [frames[s][t] for s in range(S)], vanishing_points=vps)
        for s in range(S):
            got = _group_frame(g, s)
            want = tail[t - mid][s]
            for a, b in zip(want[:5], got[:5]):
                assert a.tobytes() == b.tobytes(), (t, s)
            assert want[5] == got[5], (t, s)
    g.close()
    # play from device-resident frames
    d = torch.empty((n_frames, S, H, W), dtype=torch.uint8, device="cuda")
    for t in range(n_frames):
        for s in range(S):
            d[t, s].copy_(torch.from_numpy(frames[s][t]))
    torch.cuda.synchronize()
    tab = (C.c_void_p * (n_frames * S))(*[d[t, s].data_ptr() for t in range(n_frames) for s in range(S)])
    g = fe.GroupFrontEnd(cfg, S, calibs=calibs)
    st = g.play([seqs[0].timestamp(t) for t in range(n_frames)], tab, W, True, vanishing_points=vps)
    for s in range(S):
        assert st[s].frames == n_frames
        assert abs(st[s].checksum - chk[s]) <= 1e-6 * max(abs(chk[s]), 1.0), (s, st[s].checksum, chk[s])
    tm = g.times()
    assert tm["kernel_launches_total"] > 0 and tm["frames"] == n_frames * S
    g.close()


def test_group_bad_arguments(fe):
    cfg = fe.default_config(width=1280, height=560, **CFG1)
    with pytest.raises(fe.FrontEndError):
        fe.GroupFrontEnd(cfg, 0)
    bad = fe.default_config(width=1280, height=560, downsample=1, **CFG1)
    with pytest.raises(fe.FrontEndError):
        fe.GroupFrontEnd(bad, 2)
    g = fe.GroupFrontEnd(cfg, 2)
    with pytest.raises(fe.FrontEndError):
        g.collect()                      # nothing submitted
    img = np.zeros((560, 1280), np.uint8)
    g.submit([0.0, 0.0], [img, img])
    with pytest.raises(fe.FrontEndError):
        g.submit([0.1, 0.1], [img, img])  # lookahead 0: window full
    g.collect()
    with pytest.raises(fe.FrontEndError):
        g.set_state(0, b"\x00" * 16)
    with pytest.raises(fe.FrontEndError):
        g.set_state(5, b"\x00" * 128)
    g.close()


def test_group_set_state_rejects_inconsistent_blobs(fe, synth):
    """As a single handle (test_frontend_gpu.py test_capacity_and_boundary_guards): a blob whose per-line sizes do not add up
    to its header's entry count, or of an unknown version, is refused with the reason and leaves the stream's state as it was."""
    W, H = 1280, 560
    seq = synth.SynthSequence(seed=3, width=W, height=H, n_frames=3, hard=False)
    g = fe.GroupFrontEnd(fe.default_config(width=W, height=H, **CFG1), 2, calibs=[(seq.K, seq.D)] * 2)
    for t in range(3):
        g.feed([seq.timestamp(t)] * 2, [seq.frame(t)] * 2, vanishing_points=[seq.vanishing_points(t)] * 2)
    before = g.get_state(0)
    hdr = np.frombuffer(before[:56], fe._STATE_HDR, 1)[0]
    n_pts, n_lines = int(hdr["n_pts"]), int(hdr["n_lines"])
    assert n_lines > 0
    blob = bytearray(before)
    off = 56 + 16 * n_pts + 24 * n_lines          # the int32 sizes array
    sizes = np.frombuffer(bytes(blob[off:off + 4 * n_lines]), np.int32).copy()
    sizes[0] += 5
    blob[off:off + 4 * n_lines] = sizes.tobytes()
    with pytest.raises(fe.FrontEndError, match="line sizes do not add up"):
        g.set_state(0, bytes(blob))
    assert g.get_state(0) == before
    bad = bytearray(before)
    bad[4:8] = np.uint32(7).tobytes()             # unknown version
    with pytest.raises(fe.FrontEndError, match="foreign blob"):
        g.set_state(0, bytes(bad))
    assert g.get_state(0) == before
    g.close()
