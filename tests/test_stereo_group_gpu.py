"""Stereo group (plviwo_fe_stereo_group_*) through the C ABI.

The bar: rig r of a stereo group produces, pair by pair, EXACTLY what one FeStereoHandle produces on the same pairs —
point rows and pts_last / ids_last of both cameras, every FeStereoInfo field, the left image's line rows and line points,
the state blob — while the group batches the kernels of all rigs and runs the stereo state machine on the device.
Teacher-forced against the oracle (oracle/stereo.py), the bars of tests/test_stereo_gpu.py.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import frontend as ofe
from oracle import stereo as ost

pytestmark = pytest.mark.gpu

CFG1 = dict(num_features=200, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10, pyr_levels=3, win_size=15)
CFG2 = dict(num_features=400, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10, pyr_levels=4, win_size=15)
CFG_KAIST = dict(num_features=1500, fast_threshold=30, grid_x=15, grid_y=15, min_px_dist=15, pyr_levels=5, win_size=15)
CFG4 = dict(num_features=1000, fast_threshold=20, grid_x=10, grid_y=6, min_px_dist=15, pyr_levels=5, win_size=21)
CFG_DEEP = dict(CFG_KAIST, pyr_levels=6)   # at 1280 x 560 the pyramid stops at 6 images (40 x 18): the 15 x 15 bodies


def _info_bytes(info):
    return C.string_at(C.addressof(info), C.sizeof(info))


def _rig_seq(synth, seed, W, H, n, moving_mask=False):
    return synth.SynthSequence(seed=seed, width=W, height=H, n_frames=n, moving_mask=moving_mask)


def _k_right(seq, r):
    return tuple(v * (1.0 + 0.004 * (r + 1)) for v in seq.K)


def _pairs(seq, n, skip=False, black_at=None):
    """Per tick the rig's (left, right) pair or None: `skip` drops every second tick, `black_at` feeds a black pair."""
    out = []
    for t in range(n):
        if skip and t % 2 == 1:
            out.append(None)
        elif t == black_at:
            z = np.zeros_like(seq.frame(t, 0))
            out.append((z, z))
        else:
            out.append((seq.frame(t, 0), seq.frame(t, 1)))
    return out


def _masks(seq, t, on):
    return (seq.mask(t, 0), seq.mask(t, 1)) if on else None


def _handle_frames(fe, seq, kw, pairs, W, H, K_right, lines, masks, hist):
    """What one FeStereoHandle gives, pair by pair (None where the rig has no pair)."""
    h = fe.StereoFrontEnd(fe.default_config(width=W, height=H, K=seq.K, D=seq.D, lookahead=0, histogram_method=hist,
                                            use_lines=1 if lines else 0, **kw), K_right=K_right)
    out = []
    for t, p in enumerate(pairs):
        if p is None:
            out.append(None)
            continue
        m = _masks(seq, t, masks)
        info = h.feed_new_camera(seq.timestamp(t), p[0], p[1], m[0] if m else None, m[1] if m else None,
                                 vanishing_points=seq.vanishing_points(t) if lines else None, update_db=False)
        lr, lp = h.line_rows()
        out.append(dict(info=_info_bytes(info), rows=[h.point_rows(c).copy() for c in (0, 1)],
                        obs=[h._last(c) for c in (0, 1)], lr=lr.copy(), lp=lp.copy(), blob=h.get_state()))
    h.close()
    return out


def _assert_rig(g, r, ref, where, blob=False):
    assert _info_bytes(g.infos[r]) == ref["info"], "stereo info differs " + where
    for c in (0, 1):
        assert g.point_rows(r, c).tobytes() == ref["rows"][c].tobytes(), "point rows of camera %d differ %s" % (c, where)
        ids, uv = g.last_obs(r, c)
        assert ids.tobytes() == ref["obs"][c][0].tobytes() and uv.tobytes() == ref["obs"][c][1].tobytes(), "last obs of camera %d differ %s" % (c, where)
    lr, lp = g.line_rows(r)
    assert lr.tobytes() == ref["lr"].tobytes() and lp.tobytes() == ref["lp"].tobytes(), "line rows differ " + where
    if blob:
        assert g.get_state(r) == ref["blob"], "state blob differs " + where


def _run_group(fe, synth, kw, n_rigs, n, W=1280, H=560, lookahead=0, lines=True, masks=False, hist=1, skip_rig=None,
               black_rig=None, seed0=2000, check_blob=False):
    seqs = [_rig_seq(synth, seed0 + r, W, H, n, moving_mask=masks) for r in range(n_rigs)]
    pairs = [_pairs(q, n, skip=(r == skip_rig), black_at=(n // 2 if r == black_rig else None)) for r, q in enumerate(seqs)]
    ref = [_handle_frames(fe, q, kw, pairs[r], W, H, _k_right(q, r), lines, masks, hist) for r, q in enumerate(seqs)]
    cfg = fe.default_config(width=W, height=H, lookahead=lookahead, histogram_method=hist, use_lines=1 if lines else 0, **kw)
    g = fe.StereoGroupFrontEnd(cfg, n_rigs, calibs=[((q.K, q.D), (_k_right(q, r), q.D)) for r, q in enumerate(seqs)])
    sub = 0
    events = dict(reset=0, first=0)
    for t in range(n):
        while sub < n and sub <= t + lookahead:
            g.submit([q.timestamp(sub) for q in seqs], [pairs[r][sub] for r in range(n_rigs)],
                     vanishing_points=[q.vanishing_points(sub) for q in seqs] if lines else None,
                     masks=[_masks(q, sub, masks) if pairs[r][sub] is not None else None for r, q in enumerate(seqs)] if masks else None)
            sub += 1
        g.collect()
        for r in range(n_rigs):
            if ref[r][t] is None:
                assert g.infos[r].timestamp == -1.0, (r, t)
                continue
            _assert_rig(g, r, ref[r][t], "rig %d pair %d" % (r, t), blob=check_blob and sub == t + 1)
            if r == black_rig and t > n // 2:
                events["reset"] += int(g.infos[r].reset)
                events["first"] += int(g.infos[r].first_frame)
    g.close()
    return ref, events


@pytest.mark.parametrize("lookahead", [0, 4])
def test_stereo_group_equals_stereo_handles(fe, synth, lookahead):
    """CFG2 at 1280 x 560, 3 rigs with their own seeds and right calibrations, lines on."""
    ref, _ = _run_group(fe, synth, CFG2, 3, 12, lookahead=lookahead, check_blob=lookahead == 0)
    assert sum(len(x["rows"][1]) for r in ref for x in r if x) > 1000
    assert sum(len(x["lr"]) for r in ref for x in r if x) > 30


@pytest.mark.parametrize("kw,W,H,n", [(CFG_KAIST, 1280, 560, 6), (CFG4, 1920, 1080, 5), (CFG_DEEP, 1280, 560, 6)])
def test_stereo_group_kaist_yaml_and_wide_window(fe, synth, kw, W, H, n):
    """KAIST yaml knobs (1500 points, 15 x 15 grid), config 4 (1920 x 1080, 21 x 21 window: the generic LK kernel) and
    pyr_levels 6 at 1280 x 560 (a pyramid of 6 images: the 15 x 15 kernels, as in a handle)."""
    _run_group(fe, synth, kw, 2, n, W=W, H=H, seed0=2100)


@pytest.mark.parametrize("masks,hist,lines", [(True, 2, True), (False, 0, False)])
def test_stereo_group_masks_preprocessing_gaps_and_black_pair(fe, synth, masks, hist, lines):
    """Moving masks with CLAHE, and no equalisation with lines off; rig 1 skips every second tick, rig 2 gets a black pair
    halfway, after which the rig resets or starts over."""
    _, ev = _run_group(fe, synth, CFG1, 3, 10, masks=masks, hist=hist, lines=lines, skip_rig=1, black_rig=2, seed0=2200)
    assert ev["reset"] + ev["first"] >= 1, ev


def test_stereo_group_teacher_forced_against_oracle(fe, synth):
    """State loaded from the oracle before every pair (set_state per rig); bars of test_stereo_gpu._assert_parity."""
    from test_stereo_gpu import _assert_parity, _blob
    W, H, n, R = 1280, 560, 12, 2
    seqs = [_rig_seq(synth, 2300 + r, W, H, n) for r in range(R)]
    orc = [ost.TrackKLTStereo(ofe.FeConfig(K=q.K, D=q.D, **CFG1)) for q in seqs]
    g = fe.StereoGroupFrontEnd(fe.default_config(width=W, height=H, use_lines=0, **CFG1), R,
                               calibs=[((q.K, q.D), (q.K, q.D)) for q in seqs])
    stats = [dict(rows=0, rows_sym=0, order_equal=0, frames_equal=0, duv=[0.0], dun=[0.0]) for _ in range(R)]
    z = np.zeros((H, W), np.uint8)
    for t in range(n):
        if t > 0:
            for r in range(R):
                g.set_state(r, _blob(fe, orc[r], W, H))
        rows_o = [orc[r].feed_new_camera(seqs[r].timestamp(t), seqs[r].frame(t, 0), seqs[r].frame(t, 1), z, z) for r in range(R)]
        infos = g.feed([q.timestamp(t) for q in seqs], [(q.frame(t, 0), q.frame(t, 1)) for q in seqs])
        for r in range(R):
            o, s = orc[r], stats[r]
            assert bool(infos[r].reset) == bool(o.trace["reset"]) and bool(infos[r].first_frame) == bool(o.trace["first"]), (r, t)
            equal = True
            for cam in (0, 1):
                rows = g.point_rows(r, cam)
                ids_o = {x.id: x for x in rows_o[r][cam]}
                ids_g = {int(x["id"]): x for x in rows}
                sym = set(ids_o) ^ set(ids_g)
                s["rows"] += len(ids_o)
                s["rows_sym"] += len(sym)
                if sym:
                    equal = False
                else:
                    s["order_equal"] += int([x.id for x in rows_o[r][cam]] == [int(v) for v in rows["id"]])
                for fid in set(ids_o) & set(ids_g):
                    a, b = ids_g[fid], ids_o[fid]
                    s["duv"].append(max(abs(float(a["u"]) - b.u), abs(float(a["v"]) - b.v)))
                    s["dun"].append(max(abs(float(a["un"]) - b.un), abs(float(a["vn"]) - b.vn)))
            s["frames_equal"] += int(equal)
    g.close()
    for s in stats:
        duv, dun = np.array(s.pop("duv")), np.array(s.pop("dun"))
        s.update(duv_p99=float(np.percentile(duv, 99)), n_duv_gt_005=int((duv > 0.05).sum()), dun_p99=float(np.percentile(dun, 99)))
        print(s)
        _assert_parity(s)


def test_stereo_group_state_and_play(fe, synth):
    """get_state equals the stereo handle's blob; a handle's blob loaded into a rig continues as the handle does; play gives
    the FePlayStats and last rows of submit / collect; set_state refuses foreign, truncated and unknown-version blobs with
    the reason and leaves the rig as it was."""
    W, H, n = 1280, 560, 8
    seq = _rig_seq(synth, 2400, W, H, n)
    kw = dict(width=W, height=H, K=seq.K, D=seq.D, use_lines=0, **CFG1)
    h = fe.StereoFrontEnd(fe.default_config(**kw))
    ref = []
    for t in range(n):
        h.feed_new_camera(seq.timestamp(t), seq.frame(t, 0), seq.frame(t, 1), update_db=False)
        ref.append(([h.point_rows(c).copy() for c in (0, 1)], h.get_state()))
    h.close()
    g = fe.StereoGroupFrontEnd(fe.default_config(**kw), 2)
    for t in range(4):
        g.feed([seq.timestamp(t)] * 2, [(seq.frame(t, 0), seq.frame(t, 1)), None])
        assert g.get_state(0) == ref[t][1], t
    # rig 1 resumes from the handle's checkpoint after pair 3
    g.set_state(1, ref[3][1])
    assert g.get_state(1) == ref[3][1]
    for t in range(4, n):
        g.feed([seq.timestamp(t)] * 2, [(seq.frame(t, 0), seq.frame(t, 1))] * 2)
        for r in (0, 1):
            for c in (0, 1):
                assert g.point_rows(r, c).tobytes() == ref[t][0][c].tobytes(), (r, c, t)
            assert g.get_state(r) == ref[t][1], (r, t)
    # refusals: the rig's state is unchanged
    before = g.get_state(0)
    mono = fe.pack_state(W, H, 5, np.zeros((0, 2), np.float32), np.zeros(0, np.uint64), None, None)
    for blob, why in ((mono, "not a stereo state blob"), (before[:-100], "truncated"),
                      (before[:4] + (7).to_bytes(4, "little") + before[8:], "unknown stereo state version")):
        with pytest.raises(fe.FrontEndError) as e:
            g.set_state(0, blob)
        assert e.value.code == fe.FE_BAD_ARG and why in str(e.value), str(e.value)
        assert g.get_state(0) == before
    g.close()
    # play = submit / collect
    imgs = [[np.ascontiguousarray(seq.frame(t, c)) for c in (0, 1)] for t in range(n)]
    tab = (C.c_void_p * (n * 2 * 2))()
    for t in range(n):
        for r in range(2):
            for c in (0, 1):
                tab[(t * 2 + r) * 2 + c] = imgs[t][c].ctypes.data
    ts = [seq.timestamp(t) for t in range(n)]
    vps = [seq.vanishing_points(0)] * 2
    cfg = fe.default_config(width=W, height=H, K=seq.K, D=seq.D, use_lines=1, lookahead=3, **CFG1)
    a = fe.StereoGroupFrontEnd(cfg, 2)
    st = a.play(ts, tab, W, False, vanishing_points=vps)
    last = [[a.point_rows(r, c).copy() for c in (0, 1)] + [a.line_rows(r)[0].copy()] for r in range(2)]
    a.close()
    b = fe.StereoGroupFrontEnd(cfg, 2)
    exp = [dict(frames=0, point_rows=0, line_rows=0, resets=0, checksum=0.0) for _ in range(2)]
    for t in range(n):
        infos = b.feed([ts[t]] * 2, [(imgs[t][0], imgs[t][1])] * 2, vanishing_points=vps)
        for r in range(2):
            x = exp[r]
            x["frames"] += 1
            x["resets"] += int(infos[r].reset)
            for c in (0, 1):
                pr = b.point_rows(r, c)
                x["point_rows"] += len(pr)
                x["checksum"] += float(sum(float(p["id"]) + float(p["u"]) + float(p["v"]) for p in pr))
            lr = b.line_rows(r)[0]
            x["line_rows"] += len(lr)
            x["checksum"] += float(sum(float(l["id"]) + float(l["line"][0]) + float(l["line"][1]) + float(l["line"][2]) + float(l["line"][3]) for l in lr))
    for r in range(2):
        assert (st[r].frames, st[r].point_rows, st[r].line_rows, st[r].resets) == \
            (exp[r]["frames"], exp[r]["point_rows"], exp[r]["line_rows"], exp[r]["resets"]), r
        assert abs(st[r].checksum - exp[r]["checksum"]) <= 1e-9 * max(1.0, abs(exp[r]["checksum"])), r
        for c in (0, 1):
            assert b.point_rows(r, c).tobytes() == last[r][c].tobytes(), (r, c)
        assert b.line_rows(r)[0].tobytes() == last[r][2].tobytes(), r
    b.close()


def test_stereo_group_rig_isolation(fe, synth):
    """A rig's rows do not depend on how many other rigs share the group: 1 rig against 5 rigs."""
    W, H, n = 1280, 560, 8
    seqs = [_rig_seq(synth, 2500 + r, W, H, n) for r in range(5)]
    out = {}
    for R in (1, 5):
        g = fe.StereoGroupFrontEnd(fe.default_config(width=W, height=H, lookahead=2, **CFG1), R,
                                   calibs=[((q.K, q.D), (q.K, q.D)) for q in seqs[:R]])
        rows = []
        for t in range(n):
            g.feed([q.timestamp(t) for q in seqs[:R]], [(q.frame(t, 0), q.frame(t, 1)) for q in seqs[:R]],
                   vanishing_points=[q.vanishing_points(t) for q in seqs[:R]])
            rows.append((g.point_rows(0, 0).tobytes(), g.point_rows(0, 1).tobytes(), g.line_rows(0)[0].tobytes(), _info_bytes(g.infos[0])))
        out[R] = rows
        g.close()
    assert out[1] == out[5]


def test_stereo_group_bad_arguments(fe, synth):
    W, H = 640, 280
    seq = _rig_seq(synth, 2600, W, H, 3)
    g = fe.StereoGroupFrontEnd(fe.default_config(width=W, height=H, use_lines=0, **dict(CFG1, num_features=100)), 2)
    a, b = seq.frame(0, 0), seq.frame(0, 1)
    with pytest.raises(fe.FrontEndError) as e:
        g.submit([0.0, 0.0], [(a, b), (a, None)])                  # exactly one image of a pair
    assert e.value.code == fe.FE_BAD_ARG and "exactly one image" in str(e.value)
    with pytest.raises(fe.FrontEndError):
        g.collect()                                                # ... and nothing was enqueued
    for rig, cam in ((2, 0), (-1, 0), (0, 2)):
        with pytest.raises(fe.FrontEndError) as e:
            g.set_calib(rig, cam, seq.K, seq.D)
        assert e.value.code == fe.FE_BAD_ARG
    with pytest.raises(fe.FrontEndError) as e:
        g.set_camera(0, 1, 1, seq.K, seq.D)                        # FE_CAM_EQUI
    assert e.value.code == fe.FE_BAD_ARG and "radtan" in str(e.value)
    g.feed([0.0, 0.0], [(a, b), (a, b)])
    with pytest.raises(fe.FrontEndError):
        g.point_rows(2, 0)
    with pytest.raises(fe.FrontEndError):
        g.last_obs(0, 2)
    g.close()
