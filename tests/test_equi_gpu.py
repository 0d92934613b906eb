"""Equidistant (fisheye) camera model on the GPU: the kernel against the host form and cv2, a handle teacher-forced against
the oracle driven through cv::fisheye::undistortPoints, stream groups and stereo rigs bit for bit with handles, the model
gate of set_camera, and radtan objects from the _create_model creators equal to the old creators."""
import ctypes as C

import numpy as np
import pytest

from oracle import cvops
from oracle import frontend as ofe
from oracle import stereo as ost
from test_equi_cpu import EUROC_D, EUROC_K, STRONG_D, EquiOps, _points
from test_group_gpu import _assert_same, _group_frame
from test_stereo_group_gpu import _assert_rig, _info_bytes, _k_right
from test_stereo_gpu import _assert_parity, _blob

pytestmark = pytest.mark.gpu

CFG1 = dict(num_features=200, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10, pyr_levels=3, win_size=15)
CFG2 = dict(num_features=400, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10, pyr_levels=4, win_size=15)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32).tobytes()


def test_kernel_equals_host_form_and_cv2(fe):
    rng = np.random.default_rng(11)
    big = np.stack([rng.uniform(-400, 1150, 10 ** 6), rng.uniform(-400, 880, 10 ** 6)], 1).astype(np.float32)
    for D in (EUROC_D, STRONG_D):
        assert _bits(fe.op_undistort_equi(big, EUROC_K, D)) == _bits(fe.op_undistort_equi(big, EUROC_K, D, device=-1))
        for wide in (False, True):
            pts = _points(wide=wide)
            assert _bits(fe.op_undistort_equi(pts, EUROC_K, D)) == _bits(cvops.undistort_equi(pts, EUROC_K, D))


def _oracle_blob(fe, oracle, W, H):
    k = oracle.klt.get_state()
    l = oracle.lsd.get_state()
    return fe.pack_state(W, H, k["currid"], k["pts_last"], k["ids_last"], k["img_last"], k["mask_last"], l["currid"],
                         l["lines_last"], l["ids_last"], l["pol_last"])


def _teacher_forced(fe, synth, kw, D, n_frames, seed, K=None, W=1280, H=560):
    """A handle created with FE_CAM_EQUI against the oracle with CamEqui's undistortion, state loaded from the oracle before
    every frame.  Returns the counters the bars are asserted on."""
    seq = synth.SynthSequence(seed=seed, width=W, height=H, n_frames=n_frames, hard=True)
    K = seq.K if K is None else K
    oracle = ofe.FrontEnd(ofe.FeConfig(K=K, D=tuple(D), **kw), ops=EquiOps(cvops))
    gpu = fe.FrontEnd(fe.default_config(width=W, height=H, K=K, D=D, **kw), camera_model=fe.CAM_EQUI)
    gpu.enable_taps(True)
    s = dict(rows=0, n_feat=0, n_status_agree=0, n_klt_agree=0, gate_not_host=0, id_frames=0, id_errors=0, line_frames=0, line_errors=0, line_rows=0,
             un_not_cv2=0, line_n_not_cv2=0, failed_rows=0)
    duv = [0.0]
    for t in range(n_frames):
        if t > 0:
            gpu.set_state(_oracle_blob(fe, oracle, W, H))
        prow_o, lrow_o = oracle.feed(seq.timestamp(t), seq.frame(t), None, seq.vanishing_points(t))
        gpu.feed_new_camera(seq.timestamp(t), seq.frame(t), None, seq.vanishing_points(t), update_db=False)
        rows = gpu.point_rows()
        tr = oracle.klt.trace
        flipped = set()
        if "mask_klt" in tr:
            lk = gpu.tap(fe.TAP_LK_LAST, np.float32).reshape(-1, 6)
            assert len(lk) == len(tr["mask_klt"]), t
            rsc = tr["mask_rsc"].astype(bool) if len(tr["mask_rsc"]) else np.zeros(len(lk), bool)
            st_o = tr["mask_klt"].astype(bool) & rsc
            st_g = (lk[:, 4] > 0) & (lk[:, 5] > 0)
            s["n_feat"] += len(lk)
            s["n_status_agree"] += int((st_o == st_g).sum())
            s["n_klt_agree"] += int((tr["mask_klt"].astype(bool) == (lk[:, 4] > 0)).sum())
            # the gate's verdicts on the handle's own tracks are the host RANSAC restatement on cv2's undistortion of them
            m, _ = fe.op_ransac_fundamental(cvops.undistort_equi(lk[:, :2], K, D), cvops.undistort_equi(lk[:, 2:4], K, D),
                                            2.0 / max(K[0], K[1]))
            s["gate_not_host"] += int(not np.array_equal(m > 0, lk[:, 5] > 0))
            flipped = {int(tr["ids_old"][i]) for i in np.nonzero(st_o != st_g)[0]}
        # every row's (un, vn) is cv2.fisheye.undistortPoints of its own (u, v), bit for bit
        uv = np.stack([rows["u"], rows["v"]], 1).astype(np.float32)
        s["un_not_cv2"] += int(_bits(np.stack([rows["un"], rows["vn"]], 1)) != _bits(cvops.undistort_equi(uv, K, D)))
        s["failed_rows"] += int((rows["un"] == -1e6).sum())
        s["rows"] += len(rows)
        ids_o = {r.id: r for r in prow_o}
        ids_g = {int(r["id"]): r for r in rows}
        sym = set(ids_o) ^ set(ids_g)
        s["id_errors"] += int(not sym <= flipped)
        for fid in set(ids_o) & set(ids_g):
            a, b = ids_g[fid], ids_o[fid]
            duv.append(max(abs(float(a["u"]) - b.u), abs(float(a["v"]) - b.v)))
        lrows, lpts = gpu.line_rows()
        for r in lrows:   # line_n is cv2's result on the row's own endpoints
            e = cvops.undistort_equi(np.array(r["line"], np.float32).reshape(2, 2), K, D).reshape(4)
            s["line_n_not_cv2"] += int(_bits(r["line_n"]) != _bits(e))
        if not sym:
            s["id_frames"] += 1
            assert [r.id for r in prow_o] == [int(v) for v in rows["id"]], "row order differs at frame %d" % t
            s["line_frames"] += 1
            s["line_rows"] += len(lrow_o)
            ok = len(lrows) == len(lrow_o)
            for a, b in zip(lrows, lrow_o):
                p = lpts[a["pt_offset"]:a["pt_offset"] + a["n_pts"]]
                ok = ok and int(a["id"]) == b.id and int(a["D"]) == b.D and list(p["pid"]) == list(b.pids)
            s["line_errors"] += int(not ok)
    gpu.close()
    duv = np.array(duv)
    s.update(duv_p99=float(np.percentile(duv, 99)), n_duv_gt_005=int((duv > 0.05).sum()), n_uv=len(duv) - 1)
    print(s)
    return s


def _assert_bars(s, status=True):
    assert s["rows"] > 0 and s["id_errors"] == 0, s
    assert s["n_klt_agree"] >= 0.995 * s["n_feat"] and s["gate_not_host"] == 0, s
    if status:
        assert s["n_status_agree"] >= 0.995 * s["n_feat"], s
    assert s["duv_p99"] < 0.01 and s["n_duv_gt_005"] <= max(1, int(0.001 * s["n_uv"])), s
    assert s["line_errors"] == 0, s
    assert s["un_not_cv2"] == 0 and s["line_n_not_cv2"] == 0, s


def test_handle_teacher_forced_euroc_lens(fe, synth):
    s = _teacher_forced(fe, synth, CFG2, EUROC_D, 12, seed=1100)
    _assert_bars(s)
    assert s["line_rows"] > 10 and s["id_frames"] >= 6, s


def test_handle_teacher_forced_strong_lens(fe, synth):
    """The strong lens behind a short focal length: the image corners reach the 90 degree clamp, so rows of non-converged
    points ((-1e6, -1e6)) go through the RANSAC gate.  Near the clamp tan(theta) magnifies the 1e-4 px by which the kernel's
    LK and cv2's differ into normalised differences far above the gate's 2 / f threshold, so the gate's verdicts are compared
    with the RANSAC restatement on the handle's own tracks instead of with the oracle's verdicts on its tracks.  (On inputs
    with many (-1e6, -1e6) points that restatement and cv2.findFundamentalMat do not always agree; with real lenses such
    points are rare.)"""
    K = (400.0, 400.0, 640.0, 280.0)   # about one pixel in eight of the 1280 x 560 frame does not converge
    s = _teacher_forced(fe, synth, CFG1, STRONG_D, 6, seed=1101, K=K)
    _assert_bars(s, status=False)
    assert s["failed_rows"] > 0, s


def _handle_rows(fe, seq, kw, D, n_frames, W, H, model, create_model=True):
    h = fe.FrontEnd(fe.default_config(width=W, height=H, K=seq.K, D=D, lookahead=0, **kw), camera_model=model)
    if not create_model:   # the same object behind a handle from the creator without a model (plviwo_fe_create)
        h.close()
        fe._check(h._lib.plviwo_fe_create(C.byref(h.cfg), 0, C.byref(h._h)))
    out = []
    for t in range(n_frames):
        info = h.feed_new_camera(seq.timestamp(t), seq.frame(t), None, seq.vanishing_points(t), update_db=False)
        lr, lp = h.line_rows()
        ids, uv = h._last()
        out.append(dict(rows=h.point_rows(), lrows=lr, lpts=lp, ids=ids, uv=uv,
                        info=(info.reset, info.first_frame, info.n_detected, info.detection_ran, info.n_lk_in, info.n_klt_ok,
                              info.n_ransac_ok, info.n_lines_detected, info.n_line_matches)))
    h.close()
    return out


def _group_vs_handles(fe, synth, kw, D, lookahead, model, n_streams=3, n_frames=10, W=1280, H=560, line_samples=0,
                      create_model=True):
    seqs = [synth.SynthSequence(seed=1110 + s, width=W, height=H, n_frames=n_frames) for s in range(n_streams)]
    ref = [_handle_rows(fe, q, dict(kw, line_samples=line_samples), D, n_frames, W, H, model) for q in seqs]
    cfg = fe.default_config(width=W, height=H, lookahead=lookahead, line_samples=line_samples, **kw)
    g = fe.GroupFrontEnd(cfg, n_streams, calibs=[(q.K, D) for q in seqs], camera_model=model)
    if not create_model:   # a handle from plviwo_fe_group_create instead
        g.close()
        g._check(g._lib.plviwo_fe_group_create(C.byref(cfg), n_streams, 0, C.byref(g._h)))
        for s_, q in enumerate(seqs):
            g.set_calib(s_, q.K, D)
    sub = 0
    for t in range(n_frames):
        while sub < n_frames and sub <= t + lookahead:
            g.submit([q.timestamp(sub) for q in seqs], [q.frame(sub) for q in seqs],
                     vanishing_points=[q.vanishing_points(sub) for q in seqs])
            sub += 1
        g.collect()
        for s in range(n_streams):
            _assert_same(ref[s][t], _group_frame(g, s), "stream %d frame %d" % (s, t))
    g.close()
    return ref


@pytest.mark.parametrize("lookahead", [0, 4])
def test_group_equals_equidistant_handles(fe, synth, lookahead):
    ref = _group_vs_handles(fe, synth, CFG2, EUROC_D, lookahead, fe.CAM_EQUI)
    assert sum(len(x["lrows"]) for r in ref for x in r) > 20


def test_group_equals_equidistant_handles_line_samples(fe, synth):
    _group_vs_handles(fe, synth, CFG1, STRONG_D, 2, fe.CAM_EQUI, n_streams=2, n_frames=8, line_samples=6)


def test_stereo_handle_teacher_forced(fe, synth):
    W, H, n = 1280, 560, 16
    seq = synth.SynthSequence(seed=1120, width=W, height=H, n_frames=n, hard=True)
    kr = tuple(v * 1.01 for v in seq.K)
    o = ost.TrackKLTStereo(ofe.FeConfig(K=seq.K, D=tuple(EUROC_D), **CFG2), K_right=kr, ops=EquiOps(cvops))
    g = fe.StereoFrontEnd(fe.default_config(width=W, height=H, K=seq.K, D=EUROC_D, use_lines=0, **CFG2), K_right=kr,
                          camera_model=fe.CAM_EQUI)
    s = dict(rows=0, rows_sym=0, order_equal=0, frames_equal=0)
    duv, dun = [0.0], [0.0]
    for t in range(n):
        il, ir = seq.frame(t, 0), seq.frame(t, 1)
        if t > 0:
            g.set_state(_blob(fe, o, W, H))
        rows_o = o.feed_new_camera(seq.timestamp(t), il, ir, np.zeros_like(il), np.zeros_like(il))
        g.feed_new_camera(seq.timestamp(t), il, ir)
        eq = True
        for cam in (0, 1):
            rows = g.point_rows(cam)
            uv = np.stack([rows["u"], rows["v"]], 1).astype(np.float32)
            assert _bits(np.stack([rows["un"], rows["vn"]], 1)) == _bits(cvops.undistort_equi(uv, (seq.K, kr)[cam], EUROC_D))
            ids_o = {r.id: r for r in rows_o[cam]}
            ids_g = {int(r["id"]): r for r in rows}
            sym = set(ids_o) ^ set(ids_g)
            s["rows"] += len(ids_o)
            s["rows_sym"] += len(sym)
            eq = eq and not sym
            if not sym:
                s["order_equal"] += int([r.id for r in rows_o[cam]] == [int(v) for v in rows["id"]])
            for fid in set(ids_o) & set(ids_g):
                a, b = ids_g[fid], ids_o[fid]
                duv.append(max(abs(float(a["u"]) - b.u), abs(float(a["v"]) - b.v)))
                dun.append(max(abs(float(a["un"]) - b.un), abs(float(a["vn"]) - b.vn)))
        s["frames_equal"] += int(eq)
    g.close()
    duv, dun = np.array(duv), np.array(dun)
    s.update(duv_p99=float(np.percentile(duv, 99)), n_duv_gt_005=int((duv > 0.05).sum()), dun_p99=float(np.percentile(dun, 99)))
    print(s)
    _assert_parity(s)


@pytest.mark.parametrize("lookahead", [0, 2])
def test_stereo_group_equals_equidistant_stereo_handles(fe, synth, lookahead):
    W, H, n, n_rigs = 1280, 560, 10, 2
    seqs = [synth.SynthSequence(seed=1130 + r, width=W, height=H, n_frames=n) for r in range(n_rigs)]
    ref = []
    for r, q in enumerate(seqs):
        h = fe.StereoFrontEnd(fe.default_config(width=W, height=H, K=q.K, D=EUROC_D, lookahead=0, **CFG2), K_right=_k_right(q, r),
                              camera_model=fe.CAM_EQUI)
        out = []
        for t in range(n):
            info = h.feed_new_camera(q.timestamp(t), q.frame(t, 0), q.frame(t, 1), vanishing_points=q.vanishing_points(t),
                                     update_db=False)
            lr, lp = h.line_rows()
            out.append(dict(info=_info_bytes(info), rows=[h.point_rows(c).copy() for c in (0, 1)], obs=[h._last(c) for c in (0, 1)],
                            lr=lr.copy(), lp=lp.copy(), blob=h.get_state()))
        h.close()
        ref.append(out)
    g = fe.StereoGroupFrontEnd(fe.default_config(width=W, height=H, lookahead=lookahead, **CFG2), n_rigs,
                               calibs=[((q.K, EUROC_D), (_k_right(q, r), EUROC_D)) for r, q in enumerate(seqs)],
                               camera_model=fe.CAM_EQUI)
    sub = 0
    for t in range(n):
        while sub < n and sub <= t + lookahead:
            g.submit([q.timestamp(sub) for q in seqs], [(q.frame(sub, 0), q.frame(sub, 1)) for q in seqs],
                     vanishing_points=[q.vanishing_points(sub) for q in seqs])
            sub += 1
        g.collect()
        for r in range(n_rigs):
            _assert_rig(g, r, ref[r][t], "rig %d pair %d" % (r, t), blob=lookahead == 0)
    g.close()
    assert sum(len(x["rows"][1]) for r in ref for x in r) > 500


def test_model_gate(fe, synth):
    """The model an object was created with updates K / D and the next frame follows them; the other model is refused."""
    W, H = 640, 280
    seq = synth.SynthSequence(seed=1140, width=W, height=H, n_frames=3, hard=False)
    kw = dict(CFG1, num_features=120)
    K2 = tuple(v * 1.02 for v in seq.K)
    cfg = fe.default_config(width=W, height=H, K=seq.K, D=EUROC_D, **kw)

    def follows(rows, K, D):
        uv = np.stack([rows["u"], rows["v"]], 1).astype(np.float32)
        return len(rows) > 0 and _bits(np.stack([rows["un"], rows["vn"]], 1)) == _bits(cvops.undistort_equi(uv, K, D))

    h = fe.FrontEnd(cfg, camera_model=fe.CAM_EQUI)
    g = fe.GroupFrontEnd(fe.default_config(width=W, height=H, K=seq.K, D=EUROC_D, **kw), 1, camera_model=fe.CAM_EQUI)
    sg = fe.StereoGroupFrontEnd(fe.default_config(width=W, height=H, K=seq.K, D=EUROC_D, **kw), 1, camera_model=fe.CAM_EQUI)
    st = fe.StereoFrontEnd(fe.default_config(width=W, height=H, K=seq.K, D=EUROC_D, **kw), camera_model=fe.CAM_EQUI)
    for t in range(2):
        h.feed_new_camera(seq.timestamp(t), seq.frame(t), None, None, update_db=False)
        g.feed([seq.timestamp(t)], [seq.frame(t)])
        sg.feed([seq.timestamp(t)], [(seq.frame(t, 0), seq.frame(t, 1))])
        st.feed_new_camera(seq.timestamp(t), seq.frame(t, 0), seq.frame(t, 1), update_db=False)
    h.set_camera(fe.CAM_EQUI, K2, STRONG_D)
    g.set_camera(0, fe.CAM_EQUI, K2, STRONG_D)
    sg.set_camera(0, 0, fe.CAM_EQUI, K2, STRONG_D)
    st.set_camera(0, fe.CAM_EQUI, K2, STRONG_D)
    for refuse in (lambda: h.set_camera(fe.CAM_RADTAN, K2, STRONG_D), lambda: g.set_camera(0, fe.CAM_RADTAN, K2, STRONG_D),
                   lambda: sg.set_camera(0, 1, fe.CAM_RADTAN, K2, STRONG_D), lambda: st.set_camera(1, fe.CAM_RADTAN, K2, STRONG_D)):
        with pytest.raises(fe.FrontEndError) as e:
            refuse()
        assert e.value.code == fe.FE_BAD_ARG and "equidistant" in str(e.value), str(e.value)
    h.feed_new_camera(seq.timestamp(2), seq.frame(2), None, None, update_db=False)
    g.feed([seq.timestamp(2)], [seq.frame(2)])
    sg.feed([seq.timestamp(2)], [(seq.frame(2, 0), seq.frame(2, 1))])
    st.feed_new_camera(seq.timestamp(2), seq.frame(2, 0), seq.frame(2, 1), update_db=False)
    assert follows(h.point_rows(), K2, STRONG_D)
    assert follows(g.point_rows(0), K2, STRONG_D)
    assert follows(sg.point_rows(0, 0), K2, STRONG_D) and follows(sg.point_rows(0, 1), seq.K, EUROC_D)
    assert follows(st.point_rows(0), K2, STRONG_D) and follows(st.point_rows(1), seq.K, EUROC_D)
    for o in (h, g, sg, st):
        o.close()


def test_radtan_model_creators_equal_old_creators(fe, synth):
    """_create_model(FE_CAM_RADTAN) is the old creator: a handle and a group give the same rows, bit for bit."""
    W, H, n = 1280, 560, 8
    seq = synth.SynthSequence(seed=1150, width=W, height=H, n_frames=n)
    a = _handle_rows(fe, seq, CFG2, seq.D, n, W, H, fe.CAM_RADTAN)
    b = _handle_rows(fe, seq, CFG2, seq.D, n, W, H, fe.CAM_RADTAN, create_model=False)
    for t in range(n):
        _assert_same(a[t], (b[t]["rows"], b[t]["lrows"], b[t]["lpts"], b[t]["ids"], b[t]["uv"], b[t]["info"]), "frame %d" % t)
    # a radtan group against radtan handles, created with and without the model
    for create_model in (True, False):
        _group_vs_handles(fe, synth, CFG2, synth.KAIST_D, 2, fe.CAM_RADTAN, n_streams=2, n_frames=6, create_model=create_model)
