"""Front-end parity through the C ABI against the oracle (north_star bars: FAST corners and feature IDs
bit-exact, tracked UVs within 0.05 px, KLT/RANSAC status flags equal on >= 99.5 % of features).

Two modes (SURVEY.md 7.3 item 2):
  * teacher-forced: before every frame the GPU tracker is loaded with the oracle's state (plviwo_fe_set_state), so
    each frame is compared on IDENTICAL inputs — this is where the 0.05 px / bit-exact bars are asserted;
  * free-running: both run on their own state.  IDs and status flags must still agree; UV differences are reported
    as p99 / max because a single ill-conditioned (edge-like) feature drifts once the two trackers' inputs differ
    by 1e-3 px — OpenCV itself moves such a feature by 0.1 px for a 0.005 px change of its input.
"""
import numpy as np
import pytest

from oracle import frontend as ofe

pytestmark = pytest.mark.gpu

CFG1 = dict(num_features=200, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10, pyr_levels=3, win_size=15)
CFG2 = dict(num_features=400, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10, pyr_levels=4, win_size=15)
CFG_KAIST = dict(num_features=1500, fast_threshold=30, grid_x=15, grid_y=15, min_px_dist=15, pyr_levels=5, win_size=15)
CFG4 = dict(num_features=1000, fast_threshold=20, grid_x=10, grid_y=6, min_px_dist=15, pyr_levels=5, win_size=21)


def _oracle_state_blob(fe, oracle, W, H):
    k = oracle.klt.get_state()
    l = oracle.lsd.get_state() if oracle.lsd is not None else dict(currid=1, lines_last=None, ids_last=None, pol_last=None)
    return fe.pack_state(W, H, k["currid"], k["pts_last"], k["ids_last"], k["img_last"], k["mask_last"], l["currid"],
                         l["lines_last"], l["ids_last"], l["pol_last"])


def _compare_lines(lrows, lpts, lrow_o):
    """Line rows: ids, class, matched points bit-exact; endpoints to 2e-3 px (device vs host libm in fitLine)."""
    if len(lrows) != len(lrow_o):
        return False
    for a, b in zip(lrows, lrow_o):
        if int(a["id"]) != b.id or int(a["D"]) != b.D or int(a["n_pts"]) != len(b.pids):
            return False
        if np.abs(a["line"] - b.line).max() > 2e-3:
            return False
        if np.abs(a["line_n"] - b.line_n).max() > 1e-5:    # undistorted endpoints (2e-3 px / f = 2.4e-6)
            return False
        p = lpts[a["pt_offset"]:a["pt_offset"] + a["n_pts"]]
        if list(p["pid"]) != list(b.pids):
            return False
    return True


def _run(fe, synth, n_frames, kw, seed=1000, width=1280, height=560, line_heavy=False, moving_mask=False,
         teacher_forced=True, hard=True, use_lines=True, line_samples=0):
    from oracle import npops, cvops
    seq = synth.SynthSequence(seed=seed, width=width, height=height, n_frames=n_frames, line_heavy=line_heavy,
                              moving_mask=moving_mask, hard=hard)
    oracle = ofe.FrontEnd(ofe.FeConfig(K=seq.K, D=seq.D, use_lines=use_lines, line_samples=line_samples, **kw))
    gpu = fe.FrontEnd(fe.default_config(width=width, height=height, K=seq.K, D=seq.D, use_lines=int(use_lines),
                                        line_samples=line_samples, **kw))
    gpu.enable_taps(True)
    s = dict(frames=0, n_feat=0, n_status_agree=0, n_klt_fail=0, n_rsc_fail=0, line_frames=0, line_rows_equal=0,
             n_line_rows=0, first_divergence=None, detections=0, new_pts=0, fast_equal=0, n_fast_kps=0, id_errors=0,
             n_uv_outliers=0, n_outliers_not_scalar_exact=0, n_subpix_outliers=0, n_subpix_not_scalar_exact=0,
             min_lines_detected=10 ** 9, n_samples=0, n_sample_status_agree=0, sample_count_errors=0)
    dsmp, dsmp_n = [0.0], [0.0]
    duv, dun, dsub = [0.0], [0.0], [0.0]
    prev_eq = None
    for t in range(n_frames):
        img, mask, vps = seq.frame(t), (seq.mask(t) if moving_mask else None), seq.vanishing_points(t)
        if teacher_forced and t > 0:
            gpu.set_state(_oracle_state_blob(fe, oracle, width, height))
        prow_o, lrow_o = oracle.feed(seq.timestamp(t), img, mask, vps if use_lines else None)
        info = gpu.feed_new_camera(seq.timestamp(t), img, mask, vps if use_lines else None)
        rows = gpu.point_rows()
        tr = oracle.klt.trace
        s["frames"] += 1
        # ---- detection: FAST corner lists per cell (coordinates, scores, order) and the selected / refined / new points
        det = tr.get("det", {})
        assert bool(det.get("ran")) == bool(info.detection_ran), t
        if det.get("ran"):
            s["detections"] += 1
            s["new_pts"] += len(det.get("new_ids", []))
            ref_fast = [np.concatenate([np.full((len(c["xy"]), 2), loc, np.int32), c["xy"], c["resp"].astype(np.int32)[:, None]], 1)
                        for loc, c in zip(det["valid_locs"], det["cells"]) if c is not None]
            ref_fast = np.concatenate(ref_fast, 0) if ref_fast else np.zeros((0, 5), np.int32)
            got_fast = gpu.tap(fe.TAP_FAST_LAST, np.int32).reshape(-1, 5)
            s["n_fast_kps"] += len(ref_fast)
            s["fast_equal"] += int(got_fast.shape == ref_fast.shape and np.array_equal(got_fast, ref_fast))
            sub = gpu.tap(fe.TAP_SUBPIX_LAST, np.float32).reshape(-1, 4)
            sel_o = det.get("selected", np.zeros((0, 2), np.float32))
            assert len(sub) == len(sel_o) and np.array_equal(sub[:, :2], sel_o), "selected FAST corners differ at frame %d" % t
            if len(sub):
                ds = np.abs(sub[:, 2:] - det["refined"]).max(1)
                dsub.extend(ds.tolist())
                bad = np.nonzero(ds > 2e-2)[0]
                if len(bad):   # ill-conditioned corners: the kernel must then match the scalar restatement instead
                    img_det = prev_eq if t > 0 else tr["img_eq"]
                    sc = npops.corner_subpix(img_det, sub[bad, :2])
                    s["n_subpix_outliers"] += len(bad)
                    s["n_subpix_not_scalar_exact"] += int((np.abs(sc - sub[bad, 2:]).max(1) > 2e-3).sum())
            assert info.n_detected == len(det["new_ids"]), (t, info.n_detected, len(det["new_ids"]))
        # ---- tracking: per-feature status flags and positions
        flipped_ids = set()
        if "mask_klt" in tr:
            lk = gpu.tap(fe.TAP_LK_LAST, np.float32).reshape(-1, 6)
            assert len(lk) == len(tr["mask_klt"]), t
            rsc = tr["mask_rsc"].astype(bool) if len(tr["mask_rsc"]) else np.zeros(len(lk), bool)
            st_o = tr["mask_klt"].astype(bool) & rsc
            st_g = (lk[:, 4] > 0) & (lk[:, 5] > 0)
            s["n_feat"] += len(lk)
            s["n_status_agree"] += int((st_o == st_g).sum())
            s["n_klt_fail"] += int((~tr["mask_klt"].astype(bool)).sum())
            s["n_rsc_fail"] += int((tr["mask_klt"].astype(bool) & ~rsc).sum())
            flipped_ids = {int(tr["ids_old"][i]) for i in np.nonzero(st_o != st_g)[0]}
            if flipped_ids and "divergence_cause" not in s:
                klt_f = int((tr["mask_klt"].astype(bool) != (lk[:, 4] > 0)).sum())
                rsc_f = int(((rsc != (lk[:, 5] > 0)) & tr["mask_klt"].astype(bool) & (lk[:, 4] > 0)).sum())
                s["divergence_cause"] = {"frame": t, "klt_status_flips": klt_f, "ransac_inlier_flips": rsc_f,
                                         "max_duv_at_flip": float(np.abs(lk[:, 2:4] - tr["lk_pts1"]).max())}
            if teacher_forced:
                # UV outliers must be the features on which OpenCV itself is chaotic: there the kernel has to agree with
                # the scalar restatement of OpenCV's algorithm (oracle/npops.lk), which cv2's SIMD build does not
                d = np.abs(lk[:, 2:4] - tr["lk_pts1"]).max(1)
                bad = np.nonzero((d > 0.05) & tr["mask_klt"].astype(bool) & (lk[:, 4] > 0))[0]
                if len(bad):
                    s["n_uv_outliers"] += len(bad)
                    p0 = tr["pts_old"][bad]
                    sc, _ = npops.lk(prev_eq, tr["img_eq"], p0, p0, kw["win_size"], kw["pyr_levels"])
                    unexplained = np.abs(sc - lk[bad, 2:4]).max(1) > 2e-3
                    # ... or OpenCV itself must be unstable there: a 1e-4 px change of the input moves cv2's own answer
                    for k in np.nonzero(unexplained)[0]:
                        outs = []
                        for dx, dy in ((1e-4, 0), (-1e-4, 0), (0, 1e-4), (0, -1e-4), (2e-4, 2e-4)):
                            q = (p0[k:k + 1] + np.array([[dx, dy]], np.float32)).astype(np.float32)
                            outs.append(cvops.lk(prev_eq, tr["img_eq"], q, q, kw["win_size"], kw["pyr_levels"])[0][0])
                        spread = np.abs(np.array(outs) - tr["lk_pts1"][bad[k]]).max()
                        if spread > 0.05:
                            unexplained[k] = False
                    s["n_outliers_not_scalar_exact"] += int(unexplained.sum())
        # ---- database rows: ids must be the oracle's, except for features whose status flag flipped
        ids_o = {r.id: r for r in prow_o}
        ids_g = {int(r["id"]): r for r in rows}
        sym = set(ids_o) ^ set(ids_g)
        if not sym <= flipped_ids:
            s["id_errors"] += 1
        if sym and s["first_divergence"] is None:
            s["first_divergence"] = t
        if not sym:
            assert [r.id for r in prow_o] == [int(v) for v in rows["id"]], "row order differs at frame %d" % t
            assert np.array_equal(gpu.get_last_ids(), np.array(oracle.klt.get_last_ids(), np.uint64)), t
        for fid in set(ids_o) & set(ids_g):
            a, b = ids_g[fid], ids_o[fid]
            duv.append(max(abs(float(a["u"]) - b.u), abs(float(a["v"]) - b.v)))
            dun.append(max(abs(float(a["un"]) - b.un), abs(float(a["vn"]) - b.vn)))
        if use_lines and not sym:   # a flipped point status legitimately changes the point-on-line sets of that frame
            lrows, lpts = gpu.line_rows()
            s["line_frames"] += 1
            s["n_line_rows"] += len(lrow_o)
            s["line_rows_equal"] += int(_compare_lines(lrows, lpts, lrow_o))
        if use_lines and t > 0:
            s["min_lines_detected"] = min(s["min_lines_detected"], int(info.n_lines_detected))
        if line_samples:   # extension (BASELINE.json configs[2]): LK over points sampled along last frame's segments
            uv_g, st_g = gpu.line_samples()
            uv_o, st_o = oracle.sample_uv, oracle.sample_status
            if len(uv_g) != len(uv_o) or (len(uv_g) and not np.array_equal(uv_g[:, :2], uv_o[:, :2])):
                s["sample_count_errors"] += 1
            else:
                s["n_samples"] += len(uv_o)
                s["n_sample_status_agree"] += int((st_g.astype(bool) == st_o.astype(bool)).sum())
                both = st_g.astype(bool) & st_o.astype(bool)
                if both.any():
                    dsmp.extend(np.abs(uv_g[both, 2:] - uv_o[both, 2:]).max(1).tolist())
                    # component of the difference ACROSS the segment (the one LK can constrain on a straight edge)
                    seg = uv_o[:, :2].reshape(-1, line_samples, 2)
                    dirs = seg[:, -1] - seg[:, 0]
                    dirs = dirs / np.maximum(np.linalg.norm(dirs, axis=1, keepdims=True), 1e-9)
                    nrm = np.repeat(np.stack([-dirs[:, 1], dirs[:, 0]], 1), line_samples, 0)
                    dn = np.abs(((uv_g[:, 2:] - uv_o[:, 2:]) * nrm).sum(1))[both]
                    dsmp_n.extend(dn.tolist())
        prev_eq = tr["img_eq"]
        if sym and not teacher_forced:
            break
    gpu.close()
    duv, dun, dsub = np.array(duv), np.array(dun), np.array(dsub)
    dsmp, dsmp_n = np.array(dsmp), np.array(dsmp_n)
    s.update(sample_p99=float(np.percentile(dsmp, 99)), sample_max=float(dsmp.max()), n_sample_gt_005=int((dsmp > 0.05).sum()),
             sample_normal_p99=float(np.percentile(dsmp_n, 99)), n_sample_normal_gt_005=int((dsmp_n > 0.05).sum()))
    s.update(max_duv=float(duv.max()), duv_p99=float(np.percentile(duv, 99)), n_duv_gt_005=int((duv > 0.05).sum()),
             n_rows=len(duv) - 1, max_dun=float(dun.max()), max_dsubpix=float(dsub.max()),
             dsubpix_p99=float(np.percentile(dsub, 99)), n_subpix=len(dsub) - 1)
    print(s)
    return s


def _assert_teacher_forced(s, subpix_outlier_div=500):
    assert s["id_errors"] == 0, s                           # feature ids bit-exact (modulo flipped status flags)
    assert s["fast_equal"] == s["detections"], s            # FAST corner lists bit-exact, every detection
    # sub-pixel refinement: 1e-3 px at p99; a corner with a near-singular gradient matrix can move by a fraction of a
    # pixel for a 1e-6 change in the patch, there the kernel has to equal the scalar restatement of cv::cornerSubPix
    assert s["dsubpix_p99"] < 1e-3, s
    assert s["n_subpix_not_scalar_exact"] == 0 and s["n_subpix_outliers"] <= max(1, s["n_subpix"] // subpix_outlier_div), s
    assert s["n_status_agree"] >= 0.995 * s["n_feat"], s    # status flags >= 99.5 %
    # tracked UVs within 0.05 px — except on features where OpenCV itself is chaotic (a 1e-4 px change of the input
    # moves cv2's own answer by ~1 px, see DESIGN.md): at most 0.1 % of rows, and there the kernel must either
    # reproduce the scalar restatement of OpenCV's algorithm or cv2 must be shown to be unstable at that very point
    assert s["duv_p99"] < 0.01, s
    assert s["n_duv_gt_005"] <= max(1, int(0.001 * s["n_rows"])), s
    assert s["n_outliers_not_scalar_exact"] == 0, s
    assert s["line_rows_equal"] == s["line_frames"], s


@pytest.mark.parametrize("kw,seed", [(CFG1, 1000), (CFG2, 1001)])
def test_teacher_forced_1280x560(fe, synth, kw, seed):
    s = _run(fe, synth, 40, kw, seed=seed)
    _assert_teacher_forced(s)
    assert s["detections"] >= 10 and s["new_pts"] > 100, s    # the top-off detector really ran
    assert s["n_klt_fail"] + s["n_rsc_fail"] > 0.01 * s["n_feat"], s   # and the status bar is not vacuous


def test_teacher_forced_kaist_yaml(fe, synth):
    """Shipped KAIST settings (config_camera.yaml:11-18): 1500 pts, FAST 30, 15x15 grid, min dist 15, maxLevel 5."""
    _assert_teacher_forced(_run(fe, synth, 12, CFG_KAIST, seed=1003))


def test_teacher_forced_config3_line_heavy(fe, synth):
    """BASELINE.json configs[2]: >= 300 segments with 10 LK samples each plus 200 points, maxLevel 5.  The samples are an
    extension (not in the reference); their oracle is cv::calcOpticalFlowPyrLK on the same points (oracle/frontend.py)."""
    s = _run(fe, synth, 40, dict(CFG1, pyr_levels=5), seed=1004, line_heavy=True, line_samples=10)
    # this scene is long straight bars: many FAST corners sit on an edge, where cornerSubPix's gradient matrix is close to
    # rank 1 and cv2's own answer moves by a fraction of a pixel for a 1e-6 change of the patch — up to 1 % of the refined
    # corners may be such outliers, and each must still equal the scalar restatement (n_subpix_not_scalar_exact == 0)
    _assert_teacher_forced(s, subpix_outlier_div=100)
    assert s["n_line_rows"] > 0, s
    assert s["min_lines_detected"] >= 300, s                       # every frame after the first: >= 300 segments > 40 px
    assert s["sample_count_errors"] == 0 and s["n_samples"] >= 39 * 3000, s
    assert s["n_sample_status_agree"] >= 0.995 * s["n_samples"], s  # KLT status of the samples
    # A point ON a straight edge is LK's aperture problem: the 2 x 2 normal matrix is close to rank 1, the position along the
    # edge is barely constrained and moves by more than 0.05 px with the summation order of the mismatch vector (cv2's SIMD
    # float sums vs exact integer sums here) — 0.6 % of the samples of this scene.  The bars: p99 below 0.01 px, at most 1 %
    # of the samples over 0.05 px, and fewer still over 0.05 px ACROSS the segment (the constrained direction).
    print({k: s[k] for k in ("n_samples", "sample_p99", "sample_max", "n_sample_gt_005", "sample_normal_p99", "n_sample_normal_gt_005")})
    assert s["sample_p99"] < 0.01 and s["n_sample_gt_005"] <= int(0.01 * s["n_samples"]), s
    assert s["n_sample_normal_gt_005"] <= s["n_sample_gt_005"], s


def test_teacher_forced_config4_1920x1080(fe, synth):
    _assert_teacher_forced(_run(fe, synth, 40, CFG4, seed=1005, width=1920, height=1080))


def test_teacher_forced_moving_mask(fe, synth):
    """Moving circular mask of the reference's test_tracking.cpp:288-302, 5x3 grid."""
    _assert_teacher_forced(_run(fe, synth, 25, dict(CFG1, grid_y=3, pyr_levels=5), seed=1002, moving_mask=True))


def test_teacher_forced_clahe(fe, synth):
    """histogram_method = CLAHE (TrackKLT.cpp:60-64, TrackLSD.cpp:84-88): third pre-processing mode of the reference."""
    _assert_teacher_forced(_run(fe, synth, 8, dict(CFG1, histogram_method=2), seed=1007))


def test_teacher_forced_no_equalisation(fe, synth):
    _assert_teacher_forced(_run(fe, synth, 8, dict(CFG1, histogram_method=0), seed=1006))


@pytest.mark.parametrize("kw,seed", [(CFG1, 1000), (CFG2, 1001)])
def test_free_running_sequence(fe, synth, kw, seed):
    s = _run(fe, synth, 40, kw, seed=seed, teacher_forced=False)
    assert s["id_errors"] == 0, s
    assert s["n_status_agree"] >= 0.995 * s["n_feat"], s
    assert s["duv_p99"] < 0.05, s
    assert s["n_duv_gt_005"] <= 0.005 * s["n_rows"], s      # ill-conditioned features drift (see module docstring)


@pytest.mark.parametrize("seed", [1000, 1001, 1002])
def test_free_running_300_frames(fe, synth, seed):
    """SURVEY.md 7.2: free-running parity over 300 frames on 3 seeds.  Both sides run on their own state; one flipped status
    flag changes pts_last and with it every later id (SURVEY.md 7.3 item 2), so the run is compared up to the first frame
    whose row sets differ and that frame and its cause are reported (printed, and kept in the bench line's klt_parity)."""
    s = _run(fe, synth, 300, CFG2, seed=seed, teacher_forced=False)
    print("free-running seed %d: %d frames compared, first divergence %s, cause %s" %
          (seed, s["frames"], s["first_divergence"], s.get("divergence_cause")))
    assert s["id_errors"] == 0, s                                 # every difference is explained by a flipped status flag
    assert s["n_status_agree"] >= 0.995 * s["n_feat"], s
    assert s["duv_p99"] < 0.05, s
    assert s["n_duv_gt_005"] <= 0.005 * s["n_rows"], s
    assert s["frames"] >= 10, s                                   # the runs do not diverge at once


def test_reset_and_small_counts(fe, synth):
    """Tracker self-reset paths: < 10 points => all-fail mask (TrackKLT.cpp:848-852), then re-detection next frame."""
    seq = synth.SynthSequence(seed=1010, n_frames=6, hard=False)
    kw = dict(CFG1)
    oracle = ofe.FrontEnd(ofe.FeConfig(K=seq.K, D=seq.D, use_lines=False, **kw))
    gpu = fe.FrontEnd(fe.default_config(width=1280, height=560, K=seq.K, D=seq.D, use_lines=0, **kw))
    img0 = seq.frame(0)
    oracle.feed(1.0, img0)
    gpu.feed_new_camera(1.0, img0)
    # force 5 points only
    st = oracle.klt.get_state()
    st["pts_last"], st["ids_last"] = st["pts_last"][:5], st["ids_last"][:5]
    oracle.klt.set_state(st)
    gpu.set_state(fe.pack_state(1280, 560, st["currid"], st["pts_last"], st["ids_last"], st["img_last"], None))
    for t in range(1, 5):
        img = seq.frame(t)
        prow_o, _ = oracle.feed(seq.timestamp(t), img)
        gpu.feed_new_camera(seq.timestamp(t), img)
        rows = gpu.point_rows()
        assert list(rows["id"]) == [r.id for r in prow_o], t
        assert np.array_equal(gpu.get_last_ids(), np.array(oracle.klt.get_last_ids(), np.uint64)), t
    # a black frame kills every track: both must come back identically afterwards
    black = np.zeros_like(img0)
    for t, img in enumerate([black, seq.frame(5), seq.frame(5)]):
        prow_o, _ = oracle.feed(10.0 + t, img)
        gpu.feed_new_camera(10.0 + t, img)
        assert list(gpu.point_rows()["id"]) == [r.id for r in prow_o]
        assert np.array_equal(gpu.get_last_ids(), np.array(oracle.klt.get_last_ids(), np.uint64))
    gpu.close()


def test_grider_regrids_itself_when_features_are_fewer_than_cells(fe, synth):
    """Grider_GRID.h:88-100: with num_features < grid_x * grid_y the grider derives ITS OWN grid (15 features on a 5 x 5
    grid -> 4 x 4 cells of 320 x 140) while the valid cells still index the caller's 5 x 5 grid; cells whose origin leaves
    the image are skipped (:117-118), so 16 of the 25 locations are searched, one corner each.  The sequence also walks
    through the < 10 points all-fail mask and the reset that follows.  Teacher-forced."""
    seq = synth.SynthSequence(seed=1019, n_frames=12, hard=False)
    kw = dict(CFG1, num_features=15)
    oracle = ofe.FrontEnd(ofe.FeConfig(K=seq.K, D=seq.D, use_lines=False, **kw))
    gpu = fe.FrontEnd(fe.default_config(width=1280, height=560, K=seq.K, D=seq.D, use_lines=0, **kw))
    searched, resets = [], 0
    for t in range(12):
        if t > 0:
            gpu.set_state(_oracle_state_blob(fe, oracle, 1280, 560))
        prow_o, _ = oracle.feed(seq.timestamp(t), seq.frame(t))
        info = gpu.feed_new_camera(seq.timestamp(t), seq.frame(t))
        det = oracle.klt.trace.get("det", {})
        if det.get("ran"):
            searched.append(sum(c is not None for c in det["cells"]))
            assert info.n_detected == len(det["new_ids"]), t
        resets += int(info.reset)
        assert bool(info.reset) == bool(oracle.klt.trace.get("reset")), t
        n_in = len(oracle.klt.trace.get("pts_old", []))
        if 10 <= n_in <= 13:
            # cv::findFundamentalMat runs LMedS below 15 points and, below 14, picks its model by the rounding noise of its
            # own solver (tests/test_host_cpu.py::test_ransac_small_counts_lmeds_regime): only the structure is compared
            assert set(int(i) for i in gpu.point_rows()["id"]) <= set(oracle.klt.trace["ids_old"]), t
            continue
        assert list(gpu.point_rows()["id"]) == [r.id for r in prow_o], t
        assert np.array_equal(gpu.get_last_ids(), np.array(oracle.klt.get_last_ids(), np.uint64)), t
        if len(oracle.klt.pts_last):
            assert np.abs(gpu.get_last_obs() - oracle.klt.pts_last).max() < 0.05, t
    gpu.close()
    assert searched and max(searched) == 16, searched     # 16 of the 25 caller cells exist in the grider's own 4 x 4 grid


def test_state_roundtrip_and_pipelined_submit(fe, synth):
    """get_state/set_state round trip, and submit/collect with lookahead gives the same rows as feed()."""
    seq = synth.SynthSequence(seed=1011, n_frames=12)
    cfg = dict(width=1280, height=560, K=seq.K, D=seq.D, **CFG2)
    a = fe.FrontEnd(fe.default_config(**cfg))
    b = fe.FrontEnd(fe.default_config(lookahead=3, **cfg))
    ref = []
    for t in range(10):
        a.feed_new_camera(seq.timestamp(t), seq.frame(t), None, seq.vanishing_points(t))
        ref.append((a.point_rows().copy(), a.line_rows()[0].copy()))
        if t == 4:
            blob = a.get_state()
    frames = [seq.frame(t) for t in range(10)]
    got = []
    nsub = 0
    for t in range(10):
        while nsub < 10 and nsub <= t + 3:
            b.submit(seq.timestamp(nsub), frames[nsub], vanishing_points=seq.vanishing_points(nsub))
            nsub += 1
        b.collect()
        got.append((b.point_rows().copy(), b.line_rows()[0].copy()))
    for t in range(10):
        assert np.array_equal(ref[t][0], got[t][0]), t
        assert np.array_equal(ref[t][1], got[t][1]), t
    # resume from the frame-4 checkpoint in a fresh handle
    c = fe.FrontEnd(fe.default_config(**cfg))
    c.set_state(blob)
    for t in range(5, 10):
        c.feed_new_camera(seq.timestamp(t), frames[t], None, seq.vanishing_points(t))
        assert np.array_equal(c.point_rows(), ref[t][0]), t
        assert np.array_equal(c.line_rows()[0], ref[t][1]), t
    st = fe.unpack_state(blob)
    assert st["img_last"].shape == (560, 1280) and len(st["pts_last"]) == len(st["ids_last"]) > 0
    for h in (a, b, c):
        h.close()


@pytest.mark.parametrize("lookahead,pattern", [(8, "steady"), (16, "steady"), (8, "ragged")])
def test_batched_line_path_equals_frame_by_frame(fe, synth, lookahead, pattern):
    """With lookahead >= 8 the line paths of consecutive frames share their kernel launches (grid.y = frame, batches of
    min(4, lookahead / 2)); rows must equal the synchronous per-frame path bit for bit — also when collect() arrives before a
    batch is full (ragged: collect after every 1, 2, 3, 5, ... submits) and when a handle is closed with frames pending."""
    n = 14
    seq = synth.SynthSequence(seed=1016, n_frames=n)
    cfg = dict(width=1280, height=560, K=seq.K, D=seq.D, **CFG1)
    a = fe.FrontEnd(fe.default_config(**cfg))
    ref = []
    for t in range(n):
        a.feed_new_camera(seq.timestamp(t), seq.frame(t), None, seq.vanishing_points(t))
        lr, lp = a.line_rows()
        ref.append((a.point_rows().copy(), lr.copy(), lp.copy()))
    a.close()
    assert sum(len(r[1]) for r in ref) > 50
    b = fe.FrontEnd(fe.default_config(lookahead=lookahead, **cfg))
    frames = [seq.frame(t) for t in range(n)]
    nsub = ncol = 0
    burst = [1, 2, 3, 5, 1, 2] if pattern == "ragged" else None
    k = 0
    while ncol < n:
        if burst is not None:
            want = burst[k % len(burst)]
            k += 1
        else:
            want = lookahead + 1 - (nsub - ncol)
        for _ in range(max(want, 0)):
            if nsub < n and nsub - ncol <= lookahead:
                b.submit(seq.timestamp(nsub), frames[nsub], vanishing_points=seq.vanishing_points(nsub))
                nsub += 1
        ncoll_now = 1 if burst is None else min(nsub - ncol, 2)
        for _ in range(max(ncoll_now, 1)):
            if ncol < nsub:
                b.collect()
                lr, lp = b.line_rows()
                assert np.array_equal(b.point_rows(), ref[ncol][0]), ncol
                assert np.array_equal(lr, ref[ncol][1]), ncol
                assert np.array_equal(lp, ref[ncol][2]), ncol
                ncol += 1
    # frames pending (some in an unlaunched batch) when the handle goes away: must not hang
    for t in range(3):
        b.submit(100.0 + t, frames[t], vanishing_points=seq.vanishing_points(t))
    b.close()


def test_multi_stream_isolation(fe, synth):
    """A stream's rows do not depend on what else runs on the GPU: 4 handles interleaved == each run alone."""
    seqs = [synth.SynthSequence(seed=1020 + k, n_frames=6, hard=False) for k in range(4)]
    cfg = dict(width=1280, height=560, **CFG1)
    alone = []
    for sq in seqs:
        h = fe.FrontEnd(fe.default_config(K=sq.K, D=sq.D, **cfg))
        rows = []
        for t in range(6):
            h.feed_new_camera(sq.timestamp(t), sq.frame(t), None, sq.vanishing_points(t))
            rows.append((h.point_rows().copy(), h.line_rows()[0].copy()))
        alone.append(rows)
        h.close()
    hs = [fe.FrontEnd(fe.default_config(K=sq.K, D=sq.D, lookahead=1, **cfg)) for sq in seqs]
    for t in range(6):
        for h, sq in zip(hs, seqs):
            h.submit(sq.timestamp(t), sq.frame(t), vanishing_points=sq.vanishing_points(t))
        for k, h in enumerate(hs):
            h.collect()
            assert np.array_equal(h.point_rows(), alone[k][t][0]), (k, t)
            assert np.array_equal(h.line_rows()[0], alone[k][t][1]), (k, t)
    for h in hs:
        h.close()


def test_bad_arguments(fe):
    with pytest.raises(fe.FrontEndError):
        fe.FrontEnd(fe.default_config(win_size=14))
    with pytest.raises(fe.FrontEndError):
        fe.FrontEnd(fe.default_config(histogram_method=7))
    h = fe.FrontEnd(fe.default_config())
    with pytest.raises(fe.FrontEndError):
        h.feed_new_camera(0.0, np.zeros((100, 100), np.uint8))   # size mismatch: the reference exit()s here
    h.close()


def test_setters_between_frames_and_line_classification(fe, synth):
    """TrackBase::set_num_features / change_feat_id (TrackBase.h:150, TrackBase.cpp:267-285) and the late
    LineClassification entry point: the tracker must follow the oracle through a feature-count change, an id
    re-mapping and vanishing points that only arrive after the frame was fed (UpdaterCamera.cpp:105-110 order)."""
    seq = synth.SynthSequence(seed=1012, n_frames=10, hard=False)
    kw = dict(CFG1)
    oracle = ofe.FrontEnd(ofe.FeConfig(K=seq.K, D=seq.D, use_lines=True, **kw))
    gpu = fe.FrontEnd(fe.default_config(width=1280, height=560, K=seq.K, D=seq.D, use_lines=1, **kw))
    zeros = np.zeros((3, 2))
    for t in range(10):
        img, vps = seq.frame(t), seq.vanishing_points(t)
        if t == 3:      # ask for more features: the next top-off detection uses the new grid quota
            n_before = len(gpu.get_last_ids())
            oracle.klt.cfg.num_features = 320
            gpu.set_num_features(320)
        if t == 6:      # loop-closure style id change of an active feature
            ids = oracle.klt.get_last_ids()
            old, new = int(ids[len(ids) // 2]), 10 ** 6 + 7
            st = oracle.klt.get_state()
            st["ids_last"] = [new if int(i) == old else int(i) for i in st["ids_last"]]
            oracle.klt.set_state(st)
            gpu.change_feat_id(old, new)
            assert new in [int(v) for v in gpu.get_last_ids()]
        prow_o, lrow_o = oracle.feed(seq.timestamp(t), img, None, vps)
        gpu.feed_new_camera(seq.timestamp(t), img, None, zeros)      # vanishing points not known yet
        gpu.classify_lines(vps)                                       # ... now they are
        assert [int(v) for v in gpu.point_rows()["id"]] == [r.id for r in prow_o], t
        assert np.array_equal(gpu.get_last_ids(), np.array(oracle.klt.get_last_ids(), np.uint64)), t
        lrows, lpts = gpu.line_rows()
        assert _compare_lines(lrows, lpts, lrow_o), t
    assert len(gpu.get_last_ids()) > n_before          # the larger quota took effect
    # the setters are refused while frames are in flight
    gpu2 = fe.FrontEnd(fe.default_config(width=1280, height=560, K=seq.K, D=seq.D, lookahead=2, **kw))
    gpu2.submit(0.0, seq.frame(0), vanishing_points=zeros)
    with pytest.raises(fe.FrontEndError):
        gpu2.set_num_features(100)
    with pytest.raises(fe.FrontEndError):
        gpu2.change_feat_id(1, 2)
    gpu2.collect()
    gpu2.set_num_features(100)
    gpu2.close()
    gpu.close()


def test_play_equals_frame_by_frame(fe, synth):
    """plviwo_fe_play (whole-sequence playback inside the library) gives the rows of feeding frame by frame."""
    seq = synth.SynthSequence(seed=1013, n_frames=10)
    cfg = dict(width=1280, height=560, K=seq.K, D=seq.D, **CFG2)
    frames = [seq.frame(t) for t in range(10)]
    ts = [seq.timestamp(t) for t in range(10)]
    vps = [seq.vanishing_points(t) for t in range(10)]
    a = fe.FrontEnd(fe.default_config(lookahead=0, **cfg))
    chk, npr, nlr = 0.0, 0, 0
    for t in range(10):
        a.feed_new_camera(ts[t], frames[t], None, vps[t], update_db=False)
        rows = a.point_rows()
        lrows, _ = a.line_rows()
        npr += len(rows)
        nlr += len(lrows)
        chk += float(rows["id"].astype(np.float64).sum() + rows["u"].astype(np.float64).sum() + rows["v"].astype(np.float64).sum())
        chk += float(lrows["id"].astype(np.float64).sum() + lrows["line"].astype(np.float64).sum())
    last_ids = a.get_last_ids().copy()
    a.close()
    b = fe.FrontEnd(fe.default_config(lookahead=4, **cfg))
    st = b.play(ts, frames, vanishing_points=vps)
    assert (st.frames, st.point_rows, st.line_rows) == (10, npr, nlr)
    assert abs(st.checksum - chk) <= 1e-6 * max(1.0, abs(chk))
    assert np.array_equal(b.get_last_ids(), last_ids)
    b.close()


@pytest.mark.parametrize("size,lines", [((1280, 560), True), ((1285, 563), False)])
def test_downsample_prestep(fe, synth, size, lines):
    """cfg.downsample: UpdaterCamera::feed_measurement's cv::pyrDown of image AND mask to the truncated half size
    (UpdaterCamera.cpp:86-95) in front of both trackers; K is the halved calibration (OptionsCamera.cpp:123-126)."""
    W, H = size
    seq = synth.SynthSequence(seed=1014, width=W, height=H, n_frames=8, hard=False, moving_mask=True)
    K = tuple(v / 2.0 for v in seq.K)
    kw = dict(CFG1, num_features=150)
    oracle = ofe.FrontEnd(ofe.FeConfig(K=K, D=seq.D, use_lines=lines, downsample=True, **kw))
    gpu = fe.FrontEnd(fe.default_config(width=W, height=H, K=K, D=seq.D, use_lines=int(lines), downsample=1, **kw))
    worst = 0.0
    for t in range(8):
        img, mask, vps = seq.frame(t), seq.mask(t), [(x / 2.0, y / 2.0) for x, y in seq.vanishing_points(t)]
        prow_o, lrow_o = oracle.feed(seq.timestamp(t), img, mask, vps if lines else None)
        gpu.feed_new_camera(seq.timestamp(t), img, mask, vps if lines else None)
        assert np.array_equal(gpu.tap(fe.TAP_PYR_LEVEL0).reshape(int(H / 2.0), int(W / 2.0)), oracle.klt.trace["img_eq"]), t
        rows = gpu.point_rows()
        assert [int(v) for v in rows["id"]] == [r.id for r in prow_o], t
        if len(rows):
            uv_o = np.array([[r.u, r.v] for r in prow_o], np.float32)
            worst = max(worst, float(np.abs(np.stack([rows["u"], rows["v"]], 1) - uv_o).max()))
        if lines:
            lrows, lpts = gpu.line_rows()
            assert _compare_lines(lrows, lpts, lrow_o), t
    assert worst < 0.05, worst
    gpu.close()


@pytest.mark.parametrize("kw,lookahead", [(CFG2, 6), (CFG_KAIST, 3)])
def test_speculative_tracking_equals_synchronous(fe, synth, kw, lookahead):
    """With frames queued ahead (lookahead >= 1), LK(t -> t+1) is launched speculatively for every trackable point
    before frame t's RANSAC gate (FeContext::speculate, track_candidates).  Rows, ids and line rows must be IDENTICAL
    (bitwise) to feeding frame by frame (lookahead 0), where nothing is speculated, over a sequence long enough to
    contain detections, losses and occluders."""
    n = 40
    seq = synth.SynthSequence(seed=1015, n_frames=n)
    cfg = dict(width=1280, height=560, K=seq.K, D=seq.D, **kw)
    frames = [seq.frame(t) for t in range(n)]
    a = fe.FrontEnd(fe.default_config(lookahead=0, **cfg))
    ref = []
    for t in range(n):
        a.feed_new_camera(seq.timestamp(t), frames[t], None, seq.vanishing_points(t), update_db=False)
        ref.append((a.point_rows().copy(), a.line_rows()[0].copy(), a.get_last_ids().copy()))
    a.close()
    b = fe.FrontEnd(fe.default_config(lookahead=lookahead, **cfg))
    sub = 0
    n_spec_rows = 0
    for t in range(n):
        while sub < n and sub <= t + lookahead:
            b.submit(seq.timestamp(sub), frames[sub], vanishing_points=seq.vanishing_points(sub))
            sub += 1
        b.collect()
        assert np.array_equal(b.point_rows(), ref[t][0]), t
        assert np.array_equal(b.line_rows()[0], ref[t][1]), t
        assert np.array_equal(b.get_last_ids(), ref[t][2]), t
        n_spec_rows += len(ref[t][0])
    assert n_spec_rows > 20 * 100
    b.close()


def test_pipelined_with_masks_and_device_frames(fe, synth):
    """submit/collect with a per-frame tracking mask, and frames that already live in device memory
    (plviwo_fe_submit(on_device) / plviwo_fe_feed_device), give the rows of the synchronous host-memory feed."""
    import torch
    n = 14
    seq = synth.SynthSequence(seed=1016, n_frames=n, moving_mask=True)
    cfg = dict(width=1280, height=560, K=seq.K, D=seq.D, **CFG1)
    frames = [seq.frame(t) for t in range(n)]
    masks = [seq.mask(t) for t in range(n)]
    a = fe.FrontEnd(fe.default_config(lookahead=0, **cfg))
    ref = []
    for t in range(n):
        a.feed_new_camera(seq.timestamp(t), frames[t], masks[t], seq.vanishing_points(t), update_db=False)
        ref.append((a.point_rows().copy(), a.line_rows()[0].copy()))
    a.close()
    # pipelined, masks, host frames
    b = fe.FrontEnd(fe.default_config(lookahead=3, **cfg))
    sub = 0
    for t in range(n):
        while sub < n and sub <= t + 3:
            b.submit(seq.timestamp(sub), frames[sub], vanishing_points=seq.vanishing_points(sub), mask=masks[sub])
            sub += 1
        b.collect()
        assert np.array_equal(b.point_rows(), ref[t][0]), t
        assert np.array_equal(b.line_rows()[0], ref[t][1]), t
    b.close()
    # device-resident frames with a pitch larger than the width, no masks: compare with a mask-free synchronous run
    c0 = fe.FrontEnd(fe.default_config(lookahead=0, **cfg))
    c1 = fe.FrontEnd(fe.default_config(lookahead=0, **cfg))
    d = torch.zeros((n, 560, 1536), dtype=torch.uint8, device="cuda")
    for t in range(n):
        d[t, :, :1280] = torch.from_numpy(frames[t]).cuda()
    torch.cuda.synchronize()
    for t in range(n):
        c0.feed_new_camera(seq.timestamp(t), frames[t], None, seq.vanishing_points(t), update_db=False)
        c1.feed_device(seq.timestamp(t), d[t].data_ptr(), 1280, 560, 1536, seq.vanishing_points(t))
        assert np.array_equal(c0.point_rows(), c1.point_rows()), t
        assert np.array_equal(c0.line_rows()[0], c1.line_rows()[0]), t
    c0.close()
    c1.close()


def test_capacity_and_boundary_guards(fe, synth):
    """Round-1 advisor findings: set_num_features beyond the candidate-table capacity of the handle, state blobs whose line
    sizes do not add up, the camera-model gate and the shared id counter."""
    W, H = 640, 280
    seq = synth.SynthSequence(seed=3, width=W, height=H, n_frames=4, hard=False)
    kw = dict(num_features=150, fast_threshold=20, grid_x=1, grid_y=1, min_px_dist=10, pyr_levels=3, win_size=15)
    h = fe.FrontEnd(fe.default_config(width=W, height=H, K=seq.K, D=seq.D, **kw))
    h.feed_new_camera(seq.timestamp(0), seq.frame(0), None, seq.vanishing_points(0), update_db=False)
    h.set_num_features(600)                       # 1 cell x 601 candidates fits the 1024 slots of this handle
    with pytest.raises(fe.FrontEndError):
        h.set_num_features(2000)                  # 1 x 2001 does not: refused, not an overrun
    h.feed_new_camera(seq.timestamp(1), seq.frame(1), None, seq.vanishing_points(1), update_db=False)
    # camera model gate
    h.set_camera(0, seq.K, seq.D)
    with pytest.raises(fe.FrontEndError):
        h.set_camera(1, seq.K, seq.D)             # equidistant: not implemented, must not be silently mis-undistorted
    # id counter hand-over (TrackBase::currid is shared by the cameras of one tracker)
    c = h.get_currid()
    assert c >= 2
    h.set_currid(c + 1000)
    h.feed_new_camera(seq.timestamp(2), seq.frame(2), None, seq.vanishing_points(2), update_db=False)
    assert h.get_currid() >= c + 1000
    # a blob whose per-line sizes announce more entries than the header: rejected, the tracker state is untouched
    blob = bytearray(h.get_state())
    before = h.get_state()
    hdr = np.frombuffer(bytes(blob[:56]), fe._STATE_HDR, 1)[0]
    n_pts, n_lines = int(hdr["n_pts"]), int(hdr["n_lines"])
    if n_lines > 0:
        off = 56 + 16 * n_pts + 24 * n_lines      # the int32 sizes array
        sizes = np.frombuffer(bytes(blob[off:off + 4 * n_lines]), np.int32).copy()
        sizes[0] += 5
        blob[off:off + 4 * n_lines] = sizes.tobytes()
        with pytest.raises(fe.FrontEndError):
            h.set_state(bytes(blob))
        assert h.get_state() == before
    bad = bytearray(before)
    bad[4:8] = np.uint32(7).tobytes()             # unknown version
    with pytest.raises(fe.FrontEndError):
        h.set_state(bytes(bad))
    h.close()
