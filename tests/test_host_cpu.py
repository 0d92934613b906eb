"""CPU tests of the product's host side: the C-ABI library loads and exports every symbol include/plviwo_fe.h
declares, refuses to run without a GPU (no CPU fallback), and its host-side sequential step — the RANSAC gate —
reproduces cv2.findFundamentalMat.  No kernel is launched here."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_exported(fe):
    hdr = open(os.path.join(ROOT, "include", "plviwo_fe.h")).read()
    declared = sorted(set(re.findall(r"\b(plviwo_(?:fe|op)_[a-z0-9_]+)\s*\(", hdr)))
    assert declared == sorted(fe.EXPORTS), set(declared) ^ set(fe.EXPORTS)
    lib = fe.lib()
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert lib.plviwo_fe_abi_version() == 1


def test_struct_layouts_match_header(fe):
    import ctypes as C
    assert C.sizeof(fe.FePointRow) == 24 and fe.POINT_ROW_DTYPE.itemsize == 24
    assert C.sizeof(fe.FeLineRow) == 56 and fe.LINE_ROW_DTYPE.itemsize == 56
    assert C.sizeof(fe.FeLinePoint) == 16 and fe.LINE_POINT_DTYPE.itemsize == 16
    assert C.sizeof(fe.FeConfig) == 20 * 4 + 64
    assert C.sizeof(fe.FeStereoInfo) == 96                 # double + 21 int32, padded to 8 (checked against the C header)
    cfg = fe.default_config()
    assert (cfg.width, cfg.height, cfg.num_features, cfg.pyr_levels, cfg.win_size) == (1280, 560, 150, 5, 15)
    assert abs(cfg.K[0] - 816.90378992770002) < 1e-12 and cfg.fld_length_threshold == 20


def test_no_cpu_fallback(fe):
    if fe.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(fe.FrontEndError) as e:
        fe.FrontEnd(fe.default_config())
    assert e.value.code == fe.FE_NO_DEVICE
    with pytest.raises(fe.FrontEndError):
        fe.op_equalize_pyramid(np.zeros((64, 64), np.uint8), 2)


def test_no_cpu_fallback_stereo(fe):
    if fe.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(fe.FrontEndError) as e:
        fe.StereoFrontEnd(fe.default_config())
    assert e.value.code == fe.FE_NO_DEVICE


_SHARED_RULES = [
    (dict(width=32), "image size must be in [64, 4095]"),
    (dict(height=4096), "image size must be in [64, 4095]"),
    (dict(win_size=16), "win_size must be odd and in [3, 31]"),
    (dict(win_size=33), "win_size must be odd and in [3, 31]"),
    (dict(pyr_levels=8), "pyr_levels must be in [0, 7]"),
    (dict(grid_y=0), "bad grid / distance / feature count"),
    (dict(min_px_dist=0), "bad grid / distance / feature count"),
    (dict(num_features=0), "bad grid / distance / feature count"),
    (dict(histogram_method=7), "bad histogram_method"),
    (dict(width=642, height=281), "line tracker needs even (tracking) image dimensions (exact 2x decimation)"),
    (dict(canny_th2=60.0), "canny_th1 != canny_th2: hysteresis pass is not implemented"),
    (dict(fld_length_threshold=1), "bad fld_length_threshold"),
]
_CREATORS = ("handle", "group", "stereo")


def _create(fe, creator, cfg, n_streams=2):
    """rc and reason of a creation through the C ABI that is expected to be refused."""
    import ctypes as C
    L = fe.lib()
    h = C.c_void_p()
    if creator == "handle":
        rc, why = L.plviwo_fe_create(C.byref(cfg), 0, C.byref(h)), L.plviwo_fe_last_error(None)
    elif creator == "group":
        rc, why = L.plviwo_fe_group_create(C.byref(cfg), n_streams, 0, C.byref(h)), L.plviwo_fe_group_last_error(None)
    else:
        K, D = (C.c_double * 4)(*cfg.K), (C.c_double * 4)(*cfg.D)
        rc, why = L.plviwo_fe_stereo_create(C.byref(cfg), K, D, 0, C.byref(h)), L.plviwo_fe_stereo_last_error(None)
    assert not h.value, "created a handle from a config that must be refused"
    return rc, (why or b"").decode()


@pytest.mark.parametrize("creator", _CREATORS)
@pytest.mark.parametrize("kw,reason", _SHARED_RULES)
def test_creators_refuse_bad_configs_before_the_device_query(fe, creator, kw, reason):
    """Every creator checks the shared config rules before it looks for a device, so the refusal and its reason are the
    same with and without a GPU."""
    assert _create(fe, creator, fe.default_config(**kw)) == (fe.FE_BAD_ARG, reason)


@pytest.mark.parametrize("creator,kw,reason", [
    ("handle", dict(width=100, downsample=1), "downsampled image would be smaller than 64 pixels"),
    ("handle", dict(width=1282, downsample=1), "line tracker needs even (tracking) image dimensions (exact 2x decimation)"),
    ("group", dict(downsample=1), "cfg.downsample is not supported in a stream group"),
    ("group", dict(grid_x=16, grid_y=17), "a stream group supports at most 256 grid cells"),
])
def test_creator_specific_config_rules(fe, creator, kw, reason):
    assert _create(fe, creator, fe.default_config(**kw)) == (fe.FE_BAD_ARG, reason)


@pytest.mark.parametrize("n_streams", [0, 4097])
def test_group_refuses_bad_stream_count(fe, n_streams):
    assert _create(fe, "group", fe.default_config(), n_streams) == (fe.FE_BAD_ARG, "n_streams must be in [1, 4096]")


def test_stereo_state_blob_pack_unpack(fe):
    rng = np.random.default_rng(1)
    img = rng.integers(0, 255, (64, 96), np.uint8)
    blobs = []
    for n in (5, 3):
        pts = rng.uniform(0, 60, (n, 2)).astype(np.float32)
        blobs.append(fe.pack_state(96, 64, 77, pts, np.arange(n) + 10, img, None))
    blob = fe.pack_stereo_state(77, blobs[0], blobs[1])
    currid, left, right = fe.unpack_stereo_state(blob)
    assert currid == 77 and len(left["ids_last"]) == 5 and len(right["ids_last"]) == 3
    assert np.array_equal(left["img_last"], img) and np.array_equal(right["img_last"], img)


def test_state_blob_pack_unpack(fe):
    pts = np.random.default_rng(0).uniform(0, 500, (7, 2)).astype(np.float32)
    blob = fe.pack_state(1280, 560, 99, pts, np.arange(7) + 5, None, None, 12, np.ones((2, 4), np.float32), [3, 4],
                         [{5: 0.25, 7: 1.5}, {6: 2.0}])
    st = fe.unpack_state(blob)
    assert st["currid"] == 99 and st["line_currid"] == 12
    assert np.array_equal(st["pts_last"], pts) and list(st["ids_last"]) == list(range(5, 12))
    assert st["pol_last"] == [{5: 0.25, 7: 1.5}, {6: 2.0}] and st["img_last"] is None


def test_ransac_host_matches_opencv(fe):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(0)
    exact = 0
    for trial in range(40):
        n = int(rng.integers(15, 600))
        X = np.c_[rng.uniform(-3, 3, n), rng.uniform(-2, 2, n), rng.uniform(4, 12, n)]
        R, _ = cv2.Rodrigues(rng.normal(0, 0.03, 3))
        X2 = X @ R.T + rng.normal(0, 0.3, 3)
        p0 = (X[:, :2] / X[:, 2:]).astype(np.float32)
        p1 = (X2[:, :2] / X2[:, 2:]).astype(np.float32) + rng.normal(0, 0.5 / 800, (n, 2)).astype(np.float32)
        out = rng.random(n) < 0.15
        p1[out] += rng.normal(0, 0.05, (int(out.sum()), 2)).astype(np.float32)
        thr = 2.0 / 816.9
        _F, m = cv2.findFundamentalMat(p0, p1, cv2.FM_RANSAC, thr, 0.999)
        ref = np.zeros(n, np.uint8) if m is None else m.reshape(-1)
        mine, n_in = fe.op_ransac_fundamental(p0, p1, thr, 0.999)
        exact += int(np.array_equal(ref, mine))
        assert (ref != mine).mean() <= 0.005
    assert exact >= 38, exact
    # fewer than 7 points: OpenCV returns no mask at all (TrackKLT.cpp:877 then fails every point)
    mine, n_in = fe.op_ransac_fundamental(p0[:5], p1[:5], thr, 0.999)
    assert n_in == -1 and not mine.any()


def test_ransac_small_counts_lmeds_regime(fe):
    """cv::findFundamentalMat(FM_RANSAC) silently runs LMedS below 15 points.  With 14 points the median is the 8th
    smallest error — a point outside the 7-point sample — and the library's mask is reproduced exactly.  With 10..13
    points the median is the error of one of the model's own sample points (zero up to rounding noise, ~1e-33), so
    OpenCV's pick among the candidate models is decided by the rounding of its own solver: there the masks are only
    required to be a valid LMedS answer (at least 7 inliers, and the tracker's >= 10-point precondition of
    TrackKLT.cpp:848 keeps this regime to 10..13 points)."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(3)
    thr = 2.0 / 816.9
    exact14 = 0
    for trial in range(60):
        n = 14 if trial < 30 else int(rng.integers(10, 14))
        X = np.c_[rng.uniform(-3, 3, n), rng.uniform(-2, 2, n), rng.uniform(4, 12, n)]
        R, _ = cv2.Rodrigues(rng.normal(0, 0.03, 3))
        X2 = X @ R.T + rng.normal(0, 0.3, 3)
        p0 = (X[:, :2] / X[:, 2:]).astype(np.float32)
        p1 = (X2[:, :2] / X2[:, 2:]).astype(np.float32) + rng.normal(0, 0.5 / 800, (n, 2)).astype(np.float32)
        _F, m = cv2.findFundamentalMat(p0, p1, cv2.FM_RANSAC, thr, 0.999)
        ref = np.zeros(n, np.uint8) if m is None else m.reshape(-1)
        mine, n_in = fe.op_ransac_fundamental(p0, p1, thr, 0.999)
        if n == 14:
            exact14 += int(np.array_equal(ref, mine))
        else:
            assert n_in >= 7 and int(mine.sum()) == n_in, (n, n_in)
    assert exact14 >= 29, exact14


def test_ransac_repeated_frame(fe):
    """A repeated frame (every point tracked exactly onto itself) keeps its tracks: all points are inliers, as in the
    library's non-asserting outcome; with a few lost points among them the static ones are the inliers.  (OpenCV 4.13
    throws out of findFundamentalMat on most such inputs, which is why cv2 is not the checker here.)"""
    rng = np.random.default_rng(4)
    thr = 2.0 / 816.9
    for n in (10, 14, 15, 60, 400):
        p0 = np.c_[rng.uniform(-0.7, 0.7, n), rng.uniform(-0.3, 0.3, n)].astype(np.float32)
        mask, n_in = fe.op_ransac_fundamental(p0, p0.copy(), thr, 0.999)
        assert n_in == n and mask.all(), n
    n = 300
    p0 = np.c_[rng.uniform(-0.7, 0.7, n), rng.uniform(-0.3, 0.3, n)].astype(np.float32)
    p1 = p0.copy()
    lost = rng.choice(n, 20, replace=False)
    p1[lost] += rng.uniform(0.02, 0.05, (20, 2)).astype(np.float32) * rng.choice([-1, 1], (20, 2))
    mask, n_in = fe.op_ransac_fundamental(p0, p1, thr, 0.999)
    static = np.ones(n, bool)
    static[lost] = False
    assert mask[static].all() and n_in >= n - 20


def test_synth_sequence_is_deterministic(synth):
    a = synth.SynthSequence(seed=5, width=320, height=192, n_frames=5)
    b = synth.SynthSequence(seed=5, width=320, height=192, n_frames=5)
    assert np.array_equal(a.frame(3), b.frame(3)) and not np.array_equal(a.frame(3), a.frame(2))
    assert a.frame(0).shape == (192, 320) and a.frame(0).dtype == np.uint8
    m = synth.SynthSequence(seed=5, width=320, height=192, n_frames=5, moving_mask=True).mask(2)
    assert m.max() == 255 and m.min() == 0


def test_introsort_restatement_equals_std_sort(fe):
    """pl-viwo_b200/csrc/introsort.h (the sort the selection kernel runs) against the real libstdc++ std::sort with the
    reference's comparator (oracle shim), on tie-heavy inputs: the PERMUTATION must be identical, not just the keys."""
    from oracle import cvops
    rng = np.random.default_rng(5)
    for trial in range(300):
        n = int(rng.integers(0, 70)) if trial < 100 else int(rng.integers(70, 6000))
        span = int(rng.integers(1, 4)) if trial % 3 == 0 else int(rng.integers(1, 80))
        resp = rng.integers(20, 20 + span, n).astype(np.uint32)
        if trial % 5 == 1:
            resp = np.sort(resp)
        if trial % 5 == 2:
            resp = np.sort(resp)[::-1].copy()
        packed = (resp << 24) | np.arange(n, dtype=np.uint32)      # low bits = original index
        nfg = int(rng.integers(1, 40))
        got, pre = fe.op_sort_corners(packed, nfg, device=-1, prefix=True)
        perm = cvops.sort_perm(resp.astype(np.float32))
        assert np.array_equal(got & 0xffffff, np.asarray(perm, np.uint32)), (trial, n, span)
        # the pruned selection the kernel runs (isort::sort_prefix): the same first nfg elements, in the same order
        idx = (pre[:, 0].astype(np.uint32) | (pre[:, 1].astype(np.uint32) << 12))
        assert np.array_equal(idx, np.asarray(perm[:nfg], np.uint32)), (trial, n, span, nfg)


def test_append_new_measurements(fe):
    """The consumer side of the drop-in (UpdaterCamera.cpp:111): trackDATABASE->append_new_measurements(tracker db)."""
    trk, upd = fe.FeatureDatabase(), fe.FeatureDatabase()
    for t in (1.0, 2.0):
        trk.update_feature(7, t, 0, 10 + t, 20 + t, 0.1, 0.2)
    trk.update_feature(9, 2.0, 0, 1, 2, 0.01, 0.02)
    upd.append_new_measurements(trk)
    assert sorted(upd.get_internal_data()) == [7, 9] and upd.get_internal_data()[7].timestamps == [1.0, 2.0]
    trk.update_feature(7, 3.0, 0, 13, 23, 0.1, 0.2)
    upd.append_new_measurements(trk)                       # only the unseen timestamp is appended
    assert upd.get_internal_data()[7].timestamps == [1.0, 2.0, 3.0] and len(upd.get_internal_data()[7].uvs) == 3
    upd.append_new_measurements(trk)                       # idempotent
    assert upd.get_internal_data()[7].timestamps == [1.0, 2.0, 3.0]
    trk.get_internal_data()[9].chi_test = False
    trk.update_feature(9, 3.0, 0, 1, 2, 0.01, 0.02)
    upd.append_new_measurements(trk)                       # failed chi-square: flag copied, nothing appended
    assert upd.get_internal_data()[9].chi_test is False and upd.get_internal_data()[9].timestamps == [2.0]


def test_line_match_inverted_index_equals_reference_loop(fe):
    """The library's LineMatch (inverted index id -> last lines) against the oracle's line-by-line restatement of
    TrackLSD::LineMatch (TrackLSD.cpp:368-407: triple loop, the LAST satisfying last-frame line wins) on random line sets
    with few distinct point ids, so that lines share 0, 1 or several ids and LineSimilar decides the 1-id cases."""
    from oracle import frontend as ofe
    rng = np.random.default_rng(5)
    n_matched = 0
    for trial in range(60):
        n0, n1 = int(rng.integers(0, 25)), int(rng.integers(0, 25))
        npid = int(rng.integers(3, 40))

        def lines(n):
            a = rng.uniform(0, 300, (n, 2)).astype(np.float32)
            d = rng.uniform(-60, 60, (n, 2)).astype(np.float32)
            return np.concatenate([a, a + d], 1).astype(np.float32)

        def pols(n):
            return [{int(p): 1.0 for p in rng.choice(npid, size=min(int(rng.integers(1, 5)), npid), replace=False)} for _ in range(n)]
        l0, l1 = lines(n0), lines(n1)
        if n0 and n1 and trial % 3 == 0:      # some new lines lie on top of old ones (LineSimilar true)
            k = min(n0, n1)
            l1[:k] = l0[:k] + rng.uniform(-2, 2, (k, 4)).astype(np.float32)
        p0, p1 = pols(n0), pols(n1)
        want = ofe.TrackLSD.line_match(l1, l0, p0, p1)
        got = fe.op_line_match(p0, l0, p1, l1)
        assert got == {int(k): int(v) for k, v in want.items()}, trial
        n_matched += len(want)
    assert n_matched > 100


def test_assign_points_to_lines_equals_oracle(fe):
    """The library's AssignPointToLines (AVX2 candidate test, one bit per point, exact PointLineDistance on the survivors)
    against the oracle's restatement of TrackLSD.cpp:744-792 — including the mis-indexed bounding box of :754-757 — on
    random segments with points scattered on and around them; point counts that are not multiples of 8."""
    from oracle import frontend as ofe
    rng = np.random.default_rng(11)
    n_pairs = 0
    for trial in range(40):
        n_lines, n_pts = int(rng.integers(0, 60)), int(rng.integers(0, 333))
        a = rng.uniform(0, 560, (n_lines, 2)).astype(np.float32)
        d = rng.uniform(-300, 300, (n_lines, 2)).astype(np.float32)
        lines = np.concatenate([a, a + d], 1).astype(np.float32)
        pts = rng.uniform(0, 560, (n_pts, 2)).astype(np.float32)
        if n_lines and n_pts:      # half of the points sit within a few pixels of some segment
            k = n_pts // 2
            li = rng.integers(0, n_lines, k)
            t = rng.uniform(-0.1, 1.1, (k, 1)).astype(np.float32)
            pts[:k] = (lines[li, :2] + t * (lines[li, 2:] - lines[li, :2]) + rng.normal(0, 3.0, (k, 2))).astype(np.float32)
        pids = rng.permutation(100000)[:n_pts].astype(np.uint64)
        rel, pos, new_lines, new_ids = ofe.TrackLSD.assign_points_to_lines(lines, list(range(n_lines)), pts, [int(p) for p in pids])
        idx, pol = fe.op_assign_points(lines, pts, pids)
        assert list(idx) == list(new_ids), trial
        for got, want in zip(pol, rel):
            assert list(got.keys()) == [int(k) for k in want.keys()], trial
            assert np.allclose(list(got.values()), [float(v) for v in want.values()], rtol=0, atol=1e-6), trial
            n_pairs += len(want)
    assert n_pairs > 500


def test_ctypes_structs_match_the_c_header(fe, tmp_path):
    """sizeof / offsetof of every struct of include/plviwo_fe.h, printed by a C program compiled from the header itself,
    against the ctypes mirror the tests and bench.py use."""
    import ctypes as C
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    structs = {"FeConfig": fe.FeConfig, "FePointRow": fe.FePointRow, "FeLineRow": fe.FeLineRow, "FeLinePoint": fe.FeLinePoint,
               "FeFrameInfo": fe.FeFrameInfo, "FeStageTimes": fe.FeStageTimes, "FePlayStats": fe.FePlayStats,
               "FeStereoInfo": fe.FeStereoInfo, "FeGroupTimes": fe.FeGroupTimes}
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "plviwo_fe.h"', "int main(void) {"]
    for name, cls in structs.items():
        lines.append('  printf("%s size %%zu\\n", sizeof(%s));' % (name, name))
        for fname, _ in cls._fields_:
            lines.append('  printf("%s %s %%zu\\n", offsetof(%s, %s));' % (name, fname, name, fname))
    lines += ["  return 0;", "}"]
    src = tmp_path / "abi.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "abi"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)])
    out = subprocess.check_output([str(exe)], text=True).split("\n")
    seen = 0
    for ln in out:
        if not ln:
            continue
        name, field, value = ln.split()
        cls = structs[name]
        if field == "size":
            assert C.sizeof(cls) == int(value), ln
        else:
            assert getattr(cls, field).offset == int(value), ln
        seen += 1
    assert seen > 60
