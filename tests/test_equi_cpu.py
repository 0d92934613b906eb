"""Equidistant (fisheye) camera model without a GPU: the host form of the undistortion the handles use for their line rows
(plviwo_op_undistort_equi with device < 0, the same tracker_core.h arithmetic the kernels run) is cv2.fisheye.undistortPoints
bit for bit; every _create_model creator refuses an unknown model before it looks for a device; the oracle driven through
the equidistant undistortion gives the same rows with the NumPy restatement and with cv2."""
import ctypes as C

import numpy as np
import pytest

from oracle import cvops, npops
from oracle import frontend as ofe

EUROC_K = [458.654, 457.296, 367.215, 248.375]
EUROC_D = [-0.0348, 0.0123, -0.0071, 0.0021]
STRONG_D = [0.35, -0.6, 0.9, -0.4]   # a strongly distorting lens: many points do not converge


class EquiOps:
    """An oracle ops module whose CamBase::undistort_f is CamEqui's (cv::fisheye::undistortPoints, cam/CamEqui.h:108-129)."""

    def __init__(self, base):
        self._base = base

    def __getattr__(self, name):
        return getattr(self._base, name)

    def undistort(self, pts, K, D):
        return self._base.undistort_equi(pts, K, D)


def _points(n=3000, seed=5, wide=False):
    """Points over a 752 x 480 image and 20 px beyond it, plus the principal point (theta_d = 0); wide: out to ~400 px beyond
    the border, where theta_d reaches the 90 degree clamp."""
    rng = np.random.default_rng(seed)
    m = 400 if wide else 20
    pts = np.stack([rng.uniform(-m, 752 + m, n), rng.uniform(-m, 480 + m, n)], 1).astype(np.float32)
    pts[0] = (EUROC_K[2], EUROC_K[3])
    return pts


@pytest.mark.parametrize("wide", [False, True], ids=["image", "wide"])
@pytest.mark.parametrize("D", [EUROC_D, STRONG_D], ids=["euroc", "strong"])
def test_host_form_equals_cv2_bitwise(fe, D, wide):
    pts = _points(wide=wide)
    got = fe.op_undistort_equi(pts, EUROC_K, D, device=-1)
    ref = cvops.undistort_equi(pts, EUROC_K, D)
    assert got.view(np.uint32).tobytes() == ref.view(np.uint32).tobytes()
    failed = (ref == -1e6).all(1)
    if D is STRONG_D and wide:
        assert failed.sum() > 100, failed.sum()     # the (-1e6, -1e6) branch is exercised ...
    assert np.array_equal(got[failed], ref[failed])   # ... and matches
    assert np.signbit(got[0]).tolist() == np.signbit(ref[0]).tolist()   # -0.0 at the principal point, as OpenCV


def test_host_form_edge_inputs_follow_opencv(fe):
    """NaN and far-away inputs go where OpenCV sends them (std::max(-pi/2, NaN) is -pi/2 in OpenCV's clamp)."""
    pts = np.array([[np.nan, 10.0], [1e30, 1.0], [np.inf, 3.0], [EUROC_K[2], 200.0]], np.float32)
    for D in (EUROC_D, STRONG_D):
        got = fe.op_undistort_equi(pts, EUROC_K, D, device=-1)
        ref = cvops.undistort_equi(pts, EUROC_K, D)
        assert got.view(np.uint32).tobytes() == ref.view(np.uint32).tobytes(), (got, ref)


_MODEL_CREATORS = ("handle", "stereo", "group", "stereo_group")


def _create_model(fe, creator, model):
    L = fe.lib()
    cfg = fe.default_config()
    h = C.c_void_p()
    if creator == "handle":
        rc, why = L.plviwo_fe_create_model(C.byref(cfg), model, 0, C.byref(h)), L.plviwo_fe_last_error(None)
    elif creator == "stereo":
        rc = L.plviwo_fe_stereo_create_model(C.byref(cfg), model, None, None, 0, C.byref(h))
        why = L.plviwo_fe_stereo_last_error(None)
    elif creator == "group":
        rc, why = L.plviwo_fe_group_create_model(C.byref(cfg), 2, model, 0, C.byref(h)), L.plviwo_fe_group_last_error(None)
    else:
        rc = L.plviwo_fe_stereo_group_create_model(C.byref(cfg), 2, model, 0, C.byref(h))
        why = L.plviwo_fe_stereo_group_last_error(None)
    assert not h.value, "created an object with an unknown camera model"
    return rc, (why or b"").decode()


@pytest.mark.parametrize("creator", _MODEL_CREATORS)
@pytest.mark.parametrize("model", [2, -1])
def test_model_creators_refuse_unknown_models(fe, creator, model):
    assert _create_model(fe, creator, model) == (fe.FE_BAD_ARG, "camera model must be FE_CAM_RADTAN (0) or FE_CAM_EQUI (1)")


def test_python_creators_take_the_model(fe):
    for make in (lambda: fe.FrontEnd(camera_model=2), lambda: fe.StereoFrontEnd(camera_model=2),
                 lambda: fe.GroupFrontEnd(fe.default_config(), 2, camera_model=2),
                 lambda: fe.StereoGroupFrontEnd(fe.default_config(), 2, camera_model=2)):
        with pytest.raises(fe.FrontEndError) as e:
            make()
        assert e.value.code == fe.FE_BAD_ARG and "camera model" in str(e.value)


def test_oracle_equidistant_rows_npops_equal_cvops(synth):
    """The oracle with the equidistant undistortion, NumPy restatement vs cv2: the same point ids and line rows, positions
    within the LK restatement's 2e-3 px, and every row's (un, vn) the equidistant undistortion of its own (u, v)."""
    seq = synth.SynthSequence(seed=31, width=640, height=280, n_frames=4, hard=False)
    kw = dict(num_features=120, fast_threshold=20, grid_x=5, grid_y=5, min_px_dist=10, pyr_levels=3, win_size=15)
    runs = []
    for ops in (npops, cvops):
        o = ofe.FrontEnd(ofe.FeConfig(K=seq.K, D=tuple(EUROC_D), **kw), ops=EquiOps(ops))
        out = []
        for t in range(4):
            prow, lrow = o.feed(seq.timestamp(t), seq.frame(t), None, seq.vanishing_points(t))
            rows = np.array([(r.u, r.v, r.un, r.vn) for r in prow], np.float32).reshape(-1, 4)
            assert np.array_equal(rows[:, 2:], ops.undistort_equi(rows[:, :2], seq.K, EUROC_D)), t
            out.append(([r.id for r in prow], rows, [(r.id, r.pids, r.D) for r in lrow]))
        runs.append(out)
    assert sum(len(ids) for ids, _, _ in runs[0][1:]) > 50
    for (ids_a, rows_a, lines_a), (ids_b, rows_b, lines_b) in zip(*runs):
        assert ids_a == ids_b and lines_a == lines_b
        assert np.abs(rows_a[:, :2] - rows_b[:, :2]).max(initial=0) < 2e-3
