"""Stereo group creator (plviwo_fe_stereo_group_create): every refusal comes with its reason and before the device query,
so the same checks hold on a machine without a GPU."""
import ctypes as C

import pytest


def _create(fe, cfg, n_rigs=2):
    L = fe.lib()
    h = C.c_void_p()
    rc = L.plviwo_fe_stereo_group_create(C.byref(cfg), n_rigs, 0, C.byref(h))
    why = L.plviwo_fe_stereo_group_last_error(None)
    assert not h.value, "created a stereo group from a config that must be refused"
    return rc, (why or b"").decode()


@pytest.mark.parametrize("kw,reason", [
    (dict(width=63), "image size must be in [64, 4095]"),
    (dict(win_size=14), "win_size must be odd and in [3, 31]"),
    (dict(pyr_levels=8), "pyr_levels must be in [0, 7]"),
    (dict(num_features=0), "bad grid / distance / feature count"),
    (dict(histogram_method=7), "bad histogram_method"),
    (dict(width=642, height=281), "line tracker needs even (tracking) image dimensions (exact 2x decimation)"),
    (dict(canny_th2=60.0), "canny_th1 != canny_th2: hysteresis pass is not implemented"),
    (dict(grid_x=16, grid_y=17), "a stream group supports at most 256 grid cells"),
    (dict(downsample=1), "cfg.downsample is not supported in a stereo group"),
    (dict(line_samples=4), "cfg.line_samples is not supported in a stereo group"),
])
def test_stereo_group_refuses_bad_configs(fe, kw, reason):
    assert _create(fe, fe.default_config(**kw)) == (fe.FE_BAD_ARG, reason)


@pytest.mark.parametrize("n_rigs", [0, 2049])
def test_stereo_group_refuses_bad_rig_count(fe, n_rigs):
    assert _create(fe, fe.default_config(), n_rigs) == (fe.FE_BAD_ARG, "n_rigs must be in [1, 2048] (2 camera streams per rig, at most 4096)")


def test_stereo_group_needs_a_device(fe):
    if fe.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(fe.FrontEndError) as e:
        fe.StereoGroupFrontEnd(fe.default_config(), 2)
    assert e.value.code == fe.FE_NO_DEVICE
