"""The stream group's LK kernel (one warp per feature, k_lk15w_g's body) against the single-handle kernel (k_lk15), which
is its bit reference: positions and statuses must agree bit for bit.  A group only ever hands the warp kernel points
that a tracker produced; plviwo_op_lk_warp runs the same body on arbitrary points, so these tests aim at its border
paths: neighbourhoods and regions of the next image that cross an edge of a pyramid level at every offset and word
alignment, odd level widths, points outside the frame, flows that leave the image and flat patches.

The op's pyramids have 256-byte pitches (as the group's have), so the case of an image pointer or pitch that is not a
multiple of 4 cannot be reached from here.  In that case the kernel assembles every staged word byte by byte from
REFLECT_101 columns, which is the code the words crossing an edge take; the border cases below run it for every word
position of a staged row."""
import numpy as np
import pytest

from oracle import cvops

pytestmark = pytest.mark.gpu


def _assert_same(fe, a, b, pts0, pts1, levels):
    p_ref, s_ref = fe.op_lk(a, b, pts0, pts1, 15, levels, form="cta")
    p_got, s_got = fe.op_lk(a, b, pts0, pts1, 15, levels, form="warp")
    bad = np.flatnonzero((s_ref != s_got) | np.any(p_ref.view(np.uint32) != p_got.view(np.uint32), axis=1))
    assert bad.size == 0, "%d of %d points differ, first %s: cta %s %d, warp %s %d" % (
        bad.size, len(pts0), pts0[bad[0]], p_ref[bad[0]], s_ref[bad[0]], p_got[bad[0]], s_got[bad[0]])
    return s_ref


def _pair(synth, seed=1000, width=1280, height=560):
    seq = synth.SynthSequence(seed=seed, width=width, height=height, n_frames=3)
    return cvops.equalize_hist(seq.frame(0)), cvops.equalize_hist(seq.frame(1))


@pytest.mark.parametrize("levels", [0, 1, 2, 3, 4])
def test_lk_warp_bench_frames(fe, synth, levels):
    a, b = _pair(synth)
    xy, resp = cvops.fast_cell(a, 20)
    order = np.argsort(-resp, kind="stable")[:2400]
    rng = np.random.default_rng(levels)
    pts0 = xy[order].astype(np.float32) + rng.uniform(-0.5, 0.5, (len(order), 2)).astype(np.float32)
    assert len(pts0) >= 2000
    _assert_same(fe, a, b, pts0, pts0, levels)


def _border_points(w, h, levels, rng):
    """Level-l positions d + frac px from each border (d = 0..25, frac in quarters), mapped to level 0, so that at every
    level some window and some staged region straddle the edge at every byte offset."""
    pts = []
    for lv in range(levels + 1):
        s = float(1 << lv)
        wl, hl = (w + s - 1) // s, (h + s - 1) // s
        for d in range(26):
            for frac in (0.05, 0.3, 0.55, 0.8):
                off = d + frac
                along_x = rng.uniform(0, wl - 1)
                along_y = rng.uniform(0, hl - 1)
                for x, y in ((off, along_y), (wl - 1 - off, along_y), (along_x, off), (along_x, hl - 1 - off),
                             (off, off), (wl - 1 - off, hl - 1 - off)):
                    pts.append((x * s, y * s))
    return np.array(pts, np.float32)


def _word_offsets(p, levels):
    """rx0 & 3 of the previous-image neighbourhood at every level (rx0 = floor(x / 2^l - 7) - 1)."""
    return {int(np.floor(x / (1 << lv) - 7)) - 1 & 3 for x in p[:, 0] for lv in range(levels + 1)}


@pytest.mark.parametrize("shape", [(560, 1280), (141, 333), (97, 258), (75, 131)])
def test_lk_warp_borders(fe, synth, shape):
    h, w = shape
    levels = 4
    a, b = _pair(synth, seed=1001)
    a = np.ascontiguousarray(a[:h, :w])
    b = np.ascontiguousarray(b[:h, :w])
    rng = np.random.default_rng(w)
    pts0 = _border_points(w, h, levels, rng)
    # initial flows of up to 6 px in any direction: the region of the next image starts at every word offset and is
    # re-staged as the window moves along or across the edge
    flow = rng.uniform(-6, 6, pts0.shape).astype(np.float32)
    pts1 = pts0 + flow
    assert _word_offsets(pts0, levels) == {0, 1, 2, 3}
    reg = {int(np.floor(x / (1 << levels) - 7)) - 4 & 3 for x in pts1[:, 0]}   # reg_x0 & 3 at the first iteration
    assert reg == {0, 1, 2, 3}
    _assert_same(fe, a, b, pts0, pts1, levels)


def test_lk_warp_odd_widths(fe):
    rng = np.random.default_rng(7)
    for h, w in ((141, 333), (63, 201), (37, 85)):
        a = rng.integers(0, 256, (h, w), dtype=np.uint8)
        a = cvops.equalize_hist(np.clip(a.astype(np.int32) // 3 + np.indices((h, w)).sum(0) % 170, 0, 255).astype(np.uint8))
        b = np.roll(a, (1, 2), axis=(0, 1))
        pts0 = np.stack([rng.uniform(-3, w + 2, 3000), rng.uniform(-3, h + 2, 3000)], 1).astype(np.float32)
        for levels in (2, 3, 4):
            _assert_same(fe, a, b, pts0, pts0 + np.float32([2.0, 1.0]), levels)


def test_lk_warp_outside_flat_and_escaping(fe, synth):
    a, b = _pair(synth, seed=1002)
    a = a.copy()
    b = b.copy()
    a[200:300, 500:700] = 90          # a flat patch: minEig fails at every level
    b[200:300, 500:700] = 90
    w, h = a.shape[1], a.shape[0]
    outside = np.array([[-30, 100], [-9, -9], [1300, 200], [w + 7, h + 7], [640, -20], [640, h + 40], [-200, -200]], np.float32)
    flat = np.array([[600, 250], [550.5, 230.25], [650.75, 270.5]], np.float32)
    # initial flows that carry the window out of the frame within a few iterations, and ones that start outside
    rng = np.random.default_rng(3)
    near = np.stack([rng.uniform(1, 12, 200), rng.uniform(0, h - 1, 200)], 1).astype(np.float32)
    near_r = np.stack([rng.uniform(w - 12, w - 1, 200), rng.uniform(0, h - 1, 200)], 1).astype(np.float32)
    pts0 = np.concatenate([outside, flat, near, near_r, near[:, ::-1] * np.float32([h / w, w / h])], 0)
    pts1 = pts0.copy()
    n_o, n_f = len(outside), len(flat)
    pts1[n_o + n_f:n_o + n_f + 200, 0] -= rng.uniform(10, 40, 200).astype(np.float32)
    pts1[n_o + n_f + 200:n_o + n_f + 400, 0] += rng.uniform(10, 40, 200).astype(np.float32)
    for levels in (0, 2, 4):
        st = _assert_same(fe, a, b, pts0, pts1, levels)
        assert not st[:n_o].any()
        assert not st[n_o:n_o + n_f].any()


def test_lk_warp_rejects_other_windows(fe, synth):
    a, b = _pair(synth)
    pts = np.array([[640, 280]], np.float32)
    with pytest.raises(fe.FrontEndError):
        fe.op_lk(a, b, pts, pts, 21, 3, form="warp")
