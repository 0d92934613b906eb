"""The line detector's first labelling step (ccl_tile_body through plviwo_op_ccl_tiles): the 8-connected components of
every 64 x 16 tile on its own, against cv2.connectedComponentsWithStats per tile.  Root = the component's smallest raster
index; cnt and bbox (max y, min x, max x) at the root; the tile-local roots as a set."""
import cv2
import numpy as np
import pytest

from oracle import cvops

pytestmark = pytest.mark.gpu

TW, TH = 64, 16


def _reference(e):
    h, w = e.shape
    label = np.full((h, w), -1, np.int64)
    cnt, ymax, xmin, xmax, roots = {}, {}, {}, {}, []
    for y0 in range(0, h, TH):
        for x0 in range(0, w, TW):
            tile = e[y0:y0 + TH, x0:x0 + TW].astype(np.uint8)
            n, lab, stats, _ = cv2.connectedComponentsWithStats(tile, connectivity=8)
            for c in range(1, n):
                ys, xs = np.nonzero(lab == c)   # row-major: the first one is the smallest raster index
                root = (y0 + ys[0]) * w + x0 + xs[0]
                label[y0 + ys, x0 + xs] = root
                left, top, bw, bh, area = stats[c]
                cnt[root], ymax[root] = area, y0 + top + bh - 1
                xmin[root], xmax[root] = x0 + left, x0 + left + bw - 1
                roots.append(root)
    return label, cnt, ymax, xmin, xmax, np.sort(np.array(roots, np.int64))


def _check(fe, e, what):
    e = np.ascontiguousarray(e, bool)
    label, cnt, ymax, xmin, xmax, roots = _reference(e)
    got = fe.op_ccl_tiles(e)
    assert np.array_equal(got["label"], label), "%s: %d labels differ" % (what, int((got["label"] != label).sum()))
    assert np.array_equal(got["roots"], roots), "%s: tile-local roots differ" % what
    if len(roots):
        g_cnt = got["cnt"].reshape(-1)[roots]
        g_bb = got["bbox"].reshape(3, -1)[:, roots]
        assert np.array_equal(g_cnt, [cnt[r] for r in roots]), "%s: pixel counts differ" % what
        assert np.array_equal(g_bb[0], [ymax[r] for r in roots]), "%s: max y differs" % what
        assert np.array_equal(g_bb[1], [xmin[r] for r in roots]), "%s: min x differs" % what
        assert np.array_equal(g_bb[2], [xmax[r] for r in roots]), "%s: max x differs" % what


def _snake_rows():
    """One serpentine per tile through every even row (runs of 64 joined at alternate ends)."""
    t = np.zeros((TH, TW), bool)
    t[0::2] = True
    for k, y in enumerate(range(1, TH, 2)):
        t[y, TW - 1 if k % 2 == 0 else 0] = True
    return t


def _snake_cols():
    """One serpentine per tile through every even column: 32 one-pixel runs per row, chained through alternate ends."""
    t = np.zeros((TH, TW), bool)
    t[:, 0::2] = True
    for k, x in enumerate(range(1, TW, 2)):
        t[TH - 1 if k % 2 == 0 else 0, x] = True
    return t


def test_ccl_tiles_bench_frames(fe, synth):
    for seed in (1000, 1001):
        seq = synth.SynthSequence(seed=seed, n_frames=48)
        for t in (0, 40):
            small = cvops.half_res(cvops.equalize_hist(seq.frame(t)))
            e = cvops.canny(small) > 0
            e[:6, :6] = False
            e[-5:, -5:] = False
            _check(fe, e, "seed %d frame %d" % (seed, t))


def test_ccl_tiles_patterns(fe):
    yy, xx = np.mgrid[:TH, :TW]
    tiles = {
        "empty": np.zeros((TH, TW), bool),
        "full": np.ones((TH, TW), bool),               # 1024 edges in one tile
        "checkerboard": (yy + xx) % 2 == 0,            # 512 runs, joined through corners only
        "checkerboard_odd": (yy + xx) % 2 == 1,
        "diagonal": (xx - yy) % 4 == 0,                 # stripes connected through corners only
        "antidiagonal": (xx + yy) % 3 == 0,
        "snake_rows": _snake_rows(),
        "snake_cols": _snake_cols(),
        "comb": (yy == TH - 1) | (xx % 2 == 0),         # one run below 32 runs above it
        "rings": np.maximum(np.abs(yy - 7.5), np.abs(xx - 31.5) / 4).astype(int) % 2 == 0,
    }
    for name, t in tiles.items():
        _check(fe, np.tile(t, (3, 2)), name)
    # the patterns side by side, so tiles see different neighbours and the frame has several tile rows and columns
    _check(fe, np.vstack([np.hstack(list(tiles.values())[i:i + 5]) for i in (0, 5)]), "mosaic")


@pytest.mark.parametrize("shape", [(280, 640), (40, 100), (23, 77), (16, 64), (9, 33), (1, 1), (17, 130)])
@pytest.mark.parametrize("density", [0.25, 0.55])
def test_ccl_tiles_random_partial(fe, shape, density):
    """Partial tiles at the right and bottom edges, widths that are not a multiple of 32."""
    rng = np.random.default_rng(shape[0] * 1000 + shape[1] + int(density * 100))
    _check(fe, rng.random(shape) < density, "random %s %.2f" % (shape, density))
    _check(fe, np.ones(shape, bool), "full %s" % (shape,))
