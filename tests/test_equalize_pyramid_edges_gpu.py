"""plviwo_op_equalize_pyramid (k_hist's per-frame LUT, k_eq_pyr1, k_pyr_down) on the inputs that reach the edges of the
packed 16-bit-lane paths: widths 1, 2 and 3 mod 4 with odd heights, a frame narrower than one 64 x 16 level-1 tile, a
saturated frame (every vertical lane at its 65408 bound) and a two-valued frame (the LUT's i0 edge).  Bit-exact against
cv2; the half-resolution image against the 2 x 2 mean (a + b + c + d + 2) >> 2, which is cv2's INTER_LINEAR 0.5 resize
for even sides."""
import numpy as np
import pytest

from oracle import cvops

pytestmark = pytest.mark.gpu


def _images():
    rng = np.random.default_rng(19)
    return {
        "w1mod4": rng.integers(0, 256, (141, 333), dtype=np.uint8),
        "w2mod4": rng.integers(20, 220, (99, 258), dtype=np.uint8),
        "w3mod4": rng.integers(0, 256, (77, 259), dtype=np.uint8),
        "narrow": rng.integers(0, 256, (85, 37), dtype=np.uint8),
        "saturated": np.full((96, 160), 255, np.uint8),
        "two_valued": np.where(rng.random((120, 200)) < 0.3, 40, 200).astype(np.uint8),
    }


def _half_2x2(img):
    h, w = img.shape
    x = img[:h // 2 * 2, :w // 2 * 2].astype(np.int32)
    return ((x[0::2, 0::2] + x[0::2, 1::2] + x[1::2, 0::2] + x[1::2, 1::2] + 2) >> 2).astype(np.uint8)


@pytest.mark.parametrize("name", list(_images()))
def test_equalize_pyramid_edges_bit_exact(fe, name):
    img = _images()[name]
    levels = 5
    lv, half = fe.op_equalize_pyramid(img, levels)
    eq = cvops.equalize_hist(img)
    assert np.array_equal(lv[0], eq), "equalizeHist differs"
    ref = cvops.build_pyramid(eq, 3, levels)
    for l in range(1, min(len(ref), len(lv))):
        assert lv[l].shape == ref[l].shape
        assert np.array_equal(lv[l], ref[l]), "pyrDown level %d differs" % l
    assert np.array_equal(half, _half_2x2(eq)), "half-res differs"
    if img.shape[0] % 2 == 0 and img.shape[1] % 2 == 0:
        assert np.array_equal(half, cvops.half_res(eq)), "half-res differs from cv2"
