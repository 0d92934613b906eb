"""CPU model of the packed 16-bit-lane arithmetic of k_eq_pyr1 (pl-viwo_b200/csrc/kernels_image.cu: hpyr_words,
vpyr_words, pack_hi_bytes and the half-image sum), restated in NumPy uint32 words with __byte_perm, against
cv2.pyrDown and the 2 x 2 mean.  A carry from one lane into the other would show here as a wrong byte."""
import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")


def byte_perm(x, y, s):
    """__byte_perm(x, y, s): result byte i is byte (s >> 4i) & 7 of the 8-byte value y:x."""
    xy = (np.asarray(y, np.uint64) << np.uint64(32)) | np.asarray(x, np.uint64)
    out = np.zeros(np.broadcast(x, y).shape, np.uint64)
    for i in range(4):
        sel = (s >> (4 * i)) & 7
        out |= ((xy >> np.uint64(8 * sel)) & np.uint64(0xFF)) << np.uint64(8 * i)
    return out.astype(np.uint32)


def words(rows):
    """Bytes (..., 4k) -> little-endian uint32 words (..., k)."""
    return np.ascontiguousarray(rows).view(np.uint32)


def hpyr_words(wd):
    """hpyr_words on all pair words of a row: wd[..., k] = pixels 4k .. 4k+3; hs[..., m] centred on pixels 4m+4, 4m+6."""
    ev = byte_perm(wd, 0, 0x4240)
    od = byte_perm(wd, 0, 0x4341)
    n = wd.shape[-1] - 2
    e_m2 = byte_perm(ev[..., :n], ev[..., 1:n + 1], 0x5432)
    e_p2 = byte_perm(ev[..., 1:n + 1], ev[..., 2:n + 2], 0x5432)
    o_m1 = byte_perm(od[..., :n], od[..., 1:n + 1], 0x5432)
    return e_m2 + e_p2 + np.uint32(4) * (o_m1 + od[..., 1:n + 1]) + np.uint32(6) * ev[..., 1:n + 1]


def packed_pyr_down(img):
    """cv::pyrDown to ((w + 1) / 2, (h + 1) / 2) the way k_eq_pyr1 computes level 1: REFLECT_101 staging with pixel 2x - 4 at
    the first byte of a word, packed horizontal sums, packed vertical sums + 128, high bytes."""
    h, w = img.shape
    w1, h1 = (w + 1) // 2, (h + 1) // 2
    npair = (w1 + 1) // 2
    ncols = 4 * (npair + 2)                          # pixels -4 .. 4 * npair + 3
    xs = np.arange(-4, ncols - 4)
    ys = np.arange(-2, 2 * h1 + 3)
    ref = lambda i, n: np.where(i < 0, -i, np.where(i >= n, 2 * n - 2 - i, i))
    ok_x = (xs > -w) & (xs < 2 * w - 1)              # bytes outside REFLECT_101's range are staged as 0 and never used
    stage = np.where(ok_x[None, :], img[ref(ys, h)][:, ref(np.where(ok_x, xs, 0), w)], 0).astype(np.uint8)
    hs = hpyr_words(words(stage))                    # (rows, npair), lanes <= 16 * 255
    assert (hs & 0xFFFF).max() <= 4080 and (hs >> 16).max() <= 4080
    v = (hs[0:2 * h1:2] + hs[4:2 * h1 + 4:2] + np.uint32(4) * (hs[1:2 * h1 + 1:2] + hs[3:2 * h1 + 3:2]) +
         np.uint32(6) * hs[2:2 * h1 + 2:2] + np.uint32(0x00800080))
    assert (v & 0xFFFF).max() <= 65408 and (v >> 16).max() <= 65408
    out = np.empty((h1, 2 * npair), np.uint8)
    out[:, 0::2] = (v >> 8) & 0xFF
    out[:, 1::2] = v >> 24
    return out[:, :w1]


def packed_half(img):
    """The half-resolution image, (a + b + c + d + 2) >> 2 over 2 x 2 blocks, from the Ev / Od lane sums."""
    h, w = img.shape
    hh, wh = h // 2, w // 2
    wq = (wh + 3) // 4 * 4
    pad = np.zeros((2 * hh, 2 * wq), np.uint8)
    pad[:, :2 * wh] = img[:2 * hh, :2 * wh]
    a, b = words(pad[0::2]), words(pad[1::2])
    s = (byte_perm(a, 0, 0x4240) + byte_perm(a, 0, 0x4341) + byte_perm(b, 0, 0x4240) + byte_perm(b, 0, 0x4341) +
         np.uint32(0x00020002))
    q = s >> 2
    out = np.empty((hh, wq), np.uint8)
    out[:, 0::2] = q & 0xFF
    out[:, 1::2] = (q >> 16) & 0xFF
    return out[:, :wh]


def _cases():
    rng = np.random.default_rng(7)
    return {
        "noise": rng.integers(0, 256, (96, 160), dtype=np.uint8),
        "odd": rng.integers(0, 256, (37, 85), dtype=np.uint8),
        "w1mod4": rng.integers(0, 256, (33, 129), dtype=np.uint8),
        "w2mod4": rng.integers(0, 256, (35, 130), dtype=np.uint8),
        "w3mod4": rng.integers(0, 256, (31, 131), dtype=np.uint8),
        "saturated": np.full((40, 72), 255, np.uint8),
        "two_valued": np.where(rng.random((48, 64)) < 0.5, 0, 255).astype(np.uint8),
        "small": rng.integers(0, 256, (7, 9), dtype=np.uint8),
    }


@pytest.mark.parametrize("name", list(_cases()))
def test_packed_pyr_down_equals_cv2(name):
    img = _cases()[name]
    assert np.array_equal(packed_pyr_down(img), cv2.pyrDown(img))


@pytest.mark.parametrize("name", list(_cases()))
def test_packed_half_equals_2x2_mean(name):
    img = _cases()[name]
    h, w = img.shape
    x = img[:h // 2 * 2, :w // 2 * 2].astype(np.int32)
    ref = ((x[0::2, 0::2] + x[0::2, 1::2] + x[1::2, 0::2] + x[1::2, 1::2] + 2) >> 2).astype(np.uint8)
    assert np.array_equal(packed_half(img), ref)
    if h % 2 == 0 and w % 2 == 0:
        assert np.array_equal(packed_half(img), cv2.resize(img, None, fx=0.5, fy=0.5, interpolation=cv2.INTER_LINEAR))
