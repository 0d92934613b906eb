"""bench.py --dump-outputs: the file format two builds are compared with (no GPU: rows built from the binding's dtypes)."""
import numpy as np

import bench
import plviwo_b200 as fe


def _rows(rng, n_pts, n_lines, n_lpts):
    p = np.zeros(n_pts, fe.POINT_ROW_DTYPE)
    p["id"] = rng.integers(1, 10 ** 6, n_pts)
    for k in ("u", "v", "un", "vn"):
        p[k] = rng.uniform(-1, 1280, n_pts)
    ln = np.zeros(n_lines, fe.LINE_ROW_DTYPE)
    ln["id"], ln["D"], ln["n_pts"] = rng.integers(1, 10 ** 6, n_lines), rng.integers(0, 3, n_lines), rng.integers(0, 9, n_lines)
    ln["line"], ln["line_n"] = rng.uniform(0, 1280, (n_lines, 4)), rng.uniform(-1, 1, (n_lines, 4))
    q = np.zeros(n_lpts, fe.LINE_POINT_DTYPE)
    q["pid"], q["dist"], q["u"], q["v"] = rng.integers(0, 10 ** 6, n_lpts), rng.uniform(0, 2, n_lpts), 1.5, 2.5
    return p, ln, q


def test_dump_outputs_layout(tmp_path):
    rng = np.random.default_rng(0)
    rows = [_rows(rng, 5, 3, 7), _rows(rng, 4, 0, 0)]    # the second stream found no line
    bench.dump_outputs(str(tmp_path), [3, 9], rows)
    got = {f.stem: np.load(f) for f in tmp_path.iterdir()}
    assert sorted(got) == ["line_endpoints", "line_ids", "line_point_ids", "line_point_uv", "point_ids", "point_uv"]
    for name, a in got.items():
        assert a.dtype == (np.float64 if name.endswith("ids") else np.float32), name
    assert np.array_equal(got["point_ids"][:, 0], [3] * 5 + [9] * 4)
    assert np.array_equal(got["point_ids"][:, 1], np.concatenate([rows[0][0]["id"], rows[1][0]["id"]]).astype(np.float64))
    assert np.array_equal(got["point_uv"][5:, 2], rows[1][0]["un"])
    assert got["line_ids"].shape == (3, 6) and np.array_equal(got["line_ids"][:, 3], rows[0][1]["n_pts"])
    assert np.array_equal(got["line_endpoints"], np.concatenate([rows[0][1]["line"], rows[0][1]["line_n"]], 1))
    assert got["line_point_ids"].shape == (7, 2) and got["line_point_uv"].shape == (7, 3)
