"""MatrixMarket / Ginkgo-binary I/O of the host layer (ginkgo_b200/host/gko_b200_io.hpp, pure
C++ without CUDA) against the REAL reference's gko::read_generic_raw / write_raw /
write_binary_raw (core/base/mtx_io.cpp) through oracle/_ref, or its recorded answers
(tests/reference.py).  CPU only: the header is compiled into tests/cpp/io_check with plain g++."""
import os
import subprocess

import numpy as np
import pytest

from tests import reference as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def io_check(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("io") / "io_check")
    subprocess.run(["g++", "-O1", "-std=c++17", "-Wall", "-o", exe,
                    os.path.join(ROOT, "tests", "cpp", "io_check.cpp")], check=True)
    return exe


def ours(io_check, path, vt="f64", it="i32"):
    out = subprocess.run([io_check, "read", str(path), vt, it], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.strip().split("\n")
    rows, cols, nnz = map(int, lines[0].split())
    t = [l.split() for l in lines[1:]]
    assert len(t) == nnz
    return (rows, cols, np.array([int(x[0]) for x in t], np.int64), np.array([int(x[1]) for x in t], np.int64),
            np.array([float(x[2]) for x in t]))


FILES = {
    "coordinate_general": "%%MatrixMarket matrix coordinate real general\n% comment\n%another\n4 5 6\n"
                          "4 5 1.5\n1 1 -2\n2 3 1e-3\n1 4 7.25 trailing text\n3 2 0\n2 1 3.0e2\n",
    "coordinate_symmetric": "%%MatrixMarket matrix coordinate real symmetric\n3 3 4\n1 1 2\n2 1 -1\n3 2 -1\n3 3 2\n",
    "coordinate_skew": "%%MatrixMarket matrix coordinate real skew-symmetric\n3 3 2\n2 1 4\n3 1 -2.5\n",
    "coordinate_pattern": "%%MatrixMarket matrix coordinate pattern general\n3 4 4\n1 1\n2 4\n3 2\n3 3\n",
    "coordinate_pattern_symmetric": "%%MatrixMarket matrix coordinate pattern symmetric\n3 3 3\n1 1\n3 1\n3 2\n",
    "coordinate_integer": "%%MatrixMarket matrix coordinate integer general\n2 2 3\n1 1 4\n1 2 -7\n2 2 12\n",
    "upper_case_header": "%%MATRIXMARKET MATRIX COORDINATE REAL GENERAL\n2 2 1\n2 1 9\n",
    "array_general": "%%MatrixMarket matrix array real general\n3 2\n1\n2\n3\n4\n5\n6\n",
    "array_symmetric": "%%MatrixMarket matrix array real symmetric\n3 3\n1\n2\n3\n4\n5\n6\n",
    "array_skew": "%%MatrixMarket matrix array real skew-symmetric\n3 3\n1\n2\n3\n",
    "empty": "%%MatrixMarket matrix coordinate real general\n5 7 0\n",
}


@pytest.mark.parametrize("name", sorted(FILES))
def test_read_matches_reference(io_check, tmp_path, name):
    path = tmp_path / (name + ".mtx")
    path.write_text(FILES[name])
    rr, rc, r_rows, r_cols, r_vals = ref.read_mtx(path)
    orows, ocols, o_r, o_c, o_v = ours(io_check, path)
    assert (orows, ocols) == (rr, rc)
    assert np.array_equal(o_r, r_rows) and np.array_equal(o_c, r_cols)
    assert np.array_equal(o_v, r_vals)


def test_float_and_int64_targets(io_check, tmp_path):
    path = tmp_path / "a.mtx"
    path.write_text(FILES["coordinate_general"])
    _, _, _, _, v64 = ours(io_check, path, "f64", "i64")
    _, _, _, _, v32 = ours(io_check, path, "f32", "i32")
    assert np.array_equal(v32, v64.astype(np.float32).astype(np.float64))


@pytest.mark.parametrize("layout", ["coordinate", "array", "binary"])
def test_write_round_trips_through_the_reference(io_check, tmp_path, layout):
    rng = np.random.default_rng(3)
    n, m, nnz = 17, 23, 60
    pos = rng.choice(n * m, size=nnz, replace=False)
    rows, cols = np.sort(pos) // m, np.sort(pos) % m
    vals = rng.uniform(-1, 1, nnz)
    src = tmp_path / "src.bin"
    ref.write_mtx(src, "binary", n, m, rows, cols, vals)  # the reference writes ...
    got = ours(io_check, src)                               # ... we read its binary
    assert got[:2] == (n, m) and np.array_equal(got[2], rows) and np.array_equal(got[3], cols)
    assert np.array_equal(got[4], vals)
    out = tmp_path / ("out." + layout)
    res = subprocess.run([io_check, "write", str(src), str(out), layout], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    rr, rc, r_rows, r_cols, r_vals = ref.read_mtx(out)     # we write, the reference reads
    assert (rr, rc) == (n, m)
    if layout == "array":  # dense: explicit zeros come back as entries
        dense = np.zeros((n, m))
        dense[rows, cols] = vals
        back = np.zeros((n, m))
        back[r_rows, r_cols] = r_vals
        assert len(r_vals) == n * m and np.array_equal(back, dense)
    else:
        assert np.array_equal(r_rows, rows) and np.array_equal(r_cols, cols)
        assert np.array_equal(r_vals, vals)
    # byte-identical files for the same data
    theirs = tmp_path / ("ref." + layout)
    if layout == "array":
        ref.write_mtx(theirs, layout, n, m, rows, cols, vals)
    else:
        ref.write_mtx(theirs, layout, n, m, rows, cols, vals)
    assert out.read_bytes() == theirs.read_bytes()


@pytest.mark.parametrize("text,code", [
    ("%%MatrixMarket matrix coordinate complex general\n1 1 1\n1 1 1 0\n", 3),
    ("%%MatrixMarket matrix coordinate real hermitian\n1 1 1\n1 1 1\n", 3),
    ("%%MatrixMarket tensor coordinate real general\n1 1 1\n1 1 1\n", 1),
    ("%%MatrixMarket matrix coordinate real general\n2 2 2\n1 1 1\n", 1),
])
def test_errors(io_check, tmp_path, text, code):
    path = tmp_path / "bad.mtx"
    path.write_text(text)
    out = subprocess.run([io_check, "read", str(path), "f64", "i32"], capture_output=True, text=True)
    assert out.returncode == code, (out.returncode, out.stderr)


@pytest.mark.parametrize("name", ["coordinate_general", "coordinate_symmetric", "array_general", "empty"])
def test_csr_array_round_trip(io_check, tmp_path, name):
    """the host half of Csr::read / Csr::write: matrix_data -> (row_ptrs, col_idxs, values) ->
    matrix_data reproduces the data, and the written binary file reads back identically"""
    path = tmp_path / (name + ".mtx")
    path.write_text(FILES[name])
    out = tmp_path / "out.bin"
    res = subprocess.run([io_check, "csr", str(path), str(out)], capture_output=True, text=True)
    assert res.returncode == 0, (res.returncode, res.stderr)
    a, b = ref.read_mtx(path), ref.read_mtx(out)
    assert a[:2] == b[:2] and all(np.array_equal(x, y) for x, y in zip(a[2:], b[2:]))
