"""BiCG and its transposes (SURVEY.md 8f rank 3) without a GPU:
  * the oracle restatement of csr::transpose, jacobi::transpose_jacobi, the bicg kernels and the
    BiCG loop against the REAL reference (oracle/_ref, or its recorded answers: Csr::transpose,
    Jacobi::transpose, solver::Bicg with identity / scalar / block Jacobi);
  * a copy of ginkgo_b200/csrc/bicg_transpose.cu compiled for the host against the oracle, bit
    for bit (radix passes, chunk boundaries, empty rows / columns, duplicates, strides).
The GPU runs of the same bodies are in tests/test_zzz_dist_assembly_gpu.py."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import workloads as W
from tests import helpers as H
from tests import reference
from tests.helpers import VT
from tests.test_kernel_sources_cpu import KernelSourceBackend

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
IT = {"i32": np.int32, "i64": np.int64}


@pytest.fixture(scope="module")
def orc():
    return H.Oracle()


# execution order of the host loop that stands for the grid: ascending, descending, scrambled
@pytest.fixture(scope="module", params=[0, 1, 2], ids=["fwd", "rev", "scrambled"])
def ksrc(tmp_path_factory, request):
    d = str(tmp_path_factory.mktemp("bicg_ksrc"))
    src = os.path.join(d, "bicg_transpose.cpp")
    with open(src, "w") as f:  # + dense::compute_sqrt (dist_vector.cu), one more element-wise file
        f.write(open(os.path.join(ROOT, "ginkgo_b200", "csrc", "bicg_transpose.cu")).read())
        f.write(open(os.path.join(ROOT, "ginkgo_b200", "csrc", "dist_vector.cu")).read())
    so = os.path.join(d, "libbicg_transpose_host.so")
    subprocess.run(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-Wl,-Bsymbolic", "-Wall",
                    "-Wno-unused-function", "-DB200_SHIM_ORDER=%d" % request.param, "-ffp-contract=off",
                    "-I" + os.path.join(ROOT, "tests", "mock", "host_cuda_shim"),
                    "-I" + os.path.join(ROOT, "include"), src, "-o", so], check=True)
    return KernelSourceBackend(ctypes.CDLL(so))


def random_csr(rng, n, m, max_row, vt="f64", it="i32", sort=False):
    """rows of random length with duplicate and (unless sort) unsorted columns, some rows empty"""
    lens = rng.integers(0, max_row + 1, n)
    lens[rng.integers(0, n, max(n // 10, 1))] = 0
    rp = np.concatenate([[0], np.cumsum(lens)]).astype(IT[it])
    ci = rng.integers(0, m, int(rp[-1])).astype(IT[it])
    if sort:
        for r in range(n):
            ci[rp[r]:rp[r + 1]].sort()
    va = rng.standard_normal(int(rp[-1])).astype(VT[vt])
    return rp, ci, va


def transpose(be, rp, ci, va, m, vt, it):
    n = len(rp) - 1
    trp = np.zeros(m + 1, IT[it])
    tci = np.zeros(max(len(va), 1), IT[it])
    tva = np.zeros(max(len(va), 1), VT[vt])
    be("csr_transpose_%s_%s" % (vt, it), n, m, len(va), rp, ci if len(ci) else np.zeros(1, IT[it]),
       va if len(va) else np.zeros(1, VT[vt]), trp, tci, tva)
    return trp, tci[:len(va)], tva[:len(va)]


@pytest.mark.parametrize("vt", ["f64", "f32"])
@pytest.mark.parametrize("n,m,max_row", [(57, 43, 9), (300, 1000, 20), (1, 5, 4), (40, 1, 3)])
def test_oracle_transpose_is_the_reference_transpose(orc, vt, n, m, max_row):
    rng = np.random.default_rng(n * 7 + m)
    rp, ci, va = random_csr(rng, n, m, max_row, vt)
    want = reference.csr_transpose(rp, ci, va, m)
    got = transpose(orc, rp, ci, va, m, vt, "i32")
    for a, b in zip(got, want):
        assert reference.equal(a, b)


@pytest.mark.parametrize("vt", ["f64", "f32"])
@pytest.mark.parametrize("it", ["i32", "i64"])
@pytest.mark.parametrize("n,m,max_row", [
    (57, 43, 9),          # one chunk, one pass
    (900, 300, 12),       # several chunks, two passes
    (500, 70000, 30),     # three passes
    (3000, 255, 5), (3000, 256, 5), (3000, 257, 5),  # digit boundaries
    (1, 5, 4), (40, 1, 3), (6, 6, 0)])
def test_kernel_source_transpose_matches_oracle(orc, ksrc, vt, it, n, m, max_row):
    rng = np.random.default_rng(n + 3 * m)
    rp, ci, va = random_csr(rng, n, m, max_row, vt, it)
    a = transpose(orc, rp, ci, va, m, vt, it)
    b = transpose(ksrc, rp, ci, va, m, vt, it)
    for x, y in zip(a, b):
        assert x.dtype == y.dtype and np.array_equal(x, y)
    # transposing twice gives the matrix with each row stably sorted by column
    trp, tci, tva = b
    back = transpose(ksrc, trp, tci, tva, n, vt, it)
    assert np.array_equal(back[0], rp)
    for r in range(n):
        order = np.argsort(ci[rp[r]:rp[r + 1]], kind="stable")
        assert np.array_equal(back[1][rp[r]:rp[r + 1]], ci[rp[r]:rp[r + 1]][order])
        assert np.array_equal(back[2][rp[r]:rp[r + 1]], va[rp[r]:rp[r + 1]][order])


def _jacobi(ref, rp, ci, va, max_bs, bp=None, transposed=False):
    return ref.jacobi_generate(rp, ci, va, max_bs, bp, transposed=transposed)


def _block_entries(j):
    """the entries of every block (padding between the blocks is not defined)"""
    stride = j["block_offset"] << j["group_power"]
    mask = (1 << j["group_power"]) - 1
    out = []
    for k in range(j["num_blocks"]):
        n = int(j["block_ptrs"][k + 1] - j["block_ptrs"][k])
        ofs = j["group_offset"] * (k >> j["group_power"]) + j["block_offset"] * (k & mask)
        out.append(np.array([[j["blocks"][ofs + r + c * stride] for c in range(n)] for r in range(n)]))
    return out


@pytest.mark.parametrize("vt", ["f64", "f32"])
@pytest.mark.parametrize("max_bs", [3, 8, 32])
def test_jacobi_transpose_is_the_reference_transpose(orc, ksrc, vt, max_bs):
    ref = reference
    rp, ci, va = W.laplace(9, 2, vdtype=VT[vt])
    va = va.copy()
    rng = np.random.default_rng(max_bs)
    va *= rng.uniform(0.5, 1.5, len(va)).astype(VT[vt])  # nonsymmetric blocks
    j = _jacobi(ref, rp, ci, va, max_bs)
    jt = _jacobi(ref, rp, ci, va, max_bs, transposed=True)
    for be in (orc, ksrc):
        out = np.zeros_like(j["blocks"])
        be("jacobi_transpose_%s_i32" % vt, j["num_blocks"], 32, j["block_offset"], j["group_offset"],
           j["group_power"], j["block_ptrs"], j["blocks"], out)
        got = dict(j, blocks=out)
        for a, b, c in zip(_block_entries(got), _block_entries(jt), _block_entries(j)):
            assert np.array_equal(a, b) and np.array_equal(a, c.T)


@pytest.mark.parametrize("vt", ["f64", "f32"])
@pytest.mark.parametrize("precond", [0, 1, 2])
def test_oracle_bicg_is_the_reference_bicg(vt, precond):
    ref = reference
    rp, ci, va = W.laplace(12, 2, vdtype=VT[vt])
    rng = np.random.default_rng(5)
    va = va.copy()
    va[rng.integers(0, len(va), 60)] *= VT[vt](1.3)  # nonsymmetric
    n = len(rp) - 1
    b = rng.uniform(-1, 1, (n, 3)).astype(VT[vt])
    x0 = np.zeros((n, 3), VT[vt])
    max_bs = {0: 0, 1: 1, 2: 8}[precond]
    bp = np.arange(0, n + 1, 8, dtype=np.int32) if precond == 2 else None
    jac = ref.jacobi_generate(rp, ci, va, max_bs, bp) if precond else None
    red = 1e-10 if vt == "f64" else 1e-5
    for iter_first in (1, 0):
        xr, itr, _, _ = ref.solve("bicg", rp, ci, va, b, x0, max_bs, bp, max_iters=150, reduction=red,
                                  iter_first=iter_first)
        xo, ito, _ = H.orc_solve("bicg", vt, rp, ci, va, b, x0, precond, jac, max_iters=150, reduction=red,
                                 iter_first=iter_first)
        assert ito == itr and ito > 5
        assert reference.equal(xo, xr)


@pytest.mark.parametrize("vt", ["f64", "f32"])
@pytest.mark.parametrize("rows,cols", [(597, 43), (2001, 1), (0, 2)])
def test_kernel_source_bicg_steps_match_oracle(orc, ksrc, vt, rows, cols):
    rng = np.random.default_rng(96)
    names = ("b", "r", "z", "p", "q", "r2", "z2", "p2", "q2", "x")
    st = {k: cols + (i % 3) for i, k in enumerate(names)}
    v = {k: H.dense(rng, rows, cols, s, vt) for k, s in st.items()}
    sc = {k: rng.uniform(0.5, 1, cols).astype(VT[vt]) for k in ("rho", "prev_rho", "beta")}
    stop = np.zeros(cols, dtype=np.uint8)
    if cols > 4:
        sc["prev_rho"][2] = 0
        sc["beta"][3] = 0
        stop[1] = 1 | 0x40

    def run(be, name, args):
        args = [a.copy() if isinstance(a, np.ndarray) else a for a in args]
        be(name + "_" + vt, *args)
        return [a for a in args if isinstance(a, np.ndarray)]

    cases = [
        ("bicg_initialize", [rows, cols, v["b"], st["b"], v["r"], st["r"], v["z"], st["z"], v["p"], st["p"],
                             v["q"], st["q"], sc["prev_rho"], sc["rho"], v["r2"], st["r2"], v["z2"], st["z2"],
                             v["p2"], st["p2"], v["q2"], st["q2"], np.full(max(cols, 1), 0x81, np.uint8)]),
        ("bicg_step_1", [rows, cols, v["p"], st["p"], v["z"], st["z"], v["p2"], st["p2"], v["z2"], st["z2"],
                         sc["rho"], sc["prev_rho"], stop]),
        ("bicg_step_2", [rows, cols, v["x"], st["x"], v["r"], st["r"], v["r2"], st["r2"], v["p"], st["p"],
                         v["q"], st["q"], v["q2"], st["q2"], sc["beta"], sc["rho"], stop]),
    ]
    for name, args in cases:
        a, b = run(orc, name, args), run(ksrc, name, args)
        for x, y in zip(a, b):
            assert np.array_equal(x, y, equal_nan=True), name


@pytest.mark.parametrize("vt", ["f64", "f32"])
def test_kernel_source_compute_sqrt_matches_oracle(orc, ksrc, vt):
    rng = np.random.default_rng(2)
    data = H.dense(rng, 3, 17, 19, vt, fill=rng.uniform(0, 1e6, (3, 17)))
    a, b = data.copy(), data.copy()
    orc("dense_compute_sqrt_" + vt, 3, 17, a, 19)
    ksrc("dense_compute_sqrt_" + vt, 3, 17, b, 19)
    assert np.array_equal(a, b) and np.array_equal(a[:, :17], np.sqrt(data[:, :17]))
    assert np.array_equal(a[:, 17:], data[:, 17:])  # padding untouched
