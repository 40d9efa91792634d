"""Pins the oracle (oracle/liboracle.so, our C restatement) against the REAL reference:
oracle/_ref is the reference's own core + ReferenceExecutor + OmpExecutor sources compiled
in place (oracle/ref_build/Makefile) and driven through its public API (oracle/ref_shim.cpp).
Where oracle/_ref is not built, the reference's recorded answers stand in (tests/reference.py)."""
import ctypes

import numpy as np
import pytest

from tests import helpers as H
from tests import reference as ref
from tests.helpers import VT
from oracle import oracle  # noqa: E402

import workloads as W  # noqa: E402


@pytest.mark.parametrize("vt", ["f64", "f32"])
@pytest.mark.parametrize("fmt", ["csr", "ell", "sellp", "coo", "hybrid"])
def test_spmv_bit_identical_to_reference(orc, vt, fmt):
    rng = np.random.default_rng(21)
    n, m = 1500, 1300
    rp, ci, va = H.random_csr(rng, n, m, rng.integers(0, 40, n), vt, "i32")
    for nrhs in (1, 3):
        x = rng.uniform(-1, 1, (m, nrhs)).astype(VT[vt])
        y_ref, _ = ref.spmv(fmt, rp, ci, va, x, m)
        y = np.zeros((n, nrhs), VT[vt])
        orc("csr_spmv_%s_i32" % vt, n, m, len(va), rp, ci, va, x, nrhs, nrhs, y, nrhs)
        assert ref.equal(y, y_ref)
        y0 = rng.uniform(-1, 1, (n, nrhs)).astype(VT[vt])
        y_ref, _ = ref.spmv(fmt, rp, ci, va, x, m, alpha=-1.5, beta=0.5, y=y0.copy())
        y = y0.copy()
        orc("csr_advanced_spmv_%s_i32" % vt, n, m, len(va), rp, ci, va, np.array([-1.5], VT[vt]), x,
            nrhs, nrhs, np.array([0.5], VT[vt]), y, nrhs)
        if fmt in ("csr", "ell", "sellp"):
            assert ref.equal(y, y_ref)
        else:  # coo/hybrid scale y first, then accumulate: same values up to one rounding
            assert ref.close(y, y_ref, H.R[vt])


def test_omp_executor_matches_reference_executor():
    rp, ci, va = W.build("cfg1")
    x = W.vector(len(rp) - 1)
    y0, _ = ref.spmv("csr", rp, ci, va, x, len(rp) - 1, exec_kind=0)
    y1, _ = ref.spmv("csr", rp, ci, va, x, len(rp) - 1, exec_kind=1)
    assert ref.equal(y0, y1)


from tests.helpers import orc_solve  # noqa: E402


@pytest.mark.parametrize("kind", ["cg", "bicgstab", "gmres", "fcg", "cgs", "pipe_cg", "gcr", "minres"])
@pytest.mark.parametrize("precond", [0, 1, 2])
@pytest.mark.parametrize("vt", ["f64", "f32"])
def test_solver_loops_bit_identical_to_reference(kind, precond, vt):
    rp, ci, va = W.laplace(24, 2, vdtype=VT[vt])
    n = len(rp) - 1
    b = np.ones((n, 1), VT[vt])
    x0 = np.zeros((n, 1), VT[vt])
    red = 1e-8 if vt == "f64" else 1e-4
    bp = np.arange(0, n + 1, 8, dtype=np.int32) if precond == 2 else None
    max_bs = {0: 0, 1: 1, 2: 8}[precond]
    jac = ref.jacobi_generate(rp, ci, va, max_bs, bp) if precond else None
    for iter_first in (1, 0):
        xr, itr, _, _ = ref.solve(kind, rp, ci, va, b, x0, precond_max_bs=max_bs, block_ptrs=bp,
                                  max_iters=300, reduction=red, iter_first=iter_first, krylov_dim=12)
        xo, ito, stop = orc_solve(kind, vt, rp, ci, va, b, x0, precond, jac, max_iters=300,
                                  reduction=red, iter_first=iter_first, krylov_dim=12)
        assert itr == ito
        assert ref.equal(xo, xr)
        assert stop[0] == (0x80 | 0x40 | (2 if iter_first else 1))


@pytest.mark.parametrize("ortho", [0, 1, 2])
def test_gmres_ortho_and_multi_rhs(ortho):
    rng = np.random.default_rng(4)
    rp, ci, va = W.laplace(12, 2)
    n = len(rp) - 1
    b = rng.uniform(-1, 1, (n, 3))
    x0 = np.zeros((n, 3))
    xr, itr, _, _ = ref.solve("gmres", rp, ci, va, b, x0, max_iters=60, reduction=1e-6,
                              krylov_dim=7, ortho=ortho)
    xo, ito, _ = orc_solve("gmres", "f64", rp, ci, va, b, x0, max_iters=60, reduction=1e-6,
                           krylov_dim=7, ortho=ortho)
    assert itr == ito and ref.equal(xo, xr)


@pytest.mark.parametrize("kind", ["cg", "bicgstab"])
def test_implicit_residual_and_baselines(kind):
    rng = np.random.default_rng(5)
    rp, ci, va = W.laplace(16, 2)
    n = len(rp) - 1
    b = rng.uniform(-1, 1, (n, 2))
    x0 = rng.uniform(-1, 1, (n, 2))
    for res_kind, baseline in [(2, 0), (1, 1), (1, 2), (2, 1)]:
        xr, itr, _, _ = ref.solve(kind, rp, ci, va, b, x0, max_iters=200, res_kind=res_kind,
                                  baseline=baseline, reduction=1e-7)
        xo, ito, _ = orc_solve(kind, "f64", rp, ci, va, b, x0, max_iters=200, res_kind=res_kind,
                               baseline=baseline, reduction=1e-7)
        assert itr == ito and ref.equal(xo, xr), (res_kind, baseline)


def test_cfg1_cg_jacobi_matches_survey_probe():
    """SURVEY.md probe: 5-pt Laplacian 316^2, CG + scalar Jacobi, tol 1e-8 -> 579 iterations"""
    rp, ci, va = W.build("cfg1")
    n = len(rp) - 1
    b, x0 = np.ones((n, 1)), np.zeros((n, 1))
    jac = ref.jacobi_generate(rp, ci, va, 1)
    xo, ito, _ = orc_solve("cg", "f64", rp, ci, va, b, x0, 1, jac, max_iters=5000, reduction=1e-8)
    assert ito == 579
    xr, itr, _, _ = ref.solve("cg", rp, ci, va, b, x0, precond_max_bs=1, max_iters=5000,
                              reduction=1e-8, exec_kind=1)
    assert itr == 579
    assert ref.close(xo, xr, 1e-12)


# ---------------------------------------------------------------- conversions (SURVEY 8f-1)
def _conv_matrix(rng, vt, kind):
    n, m = 777, 650
    if kind == "empty_rows":
        lens = rng.integers(0, 3, n) * rng.integers(0, 2, n)
    elif kind == "skewed":
        lens = rng.integers(0, 12, n)
        lens[rng.integers(0, n, 5)] = rng.integers(100, 300, 5)
    else:
        lens = rng.integers(0, 40, n)
    return (n, m) + H.random_csr(rng, n, m, lens, vt, "i32")


@pytest.mark.parametrize("kind", ["uniform", "skewed", "empty_rows"])
@pytest.mark.parametrize("vt", ["f64", "f32"])
def test_convert_to_ell_matches_reference(orc, vt, kind):
    n, m, rp, ci, va = _conv_matrix(np.random.default_rng(5), vt, kind)
    r = ref.convert("ell", rp, ci, va, m)
    mx = H.OutI64()
    orc("ell_compute_max_row_nnz_i32", rp, n, mx)
    assert mx.value == r["width"] and r["stride"] == n
    cols = np.full(r["width"] * n, 77, np.int32)
    vals = np.full(r["width"] * n, 7, VT[vt])
    orc("csr_convert_to_ell_%s_i32" % vt, n, rp, ci, va, r["width"], n, cols, vals)
    assert ref.equal(cols, r["cols"]) and ref.equal(vals, r["vals"])


@pytest.mark.parametrize("kind", ["uniform", "skewed", "empty_rows"])
@pytest.mark.parametrize("slice_size,stride_factor", [(64, 1), (32, 4), (8, 3)])
def test_convert_to_sellp_matches_reference(orc, kind, slice_size, stride_factor):
    vt = "f64"
    n, m, rp, ci, va = _conv_matrix(np.random.default_rng(6), vt, kind)
    r = ref.convert("sellp", rp, ci, va, m, slice_size=slice_size, stride_factor=stride_factor)
    ns = (n + slice_size - 1) // slice_size
    ss, sl = np.zeros(ns + 1, np.uint64), np.zeros(ns, np.uint64)
    orc("sellp_compute_slice_sets_i32", rp, n, slice_size, stride_factor, ss, sl)
    assert ref.equal(ss, r["slice_sets"]) and ref.equal(sl, r["slice_lengths"])
    tot = int(ss[-1]) * slice_size
    assert (tot,) == r["cols"].shape
    # slots of rows past num_rows in the last slice are never written (the reference's answers
    # hold 0 there): compare only what it defines
    cols, vals = np.full(tot, 77, np.int32), np.full(tot, 7, VT[vt])
    orc("csr_convert_to_sellp_%s_i32" % vt, n, slice_size, ss, sl, rp, ci, va, cols, vals)
    defined = ref.sellp_defined(n, slice_size, ss, sl)
    assert ref.equal(np.where(defined, cols, 0), r["cols"])
    assert ref.equal(np.where(defined, vals, 0), r["vals"])
    assert np.all(cols[~defined] == 77)


@pytest.mark.parametrize("kind", ["uniform", "skewed", "empty_rows"])
@pytest.mark.parametrize("strategy", [(0, 0, 0, 0), (1, 3, 0, 0), (2, 0, 0.8, 0), (3, 0, 0.5, 0.01), (4, 0, 0, 0)])
def test_convert_to_hybrid_matches_reference(orc, kind, strategy):
    vt = "f64"
    n, m, rp, ci, va = _conv_matrix(np.random.default_rng(7), vt, kind)
    sk, columns, percent, ratio = strategy
    r = ref.convert("hybrid", rp, ci, va, m, strategy=sk, columns=columns, percent=percent, ratio=ratio)
    ell_lim = H.hybrid_ell_lim(orc, rp, n, m, sk, columns, percent, ratio, vbytes=8, ibytes=4)
    assert ell_lim == r["ell_lim"] and r["ell_stride"] == n
    crp = np.zeros(n + 1, np.int64)
    orc("csr_compute_hybrid_coo_row_ptrs_i32", rp, n, ell_lim, crp)
    assert crp[-1] == r["coo_nnz"]
    ec, ev = np.full(ell_lim * n, 77, np.int32), np.full(ell_lim * n, 7, VT[vt])
    cn = int(crp[-1])
    cr, cc, cv = np.zeros(cn, np.int32), np.zeros(cn, np.int32), np.zeros(cn, VT[vt])
    orc("csr_convert_to_hybrid_%s_i32" % vt, n, rp, ci, va, ell_lim, n, ec, ev, crp, cr, cc, cv)
    for a, b in ((ec, r["cols"]), (ev, r["vals"]), (cr, r["coo_rows"]), (cc, r["coo_cols"]),
                 (cv, r["coo_vals"])):
        assert ref.equal(a, b)


@pytest.mark.parametrize("vt", ["f64", "f32"])
def test_sort_by_column_index_matches_reference(orc, vt):
    rng = np.random.default_rng(8)
    n, m, rp, ci, va = _conv_matrix(rng, vt, "skewed")
    ci2, va2 = ci.copy(), va.copy()
    for r_ in range(n):  # shuffle inside the rows (columns stay distinct)
        s, e = rp[r_], rp[r_ + 1]
        perm = rng.permutation(e - s)
        ci2[s:e], va2[s:e] = ci[s:e][perm], va[s:e][perm]
    r = ref.convert("sort", rp, ci2, va2, m)
    orc("csr_sort_by_column_index_%s_i32" % vt, n, rp, ci2, va2)
    assert ref.equal(ci2, r["cols"]) and ref.equal(va2, r["vals"])
    assert np.array_equal(ci2, ci) and np.array_equal(va2, va)


# ------------------------------------------------------- block-Jacobi generate (8f-2)
def _jacobi_case(rng, vt, max_bs, singular=False):
    n = 600
    sizes = []
    while sum(sizes) < n:
        sizes.append(int(rng.integers(1, max_bs + 1)))
    sizes[-1] -= sum(sizes) - n
    if sizes[-1] == 0:
        sizes.pop()
    bp = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    lens = rng.integers(3, 40, n)
    rp, ci, va = H.random_csr(rng, n, n, lens, vt, "i32")
    if singular:  # wipe the rows of one block inside the block -> zero pivot
        b0, b1 = int(bp[3]), int(bp[4])
        for r in range(b0, b1):
            s, e = rp[r], rp[r + 1]
            va[s:e][(ci[s:e] >= b0) & (ci[s:e] < b1)] = 0
    return n, rp, ci, va, bp


@pytest.mark.parametrize("vt", ["f64", "f32"])
@pytest.mark.parametrize("max_bs", [2, 7, 16, 32])
def test_jacobi_generate_bit_identical_to_reference(orc, vt, max_bs):
    rng = np.random.default_rng(50 + max_bs)
    n, rp, ci, va, bp = _jacobi_case(rng, vt, max_bs)
    r = ref.jacobi_generate(rp, ci, va, max_bs, bp)
    assert np.array_equal(r["block_ptrs"], bp)
    blocks = np.zeros_like(r["blocks"])
    orc("jacobi_generate_%s_i32" % vt, n, rp, ci, va, len(bp) - 1, max_bs, r["block_offset"],
        r["group_offset"], r["group_power"], bp, blocks)
    # compare what the reference defines: the bs x bs part of every slot
    stride = r["block_offset"] << r["group_power"]
    for k in range(len(bp) - 1):
        bs = int(bp[k + 1] - bp[k])
        off = r["group_offset"] * (k >> r["group_power"]) + r["block_offset"] * (
            k & ((1 << r["group_power"]) - 1))
        idx = off + (np.arange(bs)[:, None] + np.arange(bs)[None, :] * stride)
        assert np.array_equal(blocks[idx], r["blocks"][idx]), k


def _blocky_matrix(rng, n, max_run, vt="f64"):
    """rows come in runs sharing one column pattern (natural blocks), run lengths 1..max_run"""
    rows_cols = []
    r = 0
    while r < n:
        run = int(rng.integers(1, max_run + 1))
        k = int(rng.integers(1, 9))
        cols = np.sort(rng.choice(n, size=k, replace=False))
        for _ in range(min(run, n - r)):
            rows_cols.append(cols)
            r += 1
    rp = np.zeros(n + 1, np.int32)
    rp[1:] = np.cumsum([len(c) for c in rows_cols])
    ci = np.concatenate(rows_cols).astype(np.int32)
    va = rng.uniform(-1, 1, len(ci)).astype(VT[vt])
    # make the diagonal blocks invertible enough: not needed for find_blocks itself
    return rp, ci, va


@pytest.mark.parametrize("max_bs", [1, 2, 5, 16, 32])
@pytest.mark.parametrize("max_run", [1, 3, 40])
def test_find_blocks_matches_reference(orc, max_bs, max_run):
    rng = np.random.default_rng(70 + max_bs + max_run)
    n = 3000
    rp, ci, va = _blocky_matrix(rng, n, max_run)
    # put a strong diagonal so the reference's generate does not hit singular blocks
    r = ref.jacobi_generate(rp, ci, va, max_bs, None)
    bp = np.full(n + 1, -1, np.int32)
    nb = H.OutI64()
    orc("jacobi_find_blocks_i32", n, rp, ci, max_bs, bp, nb)
    if max_bs == 1:
        assert nb.value == n and np.array_equal(bp[:n + 1], np.arange(n + 1))
    else:
        assert nb.value == r["num_blocks"]
        assert np.array_equal(bp[:nb.value + 1], r["block_ptrs"])


@pytest.mark.parametrize("kind,extra", [("ir", dict(relaxation_factor=1.0)), ("ir", dict(relaxation_factor=0.2)),
                                        ("chebyshev", dict(foci=(0.3, 7.9))),
                                        ("chebyshev", dict(foci=(1.0, 1.0)))])
@pytest.mark.parametrize("precond", [0, 1, 2])
@pytest.mark.parametrize("vt", ["f64", "f32"])
def test_ir_and_chebyshev_loops_bit_identical_to_reference(kind, extra, precond, vt):
    """core/solver/ir.cpp, chebyshev.cpp with update_residual.hpp (residual check ignored in the
    first criterion pass of every iteration > 0)"""
    rp, ci, va = W.laplace(16, 2, vdtype=VT[vt])
    n = len(rp) - 1
    rng = np.random.default_rng(9)
    b = rng.uniform(-1, 1, (n, 2)).astype(VT[vt])
    x0 = rng.uniform(-1, 1, (n, 2)).astype(VT[vt])
    if kind == "ir" and precond == 0:
        extra = dict(relaxation_factor=extra["relaxation_factor"] * 0.2)  # keep plain Richardson stable
    bp = np.arange(0, n + 1, 8, dtype=np.int32) if precond == 2 else None
    max_bs = {0: 0, 1: 1, 2: 8}[precond]
    jac = ref.jacobi_generate(rp, ci, va, max_bs, bp) if precond else None
    red = 1e-3
    for iter_first in (1, 0):
        xr, itr, _, _ = ref.solve(kind, rp, ci, va, b, x0, precond_max_bs=max_bs, block_ptrs=bp,
                                  max_iters=60, reduction=red, iter_first=iter_first, **extra)
        xo, ito, stop = orc_solve(kind, vt, rp, ci, va, b, x0, precond, jac, max_iters=60,
                                  reduction=red, iter_first=iter_first, **extra)
        assert itr == ito
        assert ref.equal(xo, xr, equal_nan=True)  # a diverging run must diverge alike
