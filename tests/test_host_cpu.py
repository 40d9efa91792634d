"""The C++ HOST layer (ginkgo_b200/host/*.hpp: solver loops, stopping criteria, Jacobi set-up,
format conversions, file I/O, staging) exercised WITHOUT a GPU: capi.cpp is compiled together
with tests/mock (a host-memory stand-in for the C ABI whose entry points forward to the
oracle's restatement of the same reference kernels -- test infrastructure only).  Because the
kernels underneath are the oracle's, every result must be BIT-IDENTICAL to the oracle's own
restatement of the reference host loops (which tests/test_oracle_vs_ref.py pins to the real
reference): any difference is a bug in the C++ host logic."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

import workloads as W
from tests import helpers as H
from tests.helpers import VT

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


from tests.mock_build import CpuExec as _CpuExec  # noqa: E402


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    from ginkgo_b200 import api
    from tests.mock_build import build_mock_host
    lib = build_mock_host(str(tmp_path_factory.mktemp("mock")))
    saved = api._HOST_LIB
    api._HOST_LIB = lib
    yield _CpuExec(lib)
    api._HOST_LIB = saved


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a))


def host_solve(host, kind, vt, rp, ci, va, b, x0, precond_max_bs=0, block_ptrs=None, **kw):
    from ginkgo_b200 import api
    t = [_t(va), _t(ci), _t(rp)]
    tb, tx = _t(b), _t(x0).clone()
    n = len(rp) - 1
    A = api.host_csr(host, (n, n), *t)
    s = api.HostSolver(host, kind, A, precond_max_bs=precond_max_bs, block_ptrs=block_ptrs,
                       fused=False, **kw)
    s.apply(api.host_dense(host, tb), api.host_dense(host, tx))
    return tx.numpy(), s.num_iterations, s.stop_status


@pytest.mark.parametrize("kind", ["cg", "fcg", "cgs", "pipe_cg", "minres", "bicgstab", "gmres", "gcr", "bicg"])
@pytest.mark.parametrize("precond", [0, 1, 2, 3])
@pytest.mark.parametrize("vt", ["f64", "f32"])
def test_host_solver_loops_are_the_oracle_loops(host, kind, precond, vt):
    """precond 3 = block Jacobi with blocks detected by find_blocks (no block pointers)"""
    from tests import reference as ref
    rp, ci, va = W.laplace(20, 2, vdtype=VT[vt])
    n = len(rp) - 1
    rng = np.random.default_rng(5)
    b = rng.uniform(-1, 1, (n, 2)).astype(VT[vt])
    x0 = np.zeros((n, 2), VT[vt])
    red = 1e-9 if vt == "f64" else 1e-4
    max_bs = {0: 0, 1: 1, 2: 8, 3: 4}[precond]
    bp = np.arange(0, n + 1, 8, dtype=np.int32) if precond == 2 else None
    jac = None
    if precond:
        jac = ref.jacobi_generate(rp, ci, va, max_bs, bp)
    for iter_first in (1, 0):
        xo, ito, stop_o = H.orc_solve(kind, vt, rp, ci, va, b, x0, min(precond, 2), jac, max_iters=300,
                                      reduction=red, iter_first=iter_first, krylov_dim=15)
        xh, ith, stop_h = host_solve(host, kind, vt, rp, ci, va, b, x0, max_bs, bp, max_iters=300,
                                     reduction=red, iter_first=bool(iter_first), krylov_dim=15)
        assert ith == ito
        assert stop_h == stop_o[0]
        assert np.array_equal(xh, xo)


@pytest.mark.parametrize("res_kind,baseline", [(1, 0), (1, 1), (1, 2), (2, 0), (2, 1)])
def test_host_criteria(host, res_kind, baseline):
    rp, ci, va = W.laplace(16, 2)
    n = len(rp) - 1
    b = np.ones((n, 1))
    x0 = np.full((n, 1), 0.5)
    kw = dict(max_iters=200, res_kind=res_kind, baseline=baseline, reduction=1e-6 if baseline != 2 else 1e-5,
              iter_first=1, krylov_dim=10)
    xo, ito, stop_o = H.orc_solve("cg", "f64", rp, ci, va, b, x0, 0, None, **kw)
    kw["iter_first"] = True
    xh, ith, stop_h = host_solve(host, "cg", "f64", rp, ci, va, b, x0, **kw)
    assert (ith, stop_h) == (ito, stop_o[0]) and np.array_equal(xh, xo)


@pytest.mark.parametrize("vt", ["f64", "f32"])
@pytest.mark.parametrize("fmt,kw", [("ell", {}), ("sellp", {}), ("sellp", dict(slice_size=32, stride_factor=4)),
                                    ("coo", {}), ("hybrid", {}),
                                    ("hybrid", dict(strategy="column_limit", columns=3)),
                                    ("hybrid", dict(strategy="imbalance_limit", percent=0.5)),
                                    ("hybrid", dict(strategy="minimal_storage_limit"))])
def test_host_convert_then_apply(host, orc, vt, fmt, kw):
    from ginkgo_b200 import api
    rng = np.random.default_rng(41)
    n, m = 700, 600
    rp, ci, va = H.random_csr(rng, n, m, rng.integers(0, 13, n), vt, "i32")
    x = rng.uniform(-1, 1, m).astype(VT[vt])
    A = api.host_csr(host, (n, m), _t(va), _t(ci), _t(rp))
    B = api.host_convert(A, fmt, **kw)
    tx, ty = _t(x), torch.zeros(n, dtype=_t(x).dtype)
    xd, yd = api.host_dense(host, tx), api.host_dense(host, ty)
    api._hcheck(api._host().gkob_apply(B.h, xd.h, yd.h))
    yo = np.zeros(n, VT[vt])
    orc("csr_spmv_%s_i32" % vt, n, m, len(va), rp, ci, va, x, 1, 1, yo, 1)
    assert np.array_equal(ty.numpy(), yo)
    # advanced apply through the converted operator
    al, be = torch.tensor([-1.5], dtype=tx.dtype), torch.tensor([0.25], dtype=tx.dtype)
    y0 = rng.uniform(-1, 1, n).astype(VT[vt])
    ty2 = _t(y0).clone()
    ald, bed, yd2 = api.host_dense(host, al), api.host_dense(host, be), api.host_dense(host, ty2)
    api._hcheck(api._host().gkob_apply4(B.h, ald.h, xd.h, bed.h, yd2.h))  # handles kept alive
    yo2 = y0.copy()
    orc("csr_advanced_spmv_%s_i32" % vt, n, m, len(va), rp, ci, va, np.array([-1.5], VT[vt]), x, 1, 1,
        np.array([0.25], VT[vt]), yo2, 1)
    if fmt in ("ell", "sellp"):
        assert np.array_equal(ty2.numpy(), yo2)
    else:  # coo / hybrid scale y first, then accumulate: one rounding apart at most
        assert H.rel_err(ty2.numpy(), yo2) <= H.R[vt]


def test_host_sort_and_files(host, orc, tmp_path):
    from ginkgo_b200 import api
    rng = np.random.default_rng(42)
    n, m = 300, 250
    lens = rng.integers(0, 9, n)
    lens[7] = 120
    rp, ci, va = H.random_csr(rng, n, m, lens, "f64", "i32")
    ci2, va2 = ci.copy(), va.copy()
    for r in range(n):
        s, e = rp[r], rp[r + 1]
        perm = rng.permutation(e - s)
        ci2[s:e], va2[s:e] = ci[s:e][perm], va[s:e][perm]
    t = [_t(va2), _t(ci2), _t(rp)]
    A = api.host_csr(host, (n, m), *t)
    api.host_sort_by_column_index(A)
    assert np.array_equal(t[1].numpy(), ci) and np.array_equal(t[0].numpy(), va)
    # write / read round trips of the sorted matrix, every layout that keeps the pattern
    x = rng.uniform(-1, 1, m)
    yo = np.zeros(n)
    orc("csr_spmv_f64_i32", n, m, len(va), rp, ci, va, x, 1, 1, yo, 1)
    for layout in ("coordinate", "binary"):
        out = tmp_path / ("m." + layout)
        api.host_write_csr(A, out, layout)
        B = api.host_read_csr(host, out)
        assert B.size == (n, m)
        ty = torch.zeros(n, dtype=torch.float64)
        xd, yd = api.host_dense(host, _t(x)), api.host_dense(host, ty)
        api._hcheck(api._host().gkob_apply(B.h, xd.h, yd.h))
        assert np.array_equal(ty.numpy(), yo)


def test_host_staged_apply(host, orc):
    from ginkgo_b200 import api
    rng = np.random.default_rng(43)
    n, m = 400, 300
    rp, ci, va = H.random_csr(rng, n, m, rng.integers(0, 12, n), "f64", "i32")
    A = api.host_csr(host, (n, m), _t(va), _t(ci), _t(rp))
    st = api.StagedApply(A)
    xs = [_t(rng.uniform(-1, 1, m)) for _ in range(5)]
    ys = [torch.full((n,), float("nan"), dtype=torch.float64) for _ in range(5)]
    for x, y in zip(xs, ys):
        st.apply(x, y)
    st.wait()
    for x, y in zip(xs, ys):
        yo = np.zeros(n)
        orc("csr_spmv_f64_i32", n, m, len(va), rp, ci, va, x.numpy(), 1, 1, yo, 1)
        assert np.array_equal(y.numpy(), yo)


def test_host_errors(host):
    from ginkgo_b200 import api
    rp, ci, va = W.laplace(6, 2)
    n = len(rp) - 1
    A = api.host_csr(host, (n, n), _t(va), _t(ci), _t(rp))
    bad = api.host_dense(host, torch.zeros(n + 1, dtype=torch.float64))
    y = api.host_dense(host, torch.zeros(n, dtype=torch.float64))
    with pytest.raises(api.DimensionMismatch):
        api._hcheck(api._host().gkob_apply(A.h, bad.h, y.h))
    with pytest.raises(Exception):  # block larger than max_block_size
        api.HostSolver(host, "cg", A, precond_max_bs=2, block_ptrs=np.array([0, 5, n], np.int32),
                       max_iters=5, fused=False)


@pytest.mark.parametrize("kind,extra", [("ir", dict(relaxation_factor=1.0)), ("ir", dict(relaxation_factor=0.3)),
                                        ("chebyshev", dict(foci=(0.3, 7.9))),
                                        ("chebyshev", dict(foci=(0.4, 1.7)))])
@pytest.mark.parametrize("precond", [0, 1, 2])
@pytest.mark.parametrize("vt", ["f64", "f32"])
def test_host_ir_and_chebyshev(host, kind, extra, precond, vt):
    """update_residual.hpp semantics (ignore_residual_check) + the Ir / Chebyshev host loops"""
    from tests import reference as ref
    rp, ci, va = W.laplace(14, 2, vdtype=VT[vt])
    n = len(rp) - 1
    rng = np.random.default_rng(11)
    b = rng.uniform(-1, 1, (n, 2)).astype(VT[vt])
    x0 = rng.uniform(-1, 1, (n, 2)).astype(VT[vt])
    if kind == "ir" and precond == 0:
        extra = dict(relaxation_factor=extra["relaxation_factor"] * 0.2)
    max_bs = {0: 0, 1: 1, 2: 8}[precond]
    bp = np.arange(0, n + 1, 8, dtype=np.int32)[: n // 8 + 1] if precond == 2 else None
    if precond == 2 and bp[-1] != n:
        bp = np.append(bp, n).astype(np.int32)
    jac = None
    if precond:
        jac = ref.jacobi_generate(rp, ci, va, max_bs, bp)
    for iter_first in (1, 0):
        for res_kind in (1, 0):
            kw = dict(max_iters=40, reduction=1e-3, res_kind=res_kind, krylov_dim=10, **extra)
            xo, ito, stop_o = H.orc_solve(kind, vt, rp, ci, va, b, x0, precond, jac, iter_first=iter_first, **kw)
            xh, ith, stop_h = host_solve(host, kind, vt, rp, ci, va, b, x0, max_bs, bp,
                                         iter_first=bool(iter_first), **kw)
            assert (ith, stop_h) == (ito, stop_o[0])
            assert np.array_equal(xh, xo, equal_nan=True)


@pytest.mark.parametrize("ortho", [0, 1, 2])
@pytest.mark.parametrize("krylov_dim", [5, 30])
def test_host_gmres_ortho_and_restart(host, ortho, krylov_dim):
    """GMRES orthogonalisation variants (mgs / cgs / cgs2) and restarts through the C++ host loop"""
    rp, ci, va = W.laplace(12, 2)
    n = len(rp) - 1
    rng = np.random.default_rng(4)
    b = rng.uniform(-1, 1, (n, 3))
    x0 = rng.uniform(-1, 1, (n, 3))
    kw = dict(max_iters=80, reduction=1e-10, krylov_dim=krylov_dim, ortho=ortho)
    xo, ito, stop_o = H.orc_solve("gmres", "f64", rp, ci, va, b, x0, 0, None, iter_first=1, **kw)
    xh, ith, stop_h = host_solve(host, "gmres", "f64", rp, ci, va, b, x0, iter_first=True, **kw)
    assert (ith, stop_h) == (ito, stop_o[0]) and np.array_equal(xh, xo)


def test_host_advanced_solver_apply(host):
    """x = alpha * solve(b) + beta * x  (core/solver/cg.cpp:184-200: clone, solve, scale, add_scaled)"""
    from ginkgo_b200 import api
    rp, ci, va = W.laplace(10, 2)
    n = len(rp) - 1
    rng = np.random.default_rng(8)
    b = rng.uniform(-1, 1, (n, 1))
    x0 = rng.uniform(-1, 1, (n, 1))
    A = api.host_csr(host, (n, n), _t(va), _t(ci), _t(rp))
    s = api.HostSolver(host, "cg", A, max_iters=200, reduction=1e-10, fused=False)
    tx = _t(x0).clone()
    al, be = torch.tensor([2.0], dtype=torch.float64), torch.tensor([-0.5], dtype=torch.float64)
    ald, bed, bd, xd = (api.host_dense(host, t) for t in (al, be, _t(b), tx))
    api._hcheck(api._host().gkob_apply4(s.obj.h, ald.h, bd.h, bed.h, xd.h))
    xs, _, _ = host_solve(host, "cg", "f64", rp, ci, va, b, x0, max_iters=200, reduction=1e-10)
    expect = x0 * -0.5
    expect = expect + 2.0 * xs
    assert np.array_equal(tx.numpy(), expect)


# ---------------------------------------------------------------- distributed set-up (8f rank 4)
def _random_mapping(rng, n, num_parts, run):
    out = []
    while len(out) < n:
        out += [int(rng.integers(num_parts))] * int(rng.integers(1, run + 1))
    return np.array(out[:n], np.int32)


def _ref_dist():
    from tests import reference
    return reference


def _assert_equal(a, b):
    from tests import reference
    assert reference.equal(a, b, equal_nan=True)


@pytest.mark.parametrize("seed", range(4))
def test_host_partition_is_the_reference_partition(host, seed):
    from ginkgo_b200 import api
    ref = _ref_dist()
    rng = np.random.default_rng(seed)
    num_parts = int(rng.integers(1, 7))
    mapping = _random_mapping(rng, int(rng.integers(1, 300)), num_parts, 6)
    nr = int(rng.integers(1, 10))
    ranges = np.concatenate([[0], np.cumsum(rng.integers(0 if seed % 2 else 1, 9, nr))])
    ids = rng.permutation(nr).astype(np.int32)
    cases = [(api.HostPartition.from_mapping(host, mapping, num_parts), ref.partition(0, mapping, num_parts=num_parts)),
             (api.HostPartition.from_contiguous(host, ranges), ref.partition(1, None, ranges)),
             (api.HostPartition.from_contiguous(host, ranges, ids), ref.partition(1, ids, ranges)),
             (api.HostPartition.uniform(host, num_parts, 1000 + seed), ref.partition(2, num_parts=num_parts, global_size=1000 + seed)),
             (api.HostPartition.uniform(host, 0, 5), ref.partition(2, num_parts=0, global_size=5))]
    for got, want in cases:
        got = got.info()
        for k in ("size", "num_ranges", "num_parts", "num_empty_parts", "connected", "ordered"):
            assert got[k] == want[k], k
        for k in ("range_bounds", "part_ids", "starting_indices", "part_sizes"):
            _assert_equal(got[k], want[k])
    with pytest.raises(api.DimensionMismatch):
        api.HostPartition.from_contiguous(host, ranges, np.zeros(nr + 2, np.int32))


def _dist_case(rng, square=True):
    num_parts = int(rng.integers(2, 6))
    nrows = int(rng.integers(30, 150))
    ncols = nrows if square else int(rng.integers(30, 150))
    row_map = _random_mapping(rng, nrows, num_parts, 8)
    col_map = row_map if square else _random_mapping(rng, ncols, num_parts, 8)
    nnz = int(rng.integers(50, 1200))
    order = np.unique(rng.integers(0, nrows * ncols, nnz))  # row-major sorted, no duplicates
    return num_parts, (nrows, ncols), row_map, col_map, order // ncols, order % ncols, rng.standard_normal(len(order))


@pytest.mark.parametrize("seed", range(5))
def test_host_assemble_local_is_the_reference_split(host, seed):
    """rows/values = separate_local_nonlocal's kept entries, columns = index_map's combined space"""
    from ginkgo_b200 import api
    ref = _ref_dist()
    rng = np.random.default_rng(40 + seed)
    num_parts, shape, row_map, col_map, rows, cols, vals = _dist_case(rng, square=seed % 2 == 0)
    rp = api.HostPartition.from_mapping(host, row_map, num_parts)
    cp = api.HostPartition.from_mapping(host, col_map, num_parts)
    for rank in range(num_parts):
        a = api.HostAssembly(host, rp, rank, shape, rows, cols, vals, col_part=cp)
        (lr, lc, lv), (nr_, nc, nv) = ref.separate_local_nonlocal(shape, rows, cols, vals, row_map, col_map,
                                                                 num_parts, rank)
        owned = row_map[rows] == rank
        nc_kept = cols[owned & (col_map[cols] != rank)].astype(np.int64)  # the non-local columns, in order
        _assert_equal(nc_kept, nc)
        nc = nc_kept
        im = ref.index_map(col_map, num_parts, rank, nc, 2, cols[owned])
        assert a.n_local_rows == int((row_map == rank).sum()) and a.n_local_cols == int((col_map == rank).sum())
        assert (a.n_ghost,) == im["remote_global"].shape
        _assert_equal(a.remote_global, im["remote_global"])
        _assert_equal(a.remote_local, im["remote_local"])
        want_recv = np.zeros(num_parts, np.int64)
        want_recv[im["target_ids"]] = im["remote_sizes"]
        np.testing.assert_array_equal(a.recv_counts, want_recv)
        _assert_equal(a.col_idxs, im["query_local"])
        np.testing.assert_array_equal(a.values, vals[owned])
        # row pointers = counts of the owned entries per local row
        local_row_of = np.full(shape[0], -1)
        local_row_of[row_map == rank] = np.arange(a.n_local_rows)  # one-range-per-run order == local order
        info = rp.info()
        for r in range(info["num_ranges"]):  # general: starting index + offset in range
            if info["part_ids"][r] == rank:
                b0, b1 = info["range_bounds"][r], info["range_bounds"][r + 1]
                local_row_of[b0:b1] = info["starting_indices"][r] + np.arange(b1 - b0)
        counts = np.bincount(local_row_of[rows[owned]], minlength=a.n_local_rows)
        np.testing.assert_array_equal(a.row_ptrs, np.concatenate([[0], np.cumsum(counts)]))
        for space in (0, 1, 2):
            q = rng.integers(0, shape[1], 30)
            _assert_equal(a.map_to_local(q, space), ref.index_map(col_map, num_parts, rank, nc, space, q)["query_local"])
    with pytest.raises(api.DimensionMismatch):
        api.HostAssembly(host, rp, 0, (shape[0] + 1, shape[1]), rows, cols, vals, col_part=cp)


@pytest.mark.parametrize("seed", range(4))
def test_host_send_layout_closes_the_halo_exchange(host, seed):
    """all ranks' assemblies + compute_send_layout, with the exchange itself played in numpy:
    every ghost slot receives the x entry of its global column and the local SpMVs add up to A x"""
    from ginkgo_b200 import api
    rng = np.random.default_rng(80 + seed)
    num_parts, shape, row_map, _, rows, cols, vals = _dist_case(rng)
    n = shape[0]
    part = api.HostPartition.from_mapping(host, row_map, num_parts)
    info = part.info()
    local_of = np.zeros(n, np.int64)
    for r in range(info["num_ranges"]):
        b0, b1 = info["range_bounds"][r], info["range_bounds"][r + 1]
        local_of[b0:b1] = info["starting_indices"][r] + np.arange(b1 - b0)
    asm = [api.HostAssembly(host, part, q, shape, rows, cols, vals) for q in range(num_parts)]
    S = np.array([a.recv_counts for a in asm])  # S[q][p]
    x = rng.standard_normal(n)
    x_local = []
    for p in range(num_parts):
        xl = np.zeros(asm[p].n_local_rows)
        own = np.nonzero(row_map == p)[0]
        xl[local_of[own]] = x[own]
        x_local.append(xl)
    # what every rank packs for every peer
    packed = {}
    for p in range(num_parts):
        sc, so = api.host_send_layout(num_parts, p, S)
        np.testing.assert_array_equal(sc, S[:, p])
        for q in range(num_parts):
            send_idx = asm[q].remote_local[so[q]:so[q] + sc[q]]  # read_distributed's device copy
            packed[(p, q)] = x_local[p][send_idx]
    y = np.zeros(n)
    for q in range(num_parts):
        ghosts = np.concatenate([packed[(p, q)] for p in range(num_parts)])
        np.testing.assert_array_equal(ghosts, x[asm[q].remote_global])
        x_ext = np.concatenate([x_local[q], ghosts])
        a = asm[q]
        yl = np.zeros(a.n_local_rows)
        np.add.at(yl, np.repeat(np.arange(a.n_local_rows), np.diff(a.row_ptrs)), a.values * x_ext[a.col_idxs])
        own = np.nonzero(row_map == q)[0]
        y[own] = yl[local_of[own]]
    want = np.zeros(n)
    np.add.at(want, rows, vals * x[cols])
    np.testing.assert_allclose(y, want, rtol=1e-12, atol=1e-12)


def test_host_read_distributed_on_one_rank(host):
    """world size 1 through the whole C++ path: communicator, read_distributed, Matrix::apply"""
    from ginkgo_b200 import api
    rng = np.random.default_rng(3)
    n = 200
    order = np.unique(rng.integers(0, n * n, 3000))
    rows, cols, vals = order // n, order % n, rng.standard_normal(len(order))
    part = api.HostPartition.uniform(host, 1, n)
    A = api.DistMatrix.read(host, part, (n, n), rows, cols, vals)
    assert (A.n_local, A.n_local_cols, A.n_ghost) == (n, n, 0)
    x = _t(rng.standard_normal(n))
    y = torch.zeros(n, dtype=torch.float64)
    A.apply(x, y)
    rp = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n))]).astype(np.int32)
    yo = np.zeros((n, 1))
    H.Oracle()("csr_spmv_f64_i32", n, n, len(vals), rp, cols.astype(np.int32), vals,
               x.numpy().reshape(n, 1).copy(), 1, 1, yo, 1)
    assert np.array_equal(y.numpy(), yo[:, 0])


# ------------------------------------------------------------------ transposes and BiCG (8f rank 3)
@pytest.mark.parametrize("vt", ["f64", "f32"])
def test_host_csr_transpose_applies_like_the_reference_transpose(host, vt):
    from ginkgo_b200 import api
    from tests.test_transpose_bicg_cpu import random_csr
    rng = np.random.default_rng(17)
    n, m = 300, 170
    rp, ci, va = random_csr(rng, n, m, 14, vt)
    A = api.host_csr(host, (n, m), _t(va), _t(ci), _t(rp))
    A.vt = vt
    T = api.host_transpose(A)
    h = api._host()
    assert (h.gkob_num_rows(T.h), h.gkob_num_cols(T.h)) == (m, n)
    x = rng.uniform(-1, 1, (n, 2)).astype(VT[vt])
    y = torch.zeros((m, 2), dtype=_t(va).dtype)
    xd, yd = api.host_dense(host, _t(x)), api.host_dense(host, y)  # keep the handles alive
    api._hcheck(h.gkob_apply(T.h, xd.h, yd.h))
    o = H.Oracle()
    trp, tci, tva = np.zeros(m + 1, np.int32), np.zeros(len(va), np.int32), np.zeros(len(va), VT[vt])
    o("csr_transpose_%s_i32" % vt, n, m, len(va), rp, ci, va, trp, tci, tva)
    yo = np.zeros((m, 2), VT[vt])
    o("csr_spmv_%s_i32" % vt, m, n, len(va), trp, tci, tva, x, 2, 2, yo, 2)
    assert np.array_equal(y.numpy(), yo)
    # transposing twice: the same operator again
    TT = api.host_transpose(T)
    y2 = torch.zeros((n, 2), dtype=_t(va).dtype)
    xm = rng.uniform(-1, 1, (m, 2)).astype(VT[vt])
    xmd, y2d = api.host_dense(host, _t(xm)), api.host_dense(host, y2)
    api._hcheck(h.gkob_apply(TT.h, xmd.h, y2d.h))
    # (rows of A are unsorted, A^TT has them sorted: same sums up to the order of addition)
    yo2 = np.zeros((n, 2), VT[vt])
    o("csr_spmv_%s_i32" % vt, n, m, len(va), rp, ci, va, xm, 2, 2, yo2, 2)
    np.testing.assert_allclose(y2.numpy(), yo2, rtol=1e-4 if vt == "f32" else 1e-12, atol=1e-5 if vt == "f32" else 1e-13)


@pytest.mark.parametrize("vt", ["f64", "f32"])
@pytest.mark.parametrize("precond", [0, 1, 2])
def test_host_bicg_with_transposed_preconditioner(host, vt, precond):
    """nonsymmetric values: the blocks of Jacobi::transpose differ from the blocks themselves"""
    from tests import reference as ref
    rp, ci, va = W.laplace(16, 2, vdtype=VT[vt])
    rng = np.random.default_rng(31)
    va = (va * rng.uniform(0.6, 1.4, len(va))).astype(VT[vt])
    n = len(rp) - 1
    b = rng.uniform(-1, 1, (n, 2)).astype(VT[vt])
    x0 = np.zeros((n, 2), VT[vt])
    max_bs = {0: 0, 1: 1, 2: 8}[precond]
    bp = np.arange(0, n + 1, 8, dtype=np.int32) if precond == 2 else None
    jac = None
    if precond:
        jac = ref.jacobi_generate(rp, ci, va, max_bs, bp)
    red = 1e-9 if vt == "f64" else 1e-4
    xo, ito, stop_o = H.orc_solve("bicg", vt, rp, ci, va, b, x0, precond, jac, max_iters=200, reduction=red)
    xh, ith, stop_h = host_solve(host, "bicg", vt, rp, ci, va, b, x0, max_bs, bp, max_iters=200, reduction=red)
    assert ith == ito and ito > 5
    assert stop_h == stop_o[0]
    assert np.array_equal(xh, xo)


@pytest.mark.parametrize("world,seed", [(2, 0), (3, 1), (5, 2)])
def test_host_read_distributed_multi_rank_in_threads(host, world, seed):
    """`world` ranks as threads of this process on the mock's in-process communicator (barriers +
    copies standing for NCCL): communicator::create, Matrix::read_distributed incl. the
    all-gather of counts / remote lists and the send lists cut from them, halo_create and
    Matrix::apply -- every rank's rows must equal the single-matrix SpMV bit for bit"""
    import threading
    from ginkgo_b200 import api
    h = api._host()
    api.DistMatrix._bind(h)
    rng = np.random.default_rng(60 + seed)
    n = int(rng.integers(200, 500))
    nnz = int(rng.integers(2000, 6000))
    order = np.unique(rng.integers(0, n * n, nnz))
    rows, cols, vals = order // n, order % n, rng.standard_normal(len(order))
    if seed == 1:  # one-directional coupling: strictly upper triangular + diagonal
        keep = cols >= rows
        rows, cols, vals = rows[keep], cols[keep], vals[keep]
    row_map = _random_mapping(rng, n, world, 40) if seed else None
    x = rng.standard_normal(n)
    rp = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n))]).astype(np.int32)
    want = np.zeros((n, 1))
    H.Oracle()("csr_spmv_f64_i32", n, n, len(vals), rp, cols.astype(np.int32), vals, x.reshape(n, 1).copy(), 1, 1,
               want, 1)
    idb = (ctypes.c_ubyte * 128)()
    api._hcheck(h.gkob_dist_unique_id(idb))
    results, errors = {}, []

    def run(rank):
        try:
            ex = _CpuExec(h)
            part = (api.HostPartition.from_mapping(ex, row_map, world) if row_map is not None
                    else api.HostPartition.uniform(ex, world, n))
            info = part.info()
            r64, c64 = np.ascontiguousarray(rows, np.int64), np.ascontiguousarray(cols, np.int64)
            d = h.gkob_dist_matrix_read_f64_i32(ex.h, idb, rank, world, part.h, n, n, len(vals), r64.ctypes.data,
                                                c64.ctypes.data, vals.ctypes.data, 0)
            assert d, h.gkob_last_error().decode()
            sz = np.zeros(3, np.int64)
            api._hcheck(h.gkob_dist_matrix_sizes(d, sz.ctypes.data, None))
            n_local, n_local_cols, n_ghost = (int(v) for v in sz)
            ghosts = np.zeros(max(n_ghost, 1), np.int64)
            api._hcheck(h.gkob_dist_matrix_sizes(d, sz.ctypes.data, ghosts.ctypes.data))
            # local numbering of the owned global indices
            owned = np.zeros(n_local, np.int64)
            for r in range(info["num_ranges"]):
                if info["part_ids"][r] == rank:
                    b0, b1 = info["range_bounds"][r], info["range_bounds"][r + 1]
                    owned[info["starting_indices"][r] + np.arange(b1 - b0)] = np.arange(b0, b1)
            x_ext = np.zeros(n_local + n_ghost)
            x_ext[:n_local] = x[owned]
            y = np.zeros(n_local)
            for _ in range(3):  # repeated exchanges
                x_ext[n_local:] = -1
                api._hcheck(h.gkob_dist_spmv_f64(d, x_ext.ctypes.data, y.ctypes.data))
            # distributed::read_distributed_vector of a 2-column global vector (every 3rd row set)
            vr = np.arange(0, n, 3, dtype=np.int64)
            vrows, vcols = np.repeat(vr, 2), np.tile(np.array([0, 1], np.int64), len(vr))
            vvals = (vrows * 10 + vcols).astype(np.float64)
            vout = np.zeros(max(n_local, 1) * 2)
            api._hcheck(h.gkob_dist_vector_read_f64(d, part.h, n, 2, len(vvals), vrows.ctypes.data,
                                                    vcols.ctypes.data, vvals.ctypes.data, vout.ctypes.data))
            want_v = np.zeros((n_local, 2))
            sel = owned % 3 == 0
            want_v[sel, 0], want_v[sel, 1] = owned[sel] * 10, owned[sel] * 10 + 1
            assert np.array_equal(vout[:n_local * 2].reshape(n_local, 2), want_v)
            results[rank] = (owned, y.copy(), x_ext[n_local:].copy(), ghosts[:n_ghost].copy())
            h.gkob_dist_destroy(d)
        except BaseException as e:  # noqa: BLE001
            errors.append((rank, repr(e)))

    threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(120)
    assert not errors, errors
    assert sorted(results) == list(range(world))
    for rank, (owned, y, ghost_vals, ghosts) in results.items():
        assert np.array_equal(ghost_vals, x[ghosts])
        assert np.array_equal(y, want[owned, 0])


DIST_KINDS = ["cg", "fcg", "cgs", "bicgstab", "pipe_cg", "minres", "gmres", "gmres_cgs", "gcr", "ir", "chebyshev"]


@pytest.mark.parametrize("kind", DIST_KINDS)
@pytest.mark.parametrize("precond", [0, 1, 4])
def test_host_distributed_solvers_in_threads(host, kind, precond, schwarz=0):
    """every solver of the host layer on a distributed::Matrix with distributed::Vector operands,
    3 ranks as threads: dots and norms are summed over the ranks, Jacobi comes from the local
    block.  Same iteration count (+-1) and solution as the single-matrix solver."""
    import threading
    from ginkgo_b200 import api
    h = api._host()
    api.DistMatrix._bind(h)
    world = 3
    rp, ci, va = W.laplace(12, 2)
    n = len(rp) - 1
    rng = np.random.default_rng(8)
    b = rng.uniform(-1, 1, n)
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(rp))
    cols = ci.astype(np.int64)
    skind = "gmres" if kind == "gmres_cgs" else kind
    extra = dict(ortho=1) if kind == "gmres_cgs" else {}
    if kind == "ir":  # Richardson on a spectrum in (0.1, 8): relaxation < 2 / 8
        extra = dict(relaxation_factor=0.2)
    if kind == "chebyshev":
        extra = dict(foci=(0.1, 8.0))
    # uniform partition in blocks of 4 rows so that auto-detected 4x4 blocks cannot straddle ranks
    max_bs = precond
    x1, it1, st1 = host_solve(host, skind, "f64", rp, ci, va, b.reshape(n, 1), np.zeros((n, 1)), max_bs, None,
                              max_iters=400, reduction=1e-10, krylov_dim=20, **extra)
    api._host().gkob_solver_params(extra.get("relaxation_factor", 1.0), *extra.get("foci", (0.0, 1.0)))
    idb = (ctypes.c_ubyte * 128)()
    api._hcheck(h.gkob_dist_unique_id(idb))
    out, errors = {}, []
    kinds = {"cg": 0, "bicgstab": 1, "gmres": 2, "fcg": 3, "cgs": 4, "ir": 5, "chebyshev": 6, "pipe_cg": 7,
             "gcr": 8, "minres": 9}

    def run(rank):
        try:
            ex = _CpuExec(h)
            part = api.HostPartition.from_contiguous(ex, [0, 48, 96, n])
            pb = part.info()["range_bounds"]
            q0, q1 = int(pb[rank]), int(pb[rank + 1])
            d = h.gkob_dist_matrix_read_f64_i32(ex.h, idb, rank, world, part.h, n, n, len(va), rows.ctypes.data,
                                                cols.ctypes.data, va.ctypes.data, 1)
            assert d, h.gkob_last_error().decode()
            bl, xl = b[q0:q1].copy(), np.zeros(q1 - q0)
            it, st = ctypes.c_longlong(0), ctypes.c_ubyte(0)
            rc = h.gkob_dist_solve_f64(d, kinds[skind], max_bs, schwarz, bl.ctypes.data, xl.ctypes.data, n, 400, 1,
                                       0, 1e-10, 1, 20, extra.get("ortho", 0), 1, ctypes.byref(it), ctypes.byref(st))
            assert rc == 0, h.gkob_last_error().decode()
            out[rank] = (q0, q1, xl, it.value, st.value)
            h.gkob_dist_destroy(d)
        except BaseException as e:  # noqa: BLE001
            errors.append((rank, repr(e)))

    threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(300)
    api._host().gkob_solver_params(1.0, 0.0, 1.0)
    assert not errors, errors
    x = np.zeros(n)
    for rank, (q0, q1, xl, it, st) in out.items():
        x[q0:q1] = xl
        assert abs(it - it1) <= 1, (it, it1)
        assert st == st1
    assert np.isfinite(x1).all()
    assert np.linalg.norm(x - x1[:, 0]) <= 1e-8 * np.linalg.norm(x1)


def test_host_distributed_solve_python_wrapper(host):
    """DistMatrix.read + DistMatrix.solve (the Python face) at world size 1: bit-identical to the
    plain solver except for norm2 = sqrt(sum of squares) instead of the scaled nrm2 kernel"""
    from ginkgo_b200 import api
    rp, ci, va = W.laplace(10, 2)
    n = len(rp) - 1
    rng = np.random.default_rng(12)
    b = rng.uniform(-1, 1, n)
    x1, it1, st1 = host_solve(host, "cg", "f64", rp, ci, va, b.reshape(n, 1), np.zeros((n, 1)), 1, None,
                              max_iters=300, reduction=1e-10)
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(rp))
    part = api.HostPartition.uniform(host, 1, n)
    A = api.DistMatrix.read(host, part, (n, n), rows, ci.astype(np.int64), va)
    bl, xl = _t(b), torch.zeros(n, dtype=torch.float64)
    it, st = A.solve("cg", bl, xl, n, precond_max_bs=1, max_iters=300, reduction=1e-10)
    assert abs(it - it1) <= 1 and st == st1
    assert np.linalg.norm(xl.numpy() - x1[:, 0]) <= 1e-10 * np.linalg.norm(x1)
    with pytest.raises(api.NotSupported):
        A.solve("bicg", bl, xl, n)  # no transposed distributed apply


@pytest.fixture(scope="module")
def dist_example_exe(tmp_path_factory):
    from tests.mock_build import build_mock_executable
    return build_mock_executable(str(tmp_path_factory.mktemp("dist_example")),
                                 os.path.join(ROOT, "examples", "distributed_solver.cpp"), "distributed_solver")


@pytest.mark.parametrize("solver", ["cg", "gmres", "bicgstab"])
def test_distributed_example_runs_on_the_mock(dist_example_exe, solver):
    """examples/distributed_solver.cpp (the reference's distributed-solver flow) linked against
    the host-memory mock instead of the CUDA library, one rank: read_distributed, distributed
    vectors, solver + Jacobi from the local block, residual check"""
    exe = dist_example_exe
    env = dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0")
    r = subprocess.run([exe, "10", solver], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "converged=1" in r.stdout and "n=1000" in r.stdout


@pytest.mark.parametrize("fmt", ["csr", "ell", "sellp", "coo", "hybrid", "dense"])
def test_host_read_write_every_format(host, orc, tmp_path, fmt):
    """gko::read<Format> = Csr::read + the device conversion; gko::write(Format) walks the format's
    own storage: the file written from any format equals the file written from the Csr"""
    from ginkgo_b200 import api
    rng = np.random.default_rng(44)
    n, m = 200, 170
    lens = rng.integers(0, 9, n)
    lens[5] = 90  # one long row: the hybrid split puts its tail into the COO part
    rp, ci, va = H.random_csr(rng, n, m, lens, "f64", "i32")
    A = api.host_csr(host, (n, m), _t(va), _t(ci), _t(rp))
    src = tmp_path / "a.mtx"
    api.host_write_csr(A, src, "coordinate")
    B = api.host_read(host, src, fmt)
    assert B.size == (n, m)
    x = rng.uniform(-1, 1, m)
    yo = np.zeros(n)
    orc("csr_spmv_f64_i32", n, m, len(va), rp, ci, va, x, 1, 1, yo, 1)
    ty = torch.zeros(n, dtype=torch.float64)
    xd, yd = api.host_dense(host, _t(x)), api.host_dense(host, ty)
    if fmt == "dense":  # Dense::apply (GEMM) is outside the path
        with pytest.raises(api.NotSupported):
            api._hcheck(api._host().gkob_apply(B.h, xd.h, yd.h))
    else:
        api._hcheck(api._host().gkob_apply(B.h, xd.h, yd.h))
        assert H.rel_err(ty.numpy(), yo) <= H.R["f64"]
    for layout in ("coordinate", "binary"):
        ref_file, out = tmp_path / ("ref." + layout), tmp_path / ("out." + layout)
        api.host_write_csr(A, ref_file, layout)
        api.host_write(B, out, layout)
        assert open(out, "rb").read() == open(ref_file, "rb").read()


@pytest.mark.parametrize("kind", ["cg", "gmres", "bicgstab"])
def test_host_schwarz_with_local_jacobi_is_jacobi(host, kind):
    """Schwarz(local solver = scalar Jacobi on the square local block) is the scalar Jacobi of the
    distributed matrix: same iterations and solution as the Jacobi-from-local-block run"""
    # (both run distributed on 3 threads; compared against the single-matrix solver inside)
    test_host_distributed_solvers_in_threads(host, kind, 1, schwarz=-1)


def test_host_schwarz_with_local_richardson_sweeps(host):
    """Schwarz around 3 Jacobi-preconditioned Richardson sweeps on the local block (a fixed
    polynomial, so CG stays valid): converges in fewer iterations than plain Jacobi, same x"""
    import threading
    from ginkgo_b200 import api
    h = api._host()
    api.DistMatrix._bind(h)
    world = 3
    rp, ci, va = W.laplace(12, 2)
    n = len(rp) - 1
    rng = np.random.default_rng(8)
    b = rng.uniform(-1, 1, n)
    rows, cols = np.repeat(np.arange(n, dtype=np.int64), np.diff(rp)), ci.astype(np.int64)
    x1, it1, _ = host_solve(host, "cg", "f64", rp, ci, va, b.reshape(n, 1), np.zeros((n, 1)), 1, None,
                            max_iters=400, reduction=1e-10)
    api._host().gkob_solver_params(0.8, 0.0, 1.0)
    idb = (ctypes.c_ubyte * 128)()
    api._hcheck(h.gkob_dist_unique_id(idb))
    out, errors = {}, []

    def run(rank):
        try:
            ex = _CpuExec(h)
            part = api.HostPartition.from_contiguous(ex, [0, 48, 96, n])
            pb = part.info()["range_bounds"]
            q0, q1 = int(pb[rank]), int(pb[rank + 1])
            d = h.gkob_dist_matrix_read_f64_i32(ex.h, idb, rank, world, part.h, n, n, len(va), rows.ctypes.data,
                                                cols.ctypes.data, va.ctypes.data, 1)
            assert d, h.gkob_last_error().decode()
            bl, xl = b[q0:q1].copy(), np.zeros(q1 - q0)
            it, st = ctypes.c_longlong(0), ctypes.c_ubyte(0)
            rc = h.gkob_dist_solve_f64(d, 0, 1, 3, bl.ctypes.data, xl.ctypes.data, n, 400, 1, 0, 1e-10, 1, 20, 0, 1,
                                       ctypes.byref(it), ctypes.byref(st))
            assert rc == 0, h.gkob_last_error().decode()
            out[rank] = (q0, q1, xl, it.value)
            h.gkob_dist_destroy(d)
        except BaseException as e:  # noqa: BLE001
            errors.append((rank, repr(e)))

    threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(300)
    api._host().gkob_solver_params(1.0, 0.0, 1.0)
    assert not errors, errors
    x = np.zeros(n)
    for rank, (q0, q1, xl, it) in out.items():
        x[q0:q1] = xl
        assert 3 < it < it1, (it, it1)
    assert np.linalg.norm(x - x1[:, 0]) <= 1e-8 * np.linalg.norm(x1)


def test_host_schwarz_needs_the_local_block(host):
    from ginkgo_b200 import api
    rp, ci, va = W.laplace(6, 2)
    n = len(rp) - 1
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(rp))
    part = api.HostPartition.uniform(host, 1, n)
    A = api.DistMatrix.read(host, part, (n, n), rows, ci.astype(np.int64), va)  # keep_local_block=False
    b, x = _t(np.ones(n)), torch.zeros(n, dtype=torch.float64)
    with pytest.raises(api.NotSupported):
        A.solve("cg", b, x, n, precond_max_bs=1, schwarz=-1)
    A2 = api.DistMatrix.read(host, part, (n, n), rows, ci.astype(np.int64), va, keep_local_block=True)
    it, st = A2.solve("cg", b, x, n, precond_max_bs=1, max_iters=100, reduction=1e-10, schwarz=-1)
    assert 0 < it < 100


@pytest.mark.parametrize("guess", ["zero", "rhs", "provided"])
@pytest.mark.parametrize("precond", [0, 1])
def test_host_ir_default_initial_guess(host, guess, precond):
    """Ir::with_default_initial_guess: reference == oracle == C++ host loop, bit for bit; x arrives
    filled with garbage, which only `provided` may look at"""
    from tests import reference as ref
    rp, ci, va = W.laplace(10, 2)
    n = len(rp) - 1
    rng = np.random.default_rng(3)
    b = rng.uniform(-1, 1, (n, 2))
    x0 = rng.uniform(-1, 1, (n, 2))
    jac = None
    if precond:
        jac = ref.jacobi_generate(rp, ci, va, 1, None)
    kw = dict(max_iters=40, reduction=1e-12, relaxation_factor=0.2 if not precond else 0.9, initial_guess=guess)
    xo, ito, so = H.orc_solve("ir", "f64", rp, ci, va, b, x0, precond, jac, **kw)
    xh, ith, sh = host_solve(host, "ir", "f64", rp, ci, va, b, x0, precond, None, **kw)
    assert ith == ito and sh == so[0] and np.array_equal(xh, xo)
    xr, itr, _, _ = ref.solve("ir", rp, ci, va, b, x0, precond, None, max_iters=40, reduction=1e-12,
                              relaxation_factor=kw["relaxation_factor"], initial_guess=guess)
    assert itr == ito and ref.equal(xo, xr)
    if guess == "zero":  # the same as a provided zero guess
        xz, itz, _ = H.orc_solve("ir", "f64", rp, ci, va, b, np.zeros_like(x0), precond, jac,
                                 **dict(kw, initial_guess="provided"))
        assert itz == ito and np.array_equal(xz, xo)


# ------------------------------------------------------------ fused CG and the distributed fused CG
@pytest.mark.parametrize("vt", ["f64", "f32"])
@pytest.mark.parametrize("precond", [0, 1])
@pytest.mark.parametrize("res_kind,baseline,iter_first", [(1, 0, True), (2, 1, False), (1, 2, True)])
def test_host_fused_cg_path_on_the_mock(host, vt, precond, res_kind, baseline, iter_first):
    """solver::Cg::try_fused (graph of check_every iterations, control block polling) with the
    mock's sequential restatement of the fused kernels and its recorded graphs: same iteration
    count as the kernel-by-kernel loop (+-1), same solution"""
    from ginkgo_b200 import api
    rp, ci, va = W.laplace(14, 2, vdtype=VT[vt])
    n = len(rp) - 1
    rng = np.random.default_rng(4)
    b = rng.uniform(-1, 1, n).astype(VT[vt])
    red = 1e-9 if vt == "f64" else 1e-4
    if baseline == 2:
        red *= 10  # absolute threshold
    x1, it1, st1 = host_solve(host, "cg", vt, rp, ci, va, b.reshape(n, 1), np.zeros((n, 1), VT[vt]), precond, None,
                              max_iters=300, reduction=red, res_kind=res_kind, baseline=baseline,
                              iter_first=iter_first)
    t = [_t(va), _t(ci), _t(rp)]
    tb, tx = _t(b), torch.zeros(n, dtype=_t(va).dtype)
    A = api.host_csr(host, (n, n), *t)
    s = api.HostSolver(host, "cg", A, precond_max_bs=precond, max_iters=300, reduction=red, res_kind=res_kind,
                       baseline=baseline, iter_first=iter_first, fused=True, check_every=7)
    bd, xd = api.host_dense(host, tb), api.host_dense(host, tx)
    s.apply(bd, xd)
    assert s.used_fused
    assert abs(s.num_iterations - it1) <= 1 and s.stop_status == st1
    tol = 1e-10 if vt == "f64" else 1e-4
    assert np.linalg.norm(tx.numpy() - x1[:, 0]) <= tol * 10 * np.linalg.norm(x1)
    # a second apply replays the captured graph with a new right-hand side
    tb2 = _t(rng.uniform(-1, 1, n).astype(VT[vt]))
    tx.zero_()
    bd2 = api.host_dense(host, tb2)
    s.apply(bd2, xd)
    x2, it2, _ = host_solve(host, "cg", vt, rp, ci, va, tb2.numpy().reshape(n, 1), np.zeros((n, 1), VT[vt]), precond,
                            None, max_iters=300, reduction=red, res_kind=res_kind, baseline=baseline,
                            iter_first=iter_first)
    assert abs(s.num_iterations - it2) <= 1
    assert np.linalg.norm(tx.numpy() - x2[:, 0]) <= tol * 10 * np.linalg.norm(x2)


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("scalar_jacobi", [False, True])
def test_host_distributed_fused_cg_in_threads(host, world, scalar_jacobi):
    """distributed::Cg (the fused iteration with the halo exchange and the two all-reduces inside
    the graph) on the torch-free set-up path, ranks as threads"""
    import threading
    from ginkgo_b200 import api
    h = api._host()
    api.DistMatrix._bind(h)
    rp, ci, va = W.laplace(12, 2)
    n = len(rp) - 1
    rng = np.random.default_rng(21)
    b = rng.uniform(-1, 1, n)
    rows, cols = np.repeat(np.arange(n, dtype=np.int64), np.diff(rp)), ci.astype(np.int64)
    x1, it1, st1 = host_solve(host, "cg", "f64", rp, ci, va, b.reshape(n, 1), np.zeros((n, 1)),
                              1 if scalar_jacobi else 0, None, max_iters=300, reduction=1e-10)
    idb = (ctypes.c_ubyte * 128)()
    api._hcheck(h.gkob_dist_unique_id(idb))
    out, errors = {}, []

    def run(rank):
        try:
            ex = _CpuExec(h)
            part = api.HostPartition.uniform(ex, world, n)
            pb = part.info()["range_bounds"]
            q0, q1 = int(pb[rank]), int(pb[rank + 1])
            d = h.gkob_dist_matrix_read_f64_i32(ex.h, idb, rank, world, part.h, n, n, len(va), rows.ctypes.data,
                                                cols.ctypes.data, va.ctypes.data, 0)
            assert d, h.gkob_last_error().decode()
            api._hcheck(h.gkob_dist_cg_create_f64(d, int(scalar_jacobi), 300, 1, 0, 1e-10, 1, 5))
            bl, xl = b[q0:q1].copy(), np.zeros(q1 - q0)
            it, st = ctypes.c_longlong(0), ctypes.c_ubyte(0)
            for _ in range(2):  # the second apply replays the captured graph
                xl[:] = 0
                api._hcheck(h.gkob_dist_cg_apply_f64(d, bl.ctypes.data, xl.ctypes.data, ctypes.byref(it),
                                                     ctypes.byref(st)))
            out[rank] = (q0, q1, xl, it.value, st.value)
            h.gkob_dist_destroy(d)
        except BaseException as e:  # noqa: BLE001
            errors.append((rank, repr(e)))

    threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(300)
    assert not errors, errors
    x = np.zeros(n)
    for rank, (q0, q1, xl, it, st) in out.items():
        x[q0:q1] = xl
        assert abs(it - it1) <= 1 and st == st1, (it, it1, st, st1)
    assert np.linalg.norm(x - x1[:, 0]) <= 1e-8 * np.linalg.norm(x1)


def test_cpp_user_idioms_on_the_mock(tmp_path):
    """tests/cpp/host_api_check.cpp: gko::initialize<Format> / share / clone and the reference's
    3 x 3 stencil solves (x = [1, 3, 2]) written like the reference's own tests, linked against
    the mock"""
    from tests.mock_build import build_mock_executable
    exe = build_mock_executable(str(tmp_path), os.path.join(ROOT, "tests", "cpp", "host_api_check.cpp"),
                                "host_api_check")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "ALL OK" in r.stdout, r.stdout + r.stderr


MALFORMED_FILES = {
    "empty": b"",
    "header_only": b"%%MatrixMarket matrix coordinate real general\n",
    "truncated": b"%%MatrixMarket matrix coordinate real general\n3 3 4\n1 1 1.0\n2 2",
    "bad_index": b"%%MatrixMarket matrix coordinate real general\n2 2 1\n3 1 1.0\n",
    "zero_index": b"%%MatrixMarket matrix coordinate real general\n2 2 1\n0 1 1.0\n",
    "negative_size": b"%%MatrixMarket matrix coordinate real general\n-2 2 1\n1 1 1.0\n",
    "garbage": b"\x00\x01\x02 not a matrix",
    "bad_banner": b"%%MatrixMarket matrix coordinate quaternion general\n1 1 1\n1 1 1.0\n",
    "binary_truncated": b"GINKGODI" + b"\x03\x00\x00\x00\x00\x00\x00\x00",
    "huge_nnz": b"%%MatrixMarket matrix coordinate real general\n2 2 99999999999\n1 1 1.0\n",
}


@pytest.mark.parametrize("name", sorted(MALFORMED_FILES))
def test_host_readers_reject_malformed_files(host, tmp_path, name):
    """every malformed file ends in an exception of the host layer (never a crash, never a matrix)"""
    from ginkgo_b200 import _lib, api
    p = tmp_path / "m.mtx"
    p.write_bytes(MALFORMED_FILES[name])
    for fmt in ("csr", "ell"):
        with pytest.raises(_lib.B200Error):
            api.host_read(host, p, fmt)


@pytest.mark.parametrize("kind", ["cg", "gmres", "bicgstab"])
def test_host_distributed_multiple_right_hand_sides(host, kind):
    """distributed apply and solve with 3 right-hand sides (column by column through the halo),
    3 ranks as threads, against the single-matrix multi-rhs solver"""
    import threading
    from ginkgo_b200 import api
    h = api._host()
    api.DistMatrix._bind(h)
    world, k = 3, 3
    rp, ci, va = W.laplace(12, 2)
    n = len(rp) - 1
    rng = np.random.default_rng(15)
    b = rng.uniform(-1, 1, (n, k))
    rows, cols = np.repeat(np.arange(n, dtype=np.int64), np.diff(rp)), ci.astype(np.int64)
    x1, it1, st1 = host_solve(host, kind, "f64", rp, ci, va, b, np.zeros((n, k)), 1, None, max_iters=400,
                              reduction=1e-10, krylov_dim=20)
    y1 = np.zeros((n, k))
    H.Oracle()("csr_spmv_f64_i32", n, n, len(va), rp, ci, va, b.copy(), k, k, y1, k)
    idb = (ctypes.c_ubyte * 128)()
    api._hcheck(h.gkob_dist_unique_id(idb))
    out, errors = {}, []
    kinds = {"cg": 0, "bicgstab": 1, "gmres": 2}

    def run(rank):
        try:
            ex = _CpuExec(h)
            part = api.HostPartition.uniform(ex, world, n)
            pb = part.info()["range_bounds"]
            q0, q1 = int(pb[rank]), int(pb[rank + 1])
            d = h.gkob_dist_matrix_read_f64_i32(ex.h, idb, rank, world, part.h, n, n, len(va), rows.ctypes.data,
                                                cols.ctypes.data, va.ctypes.data, 0)
            assert d, h.gkob_last_error().decode()
            bl = np.ascontiguousarray(b[q0:q1])
            yl, xl = np.zeros((q1 - q0, k)), np.zeros((q1 - q0, k))
            api._hcheck(h.gkob_dist_apply_f64(d, bl.ctypes.data, yl.ctypes.data, k))
            it, st = ctypes.c_longlong(0), ctypes.c_ubyte(0)
            rc = h.gkob_dist_solve_f64(d, kinds[kind], 1, 0, bl.ctypes.data, xl.ctypes.data, n, 400, 1, 0, 1e-10, 1,
                                       20, 0, k, ctypes.byref(it), ctypes.byref(st))
            assert rc == 0, h.gkob_last_error().decode()
            out[rank] = (q0, q1, yl, xl, it.value)
            h.gkob_dist_destroy(d)
        except BaseException as e:  # noqa: BLE001
            errors.append((rank, repr(e)))

    threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(300)
    assert not errors, errors
    x = np.zeros((n, k))
    for rank, (q0, q1, yl, xl, it) in out.items():
        assert np.array_equal(yl, y1[q0:q1])  # the SpMV rows are bit-identical
        x[q0:q1] = xl
        assert abs(it - it1) <= 1
    assert np.linalg.norm(x - x1) <= 1e-8 * np.linalg.norm(x1)
