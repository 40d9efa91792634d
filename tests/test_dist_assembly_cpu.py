"""Distributed set-up (SURVEY.md 8f rank 4) without a GPU:
  * the oracle restatement (oracle/oracle_dist.h) against the literals of the reference's own
    tests (reference/test/distributed/{partition,matrix,index_map}_kernels.cpp) and against the
    REAL reference kernels through oracle/_ref (random inputs);
  * a copy of ginkgo_b200/csrc/dist_assembly.cu compiled for the host (tests/mock/host_cuda_shim:
    lambdas become host lambdas, the device scan becomes a loop) against the oracle, bit for bit.
The same call sequences run against the CUDA library in tests/test_zz_late_gpu.py."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from tests import dist_driver as D
from tests import helpers as H
from tests import reference
from tests.test_kernel_sources_cpu import KernelSourceBackend

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def orc():
    return H.Oracle()


# execution order of the host loop that stands for the grid: ascending, descending, scrambled
@pytest.fixture(scope="module", params=[0, 1, 2], ids=["fwd", "rev", "scrambled"])
def ksrc(tmp_path_factory, request):
    d = str(tmp_path_factory.mktemp("dist_ksrc"))
    src = os.path.join(d, "dist_assembly.cpp")
    with open(src, "w") as f:
        f.write(open(os.path.join(ROOT, "ginkgo_b200", "csrc", "dist_assembly.cu")).read())
    so = os.path.join(d, "libdist_assembly_host.so")
    # -Bsymbolic: the copy's own template instantiations, not the same-named ones of the CUDA
    # library another test may have loaded into the process
    subprocess.run(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-Wl,-Bsymbolic", "-Wall",
                    "-Wno-unused-function", "-DB200_SHIM_ORDER=%d" % request.param,
                    "-I" + os.path.join(ROOT, "tests", "mock", "host_cuda_shim"),
                    "-I" + os.path.join(ROOT, "include"), src, "-o", so], check=True)
    return KernelSourceBackend(ctypes.CDLL(so))


@pytest.fixture(params=["oracle", "kernel-source"])
def be(request, orc, ksrc):
    return orc if request.param == "oracle" else ksrc


TYPES = [("i32", "i32"), ("i32", "i64"), ("i64", "i64")]


def eq(a, b):
    if isinstance(b, reference.Digest):  # a recorded answer of the reference
        assert reference.equal(a, b, equal_nan=True)
    else:
        np.testing.assert_array_equal(np.asarray(a), np.asarray(b))


# --------------------------------------------------------------------------------- partition
# literals: reference/test/distributed/partition_kernels.cpp:56-268
@pytest.mark.parametrize("lt,gt", TYPES)
def test_partition_builds_from_mapping(be, lt, gt):
    p = D.partition_from_mapping(be, [2, 2, 0, 1, 1, 2, 0, 0, 1, 0, 1, 1, 1, 2, 2, 0], 3, lt, gt)
    assert (p.size, p.num_ranges, p.num_parts, p.num_empty_parts) == (16, 10, 3, 0)
    eq(p.range_bounds, [0, 2, 3, 5, 6, 8, 9, 10, 13, 15, 16])
    eq(p.part_ids, [2, 0, 1, 2, 0, 1, 0, 1, 2, 0])
    eq(p.starting_indices, [0, 0, 0, 2, 1, 2, 3, 3, 3, 4])
    eq(p.part_sizes, [5, 6, 5])
    assert not p.ordered


def test_partition_builds_from_mapping_with_empty_parts(be):
    p = D.partition_from_mapping(be, [3, 3, 0, 1, 1, 3, 0, 0, 1, 0, 1, 1, 1, 3, 3, 0], 5)
    assert (p.num_ranges, p.num_parts, p.num_empty_parts) == (10, 5, 2)
    eq(p.part_ids, [3, 0, 1, 3, 0, 1, 0, 1, 3, 0])
    eq(p.starting_indices, [0, 0, 0, 2, 1, 2, 3, 3, 3, 4])
    eq(p.part_sizes, [5, 6, 0, 5, 0])


@pytest.mark.parametrize("lt,gt", TYPES)
def test_partition_builds_from_ranges(be, lt, gt):
    p = D.partition_from_contiguous(be, [0, 5, 5, 7, 9, 10], None, lt, gt)
    assert (p.size, p.num_ranges, p.num_parts, p.num_empty_parts) == (10, 5, 5, 1)
    eq(p.range_bounds, [0, 5, 5, 7, 9, 10])
    eq(p.part_ids, [0, 1, 2, 3, 4])
    eq(p.starting_indices, [0, 0, 0, 0, 0])
    eq(p.part_sizes, [5, 0, 2, 2, 1])
    p = D.partition_from_contiguous(be, [0, 5, 5, 7, 9, 10], [0, 4, 3, 1, 2], lt, gt)
    eq(p.part_ids, [0, 4, 3, 1, 2])
    eq(p.part_sizes, [5, 2, 1, 2, 0])
    assert p.num_empty_parts == 1 and not p.ordered


def test_partition_builds_from_single_element_range(be):
    p = D.partition_from_contiguous(be, [0])
    assert (p.size, p.num_ranges, p.num_parts, p.num_empty_parts) == (0, 0, 0, 0)
    eq(p.range_bounds, [0])


@pytest.mark.parametrize("num_parts,size,bounds,sizes,empty", [
    (5, 13, [0, 3, 6, 9, 11, 13], [3, 3, 3, 2, 2], 0),
    (5, 0, [0, 0, 0, 0, 0, 0], [0, 0, 0, 0, 0], 5),
    (5, 3, [0, 1, 2, 3, 3, 3], [1, 1, 1, 0, 0], 2),
])
def test_partition_builds_from_global_size(be, num_parts, size, bounds, sizes, empty):
    p = D.partition_uniform(be, num_parts, size)
    assert (p.size, p.num_ranges, p.num_parts, p.num_empty_parts) == (size, num_parts, num_parts, empty)
    eq(p.range_bounds, bounds)
    eq(p.part_ids, np.arange(num_parts))
    eq(p.starting_indices, np.zeros(num_parts))
    eq(p.part_sizes, sizes)
    assert p.ordered


def test_partition_zero_parts(be):
    p = D.partition_uniform(be, 0, 3)
    assert (p.size, p.num_ranges, p.num_parts, p.num_empty_parts) == (0, 0, 0, 0)


@pytest.mark.parametrize("mapping,num_parts,ordered", [
    ([0, 1, 1, 2, 2], 3, True), ([0, 2, 2, 5, 5], 6, True), ([1, 1, 0, 0, 2], 3, False),
    ([0, 1, 2, 0, 1], 3, False)])
def test_partition_is_ordered(be, mapping, num_parts, ordered):
    assert D.partition_from_mapping(be, mapping, num_parts).ordered == ordered


# -------------------------------------------------------------------- separate_local_nonlocal
# literals: reference/test/distributed/matrix_kernels.cpp:182-470 (per part: local (rows, cols,
# vals), non-local (rows, GLOBAL cols, vals))
SEPARATE_CASES = {
    "small": ([1, 0], None, 2, [0, 0, 1, 1], [0, 1, 0, 1], [1, 2, 3, 4],
              [([0], [0], [4]), ([0], [0], [1])], [([0], [0], [3]), ([0], [1], [2])]),
    "no_non_local": ([1, 2, 0, 0, 2, 1], None, 3, [0, 0, 1, 1, 2, 3, 4, 5], [0, 5, 1, 4, 3, 2, 4, 0],
                     [1, 2, 3, 4, 5, 6, 7, 8],
                     [([0, 1], [1, 0], [5, 6]), ([0, 0, 1], [0, 1, 0], [1, 2, 8]), ([0, 0, 1], [0, 1, 1], [3, 4, 7])],
                     [([], [], []), ([], [], []), ([], [], [])]),
    "no_local": ([1, 2, 0, 0, 2, 1], None, 3, [0, 0, 1, 3, 4, 5], [1, 3, 5, 1, 3, 2], [1, 2, 5, 6, 7, 8],
                 [([], [], []), ([], [], []), ([], [], [])],
                 [([1], [1], [6]), ([0, 0, 1], [1, 3, 2], [1, 2, 8]), ([0, 1], [5, 3], [5, 7])]),
    "mixed": ([1, 2, 0, 0, 2, 1], None, 3, [0, 0, 0, 0, 1, 1, 1, 2, 3, 3, 4, 4, 5, 5],
              [0, 1, 3, 5, 1, 4, 5, 3, 1, 2, 3, 4, 0, 2], [11, 1, 2, 12, 13, 14, 5, 15, 6, 16, 7, 17, 18, 8],
              [([0, 1], [1, 0], [15, 16]), ([0, 0, 1], [0, 1, 0], [11, 12, 18]), ([0, 0, 1], [0, 1, 1], [13, 14, 17])],
              [([1], [1], [6]), ([0, 0, 1], [1, 3, 2], [1, 2, 8]), ([0, 1], [5, 3], [5, 7])]),
    "small_col_partition": ([1, 0], [0, 1], 2, [0, 0, 1, 1], [0, 1, 0, 1], [1, 2, 3, 4],
                            [([0], [0], [3]), ([0], [0], [2])], [([0], [1], [4]), ([0], [0], [1])]),
    "no_local_col_partition": ([1, 2, 0, 0, 2, 1], [0, 0, 2, 2, 1, 1], 3, [2, 3, 2, 0, 5, 1, 1],
                               [2, 3, 5, 0, 1, 1, 4], [1, 2, 3, 4, 5, 6, 7],
                               [([], [], []), ([], [], []), ([], [], [])],
                               [([0, 1, 0], [2, 3, 5], [1, 2, 3]), ([0, 1], [0, 1], [4, 5]), ([0, 0], [1, 4], [6, 7])]),
    "mixed_col_partition": ([1, 2, 0, 0, 2, 1], [0, 0, 2, 2, 1, 1], 3,
                            [2, 3, 3, 0, 5, 1, 4, 2, 3, 2, 0, 0, 1, 1, 4, 4],
                            [0, 0, 1, 5, 4, 2, 2, 3, 2, 4, 1, 2, 4, 5, 0, 5],
                            [11, 12, 13, 14, 15, 16, 17, 1, 2, 3, 4, 5, 6, 7, 8, 9],
                            [([0, 1, 1], [0, 0, 1], [11, 12, 13]), ([0, 1], [1, 0], [14, 15]), ([0, 1], [0, 0], [16, 17])],
                            [([0, 1, 0], [3, 2, 4], [1, 2, 3]), ([0, 0], [1, 2], [4, 5]),
                             ([0, 0, 1, 1], [4, 5, 0, 5], [6, 7, 8, 9])]),
}


@pytest.mark.parametrize("name", sorted(SEPARATE_CASES))
@pytest.mark.parametrize("lt,gt", TYPES)
def test_separate_local_nonlocal_reference_literals(be, name, lt, gt):
    row_map, col_map, num_parts, rows, cols, vals, locals_, non_locals = SEPARATE_CASES[name]
    rp = D.partition_from_mapping(be, row_map, num_parts, lt, gt)
    cp = rp if col_map is None else D.partition_from_mapping(be, col_map, num_parts, lt, gt)
    for part in range(num_parts):
        s = D.separate(be, rp, cp, rows, cols, vals, part)
        for got, want in zip(s["local"], locals_[part]):
            eq(got, want)
        for got, want in zip(s["non_local"], non_locals[part]):
            eq(got, want)


def test_separate_empty_input(be):
    rp = D.partition_from_mapping(be, [1, 0, 2, 2, 0, 1, 1, 2], 3)
    for part in range(3):
        s = D.separate(be, rp, rp, [], [], [], part)
        assert all(len(a) == 0 for a in s["local"] + s["non_local"] + s["kept"])


# ---------------------------------------------------------------------------------- index map
# literals: reference/test/distributed/index_map_kernels.cpp:43-200
def test_index_map_build_mapping_literals(be):
    part = D.partition_from_mapping(be, [0, 0, 1, 1, 2, 2], 3)
    im = D.IndexMap(be, part, 0, [2, 3, 3, 5, 5])
    eq(im.remote_global, [2, 3, 5])
    eq(im.remote_local, [0, 1, 1])
    ids, sizes = im.target_ids()
    eq(ids, [1, 2])
    eq(sizes, [2, 1])
    im = D.IndexMap(be, part, 0, [])
    assert im.num_remote == 0 and len(im.target_ids()[0]) == 0


@pytest.mark.parametrize("space,query,want", [
    (1, [1, 1, 4, 0, 4], [1, 1, 2, 0, 2]), (1, [1, 1, 4, 3, 0, 4], [1, 1, 2, -1, 0, 2]),
    (0, [2, 3, 3, 2], [0, 1, 1, 0]), (0, [2, 4, 5, 3, 3, 2], [0, -1, -1, 1, 1, 0]),
    (2, [0, 1, 2, 3, 0, 4, 3], [2, 3, 0, 1, 2, 4, 1]), (2, [0, 1, 2, 3, 0, 4, 5, 3], [2, 3, 0, 1, 2, 4, -1, 1])])
def test_index_map_map_to_local_literals(be, space, query, want):
    part = D.partition_from_mapping(be, [0, 0, 1, 1, 2, 2], 3)
    im = D.IndexMap(be, part, 1, [0, 1, 4])
    eq(im.remote_global, [0, 1, 4])
    eq(im.map_to_local(be, query, space), want)


# ----------------------------------------------------------- random inputs, the real reference
def random_mapping(rng, n, num_parts, run):
    """owners in runs of random length (so ranges have several rows and parts several ranges)"""
    out = []
    while len(out) < n:
        out += [int(rng.integers(num_parts))] * int(rng.integers(1, run + 1))
    return np.array(out[:n], np.int32)


@pytest.mark.parametrize("seed", range(6))
def test_partition_matches_reference(be, seed):
    ref = reference
    rng = np.random.default_rng(seed)
    num_parts = int(rng.integers(1, 9))
    mapping = random_mapping(rng, int(rng.integers(1, 400)), num_parts, 7)
    got = D.partition_from_mapping(be, mapping, num_parts).as_dict()
    want = ref.partition(0, mapping, num_parts=num_parts)
    for k in ("size", "num_ranges", "num_parts", "num_empty_parts", "ordered"):
        assert got[k] == want[k], k
    for k in ("range_bounds", "part_ids", "starting_indices", "part_sizes"):
        eq(got[k], want[k])
    # contiguous with shuffled owners, uniform
    nr = int(rng.integers(1, 12))
    ranges = np.concatenate([[0], np.cumsum(rng.integers(0, 9, nr))])
    ids = rng.permutation(nr).astype(np.int32)
    got = D.partition_from_contiguous(be, ranges, ids).as_dict()
    want = ref.partition(1, ids, ranges)
    for k in ("range_bounds", "part_ids", "starting_indices", "part_sizes"):
        eq(got[k], want[k])
    assert got["num_empty_parts"] == want["num_empty_parts"] and got["ordered"] == want["ordered"]
    gs = int(rng.integers(0, 1000))
    got = D.partition_uniform(be, num_parts, gs).as_dict()
    want = ref.partition(2, num_parts=num_parts, global_size=gs)
    for k in ("range_bounds", "part_ids", "starting_indices", "part_sizes"):
        eq(got[k], want[k])


@pytest.mark.parametrize("seed", range(6))
def test_separate_and_index_map_match_reference(be, seed):
    ref = reference
    rng = np.random.default_rng(100 + seed)
    num_parts = int(rng.integers(2, 7))
    nrows, ncols = int(rng.integers(20, 200)), int(rng.integers(20, 200))
    row_map = random_mapping(rng, nrows, num_parts, 9)
    col_map = random_mapping(rng, ncols, num_parts, 9)
    nnz = int(rng.integers(1, 1500))
    order = np.sort(rng.integers(0, nrows * ncols, nnz))  # row-major, duplicates allowed
    rows, cols = order // ncols, order % ncols
    vals = rng.standard_normal(nnz)
    rp = D.partition_from_mapping(be, row_map, num_parts)
    cp = D.partition_from_mapping(be, col_map, num_parts)
    for part in range(num_parts):
        s = D.separate(be, rp, cp, rows, cols, vals, part)
        loc, nonloc = ref.separate_local_nonlocal((nrows, ncols), rows, cols, vals, row_map, col_map,
                                                  num_parts, part)
        for got, want in zip(s["local"], loc):
            eq(got, want)
        for got, want in zip(s["non_local"], nonloc):
            eq(got, want)
        nonloc_cols = np.asarray(s["non_local"][1], np.int64)  # = the reference's, checked above
        # kept = all entries of the owned rows in input order
        owned = row_map[rows] == part
        eq(s["kept"][1], cols[owned])
        eq(s["kept"][2], vals[owned])
        # the index map of the non-local columns
        im = D.IndexMap(be, cp, part, nonloc_cols)
        q = rng.integers(0, ncols, 50)
        for space in (0, 1, 2):
            r = ref.index_map(col_map, num_parts, part, nonloc_cols, space, q)
            eq(im.remote_global, r["remote_global"])
            eq(im.remote_local, r["remote_local"])
            ids, sizes = im.target_ids()
            eq(ids, r["target_ids"])
            eq(sizes, r["remote_sizes"])
            eq(im.map_to_local(be, q, space), r["query_local"])
        # marking ALL kept columns while skipping the owned ones gives the same map, and the
        # combined index space turns the kept columns into local column indices
        im2 = D.IndexMap(be, cp, part, s["kept"][1], skip_part=part)
        eq(im2.remote_global, im.remote_global)
        comb = im2.map_to_local(be, s["kept"][1], 2)
        assert (comb >= 0).all()
        n_local = int(cp.part_sizes[part])
        is_remote = comb >= n_local
        eq(im2.remote_global[comb[is_remote] - n_local], s["kept"][1][is_remote])
        eq(comb[~is_remote], s["local"][1])


# ------------------------------------------------ the kernel source against the oracle, larger
@pytest.mark.parametrize("lt,gt", TYPES)
@pytest.mark.parametrize("vt", ["f64", "f32"])
def test_kernel_source_matches_oracle(orc, ksrc, lt, gt, vt):
    rng = np.random.default_rng(7)
    num_parts, n = 5, 5000
    row_map = random_mapping(rng, n, num_parts, 200)
    nnz = 40000
    order = np.sort(rng.choice(n * n, nnz, replace=False))
    rows, cols = order // n, order % n
    vals = rng.standard_normal(nnz).astype(D.NP[vt])
    res = []
    for be in (orc, ksrc):
        rp = D.partition_from_mapping(be, row_map, num_parts, lt, gt)
        s = D.separate(be, rp, rp, rows, cols, vals, 2, vt)
        im = D.IndexMap(be, rp, 2, s["kept"][1], skip_part=2)
        comb = im.map_to_local(be, s["kept"][1], 2)
        res.append((rp.as_dict(), s, im, comb))
    (p0, s0, i0, c0), (p1, s1, i1, c1) = res
    for k in p0:
        eq(p0[k], p1[k])
    for k in ("local", "non_local", "kept"):
        for a, b in zip(s0[k], s1[k]):
            assert a.dtype == b.dtype
            eq(a, b)
    for k in ("cls", "local_rank", "non_local_rank"):
        eq(s0[k], s1[k])
    for k in ("bitmap", "word_rank", "range_offsets", "remote_sizes", "remote_global", "remote_local",
              "remote_part_ids"):
        eq(getattr(i0, k), getattr(i1, k))
    eq(c0, c1)


@pytest.mark.parametrize("lt,gt", TYPES)
@pytest.mark.parametrize("seed", range(3))
def test_vector_build_local_matches_reference(be, lt, gt, seed):
    """distributed_vector::build_local (unique (row, column) pairs)"""
    rng = np.random.default_rng(200 + seed)
    num_parts, nrows, ncols = int(rng.integers(1, 6)), int(rng.integers(5, 120)), int(rng.integers(1, 5))
    mapping = random_mapping(rng, nrows, num_parts, 6)
    order = np.unique(rng.integers(0, nrows * ncols, int(rng.integers(1, 300))))
    rows, cols, vals = order // ncols, order % ncols, rng.standard_normal(len(order))
    part = D.partition_from_mapping(be, mapping, num_parts, lt, gt)
    for p in range(num_parts):
        got = D.vector_build_local(be, part, rows, cols, vals, ncols, p)
        want = np.zeros((int((mapping == p).sum()), ncols))
        own = np.nonzero(mapping == p)[0]
        local_of = {g: i for i, g in enumerate(own)}  # mapping-built partition: local order = global order
        for r, c, v in zip(rows, cols, vals):
            if mapping[r] == p:
                want[local_of[r], c] = v
        eq(got, want)
        if (lt, gt) == ("i32", "i64"):
            eq(got, reference.vector_build_local((nrows, ncols), rows, cols, vals, mapping, num_parts, p))


def test_kernel_sources_are_race_free_under_real_threads(tmp_path):
    """ThreadSanitizer on host-compiled copies of dist_assembly.cu and bicg_transpose.cu (+
    dist_vector.cu) whose launches run on 4 real threads: no conflicting accesses inside a launch"""
    import sys
    tsan = subprocess.run(["g++", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(tsan) or not os.path.exists(tsan):
        pytest.skip("libtsan not available")
    libs = []
    for name, files in (("da", ["dist_assembly.cu"]), ("bt", ["bicg_transpose.cu", "dist_vector.cu"])):
        src = str(tmp_path / (name + ".cpp"))
        with open(src, "w") as f:
            for cu in files:
                f.write(open(os.path.join(ROOT, "ginkgo_b200", "csrc", cu)).read())
        so = str(tmp_path / ("lib%s_tsan.so" % name))
        subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-fsanitize=thread",
                        "-DB200_SHIM_THREADS=4", "-ffp-contract=off", "-Wl,-Bsymbolic",
                        "-I" + os.path.join(ROOT, "tests", "mock", "host_cuda_shim"),
                        "-I" + os.path.join(ROOT, "include"), src, "-o", so, "-lpthread"], check=True)
        libs.append(so)
    env = dict(os.environ, LD_PRELOAD=tsan, TSAN_OPTIONS="halt_on_error=0 report_signal_unsafe=0")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "tsan_runner.py")] + libs, env=env,
                       capture_output=True, text=True, timeout=900)
    if "FATAL: ThreadSanitizer" in r.stderr and "TSAN_RUNNER_DONE" not in r.stdout:
        pytest.skip("ThreadSanitizer cannot start in this environment: " + r.stderr[-200:])
    assert "TSAN_RUNNER_DONE" in r.stdout, r.stdout[-500:] + r.stderr[-2000:]
    assert "WARNING: ThreadSanitizer" not in r.stderr, r.stderr[-4000:]
