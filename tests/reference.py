"""The real reference's answers for the tests, with or without the reference at hand.

Where oracle/_ref is built (the reference's own CPU executors, compiled from its sources by
oracle/ref_build/Makefile), every call goes to it, as oracle/ref.py.  Everywhere else the answers
come from tests/golden/reference_calls.json.gz, recorded from the same calls of the same tests:

* arrays of up to SMALL entries, and whatever read_mtx returns (tests index with it), are stored as
  they are;
* larger arrays are stored as a 64-bit digest of their values (`Digest`), which `equal` / `close`
  compare with what the test computed; spmv and solver results also keep a few sampled values so that
  comparisons up to a rounding still have numbers to look at;
* jacobi_generate's blocks feed other computations, so they are recomputed by the oracle
  (oracle/liboracle.so) and accepted only when their digest is the reference's.

Padding that the reference leaves undefined (between Jacobi blocks, past the last row of a SELL-P
slice) is zeroed in every answer, recorded or live, so that digests do not depend on it.

To record after changing or adding a test that asks the reference, on a machine where oracle/_ref is
built:  B200_RECORD_REFERENCE=1 python -m pytest tests -m "not gpu"  and, for the GPU tests' calls,
B200_RECORD_REFERENCE=1 B200_TEST_SELFCHECK=1 python -m pytest tests -m gpu -k "solver_matches_oracle or
detected_blocks".  Answers are added to the file; answers of calls no test makes any more stay until
the file is deleted and recorded anew."""
import atexit
import base64
import gzip
import hashlib
import inspect
import json
import os

import numpy as np

from oracle import ref as _live

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_calls.json.gz")
SMALL = 16
SAMPLES = 16
_SAMPLED = ("spmv", "solve")
_WHOLE = ("read_mtx",)
_RECORD = os.environ.get("B200_RECORD_REFERENCE") == "1"
_answers = None
_new = {}


def live():
    return _live.available()


# ------------------------------------------------------------------------------ digests
def _canonical(a):
    """values as float64 with -0.0 -> 0.0 and one NaN: equal digests <=> np.array_equal(equal_nan=True)"""
    c = np.array(a, dtype=np.float64) + 0.0
    c[np.isnan(c)] = np.nan
    return c


def _digest(a):
    c = _canonical(a)
    return hashlib.sha256(repr(c.shape).encode() + c.tobytes()).hexdigest()[:16]


def _sample_positions(size):
    return np.random.default_rng(size).choice(size, min(size, SAMPLES), replace=False)


class Digest:
    """a large answer of the reference: its shape, the digest of its values and, for some answers,
    values at positions drawn by _sample_positions"""

    def __init__(self, shape, sha, sample=None):
        self.shape, self.sha, self.sample = tuple(shape), sha, sample

    def matches(self, a, equal_nan=False):
        a = np.asarray(a)
        if not equal_nan and a.dtype.kind in "fc" and np.isnan(a).any():
            return False
        return a.shape == self.shape and _digest(a) == self.sha


def equal(a, b, equal_nan=False):
    """np.array_equal where either side may be a recorded Digest"""
    if isinstance(a, Digest) and isinstance(b, Digest):
        return a.shape == b.shape and a.sha == b.sha
    if isinstance(a, Digest):
        a, b = b, a
    if isinstance(b, Digest):
        return b.matches(a, equal_nan)
    return np.array_equal(a, b, equal_nan=equal_nan)


def close(a, b, tol):
    """tests.helpers.rel_err(a, b) <= tol; against a Digest: equal, or within tol at its sampled positions"""
    from tests.helpers import rel_err
    if not isinstance(b, Digest):
        return rel_err(a, b) <= tol
    if b.matches(a):
        return True
    a = np.asarray(a).reshape(-1)
    return a.size == int(np.prod(b.shape)) and rel_err(a[_sample_positions(a.size)], b.sample) <= tol


# ------------------------------------------------------------------------- (de)serialising
def _encode(o, sampled, whole):
    if isinstance(o, np.ndarray):
        if o.size <= SMALL or whole:
            return {"a": o.dtype.str, "s": list(o.shape), "b": base64.b64encode(o.tobytes()).decode()}
        d = {"s": list(o.shape), "h": _digest(o)}
        if sampled and o.dtype.kind == "f":
            d["v"] = [float(v) for v in o.reshape(-1)[_sample_positions(o.size)]]
        return d
    if isinstance(o, dict):
        return {"m": {k: _encode(v, sampled, whole) for k, v in o.items()}}
    if isinstance(o, (tuple, list)):
        return {"t": [_encode(v, sampled, whole) for v in o]}
    if isinstance(o, bytes):  # a written file
        return {"f": base64.b64encode(o).decode()}
    if isinstance(o, (np.integer, np.floating, np.bool_)):
        return o.item()
    return o


def _decode(o):
    if not isinstance(o, dict):
        return o
    if "a" in o:
        return np.frombuffer(base64.b64decode(o["b"]), np.dtype(o["a"])).reshape(o["s"]).copy()
    if "h" in o:
        return Digest(o["s"], o["h"], np.array(o["v"]) if "v" in o else None)
    if "f" in o:
        return base64.b64decode(o["f"])
    if "m" in o:
        return {k: _decode(v) for k, v in o["m"].items()}
    return tuple(_decode(v) for v in o["t"])


def _key(name, fn, args, kwargs):
    bound = inspect.signature(fn).bind(*args, **kwargs)
    bound.apply_defaults()
    h = hashlib.sha256(name.encode())
    for k, v in bound.arguments.items():
        if k == "path":  # files are named by their contents
            v = open(v, "rb").read() if name == "read_mtx" else None
        h.update(k.encode())
        if isinstance(v, np.ndarray):
            v = np.ascontiguousarray(v)
            h.update(("%s%r" % (v.dtype.str, v.shape)).encode() + v.tobytes())
        elif isinstance(v, bytes):
            h.update(v)
        else:
            h.update(repr(v).encode())
    return h.hexdigest()[:20]


def _load():
    global _answers
    if _answers is None:
        _answers = json.load(gzip.open(GOLDEN, "rt")) if os.path.exists(GOLDEN) else {}
    return _answers


def _save():
    if _new:
        answers = dict(_load(), **_new)
        with gzip.GzipFile(GOLDEN, "wb", mtime=0) as f:
            f.write(json.dumps(answers, sort_keys=True, separators=(",", ":")).encode())


if _RECORD:
    atexit.register(_save)


def _recorded(name, key):
    answers = _load()
    if key not in answers:
        raise LookupError("no recorded answer of the reference for this %s call: record it where oracle/_ref "
                          "is built (tests/reference.py)" % name)
    return _decode(answers[key])


# ------------------------------------------------------------- undefined padding -> 0
def _jacobi_defined(r, value_bytes=None, precisions=None, n_values=None):
    """mask of the block storage the reference defines: the bs x bs entries of every block (in bytes of
    the stored precision when precisions are given, tests/jacobi_cases.written_mask)"""
    from tests import jacobi_cases as JC
    ptrs, bo, go, gp = r["block_ptrs"], r["block_offset"], r["group_offset"], r["group_power"]
    if value_bytes is not None:
        space = JC.scheme(bo, len(ptrs) - 1)[3]
        return JC.written_mask(ptrs, precisions, value_bytes == 8, bo, go, gp, space, value_bytes)
    mask = np.zeros(n_values, bool)
    stride = bo << gp
    for k in range(len(ptrs) - 1):
        bs = int(ptrs[k + 1] - ptrs[k])
        off = go * (k >> gp) + bo * (k & ((1 << gp) - 1))
        mask[off + (np.arange(bs)[:, None] + np.arange(bs)[None, :] * stride)] = True
    return mask


def _canon_jacobi_generate(r, max_bs):
    if max_bs > 1:
        r["blocks"] = np.where(_jacobi_defined(r, n_values=len(r["blocks"])), r["blocks"], 0).astype(r["blocks"].dtype)
    return r


def _canon_jacobi_adaptive(r, va):
    """blocks as the bytes generate writes (mask of tests/jacobi_cases.written_mask), the rest 0"""
    mask = _jacobi_defined(r, va.dtype.itemsize, r["precisions"])
    raw = r["blocks"].view(np.uint8)[:len(mask)]
    r["blocks"] = np.where(mask, raw, 0).astype(np.uint8)
    return r


def sellp_defined(n, slice_size, slice_sets, slice_lengths):
    """slots of a SELL-P matrix that belong to a row (the last slice's slots past row n-1 do not)"""
    tot = int(slice_sets[-1]) * slice_size
    defined = np.ones(tot, bool)
    for s in range(len(slice_lengths)):
        for lr in range(slice_size):
            if s * slice_size + lr >= n:
                defined[(int(slice_sets[s]) + np.arange(int(slice_lengths[s]))) * slice_size + lr] = False
    return defined


def _canon_convert(r, fmt, rp, slice_size):
    if fmt == "sellp":
        d = sellp_defined(len(rp) - 1, slice_size, r["slice_sets"], r["slice_lengths"])
        r["cols"], r["vals"] = np.where(d, r["cols"], 0).astype(r["cols"].dtype), np.where(d, r["vals"], 0)
    return r


# --------------------------------------------------------------------------- the calls
def _call(name, *args, **kwargs):
    fn = getattr(_live, name)
    key = _key(name, fn, args, kwargs)
    if not live():
        return _recorded(name, key)
    out = fn(*args, **kwargs)
    bound = inspect.signature(fn).bind(*args, **kwargs)
    bound.apply_defaults()
    a = bound.arguments
    if name == "jacobi_generate":
        out = _canon_jacobi_generate(out, a["max_bs"])
    elif name == "jacobi_adaptive":
        out = _canon_jacobi_adaptive(out, a["va"])
    elif name == "convert":
        out = _canon_convert(out, a["fmt"], a["rp"], a["slice_size"])
    elif name in ("spmv", "solve"):  # drop the time per repetition
        out = out[:-1] + (0.0,)
    elif name == "write_mtx":
        out = open(a["path"], "rb").read()
    if _RECORD:
        _new[key] = _encode(out, name in _SAMPLED, name in _WHOLE)
    return None if name == "write_mtx" else out


def spmv(*a, **k):
    return _call("spmv", *a, **k)


def solve(*a, **k):
    return _call("solve", *a, **k)


def jacobi_adaptive(*a, **k):
    return _call("jacobi_adaptive", *a, **k)


def csr_transpose(*a, **k):
    return _call("csr_transpose", *a, **k)


def convert(*a, **k):
    return _call("convert", *a, **k)


def read_mtx(*a, **k):
    return _call("read_mtx", *a, **k)


def write_mtx(path, *a, **k):
    if live():
        return _call("write_mtx", path, *a, **k)
    data = _recorded("write_mtx", _key("write_mtx", _live.write_mtx, (path,) + a, k))
    with open(path, "wb") as f:
        f.write(data)


def partition(*a, **k):
    return _call("partition", *a, **k)


def separate_local_nonlocal(*a, **k):
    return _call("separate_local_nonlocal", *a, **k)


def index_map(*a, **k):
    return _call("index_map", *a, **k)


def vector_build_local(*a, **k):
    return _call("vector_build_local", *a, **k)


def jacobi_generate(rp, ci, va, max_bs, block_ptrs=None, transposed=False):
    """live: the reference; else the oracle's generate (+ transpose), accepted when its blocks have the
    digest of the reference's"""
    if live():
        return _call("jacobi_generate", rp, ci, va, max_bs, block_ptrs, transposed)
    want = _recorded("jacobi_generate", _key("jacobi_generate", _live.jacobi_generate,
                                             (rp, ci, va, max_bs, block_ptrs, transposed), {}))
    from tests.helpers import OutI64, Oracle
    orc = Oracle()
    vt = "f64" if va.dtype == np.float64 else "f32"
    n = len(rp) - 1
    r = {k: want[k] for k in ("block_offset", "group_offset", "group_power", "num_blocks")}
    if max_bs <= 1:  # scalar Jacobi: the inverted diagonal
        diag = np.zeros(n, va.dtype)
        rows = np.repeat(np.arange(n), np.diff(rp))
        on = ci == rows
        diag[rows[on]] = va[on]
        blocks = np.zeros(n, va.dtype)
        orc("jacobi_invert_diagonal_" + vt, n, diag, blocks)
        r["block_ptrs"] = np.zeros(n + 1, np.int32)
    else:
        if block_ptrs is None:
            ptrs, nb = np.zeros(n + 1, np.int32), OutI64()
            orc("jacobi_find_blocks_i32", n, rp, ci, max_bs, ptrs, nb)
            block_ptrs = ptrs[:nb.value + 1]
        r["block_ptrs"] = np.ascontiguousarray(block_ptrs, np.int32)
        nb = len(r["block_ptrs"]) - 1
        blocks = np.zeros(want["blocks"].shape, va.dtype)
        orc("jacobi_generate_%s_i32" % vt, n, rp, ci, va, nb, max_bs, r["block_offset"], r["group_offset"],
            r["group_power"], r["block_ptrs"], blocks)
        if transposed:
            out = np.zeros_like(blocks)
            orc("jacobi_transpose_%s_i32" % vt, nb, 32, r["block_offset"], r["group_offset"], r["group_power"],
                r["block_ptrs"], blocks, out)
            blocks = out
    r["blocks"] = blocks
    r = _canon_jacobi_generate(r, max_bs)
    for k in ("blocks", "block_ptrs"):
        if not equal(r[k], want[k]):
            raise AssertionError("jacobi_generate: the oracle's %s are not the reference's" % k)
    return r
