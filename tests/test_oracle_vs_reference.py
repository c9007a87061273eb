"""Pins the numpy oracle (oracle/oracle.py) against the answers of the reference (the unmodified
superbblas, CPU build, behind oracle/ref.py): partition generators exactly, copy bit for bit,
contraction within rounding.

The compiled reference is built from sources outside the repository, so the answers are stored in
tests/golden/oracle_vs_reference/answers.npz and the comparison needs nothing else.  Each
enumeration below draws the same seeded cases it always did and yields what the library it is given
(`R`: oracle.ref or oracle.oracle, same calling convention) answers.  Exact answers (partitions,
hole sets, copies) are stored as 64-bit digests of their bits; a contraction result as its norm
and a seeded random projection of it (`sketch`).  The file names its `source`:

* "reference": recorded from the compiled reference by `python tests/golden/generate.py --answers`;
  the tests then pin the oracle to the reference.
* "oracle": `record(oracle.oracle, "oracle")`, for a tree in which the reference cannot be built.
  The tests then pin the oracle to its own earlier answers and catch any drift.  They were
  recorded with oracle/oracle.py and tests/cases.py unchanged since these comparisons last ran
  against the compiled reference and passed; the reference's own outputs that stay in the
  repository are the golden vectors of tests/test_golden.py.
"""
import hashlib
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests import cases as C

ANSWERS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_vs_reference",
                       "answers.npz")
SKETCH = 16  # random directions a contraction result is projected on


def digest(a):
    """64 bits of the sha256 of an array's dtype, shape and bytes (equal digests: C.bits_equal)"""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode() + a.tobytes()).digest()
    return int(np.frombuffer(h[:8], dtype=np.uint64)[0])


def sketch(w):
    """[norm(w), P w] with P a seeded Gaussian SKETCH x n matrix scaled so that E|P e|^2 = |e|^2:
    a difference e anywhere in w shows up in P w.  |P e|^2 / |e|^2 is chi-squared with at least
    SKETCH degrees of freedom over SKETCH, so |P e| < |e| / 2 with probability below 1e-3."""
    w = np.asarray(w, dtype=np.complex128).reshape(-1)
    p = np.random.default_rng(w.size).standard_normal((SKETCH, w.size)) / np.sqrt(SKETCH)
    return np.concatenate([[np.linalg.norm(w)], p @ w])


def close(got, want, bound):
    """Sketches of two results whose difference is at most `bound` in norm (an error up to twice
    the bound passes with probability below 1e-3, see `sketch`)"""
    return abs(got[0] - want[0]) <= bound and np.linalg.norm(got[1:] - want[1:]) <= bound


# --- enumerations: what the reference was asked, and what R answers ---------------------------------

def partitioning_random(R):
    rng = np.random.default_rng(1)
    for _ in range(200):
        n = int(rng.integers(1, 6))
        order = "".join(rng.permutation(list("xyztsc"))[:n])
        dim = [int(rng.integers(1, 13)) for _ in range(n)]
        labels = "".join(rng.permutation(list(order))[:int(rng.integers(1, n + 1))])
        nprocs = int(rng.integers(1, 25))
        procs = R.partitioning_distributed_procs(order, dim, labels, nprocs)
        ncomp = int(rng.integers(1, 4))
        P = int(np.prod(procs))
        ext = [int(rng.integers(0, 3)) for _ in range(n)]
        yield [digest(np.asarray(procs, dtype=np.int32)),
               digest(np.asarray(R.basic_partitioning(order, dim, procs, labels, P, ncomp), dtype=np.int32)),
               digest(np.asarray(R.basic_partitioning_ext(dim, procs, P, False, ext), dtype=np.int32))]


def make_hole_sets(R):
    rng = np.random.default_rng(2)
    for _ in range(100):
        n = int(rng.integers(1, 4))
        dim = [int(rng.integers(1, 7)) for _ in range(n)]
        frm = [int(rng.integers(0, d)) for d in dim]
        size = [int(rng.integers(1, d + 1)) for d in dim]
        hf = [int(rng.integers(0, d)) for d in dim]
        hs = [int(rng.integers(0, d + 1)) for d in dim]
        yield digest(np.asarray(O.box_elements(R.make_hole(frm, size, hf, hs, dim), dim), dtype=np.int64))


def copy_random(R, seed, masked=False):
    """(it, j, digest) of every output part of the cases the reference accepts"""
    rng = np.random.default_rng((300 if masked else 100) + seed)
    for it in range(80):
        case = C.random_copy_case(rng)
        if not C.safe_for_reference(case):
            continue
        m0 = m1 = None
        if masked:
            v0, v1 = C.make_copy_data(case, seed * 100 + it, consistent=True)
            m0, m1 = C.make_masks(case, seed * 100 + it, density=[0.5, 0.1, 0.9][it % 3])
        else:
            v0, v1 = C.make_copy_data(case, seed * 100 + it)
        out = [x.copy() for x in v1]
        R.copy(case["alpha"], case["p0"], case["o0"], case["from0"], case["size0"], case["dim0"], v0,
               case["p1"], case["o1"], case["from1"], case["dim1"], out, case["co"], case["copyadd"],
               mask0=m0, mask1=m1)
        for j, x in enumerate(out):
            yield it, j, digest(x)


def contraction_random(R, seed):
    """(it, j, bound, sketch) of every non-empty output part"""
    rng = np.random.default_rng(200 + seed)
    for it in range(40):
        case = C.random_contraction_case(rng)
        v0, v1, vr = C.make_contraction_data(case, seed * 100 + it)
        out = [x.copy() for x in vr]
        R.contraction(case["alpha"], case["p0"], case["from0"], case["size0"], case["dim0"],
                      case["o0"], case["conj0"], v0, case["p1"], case["from1"], case["size1"],
                      case["dim1"], case["o1"], case["conj1"], v1, case["beta"], case["pr"],
                      case["fromr"], case["sizer"], case["dimr"], case["o_r"], out, case["co"])
        tol = 1e-12 if case["T"] in (np.dtype(np.float64), np.dtype(np.complex128)) else 1e-5
        for j, w in enumerate(out):
            if w.size:
                yield it, j, tol * max(np.linalg.norm(w), 1e-30, np.sqrt(w.size)), sketch(w)


def config1_shapes(R):
    """BASELINE config 1: copy "xyztsc"->"cstzyx" (both orders) and the contraction over s,c on
    8^3x16: two copy digests and the contraction's sketch"""
    L, Lt = 8, 16
    dim0, dim1 = [L, L, L, Lt, 4, 3], [3, 4, Lt, L, L, L]
    v0 = C.fill(int(np.prod(dim0)), np.complex128, 11)
    p0, p1 = np.array([[[0] * 6, dim0]]), np.array([[[0] * 6, dim1]])
    digests = []
    for co in ("FastToSlow", "SlowToFast"):
        b = [np.zeros_like(v0)]
        R.copy(1, p0, "xyztsc", [0] * 6, dim0, dim0, [v0], p1, "cstzyx", [0] * 6, dim1, b, co, 0)
        digests.append(digest(b[0]))
    v1 = C.fill(int(np.prod(dim0)), np.complex128, 12)
    dimr = [L, L, L, Lt]
    pr = np.array([[[0] * 4, dimr]])
    b = [np.zeros(int(np.prod(dimr)), np.complex128)]
    R.contraction(1, p0, [0] * 6, dim0, dim0, "xyztsc", True, [v0], p0, [0] * 6, dim0, dim0, "xyztsc",
                  False, [v1], 0, pr, [0] * 4, dimr, dimr, "xyzt", b, "FastToSlow")
    return digests, b[0]


def record(R, source):
    """Every answer of the enumerations above given by R, as stored in ANSWERS"""
    out = {"source": np.array(source),
           "partitioning_random": np.array(list(partitioning_random(R)), dtype=np.uint64),
           "make_hole_sets": np.array(list(make_hole_sets(R)), dtype=np.uint64)}
    for masked, name, seeds in ((False, "copy_random", 6), (True, "masked_copy_random", 4)):
        for seed in range(seeds):
            out["%s_%d" % (name, seed)] = np.array(list(copy_random(R, seed, masked)), dtype=np.uint64)
    for seed in range(4):
        rows = list(contraction_random(R, seed))
        out["contraction_random_%d_at" % seed] = np.array([r[:2] for r in rows], dtype=np.int32)
        out["contraction_random_%d" % seed] = np.array([r[3] for r in rows])
    digests, r = config1_shapes(R)
    out["config1_copy"] = np.array(digests, dtype=np.uint64)
    out["config1_contraction"] = sketch(r)
    return out


@pytest.fixture(scope="module")
def answers():
    with np.load(ANSWERS) as z:
        return {k: z[k] for k in z.files}


# --- the comparisons ---------------------------------------------------------------------------------

def test_partition_known_answers():
    # the reference's own known answers: tests/dist.cpp:103-125
    for dim, labels, n, want in [([8, 8, 8, 16], "zt", 8, [1, 1, 2, 4]),
                                 ([4, 4, 4, 8], "xyzt", 6, [2, 1, 1, 3]),
                                 ([16, 16, 16, 32], "tzyx", 64, [2, 2, 2, 8]),
                                 ([3, 5, 7, 2], "xyzt", 12, [2, 2, 3, 1]),
                                 ([6, 6, 6, 6], "xy", 9, [3, 3, 1, 1]),
                                 ([48, 48, 48, 96], "zt", 8, [1, 1, 2, 4])]:
        assert O.partitioning_distributed_procs("xyzt", dim, labels, n) == want, (dim, labels, n)


def test_partitioning_random(answers):
    got = np.array(list(partitioning_random(O)), dtype=np.uint64)
    want = answers["partitioning_random"]
    assert got.shape == want.shape == (200, 3)
    bad = np.argwhere(got != want)
    assert len(bad) == 0, "case, function (procs, basic_partitioning, _ext): %s" % bad[:5].tolist()


def test_make_hole_sets(answers):
    got = np.array(list(make_hole_sets(O)), dtype=np.uint64)
    want = answers["make_hole_sets"]
    assert got.shape == want.shape == (100,)
    assert np.array_equal(got, want), np.flatnonzero(got != want)[:5].tolist()


def _copies_bit_exact(answers, name, seed, masked):
    got = np.array(list(copy_random(O, seed, masked)), dtype=np.uint64)
    want = answers["%s_%d" % (name, seed)]
    assert len(np.unique(want[:, 0])) >= 30
    assert got.shape == want.shape and np.array_equal(got[:, :2], want[:, :2])
    bad = want[got[:, 2] != want[:, 2], :2]
    assert len(bad) == 0, "(case, part) differing from the reference: %s" % bad[:5].tolist()


@pytest.mark.parametrize("seed", range(6))
def test_copy_random_bit_exact(answers, seed):
    _copies_bit_exact(answers, "copy_random", seed, False)


@pytest.mark.parametrize("seed", range(4))
def test_masked_copy_random_bit_exact(answers, seed):
    """Masked copies (MaskType masks on both tensors, tensor.h:1022-1027): the reference with
    compatible masks against the oracle, bit for bit."""
    _copies_bit_exact(answers, "masked_copy_random", seed, True)


@pytest.mark.parametrize("seed", range(4))
def test_contraction_random(answers, seed):
    at, want = answers["contraction_random_%d_at" % seed], answers["contraction_random_%d" % seed]
    rows = list(contraction_random(O, seed))
    assert [list(r[:2]) for r in rows] == at.tolist()
    for (it, j, bound, got), w in zip(rows, want):
        assert close(got, w, bound), (seed, it, j)


def test_config1_shapes(answers):
    """BASELINE config 1: copy "xyztsc"->"cstzyx" and the contraction over s,c on 8^3x16."""
    digests, r = config1_shapes(O)
    assert digests == answers["config1_copy"].tolist()
    want = answers["config1_contraction"]
    assert close(sketch(r), want, 1e-13 * abs(want[0]))
