"""The dense solvers as requests on the GPU (sbb_cholesky_begin, sbb_inversion_begin, sbb_trsm_begin,
sbb_gesm_begin).  Loopback ranks (several ranks in this process, sbb_comm_create_local) step through the
calls round by round, which runs the multi-rank plans -- matrices split across ranks, gathers of A and X,
write-back of the output from the gathered copies -- on one GPU; the output must be bit-identical to the
same call on one rank with one component."""
import os
import subprocess

import numpy as np
import pytest
import torch

import superbblas_b200 as sb
from tests import dense_cases as D
from tests.test_gpu_dense import whole, single, place, back, check

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
SQUARE = {"cholesky": sb.cholesky, "inversion": sb.inversion}
SOLVE = {"trsm": sb.trsm, "gesm": sb.gesm}
DTYPES = [np.complex128, np.complex64]
SIZES = dict(x=5, c=4, s=2, C=4, S=2, r=3)


def cut(dims, k, R):
    """R parts of a whole tensor cut along dimension k (parts beyond the extent are empty)"""
    edges = [dims[k] * i // R for i in range(R + 1)]
    out = []
    for i in range(R):
        f, s = [0] * len(dims), list(dims)
        f[k], s[k] = edges[i], edges[i + 1] - edges[i]
        out.append([f, s])
    return np.array(out, np.int32)


def cut_at(dims, k, edges):
    """Parts of a whole tensor cut along dimension k at `edges` (0 ... dims[k])"""
    out = []
    for a, b in zip(edges[:-1], edges[1:]):
        f, s = [0] * len(dims), list(dims)
        f[k], s[k] = a, b - a
        out.append([f, s])
    return np.array(out, np.int32)


# batch cuts of y (extent 5) unlike A's cut(.., R): on every R some ranks' y lies inside their own part of A
Y_EDGES = {2: [0, 3, 5], 3: [0, 1, 2, 5], 4: [0, 1, 3, 4, 5]}


def replicated(dims, R):
    return np.array([[[0] * len(dims), list(dims)]] * R, np.int32)


def rounds(reqs):
    """Every rank has begun: progress every rank once per round until all are done -> rounds taken"""
    done = [False] * len(reqs)
    n = 0
    while not all(done):
        for r, q in enumerate(reqs):
            if not done[r]:
                done[r] = q.progress()
        n += 1
        assert n < 16
    return n


def call(op, R, ops, parts, co, alpha, o, orows, ocols, ox=None, oy=None, host=(), request=True):
    """`op` on R loopback ranks (R None: one rank without a communicator) with one component per part of
    rank r at parts[r*ncomp ..]; ops = (a, x, y0) whole tensors -> (the output as a whole tensor, rounds)"""
    a, x, y0 = ops
    pa, px, py = parts
    co_ = co
    world = R or 1
    solve = op in SOLVE
    ba, ca = place(D.components(a, pa, co_), host)
    if solve:
        bx, cx = place(D.components(x, px, co_), host)
        by, cy = place(D.components(y0, py, co_), host)
    comms = sb.comm_create_local(R) if R else [None]
    n = 0
    try:
        reqs = []
        for r, comm in enumerate(comms):
            na, nx, ny = len(pa) // world, len(px) // world if solve else 0, len(py) // world if solve else 0
            sa = slice(r * na, (r + 1) * na)
            if solve:
                sx, sy = slice(r * nx, (r + 1) * nx), slice(r * ny, (r + 1) * ny)
                q = SOLVE[op](alpha, pa, na, o, orows, ocols, ba[sa], ca[sa], px, nx, ox, bx[sx], cx[sx], py, ny, oy,
                              by[sy], cy[sy], co_, comm=comm, request=request)
            else:
                q = SQUARE[op](pa, na, o, ba[sa], orows, ocols, ca[sa], co_, comm=comm, request=request)
            reqs.append(q)
        if request:
            n = rounds(reqs)
        sb.sync(sb.createGpuContext(0))
    finally:
        for c in comms:
            if c is not None:
                c.destroy()
    if solve:
        return D.assemble(back(by), py, y0, co_), n
    return D.assemble(back(ba), pa, np.full(a.shape, np.nan, a.dtype), co_), n


def same_bits(got, want):
    assert got.shape == want.shape
    assert np.array_equal(got.view(np.uint8), want.view(np.uint8))


def operands(rng, op, dtype, co, o, orows, ocols, ox=None, oy=None, sizes=SIZES):
    a = D.well_conditioned(rng, op, whole(sizes, o), o, orows, ocols, co, dtype)
    if op in SQUARE:
        return (a, None, None), None
    x = (rng.standard_normal(whole(sizes, ox)) + 1j * rng.standard_normal(whole(sizes, ox))).astype(dtype)
    y0 = np.full(whole(sizes, oy), np.nan, dtype)
    return (a, x, y0), D.oracle(op, a, o, orows, ocols, co, 0.5 - 1j, x, ox, oy, whole(sizes, oy))


def one_rank(op, ops, co, o, orows, ocols, ox=None, oy=None):
    a, x, y0 = ops
    parts = (single(a.shape), single(x.shape) if x is not None else None, single(y0.shape) if y0 is not None else None)
    return call(op, None, ops, parts, co, 0.5 - 1j, o, orows, ocols, ox, oy, request=False)[0]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("R", [2, 3, 4])
@pytest.mark.parametrize("op", ["cholesky", "inversion"])
def test_square_ops_on_loopback_ranks(op, R, dtype):
    """Matrices cut along a row label, along a column label, replicated, cut along the batch label, and with
    host components: R stepped ranks give the bits of one rank with one component"""
    rng = np.random.default_rng(60 + R)
    o, co = "xcCsS", sb.FastToSlow
    ops, _ = operands(rng, op, dtype, co, o, "cs", "CS")
    want = one_rank(op, ops, co, o, "cs", "CS")
    check(want, D.oracle(op, ops[0], o, "cs", "CS", co), dtype)
    dims = list(ops[0].shape)
    cases = [(cut(dims, o.index("c"), R), ()), (cut(dims, o.index("C"), R), (1,)), (replicated(dims, R), ()),
             (cut(dims, o.index("x"), R), (0,))]
    for pa, host in cases:
        got, n = call(op, R, ops, (pa, None, None), co, 1, o, "cs", "CS", host=host)
        same_bits(got, want)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("R", [2, 3, 4])
@pytest.mark.parametrize("left", [True, False])
@pytest.mark.parametrize("op", ["trsm", "gesm"])
def test_solves_on_loopback_ranks(op, left, R, dtype):
    """A cut along a row label or replicated (a Gram matrix every rank holds), x and y cut unlike A and
    unlike each other, some components on the host: the bits of one rank with one component, two exchanges
    (A, then x: two rounds) where both are gathered"""
    rng = np.random.default_rng(70 + R + 10 * left)
    o, co = "xcCsS", sb.SlowToFast
    ox, oy = ("rxcs", "xCrS") if left else ("rxCS", "xcrs")
    ops, oracle = operands(rng, op, dtype, co, o, "cs", "CS", ox, oy)
    want = one_rank(op, ops, co, o, "cs", "CS", ox, oy)
    check(want, oracle, dtype)
    a, x, y0 = ops
    da, dx, dy = list(a.shape), list(x.shape), list(y0.shape)
    vx = "c" if left else "C"
    cases = [
        # A cut along rows, x along its vector label, y along the batch label: A and x gathered
        ((cut(da, o.index("c"), R), cut(dx, ox.index(vx), R), cut(dy, oy.index("x"), R)), (), 2),
        # replicated Gram matrix, x and y cut along the right-hand sides: in place
        ((replicated(da, R), cut(dx, ox.index("r"), R), cut(dy, oy.index("r"), R)), (), 1),
        # replicated Gram matrix, x cut along the batch label, y along the right-hand sides, host x
        ((replicated(da, R), cut(dx, ox.index("x"), R), cut(dy, oy.index("r"), R)), (0,), None),
        # A cut along columns, x replicated, y cut along its vector label, host A
        ((cut(da, o.index("C"), R), replicated(dx, R), cut(dy, oy.index("S" if left else "s"), R)), (0,), None),
        # A cut along the batch label, x replicated, y cut along it elsewhere: the items whose matrices
        # this rank holds run during the gather of A
        ((cut(da, o.index("x"), R), replicated(dx, R), cut_at(dy, oy.index("x"), Y_EDGES[R])), (), 1),
    ]
    early = [sb.dense_steps(sb.TRSM, sb.C128, cases[-1][0][0], 1, o, "cs", "CS", co, R, r, px=cases[-1][0][1],
                            ncomponentsx=1, ox=ox, py=cases[-1][0][2], ncomponentsy=1, oy=oy)["item_steps"]
             for r in range(R)]
    assert [0] in early and [1] in early, early
    for parts, host, nrounds in cases:
        got, n = call(op, R, ops, parts, co, 0.5 - 1j, o, "cs", "CS", ox, oy, host=host)
        same_bits(got, want)
        if nrounds is not None:
            assert n == nrounds, (parts, n)


@pytest.mark.parametrize("R", [2, 3, 4])
def test_blocked_tier_on_loopback_ranks(R):
    """cholesky and trsm of n = 114 complex double (over one CTA's shared memory: the blocked tier) with the
    matrix, x and y cut along their rows: A and x gathered, y written back from temporaries"""
    rng = np.random.default_rng(80 + R)
    sizes = dict(a=114, b=114, z=2, r=6)
    o, co = "abz", sb.FastToSlow
    chol, _ = operands(rng, "cholesky", np.complex128, co, o, "a", "b", sizes=sizes)
    want = one_rank("cholesky", chol, co, o, "a", "b")
    check(want, D.oracle("cholesky", chol[0], o, "a", "b", co), np.complex128)
    got, n = call("cholesky", R, chol, (cut([114, 114, 2], 0, R), None, None), co, 1, o, "a", "b")
    same_bits(got, want)
    assert n == 1
    ops, oracle = operands(rng, "trsm", np.complex128, co, o, "a", "b", "arz", "brz", sizes=sizes)
    want = one_rank("trsm", ops, co, o, "a", "b", "arz", "brz")
    check(want, oracle, np.complex128)
    parts = (cut([114, 114, 2], 0, R), cut([114, 6, 2], 0, R), cut([114, 6, 2], 0, R))
    got, n = call("trsm", R, ops, parts, co, 0.5 - 1j, o, "a", "b", "arz", "brz")
    same_bits(got, want)
    assert n == 2


@pytest.mark.parametrize("op", ["cholesky", "inversion", "trsm", "gesm"])
def test_requests_on_one_rank(op):
    """On one rank, with one component and with the matrices cut in two components: the call and its
    begin + wait give the same bits with the same number of kernel launches; a second wait does nothing"""
    rng = np.random.default_rng(90)
    o, co = "xcCsS", sb.FastToSlow
    ox, oy = ("rxcs", "xCrS")
    ops, _ = operands(rng, op, np.complex128, co, o, "cs", "CS", ox, oy)
    a, x, y0 = ops
    for ncomp in (1, 2):
        pa = single(a.shape) if ncomp == 1 else cut(list(a.shape), o.index("c"), 2)
        px = single(x.shape) if x is not None else None
        py = single(y0.shape) if y0 is not None else None
        outs, counts = [], []
        for request in (False, True):
            sb.launch_count(reset=True)
            comps = D.components(a, pa, co)
            ba, ca = place(comps)
            if op in SOLVE:
                bx, cx = place(D.components(x, px, co))
                by, cy = place(D.components(y0, py, co))
                q = SOLVE[op](0.5 - 1j, pa, ncomp, o, "cs", "CS", ba, ca, px, 1, ox, bx, cx, py, 1, oy, by, cy, co,
                              request=request)
            else:
                q = SQUARE[op](pa, ncomp, o, ba, "cs", "CS", ca, co, request=request)
            if request:
                q.wait()
                q.wait()
                assert q.progress()
            sb.sync(sb.createGpuContext(0))
            counts.append(sb.launch_count())
            outs.append(D.assemble(back(by), py, y0, co) if op in SOLVE else
                        D.assemble(back(ba), pa, np.full(a.shape, np.nan, a.dtype), co))
        same_bits(outs[1], outs[0])
        assert counts[0] == counts[1] and counts[0] > 0, counts


def test_argument_errors_come_from_begin():
    """The begin returns the plain call's message, and nothing is left allocated"""
    o = "xcC"
    dims = whole(SIZES, o)
    a = np.zeros(dims, np.complex128)
    sb.clearCaches()
    before = sb.liveAllocations()
    bufs, ctx = place(D.components(a, single(dims), sb.FastToSlow))
    msgs = []
    for request in (False, True):
        with pytest.raises(RuntimeError) as e:
            sb.cholesky(single(dims), 1, o, bufs, "c", "c", ctx, sb.FastToSlow, request=request)
        msgs.append(str(e.value))
    assert msgs[0] == msgs[1] and msgs[0].startswith("cholesky: ")
    big = np.zeros((114, 114), np.complex128)
    bb, cb = place([big.ravel()])
    msgs = []
    for request in (False, True):
        with pytest.raises(RuntimeError, match="over the limit") as e:
            sb.inversion(single(big.shape), 1, "ab", bb, "a", "b", cb, sb.FastToSlow, request=request)
        msgs.append(str(e.value))
    assert msgs[0] == msgs[1]
    del bufs, bb
    sb.clearCaches()
    assert sb.liveAllocations() == before


def test_completing_before_every_rank_has_begun():
    """One loopback rank completes a gathering cholesky that the other has not begun: an error, and the
    request's blocks go back to the pool"""
    rng = np.random.default_rng(91)
    o = "xcCsS"
    a = D.well_conditioned(rng, "cholesky", whole(SIZES, o), o, "cs", "CS", sb.FastToSlow, np.complex128)
    pa = cut(list(a.shape), o.index("c"), 2)
    sb.clearCaches()
    before = sb.liveAllocations()
    comms = sb.comm_create_local(2)
    try:
        bufs, ctx = place(D.components(a, pa, sb.FastToSlow))
        q = sb.cholesky(pa, 1, o, bufs[:1], "cs", "CS", ctx[:1], sb.FastToSlow, comm=comms[0], request=True)
        with pytest.raises(RuntimeError, match="every rank must begin"):
            q.wait()
    finally:
        for c in comms:
            c.destroy()
    sb.sync(sb.createGpuContext(0))
    del bufs
    sb.clearCaches()
    assert sb.liveAllocations() == before


def test_loopback_requests_do_not_leak():
    rng = np.random.default_rng(92)
    o, co = "xcCsS", sb.FastToSlow
    ox, oy = "rxcs", "xCrS"
    ops, _ = operands(rng, "trsm", np.complex128, co, o, "cs", "CS", ox, oy)
    a, x, y0 = ops
    sb.clearCaches()
    before = sb.liveAllocations()
    parts = (cut(list(a.shape), o.index("c"), 2), cut(list(x.shape), ox.index("c"), 2),
             cut(list(y0.shape), oy.index("x"), 2))
    call("trsm", 2, ops, parts, co, 1, o, "cs", "CS", ox, oy, host=(1,))
    call("cholesky", 2, (a, None, None), (parts[0], None, None), co, 1, o, "cs", "CS")
    sb.clearCaches()
    assert sb.liveAllocations() == before


def test_cxx_dense_request_program(tmp_path):
    """tests/cxx/dense_request_test.cpp, compiled against include/superbblas.h and the in-tree library into a
    temporary directory, and run."""
    root = os.path.dirname(HERE)
    lib = os.path.join(root, "superbblas_b200", "lib")
    exe = str(tmp_path / "dense_request_test")
    r = subprocess.run([os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), "-std=c++17", "-O2", "-ccbin",
                        "/usr/bin/g++", "-I" + os.path.join(root, "include"),
                        os.path.join(HERE, "cxx", "dense_request_test.cpp"), "-o", exe, "-L" + lib,
                        "-lsuperbblas_b200", "-Xlinker", "-rpath", "-Xlinker", lib],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Everything went ok!" in r.stdout
