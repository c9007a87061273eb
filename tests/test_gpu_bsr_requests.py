"""bsr_krylov and create_bsr / create_kron_bsr as requests on the GPU.  Loopback ranks (several ranks in
this process, sbb_comm_create_local) step through the calls round by round, which runs the multi-rank
operator path, the halo gather with its cross-rank unpack and the write-back into a y partition unlike the
operator's, on one GPU; y must be bit-identical to the same operator on one rank and one component."""
import os
import subprocess

import numpy as np
import pytest
import torch

import superbblas_b200 as sb
from tests import bsr_cases as B
from tests import kron_bsr_cases as KB
from tests.test_gpu_bsr import single, split, dev, check
from tests.test_gpu_kron_bsr import wilson

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
DTYPES = [np.float32, np.float64, np.complex64, np.complex128]


def plain_stencil(rng, dtype, dims):
    """Nine-point operator with dense blocks along the first label, on "sxyzt" """
    blockim = [dims[0], 1, 1, 1, 1]
    ops = B.stencil_operator(rng, single(dims), dims, blockim, dtype, sb.FastToSlow)
    return dict(ops=ops, pim=single(dims), dimi=dims, dimd=dims, blockim=blockim, blockdom=blockim, imfast=True,
                co=sb.FastToSlow, oim="sxyzt", odom="SXYZT", kron=False)


def kron_stencil(rng, dtype, dims):
    op = wilson(rng, dtype, single(dims), dims)
    op["kron"] = True
    return op


def split_op(op1, pim):
    """The one-part operator op1 cut into the parts pim along its slowest label (rows stay in order)"""
    ii, jj, v = op1["ops"][0]
    bim = KB.eff(op1["blockim"], op1.get("kronim", [1] * len(op1["dimi"])))
    bsz = int(np.prod(op1["blockim"])) * int(np.prod(op1["blockdom"]))
    ptr = np.concatenate([[0], np.cumsum(ii)])
    per_slice = len(ii) // (op1["dimi"][-1] // bim[-1])
    parts = []
    for f, s in pim:
        a, b = f[-1] * per_slice, (f[-1] + s[-1]) * per_slice
        parts.append((ii[a:b], jj[ptr[a]:ptr[b]], v[ptr[a] * bsz:ptr[b] * bsz]))
    return dict(op1, ops=parts, pim=np.asarray(pim, np.int32))


def oracle(op, x, ox, y0, oy, alpha, beta, power, psize):
    if op["kron"]:
        a = KB.oracle_matrix(op["ops"], op["kronv"], op["pim"], op["dimi"], op["dimd"], op["blockim"],
                             op["blockdom"], op["kronim"], op["krondom"], op["imfast"], op["co"])
    else:
        a = B.operator_matrix(op["ops"], op["pim"], op["dimi"], op["dimd"], op["blockim"], op["blockdom"],
                              op["imfast"], op["co"])
    return B.apply(a, op["oim"], op["odom"], x, ox, y0, oy, alpha, beta, power, psize, [0] * len(oy))


def create(op, r, ncomp, comm, request):
    """Rank r's operator (components r*ncomp ..) on the GPU -> (handle, request or None, kept arrays)"""
    mine = op["ops"][r * ncomp:(r + 1) * ncomp]
    ii, jj, v = [dev(o[0]) for o in mine], [dev(o[1].reshape(-1)) for o in mine], [dev(o[2]) for o in mine]
    pdom = np.array([[[0] * len(op["dimd"]), list(op["dimd"])]] * len(op["pim"]), np.int32)
    gpu = sb.createGpuContext(0)
    if op["kron"]:
        kv = [dev(op["kronv"]) for _ in mine]
        res = sb.create_kron_bsr(op["pim"], op["dimi"], pdom, op["dimd"], ncomp, op["blockim"], op["blockdom"],
                                 op["kronim"], op["krondom"], op["imfast"], ii, jj, v, kv, gpu, op["co"], comm=comm,
                                 request=request)
    else:
        kv = []
        res = sb.create_bsr(op["pim"], op["dimi"], pdom, op["dimd"], ncomp, op["blockim"], op["blockdom"],
                            op["imfast"], ii, jj, v, gpu, op["co"], comm=comm, request=request)
    h, q = res if request else (res, None)
    return h, q, (v, kv)


def rounds(reqs):
    """Every rank has begun: progress every rank once per round until all are done"""
    done = [False] * len(reqs)
    n = 0
    while not all(done):
        for r, q in enumerate(reqs):
            if not done[r]:
                done[r] = q.progress()
        n += 1
        assert n < 64
    return n


def krylov(op, R, x, ox, px, y0, oy, py, alpha, beta, power=None):
    """create and bsr_krylov on R loopback ranks (R None: one rank without a communicator), stepped in
    rounds -> y as a whole tensor"""
    ncomp = len(op["pim"]) // (R or 1)
    comms = sb.comm_create_local(R) if R else [None]
    gpu = sb.createGpuContext(0)
    try:
        made = [create(op, r, ncomp, c, R is not None) for r, c in enumerate(comms)]
        if R:
            rounds([q for _, q, _ in made])
        xs = [dev(c) for c in B.components(x, px, op["co"])]
        ys = [dev(c) for c in B.components(y0, py, op["co"])]
        reqs = []
        for r, c in enumerate(comms):
            reqs.append(sb.bsr_krylov(alpha, made[r][0], op["oim"], op["odom"], px, ncomp, ox, [0] * len(ox),
                                      list(x.shape), list(x.shape), xs[r * ncomp:(r + 1) * ncomp], gpu, beta, py, oy,
                                      [0] * len(oy), list(y0.shape), list(y0.shape), power,
                                      ys[r * ncomp:(r + 1) * ncomp], gpu, op["co"], comm=c, ncomponentsy=ncomp,
                                      request=R is not None))
        if R:
            rounds(reqs)
        sb.sync(gpu)
        for h, _, _ in made:
            h.destroy()
    finally:
        for c in comms:
            if c is not None:
                c.destroy()
    return B.assemble([c.cpu().numpy() for c in ys], py, y0, op["co"])


def operands(rng, op, dtype, ncols, power, beta):
    dims = op["dimi"]
    x = B.rnd(rng, dtype, *dims, ncols)
    ydims = list(dims) + [ncols] + ([3] if power else [])
    y0 = np.full(ydims, np.nan, dtype) if beta == 0 else B.rnd(rng, dtype, *ydims)
    return x, op["odom"] + "n", y0, op["oim"] + "n" + ("p" if power else "")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kron", [False, True])
@pytest.mark.parametrize("R", [2, 3, 4])
def test_loopback_ranks_stepped_match_one_rank(R, kron, dtype):
    """Plain and Kronecker, powers 1 and 3, direct and written back, beta 0 and not: R loopback ranks with
    the lattice and x cut along t give the bits of one rank with one component"""
    rng = np.random.default_rng(40 + R + 10 * kron)
    dims = [4, 3, 2, 2, 2, 12] if kron else [2, 2, 2, 2, 12]
    op1 = (kron_stencil if kron else plain_stencil)(rng, dtype, dims)
    cuts = [12 * k // R for k in range(1, R)]
    op = split_op(op1, split(dims, len(dims) - 1, cuts))
    t = len(dims) - 1
    alpha = 0.75 - 0.5j if np.dtype(dtype).kind == "c" else 0.75
    for power in (None, "p"):
        for direct in (True, False):
            for beta in (0, 0.5):
                x, ox, y0, oy = operands(rng, op1, dtype, 2, power, beta)
                px = split(list(x.shape), t, cuts)
                py = split(list(y0.shape), t, cuts if direct else [c + 1 for c in cuts])
                got = krylov(op, R, x, ox, px, y0, oy, py, alpha, beta, power)
                one = krylov(op1, None, x, ox, single(x.shape), y0, oy, single(y0.shape), alpha, beta, power)
                assert np.array_equal(got.view(np.uint8), one.view(np.uint8)), (power, direct, beta)
                check(got, oracle(op1, x, ox, y0, oy, alpha, beta, power, 3 if power else 1), dtype)


def test_spin_colour_8_4_on_four_loopback_ranks():
    """The 8^4 spin-colour operator of test_gpu_kron_bsr with 12 columns, cut along t over 4 ranks"""
    rng = np.random.default_rng(12)
    dims = [4, 3, 8, 8, 8, 8]
    op1 = kron_stencil(rng, np.complex128, dims)
    op = split_op(op1, split(dims, 5, [2, 4, 6]))
    x = B.rnd(rng, np.complex128, *dims, 12)
    y0 = np.full(dims + [12], np.nan, np.complex128)
    px, py = split(list(x.shape), 5, [2, 4, 6]), split(list(y0.shape), 5, [2, 4, 6])
    got = krylov(op, 4, x, "SCXYZTn", px, y0, "scxyztn", py, 1, 0)
    one = krylov(op1, None, x, "SCXYZTn", single(x.shape), y0, "scxyztn", single(y0.shape), 1, 0)
    assert np.array_equal(got.view(np.uint8), one.view(np.uint8))
    assert B.rel_err(got, oracle(op1, x, "SCXYZTn", y0, "scxyztn", 1, 0, None, 1)) < 1e-12


def one_rank_call(op, h, x, y0, host_y, request):
    """bsr_krylov of the whole x (on the GPU) into y0's storage, on the host or the GPU, without a
    communicator -> (request or None, the y component)"""
    ox, oy = op["odom"] + "n", op["oim"] + "n"
    xc = dev(B.components(x, single(x.shape), op["co"])[0])
    yc = dev(B.components(y0, single(y0.shape), op["co"])[0], host_y)
    ctxy = sb.createCpuContext() if host_y else sb.createGpuContext(0)
    r = sb.bsr_krylov(1, h, op["oim"], op["odom"], single(x.shape), 1, ox, [0] * len(ox), list(x.shape),
                      list(x.shape), [xc], sb.createGpuContext(0), 0, single(y0.shape), oy, [0] * len(oy),
                      list(y0.shape), list(y0.shape), None, [yc], ctxy, op["co"], request=request)
    return r, yc


def test_requests_on_one_rank():
    """Host y is complete after wait and a second wait does nothing; a pending create is an error for
    bsr_krylov; the launches of a one-rank call do not change with a request; nothing leaks"""
    rng = np.random.default_rng(50)
    dims = [2, 2, 2, 2, 6]
    op = plain_stencil(rng, np.complex128, dims)
    x = B.rnd(rng, np.complex128, *dims, 3)
    y0 = np.full(dims + [3], np.nan, np.complex128)
    want = oracle(op, x, "SXYZTn", y0, "sxyztn", 1, 0, None, 1)
    sb.clearCaches()
    before = sb.liveAllocations()
    h, q, keep = create(op, 0, 1, None, True)
    with pytest.raises(RuntimeError, match="^bsr_krylov: the operator's create has not completed"):
        one_rank_call(op, h, x, y0, True, False)
    q.wait()
    q.wait()
    req, yc = one_rank_call(op, h, x, y0, True, True)
    req.wait()
    got = B.assemble([yc], single(y0.shape), y0, op["co"])
    check(got, want, np.complex128)
    first = yc.copy()
    req.wait()
    assert np.array_equal(yc.view(np.uint8), first.view(np.uint8))
    assert req.progress()
    # the launch sequence of a one-rank call is the same with and without a request
    counts = []
    for request in (False, True):
        sb.launch_count(reset=True)
        r, yd = one_rank_call(op, h, x, y0, False, request)
        if request:
            while not r.progress():
                pass
        sb.sync(sb.createGpuContext(0))
        counts.append(sb.launch_count())
        assert B.rel_err(B.assemble([yd.cpu().numpy()], single(y0.shape), y0, op["co"]), want) < 1e-12
    assert counts[0] == counts[1] and counts[0] > 0, counts
    del r, yd
    h.destroy()
    sb.clearCaches()
    assert sb.liveAllocations() == before


def test_create_errors_at_completion():
    """A bad jj on one loopback rank: begin succeeds everywhere, completion fails on every rank with the same
    message, and bsr_krylov on the handle says that its create failed"""
    rng = np.random.default_rng(51)
    dims = [2, 2, 2, 2, 4]
    op = split_op(plain_stencil(rng, np.float64, dims), split(dims, 4, [2]))
    ii, jj, v = op["ops"][1]
    jj = jj.copy()
    jj[0, 0] = 1  # not a multiple of blockdom (2) along s
    op["ops"][1] = (ii, jj, v)
    sb.clearCaches()
    before = sb.liveAllocations()
    comms = sb.comm_create_local(2)
    try:
        made = [create(op, r, 1, comms[r], True) for r in range(2)]
        for h, q, _ in made:
            with pytest.raises(RuntimeError, match="^create_bsr: a block's domain coordinate"):
                q.progress()
        with pytest.raises(RuntimeError, match="^bsr_krylov: the operator's create failed"):
            one_rank_call(op, made[0][0], np.zeros(dims + [1]), np.zeros(dims + [1]), True, False)
        for h, _, _ in made:
            h.destroy()
    finally:
        for c in comms:
            c.destroy()
    sb.clearCaches()
    assert sb.liveAllocations() == before


def test_loopback_requests_do_not_leak():
    rng = np.random.default_rng(52)
    dims = [2, 2, 2, 2, 8]
    op1 = plain_stencil(rng, np.float64, dims)
    op = split_op(op1, split(dims, 4, [4]))
    x, ox, y0, oy = operands(rng, op1, np.float64, 1, None, 0)
    sb.clearCaches()
    before = sb.liveAllocations()
    for direct in (True, False):
        py = split(list(y0.shape), 4, [4 if direct else 5])
        krylov(op, 2, x, ox, split(list(x.shape), 4, [4]), y0, oy, py, 1, 0)
    sb.clearCaches()
    assert sb.liveAllocations() == before


def test_cxx_bsr_request_program(tmp_path):
    """tests/cxx/bsr_request_test.cpp, compiled against include/superbblas.h and the in-tree library into a
    temporary directory, and run."""
    root = os.path.dirname(HERE)
    lib = os.path.join(root, "superbblas_b200", "lib")
    exe = str(tmp_path / "bsr_request_test")
    r = subprocess.run([os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), "-std=c++17", "-O2", "-ccbin",
                        "/usr/bin/g++", "-I" + os.path.join(root, "include"),
                        os.path.join(HERE, "cxx", "bsr_request_test.cpp"), "-o", exe, "-L" + lib,
                        "-lsuperbblas_b200", "-Xlinker", "-rpath", "-Xlinker", lib],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Everything went ok!" in r.stdout
