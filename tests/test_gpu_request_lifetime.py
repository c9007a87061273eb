"""What a request may outlive and what it leaves behind: a block-sparse operator cannot be destroyed while
its create or a bsr_krylov on it is open, and a request whose step failed stays failed, with its own
message, until it is released."""
import ctypes

import numpy as np
import pytest

import superbblas_b200 as sb
from superbblas_b200._lib import lib
from tests import bsr_cases as B
from tests import dense_cases as D
from tests.test_gpu_bsr import split, dev
from tests.test_gpu_bsr_requests import plain_stencil, split_op, create, rounds, operands, one_rank_call
from tests.test_gpu_dense import whole, place
from tests.test_gpu_dense_requests import SIZES, cut

pytestmark = pytest.mark.gpu


def test_destroy_refuses_an_operator_with_an_open_request():
    """destroy() under an open create or bsr_krylov request is an error that leaves the handle valid; after
    wait() it succeeds, y has the bits of the call without requests, and nothing leaks"""
    rng = np.random.default_rng(60)
    dims = [2, 2, 2, 2, 6]
    op = plain_stencil(rng, np.complex128, dims)
    x = B.rnd(rng, np.complex128, *dims, 3)
    y0 = np.full(dims + [3], np.nan, np.complex128)
    sb.clearCaches()
    before = sb.liveAllocations()
    h, _, keep = create(op, 0, 1, None, False)
    _, want = one_rank_call(op, h, x, y0, False, False)
    sb.sync(sb.createGpuContext(0))
    h.destroy()

    h, q, keep = create(op, 0, 1, None, True)
    with pytest.raises(RuntimeError, match="^destroy_bsr: .*request"):
        h.destroy()
    assert h.handle
    q.wait()
    req, got = one_rank_call(op, h, x, y0, False, True)
    with pytest.raises(RuntimeError, match="^destroy_bsr: .*request"):
        h.destroy()
    req.wait()
    h.destroy()
    sb.sync(sb.createGpuContext(0))
    assert np.array_equal(got.cpu().numpy().view(np.uint8), want.cpu().numpy().view(np.uint8))
    del got, want, keep
    sb.clearCaches()
    assert sb.liveAllocations() == before


def raw_progress(q):
    """sbb_request_progress on the request's handle, which stays with the caller on an error -> (rc, message)"""
    done = ctypes.c_int(0)
    rc = lib().sbb_request_progress(q.handle, ctypes.byref(done))
    return rc, lib().sbb_last_error().decode() if rc else ""


def fail_twice_then_release(q, name):
    """The first progress returns the step's own error, the second "<name>: the request failed"; the wait
    releases the request"""
    rc, first = raw_progress(q)
    assert rc == 1 and first.startswith("loopback communicators: every rank must begin"), first
    assert raw_progress(q) == (1, name + ": the request failed")
    h, q.handle, q._keep = q.handle, None, None
    assert lib().sbb_request_wait(h) == 1
    assert lib().sbb_last_error().decode() == name + ": the request failed"


def test_a_failed_dense_request_stays_failed():
    """A gathering cholesky on two loopback ranks, stepped on one before the other has begun"""
    rng = np.random.default_rng(61)
    o = "xcCsS"
    a = D.well_conditioned(rng, "cholesky", whole(SIZES, o), o, "cs", "CS", sb.FastToSlow, np.complex128)
    pa = cut(list(a.shape), o.index("c"), 2)
    sb.clearCaches()
    before = sb.liveAllocations()
    comms = sb.comm_create_local(2)
    try:
        bufs, ctx = place(D.components(a, pa, sb.FastToSlow))
        q = sb.cholesky(pa, 1, o, bufs[:1], "cs", "CS", ctx[:1], sb.FastToSlow, comm=comms[0], request=True)
        fail_twice_then_release(q, "cholesky")
    finally:
        for c in comms:
            c.destroy()
    sb.sync(sb.createGpuContext(0))
    del bufs
    sb.clearCaches()
    assert sb.liveAllocations() == before


def test_a_failed_bsr_krylov_request_stays_failed():
    """bsr_krylov of an operator cut over two loopback ranks, stepped on one before the other has begun; the
    operator can be destroyed once the failed request is released"""
    rng = np.random.default_rng(62)
    dims = [2, 2, 2, 2, 8]
    op1 = plain_stencil(rng, np.float64, dims)
    op = split_op(op1, split(dims, 4, [4]))
    x, ox, y0, oy = operands(rng, op1, np.float64, 1, None, 0)
    px, py = split(list(x.shape), 4, [4]), split(list(y0.shape), 4, [4])
    sb.clearCaches()
    before = sb.liveAllocations()
    comms = sb.comm_create_local(2)
    gpu = sb.createGpuContext(0)
    try:
        made = [create(op, r, 1, comms[r], True) for r in range(2)]
        rounds([q for _, q, _ in made])
        xs = [dev(c) for c in B.components(x, px, op["co"])]
        ys = [dev(c) for c in B.components(y0, py, op["co"])]
        q = sb.bsr_krylov(1, made[0][0], op["oim"], op["odom"], px, 1, ox, [0] * len(ox), list(x.shape),
                          list(x.shape), xs[:1], gpu, 0, py, oy, [0] * len(oy), list(y0.shape), list(y0.shape), None,
                          ys[:1], gpu, op["co"], comm=comms[0], ncomponentsy=1, request=True)
        with pytest.raises(RuntimeError, match="^destroy_bsr: "):
            made[0][0].destroy()
        fail_twice_then_release(q, "bsr_krylov")
        for h, _, _ in made:
            h.destroy()
    finally:
        for c in comms:
            c.destroy()
    sb.sync(gpu)
    del xs, ys, made
    sb.clearCaches()
    assert sb.liveAllocations() == before
