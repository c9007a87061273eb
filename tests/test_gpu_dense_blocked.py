"""The blocked tier of cholesky and trsm on the GPU (matrices over one CTA's shared memory), against
the numpy oracle of tests/dense_cases.py."""
import numpy as np
import pytest
import torch

import superbblas_b200 as sb
from tests import dense_cases as D
from tests.test_gpu_dense import check, run_solve, run_square, single, split, whole

pytestmark = pytest.mark.gpu
# just over the limit of each type, with its rows and columns split over two labels
OVER = {np.float32: 227, np.float64: 161, np.complex64: 161, np.complex128: 114}
FACTORS = {114: (6, 19), 161: (7, 23), 227: (227, 1), 300: (12, 25), 1000: (40, 25)}


def sizes(n, **kw):
    c, s = FACTORS[n]
    return {**dict(x=2, y=2, c=c, s=s, C=c, S=s, r=300), **kw}


def rhs_of(rng, shape, dtype):
    x = rng.standard_normal(shape)
    if np.dtype(dtype).kind == "c":
        x = x + 1j * rng.standard_normal(shape)
    return x.astype(dtype)


def blocked_cases():
    for dtype, n in OVER.items():
        for m in (n, 300):
            yield dtype, m
    yield np.float64, 1000


@pytest.mark.parametrize("dtype,n", list(blocked_cases()))
@pytest.mark.parametrize("co", [sb.FastToSlow, sb.SlowToFast])
def test_cholesky_blocked_strided(dtype, n, co):
    rng = np.random.default_rng(n)
    sz = sizes(n, x=2 if n < 1000 else 1, y=2 if n < 1000 else 1)
    o = "xCcysS"     # batch labels x, y interleaved with the matrix labels
    a = D.well_conditioned(rng, "cholesky", whole(sz, o), o, "cs", "CS", co, dtype)
    plan = sb.dense_plan(sb.CHOLESKY, {np.float32: sb.F32, np.float64: sb.F64, np.complex64: sb.C64,
                                       np.complex128: sb.C128}[dtype], single(a.shape), 1, o, "cs", "CS", co, 1, 0)
    assert "tier=blocked" in plan["items"][0]["kernel"]
    got = run_square("cholesky", a, o, "cs", "CS", co)
    check(got, D.oracle("cholesky", a, o, "cs", "CS", co), dtype)


@pytest.mark.parametrize("dtype,n", list(blocked_cases()))
@pytest.mark.parametrize("co", [sb.FastToSlow, sb.SlowToFast])
@pytest.mark.parametrize("left", [True, False])
def test_trsm_blocked_strided(dtype, n, co, left):
    rng = np.random.default_rng(n + 1)
    sz = sizes(n, x=2 if n < 1000 else 1, y=2 if n < 1000 else 1)
    o = "xCcysS"
    a = D.well_conditioned(rng, "trsm", whole(sz, o), o, "cs", "CS", co, dtype)
    ox, oy = ("sryxc", "yCSrx") if left else ("SryxC", "ycsrx")
    x = rhs_of(rng, whole(sz, ox), dtype)
    ydims = whole(sz, oy)
    alpha = 0.5 - 1j if np.dtype(dtype).kind == "c" else 0.5
    got = run_solve("trsm", alpha, a, o, "cs", "CS", x, ox, ydims, oy, co)
    check(got, D.oracle("trsm", a, o, "cs", "CS", co, alpha, x, ox, oy, ydims), dtype)


def test_cholesky_blocked_split_and_host_components():
    rng = np.random.default_rng(11)
    sz = sizes(300)
    o = "xcCsS"
    dims = whole(sz, o)
    a = D.well_conditioned(rng, "cholesky", dims, o, "cs", "CS", sb.FastToSlow, np.complex128)
    parts = split(dims, o.index("c"), 5)
    assert sb.dense_plan(sb.CHOLESKY, sb.C128, parts, 2, o, "cs", "CS", sb.FastToSlow, 1, 0)["gather_a"] == 1
    got = run_square("cholesky", a, o, "cs", "CS", sb.FastToSlow, parts=parts, host=(1,))
    check(got, D.oracle("cholesky", a, o, "cs", "CS", sb.FastToSlow), np.complex128)


@pytest.mark.parametrize("left", [True, False])
def test_trsm_blocked_split_and_host_components(left):
    rng = np.random.default_rng(12)
    sz = sizes(300)
    o = "xcCsS"
    ox, oy = ("xrcs", "xCrS") if left else ("xrCS", "xcrs")
    a = D.well_conditioned(rng, "trsm", whole(sz, o), o, "cs", "CS", sb.SlowToFast, np.complex128)
    x = rhs_of(rng, whole(sz, ox), np.complex128)
    ydims = whole(sz, oy)
    pa = split(whole(sz, o), o.index("C"), 4)
    px = split(whole(sz, ox), 1, 100)
    py = split(ydims, 3, 10)
    got = run_solve("trsm", 1, a, o, "cs", "CS", x, ox, ydims, oy, sb.SlowToFast, pa, px, py, host=(0,))
    check(got, D.oracle("trsm", a, o, "cs", "CS", sb.SlowToFast, 1, x, ox, oy, ydims), np.complex128)


def test_nan_below_the_diagonal_is_not_read():
    rng = np.random.default_rng(13)
    n = 300
    o = "xab"       # rows a, columns b
    a = D.well_conditioned(rng, "cholesky", [2, n, n], o, "a", "b", sb.FastToSlow, np.complex128)
    bad = a.copy()
    bad[:, np.tri(n, k=-1, dtype=bool)] = np.nan     # [x, row, col] with row > col
    got = run_square("cholesky", bad, o, "a", "b", sb.FastToSlow)
    assert np.all(np.isfinite(got))
    check(got, D.oracle("cholesky", a, o, "a", "b", sb.FastToSlow), np.complex128)
    x = rhs_of(rng, [2, n, 40], np.complex128)
    for ox, oy in (("xar", "xbr"), ("xbr", "xar")):
        y = run_solve("trsm", 1, bad, o, "a", "b", x, ox, [2, n, 40], oy, sb.FastToSlow)
        assert np.all(np.isfinite(y))
        check(y, D.oracle("trsm", a, o, "a", "b", sb.FastToSlow, 1, x, ox, oy, [2, n, 40]), np.complex128)


def test_blocked_results_are_deterministic():
    rng = np.random.default_rng(14)
    sz = sizes(300)
    o = "xcCsS"
    dims = whole(sz, o)
    a = D.well_conditioned(rng, "cholesky", dims, o, "cs", "CS", sb.FastToSlow, np.complex128)
    one = run_square("cholesky", a, o, "cs", "CS", sb.FastToSlow)
    assert np.array_equal(one, run_square("cholesky", a, o, "cs", "CS", sb.FastToSlow))
    two = run_square("cholesky", a, o, "cs", "CS", sb.FastToSlow, parts=split(dims, 0, 1))
    assert np.array_equal(one, two)
    ox, oy = "xrCS", "xcrs"
    x = rhs_of(rng, whole(sz, ox), np.complex128)
    ydims = whole(sz, oy)
    y1 = run_solve("trsm", 1, a, o, "cs", "CS", x, ox, ydims, oy, sb.FastToSlow)
    assert np.array_equal(y1, run_solve("trsm", 1, a, o, "cs", "CS", x, ox, ydims, oy, sb.FastToSlow))
    y2 = run_solve("trsm", 1, a, o, "cs", "CS", x, ox, ydims, oy, sb.FastToSlow, px=split(whole(sz, ox), 1, 7),
                   py=split(ydims, 1, 7))
    assert np.array_equal(y1, y2)


def test_orthonormalisation_chain_n128():
    """configs[3]'s basis at a reduced lattice: per time slice t, G = V^H V by contraction,
    U = cholesky(G) and Q = V U^-1 by trsm; Q^H Q = I and Q spans V for every t."""
    rng = np.random.default_rng(15)
    nv, m, nt = 6000, 128, 3
    v = rng.standard_normal((nv, m, nt)) + 1j * rng.standard_normal((nv, m, nt))
    gpu = sb.createGpuContext(0)
    vt = torch.from_numpy(np.ascontiguousarray(v.ravel(order="F"))).cuda()    # "ivt", first label fastest
    g = torch.zeros(m * m * nt, dtype=torch.complex128, device="cuda")        # "wvt"
    pv, pg = single([nv, m, nt]), single([m, m, nt])
    sb.contraction(1, pv, [0] * 3, [nv, m, nt], [nv, m, nt], 1, "iwt", True, [vt], gpu, pv, [0] * 3,
                   [nv, m, nt], [nv, m, nt], 1, "ivt", False, [vt], gpu, 0, pg, [0] * 3, [m, m, nt],
                   [m, m, nt], 1, "wvt", [g], gpu, sb.FastToSlow)
    sb.cholesky(pg, 1, "wvt", [g], "w", "v", gpu, sb.FastToSlow)
    q = torch.zeros_like(vt)
    sb.trsm(1, pg, 1, "wvt", "w", "v", [g], gpu, pv, 1, "ivt", [vt], gpu, pv, 1, "iwt", [q], gpu, sb.FastToSlow)
    sb.sync(gpu)
    qm = q.cpu().numpy().reshape((nv, m, nt), order="F")
    for t in range(nt):
        assert np.linalg.norm(qm[:, :, t].conj().T @ qm[:, :, t] - np.eye(m)) < 1e-10
        coef = np.linalg.lstsq(qm[:, :, t], v[:, :, t], rcond=None)[0]
        assert np.linalg.norm(qm[:, :, t] @ coef - v[:, :, t]) / np.linalg.norm(v[:, :, t]) < 1e-12


def test_blocked_workspaces_are_returned():
    rng = np.random.default_rng(16)
    n = 200
    a = D.well_conditioned(rng, "cholesky", [2, n, n], "xab", "a", "b", sb.FastToSlow, np.complex128)
    run_square("cholesky", a, "xab", "a", "b", sb.FastToSlow)
    before = sb.liveAllocations()
    run_square("cholesky", a, "xab", "a", "b", sb.FastToSlow)
    x = rhs_of(rng, [2, n, 30], np.complex128)
    run_solve("trsm", 1, a, "xab", "a", "b", x, "xar", [2, n, 30], "xbr", sb.FastToSlow)
    assert sb.liveAllocations() == before
    with pytest.raises(RuntimeError, match="dimension of label `r` does not match"):
        run_solve("trsm", 1, a, "xab", "a", "b", x, "xar", [2, n, 31], "xbr", sb.FastToSlow)
    assert sb.liveAllocations() == before
