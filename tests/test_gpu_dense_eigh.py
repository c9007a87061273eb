"""eigh, the batched Hermitian eigensolver, on the GPU through the C ABI: every type against
torch.linalg.eigvalsh in float64 within the bounds of tests/eigh_cases.py, per-site and Gram layouts,
the warp / CTA boundary and each type's limit, W partitioned and ordered unlike A, host components, the
gather path, determinism, errors, the workspace pool, the report, and the C++ drop-in program."""
import os
import subprocess

import numpy as np
import pytest
import torch

import superbblas_b200 as sb
from tests import dense_cases as D
from tests import eigh_cases as E

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
DTYPES = [np.float32, np.float64, np.complex64, np.complex128]


def single(dims):
    return np.array([[[0] * len(dims), list(dims)]], dtype=np.int32)


def place(comps, host=()):
    gpu, cpu = sb.createGpuContext(0), sb.createCpuContext()
    bufs = [c.copy() if i in host else torch.from_numpy(c).cuda() for i, c in enumerate(comps)]
    return bufs, [cpu if i in host else gpu for i in range(len(comps))]


def back(bufs):
    return [b if isinstance(b, np.ndarray) else b.cpu().numpy() for b in bufs]


def w_order(o, orows, ocols, co):
    """The labels of W in the order of as_matrices' batch and eigenvalue axes"""
    return [c for c in o if c not in orows + ocols] + list(ocols if co == sb.SlowToFast else ocols[::-1])


def run_eigh(a, o, orows, ocols, ow, co, pa=None, pw=None, host_a=(), host_w=()):
    """-> (A after the call, W) as whole tensors"""
    dims = dict(zip(o, a.shape))
    wdims = [dims[c] for c in ow]
    pa = single(a.shape) if pa is None else pa
    pw = single(wdims) if pw is None else pw
    ba, ca = place(D.components(a, pa, co), host_a)
    w0 = np.full(wdims, np.nan, E.REAL[a.dtype])
    bw, cw = place(D.components(w0, pw, co), host_w)
    sb.eigh(pa, len(ba), o, ba, orows, ocols, ca, pw, len(bw), ow, bw, cw, co)
    sb.sync(sb.createGpuContext(0))
    return D.assemble(back(ba), pa, np.full(a.shape, np.nan, a.dtype), co), D.assemble(back(bw), pw, w0, co)


def check(h, a_out, w_out, o, orows, ocols, ow, co, dtype):
    _, v = D.as_matrices(a_out, o, orows, ocols, co)
    w = np.transpose(w_out, [ow.index(c) for c in w_order(o, orows, ocols, co)]).reshape(v.shape[:-1])
    wref = torch.linalg.eigvalsh(torch.from_numpy(np.asarray(h))).numpy()
    assert np.allclose(np.linalg.eigvalsh(h), wref, rtol=0, atol=1e-12 * max(1, np.abs(wref).max(initial=0)))
    E.check(h, w, v, dtype)


def case(rng, dtype, sizes, o, orows, ocols, co, kind="random"):
    """A random Hermitian matrix tensor -> (tensor in dtype, its matrices [batch..., n, n])"""
    shape = [sizes[c] for c in o]
    _, m = D.as_matrices(np.zeros(shape), o, orows, ocols, co)
    h = E.hermitian(rng, dtype, m.shape[-1], kind, m.shape[:-2])
    return D.from_matrices(h, o, shape, orows, ocols, co).astype(dtype), h


SITE = dict(x=4, y=4, z=4, t=8, c=3, C=3, s=4, S=4)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("o,orows,ocols,ow", [
    ("xyztcC", "c", "C", "Cxyzt"),            # 3x3 per link / site, batch slowest
    ("cCxyzt", "c", "C", "xyztC"),            # batch fastest
    ("xyztcsCS", "cs", "CS", "SCtzyx"),       # 12x12 spin-colour, rows and columns over two labels
    ("csCSxyzt", "cs", "CS", "xyztCS"),
])
@pytest.mark.parametrize("co", [sb.FastToSlow, sb.SlowToFast])
def test_per_site_blocks(dtype, o, orows, ocols, ow, co):
    rng = np.random.default_rng(1)
    a, h = case(rng, dtype, SITE, o, orows, ocols, co)
    got_a, got_w = run_eigh(a, o, orows, ocols, ow, co)
    check(h, got_a, got_w, o, orows, ocols, ow, co, dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [32, 33, 64, "limit"])
def test_orders_across_the_tiers(dtype, n):
    n = E.LIMIT[np.dtype(dtype)] if n == "limit" else n
    rng = np.random.default_rng(n)
    sizes = dict(b=16 if n == 64 else 3, r=n, c=n)
    a, h = case(rng, dtype, sizes, "rcb", "r", "c", sb.FastToSlow)
    got_a, got_w = run_eigh(a, "rcb", "r", "c", "cb", sb.FastToSlow)
    check(h, got_a, got_w, "rcb", "r", "c", "cb", sb.FastToSlow, dtype)


@pytest.mark.parametrize("kind", ["repeated", "graded", "zero", "diagonal"])
def test_special_spectra(kind):
    rng = np.random.default_rng(3)
    a, h = case(rng, np.complex128, dict(b=8, r=12, c=12), "brc", "r", "c", sb.FastToSlow, kind)
    got_a, got_w = run_eigh(a, "brc", "r", "c", "bc", sb.FastToSlow)
    check(h, got_a, got_w, "brc", "r", "c", "bc", sb.FastToSlow, np.complex128)


def test_gram_batch():
    """V^H V of a block of 64 vectors per time slice, by contraction, then its eigen-decomposition"""
    rng = np.random.default_rng(4)
    nv, m, nt = 2000, 64, 8
    v = torch.from_numpy(rng.standard_normal(nv * m * nt) + 1j * rng.standard_normal(nv * m * nt)).cuda()
    g = torch.zeros(m * m * nt, dtype=torch.complex128, device="cuda")
    gpu = sb.createGpuContext(0)
    pv, pg = single([nv, m, nt]), single([m, m, nt])
    sb.contraction(1, pv, [0] * 3, [nv, m, nt], [nv, m, nt], 1, "iwt", True, [v], gpu, pv, [0] * 3, [nv, m, nt],
                   [nv, m, nt], 1, "ivt", False, [v], gpu, 0, pg, [0] * 3, [m, m, nt], [m, m, nt], 1, "wvt", [g], gpu,
                   sb.FastToSlow)
    h = g.cpu().numpy().reshape((m, m, nt), order="F").transpose(2, 0, 1)
    up = np.triu(h, 1)                         # the matrix eigh reads: the upper triangle, real diagonal
    h = up + np.conj(np.swapaxes(up, -1, -2)) + np.einsum("...ii->...i", h).real[..., None] * np.eye(m)
    w = torch.zeros(m * nt, dtype=torch.float64, device="cuda")
    sb.eigh(pg, 1, "wvt", [g], "w", "v", gpu, single([nt, m]), 1, "tv", [w], gpu, sb.FastToSlow)
    sb.sync(gpu)
    vv = g.cpu().numpy().reshape((m, m, nt), order="F").transpose(2, 0, 1)
    E.check(h, w.cpu().numpy().reshape((nt, m), order="F"), vv, np.complex128)


@pytest.mark.parametrize("dtype,s", [(np.float32, 1e-23), (np.float32, 1e20), (np.complex64, 1e-30),
                                     (np.float64, 1e-170), (np.complex128, 1e160)])
def test_extreme_scales(dtype, s):
    """Finite matrices of any magnitude, in the warp and CTA tiers, within the relative bounds"""
    rng = np.random.default_rng(10)
    for n in (4, 40):
        a, h = case(rng, dtype, dict(b=5, r=n, c=n), "brc", "r", "c", sb.FastToSlow)
        a = (a.astype(np.complex128 if np.dtype(dtype).kind == "c" else np.float64) * s).astype(dtype)
        got_a, got_w = run_eigh(a, "brc", "r", "c", "bc", sb.FastToSlow)
        _, v = D.as_matrices(got_a, "brc", "r", "c", sb.FastToSlow)
        _, hs = D.as_matrices(a.astype(np.complex128) / s, "brc", "r", "c", sb.FastToSlow)
        E.check(hs, got_w.astype(np.float64) / s, v, dtype, s)


def split(dims, k, at):
    f0, s0 = [0] * len(dims), list(dims)
    f1, s1 = [0] * len(dims), list(dims)
    s0[k], f1[k], s1[k] = at, at, dims[k] - at
    return np.array([[f0, s0], [f1, s1]], dtype=np.int32)


def test_host_components():
    rng = np.random.default_rng(5)
    o, ow = "xcCy", "yCx"
    sizes = dict(x=4, y=3, c=5, C=5)
    a, h = case(rng, np.float64, sizes, o, "c", "C", sb.SlowToFast)
    pa = split([sizes[c] for c in o], 0, 2)
    pw = split([sizes[c] for c in ow], 2, 2)        # the same batch boxes: one launch writes A and W
    assert [i["writes"] for i in sb.dense_plan(sb.EIGH, sb.F64, pa, 2, o, "c", "C", sb.SlowToFast, 1, 0, py=pw,
                                               ncomponentsy=2, oy=ow)["items"]] == ["aw", "aw"]
    got_a, got_w = run_eigh(a, o, "c", "C", ow, sb.SlowToFast, pa, pw, host_a=(1,), host_w=(0,))
    check(h, got_a, got_w, o, "c", "C", ow, sb.SlowToFast, np.float64)


def test_gather_with_w_partitioned_differently():
    """A split along a row label (gathered), W split along a batch label and along a column label"""
    rng = np.random.default_rng(6)
    o, ow = "xcsCS", "SxC"
    sizes = dict(x=5, c=3, s=2, C=3, S=2)
    a, h = case(rng, np.complex128, sizes, o, "cs", "CS", sb.FastToSlow)
    pa = split([sizes[c] for c in o], o.index("c"), 1)
    for k in ("x", "C"):
        pw = split([sizes[c] for c in ow], ow.index(k), 1)
        plan = sb.dense_plan(sb.EIGH, sb.C128, pa, 2, o, "cs", "CS", sb.FastToSlow, 1, 0, py=pw, ncomponentsy=2, oy=ow)
        assert plan["gather_a"] == 1 and "w" in [i["writes"] for i in plan["items"]]
        got_a, got_w = run_eigh(a, o, "cs", "CS", ow, sb.FastToSlow, pa, pw, host_w=(1,))
        check(h, got_a, got_w, o, "cs", "CS", ow, sb.FastToSlow, np.complex128)


def test_deterministic_and_replicated_bits():
    rng = np.random.default_rng(7)
    o, ow = "cCx", "xC"
    sizes = dict(x=40, c=20, C=20)
    a, h = case(rng, np.complex64, sizes, o, "c", "C", sb.FastToSlow)
    r1 = run_eigh(a, o, "c", "C", ow, sb.FastToSlow)
    r2 = run_eigh(a, o, "c", "C", ow, sb.FastToSlow)
    assert all(np.array_equal(x, y, equal_nan=True) for x, y in zip(r1, r2))
    # two replicated components of A and of W, and W on a third part that no launch of A serves
    dims = [sizes[c] for c in o]
    pa = np.array([[[0] * 3, dims]] * 2, dtype=np.int32)
    pw = np.array([[[0, 0], [40, 20]], [[0, 0], [40, 20]], [[10, 0], [5, 20]]], dtype=np.int32)
    ba, ca = place(D.components(a, pa, sb.FastToSlow))
    bw, cw = place([np.zeros(int(np.prod(s)), np.float32) for _, s in pw])
    sb.eigh(pa, 2, o, ba, "c", "C", ca, pw, 3, ow, bw, cw, sb.FastToSlow)
    sb.sync(sb.createGpuContext(0))
    ba, bw = back(ba), back(bw)
    assert np.array_equal(ba[0], ba[1]) and np.array_equal(bw[0], bw[1])
    assert np.array_equal(ba[0], D.components(r1[0], single(dims), sb.FastToSlow)[0])
    assert np.array_equal(bw[0], r1[1].ravel(order="F"))
    assert np.array_equal(bw[2], r1[1][10:15].ravel(order="F"))


def test_errors_and_workspaces():
    sb.clearCaches()
    before = sb.liveAllocations()
    rng = np.random.default_rng(8)
    for dtype in DTYPES:
        n = E.LIMIT[np.dtype(dtype)] + 1
        with pytest.raises(RuntimeError, match="eigh: order n = %d is over the limit" % n):
            run_eigh(np.zeros((n, n), dtype), "rc", "r", "c", "c", sb.FastToSlow)
    with pytest.raises(RuntimeError, match="eigh: w lacks the batch label `b`"):
        run_eigh(np.zeros((2, 3, 3)), "brc", "r", "c", "c", sb.FastToSlow)
    a, h = case(rng, np.float64, dict(b=3, r=5, c=5), "brc", "r", "c", sb.FastToSlow)
    run_eigh(a, "brc", "r", "c", "cb", sb.FastToSlow, pa=split([3, 5, 5], 1, 2), pw=split([5, 3], 0, 1))
    sb.clearCaches()
    assert sb.liveAllocations() == before


def test_non_finite_matrix_gives_nan():
    a = np.eye(4)[None].repeat(2, 0)
    a[1, 0, 3] = np.nan
    a[0, 3, 0] = np.nan                        # strictly lower: not read
    got_a, got_w = run_eigh(a, "brc", "r", "c", "bc", sb.FastToSlow)
    assert np.array_equal(got_w[0], np.ones(4)) and np.array_equal(got_a[0], np.eye(4))
    assert np.all(np.isnan(got_w[1])) and np.all(np.isnan(got_a[1]))


def test_report_has_an_eigh_line():
    rng = np.random.default_rng(9)
    a, _ = case(rng, np.complex128, dict(b=10, r=6, c=6), "brc", "r", "c", sb.FastToSlow)
    sb.trackTime(True)
    sb.resetTimings()
    try:
        run_eigh(a, "brc", "r", "c", "bc", sb.FastToSlow)
        t = sb.timings()
        assert t["eigh"]["calls"] == 1 and t["eigh"]["flops"] == 0
        assert t["eigh"]["bytes"] == 10 * (2 * 36 * 16 + 6 * 8)
        assert any(line.startswith("eigh") for line in sb.reportTimings().splitlines())
    finally:
        sb.trackTime(False)
        sb.resetTimings()


def test_cxx_eigh_dropin_program(tmp_path):
    """tests/cxx/dense_eigh_dropin_test.cpp, compiled against include/superbblas.h and the in-tree library
    into a temporary directory, and run."""
    root = os.path.dirname(HERE)
    lib = os.path.join(root, "superbblas_b200", "lib")
    exe = str(tmp_path / "dense_eigh_dropin_test")
    r = subprocess.run([os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), "-std=c++17", "-O2", "-ccbin",
                        "/usr/bin/g++", "-I" + os.path.join(root, "include"),
                        os.path.join(HERE, "cxx", "dense_eigh_dropin_test.cpp"), "-o", exe, "-L" + lib,
                        "-lsuperbblas_b200", "-Xlinker", "-rpath", "-Xlinker", lib],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Everything went ok!" in r.stdout
