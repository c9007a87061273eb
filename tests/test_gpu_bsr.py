"""Block-sparse operators (create_bsr / bsr_krylov / destroy_bsr) on the GPU through the C ABI, against
the oracle of tests/bsr_cases.py."""
import os
import subprocess

import numpy as np
import pytest
import torch

import superbblas_b200 as sb
from tests import bsr_cases as B

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
DTYPES = [np.float32, np.float64, np.complex64, np.complex128]


def single(dims):
    return np.array([[[0] * len(dims), list(dims)]], dtype=np.int32)


def split(dims, k, cuts):
    """Parts of a whole tensor cut along dimension k at `cuts`"""
    edges = [0] + list(cuts) + [dims[k]]
    out = []
    for a, b in zip(edges[:-1], edges[1:]):
        f, s = [0] * len(dims), list(dims)
        f[k], s[k] = a, b - a
        out.append([f, s])
    return np.array(out, dtype=np.int32)


def dev(a, host=False):
    return a.copy() if host else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run(op, x, ox, px, y0, oy, py, alpha, beta, power=None, fromy=None, sizey=None, host=(), calls=1,
        update=None):
    """create_bsr from op = dict(ops, pim, dimi, dimd, blockim, blockdom, imfast, co, oim, odom), one or
    more bsr_krylov calls, destroy; -> y as a whole tensor"""
    co, ncomp = op["co"], len(op["pim"])
    gpu, cpu = sb.createGpuContext(0), sb.createCpuContext()
    hostop = "op" in host
    ii = [dev(o[0], hostop) for o in op["ops"]]
    jj = [dev(o[1].reshape(-1), hostop) for o in op["ops"]]
    v = [dev(o[2], hostop) for o in op["ops"]]
    h = sb.create_bsr(op["pim"], op["dimi"], op["pim_dom"], op["dimd"], ncomp, op["blockim"], op["blockdom"],
                      op["imfast"], ii, jj, v, cpu if hostop else gpu, co)
    del ii, jj  # read during create_bsr only
    xs = [dev(c, "x" in host) for c in B.components(x, px, co)]
    ys = [dev(c, "y" in host) for c in B.components(y0, py, co)]
    fromy = [0] * len(oy) if fromy is None else fromy
    sizey = list(y0.shape) if sizey is None else sizey
    for k in range(calls):
        if update is not None and k > 0:
            update(v)
        sb.bsr_krylov(alpha, h, op["oim"], op["odom"], px, len(xs), ox, [0] * len(ox), list(x.shape),
                      list(x.shape), xs, cpu if "x" in host else gpu, beta, py, oy, fromy, sizey, list(y0.shape),
                      power, ys, cpu if "y" in host else gpu, co)
    sb.sync(gpu)
    h.destroy()
    got = [c if isinstance(c, np.ndarray) else c.cpu().numpy() for c in ys]
    return B.assemble(got, py, y0, co)


def make_op(rng, dtype, co, imfast, pim, dimi, dimd, blockim, blockdom, oim, odom, ops=None):
    ops = ops if ops is not None else B.random_operator(rng, pim, blockim, dimd, blockdom, dtype)
    pim_dom = np.array([[[0] * len(dimd), list(dimd)]] * len(pim), dtype=np.int32)
    return dict(ops=ops, pim=np.asarray(pim, dtype=np.int32), pim_dom=pim_dom, dimi=dimi, dimd=dimd,
                blockim=blockim, blockdom=blockdom, imfast=imfast, co=co, oim=oim, odom=odom)


def want(op, x, ox, y0, oy, alpha, beta, power=None, psize=1, fromy=None):
    a = B.operator_matrix(op["ops"], op["pim"], op["dimi"], op["dimd"], op["blockim"], op["blockdom"],
                          op["imfast"], op["co"])
    return B.apply(a, op["oim"], op["odom"], x, ox, y0, oy, alpha, beta, power, psize, fromy)


def check(got, w, dtype):
    err = B.rel_err(got, w)
    assert err < B.TOL[np.dtype(dtype)], err


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("co", [sb.FastToSlow, sb.SlowToFast])
@pytest.mark.parametrize("imfast", [True, False])
def test_rectangular_operator(dtype, co, imfast):
    """A prolongator-shaped operator: 2 image labels, 3 domain labels, different block sizes; ragged and
    empty rows; periodic jj; beta = 0 over a NaN-filled y, then beta != 0"""
    rng = np.random.default_rng(1)
    dimi, dimd = [4, 6], [6, 4, 2]
    op = make_op(rng, dtype, co, imfast, single(dimi), dimi, dimd, [2, 3], [3, 2, 1], "ab", "cde")
    x = B.rnd(rng, dtype, 6, 3, 4, 2)                      # "cgde": column label g
    y0 = np.full((3, 4, 6), np.nan, dtype)                 # "gab"
    alpha = 0.5 - 1j if np.dtype(dtype).kind == "c" else 0.5
    got = run(op, x, "cgde", single(x.shape), y0, "gab", single(y0.shape), alpha, 0)
    check(got, want(op, x, "cgde", y0, "gab", alpha, 0), dtype)
    y1 = B.rnd(rng, dtype, 3, 4, 6)
    got = run(op, x, "cgde", single(x.shape), y1, "gab", single(y1.shape), alpha, 2)
    check(got, want(op, x, "cgde", y1, "gab", alpha, 2), dtype)


def test_spin_colour_stencil_on_8_4_lattice():
    """12 x 12 blocks, periodic 9-point stencil on an 8^4 lattice, 3 columns"""
    rng = np.random.default_rng(2)
    dims = [12, 8, 8, 8, 8]
    co = sb.FastToSlow
    pim = single(dims)
    ops = B.stencil_operator(rng, pim, dims, [12, 1, 1, 1, 1], np.complex128, co)
    op = make_op(rng, np.complex128, co, True, pim, dims, dims, [12, 1, 1, 1, 1], [12, 1, 1, 1, 1], "sxyzt",
                 "SXYZT", ops)
    x = B.rnd(rng, np.complex128, 12, 8, 8, 8, 8, 3)        # "SXYZTn"
    y0 = np.full((12, 8, 8, 8, 8, 3), np.nan, np.complex128)
    got = run(op, x, "SXYZTn", single(x.shape), y0, "sxyztn", single(y0.shape), 1, 0)
    check(got, want(op, x, "SXYZTn", y0, "sxyztn", 1, 0), np.complex128)


@pytest.mark.parametrize("ncols", [1, 8, 64])
def test_large_blocks(ncols):
    """64 x 64 blocks (the CTA tier), 1, 8 and 64 columns"""
    rng = np.random.default_rng(3)
    dims = [64 * 12]
    op = make_op(rng, np.complex128, sb.FastToSlow, False, single(dims), dims, dims, [64], [64], "a", "b")
    x = B.rnd(rng, np.complex128, ncols, dims[0])           # "nb"
    y0 = B.rnd(rng, np.complex128, dims[0], ncols)          # "an"
    got = run(op, x, "nb", single(x.shape), y0, "an", single(y0.shape), 1.5, -0.5)
    check(got, want(op, x, "nb", y0, "an", 1.5, -0.5), np.complex128)
    plan = sb.bsr_plan(sb.C128, op["pim"], dims, op["pim_dom"], dims, 1, [64], [64], False,
                       *B.flat_arrays(op["ops"]), "a", "b", single(x.shape), 1, "nb", [0, 0], list(x.shape),
                       list(x.shape), single(y0.shape), 1, "an", [0, 0], list(y0.shape), list(y0.shape), None,
                       sb.FastToSlow, 1, 0)
    assert "tier=cta" in plan["items"][0]["kernel"]


def test_powers():
    """P = 3: y_p = A y_{p-1}, starting from x; the power range starts at 1 of 4"""
    rng = np.random.default_rng(4)
    dims = [6, 4]
    op = make_op(rng, np.complex128, sb.SlowToFast, True, single(dims), dims, dims, [3, 2], [3, 2], "ab", "cd")
    x = B.rnd(rng, np.complex128, 2, 6, 4)                  # "ncd"
    y0 = B.rnd(rng, np.complex128, 4, 6, 4, 2)              # "pabn"
    fromy, sizey = [1, 0, 0, 0], [3, 6, 4, 2]
    got = run(op, x, "ncd", single(x.shape), y0, "pabn", single(y0.shape), 0.7, 0.3, "p", fromy, sizey)
    check(got, want(op, x, "ncd", y0, "pabn", 0.7, 0.3, "p", 3, fromy), np.complex128)


def test_host_components_and_a_y_partition_unlike_pim():
    rng = np.random.default_rng(5)
    dimi, dimd = [4, 6], [6, 4]
    pim = split(dimi, 0, [2])
    op = make_op(rng, np.complex128, sb.FastToSlow, True, pim, dimi, dimd, [2, 3], [3, 2], "ab", "cd")
    x = B.rnd(rng, np.complex128, 6, 4, 5)                  # "cdn"
    px = split(list(x.shape), 2, [3])
    y0 = B.rnd(rng, np.complex128, 5, 4, 6)                 # "nab"
    py = split(list(y0.shape), 2, [1])                      # cut along b, unlike pim
    plan = sb.bsr_plan(sb.C128, op["pim"], dimi, op["pim_dom"], dimd, 2, [2, 3], [3, 2], True,
                       *B.flat_arrays(op["ops"]), "ab", "cd", px, 2, "cdn", [0] * 3, list(x.shape),
                       list(x.shape), py, 2, "nab", [0] * 3, list(y0.shape), list(y0.shape), None,
                       sb.FastToSlow, 1, 0)
    assert plan["direct"] == 0
    for host in [(), ("op", "x", "y")]:
        got = run(op, x, "cdn", px, y0, "nab", py, 1, 0.5, host=host)
        check(got, want(op, x, "cdn", y0, "nab", 1, 0.5), np.complex128)


@pytest.mark.parametrize("dtype", [np.float32, np.complex128])
def test_results_are_bit_identical_over_components(dtype):
    """The same operator, x and y split over 1, 2, 4 and 8 components: y identical bit for bit (direct
    writes and write-backs alike)"""
    rng = np.random.default_rng(6)
    dims = [4, 8, 8]
    bl = [4, 1, 1]
    one = single(dims)
    ops1 = B.random_operator(rng, one, bl, dims, bl, dtype)
    ii, jj, v = ops1[0]
    x = B.rnd(rng, dtype, 4, 8, 8, 3)
    y0 = B.rnd(rng, dtype, 4, 8, 8, 3)
    results = []
    for n in (1, 2, 4, 8):
        pim = split(dims, 2, list(range(8 // n, 8, 8 // n)))
        # the rows of each part: its slice of the one-part arrays (rows numbered x fastest, then y, z)
        rows_per = 8 * 8 // n
        ptr = np.concatenate([[0], np.cumsum(ii)])
        bsz = 16
        parts = []
        for k in range(n):
            r0, r1 = k * rows_per, (k + 1) * rows_per
            parts.append((ii[r0:r1], jj[ptr[r0]:ptr[r1]], v[ptr[r0] * bsz:ptr[r1] * bsz]))
        op = make_op(rng, dtype, sb.FastToSlow, True, pim, dims, dims, bl, bl, "abc", "ABC", parts)
        px = split(list(x.shape), 1, [3, 5])[: 3]
        for py in (split(list(y0.shape), 2, list(range(8 // n, 8, 8 // n))), single(y0.shape)):
            results.append(run(op, x, "ABCn", px, y0, "abcn", py, 1.25, 0.5))
    check(results[0], want(make_op(rng, dtype, sb.FastToSlow, True, one, dims, dims, bl, bl, "abc", "ABC", ops1),
                           x, "ABCn", y0, "abcn", 1.25, 0.5), dtype)
    for r in results[1:]:
        assert np.array_equal(r.view(np.uint8), results[0].view(np.uint8))


def test_v_updated_between_calls_and_no_leak():
    rng = np.random.default_rng(7)
    dims = [6, 4]
    op = make_op(rng, np.float64, sb.FastToSlow, True, single(dims), dims, dims, [3, 2], [3, 2], "ab", "cd")
    x = B.rnd(rng, np.float64, 6, 4, 2)
    y0 = np.zeros((6, 4, 2))
    sb.clearCaches()
    before = sb.liveAllocations()

    def update(v):
        for t in v:
            t.mul_(2)
    got = run(op, x, "cdn", single(x.shape), y0, "abn", single(y0.shape), 1, 0, calls=2, update=update)
    op2 = dict(op, ops=[(o[0], o[1], o[2] * 2) for o in op["ops"]])
    check(got, want(op2, x, "cdn", y0, "abn", 1, 0), np.float64)
    sb.clearCaches()
    assert sb.liveAllocations() == before


def test_errors():
    dims = [4, 4]
    gpu = sb.createGpuContext(0)
    pim = single(dims)
    ii = torch.tensor([1, 0, 0, 0], dtype=torch.int32, device="cuda")
    bad = torch.tensor([1, 0], dtype=torch.int32, device="cuda")        # not a multiple of blockdom
    v = torch.zeros(16, dtype=torch.float64, device="cuda")
    with pytest.raises(RuntimeError, match="not a multiple of blockdom"):
        sb.create_bsr(pim, dims, pim, dims, 1, [2, 2], [2, 2], True, [ii], [bad], [v], gpu, sb.FastToSlow)
    with pytest.raises(RuntimeError, match="multiples of blockim"):
        sb.create_bsr(np.array([[[1, 0], [3, 4]]], np.int32), dims, pim, dims, 1, [2, 2], [2, 2], True, [ii],
                      [bad], [v], gpu, sb.FastToSlow)


def test_cxx_bsr_dropin_program(tmp_path):
    """tests/cxx/bsr_dropin_test.cpp, compiled against include/superbblas.h and the in-tree library into a
    temporary directory, and run."""
    root = os.path.dirname(HERE)
    lib = os.path.join(root, "superbblas_b200", "lib")
    exe = str(tmp_path / "bsr_dropin_test")
    r = subprocess.run([os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), "-std=c++17", "-O2", "-ccbin",
                        "/usr/bin/g++", "-I" + os.path.join(root, "include"),
                        os.path.join(HERE, "cxx", "bsr_dropin_test.cpp"), "-o", exe, "-L" + lib,
                        "-lsuperbblas_b200", "-Xlinker", "-rpath", "-Xlinker", lib],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Everything went ok!" in r.stdout
