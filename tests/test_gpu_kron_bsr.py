"""Kronecker block-sparse operators (create_kron_bsr / bsr_krylov / destroy_bsr) on the GPU through the C
ABI, against the oracle of tests/kron_bsr_cases.py and against create_bsr on the expanded blocks."""
import os
import subprocess

import numpy as np
import pytest
import torch

import superbblas_b200 as sb
from tests import bsr_cases as B
from tests import kron_bsr_cases as KB
from tests.test_gpu_bsr import single, split, dev, check

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
DTYPES = [np.float32, np.float64, np.complex64, np.complex128]


def make_op(ops, kronv, pim, dimi, dimd, blockim, blockdom, kronim, krondom, imfast, co, oim, odom):
    pim_dom = np.array([[[0] * len(dimd), list(dimd)]] * len(pim), dtype=np.int32)
    return dict(ops=ops, kronv=kronv, pim=np.asarray(pim, dtype=np.int32), pim_dom=pim_dom, dimi=dimi, dimd=dimd,
                blockim=blockim, blockdom=blockdom, kronim=kronim, krondom=krondom, imfast=imfast, co=co, oim=oim,
                odom=odom)


def run(op, x, ox, px, y0, oy, py, alpha, beta, power=None, fromy=None, sizey=None, host=(), calls=1, update=None,
        expanded=False):
    """create_kron_bsr (or create_bsr on the expanded blocks), one or more bsr_krylov calls, destroy -> y"""
    co, ncomp = op["co"], len(op["pim"])
    gpu, cpu = sb.createGpuContext(0), sb.createCpuContext()
    hostop = "op" in host
    ctx = cpu if hostop else gpu
    ii = [dev(o[0], hostop) for o in op["ops"]]
    jj = [dev(o[1].reshape(-1), hostop) for o in op["ops"]]
    if expanded:
        ex = KB.expand(op["ops"], op["kronv"], op["blockim"], op["blockdom"], op["kronim"], op["krondom"],
                       op["imfast"], co)
        v, kv = [dev(o[2], hostop) for o in ex], []
        h = sb.create_bsr(op["pim"], op["dimi"], op["pim_dom"], op["dimd"], ncomp,
                          KB.eff(op["blockim"], op["kronim"]), KB.eff(op["blockdom"], op["krondom"]), op["imfast"],
                          ii, jj, v, ctx, co)
    else:
        v = [dev(o[2], hostop) for o in op["ops"]]
        kv = [dev(op["kronv"], hostop) for _ in op["ops"]]       # every component its own copy
        h = sb.create_kron_bsr(op["pim"], op["dimi"], op["pim_dom"], op["dimd"], ncomp, op["blockim"],
                               op["blockdom"], op["kronim"], op["krondom"], op["imfast"], ii, jj, v, kv, ctx, co)
    del ii, jj
    xs = [dev(c, "x" in host) for c in B.components(x, px, co)]
    ys = [dev(c, "y" in host) for c in B.components(y0, py, co)]
    fromy = [0] * len(oy) if fromy is None else fromy
    sizey = list(y0.shape) if sizey is None else sizey
    for k in range(calls):
        if update is not None and k > 0:
            update(v, kv)
        sb.bsr_krylov(alpha, h, op["oim"], op["odom"], px, len(xs), ox, [0] * len(ox), list(x.shape),
                      list(x.shape), xs, cpu if "x" in host else gpu, beta, py, oy, fromy, sizey, list(y0.shape),
                      power, ys, cpu if "y" in host else gpu, co)
    sb.sync(gpu)
    h.destroy()
    got = [c if isinstance(c, np.ndarray) else c.cpu().numpy() for c in ys]
    return B.assemble(got, py, y0, co)


def want(op, x, ox, y0, oy, alpha, beta, power=None, psize=1, fromy=None):
    a = KB.oracle_matrix(op["ops"], op["kronv"], op["pim"], op["dimi"], op["dimd"], op["blockim"], op["blockdom"],
                         op["kronim"], op["krondom"], op["imfast"], op["co"])
    return B.apply(a, op["oim"], op["odom"], x, ox, y0, oy, alpha, beta, power, psize, fromy)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("co", [sb.FastToSlow, sb.SlowToFast])
@pytest.mark.parametrize("imfast", [True, False])
def test_rectangular_operator(dtype, co, imfast):
    """2 image labels, 3 domain labels; the factor on one label each (3 x 2), blocks of 2 x 3; periodic jj;
    beta = 0 over a NaN-filled y, then beta != 0"""
    rng = np.random.default_rng(11)
    dimi, dimd = [4, 6], [6, 4, 2]
    blockim, kronim, blockdom, krondom = [2, 1], [1, 3], [3, 1, 1], [1, 2, 1]
    pim = single(dimi)
    ops, kronv = KB.random_kron_operator(rng, pim, blockim, dimd, blockdom, kronim, krondom, 3, dtype)
    op = make_op(ops, kronv, pim, dimi, dimd, blockim, blockdom, kronim, krondom, imfast, co, "ab", "cde")
    x = B.rnd(rng, dtype, 6, 3, 4, 2)                      # "cgde": column label g
    y0 = np.full((3, 4, 6), np.nan, dtype)                 # "gab"
    alpha = 0.5 - 1j if np.dtype(dtype).kind == "c" else 0.5
    got = run(op, x, "cgde", single(x.shape), y0, "gab", single(y0.shape), alpha, 0)
    check(got, want(op, x, "cgde", y0, "gab", alpha, 0), dtype)
    y1 = B.rnd(rng, dtype, 3, 4, 6)
    got = run(op, x, "cgde", single(x.shape), y1, "gab", single(y1.shape), alpha, 2)
    check(got, want(op, x, "cgde", y1, "gab", alpha, 2), dtype)


def wilson(rng, dtype, pim, dims, co=sb.FastToSlow):
    """4 x 4 spin factors (one per direction) ⊗ 3 x 3 colour blocks, nine points, on "scxyzt" """
    blockim, kronim = [1, 3, 1, 1, 1, 1], [4, 1, 1, 1, 1, 1]
    ops = KB.kron_stencil(rng, pim, dims, blockim, kronim, KB.NINE_POINT, dtype, co)
    kronv = B.rnd(rng, dtype, 9 * 16)
    return make_op(ops, kronv, pim, dims, dims, blockim, blockim, kronim, kronim, True, co, "scxyzt", "SCXYZT")


@pytest.mark.parametrize("ncols", [1, 8, 12])
def test_nine_point_spin_colour_on_8_4(ncols):
    """The Wilson-shaped operator on 8^4: against the oracle and against create_bsr on the 12 x 12
    expanded blocks"""
    rng = np.random.default_rng(12)
    dims = [4, 3, 8, 8, 8, 8]
    op = wilson(rng, np.complex128, single(dims), dims)
    x = B.rnd(rng, np.complex128, *dims, ncols)             # "SCXYZTn"
    y0 = np.full(dims + [ncols], np.nan, np.complex128)
    got = run(op, x, "SCXYZTn", single(x.shape), y0, "scxyztn", single(y0.shape), 1, 0)
    w = want(op, x, "SCXYZTn", y0, "scxyztn", 1, 0)
    assert B.rel_err(got, w) < 1e-12
    exp = run(op, x, "SCXYZTn", single(x.shape), y0, "scxyztn", single(y0.shape), 1, 0, expanded=True)
    assert B.rel_err(got, exp) < 1e-12
    c64 = run(dict(op, ops=[(o[0], o[1], o[2].astype(np.complex64)) for o in op["ops"]],
                   kronv=op["kronv"].astype(np.complex64)), x.astype(np.complex64), "SCXYZTn", single(x.shape),
              y0.astype(np.complex64), "scxyztn", single(y0.shape), 1, 0)
    assert B.rel_err(c64, w) < 1e-5
    plan = sb.kron_bsr_plan(sb.C128, op["pim"], dims, op["pim_dom"], dims, 1, op["blockim"], op["blockdom"],
                            op["kronim"], op["krondom"], True, *B.flat_arrays(op["ops"]), "scxyzt", "SCXYZT",
                            single(x.shape), 1, "SCXYZTn", [0] * 7, list(x.shape), list(x.shape), single(y0.shape), 1,
                            "scxyztn", [0] * 7, list(y0.shape), list(y0.shape), None, sb.FastToSlow, 1, 0)
    assert "kron_bsr tier=warp" in plan["items"][0]["kernel"]


def test_cta_tier():
    """vol(kronim) vol(blockim) = 8 x 8 > 32: the CTA tier, 3 columns"""
    rng = np.random.default_rng(13)
    dimi = dimd = [8, 8, 4]
    blockim, kronim = [1, 8, 1], [8, 1, 1]
    pim = single(dimi)
    ops, kronv = KB.random_kron_operator(rng, pim, blockim, dimd, blockim, kronim, kronim, 2, np.complex128)
    op = make_op(ops, kronv, pim, dimi, dimd, blockim, blockim, kronim, kronim, False, sb.FastToSlow, "abc", "ABC")
    x = B.rnd(rng, np.complex128, 3, 8, 8, 4)
    y0 = B.rnd(rng, np.complex128, 8, 8, 4, 3)
    got = run(op, x, "nABC", single(x.shape), y0, "abcn", single(y0.shape), 1.5, -0.5)
    check(got, want(op, x, "nABC", y0, "abcn", 1.5, -0.5), np.complex128)


def test_powers():
    """P = 3: y_p = A y_{p-1}, starting from x; the power range starts at 1 of 4"""
    rng = np.random.default_rng(14)
    dims = [6, 4]
    blockim, kronim = [3, 1], [1, 2]
    pim = single(dims)
    ops, kronv = KB.random_kron_operator(rng, pim, blockim, dims, blockim, kronim, kronim, 2, np.complex128)
    op = make_op(ops, kronv, pim, dims, dims, blockim, blockim, kronim, kronim, True, sb.SlowToFast, "ab", "cd")
    x = B.rnd(rng, np.complex128, 2, 6, 4)                  # "ncd"
    y0 = B.rnd(rng, np.complex128, 4, 6, 4, 2)              # "pabn"
    fromy, sizey = [1, 0, 0, 0], [3, 6, 4, 2]
    got = run(op, x, "ncd", single(x.shape), y0, "pabn", single(y0.shape), 0.7, 0.3, "p", fromy, sizey)
    check(got, want(op, x, "ncd", y0, "pabn", 0.7, 0.3, "p", 3, fromy), np.complex128)


def test_host_components_and_a_y_partition_unlike_pim():
    rng = np.random.default_rng(15)
    dims = [4, 3, 4, 4, 4, 4]
    pim = split(dims, 5, [2])
    op = wilson(rng, np.complex128, pim, dims)
    x = B.rnd(rng, np.complex128, *dims, 5)                 # "SCXYZTn"
    px = split(list(x.shape), 6, [3])
    y0 = B.rnd(rng, np.complex128, *dims, 5)
    py = split(list(y0.shape), 2, [1])                      # cut along x, unlike pim
    for host in [(), ("op", "x", "y")]:
        got = run(op, x, "SCXYZTn", px, y0, "scxyztn", py, 1, 0.5, host=host)
        check(got, want(op, x, "SCXYZTn", y0, "scxyztn", 1, 0.5), np.complex128)


@pytest.mark.parametrize("dtype", [np.float32, np.complex128])
def test_results_are_bit_identical_over_components(dtype):
    """The same operator, x and y split over 1, 2, 4 and 8 components: y identical bit for bit (direct
    writes and write-backs alike)"""
    rng = np.random.default_rng(16)
    dims = [4, 3, 2, 4, 2, 8]
    one = single(dims)
    op1 = wilson(rng, dtype, one, dims)
    ii, jj, v = op1["ops"][0]
    x = B.rnd(rng, dtype, *dims, 3)
    y0 = B.rnd(rng, dtype, *dims, 3)
    results = []
    for n in (1, 2, 4, 8):
        pim = split(dims, 5, list(range(8 // n, 8, 8 // n)))
        rows_per = 2 * 4 * 2 * 8 // n
        ptr = np.concatenate([[0], np.cumsum(ii)])
        bsz = 9
        parts = [(ii[k * rows_per:(k + 1) * rows_per], jj[ptr[k * rows_per]:ptr[(k + 1) * rows_per]],
                  v[ptr[k * rows_per] * bsz:ptr[(k + 1) * rows_per] * bsz]) for k in range(n)]
        op = dict(op1, ops=parts, pim=pim, pim_dom=np.array([[[0] * 6, dims]] * n, np.int32))
        px = split(list(x.shape), 3, [1, 3])
        for py in (split(list(y0.shape), 5, list(range(8 // n, 8, 8 // n))), single(y0.shape)):
            results.append(run(op, x, "SCXYZTn", px, y0, "scxyztn", py, 1.25, 0.5))
    check(results[0], want(op1, x, "SCXYZTn", y0, "scxyztn", 1.25, 0.5), dtype)
    for r in results[1:]:
        assert np.array_equal(r.view(np.uint8), results[0].view(np.uint8))


def test_v_and_kronv_updated_between_calls_and_no_leak():
    rng = np.random.default_rng(17)
    dims = [6, 4]
    blockim, kronim = [3, 1], [1, 2]
    pim = single(dims)
    ops, kronv = KB.random_kron_operator(rng, pim, blockim, dims, blockim, kronim, kronim, 2, np.float64)
    op = make_op(ops, kronv, pim, dims, dims, blockim, blockim, kronim, kronim, True, sb.FastToSlow, "ab", "cd")
    x = B.rnd(rng, np.float64, 6, 4, 2)
    y0 = np.zeros((6, 4, 2))
    sb.clearCaches()
    before = sb.liveAllocations()

    def update(v, kv):  # in place, on torch (device) and numpy (host) components alike
        for t in v:
            t *= 2
        for t in kv:
            t *= 3
    for host in [(), ("op",)]:
        got = run(op, x, "cdn", single(x.shape), y0, "abn", single(y0.shape), 1, 0, calls=2, host=host,
                  update=update)
        op2 = dict(op, ops=[(o[0], o[1], o[2] * 2) for o in op["ops"]], kronv=op["kronv"] * 3)
        check(got, want(op2, x, "cdn", y0, "abn", 1, 0), np.float64)
    sb.clearCaches()
    assert sb.liveAllocations() == before


def test_errors_on_create():
    gpu = sb.createGpuContext(0)
    dims = [4, 4]
    pim = single(dims)
    v = torch.zeros(8, dtype=torch.float64, device="cuda")
    kv = torch.zeros(4, dtype=torch.float64, device="cuda")
    ii = torch.tensor([1, 2, 1, 1], dtype=torch.int32, device="cuda")
    jj = torch.zeros(10, dtype=torch.int32, device="cuda")
    with pytest.raises(RuntimeError, match="^create_kron_bsr: every block row"):
        sb.create_kron_bsr(pim, dims, pim, dims, 1, [2, 1], [2, 1], [1, 2], [1, 2], True, [ii], [jj], [v], [kv], gpu,
                           sb.FastToSlow)
    with pytest.raises(RuntimeError, match="^create_kron_bsr: kronim and blockim exceed 1"):
        sb.create_kron_bsr(pim, dims, pim, dims, 1, [2, 2], [2, 1], [2, 1], [1, 2], True, [ii], [jj], [v], [kv], gpu,
                           sb.FastToSlow)


def test_cxx_kron_bsr_dropin_program(tmp_path):
    """tests/cxx/kron_bsr_dropin_test.cpp, compiled against include/superbblas.h and the in-tree library into
    a temporary directory, and run."""
    root = os.path.dirname(HERE)
    lib = os.path.join(root, "superbblas_b200", "lib")
    exe = str(tmp_path / "kron_bsr_dropin_test")
    r = subprocess.run([os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), "-std=c++17", "-O2", "-ccbin",
                        "/usr/bin/g++", "-I" + os.path.join(root, "include"),
                        os.path.join(HERE, "cxx", "kron_bsr_dropin_test.cpp"), "-o", exe, "-L" + lib,
                        "-lsuperbblas_b200", "-Xlinker", "-rpath", "-Xlinker", lib],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Everything went ok!" in r.stdout
