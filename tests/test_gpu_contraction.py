"""GPU parity: superbblas_b200.contraction against the oracle, within the north-star tolerances
(1e-12 relative for double / complex double, 1e-5 for float / complex float)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import superbblas_b200 as sb
from tests import cases as C

TOL = {np.dtype(np.float64): 1e-12, np.dtype(np.complex128): 1e-12,
       np.dtype(np.float32): 1e-5, np.dtype(np.complex64): 1e-5}


@pytest.fixture(scope="module")
def gu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tests import gpu_util
    return gpu_util


def close(got, want, tol):
    for g, w in zip(got, want):
        if w.size == 0:
            continue
        scale = max(float(np.linalg.norm(w)), float(np.sqrt(w.size)))
        err = float(np.linalg.norm(g.astype(np.complex128) - w.astype(np.complex128)))
        if not err <= tol * scale:
            return False, err / scale
    return True, 0.0


@pytest.mark.parametrize("kernel", ["auto", "simt", "mma"])
@pytest.mark.parametrize("seed", range(4))
def test_random_contractions(gu, seed, kernel):
    """contract.cpp-style sweep: 0..2 labels per group, shuffled orders, conj flags, partitions
    {master, replicated, block}, random from offsets, alpha/beta in {0,1,-1,other}."""
    rng = np.random.default_rng(800 + seed)
    if kernel == "auto":
        os.environ.pop("SBB_CONTRACT_KERNEL", None)
    else:
        os.environ["SBB_CONTRACT_KERNEL"] = kernel
    try:
        for it in range(40):
            case = C.random_contraction_case(rng, max_dim=5)
            v0, v1, vr = C.make_contraction_data(case, seed * 100 + it)
            want = C.oracle_contraction(case, v0, v1, vr)
            got = gu.run_contraction(case, v0, v1, vr)
            ok, err = close(got, want, TOL[case["T"]])
            assert ok, (seed, it, err, case)
    finally:
        os.environ.pop("SBB_CONTRACT_KERNEL", None)


def _single(dim):
    return np.array([[[0] * len(dim), list(dim)]], dtype=np.int32)


@pytest.mark.parametrize("co", [0, 1])
def test_config1_contractions(gu, co):
    """BASELINE config 1: contraction over s,c on 8^3x16, site-wise and with 4x4 vectors."""
    dim = [8, 8, 8, 16, 4, 3]
    for (o0, d0, o1, d1, o_r, dr) in [
            ("xyztsc", dim, "xyztsc", dim, "xyzt", dim[:4]),
            ("xyztscN", dim + [4], "xyztscn", dim + [4], "xyztNn", dim[:4] + [4, 4])]:
        case = dict(alpha=1, beta=0, p0=_single(d0), from0=[0] * len(d0), size0=d0, dim0=d0, o0=o0,
                    conj0=True, p1=_single(d1), from1=[0] * len(d1), size1=d1, dim1=d1, o1=o1,
                    conj1=False, pr=_single(dr), fromr=[0] * len(dr), sizer=dr, dimr=dr, o_r=o_r,
                    co=co, T=np.dtype(np.complex128))
        v0, v1, vr = C.make_contraction_data(case, 5)
        want = C.oracle_contraction(case, v0, v1, vr)
        got = gu.run_contraction(case, v0, v1, vr)
        ok, err = close(got, want, 1e-12)
        assert ok, (o_r, err)


@pytest.mark.parametrize("dtype", [np.complex128, np.float64, np.complex64, np.float32])
def test_distillation_shape_reduced(gu, dtype):
    """BASELINE config 2 at reduced size: V[c,x,y,z,t,n]^H V[c,x,y,z,t,m] -> [t,n,m]; also the
    z,t-partitioned variant of config 4 with 8 components (partials reduced with Add)."""
    L, Lt, nv = 8, 8, 64
    dimv, dimr = [3, L, L, L, Lt, nv], [Lt, nv, nv]
    case = dict(alpha=1, beta=0, p0=_single(dimv), from0=[0] * 6, size0=dimv, dim0=dimv, o0="cxyztn",
                conj0=True, p1=_single(dimv), from1=[0] * 6, size1=dimv, dim1=dimv, o1="cxyztm",
                conj1=False, pr=_single(dimr), fromr=[0] * 3, sizer=dimr, dimr=dimr, o_r="tnm", co=1,
                T=np.dtype(dtype))
    v0, v1, vr = C.make_contraction_data(case, 6)
    want = C.oracle_contraction(case, v0, v1, vr)
    got = gu.run_contraction(case, v0, v1, vr)
    ok, err = close(got, want, TOL[np.dtype(dtype)])
    assert ok, err
    # partitioned on z,t over 8 components; output partitioned on t
    P = 8
    pv = sb.basic_partitioning("cxyztn", dimv, [1, 1, 1, 2, 4, 1], "zt", P, 1)
    pr = sb.basic_partitioning("tnm", dimr, [P, 1, 1], "t", P, 1)
    case.update(p0=pv, p1=pv, pr=pr, beta=0.5, alpha=-1)
    v0, v1, vr = C.make_contraction_data(case, 7)
    want = C.oracle_contraction(case, v0, v1, vr)
    got = gu.run_contraction(case, v0, v1, vr)
    ok, err = close(got, want, TOL[np.dtype(dtype)])
    assert ok, err


def test_large_contraction_properties(gu):
    """At a larger size (16^3 x 32, n=m=64, complex double): agreement with a torch.einsum in
    complex128 on the GPU, and linearity in the first operand."""
    import torch
    L, Lt, nv = 16, 32, 64
    K = 3 * L ** 3
    dimv, dimr = [3, L, L, L, Lt, nv], [Lt, nv, nv]
    g = torch.Generator(device="cuda").manual_seed(5)
    mk = lambda: torch.view_as_complex(torch.rand(K * Lt * nv, 2, generator=g, device="cuda",
                                                  dtype=torch.float64) * 2 - 1)
    a, a2, b = mk(), mk(), mk()
    gpu = sb.createGpuContext(0)

    def run(x, y):
        r = torch.zeros(Lt * nv * nv, device="cuda", dtype=torch.complex128)
        sb.contraction(1, _single(dimv), [0] * 6, dimv, dimv, 1, "cxyztn", True, [x], gpu,
                       _single(dimv), [0] * 6, dimv, dimv, 1, "cxyztm", False, [y], gpu, 0,
                       _single(dimr), [0] * 3, dimr, dimr, 1, "tnm", [r], gpu, sb.FastToSlow)
        sb.sync(gpu)
        return r
    r = run(a, b)
    # FastToSlow memory order: k fastest, then t, then n  ->  torch view [n][t][k]
    A = a.view(nv, Lt, K)
    B = b.view(nv, Lt, K)
    ref = torch.einsum("ntk,mtk->mnt", A.conj(), B).contiguous().view(-1)  # r[t + Lt*(n + nv*m)]
    rel = (torch.linalg.norm(r - ref) / torch.linalg.norm(ref)).item()
    assert rel < 1e-12, rel
    r2 = run(a2, b)
    r12 = run(a + 2 * a2, b)
    rel = (torch.linalg.norm(r12 - (r + 2 * r2)) / torch.linalg.norm(r12)).item()
    assert rel < 1e-12, rel


@pytest.mark.parametrize("dtype", [np.complex128, np.complex64])
def test_skinny_shapes_of_the_reference_dist_program(gu, dtype):
    """The batched-GEMM shapes the reference's tests/dist.cpp times (there without checking them):
    "inner product" (m = n small, k long) and "update" (m long, n = k small), here against a torch
    einsum in complex128.  Whatever kernel the dispatcher picks (tensor-core split-K, generic, or the
    opt-in row / dot kernels) must agree."""
    import torch
    gpu = sb.createGpuContext(0)
    tdt = torch.complex128 if dtype == np.complex128 else torch.complex64
    tol = TOL[np.dtype(dtype)]
    g = torch.Generator(device="cuda").manual_seed(17)

    def rnd(n):
        real = torch.float64 if tdt == torch.complex128 else torch.float32
        return torch.view_as_complex(torch.rand(n, 2, generator=g, device="cuda", dtype=real) * 2 - 1)
    batch = 4
    for (m, n, k) in [(1, 1, 8192), (3, 3, 8192), (4, 4, 6000), (12, 12, 4096), (16, 5, 4096),
                      (4096, 3, 3), (4096, 12, 12), (3, 4096, 4), (2048, 16, 16)]:
        # column-major batched GEMM with op(a) = a^H:  c[i,j,b] = sum_l conj(a[l,i,b]) b[l,j,b]
        a, b = rnd(k * m * batch), rnd(k * n * batch)
        c = torch.zeros(m * n * batch, device="cuda", dtype=tdt)
        da, db, dc = [k, m, batch], [k, n, batch], [m, n, batch]
        sb.contraction(1, _single(da), [0] * 3, da, da, 1, "kmb", True, [a], gpu, _single(db), [0] * 3,
                       db, db, 1, "knb", False, [b], gpu, 0, _single(dc), [0] * 3, dc, dc, 1, "mnb", [c],
                       gpu, sb.FastToSlow)
        sb.sync(gpu)
        A = a.view(batch, m, k).to(torch.complex128)   # FastToSlow: first label fastest
        B = b.view(batch, n, k).to(torch.complex128)
        ref = torch.einsum("bmk,bnk->bnm", A.conj(), B).contiguous().view(-1)
        rel = (torch.linalg.norm(c.to(torch.complex128) - ref) / torch.linalg.norm(ref)).item()
        assert rel < tol, ((m, n, k), rel)


@pytest.mark.parametrize("shape", [
    # (m, n, k, batch dims, conj0, conj1, alpha, beta)
    (64, 64, 1536, (4,), True, False, 1, 0),            # the distillation tile, whole
    (20, 50, 1000, (3, 2), False, False, 0.5 - 2j, 1.5 + 0.5j),  # partial tiles, K tail, two batch dims
    (130, 70, 2048 + 8, (2,), False, True, -1, 0),      # several tiles per batch entry
    (64, 64, 4 * 32 * 37, (1,), True, True, 1, 1),      # no batch dim, long K (deep split-K)
    (32, 16, 512, (5,), True, False, 2, 0),             # smallest eligible tile
])
def test_tcgen05_complex_float(gu, shape):
    """Complex float contractions with a long contiguous K run on the tcgen05 path (TMA -> TF32 x 3
    split -> tensor memory).  Checked against a complex128 einsum (tolerance 1e-5, the north star's
    bound for complex float), next to the FP64 tensor-pipe kernel on the same data; the values span
    several orders of magnitude and both signs so that the hi/lo split is exercised."""
    import torch
    m, n, k, bdims, conj0, conj1, alpha, beta = shape
    gpu = sb.createGpuContext(0)
    g = torch.Generator(device="cuda").manual_seed(m * 1000 + n)
    nb = int(np.prod(bdims))

    def rnd(count):
        x = torch.randn(count, 2, generator=g, device="cuda", dtype=torch.float32)
        e = torch.rand(count, 1, generator=g, device="cuda", dtype=torch.float32) * 4 - 2
        return torch.view_as_complex((x * torch.pow(10.0, e)).contiguous())
    blabels = "tu"[:len(bdims)]
    da, db, dc = [k, *bdims, m], [k, *bdims, n], [*bdims, m, n]
    oa, ob, oc = "k" + blabels + "m", "k" + blabels + "n", blabels + "mn"
    a, b = rnd(k * nb * m), rnd(k * nb * n)
    c0 = rnd(nb * m * n)
    A = a.view(m, *reversed(bdims), k).reshape(m, nb, k).to(torch.complex128)  # first label fastest
    B = b.view(n, *reversed(bdims), k).reshape(n, nb, k).to(torch.complex128)
    ref = torch.einsum("mtk,ntk->nmt", A.conj() if conj0 else A, B.conj() if conj1 else B)
    ref = complex(alpha) * ref + complex(beta) * c0.view(n, m, nb).to(torch.complex128)
    errs = {}
    for kernel in ("auto", "mma"):
        if kernel == "auto":
            os.environ.pop("SBB_CONTRACT_KERNEL", None)
        else:
            os.environ["SBB_CONTRACT_KERNEL"] = kernel
        try:
            c = c0.clone()
            sb.profile_enable(True)
            sb.profile_read("contract_tc")
            sb.contraction(alpha, _single(da), [0] * len(da), da, da, 1, oa, conj0, [a], gpu,
                           _single(db), [0] * len(db), db, db, 1, ob, conj1, [b], gpu, beta,
                           _single(dc), [0] * len(dc), dc, dc, 1, oc, [c], gpu, sb.FastToSlow)
            sb.sync(gpu)
            _, launched = sb.profile_read("contract_tc")
            sb.profile_enable(False)
        finally:
            os.environ.pop("SBB_CONTRACT_KERNEL", None)
        assert (launched >= 1) == (kernel == "auto"), (kernel, launched)
        got = c.view(n, m, nb).to(torch.complex128)
        errs[kernel] = (torch.linalg.norm(got - ref) / torch.linalg.norm(ref)).item()
    print("tcgen05 c64 %s: rel err %.2e (FP64-pipe kernel %.2e)" % (shape[:4], errs["auto"], errs["mma"]))
    assert errs["auto"] < 1e-5, errs
    assert errs["mma"] < 1e-5, errs


def test_local_contraction_wrapper(gu):
    """local_contraction (signature of the reference's tests/local.cpp:163) against the oracle."""
    import torch
    gpu = sb.createGpuContext(0)
    for dtype, tol in ((np.complex128, 1e-12), (np.float32, 1e-5)):
        dim0, dim1, dimr = [5, 7, 3], [7, 4, 3], [3, 5, 4]  # "akt" . "kbt" -> "tab"
        case = dict(alpha=1, beta=0, p0=_single(dim0), from0=[0] * 3, size0=dim0, dim0=dim0, o0="akt",
                    conj0=True, p1=_single(dim1), from1=[0] * 3, size1=dim1, dim1=dim1, o1="kbt",
                    conj1=False, pr=_single(dimr), fromr=[0] * 3, sizer=dimr, dimr=dimr, o_r="tab",
                    co=1, T=np.dtype(dtype))
        v0, v1, vr = C.make_contraction_data(case, 9)
        want = C.oracle_contraction(case, v0, v1, vr)
        d0, d1, dr = (torch.from_numpy(x[0]).cuda() for x in (v0, v1, vr))
        sb.local_contraction(1, "akt", dim0, True, d0, "kbt", dim1, False, d1, 0, "tab", dimr, dr, gpu,
                             sb.FastToSlow)
        sb.sync(gpu)
        ok, err = close([dr.cpu().numpy()], want, tol)
        assert ok, (dtype, err)


def test_contraction_errors(gu):
    import torch
    gpu = sb.createGpuContext(0)
    x = torch.zeros(4, device="cuda", dtype=torch.float64)
    d = [2, 2]
    with pytest.raises(RuntimeError, match="unmatched"):
        sb.contraction(1, _single(d), [0, 0], d, d, 1, "ab", False, [x], gpu, _single(d), [0, 0], d,
                       d, 1, "bc", False, [x], gpu, 0, _single(d), [0, 0], d, d, 1, "cz", [x], gpu,
                       sb.FastToSlow)
    with pytest.raises(RuntimeError, match="does not match"):
        sb.contraction(1, _single(d), [0, 0], d, d, 1, "ab", False, [x], gpu, _single(d), [0, 0],
                       [2, 1], d, 1, "bc", False, [x], gpu, 0, _single(d), [0, 0], d, d, 1, "ac", [x],
                       gpu, sb.FastToSlow)


def test_contraction_error_after_staging_returns_the_workspace(gu):
    """Nine contracted labels do not fit one kernel; the call with host operands fails and leaves
    no workspace block allocated."""
    cpu = sb.createCpuContext()
    d0, d1, dr = [2] * 9 + [3], [2] * 9 + [4], [3, 4]
    v0, v1 = np.ones(int(np.prod(d0))), np.ones(int(np.prod(d1)))
    vr = np.zeros(int(np.prod(dr)))
    live = sb.liveAllocations()
    with pytest.raises(RuntimeError, match="contraction: too many labels in a group"):
        sb.contraction(1, _single(d0), [0] * 10, d0, d0, 1, "abcdefghix", False, [v0], cpu,
                       _single(d1), [0] * 10, d1, d1, 1, "abcdefghiy", False, [v1], cpu, 0,
                       _single(dr), [0, 0], dr, dr, 1, "xy", [vr], cpu, sb.FastToSlow)
    assert sb.liveAllocations() == live
