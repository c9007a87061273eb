"""The FP64 tensor-pipe contraction kernel has an instantiation for K-contiguous operands (one
contracted label of stride 1, fixed shared-memory layout) next to the generic one.  Both must give
the same bits: the same logical contraction is run with K-contiguous operands and again with the
same data laid out row-fastest or with K split over two labels, and the results must be identical.
The K split over CTAs depends only on T, M, N and K, so both runs add the same slices in the same
order.  The shapes cover rows past M and N (clamped loads) and a K tail (zero-filled loads)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import superbblas_b200 as sb

T1, T2 = 2, 3  # two batch labels
SHAPES = [(64, 64), (12, 100), (100, 12)]  # (M, N)
KS = [4096, 4099]  # 4099: a partial last stage of BK = 8
# numpy type, library type, SBB_CONTRACT_KERNEL (the float types take other kernels by default)
DTYPES = {"c128": (np.complex128, sb.C128, None), "f64": (np.float64, sb.F64, None),
          "c64": (np.complex64, sb.C64, "mma"), "f32": (np.float32, sb.F32, "mma")}
CONJ = [(False, False), (True, False), (False, True), (True, True)]


@pytest.fixture(scope="module")
def gu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tests import gpu_util
    return gpu_util


def _single(dim):
    return np.array([[[0] * len(dim), list(dim)]], dtype=np.int32)


def _random(shape, nptype, rng):
    x = rng.uniform(-1, 1, shape)
    if np.iscomplexobj(np.zeros(1, nptype)):
        x = x + 1j * rng.uniform(-1, 1, shape)
    return x.astype(nptype)


def _layouts(x, K, rows):
    """The operand x[u, t, row, k] (k fastest) in every layout the test runs, as (order, dims, data)
    with the first label fastest: k-contiguous, row-fastest and, when K is even, k split in two"""
    M = x.shape[2]
    out = {"kfast": ("k%stu" % rows, [K, M, T1, T2], x),
           "rowfast": ("%sktu" % rows, [M, K, T1, T2], x.transpose(0, 1, 3, 2))}
    if K % 2 == 0:
        K1, K2 = K // 64, 64  # k = k1 + K1 * l; l sits past the row label, so the two cannot merge
        out["ksplit"] = ("a%sltu" % rows, [K1, M, K2, T1, T2],
                         x.reshape(T2, T1, M, K2, K1).transpose(0, 1, 3, 2, 4))
    return out


def _case(a, b, M, N, conj0, conj1):
    (o0, d0, _), (o1, d1, _) = a, b
    dr = [M, N, T1, T2]
    return dict(alpha=1, beta=0, p0=_single(d0), from0=[0] * len(d0), size0=d0, dim0=d0, o0=o0,
                conj0=conj0, p1=_single(d1), from1=[0] * len(d1), size1=d1, dim1=d1, o1=o1,
                conj1=conj1, pr=_single(dr), fromr=[0] * 4, sizer=dr, dimr=dr, o_r="mntu",
                co=sb.FastToSlow)


def _describe(case, sbtype):
    """What the contraction kernel is told for this case, and the contracted labels it sees"""
    plan = sb.contraction_plan(sbtype, case["alpha"], case["p0"], case["from0"], case["size0"],
                               case["dim0"], 1, case["o0"], case["conj0"], case["p1"],
                               case["from1"], case["size1"], case["dim1"], 1, case["o1"],
                               case["conj1"], case["beta"], case["pr"], case["fromr"],
                               case["sizer"], case["dimr"], 1, case["o_r"], case["co"], 1, 0)
    (it,) = plan["items"]
    desc = sb.contract_desc(T=it["T"], M=it["M"], N=it["N"], K=it["K"], conj0=case["conj0"],
                            conj1=case["conj1"])
    return sb.contract_describe(desc, sbtype), len(it["K"])


def _run(gu, case, a, b, nptype):
    vr = [np.zeros(int(np.prod(case["dimr"])), nptype)]
    (got,) = gu.run_contraction(case, [a[2].ravel()], [b[2].ravel()], vr)
    return got


@pytest.mark.parametrize("K", KS)
@pytest.mark.parametrize("M,N", SHAPES)
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_kcontiguous_kernel_matches_generic_bitwise(gu, monkeypatch, dtype, M, N, K):
    nptype, sbtype, force = DTYPES[dtype]
    if force is None:
        monkeypatch.delenv("SBB_CONTRACT_KERNEL", raising=False)
    else:
        monkeypatch.setenv("SBB_CONTRACT_KERNEL", force)
    rng = np.random.default_rng(M * 100003 + N * 101 + K)
    A = _layouts(_random((T2, T1, M, K), nptype, rng), K, "m")
    B = _layouts(_random((T2, T1, N, K), nptype, rng), K, "n")
    for conj0, conj1 in CONJ:
        ref_case = _case(A["kfast"], B["kfast"], M, N, conj0, conj1)
        text, nk = _describe(ref_case, sbtype)
        assert text.startswith("mma ") and "a_kfast=1 b_kfast=1" in text and nk == 1, text
        ref = _run(gu, ref_case, A["kfast"], B["kfast"], nptype)
        for other in [k for k in A if k != "kfast"]:
            case = _case(A[other], B[other], M, N, conj0, conj1)
            text, nk = _describe(case, sbtype)
            if other == "rowfast":
                assert text.startswith("mma ") and "a_kfast=0 b_kfast=0" in text, text
            else:
                assert text.startswith("mma ") and "a_kfast=1 b_kfast=1" in text and nk == 2, text
            got = _run(gu, case, A[other], B[other], nptype)
            assert np.array_equal(got, ref), (other, conj0, conj1,
                                              float(np.abs(got - ref).max()))
    # the results are right, not only alike
    want = np.einsum("utmk,utnk->utnm", np.conj(A["kfast"][2]) if conj0 else A["kfast"][2],
                     np.conj(B["kfast"][2]) if conj1 else B["kfast"][2])
    tol = 1e-12 if nptype in (np.float64, np.complex128) else 1e-5
    err = np.linalg.norm(ref.astype(np.complex128) - want.ravel()) / np.linalg.norm(want)
    assert err < tol, err
