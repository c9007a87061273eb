"""The per-row body of the Kronecker block-sparse kernel (kron_row_body in superbblas_b200/csrc/bsr_kernel.hpp)
executed on the CPU through tests/cxx/bsr_kron_emul.cpp, in place of the kernel in the plan executor of
tests/test_kron_bsr_plan.py: every type and both block layouts (blockImFast), written directly, through
temporaries and over powers, against a numpy loop in the stated summation order (sum over u, then jk, of
K_u[ik, jk] t_u[jk, ib, c], t_u = sum over jb of B[ib, jb] x[jk, jb, c]).  Column chunks and block pieces
of several sizes give bit-identical results, as they do in the CUDA kernel, which calls the same function
with a warp or a CTA as the team."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import bsr_cases as B
from tests import kron_bsr_cases as KB
from tests import test_bsr_plan as P
from tests import test_kron_bsr_plan as KP

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INC = "/usr/local/cuda/include"
DTYPES = [np.float32, np.float64, np.complex64, np.complex128]


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    if not shutil.which("g++") or not os.path.exists(os.path.join(CUDA_INC, "vector_types.h")):
        pytest.skip("needs g++ and the CUDA headers")
    so = str(tmp_path_factory.mktemp("kronk") / "libkronk.so")
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-shared", "-fPIC", "-I" + CUDA_INC,
                        os.path.join(ROOT, "tests", "cxx", "bsr_kron_emul.cpp"), "-o", so],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return ctypes.CDLL(so)


def kernel(emul, kronv, m, nu):
    def run(it, v, xg, out, base, alpha, beta):
        dt = P.DT[np.dtype(out.dtype)]
        a = lambda l: np.ascontiguousarray(np.asarray(l, dtype=np.int64).reshape(-1))
        D = [(sz, ks, st) for (sz, st), ks in zip(it["D"], it["DK"])]
        I = [(nb, sz, ks, st) for (nb, sz, st), ks in zip(it["I"], it["IK"])]
        arrs = [a(it["rowptr"]), a(it["goff"] or [0]), a(D or [0]), a(I or [0]), a(it["C"] or [0])]
        p = lambda x: x.ctypes.data_as(ctypes.c_void_p)
        sc = lambda z: (ctypes.c_double * 2)(complex(z).real, complex(z).imag)
        v = np.ascontiguousarray(v.astype(out.dtype))
        kv = np.ascontiguousarray(np.asarray(kronv).astype(out.dtype))
        xg = np.ascontiguousarray(xg)
        view = out[base:]
        emul.kron_bsr_emul(dt, ctypes.c_int64(it["rows"]), p(arrs[0]), p(arrs[1]), it["bi"], it["bd"], it["ki"],
                           it["kd"], it["u"], it["imfast"], it["ncols"], len(D), p(arrs[2]), len(I), p(arrs[3]),
                           len(it["C"]), p(arrs[4]), sc(alpha), sc(beta), p(v), p(kv), p(xg),
                           view.ctypes.data_as(ctypes.c_void_p), min(m, it["ncols"]), max(1, min(nu, it["u"])))
    return run


def ordered_kernel(kronv):
    """The stated summation order as a numpy loop, one product and sum per term, in complex128"""
    def run(it, v, xg, out, base, alpha, beta):
        bi, bd, ki, kd, U, nc = it["bi"], it["bd"], it["ki"], it["kd"], it["u"], it["ncols"]
        xo, cp, rp, goff = KP.kron_points(it), P.offsets(it["C"]), it["rowptr"], it["goff"]
        kvc = np.asarray(kronv).astype(np.complex128)
        for r in range(it["rows"]):
            acc = np.zeros((ki, bi, nc), np.complex128)
            for u in range(U):
                b = rp[r] + u
                Bm = KB.mat(v[b * bi * bd:(b + 1) * bi * bd].astype(np.complex128), it["imfast"], bi, bd)
                K = KB.mat(kvc[u * ki * kd:(u + 1) * ki * kd], it["imfast"], ki, kd)
                xs = xg[(goff[b] + xo)[:, None] * nc + np.arange(nc)[None, :]].reshape(kd, bd, nc).astype(np.complex128)
                t = np.zeros((kd, bi, nc), np.complex128)
                for jb in range(bd):
                    t += Bm[None, :, jb, None] * xs[:, jb, None, :]
                for jk in range(kd):
                    acc += K[:, jk, None, None] * t[None, jk]
            o = base + KP.kron_image(it, r).reshape(ki, bi)[:, :, None] + cp[None, None, :]
            res = alpha * acc + (beta * out[o] if beta != 0 else 0)
            out[o] = res if out.dtype.kind == "c" else res.real
    return run


def close(a, b, tol):
    a, b = np.nan_to_num(a).astype(np.complex128), np.nan_to_num(b).astype(np.complex128)
    return np.linalg.norm(a - b) <= tol * np.linalg.norm(b)          # rows without blocks: both zero


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("imfast", [True, False])
def test_kron_row_body_matches_ordered_sum(emul, dtype, imfast):
    rng = np.random.default_rng(60)
    tol = B.TOL[np.dtype(dtype)]
    for k in range(6):
        kind = ["direct", "back", "power"][k % 3]
        ncomp = int(rng.integers(1, 3))
        c = KP.random_kron_case(rng, 1, ncomp, kind, dtype)
        c["imfast"] = imfast
        results = []
        for m, nu in ((64, 64), (1, 1), (2, 2)):
            _, got = KP.run_kron_plans(c, 1, ncomp, kernel(emul, c["kronv"], m, nu))
            results.append(got)
        _, want = KP.run_kron_plans(c, 1, ncomp, ordered_kernel(c["kronv"]))
        assert np.array_equal(np.isnan(results[0]), np.isnan(want))
        assert close(results[0], want, tol), (k, kind)
        assert close(results[0], KP.want_of(c), tol), (k, kind)
        for r in results[1:]:
            assert np.array_equal(r.view(np.uint8), results[0].view(np.uint8))
