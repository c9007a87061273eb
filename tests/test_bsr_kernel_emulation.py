"""The per-row body of the block-sparse kernel (superbblas_b200/csrc/bsr_kernel.hpp) executed on the CPU
through tests/cxx/bsr_kernel_emul.cpp, in place of the kernel in the plan executor of
tests/test_bsr_plan.py: every type, both block layouts (blockImFast), ragged and empty rows, written
directly and through temporaries, against the oracle.  Column chunks and domain pieces of several
sizes give bit-identical results, as they do in the CUDA kernel, which calls the same function with a
warp or a CTA as the team."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import bsr_cases as B
from tests import test_bsr_plan as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INC = "/usr/local/cuda/include"
DTYPES = [np.float32, np.float64, np.complex64, np.complex128]


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    if not shutil.which("g++") or not os.path.exists(os.path.join(CUDA_INC, "vector_types.h")):
        pytest.skip("needs g++ and the CUDA headers")
    so = str(tmp_path_factory.mktemp("bsrk") / "libbsrk.so")
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-shared", "-fPIC", "-I" + CUDA_INC,
                        os.path.join(ROOT, "tests", "cxx", "bsr_kernel_emul.cpp"), "-o", so],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return ctypes.CDLL(so)


def kernel(emul, m, kd):
    def run(it, v, xg, out, base, alpha, beta):
        dt = P.DT[np.dtype(out.dtype)]
        a = lambda l: np.ascontiguousarray(np.asarray(l, dtype=np.int64).reshape(-1))
        arrs = [a(it["rowptr"]), a(it["goff"] or [0]), a(it["D"] or [0]), a(it["I"] or [0]), a(it["C"] or [0])]
        p = lambda x: x.ctypes.data_as(ctypes.c_void_p)
        sc = lambda z: (ctypes.c_double * 2)(complex(z).real, complex(z).imag)
        v = np.ascontiguousarray(v.astype(out.dtype))
        xg = np.ascontiguousarray(xg)
        view = out[base:]
        emul.bsr_emul(dt, ctypes.c_int64(it["rows"]), p(arrs[0]), p(arrs[1]), it["bi"], it["bd"], it["imfast"],
                      it["ncols"], len(it["D"]), p(arrs[2]), len(it["I"]), p(arrs[3]), len(it["C"]), p(arrs[4]),
                      sc(alpha), sc(beta), p(v), p(xg), view.ctypes.data_as(ctypes.c_void_p),
                      min(m, it["ncols"]), min(kd, it["bd"]))
    return run


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind", ["direct", "back", "power"])
def test_row_body_matches_oracle(emul, dtype, kind):
    rng = np.random.default_rng(50)
    tol = B.TOL[np.dtype(dtype)]
    for k in range(6):
        ncomp = int(rng.integers(1, 3))
        c = P.random_case(rng, 1, ncomp, kind, dtype)
        results = []
        for m, kd in ((64, 64), (1, 1), (2, 4)):
            _, got = P.run_plans(c, 1, ncomp, kernel(emul, m, kd))
            results.append(got)
        a = B.operator_matrix(c["ops"], c["pim"], c["dimi"], c["dimd"], c["blockim"], c["blockdom"], c["imfast"],
                              c["co"])
        want = B.apply(a, c["oim"], c["odom"], c["x"], c["ox"], c["y0"], c["oy"], c["alpha"], c["beta"],
                       c["power"], 3 if c["power"] else 1, c["fromy"])
        assert np.array_equal(np.isnan(results[0]), np.isnan(want))
        assert B.rel_err(np.nan_to_num(results[0]), np.nan_to_num(want)) < tol, (k, c["imfast"])
        for r in results[1:]:
            assert np.array_equal(r.view(np.uint8), results[0].view(np.uint8))
