"""The per-matrix body of the eigh kernel (eigh_body in superbblas_b200/csrc/dense_kernel.hpp) executed
on the CPU through tests/cxx/dense_eigh_emul.cpp, against numpy.linalg.eigh: every type, orders across
the warp / CTA boundary up to each type's limit, special spectra, magnitudes near the ends of each
type's range, the unread lower triangle and non-finite input.  The CUDA kernel calls the same function with a warp or a CTA as the team."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

import superbblas_b200 as sb
from tests import eigh_cases as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INC = "/usr/local/cuda/include"
DTYPES = {np.float32: sb.F32, np.float64: sb.F64, np.complex64: sb.C64, np.complex128: sb.C128}
NS = [1, 2, 3, 5, 12, 31, 32, 33, 64, "limit"]


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    if not shutil.which("g++") or not os.path.exists(os.path.join(CUDA_INC, "vector_types.h")):
        pytest.skip("needs g++ and the CUDA headers")
    so = str(tmp_path_factory.mktemp("eighk") / "libeighk.so")
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-shared", "-fPIC", "-I" + CUDA_INC,
                        os.path.join(ROOT, "tests", "cxx", "dense_eigh_emul.cpp"), "-o", so],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return ctypes.CDLL(so)


def call(emul, dtype, a, vectors=True):
    """-> (w, V) of the row-major matrix a, as the kernel body computes them"""
    a = np.ascontiguousarray(np.asarray(a).astype(dtype))
    w = np.zeros(a.shape[0], E.REAL[np.dtype(dtype)])
    emul.eigh_emul(DTYPES[dtype], a.shape[0], a.ctypes.data_as(ctypes.c_void_p), w.ctypes.data_as(ctypes.c_void_p),
                   int(vectors))
    return w, a


def order(dtype, n):
    return E.LIMIT[np.dtype(dtype)] if n == "limit" else n


def garbage_below(rng, h, dtype):
    """h with its strict lower triangle replaced by garbage (NaN included) and, for complex types, an
    imaginary part on the diagonal: neither is read"""
    a = np.triu(h) + np.tril(E.rnd(rng, dtype, *h.shape) * 1e3, -1)
    if h.shape[0] > 1:
        a[-1, 0] = np.nan
    if np.dtype(dtype).kind == "c":
        a[np.diag_indices(h.shape[0])] += 5j
    return a


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("n", NS)
def test_random_hermitian(emul, dtype, n):
    n = order(dtype, n)
    rng = np.random.default_rng(n)
    h = E.hermitian(rng, dtype, n)
    w, v = call(emul, dtype, garbage_below(rng, h, dtype))
    E.check(h, w, v, dtype, n)


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("kind", ["repeated", "graded", "zero"])
@pytest.mark.parametrize("n", [1, 3, 12, 33, 64])
def test_special_spectra(emul, dtype, kind, n):
    rng = np.random.default_rng(10 + n)
    h = E.hermitian(rng, dtype, n, kind)
    w, v = call(emul, dtype, h)
    E.check(h, w, v, dtype, (kind, n))
    if kind == "zero":
        assert np.all(w == 0) and np.array_equal(v, np.eye(n))


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("n", [1, 5, 32, 33])
def test_diagonal_input_is_sorted_exactly(emul, dtype, n):
    rng = np.random.default_rng(20 + n)
    d = rng.standard_normal(n).astype(E.REAL[np.dtype(dtype)])
    d[n // 2] = d[0]                                     # a tie keeps index order
    w, v = call(emul, dtype, np.diag(d))
    perm = np.argsort(d, kind="stable")
    assert np.array_equal(w, d[perm])
    assert np.array_equal(v, np.eye(n)[:, perm])


@pytest.mark.parametrize("dtype", list(DTYPES))
def test_eigenvalues_without_vectors_match(emul, dtype):
    """The W-only launch skips the eigenvectors; its eigenvalues are the same bits"""
    rng = np.random.default_rng(30)
    h = E.hermitian(rng, dtype, 33)
    w1, _ = call(emul, dtype, h)
    w0, _ = call(emul, dtype, h, vectors=False)
    assert np.array_equal(w0, w1)


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("bad", [np.nan, np.inf])
def test_non_finite_entry_gives_nan(emul, dtype, bad):
    rng = np.random.default_rng(40)
    a = E.hermitian(rng, dtype, 7)
    a[2, 5] = bad
    w, v = call(emul, dtype, a)
    assert np.all(np.isnan(w)) and np.all(np.isnan(v))


SCALES = {np.float32: [1e20, 1e-20, 1e-30, 1e35], np.complex64: [1e20, 1e-20, 1e-30, 1e35],
          np.float64: [1e160, 1e-160, 1e300, 1e-300], np.complex128: [1e160, 1e-160, 1e300, 1e-300]}


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("k", range(4))
@pytest.mark.parametrize("n", [4, 33])
def test_extreme_scales(emul, dtype, k, n):
    """A finite matrix of any magnitude is diagonalised within the same relative bounds: the squares
    behind the norm and the skip test are taken on a power-of-two rescaling of the matrix"""
    s = SCALES[dtype][k]
    rng = np.random.default_rng(50 + n)
    a = (E.hermitian(rng, dtype, n) * s).astype(dtype)
    w, v = call(emul, dtype, a)
    assert np.all(np.isfinite(w)) and np.all(np.isfinite(v))
    E.check(a.astype(np.complex128) / s, w.astype(np.float64) / s, v, dtype, s)


@pytest.mark.parametrize("dtype,s", [(np.float32, 1e19), (np.float32, 1e-21), (np.float32, 1e-23),
                                     (np.complex64, 1e-23), (np.float64, 1e-170), (np.float64, 1e155),
                                     (np.complex128, 1e-170)])
def test_scaled_tridiagonal_against_exact_eigenvalues(emul, dtype, s):
    t = (2 * np.eye(4) + np.eye(4, k=1) + np.eye(4, k=-1)) * s
    w, _ = call(emul, dtype, t)
    exact = 2 + 2 * np.cos(np.pi * np.arange(4, 0, -1) / 5)
    assert np.all(np.abs(w.astype(np.float64) / s - exact) <= 20 * 4 * E.UNIT[np.dtype(dtype)] * exact[-1]), w / s
