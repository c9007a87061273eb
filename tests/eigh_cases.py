"""Inputs and acceptance bounds of eigh (the batched Hermitian eigensolver), shared by its emulation,
plan and GPU tests.  With u the unit roundoff of the element type and n the order:
    |w - w_ref| <= 20 n u ||A||_2,   ||A V - V diag(w)||_F <= 20 n u ||A||_F,   max |V^H V - I| <= 20 n u."""
import numpy as np

UNIT = {np.dtype(np.float32): 2.0 ** -24, np.dtype(np.complex64): 2.0 ** -24,
        np.dtype(np.float64): 2.0 ** -53, np.dtype(np.complex128): 2.0 ** -53}
REAL = {np.dtype(np.float32): np.float32, np.dtype(np.complex64): np.float32,
        np.dtype(np.float64): np.float64, np.dtype(np.complex128): np.float64}
LIMIT = {np.dtype(np.complex128): 80, np.dtype(np.float64): 113, np.dtype(np.complex64): 113,
         np.dtype(np.float32): 160}
KINDS = ["random", "diagonal", "repeated", "graded", "zero"]


def rnd(rng, dtype, *shape):
    x = rng.standard_normal(shape)
    if np.dtype(dtype).kind == "c":
        x = x + 1j * rng.standard_normal(shape)
    return x


def hermitian(rng, dtype, n, kind="random", batch=()):
    """Hermitian matrices [batch..., n, n] (complex128 or float64, rounded to dtype's precision)"""
    dtype = np.dtype(dtype)
    nb = int(np.prod(batch)) if batch else 1
    out = []
    for _ in range(nb):
        if kind == "random":
            b = rnd(rng, dtype, n, n)
            h = (b + b.conj().T) / 2
        elif kind == "diagonal":
            h = np.diag(rng.standard_normal(n)).astype(np.complex128 if dtype.kind == "c" else np.float64)
        else:
            if kind == "repeated":
                lam = np.repeat(rng.standard_normal((n + 2) // 3), 3)[:n]
            elif kind == "graded":
                lam = np.logspace(-8, 0, n) if n > 1 else np.ones(1)
            else:
                lam = np.zeros(n)
            q, _ = np.linalg.qr(rnd(rng, dtype, n, n)) if n else (np.zeros((0, 0)), None)
            h = (q * lam) @ q.conj().T
            h = (h + h.conj().T) / 2
        out.append(h)
    h = np.array(out).reshape(tuple(batch) + (n, n))
    return h.astype(dtype).astype(np.complex128 if dtype.kind == "c" else np.float64)


def check(h, w, v, dtype, what=""):
    """h: [..., n, n] Hermitian input; w: [..., n]; v: [..., n, n] (columns the eigenvectors) or None"""
    dtype = np.dtype(dtype)
    u = UNIT[dtype]
    h = np.asarray(h, np.complex128)
    n = h.shape[-1]
    w = np.asarray(w, np.float64)
    wref = np.linalg.eigvalsh(h)
    norm2 = np.linalg.norm(h, 2, axis=(-2, -1)) if n else np.zeros(h.shape[:-2])
    normf = np.linalg.norm(h, axis=(-2, -1))
    tol = 20 * max(n, 1) * u
    assert np.all(np.abs(w - wref) <= tol * norm2[..., None]), (what, np.max(np.abs(w - wref)), tol * np.max(norm2))
    assert np.all(np.diff(w, axis=-1) >= 0), what
    if v is None:
        return
    v = np.asarray(v, np.complex128)
    res = np.linalg.norm(h @ v - v * w[..., None, :], axis=(-2, -1))
    assert np.all(res <= tol * normf), (what, np.max(res / np.maximum(normf, 1e-300)), tol)
    orth = np.abs(np.swapaxes(v.conj(), -1, -2) @ v - np.eye(n))
    assert np.all(orth <= tol), (what, orth.max(), tol)
