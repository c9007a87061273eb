"""The blocked tier of cholesky and trsm (matrices over one CTA's shared memory) without a GPU: every
rank's plan is executed in numpy, the item's kernel by its printed `step` lines on the gathered
workspaces W and V, and compared with the oracle; the panel body runs on the CPU through
tests/cxx/dense_panel_emul.cpp against numpy."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

import superbblas_b200 as sb
from tests import dense_cases as D
from tests import test_dense_plan as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INC = "/usr/local/cuda/include"
FACTORS = {114: (6, 19), 128: (8, 16), 129: (3, 43), 200: (8, 25), 300: (12, 25)}
CTA_TIER = P.run_item


def _g(dims, which):
    return P.grid(dims, which, 0) if dims else np.zeros(1, np.int64)


def run_steps(op, it, a, x, y):
    """What the blocked tier computes for one item: its steps, one after the other, in numpy"""
    if "steps" not in it:
        return CTA_TIER(op, it, a, x, y)
    n, steps = it["n"], it["steps"]
    R, C, B, H = (it.get(k, []) for k in "RCBH")
    nb, nrhs = len(_g(B, 0)), len(_g(H, 1))
    vec = lambda w: _g(R if (it["left"] if w == 1 else not it["left"]) else C, w)
    ia = it["a"][1] + _g(B, 0)[:, None, None] + _g(R, 0)[None, :, None] + _g(C, 0)[None, None, :]
    ix = it["x"][1] + _g(B, 1)[:, None, None] + _g(H, 1)[None, :, None] + vec(1)[None, None, :] if x is not None else None
    iy = it["y"][1] + _g(B, 2)[:, None, None] + _g(H, 2)[None, :, None] + vec(2)[None, None, :] if y is not None else None
    W = np.zeros(nb * n * n, np.complex128)
    V = np.zeros(nb * nrhs * n, np.complex128)
    buf = dict(W=W, V=V)
    bw = np.arange(nb)[:, None, None] * n * n

    def block(off, rows, cols):            # [batch, rows, cols] indices of a block of W
        return bw + off + np.arange(rows)[None, :, None] * n + np.arange(cols)[None, None, :]

    for st in steps:
        s, refs = st["step"], st["refs"]
        if s == "gather" and refs[0][0] == "A":
            W[:] = a[ia].ravel()
        elif s == "gather":
            V[:] = complex(it["alpha"]) * x[ix].ravel()
        elif s == "scatter" and refs[1][0] == "A":
            a[ia] = W.reshape(nb, n, n) if a.dtype.kind == "c" else W.reshape(nb, n, n).real
        elif s == "scatter":
            y[iy] = V.reshape(nb, nrhs, n) if y.dtype.kind == "c" else V.reshape(nb, nrhs, n).real
        elif s == "zero":
            W[block(refs[0][1], st["rows"], st["cols"])] = 0
        elif s == "factor":
            i = block(refs[0][1], st["n"], st["n"])
            m = W[i]
            up = np.triu(m, 1)
            h = up + np.conj(np.swapaxes(up, 1, 2)) + np.einsum("bii->bi", m).real[:, :, None] * np.eye(st["n"])
            W[i] = np.conj(np.swapaxes(np.linalg.cholesky(h), 1, 2))
        elif s == "panel":
            u = np.triu(W[block(refs[0][1], st["n"], st["n"])])
            i = block(refs[1][1], st["n"], st["rhs"])
            W[i] = np.linalg.solve(np.conj(np.swapaxes(u, 1, 2)), W[i])
        elif s == "solve":
            u = np.triu(W[block(refs[0][1], st["n"], st["n"])])
            i = np.arange(nb)[:, None, None] * nrhs * n + refs[1][1] + np.arange(nrhs)[None, :, None] * n \
                + np.arange(st["n"])[None, None, :]
            xt = np.swapaxes(V[i], 1, 2)                        # [batch, n, rhs]
            V[i] = np.swapaxes(np.linalg.solve(u if st["left"] else np.swapaxes(u, 1, 2), xt), 1, 2)
        elif s == "update":                                      # vr -= f0(v0) v1, as the contract line says
            (b0, o0), (b1, o1), (br, orr) = refs
            T, M, N, K = (st.get(k, []) for k in "TMNK")
            i0 = o0 + _g(T, 0)[:, None, None] + _g(M, 0)[None, :, None] + _g(K, 0)[None, None, :]
            i1 = o1 + _g(T, 1)[:, None, None] + _g(N, 1)[None, :, None] + _g(K, 1)[None, None, :]
            ir = orr + _g(T, 2)[:, None, None] + _g(M, 2)[None, :, None] + _g(N, 2)[None, None, :]
            v0 = np.conj(buf[b0][i0]) if st["conj0"] else buf[b0][i0]
            buf[br][ir] -= np.einsum("tmk,tnk->tmn", v0, buf[b1][i1])
        else:
            raise AssertionError(st)


def blocked_case(rng, op, left, n, T, world):
    c, s = FACTORS[n]
    ext = dict(c=c, s=s, C=s, S=c, x=2, r=int(rng.integers(3, 41)))
    o = "".join(rng.permutation(list("xcsSC")))
    co = int(rng.integers(2))
    case = dict(op=op, T=np.dtype(T), co=co, o=o, orows="cs", ocols="SC", ext=ext,
                alpha=1.5 if np.dtype(T).kind == "f" else 0.5 + 1j)
    case["pa"] = P.random_parts(rng, [ext[k] for k in o], world)
    if op == "trsm":
        xv, yv = ("cs", "SC") if left else ("SC", "cs")
        case["ox"] = "".join(rng.permutation(list("x" + xv + "r")))
        case["oy"] = "".join(rng.permutation(list("x" + yv + "r")))
        case["px"] = P.random_parts(rng, [ext[k] for k in case["ox"]], world)
        case["py"] = P.random_parts(rng, [ext[k] for k in case["oy"]], world)
    return case


@pytest.mark.parametrize("world", [1, 2])
@pytest.mark.parametrize("T", [np.float64, np.complex128])
@pytest.mark.parametrize("n", sorted(FACTORS))
@pytest.mark.parametrize("op,left", [("cholesky", True), ("trsm", True), ("trsm", False)])
def test_blocked_steps_match_oracle(monkeypatch, op, left, n, T, world):
    monkeypatch.setattr(P, "run_item", run_steps)
    rng = np.random.default_rng(n * 10 + world + 100 * left + 1000 * (op == "trsm"))
    case = blocked_case(rng, op, left, n, T, world)
    ext, o = case["ext"], case["o"]
    a_full = D.well_conditioned(rng, op, [ext[k] for k in o], o, "cs", "SC", case["co"], T)
    x_full = None
    if op == "trsm":
        x_full = rng.standard_normal([ext[k] for k in case["ox"]]).astype(T)
    plans, got = P.run_plans(case, world, 1, a_full, x_full)
    items = [i for q in plans for i in q["items"]]
    tier = "blocked" if n * n * np.dtype(T).itemsize > 200 * 1024 else "cta"   # f64 up to n = 160
    assert items and all(i["kernel"].startswith("dense %s tier=%s n=%d " % (op, tier, n)) for i in items)
    if op == "trsm":
        want = D.oracle(op, a_full, o, "cs", "SC", case["co"], case["alpha"], x_full, case["ox"], case["oy"],
                        [ext[k] for k in case["oy"]])
    else:
        want = D.oracle(op, a_full, o, "cs", "SC", case["co"])
    assert D.rel_err(got, want) < 1e-10
    for it in items if tier == "blocked" else []:
        updates = [s for s in it["steps"] if s["step"] == "update"]
        assert updates and len([s for s in it["steps"] if s["step"] in ("factor", "solve")]) == len(updates) + 1
        # the updates run on the DMMA kernel; a trsm update needs 16 right-hand sides or more for it
        rhs = int(it["kernel"].split(" rhs=")[1].split()[0])
        if np.dtype(T) == np.complex128 and n >= 128 and (op == "cholesky" or rhs >= 16):
            assert all(s["kernel"].startswith("mma ") for s in updates), [s["kernel"] for s in updates]


def single(dims):
    return np.array([[[0] * len(dims), list(dims)]], dtype=np.int32)


def test_blocked_limits_and_errors():
    for op in (sb.CHOLESKY, sb.INVERSION):
        sb.dense_plan(op, sb.C128, single([2, 113, 113]), 1, "xcC", "c", "C", sb.FastToSlow, 1, 0)
    p = sb.dense_plan(sb.CHOLESKY, sb.C128, single([2, 114, 114]), 1, "xcC", "c", "C", sb.FastToSlow, 1, 0)
    assert p["items"][0]["kernel"].startswith("dense cholesky tier=blocked n=114 batch=2 rhs=0 nb=64 w=25992 v=0")
    kw = dict(px=single([2, 114, 5]), ncomponentsx=1, ox="xcr", py=single([2, 114, 5]), ncomponentsy=1, oy="xCr")
    p = sb.dense_plan(sb.TRSM, sb.C128, single([2, 114, 114]), 1, "xcC", "c", "C", sb.FastToSlow, 1, 0, **kw)
    assert p["items"][0]["kernel"].startswith("dense trsm tier=blocked n=114 batch=2 rhs=5 nb=64 w=25992 v=1140")
    with pytest.raises(RuntimeError, match=r"^inversion: order n = 114 is over the limit: one matrix must fit in "
                       r"shared memory, n\^2 \* sizeof\(T\) <= 204800 bytes \(n <= 113 for complex double, 160 for "
                       r"double and complex float, 226 for float\)$"):
        sb.dense_plan(sb.INVERSION, sb.C128, single([2, 114, 114]), 1, "xcC", "c", "C", sb.FastToSlow, 1, 0)
    with pytest.raises(RuntimeError, match=r"^gesm: order n = 114 is over the limit: one matrix must fit"):
        sb.dense_plan(sb.GESM, sb.C128, single([2, 114, 114]), 1, "xcC", "c", "C", sb.FastToSlow, 1, 0, **kw)
    # 8 row, 8 column and 1 batch label of extent 2: 17 box dimensions, one more than a box has; every
    # rank refuses, also the one whose part is empty
    o, rows, cols = "abcdefghABCDEFGHx", "abcdefgh", "ABCDEFGH"
    dims = [2] * 17
    pa = np.array([[[0] * 17, dims], [[0] * 17, [0] * 17]], dtype=np.int32)
    for rank in range(2):
        with pytest.raises(RuntimeError, match="cholesky: a matrix over the shared-memory limit is gathered with one "
                           "dimension per row, column, batch .* 17 labels of extent > 1 are more than 16"):
            sb.dense_plan(sb.CHOLESKY, sb.F32, pa, 1, o, rows, cols, sb.FastToSlow, 2, rank)
    with pytest.raises(RuntimeError, match="inversion: order n = 256 is over the limit"):
        sb.dense_plan(sb.INVERSION, sb.F32, pa, 1, o, rows, cols, sb.FastToSlow, 2, 0)
    # within the limit the same labels take the CTA tier and no box
    sb.dense_plan(sb.CHOLESKY, sb.F32, single([2] * 14), 1, o[:7] + o[8:15], rows[:7], cols[:7], sb.FastToSlow, 1, 0)


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    if not shutil.which("g++") or not os.path.exists(os.path.join(CUDA_INC, "vector_types.h")):
        pytest.skip("needs g++ and the CUDA headers")
    so = str(tmp_path_factory.mktemp("densepanel") / "libdensepanel.so")
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-shared", "-fPIC", "-I" + CUDA_INC,
                        os.path.join(ROOT, "tests", "cxx", "dense_panel_emul.cpp"), "-o", so],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return ctypes.CDLL(so)


@pytest.mark.parametrize("dtype,code,tol", [(np.float32, sb.F32, 1e-5), (np.float64, sb.F64, 1e-12),
                                            (np.complex64, sb.C64, 1e-5), (np.complex128, sb.C128, 1e-12)])
@pytest.mark.parametrize("n", [1, 7, 64, 65])
def test_panel_body(emul, dtype, code, tol, n):
    rng = np.random.default_rng(n)
    cplx = np.dtype(dtype).kind == "c"
    rnd = lambda *s: rng.standard_normal(s) + (1j * rng.standard_normal(s) if cplx else 0)
    u = np.triu(rnd(n, n)) + 2 * n * np.eye(n)
    a = np.where(np.tri(n, k=-1) > 0, np.nan, u).astype(dtype)   # below the diagonal is not read
    x = rnd(n, 9)
    xs = np.ascontiguousarray(x.astype(dtype))
    emul.panel_emul(code, n, np.ascontiguousarray(a).ctypes.data_as(ctypes.c_void_p),
                    xs.ctypes.data_as(ctypes.c_void_p), 9)
    want = np.linalg.solve(np.conj(u.astype(dtype).astype(np.complex128)).T, x.astype(dtype))
    assert np.linalg.norm(xs - want) / np.linalg.norm(want) < tol * n
