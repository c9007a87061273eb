"""Host logic of eigh's driver without a GPU: every rank's plan (A in place or gathered, W written by the
launch of A's batch box, by a W-only launch, or from a temporary) is executed in numpy for 1 to 4
simulated ranks and checked against the bounds of tests/eigh_cases.py; its steps; the argument errors,
which every rank throws before any data moves; and the C++ overloads compile."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import superbblas_b200 as sb
from tests import dense_cases as D
from tests import eigh_cases as E
from tests.plan_exec import _indices, run_ranks
from tests.test_dense_plan import grid, random_parts

DT = {np.dtype(np.float64): sb.F64, np.dtype(np.complex128): sb.C128}
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class Eigh:
    """numpy's eigh of the Hermitian matrix of an upper triangle, the same bits for the same input, as
    the kernel gives (replicated and redundant launches must agree)"""

    def __init__(self):
        self.memo = {}

    def __call__(self, m):
        key = m.tobytes()
        if key not in self.memo:
            self.memo[key] = np.linalg.eigh(m, UPLO="U")
        return self.memo[key]


def run_item(it, a, w, eigh):
    R, C, B = it["R"], it["C"], it.get("B", [])
    rows = grid(R, 0, 0) if R else np.zeros(1, np.int64)
    cols = grid(C, 0, 0) if C else np.zeros(1, np.int64)
    wcols = grid(C, 2, 0) if C else np.zeros(1, np.int64)
    bgrid = [grid(B, k, 0) for k in (0, 2)] if B else [np.zeros(1, np.int64)] * 2
    for ba, bw in zip(*bgrid):
        at = it["a"][1] + ba + rows[:, None] + cols[None, :]
        lam, v = eigh(a[at])
        if "a" in it["writes"]:
            a[at] = v
        if "w" in it["writes"]:
            w[it["y"][1] + bw + wcols] = lam


def aligned_w_parts(pa, o, ow):
    """W parts with the batch boxes of A's parts (whole columns): the aligned per-site case"""
    out = []
    for f, s in pa:
        if 0 in s:
            out.append([[0] * len(ow), [0] * len(ow)])
            continue
        out.append([[f[o.index(c)] if c in "xy" else 0 for c in ow],
                    [s[o.index(c)] if c in "xy" else EXT_OF[c] for c in ow]])
    return np.array(out, dtype=np.int32)


EXT_OF = {}


def random_case(rng, world, ncomp, wkind):
    T = np.dtype([np.float64, np.complex128][rng.integers(2)])
    ext = dict(c=int(rng.integers(1, 4)), s=int(rng.integers(1, 3)))
    ext.update(C=ext["s"], S=ext["c"], x=int(rng.integers(1, 4)), y=int(rng.integers(1, 3)))
    o = "".join(rng.permutation(list("xcsyCS")))
    ow = "".join(rng.permutation(list("xySC")))
    case = dict(T=T, co=int(rng.integers(2)), o=o, ow=ow, ext=ext, ncomp=ncomp)
    case["pa"] = random_parts(rng, [ext[c] for c in o], world * ncomp)
    EXT_OF.clear()
    EXT_OF.update(ext)
    if wkind == "aligned":
        case["pw"] = aligned_w_parts(case["pa"], o, ow)
    elif wkind == "replicated":
        case["pw"] = np.array([[[0] * 4, [ext[c] for c in ow]]] * (world * ncomp), dtype=np.int32)
    else:
        case["pw"] = random_parts(rng, [ext[c] for c in ow], world * ncomp)
    return case


def plan_of(case, world, rank):
    n = case["ncomp"]
    return sb.dense_plan(sb.EIGH, DT[case["T"]], case["pa"], n, case["o"], "cs", "SC", case["co"], world, rank,
                         py=case["pw"], ncomponentsy=n, oy=case["ow"])


def run_plans(case, world, a_full, eigh):
    T, co, n = case["T"], case["co"], case["ncomp"]
    plans = [plan_of(case, world, r) for r in range(world)]
    p = plans[0]
    for q in plans:
        assert all(q[f] == p[f] for f in ("nothing", "gather_a", "gather_x", "slots"))
    va = D.components(a_full, case["pa"], co)
    w0 = np.full([case["ext"][c] for c in case["ow"]], np.nan)
    vw = D.components(w0, case["pw"], co)
    if p["gather_a"]:
        aslot = [[np.zeros(max(it["a"][2], 1), T) for it in sorted(q["items"], key=lambda i: i["slot"])]
                 + [np.zeros(0, T)] * (p["slots"] - len(q["items"])) for q in plans]
        run_ranks([q["gather_a_plan"] for q in plans], va, [s for r in aslot for s in r], n, p["slots"], 1, 0, T, T)
    for r, q in enumerate(plans):
        # W-only items first: they read A in place before the other items overwrite it
        assert [it["writes"] for it in q["items"]] == sorted((it["writes"] for it in q["items"]),
                                                              key=lambda x: x != "w")
        for it in q["items"]:
            a = va[r * n + it["a"][0]] if it["a"][0] >= 0 else aslot[r][it["slot"]]
            w = None
            if "w" in it["writes"]:
                w = vw[r * n + it["y"][0]] if it["y"][0] >= 0 else np.zeros(max(it["y"][2], 1))
            else:
                assert it["y"] == (-1, 0, 0)
            run_item(it, a, w, eigh)
            if it["back"]:
                b = it["back"]
                src, dst = (w, vw) if it["writes"] == "w" else (a, va)
                dst[r * n + it["comp"]][_indices(b["size"], b["dstride"], 0)] = src[_indices(b["size"], b["sstride"],
                                                                                           b["soff"])]
    return plans, va, vw


def check_parts(comps, parts, full, co):
    """Every part holds exactly its box of `full` (replicated parts: the same bits)"""
    for c, (f, s) in zip(comps, parts):
        if 0 in s:
            continue
        box = full[tuple(slice(a, a + b) for a, b in zip(f, s))]
        assert np.array_equal(np.asarray(c).reshape(s, order="F" if co == D.FastToSlow else "C"), box)


@pytest.mark.parametrize("wkind", ["aligned", "replicated", "random"])
@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_eigh_plans(world, wkind):
    rng = np.random.default_rng(900 + world + 10 * len(wkind))
    seen = set()
    for k in range(30):
        case = random_case(rng, world, int(rng.integers(1, 3)), wkind)
        o, ow, co, T, ext = case["o"], case["ow"], case["co"], case["T"], case["ext"]
        _, h = D.as_matrices(np.zeros([ext[c] for c in o]), o, "cs", "SC", co)
        h = E.hermitian(rng, T, h.shape[-1], "random", h.shape[:-2])
        a_full = D.from_matrices(h, o, [ext[c] for c in o], "cs", "SC", co).astype(T)
        plans, va, vw = run_plans(case, world, a_full, Eigh())
        got_a = D.assemble(va, case["pa"], a_full, co)
        got_w = D.assemble(vw, case["pw"], np.full([ext[c] for c in ow], np.nan), co)
        check_parts(va, case["pa"], got_a, co)
        check_parts(vw, case["pw"], got_w, co)
        _, v = D.as_matrices(got_a, o, "cs", "SC", co)
        wt = np.transpose(got_w, [ow.index(c) for c in [c for c in o if c in "xy"] + list("SC"[::-1] if co == D.FastToSlow else "SC")])
        E.check(h, wt.reshape(h.shape[:-1]), v, T, (world, k, case))
        steps = [sb.dense_steps(sb.EIGH, DT[T], case["pa"], case["ncomp"], o, "cs", "SC", co, world, r,
                                py=case["pw"], ncomponentsy=case["ncomp"], oy=ow) for r in range(world)]
        p = plans[0]
        for r, s in enumerate(steps):
            assert s["exchanges"] == p["gather_a"] and s["steps"] == 1 + p["gather_a"]
            assert len(s["item_steps"]) == len(plans[r]["items"])
        seen.add("gather" if p["gather_a"] else "in place")
        items = [i for q in plans for i in q["items"]]
        seen |= {i["writes"] for i in items}
        if any(i["writes"] == "w" and i["back"] for i in items):
            seen.add("w back")
    want = {"in place", "gather", "aw"}
    if wkind != "aligned" and world > 1:
        want |= {"w", "a"}
    if wkind == "random":
        want.add("w back")
    assert want <= seen, seen


def single(dims):
    return np.array([[[0] * len(dims), list(dims)]], dtype=np.int32)


def plan1(o="xcC", dims=(2, 3, 3), ow="xC", wdims=(2, 3), dtype=sb.F64, orows="c", ocols="C"):
    return sb.dense_plan(sb.EIGH, dtype, single(dims), 1, o, orows, ocols, sb.FastToSlow, 1, 0,
                         py=single(wdims), ncomponentsy=1, oy=ow)


def test_eigh_plan_describe():
    p = plan1()
    assert p["op"] == "eigh" and p["gather_a"] == 0 and p["gather_x"] == 0
    (it,) = p["items"]
    assert it["writes"] == "aw" and it["back"] is None
    assert it["B"] == [(2, 1, 0, 1)] and it["C"] == [(3, 6, 0, 2)] and it["R"] == [(3, 2, 0, 0)]
    assert it["kernel"].startswith("dense eigh tier=warp n=3 batch=2 rhs=0 chunk=0 teams=2 ")
    big = plan1(dims=(1, 64, 64), wdims=(1, 64), dtype=sb.C128)["items"][0]
    assert big["kernel"].startswith("dense eigh tier=cta n=64 batch=1 ")
    assert sb.dense_steps(sb.EIGH, sb.F64, single([2, 3, 3]), 1, "xcC", "c", "C", sb.FastToSlow, 1, 0,
                          py=single([2, 3]), ncomponentsy=1, oy="xC") == dict(steps=1, exchanges=0, item_steps=[0])


def test_eigh_plan_errors():
    with pytest.raises(RuntimeError, match="eigh: w lacks the batch label `x` of the matrix"):
        plan1(ow="C", wdims=(3,))
    with pytest.raises(RuntimeError, match="eigh: w lacks the column label `C` of the matrix"):
        plan1(ow="x", wdims=(2,))
    with pytest.raises(RuntimeError, match="eigh: w has the label `c`, which is neither a batch nor a column label"):
        plan1(ow="xcC", wdims=(2, 3, 3))
    with pytest.raises(RuntimeError, match="eigh: w has the label `q`, which is neither"):
        plan1(ow="xCq", wdims=(2, 3, 4))
    with pytest.raises(RuntimeError, match="eigh: dimension of label `x` does not match"):
        plan1(wdims=(3, 3))
    with pytest.raises(RuntimeError, match="eigh: dimension of label `C` does not match"):
        plan1(wdims=(2, 4))
    with pytest.raises(RuntimeError, match="eigh: the matrix is not square: 3 rows, 2 columns"):
        plan1(dims=(2, 3, 2), wdims=(2, 2))
    with pytest.raises(RuntimeError, match="eigh: unsupported type"):
        plan1(dtype=sb.I32)
    for dtype, n in ((sb.C128, 80), (sb.F64, 113), (sb.C64, 113), (sb.F32, 160)):
        plan1(dims=(1, n, n), wdims=(1, n), dtype=dtype)
        msg = ("eigh: order n = %d is over the limit: the matrix and its eigenvectors must fit in shared memory, "
               "2 n^2 * sizeof(T) <= 204800 bytes (n <= 80 for complex double, 113 for double and complex float, "
               "160 for float)" % (n + 1))
        with pytest.raises(RuntimeError) as e:
            plan1(dims=(1, n + 1, n + 1), wdims=(1, n + 1), dtype=dtype)
        assert str(e.value) == msg


def test_every_rank_throws_when_one_ranks_w_is_wrong():
    """Rank 1's part of w has a batch extent that does not match the matrix: both ranks refuse."""
    pa = np.array([[[0, 0, 0], [2, 3, 3]]] * 2, dtype=np.int32)
    pw = np.array([[[0, 0], [2, 3]], [[0, 0], [3, 3]]], dtype=np.int32)
    for rank in range(2):
        with pytest.raises(RuntimeError, match="dimension of label `x` does not match"):
            sb.dense_plan(sb.EIGH, sb.F64, pa, 1, "xcC", "c", "C", sb.FastToSlow, 2, rank, py=pw, ncomponentsy=1,
                          oy="xC")


@pytest.mark.parametrize("mpi", [False, True])
def test_cxx_eigh_overloads_compile(mpi):
    """tests/cxx/dense_eigh_dropin_test.cpp -- superbblas::eigh without a communicator and, with
    SUPERBBLAS_USE_MPI, its MPI overload against the stand-in tests/cxx/mpi_stub/mpi.h -- is valid against
    include/superbblas.h with plain g++ (syntax and template instantiation; the GPU tests run it)."""
    cuda_inc = "/usr/local/cuda/include"
    if not shutil.which("g++") or not os.path.exists(os.path.join(cuda_inc, "cuda_runtime.h")):
        pytest.skip("needs g++ and the CUDA headers")
    cxx = os.path.join(ROOT, "tests", "cxx")
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall"] + (["-DSUPERBBLAS_USE_MPI"] if mpi else []) +
                       ["-I" + os.path.join(cxx, "mpi_stub"), "-I" + os.path.join(ROOT, "include"), "-I" + cuda_inc,
                        os.path.join(cxx, "dense_eigh_dropin_test.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
