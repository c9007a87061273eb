"""The steps of the dense solvers as requests (sbb_cholesky_begin, ...), host only: every rank of 1 to 4
simulated ranks takes the same number of steps, one per gather after the begin, and every item is queued in
the step that the printed gather plans give it -- behind the local part of a gather only when no other rank
sends into its slot."""
import numpy as np
import pytest

import superbblas_b200 as sb
from tests.test_dense_plan import OPS, DT, random_case, plan_of


def steps_of(case, world, rank, ncomp):
    kw = {}
    if "ox" in case:
        kw = dict(px=case["px"], ncomponentsx=ncomp, ox=case["ox"], py=case["py"], ncomponentsy=ncomp,
                  oy=case["oy"])
    return sb.dense_steps(OPS[case["op"]], DT[case["T"]], case["pa"], ncomp, case["o"], case["orows"],
                          case["ocols"], case["co"], world, rank, alpha=case["alpha"], **kw)


def expected_steps(plan, rank):
    """The step of every item, by brute force from the unpack ops of the printed gathers"""
    gathers = [plan[k + "_plan"][0] for k in ("gather_a", "gather_x") if plan[k]]
    remote = [{op["dst"] - rank * plan["slots"] for op in ops if op["kind"] == "unpack"} for ops in gathers]
    out = []
    for it in plan["items"]:
        k = 0
        for g, r in enumerate(remote):
            k = max(k, g + 1 if it["slot"] in r else g)
        out.append(k)
    return out


@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("ncomp", [1, 2])
def test_every_rank_takes_the_same_steps(world, ncomp):
    rng = np.random.default_rng(300 + 10 * world + ncomp)
    seen_split = 0
    for _ in range(40):
        case = random_case(rng, world, ncomp)
        plans = [plan_of(case, world, r, ncomp) for r in range(world)]
        steps = [steps_of(case, world, r, ncomp) for r in range(world)]
        if plans[0]["nothing"]:
            assert all(s is None for s in steps)
            continue
        for r, (p, s) in enumerate(zip(plans, steps)):
            assert s["exchanges"] == p["gather_a"] + p["gather_x"]
            assert s["steps"] == s["exchanges"] + 1 == steps[0]["steps"]
            assert s["item_steps"] == expected_steps(p, r)
            assert all(0 <= k <= s["exchanges"] for k in s["item_steps"])
            seen_split += 0 < len(set(s["item_steps"])) and min(s["item_steps"], default=0) < s["exchanges"]
    if world > 1:
        assert seen_split > 0  # some items run during an exchange


def test_split_matrix_and_vectors_on_two_ranks():
    """Two ranks: cholesky of matrices split along their rows gathers A in one exchange, and every item
    waits for it; trsm with replicated matrices and x, y cut along the batch label gathers nothing; with x
    cut along its rows it gathers x, and every item waits for the other rank's rows."""
    # "abx": a rows, b columns, x batch; x "arx" and y "brx" with r right-hand sides
    pa = np.array([[[0, 0, 0], [2, 4, 3]], [[2, 0, 0], [2, 4, 3]]], np.int32)
    chol = [sb.dense_steps(sb.CHOLESKY, sb.C128, pa, 1, "abx", "a", "b", sb.FastToSlow, 2, r) for r in (0, 1)]
    assert [s["steps"] for s in chol] == [2, 2]
    assert [s["item_steps"] for s in chol] == [[1], [1]]
    # replicated matrices, x and y cut along the batch label: A is in place, nothing is gathered
    pxy = np.array([[[0, 0, 0], [4, 2, 2]], [[0, 0, 2], [4, 2, 1]]], np.int32)
    pab = np.array([[[0, 0, 0], [4, 4, 3]]] * 2, np.int32)
    s = sb.dense_steps(sb.TRSM, sb.C128, pab, 1, "abx", "a", "b", sb.FastToSlow, 2, 0, px=pxy, ncomponentsx=1,
                       ox="arx", py=pxy, ncomponentsy=1, oy="brx")
    assert s == dict(steps=1, exchanges=0, item_steps=[0])
    # x cut along its row label, y along the batch label: X is gathered and every item needs the other rank
    px = np.array([[[0, 0, 0], [2, 2, 3]], [[2, 0, 0], [2, 2, 3]]], np.int32)
    for r in (0, 1):
        s = sb.dense_steps(sb.TRSM, sb.C128, pab, 1, "abx", "a", "b", sb.FastToSlow, 2, r, px=px, ncomponentsx=1,
                           ox="arx", py=pxy, ncomponentsy=1, oy="brx")
        assert s == dict(steps=2, exchanges=1, item_steps=[1])



@pytest.mark.parametrize("mpi", [False, True])
def test_cxx_request_overloads_compile(mpi):
    """tests/cxx/dense_request_test.cpp -- the C++ dense solvers with and without a Request, and with
    SUPERBBLAS_USE_MPI their MPI overloads against the stand-in tests/cxx/mpi_stub/mpi.h -- is valid
    against include/superbblas.h with plain g++ (syntax and template instantiation; the GPU tests run it)."""
    import os
    import shutil
    import subprocess
    if not shutil.which("g++"):
        pytest.skip("needs g++")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cxx = os.path.join(root, "tests", "cxx")
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall"] + (["-DSUPERBBLAS_USE_MPI"] if mpi else []) +
                       ["-I" + os.path.join(cxx, "mpi_stub"), "-I" + os.path.join(root, "include"),
                        os.path.join(cxx, "dense_request_test.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
