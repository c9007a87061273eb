"""Host logic of the contraction driver without a GPU: every rank's plan (items, the other operand
used in place or re-partitioned, the result written directly or reduced from partials, beta
scaling) is executed in numpy and compared with the oracle for 1 to 4 simulated ranks; and the
argument errors, which every rank throws before any data moves."""
import numpy as np
import pytest

import superbblas_b200 as sb
from oracle import oracle as O
from tests import cases as C
from tests.plan_exec import _indices, run_ranks
from tests.test_gpu_contraction import TOL, close

DTYPE = {np.dtype(np.float32): sb.F32, np.dtype(np.float64): sb.F64,
         np.dtype(np.complex64): sb.C64, np.dtype(np.complex128): sb.C128}


def plan_of(case, nranks, rank, ncomp):
    return sb.contraction_plan(
        DTYPE[case["T"]], case["alpha"], case["p0"], case["from0"], case["size0"], case["dim0"], ncomp,
        case["o0"], case["conj0"], case["p1"], case["from1"], case["size1"], case["dim1"], ncomp,
        case["o1"], case["conj1"], case["beta"], case["pr"], case["fromr"], case["sizer"], case["dimr"],
        ncomp, case["o_r"], case["co"], nranks, rank)


def grid_index(dims, which, off):
    """Element index, in operand `which` (0: v0, 1: v1, 2: vr), of every point of the dims' grid."""
    idx = np.full([d[0] for d in dims], off, dtype=np.int64)
    for k, d in enumerate(dims):
        shape = [1] * len(dims)
        shape[k] = d[0]
        idx = idx + (np.arange(d[0], dtype=np.int64) * d[1 + which]).reshape(shape)
    return idx


def run_item(it, case, x, x_off, y, y_off, out, out_off, beta):
    """What sbk_contract computes for the item: out = alpha * sum_K f0(x) f1(y) (+ beta * out)."""
    dims = it["T"] + it["M"] + it["N"] + it["K"]
    nfree = len(dims) - len(it["K"])
    a = x[grid_index(dims, 0, x_off)].astype(np.complex128)
    b = y[grid_index(dims, 1, y_off)].astype(np.complex128)
    acc = ((a.conj() if case["conj0"] else a) * (b.conj() if case["conj1"] else b)).sum(
        axis=tuple(range(nfree, len(dims))))
    ri = grid_index(dims[:nfree], 2, out_off)
    val = complex(case["alpha"]) * acc
    if beta is not None:
        val = val + complex(beta) * out[ri]
    out[ri] = val if case["T"].kind == "c" else val.real


def run_contraction_plans(case, world, ncomp, seed):
    """Every rank's plan in numpy, in the executor's order; -> (result parts, plans)."""
    T = case["T"]
    v0, v1, vr = C.make_contraction_data(case, seed)
    out = [x.copy() for x in vr]
    plans = [plan_of(case, world, r, ncomp) for r in range(world)]
    flags = ("nothing", "big0", "direct", "repartition", "reduction", "slots")
    for p in plans:
        assert all(p[f] == plans[0][f] for f in flags), "ranks disagree on a collective decision"
    p = plans[0]
    if p["nothing"]:
        return out, plans
    big, small = (v0, v1) if p["big0"] else (v1, v0)
    empty = lambda: [[np.zeros(0, T) for _ in range(p["slots"])] for _ in range(world)]

    # 1. the other operand into the re-partition slots
    slots = empty()
    for r, q in enumerate(plans):
        for it in q["items"]:
            if it["small"][0] < 0:
                slots[r][it["slot"]] = np.zeros(it["small_elems"], T)
    if p["repartition"]:
        run_ranks([q["repartition_plan"] for q in plans], small, [s for r in slots for s in r],
                  ncomp, p["slots"], 1, 0, T, T)
    # 2. beta, in place
    for r, q in enumerate(plans):
        for b in q["beta"]:
            part = out[r * ncomp + b["comp"]]
            i = _indices(b["size"], b["stride"], b["off"])
            part[i] = O._scale(case["beta"], part[i], T)
    # 3. the items: direct into the result, with beta; else into a partial slot
    partial = empty()
    for r, q in enumerate(plans):
        for it in q["items"]:
            (bc, boff), (sc, soff), (oc, ooff) = it["big"], it["small"], it["out"]
            xb = big[r * ncomp + bc]
            xs = small[r * ncomp + sc] if sc >= 0 else slots[r][it["slot"]]
            if oc >= 0:
                dst, beta = out[r * ncomp + oc], case["beta"]
            else:
                dst = partial[r][it["slot"]] = np.zeros(it["out_elems"], T)
                beta = None
            if p["big0"]:
                run_item(it, case, xb, boff, xs, soff, dst, ooff, beta)
            else:
                run_item(it, case, xs, soff, xb, boff, dst, ooff, beta)
    # 4. the partials added into the result
    if p["reduction"]:
        run_ranks([q["reduction_plan"] for q in plans], [x for r in partial for x in r], out,
                  p["slots"], ncomp, 1, 1, T, T)
    return out, plans


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_contraction_plans_match_oracle(world):
    rng = np.random.default_rng(900 + world)
    seen = set()
    for it in range(40):
        ncomp = int(rng.integers(1, 3))
        case = C.random_contraction_case(rng, nparts=world * ncomp)
        got, plans = run_contraction_plans(case, world, ncomp, 50 * world + it)
        want = C.oracle_contraction(case, *C.make_contraction_data(case, 50 * world + it))
        ok, err = close(got, want, TOL[case["T"]])
        assert ok, (world, it, err, case)
        p = plans[0]
        if not p["nothing"]:
            items = [i for q in plans for i in q["items"]]
            seen |= {name for name, hit in (
                ("in place", any(i["small"][0] >= 0 for i in items)),
                ("repartition", p["repartition"]), ("direct", p["direct"]),
                ("reduction", p["reduction"]), ("beta", any(q["beta"] for q in plans))) if hit}
    assert seen == {"in place", "repartition", "direct", "reduction", "beta"}, seen


def _single(dim):
    return np.array([[[0] * len(dim), list(dim)]], dtype=np.int32)


def test_group_limit_is_checked_on_every_rank():
    """Nine contracted labels of extent > 1 in rank 0's item, eight in rank 1's (there `a` has extent
    1 and is dropped): both ranks refuse the contraction, before anything is staged or exchanged."""
    d0, d1, dr = [3] + [2] * 8 + [4], [3] + [2] * 8 + [3], [4, 3]
    p0 = np.array([[[0] * 10, [2] + d0[1:]], [[2] + [0] * 9, [1] + d0[1:]]], dtype=np.int32)
    p1 = np.array([[[0] * 10, d1]] * 2, dtype=np.int32)
    pr = np.array([[[0, 0], dr]] * 2, dtype=np.int32)
    for rank in range(2):
        with pytest.raises(RuntimeError, match="contraction: too many labels in a group"):
            sb.contraction_plan(sb.F64, 1, p0, [0] * 10, d0, d0, 1, "abcdefghix", False, p1, [0] * 10, d1,
                                d1, 1, "abcdefghiy", False, 0, pr, [0, 0], dr, dr, 1, "xy", sb.FastToSlow,
                                2, rank)


def test_contraction_plan_errors():
    d = [2, 2]

    def plan(o0, o1, o_r, size1=d):
        return sb.contraction_plan(sb.F64, 1, _single(d), [0, 0], d, d, 1, o0, False, _single(d),
                                   [0, 0], size1, d, 1, o1, False, 0, _single(d), [0, 0], d, d, 1, o_r,
                                   sb.FastToSlow, 1, 0)
    with pytest.raises(RuntimeError, match="unmatched"):
        plan("ab", "bc", "cz")
    with pytest.raises(RuntimeError, match="does not match"):
        plan("ab", "bc", "ac", size1=[2, 1])
    with pytest.raises(RuntimeError, match="contraction: repeated label in an order"):
        plan("aa", "bc", "ac")
