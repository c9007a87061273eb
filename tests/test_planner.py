"""Host logic without a GPU: the copy planner (geometry in range space, exactly-once Copy, ordered
Add, zero-fill of unsupported destinations, message layout) against the oracle, for one rank and
for several ranks simulated in one process."""
import os

import numpy as np
import pytest

os.environ.setdefault("SBB_CHUNK_BYTES", "192")  # cut remote boxes in pieces even in small cases

import superbblas_b200 as sb
from tests import cases as C
from tests.plan_exec import run_ranks


def run_planned(case, v0, v1, nranks):
    """Execute the plans of all ranks; messages are exchanged through a dict."""
    P0, P1 = case["p0"].shape[0], case["p1"].shape[0]
    assert P0 % nranks == 0 and P1 % nranks == 0
    nc0, nc1 = P0 // nranks, P1 // nranks
    out = [x.copy() for x in v1]
    alpha = case["alpha"]
    zero = np.real(alpha) == 0 and np.imag(alpha) == 0
    wire_t = case["T"] if (case["copyadd"] == 1 and case["T"] != case["Q"]) else case["Q"]
    plans = [sb.copy_plan(wire_t.itemsize, case["p0"], nc0, case["o0"], case["from0"],
                          case["size0"], case["dim0"], case["p1"], nc1, case["o1"], case["from1"],
                          case["dim1"], nranks, r, case["co"], case["copyadd"], zero)
             for r in range(nranks)]
    run_ranks(plans, v0, out, nc0, nc1, alpha, case["copyadd"], case["T"], case["Q"])
    return out


@pytest.mark.parametrize("seed", range(8))
def test_plan_single_rank_matches_oracle(seed):
    rng = np.random.default_rng(300 + seed)
    for it in range(60):
        case = C.random_copy_case(rng)
        v0, v1 = C.make_copy_data(case, seed * 100 + it, consistent=case["copyadd"] == 0)
        want = C.oracle_copy(case, v0, v1)
        got = run_planned(case, v0, v1, 1)
        for j, (g, w) in enumerate(zip(got, want)):
            assert C.bits_equal(g, w), (seed, it, j, case)


@pytest.mark.parametrize("nranks", [2, 3, 4])
def test_plan_multi_rank_matches_oracle(nranks):
    rng = np.random.default_rng(400 + nranks)
    for it in range(80):
        nc0, nc1 = int(rng.integers(1, 3)), int(rng.integers(1, 3))
        case = C.random_copy_case(rng, nparts0=nranks * nc0, nparts1=nranks * nc1)
        v0, v1 = C.make_copy_data(case, 7000 + it, consistent=case["copyadd"] == 0)
        want = C.oracle_copy(case, v0, v1)
        got = run_planned(case, v0, v1, nranks)
        for j, (g, w) in enumerate(zip(got, want)):
            assert C.bits_equal(g, w), (nranks, it, j, case)


def test_redistribution_and_shift_plans():
    """BASELINE configs 3 and 5 at reduced size: t-slabs -> (z,t) blocks, and a periodic shift."""
    from oracle import oracle as O
    P = 8
    dim = [4, 4, 4, 8, 2, 3, 2]
    p0 = sb.basic_partitioning("xyztscn", dim, [1, 1, 1, P, 1, 1, 1], "t", P, 1)
    p1 = sb.basic_partitioning("xyztscn", dim, [1, 1, 2, P // 2, 1, 1, 1], "zt", P, 1)
    assert np.array_equal(p0, O.basic_partitioning("xyztscn", dim, [1, 1, 1, P, 1, 1, 1], "t", P, 1))
    case = dict(alpha=1, p0=p0, o0="xyztscn", from0=[0] * 7, size0=dim, dim0=dim, p1=p1,
                o1="xyztscn", from1=[0] * 7, dim1=dim, co=1, copyadd=0, T=np.dtype(np.complex64),
                Q=np.dtype(np.complex64))
    v0, v1 = C.make_copy_data(case, 1)
    want = C.oracle_copy(case, v0, v1)
    got = run_planned(case, v0, v1, P)
    assert all(C.bits_equal(g, w) for g, w in zip(got, want))
    # every rank sends/receives only what leaves the device
    ops, wire = sb.copy_plan(8, p0, 1, "xyztscn", [0] * 7, dim, dim, p1, 1, "xyztscn", [0] * 7, dim,
                             P, 0, 1, 0)
    assert sum(w[0] for w in wire.values()) + sum(np.prod(o["size"]) for o in ops
                                                   if o["kind"] == "local") == np.prod(p0[0, 1])

    dim = [4, 4, 4, 8, 4, 3]
    p = sb.basic_partitioning("xyztsc", dim, [1, 1, 2, 4, 1, 1], "zt", P, 1)
    for shift in ([1, 0, 0, 0, 0, 0], [0, 0, 1, 0, 0, 0], [0, 0, 0, 7, 0, 0], [1, 1, 1, 1, 0, 0]):
        case = dict(alpha=1, p0=p, o0="xyztsc", from0=[0] * 6, size0=dim, dim0=dim, p1=p,
                    o1="xyztsc", from1=shift, dim1=dim, co=1, copyadd=0, T=np.dtype(np.complex128),
                    Q=np.dtype(np.complex128))
        v0, v1 = C.make_copy_data(case, 2)
        want = C.oracle_copy(case, v0, v1)
        got = run_planned(case, v0, v1, P)
        assert all(C.bits_equal(g, w) for g, w in zip(got, want))


def test_halo_partition_plan():
    """dist.cpp:459-504: copy into / out of a halo-extended partition."""
    dim = [4, 4, 4, 8, 2]
    procs = [1, 1, 2, 2, 1]
    P = 4
    p0 = sb.basic_partitioning(dim, procs, P)
    p1 = sb.basic_partitioning(dim, procs, P, False, [1, 1, 1, 1, 0])
    for (pa, pb) in ((p0, p1), (p1, p0)):
        for copyadd in (0, 1):
            case = dict(alpha=1, p0=pa, o0="xyztc", from0=[0] * 5, size0=dim, dim0=dim, p1=pb,
                        o1="xyztc", from1=[0] * 5, dim1=dim, co=1, copyadd=copyadd,
                        T=np.dtype(np.float64), Q=np.dtype(np.float64))
            v0, v1 = C.make_copy_data(case, 3, consistent=copyadd == 0)
            want = C.oracle_copy(case, v0, v1)
            got = run_planned(case, v0, v1, P)
            assert all(C.bits_equal(g, w) for g, w in zip(got, want))


def test_errors_match_reference_messages():
    p = np.array([[[0, 0], [2, 2]]], dtype=np.int32)
    with pytest.raises(RuntimeError):
        sb.copy_plan(8, p, 1, "xyz", [0, 0], [2, 2], [2, 2], p, 1, "xy", [0, 0], [2, 2], 1, 0, 1, 0)
    with pytest.raises(RuntimeError, match="Invalid copy operation"):
        sb.copy_plan(8, p, 1, "xx", [0, 0], [2, 2], [2, 2], p, 1, "xy", [0, 0], [2, 2], 1, 0, 1, 0)
    with pytest.raises(RuntimeError, match="Invalid copy operation"):
        sb.copy_plan(8, p, 1, "xy", [0, 0], [2, 2], [2, 2], p, 1, "xz", [0, 0], [2, 2], 1, 0, 1, 0)
    with pytest.raises(RuntimeError, match="Invalid copy operation"):
        sb.copy_plan(8, p, 1, "xy", [0, 0], [3, 2], [2, 2], p, 1, "xy", [0, 0], [2, 2], 1, 0, 1, 0)
    with pytest.raises(RuntimeError, match="wtf"):
        sb.copy_plan(8, p, 2, "xy", [0, 0], [2, 2], [2, 2], p, 1, "xy", [0, 0], [2, 2], 1, 0, 1, 0)


def test_exchange_phases_are_a_proper_edge_colouring():
    """Every message of an exchange gets a phase (CopyPlan::send_phase) computed identically on all
    ranks; senders visit their receivers in phase order.  Proper: no two messages with the same
    phase share a sender or a receiver.  And the property the ordering is for: a sender with a single
    message owns phase 0 at its receiver (all senders start with their phase 0 at the same time)."""
    rng = np.random.default_rng(5)
    cases = []
    for world in (4, 8):
        dim = [4, 4, 4, 2 * world, 3]
        pa = sb.basic_partitioning("xyztc", dim, [1, 1, 1, world, 1], "t", world, 1)
        pb = sb.basic_partitioning("xyztc", dim, [1, 1, 2, world // 2, 1], "zt", world, 1)
        cases.append((world, dict(p0=pa, o0="xyztc", from0=[0] * 5, size0=dim, dim0=dim, p1=pb, o1="xyztc",
                                  from1=[0] * 5, dim1=dim, co=1, copyadd=0)))
    for _ in range(20):
        world = int(rng.integers(2, 7))
        cases.append((world, C.random_copy_case(rng, nparts0=world, nparts1=world)))
    for world, case in cases:
        edges = {}
        for rank in range(world):
            ph = {}
            _, wire = sb.copy_plan(8, case["p0"], 1, case["o0"], case["from0"], case["size0"], case["dim0"],
                                   case["p1"], 1, case["o1"], case["from1"], case["dim1"], world, rank,
                                   case["co"], case["copyadd"], phases=ph)
            for peer, phase in ph.items():
                assert peer != rank and wire[peer][0] > 0
                edges[(rank, peer)] = phase
        for (s0, r0), c0 in edges.items():
            for (s1, r1), c1 in edges.items():
                if (s0, r0) != (s1, r1) and c0 == c1:
                    assert s0 != s1 and r0 != r1, (edges,)
        outdeg = {s: sum(1 for e in edges if e[0] == s) for s in range(world)}
        for (s, r), c in edges.items():
            if outdeg[s] == 1 and all(outdeg[s2] >= 1 for (s2, r2) in edges if r2 == r):
                single_to_r = [s2 for (s2, r2) in edges if r2 == r and outdeg[s2] == 1]
                if len(single_to_r) == 1:
                    assert c == 0, (edges, s, r)
