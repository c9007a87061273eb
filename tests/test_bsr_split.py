"""Host logic of the interior / boundary split of bsr_krylov's block rows without a GPU.  With a request,
bsr_krylov runs the interior rows of power 0 while the gather of x is in flight and the boundary rows
once it is complete, so a row may be interior only if none of its blocks reads a point that the gather
fills from another rank.  For random plain and Kronecker operators on 1 to 4 simulated ranks, the split
bsr_split returns is checked against the printed gather plan by brute force over the points, and every
rank's plan is executed in numpy with the interior rows reading a slot in which every point that comes
from another rank is NaN."""
import numpy as np
import pytest

import superbblas_b200 as sb
from tests import bsr_cases as B
from tests import test_bsr_plan as P
from tests import test_kron_bsr_plan as KP
from tests.plan_exec import _indices, run_ranks


def plan_and_split(c, world, rank, ncomp, kron):
    """(plan, split) of `rank`: bsr_plan / kron_bsr_plan and bsr_split with the same arguments"""
    pdom = np.array([[[0] * len(c["dimd"]), c["dimd"]]] * world * ncomp, dtype=np.int32)
    args = (P.DT[c["T"]], c["pim"], c["dimi"], pdom, c["dimd"], ncomp, c["blockim"], c["blockdom"], c["imfast"],
            *B.flat_arrays(c["ops"]), c["oim"], c["odom"], c["px"], ncomp, c["ox"], [0] * len(c["ox"]),
            list(c["x"].shape), list(c["x"].shape), c["py"], ncomp, c["oy"], c["fromy"], c["sizey"],
            list(c["y0"].shape), c["power"], c["co"], world, rank)
    kw = dict(alpha=c["alpha"], beta=c["beta"])
    plan = KP.kron_plan_of(c, world, rank, ncomp) if kron else P.plan_of(c, world, rank, ncomp)
    if kron:
        kw.update(kronim=c["kronim"], krondom=c["krondom"])
    return plan, sb.bsr_split(*args, **kw)


def remote_elements(plan, rank, ncomp, comp):
    """Elements of the slot of `comp` that the printed gather of x fills from another rank"""
    ops = plan["gather"][0][0]
    idx = [_indices(o["size"], o["dstride"], o["doff"]) for o in ops
           if o["kind"] == "unpack" and o["dst"] == rank * ncomp + comp]
    return np.unique(np.concatenate(idx)) if idx else np.zeros(0, np.int64)


def block_points(it, kron):
    """Gathered-input points of a block relative to its first one"""
    return KP.kron_points(it) if kron else P.offsets(it["D"])


def output_index(it, r, base, kron):
    cp = P.offsets(it["C"])
    img = KP.kron_image(it, r) if kron else P.image_offsets(it, r)
    return (base + img[:, None] + cp[None, :]).reshape(-1)


def cases(seed, world, kron, n):
    rng = np.random.default_rng(seed)
    for k in range(n):
        kind = ["direct", "back", "power"][k % 3]
        ncomp = int(rng.integers(1, 3))
        make = KP.random_kron_case if kron else P.random_case
        yield k, kind, ncomp, make(rng, world, ncomp, kind)


@pytest.mark.parametrize("kron", [False, True])
@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_split_follows_the_gather_plan(world, kron):
    nsplit = 0
    for k, kind, ncomp, c in cases(3100 + world + 10 * kron, world, kron, 12):
        for rank in range(world):
            plan, split = plan_and_split(c, world, rank, ncomp, kron)
            if plan["nothing"]:
                assert split == []
                continue
            assert [s["comp"] for s in split] == [it["comp"] for it in plan["items"]]
            for it, s in zip(plan["items"], split):
                inter, bound = s["interior"], s["boundary"]
                assert inter == sorted(inter) and bound == sorted(bound)
                assert not set(inter) & set(bound)
                assert sorted(inter + bound) == list(range(it["rows"])), (world, k, rank)
                remote = set((remote_elements(plan, rank, ncomp, it["comp"]) // it["ncols"]).tolist())
                pts = block_points(it, kron)
                rp, goff = it["rowptr"], it["goff"]
                want = [r for r in range(it["rows"])
                        if any(remote & set((goff[b] + pts).tolist()) for b in range(rp[r], rp[r + 1]))]
                assert bound == want, (world, k, kind, rank, it["comp"])
                if world == 1:
                    assert bound == []
                nsplit += bool(inter) and bool(bound)
    if world > 1:
        assert nsplit > 0  # some launches do have both kinds of rows


def run_split_plans(c, world, ncomp, kron):
    """test_bsr_plan.run_plans, with power 0 computed as bsr_krylov's request runs it: the interior rows
    on a slot whose points from other ranks are still NaN, then the boundary rows on the complete slot"""
    T, co = c["T"], c["co"]
    ps = [plan_and_split(c, world, r, ncomp, kron) for r in range(world)]
    plans = [p for p, _ in ps]
    kernel = KP.kron_kernel(c["kronv"]) if kron else P.run_item
    xs = B.components(c["x"], c["px"], co)
    ys = B.components(c["y0"], c["py"], co)
    p0 = plans[0]
    if p0["nothing"]:
        return B.assemble(ys, c["py"], c["y0"], co)
    items = {(r, it["comp"]): (it, s) for r, (q, sp) in enumerate(ps) for it, s in zip(q["items"], sp)}
    slot = [np.zeros(max(items[(r, k)][0]["x"], 1) if (r, k) in items else 0, T)
            for r in range(world) for k in range(ncomp)]
    temp = [np.zeros(max(items[(r, k)][0]["y"][3], 1) if (r, k) in items else 0, T)
            for r in range(world) for k in range(ncomp)]
    for p in range(p0["powers"]):
        run_ranks([q["gather"][p] for q in plans], xs if p == 0 else ys, slot, ncomp, ncomp, 1, 0, T, T)
        if p in p0["fill"]:
            run_ranks([q["fill"][p] for q in plans], ys, temp, ncomp, ncomp, 1, 0, T, T)
        for (r, k), (it, s) in items.items():
            if p0["direct"]:
                out, base = ys[r * ncomp + it["y"][0]], it["y"][1] + p * it["y"][2]
            else:
                out, base = temp[r * ncomp + k], 0
            v, xg = c["ops"][r * ncomp + k][2], slot[r * ncomp + k]
            if p > 0:
                kernel(it, v, xg, out, base, c["alpha"], c["beta"])
                continue
            local = xg.copy()
            local[remote_elements(plans[r], r, ncomp, k)] = np.nan
            for rows, x in ((s["interior"], local), (s["boundary"], xg)):
                tmp = out.copy()
                kernel(it, v, x, tmp, base, c["alpha"], c["beta"])
                for row in rows:
                    o = output_index(it, row, base, kron)
                    out[o] = tmp[o]
        if not p0["direct"]:
            run_ranks([q["back"][p] for q in plans], temp, ys, ncomp, ncomp, 1, 0, T, T)
    return B.assemble(ys, c["py"], c["y0"], co)


@pytest.mark.parametrize("kron", [False, True])
@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_interior_then_boundary_matches_oracle(world, kron):
    for k, kind, ncomp, c in cases(3200 + world + 10 * kron, world, kron, 9):
        got = run_split_plans(c, world, ncomp, kron)
        if kron:
            want = KP.want_of(c)
        else:
            a = B.operator_matrix(c["ops"], c["pim"], c["dimi"], c["dimd"], c["blockim"], c["blockdom"],
                                  c["imfast"], c["co"])
            want = B.apply(a, c["oim"], c["odom"], c["x"], c["ox"], c["y0"], c["oy"], c["alpha"], c["beta"],
                           c["power"], 3 if c["power"] else 1, c["fromy"])
        assert np.array_equal(np.isnan(got), np.isnan(want)), (world, k, kind)
        assert B.rel_err(np.nan_to_num(got), np.nan_to_num(want)) < 1e-12, (world, k, kind)


def test_plan_text_is_unchanged_by_the_split():
    """bsr_split reads the plan; bsr_plan's text for the same arguments stays what it was"""
    rng = np.random.default_rng(3300)
    c = P.random_case(rng, 2, 1, "direct")
    before = P.plan_of(c, 2, 0, 1)
    plan_and_split(c, 2, 0, 1, False)
    assert P.plan_of(c, 2, 0, 1) == before
