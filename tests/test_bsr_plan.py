"""Host logic of the block-sparse operators without a GPU: every rank's plan of bsr_krylov (halo
gather of x or of the previous power, kernel straight into y or into temporaries added back into y) is
executed in numpy for 1 to 4 simulated ranks, with the kernel as a numpy product over the row
pointers and block offsets create_bsr computes, and compared with the oracle of tests/bsr_cases.py;
and the argument errors, which every rank throws alike."""
import numpy as np
import pytest

import superbblas_b200 as sb
from tests import bsr_cases as B
from tests.plan_exec import run_ranks

DT = {np.dtype(np.float32): sb.F32, np.dtype(np.float64): sb.F64, np.dtype(np.complex64): sb.C64,
      np.dtype(np.complex128): sb.C128}


def offsets(dims):
    """Offsets of every linear index over (size, stride..) dims, first fastest"""
    o = np.zeros(1, np.int64)
    for d in dims:
        o = (o[None, :] + (np.arange(d[0], dtype=np.int64) * d[-1])[:, None]).reshape(-1)
    return o


def image_offsets(it, r):
    o = np.zeros(1, np.int64)
    for nb, bs, st in it["I"]:
        b = r % nb
        r //= nb
        o = (o[None, :] + ((b * bs + np.arange(bs, dtype=np.int64)) * st)[:, None]).reshape(-1)
    return o


def run_item(it, v, xg, out, base, alpha, beta):
    """What the kernel computes for one item, on flat numpy storages"""
    bi, bd, nc = it["bi"], it["bd"], it["ncols"]
    dp, cp = offsets(it["D"]), offsets(it["C"])
    rp, goff = it["rowptr"], it["goff"]
    for r in range(it["rows"]):
        acc = np.zeros((bi, nc), np.complex128)
        for b in range(rp[r], rp[r + 1]):
            blk = v[b * bi * bd:(b + 1) * bi * bd]
            m = blk.reshape(bd, bi).T if it["imfast"] else blk.reshape(bi, bd)
            acc += m @ xg[(goff[b] + dp)[:, None] * nc + np.arange(nc)[None, :]]
        o = base + image_offsets(it, r)[:, None] + cp[None, :]
        res = alpha * acc + (beta * out[o] if beta != 0 else 0)
        out[o] = res if out.dtype.kind == "c" else res.real


def cuts_at(rng, n, step, parts):
    """`parts` boxes along one dimension of extent n, cut at multiples of step (some empty)"""
    cand = list(range(step, n, step))
    c = sorted(rng.choice(cand, size=min(parts - 1, len(cand)), replace=False).tolist()) if cand else []
    edges = [0] + c + [n]
    out = [(a, b - a) for a, b in zip(edges[:-1], edges[1:])]
    return out + [(0, 0)] * (parts - len(out))


def boxes(dims, k, cuts):
    out = []
    for f, s in cuts:
        ff, ss = [0] * len(dims), list(dims)
        ff[k], ss[k] = f, s
        if s == 0:
            ss = [0] * len(dims)
        out.append([ff, ss])
    return np.array(out, dtype=np.int32)


def random_case(rng, world, ncomp, kind, T=None):
    T = np.dtype([np.float64, np.complex128][rng.integers(2)] if T is None else T)
    co = int(rng.integers(2))
    imfast = bool(rng.integers(2))
    nparts = world * ncomp
    if kind == "power":
        dimi = dimd = [6, 4]
        blockim = blockdom = [3, 2]
    else:
        dimi, dimd = [8, 6], [6, 4, 2]
        blockim, blockdom = [2, 3], [3, 2, 1]
    oim, odom = "ab", "cdz"[:len(dimd)]
    pim = boxes(dimi, 0, cuts_at(rng, dimi[0], blockim[0], nparts))
    ops = B.random_operator(rng, pim, blockim, dimd, blockdom, T)
    ox = "".join(rng.permutation(list(odom + "n")))
    sizes = dict(zip(odom, dimd), n=3)
    x = B.rnd(rng, T, *[sizes[c] for c in ox])
    kx = int(rng.integers(len(ox)))
    px = boxes(list(x.shape), kx, cuts_at(rng, x.shape[kx], 1, nparts))
    oy = "".join(rng.permutation(list(oim + "n" + ("p" if kind == "power" else ""))))
    ysz = dict(zip(oim, dimi), n=3, p=4)
    ydims = [ysz[c] for c in oy]
    fromy = [0] * len(oy)
    sizey = list(ydims)
    if kind == "power":
        fromy[oy.index("p")] = int(rng.integers(4))
        sizey[oy.index("p")] = 3
    if kind == "direct":
        py = []
        for f, s in pim:
            if 0 in list(s):
                py.append([[0] * len(oy), [0] * len(oy)])
            else:
                py.append([[f[oim.index(c)] if c in oim else 0 for c in oy],
                           [s[oim.index(c)] if c in oim else ysz[c] for c in oy]])
        py = np.array(py, dtype=np.int32)
    else:
        k = int(rng.integers(len(oy)))
        py = boxes(ydims, k, cuts_at(rng, ydims[k], 1, nparts))
    beta = [0, 1, 0.5][rng.integers(3)]
    y0 = np.full(ydims, np.nan, T) if beta == 0 else B.rnd(rng, T, *ydims)
    return dict(T=T, co=co, imfast=imfast, dimi=dimi, dimd=dimd, blockim=blockim, blockdom=blockdom, oim=oim,
                odom=odom, pim=pim, ops=ops, ox=ox, x=x, px=px, oy=oy, y0=y0, py=py, fromy=fromy, sizey=sizey,
                power="p" if kind == "power" else None, alpha=1.5 if T.kind == "f" else 0.5 + 1j, beta=beta)


def plan_of(c, world, rank, ncomp):
    pdom = np.array([[[0] * len(c["dimd"]), c["dimd"]]] * world * ncomp, dtype=np.int32)
    return sb.bsr_plan(DT[c["T"]], c["pim"], c["dimi"], pdom, c["dimd"], ncomp, c["blockim"], c["blockdom"],
                       c["imfast"], *B.flat_arrays(c["ops"]), c["oim"], c["odom"], c["px"], ncomp, c["ox"],
                       [0] * len(c["ox"]), list(c["x"].shape), list(c["x"].shape), c["py"], ncomp, c["oy"],
                       c["fromy"], c["sizey"], list(c["y0"].shape), c["power"], c["co"], world, rank,
                       alpha=c["alpha"], beta=c["beta"])


def run_plans(c, world, ncomp, kernel=run_item):
    T, co = c["T"], c["co"]
    plans = [plan_of(c, world, r, ncomp) for r in range(world)]
    for p in plans:
        assert all(p[f] == plans[0][f] for f in ("nothing", "direct", "powers", "slots"))
    xs = B.components(c["x"], c["px"], co)
    ys = B.components(c["y0"], c["py"], co)
    p0 = plans[0]
    if p0["nothing"]:
        return plans, B.assemble(ys, c["py"], c["y0"], co)
    items = {(r, it["comp"]): it for r, q in enumerate(plans) for it in q["items"]}
    slot = [np.zeros(max(items[(r, k)]["x"], 1) if (r, k) in items else 0, T)
            for r in range(world) for k in range(ncomp)]
    temp = [np.zeros(max(items[(r, k)]["y"][3], 1) if (r, k) in items else 0, T)
            for r in range(world) for k in range(ncomp)]
    for p in range(p0["powers"]):
        run_ranks([q["gather"][p] for q in plans], xs if p == 0 else ys, slot, ncomp, ncomp, 1, 0, T, T)
        if p in p0["fill"]:
            run_ranks([q["fill"][p] for q in plans], ys, temp, ncomp, ncomp, 1, 0, T, T)
        for (r, k), it in items.items():
            if p0["direct"]:
                out, base = ys[r * ncomp + it["y"][0]], it["y"][1] + p * it["y"][2]
            else:
                out, base = temp[r * ncomp + k], 0
            kernel(it, c["ops"][r * ncomp + k][2], slot[r * ncomp + k], out, base, c["alpha"], c["beta"])
        if not p0["direct"]:
            run_ranks([q["back"][p] for q in plans], temp, ys, ncomp, ncomp, 1, 0, T, T)
    return plans, B.assemble(ys, c["py"], c["y0"], co)


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_bsr_plans_match_oracle(world):
    rng = np.random.default_rng(900 + world)
    seen = set()
    for k in range(24):
        kind = ["direct", "back", "power"][k % 3]
        ncomp = int(rng.integers(1, 3))
        c = random_case(rng, world, ncomp, kind)
        plans, got = run_plans(c, world, ncomp)
        a = B.operator_matrix(c["ops"], c["pim"], c["dimi"], c["dimd"], c["blockim"], c["blockdom"], c["imfast"],
                              c["co"])
        want = B.apply(a, c["oim"], c["odom"], c["x"], c["ox"], c["y0"], c["oy"], c["alpha"], c["beta"],
                       c["power"], 3 if c["power"] else 1, c["fromy"])
        assert np.array_equal(np.isnan(got), np.isnan(want)), (world, k, kind)   # NaN only outside the range
        assert B.rel_err(np.nan_to_num(got), np.nan_to_num(want)) < 1e-12, (world, k, kind)
        p = plans[0]
        seen.add("direct" if p["direct"] else "back")
        if p["fill"]:
            seen.add("fill")
        if p["powers"] > 1:
            seen.add("power " + ("direct" if p["direct"] else "back"))
    assert {"direct", "back", "fill", "power back"} <= seen, seen


def single(dims):
    return np.array([[[0] * len(dims), list(dims)]], dtype=np.int32)


def plan1(ii, jj, dims=(4, 4), blk=(2, 2), pim=None, ox="ABn", oy="abn", xdims=(4, 4, 2), ydims=(4, 4, 2),
          power=None, dtype=sb.F64, world=1, rank=0, dimd=None):
    dimd = list(dims) if dimd is None else dimd
    pim = single(dims) if pim is None else pim
    n = len(pim)
    pdom = np.array([[[0] * len(dimd), dimd]] * n, dtype=np.int32)
    px = np.array([[[0] * len(xdims), list(xdims)]] * n, dtype=np.int32)
    py = np.array([[[0] * len(ydims), list(ydims)]] * n, dtype=np.int32)
    return sb.bsr_plan(dtype, pim, list(dims), pdom, dimd, n // world, list(blk), [blk[0], blk[1]][:len(dimd)],
                       True, ii, jj, "ab", "AB"[:len(dimd)], px, n // world, ox, [0] * len(xdims), list(xdims),
                       list(xdims), py, n // world, oy, [0] * len(ydims), list(ydims), list(ydims), power,
                       sb.FastToSlow, world, rank)


def test_bsr_plan_errors():
    ok_ii, ok_jj = [1, 0, 0, 0], [2, -2]
    plan1(ok_ii, ok_jj)
    with pytest.raises(RuntimeError, match="create_bsr: a block's domain coordinate .jj. is not a multiple of blockdom"):
        plan1(ok_ii, [1, 0])
    with pytest.raises(RuntimeError, match="negative number of blocks"):
        plan1([-1, 0, 0, 0], [])
    with pytest.raises(RuntimeError, match="a block wraps around the domain lattice"):
        plan1(ok_ii, [0, 3], blk=(2, 3), dims=(4, 6), dimd=[4, 5], xdims=(4, 5, 2), ydims=(4, 6, 2))
    with pytest.raises(RuntimeError, match="multiples of blockim"):
        plan1([0, 0], [], pim=np.array([[[1, 0], [2, 4]]], np.int32))
    with pytest.raises(RuntimeError, match="the image parts must cover the image lattice"):
        plan1([0, 0], [], pim=np.array([[[0, 0], [2, 4]]], np.int32))
    with pytest.raises(RuntimeError, match="image parts overlap"):
        plan1([0] * 8, [], pim=np.array([[[0, 0], [4, 4]], [[2, 0], [2, 4]]], np.int32))
    with pytest.raises(RuntimeError, match="x lacks the label `B` of the operator"):
        plan1(ok_ii, ok_jj, ox="Anq", xdims=(4, 2, 4))
    with pytest.raises(RuntimeError, match="y lacks the column label `n` of x"):
        plan1(ok_ii, ok_jj, oy="abq")
    with pytest.raises(RuntimeError, match="dimension of label `n` does not match"):
        plan1(ok_ii, ok_jj, ydims=(4, 4, 3))
    with pytest.raises(RuntimeError, match="dimension of label `A` does not match"):
        plan1(ok_ii, ok_jj, xdims=(5, 4, 2))
    with pytest.raises(RuntimeError, match="x must not carry the power label"):
        plan1(ok_ii, ok_jj, power="n")
    with pytest.raises(RuntimeError, match="y has the label `q`"):
        plan1(ok_ii, ok_jj, oy="abnq", ydims=(4, 4, 2, 2))
    with pytest.raises(RuntimeError, match="powers above 1 need the same image and domain lattices"):
        plan1([1, 0, 0, 0], [0], dimd=[4], ox="An", xdims=(4, 2), oy="abnp", ydims=(4, 4, 2, 2), power="p")
    with pytest.raises(RuntimeError, match="unsupported type"):
        plan1(ok_ii, ok_jj, dtype=sb.I32)
    with pytest.raises(RuntimeError, match="repeated label"):
        plan1(ok_ii, ok_jj, ox="AAn")


def test_every_rank_throws_when_one_ranks_jj_is_misaligned():
    """Rank 1's only block starts off the blockdom grid; rank 0's operator is fine: both ranks refuse"""
    pim = np.array([[[0, 0], [2, 4]], [[2, 0], [2, 4]]], np.int32)
    ii = [1, 0] + [1, 0]
    jj = [0, 0] + [1, 0]
    for rank in range(2):
        with pytest.raises(RuntimeError, match="not a multiple of blockdom"):
            plan1(ii, jj, pim=pim, world=2, rank=rank)


def test_halo_is_the_shortest_periodic_arc():
    """Blocks at x = 0 and x = 14 of 16 (blockdom 2): the halo wraps, [14, 18), and the gathered input
    holds 4 points per row of the other label, not 16"""
    p = plan1([2, 0], [0, 0, 14, 0], dims=(2, 8), blk=(2, 4), dimd=[16, 4], xdims=(16, 4, 2), ydims=(2, 8, 2))
    it = p["items"][0]
    assert it["x"] == 4 * 4 * 2
    assert it["goff"] == [2, 0]
    assert "tier=warp" in it["kernel"]
