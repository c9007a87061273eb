"""Host logic of the Kronecker block-sparse operators (create_kron_bsr) without a GPU: every rank's
kron_bsr_plan is executed in numpy for 1 to 4 simulated ranks (direct, written back, powers), with the
kernel as a numpy loop over the row pointers, block offsets and Kronecker dims the plan describes,
against the oracle of the expanded operator sum_u K_u ⊗ B_{r,u}; the gather, fill and write-back copies
equal those of bsr_plan for the same operator with expanded blocks; and the argument errors, which
every rank throws alike."""
import numpy as np
import pytest

import superbblas_b200 as sb
from tests import bsr_cases as B
from tests import kron_bsr_cases as KB
from tests import test_bsr_plan as P


def kron_points(it):
    """kron_domain_point of every (jk, jb), at jb + jk * bd"""
    bd, kd = it["bd"], it["kd"]
    out = np.zeros(kd * bd, np.int64)
    for jk in range(kd):
        for jb in range(bd):
            o, a, b = 0, jk, jb
            for (sz, st), ks in zip(it["D"], it["DK"]):
                o += ((b % sz) * ks + a % ks) * st
                a, b = a // ks, b // sz
            out[jb + jk * bd] = o
    return out


def kron_image(it, r):
    """kron_image_offset of block row r for every (ik, ib), at ib + ik * bi"""
    bi, ki = it["bi"], it["ki"]
    out = np.zeros(ki * bi, np.int64)
    for ik in range(ki):
        for ib in range(bi):
            o, rr, a, b = 0, r, ik, ib
            for (nb, sz, st), ks in zip(it["I"], it["IK"]):
                o += ((rr % nb) * sz * ks + (b % sz) * ks + a % ks) * st
                rr, a, b = rr // nb, a // ks, b // sz
            out[ib + ik * bi] = o
    return out


def kron_kernel(kronv):
    """What the Kronecker kernel computes for one item, on flat numpy storages"""
    def run(it, v, xg, out, base, alpha, beta):
        bi, bd, ki, kd, U, nc = it["bi"], it["bd"], it["ki"], it["kd"], it["u"], it["ncols"]
        xo, cp, rp, goff = kron_points(it), P.offsets(it["C"]), it["rowptr"], it["goff"]
        for r in range(it["rows"]):
            acc = np.zeros((ki, bi, nc), np.complex128)
            for u in range(U):
                b = rp[r] + u
                Bm = KB.mat(v[b * bi * bd:(b + 1) * bi * bd], it["imfast"], bi, bd)
                K = KB.mat(kronv[u * ki * kd:(u + 1) * ki * kd], it["imfast"], ki, kd)
                xs = xg[(goff[b] + xo)[:, None] * nc + np.arange(nc)[None, :]].reshape(kd, bd, nc)
                t = np.einsum("ij,kjc->kic", Bm, xs)                     # [jk, ib, c]
                acc += np.einsum("lk,kic->lic", K, t)
            o = base + kron_image(it, r).reshape(ki, bi)[:, :, None] + cp[None, None, :]
            res = alpha * acc + (beta * out[o] if beta != 0 else 0)
            out[o] = res if out.dtype.kind == "c" else res.real
    return run


def random_kron_case(rng, world, ncomp, kind, T=None):
    """Like test_bsr_plan.random_case, with Kronecker labels: image "ab", domain "cd(z)"; the Kronecker
    factor lives on b / d (extent 2), the B blocks on a / c"""
    T = np.dtype([np.float64, np.complex128][rng.integers(2)] if T is None else T)
    co, imfast = int(rng.integers(2)), bool(rng.integers(2))
    nparts = world * ncomp
    if kind == "power":
        dimi = dimd = [6, 4]
        blockim = blockdom = [3, 1]
        kronim = krondom = [1, 2]
    else:
        dimi, dimd = [8, 6], [6, 4, 2]
        blockim, blockdom = [2, 1], [3, 1, 1]
        kronim, krondom = [1, 3], [1, 2, 1]
    oim, odom = "ab", "cdz"[:len(dimd)]
    pim = P.boxes(dimi, 0, P.cuts_at(rng, dimi[0], blockim[0], nparts))
    U = int(rng.integers(0, 4))
    ops, kronv = KB.random_kron_operator(rng, pim, blockim, dimd, blockdom, kronim, krondom, U, T)
    c = P.random_case(rng, world, ncomp, kind, T)                       # x, y and their partitions
    c.update(co=co, imfast=imfast, dimi=dimi, dimd=dimd, blockim=blockim, blockdom=blockdom, kronim=kronim,
             krondom=krondom, oim=oim, odom=odom, pim=pim, ops=ops, kronv=kronv, U=U)
    if kind == "direct":
        sizes = dict(zip(oim, dimi), n=3)
        c["py"] = np.array([[[f[oim.index(l)] if l in oim else 0 for l in c["oy"]],
                             [s[oim.index(l)] if l in oim else sizes[l] for l in c["oy"]]]
                            if 0 not in list(s) else [[0] * len(c["oy"]), [0] * len(c["oy"])]
                            for f, s in pim], dtype=np.int32)
    return c


def kron_plan_of(c, world, rank, ncomp):
    pdom = np.array([[[0] * len(c["dimd"]), c["dimd"]]] * world * ncomp, dtype=np.int32)
    return sb.kron_bsr_plan(P.DT[c["T"]], c["pim"], c["dimi"], pdom, c["dimd"], ncomp, c["blockim"], c["blockdom"],
                            c["kronim"], c["krondom"], c["imfast"], *B.flat_arrays(c["ops"]), c["oim"], c["odom"],
                            c["px"], ncomp, c["ox"], [0] * len(c["ox"]), list(c["x"].shape), list(c["x"].shape),
                            c["py"], ncomp, c["oy"], c["fromy"], c["sizey"], list(c["y0"].shape), c["power"],
                            c["co"], world, rank, alpha=c["alpha"], beta=c["beta"])


def run_kron_plans(c, world, ncomp, kernel=None):
    """test_bsr_plan.run_plans with the Kronecker plans and kernel"""
    saved = P.plan_of
    P.plan_of = kron_plan_of
    try:
        return P.run_plans(c, world, ncomp, kernel or kron_kernel(c["kronv"]))
    finally:
        P.plan_of = saved


def want_of(c):
    a = KB.oracle_matrix(c["ops"], c["kronv"], c["pim"], c["dimi"], c["dimd"], c["blockim"], c["blockdom"],
                         c["kronim"], c["krondom"], c["imfast"], c["co"])
    return B.apply(a, c["oim"], c["odom"], c["x"], c["ox"], c["y0"], c["oy"], c["alpha"], c["beta"], c["power"],
                   3 if c["power"] else 1, c["fromy"])


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_kron_plans_match_oracle(world):
    rng = np.random.default_rng(1900 + world)
    seen = set()
    for k in range(18):
        kind = ["direct", "back", "power"][k % 3]
        ncomp = int(rng.integers(1, 3))
        c = random_kron_case(rng, world, ncomp, kind)
        plans, got = run_kron_plans(c, world, ncomp)
        want = want_of(c)
        assert np.array_equal(np.isnan(got), np.isnan(want)), (world, k, kind)
        assert B.rel_err(np.nan_to_num(got), np.nan_to_num(want)) < 1e-12, (world, k, kind)
        p = plans[0]
        for it in (it for q in plans for it in q["items"]):
            assert it["u"] == c["U"] and it["ki"] == int(np.prod(c["kronim"])) and "kron_bsr tier=" in it["kernel"]
        seen.add("direct" if p["direct"] else "back")
        if p["fill"]:
            seen.add("fill")
        if p["powers"] > 1:
            seen.add("power " + ("direct" if p["direct"] else "back"))
    assert {"direct", "back", "fill", "power back"} <= seen, seen


@pytest.mark.parametrize("world", [1, 2, 3])
def test_copies_equal_those_of_the_expanded_operator(world):
    """The Kronecker labels are ordinary labels for the halo boxes and the copies: gather, fill and
    write-back, the row pointers, block offsets and output dims equal bsr_plan's for the expanded blocks"""
    rng = np.random.default_rng(2900 + world)
    for k in range(9):
        kind = ["direct", "back", "power"][k % 3]
        ncomp = int(rng.integers(1, 3))
        c = random_kron_case(rng, world, ncomp, kind)
        c["U"] = max(c["U"], 1)
        c["ops"], c["kronv"] = KB.random_kron_operator(rng, c["pim"], c["blockim"], c["dimd"], c["blockdom"],
                                                       c["kronim"], c["krondom"], c["U"], c["T"])
        ex = dict(c, blockim=KB.eff(c["blockim"], c["kronim"]), blockdom=KB.eff(c["blockdom"], c["krondom"]))
        for rank in range(world):
            kp, pp = kron_plan_of(c, world, rank, ncomp), P.plan_of(ex, world, rank, ncomp)
            for f in ("nothing", "direct", "powers", "slots", "gather", "fill", "back"):
                assert kp[f] == pp[f], (f, world, k, rank)
            assert len(kp["items"]) == len(pp["items"])
            for a, b in zip(kp["items"], pp["items"]):
                for f in ("comp", "y", "x", "nnz", "rows", "ncols", "C", "rowptr", "goff"):
                    assert a[f] == b[f], f
                assert a["bi"] * a["ki"] == b["bi"] and a["bd"] * a["kd"] == b["bd"]
                assert [(nb, sz * ks, st) for (nb, sz, st), ks in zip(a["I"], a["IK"])] == b["I"]
                assert [(sz * ks, st) for (sz, st), ks in zip(a["D"], a["DK"])] == b["D"]


def kplan(ii, jj, dims=(4, 4), blk=(2, 1), kron=(1, 2), dimd=None, bdom=None, kdom=None, pim=None, world=1, rank=0,
          dtype=sb.F64, ydims=None):
    dimd = list(dims) if dimd is None else dimd
    bdom = list(blk) if bdom is None else bdom
    kdom = list(kron) if kdom is None else kdom
    pim = P.single(dims) if pim is None else pim
    n = len(pim)
    xdims = list(dimd) + [2]
    ydims = list(dims) + [2] if ydims is None else ydims
    pdom = np.array([[[0] * len(dimd), dimd]] * n, dtype=np.int32)
    px = np.array([[[0] * len(xdims), xdims]] * n, dtype=np.int32)
    py = np.array([[[0] * len(ydims), ydims]] * n, dtype=np.int32)
    return sb.kron_bsr_plan(dtype, pim, list(dims), pdom, dimd, n // world, list(blk), bdom, list(kron), kdom, True,
                            ii, jj, "ab", "AB", px, n // world, "ABn", [0] * 3, xdims, xdims, py, n // world, "abn",
                            [0] * 3, ydims, ydims, None, sb.FastToSlow, world, rank)


def test_kron_plan_errors():
    ok_ii, ok_jj = [1, 1, 1, 1], [0, 0, 2, 2, 0, 2, 2, 0]             # effective blocks 2 x 2
    p = kplan(ok_ii, ok_jj)
    assert p["items"][0]["u"] == 1 and p["items"][0]["IK"] == [1, 2]
    with pytest.raises(RuntimeError, match="^create_kron_bsr: kronim and blockim exceed 1 along the same image label"):
        kplan(ok_ii, ok_jj, blk=(2, 2), kron=(2, 1), bdom=[2, 1], kdom=[1, 2])
    with pytest.raises(RuntimeError, match="^create_kron_bsr: krondom and blockdom exceed 1 along the same domain label"):
        kplan(ok_ii, ok_jj, bdom=[2, 2], kdom=[1, 2])
    with pytest.raises(RuntimeError, match="^create_kron_bsr: kronim must be positive"):
        kplan(ok_ii, ok_jj, kron=(1, 0), kdom=[1, 2])
    with pytest.raises(RuntimeError, match="^create_kron_bsr: krondom must be positive"):
        kplan(ok_ii, ok_jj, kdom=[1, 0])
    with pytest.raises(RuntimeError, match=r"^create_kron_bsr: the from and size of every image part must be "
                                           r"multiples of blockim \* kronim"):
        kplan([1, 1], [0, 0, 0, 0], pim=np.array([[[0, 1], [4, 2]]], np.int32))
    with pytest.raises(RuntimeError, match=r"^create_kron_bsr: a block's domain coordinate \(jj\) is not a multiple "
                                           r"of blockdom \* krondom"):
        kplan(ok_ii, [0, 1, 2, 2, 0, 2, 2, 0])
    with pytest.raises(RuntimeError, match=r"^create_kron_bsr: a block wraps around the domain lattice"):
        kplan(ok_ii, ok_jj, dimd=[4, 3])
    with pytest.raises(RuntimeError, match=r"^create_kron_bsr: negative number of blocks in a row \(ii\)"):
        kplan([-1, 1, 1, 1], ok_jj[2:])
    with pytest.raises(RuntimeError, match="^create_kron_bsr: the image parts must cover the image lattice"):
        kplan([1, 1], ok_jj[:4], pim=np.array([[[0, 0], [2, 4]]], np.int32))
    with pytest.raises(RuntimeError, match=r"^create_kron_bsr: every block row of every component, on every rank, "
                                           r"must have the same number of blocks \(ii\)"):
        kplan([1, 2, 1, 0], [0, 0, 2, 2, 0, 2, 2, 0])
    with pytest.raises(RuntimeError, match="^bsr_krylov: Kronecker operators need"):
        kplan([1], [0, 0], dims=(1, 8192), blk=(1, 1), kron=(1, 8192), dimd=[1, 1], bdom=[1, 1], kdom=[1, 1])


@pytest.mark.parametrize("bad_rank", [0, 1])
def test_every_rank_throws_when_one_ranks_ii_differs(bad_rank):
    """Each rank's own rows agree, but rank `bad_rank` has 2 blocks per row and the other 1: both refuse.
    Then a jj off the effective grid on one rank only: both refuse too."""
    pim = np.array([[[0, 0], [2, 4]], [[2, 0], [2, 4]]], np.int32)
    good, bad = ([1, 1], [0, 0, 0, 2]), ([2, 2], [0, 0, 2, 0, 0, 2, 2, 2])
    parts = [bad, good] if bad_rank == 0 else [good, bad]
    ii = parts[0][0] + parts[1][0]
    jj = parts[0][1] + parts[1][1]
    for rank in range(2):
        with pytest.raises(RuntimeError, match="^create_kron_bsr: every block row of every component"):
            kplan(ii, jj, pim=pim, world=2, rank=rank)
    misaligned = [0, 0, 0, 1]
    parts = [(good[0], misaligned), good] if bad_rank == 0 else [good, (good[0], misaligned)]
    for rank in range(2):
        with pytest.raises(RuntimeError, match="^create_kron_bsr: a block's domain coordinate"):
            kplan(parts[0][0] + parts[1][0], parts[0][1] + parts[1][1], pim=pim, world=2, rank=rank)
