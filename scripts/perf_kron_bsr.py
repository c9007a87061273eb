"""Throughput of bsr_krylov with a Kronecker operator (create_kron_bsr) on one GPU, next to the same
operator given to create_bsr with its blocks expanded, and to torch on the same data.

    python scripts/perf_kron_bsr.py [--out profiles/r4_perf_kron_bsr.json] [--small]

Case (complex double): the nine-point Wilson-shaped operator on a 24^3 x 48 lattice, one block row per
site, 9 blocks per row (the site and its neighbours +-1 along x, y, z, t); every block is K_u ⊗ B_{r,u}
with K_u a 4 x 4 spin factor shared by all rows and B_{r,u} a 3 x 3 colour block; 1 / 4 / 12 columns.
Tensors "scxyzt" (spin fastest, then colour) for the image and "SCXYZT" for the domain, the columns "n"
slowest.  The expanded operator has the 12 x 12 blocks K_u ⊗ B_{r,u} (16x the bytes).  torch:
`index_select` of the 9 neighbours of every site, then two `einsum`s (colour, then spin).  Time = CUDA
events around the whole call (the gather of x included), median of 5 after 2 warm-ups.  Rate = (colour
blocks + factors + x + y bytes) over that time, against the measured HBM copy bandwidth of DESIGN.md
section 4.4 (6545 GB/s); the expanded call is also given at its own bytes (its blocks instead of the
colour blocks).  The card's name and power limit come from nvidia-smi in the same run.  --small runs
everything at a tiny size (a check of the script, not a measurement)."""
import argparse
import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import superbblas_b200 as sb  # noqa: E402
from perf_bsr import HBM_COPY_GBS, timed, card, part, neighbours  # noqa: E402


def run_case(lat, ncols_list, gpu):
    nsite = int(torch.tensor(lat).prod())
    dims = [4, 3] + list(lat)
    nbr, _ = neighbours(lat)
    g = torch.Generator(device="cuda").manual_seed(1)
    v = torch.randn(nsite * 9 * 9, dtype=torch.complex128, device="cuda", generator=g)      # [site, u, jb, ib]
    kv = torch.randn(9 * 16, dtype=torch.complex128, device="cuda", generator=g)            # [u, jk, ik]
    ii = torch.full((nsite,), 9, dtype=torch.int32, device="cuda")
    nc = torch.stack([torch.stack([nbr[:, k] % lat[0], nbr[:, k] // lat[0] % lat[1],
                                   nbr[:, k] // (lat[0] * lat[1]) % lat[2], nbr[:, k] // (lat[0] * lat[1] * lat[2])], 1)
                      for k in range(9)], 1)                                   # [site, 9, 4]
    jj = torch.cat([torch.zeros(nsite, 9, 2, dtype=torch.int64, device="cuda"), nc], 2).to(torch.int32).reshape(-1)
    p = part(dims)
    one, blk, kron = [1] * 4, [1, 3] + [1] * 4, [4, 1] + [1] * 4
    op = sb.create_kron_bsr(p, dims, p, dims, 1, blk, blk, kron, kron, True, [ii], [jj], [v], [kv], gpu,
                            sb.FastToSlow)
    # expanded blocks E[site, u, jb, jk, ib, ik] = B[site, u, jb, ib] K[u, jk, ik]: element (i, j) at i + 12 j
    ve = (v.view(nsite, 9, 3, 1, 3, 1) * kv.view(1, 9, 1, 4, 1, 4)).reshape(-1)
    ope = sb.create_bsr(p, dims, p, dims, 1, [4, 3] + one, [4, 3] + one, True, [ii], [jj], [ve], gpu,
                        sb.FastToSlow)
    del ii, jj
    kbytes, ebytes = (v.numel() + kv.numel()) * 16, ve.numel() * 16
    del ve
    torch.cuda.empty_cache()
    out = {}
    for n in ncols_list:
        x = torch.randn(nsite * 12 * n, dtype=torch.complex128, device="cuda", generator=g)
        y, ye = torch.empty_like(x), torch.empty_like(x)
        px = part(dims + [n])

        def call(h, yy):
            sb.bsr_krylov(1, h, "scxyzt", "SCXYZT", px, 1, "SCXYZTn", [0] * 7, dims + [n], dims + [n], [x], gpu, 0,
                          px, "scxyztn", [0] * 7, dims + [n], dims + [n], None, [yy], gpu, sb.FastToSlow)
            sb.sync(gpu)
        t = timed(lambda: call(op, y))
        te = timed(lambda: call(ope, ye))
        xbytes = x.numel() * 16
        b4 = v.view(nsite, 9, 3, 3)
        k3 = kv.view(9, 4, 4)
        xt = x.view(n, nsite, 12)
        idx = nbr.reshape(-1)

        def torch_apply():
            xn = torch.index_select(xt, 1, idx).view(n, nsite, 9, 3, 4)            # [n, site, u, jb, jk]
            tt = torch.einsum("suji,nsujl->nsuil", b4, xn)                           # [n, site, u, ib, jk]
            return torch.einsum("ulm,nsuil->nsim", k3, tt)                           # [n, site, ib, ik]
        tt = timed(torch_apply)
        ref = torch_apply().reshape(-1)
        scale = max(ref.abs().max().item(), 1e-300)
        gbs = (kbytes + 2 * xbytes) / t / 1e9
        out["cols_%d" % n] = dict(
            seconds=t, gbs=gbs, hbm_share=gbs / HBM_COPY_GBS, expanded_seconds=te,
            expanded_gbs_own_bytes=(ebytes + 2 * xbytes) / te / 1e9, speedup_vs_expanded=te / t, torch_seconds=tt,
            speedup_vs_torch=tt / t, max_rel_diff_vs_torch=(y - ref).abs().max().item() / scale,
            max_rel_diff_vs_expanded=(y - ye).abs().max().item() / scale)
        del x, y, ye
        torch.cuda.empty_cache()
    op.destroy()
    ope.destroy()
    return dict(lattice=list(lat), sites=nsite, blocks_per_row=9, kron_bytes=kbytes, expanded_bytes=ebytes, **out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    gpu = sb.createGpuContext(0)
    res = dict(card=card(), dtype="complex128",
               bytes="colour blocks + factors + x + y; time = CUDA events around the whole call (gather of x "
                     "included), median of 5 after 2 warm-ups")
    res["wilson_4x4_kron_3x3"] = run_case([4, 4, 4, 4] if args.small else [24, 24, 24, 48], [1, 4, 12], gpu)
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
