"""Throughput of bsr_krylov on one GPU, next to torch on the same data.

    python scripts/perf_bsr.py [--out profiles/r3_perf_bsr.json] [--small]

Cases (complex double, periodic nearest-neighbour operator: 9 blocks per block row, one row per site):
  * 12 x 12 spin-colour blocks on a 24^3 x 48 lattice, 1 / 4 / 12 columns;
  * 64 x 64 coarse-operator blocks on an 8^4 lattice (4096 sites), 1 / 16 / 64 columns.
Tensors "sxyzt" (block label fastest) for the operator's image and "SXYZT" for its domain, with the
columns "n" slowest.  Rate = (matrix + x + y bytes) over the CUDA-event time of the whole call (median
of the timed repetitions after warm-ups), against the measured HBM copy bandwidth of DESIGN.md
section 4.4 (6545 GB/s).  torch: `index_select` of the 9 neighbours of every site followed by one
batched `einsum` over [site, block, i, j] blocks.  Every case's matrix is far larger than the 126 MB L2.
The card name and power limit come from nvidia-smi in the same run.  --small runs everything at a
tiny size (a check of the script, not a measurement)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import superbblas_b200 as sb  # noqa: E402

HBM_COPY_GBS = 6545.0


def timed(fn, reps=5, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    return float(np.median(ts))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown"


def part(dims):
    return np.array([[[0] * len(dims), list(dims)]], dtype=np.int32)


def neighbours(lat):
    """[site, 9] site indices (x fastest) of every site, itself first, then +-1 along x, y, z, t"""
    nsite = int(np.prod(lat))
    s = torch.arange(nsite, device="cuda")
    c, rest = [], s
    for L in lat:
        c.append(rest % L)
        rest = rest // L
    out = [s]
    for mu in range(4):
        for d in (1, -1):
            cc = list(c)
            cc[mu] = (cc[mu] + d) % lat[mu]
            idx = torch.zeros_like(s)
            for k in reversed(range(4)):
                idx = idx * lat[k] + cc[k]
            out.append(idx)
    return torch.stack(out, 1), torch.stack(c, 1)


def run_case(b, lat, ncols_list, gpu):
    nsite = int(np.prod(lat))
    dims = [b] + list(lat)
    nbr, coords = neighbours(lat)
    g = torch.Generator(device="cuda").manual_seed(1)
    v = torch.randn(nsite * 9 * b * b, dtype=torch.complex128, device="cuda", generator=g)
    ii = torch.full((nsite,), 9, dtype=torch.int32, device="cuda")
    nc = torch.stack([torch.stack([nbr[:, k] % lat[0], nbr[:, k] // lat[0] % lat[1],
                                   nbr[:, k] // (lat[0] * lat[1]) % lat[2], nbr[:, k] // (lat[0] * lat[1] * lat[2])], 1)
                      for k in range(9)], 1)                                   # [site, 9, 4]
    jj = torch.cat([torch.zeros(nsite, 9, 1, dtype=torch.int64, device="cuda"), nc], 2).to(torch.int32).reshape(-1)
    p = part(dims)
    op = sb.create_bsr(p, dims, p, dims, 1, [b, 1, 1, 1, 1], [b, 1, 1, 1, 1], True, [ii], [jj], [v], gpu,
                       sb.FastToSlow)
    del ii, jj
    out = {}
    mbytes = v.numel() * 16
    for n in ncols_list:
        x = torch.randn(nsite * b * n, dtype=torch.complex128, device="cuda", generator=g)
        y = torch.empty_like(x)
        px = part(dims + [n])
        t = timed(lambda: (sb.bsr_krylov(1, op, "sxyzt", "SXYZT", px, 1, "SXYZTn", [0] * 6, dims + [n], dims + [n],
                                         [x], gpu, 0, px, "sxyztn", [0] * 6, dims + [n], dims + [n], None, [y], gpu,
                                         sb.FastToSlow), sb.sync(gpu)))
        xbytes = x.numel() * 16
        gbs = (mbytes + 2 * xbytes) / t / 1e9
        # torch on the same data: A [site, 9, j, i] (blockImFast), X [n, site, j]
        a4 = v.view(nsite, 9, b, b)
        xt = x.view(n, nsite, b)
        idx = nbr.reshape(-1)

        def torch_apply():
            xn = torch.index_select(xt, 1, idx).view(n, nsite, 9, b)
            return torch.einsum("skji,nskj->nsi", a4, xn)
        tt = timed(torch_apply)
        err = (torch_apply().reshape(-1) - y).abs().max().item() / max(y.abs().max().item(), 1e-300)
        out["cols_%d" % n] = dict(seconds=t, gbs=gbs, hbm_share=gbs / HBM_COPY_GBS, torch_seconds=tt,
                                  speedup_vs_torch=tt / t, max_rel_diff_vs_torch=err)
        del x, y
        torch.cuda.empty_cache()
    op.destroy()
    del v
    torch.cuda.empty_cache()
    return dict(block=b, lattice=list(lat), sites=nsite, blocks_per_row=9, matrix_bytes=mbytes, **out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    gpu = sb.createGpuContext(0)
    res = dict(card=card(), dtype="complex128",
               bytes="matrix + x + y; time = CUDA events around the whole call (gather of x included)")
    res["spin_colour_12x12"] = run_case(12, [4, 4, 4, 4] if args.small else [24, 24, 24, 48], [1, 4, 12], gpu)
    res["coarse_64x64"] = run_case(64, [2, 2, 2, 2] if args.small else [8, 8, 8, 8], [1, 16, 64], gpu)
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
