"""Time of eigh (the batched Hermitian eigensolver) on one GPU, next to torch.linalg.eigh on the same
batches.

    python scripts/perf_dense_eigh.py [--out profiles/r4_perf_dense_eigh.json] [--small]

Cases (complex double, tensors FastToSlow: the batch labels have the smallest strides):
  * link: 3x3 per link of a 32^3 x 64 lattice, 4 directions, tensor "xyztdcC";
  * site: 12x12 spin-colour per site of a 32^3 x 64 lattice, tensor "xyztcsCS";
  * gram: 64x64 Gram matrices, a batch of 256, tensor "vwb" (each matrix contiguous).
For each: eigh on the labelled tensor (eigenvectors over A, eigenvalues into W with the batch labels and
the column labels), and torch.linalg.eigh on a contiguous [batch, n, n] copy, alone and with the permute
into that layout and back (V and w) that the labelled layout needs; torch's batched eigh (cuSOLVER
syevBatched) refuses batches of millions of matrices in one call, so it runs over chunks of 16384
matrices, a size it accepts for these orders on a B200 (recorded as `torch_chunk`).  Every case checks its result:
eigenvalues against torch's, and ||A V - V diag(w)|| / ||A|| and max |V^H V - I| on a sample of matrices.
Times are CUDA-event times of the whole call, median of 5 after 2 warm-ups; eigh works in place, so its
time is that of restoring the input and the call, less that of restoring alone.  The card's name and power
limit come from nvidia-smi in the same run.  --small runs everything at a tiny size (a check of the
script, not a measurement)."""
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


TORCH_CHUNK = 16384


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


def run_case(name, batch, mat, n, sample=2000):
    """batch: [(label, extent)], fastest first; mat: (row labels, column labels) with their extents"""
    (rl, rext), (cl, cext) = mat
    labels = [l for l, _ in batch] + list(rl) + list(cl)
    dims = [e for _, e in batch] + list(rext) + list(cext)
    o = "".join(labels)
    ow = "".join([l for l, _ in batch] + list(cl))
    wdims = [e for _, e in batch] + list(cext)
    nb = int(np.prod([e for _, e in batch]))
    gpu = sb.createGpuContext(0)
    g = torch.Generator(device="cuda").manual_seed(1)
    # contiguous [batch, n, n] Hermitian matrices; the labelled tensor (first label fastest) is its
    # transpose [col, row, batch] in memory
    b = torch.randn(nb, n, n, dtype=torch.complex128, device="cuda", generator=g)
    h = (b + b.mH) / 2
    del b
    lab = h.permute(2, 1, 0).contiguous().reshape(-1)
    a = lab.clone()
    w = torch.zeros(nb * n, dtype=torch.float64, device="cuda")

    def ours():
        a.copy_(lab)
        sb.eigh(part(dims), 1, o, [a], rl, cl, gpu, part(wdims), 1, ow, [w], gpu, sb.FastToSlow)

    def copy_only():
        a.copy_(lab)

    t_ours = timed(ours) - timed(copy_only)
    chunk = TORCH_CHUNK

    def torch_eigh(m):
        outs = [torch.linalg.eigh(m[i:i + chunk]) for i in range(0, nb, chunk)]
        return torch.cat([e for e, _ in outs]), torch.cat([v for _, v in outs])
    t_torch = timed(lambda: torch_eigh(h))

    def torch_permuted():
        m = lab.reshape(n, n, nb).permute(2, 1, 0).contiguous()
        ev, v = torch_eigh(m)
        v.permute(2, 1, 0).contiguous()
        ev.t().contiguous()
    t_torch_perm = timed(torch_permuted)
    ours()
    torch.cuda.synchronize()
    # result check
    wref = torch_eigh(h)[0]
    wo = w.reshape(n, nb).t()
    werr = float((wo - wref).abs().max() / wref.abs().max())
    idx = torch.arange(0, nb, max(1, nb // sample), device="cuda")
    v = a.reshape(n, n, nb).permute(2, 1, 0)[idx]
    hs = h[idx]
    res = float(torch.linalg.matrix_norm(hs @ v - v * wo[idx][:, None, :]).max() / torch.linalg.matrix_norm(hs).max())
    orth = float((v.mH @ v - torch.eye(n, dtype=v.dtype, device="cuda")).abs().max())
    ok = werr < 20 * n * 2 ** -53 * 4 and res < 20 * n * 2 ** -53 and orth < 20 * n * 2 ** -53
    bytes_moved = nb * (2 * n * n * 16 + n * 8)
    return dict(case=name, n=n, batch=nb, torch_chunk=min(chunk, nb), eigh_s=t_ours, torch_eigh_s=t_torch, torch_eigh_with_permute_s=t_torch_perm,
                eigh_GBs=bytes_moved / t_ours / 1e9, speedup_vs_torch=t_torch / t_ours,
                speedup_vs_torch_with_permute=t_torch_perm / t_ours, w_rel_err=werr, residual=res, orthogonality=orth,
                ok=bool(ok))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("perf_dense_eigh needs a CUDA device")
    L, T = (4, 4) if args.small else (32, 64)
    lat = [("x", L), ("y", L), ("z", L), ("t", T)]
    results = [
        run_case("link 3x3", lat + [("d", 4)], (("c", [3]), ("C", [3])), 3),
        run_case("site 12x12", lat, (("cs", [3, 4]), ("CS", [3, 4])), 12),
        run_case("gram 64x64", [("b", 8 if args.small else 256)], (("v", [64]), ("w", [64])), 64),
    ]
    out = dict(card=card(), small=args.small, results=results)
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    if not all(r["ok"] for r in results):
        raise SystemExit("a result check failed")


if __name__ == "__main__":
    main()
