"""How much of bsr_krylov's halo exchange the interior rows hide, one process per GPU.

    python -m torch.distributed.run --nproc_per_node N scripts/perf_bsr_overlap.py [--out F] [--small]

Cases (complex double, nine-point operator, one block row per site, 24^3 x 48 lattice cut along t over
the N ranks, x cut like the operator, y written directly; 1 and 12 columns):
  * plain: 12 x 12 blocks (create_bsr);
  * kron: 4 x 4 spin factors ⊗ 3 x 3 colour blocks (create_kron_bsr).
Per case and rank, each a median of 5 after 2 warm-ups, CUDA events on the library's stream of this rank
behind a barrier of all ranks:
  * call: the whole bsr_krylov (the interior rows run while the gather of x is in flight);
  * gather: sbb_copy of x into every rank's halo box with the layout of the gather (columns fastest);
  * kernels: the call's kernels ("bsr" / "kron_bsr" of the library's kernel profile), in a run of its own.
The overlap is gather + kernels - call; the largest value over the ranks is reported for each time.  y is
checked against the same operator on rank 0 alone (one component) in the same run.  The card's name and
power limit come from nvidia-smi in the same run.  --small runs a 4^3 x (4 N) lattice (a check of the
script, not a measurement)."""
import argparse
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import superbblas_b200 as sb  # noqa: E402
from perf_bsr import card, neighbours  # noqa: E402


def build(lat, kron, g):
    """(ii, jj, v, kronv) of the whole operator on every rank (same seed), rows x fastest"""
    nsite = int(np.prod(lat))
    nbr, _ = neighbours(lat)
    coords = [nbr % lat[0], nbr // lat[0] % lat[1], nbr // (lat[0] * lat[1]) % lat[2], nbr // (lat[0] * lat[1] * lat[2])]
    jj = torch.cat([torch.zeros(nsite, 9, 2, dtype=torch.int64, device="cuda"), torch.stack(coords, 2)], 2)
    ii = torch.full((nsite,), 9, dtype=torch.int32, device="cuda")
    bsz = 9 if kron else 144
    v = torch.randn(nsite * 9 * bsz, dtype=torch.complex128, device="cuda", generator=g)
    kv = torch.randn(9 * 16, dtype=torch.complex128, device="cuda", generator=g) if kron else None
    return ii, jj.to(torch.int32), v, kv


def create(dims, pim, rows, ops, kron, gpu, comm):
    ii, jj, v, kv = ops
    a, b = rows
    bsz = 9 if kron else 144
    blk, kr = ([1, 3] if kron else [4, 3]) + [1] * 4, [4, 1] + [1] * 4
    args = (pim, dims, pim, dims, 1)
    if kron:
        return sb.create_kron_bsr(*args, blk, blk, kr, kr, True, [ii[a:b]], [jj[a:b].reshape(-1)],
                                  [v[a * 9 * bsz:b * 9 * bsz]], [kv], gpu, sb.FastToSlow, comm=comm)
    return sb.create_bsr(*args, blk, blk, True, [ii[a:b]], [jj[a:b].reshape(-1)], [v[a * 9 * bsz:b * 9 * bsz]],
                         gpu, sb.FastToSlow, comm=comm)


def timed(fn, stream, reps=5, warmup=2):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true")
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    uid = torch.zeros(128, dtype=torch.uint8, device=dev)
    if rank == 0:
        uid.copy_(torch.frombuffer(bytearray(sb.comm_unique_id()), dtype=torch.uint8))
    dist.broadcast(uid, 0)
    comm = sb.comm_create(bytes(uid.cpu().numpy().tobytes()), world, rank, local)
    gpu = sb.createGpuContext(local)
    stream = torch.cuda.ExternalStream(sb.get_stream(local), device=dev)
    lat = [4, 4, 4, 4 * world] if args.small else [24, 24, 24, 48]
    assert lat[3] % world == 0
    tl = lat[3] // world
    per_t = lat[0] * lat[1] * lat[2]
    res = dict(card=card(), world=world, lattice=lat, dtype="complex128", cases={})
    for kron in (False, True):
        dims = [4, 3] + lat
        g = torch.Generator(device="cuda").manual_seed(3)
        ops = build(lat, kron, g)
        pim = np.array([[[0, 0, 0, 0, 0, r * tl], [4, 3] + lat[:3] + [tl]] for r in range(world)], np.int32)
        op = create(dims, pim, (rank * tl * per_t, (rank + 1) * tl * per_t), ops, kron, gpu, comm)
        op1 = create(dims, np.array([[[0] * 6, dims]], np.int32), (0, lat[3] * per_t), ops, kron, gpu,
                     None) if rank == 0 else None
        for n in (1, 12):
            xd = dims + [n]
            x = torch.randn(int(np.prod(xd)), dtype=torch.complex128, device="cuda", generator=g)
            px = np.array([[[0] * 5 + [r * tl, 0], [4, 3] + lat[:3] + [tl, n]] for r in range(world)], np.int32)
            mine = x.view(n, lat[3], -1)[:, rank * tl:(rank + 1) * tl].contiguous().view(-1)
            y = torch.empty_like(mine)

            def call():
                sb.bsr_krylov(1, op, "scxyzt", "SCXYZT", px, 1, "SCXYZTn", [0] * 7, xd, xd, [mine], gpu, 0, px,
                              "scxyztn", [0] * 7, xd, xd, None, [y], gpu, sb.FastToSlow, comm=comm)
            # the gather alone: x into every rank's halo box (t +-1), columns fastest
            hd = [n] + dims
            halo = np.array([[[0] * 6 + [(r * tl - 1) % lat[3]], [n, 4, 3] + lat[:3] + [tl + 2]]
                             for r in range(world)], np.int32)
            slot = torch.empty(n * 12 * per_t * (tl + 2), dtype=torch.complex128, device="cuda")

            def gather():
                sb.copy(1, px, 1, "SCXYZTn", [0] * 7, xd, xd, [mine], None, gpu, halo, 1, "nSCXYZT", [0] * 7, hd,
                        [slot], None, gpu, sb.FastToSlow, sb.Copy, comm=comm)
            t_call, t_gather = timed(call, stream), timed(gather, stream)
            name = "kron_bsr" if kron else "bsr"
            sb.profile_enable(True)
            sb.profile_read(name)  # since the last read: start from zero
            call()
            torch.cuda.synchronize()
            t_kern = sb.profile_read(name)[0] * 1e-3
            sb.profile_enable(False)
            # y against rank 0 alone
            full = torch.zeros(world * y.numel(), dtype=torch.complex128, device="cuda")
            dist.all_gather_into_tensor(full, y.view(n, -1).t().contiguous().view(-1))
            err = float("nan")
            if rank == 0:
                y1 = torch.empty_like(x)
                sb.bsr_krylov(1, op1, "scxyzt", "SCXYZT", np.array([[[0] * 7, xd]], np.int32), 1,
                              "SCXYZTn", [0] * 7, xd, xd, [x], gpu, 0, np.array([[[0] * 7, xd]], np.int32),
                              "scxyztn", [0] * 7, xd, xd, None, [y1], gpu, sb.FastToSlow)
                torch.cuda.synchronize()
                ref = y1.view(n, -1).t().contiguous().view(-1)
                err = (full - ref).abs().max().item() / max(ref.abs().max().item(), 1e-300)
            t = torch.tensor([t_call, t_gather, t_kern], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            t_call, t_gather, t_kern = t.tolist()
            res["cases"]["%s_cols_%d" % ("kron" if kron else "plain", n)] = dict(
                call_s=t_call, gather_s=t_gather, kernels_s=t_kern, hidden_s=t_gather + t_kern - t_call,
                max_rel_diff_vs_one_rank=err)
        op.destroy()
        if op1 is not None:
            op1.destroy()
    if rank == 0:
        print(json.dumps(res, indent=1))
        if args.out:
            with open(args.out, "w") as f:
                json.dump(res, f, indent=1)
    sb.clearCaches()
    comm.destroy()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
