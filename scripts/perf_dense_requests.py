"""How much the dense solvers' requests hide, one process per GPU: the Gram-matrix orthogonalisation of a
block of vectors with the Gram matrix split across the ranks.

    python -m torch.distributed.run --nproc_per_node N scripts/perf_dense_requests.py [--out F] [--small]

Data (complex double, the same seed on every rank): V of nv x m ("iv", i cut over the N ranks), its Gram
matrix G = V^H V ("wv", w cut over the ranks: cholesky and trsm gather it), and an unrelated tensor B of
the same size as this rank's V that a local copy permutes ("iv" -> "vi").  Per rank, each a median of 5 after
2 warm-ups, CUDA events on the library's stream of this rank behind a barrier of all ranks:
  * plain: cholesky(G) and trsm Q = V U^-1, then the copy of B, each a call without a request;
  * requests: cholesky(G) begun, the copy of B, wait; trsm begun, the copy of B, wait;
  * copy: the copy of B alone (twice), for reference.
The largest value over the ranks is reported for each time; plain - requests is what the requests hide.
Q is checked bit for bit against the same calls on rank 0 alone (one component each) in the same run.  The
card's name and power limit come from nvidia-smi in the same run.  --small runs nv = 64 N, m = 8 (a check
of the script, not a measurement)."""
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
from perf_bsr import card  # noqa: E402
from perf_bsr_overlap import timed  # noqa: E402


def cut(dims, k, world):
    out = []
    for r in range(world):
        f, s = [0] * len(dims), list(dims)
        f[k], s[k] = dims[k] * r // world, dims[k] * (r + 1) // world - dims[k] * r // world
        out.append([f, s])
    return np.array(out, np.int32)


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
    nv, m = (64 * world, 8) if args.small else (32 ** 3 * 64 * 12, 64)
    co = sb.FastToSlow
    g = torch.Generator(device="cuda").manual_seed(5)
    v = torch.randn(nv * m, dtype=torch.complex128, device="cuda", generator=g)  # "iv", i fastest
    pv, pg = cut([nv, m], 0, world), cut([m, m], 0, world)
    a, b = pv[rank][0][0], pv[rank][0][0] + pv[rank][1][0]
    mine_v = v.view(m, nv)[:, a:b].contiguous().view(-1)
    # the Gram matrix, whole on rank 0's layout "wv" (w fastest), then this rank's rows
    vm = v.view(m, nv)
    gram = (vm.conj() @ vm.t()).t().contiguous()  # [v][w]: w fastest
    ga, gb = pg[rank][0][0], pg[rank][0][0] + pg[rank][1][0]
    mine_g0 = gram[:, ga:gb].contiguous().view(-1)
    mine_g = torch.empty_like(mine_g0)
    q = torch.empty_like(mine_v)
    bsrc, bdst = torch.randn(mine_v.numel(), dtype=torch.complex128, device="cuda", generator=g), torch.empty_like(mine_v)
    nl = b - a
    pb0, pb1 = np.array([[[0, 0], [nl, m]]], np.int32), np.array([[[0, 0], [m, nl]]], np.int32)

    def copy_b():
        sb.copy(1, pb0, 1, "iv", [0, 0], [nl, m], [nl, m], [bsrc], None, gpu, pb1, 1, "vi", [0, 0], [m, nl],
                [bdst], None, gpu, co, sb.Copy)

    def fresh():
        mine_g.copy_(mine_g0)

    def plain():
        fresh()
        sb.cholesky(pg, 1, "wv", [mine_g], "w", "v", gpu, co, comm=comm)
        sb.trsm(1, pg, 1, "wv", "w", "v", [mine_g], gpu, pv, 1, "iv", [mine_v], gpu, pv, 1, "iw", [q], gpu, co,
                comm=comm)
        copy_b()
        copy_b()

    def requests():
        fresh()
        r = sb.cholesky(pg, 1, "wv", [mine_g], "w", "v", gpu, co, comm=comm, request=True)
        copy_b()
        r.wait()
        r = sb.trsm(1, pg, 1, "wv", "w", "v", [mine_g], gpu, pv, 1, "iv", [mine_v], gpu, pv, 1, "iw", [q], gpu, co,
                    comm=comm, request=True)
        copy_b()
        r.wait()

    def copies():
        copy_b()
        copy_b()

    res = dict(card=card(), world=world, nv=nv, m=m, dtype="complex128")
    t_plain, t_req, t_copy = timed(plain, stream), timed(requests, stream), timed(copies, stream)
    # Q against rank 0 alone
    requests()
    torch.cuda.synchronize()
    full = torch.zeros(world * m * max(nv // world + 1, 1), dtype=torch.complex128, device="cuda")
    rows = torch.zeros(max(nv // world + 1, 1) * m, dtype=torch.complex128, device="cuda")
    rows[:q.numel()] = q.view(m, nl).t().contiguous().view(-1)
    dist.all_gather_into_tensor(full, rows)
    same = None
    if rank == 0:
        g1 = gram.contiguous().view(-1).clone()
        q1 = torch.empty_like(v)
        p1g, p1v = np.array([[[0, 0], [m, m]]], np.int32), np.array([[[0, 0], [nv, m]]], np.int32)
        sb.cholesky(p1g, 1, "wv", [g1], "w", "v", gpu, co)
        sb.trsm(1, p1g, 1, "wv", "w", "v", [g1], gpu, p1v, 1, "iv", [v], gpu, p1v, 1, "iw", [q1], gpu, co)
        torch.cuda.synchronize()
        ref = q1.view(m, nv).t()
        parts = full.view(world, -1)
        got = torch.cat([parts[r][:(pv[r][1][0]) * m].view(int(pv[r][1][0]), m) for r in range(world)])
        same = bool(torch.equal(torch.view_as_real(got), torch.view_as_real(ref)))
    t = torch.tensor([t_plain, t_req, t_copy], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_plain, t_req, t_copy = t.tolist()
    res.update(plain_s=t_plain, requests_s=t_req, copies_s=t_copy, hidden_s=t_plain - t_req,
               q_bit_identical_to_one_rank=same)
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
