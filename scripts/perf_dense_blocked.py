"""Time of the blocked tier of cholesky and trsm (matrices over one CTA's shared memory) on one GPU,
next to torch.linalg on the same data, contiguous.

    python scripts/perf_dense_blocked.py [--out profiles/r4_perf_dense_blocked.json] [--small]

Cases:
  * `cholesky` of 64 Gram matrices of 128 x 128 complex double (configs[3]'s basis per time slice),
    against torch.linalg.cholesky;
  * `trsm` Q = V U^-1 for V of 32^3 x 64 sites x 128 vectors complex double (4.3 GB), against
    torch.linalg.solve_triangular;
  * `cholesky` and a 4096-rhs left `trsm` of one matrix of n = 1024 and 4096, complex double and double.
    For these, the DMMA contraction kernel's rate on the update steps (their 8 or 2 M N K flops over the
    time of the contract_mma launches, read with the library's CUDA-event kernel timer in a separate
    pass) is given as a share of the rate of torch.matmul on a 4096^3 product measured in the same run.
Times are CUDA-event times of the whole call, median of the timed repetitions after a warm-up.  The
card name, power limit and maximum SM clock come from nvidia-smi in the same run.  --small runs
everything at a tiny size (a check of the script, not a measurement)."""
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
from scripts.perf_dense import card, part, timed  # noqa: E402


def update_flops(plan, cplx):
    f = 0
    for it in plan["items"]:
        for st in it.get("steps", []):
            if st["step"] == "update":
                vol = lambda g: int(np.prod([d[0] for d in st.get(g, [])]))
                f += (8 if cplx else 2) * vol("T") * vol("M") * vol("N") * vol("K")
    return f


def mma_seconds(fn):
    sb.sync(sb.createGpuContext(0))
    sb.profile_read("contract_mma")
    sb.profile_enable(True)
    fn()
    sb.profile_enable(False)
    ms, _ = sb.profile_read("contract_mma")
    return ms * 1e-3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    gpu = sb.createGpuContext(0)
    co = sb.FastToSlow
    sync = lambda: sb.sync(gpu)
    g = torch.Generator(device="cuda").manual_seed(1)
    res = dict(card=card())

    # ---- 64 Gram matrices of 128 x 128, complex double --------------------------------------------
    m, nt = 128, 64
    b = torch.randn(nt, 2 * m, m, dtype=torch.complex128, device="cuda", generator=g)
    gram = b.mH @ b                                                   # [t, w, v], Hermitian
    graml = gram.transpose(1, 2).contiguous().view(-1)                # "wvt": w fastest
    u = graml.clone()
    pg = part([m, m, nt])
    chol = lambda: (u.copy_(graml), sb.cholesky(pg, 1, "wvt", [u], "w", "v", gpu, co), sync())
    res["cholesky_128x128_x64_c128"] = dict(seconds=timed(chol),
                                            copy_seconds=timed(lambda: (u.copy_(graml), torch.cuda.synchronize())),
                                            note="the call and a refreshing copy of the matrices")
    res["torch_cholesky_128x128_x64"] = dict(seconds=timed(lambda: torch.linalg.cholesky(gram)))
    um = u.view(nt, m, m)[0].t()                                      # [w, v] upper: U of slice 0
    ref = torch.linalg.cholesky(gram[0]).mH
    res["cholesky_128x128_x64_c128"]["max_abs_diff_vs_torch"] = (um - ref).abs().max().item()

    # ---- Q = V U^-1, V of 32^3 x 64 sites x 128 vectors ---------------------------------------------
    L, T = (4, 8) if args.small else (32, 64)
    nv = L * L * L * T
    v = torch.randn(nv * m, dtype=torch.complex128, device="cuda", generator=g)    # "iv": i fastest
    u1 = u[:m * m].clone()                                                          # "wv"
    p1, pv = part([m, m]), part([nv, m])
    q = torch.empty_like(v)
    trsm = lambda: (sb.trsm(1, p1, 1, "wv", "w", "v", [u1], gpu, pv, 1, "iv", [v], gpu, pv, 1, "iw", [q], gpu,
                            co), sync())
    res["trsm_VUinv_128_c128"] = dict(sites=nv, vbytes=nv * m * 16, seconds=timed(trsm, reps=3, warmup=1))
    vm, umat = v.view(m, nv).t(), u1.view(m, m).t()                  # [site, vec] (strided), [w, v]
    vc = vm.contiguous()
    res["torch_solve_triangular_VUinv_128"] = dict(seconds=timed(
        lambda: torch.linalg.solve_triangular(umat, vc, upper=True, left=False), reps=3, warmup=1))
    want = torch.linalg.solve_triangular(umat, vc, upper=True, left=False)
    res["trsm_VUinv_128_c128"]["max_abs_diff_vs_torch"] = (q.view(m, nv).t() - want).abs().max().item()
    del v, q, vm, vc, want
    torch.cuda.empty_cache()

    # ---- one large matrix: cholesky and a 4096-rhs trsm -----------------------------------------------
    big = 4096 if not args.small else 256
    for name, dt, tdt in (("c128", sb.C128, torch.complex128), ("f64", sb.F64, torch.float64)):
        cplx = tdt.is_complex
        x0 = torch.randn(big, big, dtype=tdt, device="cuda", generator=g)
        y0 = torch.randn(big, big, dtype=tdt, device="cuda", generator=g)
        t_mm = timed(lambda: torch.matmul(x0, y0))
        gemm_rate = (8 if cplx else 2) * big ** 3 / t_mm
        res["torch_matmul_%d_%s" % (big, name)] = dict(seconds=t_mm, flops_per_s=gemm_rate)
        del x0, y0
        for n in ((1024, 4096) if not args.small else (256,)):
            bm = torch.randn(n, n, dtype=tdt, device="cuda", generator=g)
            h = bm.mH @ bm + n * torch.eye(n, dtype=tdt, device="cuda")
            hl = h.t().contiguous().view(-1)                            # "ab": rows a fastest
            a = hl.clone()
            pa = part([n, n])
            plan = sb.dense_plan(sb.CHOLESKY, dt, pa, 1, "ab", "a", "b", co, 1, 0)
            fn = lambda: (a.copy_(hl), sb.cholesky(pa, 1, "ab", [a], "a", "b", gpu, co), sync())
            t = timed(fn)
            upd = update_flops(plan, cplx)
            tm = mma_seconds(fn)
            res["cholesky_%d_%s" % (n, name)] = dict(
                seconds=t, copy_seconds=timed(lambda: (a.copy_(hl), torch.cuda.synchronize())),
                update_flops=upd, mma_seconds=tm, update_share_of_gemm=upd / tm / gemm_rate if tm else None)
            res["torch_cholesky_%d_%s" % (n, name)] = dict(seconds=timed(lambda: torch.linalg.cholesky(h)))
            ua = a.view(n, n).t()                                       # [row, col] upper
            res["cholesky_%d_%s" % (n, name)]["max_abs_diff_vs_torch"] = \
                (ua - torch.linalg.cholesky(h).mH).abs().max().item()
            nr = 4096 if not args.small else 64
            x = torch.randn(nr * n, dtype=tdt, device="cuda", generator=g)   # "ar": a fastest
            y = torch.empty_like(x)
            px = part([n, nr])
            plan = sb.dense_plan(sb.TRSM, dt, pa, 1, "ab", "a", "b", co, 1, 0, px=px, ncomponentsx=1, ox="ar",
                                 py=px, ncomponentsy=1, oy="br")
            fn = lambda: (sb.trsm(1, pa, 1, "ab", "a", "b", [a], gpu, px, 1, "ar", [x], gpu, px, 1, "br", [y], gpu,
                                  co), sync())
            t = timed(fn)
            upd = update_flops(plan, cplx)
            tm = mma_seconds(fn)
            res["trsm_left_%d_%drhs_%s" % (n, nr, name)] = dict(
                seconds=t, update_flops=upd, mma_seconds=tm, update_share_of_gemm=upd / tm / gemm_rate if tm else None)
            xc = x.view(nr, n).t().contiguous()                         # [row, rhs]
            res["torch_solve_triangular_%d_%drhs_%s" % (n, nr, name)] = dict(seconds=timed(
                lambda: torch.linalg.solve_triangular(ua, xc, upper=True)))
            res["trsm_left_%d_%drhs_%s" % (n, nr, name)]["max_abs_diff_vs_torch"] = \
                (y.view(nr, n).t() - torch.linalg.solve_triangular(ua, xc, upper=True)).abs().max().item()
            del bm, h, hl, a, x, y, xc
            torch.cuda.empty_cache()
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
