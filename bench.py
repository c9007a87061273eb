#!/usr/bin/env python
"""bench.py — the tensor hot path of superbblas on B200: contraction TFLOP/s (headline) and
reshuffle GB/s, against measured rooflines, next to the reference's CPU build on the host cores.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 2|4]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload (--config 2, the default; BASELINE.json configs[1] per GPU): the distillation
contraction
    R[t,n,m] = sum_{c,x,y,z} conj(V0[c,x,y,z,t,n]) * V1[c,x,y,z,t,m],   complex double,
32^3 x 64 sites and n = m = 64 vectors PER GPU (2.0616e11 flop, 12.9 GB of operands).  With N GPUs
the lattice grows to 32 x 32 x (32*Pz) x (64*Pt), (Pz,Pt) = (1,1),(2,1),(2,2),(2,4), partitioned on
z,t like BASELINE configs[3]; the z-halves produce partial sums that are reduced across ranks into
an output partitioned on t.  Weak scaling: the work per GPU is fixed.

Every line also carries `strong_config4`: BASELINE.json configs[3] itself -- the SAME global problem
at every N (48^3 x 96 sites, n = m = 128 vectors, 4.1747e12 flop, 130.5 GB of operands, z/t
partition z1t1, z2t1, z2t2, z2t4) -- i.e. the strong-scaling curve the north star asks for
(`--config 4` makes it the headline instead, with "scaling": "strong").

A step = one `contraction` call through the public API with device-resident operands (`value`), or
with HOST operands in pinned memory, staged by the library (`e2e`).  Timing: CUDA events on the
library's stream, barrier + synchronize on both sides, max over ranks.  Operands are far larger
than the 126 MB L2, so no flush is needed between steps.  At N > 1 every rank checks its slice of
the result against a cuBLAS evaluation of the same time slices (partials of the z-halves summed
with an all-reduce) and the reshuffles against index-valued tensors; `result_check` must be true.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CPU_SAMPLE_T = 16               # time slices per part of the CPU sample (1/4 of one GPU's work)
# the committed ncu digest the headline kernel's DRAM traffic is read from
TRAFFIC_PROFILE = os.path.join("profiles", "r2_contract_mma_ncu.txt")


def grid_for(n):
    pz = 2 if n % 2 == 0 else 1
    return pz, n // pz


class Workload:
    """The distillation contraction on `world` GPUs.  config 2: weak (32^3 x 64, n = 64 per GPU);
    config 4: strong (48^3 x 96, n = 128 in total)."""

    def __init__(self, config, world):
        self.config, self.world = config, world
        self.pz, self.pt = grid_for(world)
        if config == 2:
            self.L, self.nv = 32, 64
            self.lz, self.lt = 32 * self.pz, 64 * self.pt
            self.scaling = "weak"
        else:
            self.L, self.nv = 48, 128
            self.lz, self.lt = 48, 96
            self.scaling = "strong"
        self.dimv = [3, self.L, self.L, self.lz, self.lt, self.nv]
        self.dimr = [self.lt, self.nv, self.nv]
        self.flop = 8.0 * self.lt * self.nv * self.nv * 3 * self.L * self.L * self.lz  # all GPUs
        self.flop_per_gpu = self.flop / world

    def describe(self):
        if self.config == 2:
            w = ("BASELINE configs[1] per GPU: contraction cxyztn^H . cxyztm -> tnm, 32^3x64 sites "
                 "and n=m=64 complex double per GPU")
        else:
            w = ("BASELINE configs[3]: contraction cxyztn^H . cxyztm -> tnm, 48^3x96 sites and "
                 "n=m=128 complex double in total, the same global problem at every N")
        return {"workload": w, "lattice": [self.L, self.L, self.lz, self.lt], "vectors": self.nv,
                "partition": "z%d x t%d" % (self.pz, self.pt), "coor_order": "FastToSlow",
                "l2": "operands (%.1f GB per GPU) exceed L2; no flush"
                      % (2 * np.prod(self.dimv) * 16 / self.world / 1e9)}


# ---------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the UNMODIFIED reference (oracle/_ref/libsbref.so) on the host cores
# ---------------------------------------------------------------------------------------------------

def _omp_threads_in_use():
    """What the OpenMP runtime the reference library runs on will really use"""
    import ctypes
    try:
        return int(ctypes.CDLL("libgomp.so.1").omp_get_max_threads())
    except OSError:
        return None


def cpu_contraction_sample(reps, warmup, nparts=1):
    """Times the reference's CPU contraction on a bounded sample of the headline workload: the same
    32^3 spatial block and n = m = 64 vectors per part, `nparts` parts laid out z x t like the GPU
    ranks (as components of one process, BASELINE.md §3), 16 of the 64 time slices of every part
    (5.15e10 flop per part and step: the sample grows with N like the GPU arm's work, and every
    part keeps a batch of 16 matrices for the reference's OpenMP loop over the batch)."""
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    # torch.distributed.run exports OMP_NUM_THREADS=1 to its workers: set, do not setdefault
    os.environ["OMP_NUM_THREADS"] = str(cores)
    os.environ["OPENBLAS_NUM_THREADS"] = "1"  # the reference parallelises over the batch (blas_cpu_tmpl.hpp:469)
    from oracle import ref as R
    if not R.available():
        raise RuntimeError("oracle/_ref/libsbref.so is missing (run `make -C oracle` where "
                           "/root/reference exists)")
    R.lib()
    threads = _omp_threads_in_use()
    L, NV = 32, 64
    pz, pt = grid_for(nparts)
    lt_part = CPU_SAMPLE_T
    dimv, dimr = [3, L, L, L * pz, lt_part * pt, NV], [lt_part * pt, NV, NV]
    pv = R.basic_partitioning("cxyztn", dimv, [1, 1, 1, pz, pt, 1], "zt", nparts, 1)
    pr = R.basic_partitioning("tnm", dimr, [nparts, 1, 1], "t", nparts, 1)
    rng = np.random.default_rng(0x5B5B0000 + 2 * 16)
    mk = lambda n: rng.random(n) + 1j * rng.random(n)  # noqa: E731
    a0, b0 = mk(int(np.prod(pv[0, 1]))), mk(int(np.prod(pv[0, 1])))
    a = [a0] + [a0.copy() for i in range(1, nparts)]  # (all parts have the same shape; the values do not matter here)
    b = [b0] + [b0.copy() for i in range(1, nparts)]
    c = [np.zeros(int(np.prod(pr[i, 1])), dtype=np.complex128) for i in range(nparts)]
    times = []
    for i in range(warmup + reps):
        t0 = time.perf_counter()
        R.contraction(1, pv, [0] * 6, dimv, dimv, "cxyztn", True, a, pv, [0] * 6, dimv, dimv,
                      "cxyztm", False, b, 0, pr, [0] * 3, dimr, dimr, "tnm", c, "FastToSlow")
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    flop = 8.0 * dimr[0] * NV * NV * 3 * L * L * dimv[3]
    return dict(total_s=sum(times), steps=len(times), flop_per_step=flop, cores=threads or cores,
                kind="reference", dims=dimv,
                sample="the headline contraction on a %s lattice (%d of the %d time slices of the "
                       "%d-GPU workload, %.3g flop per step) in %d CPU component(s) z%d x t%d of one "
                       "process; OpenMP threads in use = %s (host cores available %d), "
                       "OPENBLAS_NUM_THREADS=1"
                       % ("x".join(map(str, dimv[1:5])), dimr[0], 64 * pt, nparts, flop, nparts, pz,
                          pt, threads, cores))


def cpu_copy_sample(reps=5):
    """The reference's CPU copy on a bounded sample of the reshuffle workload: "xyztsc" -> "cstzyx" on
    16^3 x 32 x 4 x 3 complex double (25 MB; warm calls, i.e. with its index vectors cached)."""
    cores = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(cores)
    from oracle import ref as R
    dim0, dim1 = [16, 16, 16, 32, 4, 3], [3, 4, 32, 16, 16, 16]
    p0 = np.array([[[0] * 6, dim0]], dtype=np.int32)
    p1 = np.array([[[0] * 6, dim1]], dtype=np.int32)
    n = int(np.prod(dim0))
    rng = np.random.default_rng(1)
    a = rng.random(n) + 1j * rng.random(n)
    b = np.zeros(n, dtype=np.complex128)
    best = None
    for i in range(reps + 2):
        t0 = time.perf_counter()
        R.copy(1, p0, "xyztsc", [0] * 6, dim0, dim0, [a], p1, "cstzyx", [0] * 6, dim1, [b], "FastToSlow", 0)
        dt = time.perf_counter() - t0
        if i >= 2:
            best = dt if best is None else min(best, dt)
    return {"GB/s": 2 * n * 16 / best / 1e9, "ms": best * 1e3, "cores": cores, "kind": "reference",
            "sample": "16^3 x 32 x 4 x 3 complex double (25 MB), warm (index vectors cached)"}


def reference_gpu_comparator():
    """The unmodified reference in CUDA mode (thrust + cuBLAS, built for sm_100 by oracle/Makefile)
    timed on this GPU on the bench shapes: the bar SURVEY §2.1 sets ("beat thrust + cuBLAS on the
    same B200").  Runs in a process of its own; returns its JSON or {"unavailable": why}."""
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_gpu_bench")
    if not os.path.exists(exe):
        return {"unavailable": "oracle/_ref/ref_gpu_bench is not built (make -C oracle where /root/reference exists)"}
    blasdir = os.environ.get(
        "SBREF_BLASDIR", "/opt/prime-rl/.venv/lib/python3.12/site-packages/opencv_python_headless.libs")
    env = dict(os.environ, LD_LIBRARY_PATH=blasdir + ":" + os.environ.get("LD_LIBRARY_PATH", ""),
               OMP_NUM_THREADS="1")
    try:
        out = subprocess.run([exe, "--reps=5"], capture_output=True, text=True, timeout=300, env=env)
        line = [l for l in out.stdout.splitlines() if l.startswith("{")]
        if not line:
            return {"unavailable": "no output (rc %d): %s" % (out.returncode, out.stderr[-200:])}
        return json.loads(line[-1])
    except Exception as e:  # noqa: BLE001
        return {"unavailable": str(e)[:200]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    try:
        r = cpu_contraction_sample(args.steps, args.warmup, nparts=max(1, args.gpus))
    except Exception as e:  # noqa: BLE001
        print(json.dumps({"impl": "reference", "unavailable": str(e).splitlines()[0]}))
        return 0
    value = r["flop_per_step"] * r["steps"] / r["total_s"] / 1e12
    cfg = Workload(2, max(1, args.gpus)).describe()
    cfg["workload"] += " -- CPU arm: bounded sample, see cpu_baseline.sample"
    cfg["sample_lattice"] = r["dims"][1:5]
    line = {
        "impl": "reference", "metric": "contraction TFLOP/s (distillation V^H V -> [t,n,m])",
        "value": value, "unit": "TFLOP/s", "n_gpus": args.gpus, "steps": r["steps"],
        "warmup": args.warmup, "ms_per_step": 1e3 * r["total_s"] / r["steps"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "c128",
        "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": "TFLOP/s", "cores": r["cores"], "kind": r["kind"],
                         "sample": r["sample"]},
        "e2e": {"value": value, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def bind_host_to_gpu_numa(torch, local):
    """N > 1: keep this rank's host threads -- and therefore its pinned staging buffers (first touch)
    -- on the CPUs NVML names as local to its GPU, so that the host->device copies of the e2e leg do
    not cross sockets.  Best effort: returns the number of CPUs bound to, or None when anything is
    missing (SBB_BENCH_NUMA=0 disables it).  Not used at N = 1, where the CPU baseline needs every core."""
    if os.environ.get("SBB_BENCH_NUMA", "1") == "0":
        return None
    try:
        import pynvml
        pynvml.nvmlInit()
        u = str(torch.cuda.get_device_properties(local).uuid)
        if not u.startswith("GPU-"):
            u = "GPU-" + u
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(u)
        except TypeError:
            h = pynvml.nvmlDeviceGetHandleByUUID(u.encode())
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        return None


def traffic_from_profile():
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the headline kernel, parsed from
    the committed ncu digest (ncu --set full); None when the file is missing or unreadable."""
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    try:
        total = 0.0
        for line in open(os.path.join(ROOT, TRAFFIC_PROFILE)):
            m = re.match(r"dram__bytes_(read|write)\.sum\s+([0-9.]+)\s+(\w+)", line)
            if m:
                total += float(m.group(2)) * unit[m.group(3)]
        return total or None
    except Exception:  # noqa: BLE001
        return None


# ---------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------

class ClockSampler:
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms",
                 "50", "-i", str(self.index)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                w = [x.strip() for x in line.split(",")]
                if len(w) < 10:
                    continue
                try:
                    sm.append(float(w[2])), mx.append(float(w[3]))
                except ValueError:
                    continue
                for k, nm in enumerate(names):
                    if w[6 + k].lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except Exception:  # noqa: BLE001
            pass
        if sm:
            # under load = the upper half of the samples (the sampler also sees idle gaps)
            hi = sorted(sm)[len(sm) // 2:]
            out.update(sm_mhz=float(np.median(hi)), sm_max_mhz=max(mx), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------

class Env:
    """Process-wide state of one rank of the benchmark"""
    pass


def make_operands(E, W):
    """Two distinct random operands and a zeroed result for workload W on this rank (uniform in
    [-1,1), generated in place: a 65 GB operand has no room for temporaries)."""
    torch = E.torch
    pv = E.sb.basic_partitioning("cxyztn", W.dimv, [1, 1, 1, W.pz, W.pt, 1], "zt", E.world, 1)
    pr = E.sb.basic_partitioning("tnm", W.dimr, [E.world, 1, 1], "t", E.world, 1)
    nloc = int(np.prod(pv[E.rank, 1].astype(np.int64)))
    nout = int(np.prod(pr[E.rank, 1].astype(np.int64)))
    g = torch.Generator(device=E.dev).manual_seed(0x5B5B0000 + W.config * 16 + E.rank)

    def mk():
        x = torch.empty(nloc, 2, device=E.dev, dtype=torch.float64)
        x.uniform_(-1.0, 1.0, generator=g)
        return torch.view_as_complex(x)
    a, b = mk(), mk()
    r = torch.zeros(nout, device=E.dev, dtype=torch.complex128)
    return pv, pr, a, b, r


def contraction_step(E, W, pv, pr, va, vb, vr, ctx):
    E.sb.contraction(1, pv, [0] * 6, W.dimv, W.dimv, 1, "cxyztn", True, [va], ctx, pv, [0] * 6,
                     W.dimv, W.dimv, 1, "cxyztm", False, [vb], ctx, 0, pr, [0] * 3, W.dimr, W.dimr,
                     1, "tnm", [vr], ctx, E.sb.FastToSlow, comm=E.comm)


def check_contraction(E, W, pv, pr, a, b, r, tol=1e-12):
    """Every rank checks one time slice of ITS part of the result against cuBLAS: each rank
    evaluates, for the first time slice of every rank's output range that lies in its own lattice
    block, the partial product over its z-range; the partials are summed over ranks (all-reduce)
    and rank o compares entry o with what the library left in r.  Returns the largest relative
    error over ranks."""
    torch, dist = E.torch, E.dist
    nv = W.nv
    box, obox = pv[E.rank], pr[E.rank]
    lt_loc = int(box[1][4])
    kloc = int(np.prod(box[1][:4].astype(np.int64)))
    A, B = a.view(nv, lt_loc, kloc), b.view(nv, lt_loc, kloc)
    ref = torch.zeros(E.world, nv, nv, device=E.dev, dtype=torch.complex128)
    for o in range(E.world):
        if int(pr[o][1][0]) == 0:
            continue
        t = int(pr[o][0][0])  # first time slice of rank o's output
        tl = t - int(box[0][4])
        if 0 <= tl < lt_loc:
            ref[o] = B[:, tl, :] @ A[:, tl, :].conj().T  # [m][n]
    if E.world > 1:
        dist.all_reduce(ref)
    err = 0.0
    if int(obox[1][0]) > 0:
        got = r.view(nv, nv, int(obox[1][0]))[:, :, 0]
        err = float((torch.linalg.norm(got - ref[E.rank]) / torch.linalg.norm(ref[E.rank])).item())
    err = E.max_over_ranks(err)
    return err, bool(err < tol)


def bench_contraction(E, W, steps, warmup, profile=True):
    """Device-resident timing of workload W; returns the numbers and keeps the tensors in `out`"""
    sb = E.sb
    pv, pr, a, b, r = make_operands(E, W)
    fn = lambda: contraction_step(E, W, pv, pr, a, b, r, E.gpu)  # noqa: E731
    # The dominant kernel is timed in the SAME steps as the step itself: a pair of CUDA events around
    # every launch of it, on the stream it is launched on (two event records per 6 ms kernel do not
    # change the step; a separate pass for the kernel timing saw other clocks than the timed pass)
    sb.profile_enable(profile)

    def reset_counters():  # after the warm-up steps: only the timed steps are counted
        sb.profile_read("contract_mma")
        sb.launch_count(reset=True)
    ms = E.timed(fn, steps, warmup, after_warmup=reset_counters)
    launches = sb.launch_count()
    out = {"ms_per_step": ms / steps, "value": W.flop * steps / (ms * 1e-3) / 1e12,
           "launches": launches}
    if profile:
        kms, kn = sb.profile_read("contract_mma")
        sb.profile_enable(False)
        out["kernel_ms"] = E.max_over_ranks(kms / max(kn, 1))
        out["kernel_tflops"] = W.flop_per_gpu / (out["kernel_ms"] * 1e-3) / 1e12
    err, ok = check_contraction(E, W, pv, pr, a, b, r)
    out["rel_err"], out["check"] = err, ok
    return out, (pv, pr, a, b, r)


def dump_outputs(E, W, path, pr, r):
    """The result a caller of the timed contraction receives, as DIR/tnm.npy (DIR/tnm_rank<k>.npy
    on every rank when N > 1): float64 of shape [m, n, t, 2], the part [t, n, m] of this rank with t
    fastest and (re, im) last.  The operands are seeded, so two builds run with the same arguments
    can be compared output for output.  At most 25 MB in all (config 4)."""
    os.makedirs(path, exist_ok=True)
    lt = int(pr[E.rank][1][0])
    name = "tnm" if E.world == 1 else "tnm_rank%d" % E.rank
    out = E.torch.view_as_real(r).view(W.nv, W.nv, lt, 2).cpu().numpy()
    np.save(os.path.join(path, name + ".npy"), out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 4],
                    help="headline workload: 2 = BASELINE configs[1] per GPU (weak), 4 = configs[3] (strong)")
    ap.add_argument("--no-extras", action="store_true", help="skip the reshuffle measurements")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline contraction's result of the last timed step to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; --impl reference has none")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import superbblas_b200 as sb

    E = Env()
    E.torch, E.dist, E.sb = torch, dist, sb
    E.rank = rank = int(os.environ.get("RANK", "0"))
    E.world = world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node %d" % args.gpus)
    torch.cuda.set_device(local)
    E.dev = dev = torch.device("cuda", local)
    host_affinity = bind_host_to_gpu_numa(torch, local) if world > 1 else None
    E.comm = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(sb.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        E.comm = sb.comm_create(bytes(uid.cpu().numpy().tobytes()), world, rank, local)
    E.gpu = gpu = sb.createGpuContext(local)
    cpu = sb.createCpuContext()
    E.stream = stream = torch.cuda.ExternalStream(sb.get_stream(local), device=dev)

    def barrier():
        sb.sync(gpu)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps, warmup, after_warmup=None):
        for _ in range(warmup):
            fn()
        barrier()
        if after_warmup:
            after_warmup()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))
    E.barrier, E.max_over_ranks, E.timed = barrier, max_over_ranks, timed

    # ---- FP64 roofline denominator, measured live (MEASURED_PEAKS.json has no FP64 entry) ----------
    def zgemm_peak():
        n = 4096
        x = torch.randn(n, n, device=dev, dtype=torch.complex128)
        y = torch.randn(n, n, device=dev, dtype=torch.complex128)
        best = 1e9
        for i in range(7):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(x, y)
            e1.record()
            torch.cuda.synchronize()
            if i >= 2:
                best = min(best, e0.elapsed_time(e1))
        return 8.0 * n ** 3 / best / 1e9
    fp64_peak = zgemm_peak()

    warmup = max(args.warmup, 3)
    head = Workload(args.config, world)
    other = Workload(4 if args.config == 2 else 2, world)

    # ---- timed region: device-resident operands --------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    hd, (pv, pr, a, b, r) = bench_contraction(E, head, args.steps, warmup)
    clocks = sampler.stop() if rank == 0 else None
    checks = {"headline_contraction": hd["check"]}
    nloc, nout = a.numel(), r.numel()
    if args.dump_outputs:
        dump_outputs(E, head, args.dump_outputs, pr, r)

    # ---- the same contraction on complex float operands (N=1) --------------------------------------------
    contraction_c64 = None
    if world == 1 and not args.no_extras and args.config == 2:
        NV, LT, K = head.nv, head.lt, 3 * head.L ** 3
        A0, B0 = a.view(NV, LT, K)[:, 0, :], b.view(NV, LT, K)[:, 0, :]
        af, bf = a.to(torch.complex64), b.to(torch.complex64)
        rf = torch.zeros(nout, device=dev, dtype=torch.complex64)
        stepf = lambda: contraction_step(E, head, pv, pr, af, bf, rf, gpu)  # noqa: E731
        ms_f = timed(stepf, 10, 3)
        # the SM clock under this kernel (TMA + tensor cores + shared memory + HBM all busy: the 1 kW
        # power cap shows here first): a 2 s loop with the sampler on
        csamp = ClockSampler(local)
        csamp.start()
        t_end = time.time() + 2.0
        while time.time() < t_end:
            for _ in range(50):
                stepf()
            sb.sync(gpu)
        clocks_c64 = csamp.stop()
        sb.profile_enable(True)
        sb.profile_read("contract_tc")
        timed(stepf, 10, 1)
        kms_f, kn_f = sb.profile_read("contract_tc")
        sb.profile_enable(False)
        ref0f = (B0 @ A0.conj().T)
        got0f = rf.view(NV, NV, LT)[:, :, 0].to(torch.complex128)
        err_f = float((torch.linalg.norm(got0f - ref0f) / torch.linalg.norm(ref0f)).item())
        min_bytes = 2 * nloc * 8 + nout * 8
        hbm_floor_ms = min_bytes / 6545.3e9 * 1e3
        contraction_c64 = {"TFLOP/s": head.flop * 10 / (ms_f * 1e-3) / 1e12, "ms": ms_f / 10,
                           "rel_err_vs_c128": err_f, "min_bytes": min_bytes,
                           "kernel": "contract_tc_kernel (TMA + tcgen05 kind::tf32 x3, TMEM accumulators)",
                           "kernel_ms": kms_f / max(kn_f, 1), "clocks_under_this_kernel": clocks_c64,
                           "hbm_floor_ms": hbm_floor_ms,
                           "frac_of_hbm_roofline": hbm_floor_ms / (ms_f / 10),
                           "kernel_frac_of_hbm_roofline": hbm_floor_ms / (kms_f / max(kn_f, 1)) if kn_f else None}
        checks["contraction_c64"] = bool(err_f < 1e-5)
        del af, bf, rf

    # ---- e2e: HOST operands in pinned memory through the same public call ---------------------------------
    e2e = None
    if 2 * nloc * 16 <= 40e9:  # (config 4 on 1-2 GPUs would pin 65-130 GB of host memory per rank)
        e2e_steps = max(1, min(args.steps, 3))
        ha = torch.empty(nloc, dtype=torch.complex128, pin_memory=True)
        hb = torch.empty(nloc, dtype=torch.complex128, pin_memory=True)
        hr = torch.zeros(nout, dtype=torch.complex128, pin_memory=True)
        ha.copy_(a), hb.copy_(b)
        torch.cuda.synchronize()
        ms_e2e = timed(lambda: contraction_step(E, head, pv, pr, ha, hb, hr, cpu), e2e_steps, 1)
        e2e = {"value": head.flop * e2e_steps / (ms_e2e * 1e-3) / 1e12, "unit": "TFLOP/s",
               "h2d_bytes_per_step": 2 * nloc * 16 * world, "d2h_bytes_per_step": nout * 16 * world,
               "steps": e2e_steps, "ms_per_step": ms_e2e / e2e_steps}
        same = bool(torch.allclose(hr.to(dev), r, rtol=1e-12, atol=1e-9))
        checks["e2e_equals_device_result"] = bool(max_over_ranks(0.0 if same else 1.0) == 0.0)
        del ha, hb, hr
    del a, b, r
    torch.cuda.empty_cache()
    sb.clearCaches()

    # ---- the other contraction workload (config 4 strong scaling unless it is the headline) ---------------
    other_block = None
    if not args.no_extras:
        od, tensors = bench_contraction(E, other, max(3, min(args.steps, 10)), 3)
        del tensors
        torch.cuda.empty_cache()
        sb.clearCaches()
        other_block = {"config": other.describe(), "scaling": other.scaling, "value": od["value"],
                       "unit": "TFLOP/s", "ms_per_step": od["ms_per_step"],
                       "kernel_ms": od["kernel_ms"], "kernel_TFLOP/s_per_gpu": od["kernel_tflops"],
                       "frac_of_fp64_tensor_peak": od["kernel_tflops"] / fp64_peak,
                       "flop_per_step": other.flop, "rel_err_vs_cublas": od["rel_err"],
                       "result_check": od["check"]}
        checks["other_contraction"] = od["check"]

    # ---- extras: reshuffle GB/s -------------------------------------------------------------------------
    extras = {}
    hbm_peak, hbm_src = 6650.0, "fallback"
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        hbm_peak, hbm_src = float(mp["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:  # noqa: BLE001
        pass
    if not args.no_extras:
        extras = reshuffle_extras(E, hbm_peak, checks)

    # ---- CPU reference for the reshuffle (rank 0, N=1 only): same permutation, 16^3 x 32 x 4 x 3 ------------
    if world == 1 and not args.no_cpu and not args.no_extras:
        try:
            extras["cpu_reference_permute_xyztsc_cstzyx_c128"] = cpu_copy_sample()
        except Exception as e:  # noqa: BLE001
            extras["cpu_reference_permute_xyztsc_cstzyx_c128"] = {"unavailable": str(e)}

    # ---- the reference's own GPU path on this GPU (N=1 only; our tensors are freed by now) ----------------------
    reference_gpu = None
    if world == 1 and not args.no_extras and not args.no_cpu:
        torch.cuda.empty_cache()
        sb.clearCaches()
        reference_gpu = reference_gpu_comparator()

    # ---- CPU baseline (rank 0, N=1 only) -----------------------------------------------------------------
    cpu_baseline = None
    if world == 1 and not args.no_cpu:
        try:
            # in a process of its own (the reference arm of this script): inside this process two
            # OpenMP runtimes (torch's and the reference library's) fight over the cores and the
            # same sample runs 3x slower
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference",
                                  "--steps", "3", "--warmup", "1"], capture_output=True, text=True,
                                 timeout=600).stdout
            ref = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
            if "unavailable" in ref:
                raise RuntimeError(ref["unavailable"])
            cpu_baseline = ref["cpu_baseline"]
        except Exception as e:  # noqa: BLE001
            cpu_baseline = {"value": None, "unit": "TFLOP/s", "cores": os.cpu_count(),
                            "kind": "reference", "sample": "unavailable: %s" % e}

    result_check = all(bool(v) for v in checks.values())
    if rank == 0:
        summary = {k: {"GB/s_per_gpu": v["GB/s"] / world, "frac_of_hbm": v["per_gpu_frac_of_hbm"]}
                   for k, v in extras.items() if isinstance(v, dict) and "per_gpu_frac_of_hbm" in v}
        for k, v in (extras.get("config1") or {}).items():
            checks["config1_" + k] = v["check"]
        result_check = all(bool(v) for v in checks.values())
        line = {
            "metric": "contraction TFLOP/s (distillation V^H V -> [t,n,m])",
            "value": hd["value"], "unit": "TFLOP/s", "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": hd["ms_per_step"],
            "higher_is_better": True, "scaling": head.scaling, "vs_baseline": None, "dtype": "c128",
            "data": "synthetic", "config": head.describe(),
            "roofline": {"bound": "tensor", "achieved": hd["kernel_tflops"], "peak": fp64_peak,
                         "unit": "TFLOP/s", "frac": hd["kernel_tflops"] / fp64_peak,
                         # dram__bytes_read.sum + dram__bytes_write.sum of one launch at N = 1
                         "traffic": traffic_from_profile() if args.config == 2 else None,
                         "traffic_source": TRAFFIC_PROFILE,
                         "kernel": "contract_mma_kernel<double2>", "kernel_ms": hd["kernel_ms"],
                         "flop_per_launch": head.flop_per_gpu,
                         "peak_source": "FP64 tensor path: cuBLAS ZGEMM 4096^3 via torch.matmul, "
                                        "best of 5, measured live in this run (MEASURED_PEAKS.json "
                                        "has no FP64 entry; ncu's own peak_sustained is 37.1 and "
                                        "the nominal figure 40)",
                         "frac_of_nominal_40": hd["kernel_tflops"] / 40.0},
            "cpu_baseline": cpu_baseline,
            "e2e": e2e,
            "gpu_launches": hd["launches"], "clocks": clocks, "result_check": result_check,
            "checks": checks, "rel_err_vs_cublas": hd["rel_err"],
            "host_cpus_bound_to_gpu_numa": host_affinity,
            ("strong_config4" if args.config == 2 else "weak_config2"): other_block,
            "reshuffle_summary": summary, "reshuffle": extras, "contraction_c64": contraction_c64,
            "reference_gpu": reference_gpu,
            "hbm_peak_gbs": hbm_peak, "hbm_peak_source": hbm_src,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not result_check:
        sys.stderr.write("bench.py: RESULT CHECK FAILED: %s\n" % json.dumps(checks))
        return 3
    return 0


def index_field(torch, dev, box, dim, shift, cplx_dtype):
    """Tensor over the local box `box` = (from, size) of a lattice `dim` (first label fastest) whose
    element at global coordinate c holds the global linear index of (c - shift) mod dim, split into
    (re, im) = (index mod 2^22, index div 2^22) so that complex float carries it exactly.  With
    shift = 0 this is the reference's mock source tensor of its SB_DEBUG self-check
    (dist.h:2022-2063); with the copy's displacement it is what the destination must hold."""
    frm, size = [int(x) for x in box[0]], [int(x) for x in box[1]]
    nd = len(dim)
    idx = torch.zeros([1] * nd, dtype=torch.int64, device=dev)
    gstride = 1
    for k in range(nd):
        c = (torch.arange(size[k], device=dev, dtype=torch.int64) + frm[k] - shift[k]) % dim[k]
        shape = [1] * nd
        shape[nd - 1 - k] = size[k]  # first label fastest = last torch dimension
        idx = idx + (c * gstride).view(shape)
        gstride *= dim[k]
    idx = idx.reshape(-1)
    real = torch.float32 if cplx_dtype == torch.complex64 else torch.float64
    out = torch.empty(idx.numel(), 2, device=dev, dtype=real)
    out[:, 0] = (idx % (1 << 22)).to(real)
    out[:, 1] = (idx >> 22).to(real)
    return torch.view_as_complex(out)


def config1_block(E):
    """BASELINE configs[0] (the reference's own CPU-runnable case) on the GPU: the permutation
    "xyztsc" -> "cstzyx" and the contractions over s,c on an 8^3 x 16 complex-double lattice
    (1.5 MB tensors: launch-latency bound; microseconds per call, device time between events)."""
    sb, torch, dev, gpu, timed = E.sb, E.torch, E.dev, E.gpu, E.timed
    dim = [8, 8, 8, 16, 4, 3]
    one = lambda d: np.array([[[0] * len(d), list(d)]], dtype=np.int32)  # noqa: E731
    rnd = lambda n: torch.view_as_complex(torch.rand(n, 2, device=dev, dtype=torch.float64) * 2 - 1)  # noqa: E731
    out = {}
    n = int(np.prod(dim))
    x, y = rnd(n), torch.zeros(n, device=dev, dtype=torch.complex128)
    dim1 = dim[::-1]
    ms = timed(lambda: sb.copy(1, one(dim), 1, "xyztsc", [0] * 6, dim, dim, [x], None, gpu, one(dim1), 1,
                               "cstzyx", [0] * 6, dim1, [y], None, gpu, sb.FastToSlow, sb.Copy), 100, 10)
    ok = torch.equal(y.view(8, 8, 8, 16, 4, 3), x.view(3, 4, 16, 8, 8, 8).permute(5, 4, 3, 2, 1, 0))
    out["permute_xyztsc_cstzyx_c128"] = {"us_per_call": ms * 10, "GB/s": 2 * n * 16 / (ms / 100) / 1e6,
                                         "check": bool(ok)}
    for name, o0, d0, o1, d1, o_r, dr in (
            ("site_contraction_sc", "xyztsc", dim, "xyztsc", dim, "xyzt", dim[:4]),
            ("contract_cpp_style_n4", "xyztscN", dim + [4], "xyztscn", dim + [4], "xyztNn", dim[:4] + [4, 4])):
        a, b = rnd(int(np.prod(d0))), rnd(int(np.prod(d1)))
        r = torch.zeros(int(np.prod(dr)), device=dev, dtype=torch.complex128)
        ms = timed(lambda: sb.contraction(1, one(d0), [0] * len(d0), d0, d0, 1, o0, True, [a], gpu, one(d1),
                                          [0] * len(d1), d1, d1, 1, o1, False, [b], gpu, 0, one(dr),
                                          [0] * len(dr), dr, dr, 1, o_r, [r], gpu, sb.FastToSlow), 100, 10)
        # FastToSlow: x fastest; the contracted (s,c) are the slowest labels of the operands
        A = a.view(*(d0[::-1]))
        B = b.view(*(d1[::-1]))
        if len(d0) == 6:
            ref = torch.einsum("cstzyx,cstzyx->tzyx", A.conj(), B)
        else:
            ref = torch.einsum("Ncstzyx,ncstzyx->nNtzyx", A.conj(), B)
        err = float((torch.linalg.norm(r - ref.reshape(-1)) / torch.linalg.norm(ref)).item())
        flop = 8.0 * np.prod(dr) * 12
        out[name] = {"us_per_call": ms * 10, "GFLOP/s": flop / (ms / 100) / 1e6, "rel_err": err,
                     "check": bool(err < 1e-12)}
    return out


def reshuffle_extras(E, hbm_peak, checks):
    """Reshuffle GB/s = moved elements x (sizeof T + sizeof Q) / time (the reference's `memops`,
    tensor.h:1087): label permutation, periodic shift, and (N > 1) redistribution t -> (z,t).
    Every distributed reshuffle is also run once on index-valued tensors and compared bit for bit
    with index arithmetic on every rank (`checks`)."""
    sb, torch, dev, gpu, comm, rank, world, timed = (E.sb, E.torch, E.dev, E.gpu, E.comm, E.rank,
                                                      E.world, E.timed)
    out = {}

    def field(nbytes_elem, n):
        return torch.view_as_complex(torch.rand(n, 2, device=dev, dtype=torch.float32
                                                if nbytes_elem == 8 else torch.float64))

    def record(name, nbytes, fn, steps=20):
        ms = timed(fn, steps, 3)  # the throughput figure: no per-kernel events in the stream
        sb.profile_enable(True)   # second pass: the copy kernels alone, bracketed by events
        sb.profile_read("permute")
        timed(fn, steps, 1)
        kms, kn = sb.profile_read("permute")
        sb.profile_enable(False)
        gbs = nbytes * world * steps / (ms * 1e-3) / 1e9
        kernel_ms = kms / steps  # all permute kernels of one step (they run back to back)
        out[name] = {"GB/s": gbs, "ms": ms / steps, "per_gpu_frac_of_hbm": gbs / world / hbm_peak,
                     "kernel_ms": kernel_ms, "kernel_launches_per_step": kn / steps,
                     "kernel_GB/s_per_gpu": nbytes / kernel_ms / 1e6 if kn else None}

    def all_ranks(ok):
        return bool(E.max_over_ranks(0.0 if ok else 1.0) == 0.0)

    # (a) label permutation "xyztsc" -> "cstzyx", 32^3 x 64 x 4 x 3 complex double per GPU (config 1 scaled)
    dim0 = [32, 32, 32, 64, 4, 3]
    dim1 = [3, 4, 64, 32, 32, 32]
    p0 = np.array([[[0] * 6, dim0]] * 1, dtype=np.int32)
    p1 = np.array([[[0] * 6, dim1]] * 1, dtype=np.int32)
    n = int(np.prod(dim0))
    x, y = field(16, n), torch.zeros(n, device=dev, dtype=torch.complex128)
    record("permute_xyztsc_cstzyx_c128", 2 * n * 16,
           lambda: sb.copy(1, p0, 1, "xyztsc", [0] * 6, dim0, dim0, [x], None, gpu, p1, 1, "cstzyx",
                           [0] * 6, dim1, [y], None, gpu, sb.FastToSlow, sb.Copy))
    # "xyztsc" first-fastest is torch shape (c,s,t,z,y,x); "cstzyx" is torch shape (x,y,z,t,s,c)
    checks["permute"] = all_ranks(torch.equal(
        y.view(32, 32, 32, 64, 4, 3), x.view(3, 4, 64, 32, 32, 32).permute(5, 4, 3, 2, 1, 0)))
    if world == 1:
        # (a') the same permutation restricted to the even sites by MaskType masks on both tensors (§8f row 1);
        # bytes as the reference counts them for masked copies: mask size x (sizeof T + sizeof Q), tensor.h:1087
        idx = torch.arange(n, device=dev)
        par = (idx % 32 + (idx // 32) % 32 + (idx // 1024) % 32 + (idx // 32768) % 64) % 2
        m0 = (par == 0).to(torch.float32)
        m1 = m0.view(3, 4, 64, 32, 32, 32).permute(5, 4, 3, 2, 1, 0).contiguous().view(-1)
        del idx, par
        y.zero_()
        record("masked_even_sites_permute_xyztsc_cstzyx_c128", 2 * n * 16,
               lambda: sb.copy(1, p0, 1, "xyztsc", [0] * 6, dim0, dim0, [x], [m0], gpu, p1, 1, "cstzyx",
                               [0] * 6, dim1, [y], [m1], gpu, sb.FastToSlow, sb.Copy), steps=10)
        want = x.view(3, 4, 64, 32, 32, 32).permute(5, 4, 3, 2, 1, 0) * m1.view(32, 32, 32, 64, 4, 3)
        checks["masked_permute"] = bool(torch.equal(y.view(32, 32, 32, 64, 4, 3), want))
        del m0, m1, want
    del x, y
    if world == 1:
        out["config1"] = config1_block(E)
    # (b) periodic +1 shifts of a 64^3 x 128 x 4 x 3 field distributed on z,t (config 5): per GPU block
    pz, pt = grid_for(world)
    for es, tag in ((8, "c64"), (16, "c128")):
        cdt = torch.complex64 if es == 8 else torch.complex128
        dim = [64, 64, 32 * pz, 32 * pt, 4, 3]  # 64 x 64 x 32 x 32 x (4,3) sites per GPU
        part = sb.basic_partitioning("xyztsc", dim, [1, 1, pz, pt, 1, 1], "zt", world, 1)
        nl = int(np.prod(part[rank, 1]))
        x = index_field(torch, dev, part[rank], dim, [0] * 6, cdt)
        y = torch.zeros_like(x)
        for mu, lab in enumerate("xyzt"):
            shift = [0] * 6
            shift[mu] = 1
            record("shift_%s_%s" % (lab, tag), 2 * nl * es,
                   lambda: sb.copy(1, part, 1, "xyztsc", [0] * 6, dim, dim, [x], None, gpu, part, 1,
                                   "xyztsc", shift, dim, [y], None, gpu, sb.FastToSlow, sb.Copy,
                                   comm=comm), steps=10)
            want = index_field(torch, dev, part[rank], dim, shift, cdt)
            checks["shift_%s_%s" % (lab, tag)] = all_ranks(torch.equal(y, want))
            del want
        del x, y
    # (c) redistribution t-slabs -> (z,t) blocks of a 32^3 x 64 x (4,3) x n=128 field (config 3), N > 1
    if world > 1:
        dim = [32, 32, 32, 64, 4, 3, 128]
        pa = sb.basic_partitioning("xyztscn", dim, [1, 1, 1, world, 1, 1, 1], "t", world, 1)
        pb = sb.basic_partitioning("xyztscn", dim, [1, 1, pz, pt, 1, 1, 1], "zt", world, 1)
        nl = int(np.prod(pa[rank, 1]))
        x = index_field(torch, dev, pa[rank], dim, [0] * 7, torch.complex64)
        y = torch.zeros(int(np.prod(pb[rank, 1])), device=dev, dtype=torch.complex64)
        record("redistribute_t_to_zt_c64", 2 * nl * 8,
               lambda: sb.copy(1, pa, 1, "xyztscn", [0] * 7, dim, dim, [x], None, gpu, pb, 1,
                               "xyztscn", [0] * 7, dim, [y], None, gpu, sb.FastToSlow, sb.Copy,
                               comm=comm), steps=10)
        want = index_field(torch, dev, pb[rank], dim, [0] * 7, torch.complex64)
        checks["redistribute_t_to_zt_c64"] = all_ranks(torch.equal(y, want))
        out["redistribute_t_to_zt_c64"]["bytes_per_gpu"] = 2 * nl * 8
        out["redistribute_t_to_zt_c64"]["off_device_fraction"] = {2: 0.5, 4: 0.75, 8: 0.875}.get(world)
        del x, y, want
    return out


if __name__ == "__main__":
    sys.exit(main())
