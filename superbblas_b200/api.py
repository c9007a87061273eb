"""Python mirror of the reference's public C++ API for the tensor hot path, over the C ABI of
include/superbblas_b200.h.  Names, argument order and error behaviour follow
/root/reference/include/superbblas/dist.h (copy :3583, contraction :3701, basic_partitioning :3393
and :3477, partitioning_distributed_procs :3318, make_hole :3802) and platform.h (Context :757,
createCpuContext/createGpuContext :783-816, getGpuDevicesCount :824); errors surface as RuntimeError
with the reference's messages.

Tensor components are passed as a list with one entry per local component: a torch tensor (CUDA or
CPU), a numpy array (host) or a `(pointer, dtype)` tuple.  All compute happens in CUDA kernels; host
arrays are staged through the GPU by the library."""
import ctypes
import numpy as np

from ._lib import lib, check

SlowToFast, FastToSlow = 0, 1
Copy, Add = 0, 1
CPU, CUDA = 0, 1

F32, F64, C64, C128, I32 = 0, 1, 2, 3, 4
_NP2DT = {np.dtype(np.float32): F32, np.dtype(np.float64): F64, np.dtype(np.complex64): C64,
          np.dtype(np.complex128): C128, np.dtype(np.int32): I32}
DT_SIZE = {F32: 4, F64: 8, C64: 8, C128: 16, I32: 4}


class Context(ctypes.Structure):
    """Same layout as the reference's `Context {enum platform plat; int device;}`."""
    _fields_ = [("plat", ctypes.c_int), ("device", ctypes.c_int)]

    def __repr__(self):
        return "Context(%s, %d)" % ("CPU" if self.plat == CPU else "CUDA", self.device)


def createCpuContext():
    return Context(CPU, -1)


def createGpuContext(device=0):
    return Context(CUDA, device)


createCudaContext = createGpuContext


def getGpuDevicesCount():
    n = ctypes.c_int(0)
    check(lib().sbb_device_count(ctypes.byref(n)))
    return n.value


def sync(ctx):
    check(lib().sbb_sync(ctypes.byref(ctx)))


def syncLegacyStream(ctx):
    check(lib().sbb_sync_legacy_stream(ctypes.byref(ctx)))


def clearCaches():
    check(lib().sbb_clear_caches())


def clearHandles():
    check(lib().sbb_clear_handles())


def get_stream(device=0):
    s = ctypes.c_void_p()
    check(lib().sbb_get_stream(device, ctypes.byref(s)))
    return s.value or 0


def launch_count(reset=False):
    n = ctypes.c_longlong(0)
    check(lib().sbb_launch_count(int(reset), ctypes.byref(n)))
    return n.value


def profile_enable(on=True):
    check(lib().sbb_profile_enable(int(on)))


def profile_read(kernel):
    """-> (total milliseconds, launches) of the named kernel since the last read"""
    ms, n = ctypes.c_double(0), ctypes.c_longlong(0)
    check(lib().sbb_profile_read(kernel.encode(), ctypes.byref(ms), ctypes.byref(n)))
    return ms.value, n.value


def trackTime(on=True):
    """What the environment variable SB_TRACK_TIME does in the reference (runtime_features.h)."""
    check(lib().sbb_track_time(int(on)))


def resetTimings():
    check(lib().sbb_reset_timings())


def _text(fn, *args):
    """Call a C entry point that writes text into (buf, buflen, needed), growing buf as it asks."""
    size = 1 << 16
    while True:
        buf = ctypes.create_string_buffer(size)
        needed = ctypes.c_size_t(0)
        rc = fn(*args, buf, ctypes.c_size_t(size), ctypes.byref(needed))
        if rc == 2:
            size = needed.value + 16
            continue
        check(rc)
        return buf.value.decode()


def _report(what):
    return _text(lib().sbb_report, what)


def reportTimings():
    """reportTimings (performance.h:365) as text; empty unless tracking is on."""
    return _report(0)


def reportCacheUsage():
    """reportCacheUsage (performance.h:443) as text."""
    return _report(1)


def timings():
    """The timing report as {name: {cpu_time, gpu_time, calls, flops, bytes}}."""
    out = {}
    for line in reportTimings().splitlines()[2:]:
        name, rest = line.split(" : ", 1)
        w = rest.replace("(", " ").replace(")", " ").split()
        out[name] = dict(cpu_time=float(w[0]), gpu_time=float(w[w.index("gpu_time:") + 1]),
                         calls=int(w[w.index("calls:") + 1]), flops=float(w[w.index("flops:") + 1]),
                         bytes=float(w[w.index("bytes:") + 1]))
    return out


def liveAllocations():
    """-> (blocks, bytes) handed out by the library's allocator and not returned; what
    checkForMemoryLeaks (performance.h:494) looks at."""
    n, b = ctypes.c_longlong(0), ctypes.c_longlong(0)
    check(lib().sbb_live_allocations(ctypes.byref(n), ctypes.byref(b)))
    return n.value, b.value


# --- communicator -------------------------------------------------------------------------------

class Comm:
    """One NCCL rank bound to one GPU; stands where the reference takes an MPI_Comm."""

    def __init__(self, handle, rank, nranks):
        self.handle, self.rank, self.nranks = handle, rank, nranks

    def destroy(self):
        if self.handle:
            check(lib().sbb_comm_destroy(self.handle))
            self.handle = None


class Request:
    """Work that has been begun (reference: Request, dist.h:54): a copy, a bsr_krylov, a dense solver or the
    create of a block-sparse operator.  wait() completes it; progress() takes one step (sbb_request_progress)."""

    def __init__(self, handle, keep):
        self.handle, self._keep = handle, keep  # the marshalled arrays live as long as the request

    def wait(self):
        h, self.handle, self._keep = self.handle, None, None
        if h:
            check(lib().sbb_request_wait(h))

    def progress(self):
        """Complete the exchange in flight and begin the next one; True once the request is complete.
        Loopback ranks call it on every rank, round by round, until all are done."""
        if not self.handle:
            return True
        done = ctypes.c_int(0)
        try:
            check(lib().sbb_request_progress(self.handle, ctypes.byref(done)))
        except Exception:
            h, self.handle, self._keep = self.handle, None, None
            lib().sbb_request_wait(h)  # released; the error is the one raised
            raise
        if done.value:
            self.handle, self._keep = None, None
        return bool(done.value)


def wait(request):
    request.wait()


def comm_create_local(nranks, devices=None):
    """`nranks` loopback communicators living in this process (tests of the cross-rank path on fewer
    GPUs than ranks); rank r works on devices[r] (default: all on device 0)."""
    devices = list(devices) if devices is not None else [0] * nranks
    dv = (ctypes.c_int * nranks)(*devices)
    hs = (ctypes.c_void_p * nranks)()
    check(lib().sbb_comm_create_local(nranks, dv, hs))
    return [Comm(ctypes.c_void_p(hs[r]), r, nranks) for r in range(nranks)]


def comm_unique_id():
    buf = ctypes.create_string_buffer(128)
    check(lib().sbb_comm_unique_id(buf))
    return buf.raw


def comm_create(unique_id, nranks, rank, device):
    h = ctypes.c_void_p()
    check(lib().sbb_comm_create(ctypes.c_char_p(unique_id), nranks, rank, device, ctypes.byref(h)))
    return Comm(h, rank, nranks)


# --- helpers -------------------------------------------------------------------------------------

def _ia(x, n=None):
    a = np.ascontiguousarray(np.asarray(x, dtype=np.int32).reshape(-1))
    if n is not None and a.size != n:
        raise RuntimeError("coordinate of the wrong length")
    return a


def _ip(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int))


_IV_CACHE = {}


def _iv(x, n=None):
    """A coordinate (or a flattened partition) as a ctypes int array.  Built directly from the Python
    sequence (numpy's `.ctypes.data_as` costs ~5 us per argument, which dominated small calls) and
    remembered by value: the arrays are only ever read, by us and by the library."""
    key = x.tobytes() if isinstance(x, np.ndarray) and x.dtype == np.int32 else None
    if key is None and type(x) in (list, tuple):
        try:
            key = tuple(x)
            hash(key)
        except TypeError:         # nested lists / arrays inside
            key = None
    c = _IV_CACHE.get(key) if key is not None else None
    if c is None:
        if not isinstance(x, np.ndarray):
            try:
                c = (ctypes.c_int * len(x))(*x)
            except (TypeError, ValueError):   # nested or non-integer input: numpy flattens / rejects it
                x = np.asarray(x)
        if isinstance(x, np.ndarray):
            a = np.ascontiguousarray(x, dtype=np.int32)
            c = (ctypes.c_int * a.size).from_buffer_copy(a)
        if key is not None:
            if len(_IV_CACHE) >= 4096:
                _IV_CACHE.clear()
            _IV_CACHE[key] = c
    if n is not None and len(c) != n:
        raise RuntimeError("coordinate of the wrong length")
    return c


def _partition(p, nparts, nd):
    """int[nparts][2][nd]; a partition of the wrong length is the reference's "wtf" error
    (check_components, dist.h:709-716)."""
    a = _iv(p)
    if len(a) != nparts * 2 * nd:
        raise RuntimeError("wtf")
    return a


def _co(co):
    return {0: 0, 1: 1, "SlowToFast": 0, "FastToSlow": 1}[co]


_TORCH = None      # (torch.Tensor, {torch dtype: code}), filled on first use: torch is optional here


def _torch_types():
    global _TORCH
    if _TORCH is None:
        import torch
        _TORCH = (torch.Tensor, {torch.float32: F32, torch.float64: F64, torch.complex64: C64,
                                 torch.complex128: C128, torch.int32: I32})
    return _TORCH


def _component(x):
    """-> (pointer, dtype code)"""
    if isinstance(x, np.ndarray):
        if not x.flags.c_contiguous:
            raise RuntimeError("component arrays must be contiguous")
        return (x.__array_interface__["data"][0] if x.size else 0), _NP2DT[x.dtype]
    if isinstance(x, tuple):
        return int(x[0]), int(x[1])
    tensor, codes = _torch_types()
    if isinstance(x, tensor):
        if not x.is_contiguous():
            raise RuntimeError("component tensors must be contiguous")
        return (x.data_ptr() if x.numel() else 0), codes[x.dtype]
    raise TypeError("unsupported component type %r" % type(x))


def _components(v):
    """-> (void*[ncomponents], dtype code, keepalive)"""
    n = len(v)
    if n == 1:
        p, dt = _component(v[0])
        return (ctypes.c_void_p * 1)(p or None), dt, v
    ptrs = (ctypes.c_void_p * max(n, 1))()
    dts = set()
    for i, x in enumerate(v):
        p, dt = _component(x)
        ptrs[i] = p or None
        dts.add(dt)
    if len(dts) > 1:
        raise RuntimeError("components of a tensor must share one element type")
    return ptrs, (dts.pop() if dts else F64), v


def _contexts(ctx, n):
    if isinstance(ctx, Context):
        ctx = [ctx] * n
    if n == 0:
        return (Context * 1)()
    return (Context * n)(*ctx[:n])


def _scalar(x):
    x = complex(x)
    return (ctypes.c_double * 2)(x.real, x.imag)


def _order(o):
    return o.encode() if o is not None else None


def _check_order(o, n, name):
    if len(o) != n:
        raise RuntimeError("The length of the order should match the template argument; argument "
                           "`%s` should have length %d" % (name, n))


# --- partitions ----------------------------------------------------------------------------------

def partitioning_distributed_procs(order, dim, dist_labels, nprocs):
    n = len(dim)
    out = np.zeros(n, dtype=np.int32)
    check(lib().sbb_partitioning_distributed_procs(n, _order(order), _ip(_ia(dim)),
                                                   _order(dist_labels), int(nprocs), _ip(out)))
    return [int(x) for x in out]


def basic_partitioning(*args, **kw):
    """basic_partitioning(order, dim, procs, dist_labels, nprocs=-1, ncomponents=1)  (dist.h:3393)
    basic_partitioning(dim, procs, nprocs=-1, replicate=False, ext_power=None)      (dist.h:3477)
    Returns an int32 array [nparts][2][N]."""
    if len(args) and (args[0] is None or isinstance(args[0], str)):
        order, dim, procs, dist_labels = args[:4]
        nprocs = args[4] if len(args) > 4 else kw.get("nprocs", -1)
        ncomponents = args[5] if len(args) > 5 else kw.get("ncomponents", 1)
        n = len(dim)
        P = int(np.prod(procs)) if nprocs < 0 else nprocs
        out = np.zeros((P * ncomponents, 2, n), dtype=np.int32)
        check(lib().sbb_basic_partitioning(n, _order(order), _ip(_ia(dim, n)), _ip(_ia(procs, n)),
                                           _order(dist_labels), int(nprocs), int(ncomponents),
                                           _ip(out)))
        return out
    dim, procs = args[:2]
    nprocs = args[2] if len(args) > 2 else kw.get("nprocs", -1)
    replicate = args[3] if len(args) > 3 else kw.get("replicate", False)
    ext_power = args[4] if len(args) > 4 else kw.get("ext_power", None)
    n = len(dim)
    P = int(np.prod(procs)) if nprocs < 0 else nprocs
    out = np.zeros((P, 2, n), dtype=np.int32)
    ext = _ia(ext_power if ext_power is not None else [0] * n, n)
    check(lib().sbb_basic_partitioning_ext(n, _ip(_ia(dim, n)), _ip(_ia(procs, n)), int(nprocs),
                                           int(bool(replicate)), _ip(ext), _ip(out)))
    return out


def make_hole(frm, size, hole_from, hole_size, dim):
    n = len(dim)
    cap = 4 ** n + 1
    out = np.zeros((cap, 2, n), dtype=np.int32)
    nout = ctypes.c_int(0)
    check(lib().sbb_make_hole(n, _ip(_ia(frm, n)), _ip(_ia(size, n)), _ip(_ia(hole_from, n)),
                              _ip(_ia(hole_size, n)), _ip(_ia(dim, n)), _ip(out), cap,
                              ctypes.byref(nout)))
    return [(list(map(int, out[i, 0])), list(map(int, out[i, 1]))) for i in range(nout.value)]


# --- copy ----------------------------------------------------------------------------------------

def copy(alpha, p0, ncomponents0, o0, from0, size0, dim0, v0, mask0, ctx0,
         p1, ncomponents1, o1, from1, dim1, v1, mask1, ctx1, co, copyadd, comm=None, request=False):
    """superbblas::copy (dist.h:3583; with `comm` the MPI overload dist.h:3534).  With request=True
    the copy is only begun and a Request is returned (the reference's `Request *request` argument)."""
    n0, n1 = len(o0), len(o1)
    pv0, dt0, k0 = _components(v0)
    pv1, dt1, k1 = _components(v1)
    if len(v0) != ncomponents0 or len(v1) != ncomponents1:
        raise RuntimeError("wtf")
    # masks (MaskType = float32, one per component, laid out like the component; nonzero = active)
    pm0 = pm1 = None
    if mask0 is not None:
        if len(mask0) != ncomponents0:
            raise RuntimeError("wtf")
        pm0, mdt, km0 = _components(mask0)
        if mdt != F32:
            raise RuntimeError("masks must be float32 (MaskType)")
    if mask1 is not None:
        if len(mask1) != ncomponents1:
            raise RuntimeError("wtf")
        pm1, mdt, km1 = _components(mask1)
        if mdt != F32:
            raise RuntimeError("masks must be float32 (MaskType)")
    nr = comm.nranks if comm else 1
    a = [_partition(p0, nr * ncomponents0, n0), _iv(from0, n0), _iv(size0, n0), _iv(dim0, n0),
         _partition(p1, nr * ncomponents1, n1), _iv(from1, n1), _iv(dim1, n1)]
    call = (dt0, dt1, _scalar(alpha), n0, a[0], ncomponents0, _order(o0),
            a[1], a[2], a[3], pv0, pm0, _contexts(ctx0, ncomponents0),
            n1, a[4], ncomponents1, _order(o1), a[5], a[6], pv1, pm1,
            _contexts(ctx1, ncomponents1), comm.handle if comm else None, _co(co), int(copyadd))
    return _begun("copy", call, request, (call, a, k0, k1, v0, v1, mask0, mask1))


def local_copy(alpha, o0, from0, size0, dim0, v0, mask0, ctx0, o1, from1, dim1, v1, mask1, ctx1,
               co, copyadd):
    """local_copy (signature kept from the reference's tests/local.cpp:97): one component each."""
    n0, n1 = len(o0), len(o1)
    p0 = np.array([[[0] * n0, list(dim0)]], dtype=np.int32)
    p1 = np.array([[[0] * n1, list(dim1)]], dtype=np.int32)
    copy(alpha, p0, 1, o0, from0, size0, dim0, [v0], None if mask0 is None else [mask0], [ctx0],
         p1, 1, o1, from1, dim1, [v1], None if mask1 is None else [mask1], [ctx1], co, copyadd)


def _copy_ops(lines, phases=None):
    """(ops, wire) from the lines of CopyPlan::describe(); see copy_plan."""
    ops, wire = [], {}
    for line in lines:
        w = line.split()
        if not w:
            continue
        if w[0] == "wire":
            wire[int(w[2])] = (int(w[4]), int(w[6]))
            if phases is not None and int(w[4]) > 0:
                phases[int(w[2])] = int(w[8])
        elif w[0] == "op":
            i_size, i_ss, i_ds, i_rot = (w.index("size"), w.index("sstride"), w.index("dstride"),
                                         w.index("rot"))
            ops.append(dict(kind=w[1], src=int(w[3]), dst=int(w[5]), peer=int(w[7]),
                            soff=int(w[9]), doff=int(w[11]),
                            size=[int(x) for x in w[i_size + 1:i_ss]],
                            sstride=[int(x) for x in w[i_ss + 1:i_ds]],
                            dstride=[int(x) for x in w[i_ds + 1:i_rot]], rot=int(w[i_rot + 1])))
    return ops, wire


def copy_plan(elem_size1, p0, ncomponents0, o0, from0, size0, dim0, p1, ncomponents1, o1, from1,
              dim1, nranks, rank, co, copyadd, alpha_is_zero=False, phases=None):
    """The list of strided-box operations `copy` would run on `rank` (host only, no GPU needed).
    Returns (ops, wire) with ops = list of dicts, wire = {peer: (send_elems, recv_elems)}; if
    `phases` is a dict it receives {peer: phase of my message to that peer}."""
    n0, n1 = len(o0), len(o1)
    a = [_partition(p0, nranks * ncomponents0, n0), _iv(from0, n0), _iv(size0, n0), _iv(dim0, n0),
         _partition(p1, nranks * ncomponents1, n1), _iv(from1, n1), _iv(dim1, n1)]
    text = _text(lib().sbb_copy_plan_describe,
                 elem_size1, n0, a[0], ncomponents0, _order(o0), a[1], a[2], a[3],
                 n1, a[4], ncomponents1, _order(o1), a[5], a[6], nranks, rank, _co(co),
                 int(copyadd), int(alpha_is_zero))
    return _copy_ops(text.splitlines(), phases)


# --- contraction ---------------------------------------------------------------------------------

def contraction(alpha, p0, from0, size0, dim0, ncomponents0, o0, conj0, v0, ctx0,
                p1, from1, size1, dim1, ncomponents1, o1, conj1, v1, ctx1,
                beta, pr, fromr, sizer, dimr, ncomponentsr, o_r, vr, ctxr, co, comm=None):
    """superbblas::contraction (dist.h:3701; with `comm` the MPI overload dist.h:3628)."""
    n0, n1, nr = len(o0), len(o1), len(o_r)
    pv0, dt0, k0 = _components(v0)
    pv1, dt1, k1 = _components(v1)
    pvr, dtr, kr = _components(vr)
    if not (dt0 == dt1 == dtr):
        raise RuntimeError("contraction: operands must share one element type")
    if dt0 == I32:
        raise RuntimeError("contraction: unsupported type")
    R = comm.nranks if comm else 1
    a = [_partition(p0, R * ncomponents0, n0), _iv(from0, n0), _iv(size0, n0), _iv(dim0, n0),
         _partition(p1, R * ncomponents1, n1), _iv(from1, n1), _iv(size1, n1), _iv(dim1, n1),
         _partition(pr, R * ncomponentsr, nr), _iv(fromr, nr), _iv(sizer, nr), _iv(dimr, nr)]
    check(lib().sbb_contraction(
        dt0, _scalar(alpha), n0, a[0], a[1], a[2], a[3], ncomponents0,
        _order(o0), int(bool(conj0)), pv0, _contexts(ctx0, ncomponents0), n1, a[4], a[5],
        a[6], a[7], ncomponents1, _order(o1), int(bool(conj1)), pv1,
        _contexts(ctx1, ncomponents1), _scalar(beta), nr, a[8], a[9], a[10],
        a[11], ncomponentsr, _order(o_r), pvr, _contexts(ctxr, ncomponentsr),
        comm.handle if comm else None, _co(co)))


def contraction_plan(dtype, alpha, p0, from0, size0, dim0, ncomponents0, o0, conj0,
                     p1, from1, size1, dim1, ncomponents1, o1, conj1,
                     beta, pr, fromr, sizer, dimr, ncomponentsr, o_r, co, nranks, rank):
    """What `contraction` would do on `rank` of `nranks` (host only, no GPU needed), as a dict:
    the flags (nothing, big0, direct, repartition, reduction, slots); `items`, one per kernel launch,
    each with big / small / out = (component, element offset; component -1 = slot `slot`), the slot
    sizes small_elems / out_elems and the dims T, M, N, K as (size, stride in v0, in v1, in vr);
    `beta`, the boxes (comp, off, size, stride) scaled in place; and `repartition_plan` /
    `reduction_plan`, the (ops, wire) of those copies as copy_plan returns them, or None."""
    n0, n1, nr = len(o0), len(o1), len(o_r)
    a = [_partition(p0, nranks * ncomponents0, n0), _iv(from0, n0), _iv(size0, n0), _iv(dim0, n0),
         _partition(p1, nranks * ncomponents1, n1), _iv(from1, n1), _iv(size1, n1), _iv(dim1, n1),
         _partition(pr, nranks * ncomponentsr, nr), _iv(fromr, nr), _iv(sizer, nr), _iv(dimr, nr)]
    text = _text(lib().sbb_contraction_plan_describe,
                 int(dtype), _scalar(alpha), n0, a[0], a[1], a[2], a[3], ncomponents0, _order(o0),
                 int(bool(conj0)), n1, a[4], a[5], a[6], a[7], ncomponents1, _order(o1),
                 int(bool(conj1)), _scalar(beta), nr, a[8], a[9], a[10], a[11], ncomponentsr,
                 _order(o_r), nranks, rank, _co(co))
    sections, cur = {"": []}, ""
    for line in text.splitlines():
        if line in ("repartition", "reduction"):
            cur = line
            sections[cur] = []
        else:
            sections[cur].append(line)
    head = sections[""][0].split()
    plan = {head[i]: int(head[i + 1]) for i in range(1, len(head), 2)}
    plan["items"], plan["beta"] = [], []
    for line in sections[""][1:]:
        w = line.split()
        if w[0] == "item":
            it = dict(big=(int(w[2]), int(w[3])), small=(int(w[5]), int(w[6])), small_elems=int(w[7]),
                      out=(int(w[9]), int(w[10])), out_elems=int(w[11]), slot=int(w[13]))
            dims = {}
            for x in w[14:]:
                if x in ("T", "M", "N", "K"):
                    cur = dims[x] = []
                else:
                    cur.append(int(x))
            for g, v in dims.items():
                it[g] = [tuple(v[i:i + 4]) for i in range(0, len(v), 4)]
            plan["items"].append(it)
        elif w[0] == "beta":
            i_st = w.index("stride")
            plan["beta"].append(dict(comp=int(w[2]), off=int(w[4]),
                                     size=[int(x) for x in w[6:i_st]],
                                     stride=[int(x) for x in w[i_st + 1:]]))
    for name in ("repartition", "reduction"):
        plan[name + "_plan"] = _copy_ops(sections[name]) if name in sections else None
    return plan


# --- batched dense solvers ---------------------------------------------------------------------------

CHOLESKY, INVERSION, TRSM, GESM, EIGH = 0, 1, 2, 3, 4


def _dense_type(dt, name):
    if dt == I32:
        raise RuntimeError("%s: unsupported type" % name)
    return dt


def _begun(name, args, request, keep, result=None):
    """sbb_<name>(*args) -> `result`; or with request=True sbb_<name>_begin -> a Request that keeps `keep`
    alive, paired as (result, Request) when `result` is given"""
    if not request:
        check(getattr(lib(), "sbb_" + name)(*args))
        return result
    h = ctypes.c_void_p()
    check(getattr(lib(), "sbb_%s_begin" % name)(*args, ctypes.byref(h)))
    return Request(h, keep) if result is None else (result, Request(h, keep))


def _square(name, p, ncomponents, o, v, orows, ocols, ctx, co, comm, request):
    pv, dt, keep = _components(v)
    if len(v) != ncomponents:
        raise RuntimeError("wtf")
    R = comm.nranks if comm else 1
    args = (_dense_type(dt, name), len(o), _partition(p, R * ncomponents, len(o)), ncomponents, _order(o), pv,
            _order(orows), _order(ocols), _contexts(ctx, ncomponents), comm.handle if comm else None, _co(co))
    return _begun(name, args, request, (args, (keep, v)))


def cholesky(p, ncomponents, o, v, orows, ocols, ctx, co, comm=None, request=False):
    """superbblas::cholesky (dense.h): every matrix A (rows `orows`, columns `ocols`, one per batch
    coordinate) is replaced in place by U with A = U^H U, zeros below the diagonal.  With request=True
    the call returns a Request after its first step (sbb_cholesky_begin); A is defined once the request
    is complete."""
    return _square("cholesky", p, ncomponents, o, v, orows, ocols, ctx, co, comm, request)


def inversion(p, ncomponents, o, v, orows, ocols, ctx, co, comm=None, request=False):
    """superbblas::inversion (dense.h): every matrix A is replaced in place by its inverse.  request: as
    cholesky."""
    return _square("inversion", p, ncomponents, o, v, orows, ocols, ctx, co, comm, request)


def _solve(name, alpha, pc, ncomponentsc, oc, orows, ocols, vc, ctxc, px, ncomponentsx, ox, vx, ctxx,
           py, ncomponentsy, oy, vy, ctxy, co, comm, request):
    pvc, dtc, kc = _components(vc)
    pvx, dtx, kx = _components(vx)
    pvy, dty, ky = _components(vy)
    if len(vc) != ncomponentsc or len(vx) != ncomponentsx or len(vy) != ncomponentsy:
        raise RuntimeError("wtf")
    if not (dtc == dtx == dty):
        raise RuntimeError("%s: operands must share one element type" % name)
    R = comm.nranks if comm else 1
    args = (_dense_type(dtc, name), _scalar(alpha), len(oc), _partition(pc, R * ncomponentsc, len(oc)),
            ncomponentsc, _order(oc), _order(orows), _order(ocols), pvc, _contexts(ctxc, ncomponentsc),
            len(ox), _partition(px, R * ncomponentsx, len(ox)), ncomponentsx, _order(ox), pvx,
            _contexts(ctxx, ncomponentsx), len(oy), _partition(py, R * ncomponentsy, len(oy)), ncomponentsy,
            _order(oy), pvy, _contexts(ctxy, ncomponentsy), comm.handle if comm else None, _co(co))
    return _begun(name, args, request, (args, (kc, kx, ky, vc, vx, vy)))


def trsm(alpha, pc, ncomponentsc, oc, orows, ocols, vc, ctxc, px, ncomponentsx, ox, vx, ctxx,
         py, ncomponentsy, oy, vy, ctxy, co, comm=None, request=False):
    """superbblas::trsm (dense.h): solve with the upper triangle U of every matrix.  If x carries the
    `orows` labels, y (carrying `ocols`) gets U y = alpha x; if x carries `ocols`, y (carrying `orows`)
    gets y U = alpha x.  With request=True the call returns a Request after its first step
    (sbb_trsm_begin); y is defined once the request is complete."""
    return _solve("trsm", alpha, pc, ncomponentsc, oc, orows, ocols, vc, ctxc, px, ncomponentsx,
                  ox, vx, ctxx, py, ncomponentsy, oy, vy, ctxy, co, comm, request)


def gesm(alpha, pc, ncomponentsc, oc, orows, ocols, vc, ctxc, px, ncomponentsx, ox, vx, ctxx,
         py, ncomponentsy, oy, vy, ctxy, co, comm=None, request=False):
    """superbblas::gesm (dense.h): as trsm with a general matrix, by LU with partial pivoting."""
    return _solve("gesm", alpha, pc, ncomponentsc, oc, orows, ocols, vc, ctxc, px, ncomponentsx,
                  ox, vx, ctxx, py, ncomponentsy, oy, vy, ctxy, co, comm, request)


def eigh(p, ncomponents, o, v, orows, ocols, ctx, pw, ncomponentsw, ow, vw, ctxw, co, comm=None):
    """Eigen-decomposition of every Hermitian matrix A (rows `orows`, columns `ocols`, one per batch
    coordinate; ours, not in the reference): A is replaced in place by V with A = V diag(w) V^H, column j
    the unit eigenvector of w[j], and w (batch labels and `ocols`, element type the real type of A's, its
    own partition `pw`) gets the eigenvalues in ascending order.  Reads the upper triangle of A and the
    real part of its diagonal."""
    pv, dt, keep = _components(v)
    pvw, dtw, keepw = _components(vw)
    if len(v) != ncomponents or len(vw) != ncomponentsw:
        raise RuntimeError("wtf")
    dt = _dense_type(dt, "eigh")
    if len(vw) and dtw != {F32: F32, C64: F32, F64: F64, C128: F64}[dt]:
        raise RuntimeError("eigh: w must have the real type of the matrix's element type")
    R = comm.nranks if comm else 1
    check(lib().sbb_eigh(dt, len(o), _partition(p, R * ncomponents, len(o)), ncomponents, _order(o), pv,
                         _order(orows), _order(ocols), _contexts(ctx, ncomponents), len(ow),
                         _partition(pw, R * ncomponentsw, len(ow)), ncomponentsw, _order(ow), pvw,
                         _contexts(ctxw, ncomponentsw), comm.handle if comm else None, _co(co)))


def _dense_step(line):
    """One `step` line of the blocked tier -> dict: `step` (gather, scatter, zero, factor, panel, solve or
    update), `refs` [(buffer, element offset)] with buffers A, X, Y (the call's operands) and W, V (the
    workspaces), the integers n, rhs, left, conj0, rows, cols where given, the label groups T, M, N, K of
    an update as (size, stride in v0, in v1, in vr) and the `kernel` text of the launch it makes"""
    head, _, kernel = line.partition(" kernel ")
    w = head.split()
    st, i, g = dict(step=w[1], refs=[], kernel=kernel or None), 2, None
    while i < len(w):
        if w[i] in ("A", "X", "Y", "W", "V"):
            st["refs"].append((w[i], int(w[i + 1])))
            i += 2
        elif w[i] in ("T", "M", "N", "K"):
            g = st[w[i]] = []
            i += 1
        elif g is not None:
            g.append(int(w[i]))
            i += 1
        else:
            st[w[i]] = int(w[i + 1])
            i += 2
    for k in ("T", "M", "N", "K"):
        if k in st:
            st[k] = [tuple(st[k][j:j + 4]) for j in range(0, len(st[k]), 4)]
    return st


def dense_plan(op, dtype, pc, ncomponentsc, oc, orows, ocols, co, nranks, rank, alpha=1,
               px=None, ncomponentsx=0, ox="", py=None, ncomponentsy=0, oy=""):
    """What a dense call (op: CHOLESKY, INVERSION, TRSM, GESM or EIGH, which takes W as py / ncomponentsy
    / oy) would do on `rank` of `nranks` (host
    only, no GPU needed), as a dict: the flags (nothing, gather_a, gather_x, slots); `items`, one per
    kernel launch, each with the output component `comp`, a / x / y = (component, element offset,
    elements; component -1 = slot `slot` of the gather, or for y a temporary), `left`, `n`, the label
    groups R, C, B, H as (size, stride in A, in X, in Y), the `kernel` text, for a matrix over the
    shared-memory limit (the blocked tier of cholesky and trsm) `steps`, one dict per launch as
    _dense_step gives, for EIGH `writes` ("a", "w" or "aw"; y is then W), and, when the output is
    written from a temporary, `back` = (soff, size, sstride, dstride); and `gather_a_plan` /
    `gather_x_plan`, the (ops, wire) of the gathers as copy_plan returns them, or None."""
    nc, nx, ny = len(oc), len(ox), len(oy)
    empty = (ctypes.c_int * 1)()
    text = _text(lib().sbb_dense_plan_describe, int(op), int(dtype), _scalar(alpha), nc,
                 _partition(pc, nranks * ncomponentsc, nc), ncomponentsc, _order(oc), _order(orows),
                 _order(ocols), nx, _partition(px, nranks * ncomponentsx, nx) if px is not None else empty,
                 ncomponentsx, _order(ox), ny,
                 _partition(py, nranks * ncomponentsy, ny) if py is not None else empty, ncomponentsy,
                 _order(oy), nranks, rank, _co(co))
    sections, cur = {"": []}, ""
    for line in text.splitlines():
        if line in ("gather_a", "gather_x"):
            cur = line
            sections[cur] = []
        else:
            sections[cur].append(line)
    head = sections[""][0].split()
    plan = {head[i]: int(head[i + 1]) for i in range(2, len(head), 2)}
    plan["op"], plan["items"] = head[1], []
    for line in sections[""][1:]:
        w = line.split()
        if w[0] == "item":
            it = dict(comp=int(w[2]), a=tuple(map(int, w[4:7])), x=tuple(map(int, w[8:11])),
                      y=tuple(map(int, w[12:15])), slot=int(w[16]), left=int(w[18]), n=int(w[20]), back=None)
            groups, g = {}, None
            if "writes" in w:
                it["writes"] = w[-1]
                w = w[:-2]
            for t in w[21:]:
                if t in ("R", "C", "B", "H"):
                    g = groups[t] = []
                else:
                    g.append(int(t))
            for k, v in groups.items():
                it[k] = [tuple(v[i:i + 4]) for i in range(0, len(v), 4)]
            plan["items"].append(it)
        elif w[0] == "kernel":
            plan["items"][-1]["kernel"] = line[len("kernel "):]
        elif w[0] == "step":
            plan["items"][-1].setdefault("steps", []).append(_dense_step(line))
        elif w[0] == "back":
            i_sz, i_ss, i_ds = w.index("size"), w.index("sstride"), w.index("dstride")
            plan["items"][-1]["back"] = dict(soff=int(w[4]), size=[int(x) for x in w[i_sz + 1:i_ss]],
                                             sstride=[int(x) for x in w[i_ss + 1:i_ds]],
                                             dstride=[int(x) for x in w[i_ds + 1:]])
    for name in ("gather_a", "gather_x"):
        plan[name + "_plan"] = _copy_ops(sections[name]) if name in sections else None
    return plan


def dense_steps(op, dtype, pc, ncomponentsc, oc, orows, ocols, co, nranks, rank, alpha=1,
                px=None, ncomponentsx=0, ox="", py=None, ncomponentsy=0, oy=""):
    """The steps of the same dense call as a request (arguments of dense_plan; host only) as a dict:
    `steps` (the begin and one per gather: the same on every rank), `exchanges` (the gathers) and `item_steps`,
    for every item of dense_plan in its order the step that queues its kernels; None when the call has
    nothing to do."""
    nc, nx, ny = len(oc), len(ox), len(oy)
    empty = (ctypes.c_int * 1)()
    text = _text(lib().sbb_dense_steps_describe, int(op), int(dtype), _scalar(alpha), nc,
                 _partition(pc, nranks * ncomponentsc, nc), ncomponentsc, _order(oc), _order(orows),
                 _order(ocols), nx, _partition(px, nranks * ncomponentsx, nx) if px is not None else empty,
                 ncomponentsx, _order(ox), ny,
                 _partition(py, nranks * ncomponentsy, ny) if py is not None else empty, ncomponentsy,
                 _order(oy), nranks, rank, _co(co))
    lines = [line.split() for line in text.splitlines()]
    if not lines:
        return None
    return dict(steps=int(lines[0][1]), exchanges=int(lines[0][3]), item_steps=[int(w[3]) for w in lines[1:]])


# --- block-sparse operators ------------------------------------------------------------------------

class BSR:
    """An operator made by create_bsr.  It references the caller's `v` until destroy()."""

    def __init__(self, handle, keep):
        self.handle, self._keep = handle, keep

    def destroy(self):
        if self.handle:
            check(lib().sbb_destroy_bsr(self.handle))
            self.handle, self._keep = None, None


def _int_arrays(a):
    """-> (int*[n], keepalive) for a list of per-component int arrays (torch, numpy or None)"""
    ptrs = (ctypes.c_void_p * max(len(a), 1))()
    keep = []
    for i, x in enumerate(a):
        if x is None:
            continue
        if isinstance(x, np.ndarray) or isinstance(x, (list, tuple)):
            x = np.ascontiguousarray(np.asarray(x, dtype=np.int32).reshape(-1))
            ptrs[i] = x.ctypes.data or None if x.size else None
        else:
            p, dt = _component(x)
            if dt != I32:
                raise RuntimeError("create_bsr: ii and jj must be int32")
            ptrs[i] = p or None
        keep.append(x)
    return ptrs, keep


def create_bsr(pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, blockImFast, ii, jj, v, ctx, co,
               comm=None, request=False):
    """superbblas::create_bsr (bsr.h:2286): the operator whose component c has, per block row, ii[c]
    nonzero blocks with domain origins jj[c] (nd ints each) and values v[c]; semantics in
    include/superbblas_b200.h.  Returns a BSR handle; call .destroy() when done.  With request=True
    returns (handle, Request): the handle is usable once the request is complete."""
    return _create(False, pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, None, None, blockImFast, ii, jj, v,
                   None, ctx, co, comm, request)


def create_kron_bsr(pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, kronim, krondom, blockImFast, ii, jj,
                    v, kronv, ctx, co, comm=None, request=False):
    """create_kron_bsr: the operator of create_bsr whose u-th block of every row is kronv[c][u] ⊗ v's
    block (kronim / krondom: extents of the Kronecker factor per label); semantics in
    include/superbblas_b200.h.  Returns a BSR handle for bsr_krylov; call .destroy() when done.  With
    request=True returns (handle, Request), as create_bsr."""
    return _create(True, pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, kronim, krondom, blockImFast, ii,
                   jj, v, kronv, ctx, co, comm, request)


def _create(kron, pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, kronim, krondom, blockImFast, ii, jj, v,
            kronv, ctx, co, comm, request):
    """create_bsr, or create_kron_bsr when `kron`"""
    ni, nd = len(dimi), len(dimd)
    pv, dt, kv = _components(v)
    if kron:
        pk, dtk, kk = _components(kronv)
    if any(len(a) != ncomponents for a in (v, ii, jj, kronv if kron else v)):
        raise RuntimeError("wtf")
    if kron and dtk != dt:
        raise RuntimeError("create_kron_bsr: v and kronv must share one element type")
    R = comm.nranks if comm else 1
    pii, kii = _int_arrays(ii)
    pjj, kjj = _int_arrays(jj)
    h = ctypes.c_void_p()
    kshape, kvalues = ([_iv(kronim, ni), _iv(krondom, nd)], [pk]) if kron else ([], [])
    args = [dt, ni, _partition(pim, R * ncomponents, ni), _iv(dimi, ni), nd, _partition(pdom, R * ncomponents, nd),
            _iv(dimd, nd), ncomponents, _iv(blockim, ni), _iv(blockdom, nd), *kshape, int(bool(blockImFast)), pii,
            pjj, pv, *kvalues, _contexts(ctx, ncomponents), comm.handle if comm else None, _co(co), ctypes.byref(h)]
    op = BSR(h, (v, kv, kronv, kk) if kron else (v, kv))
    op.dtype, op.ni, op.nd = dt, ni, nd
    return _begun("create_kron_bsr" if kron else "create_bsr", args, request, None, op)


def _power(c):
    return ctypes.c_char(c.encode() if c else b"\0")


def bsr_krylov(alpha, bsr, oim, odom, px, ncomponentsx, ox, fromx, sizex, dimx, vx, ctxx,
               beta, py, oy, fromy, sizey, dimy, power_label, vy, ctxy, co, comm=None, ncomponentsy=None,
               request=False):
    """superbblas::bsr_krylov (bsr.h:2516): y_p = beta y_p + alpha A u_p, u_0 = x, u_p = y_{p-1}.
    `power_label` is a one-letter label of y or None.  With request=True the call returns a Request
    after its first step (sbb_bsr_krylov_begin); y is defined once the request is complete."""
    pvx, dtx, kx = _components(vx)
    pvy, dty, ky = _components(vy)
    ncomponentsy = len(vy) if ncomponentsy is None else ncomponentsy
    if len(vx) != ncomponentsx or len(vy) != ncomponentsy:
        raise RuntimeError("wtf")
    if dtx != dty:
        raise RuntimeError("bsr_krylov: x and y must share one element type")
    if dtx == I32:
        raise RuntimeError("bsr_krylov: unsupported type")
    nx, ny = len(ox), len(oy)
    R = comm.nranks if comm else 1
    call = (dtx, _scalar(alpha), bsr.handle, _order(oim), _order(odom), nx, _partition(px, R * ncomponentsx, nx),
            ncomponentsx, _order(ox), _iv(fromx, nx), _iv(sizex, nx), _iv(dimx, nx), pvx,
            _contexts(ctxx, ncomponentsx), _scalar(beta), ny, _partition(py, R * ncomponentsy, ny), ncomponentsy,
            _order(oy), _iv(fromy, ny), _iv(sizey, ny), _iv(dimy, ny), _power(power_label), pvy,
            _contexts(ctxy, ncomponentsy), comm.handle if comm else None, _co(co))
    return _begun("bsr_krylov", call, request, (call, kx, ky, vx, vy, bsr))


def bsr_plan(dtype, pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, blockImFast, ii_all, jj_all,
             oim, odom, px, ncomponentsx, ox, fromx, sizex, dimx, py, ncomponentsy, oy, fromy, sizey, dimy,
             power_label, co, nranks, rank, alpha=1, beta=0):
    """What bsr_krylov would do on `rank` of `nranks` (host only, no GPU needed) with the operator built
    from every rank's ii / jj (flat int arrays, concatenated in [rank][component] order), as a dict: the
    flags (nothing, direct, powers, slots); `items`, one per kernel launch, each with `comp`, y = (component,
    offset at power 0, stride of the power label, temporary elements; component -1: a temporary), the
    gathered-input elements `x`, `nnz`, `rows`, `bi`, `bd`, `imfast`, `ncols`, the dims D (size, point
    stride), I (blocks, blockim, stride), C (size, stride), `rowptr`, `goff` and the `kernel` text; and
    `gather` (x or y_{p-1} -> halo slots), `fill` (y_p -> temporaries, when beta != 0) and `back`
    (temporaries -> y_p): {power: (ops, wire)} of those copies."""
    return _bsr_plan_dict(_bsr_describe(False, dtype, pim, dimi, pdom, dimd, ncomponents, blockim, blockdom,
                                        None, None, blockImFast, ii_all, jj_all, oim, odom, px, ncomponentsx, ox,
                                        fromx, sizex, dimx, py, ncomponentsy, oy, fromy, sizey, dimy, power_label,
                                        co, nranks, rank, alpha, beta))


def kron_bsr_plan(dtype, pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, kronim, krondom, blockImFast,
                  ii_all, jj_all, oim, odom, px, ncomponentsx, ox, fromx, sizex, dimx, py, ncomponentsy, oy, fromy,
                  sizey, dimy, power_label, co, nranks, rank, alpha=1, beta=0):
    """bsr_plan for the operator create_kron_bsr would build: the same dict, and every item also has
    `ki`, `kd`, `u` and the Kronecker extents `IK` / `DK` of its I / D dims"""
    return _bsr_plan_dict(_bsr_describe(False, dtype, pim, dimi, pdom, dimd, ncomponents, blockim, blockdom,
                                        kronim, krondom, blockImFast, ii_all, jj_all, oim, odom, px, ncomponentsx,
                                        ox, fromx, sizex, dimx, py, ncomponentsy, oy, fromy, sizey, dimy,
                                        power_label, co, nranks, rank, alpha, beta))


def bsr_split(dtype, pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, blockImFast, ii_all, jj_all,
              oim, odom, px, ncomponentsx, ox, fromx, sizex, dimx, py, ncomponentsy, oy, fromy, sizey, dimy,
              power_label, co, nranks, rank, alpha=1, beta=0, kronim=None, krondom=None):
    """The block rows of every kernel launch of bsr_plan (same arguments; kronim / krondom for the
    operator of create_kron_bsr), split as bsr_krylov with a request splits power 0: a list with one
    dict per launch, {comp, interior, boundary}.  Boundary rows read a point that the gather of x
    (bsr_plan(...)["gather"][0]) fills from another rank; interior rows do not.  Host only."""
    text = _bsr_describe(True, dtype, pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, kronim, krondom,
                         blockImFast, ii_all, jj_all, oim, odom, px, ncomponentsx, ox, fromx, sizex, dimx, py,
                         ncomponentsy, oy, fromy, sizey, dimy, power_label, co, nranks, rank, alpha, beta)
    out = []
    for line in text.splitlines():
        w = line.split()
        if w[0] == "split":
            out.append(dict(comp=int(w[2])))
        else:
            out[-1][w[0]] = [int(t) for t in w[1:]]
    return out


def _bsr_describe(split, dtype, pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, kronim, krondom,
                  blockImFast, ii_all, jj_all, oim, odom, px, ncomponentsx, ox, fromx, sizex, dimx, py,
                  ncomponentsy, oy, fromy, sizey, dimy, power_label, co, nranks, rank, alpha, beta):
    ni, nd, nx, ny = len(dimi), len(dimd), len(ox), len(oy)
    ii_a = np.ascontiguousarray(np.asarray(ii_all, dtype=np.int32).reshape(-1))
    jj_a = np.ascontiguousarray(np.asarray(jj_all, dtype=np.int32).reshape(-1))
    return _text(lib().sbb_bsr_plan_describe, int(dtype), ni, _partition(pim, nranks * ncomponents, ni),
                 _iv(dimi, ni), nd, _partition(pdom, nranks * ncomponents, nd), _iv(dimd, nd), ncomponents,
                 _iv(blockim, ni), _iv(blockdom, nd), None if kronim is None else _iv(kronim, ni),
                 None if krondom is None else _iv(krondom, nd), int(bool(blockImFast)), _ip(ii_a), _ip(jj_a),
                 _scalar(alpha), _order(oim), _order(odom), nx, _partition(px, nranks * ncomponentsx, nx),
                 ncomponentsx, _order(ox), _iv(fromx, nx), _iv(sizex, nx), _iv(dimx, nx), _scalar(beta), ny,
                 _partition(py, nranks * ncomponentsy, ny), ncomponentsy, _order(oy), _iv(fromy, ny),
                 _iv(sizey, ny), _iv(dimy, ny), _power(power_label), nranks, rank, _co(co), int(split))


def _bsr_plan_dict(text):
    sections, cur = {("", 0): []}, ("", 0)
    for line in text.splitlines():
        w = line.split()
        if len(w) == 2 and w[0] in ("gather", "fill", "back"):
            cur = (w[0], int(w[1]))
            sections[cur] = []
        else:
            sections[cur].append(line)
    head = sections[("", 0)][0].split()
    plan = {head[i]: int(head[i + 1]) for i in range(1, len(head), 2)}
    plan["items"] = []
    for line in sections[("", 0)][1:]:
        w = line.split()
        if w[0] == "item":
            it = dict(comp=int(w[2]), y=tuple(map(int, w[4:8])), x=int(w[9]))
            for key in ("nnz", "rows", "bi", "bd", "imfast", "ncols"):
                it[key] = int(w[w.index(key) + 1])
            i_d, i_i, i_c = w.index("D"), w.index("I"), w.index("C")
            d, i, c = ([int(t) for t in w[a + 1:b]] for a, b in ((i_d, i_i), (i_i, i_c), (i_c, len(w))))
            it["D"] = [tuple(d[k:k + 2]) for k in range(0, len(d), 2)]
            it["I"] = [tuple(i[k:k + 3]) for k in range(0, len(i), 3)]
            it["C"] = [tuple(c[k:k + 2]) for k in range(0, len(c), 2)]
            plan["items"].append(it)
        elif w[0] in ("rowptr", "goff"):
            plan["items"][-1][w[0]] = [int(t) for t in w[1:]]
        elif w[0] == "kron":
            it, i_ik, i_dk = plan["items"][-1], w.index("IK"), w.index("DK")
            for key in ("ki", "kd", "u"):
                it[key] = int(w[w.index(key) + 1])
            it["IK"], it["DK"] = [int(t) for t in w[i_ik + 1:i_dk]], [int(t) for t in w[i_dk + 1:]]
        elif w[0] == "kernel":
            plan["items"][-1]["kernel"] = line[len("kernel "):]
    for name in ("gather", "fill", "back"):
        plan[name] = {p: _copy_ops(v) for (n, p), v in sections.items() if n == name}
    return plan


def local_contraction(alpha, o0, dim0, conj0, v0, o1, dim1, conj1, v1, beta, o_r, dimr, vr, ctx,
                      co):
    """local_contraction (signature kept from the reference's tests/local.cpp:163)."""
    def part(dim):
        return np.array([[[0] * len(dim), list(dim)]], dtype=np.int32)
    contraction(alpha, part(dim0), [0] * len(dim0), dim0, dim0, 1, o0, conj0, [v0], [ctx],
                part(dim1), [0] * len(dim1), dim1, dim1, 1, o1, conj1, [v1], [ctx], beta,
                part(dimr), [0] * len(dimr), dimr, dimr, 1, o_r, [vr], [ctx], co)


# --- kernel level ----------------------------------------------------------------------------------

class BoxDesc(ctypes.Structure):
    _fields_ = [("nd", ctypes.c_int), ("size", ctypes.c_int * 16),
                ("sstride", ctypes.c_int64 * 16), ("dstride", ctypes.c_int64 * 16),
                ("soff", ctypes.c_int64), ("doff", ctypes.c_int64), ("rot", ctypes.c_int)]


def box_desc(size, sstride, dstride, soff=0, doff=0, rot=0):
    d = BoxDesc()
    d.rot = int(rot)
    d.nd = len(size)
    for k in range(len(size)):
        d.size[k], d.sstride[k], d.dstride[k] = int(size[k]), int(sstride[k]), int(dstride[k])
    d.soff, d.doff = int(soff), int(doff)
    return d


def permute_copy(desc, src, dst, alpha=1, add=False, device=0):
    ps, dts = _component(src) if src is not None else (0, None)
    pd, dtd = _component(dst)
    if dts is None:
        dts = dtd
    check(lib().sbk_permute_copy(ctypes.byref(desc), ctypes.c_void_p(ps), dts, ctypes.c_void_p(pd),
                                 dtd, _scalar(alpha), int(add), device, None))


class ContractDim(ctypes.Structure):
    _fields_ = [("size", ctypes.c_int), ("s0", ctypes.c_int64), ("s1", ctypes.c_int64),
                ("sr", ctypes.c_int64)]


class ContractDesc(ctypes.Structure):
    _fields_ = [("nT", ctypes.c_int), ("nM", ctypes.c_int), ("nN", ctypes.c_int), ("nK", ctypes.c_int),
                ("T", ContractDim * 8), ("M", ContractDim * 8), ("N", ContractDim * 8),
                ("K", ContractDim * 8), ("conj0", ctypes.c_int), ("conj1", ctypes.c_int)]


def contract_desc(T=(), M=(), N=(), K=(), conj0=False, conj1=False):
    """sbk_contract_desc from lists of (size, stride in v0, stride in v1, stride in vr) per label."""
    d = ContractDesc()
    for name, dims in (("T", T), ("M", M), ("N", N), ("K", K)):
        setattr(d, "n" + name, len(dims))
        for i, (size, s0, s1, sr) in enumerate(dims):
            getattr(d, name)[i] = ContractDim(int(size), int(s0), int(s1), int(sr))
    d.conj0, d.conj1 = int(bool(conj0)), int(bool(conj1))
    return d


def contract_describe(desc, dtype):
    """Which kernel `sbk_contract` would launch for this problem, and how (host only)."""
    buf = ctypes.create_string_buffer(512)
    check(lib().sbk_contract_describe(ctypes.byref(desc), int(dtype), buf, ctypes.c_size_t(512)))
    return buf.value.decode()


def permute_describe(desc, dtype_src, dtype_dst, alpha=1, add=False, src_ptr=0, dst_ptr=0):
    buf = ctypes.create_string_buffer(512)
    check(lib().sbk_permute_describe(ctypes.byref(desc), dtype_src, dtype_dst, _scalar(alpha),
                                     int(add), ctypes.c_void_p(src_ptr), ctypes.c_void_p(dst_ptr),
                                     buf, ctypes.c_size_t(512)))
    return buf.value.decode()
