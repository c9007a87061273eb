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
    """A copy that has been begun (reference: Request, dist.h:54); wait() completes it."""

    def __init__(self, handle, keep):
        self.handle, self._keep = handle, keep  # the marshalled arrays live as long as the request

    def wait(self):
        h, self.handle, self._keep = self.handle, None, None
        if h:
            check(lib().sbb_request_wait(h))


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
    if not request:
        check(lib().sbb_copy(*call))
        return None
    h = ctypes.c_void_p()
    check(lib().sbb_copy_begin(*call, ctypes.byref(h)))
    return Request(h, (call, a, k0, k1, v0, v1, mask0, mask1))


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
