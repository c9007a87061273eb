"""Test-side interpreter of the planner's strided-box operations on numpy arrays.  It exists so the
host logic (box geometry, message layout, ordering of additions) can be checked without a GPU; the
product never runs it — on the GPU the same operations are executed by the CUDA kernels."""
import numpy as np

from oracle import oracle as O


def _indices(size, stride, off, rot=0):
    """Linear indices of a strided box; `rot` rotates the first listed dimension (sbk_box_desc)."""
    idx = np.full((1,), off, dtype=np.int64)
    for k, (n, s) in enumerate(zip(size, stride)):
        i = np.arange(n, dtype=np.int64)
        if k == 0 and rot:
            i = (i + rot) % n
        idx = (idx[:, None] + (i * s)[None, :]).reshape(-1)
    return idx


def run_rank(ops, wire, rank, nranks, ncomp0, ncomp1, v0_local, v1_local, alpha, copyadd, T, Q,
             exchange, mask_a=None, mask_b=None):
    """Run the ops of one rank. `exchange(send: {peer: array}) -> {peer: array}` moves messages.
    mask_a / mask_b: optional float32 masks per local destination component (laid out like it): an
    element is written only where both are nonzero; zero-fills look at mask_b only (capi.cpp,
    sbb_copy; runtime.cpp, execute_copy)."""
    T, Q = np.dtype(T), np.dtype(Q)
    one = (np.real(alpha) == 1 and np.imag(alpha) == 0)
    # wire element type: Q, except T when adding with a type change (runtime.cpp, execute_copy)
    Wt = T if (copyadd == 1 and T != Q) else Q
    send = {r: np.zeros(w[0], dtype=Wt) for r, w in wire.items() if w[0] > 0}

    def transformed(x):
        if not one:
            x = O._scale(alpha, x, T)
        return x

    def keep(comp, idx, zero=False):
        k = np.ones(idx.size, dtype=bool)
        if mask_a is not None and not zero:
            k &= mask_a[comp][idx] != 0
        if mask_b is not None:
            k &= mask_b[comp][idx] != 0
        return k

    def store(dst, idx, x, XT, comp):
        k = keep(comp, idx)
        idx, x = idx[k], x[k]
        if copyadd == 0:
            dst[idx] = x.astype(dst.dtype)
        else:
            W = np.result_type(dst.dtype, XT)
            dst[idx] = (dst[idx].astype(W) + x.astype(W)).astype(dst.dtype)

    for op in ops:
        if op["kind"] == "pack":
            src = v0_local[op["src"] - rank * ncomp0]
            x = transformed(src[_indices(op["size"], op["sstride"], op["soff"])])
            send[op["peer"]][_indices(op["size"], op["dstride"], op["doff"])] = x.astype(Wt)
    recv = exchange(send)
    for r, w in wire.items():
        if w[1] > 0:
            assert recv[r].size == w[1], "message size mismatch"
    order = ops if copyadd == 1 else \
        [o for o in ops if o["kind"] in ("local", "zero")] + [o for o in ops if o["kind"] == "unpack"]
    for op in order:
        if op["kind"] == "local":
            src = v0_local[op["src"] - rank * ncomp0]
            dst = v1_local[op["dst"] - rank * ncomp1]
            x = transformed(src[_indices(op["size"], op["sstride"], op["soff"])])
            store(dst, _indices(op["size"], op["dstride"], op["doff"], op.get("rot", 0)), x, T,
                  op["dst"] - rank * ncomp1)
        elif op["kind"] == "unpack":
            dst = v1_local[op["dst"] - rank * ncomp1]
            x = recv[op["peer"]][_indices(op["size"], op["sstride"], op["soff"])]
            store(dst, _indices(op["size"], op["dstride"], op["doff"]), x, Wt,
                  op["dst"] - rank * ncomp1)
        elif op["kind"] == "zero":
            dst = v1_local[op["dst"] - rank * ncomp1]
            idx = _indices(op["size"], op["dstride"], op["doff"])
            dst[idx[keep(op["dst"] - rank * ncomp1, idx, zero=True)]] = 0


def run_ranks(plans, v0, v1, ncomp0, ncomp1, alpha, copyadd, T, Q):
    """Execute the plans of all ranks, one (ops, wire) per rank as api.copy_plan returns them.
    v0 / v1 hold the parts of all ranks, [rank][component] flattened; v1 is updated in place.
    Messages go through a mailbox: first every rank packs, then every rank unpacks."""
    nranks = len(plans)
    # consistency of the message layout between sender and receiver
    for r in range(nranks):
        for peer, (s, _) in plans[r][1].items():
            assert plans[peer][1].get(r, (0, 0))[1] == s
    mailbox = {}
    for phase in (0, 1):
        for r in range(nranks):
            ops, wire = plans[r]

            def exchange(send, r=r, wire=wire):
                if phase == 0:
                    for peer, buf in send.items():
                        mailbox[(r, peer)] = buf.copy()
                    raise StopIteration
                return {peer: mailbox[(peer, r)] for peer, w in wire.items() if w[1] > 0}
            try:
                run_rank(ops, wire, r, nranks, ncomp0, ncomp1, v0[r * ncomp0:(r + 1) * ncomp0],
                         v1[r * ncomp1:(r + 1) * ncomp1], alpha, copyadd, T, Q, exchange)
            except StopIteration:
                pass
