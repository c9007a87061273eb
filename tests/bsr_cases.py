"""Numpy oracle and case generators of the block-sparse operators (create_bsr / bsr_krylov).

An operator is given as the arrays create_bsr takes, per part of the image partition (in [rank]
[component] order): ii (blocks per block row, rows numbered over the part's lattice of blocks with the
CoorOrder), jj (nd ints per block: the domain origin, periodic) and v (vol(blockim) * vol(blockdom)
elements per block; element (i, j) at i + j * bi if blockImFast else j + i * bd, with i and j
linearised with the CoorOrder).  The oracle turns it into a scipy sparse matrix and applies it to
whole tensors indexed in their label order."""
import numpy as np

from tests.dense_cases import components, assemble, rel_err, TOL  # noqa: F401

FastToSlow, SlowToFast = 1, 0


def _unravel(n, shape, co):
    """Coordinates (len(shape) x n) of the linear indices 0..n-1 with the CoorOrder"""
    if len(shape) == 0:
        return np.zeros((0, n), dtype=np.int64)
    return np.array(np.unravel_index(np.arange(n), shape, order="F" if co == FastToSlow else "C"))


def block_rows(part, blockim):
    f, s = part
    if 0 in list(s):
        return 0
    return int(np.prod([s[k] // blockim[k] for k in range(len(blockim))]))


def rnd(rng, dtype, *shape):
    x = rng.standard_normal(shape)
    if np.dtype(dtype).kind == "c":
        x = x + 1j * rng.standard_normal(shape)
    return x.astype(dtype)


def random_operator(rng, pim, blockim, dimd, blockdom, dtype, max_blocks=3):
    """Random ii / jj / v per part: 0..max_blocks blocks per row (empty rows included), jj anywhere on
    the periodic lattice (multiples of blockdom, shifted by random multiples of dimd)"""
    nb = [dimd[k] // blockdom[k] for k in range(len(dimd))]
    ops = []
    for part in pim:
        rows = block_rows(part, blockim)
        ii = rng.integers(0, max_blocks + 1, size=rows).astype(np.int32)
        nnz = int(ii.sum())
        jj = np.array([[rng.integers(nb[k]) * blockdom[k] + dimd[k] * int(rng.integers(-1, 2))
                        for k in range(len(dimd))] for _ in range(nnz)], dtype=np.int32).reshape(nnz, len(dimd))
        v = rnd(rng, dtype, nnz * int(np.prod(blockim)) * int(np.prod(blockdom)))
        ops.append((ii, jj, v))
    return ops


def stencil_operator(rng, pim, dims, blockim, dtype, co):
    """Periodic nearest-neighbour (9-point) operator on a lattice whose first label is the dense block
    (blockim[0] == blockdom[0] == dims[0]) and the other four are the sites: every block row (a site)
    has its own block and the blocks of the sites +-1 along each of the four site labels"""
    ops = []
    for part in pim:
        f, s = part
        rows = block_rows(part, blockim)
        ii = np.full(rows, 9, dtype=np.int32)
        nb = [s[k] // blockim[k] for k in range(len(dims))]
        coords = _unravel(rows, nb, co)
        jj = []
        for r in range(rows):
            site = [f[k] + coords[k, r] * blockim[k] for k in range(len(dims))]
            jj.append(site)
            for mu in range(1, 5):
                for d in (1, -1):
                    n = list(site)
                    n[mu] = (n[mu] + d) % dims[mu]
                    jj.append(n)
        jj = np.array(jj, dtype=np.int32).reshape(-1, len(dims))
        v = rnd(rng, dtype, len(jj) * blockim[0] * blockim[0])
        ops.append((ii, jj, v))
    return ops


def operator_matrix(ops, pim, dimi, dimd, blockim, blockdom, im_fast, co):
    """The operator as a scipy sparse matrix: rows over the image labels, columns over the domain labels,
    each linearised like numpy's C order over the labels in oim / odom order"""
    import scipy.sparse as sp
    bi, bd = int(np.prod(blockim)), int(np.prod(blockdom))
    ic, jc = _unravel(bi, blockim, co), _unravel(bd, blockdom, co)
    rows_all, cols_all, vals = [], [], []
    for (ii, jj, v), part in zip(ops, pim):
        f, s = part
        rows = block_rows(part, blockim)
        if rows == 0 or int(ii.sum()) == 0:
            continue
        nb = [s[k] // blockim[k] for k in range(len(dimi))]
        rc = _unravel(rows, nb, co)
        rb = np.repeat(np.arange(rows), ii)                                   # block row of every block
        base = np.array([f[k] + rc[k, rb] * blockim[k] for k in range(len(dimi))])       # [ni, nnz]
        org = np.array([np.asarray(jj)[:, k] % dimd[k] for k in range(len(dimd))])      # [nd, nnz]
        img = base[:, :, None, None] + ic[:, None, :, None]                   # [ni, nnz, bi, 1]
        dom = org[:, :, None, None] + jc[:, None, None, :]                    # [nd, nnz, 1, bd]
        r = np.ravel_multi_index(tuple(np.broadcast_to(img[k], img.shape[1:3] + (bd,)) for k in range(len(dimi))),
                                 dimi) if len(dimi) else np.zeros((len(rb), bi, bd), np.int64)
        c = np.ravel_multi_index(tuple(np.broadcast_to(dom[k], (dom.shape[1], bi, bd)) for k in range(len(dimd))),
                                 dimd) if len(dimd) else np.zeros((len(rb), bi, bd), np.int64)
        m = v.reshape(-1, bd, bi).transpose(0, 2, 1) if im_fast else v.reshape(-1, bi, bd)
        rows_all.append(r.ravel()), cols_all.append(c.ravel()), vals.append(m.ravel())
    vi, vd = int(np.prod(dimi)), int(np.prod(dimd))
    if not vals:
        return sp.csr_matrix((vi, vd), dtype=np.complex128)
    return sp.coo_matrix((np.concatenate(vals).astype(np.complex128),
                          (np.concatenate(rows_all), np.concatenate(cols_all))), shape=(vi, vd)).tocsr()


def apply(a, oim, odom, x, ox, y, oy, alpha, beta, power=None, psize=1, fromy=None):
    """`a` from operator_matrix; y (whole, label order oy) after y_p = beta y_p + alpha A u_p, u_0 = x, u_p = y_{p-1}"""
    ni, nd = len(oim), len(odom)
    dimi = [y.shape[oy.index(c)] for c in oim]
    vd = a.shape[1]
    am = a
    cols = [c for c in ox if c not in odom]
    y = y.astype(np.complex128).copy()
    u = x.astype(np.complex128)
    ou = ox
    for p in range(psize):
        ut = np.transpose(u, [ou.index(c) for c in odom] + [ou.index(c) for c in cols])
        csh = ut.shape[nd:]
        r = np.asarray(am @ ut.reshape(vd, -1)).reshape(tuple(dimi) + csh)          # axes oim + cols
        oy_np = [c for c in oy if c != power]
        r = np.transpose(r, [(list(oim) + cols).index(c) for c in oy_np])
        sl = [slice(None)] * len(oy)
        if power:
            sl[oy.index(power)] = (fromy[oy.index(power)] + p) % y.shape[oy.index(power)]
        sl = tuple(sl)
        old = y[sl]
        y[sl] = alpha * r + (beta * old if beta != 0 else 0)
        if power:
            u = y[sl]
            ou = "".join(odom[oim.index(c)] if c in oim else c for c in oy_np)
    return y


def flat_arrays(ops):
    """ii and jj of every part concatenated, as bsr_plan takes them"""
    ii = np.concatenate([o[0] for o in ops]) if ops else np.zeros(0, np.int32)
    jj = np.concatenate([o[1].reshape(-1) for o in ops]) if ops else np.zeros(0, np.int32)
    return ii.astype(np.int32), jj.astype(np.int32)
