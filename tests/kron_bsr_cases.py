"""Numpy oracle and case generators of the Kronecker block-sparse operators (create_kron_bsr), in the
style of tests/bsr_cases.py.

A Kronecker operator is given as create_kron_bsr takes it, per part of the image partition: ii (U
blocks in every row), jj (nd ints per block: the domain origin of the effective block, periodic), v
(the B blocks, vol(blockim) * vol(blockdom) elements each) and kronv (U factors of vol(kronim) *
vol(krondom) elements).  `expand` turns every block into K_u ⊗ B, the block of the plain operator with
the effective extents blockim * kronim and blockdom * krondom, so tests/bsr_cases.py's oracle applies
to it, and create_bsr / bsr_plan can be given the same operator."""
import numpy as np

from tests import bsr_cases as B

FastToSlow, SlowToFast = B.FastToSlow, B.SlowToFast


def eff(block, kron):
    return [b * k for b, k in zip(block, kron)]


def random_kron_operator(rng, pim, blockim, dimd, blockdom, kronim, krondom, U, dtype, kronv=None):
    """U blocks in every row, jj anywhere on the periodic lattice (multiples of the effective block,
    shifted by random multiples of dimd); the same U factors for every part -> (ops, kronv)"""
    bd_eff = eff(blockdom, krondom)
    nb = [dimd[k] // bd_eff[k] for k in range(len(dimd))]
    ki, kd = int(np.prod(kronim)), int(np.prod(krondom))
    kronv = B.rnd(rng, dtype, U * ki * kd) if kronv is None else kronv
    ops = []
    for part in pim:
        rows = B.block_rows(part, eff(blockim, kronim))
        ii = np.full(rows, U, np.int32)
        nnz = rows * U
        jj = np.array([[rng.integers(nb[k]) * bd_eff[k] + dimd[k] * int(rng.integers(-1, 2))
                        for k in range(len(dimd))] for _ in range(nnz)], dtype=np.int32).reshape(nnz, len(dimd))
        v = B.rnd(rng, dtype, nnz * int(np.prod(blockim)) * int(np.prod(blockdom)))
        ops.append((ii, jj, v))
    return ops, kronv


def _eff_index(block, kron, co):
    """[kron index, block index] -> index of the effective block, each linearised with the CoorOrder"""
    nb, nk = int(np.prod(block)), int(np.prod(kron))
    cb, ck = B._unravel(nb, block, co), B._unravel(nk, kron, co)
    if len(block) == 0:
        return np.zeros((nk, nb), np.int64)
    coords = tuple(ck[k][:, None] + cb[k][None, :] * kron[k] for k in range(len(block)))
    return np.ravel_multi_index(coords, eff(block, kron), order="F" if co == FastToSlow else "C")


def mat(a, im_fast, m, n):
    """An m x n matrix stored i-fast (i + j * m) or j-fast (j + i * n)"""
    return a.reshape(n, m).T if im_fast else a.reshape(m, n)


def expand(ops, kronv, blockim, blockdom, kronim, krondom, im_fast, co):
    """The plain operator's arrays: every block K_u ⊗ B_{r,u} over the effective extents"""
    bi, bd, ki, kd = (int(np.prod(x)) for x in (blockim, blockdom, kronim, krondom))
    iI, jI = _eff_index(blockim, kronim, co), _eff_index(blockdom, krondom, co)
    out = []
    for ii, jj, v in ops:
        vals = []
        for b in range(len(jj)):
            u = b % int(ii[0])                       # every row has ii[0] blocks
            K = mat(kronv[u * ki * kd:(u + 1) * ki * kd], im_fast, ki, kd)
            Bm = mat(v[b * bi * bd:(b + 1) * bi * bd], im_fast, bi, bd)
            E = np.zeros((ki * bi, kd * bd), v.dtype)
            E[iI.reshape(-1)[:, None], jI.reshape(-1)[None, :]] = np.kron(K, Bm)   # rows ik * bi + ib
            vals.append((E.T if im_fast else E).reshape(-1))
        out.append((ii, jj, np.concatenate(vals) if vals else np.zeros(0, v.dtype)))
    return out


def oracle_matrix(ops, kronv, pim, dimi, dimd, blockim, blockdom, kronim, krondom, im_fast, co):
    return B.operator_matrix(expand(ops, kronv, blockim, blockdom, kronim, krondom, im_fast, co), pim, dimi, dimd,
                             eff(blockim, kronim), eff(blockdom, krondom), im_fast, co)


def kron_stencil(rng, pim, dims, blockim, kronim, U_order, dtype, co):
    """Periodic nine-point operator on a lattice whose first two labels (spin, colour) are the effective
    block and the other four are the sites: every row has, in the order of U_order (0: the site itself,
    (mu, d): the site + d along site label mu), one block of the neighbour; the U factors are shared"""
    bim = eff(blockim, kronim)
    ops = []
    for f, s in pim:
        rows = B.block_rows((f, s), bim)
        nb = [s[k] // bim[k] for k in range(len(dims))]
        coords = B._unravel(rows, nb, co)
        jj = []
        for r in range(rows):
            site = [f[k] + coords[k, r] * bim[k] for k in range(len(dims))]
            for e in U_order:
                n = list(site)
                if e:
                    mu, d = e
                    n[mu] = (n[mu] + d) % dims[mu]
                jj.append(n)
        jj = np.array(jj, dtype=np.int32).reshape(-1, len(dims))
        ii = np.full(rows, len(U_order), np.int32)
        v = B.rnd(rng, dtype, len(jj) * int(np.prod(blockim)) ** 2)
        ops.append((ii, jj, v))
    return ops


NINE_POINT = [0] + [(mu, d) for mu in range(2, 6) for d in (1, -1)]
