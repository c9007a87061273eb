// Block-sparse (BSR) operator times a multi-vector: the kernel descriptor and the per-row body.
//
// One launch applies the nonzero blocks of one operator component to a gathered input whose layout
// is "columns fastest, then the domain labels of the component's halo box": the element (domain
// point q, column c) of the gathered input is at q * ncols + c.  The body is written for a team of
// `nt` threads that meet at `sync()` (a warp or a CTA on the device, one thread on the host: the CPU
// emulation, tests/cxx/bsr_kernel_emul.cpp, runs this very function).  Every output element is the
// sum over the row's blocks in `jj` order, and inside a block over the domain index in order, with
// one fused multiply-add per term in the accumulation type Acc<T>; that sequence does not depend on
// the team, the column chunk or the piece size, so results are bit-identical however the operator,
// x and y are partitioned.
// Reference counterpart: bsr_krylov (bsr.h:2516), which calls cuSPARSE bsrmm or a batched gemm.
#pragma once
#include "../../include/superbblas_b200.h"
#include "contract_scalar.hpp"
#include <cstdint>

/// One launch: block rows [0, nrows) of an operator component, or those listed in rows[0, nlist)
struct sbk_bsr_desc {
    int64_t nrows;            ///< block rows of the component
    const int64_t *rowptr;    ///< nrows + 1 prefix sums of ii (device memory)
    const int64_t *goff;      ///< per nonzero block: gathered-input point of its first domain element
    int bi, bd;               ///< vol(blockim), vol(blockdom)
    int im_fast;              ///< element (i, j) of a block at i + j * bi, else at j + i * bd
    int ncols;                ///< points of the column labels
    int nd;                   ///< domain labels, fastest first (the in-block domain index j)
    int dsize[SBK_MAX_DIMS];  ///< blockdom
    int64_t dstride[SBK_MAX_DIMS]; ///< point strides of the halo box
    int ni;                   ///< image labels, fastest first (block row r and in-block index i)
    int iblocks[SBK_MAX_DIMS], isize[SBK_MAX_DIMS]; ///< blocks of the component, blockim
    int64_t istride[SBK_MAX_DIMS]; ///< stride in the output
    int nc;                   ///< column labels, fastest first (column index c)
    int csize[SBK_MAX_DIMS];
    int64_t cstride[SBK_MAX_DIMS]; ///< stride in the output
    const int64_t *rows;      ///< optional (device memory): the block rows of the launch, else [0, nrows)
    int64_t nlist;            ///< entries of rows
};

/// The Kronecker part of a launch of a create_kron_bsr operator: the u-th block of every row is
/// K_u (ki x kd) ⊗ B (bi x bd).  Along each label at most one of the block and the Kronecker extent
/// exceeds 1; `isize` / `dsize` of sbk_bsr_desc hold the block extents, these the Kronecker ones, and
/// the in-block coordinate along a label is (block index) * ksize + (Kronecker index).
struct sbk_kron_desc {
    int ki, kd;                   ///< vol(kronim), vol(krondom)
    int u;                        ///< blocks per row (and factors)
    int iksize[SBK_MAX_DIMS];     ///< kronim, parallel to isize
    int dksize[SBK_MAX_DIMS];     ///< krondom, parallel to dsize
};

namespace sbb {
    namespace bsrk {

        template <typename T> using AccT = typename Acc<T>::type;

        /// Output offset of element i of block row r (both linearised fastest label first)
        SBB_HD int64_t image_offset(const sbk_bsr_desc &d, int64_t r, int i) {
            int64_t o = 0;
            for (int k = 0; k < d.ni; ++k) {
                const int64_t b = r % d.iblocks[k];
                r /= d.iblocks[k];
                const int e = i % d.isize[k];
                i /= d.isize[k];
                o += (b * d.isize[k] + e) * d.istride[k];
            }
            return o;
        }

        /// Output offset of column c
        SBB_HD int64_t column_offset(const sbk_bsr_desc &d, int c) {
            int64_t o = 0;
            for (int k = 0; k < d.nc; ++k) {
                o += (int64_t)(c % d.csize[k]) * d.cstride[k];
                c /= d.csize[k];
            }
            return o;
        }

        /// Gathered-input point of the in-block domain index j, relative to the block's first point
        SBB_HD int64_t domain_point(const sbk_bsr_desc &d, int j) {
            int64_t o = 0;
            for (int k = 0; k < d.nd; ++k) {
                o += (int64_t)(j % d.dsize[k]) * d.dstride[k];
                j /= d.dsize[k];
            }
            return o;
        }

        /// A team of one thread (the host emulation)
        struct SerialTeam {
            int t = 0, nt = 1;
            void sync() const {}
        };

        /// y[r, :, c0 : c0 + m] = alpha * sum_blocks A x + beta * y for block row r.  Thread t owns the
        /// outputs o = t + k * nt (k < MAXO, o < bi * m; i = o % bi, c = o / bi).  The blocks stream
        /// through the team's scratch in pieces of kd domain indices: `as` holds bi x kd elements
        /// (i fastest), `xs` kd x m; `xo` holds domain_point of every in-block domain index.
        template <int MAXO, typename T, typename Team>
        SBB_HD void row_body(const sbk_bsr_desc &d, int64_t r, int c0, int m, int kd, const T *v, const T *x,
                             T *y, AccT<T> alpha, AccT<T> beta, T *as, T *xs, const int64_t *xo, const Team &tm) {
            AccT<T> acc[MAXO];
#pragma unroll
            for (int k = 0; k < MAXO; ++k) set_zero(acc[k]);
            const int bi = d.bi, bd = d.bd, no = bi * m;
            const int64_t bvol = (int64_t)bi * bd, b1 = d.rowptr[r + 1];
            for (int64_t b = d.rowptr[r]; b < b1; ++b) {
                const T *blk = v + b * bvol;
                const int64_t g = d.goff[b] * d.ncols + c0;
                for (int j0 = 0; j0 < bd; j0 += kd) {
                    const int nk = bd - j0 < kd ? bd - j0 : kd;
                    tm.sync(); // the previous piece has been used by every thread
                    for (int e = tm.t; e < bi * nk; e += tm.nt) {
                        if (d.im_fast) { // the piece is one contiguous run of v
                            const int i = e % bi, j = e / bi;
                            as[i + j * bi] = blk[(int64_t)(j0 + j) * bi + i];
                        } else {
                            const int j = e % nk, i = e / nk;
                            as[i + j * bi] = blk[(int64_t)i * bd + j0 + j];
                        }
                    }
                    for (int e = tm.t; e < nk * m; e += tm.nt) {
                        const int j = e / m, c = e % m;
                        xs[e] = x[g + xo[j0 + j] * d.ncols + c];
                    }
                    tm.sync();
#pragma unroll
                    for (int k = 0; k < MAXO; ++k) {
                        const int o = tm.t + k * tm.nt;
                        if (o < no) {
                            const int i = o % bi, c = o / bi;
                            for (int j = 0; j < nk; ++j) fma_acc(acc[k], widen(as[i + j * bi]), widen(xs[j * m + c]));
                        }
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < MAXO; ++k) {
                const int o = tm.t + k * tm.nt;
                if (o < no) {
                    const int i = o % bi, c = o / bi;
                    epilogue(y, image_offset(d, r, i) + column_offset(d, c0 + c), acc[k], alpha, beta);
                }
            }
        }

        /// Output offset of the element (Kronecker index ik, block index ib) of block row r
        SBB_HD int64_t kron_image_offset(const sbk_bsr_desc &d, const sbk_kron_desc &kr, int64_t r, int ik,
                                         int ib) {
            int64_t o = 0;
            for (int k = 0; k < d.ni; ++k) {
                const int64_t b = r % d.iblocks[k];
                r /= d.iblocks[k];
                const int e = ib % d.isize[k], f = ik % kr.iksize[k];
                ib /= d.isize[k], ik /= kr.iksize[k];
                o += (b * d.isize[k] * kr.iksize[k] + (int64_t)e * kr.iksize[k] + f) * d.istride[k];
            }
            return o;
        }

        /// Gathered-input point of the domain element (Kronecker index jk, block index jb), relative to
        /// the block's first point
        SBB_HD int64_t kron_domain_point(const sbk_bsr_desc &d, const sbk_kron_desc &kr, int jk, int jb) {
            int64_t o = 0;
            for (int k = 0; k < d.nd; ++k) {
                const int e = jb % d.dsize[k], f = jk % kr.dksize[k];
                jb /= d.dsize[k], jk /= kr.dksize[k];
                o += (int64_t)(e * kr.dksize[k] + f) * d.dstride[k];
            }
            return o;
        }

        /// Element (i, j) of an m x n matrix stored i-fast (i + j * m) or j-fast (j + i * n)
        template <typename T> SBB_HD T elem(const T *a, int im_fast, int m, int n, int i, int j) {
            return im_fast ? a[i + (int64_t)j * m] : a[j + (int64_t)i * n];
        }

        /// y[r, :, c0 : c0 + m] = alpha * sum_u (K_u ⊗ B_{r,u}) x + beta * y for block row r of a
        /// Kronecker operator.  Thread t owns the outputs o = t + k * nt (k < MAXO, o < ki * bi * m;
        /// ib = o % bi, ik = o / bi % ki, c = o / (bi * ki)).  The row's blocks go through the team's
        /// scratch `nu` at a time: `bs` holds their B (as in v), `xs` their input slabs
        /// ([u][jk][jb][c]), `ts` (in Acc<T>, shared because lanes with different ik read it)
        /// t_u[jk, ib, c] = sum_jb B_u[ib, jb] x[jk, jb, c] ([u][jk][ib][c]).  `ks` holds the U factors
        /// (as in kronv) and `xo` kron_domain_point of every (jk, jb) at jb + jk * bd.  Every output is
        /// sum_u sum_jk K_u[ik, jk] t_u[jk, ib, c], in that order, one fused multiply-add per term.
        template <int MAXO, typename T, typename Team>
        SBB_HD void kron_row_body(const sbk_bsr_desc &d, const sbk_kron_desc &kr, int64_t r, int c0, int m, int nu,
                                  const T *v, const T *ks, const T *x, T *y, AccT<T> alpha, AccT<T> beta, T *bs,
                                  T *xs, AccT<T> *ts, const int64_t *xo, const Team &tm) {
            AccT<T> acc[MAXO];
#pragma unroll
            for (int k = 0; k < MAXO; ++k) set_zero(acc[k]);
            const int bi = d.bi, bd = d.bd, ki = kr.ki, kd = kr.kd, U = kr.u, no = ki * bi * m;
            const int64_t bvol = (int64_t)bi * bd, kvol = (int64_t)ki * kd, b0 = d.rowptr[r];
            // per output: its row of K (offset of K[ik, 0]) and its point of t (t[0, ib, c])
            int kofs[MAXO], tofs[MAXO], nown = 0;
#pragma unroll
            for (int k = 0; k < MAXO; ++k) {
                const int o = tm.t + k * tm.nt;
                const int ib = o % bi, ik = o / bi % ki, c = o / (bi * ki);
                kofs[k] = d.im_fast ? ik : ik * kd, tofs[k] = ib * m + c;
                if (o < no) nown = k + 1;
            }
            for (int u0 = 0; u0 < U; u0 += nu) {
                const int nb = U - u0 < nu ? U - u0 : nu;
                tm.sync(); // the previous blocks have been used by every thread
                for (int64_t e = tm.t; e < nb * bvol; e += tm.nt) bs[e] = v[(b0 + u0) * bvol + e];
                for (int e = tm.t; e < nb * kd * bd * m; e += tm.nt) {
                    const int c = e % m, j = e / m % (kd * bd), u = e / (m * kd * bd);
                    xs[e] = x[(d.goff[b0 + u0 + u] + xo[j]) * d.ncols + c0 + c];
                }
                tm.sync();
                for (int e = tm.t; e < nb * kd * bi * m; e += tm.nt) {
                    const int c = e % m, ib = e / m % bi, jk = e / (m * bi) % kd, u = e / (m * bi * kd);
                    const T *blk = bs + u * bvol, *xu = xs + ((int64_t)u * kd + jk) * bd * m;
                    AccT<T> t;
                    set_zero(t);
                    for (int jb = 0; jb < bd; ++jb)
                        fma_acc(t, widen(elem(blk, d.im_fast, bi, bd, ib, jb)), widen(xu[jb * m + c]));
                    ts[e] = t;
                }
                tm.sync();
                for (int u = 0; u < nb; ++u) {
                    const T *K = ks + (u0 + u) * kvol;
                    for (int jk = 0; jk < kd; ++jk) {
                        const T *Kj = K + (d.im_fast ? jk * ki : jk);
                        const AccT<T> *tj = ts + ((int64_t)u * kd + jk) * bi * m;
#pragma unroll
                        for (int k = 0; k < MAXO; ++k)
                            if (k < nown) fma_acc(acc[k], widen(Kj[kofs[k]]), tj[tofs[k]]);
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < MAXO; ++k) {
                const int o = tm.t + k * tm.nt;
                if (o < no) {
                    const int ib = o % bi, ik = o / bi % ki, c = o / (bi * ki);
                    epilogue(y, kron_image_offset(d, kr, r, ik, ib) + column_offset(d, c0 + c), acc[k], alpha, beta);
                }
            }
        }

    } // namespace bsrk
} // namespace sbb
