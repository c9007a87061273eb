// Batched dense solvers (cholesky, inversion, trsm, gesm) and the Hermitian eigensolver (eigh) on
// matrices addressed through label strides: the kernel descriptor and the per-matrix bodies.
//
// The bodies work on one n x n matrix stored row-major in (shared) memory and are written for a team
// of `nt` threads that meet at `sync()`: a warp or a CTA on the device, one thread on the host (the
// CPU emulation, tests/cxx/dense_kernel_emul.cpp, runs these very functions).  Every element is
// computed by a fixed sequence of operations, whatever the team size, so results are deterministic.
// Reference counterparts: cholesky / trsm / gesm / inversion (dense.h:1019-1290), which call cuSOLVER
// potrfBatched and cuBLAS trsmBatched / getrfBatched / getrsBatched / getriBatched.
#pragma once
#include "../../include/superbblas_b200.h"
#include "contract_scalar.hpp"
#include <cstdint>

/// One label of a dense-solver operand: extent and strides (in elements) in the matrix A and in the
/// right-hand sides X and the solutions Y; 0 where the tensor does not have the label
struct sbk_dense_dim {
    int size;
    int64_t sa, sx, sy;
};

/// One launch: for every batch entry b, the n x n matrix A[b](r, c) with r, c linearised through the
/// row and column groups (first listed label fastest).  trsm / gesm: the right-hand side j of X[b] is
/// a vector over the rows (left: A Y = alpha X) or over the columns (right: Y A = alpha X), and Y[b]
/// one over the other set.  eigh: Y is the eigenvalue tensor W (strides `sy` of the batch and column
/// labels, element type the real type of T; none when y is null), and with `vectors` the eigenvectors
/// overwrite A.
struct sbk_dense_desc {
    int op; ///< sbb_dense_op
    int n, left, vectors;
    int nrows, ncols, nbatch, nrhs;
    sbk_dense_dim rows[SBK_MAX_GROUP_DIMS], cols[SBK_MAX_GROUP_DIMS];
    sbk_dense_dim batch[SBK_MAX_GROUP_DIMS], rhs[SBK_MAX_GROUP_DIMS];
};

namespace sbb {
    namespace densek {

        /// One matrix of T must fit in one CTA's shared memory
        constexpr int64_t MAX_MATRIX_BYTES = 200 * 1024;

        /// cholesky and trsm of a larger matrix run the blocked tier (kernels_dense.cu) in blocks of
        /// BLOCK_N, through workspaces whose boxes take one dimension per label
        constexpr int BLOCK_N = 64;
        inline bool fits_cta(int64_t n, int es) { return n * n * es <= MAX_MATRIX_BYTES; }

        /// eigh keeps the matrix and its eigenvectors in shared memory: 2 n^2 sizeof(T) bytes
        inline bool fits_eigh(int64_t n, int es) { return 2 * n * n * es <= MAX_MATRIX_BYTES; }

        /// Internal op of the blocked tier (not an sbb_dense_op, outside their range): U^H y = x for
        /// every right-hand side over the rows, with U the upper triangle of the matrix
        constexpr int PANEL = 16;

        template <typename T> struct Real { using type = T; };
        template <> struct Real<float2> { using type = float; };
        template <> struct Real<double2> { using type = double; };

        SBB_HD float re(float x) { return x; }
        SBB_HD double re(double x) { return x; }
        SBB_HD float re(float2 x) { return x.x; }
        SBB_HD double re(double2 x) { return x.x; }
        SBB_HD float abs2(float x) { return x * x; }
        SBB_HD double abs2(double x) { return x * x; }
        SBB_HD float abs2(float2 x) { return x.x * x.x + x.y * x.y; }
        SBB_HD double abs2(double2 x) { return x.x * x.x + x.y * x.y; }
        SBB_HD float neg(float x) { return -x; }
        SBB_HD double neg(double x) { return -x; }
        SBB_HD float2 neg(float2 x) { return float2{-x.x, -x.y}; }
        SBB_HD double2 neg(double2 x) { return double2{-x.x, -x.y}; }
        SBB_HD float scale(float x, float r) { return x * r; }
        SBB_HD double scale(double x, double r) { return x * r; }
        SBB_HD float2 scale(float2 x, float r) { return float2{x.x * r, x.y * r}; }
        SBB_HD double2 scale(double2 x, double r) { return double2{x.x * r, x.y * r}; }
        /// 1/x; infinite or NaN for x == 0, which is how a singular matrix shows in the result
        SBB_HD float recip(float x) { return 1.0f / x; }
        SBB_HD double recip(double x) { return 1.0 / x; }
        SBB_HD float2 recip(float2 x) {
            const float d = abs2(x);
            return float2{x.x / d, -x.y / d};
        }
        SBB_HD double2 recip(double2 x) {
            const double d = abs2(x);
            return double2{x.x / d, -x.y / d};
        }
        SBB_HD float sqrt_of(float x) { return sqrtf(x); }
        SBB_HD double sqrt_of(double x) { return sqrt(x); }
        SBB_HD void set_re(float &o, float v) { o = v; }
        SBB_HD void set_re(double &o, double v) { o = v; }
        SBB_HD void set_re(float2 &o, float v) { o.x = v, o.y = 0; }
        SBB_HD void set_re(double2 &o, double v) { o.x = v, o.y = 0; }
        template <typename T> SBB_HD void swap(T &a, T &b) {
            T t = a;
            a = b, b = t;
        }
        /// Unit roundoff of the real type
        SBB_HD float unit_roundoff(float) { return 5.9604645e-8f; }      // 2^-24
        SBB_HD double unit_roundoff(double) { return 1.1102230246251565e-16; } // 2^-53
        SBB_HD void set_nan(float &o) { o = NAN; }
        SBB_HD void set_nan(double &o) { o = NAN; }
        SBB_HD void set_nan(float2 &o) { o.x = o.y = NAN; }
        SBB_HD void set_nan(double2 &o) { o.x = o.y = NAN; }
        /// max(m, |x|) over the components of x; NaN once either is NaN
        SBB_HD float max_mag(float m, float x) {
            x = fabsf(x);
            return x > m || x != x ? x : m;
        }
        SBB_HD double max_mag(double m, double x) {
            x = fabs(x);
            return x > m || x != x ? x : m;
        }
        SBB_HD float max_mag(float m, float2 x) { return max_mag(max_mag(m, x.x), x.y); }
        SBB_HD double max_mag(double m, double2 x) { return max_mag(max_mag(m, x.x), x.y); }
        /// x 2^e, exactly while the result is a normal number
        SBB_HD float pow2_scale(float x, int e) { return ldexpf(x, e); }
        SBB_HD double pow2_scale(double x, int e) { return ldexp(x, e); }
        SBB_HD float2 pow2_scale(float2 x, int e) { return float2{ldexpf(x.x, e), ldexpf(x.y, e)}; }
        SBB_HD double2 pow2_scale(double2 x, int e) { return double2{ldexp(x.x, e), ldexp(x.y, e)}; }
        /// e with x = f 2^e, f in [1/2, 1) (0 for x == 0)
        SBB_HD int binary_exponent(float x) {
            int e = 0;
            frexpf(x, &e);
            return e;
        }
        SBB_HD int binary_exponent(double x) {
            int e = 0;
            frexp(x, &e);
            return e;
        }

        /// Offset of the l-th point of a label group (first label fastest) in tensor `which`
        /// (0: A, 1: X, 2: Y)
        SBB_HD int64_t group_offset(const sbk_dense_dim *g, int ng, int64_t l, int which) {
            int64_t o = 0;
            for (int k = 0; k < ng; ++k) {
                const int64_t i = l % g[k].size;
                l /= g[k].size;
                o += i * (which == 0 ? g[k].sa : which == 1 ? g[k].sx : g[k].sy);
            }
            return o;
        }

        /// A team of one thread (the host emulation)
        struct SerialTeam {
            int t = 0, nt = 1;
            void sync() const {}
        };

        /// Row of the largest |a(i,k)|, i >= k (the first such row on ties); every thread finds the same
        template <typename T> SBB_HD int pivot_row(const T *a, int n, int k) {
            int p = k;
            auto best = abs2(a[(int64_t)k * n + k]);
            for (int i = k + 1; i < n; ++i) {
                const auto v = abs2(a[(int64_t)i * n + k]);
                if (v > best) best = v, p = i;
            }
            return p;
        }

        /// A = U^H U: reads the upper triangle and the real part of the diagonal, leaves U there and
        /// zeros below the diagonal.  A non-positive pivot gives NaN or infinity.
        template <typename T, typename Team> SBB_HD void cholesky_body(T *a, int n, const Team &tm) {
            for (int k = 0; k < n; ++k) {
                const auto d = sqrt_of(re(a[(int64_t)k * n + k]));
                tm.sync(); // everyone has read the pivot before it is overwritten
                const auto inv = (decltype(d))1 / d;
                for (int j = k + tm.t; j < n; j += tm.nt) {
                    T &x = a[(int64_t)k * n + j];
                    if (j == k) set_re(x, d);
                    else x = scale(x, inv);
                }
                tm.sync();
                const int m = n - k - 1;
                for (int e = tm.t; e < m * m; e += tm.nt) {
                    const int i = k + 1 + e / m, j = k + 1 + e % m;
                    if (j >= i) fma_acc(a[(int64_t)i * n + j], neg(cj(a[(int64_t)k * n + i])), a[(int64_t)k * n + j]);
                }
                tm.sync();
            }
            for (int e = tm.t; e < n * n; e += tm.nt)
                if (e / n > e % n) set_zero(a[e]);
            tm.sync();
        }

        /// P A = L U with partial pivoting, in place (unit L below the diagonal, U on and above);
        /// row k was swapped with row piv[k] at step k
        template <typename T, typename Team> SBB_HD void lu_body(T *a, int *piv, int n, const Team &tm) {
            for (int k = 0; k < n; ++k) {
                const int p = pivot_row(a, n, k);
                tm.sync();
                if (tm.t == 0) piv[k] = p;
                if (p != k)
                    for (int j = tm.t; j < n; j += tm.nt) swap(a[(int64_t)k * n + j], a[(int64_t)p * n + j]);
                tm.sync();
                const T inv = recip(a[(int64_t)k * n + k]);
                for (int i = k + 1 + tm.t; i < n; i += tm.nt) a[(int64_t)i * n + k] = mulc(a[(int64_t)i * n + k], inv);
                tm.sync();
                const int m = n - k - 1;
                for (int e = tm.t; e < m * m; e += tm.nt) {
                    const int i = k + 1 + e / m, j = k + 1 + e % m;
                    fma_acc(a[(int64_t)i * n + j], neg(a[(int64_t)i * n + k]), a[(int64_t)k * n + j]);
                }
                tm.sync();
            }
        }

        /// A <- A^-1 in place by Gauss-Jordan elimination with partial pivoting (the pivots of LU);
        /// `f` holds n scratch elements, `piv` n ints
        template <typename T, typename Team>
        SBB_HD void inverse_body(T *a, T *f, int *piv, int n, const Team &tm) {
            for (int k = 0; k < n; ++k) {
                const int p = pivot_row(a, n, k);
                tm.sync();
                if (tm.t == 0) piv[k] = p;
                if (p != k)
                    for (int j = tm.t; j < n; j += tm.nt) swap(a[(int64_t)k * n + j], a[(int64_t)p * n + j]);
                tm.sync();
                const T inv = recip(a[(int64_t)k * n + k]);
                tm.sync();
                for (int j = tm.t; j < n; j += tm.nt) {
                    T &x = a[(int64_t)k * n + j];
                    x = j == k ? inv : mulc(x, inv);
                    if (j != k) f[j] = a[(int64_t)j * n + k];
                }
                tm.sync();
                for (int e = tm.t; e < n * n; e += tm.nt) {
                    const int i = e / n, j = e % n;
                    if (i == k) continue;
                    T &x = a[(int64_t)i * n + j];
                    if (j == k) x = mulc(neg(f[i]), a[(int64_t)k * n + k]);
                    else fma_acc(x, neg(f[i]), a[(int64_t)k * n + j]);
                }
                tm.sync();
            }
            for (int k = n - 1; k >= 0; --k) {
                const int p = piv[k];
                if (p != k)
                    for (int i = tm.t; i < n; i += tm.nt) swap(a[(int64_t)i * n + k], a[(int64_t)i * n + p]);
                tm.sync();
            }
        }

        /// Rotation sweeps of eigh_body at most; a matrix not converged by then is returned as it stands
        constexpr int EIGH_MAX_SWEEPS = 20;

        /// Pair k of round r of the round-robin ordering of m (even) indices: every pair of indices
        /// meets once in the m - 1 rounds of a sweep, and the m / 2 pairs of a round are disjoint
        SBB_HD void round_robin_pair(int m, int r, int k, int &p, int &q) {
            const int a = k == 0 ? m - 1 : (r + k) % (m - 1), b = k == 0 ? r : (r - k + m - 1) % (m - 1);
            p = a < b ? a : b, q = a < b ? b : a;
        }

        /// Eigen-decomposition A = V diag(w) V^H of a Hermitian matrix by cyclic two-sided Jacobi in the
        /// round-robin parallel ordering.  Reads the upper triangle and the real part of the diagonal
        /// of `a`; on return w holds the eigenvalues in ascending order (ties in index order) and, with
        /// `v` given, `a` holds V (column j the unit eigenvector of w[j]) while `v` was the workspace
        /// of the rotations; without `v` the eigenvectors are not accumulated and `a` is left
        /// overwritten.  A non-finite entry in what is read gives NaN in w and in V; every finite matrix
        /// is diagonalised.  Scratch: `sig` (n elements of T), `rot` (3 * ((n + 1) / 2) reals), `ix`
        /// (n + 1 ints).
        ///
        /// The sweeps work on 2^-e A, with 2^e the power of two that brings max |a_ij| (over the real and
        /// imaginary parts of what is read) into [1/2, 1): exact, so V is that of A and w is 2^e times the
        /// eigenvalues of the scaled matrix, and the squares in ||A||_F and in the skip test neither
        /// overflow nor underflow whatever the magnitude of A.  The maximum also finds non-finite input.
        ///
        /// A sweep is n - 1 rounds (n rounded up to even; the extra index pairs with nothing) of n / 2
        /// disjoint (p, q) pairs.  A round computes, per pair, the rotation J = [[c, s], [-s^*, c]] that
        /// zeros a_pq of its 2x2 block and applies A <- J^H A to rows p and q (one thread per pair);
        /// then, after a sync, A <- A J and V <- V J to the columns.  The block itself is set to its
        /// exact rotated value: a_pp - t|a_pq|, a_qq + t|a_pq| and zeros off the diagonal.  A pair is
        /// not rotated when |a_pq| <= u ||A||_F / n (u the unit roundoff), so that what the skipped
        /// elements leave off the diagonal is below u ||A||_F in norm; the sweeps stop after one without
        /// a rotation.  Every element is updated by the same formula whatever the team size, and
        /// ||A||_F is summed row by row and then over the rows in a fixed order, so the results are
        /// bit-identical across team sizes.
        template <typename T, typename Team>
        SBB_HD void eigh_body(T *a, T *v, typename Real<T>::type *w, T *sig, typename Real<T>::type *rot, int *ix,
                              int n, const Team &tm) {
            using R = typename Real<T>::type;
            // ---- max |a_ij| of what is read, row by row; V = I -------------------------------------------
            for (int i = tm.t; i < n; i += tm.nt) {
                R m = max_mag((R)0, re(a[(int64_t)i * n + i]));
                for (int j = i + 1; j < n; ++j) m = max_mag(m, a[(int64_t)i * n + j]);
                w[i] = m;
            }
            if (v)
                for (int e = tm.t; e < n * n; e += tm.nt) set_re(v[e], e / n == e % n ? (R)1 : (R)0);
            if (tm.t == 0) ix[n] = -1;
            tm.sync();
            R amax = 0;
            for (int i = 0; i < n; ++i) amax = max_mag(amax, w[i]);
            tm.sync();
            if (!(amax - amax == 0)) { // infinite or NaN
                for (int e = tm.t; e < n * n; e += tm.nt) set_nan(a[e]);
                for (int i = tm.t; i < n; i += tm.nt) set_nan(w[i]);
                tm.sync();
                return;
            }
            const int ex = binary_exponent(amax);
            // ---- the Hermitian matrix 2^-ex A from the upper triangle; row sums of |a_ij|^2 ------------
            for (int i = tm.t; i < n; i += tm.nt) {
                T &d = a[(int64_t)i * n + i];
                const R di = pow2_scale(re(d), -ex);
                set_re(d, di);
                R s = di * di;
                for (int j = i + 1; j < n; ++j) {
                    const T x = pow2_scale(a[(int64_t)i * n + j], -ex);
                    a[(int64_t)i * n + j] = x;
                    s += 2 * abs2(x);
                    a[(int64_t)j * n + i] = cj(x);
                }
                w[i] = s;
            }
            tm.sync();
            R norm2 = 0;
            for (int i = 0; i < n; ++i) norm2 += w[i];
            tm.sync();
            const R thr = unit_roundoff(R(0)) / (n > 0 ? n : 1), thr2 = thr * thr * norm2;

            // ---- sweeps --------------------------------------------------------------------------------
            const int m = n + (n & 1), npairs = m / 2;
            for (int sweep = 0; sweep < EIGH_MAX_SWEEPS && n > 1; ++sweep) {
                for (int r = 0; r < m - 1; ++r) {
                    for (int k = tm.t; k < npairs; k += tm.nt) {
                        int p, q;
                        round_robin_pair(m, r, k, p, q);
                        R *rk = rot + 3 * k;
                        rk[0] = 0; // c = 0: the pair is not rotated
                        if (q >= n) continue;
                        const T apq = a[(int64_t)p * n + q];
                        const R g = abs2(apq);
                        if (g <= thr2) continue;
                        const R app = re(a[(int64_t)p * n + p]), aqq = re(a[(int64_t)q * n + q]);
                        const R mag = sqrt_of(g), tau = (aqq - app) / (2 * mag);
                        const R t = (tau >= 0 ? (R)1 : (R)-1) / ((tau >= 0 ? tau : -tau) + sqrt_of(1 + tau * tau));
                        const R c = 1 / sqrt_of(1 + t * t);
                        const T s = scale(apq, t * c / mag);
                        rk[0] = c, rk[1] = app - t * mag, rk[2] = aqq + t * mag;
                        sig[k] = s;
                        ix[n] = sweep;
                        // rows p and q: A <- J^H A
                        for (int j = 0; j < n; ++j) {
                            T &x = a[(int64_t)p * n + j], &y = a[(int64_t)q * n + j];
                            T xp = scale(x, c), yp = scale(y, c);
                            fma_acc(xp, neg(s), y);
                            fma_acc(yp, cj(s), x);
                            x = xp, y = yp;
                        }
                    }
                    tm.sync();
                    // columns p and q: A <- A J, V <- V J
                    const int nmat = v ? 2 : 1;
                    for (int e = tm.t; e < nmat * n * npairs; e += tm.nt) {
                        const int k = e % npairs, i = e / npairs % n;
                        const R *rk = rot + 3 * k;
                        const R c = rk[0];
                        if (c == 0) continue;
                        int p, q;
                        round_robin_pair(m, r, k, p, q);
                        T *z = e < n * npairs ? a : v;
                        T &x = z[(int64_t)i * n + p], &y = z[(int64_t)i * n + q];
                        if (z == a && (i == p || i == q)) {
                            set_re(x, i == p ? rk[1] : (R)0);
                            set_re(y, i == p ? (R)0 : rk[2]);
                            continue;
                        }
                        const T s = sig[k];
                        T xp = scale(x, c), yp = scale(y, c);
                        fma_acc(xp, neg(cj(s)), y);
                        fma_acc(yp, s, x);
                        x = xp, y = yp;
                    }
                    tm.sync();
                }
                if (ix[n] < sweep) break; // no rotation in this sweep; later sweeps only raise ix[n]
            }

            // ---- eigenvalues ascending, stable; V's columns to match ----------------------------------
            for (int i = tm.t; i < n; i += tm.nt) {
                const R di = re(a[(int64_t)i * n + i]);
                int rank = 0;
                for (int j = 0; j < n; ++j) {
                    const R dj = re(a[(int64_t)j * n + j]);
                    rank += dj < di || (dj == di && j < i);
                }
                ix[i] = rank;
            }
            tm.sync();
            for (int i = tm.t; i < n; i += tm.nt) w[ix[i]] = pow2_scale(re(a[(int64_t)i * n + i]), ex);
            tm.sync();
            if (v)
                for (int e = tm.t; e < n * n; e += tm.nt) a[(int64_t)(e / n) * n + ix[e % n]] = v[e];
            tm.sync();
        }

        /// One right-hand side x (element i at x[i * ldx]) overwritten with the solution of
        /// U y = x (left) or y U = x (right); U upper triangular, only its upper triangle is read
        template <typename T> SBB_HD void upper_solve(const T *u, T *x, int n, int ldx, bool left) {
            if (left) {
                for (int i = n - 1; i >= 0; --i) {
                    T s = x[(int64_t)i * ldx];
                    for (int j = i + 1; j < n; ++j) fma_acc(s, neg(u[(int64_t)i * n + j]), x[(int64_t)j * ldx]);
                    x[(int64_t)i * ldx] = mulc(s, recip(u[(int64_t)i * n + i]));
                }
            } else {
                for (int c = 0; c < n; ++c) {
                    T s = x[(int64_t)c * ldx];
                    for (int r = 0; r < c; ++r) fma_acc(s, neg(x[(int64_t)r * ldx]), u[(int64_t)r * n + c]);
                    x[(int64_t)c * ldx] = mulc(s, recip(u[(int64_t)c * n + c]));
                }
            }
        }

        /// One right-hand side x overwritten with the solution of U^H y = x, by forward substitution;
        /// U upper triangular, only its upper triangle is read.  This is the panel of the blocked
        /// Cholesky factorisation: U12 = U11^-H A12, one column of A12 per right-hand side.
        template <typename T> SBB_HD void upper_h_solve(const T *u, T *x, int n, int ldx) {
            for (int c = 0; c < n; ++c) {
                T s = x[(int64_t)c * ldx];
                for (int r = 0; r < c; ++r) fma_acc(s, neg(cj(u[(int64_t)r * n + c])), x[(int64_t)r * ldx]);
                x[(int64_t)c * ldx] = mulc(s, recip(cj(u[(int64_t)c * n + c])));
            }
        }

        /// The same with the LU factors of lu_body: A y = x (left) or y A = x (right)
        template <typename T> SBB_HD void lu_solve(const T *lu, const int *piv, T *x, int n, int ldx, bool left) {
            if (left) {
                for (int k = 0; k < n; ++k)
                    if (piv[k] != k) swap(x[(int64_t)k * ldx], x[(int64_t)piv[k] * ldx]);
                for (int i = 1; i < n; ++i) {
                    T s = x[(int64_t)i * ldx];
                    for (int j = 0; j < i; ++j) fma_acc(s, neg(lu[(int64_t)i * n + j]), x[(int64_t)j * ldx]);
                    x[(int64_t)i * ldx] = s;
                }
                upper_solve(lu, x, n, ldx, true);
            } else {
                upper_solve(lu, x, n, ldx, false);
                for (int c = n - 2; c >= 0; --c) {
                    T s = x[(int64_t)c * ldx];
                    for (int r = c + 1; r < n; ++r) fma_acc(s, neg(x[(int64_t)r * ldx]), lu[(int64_t)r * n + c]);
                    x[(int64_t)c * ldx] = s;
                }
                for (int k = n - 1; k >= 0; --k)
                    if (piv[k] != k) swap(x[(int64_t)k * ldx], x[(int64_t)piv[k] * ldx]);
            }
        }

    } // namespace densek
} // namespace sbb
