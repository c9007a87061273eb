// Batched dense solvers: one launch factors, inverts, solves with or diagonalises (eigh) every matrix of a batch, loading
// and storing straight through the label strides of sbk_dense_desc (no permute pass, no contiguous
// temporary).  Two tiers:
//  * warp tier (n <= 32, the per-site blocks): one warp per matrix, up to 8 matrices per CTA; the CTA
//    loads its matrices together with consecutive lanes on consecutive batch entries when the batch
//    has the smallest stride, so a warp's accesses coalesce along the site labels.
//  * CTA tier (32 < n, up to the shared-memory limit): one CTA per matrix.
// trsm / gesm: the grid covers batch entries x chunks of right-hand sides; every CTA holds the factor
// in shared memory (gesm factors it again in every chunk: deterministic, and cheap next to the
// solves of a chunk) and each thread solves one right-hand side of the chunk.
// cholesky and trsm of a matrix over the shared-memory limit run a third, blocked tier: the matrices
// and right-hand sides are gathered into contiguous workspaces and worked through in blocks of
// BLOCK_N, with the CTA (or warp) tier on the diagonal blocks and contract() for the updates.
#include "dense_kernel.hpp"
#include "runtime.hpp"
#include <algorithm>
#include <cstring>
#include <sstream>
#include <type_traits>
#include <vector>

namespace sbb {

    namespace {
        using namespace densek;

        constexpr int CTA_THREADS = 256, MAX_TEAMS = 8;
        constexpr int64_t SMEM_OPTIN = 227 * 1024; ///< B200: dynamic shared memory of one CTA
        constexpr int64_t WARP_TIER_BUDGET = 96 * 1024;

        struct Head {
            int64_t ba, bx, by;
            int mcount, active;
        };

        int64_t up16(int64_t b) { return (b + 15) & ~(int64_t)15; }

        /// Shared memory of one team: head, matrix, n scratch elements, n x m right-hand sides, their
        /// offsets in X and Y, n pivots; eigh adds the eigenvectors, the eigenvalues with the rotations
        /// (n + 3 ((n + 1) / 2) reals, each given es bytes) and n + 1 ints
        struct Layout {
            int64_t mat, f, rhs, rx, ry, piv, vec, ew, ei, bytes;
            SBB_HD Layout(int n, int m, int es, bool eigh = false) {
                mat = 16 * ((sizeof(Head) + 15) / 16);
                f = mat + (((int64_t)n * n * es + 15) & ~(int64_t)15);
                rhs = f + (((int64_t)n * es + 15) & ~(int64_t)15);
                rx = rhs + (((int64_t)n * m * es + 15) & ~(int64_t)15);
                ry = rx + 8 * (int64_t)m;
                piv = ry + 8 * (int64_t)m;
                vec = piv + (((int64_t)n * 4 + 15) & ~(int64_t)15);
                ew = vec + (eigh ? ((int64_t)n * n * es + 15) & ~(int64_t)15 : 0);
                ei = ew + (eigh ? ((int64_t)(n + 3 * ((n + 1) / 2)) * es + 15) & ~(int64_t)15 : 0);
                bytes = ei + (eigh ? ((int64_t)(n + 1) * 4 + 15) & ~(int64_t)15 : 0);
            }
        };

        struct DenseParams {
            sbk_dense_desc d;
            int64_t nbatch, nrhs; ///< points of the batch and the rhs group
            int m, nchunks, teams;
            int row_fast, batch_fast, rhs_fast; ///< which index runs along consecutive threads
            int64_t table_bytes, team_bytes;
        };

        struct WarpTeam {
            int t, nt;
            SBB_HD void sync() const {
#ifdef __CUDA_ARCH__
                __syncwarp();
#endif
            }
        };
        struct CtaTeam {
            int t, nt;
            SBB_HD void sync() const {
#ifdef __CUDA_ARCH__
                __syncthreads();
#endif
            }
        };

        template <typename T> struct TeamView {
            using R = typename Real<T>::type;
            Head *h;
            T *mat, *f, *rhs, *vec;
            int64_t *rx, *ry;
            int *piv, *ei;
            R *w, *rot; ///< eigh: eigenvalues, then the rotations
        };

        template <typename T>
        __device__ __forceinline__ TeamView<T> team_view(unsigned char *smem, const DenseParams &p, int w) {
            using R = typename Real<T>::type;
            const int n = p.d.n;
            const Layout l(n, p.m, (int)sizeof(T), p.d.op == SBB_EIGH);
            unsigned char *b = smem + p.table_bytes + (int64_t)w * p.team_bytes;
            return TeamView<T>{(Head *)b,          (T *)(b + l.mat),       (T *)(b + l.f),   (T *)(b + l.rhs),
                               (T *)(b + l.vec),   (int64_t *)(b + l.rx),  (int64_t *)(b + l.ry),
                               (int *)(b + l.piv), (int *)(b + l.ei),      (R *)(b + l.ew),  (R *)(b + l.ew) + n};
        }

        /// x == nullptr: the right-hand sides are read from y, through the strides of X, and solved in
        /// place (the blocked tier)
        /// Eigh: the instantiation of eigh alone (its body and its stores stay out of the others' registers)
        template <typename T, bool Warp, bool Eigh>
        __global__ void __launch_bounds__(CTA_THREADS, 1)
            dense_kernel(const __grid_constant__ DenseParams p, T *__restrict__ a, const T *__restrict__ x,
                         T *__restrict__ y, T alpha) {
            extern __shared__ __align__(16) unsigned char smem[];
            const sbk_dense_desc &d = p.d;
            const int n = d.n, W = p.teams, m = p.m;
            const int64_t nn = (int64_t)n * n;
            int64_t *ra = (int64_t *)smem, *ca = ra + n, *xv = ca + n, *yv = xv + n;
            for (int i = threadIdx.x; i < n; i += blockDim.x) {
                ra[i] = group_offset(d.rows, d.nrows, i, 0);
                ca[i] = group_offset(d.cols, d.ncols, i, 0);
                xv[i] = d.left ? group_offset(d.rows, d.nrows, i, 1) : group_offset(d.cols, d.ncols, i, 1);
                yv[i] = d.left ? group_offset(d.cols, d.ncols, i, 2) : group_offset(d.rows, d.nrows, i, 2);
            }
            const int team = Warp ? threadIdx.x / 32 : 0;
            const int t = Warp ? threadIdx.x % 32 : threadIdx.x, nt = Warp ? 32 : blockDim.x;
            const TeamView<T> me = team_view<T>(smem, p, team);
            const int64_t unit = (int64_t)blockIdx.x * W + team, b = unit % p.nbatch, j0 = unit / p.nbatch * m;
            const bool active = unit < p.nbatch * p.nchunks;
            if (t == 0) {
                me.h->active = active;
                me.h->ba = group_offset(d.batch, d.nbatch, b, 0);
                me.h->bx = group_offset(d.batch, d.nbatch, b, 1);
                me.h->by = group_offset(d.batch, d.nbatch, b, 2);
                me.h->mcount = (int)(p.nrhs - j0 < m ? p.nrhs - j0 : m);
            }
            for (int j = t; j < m && j0 + j < p.nrhs; j += nt) {
                me.rx[j] = group_offset(d.rhs, d.nrhs, j0 + j, 1);
                me.ry[j] = group_offset(d.rhs, d.nrhs, j0 + j, 2);
            }
            __syncthreads();

            // ---- matrices in ----------------------------------------------------------------------
            for (int64_t idx = threadIdx.x; idx < W * nn; idx += blockDim.x) {
                const int w = p.batch_fast ? (int)(idx % W) : (int)(idx / nn);
                const int64_t e = p.batch_fast ? idx / W : idx % nn;
                const TeamView<T> v = team_view<T>(smem, p, w);
                const int r = p.row_fast ? (int)(e % n) : (int)(e / n), c = p.row_fast ? (int)(e / n) : (int)(e % n);
                if (!v.h->active || ((d.op == SBB_TRSM || d.op == PANEL || d.op == SBB_EIGH) && r > c)) continue;
                v.mat[(int64_t)r * n + c] = a[v.h->ba + ra[r] + ca[c]];
            }
            __syncthreads();

            // ---- factor -----------------------------------------------------------------------------
            using Team = typename std::conditional<Warp, WarpTeam, CtaTeam>::type;
            const Team tm{t, nt};
            if (active) {
                if constexpr (Eigh) eigh_body(me.mat, d.vectors ? me.vec : nullptr, me.w, me.f, me.rot, me.ei, n, tm);
                else if (d.op == SBB_CHOLESKY) cholesky_body(me.mat, n, tm);
                else if (d.op == SBB_INVERSION) inverse_body(me.mat, me.f, me.piv, n, tm);
                else if (d.op == SBB_GESM) lu_body(me.mat, me.piv, n, tm);
            }
            __syncthreads();

            if constexpr (Eigh) { // V over A, w into W (y, through the strides sy of the columns)
                using R = typename Real<T>::type;
                if (d.vectors)
                    for (int64_t idx = threadIdx.x; idx < W * nn; idx += blockDim.x) {
                        const int w = p.batch_fast ? (int)(idx % W) : (int)(idx / nn);
                        const int64_t e = p.batch_fast ? idx / W : idx % nn;
                        const TeamView<T> v = team_view<T>(smem, p, w);
                        const int r = p.row_fast ? (int)(e % n) : (int)(e / n), c = p.row_fast ? (int)(e / n) : (int)(e % n);
                        if (v.h->active) a[v.h->ba + ra[r] + ca[c]] = v.mat[(int64_t)r * n + c];
                    }
                if (y)
                    for (int64_t idx = threadIdx.x; idx < (int64_t)W * n; idx += blockDim.x) {
                        const int w = p.batch_fast ? (int)(idx % W) : (int)(idx / n);
                        const int i = p.batch_fast ? (int)(idx / W) : (int)(idx % n);
                        const TeamView<T> v = team_view<T>(smem, p, w);
                        if (v.h->active) ((R *)y)[v.h->by + yv[i]] = v.w[i];
                    }
                return;
            }

            if (d.op == SBB_CHOLESKY || d.op == SBB_INVERSION) {
                for (int64_t idx = threadIdx.x; idx < W * nn; idx += blockDim.x) {
                    const int w = p.batch_fast ? (int)(idx % W) : (int)(idx / nn);
                    const int64_t e = p.batch_fast ? idx / W : idx % nn;
                    const TeamView<T> v = team_view<T>(smem, p, w);
                    const int r = p.row_fast ? (int)(e % n) : (int)(e / n), c = p.row_fast ? (int)(e / n) : (int)(e % n);
                    if (v.h->active) a[v.h->ba + ra[r] + ca[c]] = v.mat[(int64_t)r * n + c];
                }
                return;
            }

            // ---- solves: right-hand sides in (scaled by alpha), one per thread, out ---------------------
            const int64_t nm = (int64_t)n * m;
            for (int64_t idx = threadIdx.x; idx < W * nm; idx += blockDim.x) {
                const int w = p.batch_fast ? (int)(idx % W) : (int)(idx / nm);
                const int64_t e = p.batch_fast ? idx / W : idx % nm;
                const TeamView<T> v = team_view<T>(smem, p, w);
                const int j = p.rhs_fast ? (int)(e % m) : (int)(e / n), i = p.rhs_fast ? (int)(e / m) : (int)(e % n);
                if (!v.h->active || j >= v.h->mcount) continue;
                v.rhs[(int64_t)i * m + j] = x ? mulc(alpha, x[v.h->bx + xv[i] + v.rx[j]])
                                              : mulc(alpha, y[v.h->bx + xv[i] + v.rx[j]]);
            }
            __syncthreads();
            if (active && t < me.h->mcount) {
                if (d.op == SBB_TRSM) upper_solve(me.mat, me.rhs + t, n, m, d.left != 0);
                else if (d.op == PANEL) upper_h_solve(me.mat, me.rhs + t, n, m);
                else lu_solve(me.mat, me.piv, me.rhs + t, n, m, d.left != 0);
            }
            __syncthreads();
            for (int64_t idx = threadIdx.x; idx < W * nm; idx += blockDim.x) {
                const int w = p.batch_fast ? (int)(idx % W) : (int)(idx / nm);
                const int64_t e = p.batch_fast ? idx / W : idx % nm;
                const TeamView<T> v = team_view<T>(smem, p, w);
                const int j = p.rhs_fast ? (int)(e % m) : (int)(e / n), i = p.rhs_fast ? (int)(e / m) : (int)(e % n);
                if (!v.h->active || j >= v.h->mcount) continue;
                y[v.h->by + yv[i] + v.ry[j]] = v.rhs[(int64_t)i * m + j];
            }
        }

        int64_t points(const sbk_dense_dim *g, int ng) {
            int64_t v = 1;
            for (int k = 0; k < ng; ++k) v *= g[k].size;
            return v;
        }

        int64_t min_stride(const sbk_dense_dim *g, int ng, int which) {
            int64_t s = INT64_MAX;
            for (int k = 0; k < ng; ++k) s = std::min(s, which == 0 ? g[k].sa : which == 1 ? g[k].sx : g[k].sy);
            return s;
        }

        const char *op_name(int op) {
            return op == SBB_CHOLESKY    ? "cholesky"
                   : op == SBB_INVERSION ? "inversion"
                   : op == SBB_TRSM      ? "trsm"
                   : op == PANEL         ? "panel"
                   : op == SBB_EIGH      ? "eigh"
                                         : "gesm";
        }

        template <typename T>
        void run(const sbk_dense_desc &d, const double *alpha, void *a, const void *x, void *y,
                 cudaStream_t stream, std::string *describe) {
            const bool solve = d.op == SBB_TRSM || d.op == SBB_GESM || d.op == PANEL;
            const int n = d.n, es = (int)sizeof(T);
            DenseParams p;
            p.d = d;
            p.nbatch = points(d.batch, d.nbatch);
            p.nrhs = solve ? points(d.rhs, d.nrhs) : 1;
            p.table_bytes = up16(32 * (int64_t)n);
            const bool warp = n <= 32;
            const bool eigh = d.op == SBB_EIGH;
            if (warp) {
                p.m = solve ? (int)std::min<int64_t>(32, p.nrhs) : 0;
                p.team_bytes = Layout(n, p.m, es, eigh).bytes;
                p.teams = (int)std::max<int64_t>(1, std::min<int64_t>(MAX_TEAMS, WARP_TIER_BUDGET / p.team_bytes));
            } else {
                const int64_t room = SMEM_OPTIN - p.table_bytes - Layout(n, 0, es).bytes;
                p.m = solve ? (int)std::min<int64_t>(std::min<int64_t>(CTA_THREADS, p.nrhs), room / ((int64_t)n * es + 16))
                            : 0;
                p.team_bytes = Layout(n, p.m, es, eigh).bytes;
                p.teams = 1;
            }
            p.nchunks = !solve ? 1 : p.m > 0 ? (int)((p.nrhs + p.m - 1) / p.m) : 0;
            const int64_t units = p.nbatch * p.nchunks;
            if (warp) p.teams = (int)std::max<int64_t>(1, std::min<int64_t>(p.teams, units));
            p.row_fast = min_stride(d.rows, d.nrows, 0) <= min_stride(d.cols, d.ncols, 0);
            p.batch_fast = warp && min_stride(d.batch, d.nbatch, 0) < std::min(min_stride(d.rows, d.nrows, 0),
                                                                                 min_stride(d.cols, d.ncols, 0));
            const sbk_dense_dim *xvec = d.left ? d.rows : d.cols;
            const int nxvec = d.left ? d.nrows : d.ncols;
            p.rhs_fast = solve && min_stride(d.rhs, d.nrhs, 1) < min_stride(xvec, nxvec, 1);
            const int64_t smem = p.table_bytes + p.teams * p.team_bytes;
            const int threads = warp ? 32 * p.teams : CTA_THREADS;
            const int64_t grid = (units + p.teams - 1) / p.teams;
            if (describe) {
                std::stringstream ss;
                ss << "dense " << op_name(d.op) << " tier=" << (warp ? "warp" : "cta") << " n=" << n
                   << " batch=" << p.nbatch << " rhs=" << (solve ? p.nrhs : 0) << " chunk=" << p.m
                   << " teams=" << p.teams << " grid=" << grid << " threads=" << threads << " smem=" << smem;
                *describe = ss.str();
                return;
            }
            if (units == 0 || n == 0) return;
            if (grid > 0x7fffffff) throw std::runtime_error("dense: too many matrices in one launch");
            auto kernel = eigh ? (warp ? dense_kernel<T, true, true> : dense_kernel<T, false, true>)
                               : (warp ? dense_kernel<T, true, false> : dense_kernel<T, false, false>);
            cuda_check(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                       "cudaFuncSetAttribute");
            T al;
            narrow(scalar_of<T>(alpha), al);
            {
                KernelTimer timer("dense", stream);
                kernel<<<(unsigned)grid, threads, (size_t)smem, stream>>>(p, (T *)a, (const T *)x, (T *)y, al);
            }
            count_launch();
            cuda_check(cudaGetLastError(), "dense_kernel launch");
        }

        // ---- blocked tier ------------------------------------------------------------------------------

        /// A place in a buffer of the blocked tier: the call's matrices A, right-hand sides X or solutions
        /// Y, or the workspaces W (matrices) and V (right-hand sides); offset in elements
        struct Ref {
            char buf;
            int64_t off;
        };

        /// One launch of the blocked tier
        struct Step {
            enum Kind { Copy, Dense, Update } kind;
            const char *name; ///< Copy: gather, scatter, zero; Dense: factor, panel, solve; Update: update
            Ref p[3];         ///< Copy: source, destination; Dense: matrix, right-hand sides; Update: v0, v1, vr
            int scale;        ///< Copy: 0 zero fill, 1 plain copy, 2 times alpha
            int rows, cols;   ///< zero: the block
            sbk_box_desc box;
            sbk_dense_desc dd;
            sbk_contract_desc cd;
        };

        struct Schedule {
            int64_t nbatch, nrhs, w_elems, v_elems;
            std::vector<Step> steps;
        };

        /// Every launch of the blocked tier for cholesky or trsm with `d`, in order; both the launcher
        /// and the description run through it.  W[b][r][c] holds the matrices row-major and V[b][j][i]
        /// the right-hand sides of trsm times alpha, each one contiguous (b: the batch labels of d, j: its
        /// rhs labels, first label fastest).  Blocks of BLOCK_N; a remainder joins the last block when
        /// the two fit one CTA together, so that no update is left with a sliver.
        ///  cholesky, right-looking, for every block k: factor the diagonal block (CTA tier); panel
        ///    U12 = U11^-H A12 (PANEL); zero the block column below the diagonal; A22 -= U12^H U12
        ///    (contract, the whole square: its lower triangle is never read).
        ///  trsm left (U Y = X): blocks last to first, solve the diagonal block in V, then
        ///    V[0:i] -= U[0:i, i] Y_i; right (Y U = X): first to last, V[:, j+1:] -= Y_j U[j, j+1:].
        Schedule blocked_schedule(const sbk_dense_desc &d, int es) {
            Schedule s;
            const int n = d.n;
            const int64_t nn = (int64_t)n * n;
            const bool trsm = d.op == SBB_TRSM;
            s.nbatch = points(d.batch, d.nbatch);
            s.nrhs = trsm ? points(d.rhs, d.nrhs) : 0;
            s.w_elems = s.nbatch * nn;
            s.v_elems = s.nbatch * s.nrhs * n;
            // strides of the batch labels in W and V, of the rhs labels in V
            int64_t wb[SBK_MAX_GROUP_DIMS], vb[SBK_MAX_GROUP_DIMS], vh[SBK_MAX_GROUP_DIMS];
            for (int k = 0; k < d.nbatch; ++k)
                wb[k] = k ? wb[k - 1] * d.batch[k - 1].size : nn, vb[k] = k ? vb[k - 1] * d.batch[k - 1].size : s.nrhs * n;
            for (int k = 0; k < d.nrhs; ++k) vh[k] = k ? vh[k - 1] * d.rhs[k - 1].size : n;

            std::vector<int> edge;
            for (int k = 0; k < n; k += BLOCK_N) edge.push_back(k);
            if (n % BLOCK_N && edge.size() > 1 && fits_cta(BLOCK_N + n % BLOCK_N, es)) edge.pop_back();
            edge.push_back(n);

            auto step = [&](Step::Kind kind, const char *name) -> Step & {
                Step st;
                std::memset(&st, 0, sizeof st);
                st.kind = kind, st.name = name;
                s.steps.push_back(st);
                return s.steps.back();
            };
            auto dim = [](sbk_box_desc &b, int size, int64_t ss, int64_t ds) {
                if (b.nd >= SBK_MAX_DIMS) throw std::runtime_error("dense: too many labels for the blocked tier");
                b.size[b.nd] = size, b.sstride[b.nd] = ss, b.dstride[b.nd++] = ds;
            };
            // A <-> W: every row, column and batch label one dimension
            auto matrices = [&](const char *name, Ref src, Ref dst, bool to_w) {
                Step &st = step(Step::Copy, name);
                st.p[0] = src, st.p[1] = dst, st.scale = 1;
                int64_t c = n;
                for (int k = 0; k < d.nrows; c *= d.rows[k++].size)
                    dim(st.box, d.rows[k].size, to_w ? d.rows[k].sa : c, to_w ? c : d.rows[k].sa);
                c = 1;
                for (int k = 0; k < d.ncols; c *= d.cols[k++].size)
                    dim(st.box, d.cols[k].size, to_w ? d.cols[k].sa : c, to_w ? c : d.cols[k].sa);
                for (int k = 0; k < d.nbatch; ++k)
                    dim(st.box, d.batch[k].size, to_w ? d.batch[k].sa : wb[k], to_w ? wb[k] : d.batch[k].sa);
            };
            // X -> V (times alpha) and V -> Y, through the strides of X resp. Y
            auto vectors = [&](const char *name, Ref src, Ref dst, bool to_v) {
                Step &st = step(Step::Copy, name);
                st.p[0] = src, st.p[1] = dst, st.scale = to_v ? 2 : 1;
                const bool rows = d.left ? to_v : !to_v; // X carries the rows when left, Y the rows when right
                const sbk_dense_dim *vec = rows ? d.rows : d.cols;
                const int nvec = rows ? d.nrows : d.ncols;
                auto sv = [&](const sbk_dense_dim &x) { return to_v ? x.sx : x.sy; };
                int64_t c = 1;
                for (int k = 0; k < nvec; c *= vec[k++].size)
                    dim(st.box, vec[k].size, to_v ? sv(vec[k]) : c, to_v ? c : sv(vec[k]));
                for (int k = 0; k < d.nrhs; ++k)
                    dim(st.box, d.rhs[k].size, to_v ? sv(d.rhs[k]) : vh[k], to_v ? vh[k] : sv(d.rhs[k]));
                for (int k = 0; k < d.nbatch; ++k)
                    dim(st.box, d.batch[k].size, to_v ? sv(d.batch[k]) : vb[k], to_v ? vb[k] : sv(d.batch[k]));
            };
            // the CTA (or warp) tier on the diagonal block [i0, i1) of W, right-hand sides at `rhs`
            auto diagonal = [&](const char *name, int op, int i0, int i1, Ref rhs) {
                Step &st = step(Step::Dense, name);
                const int bs = i1 - i0;
                st.p[0] = Ref{'W', (int64_t)i0 * n + i0}, st.p[1] = rhs;
                sbk_dense_desc &e = st.dd;
                e.op = op, e.n = bs, e.left = op == PANEL ? 1 : d.left;
                e.nrows = e.ncols = 1;
                if (op == PANEL) { // columns i1.. of the block rows: vectors over the rows, stride n
                    e.rows[0] = sbk_dense_dim{bs, n, n, 0}, e.cols[0] = sbk_dense_dim{bs, 1, 0, n};
                    e.nrhs = 1, e.rhs[0] = sbk_dense_dim{n - i1, 0, 1, 1};
                } else {
                    e.rows[0] = sbk_dense_dim{bs, n, 1, 1}, e.cols[0] = sbk_dense_dim{bs, 1, 1, 1};
                    e.nrhs = trsm ? d.nrhs : 0;
                    for (int k = 0; k < e.nrhs; ++k) e.rhs[k] = sbk_dense_dim{d.rhs[k].size, 0, vh[k], vh[k]};
                }
                e.nbatch = d.nbatch;
                for (int k = 0; k < d.nbatch; ++k)
                    e.batch[k] = sbk_dense_dim{d.batch[k].size, wb[k], trsm ? vb[k] : wb[k], trsm ? vb[k] : wb[k]};
            };
            // vr -= f0(v0) v1 with the batch labels in T; the caller adds M, N and K
            auto update = [&](Ref v0, Ref v1, Ref vr, int conj0) -> sbk_contract_desc & {
                Step &st = step(Step::Update, "update");
                st.p[0] = v0, st.p[1] = v1, st.p[2] = vr;
                sbk_contract_desc &c = st.cd;
                c.conj0 = conj0;
                auto bs = [&](char b, int k) { return b == 'W' ? wb[k] : vb[k]; };
                c.nT = d.nbatch;
                for (int k = 0; k < d.nbatch; ++k)
                    c.T[k] = sbk_contract_dim{d.batch[k].size, bs(v0.buf, k), bs(v1.buf, k), bs(vr.buf, k)};
                return c;
            };

            const Ref A{'A', 0}, W{'W', 0}, V{'V', 0};
            const int nblocks = (int)edge.size() - 1;
            if (!trsm) {
                matrices("gather", A, W, true);
                for (int b = 0; b < nblocks; ++b) {
                    const int k0 = edge[b], k1 = edge[b + 1], bs = k1 - k0, rest = n - k1;
                    diagonal("factor", SBB_CHOLESKY, k0, k1, Ref{'W', (int64_t)k0 * n + k0});
                    if (rest == 0) break;
                    diagonal("panel", PANEL, k0, k1, Ref{'W', (int64_t)k0 * n + k1});
                    Step &z = step(Step::Copy, "zero");
                    z.p[0] = z.p[1] = Ref{'W', (int64_t)k1 * n + k0}, z.scale = 0, z.rows = rest, z.cols = bs;
                    dim(z.box, bs, 1, 1), dim(z.box, rest, n, n);
                    for (int k = 0; k < d.nbatch; ++k) dim(z.box, d.batch[k].size, wb[k], wb[k]);
                    const Ref u12{'W', (int64_t)k0 * n + k1};
                    sbk_contract_desc &c = update(u12, u12, Ref{'W', (int64_t)k1 * n + k1}, 1);
                    c.nK = c.nM = c.nN = 1;
                    c.K[0] = sbk_contract_dim{bs, n, n, 0};
                    c.M[0] = sbk_contract_dim{rest, 1, 0, n};
                    c.N[0] = sbk_contract_dim{rest, 0, 1, 1};
                }
                matrices("scatter", W, A, false);
                return s;
            }
            matrices("gather", A, W, true);
            vectors("gather", Ref{'X', 0}, V, true);
            for (int t = 0; t < nblocks; ++t) {
                const int b = d.left ? nblocks - 1 - t : t;
                const int i0 = edge[b], i1 = edge[b + 1], bs = i1 - i0;
                diagonal("solve", SBB_TRSM, i0, i1, Ref{'V', i0});
                if (d.left && i0 > 0) { // V[0:i0] -= U[0:i0, i0:i1] Y_b
                    sbk_contract_desc &c = update(Ref{'W', i0}, Ref{'V', i0}, V, 0);
                    c.nM = c.nK = 1, c.nN = d.nrhs;
                    c.M[0] = sbk_contract_dim{i0, n, 0, 1};
                    c.K[0] = sbk_contract_dim{bs, 1, 1, 0};
                    for (int k = 0; k < d.nrhs; ++k) c.N[k] = sbk_contract_dim{d.rhs[k].size, 0, vh[k], vh[k]};
                } else if (!d.left && i1 < n) { // V[:, i1:] -= Y_b U[i0:i1, i1:]
                    sbk_contract_desc &c = update(Ref{'V', i0}, Ref{'W', (int64_t)i0 * n + i1}, Ref{'V', i1}, 0);
                    c.nM = d.nrhs, c.nK = c.nN = 1;
                    for (int k = 0; k < d.nrhs; ++k) c.M[k] = sbk_contract_dim{d.rhs[k].size, vh[k], 0, vh[k]};
                    c.K[0] = sbk_contract_dim{bs, 1, n, 0};
                    c.N[0] = sbk_contract_dim{n - i1, 0, 1, 1};
                }
            }
            vectors("scatter", V, Ref{'Y', 0}, false);
            return s;
        }

        void blocked(const sbk_dense_desc &d, int dtype, int es, const double *alpha, void *a, const void *x,
                     void *y, cudaStream_t stream, std::string *describe) {
            const Schedule s = blocked_schedule(d, es);
            const double one[2] = {1, 0}, zero[2] = {0, 0}, minus_one[2] = {-1, 0};
            std::stringstream ss;
            ss << "dense " << op_name(d.op) << " tier=blocked n=" << d.n << " batch=" << s.nbatch
               << " rhs=" << s.nrhs << " nb=" << BLOCK_N << " w=" << s.w_elems << " v=" << s.v_elems;
            if (!describe && (s.w_elems == 0 || (d.op == SBB_TRSM && s.v_elems == 0))) return;
            int dev = 0;
            if (!describe) cuda_check(cudaGetDevice(&dev), "cudaGetDevice");
            PoolGuard pool;
            char *w = describe ? nullptr : (char *)pool.alloc(dev, (size_t)s.w_elems * es);
            char *v = describe || s.v_elems == 0 ? nullptr : (char *)pool.alloc(dev, (size_t)s.v_elems * es);
            auto at = [&](const Ref &r) {
                char *b = r.buf == 'A' ? (char *)a : r.buf == 'X' ? (char *)x : r.buf == 'Y' ? (char *)y : r.buf == 'W' ? w : v;
                return b + r.off * es;
            };
            auto ref = [&](const Ref &r) { ss << " " << r.buf << " " << r.off; };
            for (const Step &st : s.steps) {
                std::string k;
                if (st.kind == Step::Copy) {
                    if (describe) {
                        ss << "\nstep " << st.name;
                        ref(st.p[0]);
                        if (st.scale == 0) ss << " rows " << st.rows << " cols " << st.cols;
                        else ref(st.p[1]);
                        continue;
                    }
                    permute_copy(st.box, at(st.p[0]), dtype, at(st.p[1]), dtype,
                                 st.scale == 0 ? zero : st.scale == 1 ? one : alpha, false, dev, stream);
                } else if (st.kind == Step::Dense) {
                    if (describe) {
                        dense(st.dd, dtype, one, nullptr, nullptr, nullptr, nullptr, &k);
                        ss << "\nstep " << st.name;
                        ref(st.p[0]);
                        if (st.dd.op != SBB_CHOLESKY) ref(st.p[1]);
                        ss << " n " << st.dd.n;
                        if (st.dd.op == PANEL) ss << " rhs " << st.dd.rhs[0].size;
                        if (st.dd.op == SBB_TRSM) ss << " left " << st.dd.left;
                        ss << " kernel " << k;
                        continue;
                    }
                    dense(st.dd, dtype, one, at(st.p[0]), nullptr, at(st.p[1]), stream);
                } else {
                    if (describe) {
                        contract(st.cd, dtype, minus_one, nullptr, nullptr, one, nullptr, dev, nullptr, &k);
                        const sbk_contract_desc &c = st.cd;
                        ss << "\nstep update";
                        for (const Ref &r : st.p) ref(r);
                        ss << " conj0 " << c.conj0;
                        const struct {
                            const char *name;
                            int n;
                            const sbk_contract_dim *dims;
                        } groups[] = {{"T", c.nT, c.T}, {"M", c.nM, c.M}, {"N", c.nN, c.N}, {"K", c.nK, c.K}};
                        for (const auto &g : groups) {
                            ss << " " << g.name;
                            for (int i = 0; i < g.n; ++i)
                                ss << " " << g.dims[i].size << " " << g.dims[i].s0 << " " << g.dims[i].s1 << " " << g.dims[i].sr;
                        }
                        ss << " kernel " << k;
                        continue;
                    }
                    contract(st.cd, dtype, minus_one, at(st.p[0]), at(st.p[1]), one, at(st.p[2]), dev, stream);
                }
            }
            if (describe) *describe = ss.str();
        }
    } // namespace

    void dense(const sbk_dense_desc &d, int dtype, const double *alpha, void *a, const void *x, void *y,
               cudaStream_t stream, std::string *describe) {
        const int es = dtype == SBB_F32 ? 4 : dtype == SBB_F64 || dtype == SBB_C64 ? 8 : 16;
        if ((d.op == SBB_CHOLESKY || d.op == SBB_TRSM) && !densek::fits_cta(d.n, es) &&
            (dtype == SBB_F32 || dtype == SBB_F64 || dtype == SBB_C64 || dtype == SBB_C128))
            return blocked(d, dtype, es, alpha, a, x, y, stream, describe);
        switch (dtype) {
        case SBB_F32: return run<float>(d, alpha, a, x, y, stream, describe);
        case SBB_F64: return run<double>(d, alpha, a, x, y, stream, describe);
        case SBB_C64: return run<float2>(d, alpha, a, x, y, stream, describe);
        case SBB_C128: return run<double2>(d, alpha, a, x, y, stream, describe);
        default: throw std::runtime_error("dense: unsupported type");
        }
    }

} // namespace sbb
