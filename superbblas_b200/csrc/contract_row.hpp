// Row kernel of the contraction: one thread per output ROW for problems with a short contracted
// range and one small free group ("update" shapes of the reference's tests/dist.cpp: m = 49152,
// n = k = 3..16; colour/spin matrices applied to every site).  Such problems are bound by reading the
// big operand and writing the result once; the generic one-thread-per-output kernel re-reads the
// big operand for every column and, for column-major results, writes uncoalesced.  Here a thread
// walks its row of the big operand once, keeps the S <= 16 partial sums in registers and reads the
// small operand through L1 (every lane of a warp reads the same word: a broadcast).
//
// The body is written as a host/device function so that the indexing and the arithmetic are
// checked on the CPU by tests/test_row_kernel_emulation.py (the same code runs one row per call);
// only the launch itself needs a GPU.  Validated on a B200 in round 2; default dispatch for these shapes
// (kernels_contract.cu also has the variant that stages the small operand in shared memory).
#pragma once
#include "../../include/superbblas_b200.h"
#include "contract_scalar.hpp"
#include <cstring>
#include <stdexcept>
#include <vector>

namespace sbb {
    namespace rowk {

        using namespace sbb; // code that uses namespace rowk also sees the scalar helpers (contract_scalar.hpp)

        constexpr int RD = 2 * SBK_MAX_GROUP_DIMS; // dims of a row index (batch labels + big free group)
        constexpr int SMAX = 16;                   // extent of the small free group (partial sums per thread)
        constexpr int KMAX = 64;                   // contracted extent

        struct RowParams {
            int nd;                              ///< dims of the row index, fastest thread index first
            int size[RD];
            long long sa[RD], sb[RD], sr[RD];    ///< strides in the big operand, the small operand, the result
            long long rows;                      ///< number of rows
            int ns, nk;                          ///< extents of the small free group and of the contraction
            long long koff_a[KMAX], koff_b[KMAX]; ///< offset of contracted index k in the big / small operand
            long long soff_b[SMAX], soff_r[SMAX]; ///< offset of small index s in the small operand / result
            int conj_a, conj_b;                  ///< conjugate the big / small operand
        };

        /// One row: vr[row, s] = alpha * sum_k fa(va[row, k]) * fb(vb[row's batch, k, s]) + beta * vr[row, s]
        template <typename T>
        SBB_HD void row_body(const RowParams &p, long long row, const T *va, const T *vb, T *vr,
                             typename Acc<T>::type alpha, typename Acc<T>::type beta) {
            using A = typename Acc<T>::type;
            long long oa = 0, ob = 0, orr = 0, rem = row;
#pragma unroll 1
            for (int d = 0; d < p.nd; ++d) {
                const long long c = rem % p.size[d];
                rem /= p.size[d];
                oa += c * p.sa[d], ob += c * p.sb[d], orr += c * p.sr[d];
            }
            using F = typename Fast<T>::type;
            F acc[SMAX];
#pragma unroll
            for (int s = 0; s < SMAX; ++s) set_zero(acc[s]);
            constexpr int KB = 8; // loads of the row in flight per thread
            for (int k0 = 0; k0 < p.nk; k0 += KB) {
                F a[KB];
#pragma unroll
                for (int j = 0; j < KB; ++j)
                    if (k0 + j < p.nk) {
                        a[j] = va[oa + p.koff_a[k0 + j]];
                        if (p.conj_a) a[j] = cj(a[j]);
                    }
#pragma unroll
                for (int j = 0; j < KB; ++j)
                    if (k0 + j < p.nk) {
                        const T *bk = vb + ob + p.koff_b[k0 + j];
#pragma unroll
                        for (int s = 0; s < SMAX; ++s)
                            if (s < p.ns) {
                                F b = bk[p.soff_b[s]];
                                if (p.conj_b) b = cj(b);
                                fma_acc(acc[s], a[j], b);
                            }
                    }
            }
            // (the epilogue written out rather than sbb::epilogue: that call would read p.soff_r[s] before
            // the product, which reorders the complex kernels' code)
#pragma unroll
            for (int s = 0; s < SMAX; ++s)
                if (s < p.ns) {
                    A r = mulc(alpha, widen(acc[s]));
                    T *w = vr + orr + p.soff_r[s];
                    if (!is_zero(beta)) r = addc(r, mulc(beta, widen(*w)));
                    narrow(r, *w);
                }
        }

        // ---- output enumeration of the generic kernel ---------------------------------------------------
        /// Thread index -> (t, m, n) with the groups listed in `order` (0 = T, 1 = M, 2 = N) from the
        /// fastest to the slowest; {2, 1, 0} is the kernel's default (n fastest, then m, then t)
        SBB_HD void output_index(const int *order, long long tvol, long long mvol, long long nvol,
                                 long long idx, long long &t, long long &m, long long &n) {
            long long g[3] = {0, 0, 0};
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                const int grp = order[q];
                const long long vol = grp == 0 ? tvol : grp == 1 ? mvol : nvol;
                const long long c = idx % vol;
                idx /= vol;
                if (grp == 0) g[0] = c;
                else if (grp == 1) g[1] = c;
                else g[2] = c;
            }
            t = g[0], m = g[1], n = g[2];
        }

        /// Groups ordered by their smallest result stride (ties and absent groups keep {N, M, T})
        inline void output_order(const long long min_sr[3], int *order) {
            order[0] = 2, order[1] = 1, order[2] = 0;
            for (int i = 1; i < 3; ++i)
                for (int j = i; j > 0 && min_sr[order[j]] < min_sr[order[j - 1]]; --j) {
                    const int x = order[j];
                    order[j] = order[j - 1], order[j - 1] = x;
                }
        }

        // ---- host: parameters from a contraction descriptor -------------------------------------------

        struct Dim {
            int size;
            long long sa, sb, sr;
        };

        inline long long volume_of(const sbk_contract_dim *d, int n) {
            long long v = 1;
            for (int i = 0; i < n; ++i) v *= d[i].size;
            return v;
        }

        /// Offsets of every index of a label group (first label fastest) for one stride selector
        inline void group_offsets(const sbk_contract_dim *d, int n, int which, long long *out) {
            const long long vol = volume_of(d, n);
            for (long long i = 0; i < vol; ++i) {
                long long rem = i, off = 0;
                for (int k = 0; k < n; ++k) {
                    const long long c = rem % d[k].size;
                    rem /= d[k].size;
                    off += c * (which == 0 ? d[k].s0 : which == 1 ? d[k].s1 : d[k].sr);
                }
                out[i] = off;
            }
        }

        /// Can the row kernel run this problem?  (short contraction, one small free group, nothing empty)
        inline bool eligible(const sbk_contract_desc &c) {
            const long long m = volume_of(c.M, c.nM), n = volume_of(c.N, c.nN), k = volume_of(c.K, c.nK),
                            t = volume_of(c.T, c.nT);
            if (m <= 0 || n <= 0 || t <= 0 || k <= 0 || k > KMAX) return false;
            return (m >= n ? n : m) <= SMAX;
        }

        /// Fill RowParams; `swapped` tells the caller that the big operand is v1 (the big free group is N)
        inline void build(const sbk_contract_desc &c, RowParams &p, bool &swapped) {
            if (!eligible(c)) throw std::runtime_error("row kernel: shape not supported");
            std::memset(&p, 0, sizeof p);
            const long long m = volume_of(c.M, c.nM), n = volume_of(c.N, c.nN);
            swapped = n > m; // rows run over the bigger free group
            const sbk_contract_dim *big = swapped ? c.N : c.M, *small = swapped ? c.M : c.N;
            const int nbig = swapped ? c.nN : c.nM, nsmall = swapped ? c.nM : c.nN;
            const int wa = swapped ? 1 : 0, wb = swapped ? 0 : 1; // stride selectors of the big / small operand
            p.conj_a = swapped ? c.conj1 : c.conj0;
            p.conj_b = swapped ? c.conj0 : c.conj1;
            // row dims: batch labels and the big free group, the smallest result stride first
            std::vector<Dim> rows;
            auto pick = [](const sbk_contract_dim &d, int w) { return w == 0 ? d.s0 : d.s1; };
            for (int i = 0; i < c.nT; ++i)
                if (c.T[i].size > 1) rows.push_back({c.T[i].size, pick(c.T[i], wa), pick(c.T[i], wb), c.T[i].sr});
            for (int i = 0; i < nbig; ++i)
                if (big[i].size > 1) rows.push_back({big[i].size, pick(big[i], wa), 0, big[i].sr});
            for (size_t i = 1; i < rows.size(); ++i) // insertion sort by |result stride| (stable)
                for (size_t j = i; j > 0 && std::llabs(rows[j].sr) < std::llabs(rows[j - 1].sr); --j)
                    std::swap(rows[j], rows[j - 1]);
            if ((int)rows.size() > RD) throw std::runtime_error("row kernel: too many labels");
            p.nd = (int)rows.size();
            p.rows = 1;
            for (int d = 0; d < p.nd; ++d) {
                p.size[d] = rows[d].size, p.sa[d] = rows[d].sa, p.sb[d] = rows[d].sb, p.sr[d] = rows[d].sr;
                p.rows *= rows[d].size;
            }
            p.ns = (int)volume_of(small, nsmall);
            p.nk = (int)volume_of(c.K, c.nK);
            group_offsets(c.K, c.nK, wa, p.koff_a);
            group_offsets(c.K, c.nK, wb, p.koff_b);
            group_offsets(small, nsmall, wb, p.soff_b);
            group_offsets(small, nsmall, 2, p.soff_r);
        }

    } // namespace rowk
} // namespace sbb
