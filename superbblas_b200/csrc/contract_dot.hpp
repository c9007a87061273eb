// Dot kernel of the contraction: long contracted range, both free groups small ("inner product" shapes
// of the reference's tests/dist.cpp: m, n <= 16, k = 49152; V^H V with a handful of vectors).  Such
// problems are bound by reading both operands once; the tensor-core kernel wastes most of its 64x64
// tile on them and the generic kernel has no parallelism over K.  Here the contracted range is cut in
// `slices` interleaved slices (consecutive threads take consecutive k, so the loads are coalesced when
// K is contiguous); a thread keeps a 4x4 block of partial sums in registers; the 128 threads of a CTA
// (128 consecutive slices of the same outputs) add their blocks with a fixed shuffle / shared-memory
// tree and write ONE block per CTA to the workspace; a second pass sums the remaining slices/128
// blocks in a fixed order (deterministic) and applies alpha, beta.
//
// The per-thread parts are host/device functions: tests/test_row_kernel_emulation.py runs them
// thread by thread on the CPU against numpy (the CTA tree is emulated there by summing 128
// consecutive threads; the second pass with the kernel's own lane sums and shuffle tree).
// Validated on a B200 in round 2 (tests/test_gpu_contraction.py).
#pragma once
#include "contract_row.hpp"

namespace sbb {
    namespace dotk {

        constexpr int GD = SBK_MAX_GROUP_DIMS;
        constexpr int FMAX = 16; // largest free group
        constexpr int SB = 4;    // a thread owns an SB x SB block of outputs
        constexpr int CTA = 128; // threads per CTA of the first pass = slices added inside a CTA

        struct DotParams {
            int nd_t;                                 ///< batch dims (first fastest)
            int size_t_[GD];
            long long sa_t[GD], sb_t[GD], sr_t[GD];
            long long tvol;
            int m, n;                                 ///< extents of the free groups (v0 x vr, v1 x vr)
            long long moff_a[FMAX], moff_r[FMAX], noff_b[FMAX], noff_r[FMAX];
            int nd_k;                                 ///< contracted dims (first fastest)
            int size_k[GD];
            long long sa_k[GD], sb_k[GD];
            long long kvol;
            int slices, pgm, pgn;                     ///< k slices and blocks of SB rows / SB columns
            int conj_a, conj_b;
        };

        SBB_HD long long threads_of(const DotParams &p) {
            return p.tvol * (long long)(p.pgm * p.pgn) * p.slices;
        }
        SBB_HD long long outputs_of(const DotParams &p) { return p.tvol * (long long)(p.m * p.n); }

        /// Pass 1, one thread: partial sums of its k slice for its SB x SB block
        template <typename T>
        SBB_HD void dot_partial_acc(const DotParams &p, long long thread, const T *va, const T *vb,
                                    typename Fast<T>::type (&acc)[SB][SB]) {
            using A = typename Fast<T>::type;
            const int slice = (int)(thread % p.slices);
            long long rem = thread / p.slices;
            const int pg = (int)(rem % (p.pgm * p.pgn));
            long long t = rem / (p.pgm * p.pgn);
            const int m0 = (pg / p.pgn) * SB, n0 = (pg % p.pgn) * SB;
            long long oa = 0, ob = 0;
#pragma unroll 1
            for (int d = 0; d < p.nd_t; ++d) {
                const long long c = t % p.size_t_[d];
                t /= p.size_t_[d];
                oa += c * p.sa_t[d], ob += c * p.sb_t[d];
            }
#pragma unroll
            for (int i = 0; i < SB; ++i)
#pragma unroll
                for (int j = 0; j < SB; ++j) set_zero(acc[i][j]);
            for (long long k = slice; k < p.kvol; k += p.slices) {
                long long ka, kb;
                if (p.nd_k == 1) {
                    ka = k * p.sa_k[0], kb = k * p.sb_k[0];
                } else {
                    long long r = k;
                    ka = kb = 0;
#pragma unroll 1
                    for (int d = 0; d < p.nd_k; ++d) {
                        const long long c = r % p.size_k[d];
                        r /= p.size_k[d];
                        ka += c * p.sa_k[d], kb += c * p.sb_k[d];
                    }
                }
                A a[SB], b[SB];
#pragma unroll
                for (int i = 0; i < SB; ++i) {
                    set_zero(a[i]);
                    if (m0 + i < p.m) {
                        a[i] = va[oa + ka + p.moff_a[m0 + i]];
                        if (p.conj_a) a[i] = cj(a[i]);
                    }
                }
#pragma unroll
                for (int j = 0; j < SB; ++j) {
                    set_zero(b[j]);
                    if (n0 + j < p.n) {
                        b[j] = vb[ob + kb + p.noff_b[n0 + j]];
                        if (p.conj_b) b[j] = cj(b[j]);
                    }
                }
#pragma unroll
                for (int i = 0; i < SB; ++i)
#pragma unroll
                    for (int j = 0; j < SB; ++j) fma_acc(acc[i][j], a[i], b[j]);
            }
        }

        /// Pass 1 without the CTA tree (slices not a multiple of 128): every thread writes its block
        template <typename T>
        SBB_HD void dot_partial(const DotParams &p, long long thread, const T *va, const T *vb,
                                typename Acc<T>::type *ws) {
            typename Fast<T>::type acc[SB][SB];
            dot_partial_acc<T>(p, thread, va, vb, acc);
            typename Acc<T>::type *out = ws + thread * (SB * SB);
#pragma unroll
            for (int i = 0; i < SB; ++i)
#pragma unroll
                for (int j = 0; j < SB; ++j) out[i * SB + j] = widen(acc[i][j]);
        }

        /// True when every CTA of the first pass holds 128 slices of one block of outputs, so that
        /// the CTA adds them itself; the workspace then holds slices / 128 blocks per output block
        SBB_HD bool cta_tree(const DotParams &p) { return p.slices % CTA == 0; }
        SBB_HD int ws_slices(const DotParams &p) { return cta_tree(p) ? p.slices / CTA : p.slices; }

        /// Pass 2: output `out` as (row mm, column nn, batch entry t), the column fastest
        struct Output {
            int nn, mm;
            long long t;
        };
        SBB_HD Output output_of(const DotParams &p, long long out) {
            Output o;
            o.nn = (int)(out % p.n);
            const long long rem = out / p.n;
            o.mm = (int)(rem % p.m);
            o.t = rem / p.m;
            return o;
        }

        /// Pass 2: the first of the nsl = ws_slices(p) workspace entries of an output (slice s at + s * SB * SB)
        template <typename A>
        SBB_HD const A *ws_column(const DotParams &p, const A *ws, int nsl, const Output &o) {
            const int pg = (o.mm / SB) * p.pgn + o.nn / SB;
            return ws + ((o.t * (p.pgm * p.pgn) + pg) * (long long)nsl) * (SB * SB) + (o.mm % SB) * SB + o.nn % SB;
        }

        /// Pass 2: offset of an output in the result
        SBB_HD long long result_offset(const DotParams &p, const Output &o) {
            long long orr = p.moff_r[o.mm] + p.noff_r[o.nn], t = o.t;
            for (int d = 0; d < p.nd_t; ++d) {
                const long long c = t % p.size_t_[d];
                t /= p.size_t_[d];
                orr += c * p.sr_t[d];
            }
            return orr;
        }

        /// Pass 2 of output `out` on the CPU, added in the kernel's order: lane l (of 32) sums the slices
        /// l, l + 32, ... from zero, then the lanes are folded by the shuffle tree (lane l += lane l + off
        /// for off = 16, 8, 4, 2, 1) and lane 0 applies alpha and beta
        template <typename T>
        inline void dot_reduce(const DotParams &p, long long out, const typename Acc<T>::type *ws, T *vr,
                               typename Acc<T>::type alpha, typename Acc<T>::type beta) {
            using A = typename Acc<T>::type;
            const int nsl = ws_slices(p);
            const Output o = output_of(p, out);
            const A *src = ws_column(p, ws, nsl, o);
            A v[32];
            for (int l = 0; l < 32; ++l) {
                set_zero(v[l]);
                for (int s = l; s < nsl; s += 32) v[l] = addc(v[l], src[(long long)s * (SB * SB)]);
            }
            for (int off = 16; off > 0; off >>= 1)
                for (int l = 0; l < off; ++l) v[l] = addc(v[l], v[l + off]);
            epilogue(vr, result_offset(p, o), v[0], alpha, beta);
        }

        // ---- host -----------------------------------------------------------------------------------

        inline bool eligible(const sbk_contract_desc &c) {
            const long long m = rowk::volume_of(c.M, c.nM), n = rowk::volume_of(c.N, c.nN),
                            k = rowk::volume_of(c.K, c.nK), t = rowk::volume_of(c.T, c.nT);
            return m >= 1 && n >= 1 && t >= 1 && k >= 1 && m <= FMAX && n <= FMAX;
        }

        /// `target_threads`: how many threads should be busy (a few per core of the machine)
        inline void build(const sbk_contract_desc &c, DotParams &p, long long target_threads) {
            if (!eligible(c)) throw std::runtime_error("dot kernel: shape not supported");
            std::memset(&p, 0, sizeof p);
            p.tvol = 1;
            for (int i = 0; i < c.nT; ++i)
                if (c.T[i].size > 1) {
                    const int d = p.nd_t++;
                    p.size_t_[d] = c.T[i].size, p.sa_t[d] = c.T[i].s0, p.sb_t[d] = c.T[i].s1,
                    p.sr_t[d] = c.T[i].sr;
                    p.tvol *= c.T[i].size;
                }
            p.kvol = 1;
            for (int i = 0; i < c.nK; ++i)
                if (c.K[i].size > 1) {
                    // merge with the previous contracted dim when both operands stay affine
                    if (p.nd_k > 0 && p.sa_k[p.nd_k - 1] * p.size_k[p.nd_k - 1] == c.K[i].s0 &&
                        p.sb_k[p.nd_k - 1] * p.size_k[p.nd_k - 1] == c.K[i].s1 &&
                        (long long)p.size_k[p.nd_k - 1] * c.K[i].size < (1ll << 31)) {
                        p.size_k[p.nd_k - 1] *= c.K[i].size;
                    } else {
                        const int d = p.nd_k++;
                        p.size_k[d] = c.K[i].size, p.sa_k[d] = c.K[i].s0, p.sb_k[d] = c.K[i].s1;
                    }
                    p.kvol *= c.K[i].size;
                }
            if (p.nd_k == 0) p.nd_k = 1, p.size_k[0] = 1; // a single term
            p.m = (int)rowk::volume_of(c.M, c.nM), p.n = (int)rowk::volume_of(c.N, c.nN);
            rowk::group_offsets(c.M, c.nM, 0, p.moff_a);
            rowk::group_offsets(c.M, c.nM, 2, p.moff_r);
            rowk::group_offsets(c.N, c.nN, 1, p.noff_b);
            rowk::group_offsets(c.N, c.nN, 2, p.noff_r);
            p.pgm = (p.m + SB - 1) / SB, p.pgn = (p.n + SB - 1) / SB;
            p.conj_a = c.conj0, p.conj_b = c.conj1;
            long long s = target_threads / (p.tvol * p.pgm * p.pgn);
            s = s / 32 * 32;
            if (s < 32) s = 32;
            if (s > 8192) s = 8192;
            if (s > p.kvol) s = p.kvol;
            if (s >= CTA) s = s / CTA * CTA; // whole CTAs per block of outputs (see cta_tree)
            p.slices = (int)s;
        }

    } // namespace dotk
} // namespace sbb
