// Contraction kernels for sm_100a:  vr = alpha * sum_K f0(v0) * f1(v1) + beta * vr
//
// Replaces the reference's lowering "permute both operands -> xgemm_batch_strided -> add-copy"
// (tensor.h:1271-1429 suggested_orders_for_contraction, tensor.h:1475-1598
// local_contraction_normalized, blas.h:662-810 cublasGemmStridedBatchedEx).  Here the operands are
// never re-laid-out: every label keeps its own stride (sbk_contract_desc) and the tile loaders
// gather straight from the caller's layout, so the permutation is fused into the GEMM.
//
// Kernels:
//  * contract_mma_kernel (double, complex double; float and complex float with their tiles kept in
//    float and widened at the fragment loads): FP64 tensor-core path.  tcgen05 has no f64 kind,
//    so on Blackwell FP64 matrix math is issued as warp-level DMMA (mma.sync.m8n8k4.f64).  A CTA
//    owns a 64x64 output tile of one batch entry and one K-slice; operands flow
//    global --cp.async (16 B per complex element, any stride)--> 4-stage shared-memory ring -->
//    LDS.128 fragments --> DMMA, a complex product being four real DMMAs (the sign of the
//    imaginary parts carries conj and the minus of i*i).  K is split across CTAs so that the grid
//    fills 148 SMs x 2 CTAs for several waves even when the output is a single tile per batch
//    entry (distillation shapes: M=N=64..128, K~1e5); partial tiles go to a workspace and
//  * contract_reduce_kernel sums them in a fixed order (deterministic), applies alpha/beta/output
//    strides (the reference's final add-copy, dist.h:3184, fused here).
//  * contract_simt_kernel: any type, any shape; one thread per output element, K loop in registers,
//    float types accumulate in double.  Used for short contractions (e.g. site-wise colour-spin
//    contractions with M=N=1) and small tiles with many outputs.
//  * contract_row_kernel / contract_row_smem_kernel (contract_row.hpp: short K and one small free
//    group; the small operand staged in shared memory when a CTA's rows share it) and
//    contract_dot_*_kernel (contract_dot.hpp: long K and two small free groups; CTA tree + a warp per
//    output in the second pass): the skinny shapes the reference hands to GEMV / dot calls
//    (blas.h:686-699).  Bodies also run on the CPU (tests/test_row_kernel_emulation.py).
//  * complex float with a long contiguous K goes to the tcgen05 kernel (kernels_contract_tc.cu).
#include "contract_dot.hpp"
#include "contract_row.hpp"
#include "contract_tc.hpp"
#include "kernels.hpp"
#include "runtime.hpp"
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <sstream>
#include <type_traits>
#include <vector>

namespace sbb {

    namespace {

        constexpr int GD = SBK_MAX_GROUP_DIMS;

        struct Group {
            int n;
            int size[GD];
            long long s0[GD], s1[GD], sr[GD];
            long long vol;
        };

        struct ContractParams {
            Group T, M, N, K;
            int conj0, conj1;
            int bn; // columns of an output tile of the mma kernel
            int out_order[3]; // generic kernel: groups (0 = T, 1 = M, 2 = N) from fastest to slowest thread index
            // mma kernel
            int mtiles, ntiles, ksplit, ksteps; // ksteps = ceil(K/BK)
            int a_sr, a_sk, b_sr, b_sk;         // shared-memory strides (elements) of the operand tiles
            int a_kfast, b_kfast;               // loader enumeration: 1 = k fastest, 0 = row fastest
        };

        __host__ __device__ inline long long group_offset(const Group &g, long long idx,
                                                          const long long *stride) {
            long long off = 0;
#pragma unroll
            for (int d = 0; d < GD; ++d)
                if (d < g.n) {
                    const long long c = idx % g.size[d];
                    idx /= g.size[d];
                    off += c * stride[d];
                }
            return off;
        }

        // ---- generic kernel ------------------------------------------------------------------------

        template <typename T>
        __global__ void __launch_bounds__(256)
            contract_simt_kernel(const __grid_constant__ ContractParams p, const T *__restrict__ v0,
                                 const T *__restrict__ v1, T *vr, typename Acc<T>::type alpha,
                                 typename Acc<T>::type beta) {
            using A = typename Acc<T>::type;
            const long long total = p.T.vol * p.M.vol * p.N.vol;
            for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
                 idx += (long long)gridDim.x * blockDim.x) {
                // output enumeration: the group with the smallest output stride fastest, so that the
                // stores are coalesced (default order: n fastest, then m, then t)
                long long n = idx % p.N.vol, m = (idx / p.N.vol) % p.M.vol,
                          t = idx / (p.N.vol * p.M.vol);
                if (p.out_order[0] != 2 || p.out_order[1] != 1)
                    rowk::output_index(p.out_order, p.T.vol, p.M.vol, p.N.vol, idx, t, m, n);
                const long long o0 = group_offset(p.T, t, p.T.s0) + group_offset(p.M, m, p.M.s0);
                const long long o1 = group_offset(p.T, t, p.T.s1) + group_offset(p.N, n, p.N.s1);
                const long long orr = group_offset(p.T, t, p.T.sr) + group_offset(p.M, m, p.M.sr) +
                                      group_offset(p.N, n, p.N.sr);
                A acc;
                set_zero(acc);
                if (p.K.n <= 1) {
                    const long long k0 = p.K.n ? p.K.s0[0] : 0, k1 = p.K.n ? p.K.s1[0] : 0;
                    for (long long k = 0; k < p.K.vol; ++k) {
                        A a = widen(v0[o0 + k * k0]), b = widen(v1[o1 + k * k1]);
                        if (p.conj0) a = cj(a);
                        if (p.conj1) b = cj(b);
                        fma_acc(acc, a, b);
                    }
                } else {
                    for (long long k = 0; k < p.K.vol; ++k) {
                        A a = widen(v0[o0 + group_offset(p.K, k, p.K.s0)]),
                          b = widen(v1[o1 + group_offset(p.K, k, p.K.s1)]);
                        if (p.conj0) a = cj(a);
                        if (p.conj1) b = cj(b);
                        fma_acc(acc, a, b);
                    }
                }
                epilogue(vr, orr, acc, alpha, beta);
            }
        }

        // ---- row kernel (short contraction, one small free group; body in contract_row.hpp) ----------

        template <typename T>
        __global__ void __launch_bounds__(128)
            contract_row_kernel(const __grid_constant__ rowk::RowParams p, const T *__restrict__ va,
                                const T *__restrict__ vb, T *vr, typename Acc<T>::type alpha,
                                typename Acc<T>::type beta) {
            for (long long row = blockIdx.x * (long long)blockDim.x + threadIdx.x; row < p.rows;
                 row += (long long)gridDim.x * blockDim.x)
                rowk::row_body<T>(p, row, va, vb, vr, alpha, beta);
        }

        /// The same with the small operand staged in shared memory: when the 128 rows of a CTA share
        /// one K x S block of it (`inner` = rows per block is a multiple of 128), the block is loaded
        /// once per CTA and every product reads it with a broadcast LDS instead of a load through L1
        /// (S x K loads per row: they, not the big operand, bound the kernel -- 49152 x 16 x 16
        /// "update" shapes ran at 14 % of the HBM floor).
        template <typename T>
        __global__ void __launch_bounds__(128)
            contract_row_smem_kernel(const __grid_constant__ rowk::RowParams p, const T *__restrict__ va,
                                     const T *__restrict__ vb, T *vr, typename Acc<T>::type alpha,
                                     typename Acc<T>::type beta) {
            using F = typename Fast<T>::type;
            __shared__ F sb[rowk::KMAX * rowk::SMAX];
            const long long nblocks = (p.rows + 127) / 128;
            for (long long blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
                const long long row = blk * 128 + threadIdx.x;
                // offsets of this row (the small operand's offset is the same for the whole CTA)
                long long oa = 0, ob = 0, orr = 0, rem = row < p.rows ? row : p.rows - 1;
#pragma unroll 1
                for (int d = 0; d < p.nd; ++d) {
                    const long long c = rem % p.size[d];
                    rem /= p.size[d];
                    oa += c * p.sa[d], ob += c * p.sb[d], orr += c * p.sr[d];
                }
                __syncthreads(); // the previous block's products are done with sb
                for (int i = threadIdx.x; i < p.nk * p.ns; i += 128) {
                    F b = vb[ob + p.koff_b[i / p.ns] + p.soff_b[i % p.ns]];
                    if (p.conj_b) b = cj(b);
                    sb[i] = b;
                }
                __syncthreads();
                if (row >= p.rows) continue;
                F acc[rowk::SMAX];
#pragma unroll
                for (int s = 0; s < rowk::SMAX; ++s) set_zero(acc[s]);
                constexpr int KB = 8;
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
                            const F *bk = sb + (k0 + j) * p.ns;
#pragma unroll
                            for (int s = 0; s < rowk::SMAX; ++s)
                                if (s < p.ns) fma_acc(acc[s], a[j], bk[s]);
                        }
                }
#pragma unroll
                for (int s = 0; s < rowk::SMAX; ++s)
                    if (s < p.ns) epilogue(vr + orr, p.soff_r[s], widen(acc[s]), alpha, beta);
            }
        }

        // ---- dot kernel (long contraction, both free groups small; bodies in contract_dot.hpp) -------

        __device__ __forceinline__ double shfl_down(double v, int off) { return __shfl_down_sync(0xffffffffu, v, off); }
        __device__ __forceinline__ double2 shfl_down(double2 v, int off) {
            return make_double2(__shfl_down_sync(0xffffffffu, v.x, off), __shfl_down_sync(0xffffffffu, v.y, off));
        }

        template <typename T>
        __global__ void __launch_bounds__(dotk::CTA)
            contract_dot_partial_kernel(const __grid_constant__ dotk::DotParams p,
                                        const T *__restrict__ va, const T *__restrict__ vb,
                                        typename Acc<T>::type *__restrict__ ws) {
            using A = typename Acc<T>::type;
            constexpr int SB = dotk::SB;
            const long long thread = blockIdx.x * (long long)blockDim.x + threadIdx.x;
            if (!dotk::cta_tree(p)) { // few slices: every thread writes its own block
                if (thread < dotk::threads_of(p)) dotk::dot_partial<T>(p, thread, va, vb, ws);
                return;
            }
            // the CTA holds 128 slices of the same outputs: add them here (fixed tree: deterministic)
            typename Fast<T>::type acc[SB][SB];
            dotk::dot_partial_acc<T>(p, thread, va, vb, acc);
            __shared__ A part[dotk::CTA / 32][SB * SB];
            const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
            // (only the live entries of the block: for m = n = 1 the 15 dead ones cost 300 shuffles
            // per thread, most of the kernel; the condition is uniform over the CTA)
            const int pgi = (int)((blockIdx.x / (p.slices / dotk::CTA)) % (p.pgm * p.pgn));
            const int mlive = min(SB, p.m - (pgi / p.pgn) * SB), nlive = min(SB, p.n - (pgi % p.pgn) * SB);
#pragma unroll
            for (int q = 0; q < SB * SB; ++q) {
                A v = widen(acc[q / SB][q % SB]);
                if (q / SB < mlive && q % SB < nlive) {
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) v = addc(v, shfl_down(v, off));
                }
                if (lane == 0) part[warp][q] = v;
            }
            __syncthreads();
            if (threadIdx.x < SB * SB) {
                A v = part[0][threadIdx.x];
#pragma unroll
                for (int w = 1; w < dotk::CTA / 32; ++w) v = addc(v, part[w][threadIdx.x]);
                ws[blockIdx.x * (long long)(SB * SB) + threadIdx.x] = v;
            }
        }

        /// Second pass of the dot kernel: one WARP per output -- the lanes stride over the slices left
        /// by the first pass and add their sums with a fixed shuffle tree (deterministic).  (One thread
        /// per output walked the slices one dependent load after the other: 38 of the 40 us of an
        /// m = n = 1, k = 49152, batch 32 call.)
        template <typename T>
        __global__ void __launch_bounds__(256)
            contract_dot_reduce_kernel(const __grid_constant__ dotk::DotParams p,
                                       const typename Acc<T>::type *__restrict__ ws, T *vr,
                                       typename Acc<T>::type alpha,
                                       typename Acc<T>::type beta) {
            using A = typename Acc<T>::type;
            constexpr int SB = dotk::SB;
            const long long total = dotk::outputs_of(p);
            const int lane = threadIdx.x & 31, nsl = dotk::ws_slices(p);
            const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
            for (long long out = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5; out < total;
                 out += nwarps) {
                const dotk::Output o = dotk::output_of(p, out);
                const A *src = dotk::ws_column(p, ws, nsl, o);
                A acc;
                set_zero(acc);
                for (int s = lane; s < nsl; s += 32) acc = addc(acc, src[(long long)s * (SB * SB)]);
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) acc = addc(acc, shfl_down(acc, off));
                if (lane == 0) epilogue(vr, dotk::result_offset(p, o), acc, alpha, beta);
            }
        }

        // ---- FP64 tensor-core kernel -----------------------------------------------------------------

        constexpr int BM = 64, MMA_THREADS = 128;
        // BN (tile columns), pipeline depth and resident CTAs are template parameters: 64/4/2 and 32/4/3 are built

        __device__ __forceinline__ void dmma(double &d0, double &d1, double a, double b) {
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                         : "+d"(d0), "+d"(d1)
                         : "d"(a), "d"(b));
        }

        template <int BYTES>
        __device__ __forceinline__ void cp_async(void *smem, const void *gmem, bool valid) {
            const unsigned saddr = (unsigned)__cvta_generic_to_shared(smem);
            const int src = valid ? BYTES : 0; // src-size 0: the destination is zero filled
            asm volatile("cp.async.ca.shared.global [%0], [%1], %2, %3;" ::"r"(saddr), "l"(gmem),
                         "n"(BYTES), "r"(src));
        }
        __device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
        template <int N> __device__ __forceinline__ void cp_async_wait() {
            asm volatile("cp.async.wait_group %0;" ::"n"(N));
        }

        template <typename T> struct Frag; // fragment element as loaded from shared memory
        template <> struct Frag<double> {
            static constexpr bool cplx = false;
        };
        template <> struct Frag<double2> {
            static constexpr bool cplx = true;
        };
        // float and complex float operands stay in their own type up to shared memory (half the HBM
        // and shared-memory traffic) and are widened when the fragments are read: the products and
        // the whole K sum are done by the FP64 tensor pipe, only the final result is rounded to float
        template <> struct Frag<float> {
            static constexpr bool cplx = false;
        };
        template <> struct Frag<float2> {
            static constexpr bool cplx = true;
        };

        /// Offset of contracted index k in an operand
        __device__ __forceinline__ long long k_offset(const Group &K, long long k,
                                                      const long long *stride) {
            if (K.n == 1) return k * stride[0];
            return group_offset(K, k, stride);
        }

        /// Shared-memory row stride of a k-contiguous operand tile ([row][k], see tile_layout)
        __host__ __device__ constexpr int kfast_row_stride(int bk) { return bk + 4; }

        /// Stage loader of contract_mma_kernel for any layout: 4 elements of A and 4 of B per thread
        /// and stage, each slot with its own source row, k and shared-memory offset.
        template <typename T, int BN, int BK> struct MmaLoader {
            static constexpr int A_SLOTS = BM * BK / MMA_THREADS, B_SLOTS = BN * BK / MMA_THREADS;
            const ContractParams &p;
            const T *a_base, *b_base;
            long long a_row[A_SLOTS], b_row[B_SLOTS];
            int a_kk[A_SLOTS], b_kk[B_SLOTS], a_sm[A_SLOTS], b_sm[B_SLOTS];
            const T *a_ptr[A_SLOTS], *b_ptr[B_SLOTS];
            long long a_step, b_step;

            __device__ MmaLoader(const ContractParams &p_, const T *a_base_, const T *b_base_, int tid,
                                 int mt, int nt, int kstep0, int a_stage)
                : p(p_), a_base(a_base_), b_base(b_base_) {
#pragma unroll
                for (int i = 0; i < A_SLOTS; ++i) {
                    const int slot = tid + i * MMA_THREADS;
                    const int r = p.a_kfast ? slot / BK : slot % BM, kk = p.a_kfast ? slot % BK : slot / BM;
                    const long long m = min((long long)mt * BM + r, p.M.vol - 1); // clamp: rows past M are never read back
                    a_row[i] = group_offset(p.M, m, p.M.s0);
                    a_kk[i] = kk;
                    a_sm[i] = r * p.a_sr + kk * p.a_sk;
                }
#pragma unroll
                for (int i = 0; i < B_SLOTS; ++i) {
                    const int slot = tid + i * MMA_THREADS;
                    const int r = p.b_kfast ? slot / BK : slot % BN, kk = p.b_kfast ? slot % BK : slot / BN;
                    const long long n = min((long long)nt * BN + r, p.N.vol - 1);
                    b_row[i] = group_offset(p.N, n, p.N.s1);
                    b_kk[i] = kk;
                    b_sm[i] = a_stage + r * p.b_sr + kk * p.b_sk;
                }
                // When the contracted labels merge into one dimension (the common case) every slot
                // walks its row with a constant pointer increment; otherwise the K offset is
                // decomposed per load.
                a_step = (p.K.n ? p.K.s0[0] : 0) * BK, b_step = (p.K.n ? p.K.s1[0] : 0) * BK;
#pragma unroll
                for (int i = 0; i < A_SLOTS; ++i)
                    a_ptr[i] = a_base + a_row[i] + ((long long)kstep0 * BK + a_kk[i]) * (p.K.n ? p.K.s0[0] : 0);
#pragma unroll
                for (int i = 0; i < B_SLOTS; ++i)
                    b_ptr[i] = b_base + b_row[i] + ((long long)kstep0 * BK + b_kk[i]) * (p.K.n ? p.K.s1[0] : 0);
            }

            /// Issue the cp.async of stage `kstep` into the slot at `s`
            __device__ __forceinline__ void operator()(T *s, int kstep, const T *, const T *) {
                const long long kbase = (long long)kstep * BK;
                if (p.K.n <= 1) {
                    // stages are loaded in k order, so the pointers simply advance
                    const bool tail = kbase + BK > p.K.vol;
#pragma unroll
                    for (int i = 0; i < A_SLOTS; ++i) {
                        const bool ok = !tail || kbase + a_kk[i] < p.K.vol;
                        cp_async<sizeof(T)>(s + a_sm[i], ok ? a_ptr[i] : a_base, ok);
                        a_ptr[i] += a_step;
                    }
#pragma unroll
                    for (int i = 0; i < B_SLOTS; ++i) {
                        const bool ok = !tail || kbase + b_kk[i] < p.K.vol;
                        cp_async<sizeof(T)>(s + b_sm[i], ok ? b_ptr[i] : b_base, ok);
                        b_ptr[i] += b_step;
                    }
                    return;
                }
#pragma unroll
                for (int i = 0; i < A_SLOTS; ++i) {
                    const long long k = kbase + a_kk[i];
                    const bool ok = k < p.K.vol;
                    const long long off = ok ? a_row[i] + k_offset(p.K, k, p.K.s0) : 0;
                    cp_async<sizeof(T)>(s + a_sm[i], a_base + off, ok);
                }
#pragma unroll
                for (int i = 0; i < B_SLOTS; ++i) {
                    const long long k = kbase + b_kk[i];
                    const bool ok = k < p.K.vol;
                    const long long off = ok ? b_row[i] + k_offset(p.K, k, p.K.s1) : 0;
                    cp_async<sizeof(T)>(s + b_sm[i], b_base + off, ok);
                }
            }
        };

        /// Stage loader for K-contiguous operands (the KC kernel).  Slot tid + 128 i of a thread holds
        /// row tid / BK + i * 128 / BK and k = tid % BK, so all slots of a thread share their k and one
        /// pointer per operand, advanced by BK per stage, reaches every source.  Rows past M (N) are
        /// clamped to the last row, as in MmaLoader; a thread's k past the end of K is zero filled.
        template <typename T, int BN, int BK> struct MmaLoaderKC {
            static constexpr int ROWS = MMA_THREADS / BK; // rows loaded per pass of the CTA
            static constexpr int A_SLOTS = BM / ROWS, B_SLOTS = BN / ROWS;
            static constexpr int SR = kfast_row_stride(BK), A_STAGE = BM * SR;
            static_assert(MMA_THREADS % BK == 0, "every slot of a thread has the same k");
            const T *a_ptr, *b_ptr;   // slot 0's source at the next stage
            long long a_rs, b_rs;     // row strides in global memory (0 for an empty row group)
            int a_lim, b_lim;         // rows after slot 0's that are inside M (N); further rows are clamped
            int sm;                   // shared-memory offset of slot 0 in the A tile (B: + A_STAGE)
            int kfull;                // stages without a K tail
            bool tail_ok;             // this thread's k is inside K in the partial last stage

            __device__ MmaLoaderKC(const ContractParams &p, const T *a_base, const T *b_base, int tid,
                                   int mt, int nt, int kstep0, int) {
                const int kk = tid % BK, r = tid / BK;
                a_rs = p.M.s0[0], b_rs = p.N.s1[0];
                const long long m = min((long long)mt * BM + r, p.M.vol - 1);
                const long long n = min((long long)nt * BN + r, p.N.vol - 1);
                a_lim = (int)min(p.M.vol - 1 - m, (long long)BM);
                b_lim = (int)min(p.N.vol - 1 - n, (long long)BN);
                a_ptr = a_base + m * a_rs + (long long)kstep0 * BK + kk;
                b_ptr = b_base + n * b_rs + (long long)kstep0 * BK + kk;
                sm = r * SR + kk;
                kfull = (int)(p.K.vol / BK);
                tail_ok = kk < (int)(p.K.vol % BK);
            }

            /// Issue the cp.async of stage `kstep` into the slot at `s`; a zero-filled element is
            /// "read" from the operand's start (v0, v1)
            __device__ __forceinline__ void operator()(T *s, int kstep, const T *v0, const T *v1) {
                const bool ok = kstep < kfull || tail_ok;
#pragma unroll
                for (int i = 0; i < A_SLOTS; ++i) {
                    const T *src = a_ptr + (i ? min(i * ROWS, a_lim) * a_rs : 0);
                    cp_async<sizeof(T)>(s + sm + i * ROWS * SR, ok ? src : v0, ok);
                }
#pragma unroll
                for (int i = 0; i < B_SLOTS; ++i) {
                    const T *src = b_ptr + (i ? min(i * ROWS, b_lim) * b_rs : 0);
                    cp_async<sizeof(T)>(s + A_STAGE + sm + i * ROWS * SR, ok ? src : v1, ok);
                }
                a_ptr += BK, b_ptr += BK;
            }
        };

        /// KC: both operands k-contiguous with one contracted label of stride 1 and at most one label
        /// per row group (launch_mma decides).  The shared-memory layout is then a compile-time
        /// constant and each operand is loaded through one pointer; every other layout runs KC = false.
        template <typename T, int BN, int BK, int STAGES, int MINB, bool KC>
        __global__ void __launch_bounds__(MMA_THREADS, MINB)
            contract_mma_kernel(const __grid_constant__ ContractParams p, const T *__restrict__ v0,
                                const T *__restrict__ v1, typename Acc<T>::type *__restrict__ ws) {
            using A = typename Acc<T>::type; // double or double2: what the partial tiles are stored as
            constexpr bool CPLX = Frag<T>::cplx;
            constexpr int ACC = CPLX ? 4 : 2; // doubles per 8x8 block per lane
            constexpr int WN = BN / 16;       // 8-column blocks per warp (warp tile = 32 x BN/2)
            constexpr int KB = BK / 4;        // k4 blocks per stage
            static_assert(KB % 2 == 0, "the fragment double buffer alternates within a stage");
            extern __shared__ __align__(16) unsigned char smem_raw[];
            // stage layout: [A tile | B tile], sizes fixed by the host (a_stage, b_stage elements)
            constexpr int KC_SR = kfast_row_stride(BK);
            const int a_sr = KC ? KC_SR : p.a_sr, a_sk = KC ? 1 : p.a_sk;
            const int b_sr = KC ? KC_SR : p.b_sr, b_sk = KC ? 1 : p.b_sk;
            const int a_stage = KC ? BM * KC_SR : p.a_kfast ? BM * p.a_sr : BK * p.a_sk;
            const int b_stage = KC ? BN * KC_SR : p.b_kfast ? BN * p.b_sr : BK * p.b_sk;
            T *smem = reinterpret_cast<T *>(smem_raw);
            const int stage_elems = a_stage + b_stage;

            const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
            const int wm = warp >> 1, wn = warp & 1; // 2x2 warps, 32 x BN/2 each

            // ---- which tile / K slice ------------------------------------------------------------
            long long bid = blockIdx.x;
            const int nt = (int)(bid % p.ntiles);
            bid /= p.ntiles;
            const int mt = (int)(bid % p.mtiles);
            bid /= p.mtiles;
            const int ks = (int)(bid % p.ksplit);
            const long long t = bid / p.ksplit;
            const int kstep0 = (int)((long long)p.ksteps * ks / p.ksplit);
            const int kstep1 = (int)((long long)p.ksteps * (ks + 1) / p.ksplit);
            const int nsteps = kstep1 - kstep0;

            const T *a_base = v0 + group_offset(p.T, t, p.T.s0);
            const T *b_base = v1 + group_offset(p.T, t, p.T.s1);

            using Loader = std::conditional_t<KC, MmaLoaderKC<T, BN, BK>, MmaLoader<T, BN, BK>>;
            Loader load = Loader(p, a_base, b_base, tid, mt, nt, kstep0, a_stage);
            auto load_stage = [&](int kstep) {
                load(smem + (size_t)((kstep - kstep0) % STAGES) * stage_elems, kstep, v0, v1);
            };

            // ---- accumulators: 4x4 blocks of 8x8 per warp ---------------------------------------------
            double acc[4][WN][ACC];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < WN; ++j)
#pragma unroll
                    for (int c = 0; c < ACC; ++c) acc[i][j][c] = 0.0;

            // fragment addresses inside a stage: element (row = base + lane/4, k = lane%4) of the
            // warp's first 8-row block; block i is 8 i rows further, k4 block kb is 4 kb k further
            const int a_frag = (wm * 32 + (lane >> 2)) * a_sr + (lane & 3) * a_sk;
            const int b_frag = a_stage + (wn * (BN / 2) + (lane >> 2)) * b_sr + (lane & 3) * b_sk;
            // raw fragments of a k4 block; with AHEAD (below) double buffered: block kb uses buffer kb % 2
            T fa[2][4], fb[2][WN];
            auto load_frags = [&](const T *s, int kb, T(&a)[4], T(&b)[WN]) {
#pragma unroll
                for (int i = 0; i < 4; ++i) a[i] = s[a_frag + i * 8 * a_sr + kb * 4 * a_sk];
#pragma unroll
                for (int j = 0; j < WN; ++j) b[j] = s[b_frag + j * 8 * b_sr + kb * 4 * b_sk];
            };
            // conj and the minus of i*i are sign flips of the imaginary fragments.  They are done on
            // the integer pipe (XOR of the sign bit): as FP64 multiplies / negations (8 per 64 DMMAs)
            // they shared the FP64 pipe with the DMMAs and drew 23 % of the stall samples
            // (profiles/r2_contract_mma_ncu.txt: DADD), with the tensor pipe at 88 %.
            const unsigned sa = p.conj0 ? 0x80000000u : 0u, sb = p.conj1 ? 0x80000000u : 0u;
            auto flip = [](double x, unsigned m) {
                return __hiloint2double(__double2hiint(x) ^ (int)m, __double2loint(x));
            };
            // the DMMAs of one k4 block, in the same order in both schedules
            auto mma_block = [&](const T(&fa)[4], const T(&fb)[WN]) {
                if constexpr (CPLX) {
                    double ar[4], ai[4], nai[4], br[WN], bi[WN];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const double2 a = widen(fa[i]);
                        ar[i] = a.x, ai[i] = flip(a.y, sa), nai[i] = flip(a.y, sa ^ 0x80000000u);
                    }
#pragma unroll
                    for (int j = 0; j < WN; ++j) {
                        const double2 b = widen(fb[j]);
                        br[j] = b.x, bi[j] = flip(b.y, sb);
                    }
                    // four passes over the 16 blocks: the two DMMAs that accumulate into the
                    // same registers are 32 instructions apart, so none waits for the other
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < WN; ++j) {
                            dmma(acc[i][j][0], acc[i][j][1], ar[i], br[j]);
                            dmma(acc[i][j][2], acc[i][j][3], ar[i], bi[j]);
                        }
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < WN; ++j) {
                            dmma(acc[i][j][0], acc[i][j][1], nai[i], bi[j]);
                            dmma(acc[i][j][2], acc[i][j][3], ai[i], br[j]);
                        }
                } else {
                    double a[4], b[WN];
#pragma unroll
                    for (int i = 0; i < 4; ++i) a[i] = widen(fa[i]);
#pragma unroll
                    for (int j = 0; j < WN; ++j) b[j] = widen(fb[j]);
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < WN; ++j) dmma(acc[i][j][0], acc[i][j][1], a[i], b[j]);
                }
            };

            // ---- pipeline -----------------------------------------------------------------------------
            // Stage kstep0 + it lives in slot it % STAGES, and commit group g holds stage kstep0 + g
            // (empty past the end of the slice).  The loads of stage it+STAGES-1 go to the slot of
            // stage it-1.
            // Invariant: cp.async overwrites a slot only after a barrier that every warp reaches after
            // its last LDS from that slot.
            //  * generic: the barrier at the top of iteration it follows every LDS of stage it-1, and
            //    the loads are issued after it.  There groups 0..it+STAGES-2 have been committed and
            //    stage it must have landed: STAGES-2 groups may stay in flight.
            //  * KC (AHEAD): the fragments of the next k4 block are read before the DMMAs of the
            //    current one, so no LDS sits between a barrier and the DMMAs after it; the registers
            //    freed by the KC loader pay for the second fragment buffer (the generic kernel would
            //    spill).  The barrier comes before the last k4 block of stage it, after the warp's
            //    last LDS of stage it and before its first LDS of stage it+1.  Stage it-1 was last read
            //    before the barrier of iteration it-1, so the loads can be issued at the start of
            //    iteration it.  At the barrier of iteration it, groups 0..it+STAGES-1 have been
            //    committed and stage it+1 must have landed: STAGES-2 groups may stay in flight.
            constexpr bool AHEAD = KC;
            auto load_ahead = [&](int it) {
                const int ahead = it + STAGES - 1;
                if (ahead < nsteps) load_stage(kstep0 + ahead);
                cp_async_commit();
            };
#pragma unroll
            for (int s = 0; s < STAGES - 1; ++s) {
                if (s < nsteps) load_stage(kstep0 + s);
                cp_async_commit();
            }
            if constexpr (AHEAD) {
                cp_async_wait<STAGES - 2>();
                __syncthreads();
                load_frags(smem, 0, fa[0], fb[0]);
            }
            for (int it = 0; it < nsteps; ++it) {
                const T *s = smem + (size_t)(it % STAGES) * stage_elems;
                if constexpr (!AHEAD) {
                    cp_async_wait<STAGES - 2>();
                    __syncthreads();
                }
#pragma unroll
                for (int kb = 0; kb < KB; ++kb) {
                    if constexpr (AHEAD) {
                        const int cur = kb % 2, nxt = cur ^ 1;
                        if (kb + 1 < KB) {
                            load_frags(s, kb + 1, fa[nxt], fb[nxt]);
                        } else if (it + 1 < nsteps) {
                            cp_async_wait<STAGES - 2>();
                            __syncthreads();
                            load_frags(smem + (size_t)((it + 1) % STAGES) * stage_elems, 0, fa[nxt], fb[nxt]);
                        }
                        if (kb == 0) load_ahead(it);
                        mma_block(fa[cur], fb[cur]);
                    } else {
                        // the loads are issued in the shadow of the first block of DMMAs
                        if (kb == (KB > 1 ? 1 : 0)) load_ahead(it);
                        load_frags(s, kb, fa[0], fb[0]);
                        mma_block(fa[0], fb[0]);
                    }
                }
            }
            cp_async_wait<0>();

            // ---- partial tile to the workspace: ws[((t*mt*nt tile) * ksplit + ks)][m][n] -------------
            const long long tile_id = ((t * p.mtiles + mt) * p.ntiles + nt) * p.ksplit + ks;
            A *out = ws + tile_id * (long long)(BM * BN);
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < WN; ++j) {
                    const int row = wm * 32 + i * 8 + (lane >> 2);
                    const int col = wn * (BN / 2) + j * 8 + (lane & 3) * 2;
                    if constexpr (CPLX) {
                        double4 v0 = make_double4(acc[i][j][0], acc[i][j][2], acc[i][j][1],
                                                  acc[i][j][3]);
                        *reinterpret_cast<double4 *>(out + row * BN + col) = v0;
                    } else {
                        *reinterpret_cast<double2 *>(out + row * BN + col) =
                            make_double2(acc[i][j][0], acc[i][j][1]);
                    }
                }
        }

        /// Sum the K-slices of every output tile in a fixed order and write alpha*sum + beta*vr
        template <typename T>
        __global__ void __launch_bounds__(256)
            contract_reduce_kernel(const __grid_constant__ ContractParams p,
                                   const typename Acc<T>::type *__restrict__ ws, T *vr,
                                   typename Acc<T>::type alpha, typename Acc<T>::type beta) {
            using A = typename Acc<T>::type;
            const long long total = p.T.vol * p.M.vol * p.N.vol;
            for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
                 idx += (long long)gridDim.x * blockDim.x) {
                const long long n = idx % p.N.vol, m = (idx / p.N.vol) % p.M.vol,
                                t = idx / (p.N.vol * p.M.vol);
                const int BN = p.bn;
                const int mt = (int)(m / BM), nt = (int)(n / BN);
                const long long tile0 = ((t * p.mtiles + mt) * p.ntiles + nt) * p.ksplit;
                const A *src = ws + tile0 * (long long)(BM * BN) + (m % BM) * BN + (n % BN);
                A acc = src[0];
                for (int s = 1; s < p.ksplit; ++s) acc = addc(acc, src[(long long)s * BM * BN]);
                const long long orr = group_offset(p.T, t, p.T.sr) + group_offset(p.M, m, p.M.sr) +
                                      group_offset(p.N, n, p.N.sr);
                epilogue(vr, orr, acc, alpha, beta);
            }
        }

        // ---- host ----------------------------------------------------------------------------------

        /// Copy one label group, dropping extent-1 labels and merging neighbours that stay affine in
        /// every tensor; dims are sorted by the stride in `key` (0: s0, 1: s1, 2: sr)
        Group make_group(const sbk_contract_dim *d, int n, int key) {
            std::vector<sbk_contract_dim> v;
            for (int i = 0; i < n; ++i) {
                if (d[i].size <= 0) {
                    Group g;
                    std::memset(&g, 0, sizeof g);
                    g.vol = 0;
                    return g;
                }
                if (d[i].size > 1) v.push_back(d[i]);
            }
            auto keyof = [&](const sbk_contract_dim &x) { return key == 0 ? x.s0 : key == 1 ? x.s1 : x.sr; };
            std::stable_sort(v.begin(), v.end(), [&](const sbk_contract_dim &a, const sbk_contract_dim &b) {
                return keyof(a) < keyof(b);
            });
            std::vector<sbk_contract_dim> m;
            for (const auto &x : v) {
                if (!m.empty()) {
                    auto &l = m.back();
                    const long long s = l.size;
                    if (l.s0 * s == x.s0 && l.s1 * s == x.s1 && l.sr * s == x.sr &&
                        s * (long long)x.size < (1ll << 31)) {
                        l.size *= x.size;
                        continue;
                    }
                }
                m.push_back(x);
            }
            if ((int)m.size() > GD) throw std::runtime_error("contraction: too many labels in a group");
            Group g;
            std::memset(&g, 0, sizeof g);
            g.n = (int)m.size();
            g.vol = 1;
            for (int i = 0; i < g.n; ++i) {
                g.size[i] = m[i].size, g.s0[i] = m[i].s0, g.s1[i] = m[i].s1, g.sr[i] = m[i].sr;
                g.vol *= m[i].size;
            }
            return g;
        }

        template <typename T>
        void launch_row(const rowk::RowParams &rp, bool swapped, const double *alpha, const void *v0,
                        const void *v1, const double *beta, void *vr, int device, cudaStream_t stream,
                        std::string *describe) {
            if (describe) {
                std::stringstream ss;
                ss << "row rows=" << rp.rows << " small=" << rp.ns << " K=" << rp.nk
                   << " big_operand=" << (swapped ? "v1" : "v0");
                *describe = ss.str();
                return;
            }
            const unsigned grid =
                (unsigned)std::min<long long>((rp.rows + 127) / 128, (long long)sm_count(device) * 12);
            // rows that share one block of the small operand: the leading row dims it does not depend on
            long long inner = 1;
            for (int d = 0; d < rp.nd && rp.sb[d] == 0; ++d) inner *= rp.size[d];
            if (inner % 128 == 0 && rp.ns * rp.nk >= 4)
                contract_row_smem_kernel<T><<<grid, 128, 0, stream>>>(rp, (const T *)(swapped ? v1 : v0),
                                                                     (const T *)(swapped ? v0 : v1), (T *)vr,
                                                                     scalar_of<T>(alpha), scalar_of<T>(beta));
            else
                contract_row_kernel<T><<<grid, 128, 0, stream>>>(rp, (const T *)(swapped ? v1 : v0),
                                                                (const T *)(swapped ? v0 : v1), (T *)vr,
                                                                scalar_of<T>(alpha), scalar_of<T>(beta));
            count_launch();
            cuda_check(cudaGetLastError(), "contract_row_kernel launch");
        }

        template <typename T>
        void launch_dot(const dotk::DotParams &dp, const double *alpha, const void *v0, const void *v1,
                        const double *beta, void *vr, int device, cudaStream_t stream,
                        std::string *describe) {
            if (describe) {
                std::stringstream ss;
                ss << "dot T=" << dp.tvol << " M=" << dp.m << " N=" << dp.n << " K=" << dp.kvol
                   << " slices=" << dp.slices << " blocks=" << dp.pgm << "x" << dp.pgn;
                *describe = ss.str();
                return;
            }
            using A = typename Acc<T>::type;
            const long long threads = dotk::threads_of(dp);
            PoolGuard guard;
            A *ws = (A *)guard.alloc(device, (size_t)threads * dotk::SB * dotk::SB * sizeof(A));
            contract_dot_partial_kernel<T><<<(unsigned)((threads + dotk::CTA - 1) / dotk::CTA), dotk::CTA, 0, stream>>>(
                dp, (const T *)v0, (const T *)v1, ws);
            count_launch();
            cuda_check(cudaGetLastError(), "contract_dot_partial_kernel launch");
            const long long outs = dotk::outputs_of(dp); // one warp each
            const unsigned grid =
                (unsigned)std::min<long long>((outs * 32 + 255) / 256, (long long)sm_count(device) * 8);
            contract_dot_reduce_kernel<T><<<grid, 256, 0, stream>>>(dp, ws, (T *)vr, scalar_of<T>(alpha),
                                                                  scalar_of<T>(beta));
            count_launch();
            cuda_check(cudaGetLastError(), "contract_dot_reduce_kernel launch");
        }

        template <typename T>
        void launch_simt(const ContractParams &p, const double *alpha, const void *v0, const void *v1,
                         const double *beta, void *vr, int device, cudaStream_t stream,
                         std::string *describe) {
            if (describe) {
                std::stringstream ss;
                ss << "simt T=" << p.T.vol << " M=" << p.M.vol << " N=" << p.N.vol << " K=" << p.K.vol;
                *describe = ss.str();
                return;
            }
            const long long total = p.T.vol * p.M.vol * p.N.vol;
            const unsigned grid =
                (unsigned)std::min<long long>((total + 255) / 256, (long long)sm_count(device) * 16);
            contract_simt_kernel<T><<<grid, 256, 0, stream>>>(p, (const T *)v0, (const T *)v1, (T *)vr,
                                                             scalar_of<T>(alpha), scalar_of<T>(beta));
            count_launch();
            cuda_check(cudaGetLastError(), "contract_simt_kernel launch");
        }

        /// Shared-memory layout of an operand tile: k-contiguous operands are stored [row][k] with
        /// row stride = BK + pad, row-contiguous operands [k][row]; the pads make the fragment
        /// LDS conflict free (see the derivation in DESIGN.md).
        void tile_layout(bool kfast, int esize, int rows, int bk, int &sr, int &sk) {
            if (kfast) {
                sr = kfast_row_stride(bk); // 12: = 4 mod 8 (16 B elements), in {4,12} mod 16 (8 B) and in {12,20} mod 32 (4 B)
                sk = 1;
            } else {
                sk = rows + (esize == 16 ? 2 : esize == 8 ? 4 : 8); // = 2 mod 8, 4 mod 16, 8 mod 32 elements
                sr = 1;
            }
        }

        template <typename T, int BN, int BK, int STAGES, int MINB>
        void launch_mma(ContractParams p, const double *alpha, const void *v0, const void *v1,
                        const double *beta, void *vr, int device, cudaStream_t stream,
                        std::string *describe) {
            using A = typename Acc<T>::type;
            p.bn = BN;
            p.mtiles = (int)((p.M.vol + BM - 1) / BM);
            p.ntiles = (int)((p.N.vol + BN - 1) / BN);
            p.ksteps = (int)((p.K.vol + BK - 1) / BK);
            // operand enumeration: follow the contiguous direction in global memory
            p.a_kfast = p.K.n > 0 && (p.M.n == 0 || p.K.s0[0] <= p.M.s0[0]);
            p.b_kfast = p.K.n > 0 && (p.N.n == 0 || p.K.s1[0] <= p.N.s1[0]);
            tile_layout(p.a_kfast, sizeof(T), BM, BK, p.a_sr, p.a_sk);
            tile_layout(p.b_kfast, sizeof(T), BN, BK, p.b_sr, p.b_sk);
            const int a_stage = p.a_kfast ? BM * p.a_sr : BK * p.a_sk;
            const int b_stage = p.b_kfast ? BN * p.b_sr : BK * p.b_sk;
            const size_t smem = (size_t)(a_stage + b_stage) * STAGES * sizeof(T);

            // K split: fill the machine for several waves, keep every slice long
            const long long tiles = p.T.vol * p.mtiles * p.ntiles;
            const long long slots = (long long)sm_count(device, describe != nullptr) * MINB;
            int best = 1;
            double best_eff = -1;
            const int smax = std::max(1, p.ksteps / 32);
            for (int s = 1; s <= smax && s <= 1024; ++s) {
                const long long ctas = tiles * s;
                const long long waves = (ctas + slots - 1) / slots;
                double eff = (double)ctas / (double)(waves * slots);
                if (waves >= 6) eff += 1e-3; // prefer enough waves to hide the ragged tail
                if (eff > best_eff + 1e-9) best_eff = eff, best = s;
                if (waves >= 16) break;
            }
            p.ksplit = best;
            const long long ctas = tiles * p.ksplit;
            if (ctas >= (1ll << 31)) throw std::runtime_error("contraction: grid too large");
            if (describe) {
                std::stringstream ss;
                ss << "mma f64" << (sizeof(A) != sizeof(T) ? " (float operands)" : "") << " tile=" << BM << "x" << BN << "x" << BK << " stages=" << STAGES
                   << " T=" << p.T.vol << " M=" << p.M.vol << " N=" << p.N.vol << " K=" << p.K.vol
                   << " ksplit=" << p.ksplit << " ctas=" << ctas << " smem=" << smem
                   << " a_kfast=" << p.a_kfast << " b_kfast=" << p.b_kfast << " loader=cp.async";
                *describe = ss.str();
                return;
            }
            PoolGuard guard;
            A *ws = (A *)guard.alloc(device, (size_t)ctas * BM * BN * sizeof(A));
            // K-contiguous operands (the distillation shapes) run the KC instantiation, whose tile
            // layout is fixed at compile time; it must match tile_layout above
            const bool kc = p.a_kfast && p.b_kfast && p.K.n == 1 && p.K.s0[0] == 1 && p.K.s1[0] == 1 &&
                            p.M.n <= 1 && p.N.n <= 1;
            auto *kernel = kc ? contract_mma_kernel<T, BN, BK, STAGES, MINB, true>
                              : contract_mma_kernel<T, BN, BK, STAGES, MINB, false>;
            static size_t attr_smem[2][64] = {};
            if (smem > attr_smem[kc][device]) {
                cuda_check(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                           "cudaFuncSetAttribute");
                attr_smem[kc][device] = smem;
            }
            {
                KernelTimer timer("contract_mma", stream);
                kernel<<<(unsigned)ctas, MMA_THREADS, smem, stream>>>(p, (const T *)v0, (const T *)v1, ws);
            }
            count_launch();
            cuda_check(cudaGetLastError(), "contract_mma_kernel launch");
            const long long total = p.T.vol * p.M.vol * p.N.vol;
            const unsigned grid =
                (unsigned)std::min<long long>((total + 255) / 256, (long long)sm_count(device) * 8);
            contract_reduce_kernel<T><<<grid, 256, 0, stream>>>(p, ws, (T *)vr, scalar_of<T>(alpha),
                                                               scalar_of<T>(beta));
            count_launch();
            cuda_check(cudaGetLastError(), "contract_reduce_kernel launch");
        }

        /// SBB_CONTRACT_KERNEL = simt | mma | tc | row | dot forces a path (tests); read on every call
        enum class Forced { None, Simt, Mma, Tc, Row, Dot, Other };

        Forced forced_kernel() {
            const char *e = std::getenv("SBB_CONTRACT_KERNEL");
            if (!e) return Forced::None;
            const std::string f = e;
            return f == "simt" ? Forced::Simt : f == "mma" ? Forced::Mma : f == "tc" ? Forced::Tc
                   : f == "row" ? Forced::Row : f == "dot" ? Forced::Dot : Forced::Other;
        }

        /// The kernel a contraction takes and the parameters it runs (or is described) with
        struct Choice {
            enum Path { Empty, Tc, Dot, Row, Mma, Simt } path;
            ContractParams p;   ///< mma, simt
            tc::Problem tp;     ///< tc
            dotk::DotParams dp; ///< dot
            rowk::RowParams rp; ///< row
            bool swapped;       ///< row: the big operand is v1
        };

        /// The paths are tried in the order empty, tc, dot, row, mma, simt.  A forced tc, dot or row
        /// kernel that cannot take the problem, and a value that names no kernel, leave the choice
        /// between mma and simt to the default rule.  `describe`: v0 and v1 are not real operands.
        Choice choose(const sbk_contract_desc &desc, int dtype, const void *v0, const void *v1, int device,
                      bool describe) {
            Choice c;
            std::memset(&c, 0, sizeof c);
            ContractParams &p = c.p;
            p.T = make_group(desc.T, desc.nT, 2);
            p.M = make_group(desc.M, desc.nM, 0);
            p.N = make_group(desc.N, desc.nN, 1);
            p.K = make_group(desc.K, desc.nK, 0);
            p.conj0 = desc.conj0 != 0, p.conj1 = desc.conj1 != 0;
            if (p.T.vol == 0 || p.M.vol == 0 || p.N.vol == 0) {
                c.path = Choice::Empty;
                return c;
            }
            // An empty contracted range leaves vr = beta*vr: the generic kernel handles K.vol == 0
            const Forced force = forced_kernel();
            const bool forced = force != Forced::None;
            // The tensor-core kernel wants a real tile (M, N >= 8, M*N >= 256) -- or a long contraction
            // with few outputs ("inner product" shapes, e.g. m = n = 1..12, k = 49152 of the reference's
            // tests/dist.cpp): there the generic kernel has one thread per output and no parallelism
            // over K, while the split-K of the tensor-core kernel fills the machine (the rows of the
            // 64x64 tile beyond M, N are clamped re-reads of the last row: wasted DMMA work, but the
            // operands are still read once).  The forced-"mma" parity tests cover tiny M and N.
            const long long outputs = p.T.vol * p.M.vol * p.N.vol;
            bool use_mma = p.K.vol >= 64 &&
                           ((p.M.vol * p.N.vol >= 256 && p.M.vol >= 8 && p.N.vol >= 8) ||
                            (p.K.vol >= 2048 && outputs < 148ll * 2048));
            if (force == Forced::Simt) use_mma = false;
            if (force == Forced::Mma && p.K.vol > 0) use_mma = true;
            // Complex float with real tiles and a long, contiguous contracted index: the tcgen05 path
            // (TF32 x 3 split, FP32 accumulation in tensor memory; kernels_contract_tc.cu).  The FP64
            // tensor-pipe kernel stays the path for everything else (and SBB_CONTRACT_KERNEL=mma
            // selects it for the accuracy comparison in the tests).
            if (dtype == SBB_C64 && (!forced || force == Forced::Tc) && p.K.n == 1 &&
                p.K.s0[0] == 1 && p.K.s1[0] == 1 && p.M.n <= 1 && p.N.n <= 1 && p.T.n <= 2 &&
                p.K.vol >= 256 && p.M.vol >= 16 && p.N.vol >= 16 && p.M.vol < (1 << 30) && p.N.vol < (1 << 30)) {
                tc::Problem &tp = c.tp;
                tp.nT = p.T.n;
                for (int d = 0; d < p.T.n; ++d)
                    tp.T[d] = tc::Dim{p.T.size[d], p.T.s0[d], p.T.s1[d], p.T.sr[d]};
                tp.M = tc::Dim{(int)p.M.vol, p.M.n ? p.M.s0[0] : 0, 0, p.M.n ? p.M.sr[0] : 0};
                tp.N = tc::Dim{(int)p.N.vol, 0, p.N.n ? p.N.s1[0] : 0, p.N.n ? p.N.sr[0] : 0};
                tp.K = p.K.vol, tp.conj0 = p.conj0, tp.conj1 = p.conj1;
                // (a description assumes 16-byte aligned operands)
                const void *a = describe ? (const void *)16 : v0, *b = describe ? (const void *)16 : v1;
                if (tc::eligible(tp, a, b)) {
                    c.path = Choice::Tc;
                    return c;
                }
            }
            // Small-tile regimes (validated on a B200 in round 2; bodies also checked on the CPU by
            // tests/test_row_kernel_emulation.py): long contractions whose free groups are both small go
            // to the dot kernel, short contractions with one small free group to the row kernel.
            if ((!forced || force == Forced::Dot) && (forced || p.K.vol >= 1024) && dotk::eligible(desc)) {
                dotk::build(desc, c.dp, (long long)sm_count(device, describe) * 2048);
                // (bounds the workspace: 2 bytes per thread with the CTA tree, 256 without)
                if (dotk::threads_of(c.dp) <= (dotk::cta_tree(c.dp) ? (1ll << 26) : (1ll << 20))) {
                    c.path = Choice::Dot;
                    return c;
                }
            }
            if ((!forced || force == Forced::Row) && (forced || !use_mma) && rowk::eligible(desc)) {
                rowk::build(desc, c.rp, c.swapped);
                c.path = Choice::Row;
                return c;
            }
            if (use_mma) {
                c.path = Choice::Mma;
                return c;
            }
            // enumerate the outputs along the smallest result stride, so that the stores coalesce
            auto min_sr = [](const Group &g) {
                long long s = 1ll << 62;
                for (int d = 0; d < g.n; ++d) s = std::min(s, g.sr[d] < 0 ? -g.sr[d] : g.sr[d]);
                return s;
            };
            const long long key[3] = {min_sr(p.T), min_sr(p.M), min_sr(p.N)};
            rowk::output_order(key, p.out_order);
            c.path = Choice::Simt;
            return c;
        }

        /// Launch the chosen kernel on operands of type T, or describe it
        template <typename T>
        void run(const Choice &c, const double *alpha, const void *v0, const void *v1, const double *beta,
                 void *vr, int device, cudaStream_t stream, std::string *describe) {
            switch (c.path) {
            case Choice::Empty:
                if (describe) *describe = "empty";
                return;
            case Choice::Tc: return tc::launch_c64(c.tp, alpha, v0, v1, beta, vr, device, stream, describe);
            case Choice::Dot: return launch_dot<T>(c.dp, alpha, v0, v1, beta, vr, device, stream, describe);
            case Choice::Row:
                return launch_row<T>(c.rp, c.swapped, alpha, v0, v1, beta, vr, device, stream, describe);
            case Choice::Mma:
                // 64x64 tile, BK = 8, 4 stages, 2 CTAs per SM (round 1 also measured 64x32 with 3 CTAs per
                // SM, BK = 16 with 2 stages and a cp.async.bulk row loader: all slower, removed)
                return launch_mma<T, 64, 8, 4, 2>(c.p, alpha, v0, v1, beta, vr, device, stream, describe);
            case Choice::Simt: return launch_simt<T>(c.p, alpha, v0, v1, beta, vr, device, stream, describe);
            }
        }

    } // namespace

    int sm_count(int device, bool describe_only) {
        static int sms[64] = {0};
        if (device < 0 || device >= 64) throw std::runtime_error("invalid device");
        if (!sms[device]) {
            int n = 0;
            const cudaError_t e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device);
            if (e != cudaSuccess && describe_only) {
                cudaGetLastError();
                return 148; // B200; not remembered: a real launch must ask the device
            }
            cuda_check(e, "cudaDeviceGetAttribute");
            sms[device] = n;
        }
        return sms[device];
    }

    void contract(const sbk_contract_desc &desc, int dtype, const double *alpha, const void *v0,
                  const void *v1, const double *beta, void *vr, int device, cudaStream_t stream,
                  std::string *describe) {
        if (dtype != SBB_F32 && dtype != SBB_F64 && dtype != SBB_C64 && dtype != SBB_C128)
            throw std::runtime_error("contraction: unsupported type");
        if (desc.nT > GD || desc.nM > GD || desc.nN > GD || desc.nK > GD || desc.nT < 0 ||
            desc.nM < 0 || desc.nN < 0 || desc.nK < 0)
            throw std::runtime_error("contraction: too many labels in a group");
        const Choice c = choose(desc, dtype, v0, v1, device, describe != nullptr);
        switch (dtype) {
        case SBB_F32: return run<float>(c, alpha, v0, v1, beta, vr, device, stream, describe);
        case SBB_F64: return run<double>(c, alpha, v0, v1, beta, vr, device, stream, describe);
        case SBB_C64: return run<float2>(c, alpha, v0, v1, beta, vr, device, stream, describe);
        case SBB_C128: return run<double2>(c, alpha, v0, v1, beta, vr, device, stream, describe);
        }
    }

} // namespace sbb
