// Complex-float contraction on the 5th-generation tensor cores of sm_100a.
//
//   vr[t,m,n] = alpha * sum_k f0(v0[t,m,k]) * f1(v1[t,n,k]) + beta * vr[t,m,n]      (k contiguous)
//
// Reference semantics: the complex-float GEMM of xgemm_batch_strided, computed by cuBLAS in
// CUBLAS_COMPUTE_32F (blas.h:559-565, :766).  Here:
//
//  * A complex product is four real products.  The operands are de-interleaved on the fly into
//    A' = [Re v0; Im v0] (2 x 64 rows) and B' = [Re v1; Im v1] (2 x 64 rows), so that ONE real
//    128 x 128 x K product A' B'^T holds all four blocks (rr, ri, ir, ii) of a 64 x 64 complex tile.
//  * FP32 accuracy from TF32 tensor cores: every element is split x = hi + lo with hi, lo exactly
//    representable in TF32 (hi = x rounded to the nearest TF32 value, lo = x - hi, exact in FP32,
//    rounded the same way) and D += Ahi Bhi + Ahi Blo + Alo Bhi accumulates in FP32 in tensor
//    memory; the dropped lo*lo term and the rounding of lo are O(2^-23) relative.
//  * Measured on B200: the FP32 accumulation inside tcgen05.mma is much less accurate than an IEEE
//    add -- every instruction that adds into a NON-ZERO accumulator leaves an error of about
//    2^-19 |accumulator| (relative error of a chain of n instructions ~ 1.9e-6 sqrt(n/2); the first
//    version of this kernel, one chain of 4096 instructions per CTA, was off by 8e-5).  So the
//    tensor core only sums SHORT chains: the hi*hi products go to an accumulator H that is drained
//    ("promoted") every `promote` stages by eight accumulation warps, which keep the running sums in
//    FP32 registers (IEEE adds on the CUDA cores); H is double buffered in TMEM so that the tensor
//    core never waits for the drain.  The hi*lo + lo*hi products, 2^-11 smaller, accumulate in a
//    third TMEM region S for the whole K slice (their accumulation error is 2^-11 smaller too).
//    K is also split across CTAs and the slices are summed in double by the reduce kernel.
//  * Data path per CTA (one 64 x 64 complex tile of one batch entry and one K slice; 1 CTA per SM):
//      TMA (cp.async.bulk.tensor, 64 rows x 32 complex per operand) -> raw ring (3 stages)
//      -> 8 transform warps (LDS.128 / split / STS.128 into the K-major SWIZZLE_128B layout the
//         tensor core reads) -> operand ring (2 stages x {Ahi, Alo, Bhi, Blo})
//      -> 1 thread issues tcgen05.mma.kind::tf32 (M = N = 128, K = 8 per instruction, 12 per stage)
//      -> 128 x 128 FP32 accumulators in TMEM (H[2], S) -> tcgen05.ld by 8 accumulation warps
//         -> FP32 running sums in registers -> workspace.
//    All hand-offs are mbarriers (TMA transaction counts, tcgen05.commit); no __syncthreads in the
//    main loop.
//  * contract_tc_reduce_kernel sums the K slices in a fixed order in double, combines the four
//    blocks into the complex result with the conj flags as signs, applies alpha, beta and the
//    output strides (the reference's final add-copy, fused).
//
// Roofline: the operands are read once (HBM floor: bytes / 6.5 TB/s); the tensor work is 3 x the
// algorithmic flop count at TF32 rate.  DESIGN.md §4.2b has the numbers.
#include "contract_tc.hpp"
#include "runtime.hpp"
#include <cuda.h>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <sstream>

namespace sbb {
    namespace tc {

        namespace {

            constexpr int TM = 64, TN = 64;         // complex tile
            constexpr int BKC = 32;                 // complex k per stage (= 32 TF32 per tile row = 128 B)
            constexpr int RAW_STAGES = 3, OP_STAGES = 2;
            constexpr int RAW_TILE = TM * BKC * 8;  // bytes of one operand's raw tile (16 KB)
            constexpr int OP_TILE = 128 * BKC * 4;  // bytes of one de-interleaved tile (128 rows x 128 B)
            constexpr int RAW_STAGE = 2 * RAW_TILE, OP_STAGE = 4 * OP_TILE;
            constexpr int SMEM_DATA = OP_STAGES * OP_STAGE + RAW_STAGES * RAW_STAGE;
            constexpr int SMEM_BYTES = SMEM_DATA + 1024 /* alignment slack */ + 256 /* barriers */;
            // warps 0-7 transform, 8-15 accumulate (two per TMEM lane quadrant), 16 TMA, 17 MMA.  With four
            // transform warps (one per scheduler) the split -- ~530 dependent instructions per thread
            // and stage -- took longer than the 768 cycles of the stage's MMAs and bound the kernel
            // (ncu: issue slots 44 % busy, tensor pipe 53 %, shared memory 53 %, DRAM 61 %).
            constexpr int THREADS = 576;
            constexpr int NTR = 256, NACC = 256;    // transform / accumulation threads
            constexpr int TMEM_COLS = 512;          // H[0] at column 0, H[1] at 128, S at 256

            struct Params {
                int nT, tsize[2];
                long long tsr[2];
                int M, N;
                long long msr, nsr;
                long long K;
                int mtiles, ntiles, ksplit, ksteps;
                int conj0, conj1;
                int promote; ///< stages per accumulation chain of the tensor core (see the header)
            };

            // ---- PTX wrappers ----------------------------------------------------------------------
            __device__ __forceinline__ unsigned smem_u32(const void *p) {
                return (unsigned)__cvta_generic_to_shared(p);
            }
            __device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
                asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
            }
            __device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
                             : "memory");
            }
            __device__ __forceinline__ void mbar_arrive(unsigned bar) {
                asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
            }
            __device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
                asm volatile("{\n\t"
                             ".reg .pred p;\n\t"
                             "WAIT_%=:\n\t"
                             "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                             "@p bra DONE_%=;\n\t"
                             "bra WAIT_%=;\n\t"
                             "DONE_%=:\n\t"
                             "}" ::"r"(bar),
                             "r"(parity)
                             : "memory");
            }
            __device__ __forceinline__ void tma_load_4d(unsigned dst, const CUtensorMap *map, int c0, int c1,
                                                        int c2, int c3, unsigned bar) {
                asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
                             " [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(dst),
                             "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar)
                             : "memory");
            }
            __device__ __forceinline__ void mma_tf32(unsigned d_tmem, unsigned long long adesc,
                                                     unsigned long long bdesc, unsigned idesc, unsigned accumulate) {
                asm volatile("{\n\t"
                             ".reg .pred p;\n\t"
                             "setp.ne.b32 p, %4, 0;\n\t"
                             "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
                             "}" ::"r"(d_tmem),
                             "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
                             : "memory");
            }
            /// The mbarrier receives one arrival when every tcgen05.mma issued so far by this thread is done
            __device__ __forceinline__ void mma_commit(unsigned bar) {
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
                             : "memory");
            }
            __device__ __forceinline__ void tmem_ld32(unsigned taddr, unsigned *r) {
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                             "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                             "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                             : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
                               "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]),
                               "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
                               "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
                               "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
                               "=r"(r[31])
                             : "r"(taddr)
                             : "memory");
            }

            __device__ __forceinline__ void tmem_ld16(unsigned taddr, unsigned *r) {
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                             "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                             : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
                               "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]),
                               "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                             : "r"(taddr)
                             : "memory");
            }

            /// Shared-memory matrix descriptor of a K-major tile in the canonical SWIZZLE_128B layout:
            /// rows of 128 bytes, groups of 8 rows 1024 bytes apart, 16-byte chunk c of row r stored at
            /// chunk c ^ (r % 8).  Fields: start address >> 4 (bits 0-13), leading byte offset >> 4
            /// (16-29; unused for swizzled K-major tiles), stride byte offset >> 4 (32-45) = 1024 >> 4,
            /// descriptor version 1 (46-47), layout type 2 = SWIZZLE_128B (61-63).
            __device__ __forceinline__ unsigned long long op_desc(unsigned smem_addr) {
                return (unsigned long long)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) |
                       (1ull << 46) | (2ull << 61);
            }
            /// Instruction descriptor of kind::tf32: D = F32 (bits 4-5 = 1), A and B = TF32 (7-9, 10-12
            /// = 2), both K-major (15, 16 = 0), N >> 3 (17-22), M >> 4 (24-28)
            constexpr unsigned IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);

            __device__ __forceinline__ float4 lds128(unsigned addr) {
                float4 v;
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                             : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                             : "r"(addr));
                return v;
            }
            __device__ __forceinline__ void sts128(unsigned addr, float a, float b, float c, float d) {
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d)
                             : "memory");
            }

            /// x rounded to the nearest TF32 value (10 explicit mantissa bits, ties away from zero; the
            /// low 13 bits of the result are zero, so the tensor core reads it exactly whatever it
            /// does with those bits).  Two full-rate integer instructions: cvt.rna.tf32.f32 computes
            /// the same but is a quarter-rate conversion (measured: 1.26 -> 1.46 ms for config 2).
            __device__ __forceinline__ float tf32_hi(float x) {
                return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
            }

            /// Split 4 consecutive complex numbers of one row into TF32 hi / lo parts and store them,
            /// de-interleaved, into the hi and lo tiles (re at row r, im at row r + 64)
            __device__ __forceinline__ void split_store(const float4 c0, const float4 c1, unsigned hi,
                                                        unsigned lo, unsigned off) {
                const float re[4] = {c0.x, c0.z, c1.x, c1.z}, im[4] = {c0.y, c0.w, c1.y, c1.w};
                float rh[4], rl[4], ih[4], il[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    rh[q] = tf32_hi(re[q]), rl[q] = tf32_hi(re[q] - rh[q]);
                    ih[q] = tf32_hi(im[q]), il[q] = tf32_hi(im[q] - ih[q]);
                }
                sts128(hi + off, rh[0], rh[1], rh[2], rh[3]);
                sts128(hi + off + 64 * 128, ih[0], ih[1], ih[2], ih[3]);
                sts128(lo + off, rl[0], rl[1], rl[2], rl[3]);
                sts128(lo + off + 64 * 128, il[0], il[1], il[2], il[3]);
            }

            __global__ void __launch_bounds__(THREADS, 1)
                contract_tc_kernel(const __grid_constant__ CUtensorMap map_a,
                                   const __grid_constant__ CUtensorMap map_b,
                                   const __grid_constant__ Params p, float *__restrict__ ws) {
                extern __shared__ unsigned char smem_raw[];
                // the operand tiles need 1024-byte alignment (swizzle atom); the raw tiles 128
                unsigned char *smem = reinterpret_cast<unsigned char *>(
                    (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
                unsigned char *ops = smem;                         // [OP_STAGES][Ahi, Alo, Bhi, Blo]
                unsigned char *raw = smem + OP_STAGES * OP_STAGE;  // [RAW_STAGES][A, B]
                unsigned long long *bars = reinterpret_cast<unsigned long long *>(smem + SMEM_DATA);
                // barriers: raw_full[3], raw_empty[3], op_full[2], op_empty[2], acc_full[2], acc_empty[2]
                const unsigned bar0 = smem_u32(bars);
                auto raw_full = [&](int s) { return bar0 + 8u * s; };
                auto raw_empty = [&](int s) { return bar0 + 8u * (RAW_STAGES + s); };
                auto op_full = [&](int u) { return bar0 + 8u * (2 * RAW_STAGES + u); };
                auto op_empty = [&](int u) { return bar0 + 8u * (2 * RAW_STAGES + OP_STAGES + u); };
                auto acc_full = [&](int b) { return bar0 + 8u * (2 * RAW_STAGES + 2 * OP_STAGES + b); };
                auto acc_empty = [&](int b) { return bar0 + 8u * (2 * RAW_STAGES + 2 * OP_STAGES + 2 + b); };
                unsigned *tmem_slot = reinterpret_cast<unsigned *>(bars + 2 * RAW_STAGES + 2 * OP_STAGES + 4);

                const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

                // ---- which tile / K slice ----------------------------------------------------------
                long long bid = blockIdx.x;
                const int nt = (int)(bid % p.ntiles);
                bid /= p.ntiles;
                const int mt = (int)(bid % p.mtiles);
                bid /= p.mtiles;
                const int ks = (int)(bid % p.ksplit);
                const long long t = bid / p.ksplit;
                const int t0 = (int)(t % p.tsize[0]), t1 = (int)(t / p.tsize[0]);
                const int kstep0 = (int)((long long)p.ksteps * ks / p.ksplit);
                const int kstep1 = (int)((long long)p.ksteps * (ks + 1) / p.ksplit);
                const int nsteps = kstep1 - kstep0;

                // ---- set-up ------------------------------------------------------------------------
                if (tid == 0) {
                    for (int s = 0; s < RAW_STAGES; ++s) mbar_init(raw_full(s), 1), mbar_init(raw_empty(s), NTR);
                    for (int u = 0; u < OP_STAGES; ++u) mbar_init(op_full(u), NTR), mbar_init(op_empty(u), 1);
                    for (int b = 0; b < 2; ++b) mbar_init(acc_full(b), 1), mbar_init(acc_empty(b), NACC);
                    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
                }
                if (warp == 17) { // the MMA warp owns the tensor memory
                    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                                     smem_u32(tmem_slot)),
                                 "n"(TMEM_COLS)
                                 : "memory");
                    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
                }
                if (warp == 16 && lane == 0) {
                    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
                    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncthreads();
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const unsigned tmem = *tmem_slot;
                const int P = p.promote > 0 ? p.promote : nsteps; // stages per chain
                const int nchunks = (nsteps + P - 1) / P;

                if (warp == 16) {
                    // ===== TMA producer =================================================================
                    if (lane == 0) {
                        for (int it = 0; it < nsteps; ++it) {
                            const int s = it % RAW_STAGES;
                            mbar_wait(raw_empty(s), ((it / RAW_STAGES) & 1) ^ 1);
                            mbar_expect_tx(raw_full(s), RAW_STAGE);
                            const int kc = (kstep0 + it) * (2 * BKC); // in floats
                            const unsigned dst = smem_u32(raw + s * RAW_STAGE);
                            tma_load_4d(dst, &map_a, kc, mt * TM, t0, t1, raw_full(s));
                            tma_load_4d(dst + RAW_TILE, &map_b, kc, nt * TN, t0, t1, raw_full(s));
                        }
                    }
                } else if (warp == 17) {
                    // ===== MMA issuer ===================================================================
                    if (lane == 0) {
                        for (int it = 0; it < nsteps; ++it) {
                            const int u = it % OP_STAGES;
                            const int c = it / P, b = c & 1;
                            const bool first = it % P == 0, last = (it % P == P - 1) || it == nsteps - 1;
                            mbar_wait(op_full(u), (it / OP_STAGES) & 1);
                            if (first) mbar_wait(acc_empty(b), ((c >> 1) & 1) ^ 1); // H[b] drained
                            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                            const unsigned base = smem_u32(ops + u * OP_STAGE);
                            const unsigned long long ahi = op_desc(base), alo = op_desc(base + OP_TILE),
                                                     bhi = op_desc(base + 2 * OP_TILE),
                                                     blo = op_desc(base + 3 * OP_TILE);
                            const unsigned H = tmem + (unsigned)(b * 128), S = tmem + 256u;
#pragma unroll
                            for (int k4 = 0; k4 < BKC / 8; ++k4) { // 8 TF32 = 32 bytes per instruction
                                const unsigned long long adv = (unsigned long long)(k4 * 2);
                                mma_tf32(H, ahi + adv, bhi + adv, IDESC, !(first && k4 == 0));
                                mma_tf32(S, ahi + adv, blo + adv, IDESC, (it | k4) != 0);
                                mma_tf32(S, alo + adv, bhi + adv, IDESC, 1);
                            }
                            mma_commit(op_empty(u)); // the stage is free once these MMAs have read it
                            if (last) mma_commit(acc_full(b)); // (the last one also covers S)
                        }
                    }
                } else if (warp >= 8) {
                    // ===== accumulation warps (8-15): TMEM lanes 32 (warp % 4) .. +31, one row per thread,
                    //       columns 64 h .. 64 h + 63 of the 128 with h = (warp - 8) / 4 =====================
                    const unsigned lane_base = (unsigned)((warp & 3) * 32) << 16;
                    const unsigned col0 = (unsigned)(((warp - 8) >> 2) * 64);
                    float sum[64];
#pragma unroll
                    for (int j = 0; j < 64; ++j) sum[j] = 0.f;
                    for (int c = 0; c < nchunks; ++c) {
                        const int b = c & 1;
                        mbar_wait(acc_full(b), (c >> 1) & 1);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                        for (int q = 0; q < 4; ++q) { // (16 columns at a time: 64 sums + 16 values fit the registers)
                            unsigned v[16];
                            tmem_ld16(tmem + lane_base + (unsigned)(b * 128) + col0 + (unsigned)(q * 16), v);
                            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                            for (int j = 0; j < 16; ++j) sum[q * 16 + j] += __uint_as_float(v[j]);
                        }
                        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                        mbar_arrive(acc_empty(b));
                    }
                    // the small terms (complete: the last acc_full covered them), then the partial tile
                    const long long tile_id = ((t * p.mtiles + mt) * p.ntiles + nt) * (long long)p.ksplit + ks;
                    float *out = ws + tile_id * (128 * 128) + ((warp & 3) * 32 + lane) * 128 + col0;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        unsigned v[16];
                        tmem_ld16(tmem + lane_base + 256u + col0 + (unsigned)(q * 16), v);
                        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            *reinterpret_cast<float4 *>(out + q * 16 + j * 4) =
                                make_float4(sum[q * 16 + 4 * j] + __uint_as_float(v[4 * j]),
                                            sum[q * 16 + 4 * j + 1] + __uint_as_float(v[4 * j + 1]),
                                            sum[q * 16 + 4 * j + 2] + __uint_as_float(v[4 * j + 2]),
                                            sum[q * 16 + 4 * j + 3] + __uint_as_float(v[4 * j + 3]));
                    }
                } else {
                    // ===== transform warps (0-7) ==========================================================
                    // item = (row r, group g of 4 complex): lanes of a quarter warp share r and cover
                    // g = 0..7, i.e. one 256-byte raw row and one 128-byte row of each output tile.
                    // The two 16-byte loads of a thread are issued in swapped order by the upper four
                    // lanes so that every quarter-warp request touches 8 distinct bank groups.
                    const int g = tid & 7, swap = (g >> 2) & 1;
                    for (int it = 0; it < nsteps; ++it) {
                        const int s = it % RAW_STAGES, u = it % OP_STAGES;
                        mbar_wait(raw_full(s), (it / RAW_STAGES) & 1);
                        mbar_wait(op_empty(u), ((it / OP_STAGES) & 1) ^ 1);
                        const unsigned ra = smem_u32(raw + s * RAW_STAGE);
                        const unsigned op = smem_u32(ops + u * OP_STAGE);
#pragma unroll
                        for (int half = 0; half < 2; ++half) { // A then B
                            const unsigned src = ra + half * RAW_TILE;
                            const unsigned hi = op + (2 * half) * OP_TILE, lo = hi + OP_TILE;
                            float4 f[2], h[2];
#pragma unroll
                            for (int i = 0; i < 2; ++i) {
                                const int r = (tid >> 3) + 32 * i;
                                const unsigned b = src + r * (BKC * 8) + g * 32;
                                f[i] = lds128(b + swap * 16);
                                h[i] = lds128(b + 16 - swap * 16);
                            }
#pragma unroll
                            for (int i = 0; i < 2; ++i) {
                                const int r = (tid >> 3) + 32 * i;
                                const unsigned off = (unsigned)((r >> 3) * 1024 + (r & 7) * 128 + ((g ^ (r & 7)) << 4));
                                split_store(swap ? h[i] : f[i], swap ? f[i] : h[i], hi, lo, off);
                            }
                        }
                        // generic-proxy writes -> visible to the tensor core (async proxy), then hand over
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        mbar_arrive(op_full(u));
                        mbar_arrive(raw_empty(s));
                    }
                }

                // ---- teardown ----------------------------------------------------------------------------
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncthreads();
                if (warp == 17) {
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TMEM_COLS)
                                 : "memory");
                }
            }


            /// Sum the K slices (fixed order, double), combine the four real blocks, alpha, beta, strides
            __global__ void __launch_bounds__(256)
                contract_tc_reduce_kernel(const __grid_constant__ Params p, const float *__restrict__ ws,
                                          float2 *vr, double2 alpha, double2 beta) {
                const long long tvol = (long long)p.tsize[0] * p.tsize[1];
                const long long total = tvol * p.M * p.N;
                const double sa = p.conj0 ? -1.0 : 1.0, sb = p.conj1 ? -1.0 : 1.0;
                for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
                     idx += (long long)gridDim.x * blockDim.x) {
                    const int n = (int)(idx % p.N);
                    const int m = (int)((idx / p.N) % p.M);
                    const long long t = idx / ((long long)p.N * p.M);
                    const int mt = m / TM, ntile = n / TN, mi = m % TM, ni = n % TN;
                    const float *src = ws + (((t * p.mtiles + mt) * p.ntiles + ntile) * (long long)p.ksplit) * (128 * 128);
                    double rr = 0, ri = 0, ir = 0, ii = 0;
                    for (int s = 0; s < p.ksplit; ++s, src += 128 * 128) {
                        rr += (double)src[mi * 128 + ni];
                        ri += (double)src[mi * 128 + 64 + ni];
                        ir += (double)src[(64 + mi) * 128 + ni];
                        ii += (double)src[(64 + mi) * 128 + 64 + ni];
                    }
                    // (ar + i sa ai)(br + i sb bi)
                    const double re = rr - sa * sb * ii, im = sb * ri + sa * ir;
                    double2 r = make_double2(alpha.x * re - alpha.y * im, alpha.x * im + alpha.y * re);
                    const long long orr = (t % p.tsize[0]) * p.tsr[0] + (t / p.tsize[0]) * p.tsr[1] +
                                          m * p.msr + n * p.nsr;
                    if (beta.x != 0 || beta.y != 0) {
                        const float2 old = vr[orr];
                        r.x += beta.x * old.x - beta.y * old.y;
                        r.y += beta.x * old.y + beta.y * old.x;
                    }
                    vr[orr] = make_float2((float)r.x, (float)r.y);
                }
            }

            // ---- host ------------------------------------------------------------------------------

            using EncodeFn = CUresult (*)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                          const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                          const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                          CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

            EncodeFn encoder() {
                static EncodeFn fn = nullptr;
                static std::once_flag once;
                std::call_once(once, [] {
                    void *p = nullptr;
                    cudaDriverEntryPointQueryResult q;
                    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
                        q == cudaDriverEntryPointSuccess)
                        fn = (EncodeFn)p;
                    else
                        cudaGetLastError();
                });
                if (!fn) throw std::runtime_error("cuTensorMapEncodeTiled is not available in this driver");
                return fn;
            }

            /// The operand as a 4-d float tensor (2k, row, t0, t1); out-of-range rows and k read as zero
            CUtensorMap make_map(const void *base, long long K, int rows, long long row_stride, const Problem &p,
                                 bool second) {
                CUtensorMap m;
                const cuuint64_t dims[4] = {(cuuint64_t)(2 * K), (cuuint64_t)rows,
                                            (cuuint64_t)(p.nT > 0 ? p.T[0].size : 1),
                                            (cuuint64_t)(p.nT > 1 ? p.T[1].size : 1)};
                auto ts = [&](int i) { return second ? p.T[i].s1 : p.T[i].s0; };
                // byte strides of dims 1..3 (multiples of 16; a size-1 dim may carry any valid value)
                const cuuint64_t strides[3] = {(cuuint64_t)((rows > 1 ? row_stride : K) * 8),
                                               (cuuint64_t)((p.nT > 0 ? ts(0) : K) * 8),
                                               (cuuint64_t)((p.nT > 1 ? ts(1) : K) * 8)};
                const cuuint32_t box[4] = {2 * BKC, (cuuint32_t)TM, 1, 1}, estr[4] = {1, 1, 1, 1};
                const CUresult r = encoder()(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void *>(base), dims,
                                             strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                             CU_TENSOR_MAP_SWIZZLE_NONE,
                                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
                if (r != CUDA_SUCCESS)
                    throw std::runtime_error("cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
                return m;
            }

        } // namespace

        bool eligible(const Problem &p, const void *v0, const void *v1) {
            if (p.K < 1 || p.K >= (1ll << 30) || p.nT < 0 || p.nT > 2) return false;
            if (((uintptr_t)v0 | (uintptr_t)v1) & 15) return false;
            auto even = [](long long s) { return s > 0 && s % 2 == 0; }; // 8-byte elements, 16-byte strides
            // TMA also wants ascending, non-overlapping dims only in the sense of valid strides < 2^40 bytes
            auto ok = [&](long long s) { return even(s) && s < (1ll << 36); };
            if (p.M.size > 1 && !ok(p.M.s0)) return false;
            if (p.N.size > 1 && !ok(p.N.s1)) return false;
            for (int i = 0; i < p.nT; ++i)
                if (!ok(p.T[i].s0) || !ok(p.T[i].s1)) return false;
            return true;
        }

        void launch_c64(const Problem &pr, const double *alpha, const void *v0, const void *v1,
                        const double *beta, void *vr, int device, cudaStream_t stream,
                        std::string *describe) {
            Params p;
            std::memset(&p, 0, sizeof p);
            p.nT = pr.nT;
            p.tsize[0] = pr.nT > 0 ? pr.T[0].size : 1, p.tsize[1] = pr.nT > 1 ? pr.T[1].size : 1;
            p.tsr[0] = pr.nT > 0 ? pr.T[0].sr : 0, p.tsr[1] = pr.nT > 1 ? pr.T[1].sr : 0;
            p.M = pr.M.size, p.N = pr.N.size, p.msr = pr.M.sr, p.nsr = pr.N.sr;
            p.K = pr.K, p.conj0 = pr.conj0, p.conj1 = pr.conj1;
            p.mtiles = (p.M + TM - 1) / TM, p.ntiles = (p.N + TN - 1) / TN;
            p.ksteps = (int)((p.K + BKC - 1) / BKC);
            const long long tvol = (long long)p.tsize[0] * p.tsize[1];
            const long long tiles = tvol * p.mtiles * p.ntiles;
            // K split: one CTA per SM; fill the machine in whole waves, keep slices >= 8 stages and
            // the workspace small (fewest slices within 3 % of the best wave efficiency)
            const long long slots = sm_count(device, describe != nullptr);
            const int smax = std::max(1, std::min(p.ksteps / 8, 4096));
            double best_eff = -1;
            for (int s = 1; s <= smax; ++s) {
                const long long ctas = tiles * s, waves = (ctas + slots - 1) / slots;
                best_eff = std::max(best_eff, (double)ctas / (double)(waves * slots));
                if (waves >= 32) break;
            }
            p.ksplit = 1;
            for (int s = 1; s <= smax; ++s) {
                const long long ctas = tiles * s, waves = (ctas + slots - 1) / slots;
                if ((double)ctas / (double)(waves * slots) >= best_eff - 0.03) {
                    p.ksplit = s;
                    break;
                }
                if (waves >= 32) break;
            }
            {
                // experiments: SBB_TC_KSPLIT forces the K split, SBB_TC_PROMOTE the chain length in
                // stages (0 = never drain: one chain per CTA, the inaccurate first version)
                static int ks_env = -1, pr_env = -2;
                if (ks_env < 0) {
                    const char *e = std::getenv("SBB_TC_KSPLIT");
                    ks_env = e ? std::atoi(e) : 0;
                    const char *q = std::getenv("SBB_TC_PROMOTE");
                    pr_env = q ? std::atoi(q) : -1;
                }
                if (ks_env > 0) p.ksplit = std::min(ks_env, p.ksteps);
                p.promote = pr_env >= 0 ? pr_env : 4;
            }
            const long long ctas = tiles * p.ksplit;
            if (ctas >= (1ll << 31)) throw std::runtime_error("contraction: grid too large");
            if (describe) {
                std::stringstream ss;
                ss << "tcgen05 tf32x3 tile=" << TM << "x" << TN << "x" << BKC << " (complex) T=" << tvol
                   << " M=" << p.M << " N=" << p.N << " K=" << p.K << " ksplit=" << p.ksplit
                   << " ctas=" << ctas << " promote=" << p.promote << " smem=" << SMEM_BYTES << " loader=tma";
                *describe = ss.str();
                return;
            }
            const CUtensorMap ma = make_map(v0, p.K, p.M, pr.M.s0, pr, false);
            const CUtensorMap mb = make_map(v1, p.K, p.N, pr.N.s1, pr, true);
            PoolGuard guard;
            float *ws = (float *)guard.alloc(device, (size_t)ctas * 128 * 128 * sizeof(float));
            static bool attr_set[64] = {false};
            if (!attr_set[device]) {
                cuda_check(cudaFuncSetAttribute(contract_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                SMEM_BYTES),
                           "cudaFuncSetAttribute");
                attr_set[device] = true;
            }
            {
                KernelTimer timer("contract_tc", stream);
                contract_tc_kernel<<<(unsigned)ctas, THREADS, SMEM_BYTES, stream>>>(ma, mb, p, ws);
            }
            count_launch();
            cuda_check(cudaGetLastError(), "contract_tc_kernel launch");
            const long long total = tvol * p.M * p.N;
            const unsigned grid = (unsigned)std::min<long long>((total + 255) / 256, slots * 8);
            contract_tc_reduce_kernel<<<grid, 256, 0, stream>>>(p, ws, (float2 *)vr,
                                                                make_double2(alpha[0], alpha[1]),
                                                                make_double2(beta[0], beta[1]));
            count_launch();
            cuda_check(cudaGetLastError(), "contract_tc_reduce_kernel launch");
        }

    } // namespace tc
} // namespace sbb
