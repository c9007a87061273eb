// Permutation / reshuffle copy kernels for sm_100a.
//
// Replaces the reference's index-vector machinery: get_permutation (tensor.h:815-961, thrust K1),
// copy_n / copy_n_blocking gather-scatter (copy_n.h:283-351, :752-987, thrust K2-K4) and zero_n
// (copy_n.h:379).  No index vector exists here: a copy is a strided box (sbk_box_desc), and the
// kernel walks it tile by tile.
//
// Kernel design (HBM-bound byte work; the rules that matter are coalescing, bytes in flight and
// grid sizing, not tensor cores):
//   * The box is canonicalised on the host: extent-1 dims dropped, dims sorted by destination
//     stride, neighbouring dims merged when both sides stay affine, and the element widened to 8 or
//     16 bytes when the fastest dim is shared and aligned (128-bit ld/st whenever possible).
//   * A tile is a small sub-box chosen so that it holds a long contiguous run of the destination
//     AND a long contiguous run of the source (>=256-512 B each when the geometry allows).
//     CTAs are persistent (grid = SMs x resident CTAs) and stride over the tiles.
//   * Inside a tile every thread owns up to EPT "slots".  The slot -> (source offset, shared-memory
//     position) map for the load phase (threads consecutive along the SOURCE-contiguous direction)
//     and the slot -> (destination offset, shared-memory position) map for the store phase
//     (threads consecutive along the DESTINATION-contiguous direction) are tile invariant, so they
//     are computed once per CTA and kept in registers: the per-element cost in the steady state
//     is one load, one st.shared, one ld.shared, one store.  Tile coordinates advance with
//     carry arithmetic (no division in the loop).
//   * Shared memory is laid out in destination order; the stride of the source-fastest dim is
//     padded to an odd number of elements so the transposing st.shared is bank-conflict free.
//   * When source and destination enumerate the tile in the same order no staging is needed and
//     the direct variant (no shared memory, no barrier) is used.
//   * Typed variants apply alpha (without fused multiply-add, so results are bit-identical to the
//     reference's CPU loops built with -ffp-contract=off), convert T->Q and add.
#include "kernels.hpp"
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cuda_runtime.h>
#include <map>
#include <numeric>
#include <sstream>
#include <vector>

namespace sbb {

    void permute_cache_clear();

    namespace {
        size_t g_table_bytes = 0; // device memory held by the cached launch tables
        constexpr size_t kTableBudget = (size_t)1 << 30;

        constexpr int KD = 8;   // dims handled inside one launch (after merging)
        constexpr int MAXT = 6; // tiled dims
        constexpr int NT = 256; // threads per CTA
        constexpr int EPT = 8;  // slots (elements of a tile) per thread; 16 was measured slower for transposing tiles
        // Masked copies carry up to three mask words per slot besides the element and the slot maps:
        // with 8 slots the 16-byte variant needs > 128 registers (measured: spills, 2 CTAs per SM,
        // 25 % occupancy, 0.43 ms for the even-site permutation).  4 slots: 3 CTAs per SM.
        constexpr int MASK_EPT = 4;

        struct PermParams {
            int nd, nt, tile_elems, smem_elems;
            int rot, rot_q; // rotation of the fastest dim in the destination, and its tiled-dim slot (-1: none)
            unsigned ntiles;
            int size[KD];
            int te[KD];
            unsigned ntile[KD];
            long long tsstride[KD], tdstride[KD]; // te*stride: jump between tiles
            int tdim[MAXT];                       // tiled dims, destination order
            int text[MAXT];                       // their tile extents
            int sord[MAXT];                       // positions in tdim[], sorted by source stride
            int smem_stride[MAXT];
            long long tss[MAXT], tds[MAXT]; // element strides of the tiled dims
        };

        // ---- element functors -----------------------------------------------------------------

        __device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
        __device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
        __device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
        __device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
        __device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
        __device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }

        // alpha * x in T, each real operation rounded once (no contraction into FMA)
        __device__ __forceinline__ float scale(float a, float x) { return mul_rn(a, x); }
        __device__ __forceinline__ double scale(double a, double x) { return mul_rn(a, x); }
        __device__ __forceinline__ int scale(int a, int x) { return a * x; }
        __device__ __forceinline__ float2 scale(float2 a, float2 x) {
            return make_float2(sub_rn(mul_rn(a.x, x.x), mul_rn(a.y, x.y)),
                               add_rn(mul_rn(a.x, x.y), mul_rn(a.y, x.x)));
        }
        __device__ __forceinline__ double2 scale(double2 a, double2 x) {
            return make_double2(sub_rn(mul_rn(a.x, x.x), mul_rn(a.y, x.y)),
                                add_rn(mul_rn(a.x, x.y), mul_rn(a.y, x.x)));
        }

        template <typename Q, typename T> struct Cvt;
        template <typename T> struct Cvt<T, T> {
            __device__ static __forceinline__ T to(T x) { return x; }
        };
        template <> struct Cvt<double, float> {
            __device__ static __forceinline__ double to(float x) { return (double)x; }
        };
        template <> struct Cvt<float, double> {
            __device__ static __forceinline__ float to(double x) { return __double2float_rn(x); }
        };
        template <> struct Cvt<double2, float2> {
            __device__ static __forceinline__ double2 to(float2 x) {
                return make_double2((double)x.x, (double)x.y);
            }
        };
        template <> struct Cvt<float2, double2> {
            __device__ static __forceinline__ float2 to(double2 x) {
                return make_float2(__double2float_rn(x.x), __double2float_rn(x.y));
            }
        };

        // the wider of two element types (C's usual arithmetic conversions for `w += x`)
        template <typename Q, typename T> struct Wider { using type = Q; };
        template <> struct Wider<float, double> { using type = double; };
        template <> struct Wider<float2, double2> { using type = double2; };

        __device__ __forceinline__ float plus(float a, float b) { return add_rn(a, b); }
        __device__ __forceinline__ double plus(double a, double b) { return add_rn(a, b); }
        __device__ __forceinline__ int plus(int a, int b) { return a + b; }
        __device__ __forceinline__ float2 plus(float2 a, float2 b) {
            return make_float2(add_rn(a.x, b.x), add_rn(a.y, b.y));
        }
        __device__ __forceinline__ double2 plus(double2 a, double2 b) {
            return make_double2(add_rn(a.x, b.x), add_rn(a.y, b.y));
        }

        /// w = Q(alpha*x)   or   w = Q(W(w) + W(alpha*x)); `scale` and `add` are uniform run-time flags
        template <typename T_, typename Q_> struct ElemOp {
            using T = T_;
            using Q = Q_;
            T alpha;
            bool scale_, add_;
            __device__ __forceinline__ bool add() const { return add_; }
            __device__ __forceinline__ Q apply(T x) const {
                if (scale_) x = scale(alpha, x);
                return Cvt<Q, T>::to(x);
            }
            __device__ __forceinline__ Q combine(Q old, T x) const {
                if (scale_) x = scale(alpha, x);
                using W = typename Wider<Q, T>::type;
                return Cvt<Q, W>::to(plus(Cvt<W, Q>::to(old), Cvt<W, T>::to(x)));
            }
        };

        /// Raw move of 4, 8 or 16 bytes
        template <typename V> struct MoveOp {
            using T = V;
            using Q = V;
            __device__ __forceinline__ constexpr bool add() const { return false; }
            __device__ __forceinline__ V apply(V x) const { return x; }
            __device__ __forceinline__ V combine(V, V x) const { return x; }
        };

        // ---- global memory accessors ----------------------------------------------------------------
        // address = base + 32-bit slot offset x element size in ONE instruction (IMAD.WIDE.U32), then
        // the memory instruction itself; written in PTX because the compiler otherwise carries every
        // slot offset as a 64-bit pair and spends 4-5 integer instructions per access, which made the
        // kernel issue bound for 4- and 8-byte elements (profiles/r1_permute64_ncu.txt).
        template <typename T>
        __device__ __forceinline__ unsigned long long elem_addr(const T *base, unsigned off) {
            unsigned long long a;
            asm("mad.wide.u32 %0, %1, %2, %3;"
                : "=l"(a)
                : "r"(off), "n"((unsigned)sizeof(T)), "l"(base));
            return a;
        }
        /// NC: read-only path (ld.global.nc) for the source; the destination of an Add is read coherently
        template <bool NC, typename T> __device__ __forceinline__ T ld_elem(const T *base, unsigned off) {
            static_assert(sizeof(T) == 4 || sizeof(T) == 8 || sizeof(T) == 16, "element size");
            const unsigned long long a = elem_addr(base, off);
            T v;
            if constexpr (sizeof(T) == 4) {
                unsigned x;
                if (NC) asm volatile("ld.global.nc.b32 %0, [%1];" : "=r"(x) : "l"(a));
                else asm volatile("ld.global.b32 %0, [%1];" : "=r"(x) : "l"(a));
                memcpy(&v, &x, 4);
            } else if constexpr (sizeof(T) == 8) {
                uint2 x;
                if (NC) asm volatile("ld.global.nc.v2.b32 {%0,%1}, [%2];" : "=r"(x.x), "=r"(x.y) : "l"(a));
                else asm volatile("ld.global.v2.b32 {%0,%1}, [%2];" : "=r"(x.x), "=r"(x.y) : "l"(a));
                memcpy(&v, &x, 8);
            } else {
                uint4 x;
                if (NC)
                    asm volatile("ld.global.nc.v4.b32 {%0,%1,%2,%3}, [%4];"
                                 : "=r"(x.x), "=r"(x.y), "=r"(x.z), "=r"(x.w)
                                 : "l"(a));
                else
                    asm volatile("ld.global.v4.b32 {%0,%1,%2,%3}, [%4];"
                                 : "=r"(x.x), "=r"(x.y), "=r"(x.z), "=r"(x.w)
                                 : "l"(a));
                memcpy(&v, &x, 16);
            }
            return v;
        }
        template <typename T> __device__ __forceinline__ void st_elem(T *base, unsigned off, const T &v) {
            static_assert(sizeof(T) == 4 || sizeof(T) == 8 || sizeof(T) == 16, "element size");
            const unsigned long long a = elem_addr(base, off);
            if constexpr (sizeof(T) == 4) {
                unsigned x;
                memcpy(&x, &v, 4);
                asm volatile("st.global.b32 [%0], %1;" ::"l"(a), "r"(x));
            } else if constexpr (sizeof(T) == 8) {
                uint2 x;
                memcpy(&x, &v, 8);
                asm volatile("st.global.v2.b32 [%0], {%1,%2};" ::"l"(a), "r"(x.x), "r"(x.y));
            } else {
                uint4 x;
                memcpy(&x, &v, 16);
                asm volatile("st.global.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(a), "r"(x.x), "r"(x.y),
                             "r"(x.z), "r"(x.w));
            }
        }

        // ---- the kernel -------------------------------------------------------------------------

        /// Decompose slot index e following the enumeration `ord` (positions in tdim[]).
        /// Returns false if e is outside the tile.
        __device__ __forceinline__ void slot_coords(const PermParams &p, unsigned e,
                                                    const int *ord, int c[MAXT]) {
#pragma unroll
            for (int q = 0; q < MAXT; ++q) c[q] = 0;
#pragma unroll
            for (int q = 0; q < MAXT; ++q) {
                if (q < p.nt) {
                    const int t = ord[q];
                    const unsigned ext = (unsigned)p.text[t];
                    const int v = (int)(e % ext);
                    e /= ext;
                    // c[t] = v without dynamic register indexing
#pragma unroll
                    for (int j = 0; j < MAXT; ++j)
                        if (j == t) c[j] = v;
                }
            }
        }

        /// Per-geometry tables, built on the host once and cached on the device (see build_tables):
        /// the slot maps of a tile and the origin of every tile.
        struct Tables {
            const unsigned *so, *dof, *sp; // per slot: source offset, destination offset, shared-memory
                                           // positions (load position << 16 | store position)
            const longlong2 *tiles;        // per tile: {source origin | boundary flag in bit 63, destination origin}
        };

        /// MASK: the destination element is written only where the masks (MaskType = float, nonzero =
        /// active; laid out like the destination, either may be null) are nonzero.  This is the
        /// reference's `select` on the index vectors (tensor.h:1022-1027, blas.h:877-923) done as a
        /// predicate on the store instead of a stream compaction.
        template <class Op, bool SMEM, int EPT, int MINB, bool MASK>
        __global__ void __launch_bounds__(NT, MINB)
            permute_kernel(const __grid_constant__ PermParams p, const Tables tab,
                           const typename Op::T *__restrict__ src, typename Op::Q *dst, Op op,
                           const float *__restrict__ ma, const float *__restrict__ mb,
                           const bool ma_src, const ExchangeSync xs) {
            using T = typename Op::T;
            using Q = typename Op::Q;
            extern __shared__ __align__(16) unsigned char smem_raw[];
            T *smem = reinterpret_cast<T *>(smem_raw);
            // ma_src: `ma` is the SOURCE's mask (laid out like the source): it is read with the source
            // elements and, in the transposing variant, travels to the store slot as one byte per
            // element through shared memory (after the element tile) -- a masked local copy in one
            // pass, without first carrying the mask to the destination layout
            unsigned char *flg = smem_raw + (size_t)p.smem_elems * sizeof(T);

            const unsigned tid = threadIdx.x;
            if (blockIdx.x >= p.ntiles) return; // (never taken: the grid is at most ntiles)

            // ---- per-slot maps: tile invariant, kept in registers ---------------------------------
            unsigned so[EPT], dof[EPT], sp[EPT];
            unsigned live = 0; // bit k set: slot k is inside the tile
#pragma unroll
            for (int k = 0; k < EPT; ++k) {
                const unsigned e = tid + k * NT;
                so[k] = dof[k] = sp[k] = 0;
                if (e < (unsigned)p.tile_elems) {
                    live |= 1u << k;
                    so[k] = tab.so[e];
                    dof[k] = tab.dof[e];
                    if (SMEM) sp[k] = tab.sp[e];
                }
            }

            // ---- tile loop, software pipelined -----------------------------------------------------
            // The loads of the next tile are in flight while the current tile is being stored, so a
            // CTA always has a tile's worth of bytes outstanding (HBM latency x bandwidth needs
            // ~40 KB per SM in flight).  Tile origins come from the table, two tiles ahead.
            struct Tile {
                long long sbase, dbase;
                unsigned mask_l, mask_s; // slots to load / to store (all live slots on full tiles)
            };
            auto make_tile = [&](longlong2 e, unsigned tile) {
                Tile t;
                t.sbase = e.x & 0x7fffffffffffffffll;
                t.dbase = e.y;
                t.mask_l = t.mask_s = live;
                if (e.x < 0) {
                    // boundary tile (rare): mask the slots that fall outside the box
                    int dord[MAXT];
#pragma unroll
                    for (int q = 0; q < MAXT; ++q) dord[q] = q;
                    unsigned tc[KD];
                    unsigned rem = tile;
#pragma unroll
                    for (int d = 0; d < KD; ++d) {
                        tc[d] = 0;
                        if (d < p.nd) {
                            tc[d] = rem % p.ntile[d];
                            rem /= p.ntile[d];
                        }
                    }
                    int lim[MAXT];
#pragma unroll
                    for (int q = 0; q < MAXT; ++q) {
                        lim[q] = 1;
                        if (q < p.nt) {
                            const int d = p.tdim[q];
                            unsigned tcd = 0;
#pragma unroll
                            for (int dd = 0; dd < KD; ++dd)
                                if (dd == d) tcd = tc[dd];
                            lim[q] = min(p.text[q], p.size[d] - (int)(tcd * (unsigned)p.te[d]));
                        }
                    }
                    auto inside = [&](unsigned slot, const int *ord) {
                        int c[MAXT];
                        slot_coords(p, slot, ord, c);
                        bool ok = true;
#pragma unroll
                        for (int q = 0; q < MAXT; ++q) ok = ok && (c[q] < lim[q]);
                        return ok;
                    };
                    t.mask_l = t.mask_s = 0;
#pragma unroll
                    for (int k = 0; k < EPT; ++k)
                        if (live >> k & 1) {
                            if (inside(tid + k * NT, dord)) t.mask_s |= 1u << k;
                            if (SMEM && inside(tid + k * NT, p.sord)) t.mask_l |= 1u << k;
                        }
                    if (!SMEM) t.mask_l = t.mask_s;
                }
                return t;
            };
            constexpr int NFS = (MASK && SMEM) ? EPT : 1;
            float fsrc[NFS]; // source mask words, paired with the elements in r
            auto load = [&](const Tile &t, T(&r)[EPT], float(&fs)[NFS]) {
                const T *s = src + t.sbase;
#pragma unroll
                for (int k = 0; k < EPT; ++k)
                    if (t.mask_l >> k & 1) r[k] = ld_elem<true>(s, so[k]);
                if (MASK && SMEM && ma_src) {
#pragma unroll
                    for (int k = 0; k < NFS; ++k)
                        if (t.mask_l >> k & 1) fs[k] = ld_elem<true>(ma + t.sbase, so[k]);
                }
            };

            const unsigned G = gridDim.x;
            const unsigned my_tiles = (p.ntiles - blockIdx.x + G - 1) / G;
            unsigned tile = blockIdx.x;
            longlong2 e_nxt = my_tiles > 1 ? tab.tiles[tile + G] : tab.tiles[tile];
            Tile cur = make_tile(tab.tiles[tile], tile);
            // Masks travel like the data: the mask words of tile i+1 are requested together with its
            // source elements, and turned into store predicates when tile i+1 becomes current.
            float fa[MASK ? EPT : 1], fb[MASK ? EPT : 1];
            auto load_masks = [&](const Tile &t) {
                if (!MASK) return;
#pragma unroll
                for (int k = 0; k < (MASK ? EPT : 1); ++k) {
                    fa[k] = fb[k] = 1.0f;
                    if (t.mask_s >> k & 1) {
                        if (ma && !ma_src) fa[k] = ld_elem<true>(ma + t.dbase, dof[k]);
                        if (ma && ma_src && !SMEM) fa[k] = ld_elem<true>(ma + t.sbase, so[k]); // same slot on both sides
                        if (mb) fb[k] = ld_elem<true>(mb + t.dbase, dof[k]);
                    }
                }
            };
            T r[EPT];
            load(cur, r, fsrc);
            load_masks(cur);
            for (unsigned i = 0; i < my_tiles; ++i, tile += G) {
                const bool has_next = i + 1 < my_tiles;
                const longlong2 e_nn = i + 2 < my_tiles ? tab.tiles[tile + 2 * G] : e_nxt;
                Tile nxt = cur;
                if (has_next) nxt = make_tile(e_nxt, tile + G);
                Q *w = dst + cur.dbase;
                if (MASK) {
                    // masked-out destination elements are left untouched
#pragma unroll
                    for (int k = 0; k < (MASK ? EPT : 1); ++k)
                        if (fa[k] == 0.0f || fb[k] == 0.0f) cur.mask_s &= ~(1u << k);
                }
                if (SMEM) {
#pragma unroll
                    for (int k = 0; k < EPT; ++k)
                        if (cur.mask_l >> k & 1) smem[sp[k] >> 16] = r[k];
                    if (MASK && ma_src) {
#pragma unroll
                        for (int k = 0; k < NFS; ++k)
                            if (cur.mask_l >> k & 1) flg[sp[k] >> 16] = fsrc[k] != 0.0f;
                    }
                    __syncthreads();
                    if (MASK && ma_src) {
#pragma unroll
                        for (int k = 0; k < EPT; ++k)
                            if ((cur.mask_s >> k & 1) && !flg[sp[k] & 0xffffu]) cur.mask_s &= ~(1u << k);
                    }
                    if (has_next) load(nxt, r, fsrc), load_masks(nxt); // in flight during the store phase
                    if (op.add()) {
                        Q o[EPT];
#pragma unroll
                        for (int k = 0; k < EPT; ++k)
                            if (cur.mask_s >> k & 1) o[k] = ld_elem<false>(w, dof[k]);
#pragma unroll
                        for (int k = 0; k < EPT; ++k)
                            if (cur.mask_s >> k & 1)
                                st_elem(w, dof[k], op.combine(o[k], smem[sp[k] & 0xffffu]));
                    } else {
#pragma unroll
                        for (int k = 0; k < EPT; ++k)
                            if (cur.mask_s >> k & 1) st_elem(w, dof[k], op.apply(smem[sp[k] & 0xffffu]));
                    }
                    __syncthreads();
                } else {
                    T r2[EPT];
                    if (has_next) load(nxt, r2, fsrc), load_masks(nxt);
                    if (op.add()) {
                        Q o[EPT];
#pragma unroll
                        for (int k = 0; k < EPT; ++k)
                            if (cur.mask_s >> k & 1) o[k] = ld_elem<false>(w, dof[k]);
#pragma unroll
                        for (int k = 0; k < EPT; ++k)
                            if (cur.mask_s >> k & 1) st_elem(w, dof[k], op.combine(o[k], r[k]));
                    } else {
#pragma unroll
                        for (int k = 0; k < EPT; ++k)
                            if (cur.mask_s >> k & 1) st_elem(w, dof[k], op.apply(r[k]));
                    }
#pragma unroll
                    for (int k = 0; k < EPT; ++k) r[k] = r2[k];
                }
                cur = nxt;
                e_nxt = e_nn;
            }

            // Pack side of an exchange: when the last CTA of this kernel has finished, all its stores
            // (which went to the receivers' arenas over NVLink) are complete: raise this rank's flag
            // at every receiver (fused signal: no kernel boundary, no NCCL barrier)
            if (xs.peer_flags) {
                __threadfence_system();
                __syncthreads();
                if (tid == 0) {
                    const unsigned prev = atomicAdd(xs.done, 1u);
                    if (prev + 1 == gridDim.x) {
                        // one system-scope fence orders every CTA's stores (each fenced before its
                        // atomicAdd) before the flag stores, which can then be relaxed and pipelined
                        // (a release store per peer would pay the fence once per peer)
                        __threadfence_system();
                        atomicExch(xs.done, 0u); // the next user is ordered behind this kernel
                        for (int q = 0; q < xs.nranks; ++q) {
                            unsigned long long *f = xs.peer_flags[q] + xs.me;
                            asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(f), "l"(xs.sig_seq)
                                         : "memory");
                        }
                    }
                }
            }
        }

        /// Zero fill of a strided box (direct variant without source)
        template <class V>
        __global__ void __launch_bounds__(NT)
            zero_kernel(const __grid_constant__ PermParams p, V *dst, const float *__restrict__ ma,
                        const float *__restrict__ mb) {
            const unsigned tid = threadIdx.x;
            int dord[MAXT];
#pragma unroll
            for (int q = 0; q < MAXT; ++q) dord[q] = q;
            V zero;
            memset(&zero, 0, sizeof(V));
            for (unsigned tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
                long long dbase = 0;
                unsigned t = tile;
                int lim[MAXT];
                unsigned tcs[KD];
#pragma unroll
                for (int d = 0; d < KD; ++d) {
                    tcs[d] = 0;
                    if (d < p.nd) {
                        tcs[d] = t % p.ntile[d];
                        t /= p.ntile[d];
                        dbase += tcs[d] * p.tdstride[d];
                    }
                }
#pragma unroll
                for (int q = 0; q < MAXT; ++q) {
                    lim[q] = 1;
                    if (q < p.nt) {
                        const int d = p.tdim[q];
                        unsigned tcd = 0;
#pragma unroll
                        for (int dd = 0; dd < KD; ++dd)
                            if (dd == d) tcd = tcs[dd];
                        lim[q] = min(p.text[q], p.size[d] - (int)(tcd * (unsigned)p.te[d]));
                    }
                }
#pragma unroll
                for (int k = 0; k < EPT; ++k) {
                    const unsigned e = tid + k * NT;
                    if (e < (unsigned)p.tile_elems) {
                        int c[MAXT];
                        slot_coords(p, e, dord, c);
                        bool ok = true;
                        long long d = 0;
#pragma unroll
                        for (int q = 0; q < MAXT; ++q) {
                            ok = ok && (c[q] < lim[q]);
                            if (q < p.nt) d += c[q] * p.tds[q];
                        }
                        if (ok && ma && ma[dbase + d] == 0.0f) ok = false;
                        if (ok && mb && mb[dbase + d] == 0.0f) ok = false;
                        if (ok) dst[dbase + d] = zero;
                    }
                }
            }
        }

        // ---- host side: canonical form, tiling, launch --------------------------------------------

        struct Canon {
            int nd = 0;
            std::vector<int> size;
            std::vector<int64_t> ss, ds;
            int64_t soff = 0, doff = 0;
            int rot = 0; ///< rotation of canonical dim 0 (which then has unit strides and is not merged)
        };

        Canon canonicalize(const sbk_box_desc &b, bool has_src) {
            Canon c;
            c.soff = b.soff, c.doff = b.doff;
            std::vector<int> idx;
            for (int k = 0; k < b.nd; ++k) {
                if (b.size[k] <= 0) {
                    c.nd = -1; // empty
                    return c;
                }
                if (b.size[k] > 1) idx.push_back(k);
            }
            std::stable_sort(idx.begin(), idx.end(),
                             [&](int x, int y) { return b.dstride[x] < b.dstride[y]; });
            if (b.rot != 0 && b.nd > 0 && b.size[0] > 1) {
                if (!has_src || b.sstride[0] != 1 || b.dstride[0] != 1 || idx.empty() || idx[0] != 0)
                    throw std::runtime_error("permute copy: rotation needs unit strides on dim 0");
                c.rot = ((b.rot % b.size[0]) + b.size[0]) % b.size[0];
            }
            for (int k : idx) {
                const int64_t ss = has_src ? b.sstride[k] : 0, ds = b.dstride[k];
                if (!c.size.empty() && !(c.rot != 0 && c.size.size() == 1)) {
                    const int64_t n = c.size.back();
                    if (c.ds.back() * n == ds && c.ss.back() * n == ss &&
                        n * (int64_t)b.size[k] < (1ll << 30)) {
                        c.size.back() *= b.size[k];
                        continue;
                    }
                }
                c.size.push_back(b.size[k]);
                c.ss.push_back(ss);
                c.ds.push_back(ds);
            }
            c.nd = (int)c.size.size();
            return c;
        }

        struct Tiling {
            std::vector<int> te;
            int64_t run_d = 1, run_s = 1, total = 1;
        };

        /// Greedy tile: cover `want_d` contiguous destination elements and `want_s` contiguous
        /// source elements.
        Tiling build_tile(const Canon &c, const std::vector<int> &sorder, int64_t want_d,
                          int64_t want_s) {
            Tiling t;
            t.te.assign(c.nd, 1);
            // extent close to `need` that divides the dimension when there is one (full tiles only)
            auto pick = [](int size, int64_t need) {
                int ext = (int)std::min<int64_t>(size, need);
                if (size % ext == 0) return ext;
                for (int e = ext; e <= std::min<int64_t>(size, 2 * (int64_t)ext); ++e)
                    if (size % e == 0) return e;
                for (int e = ext; e > ext / 2 && e >= 1; --e)
                    if (size % e == 0) return e;
                return ext;
            };
            int64_t acc = 1;
            for (int d = 0; d < c.nd && acc < want_d; ++d) {
                if (d == 0 ? false : c.ds[d] != c.ds[d - 1] * c.size[d - 1]) break;
                const int64_t need = (want_d + acc - 1) / acc;
                const int ext = pick(c.size[d], need);
                t.te[d] = ext;
                acc *= ext;
                if (ext < c.size[d]) break;
            }
            acc = 1;
            for (size_t q = 0; q < sorder.size() && acc < want_s; ++q) {
                const int d = sorder[q];
                if (q > 0 && c.ss[d] != c.ss[sorder[q - 1]] * c.size[sorder[q - 1]]) break;
                if (q > 0 && t.te[sorder[q - 1]] < c.size[sorder[q - 1]]) break;
                const int64_t need = (want_s + acc - 1) / acc;
                const int ext = std::max<int>(t.te[d], pick(c.size[d], need));
                t.te[d] = ext;
                acc *= ext;
                if (ext < c.size[d]) break;
            }
            // actual runs
            t.run_d = 1;
            for (int d = 0; d < c.nd; ++d) {
                if (d > 0 && (c.ds[d] != c.ds[d - 1] * c.size[d - 1] || t.te[d - 1] < c.size[d - 1]))
                    break;
                t.run_d *= t.te[d];
            }
            t.run_s = 1;
            for (size_t q = 0; q < sorder.size(); ++q) {
                const int d = sorder[q];
                if (q > 0) {
                    const int pd = sorder[q - 1];
                    if (c.ss[d] != c.ss[pd] * c.size[pd] || t.te[pd] < c.size[pd]) break;
                }
                t.run_s *= t.te[d];
            }
            t.total = 1;
            for (int d = 0; d < c.nd; ++d) t.total *= t.te[d];
            return t;
        }

        struct LaunchPlan {
            PermParams p;
            bool smem = false;
            int es = 0; // element size in bytes seen by the kernel
            int64_t run_d = 0, run_s = 0;
            bool empty = false;
            Tables tab{nullptr, nullptr, nullptr, nullptr}; // device tables (owned by the launch cache)
            void *tab_mem = nullptr;
            int tab_device = -1;
        };

        /// Host-side construction of the kernel's tables: the slot maps of one tile (load phase
        /// enumerates along the source-contiguous direction, store phase along the destination-
        /// contiguous one; `rot` rotates whole rows in the destination) and the origin of every
        /// tile.  They depend on the geometry only, so they are built once per distinct copy,
        /// uploaded and cached; the kernel then does no index arithmetic beyond one add per access.
        void build_tables(LaunchPlan &lp, bool has_src, int device, cudaStream_t stream) {
            const PermParams &p = lp.p;
            const size_t ne = (size_t)p.tile_elems, nt = p.ntiles;
            std::vector<unsigned> so(ne), dof(ne), sp(ne, 0);
            auto coords = [&](size_t e, const int *ord, int *c) {
                for (int q = 0; q < MAXT; ++q) c[q] = 0;
                for (int q = 0; q < p.nt; ++q) {
                    const int t = ord ? ord[q] : q;
                    c[t] = (int)(e % (size_t)p.text[t]);
                    e /= (size_t)p.text[t];
                }
            };
            for (size_t e = 0; e < ne; ++e) {
                int c[MAXT];
                coords(e, nullptr, c); // destination enumeration
                long long d = 0, sd = 0;
                int pos = 0;
                for (int q = 0; q < p.nt; ++q) {
                    int cd = c[q];
                    if (q == p.rot_q) cd = (cd + p.rot) % p.text[q];
                    d += cd * p.tds[q];
                    sd += c[q] * p.tss[q];
                    pos += c[q] * p.smem_stride[q];
                }
                dof[e] = (unsigned)d;
                so[e] = (unsigned)sd;
                if (lp.smem) {
                    coords(e, p.sord, c); // source enumeration
                    long long ssrc = 0;
                    int posl = 0;
                    for (int q = 0; q < p.nt; ++q) {
                        ssrc += c[q] * p.tss[q];
                        posl += c[q] * p.smem_stride[q];
                    }
                    so[e] = (unsigned)ssrc;
                    sp[e] = ((unsigned)posl << 16) | (unsigned)pos;
                }
            }
            std::vector<long long> tiles(2 * nt);
            {
                unsigned tc[KD] = {0};
                long long sb = 0, db = 0;
                for (size_t t = 0; t < nt; ++t) {
                    bool boundary = false;
                    for (int d = 0; d < p.nd; ++d)
                        if ((long long)(tc[d] + 1) * p.te[d] > p.size[d]) boundary = true;
                    tiles[2 * t] = sb | (boundary ? (long long)(1ull << 63) : 0ll);
                    tiles[2 * t + 1] = db;
                    // next tile: increment the odometer
                    for (int d = 0; d < p.nd; ++d) {
                        sb += p.tsstride[d], db += p.tdstride[d];
                        if (++tc[d] < p.ntile[d]) break;
                        sb -= (long long)p.ntile[d] * p.tsstride[d];
                        db -= (long long)p.ntile[d] * p.tdstride[d];
                        tc[d] = 0;
                    }
                }
            }
            (void)has_src;
            const size_t slot_bytes = (ne * sizeof(unsigned) + 255) / 256 * 256;
            const size_t total = 3 * slot_bytes + tiles.size() * sizeof(long long);
            char *mem = nullptr;
            if (g_table_bytes + total > kTableBudget) permute_cache_clear(); // bounded: the cache is a convenience
            cuda_check(cudaMalloc((void **)&mem, total), "cudaMalloc (copy tables)");
            g_table_bytes += total;
            cuda_check(cudaMemcpyAsync(mem, so.data(), ne * sizeof(unsigned), cudaMemcpyHostToDevice, stream), "table upload");
            cuda_check(cudaMemcpyAsync(mem + slot_bytes, dof.data(), ne * sizeof(unsigned), cudaMemcpyHostToDevice, stream), "table upload");
            cuda_check(cudaMemcpyAsync(mem + 2 * slot_bytes, sp.data(), ne * sizeof(unsigned), cudaMemcpyHostToDevice, stream), "table upload");
            cuda_check(cudaMemcpyAsync(mem + 3 * slot_bytes, tiles.data(), tiles.size() * sizeof(long long), cudaMemcpyHostToDevice, stream), "table upload");
            // The cached launch may later run on other streams (auxiliary stream, another call's
            // stream, a caller's stream through sbk_permute_copy): the tables must be complete in
            // device memory before anybody can see them.  Once per distinct geometry.
            cuda_check(cudaStreamSynchronize(stream), "table upload");
            lp.tab.so = (const unsigned *)mem;
            lp.tab.dof = (const unsigned *)(mem + slot_bytes);
            lp.tab.sp = (const unsigned *)(mem + 2 * slot_bytes);
            lp.tab.tiles = (const longlong2 *)(mem + 3 * slot_bytes);
            lp.tab_mem = mem;
            lp.tab_device = device;
        }

        /// Fill PermParams for a canonical box; `es` = bytes per element, `max_tile` = NT*EPT.
        LaunchPlan plan_launch(const Canon &c, int es, int max_tile, bool has_src) {
            LaunchPlan lp;
            lp.es = es;
            PermParams &p = lp.p;
            memset(&p, 0, sizeof p);
            p.nd = std::max(c.nd, 1);
            Canon cc = c;
            if (c.nd == 0) { // single element
                cc.nd = 1;
                cc.size = {1};
                cc.ss = {1};
                cc.ds = {1};
            }
            std::vector<int> sorder(cc.nd);
            std::iota(sorder.begin(), sorder.end(), 0);
            if (has_src)
                std::stable_sort(sorder.begin(), sorder.end(),
                                 [&](int x, int y) { return cc.ss[x] < cc.ss[y]; });
            // The fastest source dim must be contiguous for a source run to exist at all
            const bool src_contig = has_src && cc.ss[sorder[0]] == 1;
            const bool dst_contig = cc.ds[0] == 1;

            // candidate search: maximise covered bytes per side (capped at 512 B), then tile size
            Tiling best;
            double best_score = -1;
            if (cc.rot != 0) {
                // rotated rows: a tile holds whole rows
                if (cc.size[0] > max_tile) throw std::runtime_error("permute copy: row too long to rotate");
                best.te.assign(cc.nd, 1);
                best.te[0] = cc.size[0];
                best.total = best.run_d = best.run_s = cc.size[0];
                best_score = 0;
            }
            for (int64_t wd = 1; wd <= max_tile && cc.rot == 0; wd *= 2)
                for (int64_t ws = 1; ws <= max_tile; ws *= 2) {
                    Tiling t = build_tile(cc, sorder, dst_contig ? wd : 1, src_contig ? ws : 1);
                    if (t.total > max_tile) continue;
                    // count tiled dims
                    int nt = 0;
                    for (int d = 0; d < cc.nd; ++d) nt += t.te[d] > 1;
                    if (nt > MAXT) continue;
                    const double sd = (double)std::min<int64_t>(t.run_d * es, 512);
                    const double ssrc = has_src ? (double)std::min<int64_t>(t.run_s * es, 512) : 512;
                    const double score = (sd + ssrc) * 1e6 + (double)t.total;
                    if (score > best_score) best_score = score, best = t;
                }
            // grow small tiles along further destination dims so that a CTA has enough in flight
            for (int d = 0; d < cc.nd; ++d) {
                while (best.te[d] < cc.size[d] && best.total * 2 <= max_tile) {
                    int nt = 0;
                    for (int k = 0; k < cc.nd; ++k) nt += best.te[k] > 1;
                    if (best.te[d] == 1 && nt >= MAXT) break;
                    const int ne = std::min(cc.size[d], best.te[d] * 2);
                    if (best.total / best.te[d] * ne > max_tile) break;
                    best.total = best.total / best.te[d] * ne;
                    best.te[d] = ne;
                }
            }
            // 32-bit in-tile offsets: shrink extents on huge-stride dims if needed
            for (;;) {
                int64_t ms = 0, md = 0;
                int worst = -1;
                int64_t worst_v = 0;
                for (int d = 0; d < cc.nd; ++d) {
                    const int64_t vs = (best.te[d] - 1) * cc.ss[d], vd = (best.te[d] - 1) * cc.ds[d];
                    ms += vs, md += vd;
                    if (std::max(vs, vd) > worst_v) worst_v = std::max(vs, vd), worst = d;
                }
                if (ms < (1ll << 31) && md < (1ll << 31)) break;
                best.total /= best.te[worst];
                best.te[worst] = std::max(1, best.te[worst] / 2);
                best.total *= best.te[worst];
            }

            int64_t ntiles = 1;
            for (int d = 0; d < cc.nd; ++d) {
                p.size[d] = cc.size[d];
                p.te[d] = best.te[d];
                p.ntile[d] = (unsigned)((cc.size[d] + best.te[d] - 1) / best.te[d]);
                p.tsstride[d] = (long long)best.te[d] * cc.ss[d];
                p.tdstride[d] = (long long)best.te[d] * cc.ds[d];
                ntiles *= p.ntile[d];
            }
            if (ntiles >= (1ll << 31)) throw std::runtime_error("permute copy: too many tiles");
            p.ntiles = (unsigned)ntiles;
            p.nt = 0;
            for (int d = 0; d < cc.nd; ++d)
                if (best.te[d] > 1) {
                    p.tdim[p.nt] = d;
                    p.text[p.nt] = best.te[d];
                    p.tss[p.nt] = cc.ss[d];
                    p.tds[p.nt] = cc.ds[d];
                    ++p.nt;
                }
            p.tile_elems = (int)best.total;
            p.rot = cc.rot;
            p.rot_q = cc.rot != 0 ? 0 : -1; // dim 0 is tiled (te = size > 1), so it is tiled-dim slot 0
            // source enumeration order of the tiled dims
            std::vector<int> so(p.nt);
            std::iota(so.begin(), so.end(), 0);
            std::stable_sort(so.begin(), so.end(), [&](int x, int y) { return p.tss[x] < p.tss[y]; });
            bool same_order = true;
            for (int q = 0; q < p.nt; ++q) {
                p.sord[q] = so[q];
                if (so[q] != q) same_order = false;
            }
            lp.smem = has_src && !same_order;
            // shared memory layout: destination order, odd stride for the source-fastest dim
            int stride = 1;
            for (int q = 0; q < p.nt; ++q) {
                if (lp.smem && q > 0 && q == so[0] && stride % 2 == 0) stride += 1;
                p.smem_stride[q] = stride;
                stride *= p.text[q];
            }
            p.smem_elems = lp.smem ? stride : 0;
            if (p.smem_elems > 65535) throw std::runtime_error("permute copy: tile too large");
            lp.run_d = best.run_d, lp.run_s = best.run_s;
            return lp;
        }

        struct DevInfo {
            int sms = 0;
        };
        DevInfo &dev_info(int device) {
            static DevInfo info[64];
            if (info[device].sms == 0) {
                cudaDeviceProp prop;
                cuda_check(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties");
                info[device].sms = prop.multiProcessorCount;
            }
            return info[device];
        }

        template <class Kernel> int resident_ctas(Kernel k, size_t smem_bytes) {
            if (smem_bytes > 48 * 1024)
                cuda_check(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                (int)smem_bytes),
                           "cudaFuncSetAttribute");
            int n = 0;
            cuda_check(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k, NT, smem_bytes),
                       "cudaOccupancyMaxActiveBlocksPerMultiprocessor");
            return std::max(n, 1);
        }

        /// Returns true when `xs` rode on the launched kernel
        template <class Op, bool MASK = false, int EPT_ = EPT>
        bool launch_perm(LaunchPlan &lp, const void *src, void *dst, Op op, int device,
                         cudaStream_t stream, int cap, const ExchangeSync *xs,
                         const float *ma = nullptr, const float *mb = nullptr, bool ma_src = false) {
            using T = typename Op::T;
            using Q = typename Op::Q;
            // (masked, transposing: one flag byte per tile element behind the element tile)
            const size_t smem_bytes = (size_t)lp.p.smem_elems * sizeof(T) + (MASK ? (size_t)lp.p.smem_elems : 0);
            auto go = [&](auto kernel) {
                // resident CTAs per SM for this kernel, cached by dynamic shared-memory size
                static std::map<size_t, int> ctas;
                auto it = ctas.find(smem_bytes);
                if (it == ctas.end()) it = ctas.emplace(smem_bytes, resident_ctas(kernel, smem_bytes)).first;
                unsigned grid = (unsigned)std::min<int64_t>(
                    lp.p.ntiles, (int64_t)dev_info(device).sms * it->second);
                if (cap > 0) grid = std::min<unsigned>(grid, (unsigned)cap);
                {
                    KernelTimer timer("permute", stream);
                    kernel<<<grid, NT, smem_bytes, stream>>>(lp.p, lp.tab, (const T *)src, (Q *)dst, op,
                                                             ma, mb, ma_src, xs ? *xs : ExchangeSync{});
                }
                count_launch();
                cuda_check(cudaGetLastError(), "permute_kernel launch");
            };
            // small elements: three resident CTAs per SM (more loads in flight per SM for the same bytes)
            constexpr int MINB = ((sizeof(T) <= 8 && sizeof(Q) <= 8 && EPT_ <= 8 && !MASK) || (MASK && EPT_ <= 4)) ? 3 : 2;
            if (lp.smem)
                go(permute_kernel<Op, true, EPT_, MINB, MASK>);
            else
                go(permute_kernel<Op, false, EPT_, MINB, MASK>);
            return xs != nullptr;
        }

        template <class V>
        void launch_zero(LaunchPlan &lp, void *dst, int device, cudaStream_t stream,
                         const float *ma = nullptr, const float *mb = nullptr) {
            const unsigned grid =
                (unsigned)std::min<int64_t>(lp.p.ntiles, (int64_t)dev_info(device).sms * 8);
            zero_kernel<V><<<grid, NT, 0, stream>>>(lp.p, (V *)dst, ma, mb);
            count_launch();
            cuda_check(cudaGetLastError(), "zero_kernel launch");
        }

        /// Slots per thread of the raw-move kernels: 4- and 8-byte elements get 16 when the tile is
        /// transposed through shared memory (a tile must hold runs of >= 256 B on both sides and
        /// enough bytes in flight; measured +17 % for float, +7 % for 8-byte transposes), 8 otherwise
        /// (the direct variant double-buffers in registers)
        int ept_for(int es) { return es == 4 || es == 8 ? 16 : EPT; }
        int max_tile_for(int es) { return NT * ept_for(es); }

        /// Widen the element when the fastest dim is shared, contiguous and aligned
        int promote(Canon &c, int es, const void *src, const void *dst, bool has_src) {
            if (c.nd < 1 || c.ds[0] != 1 || (has_src && c.ss[0] != 1)) return es;
            int f = 16 / es;
            for (; f > 1; f /= 2) {
                bool ok = true;
                if (c.size[0] % f || c.rot % f) ok = false;
                for (int d = 1; ok && d < c.nd; ++d)
                    if (c.ds[d] % f || (has_src && c.ss[d] % f)) ok = false;
                if (ok && (c.doff % f || (has_src && c.soff % f))) ok = false;
                if (ok && ((uintptr_t)dst + (uintptr_t)c.doff * es) % ((size_t)f * es)) ok = false;
                if (ok && has_src && ((uintptr_t)src + (uintptr_t)c.soff * es) % ((size_t)f * es))
                    ok = false;
                if (ok) break;
            }
            if (f <= 1) return es;
            c.rot /= f;
            c.size[0] /= f;
            for (int d = 1; d < c.nd; ++d) {
                c.ds[d] /= f;
                if (has_src) c.ss[d] /= f;
            }
            c.doff /= f;
            if (has_src) c.soff /= f;
            // the widened dim may now merge with the next one, or vanish
            if (c.size[0] == 1) {
                c.size.erase(c.size.begin());
                c.ss.erase(c.ss.begin());
                c.ds.erase(c.ds.begin());
                c.nd--;
            }
            return es * f;
        }

        template <typename T> T make_elem(const double *a);
        template <> float make_elem<float>(const double *a) { return (float)a[0]; }
        template <> double make_elem<double>(const double *a) { return a[0]; }
        template <> int make_elem<int>(const double *a) { return (int)a[0]; }
        template <> float2 make_elem<float2>(const double *a) {
            return make_float2((float)a[0], (float)a[1]);
        }
        template <> double2 make_elem<double2>(const double *a) { return make_double2(a[0], a[1]); }

        template <typename T, typename Q>
        bool launch_typed(LaunchPlan &lp, const void *src, void *dst, const double *alpha,
                          bool scale, bool add, int device, cudaStream_t stream, int cap,
                          const ExchangeSync *xs, const float *ma, const float *mb, bool ma_src) {
            if (ma || mb) // (planned with MASK_EPT slots per thread, see prepare)
                return launch_perm<ElemOp<T, Q>, true, MASK_EPT>(lp, src, dst, {make_elem<T>(alpha), scale, add},
                                                                 device, stream, cap, xs, ma, mb, ma_src);
            return launch_perm<ElemOp<T, Q>>(lp, src, dst, {make_elem<T>(alpha), scale, add}, device,
                                             stream, cap, xs);
        }

        bool convertible(int dt0, int dt1) {
            if (dt0 == dt1) return true;
            return (dt0 == SBB_F32 && dt1 == SBB_F64) || (dt0 == SBB_F64 && dt1 == SBB_F32) ||
                   (dt0 == SBB_C64 && dt1 == SBB_C128) || (dt0 == SBB_C128 && dt1 == SBB_C64);
        }

        /// Kernel of a box: fill with zeros, move raw (widened) elements, or scale / convert / add
        enum Kind { Zero, Move, Typed };

        struct Prepared {
            Canon c;
            LaunchPlan lp;
            int es; ///< destination element size after widening
        };
        std::map<std::string, Prepared> &prepared_cache() {
            static std::map<std::string, Prepared> cache;
            return cache;
        }

        /// The launch of one box: from the cache, or planned (with the tables the kernel reads).
        /// The offsets of the result are c0's, in elements of the widened size.
        Prepared prepare(Kind kind, const Canon &c0, const void *src, int dt0, void *dst, int dt1,
                         bool masked, bool is_zero, bool is_one, bool add, int device,
                         cudaStream_t stream, bool describe) {
            // Prepared launches are cached by geometry, types, flags and pointer alignment: the
            // tiling search runs once per distinct copy (the reference caches its index vectors
            // the same way, tensor.h:946-951 -- here the cached object is ~0.5 KB, not the index).
            auto &cache = prepared_cache();
            std::string key;
            {
                auto put = [&](const void *ptr, size_t n) { key.append((const char *)ptr, n); };
                const int flags[8] = {dt0, dt1, is_zero, is_one, add,
                                      (int)(((uintptr_t)src & 15) | (((uintptr_t)dst & 15) << 4)),
                                      device, masked};
                put(flags, sizeof flags);
                put(&c0.nd, sizeof c0.nd);
                put(c0.size.data(), c0.size.size() * sizeof(int));
                put(c0.ss.data(), c0.ss.size() * sizeof(int64_t));
                put(c0.ds.data(), c0.ds.size() * sizeof(int64_t));
                put(&c0.rot, sizeof c0.rot);
                // the offsets only matter through what the widening of the element may assume about
                // them (promote): their residues, not their values -- a sweep of sub-boxes over a big
                // tensor shares one entry (and one device table) instead of creating one per offset
                const int res[2] = {(int)(c0.soff & 15), (int)(c0.doff & 15)};
                put(res, sizeof res);
            }
            auto hit = describe ? cache.end() : cache.find(key);
            Prepared p;
            if (hit != cache.end()) {
                p = hit->second;
            } else {
                p.c = c0;
                switch (kind) {
                case Zero: // (masks are per element: no widening)
                    p.es = masked ? dtype_bytes(dt1) : promote(p.c, dtype_bytes(dt1), nullptr, dst, false);
                    p.lp = plan_launch(p.c, p.es, NT * EPT, false);
                    break;
                case Move:
                    p.es = promote(p.c, dtype_bytes(dt0), src, dst, true);
                    p.lp = plan_launch(p.c, p.es, max_tile_for(p.es), true);
                    if (!p.lp.smem && p.lp.p.tile_elems > NT * EPT) p.lp = plan_launch(p.c, p.es, NT * EPT, true);
                    break;
                case Typed: // native elements
                    p.es = dtype_bytes(dt1);
                    p.lp = plan_launch(p.c, std::max(dtype_bytes(dt0), p.es), NT * (masked ? MASK_EPT : EPT), true);
                    break;
                }
                if (!describe) {
                    if (kind != Zero) build_tables(p.lp, true, device, stream);
                    if (cache.size() > 8192) permute_cache_clear();
                    cache[key] = p;
                }
            }
            // (a cached entry may come from another offset with the same residue)
            const int f = p.es / dtype_bytes(dt1);
            p.c.soff = c0.soff / f, p.c.doff = c0.doff / f;
            return p;
        }

        /// Run (or describe) one box of at most KD (canonical) dims; true when `opt.xs` rode on its kernel
        bool run_box(const Canon &c0, const void *src, int dt0, void *dst, int dt1, const double *alpha,
                     bool add, int device, cudaStream_t stream, const PermuteOptions &opt,
                     std::string *describe) {
            const bool ma_src = opt.mask_src != nullptr;
            const float *ma = ma_src ? opt.mask_src : opt.mask_a, *mb = opt.mask_b;
            const bool masked = ma || mb; // masks are per element: typed kernel
            const bool is_zero = scalar_is(dt0, alpha, 0), is_one = scalar_is(dt0, alpha, 1);
            if (is_zero && add) return false;
            const Kind kind = is_zero ? Zero : dt0 == dt1 && is_one && !add && !masked ? Move : Typed;
            Prepared pr = prepare(kind, c0, src, dt0, dst, dt1, masked, is_zero, is_one, add, device,
                                  stream, describe != nullptr);
            const Canon &c = pr.c;
            LaunchPlan &lp = pr.lp;
            const int es = pr.es, es0 = dtype_bytes(dt0);
            if (describe) {
                std::stringstream ds;
                if (kind == Zero)
                    ds << (masked ? "masked " : "") << "zero es=" << es << " tile=" << lp.p.tile_elems
                       << " ntiles=" << lp.p.ntiles;
                else if (kind == Move)
                    ds << (lp.smem ? "move tiled" : "move direct") << " es=" << es
                       << " tile=" << lp.p.tile_elems << " ntiles=" << lp.p.ntiles
                       << " run_dst=" << lp.run_d * es << "B run_src=" << lp.run_s * es << "B nd="
                       << lp.p.nd;
                else
                    ds << (masked ? "masked " : "") << (lp.smem ? "typed tiled" : "typed direct") << " es=" << es0
                       << "->" << es << " tile=" << lp.p.tile_elems << " ntiles=" << lp.p.ntiles
                       << " scale=" << !is_one << " add=" << add;
                *describe = ds.str();
                return false;
            }
            char *d = (char *)dst + c.doff * es;
            if (kind == Zero) {
                // (no source here: a source-layout mask does not apply to a zero fill)
                const float *xa = ma && !ma_src ? ma + c.doff : nullptr, *xb = mb ? mb + c.doff : nullptr;
                if (es == 16) launch_zero<uint4>(lp, d, device, stream, xa, xb);
                else if (es == 8) launch_zero<uint2>(lp, d, device, stream, xa, xb);
                else launch_zero<unsigned>(lp, d, device, stream, xa, xb);
                return false;
            }
            const char *s = (const char *)src + c.soff * (kind == Move ? es : es0);
            const int cap = opt.grid_cap;
            const ExchangeSync *xs = opt.xs;
            if (kind == Move) {
                const bool wide = lp.p.tile_elems > NT * EPT; // planned with 16 slots per thread
                if (es == 16) return launch_perm<MoveOp<uint4>>(lp, s, d, {}, device, stream, cap, xs);
                if (es == 8 && wide) return launch_perm<MoveOp<uint2>, false, 16>(lp, s, d, {}, device, stream, cap, xs);
                if (es == 8) return launch_perm<MoveOp<uint2>>(lp, s, d, {}, device, stream, cap, xs);
                if (wide) return launch_perm<MoveOp<unsigned>, false, 16>(lp, s, d, {}, device, stream, cap, xs);
                return launch_perm<MoveOp<unsigned>>(lp, s, d, {}, device, stream, cap, xs);
            }
#define SBB_TYPED(DT0, DT1, T, Q)                                                                  \
    if (dt0 == DT0 && dt1 == DT1)                                                                  \
        return launch_typed<T, Q>(lp, s, d, alpha, !is_one, add, device, stream, cap, xs,          \
                                  ma ? ma + (ma_src ? c.soff : c.doff) : nullptr,                  \
                                  mb ? mb + c.doff : nullptr, ma_src);
            SBB_TYPED(SBB_F32, SBB_F32, float, float)
            SBB_TYPED(SBB_F64, SBB_F64, double, double)
            SBB_TYPED(SBB_C64, SBB_C64, float2, float2)
            SBB_TYPED(SBB_C128, SBB_C128, double2, double2)
            SBB_TYPED(SBB_I32, SBB_I32, int, int)
            SBB_TYPED(SBB_F32, SBB_F64, float, double)
            SBB_TYPED(SBB_F64, SBB_F32, double, float)
            SBB_TYPED(SBB_C64, SBB_C128, float2, double2)
            SBB_TYPED(SBB_C128, SBB_C64, double2, float2)
#undef SBB_TYPED
            throw std::runtime_error("permute copy: unsupported type combination");
        }

    } // namespace

    // ---- peer-memory signalling (the "barrier" of an exchange, without NCCL on the data path) ---------
    namespace {
        /// After the pack kernels of a round (same stream, so their stores -- including the ones that
        /// went to peer memory over NVLink -- are complete): raise my flag in every rank's arena.
        __global__ void signal_kernel(unsigned long long *const *peer_flags, int me, int nranks,
                                      unsigned long long seq) {
            const int q = threadIdx.x;
            if (q < nranks) {
                unsigned long long *f = peer_flags[q] + me;
                asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(f), "l"(seq) : "memory");
            }
        }
        /// Before the unpack kernels of a round: wait until every rank has raised its flag to `seq`.
        /// The spin is bounded: after `timeout_ns` without the flags the kernel gives up and writes the
        /// missing rank + 1 to `*error` (host-mapped), which the next library call turns into an
        /// exception instead of a wedged GPU.
        __global__ void wait_kernel(const unsigned long long *flags, int nranks, unsigned long long seq,
                                    unsigned long long timeout_ns, int *error) {
            const int r = threadIdx.x;
            if (r < nranks) {
                unsigned long long v, t0 = 0;
                unsigned spins = 0;
                for (;;) { // relaxed polling (served by L2, where the peers' stores land); one fence at the end
                    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flags + r) : "memory");
                    if (v >= seq) break;
                    __nanosleep(100);
                    if ((++spins & 1023u) == 0) {
                        unsigned long long now;
                        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                        if (t0 == 0) t0 = now;
                        else if (now - t0 > timeout_ns) {
                            if (error) *(volatile int *)error = r + 1;
                            break;
                        }
                    }
                }
            }
            __syncthreads();
            __threadfence_system();
        }
    }

    void launch_signal(unsigned long long *const *peer_flags, int me, int nranks,
                       unsigned long long seq, cudaStream_t stream) {
        signal_kernel<<<1, std::max(32, (nranks + 31) / 32 * 32), 0, stream>>>(peer_flags, me, nranks, seq);
        count_launch();
        cuda_check(cudaGetLastError(), "signal_kernel launch");
    }

    void launch_wait(const unsigned long long *flags, int nranks, unsigned long long seq,
                     cudaStream_t stream, unsigned long long timeout_ns, int *error) {
        wait_kernel<<<1, std::max(32, (nranks + 31) / 32 * 32), 0, stream>>>(flags, nranks, seq,
                                                                            timeout_ns, error);
        count_launch();
        cuda_check(cudaGetLastError(), "wait_kernel launch");
    }

    void permute_cache_clear() {
        for (auto &kv : prepared_cache()) {
            LaunchPlan &lp = kv.second.lp;
            if (lp.tab_mem) {
                cudaSetDevice(lp.tab_device);
                cudaDeviceSynchronize();
                cudaFree(lp.tab_mem);
            }
        }
        prepared_cache().clear();
        g_table_bytes = 0;
    }

    bool permute_copy(const sbk_box_desc &box, const void *src, int dt0, void *dst, int dt1,
                      const double *alpha, bool add, int device, cudaStream_t stream,
                      const PermuteOptions &opt, std::string *describe) {
        if (box.nd < 0 || box.nd > SBK_MAX_DIMS) throw std::runtime_error("permute copy: bad nd");
        if (opt.mask_src && opt.mask_a) throw std::runtime_error("permute copy: the source mask is given twice");
        if (!convertible(dt0, dt1))
            throw std::runtime_error("permute copy: unsupported type combination");
        Canon c = canonicalize(box, !scalar_is(dt0, alpha, 0));
        if (c.nd < 0) {
            if (describe) *describe = "empty";
            return false;
        }
        if (c.nd <= KD) return run_box(c, src, dt0, dst, dt1, alpha, add, device, stream, opt, describe);
        // More than KD irreducible dims: iterate over the slowest ones on the host (a signal must not
        // ride on a partial launch)
        PermuteOptions part = opt;
        part.xs = nullptr;
        const int outer = c.nd - KD;
        std::vector<int> idx(outer, 0);
        for (;;) {
            Canon sub = c;
            sub.nd = KD;
            sub.size.resize(KD), sub.ss.resize(KD), sub.ds.resize(KD);
            for (int k = 0; k < outer; ++k) {
                sub.soff += idx[k] * c.ss[KD + k];
                sub.doff += idx[k] * c.ds[KD + k];
            }
            run_box(sub, src, dt0, dst, dt1, alpha, add, device, stream, part, describe);
            if (describe) return false;
            int k = 0;
            for (; k < outer; ++k) {
                if (++idx[k] < c.size[KD + k]) break;
                idx[k] = 0;
            }
            if (k == outer) break;
        }
        return false;
    }

} // namespace sbb
