// Block-sparse operator times a multi-vector (bsr_kernel.hpp): one launch per operator component.
// Two tiers, chosen from the block sizes and the column count:
//  * warp tier (vol(blockim) <= 32: the 12 x 12 spin-colour blocks, 4 x 4, ...): one warp per block
//    row and column chunk, up to 8 per CTA.  A warp loads each block's contiguous run of v with
//    consecutive lanes on consecutive elements and the block's input slab (columns fastest, so one
//    contiguous run per domain point) into its shared-memory scratch, then each lane accumulates up
//    to 8 outputs in registers.
//  * CTA tier (larger blocks: coarse operators): one CTA of 256 threads per block row and column
//    chunk, up to 16 outputs per thread in registers; blocks stream through shared memory in pieces
//    of the domain index that fit the budget.
// Every matrix block is read from HBM once per column chunk; offsets are 64-bit throughout.  A launch
// covers the block rows [0, nrows), or the list `rows` when one is given (bsr_krylov's interior and
// boundary rows, bsr_plan.cpp); the list only changes which row a team takes.
// Kronecker operators (kron_bsr_kernel, profile name "kron_bsr") have the same two tiers, chosen by
// vol(kronim) * vol(blockim) <= 32 (spin-colour: 4 x 3 = 12).  A CTA first loads the U factors and the
// input-point table into shared memory; each team then streams its row's blocks through its scratch a
// piece of `nu` blocks at a time (B, the x slab, t in Acc<T>) and accumulates the Kronecker sum in
// registers.  There are no domain pieces: one block and one column of its input must fit the team's
// budget, and the factors 64 KiB.
#include "bsr_kernel.hpp"
#include "kernels.hpp"
#include <algorithm>
#include <sstream>

namespace sbb {

    namespace {
        using namespace bsrk;

        constexpr int CTA_THREADS = 256, MAX_WARPS = 8, WARP_OUT = 8, CTA_OUT = 16;
        constexpr int64_t WARP_TEAM_BUDGET = 12 * 1024, CTA_TEAM_BUDGET = 96 * 1024;

        struct BsrParams {
            sbk_bsr_desc d;
            int m, nchunks, kd, teams;
            int64_t team_bytes, table_bytes;
        };

        struct WarpTeam {
            int t, nt;
            __device__ void sync() const { __syncwarp(); }
        };
        struct CtaTeam {
            int t, nt;
            __device__ void sync() const { __syncthreads(); }
        };

        /// A team's unit of work: block row r (from the list when there is one), columns [c0, c0 + m)
        struct Unit {
            int team, c0, m;
            int64_t r;
        };

        /// The unit of this thread's team (a warp, or the CTA); false when the team has none
        template <bool Warp>
        __device__ bool team_unit(const sbk_bsr_desc &d, int teams, int nchunks, int chunk, Unit &u) {
            u.team = Warp ? threadIdx.x / 32 : 0;
            const int64_t unit = (int64_t)blockIdx.x * teams + u.team;
            if (unit >= (d.rows ? d.nlist : d.nrows) * nchunks) return false;
            u.r = d.rows ? d.rows[unit / nchunks] : unit / nchunks;
            u.c0 = (int)(unit % nchunks) * chunk;
            u.m = d.ncols - u.c0 < chunk ? d.ncols - u.c0 : chunk;
            return true;
        }

        template <typename T, bool Warp>
        __global__ void __launch_bounds__(CTA_THREADS)
            bsr_kernel(const __grid_constant__ BsrParams p, const T *__restrict__ v, const T *__restrict__ x,
                       T *__restrict__ y, AccT<T> alpha, AccT<T> beta) {
            extern __shared__ __align__(16) unsigned char smem[];
            const sbk_bsr_desc &d = p.d;
            int64_t *xo = (int64_t *)smem;
            for (int j = threadIdx.x; j < d.bd; j += blockDim.x) xo[j] = domain_point(d, j);
            __syncthreads();
            Unit u;
            if (!team_unit<Warp>(d, p.teams, p.nchunks, p.m, u)) return; // a whole team leaves: no barrier of the CTA follows
            T *as = (T *)(smem + p.table_bytes + u.team * p.team_bytes);
            T *xs = as + (int64_t)d.bi * p.kd;
            if (Warp) {
                const WarpTeam tm{(int)(threadIdx.x % 32), 32};
                row_body<WARP_OUT>(d, u.r, u.c0, u.m, p.kd, v, x, y, alpha, beta, as, xs, xo, tm);
            } else {
                const CtaTeam tm{(int)threadIdx.x, (int)blockDim.x};
                row_body<CTA_OUT>(d, u.r, u.c0, u.m, p.kd, v, x, y, alpha, beta, as, xs, xo, tm);
            }
        }

        int64_t up16(int64_t b) { return (b + 15) & ~(int64_t)15; }

        /// Launches `kernel` (profile name `name`) over the units of p (block rows times column chunks): in
        /// the warp tier one warp per unit, up to MAX_WARPS per CTA, else one CTA per unit, with `fixed`
        /// bytes of shared memory plus `team` per team.  Sets p.teams.  With `describe` the sizes of the
        /// launch are appended to the text there instead; nothing is launched without units or if `empty`.
        template <typename K, typename P, typename... A>
        void launch(K kernel, const char *name, bool warp, int64_t fixed, int64_t team, bool empty, P &p,
                    cudaStream_t stream, std::string *describe, A... args) {
            const int64_t units = (p.d.rows ? p.d.nlist : p.d.nrows) * p.nchunks;
            p.teams = warp ? (int)std::max<int64_t>(1, std::min<int64_t>(MAX_WARPS, units)) : 1;
            const int threads = warp ? 32 * p.teams : CTA_THREADS;
            const int64_t smem = fixed + p.teams * team;
            const int64_t grid = (units + p.teams - 1) / p.teams;
            if (describe) {
                std::stringstream ss;
                ss << " teams=" << p.teams << " grid=" << grid << " threads=" << threads << " smem=" << smem;
                *describe += ss.str();
                return;
            }
            if (units == 0 || empty) return;
            if (grid > 0x7fffffff) throw std::runtime_error("bsr_krylov: too many block rows in one launch");
            cuda_check(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                       "cudaFuncSetAttribute");
            {
                KernelTimer timer(name, stream);
                kernel<<<(unsigned)grid, threads, (size_t)smem, stream>>>(p, args...);
            }
            count_launch();
            if (const cudaError_t e = cudaGetLastError()) cuda_check(e, (std::string(name) + "_kernel launch").c_str());
        }

        template <typename T>
        void run(const sbk_bsr_desc &d, const double *alpha, const double *beta, const void *v, const void *x,
                 void *y, cudaStream_t stream, std::string *describe) {
            const int es = (int)sizeof(T);
            if (d.bi > CTA_THREADS * CTA_OUT || d.bd > 4096)
                throw std::runtime_error("bsr_krylov: blocks larger than 4096 x 4096 elements are not supported");
            BsrParams p;
            p.d = d;
            const bool warp = d.bi <= 32;
            const int out = warp ? 32 * WARP_OUT : CTA_THREADS * CTA_OUT;
            p.m = std::max(1, std::min(d.ncols, out / std::max(d.bi, 1)));
            p.nchunks = d.ncols > 0 ? (d.ncols + p.m - 1) / p.m : 0;
            const int64_t budget = warp ? WARP_TEAM_BUDGET : CTA_TEAM_BUDGET;
            p.kd = (int)std::max<int64_t>(1, std::min<int64_t>(d.bd, budget / ((int64_t)(d.bi + p.m) * es)));
            p.team_bytes = up16((int64_t)(d.bi + p.m) * p.kd * es);
            p.table_bytes = up16(8 * (int64_t)std::max(d.bd, 1));
            if (describe) {
                std::stringstream ss;
                ss << "bsr tier=" << (warp ? "warp" : "cta") << " rows=" << d.nrows << " bi=" << d.bi
                   << " bd=" << d.bd << " cols=" << d.ncols << " chunk=" << p.m << " kd=" << p.kd;
                *describe = ss.str();
            }
            launch(warp ? bsr_kernel<T, true> : bsr_kernel<T, false>, "bsr", warp, p.table_bytes, p.team_bytes,
                   d.bi == 0, p, stream, describe, (const T *)v, (const T *)x, (T *)y, scalar_of<T>(alpha),
                   scalar_of<T>(beta));
        }

        // ---- Kronecker operators (create_kron_bsr) ----------------------------------------------------

        struct KronParams {
            sbk_bsr_desc d;
            sbk_kron_desc k;
            int m, nchunks, nu, teams;
            int64_t team_bytes, table_bytes, factor_bytes, xs_off, ts_off; ///< xs, ts: offsets in a team's scratch
        };

        /// Shared memory: the factors, the xo table, then per team bs | xs | ts (16-byte aligned each)
        template <typename T, bool Warp>
        __global__ void __launch_bounds__(CTA_THREADS)
            kron_bsr_kernel(const __grid_constant__ KronParams p, const T *__restrict__ v, const T *__restrict__ kv,
                            const T *__restrict__ x, T *__restrict__ y, AccT<T> alpha, AccT<T> beta) {
            extern __shared__ __align__(16) unsigned char smem[];
            const sbk_bsr_desc &d = p.d;
            const sbk_kron_desc &kr = p.k;
            T *ks = (T *)smem;
            int64_t *xo = (int64_t *)(smem + p.factor_bytes);
            for (int e = threadIdx.x; e < kr.u * kr.ki * kr.kd; e += blockDim.x) ks[e] = kv[e];
            for (int j = threadIdx.x; j < kr.kd * d.bd; j += blockDim.x) xo[j] = kron_domain_point(d, kr, j / d.bd, j % d.bd);
            __syncthreads();
            Unit u;
            if (!team_unit<Warp>(d, p.teams, p.nchunks, p.m, u)) return; // a whole team leaves: no barrier of the CTA follows
            unsigned char *base = smem + p.factor_bytes + p.table_bytes + u.team * p.team_bytes;
            T *bs = (T *)base;
            T *xs = (T *)(base + p.xs_off);
            AccT<T> *ts = (AccT<T> *)(base + p.ts_off);
            if (Warp) {
                const WarpTeam tm{(int)(threadIdx.x % 32), 32};
                kron_row_body<WARP_OUT>(d, kr, u.r, u.c0, u.m, p.nu, v, ks, x, y, alpha, beta, bs, xs, ts, xo, tm);
            } else {
                const CtaTeam tm{(int)threadIdx.x, (int)blockDim.x};
                kron_row_body<CTA_OUT>(d, kr, u.r, u.c0, u.m, p.nu, v, ks, x, y, alpha, beta, bs, xs, ts, xo, tm);
            }
        }

        constexpr int64_t KRON_FACTOR_BUDGET = 64 * 1024;

        template <typename T>
        void run_kron(const sbk_bsr_desc &d, const sbk_kron_desc &k, const double *alpha, const double *beta,
                      const void *v, const void *kv, const void *x, void *y, cudaStream_t stream,
                      std::string *describe) {
            const int64_t es = sizeof(T), as = sizeof(AccT<T>);
            KronParams p;
            p.d = d, p.k = k;
            const int bi = std::max(d.bi, 1), bd = std::max(d.bd, 1);
            const int64_t kib = (int64_t)k.ki * bi;
            const bool warp = kib <= 32;
            const int64_t budget = warp ? WARP_TEAM_BUDGET : CTA_TEAM_BUDGET;
            // per block of a piece: B, then its input slab and t for m columns
            auto per_block = [&](int64_t m) { return up16((int64_t)bi * bd * es) + up16((int64_t)k.kd * bd * m * es) +
                                                     up16((int64_t)k.kd * bi * m * as); };
            p.factor_bytes = up16((int64_t)k.u * k.ki * k.kd * es);
            if (kib > CTA_THREADS * CTA_OUT || per_block(1) > budget || p.factor_bytes > KRON_FACTOR_BUDGET)
                throw std::runtime_error(
                    "bsr_krylov: Kronecker operators need vol(kronim) * vol(blockim) <= 4096, the U factors within "
                    "64 KiB and one block with one column of its input within 96 KiB");
            const int64_t out = warp ? 32 * WARP_OUT : CTA_THREADS * CTA_OUT;
            p.m = (int)std::max<int64_t>(1, std::min<int64_t>(d.ncols, out / kib));
            while (p.m > 1 && per_block(p.m) > budget) p.m = (p.m + 1) / 2;
            p.nchunks = d.ncols > 0 ? (d.ncols + p.m - 1) / p.m : 0;
            p.nu = (int)std::max<int64_t>(1, std::min<int64_t>(k.u, budget / per_block(p.m)));
            p.xs_off = up16(p.nu * (int64_t)bi * bd * es);
            p.ts_off = p.xs_off + up16(p.nu * (int64_t)k.kd * bd * p.m * es);
            p.team_bytes = p.ts_off + up16(p.nu * (int64_t)k.kd * bi * p.m * as);
            p.table_bytes = up16(8 * (int64_t)k.kd * bd);
            if (describe) {
                std::stringstream ss;
                ss << "kron_bsr tier=" << (warp ? "warp" : "cta") << " rows=" << d.nrows << " bi=" << d.bi
                   << " bd=" << d.bd << " ki=" << k.ki << " kd=" << k.kd << " u=" << k.u << " cols=" << d.ncols
                   << " chunk=" << p.m << " nu=" << p.nu;
                *describe = ss.str();
            }
            launch(warp ? kron_bsr_kernel<T, true> : kron_bsr_kernel<T, false>, "kron_bsr", warp,
                   p.factor_bytes + p.table_bytes, p.team_bytes, d.bi == 0 || k.ki == 0, p, stream, describe,
                   (const T *)v, (const T *)kv, (const T *)x, (T *)y, scalar_of<T>(alpha), scalar_of<T>(beta));
        }
    } // namespace

    void bsr(const sbk_bsr_desc &d, int dtype, const double *alpha, const double *beta, const void *v,
             const void *x, void *y, cudaStream_t stream, std::string *describe) {
        switch (dtype) {
        case SBB_F32: return run<float>(d, alpha, beta, v, x, y, stream, describe);
        case SBB_F64: return run<double>(d, alpha, beta, v, x, y, stream, describe);
        case SBB_C64: return run<float2>(d, alpha, beta, v, x, y, stream, describe);
        case SBB_C128: return run<double2>(d, alpha, beta, v, x, y, stream, describe);
        default: throw std::runtime_error("bsr_krylov: unsupported type");
        }
    }

    void kron_bsr(const sbk_bsr_desc &d, const sbk_kron_desc &k, int dtype, const double *alpha,
                  const double *beta, const void *v, const void *kv, const void *x, void *y, cudaStream_t stream,
                  std::string *describe) {
        switch (dtype) {
        case SBB_F32: return run_kron<float>(d, k, alpha, beta, v, kv, x, y, stream, describe);
        case SBB_F64: return run_kron<double>(d, k, alpha, beta, v, kv, x, y, stream, describe);
        case SBB_C64: return run_kron<float2>(d, k, alpha, beta, v, kv, x, y, stream, describe);
        case SBB_C128: return run_kron<double2>(d, k, alpha, beta, v, kv, x, y, stream, describe);
        default: throw std::runtime_error("bsr_krylov: unsupported type");
        }
    }

} // namespace sbb
