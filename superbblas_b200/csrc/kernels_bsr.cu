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
// Every matrix block is read from HBM once per column chunk; offsets are 64-bit throughout.
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

        template <typename T, bool Warp>
        __global__ void __launch_bounds__(CTA_THREADS)
            bsr_kernel(const __grid_constant__ BsrParams p, const T *__restrict__ v, const T *__restrict__ x,
                       T *__restrict__ y, AccT<T> alpha, AccT<T> beta) {
            extern __shared__ __align__(16) unsigned char smem[];
            const sbk_bsr_desc &d = p.d;
            int64_t *xo = (int64_t *)smem;
            for (int j = threadIdx.x; j < d.bd; j += blockDim.x) xo[j] = domain_point(d, j);
            __syncthreads();
            const int team = Warp ? threadIdx.x / 32 : 0;
            const int64_t unit = (int64_t)blockIdx.x * p.teams + team;
            if (unit >= d.nrows * p.nchunks) return; // a whole team leaves: no barrier of the CTA follows
            const int64_t r = unit / p.nchunks;
            const int c0 = (int)(unit % p.nchunks) * p.m;
            const int m = d.ncols - c0 < p.m ? d.ncols - c0 : p.m;
            T *as = (T *)(smem + p.table_bytes + team * p.team_bytes);
            T *xs = as + (int64_t)d.bi * p.kd;
            if (Warp) {
                const WarpTeam tm{(int)(threadIdx.x % 32), 32};
                row_body<WARP_OUT>(d, r, c0, m, p.kd, v, x, y, alpha, beta, as, xs, xo, tm);
            } else {
                const CtaTeam tm{(int)threadIdx.x, (int)blockDim.x};
                row_body<CTA_OUT>(d, r, c0, m, p.kd, v, x, y, alpha, beta, as, xs, xo, tm);
            }
        }

        int64_t up16(int64_t b) { return (b + 15) & ~(int64_t)15; }

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
            const int64_t units = d.nrows * p.nchunks;
            p.teams = warp ? (int)std::max<int64_t>(1, std::min<int64_t>(MAX_WARPS, units)) : 1;
            const int threads = warp ? 32 * p.teams : CTA_THREADS;
            const int64_t smem = p.table_bytes + p.teams * p.team_bytes;
            const int64_t grid = (units + p.teams - 1) / p.teams;
            if (describe) {
                std::stringstream ss;
                ss << "bsr tier=" << (warp ? "warp" : "cta") << " rows=" << d.nrows << " bi=" << d.bi
                   << " bd=" << d.bd << " cols=" << d.ncols << " chunk=" << p.m << " kd=" << p.kd
                   << " teams=" << p.teams << " grid=" << grid << " threads=" << threads << " smem=" << smem;
                *describe = ss.str();
                return;
            }
            if (units == 0 || d.bi == 0) return;
            if (grid > 0x7fffffff) throw std::runtime_error("bsr_krylov: too many block rows in one launch");
            auto kernel = warp ? bsr_kernel<T, true> : bsr_kernel<T, false>;
            cuda_check(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                       "cudaFuncSetAttribute");
            {
                KernelTimer timer("bsr", stream);
                kernel<<<(unsigned)grid, threads, (size_t)smem, stream>>>(p, (const T *)v, (const T *)x, (T *)y,
                                                                          scalar_of<T>(alpha), scalar_of<T>(beta));
            }
            count_launch();
            cuda_check(cudaGetLastError(), "bsr_kernel launch");
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

} // namespace sbb
