// CPU emulation of the per-row body of the block-sparse kernel (superbblas_b200/csrc/bsr_kernel.hpp), run
// by tests/test_bsr_kernel_emulation.py: the very function the CUDA kernel calls, on a team of one thread,
// over column chunks and domain pieces like the kernel's.
#include "../../superbblas_b200/csrc/bsr_kernel.hpp"
#include <algorithm>
#include <vector>

using namespace sbb;
using namespace sbb::bsrk;

namespace {
    constexpr int MAXO = 4096;

    template <typename T>
    void run(const sbk_bsr_desc &d, const double *alpha, const double *beta, const void *v, const void *x, void *y,
             int m, int kd) {
        std::vector<T> as((size_t)d.bi * kd), xs((size_t)kd * m);
        std::vector<int64_t> xo(std::max(d.bd, 1));
        for (int j = 0; j < d.bd; ++j) xo[j] = domain_point(d, j);
        const SerialTeam tm;
        for (int64_t r = 0; r < d.nrows; ++r)
            for (int c0 = 0; c0 < d.ncols; c0 += m)
                row_body<MAXO>(d, r, c0, std::min(m, d.ncols - c0), kd, (const T *)v, (const T *)x, (T *)y,
                               scalar_of<T>(alpha), scalar_of<T>(beta), as.data(), xs.data(), xo.data(), tm);
    }
}

/// dims: D as (size, stride) pairs, I as (blocks, size, stride) triples, C as (size, stride) pairs
extern "C" void bsr_emul(int dtype, int64_t nrows, const int64_t *rowptr, const int64_t *goff, int bi, int bd,
                         int im_fast, int ncols, int nd, const int64_t *D, int ni, const int64_t *I, int nc,
                         const int64_t *C, const double *alpha, const double *beta, const void *v, const void *x,
                         void *y, int m, int kd) {
    sbk_bsr_desc d{};
    d.nrows = nrows, d.rowptr = rowptr, d.goff = goff, d.bi = bi, d.bd = bd, d.im_fast = im_fast, d.ncols = ncols;
    d.nd = nd, d.ni = ni, d.nc = nc;
    for (int k = 0; k < nd; ++k) d.dsize[k] = (int)D[2 * k], d.dstride[k] = D[2 * k + 1];
    for (int k = 0; k < ni; ++k) d.iblocks[k] = (int)I[3 * k], d.isize[k] = (int)I[3 * k + 1], d.istride[k] = I[3 * k + 2];
    for (int k = 0; k < nc; ++k) d.csize[k] = (int)C[2 * k], d.cstride[k] = C[2 * k + 1];
    switch (dtype) {
    case SBB_F32: return run<float>(d, alpha, beta, v, x, y, m, kd);
    case SBB_F64: return run<double>(d, alpha, beta, v, x, y, m, kd);
    case SBB_C64: return run<float2>(d, alpha, beta, v, x, y, m, kd);
    case SBB_C128: return run<double2>(d, alpha, beta, v, x, y, m, kd);
    }
}
