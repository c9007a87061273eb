// CPU emulation of the per-row body of the Kronecker block-sparse kernel (kron_row_body in
// superbblas_b200/csrc/bsr_kernel.hpp), run by tests/test_bsr_kron_kernel_emulation.py: the very function
// the CUDA kernel calls, on a team of one thread, over column chunks and block pieces like the kernel's.
#include "../../superbblas_b200/csrc/bsr_kernel.hpp"
#include <algorithm>
#include <vector>

using namespace sbb;
using namespace sbb::bsrk;

namespace {
    constexpr int MAXO = 4096;

    template <typename T>
    void run(const sbk_bsr_desc &d, const sbk_kron_desc &k, const double *alpha, const double *beta, const void *v,
             const void *kv, const void *x, void *y, int m, int nu) {
        std::vector<T> bs((size_t)nu * d.bi * d.bd + 1), xs((size_t)nu * k.kd * d.bd * m + 1);
        std::vector<AccT<T>> ts((size_t)nu * k.kd * d.bi * m + 1);
        std::vector<int64_t> xo((size_t)k.kd * d.bd + 1);
        for (int j = 0; j < k.kd * d.bd; ++j) xo[j] = kron_domain_point(d, k, j / d.bd, j % d.bd);
        const SerialTeam tm;
        for (int64_t r = 0; r < d.nrows; ++r)
            for (int c0 = 0; c0 < d.ncols; c0 += m)
                kron_row_body<MAXO>(d, k, r, c0, std::min(m, d.ncols - c0), nu, (const T *)v, (const T *)kv,
                                    (const T *)x, (T *)y, scalar_of<T>(alpha), scalar_of<T>(beta), bs.data(),
                                    xs.data(), ts.data(), xo.data(), tm);
    }
}

/// dims: D as (size, ksize, stride) triples, I as (blocks, size, ksize, stride) quadruples, C as (size, stride)
extern "C" void kron_bsr_emul(int dtype, int64_t nrows, const int64_t *rowptr, const int64_t *goff, int bi, int bd,
                              int ki, int kd, int u, int im_fast, int ncols, int nd, const int64_t *D, int ni,
                              const int64_t *I, int nc, const int64_t *C, const double *alpha, const double *beta,
                              const void *v, const void *kv, const void *x, void *y, int m, int nu) {
    sbk_bsr_desc d{};
    sbk_kron_desc k{};
    d.nrows = nrows, d.rowptr = rowptr, d.goff = goff, d.bi = bi, d.bd = bd, d.im_fast = im_fast, d.ncols = ncols;
    d.nd = nd, d.ni = ni, d.nc = nc;
    k.ki = ki, k.kd = kd, k.u = u;
    for (int e = 0; e < nd; ++e) d.dsize[e] = (int)D[3 * e], k.dksize[e] = (int)D[3 * e + 1], d.dstride[e] = D[3 * e + 2];
    for (int e = 0; e < ni; ++e)
        d.iblocks[e] = (int)I[4 * e], d.isize[e] = (int)I[4 * e + 1], k.iksize[e] = (int)I[4 * e + 2],
        d.istride[e] = I[4 * e + 3];
    for (int e = 0; e < nc; ++e) d.csize[e] = (int)C[2 * e], d.cstride[e] = C[2 * e + 1];
    switch (dtype) {
    case SBB_F32: return run<float>(d, k, alpha, beta, v, kv, x, y, m, nu);
    case SBB_F64: return run<double>(d, k, alpha, beta, v, kv, x, y, m, nu);
    case SBB_C64: return run<float2>(d, k, alpha, beta, v, kv, x, y, m, nu);
    case SBB_C128: return run<double2>(d, k, alpha, beta, v, kv, x, y, m, nu);
    }
}
