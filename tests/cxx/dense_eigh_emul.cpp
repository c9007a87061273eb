// CPU emulation of the per-matrix body of the eigh kernel (eigh_body in superbblas_b200/csrc/
// dense_kernel.hpp), run by tests/test_dense_eigh_emulation.py: the very function the CUDA kernel calls,
// on a team of one thread.
#include "../../superbblas_b200/csrc/dense_kernel.hpp"
#include <vector>

using namespace sbb::densek;

namespace {
    /// a: n x n row-major, overwritten with V (vectors != 0); w: n eigenvalues
    template <typename T> void run(int n, void *av, void *wv, int vectors) {
        using R = typename Real<T>::type;
        const int m = n > 0 ? n : 1;
        std::vector<T> v(vectors ? (size_t)m * m : 0), sig(m);
        std::vector<R> rot(3 * ((m + 1) / 2));
        std::vector<int> ix(m + 1);
        eigh_body((T *)av, vectors ? v.data() : nullptr, (R *)wv, sig.data(), rot.data(), ix.data(), n, SerialTeam());
    }
}

extern "C" void eigh_emul(int dtype, int n, void *a, void *w, int vectors) {
    switch (dtype) {
    case SBB_F32: return run<float>(n, a, w, vectors);
    case SBB_F64: return run<double>(n, a, w, vectors);
    case SBB_C64: return run<float2>(n, a, w, vectors);
    case SBB_C128: return run<double2>(n, a, w, vectors);
    }
}
