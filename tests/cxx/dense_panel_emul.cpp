// CPU emulation of the panel body of the blocked dense-solver tier (upper_h_solve in superbblas_b200/
// csrc/dense_kernel.hpp), run by tests/test_dense_blocked_plan.py: the function the CUDA kernel calls.
#include "../../superbblas_b200/csrc/dense_kernel.hpp"

using namespace sbb::densek;

namespace {
    /// u: n x n row-major; x: n x m (right-hand side j at x + j, stride m), overwritten with U^-H x
    template <typename T> void run(int n, const void *u, void *x, int m) {
        for (int j = 0; j < m; ++j) upper_h_solve((const T *)u, (T *)x + j, n, m);
    }
}

extern "C" void panel_emul(int dtype, int n, const void *u, void *x, int m) {
    switch (dtype) {
    case SBB_F32: return run<float>(n, u, x, m);
    case SBB_F64: return run<double>(n, u, x, m);
    case SBB_C64: return run<float2>(n, u, x, m);
    case SBB_C128: return run<double2>(n, u, x, m);
    }
}
