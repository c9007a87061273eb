// TEST INFRASTRUCTURE: runs the body of the contraction row kernel (superbblas_b200/csrc/contract_row.hpp,
// the same host/device function the CUDA kernel calls) one row at a time on the CPU, so that its indexing
// and arithmetic are checked without a GPU (tests/test_row_kernel_emulation.py).  Not part of the product.
#include "../../superbblas_b200/csrc/contract_dot.hpp"

using namespace sbb::rowk;

template <typename T>
static void run(const RowParams &p, bool swapped, const double *alpha, const void *v0, const void *v1,
                const double *beta, void *vr) {
    const T *va = (const T *)(swapped ? v1 : v0), *vb = (const T *)(swapped ? v0 : v1);
    for (long long row = 0; row < p.rows; ++row)
        row_body<T>(p, row, va, vb, (T *)vr, scalar_of<T>(alpha), scalar_of<T>(beta));
}

extern "C" int rowk_eligible(const sbk_contract_desc *desc) { return eligible(*desc) ? 1 : 0; }

extern "C" int rowk_emulate(const sbk_contract_desc *desc, int dtype, const double *alpha, const void *v0,
                            const void *v1, const double *beta, void *vr) {
    try {
        RowParams p;
        bool swapped = false;
        build(*desc, p, swapped);
        switch (dtype) {
        case SBB_F32: run<float>(p, swapped, alpha, v0, v1, beta, vr); break;
        case SBB_F64: run<double>(p, swapped, alpha, v0, v1, beta, vr); break;
        case SBB_C64: run<float2>(p, swapped, alpha, v0, v1, beta, vr); break;
        case SBB_C128: run<double2>(p, swapped, alpha, v0, v1, beta, vr); break;
        default: return 2;
        }
        return 0;
    } catch (const std::exception &) { return 1; }
}

// generic kernel's opt-in output enumeration: (order chosen from the strides, then idx -> t, m, n)
extern "C" void rowk_output_order(const long long *min_sr, int *order) { output_order(min_sr, order); }
extern "C" void rowk_output_index(const int *order, long long tvol, long long mvol, long long nvol,
                                  long long idx, long long *tmn) {
    output_index(order, tvol, mvol, nvol, idx, tmn[0], tmn[1], tmn[2]);
}

// ---- dot kernel (long contraction, both free groups small): both passes, thread by thread -----------------
template <typename T>
static void run_dot(const sbb::dotk::DotParams &p, const double *alpha, const void *v0, const void *v1,
                    const double *beta, void *vr) {
    using A = typename Acc<T>::type;
    constexpr int SB = sbb::dotk::SB;
    std::vector<A> ws((size_t)sbb::dotk::threads_of(p) * SB * SB);
    if (sbb::dotk::cta_tree(p)) {
        // what a CTA of the CUDA kernel does: its 128 threads add their blocks, one block is written
        for (long long th = 0; th < sbb::dotk::threads_of(p); th += sbb::dotk::CTA) {
            A sum[SB * SB];
            for (int q = 0; q < SB * SB; ++q) set_zero(sum[q]);
            for (int l = 0; l < sbb::dotk::CTA; ++l) {
                typename Fast<T>::type acc[SB][SB];
                sbb::dotk::dot_partial_acc<T>(p, th + l, (const T *)v0, (const T *)v1, acc);
                for (int q = 0; q < SB * SB; ++q) sum[q] = addc(sum[q], widen(acc[q / SB][q % SB]));
            }
            for (int q = 0; q < SB * SB; ++q) ws[(size_t)(th / sbb::dotk::CTA) * SB * SB + q] = sum[q];
        }
    } else {
        for (long long th = 0; th < sbb::dotk::threads_of(p); ++th)
            sbb::dotk::dot_partial<T>(p, th, (const T *)v0, (const T *)v1, ws.data());
    }
    for (long long o = 0; o < sbb::dotk::outputs_of(p); ++o)
        sbb::dotk::dot_reduce<T>(p, o, ws.data(), (T *)vr, scalar_of<T>(alpha), scalar_of<T>(beta));
}

extern "C" int dotk_eligible(const sbk_contract_desc *desc) { return sbb::dotk::eligible(*desc) ? 1 : 0; }

extern "C" int dotk_emulate(const sbk_contract_desc *desc, int dtype, long long target_threads,
                            const double *alpha, const void *v0, const void *v1, const double *beta,
                            void *vr) {
    try {
        sbb::dotk::DotParams p;
        sbb::dotk::build(*desc, p, target_threads);
        switch (dtype) {
        case SBB_F32: run_dot<float>(p, alpha, v0, v1, beta, vr); break;
        case SBB_F64: run_dot<double>(p, alpha, v0, v1, beta, vr); break;
        case SBB_C64: run_dot<float2>(p, alpha, v0, v1, beta, vr); break;
        case SBB_C128: run_dot<double2>(p, alpha, v0, v1, beta, vr); break;
        default: return 2;
        }
        return 0;
    } catch (const std::exception &) { return 1; }
}
