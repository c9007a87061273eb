// Scalar arithmetic of the contraction kernels on real and complex elements (float, double, float2,
// double2), for the host and the device: every contraction kernel uses these, and the CPU emulation of
// the row and dot kernels (tests/test_row_kernel_emulation.py) runs the same functions.
#pragma once
#include <cmath>
#include <type_traits>
#include <vector_types.h>

#if defined(__CUDACC__)
#    define SBB_HD __host__ __device__ __forceinline__
#else
#    define SBB_HD inline
#endif

namespace sbb {

    /// Type of alpha, beta and the long sums: double for the float types
    template <typename T> struct Acc { using type = T; };
    template <> struct Acc<float> { using type = double; };
    template <> struct Acc<float2> { using type = double2; };

    /// Type of the products and of the short sums a thread keeps in registers: the operand type
    /// itself (float types stay float: at most KMAX terms per sum in the row kernel, and slices of a
    /// few dozen terms in the dot kernel; alpha, beta and the sums over slices are done in Acc<T>)
    template <typename T> struct Fast { using type = T; };

    SBB_HD float cj(float x) { return x; }
    SBB_HD float2 cj(float2 x) {
        x.y = -x.y;
        return x;
    }
    SBB_HD void fma_acc(float &acc, float a, float b) { acc = fmaf(a, b, acc); }
    SBB_HD void fma_acc(float2 &acc, float2 a, float2 b) {
        acc.x = fmaf(a.x, b.x, acc.x);
        acc.x = fmaf(-a.y, b.y, acc.x);
        acc.y = fmaf(a.x, b.y, acc.y);
        acc.y = fmaf(a.y, b.x, acc.y);
    }
    SBB_HD void set_zero(float &x) { x = 0; }
    SBB_HD void set_zero(float2 &x) { x.x = x.y = 0; }

    SBB_HD double widen(float x) { return (double)x; }
    SBB_HD double widen(double x) { return x; }
    SBB_HD double2 widen(float2 x) {
        double2 r;
        r.x = x.x, r.y = x.y;
        return r;
    }
    SBB_HD double2 widen(double2 x) { return x; }
    SBB_HD double cj(double x) { return x; }
    SBB_HD double2 cj(double2 x) {
        x.y = -x.y;
        return x;
    }
    SBB_HD void fma_acc(double &acc, double a, double b) { acc = fma(a, b, acc); }
    SBB_HD void fma_acc(double2 &acc, double2 a, double2 b) {
        acc.x = fma(a.x, b.x, acc.x);
        acc.x = fma(-a.y, b.y, acc.x);
        acc.y = fma(a.x, b.y, acc.y);
        acc.y = fma(a.y, b.x, acc.y);
    }
    SBB_HD double mulc(double a, double b) { return a * b; }
    SBB_HD double2 mulc(double2 a, double2 b) {
        double2 r;
        r.x = a.x * b.x - a.y * b.y, r.y = a.x * b.y + a.y * b.x;
        return r;
    }
    SBB_HD double addc(double a, double b) { return a + b; }
    SBB_HD double2 addc(double2 a, double2 b) {
        a.x += b.x, a.y += b.y;
        return a;
    }
    SBB_HD bool is_zero(double x) { return x == 0; }
    SBB_HD bool is_zero(double2 x) { return x.x == 0 && x.y == 0; }
    SBB_HD void set_zero(double &x) { x = 0; }
    SBB_HD void set_zero(double2 &x) { x.x = x.y = 0; }
    SBB_HD void narrow(double x, float &o) { o = (float)x; }
    SBB_HD void narrow(double x, double &o) { o = x; }
    SBB_HD void narrow(double2 x, float2 &o) { o.x = (float)x.x, o.y = (float)x.y; }
    SBB_HD void narrow(double2 x, double2 &o) { o = x; }

    /// vr[off] = alpha * acc + beta * vr[off], rounded to T; vr[off] is not read when beta is zero
    /// (it may hold NaNs)
    template <typename T>
    SBB_HD void epilogue(T *vr, long long off, typename Acc<T>::type acc, typename Acc<T>::type alpha,
                         typename Acc<T>::type beta) {
        typename Acc<T>::type r = mulc(alpha, acc);
        T *w = vr + off;
        if (!is_zero(beta)) r = addc(r, mulc(beta, widen(*w)));
        narrow(r, *w);
    }

    /// alpha or beta of the C ABI ({re, im}) as the kernels of element type T take it
    template <typename T> inline typename Acc<T>::type scalar_of(const double *a) {
        typename Acc<T>::type r;
        if constexpr (std::is_same<typename Acc<T>::type, double2>::value) r.x = a[0], r.y = a[1];
        else r = a[0];
        return r;
    }

} // namespace sbb
