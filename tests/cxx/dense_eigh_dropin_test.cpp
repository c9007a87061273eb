// Drop-in check of eigh in include/superbblas.h: a batch of Hermitian matrices diagonalised on the GPU
// through the template, with A V = V diag(w), V^H V = I and the ascending order checked on the host.  With
// SUPERBBLAS_USE_MPI the MPI overload is instantiated as well (against tests/cxx/mpi_stub/mpi.h; it is
// never called).
#include "superbblas.h"
#include <algorithm>
#include <cmath>
#include <complex>
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>
#include <vector>

using namespace superbblas;
using Z = std::complex<double>;

#define CHECK(cond)                                                                                \
    do {                                                                                           \
        if (!(cond)) {                                                                             \
            std::printf("FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond);                          \
            return 1;                                                                              \
        }                                                                                          \
    } while (0)

template <typename T> T *to_device(const std::vector<T> &h) {
    T *d = nullptr;
    if (cudaMalloc((void **)&d, sizeof(T) * std::max<std::size_t>(h.size(), 1)) != cudaSuccess) std::abort();
    cudaMemcpy(d, h.data(), sizeof(T) * h.size(), cudaMemcpyHostToDevice);
    return d;
}
template <typename T> std::vector<T> to_host(const T *d, std::size_t n) {
    std::vector<T> h(n);
    cudaMemcpy(h.data(), d, sizeof(T) * n, cudaMemcpyDeviceToHost);
    return h;
}

#ifdef SUPERBBLAS_USE_MPI
// The MPI overload (instantiation only)
void mpi_overload(const PartitionItem<3> &p, const PartitionItem<2> &pw, Z **a, double **w, const Context *ctx) {
    eigh<3, 2>(&p, 1, "brc", a, "r", "c", ctx, &pw, 1, "bc", w, ctx, MPI_COMM_WORLD, FastToSlow);
}
#endif

int main() {
    if (getGpuDevicesCount() == 0) {
        std::printf("no GPU\n");
        return 2;
    }
    Context gpu = createGpuContext(0);
    const int n = 12, B = 64; // "brc" matrices (first label fastest), "bc" eigenvalues
    std::vector<Z> a(B * n * n);
    std::srand(11);
    auto rnd = [] { return std::rand() / (double)RAND_MAX - 0.5; };
    auto at = [&](int b, int r, int c) { return b + B * (r + n * c); };
    for (int b = 0; b < B; ++b)
        for (int r = 0; r < n; ++r)
            for (int c = r; c < n; ++c) {
                const Z x = r == c ? Z(rnd(), 0) : Z(rnd(), rnd());
                a[at(b, r, c)] = x, a[at(b, c, r)] = std::conj(x);
            }
    Z *da = to_device(a);
    double *dw = to_device(std::vector<double>(B * n));
    PartitionItem<3> pa{Coor<3>{}, Coor<3>{B, n, n}};
    PartitionItem<2> pw{Coor<2>{}, Coor<2>{B, n}};
    eigh<3, 2>(&pa, 1, "brc", &da, "r", "c", &gpu, &pw, 1, "bc", &dw, &gpu, FastToSlow);
    sync(gpu);
    std::vector<Z> v = to_host(da, a.size());
    std::vector<double> w = to_host(dw, (std::size_t)B * n);
    double res = 0, orth = 0;
    for (int b = 0; b < B; ++b) {
        for (int j = 0; j + 1 < n; ++j) CHECK(w[b + B * j] <= w[b + B * (j + 1)]);
        for (int j = 0; j < n; ++j)
            for (int r = 0; r < n; ++r) {
                Z s = 0, g = 0;
                for (int k = 0; k < n; ++k) s += a[at(b, r, k)] * v[at(b, k, j)];
                res = std::max(res, std::abs(s - w[b + B * j] * v[at(b, r, j)]));
                for (int k = 0; k < n; ++k) g += std::conj(v[at(b, k, r)]) * v[at(b, k, j)];
                orth = std::max(orth, std::abs(g - (r == j ? Z(1) : Z(0))));
            }
    }
    CHECK(res < 1e-12);
    CHECK(orth < 1e-12);
    cudaFree(da), cudaFree(dw);
    std::printf("Everything went ok!\n");
    return 0;
}
