// Drop-in check of the block-sparse operators of include/superbblas.h: create_bsr, bsr_krylov (with and
// without a power label) and destroy_bsr called through the templates on a periodic 1-D lattice of 4 x 4
// blocks with three blocks per row, the result checked on the host.
#include "superbblas.h"
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

int main() {
    if (getGpuDevicesCount() == 0) {
        std::printf("no GPU\n");
        return 2;
    }
    Context gpu = createGpuContext(0);
    const int b = 4, L = 16, N = 2, P = 2; // lattice "sx" (s: block, x: sites); columns n; powers p
    std::srand(11);
    auto rnd = [] { return Z(std::rand() / (double)RAND_MAX - 0.5, std::rand() / (double)RAND_MAX - 0.5); };
    std::vector<int> ii(L, 3);
    std::vector<Coor<2>> jj;
    for (int x = 0; x < L; ++x)
        for (int d : {-1, 0, 1}) jj.push_back(Coor<2>{0, x + d}); // x - 1 = -1 is taken modulo L
    std::vector<Z> v(jj.size() * b * b), xv(b * L * N);
    for (auto &e : v) e = rnd();
    for (auto &e : xv) e = rnd();
    // host reference: y(s, x, n) = sum_d sum_t A_{x,d}(s, t) x(t, x + d, n); element (i, j) at i + j * b
    auto apply = [&](const std::vector<Z> &in) {
        std::vector<Z> out(b * L * N);
        for (int n = 0; n < N; ++n)
            for (int x = 0; x < L; ++x)
                for (int k = 0; k < 3; ++k) {
                    const int xs = ((jj[x * 3 + k][1] % L) + L) % L;
                    for (int s = 0; s < b; ++s)
                        for (int t = 0; t < b; ++t)
                            out[s + b * (x + L * n)] += v[(x * 3 + k) * b * b + s + t * b] * in[t + b * (xs + L * n)];
                }
        return out;
    };
    std::vector<Z> want1 = apply(xv), want2 = apply(want1);

    int *dii = to_device(ii);
    Coor<2> *djj = to_device(jj);
    Z *dv = to_device(v);
    const Z *cv = dv;
    PartitionItem<2> pim{Coor<2>{}, Coor<2>{b, L}};
    BSR_handle *op = nullptr;
    create_bsr<2, 2, Z>(&pim, Coor<2>{b, L}, &pim, Coor<2>{b, L}, 1, Coor<2>{b, 1}, Coor<2>{b, 1}, true, &dii, &djj,
                        &cv, &gpu, FastToSlow, &op);
    cudaFree(dii), cudaFree(djj); // read during create_bsr only

    Z *dx = to_device(xv), *dy = to_device(std::vector<Z>(b * L * N)), *dyp = to_device(std::vector<Z>(b * L * N * P));
    const Z *cx = dx;
    PartitionItem<3> px{Coor<3>{}, Coor<3>{b, L, N}};
    PartitionItem<4> py{Coor<4>{}, Coor<4>{b, L, N, P}};
    Request req;
    bsr_krylov<2, 2, 3, 3, Z>(Z{1}, op, "sx", "SX", &px, 1, "SXn", Coor<3>{}, Coor<3>{b, L, N}, Coor<3>{b, L, N}, &cx,
                              Z{0}, &px, "sxn", Coor<3>{}, Coor<3>{b, L, N}, Coor<3>{b, L, N}, 0, &dy, &gpu,
                              FastToSlow, &req);
    wait(req);
    bsr_krylov<2, 2, 3, 4, Z>(Z{1}, op, "sx", "SX", &px, 1, "SXn", Coor<3>{}, Coor<3>{b, L, N}, Coor<3>{b, L, N}, &cx,
                              Z{0}, &py, "sxnp", Coor<4>{}, Coor<4>{b, L, N, P}, Coor<4>{b, L, N, P}, 'p', &dyp,
                              &gpu, FastToSlow);
    sync(gpu);
    std::vector<Z> y = to_host(dy, want1.size()), yp = to_host(dyp, 2 * want1.size());
    double err = 0, nrm = 0;
    for (std::size_t i = 0; i < want1.size(); ++i) {
        err += std::norm(y[i] - want1[i]) + std::norm(yp[i] - want1[i]) + std::norm(yp[i + want1.size()] - want2[i]);
        nrm += std::norm(want1[i]) + std::norm(want2[i]);
    }
    CHECK(std::sqrt(err / nrm) < 1e-12);
    destroy_bsr(op);

    bool threw = false; // a jj that is not a multiple of blockdom
    try {
        std::vector<int> ii1(L, 0);
        ii1[0] = 1;
        std::vector<Coor<2>> jj1{Coor<2>{1, 0}};
        int *pi = ii1.data();
        Coor<2> *pj = jj1.data();
        const Z *hv = v.data();
        Context cpu = createCpuContext();
        create_bsr<2, 2, Z>(&pim, Coor<2>{b, L}, &pim, Coor<2>{b, L}, 1, Coor<2>{b, 1}, Coor<2>{b, 1}, true, &pi, &pj,
                            &hv, &cpu, FastToSlow, &op);
    } catch (const std::exception &e) { threw = true; }
    CHECK(threw);

    cudaFree(dv), cudaFree(dx), cudaFree(dy), cudaFree(dyp);
    clearCaches();
    long long blocks = 0, bytes = 0;
    CHECK(sbb_live_allocations(&blocks, &bytes) == 0 && blocks == 0);
    std::printf("Everything went ok!\n");
    return 0;
}
