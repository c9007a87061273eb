// bsr_krylov with a Request through include/superbblas.h: the operator on the GPU, x and y on the host.
// y is complete after wait(request); a request dropped without wait completes when it goes away; a
// second wait does nothing.  A periodic 1-D lattice of 4 x 4 blocks with three blocks per row.
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

int main() {
    if (getGpuDevicesCount() == 0) {
        std::printf("no GPU\n");
        return 2;
    }
    Context gpu = createGpuContext(0), cpu = createCpuContext();
    const int b = 4, L = 16, N = 3; // lattice "sx" (s: block, x: sites); columns n
    std::srand(7);
    auto rnd = [] { return Z(std::rand() / (double)RAND_MAX - 0.5, std::rand() / (double)RAND_MAX - 0.5); };
    std::vector<int> ii(L, 3);
    std::vector<Coor<2>> jj;
    for (int x = 0; x < L; ++x)
        for (int d : {-1, 0, 1}) jj.push_back(Coor<2>{0, x + d});
    std::vector<Z> v(jj.size() * b * b), xv(b * L * N);
    for (auto &e : v) e = rnd();
    for (auto &e : xv) e = rnd();
    std::vector<Z> want(b * L * N);
    for (int n = 0; n < N; ++n)
        for (int x = 0; x < L; ++x)
            for (int k = 0; k < 3; ++k) {
                const int xs = ((jj[x * 3 + k][1] % L) + L) % L;
                for (int s = 0; s < b; ++s)
                    for (int t = 0; t < b; ++t)
                        want[s + b * (x + L * n)] += v[(x * 3 + k) * b * b + s + t * b] * xv[t + b * (xs + L * n)];
            }

    int *dii = to_device(ii);
    Coor<2> *djj = to_device(jj);
    Z *dv = to_device(v);
    const Z *cv = dv;
    PartitionItem<2> pim{Coor<2>{}, Coor<2>{b, L}};
    BSR_handle *op = nullptr;
    create_bsr<2, 2, Z>(&pim, Coor<2>{b, L}, &pim, Coor<2>{b, L}, 1, Coor<2>{b, 1}, Coor<2>{b, 1}, true, &dii, &djj,
                        &cv, &gpu, FastToSlow, &op);
    cudaFree(dii), cudaFree(djj);

    const Z *cx = xv.data();
    PartitionItem<3> px{Coor<3>{}, Coor<3>{b, L, N}};
    auto relerr = [&](const std::vector<Z> &y) {
        double err = 0, nrm = 0;
        for (std::size_t i = 0; i < want.size(); ++i) err += std::norm(y[i] - want[i]), nrm += std::norm(want[i]);
        return std::sqrt(err / nrm);
    };
    std::vector<Z> y(b * L * N, Z{NAN, NAN});
    Z *py = y.data();
    Request req;
    bsr_krylov<2, 2, 3, 3, Z>(Z{1}, op, "sx", "SX", &px, 1, "SXn", Coor<3>{}, Coor<3>{b, L, N}, Coor<3>{b, L, N}, &cx,
                              Z{0}, &px, "sxn", Coor<3>{}, Coor<3>{b, L, N}, Coor<3>{b, L, N}, 0, &py, &cpu,
                              FastToSlow, &req);
    wait(req);
    CHECK(relerr(y) < 1e-12);
    wait(req); // completed: nothing left to do
    CHECK(relerr(y) < 1e-12);

    std::vector<Z> y2(b * L * N, Z{NAN, NAN});
    Z *py2 = y2.data();
    {
        Request dropped;
        bsr_krylov<2, 2, 3, 3, Z>(Z{1}, op, "sx", "SX", &px, 1, "SXn", Coor<3>{}, Coor<3>{b, L, N}, Coor<3>{b, L, N},
                                  &cx, Z{0}, &px, "sxn", Coor<3>{}, Coor<3>{b, L, N}, Coor<3>{b, L, N}, 0, &py2, &cpu,
                                  FastToSlow, &dropped);
    }
    CHECK(relerr(y2) < 1e-12);
    for (std::size_t i = 0; i < y.size(); ++i) CHECK(y[i] == y2[i]);

    destroy_bsr(op);
    cudaFree(dv);
    clearCaches();
    long long blocks = 0, bytes = 0;
    CHECK(sbb_live_allocations(&blocks, &bytes) == 0 && blocks == 0);
    std::printf("Everything went ok!\n");
    return 0;
}
