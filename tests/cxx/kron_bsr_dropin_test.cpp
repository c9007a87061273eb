// Drop-in check of the Kronecker block-sparse operator of include/superbblas.h: create_kron_bsr, bsr_krylov
// (with and without a power label) and destroy_bsr called through the templates on a periodic 1-D lattice
// "scx" (spin: the 2 x 2 Kronecker factor, colour: 2 x 2 blocks, x: sites) with three blocks per row, the
// result checked on the host.
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
    const int S = 2, C = 2, L = 16, N = 2, P = 2, U = 3, E = S * C * L * N;
    std::srand(12);
    auto rnd = [] { return Z(std::rand() / (double)RAND_MAX - 0.5, std::rand() / (double)RAND_MAX - 0.5); };
    std::vector<int> ii(L, U);
    std::vector<Coor<3>> jj;
    for (int x = 0; x < L; ++x)
        for (int d : {-1, 0, 1}) jj.push_back(Coor<3>{0, 0, x + d}); // x - 1 = -1 is taken modulo L
    std::vector<Z> v(jj.size() * C * C), kv(U * S * S), xv(E);
    for (auto &e : v) e = rnd();
    for (auto &e : kv) e = rnd();
    for (auto &e : xv) e = rnd();
    // host reference: y(s, c, x, n) = sum_u sum_t sum_e K_u(s, t) B_{x,u}(c, e) x(t, e, x + d_u, n)
    auto apply = [&](const std::vector<Z> &in) {
        std::vector<Z> out(E);
        for (int n = 0; n < N; ++n)
            for (int x = 0; x < L; ++x)
                for (int u = 0; u < U; ++u) {
                    const int xs = ((jj[x * U + u][2] % L) + L) % L;
                    for (int s = 0; s < S; ++s)
                        for (int c = 0; c < C; ++c)
                            for (int t = 0; t < S; ++t)
                                for (int e = 0; e < C; ++e)
                                    out[s + S * (c + C * (x + L * n))] += kv[u * S * S + s + t * S] *
                                                                          v[(x * U + u) * C * C + c + e * C] *
                                                                          in[t + S * (e + C * (xs + L * n))];
                }
        return out;
    };
    std::vector<Z> want1 = apply(xv), want2 = apply(want1);

    int *dii = to_device(ii);
    Coor<3> *djj = to_device(jj);
    Z *dv = to_device(v), *dkv = to_device(kv);
    const Z *cv = dv, *ckv = dkv;
    const Coor<3> dim{S, C, L};
    PartitionItem<3> pim{Coor<3>{}, dim};
    BSR_handle *op = nullptr;
    create_kron_bsr<3, 3, Z>(&pim, dim, &pim, dim, 1, Coor<3>{1, C, 1}, Coor<3>{1, C, 1}, Coor<3>{S, 1, 1},
                             Coor<3>{S, 1, 1}, true, &dii, &djj, &cv, &ckv, &gpu, FastToSlow, &op);
    cudaFree(dii), cudaFree(djj); // read during create_kron_bsr only

    Z *dx = to_device(xv), *dy = to_device(std::vector<Z>(E)), *dyp = to_device(std::vector<Z>(E * P));
    const Z *cx = dx;
    PartitionItem<4> px{Coor<4>{}, Coor<4>{S, C, L, N}};
    PartitionItem<5> py{Coor<5>{}, Coor<5>{S, C, L, N, P}};
    Request req;
    bsr_krylov<3, 3, 4, 4, Z>(Z{1}, op, "scx", "SCX", &px, 1, "SCXn", Coor<4>{}, Coor<4>{S, C, L, N},
                              Coor<4>{S, C, L, N}, &cx, Z{0}, &px, "scxn", Coor<4>{}, Coor<4>{S, C, L, N},
                              Coor<4>{S, C, L, N}, 0, &dy, &gpu, FastToSlow, &req);
    wait(req);
    bsr_krylov<3, 3, 4, 5, Z>(Z{1}, op, "scx", "SCX", &px, 1, "SCXn", Coor<4>{}, Coor<4>{S, C, L, N},
                              Coor<4>{S, C, L, N}, &cx, Z{0}, &py, "scxnp", Coor<5>{}, Coor<5>{S, C, L, N, P},
                              Coor<5>{S, C, L, N, P}, 'p', &dyp, &gpu, FastToSlow);
    sync(gpu);
    std::vector<Z> y = to_host(dy, E), yp = to_host(dyp, 2 * E);
    double err = 0, nrm = 0;
    for (int i = 0; i < E; ++i) {
        err += std::norm(y[i] - want1[i]) + std::norm(yp[i] - want1[i]) + std::norm(yp[i + E] - want2[i]);
        nrm += std::norm(want1[i]) + std::norm(want2[i]);
    }
    CHECK(std::sqrt(err / nrm) < 1e-12);
    destroy_bsr(op);

    bool threw = false; // rows with different block counts
    try {
        std::vector<int> ii1(L, 0);
        ii1[0] = 1;
        std::vector<Coor<3>> jj1{Coor<3>{0, 0, 0}};
        int *pi = ii1.data();
        Coor<3> *pj = jj1.data();
        const Z *hv = v.data(), *hk = kv.data();
        Context cpu = createCpuContext();
        create_kron_bsr<3, 3, Z>(&pim, dim, &pim, dim, 1, Coor<3>{1, C, 1}, Coor<3>{1, C, 1}, Coor<3>{S, 1, 1},
                                 Coor<3>{S, 1, 1}, true, &pi, &pj, &hv, &hk, &cpu, FastToSlow, &op);
    } catch (const std::exception &e) { threw = true; }
    CHECK(threw);

    cudaFree(dv), cudaFree(dkv), cudaFree(dx), cudaFree(dy), cudaFree(dyp);
    clearCaches();
    long long blocks = 0, bytes = 0;
    CHECK(sbb_live_allocations(&blocks, &bytes) == 0 && blocks == 0);
    std::printf("Everything went ok!\n");
    return 0;
}
