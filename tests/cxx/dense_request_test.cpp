// The dense solvers with a Request through include/superbblas.h: cholesky, inversion, trsm and gesm on a
// batch of matrices on the GPU, y of the solves on the host.  Each request's result is bit-identical to the
// call without one; host y is complete after wait(request); a request dropped without wait completes when
// it goes away; a second wait does nothing.  With SUPERBBLAS_USE_MPI the MPI overloads, with and without a
// request, are instantiated too (compile-checked against a stand-in mpi.h; never run that way).
#include "superbblas.h"
#include <cmath>
#include <complex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
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

static Context g_cpu = createCpuContext();

template <typename T> T *to_device(const std::vector<T> &h, Context gpu) {
    T *d = allocate<T>(h.size(), gpu);
    detail::check(sbb_memcpy(d, detail::ctx_ptr(&gpu), h.data(), detail::ctx_ptr(&g_cpu), sizeof(T) * h.size()));
    return d;
}
template <typename T> std::vector<T> to_host(const T *d, std::size_t n, Context gpu) {
    std::vector<T> h(n);
    detail::check(sbb_memcpy(h.data(), detail::ctx_ptr(&g_cpu), d, detail::ctx_ptr(&gpu), sizeof(T) * n));
    return h;
}
static bool same_bits(const std::vector<Z> &a, const std::vector<Z> &b) {
    return a.size() == b.size() && std::memcmp(a.data(), b.data(), sizeof(Z) * a.size()) == 0;
}

#ifdef SUPERBBLAS_USE_MPI
// The MPI overloads with and without a request (instantiation only)
void mpi_overloads(Z **a, const Z **ca, const Z **x, Z **y, const Context *ctx) {
    PartitionItem<3> p{Coor<3>{}, Coor<3>{1, 2, 2}};
    Request r;
    cholesky<3>(&p, 1, "brc", a, "r", "c", ctx, MPI_COMM_WORLD, FastToSlow);
    cholesky<3>(&p, 1, "brc", a, "r", "c", ctx, MPI_COMM_WORLD, FastToSlow, &r);
    inversion<3>(&p, 1, "brc", a, "r", "c", ctx, MPI_COMM_WORLD, FastToSlow, &r);
    trsm<3, 3, 3>(Z{1}, &p, 1, "brc", "r", "c", ca, ctx, &p, 1, "bxr", x, ctx, &p, 1, "bxc", y, ctx,
                  MPI_COMM_WORLD, FastToSlow, &r);
    gesm<3, 3, 3>(Z{1}, &p, 1, "brc", "r", "c", ca, ctx, &p, 1, "bxr", x, ctx, &p, 1, "bxc", y, ctx,
                  MPI_COMM_WORLD, FastToSlow, nullptr, 0);
    wait(r);
}
#endif

int main(int argc, char **) {
    if (getGpuDevicesCount() == 0) {
        std::printf("no GPU\n");
        return 2;
    }
    Context gpu = createGpuContext(0), cpu = createCpuContext();
    const int n = 12, B = 16, R = 5; // "brc" matrices (first label fastest), "bxr" / "bxc" vectors
    std::vector<Z> a(B * n * n), x(B * R * n);
    std::srand(11);
    auto rnd = [] { return Z(std::rand() / (double)RAND_MAX - 0.5, std::rand() / (double)RAND_MAX - 0.5); };
    for (int b = 0; b < B; ++b)
        for (int r = 0; r < n; ++r)
            for (int c = 0; c < n; ++c) a[b + B * (r + n * c)] = rnd() + (r == c ? Z(2.0 * n) : Z(0));
    for (auto &v : x) v = rnd();
    // Hermitian positive definite matrices for cholesky: A + A^H
    std::vector<Z> h(a.size());
    for (int b = 0; b < B; ++b)
        for (int r = 0; r < n; ++r)
            for (int c = 0; c < n; ++c) h[b + B * (r + n * c)] = a[b + B * (r + n * c)] + std::conj(a[b + B * (c + n * r)]);
    PartitionItem<3> pa{Coor<3>{}, Coor<3>{B, n, n}}, pv{Coor<3>{}, Coor<3>{B, R, n}};
#ifdef SUPERBBLAS_USE_MPI
    if (argc < 0) {
        Z *d = nullptr;
        const Z *cd = nullptr;
        mpi_overloads(&d, &cd, &cd, &d, &gpu);
    }
#else
    (void)argc;
#endif

    // cholesky and inversion in place: plain, then with a request (waited), then with a dropped request
    for (int inv = 0; inv < 2; ++inv) {
        const std::vector<Z> &m = inv ? a : h;
        std::vector<Z> out[3];
        for (int mode = 0; mode < 3; ++mode) {
            Z *d = to_device(m, gpu);
            if (mode == 0) {
                if (inv) inversion<3>(&pa, 1, "brc", &d, "r", "c", &gpu, FastToSlow);
                else cholesky<3>(&pa, 1, "brc", &d, "r", "c", &gpu, FastToSlow);
            } else {
                Request req;
                if (inv) inversion<3>(&pa, 1, "brc", &d, "r", "c", &gpu, FastToSlow, &req);
                else cholesky<3>(&pa, 1, "brc", &d, "r", "c", &gpu, FastToSlow, &req);
                if (mode == 1) wait(req), wait(req);
            }
            sync(gpu);
            out[mode] = to_host(d, m.size(), gpu);
            deallocate(d, gpu);
        }
        CHECK(same_bits(out[0], out[1]) && same_bits(out[0], out[2]));
        for (const Z &v : out[0]) CHECK(std::isfinite(v.real()) && std::isfinite(v.imag()));
    }

    // trsm and gesm with x on the GPU and y on the host
    Z *da = to_device(a, gpu), *dx = to_device(x, gpu);
    const Z *ca = da, *cx = dx;
    for (int ge = 0; ge < 2; ++ge) {
        std::vector<Z> y[3];
        for (int mode = 0; mode < 3; ++mode) {
            y[mode].assign(x.size(), Z{NAN, NAN});
            Z *py = y[mode].data();
            Request req;
            Request *q = mode ? &req : nullptr;
            if (ge)
                gesm<3, 3, 3>(Z{0.5, -1}, &pa, 1, "brc", "r", "c", &ca, &gpu, &pv, 1, "bxr", &cx, &gpu, &pv, 1, "bxc",
                              &py, &cpu, FastToSlow, q);
            else
                trsm<3, 3, 3>(Z{0.5, -1}, &pa, 1, "brc", "r", "c", &ca, &gpu, &pv, 1, "bxr", &cx, &gpu, &pv, 1, "bxc",
                              &py, &cpu, FastToSlow, q);
            if (mode == 1) wait(req), wait(req);
            if (mode == 2) req = Request{}; // dropped: completed when its last copy goes away
        }
        CHECK(same_bits(y[0], y[1]) && same_bits(y[0], y[2]));
        // residual of A y = alpha x (trsm: the upper triangle of A)
        double err = 0, nrm = 0;
        for (int b = 0; b < B; ++b)
            for (int j = 0; j < R; ++j)
                for (int r = 0; r < n; ++r) {
                    Z s = 0;
                    for (int c = ge ? 0 : r; c < n; ++c) s += a[b + B * (r + n * c)] * y[0][b + B * (j + R * c)];
                    const Z want = Z{0.5, -1} * x[b + B * (j + R * r)];
                    err += std::norm(s - want), nrm += std::norm(want);
                }
        CHECK(std::sqrt(err / nrm) < 1e-12);
    }

    // an argument error comes back from the begin, with the message of the call without a request
    {
        Request req;
        std::string plain, begun;
        try {
            trsm<3, 3, 3>(Z{1}, &pa, 1, "brc", "r", "c", &ca, &gpu, &pv, 1, "bxr", &cx, &gpu, &pv, 1, "bxr", &dx, &gpu,
                          FastToSlow);
        } catch (const std::exception &e) {
            plain = e.what();
        }
        try {
            trsm<3, 3, 3>(Z{1}, &pa, 1, "brc", "r", "c", &ca, &gpu, &pv, 1, "bxr", &cx, &gpu, &pv, 1, "bxr", &dx, &gpu,
                          FastToSlow, &req);
        } catch (const std::exception &e) {
            begun = e.what();
        }
        CHECK(!plain.empty() && plain == begun);
        CHECK(!req);
    }
    deallocate(da, gpu), deallocate(dx, gpu);
    clearCaches();
    long long blocks = 0, bytes = 0;
    CHECK(sbb_live_allocations(&blocks, &bytes) == 0 && blocks == 0);
    std::printf("Everything went ok!\n");
    return 0;
}
