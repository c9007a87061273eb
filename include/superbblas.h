// superbblas.h — drop-in C++ front end of the B200-native tensor hot path.
//
// Same namespace, names, template parameters, argument order and defaults as the reference's public
// API for this path, so that Chroma-style callers compile unchanged; every function only marshals
// into the C ABI of superbblas_b200.h (libsuperbblas_b200.so).  Reference declarations mirrored
// (eromero-vlc/superbblas, include/superbblas/):
//   Coor, Order, IndexType, MaskType, CoorOrder, CopyAdd            tensor.h:47-66
//   platform, Context, createCpuContext/CudaContext/GpuContext,
//   getGpuDevicesCount, clearHandles, Session                       platform.h:108-125,:757-841
//   sync, syncLegacyStream                                          blas.h:965-988
//   PartitionItem, Request, wait                                    dist.h:39-61
//   partitioning_distributed_procs, basic_partitioning (x2)         dist.h:3318,:3393,:3477
//   make_hole                                                       dist.h:3802
//   copy                                                            dist.h:3583 (MPI overload :3534)
//   contraction                                                     dist.h:3701 (MPI overload :3628)
//   local_copy, local_contraction                                   tests/local.cpp:97,:163
//   clearCaches                                                     alloc.h:440
//   create_bsr, bsr_krylov, destroy_bsr                             bsr.h:2286,:2352,:2516
//   create_kron_bsr                                                 bsr.h (not checked against it)
//   getDebugLevel, resetTimings, reportTimings, reportCacheUsage,
//   checkForMemoryLeaks                                             runtime_features.h:31, performance.h:357-518
// Errors are reported like the reference does: std::runtime_error.
//
// Where the reference's MPI overloads take an `MPI_Comm`, this header takes an `sbb_comm_t`
// (one NCCL rank per GPU, see superbblas_b200.h); with SUPERBBLAS_USE_MPI defined, overloads taking
// an MPI_Comm are provided as well and bootstrap the NCCL communicator over MPI once per communicator.
#ifndef SUPERBBLAS_B200_CXX_H
#define SUPERBBLAS_B200_CXX_H

// this build always has the GPU path (the reference defines these from its build flags, platform.h:76)
#ifndef SUPERBBLAS_USE_CUDA
#    define SUPERBBLAS_USE_CUDA
#endif
#ifndef SUPERBBLAS_USE_GPU
#    define SUPERBBLAS_USE_GPU
#endif

#include "superbblas_b200.h"
#include <algorithm>
#include <array>
#include <chrono>
#include <complex>
#include <cstring>
#include <cstdlib>
#include <functional>
#include <iostream>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>
#ifdef SUPERBBLAS_USE_MPI
#    include <mpi.h>
#endif

namespace superbblas {

    using IndexType = int;
    template <std::size_t Nd, typename Idx = IndexType> using Coor = std::array<Idx, Nd>;
    template <std::size_t Nd> using Order = std::array<char, Nd>;
    using MaskType = float;
    using Session = unsigned int;

    enum CoorOrder { SlowToFast, FastToSlow };
    enum CopyAdd { Copy, Add };
    enum platform { CPU, CUDA, HIP };
    constexpr int CPU_DEVICE_ID = -1;
    const platform GPU = platform::CUDA;

    /// Where a component lives; same layout as sbb_context (and as the reference's Context)
    namespace detail {
        /// Low-level contexts of the reference (platform.h:173-217); here they only carry the Context
        struct Cpu {
            Session session = 0;
        };
        struct Gpu {
            int device = 0;
            Session session = 0;
        };
    }

    class Context {
    public:
        enum platform plat;
        int device;
        Context(enum platform plat, int device) : plat(plat), device(device) {}
        detail::Cpu toCpu(Session session) const { return detail::Cpu{session}; }
        detail::Gpu toGpu(Session session) const { return detail::Gpu{device, session}; }
    };
    static_assert(sizeof(Context) == sizeof(sbb_context), "Context must match sbb_context");

    inline Context createCpuContext() { return Context{CPU, CPU_DEVICE_ID}; }
    inline Context createCudaContext(int device = 0) { return Context{CUDA, device}; }
    inline Context createGpuContext(int device = 0) { return Context{GPU, device}; }

    template <std::size_t N> using PartitionItem = std::array<Coor<N>, 2>;
    using Request = std::function<void(void)>;
    inline void wait(const Request &request) {
        if (request) request();
    }

    namespace detail {
        inline void check(int rc) {
            if (rc != 0) throw std::runtime_error(sbb_last_error());
        }

        /// A Request that completes (and releases) the begun `h` exactly once, on its first call or,
        /// when dropped without one, when its last copy goes away
        inline Request make_request(sbb_request_t h) {
            std::shared_ptr<sbb_request_t> once(new sbb_request_t(h), [](sbb_request_t *q) {
                if (*q) sbb_request_wait(*q); // dropped without wait: complete it anyway
                delete q;
            });
            return [once]() {
                sbb_request_t q = *once;
                *once = nullptr;
                if (q) check(sbb_request_wait(q));
            };
        }

        template <typename T> struct dtype_of;
        template <> struct dtype_of<float> { static constexpr int value = SBB_F32; };
        template <> struct dtype_of<double> { static constexpr int value = SBB_F64; };
        template <> struct dtype_of<std::complex<float>> { static constexpr int value = SBB_C64; };
        template <> struct dtype_of<std::complex<double>> { static constexpr int value = SBB_C128; };
        template <> struct dtype_of<int> { static constexpr int value = SBB_I32; };
        template <typename T> struct dtype_of<const T> : dtype_of<T> {};

        template <typename T> inline std::array<double, 2> scalar(const T &a) {
            return {(double)a, 0.0};
        }
        template <typename T> inline std::array<double, 2> scalar(const std::complex<T> &a) {
            return {(double)a.real(), (double)a.imag()};
        }

        template <std::size_t N> inline std::size_t volume(const Coor<N> &c) {
            std::size_t v = 1;
            for (auto x : c) v *= (std::size_t)x;
            return v;
        }

        /// Return an array from a string (reference: tensor.h:266)
        template <std::size_t Nd> inline void check_order(const char *o, const char *name) {
            if ((o == nullptr && Nd > 0) || (o != nullptr && std::strlen(o) != Nd))
                throw std::runtime_error(
                    std::string("The length of the order should match the template argument; "
                                "argument `") +
                    name + "` should have length " + std::to_string(Nd));
        }

        inline const sbb_context *ctx_ptr(const Context *c) {
            return reinterpret_cast<const sbb_context *>(c);
        }

        template <std::size_t N>
        std::vector<PartitionItem<N>> boxes_from(const std::vector<int> &flat) {
            std::vector<PartitionItem<N>> r(flat.size() / (2 * N));
            for (std::size_t i = 0; i < r.size(); ++i)
                for (int j = 0; j < 2; ++j)
                    for (std::size_t k = 0; k < N; ++k) r[i][j][k] = flat[(i * 2 + j) * N + k];
            return r;
        }

        /// Element type used to express alpha (reference: elem<T>, blas.h:100)
        template <typename T> struct elem { using type = T; };
    }

    // ---- detail:: helpers that the reference's own tests reach into (tests/contract.cpp:84-116,
    //      tests/dist.cpp:93-97); kept source compatible so those tests compile unchanged -----------
    namespace detail {
        inline Context to_context(const Cpu &) { return Context{CPU, CPU_DEVICE_ID}; }
        inline Context to_context(const Gpu &g) { return Context{CUDA, g.device}; }

        /// Reference-counted buffer in the space of a context (reference: blas.h:240-358)
        template <typename T, typename XPU> struct vector {
            using T_no_const = typename std::remove_const<T>::type;
            vector() : n(0), xpu() {}
            vector(std::size_t n, XPU xpu) : n(n), xpu(xpu) {
                Context c = to_context(xpu);
                T_no_const *p = n ? superbblas_b200_alloc<T_no_const>(n, c) : nullptr;
                ptr = std::shared_ptr<T_no_const>(p, [c](T_no_const *q) {
                    if (q) sbb_deallocate(ctx_ptr(&c), (void *)q);
                });
            }
            T *data() const { return ptr.get(); }
            T *begin() const { return ptr.get(); }
            T *end() const { return ptr.get() + n; }
            std::size_t size() const { return n; }
            XPU ctx() const { return xpu; }
            /// Element access (meaningful for host vectors only, as in the reference)
            T &operator[](std::size_t i) const { return ptr.get()[i]; }
            void clear() {
                n = 0;
                ptr.reset();
            }

        private:
            template <typename U> static U *superbblas_b200_alloc(std::size_t n, Context c) {
                void *p = nullptr;
                check(sbb_allocate(ctx_ptr(&c), n * sizeof(U), &p));
                return (U *)p;
            }
            std::size_t n;
            std::shared_ptr<T_no_const> ptr;
            XPU xpu;
        };

        /// Contiguous copy between contexts (reference: blas.h:170-231)
        template <typename T, typename XPU0, typename XPU1>
        void copy_n(const T *v, XPU0 xpu0, std::size_t n, T *w, XPU1 xpu1) {
            Context c0 = to_context(xpu0), c1 = to_context(xpu1);
            check(sbb_memcpy((void *)w, ctx_ptr(&c1), (const void *)v, ctx_ptr(&c0), n * sizeof(T)));
        }

        template <std::size_t N, typename I> Coor<N, I> operator+(const Coor<N, I> &a, const Coor<N, I> &b) {
            Coor<N, I> r;
            for (std::size_t i = 0; i < N; ++i) r[i] = a[i] + b[i];
            return r;
        }
        template <std::size_t N, typename I> Coor<N, I> operator-(const Coor<N, I> &a, const Coor<N, I> &b) {
            Coor<N, I> r;
            for (std::size_t i = 0; i < N; ++i) r[i] = a[i] - b[i];
            return r;
        }

        /// Jumps between consecutive coordinates (reference: tensor.h:282)
        template <typename SIdx, std::size_t Nd, typename CIdx>
        Coor<Nd, SIdx> get_strides(const Coor<Nd, CIdx> dim, CoorOrder co) {
            Coor<Nd, SIdx> p;
            if (Nd > 0) {
                if (co == SlowToFast) {
                    p[Nd - 1] = 1;
                    for (std::size_t i = Nd - 1; i >= 1; --i) p[i - 1] = p[i] * dim[i];
                } else {
                    p[0] = 1;
                    for (std::size_t i = 1; i < Nd; ++i) p[i] = p[i - 1] * dim[i - 1];
                }
            }
            return p;
        }
        /// Linear index of a coordinate / coordinate of an index (reference: tensor.h:304, :334)
        template <std::size_t Nd, typename CIdx, typename SIdx>
        SIdx coor2index(const Coor<Nd, CIdx> &coor, const Coor<Nd, CIdx> &dim, const Coor<Nd, SIdx> &stride) {
            SIdx r = 0;
            for (std::size_t j = 0; j < Nd; ++j) r += (coor[j] % dim[j]) * stride[j];
            return r;
        }
        template <std::size_t Nd, typename CIdx, typename SIdx>
        Coor<Nd, CIdx> index2coor(const SIdx &index, const Coor<Nd, CIdx> &dim, const Coor<Nd, SIdx> &stride) {
            Coor<Nd, CIdx> r;
            for (std::size_t j = 0; j < Nd; ++j) r[j] = (CIdx)((index / stride[j]) % (SIdx)dim[j]);
            return r;
        }
    }

    inline unsigned int getGpuDevicesCount() {
        int n = 0;
        detail::check(sbb_device_count(&n));
        return (unsigned int)n;
    }
    inline void clearHandles() { detail::check(sbb_clear_handles()); }
    inline void clearCaches() { detail::check(sbb_clear_caches()); }
    inline void sync(Context ctx) { detail::check(sbb_sync(detail::ctx_ptr(&ctx))); }
    inline void syncLegacyStream(Context ctx) {
        detail::check(sbb_sync_legacy_stream(detail::ctx_ptr(&ctx)));
    }

    /// Allocate / free memory in the space of a context (reference: alloc.h:398-425)
    template <typename T> T *allocate(std::size_t n, Context ctx) {
        void *p = nullptr;
        detail::check(sbb_allocate(detail::ctx_ptr(&ctx), n * sizeof(T), &p));
        return (T *)p;
    }
    template <typename T> void deallocate(T *ptr, Context ctx) {
        detail::check(sbb_deallocate(detail::ctx_ptr(&ctx), (void *)ptr));
    }

    // ---- helpers of namespace detail that the reference's own tests/dist.cpp uses ----------------------
    namespace detail {
        /// Lists of ranges (reference: dist.h:36-51)
        template <std::size_t N> using From_size_item = PartitionItem<N>;
        template <std::size_t N> using From_size = std::vector<PartitionItem<N>>;

        /// Total number of sites of a list of ranges
        template <std::size_t N> std::size_t volume(const From_size<N> &fs) {
            std::size_t v = 0;
            for (const auto &it : fs) v += volume<N>(it[1]);
            return v;
        }

        /// Intersection of two ranges on a periodic lattice, as a list of plain ranges (semantics of
        /// the reference's dist.h:353-495; written from the definition: a site belongs to a range
        /// iff (site - from) mod dim < size).  Per dimension the common sites form at most two runs.
        template <std::size_t N>
        From_size<N> intersection(const Coor<N> &from0, const Coor<N> &size0, const Coor<N> &from1,
                                  const Coor<N> &size1, const Coor<N> &dim) {
            std::array<std::vector<std::array<int, 2>>, N> runs; // per dimension: {first site, length}
            for (std::size_t k = 0; k < N; ++k) {
                const int d = dim[k];
                if (d <= 0) return {};
                auto inside = [&](int site, int from, int size) {
                    return ((site - from) % d + d) % d < size;
                };
                std::vector<char> in((std::size_t)d);
                bool all = true, any = false;
                for (int i = 0; i < d; ++i) {
                    in[i] = inside(i, from0[k], size0[k]) && inside(i, from1[k], size1[k]);
                    all = all && in[i];
                    any = any || in[i];
                }
                if (!any) return {};
                if (all) {
                    runs[k].push_back({((from0[k] % d) + d) % d, d});
                    continue;
                }
                // start at a site that is outside, so that no run wraps around the scan
                int start = 0;
                while (in[start]) ++start;
                for (int j = 1; j <= d;) {
                    const int i = (start + j) % d;
                    if (!in[i]) {
                        ++j;
                        continue;
                    }
                    int len = 0;
                    while (j + len <= d && in[(start + j + len) % d]) ++len;
                    runs[k].push_back({i, len});
                    j += len;
                }
            }
            From_size<N> r(1);
            for (std::size_t k = 0; k < N; ++k) {
                From_size<N> next;
                for (const auto &box : r)
                    for (const auto &run : runs[k]) {
                        PartitionItem<N> b = box;
                        b[0][k] = run[0], b[1][k] = run[1];
                        next.push_back(b);
                    }
                r.swap(next);
            }
            return r;
        }

        /// Intersection of every range of a list with one range
        template <std::size_t N>
        From_size<N> intersection(const From_size<N> &fs0, const Coor<N> &from1, const Coor<N> &size1,
                                  const Coor<N> &dim) {
            From_size<N> r;
            for (const auto &it : fs0) {
                From_size<N> p = intersection<N>(it[0], it[1], from1, size1, dim);
                r.insert(r.end(), p.begin(), p.end());
            }
            return r;
        }

        /// Wall-clock time in seconds (reference: performance.h:228)
        inline double w_time() {
            return std::chrono::duration<double>(std::chrono::system_clock::now().time_since_epoch())
                .count();
        }

        inline int deviceId(const Cpu &) { return CPU_DEVICE_ID; }
        inline int deviceId(const Gpu &g) { return g.device; }
        inline void sync(const Cpu &) {}
        inline void sync(const Gpu &g) { superbblas::sync(to_context(g)); }

        /// Batched strided GEMM with the BLAS column-major convention (reference: blas.h:662 on GPUs,
        /// blas_cpu_tmpl.hpp:376 on CPUs): c_i = alpha * op(a_i) * op(b_i) + beta * c_i.  Here it is
        /// one launch of the fused contraction kernel: the transpositions are strides, 'c' is a flag.
        template <typename T>
        void xgemm_batch_strided(char transa, char transb, int m, int n, int k, T alpha, const T *a,
                                 int lda, int stridea, const T *b, int ldb, int strideb, T beta, T *c,
                                 int ldc, int stridec, int batch_size, Gpu xpu) {
            if (m == 0 || n == 0 || batch_size == 0) return;
            const bool ta = !(transa == 'n' || transa == 'N'), tb = !(transb == 'n' || transb == 'N');
            sbk_contract_desc d;
            std::memset(&d, 0, sizeof d);
            d.nT = d.nM = d.nN = d.nK = 1;
            d.T[0].size = batch_size, d.T[0].s0 = stridea, d.T[0].s1 = strideb, d.T[0].sr = stridec;
            d.M[0].size = m, d.M[0].s0 = ta ? lda : 1, d.M[0].sr = 1;
            d.N[0].size = n, d.N[0].s1 = tb ? 1 : ldb, d.N[0].sr = ldc;
            d.K[0].size = k, d.K[0].s0 = ta ? 1 : lda, d.K[0].s1 = tb ? ldb : 1;
            d.conj0 = transa == 'c' || transa == 'C', d.conj1 = transb == 'c' || transb == 'C';
            const std::array<double, 2> al = scalar(alpha), be = scalar(beta);
            check(sbk_contract(&d, dtype_of<T>::value, al.data(), (const void *)a, (const void *)b,
                               be.data(), (void *)c, xpu.device, nullptr));
        }

        /// Host operands: staged through the GPU (there is no CPU compute path)
        template <typename T>
        void xgemm_batch_strided(char transa, char transb, int m, int n, int k, T alpha, const T *a,
                                 int lda, int stridea, const T *b, int ldb, int strideb, T beta, T *c,
                                 int ldc, int stridec, int batch_size, Cpu) {
            if (m == 0 || n == 0 || batch_size == 0) return;
            const bool ta = !(transa == 'n' || transa == 'N'), tb = !(transb == 'n' || transb == 'N');
            auto extent = [&](int rows, int cols, int ld, int stride) {
                return (std::size_t)(batch_size - 1) * stride + (std::size_t)(cols - 1) * ld + rows;
            };
            const std::size_t na = extent(ta ? k : m, ta ? m : k, lda, stridea),
                              nb = extent(tb ? n : k, tb ? k : n, ldb, strideb),
                              nc = extent(m, n, ldc, stridec);
            Gpu gpu{0, 0};
            Cpu cpu{};
            vector<T, Gpu> da(na, gpu), db(nb, gpu), dc(nc, gpu);
            copy_n<T>(a, cpu, na, da.data(), gpu);
            copy_n<T>(b, cpu, nb, db.data(), gpu);
            copy_n<T>(c, cpu, nc, dc.data(), gpu);
            xgemm_batch_strided<T>(transa, transb, m, n, k, alpha, da.data(), lda, stridea, db.data(), ldb,
                                   strideb, beta, dc.data(), ldc, stridec, batch_size, gpu);
            copy_n<T>(dc.data(), gpu, nc, c, cpu);
        }
    }

    // Diagnostics of the reference that callers and its tests reference
    /// SB_DEBUG (runtime_features.h:31): 0 = none; >= 2 makes every copy verify itself on
    /// index-valued mock tensors first (dist.h:2282-2285), which the library does in sbb_copy
    inline int getDebugLevel() {
        static int level = [] {
            const char *e = std::getenv("SB_DEBUG");
            return e ? std::atoi(e) : 0;
        }();
        return level;
    }
    /// SB_TRACK_TIME / SB_TRACK_MEMORY (runtime_features.h): nonzero turns the reports below on
    inline bool getTrackingTime() {
        static bool on = [] {
            const char *e = std::getenv("SB_TRACK_TIME");
            return e && std::atoi(e) != 0;
        }();
        return on;
    }
    inline bool getTrackingMemory() {
        static bool on = [] {
            const char *e = std::getenv("SB_TRACK_MEMORY");
            return e && std::atoi(e) != 0;
        }();
        return on;
    }
    namespace detail {
        /// Text of one of the library's reports (sbb_report)
        inline std::string report_text(int what) {
            std::string buf(1 << 14, '\0');
            for (;;) {
                std::size_t needed = 0;
                const int rc = sbb_report(what, &buf[0], buf.size(), &needed);
                if (rc == 2) {
                    buf.assign(needed + 16, '\0');
                    continue;
                }
                if (rc != 0) throw std::runtime_error(sbb_last_error());
                buf.resize(std::strlen(buf.c_str()));
                return buf;
            }
        }
    }
    /// performance.h:357: forget what has been tracked so far
    inline void resetTimings() {
        if (sbb_reset_timings() != 0) throw std::runtime_error(sbb_last_error());
    }
    /// performance.h:365: per public call, host and device time, calls, flops and bytes (SB_TRACK_TIME)
    template <typename OStream> void reportTimings(OStream &s) {
        if (!getTrackingTime()) return;
        s << detail::report_text(0);
    }
    /// performance.h:443: cached plans and pooled workspaces (SB_TRACK_MEMORY)
    template <typename OStream> void reportCacheUsage(OStream &s) {
        if (!getTrackingMemory()) return;
        s << detail::report_text(1);
    }
    /// performance.h:476
    template <typename OStream> void reportCurrentMemoryAllocations(OStream &s) {
        if (!getTrackingMemory()) return;
        s << detail::report_text(2);
    }
    /// performance.h:494: after clearCaches() nothing handed out by the library's allocator
    /// (detail::vector, allocate) may still be around (SB_TRACK_MEMORY)
    template <typename OStream> void checkForMemoryLeaks(OStream &s) {
        if (!getTrackingMemory()) return;
        long long blocks = 0, bytes = 0;
        if (sbb_live_allocations(&blocks, &bytes) != 0) throw std::runtime_error(sbb_last_error());
        if (blocks == 0) return;
        reportCurrentMemoryAllocations(s);
        throw std::runtime_error("checkForMemoryLeaks: some allocations are still around");
    }

    // ---- partitions ---------------------------------------------------------------------------------

    template <std::size_t Nd, typename std::enable_if<(Nd > 0), bool>::type = true>
    Coor<Nd> partitioning_distributed_procs(const char *order, const Coor<Nd> &dim,
                                            const char *dist_labels, unsigned int nprocs) {
        Coor<Nd> r;
        detail::check(sbb_partitioning_distributed_procs((int)Nd, order, dim.data(), dist_labels,
                                                         (int)nprocs, r.data()));
        return r;
    }

    template <std::size_t Nd>
    std::vector<PartitionItem<Nd>> basic_partitioning(const char *order, Coor<Nd> dim,
                                                      Coor<Nd> procs, const char *dist_labels,
                                                      int nprocs = -1, int ncomponents = 1) {
        const int vol_procs = (int)detail::volume<Nd>(procs);
        std::vector<int> flat((std::size_t)(nprocs < 0 ? vol_procs : nprocs) * ncomponents * 2 * Nd);
        detail::check(sbb_basic_partitioning((int)Nd, order, dim.data(), procs.data(), dist_labels,
                                             nprocs, ncomponents, flat.data()));
        return detail::boxes_from<Nd>(flat);
    }

    template <std::size_t Nd>
    std::vector<PartitionItem<Nd>> basic_partitioning(Coor<Nd> dim, Coor<Nd> procs, int nprocs = -1,
                                                      bool replicate = false,
                                                      Coor<Nd> ext_power = {{}}) {
        const int vol_procs = (int)detail::volume<Nd>(procs);
        std::vector<int> flat((std::size_t)(nprocs < 0 ? vol_procs : nprocs) * 2 * Nd);
        detail::check(sbb_basic_partitioning_ext((int)Nd, dim.data(), procs.data(), nprocs,
                                                 replicate ? 1 : 0, ext_power.data(), flat.data()));
        return detail::boxes_from<Nd>(flat);
    }

    template <std::size_t N>
    std::vector<std::array<Coor<N>, 2>> make_hole(const Coor<N> &from, const Coor<N> &size,
                                                  const Coor<N> &hole_from,
                                                  const Coor<N> &hole_size, const Coor<N> &dim) {
        if (N == 0) return {};
        std::size_t cap = 1;
        for (std::size_t i = 0; i < N; ++i) cap *= 4;
        std::vector<int> flat((cap + 1) * 2 * N);
        int n = 0;
        detail::check(sbb_make_hole((int)N, from.data(), size.data(), hole_from.data(),
                                    hole_size.data(), dim.data(), flat.data(), (int)cap + 1, &n));
        flat.resize((std::size_t)n * 2 * N);
        return detail::boxes_from<N>(flat);
    }

    // ---- communicator ----------------------------------------------------------------------------------

#ifdef SUPERBBLAS_USE_MPI
    namespace detail {
        /// One NCCL communicator per MPI communicator, created on first use: rank 0 makes the unique
        /// id and MPI broadcasts it; the GPU is the one of the first GPU context of the call
        inline sbb_comm_t comm_for(MPI_Comm mpicomm, int device) {
            static std::map<MPI_Comm, sbb_comm_t> comms;
            auto it = comms.find(mpicomm);
            if (it != comms.end()) return it->second;
            int rank = 0, nranks = 1;
            MPI_Comm_rank(mpicomm, &rank);
            MPI_Comm_size(mpicomm, &nranks);
            char id[128];
            if (rank == 0) check(sbb_comm_unique_id(id));
            MPI_Bcast(id, 128, MPI_BYTE, 0, mpicomm);
            sbb_comm_t c = nullptr;
            check(sbb_comm_create(id, nranks, rank, device, &c));
            comms[mpicomm] = c;
            return c;
        }
        inline int first_device(const Context *ctx, int n) {
            for (int i = 0; i < n; ++i)
                if (ctx[i].plat != CPU) return ctx[i].device;
            return 0;
        }
    }
#endif

    // ---- SB_DEBUG >= 2: every copy first verifies itself on mock tensors (reference: ns_copy_test,
    //      dist.h:1919-2116, called from copy_request at dist.h:2282-2285) ------------------------------
    template <std::size_t Nd0, std::size_t Nd1, typename T, typename Q>
    void copy(typename detail::elem<T>::type alpha, const PartitionItem<Nd0> *p0, int ncomponents0,
              const char *o0, const Coor<Nd0> &from0, const Coor<Nd0> &size0, const Coor<Nd0> &dim0,
              const T **v0, const MaskType **mask0, const Context *ctx0,
              const PartitionItem<Nd1> *p1, int ncomponents1, const char *o1,
              const Coor<Nd1> &from1, const Coor<Nd1> &dim1, Q **v1, const MaskType **mask1,
              const Context *ctx1, sbb_comm_t comm, CoorOrder co, CopyAdd copyadd,
              Request *request = nullptr, Session session = 0);

    namespace detail {
        inline bool &inside_self_check() {
            static bool v = false;
            return v;
        }

        /// The same copy on host tensors of doubles whose elements hold the global linear index of
        /// their own coordinate; afterwards every local destination element must hold the index of
        /// the source coordinate it comes from (times the number of holders for Add; 0 where a Copy
        /// has no holder; the sentinel outside the range).  The mock tensors go through the whole
        /// path (staging, kernels, exchange between ranks).  Collective like the copy itself.
        template <std::size_t Nd0, std::size_t Nd1>
        void self_check_copy(const PartitionItem<Nd0> *p0, int nc0, const char *o0, const Coor<Nd0> &from0,
                             const Coor<Nd0> &size0, const Coor<Nd0> &dim0, const PartitionItem<Nd1> *p1,
                             int nc1, const char *o1, const Coor<Nd1> &from1, const Coor<Nd1> &dim1,
                             sbb_comm_t comm, CoorOrder co, CopyAdd copyadd) {
            if (inside_self_check()) return;
            struct Guard {
                Guard() { inside_self_check() = true; }
                ~Guard() { inside_self_check() = false; }
            } guard;
            int rank = 0, nranks = 1;
            if (comm) check(sbb_comm_rank(comm, &rank, &nranks));
            const double sentinel = -1.0;
            const Coor<Nd0, long long> g0 = get_strides<long long>(dim0, co);
            std::vector<std::vector<double>> m0(nc0), m1(nc1);
            for (int c = 0; c < nc0; ++c) {
                const PartitionItem<Nd0> &b = p0[(std::size_t)rank * nc0 + c];
                const std::size_t vol = volume<Nd0>(b[1]);
                const Coor<Nd0, long long> ls = get_strides<long long>(b[1], co);
                m0[c].resize(vol);
                for (std::size_t i = 0; i < vol; ++i) {
                    Coor<Nd0> x = index2coor<Nd0, int, long long>((long long)i, b[1], ls);
                    for (std::size_t k = 0; k < Nd0; ++k) x[k] = (x[k] + b[0][k]) % dim0[k];
                    m0[c][i] = (double)coor2index<Nd0, int, long long>(x, dim0, g0);
                }
            }
            for (int c = 0; c < nc1; ++c)
                m1[c].assign(volume<Nd1>(p1[(std::size_t)rank * nc1 + c][1]), sentinel);
            std::vector<const double *> s(nc0);
            std::vector<double *> d(nc1);
            for (int c = 0; c < nc0; ++c) s[c] = m0[c].data();
            for (int c = 0; c < nc1; ++c) d[c] = m1[c].data();
            std::vector<Context> c0(nc0, Context{CPU, CPU_DEVICE_ID}), c1(nc1, Context{CPU, CPU_DEVICE_ID});
            superbblas::copy<Nd0, Nd1, double, double>(1.0, p0, nc0, o0, from0, size0, dim0, s.data(), nullptr,
                                                       c0.data(), p1, nc1, o1, from1, dim1, d.data(), nullptr,
                                                       c1.data(), comm, co, copyadd, nullptr, 0);
            // position of every destination label in the source order (-1: absent, extent 1)
            int pos0[Nd1 ? Nd1 : 1];
            for (std::size_t k1 = 0; k1 < Nd1; ++k1) {
                pos0[k1] = -1;
                for (std::size_t k0 = 0; k0 < Nd0; ++k0)
                    if (o0[k0] == o1[k1]) pos0[k1] = (int)k0;
            }
            for (int c = 0; c < nc1; ++c) {
                const PartitionItem<Nd1> &b = p1[(std::size_t)rank * nc1 + c];
                const Coor<Nd1, long long> ls = get_strides<long long>(b[1], co);
                for (std::size_t i = 0; i < m1[c].size(); ++i) {
                    Coor<Nd1> y = index2coor<Nd1, int, long long>((long long)i, b[1], ls);
                    Coor<Nd0> x = from0;
                    bool in_range = true;
                    for (std::size_t k1 = 0; k1 < Nd1 && in_range; ++k1) {
                        const int g = (y[k1] + b[0][k1]) % dim1[k1];
                        const int rel = ((g - from1[k1]) % dim1[k1] + dim1[k1]) % dim1[k1];
                        const int extent = pos0[k1] >= 0 ? size0[pos0[k1]] : 1;
                        if (rel >= extent) in_range = false;
                        else if (pos0[k1] >= 0) x[pos0[k1]] = (from0[pos0[k1]] + rel) % dim0[pos0[k1]];
                    }
                    double want = sentinel;
                    if (in_range) {
                        int rep = 0;
                        for (std::size_t q = 0; q < (std::size_t)nranks * nc0; ++q) {
                            bool holds = true;
                            for (std::size_t k = 0; k < Nd0 && holds; ++k) {
                                const int sz = p0[q][1][k];
                                const int rel = ((x[k] - p0[q][0][k]) % dim0[k] + dim0[k]) % dim0[k];
                                holds = sz > 0 && (sz >= dim0[k] || rel < sz);
                            }
                            rep += holds;
                        }
                        const double idx = (double)coor2index<Nd0, int, long long>(x, dim0, g0);
                        want = copyadd == Copy ? (rep ? idx : 0.0) : sentinel + rep * idx;
                    }
                    if (m1[c][i] != want)
                        throw std::runtime_error("SB_DEBUG self-check of copy failed: component " +
                                                 std::to_string(c) + " element " + std::to_string(i) + " holds " +
                                                 std::to_string(m1[c][i]) + ", expected " + std::to_string(want));
                }
            }
        }
    }

    // ---- copy ------------------------------------------------------------------------------------------

    /// Copy the content of plural tensor v0 into v1 (reference: dist.h:3534 with the communicator
    /// being an NCCL rank instead of an MPI_Comm)
    template <std::size_t Nd0, std::size_t Nd1, typename T, typename Q>
    void copy(typename detail::elem<T>::type alpha, const PartitionItem<Nd0> *p0, int ncomponents0,
              const char *o0, const Coor<Nd0> &from0, const Coor<Nd0> &size0, const Coor<Nd0> &dim0,
              const T **v0, const MaskType **mask0, const Context *ctx0,
              const PartitionItem<Nd1> *p1, int ncomponents1, const char *o1,
              const Coor<Nd1> &from1, const Coor<Nd1> &dim1, Q **v1, const MaskType **mask1,
              const Context *ctx1, sbb_comm_t comm, CoorOrder co, CopyAdd copyadd,
              Request *request, Session session) {
        if (session != 0) throw std::runtime_error("unsupported session");
        detail::check_order<Nd0>(o0, "o0");
        detail::check_order<Nd1>(o1, "o1");
        if (getDebugLevel() >= 2 && !mask0 && !mask1)
            detail::self_check_copy<Nd0, Nd1>(p0, ncomponents0, o0, from0, size0, dim0, p1, ncomponents1, o1,
                                              from1, dim1, comm, co, copyadd);
        const auto a = detail::scalar(alpha);
        if (request) {
            // deferred completion (dist.h:3554-3557): the packs, their signal and the local part are
            // queued now; wait(request) queues the unpack side and completes host destinations
            sbb_request_t h = nullptr;
            detail::check(sbb_copy_begin(detail::dtype_of<T>::value, detail::dtype_of<Q>::value, a.data(),
                                         (int)Nd0, (const int *)p0, ncomponents0, o0, from0.data(),
                                         size0.data(), dim0.data(), (const void *const *)v0,
                                         (const float *const *)mask0, detail::ctx_ptr(ctx0), (int)Nd1,
                                         (const int *)p1, ncomponents1, o1, from1.data(), dim1.data(),
                                         (void *const *)v1, (const float *const *)mask1,
                                         detail::ctx_ptr(ctx1), comm, co == SlowToFast ? 0 : 1,
                                         copyadd == Copy ? 0 : 1, &h));
            *request = detail::make_request(h);
            return;
        }
        detail::check(sbb_copy(detail::dtype_of<T>::value, detail::dtype_of<Q>::value, a.data(),
                               (int)Nd0, (const int *)p0, ncomponents0, o0, from0.data(),
                               size0.data(), dim0.data(), (const void *const *)v0,
                               (const float *const *)mask0, detail::ctx_ptr(ctx0), (int)Nd1,
                               (const int *)p1, ncomponents1, o1, from1.data(), dim1.data(),
                               (void *const *)v1, (const float *const *)mask1,
                               detail::ctx_ptr(ctx1), comm, co == SlowToFast ? 0 : 1,
                               copyadd == Copy ? 0 : 1));
    }

    /// No-communicator overload (reference: dist.h:3583)
    template <std::size_t Nd0, std::size_t Nd1, typename T, typename Q>
    void copy(typename detail::elem<T>::type alpha, const PartitionItem<Nd0> *p0, int ncomponents0,
              const char *o0, const Coor<Nd0> from0, const Coor<Nd0> size0, const Coor<Nd0> dim0,
              const T **v0, const MaskType **mask0, const Context *ctx0,
              const PartitionItem<Nd1> *p1, int ncomponents1, const char *o1, const Coor<Nd1> from1,
              const Coor<Nd1> dim1, Q **v1, const MaskType **mask1, const Context *ctx1,
              CoorOrder co, CopyAdd copyadd, Request *request = nullptr, Session session = 0) {
        copy<Nd0, Nd1, T, Q>(alpha, p0, ncomponents0, o0, from0, size0, dim0, v0, mask0, ctx0, p1,
                             ncomponents1, o1, from1, dim1, v1, mask1, ctx1, (sbb_comm_t) nullptr,
                             co, copyadd, request, session);
    }

#ifdef SUPERBBLAS_USE_MPI
    template <std::size_t Nd0, std::size_t Nd1, typename T, typename Q>
    void copy(typename detail::elem<T>::type alpha, const PartitionItem<Nd0> *p0, int ncomponents0,
              const char *o0, const Coor<Nd0> &from0, const Coor<Nd0> &size0, const Coor<Nd0> &dim0,
              const T **v0, const MaskType **mask0, const Context *ctx0,
              const PartitionItem<Nd1> *p1, int ncomponents1, const char *o1,
              const Coor<Nd1> &from1, const Coor<Nd1> &dim1, Q **v1, const MaskType **mask1,
              const Context *ctx1, MPI_Comm mpicomm, CoorOrder co, CopyAdd copyadd,
              Request *request = nullptr, Session session = 0) {
        copy<Nd0, Nd1, T, Q>(alpha, p0, ncomponents0, o0, from0, size0, dim0, v0, mask0, ctx0, p1,
                             ncomponents1, o1, from1, dim1, v1, mask1, ctx1,
                             detail::comm_for(mpicomm, detail::first_device(ctx1, ncomponents1)),
                             co, copyadd, request, session);
    }
#endif

    /// Copy between two single-component tensors (signature of the reference's tests/local.cpp:97)
    template <std::size_t Nd0, std::size_t Nd1, typename T, typename Q>
    void local_copy(typename detail::elem<T>::type alpha, const char *o0, const Coor<Nd0> &from0,
                    const Coor<Nd0> &size0, const Coor<Nd0> &dim0, const T *v0,
                    const MaskType *mask0, Context ctx0, const char *o1, const Coor<Nd1> &from1,
                    const Coor<Nd1> &dim1, Q *v1, const MaskType *mask1, Context ctx1, CoorOrder co,
                    CopyAdd copyadd) {
        PartitionItem<Nd0> p0{Coor<Nd0>{{}}, dim0};
        PartitionItem<Nd1> p1{Coor<Nd1>{{}}, dim1};
        const MaskType **m0 = mask0 ? &mask0 : nullptr, **m1 = mask1 ? &mask1 : nullptr;
        copy<Nd0, Nd1, T, Q>(alpha, &p0, 1, o0, from0, size0, dim0, &v0, m0, &ctx0, &p1, 1, o1, from1,
                             dim1, &v1, m1, &ctx1, co, copyadd);
    }

    // ---- contraction ---------------------------------------------------------------------------------------

    /// vr = alpha * contraction(v0, v1) + beta * vr (reference: dist.h:3628 with an NCCL communicator)
    template <std::size_t Nd0, std::size_t Nd1, std::size_t Ndo, typename T>
    void contraction(T alpha, const PartitionItem<Nd0> *p0, const Coor<Nd0> &from0,
                     const Coor<Nd0> &size0, const Coor<Nd0> &dim0, int ncomponents0,
                     const char *o0, bool conj0, const T **v0, const Context *ctx0,
                     const PartitionItem<Nd1> *p1, const Coor<Nd1> &from1, const Coor<Nd1> &size1,
                     const Coor<Nd1> &dim1, int ncomponents1, const char *o1, bool conj1,
                     const T **v1, const Context *ctx1, T beta, const PartitionItem<Ndo> *pr,
                     const Coor<Ndo> &fromr, const Coor<Ndo> &sizer, const Coor<Ndo> &dimr,
                     int ncomponentsr, const char *o_r, T **vr, const Context *ctxr,
                     sbb_comm_t comm, CoorOrder co, Request *request = nullptr,
                     Session session = 0) {
        if (session != 0) throw std::runtime_error("unsupported session");
        if (detail::dtype_of<T>::value == SBB_I32)
            throw std::runtime_error("contraction: unsupported type");
        detail::check_order<Nd0>(o0, "o0");
        detail::check_order<Nd1>(o1, "o1");
        detail::check_order<Ndo>(o_r, "o_r");
        const auto a = detail::scalar(alpha), b = detail::scalar(beta);
        detail::check(sbb_contraction(
            detail::dtype_of<T>::value, a.data(), (int)Nd0, (const int *)p0, from0.data(),
            size0.data(), dim0.data(), ncomponents0, o0, conj0 ? 1 : 0, (const void *const *)v0,
            detail::ctx_ptr(ctx0), (int)Nd1, (const int *)p1, from1.data(), size1.data(),
            dim1.data(), ncomponents1, o1, conj1 ? 1 : 0, (const void *const *)v1,
            detail::ctx_ptr(ctx1), b.data(), (int)Ndo, (const int *)pr, fromr.data(), sizer.data(),
            dimr.data(), ncomponentsr, o_r, (void *const *)vr, detail::ctx_ptr(ctxr), comm,
            co == SlowToFast ? 0 : 1));
        if (request) *request = Request{};
    }

    /// No-communicator overload (reference: dist.h:3701)
    template <std::size_t Nd0, std::size_t Nd1, std::size_t Ndo, typename T>
    void contraction(T alpha, const PartitionItem<Nd0> *p0, const Coor<Nd0> from0,
                     const Coor<Nd0> size0, const Coor<Nd0> &dim0, int ncomponents0, const char *o0,
                     bool conj0, const T **v0, const Context *ctx0, const PartitionItem<Nd1> *p1,
                     const Coor<Nd1> &from1, const Coor<Nd1> &size1, const Coor<Nd1> &dim1,
                     int ncomponents1, const char *o1, bool conj1, const T **v1,
                     const Context *ctx1, T beta, const PartitionItem<Ndo> *pr,
                     const Coor<Ndo> &fromr, const Coor<Ndo> &sizer, const Coor<Ndo> &dimr,
                     int ncomponentsr, const char *o_r, T **vr, const Context *ctxr, CoorOrder co,
                     Request *request = nullptr, Session session = 0) {
        contraction<Nd0, Nd1, Ndo, T>(alpha, p0, from0, size0, dim0, ncomponents0, o0, conj0, v0,
                                      ctx0, p1, from1, size1, dim1, ncomponents1, o1, conj1, v1,
                                      ctx1, beta, pr, fromr, sizer, dimr, ncomponentsr, o_r, vr,
                                      ctxr, (sbb_comm_t) nullptr, co, request, session);
    }

#ifdef SUPERBBLAS_USE_MPI
    template <std::size_t Nd0, std::size_t Nd1, std::size_t Ndo, typename T>
    void contraction(T alpha, const PartitionItem<Nd0> *p0, const Coor<Nd0> &from0,
                     const Coor<Nd0> &size0, const Coor<Nd0> &dim0, int ncomponents0,
                     const char *o0, bool conj0, const T **v0, const Context *ctx0,
                     const PartitionItem<Nd1> *p1, const Coor<Nd1> &from1, const Coor<Nd1> &size1,
                     const Coor<Nd1> &dim1, int ncomponents1, const char *o1, bool conj1,
                     const T **v1, const Context *ctx1, T beta, const PartitionItem<Ndo> *pr,
                     const Coor<Ndo> &fromr, const Coor<Ndo> &sizer, const Coor<Ndo> &dimr,
                     int ncomponentsr, const char *o_r, T **vr, const Context *ctxr,
                     MPI_Comm mpicomm, CoorOrder co, Request *request = nullptr,
                     Session session = 0) {
        contraction<Nd0, Nd1, Ndo, T>(
            alpha, p0, from0, size0, dim0, ncomponents0, o0, conj0, v0, ctx0, p1, from1, size1, dim1,
            ncomponents1, o1, conj1, v1, ctx1, beta, pr, fromr, sizer, dimr, ncomponentsr, o_r, vr,
            ctxr, detail::comm_for(mpicomm, detail::first_device(ctxr, ncomponentsr)), co, request,
            session);
    }
#endif

    /// Contraction of single-component tensors (signature of the reference's tests/local.cpp:163)
    template <std::size_t Nd0, std::size_t Nd1, std::size_t Ndo, typename T>
    void local_contraction(T alpha, const char *o0, const Coor<Nd0> &dim0, bool conj0, const T *v0,
                           const char *o1, const Coor<Nd1> &dim1, bool conj1, const T *v1, T beta,
                           const char *o_r, const Coor<Ndo> &dimr, T *vr, Context ctx,
                           CoorOrder co) {
        PartitionItem<Nd0> p0{Coor<Nd0>{{}}, dim0};
        PartitionItem<Nd1> p1{Coor<Nd1>{{}}, dim1};
        PartitionItem<Ndo> pr{Coor<Ndo>{{}}, dimr};
        contraction<Nd0, Nd1, Ndo, T>(alpha, &p0, Coor<Nd0>{{}}, dim0, dim0, 1, o0, conj0, &v0, &ctx,
                                      &p1, Coor<Nd1>{{}}, dim1, dim1, 1, o1, conj1, &v1, &ctx, beta,
                                      &pr, Coor<Ndo>{{}}, dimr, dimr, 1, o_r, &vr, &ctx, co);
    }

    // ---- batched dense solvers (reference: dense.h:1019-1290; semantics in superbblas_b200.h) -----------

    namespace detail {
        using SquareFn = int (*)(int, int, const int *, int, const char *, void *const *, const char *,
                                 const char *, const sbb_context *, sbb_comm_t, int);
        using SquareBeginFn = int (*)(int, int, const int *, int, const char *, void *const *, const char *,
                                      const char *, const sbb_context *, sbb_comm_t, int, sbb_request_t *);

        /// With a request the call is begun (fn_begin) and `*request` completes it
        template <std::size_t N, typename T>
        void square_op(SquareFn fn, SquareBeginFn fn_begin, const char *name, const PartitionItem<N> *p,
                       int ncomponents, const char *o, T **v, const char *orows, const char *ocols,
                       const Context *ctx, sbb_comm_t comm, CoorOrder co, Request *request, Session session) {
            if (session != 0) throw std::runtime_error("unsupported session");
            if (dtype_of<T>::value == SBB_I32) throw std::runtime_error(std::string(name) + ": unsupported type");
            check_order<N>(o, "o");
            if (request) {
                sbb_request_t h = nullptr;
                check(fn_begin(dtype_of<T>::value, (int)N, (const int *)p, ncomponents, o, (void *const *)v, orows,
                               ocols, ctx_ptr(ctx), comm, co == SlowToFast ? 0 : 1, &h));
                *request = make_request(h);
                return;
            }
            check(fn(dtype_of<T>::value, (int)N, (const int *)p, ncomponents, o, (void *const *)v, orows, ocols,
                     ctx_ptr(ctx), comm, co == SlowToFast ? 0 : 1));
        }

        using SolveFn = int (*)(int, const double *, int, const int *, int, const char *, const char *,
                                const char *, const void *const *, const sbb_context *, int, const int *, int,
                                const char *, const void *const *, const sbb_context *, int, const int *,
                                int, const char *, void *const *, const sbb_context *, sbb_comm_t, int);
        using SolveBeginFn = int (*)(int, const double *, int, const int *, int, const char *, const char *,
                                     const char *, const void *const *, const sbb_context *, int, const int *,
                                     int, const char *, const void *const *, const sbb_context *, int,
                                     const int *, int, const char *, void *const *, const sbb_context *,
                                     sbb_comm_t, int, sbb_request_t *);

        /// With a request the call is begun (fn_begin) and `*request` completes it
        template <std::size_t Nc, std::size_t Nx, std::size_t Ny, typename T>
        void solve_op(SolveFn fn, SolveBeginFn fn_begin, const char *name, T alpha, const PartitionItem<Nc> *pc,
                      int ncomponentsc, const char *oc, const char *orows, const char *ocols, const T **vc,
                      const Context *ctxc, const PartitionItem<Nx> *px, int ncomponentsx, const char *ox,
                      const T **vx, const Context *ctxx, const PartitionItem<Ny> *py, int ncomponentsy,
                      const char *oy, T **vy, const Context *ctxy, sbb_comm_t comm, CoorOrder co,
                      Request *request, Session session) {
            if (session != 0) throw std::runtime_error("unsupported session");
            if (dtype_of<T>::value == SBB_I32) throw std::runtime_error(std::string(name) + ": unsupported type");
            check_order<Nc>(oc, "oc");
            check_order<Nx>(ox, "ox");
            check_order<Ny>(oy, "oy");
            const auto a = scalar(alpha);
            const int cco = co == SlowToFast ? 0 : 1;
            if (request) {
                sbb_request_t h = nullptr;
                check(fn_begin(dtype_of<T>::value, a.data(), (int)Nc, (const int *)pc, ncomponentsc, oc, orows,
                               ocols, (const void *const *)vc, ctx_ptr(ctxc), (int)Nx, (const int *)px,
                               ncomponentsx, ox, (const void *const *)vx, ctx_ptr(ctxx), (int)Ny, (const int *)py,
                               ncomponentsy, oy, (void *const *)vy, ctx_ptr(ctxy), comm, cco, &h));
                *request = make_request(h);
                return;
            }
            check(fn(dtype_of<T>::value, a.data(), (int)Nc, (const int *)pc, ncomponentsc, oc, orows, ocols,
                     (const void *const *)vc, ctx_ptr(ctxc), (int)Nx, (const int *)px, ncomponentsx, ox,
                     (const void *const *)vx, ctx_ptr(ctxx), (int)Ny, (const int *)py, ncomponentsy, oy,
                     (void *const *)vy, ctx_ptr(ctxy), comm, cco));
        }
    }

#define SUPERBBLAS_B200_SQUARE_OP(NAME)                                                                        \
    /** NAME of every matrix (rows orows, columns ocols) in place, with an NCCL communicator */                 \
    template <std::size_t N, typename T>                                                                       \
    void NAME(const PartitionItem<N> *p, int ncomponents, const char *o, T **v, const char *orows,              \
              const char *ocols, const Context *ctx, sbb_comm_t comm, CoorOrder co, Request *request = nullptr, \
              Session session = 0) {                                                                           \
        detail::square_op<N, T>(sbb_##NAME, sbb_##NAME##_begin, #NAME, p, ncomponents, o, v, orows, ocols, ctx, \
                                comm, co, request, session);                                                   \
    }                                                                                                          \
    /** No-communicator overload */                                                                            \
    template <std::size_t N, typename T>                                                                       \
    void NAME(const PartitionItem<N> *p, int ncomponents, const char *o, T **v, const char *orows,              \
              const char *ocols, const Context *ctx, CoorOrder co, Request *request = nullptr,                 \
              Session session = 0) {                                                                           \
        detail::square_op<N, T>(sbb_##NAME, sbb_##NAME##_begin, #NAME, p, ncomponents, o, v, orows, ocols, ctx, \
                                (sbb_comm_t) nullptr, co, request, session);                                   \
    }

#define SUPERBBLAS_B200_SOLVE_OP(NAME)                                                                         \
    /** Solve with every matrix of c (rows orows, columns ocols); with an NCCL communicator */                \
    template <std::size_t Nc, std::size_t Nx, std::size_t Ny, typename T>                                      \
    void NAME(T alpha, const PartitionItem<Nc> *pc, int ncomponentsc, const char *oc, const char *orows,       \
              const char *ocols, const T **vc, const Context *ctxc, const PartitionItem<Nx> *px,               \
              int ncomponentsx, const char *ox, const T **vx, const Context *ctxx,                             \
              const PartitionItem<Ny> *py, int ncomponentsy, const char *oy, T **vy, const Context *ctxy,      \
              sbb_comm_t comm, CoorOrder co, Request *request = nullptr, Session session = 0) {                \
        detail::solve_op<Nc, Nx, Ny, T>(sbb_##NAME, sbb_##NAME##_begin, #NAME, alpha, pc, ncomponentsc, oc,   \
                                        orows, ocols, vc, ctxc, px, ncomponentsx, ox, vx, ctxx, py,           \
                                        ncomponentsy, oy, vy, ctxy, comm, co, request, session);              \
    }                                                                                                          \
    /** No-communicator overload */                                                                            \
    template <std::size_t Nc, std::size_t Nx, std::size_t Ny, typename T>                                      \
    void NAME(T alpha, const PartitionItem<Nc> *pc, int ncomponentsc, const char *oc, const char *orows,       \
              const char *ocols, const T **vc, const Context *ctxc, const PartitionItem<Nx> *px,               \
              int ncomponentsx, const char *ox, const T **vx, const Context *ctxx,                             \
              const PartitionItem<Ny> *py, int ncomponentsy, const char *oy, T **vy, const Context *ctxy,      \
              CoorOrder co, Request *request = nullptr, Session session = 0) {                                 \
        detail::solve_op<Nc, Nx, Ny, T>(sbb_##NAME, sbb_##NAME##_begin, #NAME, alpha, pc, ncomponentsc, oc,   \
                                        orows, ocols, vc, ctxc, px, ncomponentsx, ox, vx, ctxx, py,           \
                                        ncomponentsy, oy, vy, ctxy, (sbb_comm_t) nullptr, co, request,        \
                                        session);                                                              \
    }

    /// A = U^H U, U upper triangular, in place
    SUPERBBLAS_B200_SQUARE_OP(cholesky)
    /// A <- A^-1, in place
    SUPERBBLAS_B200_SQUARE_OP(inversion)
    /// Solve with the upper triangle of c: c y = alpha x (x carries orows) or y c = alpha x (x carries ocols)
    SUPERBBLAS_B200_SOLVE_OP(trsm)
    /// The same with a general matrix, by LU with partial pivoting
    SUPERBBLAS_B200_SOLVE_OP(gesm)

#undef SUPERBBLAS_B200_SQUARE_OP
#undef SUPERBBLAS_B200_SOLVE_OP

    namespace detail {
        template <typename T> struct real_of { using type = T; };
        template <typename T> struct real_of<std::complex<T>> { using type = T; };

        template <std::size_t N, std::size_t Nw, typename T>
        void eigh(const PartitionItem<N> *p, int ncomponents, const char *o, T **v, const char *orows,
                  const char *ocols, const Context *ctx, const PartitionItem<Nw> *pw, int ncomponentsw, const char *ow,
                  typename real_of<T>::type **vw, const Context *ctxw, sbb_comm_t comm, CoorOrder co, Session session) {
            if (session != 0) throw std::runtime_error("unsupported session");
            if (dtype_of<T>::value == SBB_I32) throw std::runtime_error("eigh: unsupported type");
            check_order<N>(o, "o");
            check_order<Nw>(ow, "ow");
            check(sbb_eigh(dtype_of<T>::value, (int)N, (const int *)p, ncomponents, o, (void *const *)v, orows, ocols,
                           ctx_ptr(ctx), (int)Nw, (const int *)pw, ncomponentsw, ow, (void *const *)vw, ctx_ptr(ctxw),
                           comm, co == SlowToFast ? 0 : 1));
        }
    }

    /// (ours) Every Hermitian matrix of v (rows orows, columns ocols; the upper triangle is read) is replaced
    /// in place by its eigenvectors V, A = V diag(w) V^H, and w (the batch labels and ocols, element type the
    /// real type of T) gets the eigenvalues in ascending order; with an NCCL communicator
    template <std::size_t N, std::size_t Nw, typename T>
    void eigh(const PartitionItem<N> *p, int ncomponents, const char *o, T **v, const char *orows, const char *ocols,
              const Context *ctx, const PartitionItem<Nw> *pw, int ncomponentsw, const char *ow,
              typename detail::real_of<T>::type **vw, const Context *ctxw, sbb_comm_t comm, CoorOrder co,
              Session session = 0) {
        detail::eigh<N, Nw, T>(p, ncomponents, o, v, orows, ocols, ctx, pw, ncomponentsw, ow, vw, ctxw, comm, co,
                               session);
    }
    /// No-communicator overload
    template <std::size_t N, std::size_t Nw, typename T>
    void eigh(const PartitionItem<N> *p, int ncomponents, const char *o, T **v, const char *orows, const char *ocols,
              const Context *ctx, const PartitionItem<Nw> *pw, int ncomponentsw, const char *ow,
              typename detail::real_of<T>::type **vw, const Context *ctxw, CoorOrder co, Session session = 0) {
        detail::eigh<N, Nw, T>(p, ncomponents, o, v, orows, ocols, ctx, pw, ncomponentsw, ow, vw, ctxw,
                               (sbb_comm_t) nullptr, co, session);
    }

#ifdef SUPERBBLAS_USE_MPI
    template <std::size_t N, typename T>
    void cholesky(const PartitionItem<N> *p, int ncomponents, const char *o, T **v, const char *orows,
                  const char *ocols, const Context *ctx, MPI_Comm mpicomm, CoorOrder co, Request *request = nullptr,
                  Session session = 0) {
        detail::square_op<N, T>(sbb_cholesky, sbb_cholesky_begin, "cholesky", p, ncomponents, o, v, orows, ocols, ctx,
                                detail::comm_for(mpicomm, detail::first_device(ctx, ncomponents)), co, request,
                                session);
    }
    template <std::size_t N, typename T>
    void inversion(const PartitionItem<N> *p, int ncomponents, const char *o, T **v, const char *orows,
                   const char *ocols, const Context *ctx, MPI_Comm mpicomm, CoorOrder co, Request *request = nullptr,
                   Session session = 0) {
        detail::square_op<N, T>(sbb_inversion, sbb_inversion_begin, "inversion", p, ncomponents, o, v, orows, ocols, ctx,
                                detail::comm_for(mpicomm, detail::first_device(ctx, ncomponents)), co, request,
                                session);
    }
    template <std::size_t Nc, std::size_t Nx, std::size_t Ny, typename T>
    void trsm(T alpha, const PartitionItem<Nc> *pc, int ncomponentsc, const char *oc, const char *orows,
              const char *ocols, const T **vc, const Context *ctxc, const PartitionItem<Nx> *px,
              int ncomponentsx, const char *ox, const T **vx, const Context *ctxx, const PartitionItem<Ny> *py,
              int ncomponentsy, const char *oy, T **vy, const Context *ctxy, MPI_Comm mpicomm, CoorOrder co,
              Request *request = nullptr, Session session = 0) {
        detail::solve_op<Nc, Nx, Ny, T>(sbb_trsm, sbb_trsm_begin, "trsm", alpha, pc, ncomponentsc, oc, orows, ocols, vc, ctxc,
                                        px, ncomponentsx, ox, vx, ctxx, py, ncomponentsy, oy, vy, ctxy,
                                        detail::comm_for(mpicomm, detail::first_device(ctxy, ncomponentsy)),
                                        co, request, session);
    }
    template <std::size_t Nc, std::size_t Nx, std::size_t Ny, typename T>
    void gesm(T alpha, const PartitionItem<Nc> *pc, int ncomponentsc, const char *oc, const char *orows,
              const char *ocols, const T **vc, const Context *ctxc, const PartitionItem<Nx> *px,
              int ncomponentsx, const char *ox, const T **vx, const Context *ctxx, const PartitionItem<Ny> *py,
              int ncomponentsy, const char *oy, T **vy, const Context *ctxy, MPI_Comm mpicomm, CoorOrder co,
              Request *request = nullptr, Session session = 0) {
        detail::solve_op<Nc, Nx, Ny, T>(sbb_gesm, sbb_gesm_begin, "gesm", alpha, pc, ncomponentsc, oc, orows, ocols, vc, ctxc,
                                        px, ncomponentsx, ox, vx, ctxx, py, ncomponentsy, oy, vy, ctxy,
                                        detail::comm_for(mpicomm, detail::first_device(ctxy, ncomponentsy)),
                                        co, request, session);
    }
    template <std::size_t N, std::size_t Nw, typename T>
    void eigh(const PartitionItem<N> *p, int ncomponents, const char *o, T **v, const char *orows, const char *ocols,
              const Context *ctx, const PartitionItem<Nw> *pw, int ncomponentsw, const char *ow,
              typename detail::real_of<T>::type **vw, const Context *ctxw, MPI_Comm mpicomm, CoorOrder co,
              Session session = 0) {
        detail::eigh<N, Nw, T>(p, ncomponents, o, v, orows, ocols, ctx, pw, ncomponentsw, ow, vw, ctxw,
                               detail::comm_for(mpicomm, detail::first_device(ctx, ncomponents)), co, session);
    }
#endif

    // ---- block-sparse operators (reference: bsr.h:2286, :2352, :2516; semantics in superbblas_b200.h) ----

    /// An operator made by create_bsr; it references the caller's v until destroy_bsr
    struct BSR_handle;

    namespace detail {
        template <std::size_t ND, std::size_t NI, typename T>
        void create_bsr(const PartitionItem<NI> *pim, const Coor<NI> &dimi, const PartitionItem<ND> *pdom,
                        const Coor<ND> &dimd, int ncomponents, const Coor<NI> &blockim, const Coor<ND> &blockdom,
                        bool blockImFast, IndexType **ii, Coor<ND> **jj, const T **v, const Context *ctx,
                        sbb_comm_t comm, CoorOrder co, BSR_handle **bsrh, Session session) {
            if (session != 0) throw std::runtime_error("unsupported session");
            if (dtype_of<T>::value == SBB_I32) throw std::runtime_error("create_bsr: unsupported type");
            sbb_bsr_t h = nullptr;
            check(sbb_create_bsr(dtype_of<T>::value, (int)NI, (const int *)pim, dimi.data(), (int)ND,
                                 (const int *)pdom, dimd.data(), ncomponents, blockim.data(), blockdom.data(),
                                 blockImFast ? 1 : 0, (const int *const *)ii, (const int *const *)jj,
                                 (const void *const *)v, ctx_ptr(ctx), comm, co == SlowToFast ? 0 : 1, &h));
            *bsrh = (BSR_handle *)h;
        }

        template <std::size_t ND, std::size_t NI, typename T>
        void create_kron_bsr(const PartitionItem<NI> *pim, const Coor<NI> &dimi, const PartitionItem<ND> *pdom,
                             const Coor<ND> &dimd, int ncomponents, const Coor<NI> &blockim,
                             const Coor<ND> &blockdom, const Coor<NI> &kronim, const Coor<ND> &krondom,
                             bool blockImFast, IndexType **ii, Coor<ND> **jj, const T **v, const T **kronv,
                             const Context *ctx, sbb_comm_t comm, CoorOrder co, BSR_handle **bsrh,
                             Session session) {
            if (session != 0) throw std::runtime_error("unsupported session");
            if (dtype_of<T>::value == SBB_I32) throw std::runtime_error("create_kron_bsr: unsupported type");
            sbb_bsr_t h = nullptr;
            check(sbb_create_kron_bsr(dtype_of<T>::value, (int)NI, (const int *)pim, dimi.data(), (int)ND,
                                      (const int *)pdom, dimd.data(), ncomponents, blockim.data(), blockdom.data(),
                                      kronim.data(), krondom.data(), blockImFast ? 1 : 0, (const int *const *)ii,
                                      (const int *const *)jj, (const void *const *)v, (const void *const *)kronv,
                                      ctx_ptr(ctx), comm, co == SlowToFast ? 0 : 1, &h));
            *bsrh = (BSR_handle *)h;
        }

        template <std::size_t ND, std::size_t NI, std::size_t NX, std::size_t NY, typename T>
        void bsr_krylov(T alpha, BSR_handle *bsrh, const char *oim, const char *odom, const PartitionItem<NX> *px,
                        int ncomponents, const char *ox, const Coor<NX> &fromx, const Coor<NX> &sizex,
                        const Coor<NX> &dimx, const T **vx, T beta, const PartitionItem<NY> *py, const char *oy,
                        const Coor<NY> &fromy, const Coor<NY> &sizey, const Coor<NY> &dimy, char power_label,
                        T **vy, const Context *ctx, sbb_comm_t comm, CoorOrder co, Request *request,
                        Session session) {
            if (session != 0) throw std::runtime_error("unsupported session");
            if (dtype_of<T>::value == SBB_I32) throw std::runtime_error("bsr_krylov: unsupported type");
            check_order<NI>(oim, "oim");
            check_order<ND>(odom, "odom");
            check_order<NX>(ox, "ox");
            check_order<NY>(oy, "oy");
            const auto a = scalar(alpha), b = scalar(beta);
            if (request) {
                // the first step is queued now (the gather of x begun, the interior rows behind its local
                // part); wait(request) runs the rest, and y is defined after it
                sbb_request_t h = nullptr;
                check(sbb_bsr_krylov_begin(dtype_of<T>::value, a.data(), (sbb_bsr_t)bsrh, oim, odom, (int)NX,
                                           (const int *)px, ncomponents, ox, fromx.data(), sizex.data(), dimx.data(),
                                           (const void *const *)vx, ctx_ptr(ctx), b.data(), (int)NY, (const int *)py,
                                           ncomponents, oy, fromy.data(), sizey.data(), dimy.data(), power_label,
                                           (void *const *)vy, ctx_ptr(ctx), comm, co == SlowToFast ? 0 : 1, &h));
                *request = make_request(h);
                return;
            }
            check(sbb_bsr_krylov(dtype_of<T>::value, a.data(), (sbb_bsr_t)bsrh, oim, odom, (int)NX, (const int *)px,
                                 ncomponents, ox, fromx.data(), sizex.data(), dimx.data(), (const void *const *)vx,
                                 ctx_ptr(ctx), b.data(), (int)NY, (const int *)py, ncomponents, oy, fromy.data(),
                                 sizey.data(), dimy.data(), power_label, (void *const *)vy, ctx_ptr(ctx), comm,
                                 co == SlowToFast ? 0 : 1));
        }
    }

    /// Create a block-sparse operator (reference: bsr.h:2286) with an NCCL communicator
    template <std::size_t ND, std::size_t NI, typename T>
    void create_bsr(const PartitionItem<NI> *pim, const Coor<NI> &dimi, const PartitionItem<ND> *pdom,
                    const Coor<ND> &dimd, int ncomponents, const Coor<NI> &blockim, const Coor<ND> &blockdom,
                    bool blockImFast, IndexType **ii, Coor<ND> **jj, const T **v, const Context *ctx,
                    sbb_comm_t comm, CoorOrder co, BSR_handle **bsrh, Session session = 0) {
        detail::create_bsr<ND, NI, T>(pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, blockImFast, ii, jj, v,
                                      ctx, comm, co, bsrh, session);
    }
    /// No-communicator overload (reference: bsr.h:2352)
    template <std::size_t ND, std::size_t NI, typename T>
    void create_bsr(const PartitionItem<NI> *pim, const Coor<NI> &dimi, const PartitionItem<ND> *pdom,
                    const Coor<ND> &dimd, int ncomponents, const Coor<NI> &blockim, const Coor<ND> &blockdom,
                    bool blockImFast, IndexType **ii, Coor<ND> **jj, const T **v, const Context *ctx,
                    CoorOrder co, BSR_handle **bsrh, Session session = 0) {
        detail::create_bsr<ND, NI, T>(pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, blockImFast, ii, jj, v,
                                      ctx, (sbb_comm_t) nullptr, co, bsrh, session);
    }

    /// Create a Kronecker block-sparse operator (reference: create_kron_bsr in bsr.h) with an NCCL
    /// communicator: the u-th block of every row is kronv[u] ⊗ its block of v (superbblas_b200.h)
    template <std::size_t ND, std::size_t NI, typename T>
    void create_kron_bsr(const PartitionItem<NI> *pim, const Coor<NI> &dimi, const PartitionItem<ND> *pdom,
                         const Coor<ND> &dimd, int ncomponents, const Coor<NI> &blockim, const Coor<ND> &blockdom,
                         const Coor<NI> &kronim, const Coor<ND> &krondom, bool blockImFast, IndexType **ii,
                         Coor<ND> **jj, const T **v, const T **kronv, const Context *ctx, sbb_comm_t comm,
                         CoorOrder co, BSR_handle **bsrh, Session session = 0) {
        detail::create_kron_bsr<ND, NI, T>(pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, kronim, krondom,
                                           blockImFast, ii, jj, v, kronv, ctx, comm, co, bsrh, session);
    }
    /// No-communicator overload
    template <std::size_t ND, std::size_t NI, typename T>
    void create_kron_bsr(const PartitionItem<NI> *pim, const Coor<NI> &dimi, const PartitionItem<ND> *pdom,
                         const Coor<ND> &dimd, int ncomponents, const Coor<NI> &blockim, const Coor<ND> &blockdom,
                         const Coor<NI> &kronim, const Coor<ND> &krondom, bool blockImFast, IndexType **ii,
                         Coor<ND> **jj, const T **v, const T **kronv, const Context *ctx, CoorOrder co,
                         BSR_handle **bsrh, Session session = 0) {
        detail::create_kron_bsr<ND, NI, T>(pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, kronim, krondom,
                                           blockImFast, ii, jj, v, kronv, ctx, (sbb_comm_t) nullptr, co, bsrh,
                                           session);
    }

    inline void destroy_bsr(BSR_handle *bsrh) { detail::check(sbb_destroy_bsr((sbb_bsr_t)bsrh)); }

    /// y_p = beta y_p + alpha A u_p, u_0 = x, u_p = y_{p-1} (reference: bsr.h:2516), NCCL communicator
    template <std::size_t ND, std::size_t NI, std::size_t NX, std::size_t NY, typename T>
    void bsr_krylov(T alpha, BSR_handle *bsrh, const char *oim, const char *odom, const PartitionItem<NX> *px,
                    int ncomponents, const char *ox, const Coor<NX> &fromx, const Coor<NX> &sizex,
                    const Coor<NX> &dimx, const T **vx, T beta, const PartitionItem<NY> *py, const char *oy,
                    const Coor<NY> &fromy, const Coor<NY> &sizey, const Coor<NY> &dimy, char power_label, T **vy,
                    const Context *ctx, sbb_comm_t comm, CoorOrder co, Request *request = nullptr,
                    Session session = 0) {
        detail::bsr_krylov<ND, NI, NX, NY, T>(alpha, bsrh, oim, odom, px, ncomponents, ox, fromx, sizex, dimx, vx,
                                              beta, py, oy, fromy, sizey, dimy, power_label, vy, ctx, comm, co,
                                              request, session);
    }
    /// No-communicator overload
    template <std::size_t ND, std::size_t NI, std::size_t NX, std::size_t NY, typename T>
    void bsr_krylov(T alpha, BSR_handle *bsrh, const char *oim, const char *odom, const PartitionItem<NX> *px,
                    int ncomponents, const char *ox, const Coor<NX> &fromx, const Coor<NX> &sizex,
                    const Coor<NX> &dimx, const T **vx, T beta, const PartitionItem<NY> *py, const char *oy,
                    const Coor<NY> &fromy, const Coor<NY> &sizey, const Coor<NY> &dimy, char power_label, T **vy,
                    const Context *ctx, CoorOrder co, Request *request = nullptr, Session session = 0) {
        detail::bsr_krylov<ND, NI, NX, NY, T>(alpha, bsrh, oim, odom, px, ncomponents, ox, fromx, sizex, dimx, vx,
                                              beta, py, oy, fromy, sizey, dimy, power_label, vy, ctx,
                                              (sbb_comm_t) nullptr, co, request, session);
    }

#ifdef SUPERBBLAS_USE_MPI
    template <std::size_t ND, std::size_t NI, typename T>
    void create_bsr(const PartitionItem<NI> *pim, const Coor<NI> &dimi, const PartitionItem<ND> *pdom,
                    const Coor<ND> &dimd, int ncomponents, const Coor<NI> &blockim, const Coor<ND> &blockdom,
                    bool blockImFast, IndexType **ii, Coor<ND> **jj, const T **v, const Context *ctx,
                    MPI_Comm mpicomm, CoorOrder co, BSR_handle **bsrh, Session session = 0) {
        detail::create_bsr<ND, NI, T>(pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, blockImFast, ii, jj, v,
                                      ctx, detail::comm_for(mpicomm, detail::first_device(ctx, ncomponents)), co,
                                      bsrh, session);
    }
    template <std::size_t ND, std::size_t NI, typename T>
    void create_kron_bsr(const PartitionItem<NI> *pim, const Coor<NI> &dimi, const PartitionItem<ND> *pdom,
                         const Coor<ND> &dimd, int ncomponents, const Coor<NI> &blockim, const Coor<ND> &blockdom,
                         const Coor<NI> &kronim, const Coor<ND> &krondom, bool blockImFast, IndexType **ii,
                         Coor<ND> **jj, const T **v, const T **kronv, const Context *ctx, MPI_Comm mpicomm,
                         CoorOrder co, BSR_handle **bsrh, Session session = 0) {
        detail::create_kron_bsr<ND, NI, T>(pim, dimi, pdom, dimd, ncomponents, blockim, blockdom, kronim, krondom,
                                           blockImFast, ii, jj, v, kronv, ctx,
                                           detail::comm_for(mpicomm, detail::first_device(ctx, ncomponents)), co,
                                           bsrh, session);
    }
    template <std::size_t ND, std::size_t NI, std::size_t NX, std::size_t NY, typename T>
    void bsr_krylov(T alpha, BSR_handle *bsrh, const char *oim, const char *odom, const PartitionItem<NX> *px,
                    int ncomponents, const char *ox, const Coor<NX> &fromx, const Coor<NX> &sizex,
                    const Coor<NX> &dimx, const T **vx, T beta, const PartitionItem<NY> *py, const char *oy,
                    const Coor<NY> &fromy, const Coor<NY> &sizey, const Coor<NY> &dimy, char power_label, T **vy,
                    const Context *ctx, MPI_Comm mpicomm, CoorOrder co, Request *request = nullptr,
                    Session session = 0) {
        detail::bsr_krylov<ND, NI, NX, NY, T>(alpha, bsrh, oim, odom, px, ncomponents, ox, fromx, sizex, dimx, vx,
                                              beta, py, oy, fromy, sizey, dimy, power_label, vy, ctx,
                                              detail::comm_for(mpicomm, detail::first_device(ctx, ncomponents)), co,
                                              request, session);
    }
#endif

} // namespace superbblas

#endif // SUPERBBLAS_B200_CXX_H
