// extern "C" entry points (include/superbblas_b200.h). Nothing here throws across the boundary.
#include "contract_plan.hpp"
#include "bsr_plan.hpp"
#include "dense_plan.hpp"
#include "runtime.hpp"
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>

using namespace sbb;

static thread_local std::string g_error;

#define SBB_TRY(...)                                                                               \
    try {                                                                                          \
        __VA_ARGS__;                                                                               \
        return 0;                                                                                  \
    } catch (const std::exception &e) {                                                            \
        g_error = e.what();                                                                        \
        return 1;                                                                                  \
    } catch (...) {                                                                                \
        g_error = "unknown error";                                                                 \
        return 1;                                                                                  \
    }

namespace {
    Coor coor(const int *v, int n) { return v ? Coor(v, v + n) : Coor(n, 0); }

    void store_boxes(const std::vector<Box> &b, int nd, int *out) {
        for (size_t i = 0; i < b.size(); ++i) {
            std::memcpy(out + (2 * i) * nd, b[i].from.data(), sizeof(int) * nd);
            std::memcpy(out + (2 * i + 1) * nd, b[i].size.data(), sizeof(int) * nd);
        }
    }

    std::string order_string(const char *o, int nd, const char *name) {
        if ((o == nullptr && nd > 0) || (o != nullptr && (int)std::strlen(o) != nd))
            throw std::runtime_error(
                std::string("The length of the order should match the template argument; argument `") +
                name + "` should have length " + std::to_string(nd));
        return o ? std::string(o) : std::string();
    }

    /// `s` into buf; 2 (with *needed set) when buf is too small
    int put_text(const std::string &s, char *buf, size_t buflen, size_t *needed) {
        if (needed) *needed = s.size() + 1;
        if (s.size() + 1 > buflen) {
            g_error = "buffer too small";
            return 2;
        }
        std::memcpy(buf, s.c_str(), s.size() + 1);
        return 0;
    }

    void check_co(int co) {
        if (co != SBB_SLOW_TO_FAST && co != SBB_FAST_TO_SLOW) throw std::runtime_error("invalid coordinate order");
    }

    /// A tensor argument of a C call; from, size and dim are zeros when not given
    TensorArg read_tensor(int nd, const int *p, int ncomp, const char *o, const char *name, int nranks,
                          const int *from = nullptr, const int *size = nullptr, const int *dim = nullptr) {
        TensorArg t;
        t.nd = nd;
        t.o = order_string(o, nd, name);
        t.ncomp = ncomp;
        t.p = read_partition(p, nranks * ncomp, nd);
        t.from = coor(from, nd), t.size = coor(size, nd), t.dim = coor(dim, nd);
        return t;
    }

    CopyArgs make_copy_args(int nd0, const int *p0, int ncomp0, const char *o0, const int *from0,
                            const int *size0, const int *dim0, int nd1, const int *p1, int ncomp1,
                            const char *o1, const int *from1, const int *dim1, int nranks, int rank,
                            int co, int copyadd) {
        check_co(co);
        if (copyadd != SBB_COPY && copyadd != SBB_ADD) throw std::runtime_error("invalid CopyAdd");
        if (ncomp0 < 0 || ncomp1 < 0) throw std::runtime_error("wtf");
        CopyArgs a;
        a.nd0 = nd0, a.nd1 = nd1;
        a.o0 = order_string(o0, nd0, "o0");
        a.o1 = order_string(o1, nd1, "o1");
        a.ncomp0 = ncomp0, a.ncomp1 = ncomp1;
        a.nranks = nranks, a.rank = rank;
        a.p0 = read_partition(p0, nranks * ncomp0, nd0);
        a.p1 = read_partition(p1, nranks * ncomp1, nd1);
        a.from0 = coor(from0, nd0), a.size0 = coor(size0, nd0), a.dim0 = coor(dim0, nd0);
        a.from1 = coor(from1, nd1), a.dim1 = coor(dim1, nd1);
        a.co = co;
        a.add = copyadd == SBB_ADD;
        return a;
    }

    ContractionArgs make_contraction_args(int dtype, const double *alpha, int nd0, const int *p0,
                                          const int *from0, const int *size0, const int *dim0,
                                          int ncomponents0, const char *o0, int conj0, int nd1,
                                          const int *p1, const int *from1, const int *size1,
                                          const int *dim1, int ncomponents1, const char *o1, int conj1,
                                          const double *beta, int ndo, const int *pr, const int *fromr,
                                          const int *sizer, const int *dimr, int ncomponentsr,
                                          const char *o_r, int nranks, int rank, int co) {
        check_co(co);
        ContractionArgs a;
        a.dtype = dtype;
        a.alpha[0] = alpha[0], a.alpha[1] = alpha[1];
        a.beta[0] = beta[0], a.beta[1] = beta[1];
        a.co = co, a.nranks = nranks, a.rank = rank;
        a.t0 = read_tensor(nd0, p0, ncomponents0, o0, "o0", nranks, from0, size0, dim0);
        a.t1 = read_tensor(nd1, p1, ncomponents1, o1, "o1", nranks, from1, size1, dim1);
        a.tr = read_tensor(ndo, pr, ncomponentsr, o_r, "o_r", nranks, fromr, sizer, dimr);
        a.conj0 = conj0 != 0, a.conj1 = conj1 != 0;
        return a;
    }

    /// Arguments of the dense solvers; x and y are absent (nd 0, no partition) for cholesky and inversion;
    /// eigh takes W in the y arguments
    DenseArgs make_dense_args(int op, int dtype, const double *alpha, int ndc, const int *pc, int ncomponentsc,
                              const char *oc, const char *orows, const char *ocols, int ndx, const int *px,
                              int ncomponentsx, const char *ox, int ndy, const int *py, int ncomponentsy,
                              const char *oy, int nranks, int rank, int co) {
        check_co(co);
        if (ncomponentsc < 0 || ncomponentsx < 0 || ncomponentsy < 0) throw std::runtime_error("wtf");
        DenseArgs a;
        a.op = op, a.dtype = dtype;
        if (alpha) a.alpha[0] = alpha[0], a.alpha[1] = alpha[1];
        a.co = co, a.nranks = nranks, a.rank = rank;
        a.orows = orows ? orows : "", a.ocols = ocols ? ocols : "";
        a.a = read_tensor(ndc, pc, ncomponentsc, oc, "o", nranks);
        if (op == SBB_TRSM || op == SBB_GESM) {
            a.x = read_tensor(ndx, px, ncomponentsx, ox, "ox", nranks);
            a.y = read_tensor(ndy, py, ncomponentsy, oy, "oy", nranks);
        }
        if (op == SBB_EIGH) a.w = read_tensor(ndy, py, ncomponentsy, oy, "ow", nranks);
        return a;
    }

    std::vector<Buffer> buffers(const void *const *v, const sbb_context *ctx, int n) {
        std::vector<Buffer> r(n);
        for (int i = 0; i < n; ++i) {
            r[i].ptr = v ? const_cast<void *>(v[i]) : nullptr;
            if (ctx[i].plat == SBB_CPU)
                r[i].host = true;
            else if (ctx[i].plat == SBB_CUDA)
                r[i].host = false, r[i].device = ctx[i].device;
            else
                throw std::runtime_error("Unsupported platform");
        }
        return r;
    }

    // ---- SB_TRACK_TIME: what the public calls cost (reference: performance.h:357-441) -------------
    struct Timing {
        double cpu_s = 0, gpu_s = 0, flops = 0, bytes = 0;
        long long calls = 0;
    };
    struct Interval { ///< device time of one call, not yet read back
        std::string name;
        int device;
        cudaEvent_t start, stop;
    };
    std::map<std::string, Timing> g_timings;
    std::vector<Interval> g_open;
    std::map<int, std::vector<cudaEvent_t>> g_spare_events;
    int g_track_time = -1;

    bool track_time() {
        if (g_track_time < 0) {
            const char *e = std::getenv("SB_TRACK_TIME");
            g_track_time = e && std::atoi(e) != 0;
        }
        return g_track_time != 0;
    }

    double now_s() {
        return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
    }

    cudaEvent_t timing_event(int device) {
        auto &spare = g_spare_events[device];
        if (!spare.empty()) {
            cudaEvent_t e = spare.back();
            spare.pop_back();
            return e;
        }
        cudaEvent_t e = nullptr;
        if (cudaEventCreate(&e) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        return e;
    }

    /// Read the device times of the finished calls back (waits for them)
    void resolve_intervals() {
        for (Interval &i : g_open) {
            float ms = 0;
            cudaSetDevice(i.device);
            if (cudaEventSynchronize(i.stop) == cudaSuccess &&
                cudaEventElapsedTime(&ms, i.start, i.stop) == cudaSuccess)
                g_timings[i.name].gpu_s += ms * 1e-3;
            else
                cudaGetLastError();
            g_spare_events[i.device].push_back(i.start);
            g_spare_events[i.device].push_back(i.stop);
        }
        g_open.clear();
    }

    /// The device whose library stream brackets a call: the communicator's, else the first GPU
    /// component (destination first, as the executors choose their home device), else the staging
    /// device of an all-host call
    int tracked_device(Comm *c, std::initializer_list<std::pair<const sbb_context *, int>> tensors) {
        if (c) return c->device;
        for (const auto &t : tensors)
            for (int i = 0; t.first && i < t.second; ++i)
                if (t.first[i].plat == SBB_CUDA) return t.first[i].device;
        return default_device(nullptr);
    }

    /// One tracked public call; does nothing when tracking is off or without a name
    struct Tracker {
        const char *name;
        bool on;
        int device = -1;
        cudaStream_t stream = nullptr;
        cudaEvent_t start = nullptr, stop = nullptr;
        double t0 = 0;
        WorkCounters w0;
        template <typename PickDevice> Tracker(const char *name_, PickDevice pick) : name(name_), on(name_ && track_time()) {
            if (!on) return;
            w0 = work_counters();
            try {
                device = pick();
                if (device >= 0) {
                    stream = device_state(device).stream;
                    use_device(device);
                    start = timing_event(device), stop = timing_event(device);
                    if (!start || !stop || cudaEventRecord(start, stream) != cudaSuccess) {
                        cudaGetLastError();
                        start = stop = nullptr;
                    }
                }
            } catch (...) { // no usable device: the call itself will say so; host time is still counted
                start = stop = nullptr;
            }
            t0 = now_s();
        }
        ~Tracker() {
            if (!on) return;
            Timing &t = g_timings[name];
            t.cpu_s += now_s() - t0;
            t.calls += 1;
            t.flops += work_counters().flops - w0.flops;
            t.bytes += work_counters().bytes - w0.bytes;
            if (start && stop) {
                cudaSetDevice(device);
                if (cudaEventRecord(stop, stream) == cudaSuccess)
                    g_open.push_back(Interval{name, device, start, stop});
                else
                    cudaGetLastError();
                if (g_open.size() >= 1024) resolve_intervals(); // bounded: tracking is a diagnostic mode
            }
        }
    };

    /// The body of every public call that makes a request; `make` returns the request begun.  A `_begin`
    /// (named `begun`) hands it out in `*request`, and the plain call (`begun` and `request` null) completes
    /// it here.  The SB_TRACK_TIME report counts the call as `begun` or `name`, on the device `pick`
    /// returns; a call without a `name` is not counted.
    template <typename Pick, typename Make>
    int begin_or_complete(const char *name, const char *begun, sbb_request_t *request, Pick pick, Make make) {
        SBB_TRY({
            if (begun && !request) throw std::runtime_error(std::string(begun) + ": null request");
            if (request) *request = nullptr;
            Tracker tracker(name && begun ? begun : name, pick);
            std::unique_ptr<Request> q = make();
            if (begun) *request = (sbb_request_t)q.release();
            else q->wait();
        });
    }

    std::string timings_report() {
        if (!track_time()) return std::string();
        resolve_intervals();
        std::string s = "Timing of superbblas kernels:\n-----------------------------\n";
        char line[512];
        for (const auto &it : g_timings) { // std::map: alphabetical, like the reference's report
            const Timing &t = it.second;
            const double time = t.gpu_s > 0 ? t.gpu_s : t.cpu_s;
            const double gflops = time > 0 ? t.flops / time / 1e9 : 0;
            const double gbytes = time > 0 ? t.bytes / time / (1024.0 * 1024.0 * 1024.0) : 0;
            const double intensity = t.bytes > 0 ? t.flops / (t.bytes / sizeof(float)) : 0;
            std::snprintf(line, sizeof line,
                          "%s : %.6f s (gpu_time: %.6f calls: %lld flops: %.0f bytes: %.0f GFLOPs_single: %.3e "
                          "GBYTES/s: %.3e intensity: %.1f )\n",
                          it.first.c_str(), t.cpu_s, t.gpu_s, t.calls, t.flops, t.bytes, gflops, gbytes,
                          intensity);
            s += line;
        }
        return s;
    }

    std::string cache_report() {
        std::string s = "Cache usage of superbblas kernels:\n-----------------------------\n";
        char line[256];
        std::snprintf(line, sizeof line, "copy plans : %zu entries\n", plan_cache_size());
        s += line;
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess) cudaGetLastError(), ndev = 0;
        for (int d = 0; d < ndev; ++d) {
            const PoolStats p = pool_stats(d);
            if (p.cached_blocks == 0 && p.live_blocks == 0) continue;
            std::snprintf(line, sizeof line, "workspace pool, device %d : %g GiB cached in %zu blocks, %g GiB in use in %zu blocks\n",
                          d, p.cached_bytes / 1073741824.0, p.cached_blocks, p.live_bytes / 1073741824.0,
                          p.live_blocks);
            s += line;
        }
        return s;
    }

    void live_allocations(long long *blocks, long long *bytes) {
        *blocks = *bytes = 0;
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess) cudaGetLastError(), ndev = 0;
        for (int d = 0; d < ndev; ++d) {
            const PoolStats p = pool_stats(d);
            *blocks += (long long)p.live_blocks, *bytes += (long long)p.live_bytes;
        }
    }

    std::string allocations_report() {
        long long blocks = 0, bytes = 0;
        live_allocations(&blocks, &bytes);
        if (blocks == 0) return std::string();
        std::string s = "Current memory allocation from superbblas:\n-----------------------------\n";
        char line[256];
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess) cudaGetLastError(), ndev = 0;
        for (int d = 0; d < ndev; ++d) {
            const PoolStats p = pool_stats(d);
            if (p.live_blocks == 0) continue;
            std::snprintf(line, sizeof line, "device %d: %zu blocks, %g GiB\n", d, p.live_blocks,
                          p.live_bytes / 1073741824.0);
            s += line;
        }
        return s;
    }
}

extern "C" {

const char *sbb_last_error(void) { return g_error.c_str(); }
const char *sbb_version(void) { return "superbblas_b200 0.2 (sm_100a)"; }
#ifndef SBB_SOURCE_HASH
#define SBB_SOURCE_HASH "unknown"
#endif
const char *sbb_source_hash(void) { return SBB_SOURCE_HASH; }

int sbb_device_count(int *count) {
    SBB_TRY({
        *count = 0;
        cudaError_t e = cudaGetDeviceCount(count);
        if (e != cudaSuccess) {
            cudaGetLastError();
            *count = 0;
        }
    });
}

int sbb_sync(const sbb_context *ctx) {
    SBB_TRY({
        if (ctx->plat == SBB_CUDA) {
            DeviceState &d = device_state(ctx->device);
            use_device(ctx->device);
            cuda_check(cudaStreamSynchronize(d.stream), "cudaStreamSynchronize");
        }
    });
}

int sbb_sync_legacy_stream(const sbb_context *ctx) {
    SBB_TRY({
        if (ctx->plat == SBB_CUDA) {
            DeviceState &d = device_state(ctx->device);
            use_device(ctx->device);
            cuda_check(cudaEventRecord(d.ev_a, cudaStreamLegacy), "cudaEventRecord");
            cuda_check(cudaStreamWaitEvent(d.stream, d.ev_a, 0), "cudaStreamWaitEvent");
        }
    });
}

int sbb_clear_caches(void) {
    SBB_TRY({
        clear_plan_cache();
        permute_cache_clear();
        pool_clear();
    });
}

int sbb_clear_handles(void) { SBB_TRY(destroy_all_streams()); }

int sbb_get_stream(int device, void **stream) { SBB_TRY(*stream = device_state(device).stream); }

int sbb_launch_count(int reset, long long *count) { SBB_TRY(*count = launch_count(reset != 0)); }

int sbb_allocate(const sbb_context *ctx, size_t bytes, void **ptr) {
    SBB_TRY({
        *ptr = nullptr;
        if (ctx->plat == SBB_CPU) {
            // pageable, 64-byte aligned (pinning is the caller's choice: it costs ~1 ms per call)
            if (posix_memalign(ptr, 64, bytes ? bytes : 64) != 0) throw std::runtime_error("out of memory");
        } else if (ctx->plat == SBB_CUDA) {
            device_state(ctx->device);
            *ptr = pool_alloc(ctx->device, bytes);
        } else {
            throw std::runtime_error("Unsupported platform");
        }
    });
}

int sbb_deallocate(const sbb_context *ctx, void *ptr) {
    SBB_TRY({
        if (!ptr) return 0;
        if (ctx->plat == SBB_CPU) {
            std::free(ptr);
        } else {
            pool_free(ctx->device, ptr);
        }
    });
}

int sbb_memcpy(void *dst, const sbb_context *dst_ctx, const void *src, const sbb_context *src_ctx,
               size_t bytes) {
    SBB_TRY({
        if (bytes == 0) return 0;
        const bool dh = dst_ctx->plat == SBB_CPU, sh = src_ctx->plat == SBB_CPU;
        if (dh && sh) {
            std::memcpy(dst, src, bytes);
            return 0;
        }
        const int dev = dh ? src_ctx->device : dst_ctx->device;
        DeviceState &d = device_state(dev);
        use_device(dev);
        cuda_check(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, d.stream), "cudaMemcpyAsync");
        if (dh) cuda_check(cudaStreamSynchronize(d.stream), "cudaStreamSynchronize");
    });
}

int sbb_profile_enable(int on) { SBB_TRY(profile_enable(on != 0)); }

int sbb_profile_read(const char *kernel, double *total_ms, long long *count) {
    SBB_TRY(profile_read(kernel, total_ms, count));
}

int sbb_track_time(int on) { SBB_TRY(g_track_time = on != 0); }

int sbb_reset_timings(void) {
    SBB_TRY({
        resolve_intervals();
        g_timings.clear();
    });
}

int sbb_report(int what, char *buf, size_t buflen, size_t *needed) {
    SBB_TRY({
        const std::string s = what == 0   ? timings_report()
                              : what == 1 ? cache_report()
                              : what == 2 ? allocations_report()
                                          : throw std::runtime_error("sbb_report: unknown report");
        return put_text(s, buf, buflen, needed);
    });
}

int sbb_live_allocations(long long *blocks, long long *bytes) { SBB_TRY(live_allocations(blocks, bytes)); }

int sbb_comm_unique_id(void *id128) { SBB_TRY(nccl_unique_id(id128)); }

int sbb_comm_create(const void *id128, int nranks, int rank, int device, sbb_comm_t *comm) {
    SBB_TRY(*comm = (sbb_comm_t)comm_create(id128, nranks, rank, device));
}

int sbb_comm_create_local(int nranks, const int *devices, sbb_comm_t *comms) {
    SBB_TRY({
        auto v = comm_create_local(nranks, devices);
        for (int r = 0; r < nranks; ++r) comms[r] = (sbb_comm_t)v[r];
    });
}

int sbb_comm_destroy(sbb_comm_t comm) { SBB_TRY(comm_destroy((Comm *)comm)); }

int sbb_comm_rank(sbb_comm_t comm, int *rank, int *nranks) {
    SBB_TRY({
        Comm *c = (Comm *)comm;
        *rank = c ? c->rank : 0;
        *nranks = c ? c->nranks : 1;
    });
}

int sbb_partitioning_distributed_procs(int nd, const char *order, const int *dim,
                                       const char *dist_labels, int nprocs, int *out) {
    SBB_TRY({
        Coor r = partitioning_distributed_procs(order_string(order, nd, "order"), coor(dim, nd),
                                                dist_labels ? dist_labels : "", (unsigned)nprocs);
        std::memcpy(out, r.data(), sizeof(int) * nd);
    });
}

int sbb_basic_partitioning(int nd, const char *order, const int *dim, const int *procs,
                           const char *dist_labels, int nprocs, int ncomponents, int *out) {
    SBB_TRY(store_boxes(
        basic_partitioning(order, coor(dim, nd), coor(procs, nd), dist_labels, nprocs, ncomponents),
        nd, out));
}

int sbb_basic_partitioning_ext(int nd, const int *dim, const int *procs, int nprocs, int replicate,
                               const int *ext_power, int *out) {
    SBB_TRY(store_boxes(basic_partitioning_ext(coor(dim, nd), coor(procs, nd), nprocs,
                                               replicate != 0, coor(ext_power, nd)),
                        nd, out));
}

int sbb_make_hole(int nd, const int *from, const int *size, const int *hole_from,
                  const int *hole_size, const int *dim, int *out, int max_out, int *nout) {
    SBB_TRY({
        auto r = make_hole(coor(from, nd), coor(size, nd), coor(hole_from, nd), coor(hole_size, nd),
                           coor(dim, nd));
        if ((int)r.size() > max_out) throw std::runtime_error("make_hole: output buffer too small");
        *nout = (int)r.size();
        store_boxes(r, nd, out);
    });
}

namespace {
    /// Everything of a copy up to the executor (for masked copies that includes carrying mask0 to
    /// the destination layout, which is a complete copy of its own)
    std::unique_ptr<CopyExec> make_copy(int dtype0, int dtype1, const double *alpha, int nd0, const int *p0,
                                        int ncomponents0, const char *o0, const int *from0,
                                        const int *size0, const int *dim0, const void *const *v0,
                                        const float *const *mask0, const sbb_context *ctx0, int nd1,
                                        const int *p1, int ncomponents1, const char *o1, const int *from1,
                                        const int *dim1, void *const *v1, const float *const *mask1,
                                        const sbb_context *ctx1, Comm *c, int co, int copyadd) {
        // Whether a copy is masked must not depend on the rank (a rank whose components are all
        // empty passes null entries): it is decided by the mask ARRAYS being given.
        const bool has_m0 = mask0 != nullptr, has_m1 = mask1 != nullptr;
        CopyArgs a = make_copy_args(nd0, p0, ncomponents0, o0, from0, size0, dim0, nd1, p1, ncomponents1,
                                    o1, from1, dim1, c ? c->nranks : 1, c ? c->rank : 0, co, copyadd);
        dtype_bytes(dtype0);
        a.alpha_is_zero = scalar_is(dtype0, alpha, 0);
        a.wire_align = 16 / dtype_bytes((a.add && dtype0 != dtype1) ? dtype0 : dtype1);
        a.chunk_bytes = exchange_chunk_bytes();
        auto plan = get_copy_plan(a);
        if (!has_m0 && !has_m1)
            return std::unique_ptr<CopyExec>(new CopyExec(plan, a, dtype0, dtype1, alpha,
                                                          buffers(v0, ctx0, ncomponents0),
                                                          buffers((const void *const *)v1, ctx1, ncomponents1), c));
        // Masked copy (reference: tensor.h:1022-1027, dist.h:944-970, :1240-1243): an element moves
        // iff the source mask at its origin and the destination mask at its target are nonzero.
        // Purely local copies apply both masks in ONE pass: the source's mask is read with the source
        // elements (permute_kernel, ma_src).  When parts of the copy are remote, step 1 carries mask0
        // to the destination layout with the copy engine itself (a float copy with the same
        // geometry, exchange included) and step 2 is the data copy with the two masks as a predicate
        // on every destination store.
        std::vector<Buffer> m0b, m1b, tmp;
        if (has_m1) m1b = buffers((const void *const *)mask1, ctx1, ncomponents1);
        if (has_m0 && !a.alpha_is_zero && !plan->any_comm) {
            m0b = buffers((const void *const *)mask0, ctx0, ncomponents0);
            return std::unique_ptr<CopyExec>(new CopyExec(plan, a, dtype0, dtype1, alpha,
                                                          buffers(v0, ctx0, ncomponents0),
                                                          buffers((const void *const *)v1, ctx1, ncomponents1), c,
                                                          nullptr, has_m1 ? &m1b : nullptr, &m0b));
        }
        PoolGuard blocks;
        if (has_m0 && !a.alpha_is_zero) {
            m0b = buffers((const void *const *)mask0, ctx0, ncomponents0);
            tmp.resize(ncomponents1);
            for (int i = 0; i < ncomponents1; ++i) {
                const int64_t vol = volume(a.p1[(size_t)a.rank * ncomponents1 + i].size);
                const int dev = ctx1[i].plat == SBB_CUDA ? ctx1[i].device : default_device(c);
                tmp[i].host = false, tmp[i].device = dev;
                tmp[i].ptr = blocks.alloc(dev, (size_t)std::max<int64_t>(vol, 1) * sizeof(float));
            }
            CopyArgs am = a;
            am.add = false;
            am.wire_align = 16 / (int)sizeof(float);
            const double one[2] = {1, 0};
            execute_copy(*get_copy_plan(am), am, SBB_F32, SBB_F32, one, m0b, tmp, c);
        }
        std::unique_ptr<CopyExec> e(new CopyExec(plan, a, dtype0, dtype1, alpha, buffers(v0, ctx0, ncomponents0),
                                                 buffers((const void *const *)v1, ctx1, ncomponents1), c,
                                                 tmp.empty() ? nullptr : &tmp, has_m1 ? &m1b : nullptr));
        e->adopt(blocks);
        return e;
    }

    /// sbb_copy, or sbb_copy_begin (`begun`) into `*request`
    int copy_call(const char *begun, sbb_request_t *request, int dtype0, int dtype1, const double *alpha, int nd0,
                  const int *p0, int ncomponents0, const char *o0, const int *from0, const int *size0,
                  const int *dim0, const void *const *v0, const float *const *mask0, const sbb_context *ctx0,
                  int nd1, const int *p1, int ncomponents1, const char *o1, const int *from1, const int *dim1,
                  void *const *v1, const float *const *mask1, const sbb_context *ctx1, sbb_comm_t comm, int co,
                  int copyadd) {
        Comm *c = (Comm *)comm;
        return begin_or_complete(
            "copy", begun, request, [&] { return tracked_device(c, {{ctx1, ncomponents1}, {ctx0, ncomponents0}}); },
            [&]() -> std::unique_ptr<Request> {
                auto e = make_copy(dtype0, dtype1, alpha, nd0, p0, ncomponents0, o0, from0, size0, dim0, v0, mask0,
                                   ctx0, nd1, p1, ncomponents1, o1, from1, dim1, v1, mask1, ctx1, c, co, copyadd);
                e->begin();
                return e;
            });
    }
}

int sbb_copy(int dtype0, int dtype1, const double *alpha, int nd0, const int *p0, int ncomponents0,
             const char *o0, const int *from0, const int *size0, const int *dim0,
             const void *const *v0, const float *const *mask0, const sbb_context *ctx0, int nd1,
             const int *p1, int ncomponents1, const char *o1, const int *from1, const int *dim1,
             void *const *v1, const float *const *mask1, const sbb_context *ctx1, sbb_comm_t comm,
             int co, int copyadd) {
    return copy_call(nullptr, nullptr, dtype0, dtype1, alpha, nd0, p0, ncomponents0, o0, from0, size0, dim0, v0,
                     mask0, ctx0, nd1, p1, ncomponents1, o1, from1, dim1, v1, mask1, ctx1, comm, co, copyadd);
}

int sbb_copy_begin(int dtype0, int dtype1, const double *alpha, int nd0, const int *p0,
                   int ncomponents0, const char *o0, const int *from0, const int *size0,
                   const int *dim0, const void *const *v0, const float *const *mask0,
                   const sbb_context *ctx0, int nd1, const int *p1, int ncomponents1, const char *o1,
                   const int *from1, const int *dim1, void *const *v1, const float *const *mask1,
                   const sbb_context *ctx1, sbb_comm_t comm, int co, int copyadd,
                   sbb_request_t *request) {
    return copy_call("copy_begin", request, dtype0, dtype1, alpha, nd0, p0, ncomponents0, o0, from0, size0, dim0,
                     v0, mask0, ctx0, nd1, p1, ncomponents1, o1, from1, dim1, v1, mask1, ctx1, comm, co, copyadd);
}

int sbb_request_wait(sbb_request_t request) {
    if (!request) return 0;
    std::unique_ptr<Request> e((Request *)request); // released whether or not the completion works
    SBB_TRY({
        Tracker tracker("wait", [] { return -1; }); // host time, bytes of the unpack kernels
        e->wait();
    });
}

int sbb_request_progress(sbb_request_t request, int *done) {
    SBB_TRY({
        *done = 0;
        if (!request) {
            *done = 1;
            return 0;
        }
        Tracker tracker("wait", [] { return -1; });
        Request *e = (Request *)request;
        if (e->progress()) {
            delete e;
            *done = 1;
        }
    });
}

int sbb_copy_plan_describe(int elem_size1, int nd0, const int *p0, int ncomponents0, const char *o0,
                           const int *from0, const int *size0, const int *dim0, int nd1,
                           const int *p1, int ncomponents1, const char *o1, const int *from1,
                           const int *dim1, int nranks, int rank, int co, int copyadd,
                           int alpha_is_zero, char *buf, size_t buflen, size_t *needed) {
    SBB_TRY({
        CopyArgs a = make_copy_args(nd0, p0, ncomponents0, o0, from0, size0, dim0, nd1, p1,
                                    ncomponents1, o1, from1, dim1, nranks, rank, co, copyadd);
        a.alpha_is_zero = alpha_is_zero != 0;
        a.wire_align = elem_size1 > 0 && elem_size1 <= 16 ? 16 / elem_size1 : 1;
        a.chunk_bytes = exchange_chunk_bytes();
        return put_text(make_copy_plan(a)->describe(), buf, buflen, needed);
    });
}

int sbb_contraction(int dtype, const double *alpha, int nd0, const int *p0, const int *from0,
                    const int *size0, const int *dim0, int ncomponents0, const char *o0, int conj0,
                    const void *const *v0, const sbb_context *ctx0, int nd1, const int *p1,
                    const int *from1, const int *size1, const int *dim1, int ncomponents1,
                    const char *o1, int conj1, const void *const *v1, const sbb_context *ctx1,
                    const double *beta, int ndo, const int *pr, const int *fromr, const int *sizer,
                    const int *dimr, int ncomponentsr, const char *o_r, void *const *vr,
                    const sbb_context *ctxr, sbb_comm_t comm, int co) {
    SBB_TRY({
        Comm *c = (Comm *)comm;
        Tracker tracker("contraction", [&] {
            return tracked_device(c, {{ctxr, ncomponentsr}, {ctx0, ncomponents0}, {ctx1, ncomponents1}});
        });
        const ContractionArgs a = make_contraction_args(
            dtype, alpha, nd0, p0, from0, size0, dim0, ncomponents0, o0, conj0, nd1, p1, from1, size1,
            dim1, ncomponents1, o1, conj1, beta, ndo, pr, fromr, sizer, dimr, ncomponentsr, o_r,
            c ? c->nranks : 1, c ? c->rank : 0, co);
        execute_contraction(a, buffers(v0, ctx0, ncomponents0), buffers(v1, ctx1, ncomponents1),
                            buffers((const void *const *)vr, ctxr, ncomponentsr), c);
    });
}

int sbb_contraction_plan_describe(int dtype, const double *alpha, int nd0, const int *p0,
                                  const int *from0, const int *size0, const int *dim0,
                                  int ncomponents0, const char *o0, int conj0, int nd1,
                                  const int *p1, const int *from1, const int *size1, const int *dim1,
                                  int ncomponents1, const char *o1, int conj1, const double *beta,
                                  int ndo, const int *pr, const int *fromr, const int *sizer,
                                  const int *dimr, int ncomponentsr, const char *o_r, int nranks,
                                  int rank, int co, char *buf, size_t buflen, size_t *needed) {
    SBB_TRY({
        const ContractionArgs a = make_contraction_args(
            dtype, alpha, nd0, p0, from0, size0, dim0, ncomponents0, o0, conj0, nd1, p1, from1, size1,
            dim1, ncomponents1, o1, conj1, beta, ndo, pr, fromr, sizer, dimr, ncomponentsr, o_r,
            nranks, rank, co);
        return put_text(make_contraction_plan(a).describe(), buf, buflen, needed);
    });
}

namespace {
    /// A dense call, begun into `*request` (name `begun` in the reports) or completed here without one;
    /// eigh passes W as y
    int dense_call(const char *name, const char *begun, int op, int dtype, const double *alpha, int ndc,
                   const int *pc, int ncomponentsc, const char *oc, const char *orows, const char *ocols,
                   const void *const *vc, const sbb_context *ctxc, int ndx, const int *px, int ncomponentsx,
                   const char *ox, const void *const *vx, const sbb_context *ctxx, int ndy, const int *py,
                   int ncomponentsy, const char *oy, void *const *vy, const sbb_context *ctxy, sbb_comm_t comm,
                   int co, sbb_request_t *request) {
        Comm *c = (Comm *)comm;
        return begin_or_complete(
            name, begun, request,
            [&] { return tracked_device(c, {{ctxy, ncomponentsy}, {ctxc, ncomponentsc}, {ctxx, ncomponentsx}}); },
            [&] {
                const DenseArgs a = make_dense_args(op, dtype, alpha, ndc, pc, ncomponentsc, oc, orows, ocols, ndx,
                                                    px, ncomponentsx, ox, ndy, py, ncomponentsy, oy,
                                                    c ? c->nranks : 1, c ? c->rank : 0, co);
                const std::vector<Buffer> y = buffers((const void *const *)vy, ctxy, ncomponentsy);
                return begin_dense(a, buffers(vc, ctxc, ncomponentsc), buffers(vx, ctxx, ncomponentsx),
                                   op == SBB_EIGH ? std::vector<Buffer>() : y, op == SBB_EIGH ? y : std::vector<Buffer>(),
                                   c);
            });
    }

    int square_call(const char *name, const char *begun, int op, int dtype, int nd, const int *p, int ncomponents,
                    const char *o, void *const *v, const char *orows, const char *ocols, const sbb_context *ctx,
                    sbb_comm_t comm, int co, sbb_request_t *request) {
        return dense_call(name, begun, op, dtype, nullptr, nd, p, ncomponents, o, orows, ocols,
                          (const void *const *)v, ctx, 0, nullptr, 0, nullptr, nullptr, nullptr, 0, nullptr, 0,
                          nullptr, nullptr, nullptr, comm, co, request);
    }
}

int sbb_cholesky(int dtype, int nd, const int *p, int ncomponents, const char *o, void *const *v,
                 const char *orows, const char *ocols, const sbb_context *ctx, sbb_comm_t comm, int co) {
    return square_call("cholesky", nullptr, SBB_CHOLESKY, dtype, nd, p, ncomponents, o, v, orows, ocols, ctx, comm,
                       co, nullptr);
}

int sbb_cholesky_begin(int dtype, int nd, const int *p, int ncomponents, const char *o, void *const *v,
                       const char *orows, const char *ocols, const sbb_context *ctx, sbb_comm_t comm, int co,
                       sbb_request_t *request) {
    return square_call("cholesky", "cholesky_begin", SBB_CHOLESKY, dtype, nd, p, ncomponents, o, v, orows, ocols,
                       ctx, comm, co, request);
}

int sbb_inversion(int dtype, int nd, const int *p, int ncomponents, const char *o, void *const *v,
                  const char *orows, const char *ocols, const sbb_context *ctx, sbb_comm_t comm, int co) {
    return square_call("inversion", nullptr, SBB_INVERSION, dtype, nd, p, ncomponents, o, v, orows, ocols, ctx,
                       comm, co, nullptr);
}

int sbb_inversion_begin(int dtype, int nd, const int *p, int ncomponents, const char *o, void *const *v,
                        const char *orows, const char *ocols, const sbb_context *ctx, sbb_comm_t comm, int co,
                        sbb_request_t *request) {
    return square_call("inversion", "inversion_begin", SBB_INVERSION, dtype, nd, p, ncomponents, o, v, orows,
                       ocols, ctx, comm, co, request);
}

int sbb_trsm(int dtype, const double *alpha, int ndc, const int *pc, int ncomponentsc, const char *oc,
             const char *orows, const char *ocols, const void *const *vc, const sbb_context *ctxc,
             int ndx, const int *px, int ncomponentsx, const char *ox, const void *const *vx,
             const sbb_context *ctxx, int ndy, const int *py, int ncomponentsy, const char *oy,
             void *const *vy, const sbb_context *ctxy, sbb_comm_t comm, int co) {
    return dense_call("trsm", nullptr, SBB_TRSM, dtype, alpha, ndc, pc, ncomponentsc, oc, orows, ocols, vc, ctxc,
                      ndx, px, ncomponentsx, ox, vx, ctxx, ndy, py, ncomponentsy, oy, vy, ctxy, comm, co, nullptr);
}

int sbb_trsm_begin(int dtype, const double *alpha, int ndc, const int *pc, int ncomponentsc, const char *oc,
                   const char *orows, const char *ocols, const void *const *vc, const sbb_context *ctxc,
                   int ndx, const int *px, int ncomponentsx, const char *ox, const void *const *vx,
                   const sbb_context *ctxx, int ndy, const int *py, int ncomponentsy, const char *oy,
                   void *const *vy, const sbb_context *ctxy, sbb_comm_t comm, int co, sbb_request_t *request) {
    return dense_call("trsm", "trsm_begin", SBB_TRSM, dtype, alpha, ndc, pc, ncomponentsc, oc, orows, ocols, vc,
                      ctxc, ndx, px, ncomponentsx, ox, vx, ctxx, ndy, py, ncomponentsy, oy, vy, ctxy, comm, co,
                      request);
}

int sbb_gesm(int dtype, const double *alpha, int ndc, const int *pc, int ncomponentsc, const char *oc,
             const char *orows, const char *ocols, const void *const *vc, const sbb_context *ctxc,
             int ndx, const int *px, int ncomponentsx, const char *ox, const void *const *vx,
             const sbb_context *ctxx, int ndy, const int *py, int ncomponentsy, const char *oy,
             void *const *vy, const sbb_context *ctxy, sbb_comm_t comm, int co) {
    return dense_call("gesm", nullptr, SBB_GESM, dtype, alpha, ndc, pc, ncomponentsc, oc, orows, ocols, vc, ctxc,
                      ndx, px, ncomponentsx, ox, vx, ctxx, ndy, py, ncomponentsy, oy, vy, ctxy, comm, co, nullptr);
}

int sbb_gesm_begin(int dtype, const double *alpha, int ndc, const int *pc, int ncomponentsc, const char *oc,
                   const char *orows, const char *ocols, const void *const *vc, const sbb_context *ctxc,
                   int ndx, const int *px, int ncomponentsx, const char *ox, const void *const *vx,
                   const sbb_context *ctxx, int ndy, const int *py, int ncomponentsy, const char *oy,
                   void *const *vy, const sbb_context *ctxy, sbb_comm_t comm, int co, sbb_request_t *request) {
    return dense_call("gesm", "gesm_begin", SBB_GESM, dtype, alpha, ndc, pc, ncomponentsc, oc, orows, ocols, vc,
                      ctxc, ndx, px, ncomponentsx, ox, vx, ctxx, ndy, py, ncomponentsy, oy, vy, ctxy, comm, co,
                      request);
}

int sbb_eigh(int dtype, int nd, const int *p, int ncomponents, const char *o, void *const *v,
             const char *orows, const char *ocols, const sbb_context *ctx,
             int ndw, const int *pw, int ncomponentsw, const char *ow, void *const *vw,
             const sbb_context *ctxw, sbb_comm_t comm, int co) {
    return dense_call("eigh", nullptr, SBB_EIGH, dtype, nullptr, nd, p, ncomponents, o, orows, ocols,
                      (const void *const *)v, ctx, 0, nullptr, 0, nullptr, nullptr, nullptr, ndw, pw, ncomponentsw, ow,
                      vw, ctxw, comm, co, nullptr);
}

int sbb_dense_plan_describe(int op, int dtype, const double *alpha, int ndc, const int *pc,
                            int ncomponentsc, const char *oc, const char *orows, const char *ocols,
                            int ndx, const int *px, int ncomponentsx, const char *ox, int ndy,
                            const int *py, int ncomponentsy, const char *oy, int nranks, int rank,
                            int co, char *buf, size_t buflen, size_t *needed) {
    SBB_TRY({
        const DenseArgs a = make_dense_args(op, dtype, alpha, ndc, pc, ncomponentsc, oc, orows, ocols, ndx, px,
                                            ncomponentsx, ox, ndy, py, ncomponentsy, oy, nranks, rank, co);
        return put_text(make_dense_plan(a).describe(), buf, buflen, needed);
    });
}

int sbb_dense_steps_describe(int op, int dtype, const double *alpha, int ndc, const int *pc,
                             int ncomponentsc, const char *oc, const char *orows, const char *ocols,
                             int ndx, const int *px, int ncomponentsx, const char *ox, int ndy,
                             const int *py, int ncomponentsy, const char *oy, int nranks, int rank,
                             int co, char *buf, size_t buflen, size_t *needed) {
    SBB_TRY({
        const DenseArgs a = make_dense_args(op, dtype, alpha, ndc, pc, ncomponentsc, oc, orows, ocols, ndx, px,
                                            ncomponentsx, ox, ndy, py, ncomponentsy, oy, nranks, rank, co);
        const DensePlan plan = make_dense_plan(a);
        return put_text(plan.nothing ? std::string() : dense_steps(plan).describe(), buf, buflen, needed);
    });
}

namespace {
    BsrShape make_bsr_shape(int dtype, int ni, const int *pim, const int *dimi, int nd, const int *pdom,
                            const int *dimd, int ncomponents, const int *blockim, const int *blockdom,
                            int blockImFast, int nranks, int rank, int co, const int *kronim, const int *krondom,
                            bool kron) {
        check_co(co);
        if (ni < 0 || nd < 0 || ncomponents < 0) throw std::runtime_error("wtf");
        BsrShape s;
        s.dtype = dtype, s.ni = ni, s.nd = nd, s.ncomp = ncomponents, s.co = co, s.nranks = nranks, s.rank = rank;
        s.dimi = coor(dimi, ni), s.dimd = coor(dimd, nd), s.blockim = coor(blockim, ni), s.blockdom = coor(blockdom, nd);
        s.kron = kron;
        s.kronim = kron ? coor(kronim, ni) : Coor(ni, 1), s.krondom = kron ? coor(krondom, nd) : Coor(nd, 1);
        s.im_fast = blockImFast != 0;
        s.pim = read_partition(pim, nranks * ncomponents, ni);
        s.pdom = read_partition(pdom, nranks * ncomponents, nd);
        return s;
    }

    BsrCall make_bsr_call(int dtype, const double *alpha, const char *oim, const char *odom, int ni, int nd,
                          int ndx, const int *px, int ncomponentsx, const char *ox, const int *fromx,
                          const int *sizex, const int *dimx, const double *beta, int ndy, const int *py,
                          int ncomponentsy, const char *oy, const int *fromy, const int *sizey, const int *dimy,
                          char power_label, int nranks, int rank, int co) {
        check_co(co);
        if (ncomponentsx < 0 || ncomponentsy < 0) throw std::runtime_error("wtf");
        BsrCall c;
        c.dtype = dtype;
        c.alpha[0] = alpha[0], c.alpha[1] = alpha[1], c.beta[0] = beta[0], c.beta[1] = beta[1];
        c.oim = order_string(oim, ni, "oim"), c.odom = order_string(odom, nd, "odom");
        c.power = power_label, c.co = co, c.nranks = nranks, c.rank = rank;
        c.x = read_tensor(ndx, px, ncomponentsx, ox, "ox", nranks, fromx, sizex, dimx);
        c.y = read_tensor(ndy, py, ncomponentsy, oy, "oy", nranks, fromy, sizey, dimy);
        return c;
    }
}

namespace {
    /// create_bsr and create_kron_bsr (`kron`), or their `_begin` (`begun`): the handle at once, completed by
    /// `*request`, or here without one
    int create(const char *begun, sbb_request_t *request, bool kron, int dtype, int ni, const int *pim,
               const int *dimi, int nd, const int *pdom, const int *dimd, int ncomponents, const int *blockim,
               const int *blockdom, const int *kronim, const int *krondom, int blockImFast, const int *const *ii,
               const int *const *jj, const void *const *v, const void *const *kronv, const sbb_context *ctx,
               sbb_comm_t comm, int co, sbb_bsr_t *bsr) {
        std::unique_ptr<BsrOperator> op;
        const int r = begin_or_complete(nullptr, begun, request, [] { return -1; }, [&] {
            *bsr = nullptr;
            Comm *c = (Comm *)comm;
            const BsrShape s = make_bsr_shape(dtype, ni, pim, dimi, nd, pdom, dimd, ncomponents, blockim, blockdom,
                                              blockImFast, c ? c->nranks : 1, c ? c->rank : 0, co, kronim, krondom,
                                              kron);
            std::unique_ptr<Request> q;
            op.reset(create_bsr_begin(s, ii, jj, buffers(v, ctx, ncomponents),
                                      kron ? buffers(kronv, ctx, ncomponents) : std::vector<Buffer>(), c, &q));
            return q;
        });
        if (r == 0) *bsr = (sbb_bsr_t)op.release();
        return r;
    }
}

int sbb_create_bsr(int dtype, int ni, const int *pim, const int *dimi, int nd, const int *pdom, const int *dimd,
                   int ncomponents, const int *blockim, const int *blockdom, int blockImFast,
                   const int *const *ii, const int *const *jj, const void *const *v, const sbb_context *ctx,
                   sbb_comm_t comm, int co, sbb_bsr_t *bsr) {
    return create(nullptr, nullptr, false, dtype, ni, pim, dimi, nd, pdom, dimd, ncomponents, blockim, blockdom,
                  nullptr, nullptr, blockImFast, ii, jj, v, nullptr, ctx, comm, co, bsr);
}

int sbb_create_bsr_begin(int dtype, int ni, const int *pim, const int *dimi, int nd, const int *pdom,
                         const int *dimd, int ncomponents, const int *blockim, const int *blockdom, int blockImFast,
                         const int *const *ii, const int *const *jj, const void *const *v, const sbb_context *ctx,
                         sbb_comm_t comm, int co, sbb_bsr_t *bsr, sbb_request_t *request) {
    return create("create_bsr_begin", request, false, dtype, ni, pim, dimi, nd, pdom, dimd, ncomponents, blockim,
                  blockdom, nullptr, nullptr, blockImFast, ii, jj, v, nullptr, ctx, comm, co, bsr);
}

int sbb_create_kron_bsr(int dtype, int ni, const int *pim, const int *dimi, int nd, const int *pdom,
                        const int *dimd, int ncomponents, const int *blockim, const int *blockdom,
                        const int *kronim, const int *krondom, int blockImFast, const int *const *ii,
                        const int *const *jj, const void *const *v, const void *const *kronv,
                        const sbb_context *ctx, sbb_comm_t comm, int co, sbb_bsr_t *bsr) {
    return create(nullptr, nullptr, true, dtype, ni, pim, dimi, nd, pdom, dimd, ncomponents, blockim, blockdom,
                  kronim, krondom, blockImFast, ii, jj, v, kronv, ctx, comm, co, bsr);
}

int sbb_create_kron_bsr_begin(int dtype, int ni, const int *pim, const int *dimi, int nd, const int *pdom,
                              const int *dimd, int ncomponents, const int *blockim, const int *blockdom,
                              const int *kronim, const int *krondom, int blockImFast, const int *const *ii,
                              const int *const *jj, const void *const *v, const void *const *kronv,
                              const sbb_context *ctx, sbb_comm_t comm, int co, sbb_bsr_t *bsr,
                              sbb_request_t *request) {
    return create("create_kron_bsr_begin", request, true, dtype, ni, pim, dimi, nd, pdom, dimd, ncomponents,
                  blockim, blockdom, kronim, krondom, blockImFast, ii, jj, v, kronv, ctx, comm, co, bsr);
}

int sbb_destroy_bsr(sbb_bsr_t bsr) {
    SBB_TRY({
        if (bsr && ((BsrOperator *)bsr)->requests > 0)
            throw std::runtime_error("destroy_bsr: a request on the operator is still open (wait for it first)");
        delete (BsrOperator *)bsr;
    });
}

namespace {
    /// bsr_krylov, or its `_begin` (`begun`) into `*request`
    int bsr_call(const char *begun, sbb_request_t *request, int dtype, const double *alpha, sbb_bsr_t bsr,
                 const char *oim, const char *odom, int ndx, const int *px, int ncomponentsx, const char *ox,
                 const int *fromx, const int *sizex, const int *dimx, const void *const *vx, const sbb_context *ctxx,
                 const double *beta, int ndy, const int *py, int ncomponentsy, const char *oy, const int *fromy,
                 const int *sizey, const int *dimy, char power_label, void *const *vy, const sbb_context *ctxy,
                 sbb_comm_t comm, int co) {
        Comm *c = (Comm *)comm;
        return begin_or_complete(
            "bsr_krylov", begun, request,
            [&] { return tracked_device(c, {{ctxy, ncomponentsy}, {ctxx, ncomponentsx}}); },
            [&] {
                if (!bsr) throw std::runtime_error("bsr_krylov: null operator");
                const BsrOperator &op = *(const BsrOperator *)bsr;
                const BsrCall call = make_bsr_call(dtype, alpha, oim, odom, op.g.s.ni, op.g.s.nd, ndx, px,
                                                   ncomponentsx, ox, fromx, sizex, dimx, beta, ndy, py, ncomponentsy,
                                                   oy, fromy, sizey, dimy, power_label, c ? c->nranks : 1,
                                                   c ? c->rank : 0, co);
                if (co != op.g.s.co)
                    throw std::runtime_error("bsr_krylov: the coordinate order differs from the operator's");
                return begin_bsr(op, call, buffers(vx, ctxx, ncomponentsx),
                                 buffers((const void *const *)vy, ctxy, ncomponentsy), c);
            });
    }
}

int sbb_bsr_krylov(int dtype, const double *alpha, sbb_bsr_t bsr, const char *oim, const char *odom, int ndx,
                   const int *px, int ncomponentsx, const char *ox, const int *fromx, const int *sizex,
                   const int *dimx, const void *const *vx, const sbb_context *ctxx, const double *beta, int ndy,
                   const int *py, int ncomponentsy, const char *oy, const int *fromy, const int *sizey,
                   const int *dimy, char power_label, void *const *vy, const sbb_context *ctxy, sbb_comm_t comm,
                   int co) {
    return bsr_call(nullptr, nullptr, dtype, alpha, bsr, oim, odom, ndx, px, ncomponentsx, ox, fromx, sizex, dimx, vx,
                    ctxx, beta, ndy, py, ncomponentsy, oy, fromy, sizey, dimy, power_label, vy, ctxy, comm, co);
}

int sbb_bsr_krylov_begin(int dtype, const double *alpha, sbb_bsr_t bsr, const char *oim, const char *odom, int ndx,
                         const int *px, int ncomponentsx, const char *ox, const int *fromx, const int *sizex,
                         const int *dimx, const void *const *vx, const sbb_context *ctxx, const double *beta, int ndy,
                         const int *py, int ncomponentsy, const char *oy, const int *fromy, const int *sizey,
                         const int *dimy, char power_label, void *const *vy, const sbb_context *ctxy,
                         sbb_comm_t comm, int co, sbb_request_t *request) {
    return bsr_call("bsr_krylov_begin", request, dtype, alpha, bsr, oim, odom, ndx, px, ncomponentsx, ox, fromx,
                    sizex, dimx, vx, ctxx, beta, ndy, py, ncomponentsy, oy, fromy, sizey, dimy, power_label, vy, ctxy,
                    comm, co);
}

int sbb_bsr_plan_describe(int dtype, int ni, const int *pim, const int *dimi, int nd, const int *pdom,
                          const int *dimd, int ncomponents, const int *blockim, const int *blockdom,
                          const int *kronim, const int *krondom, int blockImFast, const int *ii_all,
                          const int *jj_all, const double *alpha, const char *oim, const char *odom, int ndx,
                          const int *px, int ncomponentsx, const char *ox, const int *fromx, const int *sizex,
                          const int *dimx, const double *beta, int ndy, const int *py, int ncomponentsy,
                          const char *oy, const int *fromy, const int *sizey, const int *dimy, char power_label,
                          int nranks, int rank, int co, int split, char *buf, size_t buflen, size_t *needed) {
    SBB_TRY({
        const BsrShape s = make_bsr_shape(dtype, ni, pim, dimi, nd, pdom, dimd, ncomponents, blockim, blockdom,
                                          blockImFast, nranks, rank, co, kronim, krondom,
                                          kronim != nullptr || krondom != nullptr);
        const BsrGeometry g = bsr_geometry_from_all(s, ii_all, jj_all);
        const BsrCall call = make_bsr_call(dtype, alpha, oim, odom, ni, nd, ndx, px, ncomponentsx, ox, fromx, sizex,
                                           dimx, beta, ndy, py, ncomponentsy, oy, fromy, sizey, dimy, power_label,
                                           nranks, rank, co);
        const BsrPlan plan = make_bsr_plan(g, call);
        if (!split) return put_text(plan.describe(g), buf, buflen, needed);
        if (plan.nothing) return put_text("", buf, buflen, needed);
        return put_text(describe_bsr_split(plan, make_bsr_split(g, plan, *get_copy_plan(plan.gather_x))), buf, buflen,
                        needed);
    });
}

int sbk_permute_copy(const sbk_box_desc *box, const void *src, int dtype_src, void *dst,
                     int dtype_dst, const double *alpha, int add, int device, void *stream) {
    SBB_TRY({
        DeviceState &d = device_state(device);
        use_device(device);
        permute_copy(*box, src, dtype_src, dst, dtype_dst, alpha, add != 0, device,
                     stream ? (cudaStream_t)stream : d.stream);
    });
}

int sbk_permute_describe(const sbk_box_desc *box, int dtype_src, int dtype_dst, const double *alpha,
                         int add, const void *src, const void *dst, char *buf, size_t buflen) {
    SBB_TRY({
        std::string s;
        permute_copy(*box, src, dtype_src, const_cast<void *>(dst), dtype_dst, alpha, add != 0, 0,
                     nullptr, {}, &s);
        std::snprintf(buf, buflen, "%s", s.c_str());
    });
}

int sbk_contract(const sbk_contract_desc *desc, int dtype, const double *alpha, const void *v0,
                 const void *v1, const double *beta, void *vr, int device, void *stream) {
    SBB_TRY({
        DeviceState &d = device_state(device);
        use_device(device);
        contract(*desc, dtype, alpha, v0, v1, beta, vr, device,
                 stream ? (cudaStream_t)stream : d.stream);
    });
}

int sbk_contract_describe(const sbk_contract_desc *desc, int dtype, char *buf, size_t buflen) {
    SBB_TRY({
        std::string s;
        const double one[2] = {1, 0};
        contract(*desc, dtype, one, nullptr, nullptr, one, nullptr, 0, nullptr, &s);
        std::snprintf(buf, buflen, "%s", s.c_str());
    });
}
}
