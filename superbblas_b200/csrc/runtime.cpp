// Host runtime. See runtime.hpp.
#include "runtime.hpp"
#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <map>
#include <mutex>
#include <set>
#include <string>
#include <vector>

namespace sbb {

    // ---------------------------------------------------------------------------------------------
    // Devices, streams, launch counter
    // ---------------------------------------------------------------------------------------------

    static std::atomic<long long> g_launches{0};
    void count_launch() { ++g_launches; }
    long long launch_count(bool reset) {
        long long v = g_launches.load();
        if (reset) g_launches = 0;
        return v;
    }

    namespace {
        bool g_profile = false;
        struct TimedLaunch {
            cudaEvent_t a, b;
        };
        std::map<std::string, std::vector<TimedLaunch>> g_timed;
    }

    void profile_enable(bool on) { g_profile = on; }

    KernelTimer::KernelTimer(const char *name_, cudaStream_t stream_)
        : name(name_), stream(stream_), on(g_profile) {
        if (!on) return;
        TimedLaunch t;
        cuda_check(cudaEventCreate(&t.a), "cudaEventCreate");
        cuda_check(cudaEventCreate(&t.b), "cudaEventCreate");
        cuda_check(cudaEventRecord(t.a, stream), "cudaEventRecord");
        g_timed[name].push_back(t);
    }

    KernelTimer::~KernelTimer() {
        if (!on) return;
        cudaEventRecord(g_timed[name].back().b, stream);
    }

    void profile_read(const char *name, double *total_ms, long long *count) {
        *total_ms = 0, *count = 0;
        auto it = g_timed.find(name);
        if (it == g_timed.end()) return;
        for (auto &t : it->second) {
            cuda_check(cudaEventSynchronize(t.b), "cudaEventSynchronize");
            float ms = 0;
            cuda_check(cudaEventElapsedTime(&ms, t.a, t.b), "cudaEventElapsedTime");
            *total_ms += ms;
            ++*count;
            cudaEventDestroy(t.a);
            cudaEventDestroy(t.b);
        }
        it->second.clear();
    }

    int dtype_bytes(int dt) {
        switch (dt) {
        case SBB_F32: return 4;
        case SBB_F64: return 8;
        case SBB_C64: return 8;
        case SBB_C128: return 16;
        case SBB_I32: return 4;
        default: throw std::runtime_error("unsupported element type");
        }
    }

    namespace {
        constexpr int MAX_DEVICES = 64;
        DeviceState g_dev[MAX_DEVICES];
        bool g_peer[MAX_DEVICES][MAX_DEVICES];
    }

    void use_device(int device) { cuda_check(cudaSetDevice(device), "cudaSetDevice"); }

    DeviceState &device_state(int device) {
        if (device < 0 || device >= MAX_DEVICES) throw std::runtime_error("invalid device id");
        DeviceState &d = g_dev[device];
        if (d.stream == nullptr) {
            int count = 0;
            cuda_check(cudaGetDeviceCount(&count), "cudaGetDeviceCount");
            if (device >= count)
                throw std::runtime_error("superbblas_b200: no such CUDA device (this build has no "
                                         "CPU compute path; a B200 is required)");
            use_device(device);
            d.id = device;
            // The compute stream is a *blocking* stream like the reference's (cudaStreamCreate,
            // platform.h:304-309): it orders itself with the legacy default stream, so inputs produced
            // there (thrust, torch's default stream, QDP-JIT) are seen without an explicit
            // syncLegacyStream.  The communication and auxiliary streams are internal.
            cuda_check(cudaStreamCreate(&d.stream), "stream");
            cuda_check(cudaStreamCreateWithFlags(&d.comm_stream, cudaStreamNonBlocking), "stream");
            cuda_check(cudaStreamCreateWithFlags(&d.aux_stream, cudaStreamNonBlocking), "stream");
            cuda_check(cudaEventCreateWithFlags(&d.ev_c, cudaEventDisableTiming), "event");
            cuda_check(cudaEventCreateWithFlags(&d.ev_a, cudaEventDisableTiming), "event");
        }
        return d;
    }

    void enable_peer(int a, int b) {
        if (a == b || g_peer[a][b]) return;
        int can = 0;
        cuda_check(cudaDeviceCanAccessPeer(&can, a, b), "cudaDeviceCanAccessPeer");
        if (!can) throw std::runtime_error("devices cannot access each other's memory (no NVLink/P2P)");
        use_device(a);
        cudaError_t e = cudaDeviceEnablePeerAccess(b, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled)
            cudaGetLastError();
        else
            cuda_check(e, "cudaDeviceEnablePeerAccess");
        g_peer[a][b] = true;
    }

    // ---------------------------------------------------------------------------------------------
    // Workspace pool
    // ---------------------------------------------------------------------------------------------

    namespace {
        struct Pool {
            std::multimap<size_t, void *> free_blocks;
            std::map<void *, size_t> live;
        };
        Pool g_pool[MAX_DEVICES];
    }

    void *pool_alloc(int device, size_t bytes) {
        if (bytes == 0) bytes = 256;
        bytes = (bytes + 255) / 256 * 256;
        Pool &p = g_pool[device];
        auto it = p.free_blocks.lower_bound(bytes);
        if (it != p.free_blocks.end() && it->first <= bytes * 2) {
            void *ptr = it->second;
            p.live[ptr] = it->first;
            p.free_blocks.erase(it);
            return ptr;
        }
        use_device(device);
        void *ptr = nullptr;
        cudaError_t e = cudaMalloc(&ptr, bytes);
        if (e != cudaSuccess) { // release the cache and retry once (alloc.h:104-168)
            cudaGetLastError();
            for (auto &b : p.free_blocks) cudaFree(b.second);
            p.free_blocks.clear();
            permute_cache_clear(); // the launch tables of the copy kernels are cached device memory too
            use_device(device);
            cuda_check(cudaMalloc(&ptr, bytes), "cudaMalloc (workspace)");
        }
        p.live[ptr] = bytes;
        return ptr;
    }

    void pool_free(int device, void *ptr) {
        if (!ptr) return;
        Pool &p = g_pool[device];
        auto it = p.live.find(ptr);
        if (it == p.live.end()) return;
        p.free_blocks.emplace(it->second, ptr);
        p.live.erase(it);
    }

    PoolStats pool_stats(int device) {
        PoolStats r;
        if (device < 0 || device >= MAX_DEVICES) return r;
        const Pool &p = g_pool[device];
        for (const auto &b : p.live) r.live_bytes += b.second, ++r.live_blocks;
        for (const auto &b : p.free_blocks) r.cached_bytes += b.first, ++r.cached_blocks;
        return r;
    }

    WorkCounters &work_counters() {
        static WorkCounters w;
        return w;
    }

    void pool_clear() {
        for (int d = 0; d < MAX_DEVICES; ++d) {
            Pool &p = g_pool[d];
            if (p.free_blocks.empty()) continue;
            use_device(d);
            cudaStreamSynchronize(g_dev[d].stream);
            for (auto &b : p.free_blocks) cudaFree(b.second);
            p.free_blocks.clear();
        }
    }

    void destroy_all_streams() {
        for (int d = 0; d < MAX_DEVICES; ++d) {
            DeviceState &s = g_dev[d];
            if (!s.stream) continue;
            use_device(d);
            cudaStreamSynchronize(s.stream);
            cudaStreamSynchronize(s.comm_stream);
            cudaStreamSynchronize(s.aux_stream);
            cudaStreamDestroy(s.stream);
            cudaStreamDestroy(s.comm_stream);
            cudaStreamDestroy(s.aux_stream);
            cudaEventDestroy(s.ev_c);
            cudaEventDestroy(s.ev_a);
            s = DeviceState{};
        }
    }

    // ---------------------------------------------------------------------------------------------
    // NCCL, loaded at run time so that the library itself has no link-time dependency on it
    // ---------------------------------------------------------------------------------------------

    namespace {
        struct Id128 { // ncclUniqueId
            char bytes[128];
        };
        struct NcclApi {
            void *handle = nullptr;
            int (*GetUniqueId)(void *) = nullptr;
            int (*CommInitRank)(void **, int, Id128, int) = nullptr;
            int (*CommDestroy)(void *) = nullptr;
            int (*Send)(const void *, size_t, int, int, void *, cudaStream_t) = nullptr;
            int (*Recv)(void *, size_t, int, int, void *, cudaStream_t) = nullptr;
            int (*AllGather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
            int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
            int (*GroupStart)() = nullptr;
            int (*GroupEnd)() = nullptr;
            const char *(*GetErrorString)(int) = nullptr;
        };
    }
    namespace {
        NcclApi &nccl() {
            static NcclApi api;
            if (api.handle) return api;
            const char *names[] = {"libnccl.so.2", "libnccl.so"};
            for (const char *n : names) {
                api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
                if (api.handle) break;
            }
            if (!api.handle)
                throw std::runtime_error("cannot load libnccl.so.2 (needed for multi-GPU copies)");
            auto sym = [&](const char *name) {
                void *p = dlsym(api.handle, name);
                if (!p) throw std::runtime_error(std::string("NCCL symbol missing: ") + name);
                return p;
            };
            api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
            api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
            api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
            api.Send = (decltype(api.Send))sym("ncclSend");
            api.Recv = (decltype(api.Recv))sym("ncclRecv");
            api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
            api.AllReduce = (decltype(api.AllReduce))sym("ncclAllReduce");
            api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
            api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
            api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
            return api;
        }
        void nccl_check(int r, const char *what) {
            if (r != 0)
                throw std::runtime_error(std::string("NCCL error in ") + what + ": " +
                                         nccl().GetErrorString(r));
        }
        constexpr int kNcclChar = 0; // ncclInt8 / ncclChar
        constexpr int kNcclInt32 = 2, kNcclSum = 0, kNcclMin = 3;
    }

    void nccl_unique_id(void *id128) { nccl_check(nccl().GetUniqueId(id128), "ncclGetUniqueId"); }

    namespace {
        /// All ranks agree on min(value) (used to decide collectively whether a step worked)
        int agree_min(Comm *c, int value) {
            DeviceState &d = device_state(c->device);
            use_device(c->device);
            cuda_check(cudaMemcpyAsync(c->flag, &value, sizeof(int), cudaMemcpyHostToDevice, d.comm_stream), "memcpy");
            nccl_check(nccl().AllReduce(c->flag, c->flag, 1, kNcclInt32, kNcclMin, c->nccl, d.comm_stream), "ncclAllReduce");
            int out = 0;
            cuda_check(cudaMemcpyAsync(&out, c->flag, sizeof(int), cudaMemcpyDeviceToHost, d.comm_stream), "memcpy");
            cuda_check(cudaStreamSynchronize(d.comm_stream), "cudaStreamSynchronize");
            return out;
        }

        void release_arena(Comm *c) {
            use_device(c->device);
            if (!c->local)
                for (int r = 0; r < (int)c->peer.size(); ++r)
                    if (r != c->rank && c->peer[r]) cudaIpcCloseMemHandle(c->peer[r]);
            c->peer.clear();
            if (c->arena) cudaFree(c->arena);
            c->arena = nullptr, c->half_bytes = 0;
        }

        /// Loopback group: all arenas grow together (one host thread owns every member)
        void ensure_arena_local(Comm *c, size_t half_bytes) {
            if (half_bytes <= c->half_bytes) return;
            LocalGroup *g = c->local;
            for (Comm *m : g->members) { // nobody may still be using the old arenas
                use_device(m->device);
                cuda_check(cudaDeviceSynchronize(), "cudaDeviceSynchronize");
            }
            half_bytes = (half_bytes + half_bytes / 4 + (1 << 20) - 1) >> 20 << 20;
            std::vector<char *> arenas(g->members.size(), nullptr);
            for (size_t r = 0; r < g->members.size(); ++r) {
                Comm *m = g->members[r];
                release_arena(m);
                use_device(m->device);
                cuda_check(cudaMalloc((void **)&arenas[r], 2 * half_bytes), "cudaMalloc (arena)");
            }
            for (size_t r = 0; r < g->members.size(); ++r) {
                Comm *m = g->members[r];
                m->arena = arenas[r], m->half_bytes = half_bytes, m->peer = arenas;
                for (Comm *o : g->members) enable_peer(m->device, o->device);
            }
        }

        /// Make every rank's arena at least 2 x half_bytes and map it everywhere. Collective.
        void ensure_arena(Comm *c, size_t half_bytes) {
            if (c->local) return ensure_arena_local(c, half_bytes);
            if (half_bytes <= c->half_bytes) return;
            DeviceState &d = device_state(c->device);
            use_device(c->device);
            // nobody may still be using the old arenas
            cuda_check(cudaStreamSynchronize(d.stream), "cudaStreamSynchronize");
            agree_min(c, 1);
            release_arena(c);
            half_bytes = (half_bytes + half_bytes / 4 + (1 << 20) - 1) >> 20 << 20; // grow with slack
            // [half 0 | half 1 | one 64-bit flag per rank]
            const size_t flag_bytes = ((size_t)c->nranks * sizeof(unsigned long long) + 255) / 256 * 256;
            int ok = cudaMalloc((void **)&c->arena, 2 * half_bytes + flag_bytes) == cudaSuccess ? 1 : 0;
            if (!ok) cudaGetLastError(), c->arena = nullptr;
            if (ok) // flags start at zero (sequence numbers only grow); queued before the handles leave
                cuda_check(cudaMemsetAsync(c->arena + 2 * half_bytes, 0, flag_bytes, d.comm_stream), "memset");
            cudaIpcMemHandle_t mine;
            std::memset(&mine, 0, sizeof mine);
            if (ok && cudaIpcGetMemHandle(&mine, c->arena) != cudaSuccess) cudaGetLastError(), ok = 0;
            // exchange the handles with an all-gather (they are 64 opaque bytes each); the scratch was
            // allocated with the communicator, so nothing here can fail on one rank only before the
            // collective (a CUDA error in these copies is sticky and fatal on every later call anyway)
            char *dev = (char *)c->flag + 256;
            cuda_check(cudaMemcpyAsync(dev, &mine, sizeof mine, cudaMemcpyHostToDevice, d.comm_stream), "memcpy");
            nccl_check(nccl().AllGather(dev, dev + sizeof mine, sizeof mine, kNcclChar, c->nccl, d.comm_stream), "ncclAllGather");
            std::vector<cudaIpcMemHandle_t> all(c->nranks);
            cuda_check(cudaMemcpyAsync(all.data(), dev + sizeof mine, sizeof(mine) * c->nranks, cudaMemcpyDeviceToHost, d.comm_stream), "memcpy");
            cuda_check(cudaStreamSynchronize(d.comm_stream), "cudaStreamSynchronize");
            ok = agree_min(c, ok);
            c->peer.assign(c->nranks, nullptr);
            for (int r = 0; ok && r < c->nranks; ++r) {
                if (r == c->rank) {
                    c->peer[r] = c->arena;
                    continue;
                }
                void *p = nullptr;
                if (cudaIpcOpenMemHandle(&p, all[r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                    cudaGetLastError();
                    ok = 0;
                }
                c->peer[r] = (char *)p;
            }
            ok = agree_min(c, ok);
            if (!ok) {
                release_arena(c);
                c->p2p = false; // every rank takes this branch: fall back to ncclSend/ncclRecv
                return;
            }
            c->half_bytes = half_bytes;
            c->flags = (unsigned long long *)(c->arena + 2 * half_bytes);
            std::vector<unsigned long long *> pf(c->nranks);
            for (int r = 0; r < c->nranks; ++r) pf[r] = (unsigned long long *)(c->peer[r] + 2 * half_bytes);
            cuda_check(cudaMemcpyAsync(c->peer_flags, pf.data(), sizeof(void *) * c->nranks,
                                       cudaMemcpyHostToDevice, d.comm_stream), "memcpy");
            cuda_check(cudaStreamSynchronize(d.comm_stream), "cudaStreamSynchronize");
            agree_min(c, 1); // nobody signals before every rank's flags are zeroed and mapped
        }
    }

    Comm *comm_create(const void *id128, int nranks, int rank, int device) {
        if (nranks < 1 || rank < 0 || rank >= nranks) throw std::runtime_error("invalid rank");
        device_state(device);
        use_device(device);
        Comm *c = new Comm;
        c->nranks = nranks, c->rank = rank, c->device = device;
        if (nranks > 1) {
            Id128 id;
            std::memcpy(id.bytes, id128, 128);
            nccl_check(nccl().CommInitRank(&c->nccl, nranks, id, rank), "ncclCommInitRank");
            // [0,256): barrier words and the CTA counter of the fused signal; then the scratch of the
            // IPC handle exchange (64 bytes per rank + mine) and the table of the peers' flag arrays
            const size_t scratch = 256 + sizeof(cudaIpcMemHandle_t) * (nranks + 1);
            cuda_check(cudaMalloc((void **)&c->flag, scratch), "cudaMalloc");
            cuda_check(cudaMemset(c->flag, 0, scratch), "cudaMemset");
            cuda_check(cudaMalloc((void **)&c->peer_flags, sizeof(void *) * nranks), "cudaMalloc");
            cuda_check(cudaHostAlloc((void **)&c->error_host, sizeof(int), cudaHostAllocMapped), "cudaHostAlloc");
            *c->error_host = 0;
            cuda_check(cudaHostGetDevicePointer((void **)&c->error_dev, c->error_host, 0),
                       "cudaHostGetDevicePointer");
            const char *e = std::getenv("SBB_P2P");
            c->p2p = !(e && std::atoi(e) == 0);
            // every rank must take the same decision
            c->p2p = agree_min(c, c->p2p ? 1 : 0) != 0;
        }
        return c;
    }

    std::vector<Comm *> comm_create_local(int nranks, const int *devices) {
        if (nranks < 1) throw std::runtime_error("invalid number of ranks");
        LocalGroup *g = new LocalGroup;
        g->begun.assign(nranks, 0);
        g->round_ev.resize(nranks);
        for (int r = 0; r < nranks; ++r) {
            device_state(devices[r]);
            Comm *c = new Comm;
            c->nranks = nranks, c->rank = r, c->device = devices[r];
            c->local = g, c->p2p = true;
            g->members.push_back(c);
        }
        return g->members;
    }

    void comm_destroy(Comm *c) {
        if (!c) return;
        if (c->pending) {
            try {
                c->pending->wait();
            } catch (...) {
            }
            c->pending = nullptr;
        }
        use_device(c->device);
        for (auto e : c->events) cudaEventDestroy(e);
        c->events.clear();
        if (c->local) {
            LocalGroup *g = c->local;
            cudaDeviceSynchronize();
            release_arena(c);
            for (auto e : g->round_ev[c->rank]) cudaEventDestroy(e);
            g->round_ev[c->rank].clear();
            g->members[c->rank] = nullptr;
            bool last = true;
            for (Comm *m : g->members) last = last && m == nullptr;
            if (last) delete g;
            delete c;
            return;
        }
        if (c->nccl) {
            use_device(c->device);
            cudaStreamSynchronize(device_state(c->device).stream);
            cudaStreamSynchronize(device_state(c->device).comm_stream);
            release_arena(c);
            if (c->flag) cudaFree(c->flag);
            if (c->peer_flags) cudaFree(c->peer_flags);
            if (c->error_host) cudaFreeHost(c->error_host);
            nccl().CommDestroy(c->nccl);
        }
        delete c;
    }

    void comm_check(Comm *c) {
        if (!c || !c->usable()) return;
        if (c->error_host && *(volatile int *)c->error_host != 0) {
            c->poisoned = true;
            throw std::runtime_error("exchange timed out waiting for rank " +
                                     std::to_string(*(volatile int *)c->error_host - 1) +
                                     " (its flag never arrived); the communicator is unusable");
        }
        if (c->poisoned)
            throw std::runtime_error("the communicator is unusable after an earlier error inside an "
                                     "exchange (ranks no longer agree on its state); create a new one");
    }

    namespace {
        unsigned long long wait_timeout_ns() {
            static unsigned long long v = 0;
            if (!v) {
                const char *e = std::getenv("SBB_WAIT_TIMEOUT_S");
                const double s = e ? std::atof(e) : 60.0;
                v = (unsigned long long)((s > 0 ? s : 60.0) * 1e9);
            }
            return v;
        }
    }

    int64_t exchange_chunk_bytes() {
        static int64_t v = -1;
        if (v < 0) {
            const char *e = std::getenv("SBB_CHUNK_MB"), *b = std::getenv("SBB_CHUNK_BYTES");
            v = b ? std::atoll(b) : (e ? std::atoll(e) : 256) * (1ll << 20);
        }
        return v;
    }

    int default_device(Comm *comm) {
        if (comm) return comm->device;
        int dev = 0;
        cudaGetDevice(&dev);
        return dev;
    }

    void order_streams(const std::set<int> &devs) {
        if (devs.size() < 2) return;
        for (int a : devs) {
            DeviceState &da = device_state(a);
            use_device(a);
            cuda_check(cudaEventRecord(da.ev_a, da.stream), "cudaEventRecord");
        }
        for (int a : devs)
            for (int b : devs) {
                if (a == b) continue;
                use_device(a);
                cuda_check(cudaStreamWaitEvent(device_state(a).stream, device_state(b).ev_a, 0),
                           "cudaStreamWaitEvent");
            }
    }

    // ---------------------------------------------------------------------------------------------
    // Copy executor
    // ---------------------------------------------------------------------------------------------

    namespace {
        sbk_box_desc to_desc(const BoxOp &op) {
            sbk_box_desc d;
            std::memset(&d, 0, sizeof d);
            if (op.size.size() > SBK_MAX_DIMS) throw std::runtime_error("too many dimensions");
            d.nd = (int)op.size.size();
            for (int k = 0; k < d.nd; ++k) {
                d.size[k] = op.size[k];
                d.sstride[k] = op.sstride[k];
                d.dstride[k] = op.dstride[k];
            }
            d.rot = op.rot;
            return d;
        }

        struct Resolved {
            char *ptr = nullptr;
            int device = 0;
            void *host = nullptr; ///< the caller's buffer when it is host memory (ptr is then a pool block)
            size_t bytes = 0;
            bool used = false;
        };

        /// CTAs of the pack kernels of a peer-memory exchange (NVLink, not HBM, bounds them) and of
        /// the kernels that run beside them on the auxiliary stream; measured in round 1 on 2 and 4
        /// GPUs (pack 24..296 tried; auxiliary 0 = no limit 3.18 ms, 148 2.69, 222 2.57)
        int pack_grid() {
            static int v = -1;
            if (v < 0) {
                const char *e = std::getenv("SBB_P2P_PACK_GRID");
                v = e ? std::atoi(e) : 74;
            }
            return v;
        }
        int aux_grid_default() {
            static int v = -1;
            if (v < 0) {
                const char *e = std::getenv("SBB_P2P_AUX_GRID");
                v = e ? std::atoi(e) : 222;
            }
            return v;
        }

        /// Event `slot` of `v`, created on `device` (with the ones before it) if missing
        cudaEvent_t event_slot(std::vector<cudaEvent_t> &v, size_t slot, int device) {
            use_device(device);
            while (v.size() <= slot) {
                cudaEvent_t e;
                cuda_check(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "event");
                v.push_back(e);
            }
            return v[slot];
        }
        /// Event i of the communicator's set `which` (0 / 1, alternating per exchange)
        cudaEvent_t comm_event(Comm *c, int which, int i) {
            // sets are interleaved so that growing the vector keeps the earlier assignments
            return event_slot(c->events, (size_t)2 * i + which, c->device);
        }
        cudaEvent_t local_round_event(LocalGroup *g, int rank, int device, size_t slot) {
            return event_slot(g->round_ev[rank], slot, device);
        }
    }

    struct CopyExec::Impl {
        std::shared_ptr<const CopyPlan> plan_ptr;
        CopyArgs args;
        int dtype0, dtype1;
        double alpha[2];
        std::vector<Buffer> v0, v1, mask_a, mask_b, mask_s;
        bool has_mask_a = false, has_mask_b = false, has_mask_s = false;
        Comm *comm;
        Request *owner = nullptr; ///< what comm->pending points to while the exchange is open
        enum State { Created, Begun, Finished, Failed } state = Created;

        // ---- derived in begin() -------------------------------------------------------------------
        int es0 = 0, es1 = 0, wire_dtype = 0, esw = 0, me = 0, home = -1;
        PoolGuard pool;
        std::vector<Resolved> s, d;
        std::set<int> devs;
        std::vector<const float *> mA, mB, mS;
        enum Transport { None, Peer, Nccl } transport = None;
        bool exchange_open = false; ///< between the first and the last step of an exchange on `comm`
        std::vector<size_t> seg_send, seg_recv;
        char *sendbuf = nullptr, *recvbuf = nullptr;
        std::vector<char *> p2p_send_base, p2p_recv_base;
        bool use_aux = false;
        int aux_grid = 0, nrounds = 0, evset = 0;
        unsigned long long seq0 = 0, exchange_id = 0;
        bool local_done = false, nothing_to_do = false;
        std::vector<char> waited; ///< rounds whose wait kernel was already queued by begin() (pacing)
        std::vector<std::vector<int64_t>> rlo, rhi; // NCCL transport: receive windows per (round, peer)

        const CopyPlan &plan() const { return *plan_ptr; }
        DeviceState &hs() { return device_state(home); }
        cudaStream_t stream_for(int dev) {
            return use_aux && dev == home ? hs().aux_stream : device_state(dev).stream;
        }
        int round_of(const BoxOp &op) const {
            const int64_t chunk = std::max<int64_t>(args.chunk_bytes, 1);
            const int64_t off = (op.kind == BoxOp::Pack ? op.doff : op.soff) * esw;
            return args.chunk_bytes > 0 ? (int)(off / chunk) : 0;
        }

        /// Queue one box op; true when `xs` (last pack of a round) rode on its kernel
        bool run(const BoxOp &op, const ExchangeSync *xs = nullptr) {
            PermuteOptions opt;
            if (op.kind == BoxOp::Pack)
                opt.grid_cap = transport == Peer ? pack_grid() : 0;
            else if (use_aux && aux_grid > 0)
                // while an exchange is in flight the kernels on the auxiliary stream (local part,
                // unpack) run on a reduced grid: they are persistent, and at full width they would
                // hold every SM until they end, so that the pack kernels of the next round could not
                // start beside them
                opt.grid_cap = aux_grid;
            const double one[2] = {1, 0}, zero[2] = {0, 0};
            sbk_box_desc desc = to_desc(op);
            {
                // the reference's `memops`: every moved element counts sizeof(T) + sizeof(Q) once,
                // wherever its two ends are (the hop through an arena or a send buffer does not count)
                const int from = op.kind == BoxOp::Local || op.kind == BoxOp::Pack ? es0 : 0;
                const int to = op.kind == BoxOp::Pack ? 0 : es1;
                work_counters().bytes += (double)op.volume() * (double)(from + to);
            }
            switch (op.kind) {
            case BoxOp::Local: {
                const Resolved &a = s[op.src_comp], &b = d[op.dst_comp];
                enable_peer(b.device, a.device);
                use_device(b.device);
                desc.soff = op.soff, desc.doff = op.doff;
                opt.mask_a = mA[op.dst_comp], opt.mask_b = mB[op.dst_comp], opt.mask_src = mS[op.src_comp];
                return permute_copy(desc, a.ptr, dtype0, b.ptr, dtype1, alpha, args.add, b.device,
                                    stream_for(b.device), opt);
            }
            case BoxOp::Pack: {
                const Resolved &a = s[op.src_comp];
                enable_peer(home, a.device);
                use_device(home);
                desc.soff = op.soff, desc.doff = op.doff;
                // scaled (and normally converted) before it leaves; with the peer-memory transport
                // the kernel's stores go straight into the receiver's arena over NVLink
                char *to = transport == Peer ? p2p_send_base[op.peer] : sendbuf + seg_send[op.peer];
                opt.xs = xs;
                return permute_copy(desc, a.ptr, dtype0, to, wire_dtype, alpha, false, home, hs().stream, opt);
            }
            case BoxOp::Unpack: {
                const Resolved &b = d[op.dst_comp];
                enable_peer(b.device, home);
                use_device(b.device);
                desc.soff = op.soff, desc.doff = op.doff;
                const char *from = transport == Peer ? p2p_recv_base[op.peer] : recvbuf + seg_recv[op.peer];
                opt.mask_a = mA[op.dst_comp], opt.mask_b = mB[op.dst_comp];
                return permute_copy(desc, from, wire_dtype, b.ptr, dtype1, one, args.add, b.device,
                                    stream_for(b.device), opt);
            }
            case BoxOp::Zero: {
                const Resolved &b = d[op.dst_comp];
                use_device(b.device);
                desc.doff = op.doff;
                // uncovered destination: only the destination's own mask applies (dist.h:2363-2367)
                opt.mask_b = mB[op.dst_comp];
                return permute_copy(desc, nullptr, dtype1, b.ptr, dtype1, zero, false, b.device,
                                    stream_for(b.device), opt);
            }
            }
            return false;
        }
        void run_local_part() {
            for (const auto &op : plan().ops)
                if (op.kind == BoxOp::Local || op.kind == BoxOp::Zero) run(op);
        }

        void resolve_buffers();
        void begin();
        void begin_peer();
        void begin_nccl();
        void finish();
        void finish_peer();
        void finish_nccl();
        void fail() {
            state = Failed;
            if (exchange_open && comm) {
                comm->poisoned = true;
                if (comm->pending == owner) comm->pending = nullptr;
            }
        }
    };

    void CopyExec::Impl::resolve_buffers() {
        // Which components take part, and how much of every destination is overwritten
        s.assign(v0.size(), Resolved()), d.assign(v1.size(), Resolved());
        std::vector<int64_t> written(v1.size(), 0);
        for (const auto &op : plan().ops) {
            if (op.src_comp >= 0) s[op.src_comp].used = true;
            if (op.dst_comp >= 0) d[op.dst_comp].used = true, written[op.dst_comp] += op.volume();
        }
        // Home device: where host buffers are staged and where messages are packed
        home = -1;
        if (comm) home = comm->device;
        for (size_t c = 0; c < v1.size() && home < 0; ++c)
            if (d[c].used && !v1[c].host) home = v1[c].device;
        for (size_t c = 0; c < v0.size() && home < 0; ++c)
            if (s[c].used && !v0[c].host) home = v0[c].device;
        if (home < 0) home = default_device(comm);
        device_state(home);
        devs.insert(home);
        // A pool block on `device` holding a copy of a host buffer (H2D on the device's stream)
        auto stage = [&](int device, const void *host, size_t bytes) {
            void *p = pool.alloc(device, bytes);
            use_device(device);
            cuda_check(cudaMemcpyAsync(p, host, bytes, cudaMemcpyHostToDevice, device_state(device).stream),
                       "cudaMemcpyAsync H2D");
            return p;
        };
        // Host components are staged on the home device; `copy_in`: their contents are needed
        auto resolve = [&](Resolved &r, const Buffer &b, size_t bytes, bool copy_in) {
            r.bytes = bytes;
            if (b.ptr == nullptr) throw std::runtime_error("null pointer for a non-empty component");
            if (b.host) {
                r.host = b.ptr;
                r.device = home;
                r.ptr = (char *)(copy_in ? stage(home, b.ptr, bytes) : pool.alloc(home, bytes));
            } else {
                r.ptr = (char *)b.ptr, r.device = b.device;
                device_state(r.device);
            }
            devs.insert(r.device);
        };
        for (size_t c = 0; c < v0.size(); ++c)
            if (s[c].used) resolve(s[c], v0[c], (size_t)volume(args.p0[me * args.ncomp0 + c].size) * es0, true);
        const bool masked = has_mask_a || has_mask_b || has_mask_s;
        for (size_t c = 0; c < v1.size(); ++c) {
            if (!d[c].used) continue;
            const int64_t vol = volume(args.p1[me * args.ncomp1 + c].size);
            // keep what the copy does not overwrite (Copy ops never overlap, see plan.cpp)
            resolve(d[c], v1[c], (size_t)vol * es1, args.add || written[c] < vol || masked);
        }
        // Masks (MaskType = float, laid out like the component they belong to): host masks are
        // staged next to the component's data
        auto resolve_mask = [&](const Buffer &b, const Resolved &r, int es) {
            if (!b.ptr) throw std::runtime_error("copy: null mask for a non-empty component");
            if (b.host) return (const float *)stage(r.device, b.ptr, r.bytes / es * sizeof(float));
            devs.insert(b.device);
            return (const float *)b.ptr;
        };
        mA.assign(v1.size(), nullptr), mB.assign(v1.size(), nullptr);
        for (int which = 0; which < 2; ++which) {
            if (!(which ? has_mask_b : has_mask_a)) continue;
            const std::vector<Buffer> &m = which ? mask_b : mask_a;
            if (m.size() != v1.size()) throw std::runtime_error("copy: one mask per component expected");
            for (size_t c = 0; c < v1.size(); ++c) {
                if (!d[c].used) continue;
                (which ? mB : mA)[c] = resolve_mask(m[c], d[c], es1);
                if (!m[c].host) enable_peer(d[c].device, m[c].device);
            }
        }
        // The source's mask in its own layout (purely local copies)
        mS.assign(v0.size(), nullptr);
        if (has_mask_s) {
            if (plan().any_comm) throw std::runtime_error("copy: source-layout masks need a local copy");
            if (mask_s.size() != v0.size()) throw std::runtime_error("copy: one mask per component expected");
            for (size_t c = 0; c < v0.size(); ++c)
                if (s[c].used) mS[c] = resolve_mask(mask_s[c], s[c], es0);
        }
    }

    void CopyExec::Impl::begin() {
        if (state != Created) throw std::runtime_error("copy request: begun twice");
        comm_check(comm);
        const CopyPlan &pl = plan();
        const bool peer_capable = comm && comm->usable() && comm->p2p && pl.any_comm;
        // a rank without work still takes part in the synchronisation of the peer-memory transport
        if (pl.ops.empty() && !peer_capable) {
            nothing_to_do = true;
            state = Begun;
            return;
        }
        es0 = dtype_bytes(dtype0), es1 = dtype_bytes(dtype1);
        // Element type on the wire: the destination type, so that conversions happen once, before
        // sending (as the reference does, dist.h:1450-1451) -- except when adding with a type
        // change, where the scaled source type travels so that the receiver performs exactly the
        // arithmetic of a local `w += alpha*v` (copy_n.h:216-232)
        wire_dtype = (args.add && dtype0 != dtype1) ? dtype0 : dtype1;
        esw = dtype_bytes(wire_dtype);
        me = pl.rank;
        if (pl.needs_comm && (!comm || !comm->usable()))
            throw std::runtime_error("copy needs communication but no communicator was given");
        // one exchange at a time per communicator: complete the previous one first
        if (comm && comm->pending && comm->pending != owner && (peer_capable || pl.needs_comm)) comm->pending->wait();

        resolve_buffers();
        // several devices in one process: order their streams before and after (the reference's
        // causalConnectTo, platform.h:371-409)
        order_streams(devs);

        // Transport: all ranks take the same decision from plan-wide quantities
        if (peer_capable || pl.needs_comm) exchange_open = true;
        if (peer_capable) ensure_arena(comm, (size_t)pl.arena_elems * esw);
        if (peer_capable && comm->p2p) // ensure_arena may have disabled it (collectively)
            transport = Peer;
        else if (pl.needs_comm)
            transport = Nccl;
        if (transport == Nccl && comm->local)
            throw std::runtime_error("loopback communicators only have the peer-memory transport");
        if (transport == None) exchange_open = false;

        if (transport == Peer) begin_peer();
        else if (transport == Nccl) begin_nccl();
        else
            for (const auto &op : pl.ops) run(op);
        state = Begun;
    }

    // ---- peer-memory exchange --------------------------------------------------------------------
    // Pack kernels write into the receivers' arenas; the last CTA of a round's last pack kernel
    // raises this rank's flag at every receiver (processes) or an event is recorded behind it
    // (loopback).  The arena halves alternate, and every exchange ends with the compute stream
    // waiting for every rank's last signal, so a sender can only overwrite a half after its previous
    // readers have finished (DESIGN.md §5).  The exchange is cut in rounds (windows of `chunk` bytes
    // of every segment): round k's unpack kernels (auxiliary stream) overlap the pack kernels of the
    // later rounds (compute stream); the pack kernels run on a reduced grid because NVLink, not
    // HBM, bounds them, which leaves SM resources for the kernels on the auxiliary stream.  Queue
    // order matters (the kernels are persistent): packs of round 0 and their signal first, then the
    // local part on the auxiliary stream.
    void CopyExec::Impl::begin_peer() {
        const CopyPlan &pl = plan();
        const int64_t chunk = std::max<int64_t>(args.chunk_bytes, 1);
        p2p_send_base.assign(pl.nranks, nullptr), p2p_recv_base.assign(pl.nranks, nullptr);
        const size_t half = (comm->epoch & 1) * comm->half_bytes;
        for (int r = 0; r < pl.nranks; ++r) {
            p2p_send_base[r] = comm->peer[r] + half + (size_t)pl.send_seg_off[r] * esw;
            p2p_recv_base[r] = comm->arena + half + (size_t)pl.recv_seg_off[r] * esw;
        }
        exchange_id = comm->epoch;
        evset = (int)(comm->epoch & 1);
        ++comm->epoch;
        // all ranks run the same number of rounds: it comes from the largest message of the exchange
        nrounds = args.chunk_bytes > 0
                      ? (int)std::max<int64_t>(1, (pl.max_pair_elems * esw + chunk - 1) / chunk)
                      : 1;
        // only worth it when there are several rounds of NVLink-bound packs to overlap with
        aux_grid = nrounds > 1 ? aux_grid_default() : 0;
        DeviceState &h = hs();
        use_device(home);
        cuda_check(cudaEventRecord(h.ev_a, h.stream), "cudaEventRecord");
        cuda_check(cudaStreamWaitEvent(h.aux_stream, h.ev_a, 0), "cudaStreamWaitEvent");
        use_aux = true;
        const bool flags = comm->local == nullptr;
        seq0 = comm->seq;
        if (flags) comm->seq += (unsigned long long)nrounds;
        local_done = args.add; // additions keep plan order: everything after the last wait
        // Pacing: nothing aligns the rounds of different senders in time.  A sender with fewer messages
        // than the exchange has phases (a rank that keeps part of its data) would run ahead and meet
        // the other sender of its receiver for half of the exchange (measured: the pack kernels alone
        // of t-slabs -> (z,t) blocks take 6.0 ms on 4 and 8 GPUs where the busiest receiver's ingress
        // allows 4.9).  Such a sender starts round k only when every rank has finished round k - 1
        // (the flags it waits for anyway, one round earlier); balanced senders are not held back.
        int my_peers = 0;
        for (int r = 0; r < pl.nranks; ++r) my_peers += r != me && pl.send_elems[r] > 0;
        const bool pace = flags && nrounds > 1 && my_peers > 0 && my_peers < pl.nphases;
        waited.assign(nrounds, 0);
        for (int k = 0; k < nrounds; ++k) {
            if (pace && k > 0) {
                cuda_check(cudaStreamWaitEvent(h.comm_stream, comm_event(comm, evset, 2 * (k - 1)), 0),
                           "cudaStreamWaitEvent");
                launch_wait(comm->flags, comm->nranks, seq0 + k, h.comm_stream, wait_timeout_ns(), comm->error_dev);
                cuda_check(cudaEventRecord(comm_event(comm, evset, 2 * (k - 1) + 1), h.comm_stream),
                           "cudaEventRecord");
                cuda_check(cudaStreamWaitEvent(h.stream, comm_event(comm, evset, 2 * (k - 1) + 1), 0),
                           "cudaStreamWaitEvent");
                waited[k - 1] = 1;
            }
            // Order of the receivers inside a round: by the phase the planner gave every message (a
            // proper colouring of the sender -> receiver pairs, identical on all ranks).  With the
            // same order on every rank all senders of a redistribution hit the same receivers at the
            // same time (t-slabs -> (z,t) blocks on 8 GPUs: everybody first sends to the z = 0 ranks,
            // two senders per receiver at half the link rate each, while the z = 1 ranks idle:
            // 312 GB/s per direction; rotating the order by the rank left two such collisions: 444).
            std::vector<const BoxOp *> packs;
            {
                std::vector<int> peers;
                for (const auto &op : pl.ops)
                    if (op.kind == BoxOp::Pack && round_of(op) == k &&
                        std::find(peers.begin(), peers.end(), op.peer) == peers.end())
                        peers.push_back(op.peer);
                std::sort(peers.begin(), peers.end(), [&](int x, int y) {
                    const int px = pl.send_phase[x], py = pl.send_phase[y];
                    return px != py ? px < py : x < y;
                });
                for (int peer : peers)
                    for (const auto &op : pl.ops)
                        if (op.kind == BoxOp::Pack && round_of(op) == k && op.peer == peer) packs.push_back(&op);
            }
            const BoxOp *last_pack = packs.empty() ? nullptr : packs.back();
            ExchangeSync xs;
            if (flags) {
                xs.peer_flags = comm->peer_flags, xs.sig_seq = seq0 + k + 1;
                xs.done = (unsigned *)comm->flag + 32, xs.nranks = comm->nranks, xs.me = comm->rank;
            }
            bool signalled = false;
            for (const BoxOp *op : packs) signalled = run(*op, flags && op == last_pack ? &xs : nullptr);
            use_device(home);
            if (flags) {
                // my stores of this round are complete (stream order): tell every rank
                if (!signalled)
                    launch_signal(comm->peer_flags, comm->rank, comm->nranks, seq0 + k + 1, h.stream);
                // the wait kernel of this round may only become resident once my own packs are done:
                // queued without this dependency it would sit on an SM through whatever long kernel
                // precedes the pack on the compute stream (a contraction whose grid is an exact number
                // of waves then needs one wave more)
                cuda_check(cudaEventRecord(comm_event(comm, evset, 2 * k), h.stream),
                           "cudaEventRecord");
            } else {
                cuda_check(cudaEventRecord(local_round_event(comm->local, comm->rank, home,
                                                             (size_t)2 * k + evset),
                                           h.stream),
                           "cudaEventRecord");
            }
            if (!local_done) {
                run_local_part();
                local_done = true;
            }
        }
        if (comm->local) comm->local->begun[comm->rank] = exchange_id + 1;
    }

    void CopyExec::Impl::finish_peer() {
        const CopyPlan &pl = plan();
        DeviceState &h = hs();
        const bool flags = comm->local == nullptr;
        if (!flags) {
            for (int q = 0; q < comm->nranks; ++q)
                if (comm->local->begun[q] < exchange_id + 1)
                    throw std::runtime_error("loopback communicators: every rank must begin a copy "
                                             "(with a Request) before any rank completes it");
        }
        auto wait_round = [&](int k) {
            use_device(home);
            cudaEvent_t arrived = comm_event(comm, evset, 2 * k + 1);
            if (flags && waited[k]) {
                // (already queued by begin(): the sender paced itself on this round)
            } else if (flags) {
                // every rank's stores of round k have landed in my arena once all flags reached the
                // sequence number.  The one-warp wait kernel spins on the communication stream
                cuda_check(cudaStreamWaitEvent(h.comm_stream, comm_event(comm, evset, 2 * k), 0),
                           "cudaStreamWaitEvent");
                launch_wait(comm->flags, comm->nranks, seq0 + k + 1, h.comm_stream, wait_timeout_ns(),
                            comm->error_dev);
            } else {
                for (int q = 0; q < comm->nranks; ++q)
                    cuda_check(cudaStreamWaitEvent(h.comm_stream,
                                                   local_round_event(comm->local, q, comm->local->members[q]->device,
                                                                     (size_t)2 * k + evset),
                                                   0),
                               "cudaStreamWaitEvent");
            }
            if (!(flags && waited[k])) cuda_check(cudaEventRecord(arrived, h.comm_stream), "cudaEventRecord");
            for (int a : devs) {
                use_device(a);
                cuda_check(cudaStreamWaitEvent(stream_for(a), arrived, 0), "cudaStreamWaitEvent");
            }
        };
        if (args.add) {
            for (int k = 0; k < nrounds; ++k) wait_round(k);
            for (const auto &op : pl.ops)
                if (op.kind != BoxOp::Pack) run(op);
        } else {
            for (int k = 0; k < nrounds; ++k) {
                wait_round(k);
                for (const auto &op : pl.ops)
                    if (op.kind == BoxOp::Unpack && round_of(op) == k) run(op);
            }
        }
        // the compute stream continues after everything of this call: every rank has then seen every
        // other rank's last signal of this call, which is what makes the alternation of the arena
        // halves safe (a rank packs call e+1 only after all ranks finished unpacking call e-1)
        use_device(home);
        cuda_check(cudaEventRecord(h.ev_c, h.aux_stream), "cudaEventRecord");
        cuda_check(cudaStreamWaitEvent(h.stream, h.ev_c, 0), "cudaStreamWaitEvent");
        cuda_check(cudaStreamWaitEvent(h.stream, comm_event(comm, evset, 2 * nrounds - 1), 0),
                   "cudaStreamWaitEvent");
        use_aux = false;
    }

    // ---- NCCL transport (SBB_P2P=0, or when the arenas cannot be mapped) ----------------------------
    // Round k: pack (compute stream) -> event -> grouped ncclSend/ncclRecv of that window
    // (communication stream) -> event -> unpack.  All packs are queued first, so the transfer of
    // round k overlaps the packing of rounds > k and the unpacking of rounds < k; the local part of
    // a Copy is queued right after the first pack.
    void CopyExec::Impl::begin_nccl() {
        const CopyPlan &pl = plan();
        DeviceState &h = hs();
        seg_send.assign(pl.nranks + 1, 0), seg_recv.assign(pl.nranks + 1, 0);
        for (int r = 0; r < pl.nranks; ++r) {
            seg_send[r + 1] = seg_send[r] + ((size_t)pl.send_elems[r] * esw + 255) / 256 * 256;
            seg_recv[r + 1] = seg_recv[r] + ((size_t)pl.recv_elems[r] * esw + 255) / 256 * 256;
        }
        if (seg_send[pl.nranks]) sendbuf = (char *)pool.alloc(home, seg_send[pl.nranks]);
        if (seg_recv[pl.nranks]) recvbuf = (char *)pool.alloc(home, seg_recv[pl.nranks]);
        evset = (int)(comm->epoch & 1);
        ++comm->epoch;
        nrounds = 0;
        for (const auto &op : pl.ops)
            if (op.kind == BoxOp::Pack || op.kind == BoxOp::Unpack) nrounds = std::max(nrounds, round_of(op) + 1);
        // byte window of every (round, peer): [lo, hi)
        std::vector<std::vector<int64_t>> slo(nrounds, std::vector<int64_t>(pl.nranks, -1)), shi = slo;
        rlo = slo, rhi = slo;
        for (const auto &op : pl.ops) {
            if (op.kind != BoxOp::Pack && op.kind != BoxOp::Unpack) continue;
            const int k = round_of(op);
            const bool snd = op.kind == BoxOp::Pack;
            const int64_t b0 = (snd ? op.doff : op.soff) * esw, b1 = b0 + op.volume() * esw;
            auto &lo = (snd ? slo : rlo)[k][op.peer];
            auto &hi = (snd ? shi : rhi)[k][op.peer];
            lo = lo < 0 ? b0 : std::min(lo, b0);
            hi = std::max(hi, b1);
        }
        NcclApi &n = nccl();
        local_done = args.add;
        for (int k = 0; k < nrounds; ++k) {
            for (const auto &op : pl.ops)
                if (op.kind == BoxOp::Pack && round_of(op) == k) run(op);
            use_device(home);
            cudaEvent_t packed = comm_event(comm, evset, 2 * k),
                        arrived = comm_event(comm, evset, 2 * k + 1);
            cuda_check(cudaEventRecord(packed, h.stream), "cudaEventRecord");
            cuda_check(cudaStreamWaitEvent(h.comm_stream, packed, 0), "cudaStreamWaitEvent");
            nccl_check(n.GroupStart(), "ncclGroupStart");
            for (int r = 0; r < pl.nranks; ++r) {
                if (slo[k][r] >= 0)
                    nccl_check(n.Send(sendbuf + seg_send[r] + slo[k][r], (size_t)(shi[k][r] - slo[k][r]),
                                      kNcclChar, r, comm->nccl, h.comm_stream),
                               "ncclSend");
                if (rlo[k][r] >= 0)
                    nccl_check(n.Recv(recvbuf + seg_recv[r] + rlo[k][r], (size_t)(rhi[k][r] - rlo[k][r]),
                                      kNcclChar, r, comm->nccl, h.comm_stream),
                               "ncclRecv");
            }
            nccl_check(n.GroupEnd(), "ncclGroupEnd");
            cuda_check(cudaEventRecord(arrived, h.comm_stream), "cudaEventRecord");
            if (!local_done) { // the local part overlaps the transfers
                run_local_part();
                local_done = true;
            }
        }
    }

    void CopyExec::Impl::finish_nccl() {
        const CopyPlan &pl = plan();
        auto wait_round = [&](int k) {
            for (int a : devs) {
                use_device(a);
                cuda_check(cudaStreamWaitEvent(device_state(a).stream,
                                               comm_event(comm, evset, 2 * k + 1), 0),
                           "cudaStreamWaitEvent");
            }
        };
        if (args.add) {
            // additions are applied in plan order (ascending source part) so that the result does not
            // depend on which contributions were remote
            for (int k = 0; k < nrounds; ++k) wait_round(k);
            for (const auto &op : pl.ops)
                if (op.kind != BoxOp::Pack) run(op);
        } else {
            if (!local_done) run_local_part();
            for (int k = 0; k < nrounds; ++k) {
                wait_round(k);
                for (const auto &op : pl.ops)
                    if (op.kind == BoxOp::Unpack && round_of(op) == k) run(op);
            }
        }
    }

    void CopyExec::Impl::finish() {
        if (state == Finished) return;
        if (state != Begun) throw std::runtime_error("copy request: not begun (or failed)");
        if (nothing_to_do) {
            state = Finished;
            return;
        }
        if (transport == Peer) finish_peer();
        else if (transport == Nccl) finish_nccl();
        order_streams(devs);
        // Host destinations are complete when the request is
        bool host_out = false;
        for (size_t c = 0; c < v1.size(); ++c)
            if (d[c].used && d[c].host) {
                use_device(home);
                cuda_check(cudaMemcpyAsync(d[c].host, d[c].ptr, d[c].bytes, cudaMemcpyDeviceToHost, hs().stream),
                           "cudaMemcpyAsync D2H");
                host_out = true;
            }
        if (host_out) {
            use_device(home);
            cuda_check(cudaStreamSynchronize(hs().stream), "cudaStreamSynchronize");
        }
        pool.release();
        if (exchange_open) {
            exchange_open = false;
            if (comm->pending == owner) comm->pending = nullptr;
        }
        state = Finished;
    }

    CopyExec::CopyExec(std::shared_ptr<const CopyPlan> plan, const CopyArgs &args, int dtype0, int dtype1,
                       const double *alpha, std::vector<Buffer> v0, std::vector<Buffer> v1, Comm *comm,
                       const std::vector<Buffer> *mask_a, const std::vector<Buffer> *mask_b,
                       const std::vector<Buffer> *mask_src)
        : impl(new Impl) {
        impl->owner = this;
        impl->plan_ptr = std::move(plan), impl->args = args, impl->dtype0 = dtype0, impl->dtype1 = dtype1;
        impl->alpha[0] = alpha[0], impl->alpha[1] = alpha[1];
        impl->v0 = std::move(v0), impl->v1 = std::move(v1), impl->comm = comm;
        if (mask_a) impl->mask_a = *mask_a, impl->has_mask_a = true;
        if (mask_b) impl->mask_b = *mask_b, impl->has_mask_b = true;
        if (mask_src) impl->mask_s = *mask_src, impl->has_mask_s = true;
    }

    CopyExec::~CopyExec() {
        // a request dropped between begin and finish leaves the ranks out of step
        if (impl->state == Impl::Begun && impl->exchange_open) impl->fail();
        delete impl;
    }

    void CopyExec::begin() {
        try {
            impl->begin();
            if (impl->exchange_open) impl->comm->pending = impl->owner;
        } catch (...) {
            impl->fail();
            throw;
        }
    }

    void CopyExec::finish() {
        try {
            impl->finish();
        } catch (...) {
            impl->fail();
            throw;
        }
    }

    void CopyExec::set_owner(Request *owner) { impl->owner = owner; }

    void CopyExec::wait_local() {
        Impl &m = *impl;
        if (m.state != Impl::Begun || m.nothing_to_do || !m.use_aux) return; // otherwise in stream order
        DeviceState &h = m.hs();
        use_device(m.home);
        cuda_check(cudaEventRecord(h.ev_c, h.aux_stream), "cudaEventRecord");
        cuda_check(cudaStreamWaitEvent(h.stream, h.ev_c, 0), "cudaStreamWaitEvent");
    }

    void CopyExec::adopt(PoolGuard &g) {
        impl->pool.blocks.insert(impl->pool.blocks.end(), g.blocks.begin(), g.blocks.end());
        g.blocks.clear();
    }

    void execute_copy(const CopyPlan &plan, const CopyArgs &args, int dtype0, int dtype1,
                      const double *alpha, const std::vector<Buffer> &v0, const std::vector<Buffer> &v1,
                      Comm *comm, const std::vector<Buffer> *mask_a, const std::vector<Buffer> *mask_b) {
        // (the plan outlives the call: wrap it without taking ownership)
        CopyExec e(std::shared_ptr<const CopyPlan>(std::shared_ptr<const CopyPlan>(), &plan), args, dtype0,
                   dtype1, alpha, v0, v1, comm, mask_a, mask_b);
        e.begin();
        e.finish();
    }

} // namespace sbb
