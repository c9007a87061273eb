// Host runtime: per-device streams, workspace pool, NCCL communicator, and the executors that turn
// a plan into kernel launches.
//
// Reference counterparts: one persistent stream per device (platform.h:456-467), buffer pool
// (alloc.h:323-391), causalConnectTo (platform.h:371-409), send_receive (dist.h:1426-1573).
#pragma once
#include "kernels.hpp"
#include "plan.hpp"
#include <memory>
#include <set>
#include <vector>

namespace sbb {

    struct DeviceState {
        int id = -1;
        cudaStream_t stream = nullptr;      ///< all kernels of the library for this device
        cudaStream_t comm_stream = nullptr; ///< NCCL traffic, overlapped with `stream`
        cudaStream_t aux_stream = nullptr;  ///< unpack / local kernels that overlap the pack kernels of an exchange
        cudaEvent_t ev_a = nullptr, ev_c = nullptr;
    };

    DeviceState &device_state(int device);
    void use_device(int device);
    void enable_peer(int a, int b);
    void destroy_all_streams();
    /// Make every listed device's stream wait for the work already queued on the others
    void order_streams(const std::set<int> &devs);

    /// Cached device allocations (reused by later calls on the same stream)
    void *pool_alloc(int device, size_t bytes);
    void pool_free(int device, void *p);
    void pool_clear();
    /// Bytes / blocks handed out and not returned, and cached for reuse, on one device
    struct PoolStats {
        size_t live_bytes = 0, live_blocks = 0, cached_bytes = 0, cached_blocks = 0;
    };
    PoolStats pool_stats(int device);

    /// Pool blocks of one call: returned to the pool when the guard ends, normally or by an exception
    struct PoolGuard {
        std::vector<std::pair<int, void *>> blocks;
        PoolGuard() = default;
        PoolGuard(const PoolGuard &) = delete;
        PoolGuard &operator=(const PoolGuard &) = delete;
        void *alloc(int device, size_t bytes) {
            void *p = pool_alloc(device, bytes);
            blocks.emplace_back(device, p);
            return p;
        }
        void release() {
            for (auto &b : blocks) pool_free(b.first, b.second);
            blocks.clear();
        }
        ~PoolGuard() { release(); }
    };

    /// Work queued by the executors so far, in the reference's units (tensor.h:1087-1088, :1593):
    /// bytes = elements moved x (sizeof source + sizeof destination element) per copy kernel,
    /// flops = 8 (complex) or 2 (real) x T.M.N.K per contraction kernel.  Read by the SB_TRACK_TIME
    /// report of the public calls (capi.cpp); plain process-wide counters, like every other state here.
    struct WorkCounters {
        double flops = 0, bytes = 0;
    };
    WorkCounters &work_counters();

    /// A request of the public API (sbb_request_t, the reference's Request): a sequence of exchanges.
    /// Every step completes the exchange in flight, queues what follows up to the next exchange and
    /// begins it.  A copy is one step; bsr_krylov and create_bsr take several.
    class Request {
    public:
        virtual ~Request() = default;
        /// One step; true when nothing is left (the request is complete)
        virtual bool progress() = 0;
        void wait() {
            while (!progress()) {
            }
        }
    };

    class CopyExec;
    struct Comm;

    /// Several ranks living in ONE process ("loopback" communicators, sbb_comm_create_local): the
    /// same exchange as between processes -- pack kernels store into the receiver's arena, unpack
    /// kernels read it -- with plain device pointers instead of IPC mappings and CUDA events instead
    /// of flags in peer memory (a kernel that spins on a flag must never wait for a kernel of the
    /// same process that may not have been launched yet).  This is how the cross-rank path is
    /// exercised on a box with fewer GPUs than ranks; the ranks are driven by one host thread in
    /// phases: every rank begins the copy (Request), then every rank completes it.
    struct LocalGroup {
        std::vector<Comm *> members;
        std::vector<unsigned long long> begun; ///< exchanges begun by every rank
        /// [rank][slot]: recorded on the rank's compute stream behind the pack kernels of a round
        std::vector<std::vector<cudaEvent_t>> round_ev;
    };

    struct Comm {
        void *nccl = nullptr; ///< ncclComm_t (ranks in different processes)
        LocalGroup *local = nullptr; ///< ranks in this process (shared by the members)
        int nranks = 1, rank = 0, device = 0;
        // Peer-memory transport: every rank owns a receive arena (two halves, used alternately) that
        // all other ranks can store into (CUDA IPC mappings between processes); pack kernels write
        // straight into the receiver's arena over NVLink.
        bool p2p = false;          ///< transport usable (decided collectively at creation)
        char *arena = nullptr;     ///< my arena
        size_t half_bytes = 0;     ///< size of one half
        std::vector<char *> peer;  ///< every rank's arena as mapped here (peer[rank] == arena)
        unsigned long long epoch = 0; ///< exchanges begun (selects the arena half)
        int *flag = nullptr;       ///< device scratch: collective yes/no decisions, handle exchange, CTA counter
        // Signalling between processes: every arena ends with one 64-bit slot per rank; a sender
        // raises its slot in every receiver's arena to the sequence number of the round once its
        // pack kernels are done (the last CTA of the last pack kernel does it), receivers spin on
        // their own slots with a one-warp kernel.
        unsigned long long seq = 0;              ///< rounds signalled so far (all ranks agree)
        unsigned long long *flags = nullptr;     ///< my slots (inside my arena allocation)
        unsigned long long **peer_flags = nullptr; ///< device array: every rank's slots as mapped here
        // Failure handling: a wait kernel that gives up (SBB_WAIT_TIMEOUT_S, default 60 s) writes the
        // missing rank + 1 here (pinned host memory mapped into the device); an exception inside an
        // exchange poisons the communicator, because the ranks no longer agree on epoch / seq.
        int *error_host = nullptr, *error_dev = nullptr;
        bool poisoned = false;
        /// The request whose exchange has been begun and not completed (at most one per communicator:
        /// the next exchange completes the whole request first, which keeps the alternation of the
        /// arena halves safe)
        Request *pending = nullptr;
        std::vector<cudaEvent_t> events; ///< per-exchange events (two sets, alternating like the arena halves)
        bool usable() const { return nccl != nullptr || local != nullptr; }
    };

    /// Throws when the communicator is poisoned or one of its wait kernels timed out
    void comm_check(Comm *c);

    void nccl_unique_id(void *id128);
    Comm *comm_create(const void *id128, int nranks, int rank, int device);
    /// `nranks` loopback communicators of one group; rank r works on devices[r]
    std::vector<Comm *> comm_create_local(int nranks, const int *devices);
    void comm_destroy(Comm *c);

    /// A component buffer as given by the caller
    struct Buffer {
        void *ptr = nullptr;
        bool host = false;
        int device = 0;
    };

    /// Masks: `mask_b` is the destination's mask; the source's mask comes either as `mask_a`, already
    /// carried to the destination layout (one per destination component: copies with remote parts),
    /// or as `mask_src`, one per SOURCE component in the source's own layout (purely local copies:
    /// applied in the same pass).
    /// A copy in two steps (the reference's Request, dist.h:54-61): begin() queues everything that
    /// does not depend on other ranks -- staging of host components, the pack kernels with their
    /// signal, the local part -- and finish() the rest: waiting for the other ranks' data, the
    /// unpack kernels, the copy-back of host destinations (with the only host synchronisation).
    class CopyExec : public Request {
    public:
        CopyExec(std::shared_ptr<const CopyPlan> plan, const CopyArgs &args, int dtype0, int dtype1,
                 const double *alpha, std::vector<Buffer> v0, std::vector<Buffer> v1, Comm *comm,
                 const std::vector<Buffer> *mask_a = nullptr, const std::vector<Buffer> *mask_b = nullptr,
                 const std::vector<Buffer> *mask_src = nullptr);
        ~CopyExec();
        CopyExec(const CopyExec &) = delete;
        CopyExec &operator=(const CopyExec &) = delete;
        void begin();
        void finish();
        bool progress() override {
            finish();
            return true;
        }
        /// The request this copy is one step of (default: itself); it is the communicator's pending
        /// request while the copy's exchange is open
        void set_owner(Request *owner);
        /// Make every compute stream the copy writes on wait for the local part queued by begin(), so
        /// that kernels queued next may read the destination points that do not come from other ranks
        void wait_local();
        /// Take over the blocks of `g` (e.g. the carried mask): they live until the copy is complete
        void adopt(PoolGuard &g);
        struct Impl;

    private:
        Impl *impl;
    };

    /// begin() + finish()
    void execute_copy(const CopyPlan &plan, const CopyArgs &args, int dtype0, int dtype1,
                      const double *alpha, const std::vector<Buffer> &v0,
                      const std::vector<Buffer> &v1, Comm *comm,
                      const std::vector<Buffer> *mask_a = nullptr,
                      const std::vector<Buffer> *mask_b = nullptr);

    long long launch_count(bool reset);

    /// Granularity of the pipelined exchange (bytes per peer and round); SBB_CHUNK_MB overrides
    int64_t exchange_chunk_bytes();

    /// Default device for staging host buffers when no GPU component takes part
    int default_device(Comm *comm);

} // namespace sbb
