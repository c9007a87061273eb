// The call frame of the operator drivers. See driver.hpp.
#include "driver.hpp"

namespace sbb {

    void check_float_dtype(int dtype, const std::string &what) {
        if (dtype != SBB_F32 && dtype != SBB_F64 && dtype != SBB_C64 && dtype != SBB_C128)
            throw std::runtime_error(what + ": unsupported type");
    }

    int home_device(Comm *comm, std::initializer_list<const std::vector<Buffer> *> bufs, int fallback,
                    bool need_ptr) {
        int home = comm ? comm->device : -1;
        for (const auto *bv : bufs)
            for (const auto &b : *bv)
                if (home < 0 && !b.host && (b.ptr || !need_ptr)) home = b.device;
        if (home < 0) home = fallback;
        device_state(home);
        return home;
    }

    Staged stage_in(const std::vector<Buffer> &v, const std::vector<size_t> &bytes, int home, PoolGuard &pool) {
        Staged s;
        s.dev = v;
        s.temps.assign(v.size(), nullptr);
        s.bytes = bytes;
        for (size_t c = 0; c < v.size(); ++c) {
            if (!v[c].host || bytes[c] == 0) continue;
            if (!v[c].ptr) throw std::runtime_error("null pointer for a non-empty component");
            s.temps[c] = pool.alloc(home, bytes[c]);
            s.dev[c].ptr = s.temps[c], s.dev[c].host = false, s.dev[c].device = home;
            use_device(home);
            cuda_check(cudaMemcpyAsync(s.temps[c], v[c].ptr, bytes[c], cudaMemcpyHostToDevice,
                                       device_state(home).stream),
                       "cudaMemcpyAsync H2D");
        }
        return s;
    }

    Staged stage_in(const std::vector<Buffer> &v, const TensorArg &t, int me, int es, int home,
                    PoolGuard &pool) {
        std::vector<size_t> bytes(v.size());
        for (size_t c = 0; c < v.size(); ++c) bytes[c] = (size_t)volume(t.p[me * t.ncomp + c].size) * es;
        return stage_in(v, bytes, home, pool);
    }

    std::set<int> call_devices(int home, std::initializer_list<const Staged *> staged) {
        std::set<int> devs{home};
        for (const Staged *s : staged)
            for (const auto &b : s->dev)
                if (b.ptr) devs.insert(b.device);
        return devs;
    }

    std::vector<Buffer> alloc_slots(int nslots, const std::vector<SlotNeed> &need, int es, int home,
                                    PoolGuard &pool) {
        std::vector<Buffer> slot(nslots, Buffer{nullptr, false, home}); // unused slots: bookkeeping only
        for (const SlotNeed &n : need) slot[n.slot] = Buffer{pool.alloc(n.device, (size_t)n.elems * es), false, n.device};
        return slot;
    }

    void stage_out(const std::vector<Buffer> &v, const Staged &s, int home) {
        bool host_out = false;
        for (size_t c = 0; c < v.size(); ++c)
            if (s.temps[c]) {
                use_device(home);
                cuda_check(cudaMemcpyAsync(v[c].ptr, s.temps[c], s.bytes[c], cudaMemcpyDeviceToHost,
                                           device_state(home).stream),
                           "cudaMemcpyAsync D2H");
                host_out = true;
            }
        if (host_out) cuda_check(cudaStreamSynchronize(device_state(home).stream), "sync");
    }

    CopyArgs copy_args(int nranks, int rank, int co, int es) {
        CopyArgs ca;
        ca.nranks = nranks, ca.rank = rank, ca.co = co;
        ca.wire_align = 16 / es;
        ca.chunk_bytes = exchange_chunk_bytes();
        return ca;
    }

    CopyArgs gather_to_slots_args(const TensorArg &t, int slots, int nranks, int rank, int co, int es) {
        CopyArgs ca = copy_args(nranks, rank, co, es);
        ca.nd0 = ca.nd1 = t.nd;
        ca.o0 = ca.o1 = t.o;
        ca.p0 = t.p, ca.ncomp0 = t.ncomp;
        ca.from0 = t.from, ca.size0 = t.size, ca.dim0 = t.dim;
        ca.from1.assign(t.nd, 0), ca.dim1 = t.size;
        ca.ncomp1 = slots;
        ca.p1.assign((size_t)nranks * slots, Box{Coor(t.nd, 0), Coor(t.nd, 0)});
        return ca;
    }

    bool StepRequest::progress() {
        if (state == Done) return true;
        if (state == Failed) throw std::runtime_error(std::string(name) + ": the request failed");
        try {
            if (exchange) exchange->finish();
            exchange.reset();
            if (!step()) return false;
        } catch (...) {
            state = Failed;
            on_failure();
            throw;
        }
        state = Done;
        return true;
    }

    void StepRequest::begin_exchange(const CopyArgs &ca, int dtype, const std::vector<Buffer> &from,
                                     const std::vector<Buffer> &to, Comm *comm) {
        const double one[2] = {1, 0};
        exchange.reset(new CopyExec(get_copy_plan(ca), ca, dtype, dtype, one, from, to, comm));
        exchange->set_owner(this);
        exchange->begin();
    }

} // namespace sbb
