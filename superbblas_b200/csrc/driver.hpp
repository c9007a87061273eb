// The call frame shared by the operator drivers (contraction, dense solvers, block-sparse): the home
// device of a call, host components staged on it, pool slots for gathered operands, and host results
// copied back; and the step engine of the drivers whose requests take several exchanges.  Each driver
// keeps its own argument checks, items, kernel descriptors and counters.
#pragma once
#include "runtime.hpp"
#include <initializer_list>
#include <set>

namespace sbb {

    struct TensorArg {
        int nd = 0;
        std::string o;
        int ncomp = 1;
        std::vector<Box> p; ///< all parts of all ranks
        Coor from, size, dim;
    };

    /// Caller's components with the host ones replaced by device copies (blocks of a PoolGuard)
    struct Staged {
        std::vector<Buffer> dev; ///< device-resident version of the caller's components
        std::vector<void *> temps;
        std::vector<size_t> bytes;
    };

    /// Throws "<what>: unsupported type" unless `dtype` is F32, F64, C64 or C128
    void check_float_dtype(int dtype, const std::string &what);

    /// The device a call stages host components on: the communicator's, else that of the first device
    /// buffer of `bufs` (in the order given) with a pointer, else `fallback`.  With `need_ptr` false a
    /// device buffer counts without a pointer too.  Creates the device's state.
    int home_device(Comm *comm, std::initializer_list<const std::vector<Buffer> *> bufs, int fallback,
                    bool need_ptr = true);

    /// Host components of `v` with `bytes[c] > 0` copied into blocks of `pool` on `home`, in order
    Staged stage_in(const std::vector<Buffer> &v, const std::vector<size_t> &bytes, int home, PoolGuard &pool);
    /// Host components of this rank (`me`) of tensor `t` copied into blocks of `pool` on `home`
    Staged stage_in(const std::vector<Buffer> &v, const TensorArg &t, int me, int es, int home,
                    PoolGuard &pool);

    /// Every device a call touches, for order_streams
    std::set<int> call_devices(int home, std::initializer_list<const Staged *> staged);

    /// A pool block that slot `slot` needs: `elems` elements on `device`
    struct SlotNeed {
        int slot, device;
        int64_t elems;
    };
    /// One block of `pool` per need; slots without a need stay empty, with `home` as their device
    std::vector<Buffer> alloc_slots(int nslots, const std::vector<SlotNeed> &need, int es, int home,
                                    PoolGuard &pool);

    /// The staged host components of `s` copied back into the caller's `v`, then one synchronisation
    /// of `home`'s stream (none without a host component)
    void stage_out(const std::vector<Buffer> &v, const Staged &s, int home);

    /// CopyArgs with the fields every driver sets alike; the tensors are the caller's to fill
    CopyArgs copy_args(int nranks, int rank, int co, int es);
    /// Copy of the range of `t` into `slots` boxes per rank, each from 0 in the range's own extents;
    /// the boxes (p1) are empty for the caller to fill
    CopyArgs gather_to_slots_args(const TensorArg &t, int slots, int nranks, int rank, int co, int es);

    /// The step engine of a request with several exchanges.  A driver supplies its name and step(): queue
    /// everything up to and including the beginning of the next exchange (begin_exchange), and return true
    /// when nothing is left.  progress() completes the exchange in flight and takes the next step, so one
    /// exchange is in flight at a time, with the request as the communicator's pending one.  An exception
    /// fails the request for good: on_failure() runs, the exception goes on, and every later progress()
    /// throws "<name>: the request failed".
    class StepRequest : public Request {
    public:
        bool progress() final;
        /// Begin the copy `ca` of `from` into `to` (elements of `dtype`) as this request's exchange, the one
        /// in flight until the next progress()
        void begin_exchange(const CopyArgs &ca, int dtype, const std::vector<Buffer> &from,
                            const std::vector<Buffer> &to, Comm *comm);

    protected:
        explicit StepRequest(const char *name) : name(name) {}
        virtual bool step() = 0;
        virtual void on_failure() {}
        /// Make the compute streams wait for the local part of the exchange begun in this step, if any
        /// (CopyExec::wait_local), so that what is queued next may read it
        void wait_local() {
            if (exchange) exchange->wait_local();
        }

    private:
        const char *name;
        std::unique_ptr<CopyExec> exchange; ///< the exchange in flight
        enum { Running, Done, Failed } state = Running;
    };

} // namespace sbb
