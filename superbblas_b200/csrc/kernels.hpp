// Internal interface between the host runtime and the CUDA kernels.
#pragma once
#include "../../include/superbblas_b200.h"
#include <cuda_runtime.h>
#include <stdexcept>
#include <string>

struct sbk_dense_desc;
struct sbk_bsr_desc;
struct sbk_kron_desc;

namespace sbb {

    inline void cuda_check(cudaError_t e, const char *what) {
        if (e != cudaSuccess)
            throw std::runtime_error(std::string("CUDA error in ") + what + ": " +
                                     cudaGetErrorString(e));
    }

    /// Count a kernel launch (reported by sbb_launch_count; bench.py's `gpu_launches`)
    void count_launch();

    int dtype_bytes(int dtype);

    /// The scalar `a` ({re, im}) of element type `dtype` is exactly `v`; a real type ignores `im`
    inline bool scalar_is(int dtype, const double *a, double v) {
        return a[0] == v && (a[1] == 0 || dtype == SBB_F32 || dtype == SBB_F64 || dtype == SBB_I32);
    }

    /// Optional device-side timing of the library's own kernels (bench.py's roofline numbers):
    /// when enabled, a pair of CUDA events brackets every launch of the named kernel on the stream
    /// it is launched on.
    struct KernelTimer {
        KernelTimer(const char *name, cudaStream_t stream);
        ~KernelTimer();
        const char *name;
        cudaStream_t stream;
        bool on;
    };
    void profile_enable(bool on);
    /// Synchronise, sum and clear the recorded launches of `name`
    void profile_read(const char *name, double *total_ms, long long *count);

    /// Peer-memory signalling of an exchange round: `launch_signal` (queued behind the pack kernels)
    /// stores `seq` into slot `me` of every rank's flag array; `launch_wait` (queued before the unpack
    /// kernels) spins until all `nranks` slots of this rank's flag array have reached `seq`.
    void launch_signal(unsigned long long *const *peer_flags, int me, int nranks,
                       unsigned long long seq, cudaStream_t stream);
    /// The spin is bounded by `timeout_ns`; on expiry the missing rank + 1 is written to `*error`.
    void launch_wait(const unsigned long long *flags, int nranks, unsigned long long seq,
                     cudaStream_t stream, unsigned long long timeout_ns, int *error);

    /// Exchange signal fused into a pack kernel: the last CTA of the kernel to finish stores `sig_seq`
    /// into slot `me` of every rank's flag array (`done` counts finished CTAs and is left at zero).
    /// (The wait side stays a one-warp kernel of its own: a persistent, SM-filling unpack kernel
    /// that spins could keep this rank's next pack kernel off the SMs while the peer does the same.)
    struct ExchangeSync {
        unsigned long long *const *peer_flags = nullptr;
        unsigned long long sig_seq = 0;
        unsigned *done = nullptr;
        int nranks = 0, me = 0;
    };

    struct PermuteOptions {
        /// mask_a / mask_b (MaskType = float, laid out exactly like dst): an element of dst is written
        /// only where every given mask is nonzero.  mask_src (instead of mask_a): the source's mask,
        /// laid out exactly like src, applied in the same pass.
        const float *mask_a = nullptr, *mask_b = nullptr, *mask_src = nullptr;
        /// Upper bound on the CTAs of the permute kernel (0 = none).  While an exchange is in flight
        /// the runtime leaves SMs free for the kernels that run beside the pack / unpack kernels.
        int grid_cap = 0;
        /// Signal to fuse into the permute kernel; only a box that takes ONE launch carries it
        const ExchangeSync *xs = nullptr;
    };

    /// dst (+)= Q(alpha*src) over a strided box. The current device must be `device`.
    /// If `describe` is given nothing is launched and the chosen variant is described instead.
    /// Returns true when `opt.xs` rode on a launched kernel (the caller then needs no signal kernel).
    bool permute_copy(const sbk_box_desc &box, const void *src, int dtype_src, void *dst,
                      int dtype_dst, const double *alpha, bool add, int device, cudaStream_t stream,
                      const PermuteOptions &opt = {}, std::string *describe = nullptr);

    /// Drop the cached launches of permute_copy (and their device tables)
    void permute_cache_clear();

    /// SMs of a device.  When only a description of a launch is asked for (`describe_only`) and there
    /// is no usable device, the B200's 148 -- the one target of this library -- so that the dispatch
    /// and the K split of the contraction kernels can be examined (and are tested) on any host.
    int sm_count(int device, bool describe_only = false);

    /// vr = alpha * sum_K f0(v0) f1(v1) + beta * vr. The current device must be `device`.
    void contract(const sbk_contract_desc &desc, int dtype, const double *alpha, const void *v0,
                  const void *v1, const double *beta, void *vr, int device, cudaStream_t stream,
                  std::string *describe = nullptr);

    /// Every matrix of the batch factored, inverted or solved with (dense_kernel.hpp). The current
    /// device must be the one of a, x and y.
    void dense(const sbk_dense_desc &desc, int dtype, const double *alpha, void *a, const void *x, void *y,
               cudaStream_t stream, std::string *describe = nullptr);

    /// y = alpha * A x + beta * y for the block rows of one operator component (bsr_kernel.hpp); the
    /// current device must be the one of v, x and y.  y is not read when beta is zero.
    void bsr(const sbk_bsr_desc &desc, int dtype, const double *alpha, const double *beta, const void *v,
             const void *x, void *y, cudaStream_t stream, std::string *describe = nullptr);
    /// The same for a Kronecker operator: kv holds its U factors (bsr_kernel.hpp, kron_row_body)
    void kron_bsr(const sbk_bsr_desc &desc, const sbk_kron_desc &kron, int dtype, const double *alpha,
                  const double *beta, const void *v, const void *kv, const void *x, void *y, cudaStream_t stream,
                  std::string *describe = nullptr);

} // namespace sbb
