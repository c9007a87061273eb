/* superbblas_b200.h — C ABI of the B200-native implementation of superbblas's tensor hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++ or torch types.  The C++ header
 * include/superbblas.h (namespace superbblas, same templates as the reference) and the Python mirror
 * (superbblas_b200/api.py) are thin marshalling layers over these entry points.
 *
 * Every function returns 0 on success and non-zero on error; the message is retrievable with
 * sbb_last_error() (thread local).  Nothing here throws.  There is no CPU compute path: every
 * element is moved or multiplied by a CUDA kernel; SBB_CPU contexts only name where a buffer lives
 * (host memory is staged through the GPU).
 *
 * "Reference" below = eromero-vlc/superbblas, include/superbblas/<file>:<line>.
 */
#ifndef SUPERBBLAS_B200_H
#define SUPERBBLAS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- vocabulary (reference: tensor.h:47-66, platform.h:757-816) ------------------------------ */

/* element types: T,Q of reference templates (platform.h:686-712) */
enum sbb_dtype { SBB_F32 = 0, SBB_F64 = 1, SBB_C64 = 2, SBB_C128 = 3, SBB_I32 = 4 };
/* CoorOrder (tensor.h:56-59) */
enum sbb_coor_order { SBB_SLOW_TO_FAST = 0, SBB_FAST_TO_SLOW = 1 };
/* CopyAdd (tensor.h:62-65) */
enum sbb_copy_add { SBB_COPY = 0, SBB_ADD = 1 };
/* enum platform (platform.h:66-76): CPU, CUDA */
enum sbb_platform { SBB_CPU = 0, SBB_CUDA = 1 };

/* Same layout as the reference's `class Context {enum platform plat; int device;}` (platform.h:757) */
typedef struct sbb_context {
    int plat;   /* SBB_CPU: `v` is host memory; SBB_CUDA: device memory on `device` */
    int device; /* CUDA device ordinal (ignored for SBB_CPU) */
} sbb_context;

/* Communicator: replaces the MPI_Comm argument of the reference's MPI overloads (dist.h:3534,
 * :3628).  NULL means "this process only" (the reference's SelfComm, dist.h:143-149).  A non-NULL
 * communicator is one NCCL rank bound to one GPU; partitions then have nranks*ncomponents items,
 * ordered [rank][component] exactly like the reference (dist.h:3252-3261). */
typedef struct sbb_comm_s *sbb_comm_t;
/* A copy that has been begun and not completed (the reference's Request, dist.h:54-61) */
typedef struct sbb_request_s *sbb_request_t;

/* ---- library ----------------------------------------------------------------------------------- */

const char *sbb_last_error(void);
const char *sbb_version(void);
/** sha1 of the sources this binary was built from (the loader refuses a binary that does not match
 *  the sources next to it) */
const char *sbb_source_hash(void);
/* getGpuDevicesCount (platform.h:824) */
int sbb_device_count(int *count);
/* sync(ctx) (blas.h:965): wait for the library stream of the context's device */
int sbb_sync(const sbb_context *ctx);
/* syncLegacyStream(ctx) (blas.h:979): make the library stream wait for the legacy default stream */
int sbb_sync_legacy_stream(const sbb_context *ctx);
/* clearCaches (alloc.h:440): drop cached plans and pooled workspaces */
int sbb_clear_caches(void);
/* clearHandles (platform.h:833): destroy streams, events and communicators' streams */
int sbb_clear_handles(void);
/* The library's stream for a device (cudaStream_t), for callers that want to order their own work */
int sbb_get_stream(int device, void **stream);
/* Number of CUDA kernels launched by the library since the last call with reset != 0 */
int sbb_launch_count(int reset, long long *count);

/* allocate / deallocate (alloc.h:398-425): memory in the context's space (pooled device memory or
 * 64-byte aligned host memory).  sbb_memcpy copies bytes between two contexts in stream order of the
 * library stream; it returns when host destinations are complete. */
int sbb_allocate(const sbb_context *ctx, size_t bytes, void **ptr);
int sbb_deallocate(const sbb_context *ctx, void *ptr);
int sbb_memcpy(void *dst, const sbb_context *dst_ctx, const void *src, const sbb_context *src_ctx,
               size_t bytes);

/* Device-side timing of the library's own kernels: when enabled every launch of the copy kernel
 * ("permute") and of the tensor-core contraction kernel ("contract_mma") is bracketed by CUDA events
 * on its stream; sbb_profile_read synchronises, returns the summed duration and clears the list. */
int sbb_profile_enable(int on);
int sbb_profile_read(const char *kernel, double *total_ms, long long *count);

/* Reports of the public calls (performance.h:357-518).  With tracking on -- the environment variable
 * SB_TRACK_TIME set to a nonzero number, or sbb_track_time(1) -- sbb_copy, sbb_copy_begin,
 * sbb_request_wait and sbb_contraction accumulate per name: host seconds, device seconds (CUDA events
 * on the library stream around the call, resolved when the report is read), calls, flops and bytes
 * in the reference's units (tensor.h:1087-1088, :1593).  sbb_report writes text into buf:
 *   what = 0  reportTimings: "name : S s (gpu_time: S calls: N flops: F bytes: B GFLOPs_single: ..
 *             GBYTES/s: .. intensity: .. )", one line per name, alphabetically (empty when tracking is off)
 *   what = 1  reportCacheUsage: cached plans, workspace pool per device
 *   what = 2  reportCurrentMemoryAllocations: the pool blocks handed out and not returned
 * It returns 2 and sets *needed when buf is too small.  sbb_live_allocations is what
 * checkForMemoryLeaks (performance.h:494) looks at after clearCaches(). */
int sbb_track_time(int on);
int sbb_reset_timings(void);
int sbb_report(int what, char *buf, size_t buflen, size_t *needed);
int sbb_live_allocations(long long *blocks, long long *bytes);

/* ---- communicator (NCCL over NVLink) ------------------------------------------------------------ */

/* Write a 128-byte NCCL unique id (rank 0 calls it and broadcasts the bytes by any means) */
int sbb_comm_unique_id(void *id128);
int sbb_comm_create(const void *id128, int nranks, int rank, int device, sbb_comm_t *comm);
/* `nranks` "loopback" communicators whose ranks all live in THIS process (rank r works on
 * devices[r]; devices may repeat).  The exchange is the same as between processes -- pack kernels
 * store into the receiver's arena, unpack kernels read it -- with CUDA events for the
 * synchronisation.  One host thread drives the ranks in phases: every rank begins a copy
 * (sbb_copy_begin), then every rank completes it (sbb_request_wait); completing a copy before every
 * rank has begun it is an error.  Masked copies are not supported on loopback communicators.
 * This is how the cross-rank path is tested on a box with fewer GPUs than ranks. */
int sbb_comm_create_local(int nranks, const int *devices, sbb_comm_t *comms);
int sbb_comm_destroy(sbb_comm_t comm);
int sbb_comm_rank(sbb_comm_t comm, int *rank, int *nranks);

/* ---- partitions (host only; reference: dist.h:3318-3509, :3802) ---------------------------------- */

/* partitioning_distributed_procs (dist.h:3318). out: [nd] */
int sbb_partitioning_distributed_procs(int nd, const char *order, const int *dim,
                                       const char *dist_labels, int nprocs, int *out);
/* basic_partitioning(order, dim, procs, dist_labels, nprocs, ncomponents) (dist.h:3393).
 * out: [(nprocs<0 ? prod(procs) : nprocs) * ncomponents][2][nd] */
int sbb_basic_partitioning(int nd, const char *order, const int *dim, const int *procs,
                           const char *dist_labels, int nprocs, int ncomponents, int *out);
/* basic_partitioning(dim, procs, nprocs, replicate, ext_power) (dist.h:3477). out: [nprocs][2][nd] */
int sbb_basic_partitioning_ext(int nd, const int *dim, const int *procs, int nprocs, int replicate,
                               const int *ext_power, int *out);
/* make_hole (dist.h:3802). out: room for max_out boxes [max_out][2][nd]; *nout = boxes written */
int sbb_make_hole(int nd, const int *from, const int *size, const int *hole_from,
                  const int *hole_size, const int *dim, int *out, int max_out, int *nout);

/* ---- copy (reference: superbblas::copy, dist.h:3583 / :3534) ------------------------------------- */

/* v1[from1 + perm(c - from0)] (+)= Q(alpha * v0[c]) for c in [from0, from0+size0) (periodic).
 *   p0, p1 : partitions, int[nparts][2][nd] with nparts = nranks*ncomponents
 *   o0, o1 : label strings of length nd0, nd1
 *   v0, v1 : one pointer per LOCAL component
 *   mask0, mask1 : NULL, or one MaskType (float) array per LOCAL component, laid out exactly like
 *            the component and living in the same context (reference: Mask<XPU>, dist.h:169,
 *            tensor.h:1022-1027).  An element moves iff mask0 is nonzero at its source and mask1
 *            is nonzero at its destination; everything else in v1 is left untouched.  Replicated
 *            source parts must carry consistent masks.  The reference only accepts "compatible"
 *            pairs (mask1 = mask0 carried to the destination); for those the results are
 *            identical.
 *   alpha  : {re, im} (im ignored for real T); the value is converted to T
 * The call is asynchronous with respect to GPU components (use sbb_sync); host (SBB_CPU) destination
 * components are complete on return. */
int sbb_copy(int dtype0, int dtype1, const double *alpha, int nd0, const int *p0, int ncomponents0,
             const char *o0, const int *from0, const int *size0, const int *dim0,
             const void *const *v0, const float *const *mask0, const sbb_context *ctx0, int nd1,
             const int *p1, int ncomponents1, const char *o1, const int *from1, const int *dim1,
             void *const *v1, const float *const *mask1, const sbb_context *ctx1, sbb_comm_t comm,
             int co, int copyadd);

/* The same copy in two steps (reference: the `Request *request` argument of copy, dist.h:3534-3558,
 * and wait(request), dist.h:61).  sbb_copy_begin queues everything that does not depend on other
 * ranks (staging of host components, pack kernels and their signal, the local part) and returns;
 * sbb_request_wait queues the rest (wait for the other ranks' data, unpack kernels), copies host
 * destinations back and returns when those are complete.  The request is released by the wait
 * whatever its outcome.  Sources must not be modified and destinations not be read in between.  A
 * communicator carries one outstanding copy at a time: beginning another one completes it first. */
int sbb_copy_begin(int dtype0, int dtype1, const double *alpha, int nd0, const int *p0,
                   int ncomponents0, const char *o0, const int *from0, const int *size0,
                   const int *dim0, const void *const *v0, const float *const *mask0,
                   const sbb_context *ctx0, int nd1, const int *p1, int ncomponents1, const char *o1,
                   const int *from1, const int *dim1, void *const *v1, const float *const *mask1,
                   const sbb_context *ctx1, sbb_comm_t comm, int co, int copyadd,
                   sbb_request_t *request);
int sbb_request_wait(sbb_request_t request);

/* Describe, without touching any data, the operations sbb_copy would run on `rank` of `nranks`:
 * writes a text description (one op per line) into buf.  Host only; used by the CPU-side tests to
 * check the planner against the oracle.  Returns 2 if buf is too small (*needed is set). */
int sbb_copy_plan_describe(int elem_size1, int nd0, const int *p0, int ncomponents0, const char *o0,
                           const int *from0, const int *size0, const int *dim0, int nd1,
                           const int *p1, int ncomponents1, const char *o1, const int *from1,
                           const int *dim1, int nranks, int rank, int co, int copyadd,
                           int alpha_is_zero, char *buf, size_t buflen, size_t *needed);

/* ---- contraction (reference: superbblas::contraction, dist.h:3701 / :3628) ----------------------- */

/* vr[fromr..] = alpha * sum_A f0(v0[from0..]) * f1(v1[from1..]) + beta * vr[fromr..]
 * Labels in o0,o1,o_r: T = in all three (batch), A = o0 and o1 only (contracted), B = o0 and o_r,
 * C = o1 and o_r; anything else is an error (tensor.h:1349-1354). dtype: F32, F64, C64 or C128. */
int sbb_contraction(int dtype, const double *alpha, int nd0, const int *p0, const int *from0,
                    const int *size0, const int *dim0, int ncomponents0, const char *o0, int conj0,
                    const void *const *v0, const sbb_context *ctx0, int nd1, const int *p1,
                    const int *from1, const int *size1, const int *dim1, int ncomponents1,
                    const char *o1, int conj1, const void *const *v1, const sbb_context *ctx1,
                    const double *beta, int ndo, const int *pr, const int *fromr, const int *sizer,
                    const int *dimr, int ncomponentsr, const char *o_r, void *const *vr,
                    const sbb_context *ctxr, sbb_comm_t comm, int co);

/* Describe, without touching any data, what sbb_contraction would do on `rank` of `nranks` (the
 * arguments of sbb_contraction without buffers, contexts and communicator): the decisions, one line
 * per kernel launch with its T/M/N/K dimensions, the boxes scaled by beta, and the sbb_copy_plan_describe
 * text of the re-partition of the other operand and of the reduction of the partial results.  Host
 * only; throws the argument errors sbb_contraction throws.  Returns 2 if buf is too small (*needed is
 * set). */
int sbb_contraction_plan_describe(int dtype, const double *alpha, int nd0, const int *p0,
                                  const int *from0, const int *size0, const int *dim0,
                                  int ncomponents0, const char *o0, int conj0, int nd1,
                                  const int *p1, const int *from1, const int *size1, const int *dim1,
                                  int ncomponents1, const char *o1, int conj1, const double *beta,
                                  int ndo, const int *pr, const int *fromr, const int *sizer,
                                  const int *dimr, int ncomponentsr, const char *o_r, int nranks,
                                  int rank, int co, char *buf, size_t buflen, size_t *needed);

/* ---- kernel level (what the planner launches; exposed for tests and micro-benchmarks) ------------ */

#define SBK_MAX_DIMS 16

/* A strided box: element e=(i_0..i_{nd-1}), 0<=i_k<size[k], lives at src[soff + sum i_k*sstride[k]]
 * and goes to dst[doff + sum i_k*dstride[k]] (strides and offsets in elements of T resp. Q). */
typedef struct sbk_box_desc {
    int nd;
    int size[SBK_MAX_DIMS];
    int64_t sstride[SBK_MAX_DIMS];
    int64_t dstride[SBK_MAX_DIMS];
    int64_t soff, doff;
    /* Periodic rotation of dimension 0: element i_0 goes to destination index (i_0 + rot) mod
     * size[0] (0 = none).  Requires sstride[0] == dstride[0] == 1.  This is how a +-1 shift along
     * the fastest label is done in one pass over whole rows instead of two boxes. */
    int rot;
} sbk_box_desc;

/* dst (+)= Q(alpha*src) over the box; alpha==0 with add==0 zero-fills without reading src.
 * Replaces the reference's index-vector gather/scatter copy_n / copy_n_blocking (copy_n.h:541,
 * :1031) and get_permutation (tensor.h:815-961).  stream: cudaStream_t (NULL = library stream). */
int sbk_permute_copy(const sbk_box_desc *box, const void *src, int dtype_src, void *dst,
                     int dtype_dst, const double *alpha, int add, int device, void *stream);
/* Which kernel variant sbk_permute_copy would use: writes a short text ("tiled es=16 tile=...") */
int sbk_permute_describe(const sbk_box_desc *box, int dtype_src, int dtype_dst, const double *alpha,
                         int add, const void *src, const void *dst, char *buf, size_t buflen);

#define SBK_MAX_GROUP_DIMS 8
/* One label of a contraction: extent and strides (in elements) in the tensors that carry it */
typedef struct sbk_contract_dim {
    int size;
    int64_t s0, s1, sr; /* stride in v0, v1, vr; 0 when the tensor does not have the label */
} sbk_contract_dim;

typedef struct sbk_contract_desc {
    int nT, nM, nN, nK;
    sbk_contract_dim T[SBK_MAX_GROUP_DIMS]; /* batch labels   : v0, v1, vr */
    sbk_contract_dim M[SBK_MAX_GROUP_DIMS]; /* labels of v0 and vr (reference's B) */
    sbk_contract_dim N[SBK_MAX_GROUP_DIMS]; /* labels of v1 and vr (reference's C) */
    sbk_contract_dim K[SBK_MAX_GROUP_DIMS]; /* contracted labels: v0, v1 (reference's A) */
    int conj0, conj1;
} sbk_contract_desc;

/* vr = alpha * sum_K f0(v0) f1(v1) + beta * vr with operands addressed through the strides above
 * (the permutation is folded into the tile loaders).  Replaces local_contraction_normalized
 * (tensor.h:1475) + xgemm_batch_strided (blas.h:662).  workspace may be NULL (library pool). */
int sbk_contract(const sbk_contract_desc *desc, int dtype, const double *alpha, const void *v0,
                 const void *v1, const double *beta, void *vr, int device, void *stream);
int sbk_contract_describe(const sbk_contract_desc *desc, int dtype, char *buf, size_t buflen);

#ifdef __cplusplus
}
#endif
#endif /* SUPERBBLAS_B200_H */
