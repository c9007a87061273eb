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
/* Work that has been begun and not completed (the reference's Request, dist.h:54-61): a copy, a
 * bsr_krylov, a dense solver or the create of a block-sparse operator.  Every sbb_*_begin returns 1 with
 * "<name>_begin: null request" for a null `request`, and then begins and writes nothing. */
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
 * ("permute"), of the tensor-core contraction kernel ("contract_mma"), of the dense-solver kernel ("dense"), of the
 * block-sparse kernel ("bsr") and of the Kronecker block-sparse kernel ("kron_bsr") is bracketed by CUDA events
 * on its stream; sbb_profile_read synchronises, returns the summed duration and clears the list. */
int sbb_profile_enable(int on);
int sbb_profile_read(const char *kernel, double *total_ms, long long *count);

/* Reports of the public calls (performance.h:357-518).  With tracking on -- the environment variable
 * SB_TRACK_TIME set to a nonzero number, or sbb_track_time(1) -- sbb_copy, sbb_copy_begin,
 * sbb_request_wait, sbb_contraction the dense solvers (names cholesky, trsm, gesm, inversion; flops
 * n^3/3, n^2 nrhs, 2n^3/3 + 2n^2 nrhs and 2n^3 per matrix, x4 for complex types; eigh, with flops 0
 * because its number of sweeps is decided on the device, and bytes the matrices plus W; their _begin forms
 * count as cholesky_begin, ..., and what their later steps queue as wait) and sbb_bsr_krylov
 * (name bsr_krylov; flops 8 (complex) or 2 x nnz blocks x vol(blockim) vol(blockdom) x columns x P,
 * bytes the matrix + the gathered x + y; for a Kronecker operator 8 or 2 x rows x U x (vol(blockim)
 * vol(blockdom) vol(krondom) + vol(kronim) vol(krondom) vol(blockim)) x columns x P, bytes the blocks + the
 * factors + the gathered x + y) accumulate per name: host seconds, device seconds (CUDA events
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
 * rank has begun it is an error.  Requests with several exchanges (sbb_bsr_krylov_begin,
 * sbb_create_bsr_begin, sbb_create_kron_bsr_begin, sbb_cholesky_begin, sbb_inversion_begin,
 * sbb_trsm_begin, sbb_gesm_begin) go round by round: every rank begins, then every rank calls
 * sbb_request_progress once per round until all are done.  The collective calls that complete their
 * exchanges inside (sbb_create_bsr, sbb_bsr_krylov, sbb_cholesky, ...) cannot be used on loopback
 * ranks.  Masked copies are not supported on loopback communicators.  This is how the cross-rank path
 * is tested on a box with fewer GPUs than ranks. */
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
 * communicator carries one outstanding request at a time: beginning another exchange on it completes
 * the whole request first. */
int sbb_copy_begin(int dtype0, int dtype1, const double *alpha, int nd0, const int *p0,
                   int ncomponents0, const char *o0, const int *from0, const int *size0,
                   const int *dim0, const void *const *v0, const float *const *mask0,
                   const sbb_context *ctx0, int nd1, const int *p1, int ncomponents1, const char *o1,
                   const int *from1, const int *dim1, void *const *v1, const float *const *mask1,
                   const sbb_context *ctx1, sbb_comm_t comm, int co, int copyadd,
                   sbb_request_t *request);
int sbb_request_wait(sbb_request_t request);
/* One step of a request: completes the exchange in flight, queues everything up to the next exchange and
 * begins it, or sets *done when nothing is left.  When *done is set the request is complete (host results
 * included) and released; on an error it is not released (sbb_request_wait releases it).  A copy is one
 * step; sbb_request_wait is sbb_request_progress until done.  A process-per-GPU program just waits;
 * loopback ranks step in rounds (sbb_comm_create_local). */
int sbb_request_progress(sbb_request_t request, int *done);

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

/* ---- batched dense solvers (reference: cholesky, trsm, gesm, inversion; dense.h:1019-1290) ------- */

enum sbb_dense_op { SBB_CHOLESKY = 0, SBB_INVERSION = 1, SBB_TRSM = 2, SBB_GESM = 3, SBB_EIGH = 4 };

/* A dense-solver tensor is a whole tensor: its extent along each label is max(from + size) over all
 * parts (parts do not wrap).  `orows` / `ocols` (disjoint subsets of `o`) pick out the matrix: the
 * row index linearises the orows labels in the order of that string with the call's CoorOrder
 * (FastToSlow: first label fastest), columns likewise, n = vol(orows) = vol(ocols).  Every other label
 * of the matrix tensor is a batch label: one matrix per batch coordinate.  dtype: F32, F64, C64 or
 * C128; float types compute in their own type.  gesm and inversion: one matrix must fit in one CTA's
 * shared memory, n^2 * sizeof(T) <= 200 KiB (n <= 113 for C128, 160 for F64 and C64, 226 for F32).
 * cholesky and trsm have no limit beyond device memory: a larger matrix runs a blocked tier on two
 * pooled workspaces, the item's matrices and (trsm) a copy of the item's X box, with its updates
 * on the contraction kernels.
 *
 * Where every part holds whole matrices (all rows and columns) the kernels work in place; otherwise
 * every part's matrices are gathered with the copy engine, each part factors the matrices it touches
 * (redundant work, identical bits) and writes back its own box.
 *
 * Singular or indefinite matrices raise no error (that would need a device-to-host synchronisation):
 * their results come out non-finite.  Results are deterministic; replicated parts compute identical
 * bits.  Argument errors are thrown by every rank alike, before any data moves. */

/* A = U^H U with U upper triangular (row <= col): reads the upper triangle and the real part of the
 * diagonal, writes U there and zeros strictly below the diagonal.  In place. */
int sbb_cholesky(int dtype, int nd, const int *p, int ncomponents, const char *o, void *const *v,
                 const char *orows, const char *ocols, const sbb_context *ctx, sbb_comm_t comm, int co);
/* A <- A^-1 in place, by Gauss-Jordan elimination with partial pivoting (largest |.| in the column). */
int sbb_inversion(int dtype, int nd, const int *p, int ncomponents, const char *o, void *const *v,
                  const char *orows, const char *ocols, const sbb_context *ctx, sbb_comm_t comm, int co);
/* Solve with the upper triangle of C (trsm) or with a general A by LU with partial pivoting (gesm).
 * If X carries the orows labels, Y carries the ocols labels and A Y = alpha X is solved; if X carries
 * the ocols labels, Y carries the orows labels and Y A = alpha X is solved.  Any other label of X is a
 * batch label when the matrix has it and a right-hand-side label otherwise; Y has exactly those labels
 * too, with the same extents.  Label orders are arbitrary. */
int sbb_trsm(int dtype, const double *alpha, int ndc, const int *pc, int ncomponentsc, const char *oc,
             const char *orows, const char *ocols, const void *const *vc, const sbb_context *ctxc,
             int ndx, const int *px, int ncomponentsx, const char *ox, const void *const *vx,
             const sbb_context *ctxx, int ndy, const int *py, int ncomponentsy, const char *oy,
             void *const *vy, const sbb_context *ctxy, sbb_comm_t comm, int co);
int sbb_gesm(int dtype, const double *alpha, int ndc, const int *pc, int ncomponentsc, const char *oc,
             const char *orows, const char *ocols, const void *const *vc, const sbb_context *ctxc,
             int ndx, const int *px, int ncomponentsx, const char *ox, const void *const *vx,
             const sbb_context *ctxx, int ndy, const int *py, int ncomponentsy, const char *oy,
             void *const *vy, const sbb_context *ctxy, sbb_comm_t comm, int co);
/* Eigen-decomposition of every Hermitian matrix of A (ours; cuSOLVER's heevjBatched is the vendor
 * counterpart): A = V diag(w) V^H by cyclic two-sided Jacobi.  Reads the upper triangle and the real
 * part of the diagonal, as cholesky; the strict lower triangle is never read.  A is overwritten with
 * the eigenvectors V: column j (linearised over ocols) is the unit eigenvector of w[j], defined up to a
 * phase as in LAPACK.  The eigenvalues go to W, ascending (ties keep index order).  W's element type is
 * the real type of dtype (F32 for F32 and C64, F64 for F64 and C128); it carries every batch label of A
 * with the same extent and the ocols labels, which linearise the eigenvalue index like the columns, in
 * any label order, with its own partition `pw` / `ncomponentsw` and contexts `ctxw` (host components
 * allowed); any other label, or a missing one, is an argument error.  A and V must both fit in one
 * CTA's shared memory, 2 n^2 * sizeof(T) <= 200 KiB: n <= 80 for C128, 113 for F64 and C64, 160 for F32.
 * Every part of W gets the eigenvalues of its batch range: from the launch that writes the same batch
 * box of A on its rank, or else from a launch of its own on the matrices (in place or gathered as for
 * A), so W does not depend on the partitions.  Every finite matrix is diagonalised, whatever its
 * magnitude (it is scaled by a power of two for the sweeps); a matrix with a non-finite entry in what is
 * read gives NaN eigenvalues and eigenvectors, and no error.  There is no request form. */
int sbb_eigh(int dtype, int nd, const int *p, int ncomponents, const char *o, void *const *v,
             const char *orows, const char *ocols, const sbb_context *ctx,
             int ndw, const int *pw, int ncomponentsw, const char *ow, void *const *vw,
             const sbb_context *ctxw, sbb_comm_t comm, int co);
/* The dense calls as requests (reference: the `Request *request` argument of cholesky, trsm, gesm and
 * inversion), with the arguments of the calls above.  Argument errors are returned here, by every rank
 * alike, before any data moves, with the messages of the calls without a request.  On return the host
 * components are staged, the gather of the matrices has begun where the call gathers them (pack kernels,
 * signal, local part), and behind its local part the kernels of every item whose gathered operands come
 * from this rank's own parts alone are queued (without gathers: every kernel).  Each later step completes
 * one gather and queues what it unblocks: the gather of X (trsm, gesm) begins in the step after that of
 * the matrices, one exchange at a time, and the last step runs the remaining items, blocked tier
 * included, their write-back from the gathered copies and the copy of host outputs back.  The outputs
 * (A for cholesky and inversion, Y for trsm and gesm) are defined only when the request is complete,
 * and bit-identical to the call's without a request; until then the inputs must not be modified nor the
 * outputs read.  sbb_dense_steps_describe lists the steps. */
int sbb_cholesky_begin(int dtype, int nd, const int *p, int ncomponents, const char *o, void *const *v,
                       const char *orows, const char *ocols, const sbb_context *ctx, sbb_comm_t comm, int co,
                       sbb_request_t *request);
int sbb_inversion_begin(int dtype, int nd, const int *p, int ncomponents, const char *o, void *const *v,
                        const char *orows, const char *ocols, const sbb_context *ctx, sbb_comm_t comm, int co,
                        sbb_request_t *request);
int sbb_trsm_begin(int dtype, const double *alpha, int ndc, const int *pc, int ncomponentsc, const char *oc,
                   const char *orows, const char *ocols, const void *const *vc, const sbb_context *ctxc,
                   int ndx, const int *px, int ncomponentsx, const char *ox, const void *const *vx,
                   const sbb_context *ctxx, int ndy, const int *py, int ncomponentsy, const char *oy,
                   void *const *vy, const sbb_context *ctxy, sbb_comm_t comm, int co, sbb_request_t *request);
int sbb_gesm_begin(int dtype, const double *alpha, int ndc, const int *pc, int ncomponentsc, const char *oc,
                   const char *orows, const char *ocols, const void *const *vc, const sbb_context *ctxc,
                   int ndx, const int *px, int ncomponentsx, const char *ox, const void *const *vx,
                   const sbb_context *ctxx, int ndy, const int *py, int ncomponentsy, const char *oy,
                   void *const *vy, const sbb_context *ctxy, sbb_comm_t comm, int co, sbb_request_t *request);
/* Describe, without touching any data, what the dense call `op` would do on `rank` of `nranks` (its
 * arguments without buffers, contexts and communicator; cholesky and inversion pass ndx = ndy = 0;
 * for SBB_EIGH, pass ndx = 0 and W in the y arguments, and each item line ends with what it writes,
 * "writes a", "writes w" or "writes aw"):
 * in place or re-partitioned, one line per kernel launch with its tier and label groups (a blocked
 * cholesky or trsm follows it with one `step` line per launch of the tier), the boxes written back
 * from the gathered copies, and the sbb_copy_plan_describe text of each gather.  Host
 * only; throws the argument errors of the call.  Returns 2 if buf is too small (*needed is set). */
int sbb_dense_plan_describe(int op, int dtype, const double *alpha, int ndc, const int *pc,
                            int ncomponentsc, const char *oc, const char *orows, const char *ocols,
                            int ndx, const int *px, int ncomponentsx, const char *ox, int ndy,
                            const int *py, int ncomponentsy, const char *oy, int nranks, int rank,
                            int co, char *buf, size_t buflen, size_t *needed);
/* The steps of the same call as a request (sbb_cholesky_begin, ...), with the arguments of
 * sbb_dense_plan_describe: a line "steps <S> exchanges <E>" (S = E + 1: the begin, then one step per
 * gather; every rank has the same), then per item of sbb_dense_plan_describe, in its order, a line
 * "item <i> step <s>" with the step that queues its kernels.  Empty when the call has nothing to do. */
int sbb_dense_steps_describe(int op, int dtype, const double *alpha, int ndc, const int *pc,
                             int ncomponentsc, const char *oc, const char *orows, const char *ocols,
                             int ndx, const int *px, int ncomponentsx, const char *ox, int ndy,
                             const int *py, int ncomponentsy, const char *oy, int nranks, int rank,
                             int co, char *buf, size_t buflen, size_t *needed);

/* ---- block-sparse operators (reference: create_bsr, bsr_krylov; bsr.h:2286, :2352, :2516) ----------- */

/* An operator A from the domain lattice (nd labels, extents dimd) to the image lattice (ni labels,
 * extents dimi) made of dense blocks of blockim x blockdom elements.
 *   pim      : image parts, int[nranks*ncomponents][2][ni], [rank][component] order.  The from and size
 *              of every non-empty part are multiples of blockim; the parts cover the image lattice
 *              without overlapping.
 *   pdom     : domain partition, checked for shape only (x is gathered from its own partition).
 *   ii[c]    : one int per block row of component c: its number of nonzero blocks (zero allowed).  The
 *              block rows of a part are the points of its lattice of blocks (size / blockim), numbered
 *              with the CoorOrder `co`.
 *   jj[c]    : nd ints per nonzero block, in row order: the global domain coordinate of the block's first
 *              element, taken modulo dimd (periodic).  It must be a multiple of blockdom and the block
 *              must not wrap: (jj mod dimd) + blockdom <= dimd.
 *   v[c]     : sum(ii) blocks of vol(blockim) * vol(blockdom) elements, in the order of jj.  In a block,
 *              with i the image index and j the domain index (each linearised with `co`), element (i, j)
 *              is at i + j * vol(blockim) if blockImFast, and at j + i * vol(blockdom) otherwise.
 *   ii, jj, v live in the memory of the component's context.  ii and jj are read during the call; v is
 *   referenced (not copied) until sbb_destroy_bsr, and later changes to its values are seen by later
 *   calls.  With a communicator the call is collective and every rank throws the same error, even
 *   when only one rank's jj is wrong: the halo boxes and an error code of every rank are shared with
 *   one small copy. */
typedef struct sbb_bsr_s *sbb_bsr_t;
int sbb_create_bsr(int dtype, int ni, const int *pim, const int *dimi, int nd, const int *pdom, const int *dimd,
                   int ncomponents, const int *blockim, const int *blockdom, int blockImFast,
                   const int *const *ii, const int *const *jj, const void *const *v, const sbb_context *ctx,
                   sbb_comm_t comm, int co, sbb_bsr_t *bsr);
/* Releases the operator.  While a request on it (its create, a sbb_bsr_krylov_begin) has not been
 * released, it is an error ("destroy_bsr: ...") that leaves the handle valid: wait, then destroy again. */
int sbb_destroy_bsr(sbb_bsr_t bsr);
/* sbb_create_bsr in two steps: the handle is returned at once and becomes usable when `*request`
 * completes (sbb_request_wait / sbb_request_progress).  ii and jj are read before it returns.  Argument
 * errors that need no exchange are returned here; those that need every rank's data (a bad jj or ii on
 * any rank) are returned by the completion, with the same message on every rank, and leave the handle
 * unusable (sbb_destroy_bsr still releases it).  sbb_bsr_krylov on a handle whose create has not
 * completed is an error.  Destroy the handle only after its request has been released (completed, or
 * waited for after an error). */
int sbb_create_bsr_begin(int dtype, int ni, const int *pim, const int *dimi, int nd, const int *pdom,
                         const int *dimd, int ncomponents, const int *blockim, const int *blockdom, int blockImFast,
                         const int *const *ii, const int *const *jj, const void *const *v, const sbb_context *ctx,
                         sbb_comm_t comm, int co, sbb_bsr_t *bsr, sbb_request_t *request);

/* A Kronecker block-sparse operator (reference: create_kron_bsr in bsr.h; this contract follows the
 * reference's names and argument order as far as they are known, and was not checked against the
 * reference itself).  It is the operator of sbb_create_bsr whose blocks have the effective extents
 * blockim[k] * kronim[k] and blockdom[k] * krondom[k]: every rule above holds with those extents
 * (parts and jj are multiples of them, blocks do not wrap).  Along any one label at most one of blockim
 * and kronim (blockdom and krondom) exceeds 1.
 *   ii[c]    : every block row of every component, on every rank, has the same number U of blocks.
 *   v[c]     : the B blocks, vol(blockim) x vol(blockdom) elements each, laid out as for sbb_create_bsr.
 *   kronv[c] : U factors K_u of vol(kronim) x vol(krondom) elements, in the same layout rule; factor u
 *              applies to the u-th block of every row.  Referenced like v (not copied, valid until
 *              sbb_destroy_bsr, later changes seen).  Each component reads its own kronv; the results
 *              are independent of the partition only when every component holds the same values.
 * The u-th block of row r is K_u ⊗ B_{r,u}: the element at image offset (kron ik, block ib) and domain
 * offset (kron jk, block jb), each linearised with `co` over its own labels, is K_u[ik, jk] B_{r,u}[ib, jb].
 * sbb_bsr_krylov and sbb_destroy_bsr take the handle unchanged.  Every output element is
 *   sum over u in jj order, then over jk in order, of K_u[ik, jk] t_u[jk, ib, c], with
 *   t_u[jk, ib, c] = the sum over jb in order of B_{r,u}[ib, jb] x[jk, jb, c],
 * one fused multiply-add per term in the accumulation type, then the alpha / beta epilogue: bit-identical
 * however x, y and the operator are partitioned (not to sbb_create_bsr on the expanded blocks, whose sum
 * runs in another order).  Limits of the kernel: vol(kronim) vol(blockim) <= 4096, the U factors within
 * 64 KiB, and one B block with one column of its input slab (vol(krondom) vol(blockdom)) and its partial
 * sums within 96 KiB.  Errors start with "create_kron_bsr:", and every rank throws the same one. */
int sbb_create_kron_bsr(int dtype, int ni, const int *pim, const int *dimi, int nd, const int *pdom,
                        const int *dimd, int ncomponents, const int *blockim, const int *blockdom,
                        const int *kronim, const int *krondom, int blockImFast,
                        const int *const *ii, const int *const *jj, const void *const *v,
                        const void *const *kronv, const sbb_context *ctx, sbb_comm_t comm, int co,
                        sbb_bsr_t *bsr);
/* sbb_create_kron_bsr in two steps, as sbb_create_bsr_begin; a mismatch of U between ranks is returned by
 * the completion. */
int sbb_create_kron_bsr_begin(int dtype, int ni, const int *pim, const int *dimi, int nd, const int *pdom,
                              const int *dimd, int ncomponents, const int *blockim, const int *blockdom,
                              const int *kronim, const int *krondom, int blockImFast, const int *const *ii,
                              const int *const *jj, const void *const *v, const void *const *kronv,
                              const sbb_context *ctx, sbb_comm_t comm, int co, sbb_bsr_t *bsr,
                              sbb_request_t *request);

/* y_p <- beta * y_p + alpha * A u_p for p = 0 .. P-1, with u_0 = x and u_p = the finished y_{p-1}.
 *   oim (ni letters) names the image labels, odom (nd letters) the domain labels; they may share letters.
 *   x carries every odom label with extent dimd and y every oim label with extent dimi; along them
 *   from = 0 and size = dim.  Every other label of x is a column label and appears in y with the same
 *   size, in any order.  y may also carry `power_label` (0: none), which x must not have; its size is P.
 *   P > 1 needs ni == nd and dimi == dimd; y_{p-1} is read with oim[k] as odom[k].
 *   When beta is zero y is not read.  dtype: F32, F64, C64 or C128 (as given to sbb_create_bsr); float
 *   types accumulate in double.  Every output element sums its row's blocks in jj order, and each block's
 *   domain index in order, so y is bit-identical however x, y and the operator are partitioned.
 *   The kernel writes y directly when y's parts are the operator's image parts with every column and
 *   power; otherwise it works on temporaries that receive y's box of each image part (when beta is
 *   nonzero) and are copied back into y, with the same arithmetic. */
int sbb_bsr_krylov(int dtype, const double *alpha, sbb_bsr_t bsr, const char *oim, const char *odom, int ndx,
                   const int *px, int ncomponentsx, const char *ox, const int *fromx, const int *sizex,
                   const int *dimx, const void *const *vx, const sbb_context *ctxx, const double *beta, int ndy,
                   const int *py, int ncomponentsy, const char *oy, const int *fromy, const int *sizey,
                   const int *dimy, char power_label, void *const *vy, const sbb_context *ctxy, sbb_comm_t comm,
                   int co);
/* sbb_bsr_krylov as a request (reference: the `Request *request` argument of bsr_krylov).  It returns
 * after the first step: host components staged, the gather of x begun (packs, signal, local part) and,
 * behind the local part, the kernels of power 0 for the interior rows of every component -- the block
 * rows all of whose blocks read only points that the gather fills from this rank's own parts.  The next
 * step completes the gather and runs the boundary rows; the write-back and the powers p >= 1 follow, one
 * exchange per step.  Without temporaries to fill (beta == 0 or y written directly) that is the split;
 * with them every row runs after the fill.  y is defined once the request is complete, and bit-identical
 * to sbb_bsr_krylov's.  x, y and the operator must not be modified, nor y read, before then. */
int sbb_bsr_krylov_begin(int dtype, const double *alpha, sbb_bsr_t bsr, const char *oim, const char *odom, int ndx,
                         const int *px, int ncomponentsx, const char *ox, const int *fromx, const int *sizex,
                         const int *dimx, const void *const *vx, const sbb_context *ctxx, const double *beta, int ndy,
                         const int *py, int ncomponentsy, const char *oy, const int *fromy, const int *sizey,
                         const int *dimy, char power_label, void *const *vy, const sbb_context *ctxy,
                         sbb_comm_t comm, int co, sbb_request_t *request);
/* Describe, without touching any device, what sbb_bsr_krylov would do on `rank` of `nranks` with the
 * operator sbb_create_bsr (kronim and krondom NULL) or sbb_create_kron_bsr would build from every rank's
 * ii and jj (host arrays, concatenated in [rank][component] order).  Throws the argument errors of both
 * calls.  With split == 0: direct or written back, one line per kernel launch with its dims, row pointers
 * and block offsets (and, for a Kronecker operator, a `kron` line with vol(kronim), vol(krondom), U and
 * the Kronecker extents of its image and domain labels), the boxes scaled by beta, and the
 * sbb_copy_plan_describe text of the gather of every power and of the write-back.  With split == 1: the
 * interior and boundary rows (sbb_bsr_krylov_begin) of every kernel launch, from the gather of x: per
 * launch a line "split comp <c>", then "interior" and "boundary" lines with the block rows. */
int sbb_bsr_plan_describe(int dtype, int ni, const int *pim, const int *dimi, int nd, const int *pdom,
                          const int *dimd, int ncomponents, const int *blockim, const int *blockdom,
                          const int *kronim, const int *krondom, int blockImFast, const int *ii_all,
                          const int *jj_all, const double *alpha, const char *oim, const char *odom, int ndx,
                          const int *px, int ncomponentsx, const char *ox, const int *fromx, const int *sizex,
                          const int *dimx, const double *beta, int ndy, const int *py, int ncomponentsy,
                          const char *oy, const int *fromy, const int *sizey, const int *dimy, char power_label,
                          int nranks, int rank, int co, int split, char *buf, size_t buflen, size_t *needed);

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
