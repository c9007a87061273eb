// Driver of the batched dense solvers (cholesky, inversion, trsm, gesm) and of eigh: argument checks,
// the items of every rank, and the gather of whole matrices with the copy engine where a part does not
// hold them.
//
// Reference counterparts: cholesky, trsm, gesm, inversion (dense.h:1019-1290).
#pragma once
#include "dense_kernel.hpp"
#include "driver.hpp"
#include <memory>

namespace sbb {

    struct DenseArgs {
        int op = SBB_CHOLESKY, dtype = SBB_C128;
        double alpha[2] = {1, 0};
        TensorArg a, x, y; ///< x, y: trsm and gesm only; from / size / dim are filled by the plan
        TensorArg w;       ///< eigh only: the eigenvalues
        std::string orows, ocols;
        int co = FastToSlow, nranks = 1, rank = 0;
    };

    /// One kernel launch of this rank, driven by one part of the output (A for cholesky and
    /// inversion, Y for trsm and gesm).  Components are local indices, offsets and counts in elements;
    /// a component -1 means the operand is in slot `slot` of its gather (or, for the output, in a
    /// temporary of `*_elems` elements whose box `back` is then copied into component `comp`).
    /// eigh: an item is driven by a part of A (it writes V there, and W through `y_*` when a part of
    /// W on the rank has exactly its batch box: writes = a or aw) or by a part of W that no such item
    /// serves (writes = w: the eigenvalues alone, into `y_*` or a temporary written back into `comp`,
    /// a component of W).  W-only items come first, so that they read A before any item of the rank
    /// overwrites it in place.
    struct DenseItem {
        int comp;   ///< component of the output part
        int writes; ///< eigh: WRITES_A | WRITES_W; 0 for the other ops
        int a_comp; int64_t a_off, a_elems;
        int x_comp; int64_t x_off, x_elems;
        int y_comp; int64_t y_off, y_elems;
        int slot;
        bool write_back; ///< the kernel works on a temporary: copy `back` from it into `comp`
        sbk_box_desc back;
        sbk_dense_desc desc;
    };

    constexpr int WRITES_A = 1, WRITES_W = 2;

    /// What a dense call does on one rank, decided from geometry alone; no device is touched
    struct DensePlan {
        int op = SBB_CHOLESKY, dtype = SBB_C128;
        bool nothing = false;              ///< no element in the output
        bool gather_a = false, gather_x = false; ///< some part lacks whole matrices / vectors
        int slots = 0;                     ///< largest number of items of one rank
        std::vector<DenseItem> items;      ///< this rank's, in launch order
        int w_only = 0;                    ///< eigh: the first w_only items write W alone
        CopyArgs a_args, x_args;           ///< A / X -> the gather slots
        std::string describe() const;
    };

    /// Throws the call's argument errors; every rank throws the same ones
    DensePlan make_dense_plan(const DenseArgs &a);

    /// The steps of a dense call as a request: the gather of A, then that of X, one exchange per step
    /// (only those the plan has; every rank has the same ones), and the step in which each item of this
    /// rank is queued.  Step k < exchanges begins gather k and queues, behind its local part, the items
    /// whose gathered slots are then filled: those of earlier gathers, and of gather k only where its
    /// local part alone fills them (no unpack into the slot).  Step `exchanges` completes the last
    /// gather and queues the rest.  Without gathers every item is queued in step 0.
    struct DenseSteps {
        int exchanges = 0;
        std::vector<int> step; ///< per item of DensePlan::items
        std::string describe() const;
    };
    DenseSteps dense_steps(const DensePlan &plan);

    /// The call begun: host components staged, the first step taken; the argument errors are thrown
    /// before anything is staged.  vw: eigh's W (empty otherwise)
    std::unique_ptr<Request> begin_dense(const DenseArgs &a, const std::vector<Buffer> &va,
                                         const std::vector<Buffer> &vx, const std::vector<Buffer> &vy,
                                         const std::vector<Buffer> &vw, Comm *comm);

} // namespace sbb
