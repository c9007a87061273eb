// Driver of the batched dense solvers (cholesky, inversion, trsm, gesm): argument checks, the items
// of every rank, and the gather of whole matrices with the copy engine where a part does not hold
// them.
//
// Reference counterparts: cholesky, trsm, gesm, inversion (dense.h:1019-1290).
#pragma once
#include "dense_kernel.hpp"
#include "driver.hpp"

namespace sbb {

    struct DenseArgs {
        int op = SBB_CHOLESKY, dtype = SBB_C128;
        double alpha[2] = {1, 0};
        TensorArg a, x, y; ///< x, y: trsm and gesm only; from / size / dim are filled by the plan
        std::string orows, ocols;
        int co = FastToSlow, nranks = 1, rank = 0;
    };

    /// One kernel launch of this rank, driven by one part of the output (A for cholesky and
    /// inversion, Y for trsm and gesm).  Components are local indices, offsets and counts in elements;
    /// a component -1 means the operand is in slot `slot` of its gather (or, for the output, in a
    /// temporary of `*_elems` elements whose box `back` is then copied into component `comp`).
    struct DenseItem {
        int comp;   ///< component of the output part
        int a_comp; int64_t a_off, a_elems;
        int x_comp; int64_t x_off, x_elems;
        int y_comp; int64_t y_off, y_elems;
        int slot;
        bool write_back; ///< the kernel works on a temporary: copy `back` from it into `comp`
        sbk_box_desc back;
        sbk_dense_desc desc;
    };

    /// What a dense call does on one rank, decided from geometry alone; no device is touched
    struct DensePlan {
        int op = SBB_CHOLESKY, dtype = SBB_C128;
        bool nothing = false;              ///< no element in the output
        bool gather_a = false, gather_x = false; ///< some part lacks whole matrices / vectors
        int slots = 0;                     ///< largest number of items of one rank
        std::vector<DenseItem> items;      ///< this rank's, in launch order
        CopyArgs a_args, x_args;           ///< A / X -> the gather slots
        std::string describe() const;
    };

    /// Throws the call's argument errors; every rank throws the same ones
    DensePlan make_dense_plan(const DenseArgs &a);

    void execute_dense(const DenseArgs &a, const std::vector<Buffer> &va, const std::vector<Buffer> &vx,
                       const std::vector<Buffer> &vy, Comm *comm);

} // namespace sbb
