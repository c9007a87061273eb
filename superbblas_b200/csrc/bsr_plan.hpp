// Distributed block-sparse operators (create_bsr, bsr_krylov, destroy_bsr): the operator's host
// geometry, the plan of a call and its execution.
//
// At create time every operator component computes its halo box -- per domain label the shortest
// periodic arc that covers every referenced [jj, jj + blockdom) -- and turns each block's jj into the
// point of the gathered input where the block's domain starts.  The boxes of every rank (and a
// per-rank error code) are shared with one copy of a small int32 tensor, so every rank can plan the
// gather and every rank throws the same error.  At call time x is gathered into the halo boxes with
// the copy engine (columns fastest, then the domain labels), the kernel runs straight into y when
// y's parts are the operator's image parts, and otherwise into temporaries that hold y's box of the
// part (when beta is nonzero) and are copied back into y: the same epilogue either way, so y is
// bit-identical whichever path runs.
//
// A Kronecker operator (create_kron_bsr) is planned as the plain operator of its effective blocks
// (blockim * kronim, blockdom * krondom): the Kronecker labels are ordinary labels for the halo boxes,
// the gathers and the write-back; only the kernel and the values differ.
//
// Reference counterparts: create_bsr (bsr.h:2286, :2352), create_kron_bsr, bsr_krylov (bsr.h:2516),
// destroy_bsr.
#pragma once
#include "bsr_kernel.hpp"
#include "driver.hpp"

namespace sbb {

    /// What create_bsr is given, apart from the arrays of this rank
    struct BsrShape {
        int dtype = SBB_C128, ni = 0, nd = 0, ncomp = 1, co = FastToSlow, nranks = 1, rank = 0;
        Coor dimi, dimd, blockim, blockdom;
        Coor kronim, krondom;       ///< all ones for a plain operator
        bool kron = false;          ///< made by create_kron_bsr
        bool im_fast = true;
        std::vector<Box> pim, pdom; ///< all ranks, [rank][component]
        Coor effim() const;         ///< blockim * kronim
        Coor effdom() const;        ///< blockdom * krondom
        const char *name() const { return kron ? "create_kron_bsr" : "create_bsr"; }
    };

    /// One operator component as create_bsr leaves it (host copies)
    struct BsrPart {
        int error = 0;               ///< 0, or a code of bsr_error()
        Box halo;                    ///< in the domain labels; empty without blocks
        std::vector<int64_t> rowptr; ///< block rows + 1
        std::vector<int64_t> goff;   ///< per nonzero block, point of the halo box
        int u = -1;                  ///< Kronecker: blocks of every row, -1 without rows
    };

    /// Geometry of an operator: the shape, this rank's parts and every part's halo box
    struct BsrGeometry {
        BsrShape s;
        std::vector<BsrPart> mine;   ///< this rank's components
        std::vector<Box> halo;       ///< all ranks, [rank][component]
    };

    /// Argument checks that need no array; the same on every rank
    void check_bsr_shape(const BsrShape &s);
    /// Block rows of the part (lattice of blocks of the image box)
    int64_t bsr_rows(const BsrShape &s, const Box &part);
    /// One component from its ii (block rows) and jj (nnz * nd) on the host
    BsrPart make_bsr_part(const BsrShape &s, const Box &part, const int *ii, const int *jj);
    /// Every part computed here from all ranks' ii and jj (concatenated in [rank][component] order)
    BsrGeometry bsr_geometry_from_all(const BsrShape &s, const int *ii_all, const int *jj_all);

    struct BsrCall {
        int dtype = SBB_C128;
        double alpha[2] = {1, 0}, beta[2] = {0, 0};
        std::string oim, odom;
        TensorArg x, y;
        char power = 0;
        int co = FastToSlow, nranks = 1, rank = 0;
    };

    /// One kernel launch (per power) of this rank, for operator component `comp`
    struct BsrItem {
        int comp;
        int y_comp;               ///< direct: the y component; -1: a temporary of y_elems elements
        int64_t y_off, y_pstride; ///< direct: offset at power 0, stride of the power label
        int64_t y_elems, x_elems; ///< temporary and gathered input, in elements
        int64_t nnz;
        sbk_bsr_desc desc;        ///< rowptr and goff are filled at execution
        sbk_kron_desc kdesc;      ///< Kronecker operators only
    };

    struct BsrPlan {
        bool nothing = false, direct = false;
        int powers = 1, slots = 0;
        std::vector<BsrItem> items;  ///< this rank's, in launch order
        CopyArgs gather_x, gather_y; ///< x (or y_{p-1}, power from0 set per call) -> slots
        CopyArgs fill;               ///< y_p -> temporaries (power from0 set per call), when beta != 0
        CopyArgs back;               ///< temporaries -> y_p (power from1 set per call)
        bool fill_temps = false, kron = false;
        int y_power_pos = -1;
        std::string odom;
        CopyArgs fill_args(int p) const; ///< fill / back with the power label at p
        CopyArgs back_args(int p) const;
        std::string describe(const BsrGeometry &g) const;
    };

    /// Throws the call's argument errors; every rank throws the same ones
    BsrPlan make_bsr_plan(const BsrGeometry &g, const BsrCall &c);

    /// The block rows of one item (plan.items order), by what they read of the gathered input: a row is
    /// a boundary row iff one of its blocks' domain boxes meets a box of the slot that `gather` fills
    /// from another rank, else an interior row, which the local part of the gather completes
    struct BsrRowSplit {
        std::vector<int64_t> interior, boundary; ///< ascending
    };
    std::vector<BsrRowSplit> make_bsr_split(const BsrGeometry &g, const BsrPlan &plan, const CopyPlan &gather);
    /// The items' interior and boundary rows as text (sbb_bsr_plan_describe with split = 1)
    std::string describe_bsr_split(const BsrPlan &plan, const std::vector<BsrRowSplit> &split);

    /// An operator: its geometry and, per component of this rank, the caller's v (and kronv) and
    /// device copies of the row pointers and block offsets
    struct BsrOperator {
        BsrGeometry g;
        std::vector<Buffer> v, kronv; ///< kronv: Kronecker operators only
        std::vector<Buffer> rowptr, goff; ///< pool blocks
        int home = 0;
        /// Pending until the request of its create completes; Failed when that completion threw
        enum State { Pending, Ready, Failed } state = Pending;
        /// Requests on the operator not yet released (its create, bsr_krylov calls): they read and write
        /// it in their later steps, so it must not be destroyed while there is one
        mutable int requests = 0;
        /// Row splits of recent gather plans (the plan is held, so its address is not reused): per item,
        /// a pool block on the device of the item's row pointers with the interior rows, then the
        /// boundary rows; null for an item whose split is trivial (one of the lists is empty)
        struct Split {
            std::shared_ptr<const CopyPlan> gather;
            std::vector<int64_t> ninterior;
            std::vector<Buffer> rows;
            ~Split();
        };
        mutable std::vector<std::shared_ptr<const Split>> splits;
        ~BsrOperator();
    };

    /// kronv: one buffer per component for a Kronecker operator (s.kron), else empty.  Throws the
    /// argument errors that need no exchange; the operator is usable once `*request` completes (which
    /// throws the errors that need every rank's data)
    BsrOperator *create_bsr_begin(const BsrShape &s, const int *const *ii, const int *const *jj,
                                  const std::vector<Buffer> &v, const std::vector<Buffer> &kronv, Comm *comm,
                                  std::unique_ptr<Request> *request);

    /// bsr_krylov as a request: the first step is queued when it returns (stage, begin the gather of x,
    /// the interior rows of power 0)
    std::unique_ptr<Request> begin_bsr(const BsrOperator &op, const BsrCall &c, const std::vector<Buffer> &vx,
                                       const std::vector<Buffer> &vy, Comm *comm);

} // namespace sbb
