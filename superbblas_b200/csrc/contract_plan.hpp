// Contraction driver: label classification, owner-computes decomposition over the partition of the
// larger operand, optional re-partition of the other operand, local fused kernels, reduction of the
// partial results into the caller's output partition.
//
// Reference counterparts: contraction_normalized (dist.h:3092-3196), get_partitions_for_contraction
// (dist.h:3039-3090), remove_repetitions (dist.h:3001-3028), suggested_orders_for_contraction
// (tensor.h:1271-1429; only its label classification and error rules survive here, the re-ordering
// is unnecessary because the kernels take arbitrary strides).
#pragma once
#include "driver.hpp"

namespace sbb {

    struct ContractionArgs {
        int dtype = SBB_C128;
        double alpha[2] = {1, 0}, beta[2] = {0, 0};
        TensorArg t0, t1, tr;
        bool conj0 = false, conj1 = false;
        int co = FastToSlow, nranks = 1, rank = 0;
    };

    /// One kernel launch of this rank. Components are local component indices; offsets and element
    /// counts are in elements.
    struct ContractionItem {
        int big_comp;          ///< component of the driving operand
        int64_t big_off;
        int small_comp;        ///< component of the other operand, or -1: re-partition slot `slot`
        int64_t small_off;
        int out_comp;          ///< result component (direct), or -1: partial slot `slot`
        int64_t out_off;
        int slot;              ///< index among this rank's items
        int64_t small_elems, out_elems; ///< sizes of the slots
        sbk_contract_desc desc;
    };

    /// What a contraction does on one rank, decided from the call's geometry alone: every argument
    /// check, the items, where their operands come from and where their results go. No device is
    /// touched, so every rank's plan can be built and checked on any host.
    struct ContractionPlan {
        bool nothing = false;    ///< empty output range: nothing to do
        bool big0 = true;        ///< operand 0 drives the decomposition
        bool direct = false;     ///< the kernel writes the result (with beta); no partials
        bool repartition = false, reduction = false;
        int slots = 0;           ///< largest number of items of one rank
        std::vector<ContractionItem> items;              ///< this rank's, in launch order
        std::vector<std::pair<int, sbk_box_desc>> beta;  ///< (result component, box) scaled in place
        CopyArgs repart_args;    ///< other operand -> re-partition slots
        CopyArgs reduce_args;    ///< partial slots -> result, with Add
        std::string describe() const;
    };

    /// Throws the contraction's argument errors; every rank throws the same ones
    ContractionPlan make_contraction_plan(const ContractionArgs &a);

    void execute_contraction(const ContractionArgs &a, const std::vector<Buffer> &v0,
                             const std::vector<Buffer> &v1, const std::vector<Buffer> &vr,
                             Comm *comm);

} // namespace sbb
