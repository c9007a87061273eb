// Contraction driver. See contract_plan.hpp.
#include "contract_plan.hpp"
#include <algorithm>
#include <cstring>
#include <map>
#include <numeric>
#include <set>
#include <sstream>

namespace sbb {

    namespace {

        struct Label {
            char c;
            int i0 = -1, i1 = -1, ir = -1; ///< position in o0, o1, o_r
            int size = 1;
        };

        std::vector<Label> classify(const ContractionArgs &a) {
            if (!labels_unique(a.t0.o) || !labels_unique(a.t1.o) || !labels_unique(a.tr.o))
                throw std::runtime_error("contraction: repeated label in an order");
            std::map<char, Label> m;
            auto add = [&](const TensorArg &t, int which) {
                for (int k = 0; k < t.nd; ++k) {
                    auto it = m.find(t.o[k]);
                    if (it == m.end()) {
                        Label l;
                        l.c = t.o[k];
                        l.size = t.size[k];
                        it = m.emplace(t.o[k], l).first;
                    } else if (it->second.size != t.size[k]) {
                        throw std::runtime_error("some dimension does not match");
                    }
                    (which == 0 ? it->second.i0 : which == 1 ? it->second.i1 : it->second.ir) = k;
                }
            };
            add(a.t0, 0), add(a.t1, 1), add(a.tr, 2);
            std::vector<Label> out;
            for (auto &kv : m) {
                const Label &l = kv.second;
                const int n = (l.i0 >= 0) + (l.i1 >= 0) + (l.ir >= 0);
                if (n < 2) {
                    if (l.i0 >= 0) throw std::runtime_error("o0 has unmatched dimensions");
                    if (l.i1 >= 0) throw std::runtime_error("o1 has unmatched directions");
                    throw std::runtime_error("o_r has unmatched dimensions");
                }
                out.push_back(l);
            }
            return out;
        }

        std::vector<int> identity(int n) {
            std::vector<int> v(n);
            std::iota(v.begin(), v.end(), 0);
            return v;
        }

        /// (part ∩ range) boxes in the tensor's own label order
        std::vector<RBox> range_boxes(const TensorArg &t, const Box &part) {
            return part_boxes(part, t.from, t.size, t.dim, identity(t.nd), t.nd);
        }

        bool contains(const RBox &outer, const Box &b) {
            for (size_t k = 0; k < b.from.size(); ++k)
                if (b.from[k] < outer.u[k] || b.from[k] + b.size[k] > outer.u[k] + outer.len[k])
                    return false;
            return true;
        }

        /// A piece of work: one box of the partition-driving operand, owned by `part`
        struct Item {
            int part;  ///< global part index of the driving operand
            RBox box;  ///< in the driving operand's label order
        };

    }

    ContractionPlan make_contraction_plan(const ContractionArgs &a) {
        check_float_dtype(a.dtype, "contraction");
        const std::vector<Label> labels = classify(a);
        for (const TensorArg *t : {&a.t0, &a.t1, &a.tr}) {
            if ((int)t->p.size() != a.nranks * t->ncomp) throw std::runtime_error("wtf");
            for (int k = 0; k < t->nd; ++k)
                if (t->size[k] < 0 || t->size[k] > t->dim[k])
                    throw std::runtime_error("contraction: range larger than the tensor");
        }
        ContractionPlan plan;
        if (volume(a.tr.size) == 0) {
            plan.nothing = true;
            return plan;
        }
        const int es = dtype_bytes(a.dtype);
        const int me = a.rank;

        // ---- items of every rank: the larger operand drives the decomposition ---------------------
        plan.big0 = volume(a.t0.size) >= volume(a.t1.size);
        const TensorArg &tb = plan.big0 ? a.t0 : a.t1, &ts = plan.big0 ? a.t1 : a.t0;

        std::vector<Item> items; // all ranks, ascending part
        if (volume(tb.size) > 0 && volume(ts.size) > 0) {
            const std::vector<int> ident = identity(tb.nd);
            std::vector<std::vector<RBox>> raw(tb.p.size());
            for (size_t i = 0; i < tb.p.size(); ++i) raw[i] = range_boxes(tb, tb.p[i]);
            for (size_t i = 0; i < tb.p.size(); ++i) {
                std::vector<RBox> mine = raw[i];
                // every element of the range is contracted once: drop what earlier parts already hold
                for (size_t j = 0; j < i && !mine.empty(); ++j)
                    for (const auto &other : raw[j]) {
                        std::vector<RBox> next;
                        for (const auto &b : mine) {
                            auto left = subtract(b, other, ident);
                            next.insert(next.end(), left.begin(), left.end());
                        }
                        mine.swap(next);
                    }
                for (auto &b : mine)
                    if (!b.empty()) items.push_back(Item{(int)i, b});
            }
        }

        // Range-space box of `t` that an item needs: shared labels follow the item, the others are full
        auto box_in = [&](const TensorArg &t, const Item &it) {
            Box b{Coor(t.nd, 0), t.size};
            for (int k = 0; k < t.nd; ++k) {
                const int kb = label_pos(tb.o, t.o[k]);
                if (kb >= 0) b.from[k] = it.box.u[kb], b.size[k] = it.box.len[kb];
            }
            return b;
        };

        // ---- is the other operand already where every item needs it? ------------------------------
        struct Found {
            int part = -1;
            RBox box;
        };
        std::vector<Found> small_at(items.size());
        bool inplace = true;
        for (size_t q = 0; q < items.size() && inplace; ++q) {
            const int r = items[q].part / tb.ncomp;
            const Box need = box_in(ts, items[q]);
            bool ok = false;
            for (int c = 0; c < ts.ncomp && !ok; ++c) {
                const int part = r * ts.ncomp + c;
                for (const auto &b : range_boxes(ts, ts.p[part]))
                    if (contains(b, need)) {
                        small_at[q].part = part, small_at[q].box = b;
                        ok = true;
                        break;
                    }
            }
            if (!ok) inplace = false;
        }

        // ---- where does the result go? ------------------------------------------------------------
        // Direct: a single item whose output box lies inside the only part that owns that range.
        int direct_part = -1;
        RBox direct_box;
        if (items.size() == 1) {
            const Box out = box_in(a.tr, items[0]);
            RBox want;
            want.u = out.from, want.len = out.size;
            int owners = 0;
            for (size_t i = 0; i < a.tr.p.size(); ++i)
                for (const auto &b : range_boxes(a.tr, a.tr.p[i])) {
                    Coor iu, il;
                    if (intersect(b, want, iu, il)) {
                        ++owners;
                        if (contains(b, out)) direct_part = (int)i, direct_box = b;
                    }
                }
            plan.direct = owners == 1 && direct_part >= 0 &&
                          direct_part / a.tr.ncomp == items[0].part / tb.ncomp;
        }
        plan.repartition = !inplace && !items.empty();
        plan.reduction = !plan.direct && !items.empty();

        // ---- slots: the items of a rank, numbered in order -----------------------------------------
        std::vector<int> slot(items.size()), per_rank(a.nranks, 0);
        for (size_t q = 0; q < items.size(); ++q) slot[q] = per_rank[items[q].part / tb.ncomp]++;
        plan.slots = items.empty() ? 0 : *std::max_element(per_rank.begin(), per_rank.end());

        if (plan.repartition) { // the other operand -> one compact box per slot
            CopyArgs &ca = plan.repart_args = gather_to_slots_args(ts, plan.slots, a.nranks, me, a.co, es);
            for (size_t q = 0; q < items.size(); ++q)
                ca.p1[(size_t)(items[q].part / tb.ncomp) * plan.slots + slot[q]] = box_in(ts, items[q]);
        }
        if (plan.reduction) { // partial slots -> the caller's output partition
            CopyArgs &ra = plan.reduce_args = copy_args(a.nranks, me, a.co, es);
            ra.nd0 = ra.nd1 = a.tr.nd;
            ra.o0 = ra.o1 = a.tr.o;
            ra.ncomp0 = plan.slots;
            ra.p0.assign((size_t)a.nranks * plan.slots, Box{Coor(a.tr.nd, 0), Coor(a.tr.nd, 0)});
            ra.from0.assign(a.tr.nd, 0), ra.size0 = a.tr.size, ra.dim0 = a.tr.size;
            ra.p1 = a.tr.p, ra.ncomp1 = a.tr.ncomp, ra.from1 = a.tr.from, ra.dim1 = a.tr.dim;
            ra.add = true;
            for (size_t q = 0; q < items.size(); ++q)
                ra.p0[(size_t)(items[q].part / tb.ncomp) * plan.slots + slot[q]] = box_in(a.tr, items[q]);
        }

        // ---- the kernel of every item; every rank checks every item, so all ranks throw alike ------
        for (size_t q = 0; q < items.size(); ++q) {
            const Item &it = items[q];
            ContractionItem ci;
            ci.big_comp = it.part % tb.ncomp, ci.slot = slot[q];
            const auto bstr = get_strides(tb.p[it.part].size, a.co);
            ci.big_off = 0;
            for (int k = 0; k < tb.nd; ++k) ci.big_off += (int64_t)it.box.lfrom[k] * bstr[k];

            const Box need = box_in(ts, it);
            std::vector<int64_t> sstr;
            ci.small_comp = -1, ci.small_off = 0, ci.small_elems = 0;
            if (plan.repartition) {
                sstr = get_strides(need.size, a.co);
                ci.small_elems = volume(need.size);
            } else {
                const Found &f = small_at[q];
                ci.small_comp = f.part % ts.ncomp;
                sstr = get_strides(ts.p[f.part].size, a.co);
                for (int k = 0; k < ts.nd; ++k)
                    ci.small_off += (int64_t)(f.box.lfrom[k] + need.from[k] - f.box.u[k]) * sstr[k];
            }

            const Box out = box_in(a.tr, it);
            std::vector<int64_t> ostr;
            ci.out_comp = -1, ci.out_off = 0, ci.out_elems = 0;
            if (plan.direct) {
                ci.out_comp = direct_part % a.tr.ncomp;
                ostr = get_strides(a.tr.p[direct_part].size, a.co);
                for (int k = 0; k < a.tr.nd; ++k)
                    ci.out_off += (int64_t)(direct_box.lfrom[k] + out.from[k] - direct_box.u[k]) * ostr[k];
            } else {
                ostr = get_strides(out.size, a.co);
                ci.out_elems = volume(out.size);
            }

            sbk_contract_desc &d = ci.desc;
            std::memset(&d, 0, sizeof d);
            d.conj0 = a.conj0, d.conj1 = a.conj1;
            for (const Label &l : labels) {
                sbk_contract_dim x;
                // extent of this label inside the item
                const int kb = label_pos(tb.o, l.c), ks = label_pos(ts.o, l.c);
                x.size = kb >= 0 ? it.box.len[kb] : l.size;
                const int64_t big_stride = kb >= 0 ? bstr[kb] : 0;
                const int64_t small_stride = ks >= 0 ? sstr[ks] : 0;
                x.s0 = plan.big0 ? big_stride : small_stride;
                x.s1 = plan.big0 ? small_stride : big_stride;
                x.sr = l.ir >= 0 ? ostr[l.ir] : 0;
                sbk_contract_dim *grp;
                int *n;
                if (l.i0 >= 0 && l.i1 >= 0 && l.ir >= 0) grp = d.T, n = &d.nT;
                else if (l.i0 >= 0 && l.i1 >= 0) grp = d.K, n = &d.nK;
                else if (l.i0 >= 0) grp = d.M, n = &d.nM;
                else grp = d.N, n = &d.nN;
                if (x.size == 1) continue;
                if (*n >= SBK_MAX_GROUP_DIMS)
                    throw std::runtime_error("contraction: too many labels in a group");
                grp[(*n)++] = x;
            }
            if (it.part / tb.ncomp == me) plan.items.push_back(ci);
        }

        // ---- beta scaling of my output range, unless the kernel epilogue applies beta ---------------
        if (!plan.direct && !scalar_is(a.dtype, a.beta, 1)) {
            for (int c = 0; c < a.tr.ncomp; ++c) {
                const int part = me * a.tr.ncomp + c;
                const auto strides = get_strides(a.tr.p[part].size, a.co);
                for (const auto &b : range_boxes(a.tr, a.tr.p[part])) {
                    sbk_box_desc d;
                    std::memset(&d, 0, sizeof d);
                    d.nd = a.tr.nd;
                    int64_t off = 0;
                    for (int k = 0; k < a.tr.nd; ++k) {
                        d.size[k] = b.len[k];
                        d.sstride[k] = d.dstride[k] = strides[k];
                        off += (int64_t)b.lfrom[k] * strides[k];
                    }
                    d.soff = d.doff = off;
                    plan.beta.emplace_back(c, d);
                }
            }
        }
        return plan;
    }

    std::string ContractionPlan::describe() const {
        std::stringstream ss;
        ss << "contraction nothing " << nothing << " big0 " << big0 << " direct " << direct
           << " repartition " << repartition << " reduction " << reduction << " slots " << slots
           << "\n";
        for (const auto &it : items) {
            ss << "item big " << it.big_comp << " " << it.big_off << " small " << it.small_comp << " "
               << it.small_off << " " << it.small_elems << " out " << it.out_comp << " " << it.out_off
               << " " << it.out_elems << " slot " << it.slot;
            const sbk_contract_desc &d = it.desc;
            const struct {
                const char *name;
                int n;
                const sbk_contract_dim *dims;
            } groups[] = {{"T", d.nT, d.T}, {"M", d.nM, d.M}, {"N", d.nN, d.N}, {"K", d.nK, d.K}};
            for (const auto &g : groups) {
                ss << " " << g.name;
                for (int i = 0; i < g.n; ++i)
                    ss << " " << g.dims[i].size << " " << g.dims[i].s0 << " " << g.dims[i].s1 << " "
                       << g.dims[i].sr;
            }
            ss << "\n";
        }
        for (const auto &b : beta) {
            ss << "beta comp " << b.first << " off " << b.second.soff << " size";
            for (int k = 0; k < b.second.nd; ++k) ss << " " << b.second.size[k];
            ss << " stride";
            for (int k = 0; k < b.second.nd; ++k) ss << " " << b.second.sstride[k];
            ss << "\n";
        }
        if (repartition) ss << "repartition\n" << make_copy_plan(repart_args)->describe();
        if (reduction) ss << "reduction\n" << make_copy_plan(reduce_args)->describe();
        return ss.str();
    }

    void execute_contraction(const ContractionArgs &a, const std::vector<Buffer> &v0,
                             const std::vector<Buffer> &v1, const std::vector<Buffer> &vr,
                             Comm *comm) {
        const ContractionPlan plan = make_contraction_plan(a);
        if (plan.nothing) return;
        const int es = dtype_bytes(a.dtype);
        const double one[2] = {1, 0}, zero[2] = {0, 0};

        // ---- 1. home device of this rank -------------------------------------------------------------
        const int home = home_device(comm, {&vr, &v0, &v1}, default_device(comm));

        // ---- 2. host operands staged on it; every workspace of the call comes from `pool` ------------
        PoolGuard pool;
        Staged s0 = stage_in(v0, a.t0, a.rank, es, home, pool);
        Staged s1 = stage_in(v1, a.t1, a.rank, es, home, pool);
        Staged sr = stage_in(vr, a.tr, a.rank, es, home, pool);
        const Staged &sb = plan.big0 ? s0 : s1, &ss = plan.big0 ? s1 : s0;

        // ---- 3. re-partition the other operand: one slot per item, on the item's device --------------
        std::vector<SlotNeed> small_need, out_need; // the partials are allocated after the re-partition
        for (const auto &it : plan.items) {
            const int dev = sb.dev[it.big_comp].device;
            if (it.small_comp < 0) small_need.push_back({it.slot, dev, it.small_elems});
            if (it.out_comp < 0) out_need.push_back({it.slot, dev, it.out_elems});
        }
        const std::vector<Buffer> small = alloc_slots(plan.slots, small_need, es, home, pool);
        if (plan.repartition)
            execute_copy(*get_copy_plan(plan.repart_args), plan.repart_args, a.dtype, a.dtype, one,
                         ss.dev, small, comm);

        // ---- 4. vr <- beta * vr on the output range, in place ----------------------------------------
        for (const auto &b : plan.beta) {
            const Buffer &r = sr.dev[b.first];
            use_device(r.device);
            permute_copy(b.second, r.ptr, a.dtype, r.ptr, a.dtype, a.beta, false, r.device,
                         device_state(r.device).stream);
        }

        // ---- 5. local kernels; several devices in this process: order their streams around them -------
        const std::vector<Buffer> partial = alloc_slots(plan.slots, out_need, es, home, pool);
        const std::set<int> devs = call_devices(home, {&s0, &s1, &sr});
        order_streams(devs);

        for (const auto &it : plan.items) {
            const int dev = sb.dev[it.big_comp].device;
            const Buffer &small_buf = it.small_comp >= 0 ? ss.dev[it.small_comp] : small[it.slot];
            enable_peer(dev, small_buf.device);
            char *out = (char *)partial[it.slot].ptr;
            if (it.out_comp >= 0) {
                out = (char *)sr.dev[it.out_comp].ptr + it.out_off * es;
                enable_peer(dev, sr.dev[it.out_comp].device);
            }
            const char *bptr = (const char *)sb.dev[it.big_comp].ptr + it.big_off * es;
            const char *sptr = (const char *)small_buf.ptr + it.small_off * es;
            use_device(dev);
            contract(it.desc, a.dtype, a.alpha, plan.big0 ? bptr : sptr, plan.big0 ? sptr : bptr,
                     plan.direct ? a.beta : zero, out, dev, device_state(dev).stream);
            {
                const sbk_contract_desc &d = it.desc;
                double vt = 1, vm = 1, vn = 1, vk = 1;
                for (int i = 0; i < d.nT; ++i) vt *= d.T[i].size;
                for (int i = 0; i < d.nM; ++i) vm *= d.M[i].size;
                for (int i = 0; i < d.nN; ++i) vn *= d.N[i].size;
                for (int i = 0; i < d.nK; ++i) vk *= d.K[i].size;
                const bool cplx = a.dtype == SBB_C64 || a.dtype == SBB_C128;
                work_counters().flops += (cplx ? 8.0 : 2.0) * vt * vm * vn * vk;
                work_counters().bytes += vt * (vm * vk + vn * vk + vm * vn) * (double)es;
            }
        }

        order_streams(devs);

        // ---- 6. add the partial results into the caller's partition ------------------------------------
        if (plan.reduction)
            execute_copy(*get_copy_plan(plan.reduce_args), plan.reduce_args, a.dtype, a.dtype, one,
                         partial, sr.dev, comm);

        // ---- 7. host results back (the workspace returns to the pool when `pool` ends) ------------------
        stage_out(vr, sr, home);
    }

} // namespace sbb
