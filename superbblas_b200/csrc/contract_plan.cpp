// Contraction driver. See contract_plan.hpp.
#include "contract_plan.hpp"
#include <algorithm>
#include <cstring>
#include <map>
#include <set>

namespace sbb {

    namespace {

        struct Label {
            char c;
            int i0 = -1, i1 = -1, ir = -1; ///< position in o0, o1, o_r
            int size = 1;
        };

        std::vector<Label> classify(const ContractionArgs &a) {
            auto unique = [](const std::string &o) {
                for (size_t i = 0; i < o.size(); ++i)
                    if (o.find(o[i], i + 1) != std::string::npos) return false;
                return true;
            };
            if (!unique(a.t0.o) || !unique(a.t1.o) || !unique(a.tr.o))
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

        /// (part ∩ range) boxes in the tensor's own label order
        std::vector<RBox> own_boxes(const TensorArg &t, const Box &part) {
            std::vector<int> ident(t.nd);
            for (int k = 0; k < t.nd; ++k) ident[k] = k;
            if (part.empty()) return {};
            // part_boxes lives in plan.cpp's anonymous namespace; restate it through ring_pieces
            std::vector<std::vector<Piece>> pieces(t.nd);
            for (int k = 0; k < t.nd; ++k) {
                pieces[k] = ring_pieces(part.from[k], part.size[k], t.from[k], t.size[k], t.dim[k]);
                if (pieces[k].empty()) return {};
            }
            std::vector<RBox> out;
            std::vector<int> idx(t.nd, 0);
            for (;;) {
                RBox b;
                b.u.resize(t.nd), b.len.resize(t.nd), b.lfrom.resize(t.nd);
                for (int k = 0; k < t.nd; ++k) {
                    const Piece &pc = pieces[k][idx[k]];
                    b.u[k] = pc.u, b.len[k] = pc.len, b.lfrom[k] = pc.local;
                }
                out.push_back(b);
                int k = 0;
                for (; k < t.nd; ++k) {
                    if (++idx[k] < (int)pieces[k].size()) break;
                    idx[k] = 0;
                }
                if (k == t.nd) break;
            }
            return out;
        }

        bool contains(const RBox &outer, const Coor &u, const Coor &len) {
            for (size_t k = 0; k < u.size(); ++k)
                if (u[k] < outer.u[k] || u[k] + len[k] > outer.u[k] + outer.len[k]) return false;
            return true;
        }

        /// A piece of work: one box of the partition-driving operand, owned by `part`
        struct Item {
            int part;  ///< global part index of the driving operand
            RBox box;  ///< in the driving operand's label order
        };

        struct View { ///< where an operand box lives
            char *ptr = nullptr;
            int device = 0;
            std::vector<int64_t> stride; ///< per label of the tensor's order
            int64_t off = 0;
        };

        struct Staged {
            std::vector<Buffer> dev; ///< device-resident version of the caller's components
            std::vector<void *> temps;
            std::vector<size_t> bytes;
        };

        /// Host components copied into blocks of `pool` on `home`
        Staged stage_in(const std::vector<Buffer> &v, const TensorArg &t, int me, int es, int home,
                        PoolGuard &pool) {
            Staged s;
            s.dev = v;
            s.temps.assign(v.size(), nullptr);
            s.bytes.assign(v.size(), 0);
            for (size_t c = 0; c < v.size(); ++c) {
                const int64_t vol = volume(t.p[me * t.ncomp + c].size);
                s.bytes[c] = (size_t)vol * es;
                if (!v[c].host || vol == 0) continue;
                if (!v[c].ptr) throw std::runtime_error("null pointer for a non-empty component");
                s.temps[c] = pool.alloc(home, s.bytes[c]);
                s.dev[c].ptr = s.temps[c], s.dev[c].host = false, s.dev[c].device = home;
                use_device(home);
                cuda_check(cudaMemcpyAsync(s.temps[c], v[c].ptr, s.bytes[c], cudaMemcpyHostToDevice,
                                           device_state(home).stream),
                           "cudaMemcpyAsync H2D");
            }
            return s;
        }
    }

    void execute_contraction(const ContractionArgs &a, const std::vector<Buffer> &v0,
                             const std::vector<Buffer> &v1, const std::vector<Buffer> &vr,
                             Comm *comm) {
        if (a.dtype != SBB_F32 && a.dtype != SBB_F64 && a.dtype != SBB_C64 && a.dtype != SBB_C128)
            throw std::runtime_error("contraction: unsupported type");
        const std::vector<Label> labels = classify(a);
        for (const TensorArg *t : {&a.t0, &a.t1, &a.tr}) {
            if ((int)t->p.size() != a.nranks * t->ncomp) throw std::runtime_error("wtf");
            for (int k = 0; k < t->nd; ++k)
                if (t->size[k] < 0 || t->size[k] > t->dim[k])
                    throw std::runtime_error("contraction: range larger than the tensor");
        }
        const int es = dtype_bytes(a.dtype);
        const int me = a.rank;
        if (volume(a.tr.size) == 0) return;

        // Home device of this rank
        int home = -1;
        if (comm) home = comm->device;
        for (const auto *bv : {&vr, &v0, &v1})
            for (const auto &b : *bv)
                if (home < 0 && !b.host && b.ptr) home = b.device;
        if (home < 0) home = default_device(comm);
        device_state(home);

        // every workspace of the call: staged operands, re-partitioned operand, partial results
        PoolGuard pool;
        Staged s0 = stage_in(v0, a.t0, me, es, home, pool);
        Staged s1 = stage_in(v1, a.t1, me, es, home, pool);
        Staged sr = stage_in(vr, a.tr, me, es, home, pool);

        // ---- 1. vr <- beta * vr on the output range, part by part, in place ---------------------------
        const bool beta_one = scalar_is(a.dtype, a.beta, 1);
        // (done below, after deciding whether the kernel epilogue can take care of beta)

        // ---- 2. items: the larger operand drives the decomposition -------------------------------------
        const bool big0 = volume(a.t0.size) >= volume(a.t1.size);
        const TensorArg &tb = big0 ? a.t0 : a.t1, &ts = big0 ? a.t1 : a.t0;
        const Staged &sb = big0 ? s0 : s1, &ss = big0 ? s1 : s0;
        std::vector<int> ident(tb.nd);
        for (int k = 0; k < tb.nd; ++k) ident[k] = k;

        std::vector<Item> items; // all ranks, ascending part
        if (volume(tb.size) > 0 && volume(ts.size) > 0) {
            std::vector<std::vector<RBox>> raw(tb.p.size());
            for (size_t i = 0; i < tb.p.size(); ++i) raw[i] = own_boxes(tb, tb.p[i]);
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

        // label lookups between tensors
        auto pos_in = [](const TensorArg &t, char c) {
            const auto p = t.o.find(c);
            return p == std::string::npos ? -1 : (int)p;
        };

        // Box of the other operand needed by an item: shared labels follow the item, private ones are full
        auto needed_small = [&](const Item &it, Coor &u, Coor &len) {
            u.assign(ts.nd, 0), len = ts.size;
            for (int k = 0; k < ts.nd; ++k) {
                const int kb = pos_in(tb, ts.o[k]);
                if (kb >= 0) u[k] = it.box.u[kb], len[k] = it.box.len[kb];
            }
        };
        // Output box of an item in o_r order
        auto output_box = [&](const Item &it, Coor &u, Coor &len) {
            u.assign(a.tr.nd, 0), len = a.tr.size;
            for (int k = 0; k < a.tr.nd; ++k) {
                const int kb = pos_in(tb, a.tr.o[k]);
                if (kb >= 0) u[k] = it.box.u[kb], len[k] = it.box.len[kb];
            }
        };

        // ---- 3. is the other operand already where every item needs it? ---------------------------------
        struct Found {
            int part = -1;
            RBox box;
        };
        std::vector<Found> small_at(items.size());
        bool inplace = true;
        for (size_t q = 0; q < items.size() && inplace; ++q) {
            const int r = items[q].part / tb.ncomp;
            Coor u, len;
            needed_small(items[q], u, len);
            bool ok = false;
            for (int c = 0; c < ts.ncomp && !ok; ++c) {
                const int part = r * ts.ncomp + c;
                for (const auto &b : own_boxes(ts, ts.p[part]))
                    if (contains(b, u, len)) {
                        small_at[q].part = part, small_at[q].box = b;
                        ok = true;
                        break;
                    }
            }
            if (!ok) inplace = false;
        }

        // my items
        std::vector<size_t> my;
        for (size_t q = 0; q < items.size(); ++q)
            if (items[q].part / tb.ncomp == me) my.push_back(q);
        std::vector<int> per_rank(a.nranks, 0);
        for (const auto &it : items) per_rank[it.part / tb.ncomp]++;
        const int max_items = items.empty() ? 0 : *std::max_element(per_rank.begin(), per_rank.end());

        // ---- 4. re-partition the other operand when needed ------------------------------------------------
        std::vector<View> small_view(items.size());
        if (!inplace && !items.empty()) {
            CopyArgs ca;
            ca.nd0 = ca.nd1 = ts.nd;
            ca.o0 = ca.o1 = ts.o;
            ca.p0 = ts.p, ca.ncomp0 = ts.ncomp;
            ca.from0 = ts.from, ca.size0 = ts.size, ca.dim0 = ts.dim;
            ca.from1.assign(ts.nd, 0), ca.dim1 = ts.size;
            ca.ncomp1 = max_items;
            ca.p1.assign((size_t)a.nranks * max_items, Box{Coor(ts.nd, 0), Coor(ts.nd, 0)});
            ca.nranks = a.nranks, ca.rank = me, ca.co = a.co;
            ca.wire_align = 16 / es;
            ca.chunk_bytes = exchange_chunk_bytes();
            std::vector<int> slot(a.nranks, 0);
            std::vector<Buffer> dst(max_items);
            for (size_t q = 0; q < items.size(); ++q) {
                const int r = items[q].part / tb.ncomp;
                Coor u, len;
                needed_small(items[q], u, len);
                const int c = slot[r]++;
                ca.p1[(size_t)r * max_items + c] = Box{u, len};
                if (r == me) {
                    const int dev = sb.dev[items[q].part % tb.ncomp].device;
                    void *t = pool.alloc(dev, (size_t)volume(len) * es);
                    dst[c].ptr = t, dst[c].device = dev, dst[c].host = false;
                    View &v = small_view[q];
                    v.ptr = (char *)t, v.device = dev, v.stride = get_strides(len, a.co), v.off = 0;
                }
            }
            // unused slots need a device for bookkeeping only
            for (auto &b : dst)
                if (!b.ptr) b.device = home;
            const double one[2] = {1, 0};
            auto plan = get_copy_plan(ca);
            execute_copy(*plan, ca, a.dtype, a.dtype, one, ss.dev, dst, comm);
        } else {
            for (size_t q : my) {
                const Found &f = small_at[q];
                const int c = f.part % ts.ncomp;
                View &v = small_view[q];
                v.ptr = (char *)ss.dev[c].ptr, v.device = ss.dev[c].device;
                v.stride = get_strides(ts.p[f.part].size, a.co);
                Coor u, len;
                needed_small(items[q], u, len);
                v.off = 0;
                for (int k = 0; k < ts.nd; ++k)
                    v.off += (int64_t)(f.box.lfrom[k] + u[k] - f.box.u[k]) * v.stride[k];
            }
        }

        // ---- 5. where does the result go? -------------------------------------------------------------------
        // Direct: a single item whose output box lies inside the only part that owns that range.
        bool direct = false;
        int direct_part = -1;
        RBox direct_box;
        if (items.size() == 1) {
            Coor u, len;
            output_box(items[0], u, len);
            int owners = 0;
            for (size_t i = 0; i < a.tr.p.size(); ++i)
                for (const auto &b : own_boxes(a.tr, a.tr.p[i])) {
                    Coor iu, il;
                    RBox want;
                    want.u = u, want.len = len;
                    if (intersect(b, want, iu, il)) {
                        ++owners;
                        if (contains(b, u, len)) direct_part = (int)i, direct_box = b;
                    }
                }
            direct = owners == 1 && direct_part >= 0 &&
                     direct_part / a.tr.ncomp == items[0].part / tb.ncomp;
        }

        // beta scaling of the output range (skipped when the epilogue applies beta itself)
        if (!direct && !beta_one) {
            for (int c = 0; c < a.tr.ncomp; ++c) {
                const int part = me * a.tr.ncomp + c;
                const auto strides = get_strides(a.tr.p[part].size, a.co);
                for (const auto &b : own_boxes(a.tr, a.tr.p[part])) {
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
                    const int dev = sr.dev[c].device;
                    use_device(dev);
                    permute_copy(d, sr.dev[c].ptr, a.dtype, sr.dev[c].ptr, a.dtype, a.beta, false, dev,
                                 device_state(dev).stream);
                }
            }
        }

        // ---- 6. local kernels ----------------------------------------------------------------------------------
        std::vector<Buffer> partial(max_items);
        for (auto &b : partial) b.device = home;
        CopyArgs ra; // reduction of the partial results
        if (!direct && !items.empty()) {
            ra.nd0 = ra.nd1 = a.tr.nd;
            ra.o0 = ra.o1 = a.tr.o;
            ra.ncomp0 = max_items;
            ra.p0.assign((size_t)a.nranks * max_items, Box{Coor(a.tr.nd, 0), Coor(a.tr.nd, 0)});
            ra.from0.assign(a.tr.nd, 0), ra.size0 = a.tr.size, ra.dim0 = a.tr.size;
            ra.p1 = a.tr.p, ra.ncomp1 = a.tr.ncomp, ra.from1 = a.tr.from, ra.dim1 = a.tr.dim;
            ra.nranks = a.nranks, ra.rank = me, ra.co = a.co, ra.add = true;
            ra.wire_align = 16 / es;
            ra.chunk_bytes = exchange_chunk_bytes();
            std::vector<int> slot(a.nranks, 0);
            for (size_t q = 0; q < items.size(); ++q) {
                const int r = items[q].part / tb.ncomp;
                Coor u, len;
                output_box(items[q], u, len);
                ra.p0[(size_t)r * max_items + slot[r]++] = Box{u, len};
            }
        }

        // several devices in this process: order their streams around the kernels
        std::set<int> devs{home};
        for (const auto *bv : {&s0.dev, &s1.dev, &sr.dev})
            for (const auto &b : *bv)
                if (b.ptr) devs.insert(b.device);
        order_streams(devs);

        int my_slot = 0;
        for (size_t q : my) {
            const Item &it = items[q];
            const int cb = it.part % tb.ncomp;
            const int dev = sb.dev[cb].device;
            const auto bstr = get_strides(tb.p[it.part].size, a.co);
            int64_t boff = 0;
            for (int k = 0; k < tb.nd; ++k) boff += (int64_t)it.box.lfrom[k] * bstr[k];
            const View &sv = small_view[q];
            enable_peer(dev, sv.device);

            // output view
            Coor ou, olen;
            output_box(it, ou, olen);
            View ov;
            if (direct) {
                const int c = direct_part % a.tr.ncomp;
                ov.ptr = (char *)sr.dev[c].ptr, ov.device = sr.dev[c].device;
                ov.stride = get_strides(a.tr.p[direct_part].size, a.co);
                for (int k = 0; k < a.tr.nd; ++k)
                    ov.off += (int64_t)(direct_box.lfrom[k] + ou[k] - direct_box.u[k]) * ov.stride[k];
                enable_peer(dev, ov.device);
            } else {
                void *t = pool.alloc(dev, (size_t)volume(olen) * es);
                ov.ptr = (char *)t, ov.device = dev, ov.stride = get_strides(olen, a.co);
                partial[my_slot].ptr = t, partial[my_slot].device = dev;
            }
            ++my_slot;

            sbk_contract_desc d;
            std::memset(&d, 0, sizeof d);
            d.conj0 = a.conj0, d.conj1 = a.conj1;
            for (const Label &l : labels) {
                sbk_contract_dim x;
                x.s0 = x.s1 = x.sr = 0;
                // extent of this label inside the item
                const int kb = pos_in(tb, l.c);
                x.size = kb >= 0 ? it.box.len[kb] : l.size;
                const int k_in_big = kb, k_in_small = pos_in(ts, l.c);
                const int64_t big_stride = k_in_big >= 0 ? bstr[k_in_big] : 0;
                const int64_t small_stride = k_in_small >= 0 ? sv.stride[k_in_small] : 0;
                x.s0 = big0 ? big_stride : small_stride;
                x.s1 = big0 ? small_stride : big_stride;
                x.sr = l.ir >= 0 ? ov.stride[l.ir] : 0;
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
            const char *bptr = (const char *)sb.dev[cb].ptr + boff * es;
            const char *sptr = sv.ptr + sv.off * es;
            const double zero[2] = {0, 0};
            use_device(dev);
            contract(d, a.dtype, a.alpha, big0 ? bptr : sptr, big0 ? sptr : bptr,
                     direct ? a.beta : zero, ov.ptr + ov.off * es, dev, device_state(dev).stream);
            {
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

        // ---- 7. add the partial results into the caller's partition ---------------------------------------------
        if (!direct && !items.empty()) {
            const double one[2] = {1, 0};
            auto plan = get_copy_plan(ra);
            execute_copy(*plan, ra, a.dtype, a.dtype, one, partial, sr.dev, comm);
        }

        // ---- 8. host results back (the workspace returns to the pool when `pool` ends) ---------------------------
        bool host_out = false;
        for (size_t c = 0; c < vr.size(); ++c)
            if (sr.temps[c]) {
                use_device(home);
                cuda_check(cudaMemcpyAsync(vr[c].ptr, sr.temps[c], sr.bytes[c], cudaMemcpyDeviceToHost,
                                           device_state(home).stream),
                           "cudaMemcpyAsync D2H");
                host_out = true;
            }
        if (host_out) cuda_check(cudaStreamSynchronize(device_state(home).stream), "sync");
    }

} // namespace sbb
