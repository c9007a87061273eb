// Driver of the batched dense solvers. See dense_plan.hpp.
#include "dense_plan.hpp"
#include <algorithm>
#include <cstring>
#include <set>
#include <sstream>

namespace sbb {

    namespace {

        const char *op_name(int op) {
            switch (op) {
            case SBB_CHOLESKY: return "cholesky";
            case SBB_INVERSION: return "inversion";
            case SBB_TRSM: return "trsm";
            case SBB_GESM: return "gesm";
            case SBB_EIGH: return "eigh";
            default: throw std::runtime_error("dense: unknown operation");
            }
        }

        bool solves(int op) { return op == SBB_TRSM || op == SBB_GESM; }

        /// A whole tensor: its extent along each label is max(from + size) over all parts
        void make_whole(TensorArg &t) {
            t.dim.assign(t.nd, 0);
            for (const Box &b : t.p)
                for (int k = 0; k < t.nd; ++k) t.dim[k] = std::max(t.dim[k], b.from[k] + b.size[k]);
            t.from.assign(t.nd, 0);
            t.size = t.dim;
        }

        /// Local offset of `need` inside the storage of `part` (strides `str`)
        int64_t offset_in(const Box &part, const Box &need, const std::vector<int64_t> &str) {
            int64_t off = 0;
            for (size_t k = 0; k < str.size(); ++k) off += (int64_t)(need.from[k] - part.from[k]) * str[k];
            return off;
        }

        bool contains(const Box &outer, const Box &b) {
            for (size_t k = 0; k < b.from.size(); ++k)
                if (b.from[k] < outer.from[k] || b.from[k] + b.size[k] > outer.from[k] + outer.size[k]) return false;
            return true;
        }

        bool same(const Box &a, const Box &b) { return a.from == b.from && a.size == b.size; }

        /// The part of `t` on rank r holding `need`, as (global part index), or -1
        int holder(const TensorArg &t, int r, const Box &need) {
            for (int c = 0; c < t.ncomp; ++c) {
                const Box &b = t.p[(size_t)r * t.ncomp + c];
                if (!b.empty() && contains(b, need)) return r * t.ncomp + c;
            }
            return -1;
        }
    }

    DensePlan make_dense_plan(const DenseArgs &in) {
        DenseArgs a = in;
        const std::string name = op_name(a.op);
        auto fail = [&](const std::string &m) { throw std::runtime_error(name + ": " + m); };
        check_float_dtype(a.dtype, name);
        const bool solve = solves(a.op), eigh = a.op == SBB_EIGH;
        std::vector<TensorArg *> ts{&a.a};
        if (solve) ts.push_back(&a.x), ts.push_back(&a.y);
        if (eigh) ts.push_back(&a.w);
        for (TensorArg *t : ts) {
            if ((int)t->p.size() != a.nranks * t->ncomp) throw std::runtime_error("wtf");
            if (!labels_unique(t->o)) fail("repeated label in an order");
            make_whole(*t);
        }
        if (!labels_unique(a.orows) || !labels_unique(a.ocols)) fail("repeated label in orows or ocols");
        for (char c : a.orows)
            if (label_pos(a.ocols, c) >= 0) fail(std::string("orows and ocols share the label `") + c + "`");
        for (const std::string *s : {&a.orows, &a.ocols})
            for (char c : *s)
                if (label_pos(a.a.o, c) < 0) fail(std::string("label `") + c + "` of orows / ocols is not in the matrix's order");
        const TensorArg &A = a.a;
        auto ext = [](const TensorArg &t, char c) { return t.dim[label_pos(t.o, c)]; };
        int64_t n = 1, ncols = 1;
        for (char c : a.orows) n *= ext(A, c);
        for (char c : a.ocols) ncols *= ext(A, c);
        if (n != ncols)
            fail("the matrix is not square: " + std::to_string(n) + " rows, " + std::to_string(ncols) + " columns");
        const int es = dtype_bytes(a.dtype);
        // cholesky and trsm of a larger matrix run the blocked tier of dense()
        const bool blocked = !densek::fits_cta(n, es);
        if (blocked && (a.op == SBB_GESM || a.op == SBB_INVERSION))
            fail("order n = " + std::to_string(n) +
                 " is over the limit: one matrix must fit in shared memory, n^2 * sizeof(T) <= 204800 bytes (n <= 113 "
                 "for complex double, 160 for double and complex float, 226 for float)");

        if (eigh && !densek::fits_eigh(n, es))
            fail("order n = " + std::to_string(n) +
                 " is over the limit: the matrix and its eigenvectors must fit in shared memory, 2 n^2 * sizeof(T) <= "
                 "204800 bytes (n <= 80 for complex double, 113 for double and complex float, 160 for float)");
        if (eigh) {
            // w: every batch and column label of the matrix with its extent, nothing else
            for (char c : A.o) {
                if (label_pos(a.orows, c) >= 0) continue;
                if (label_pos(a.w.o, c) < 0)
                    fail(std::string("w lacks the ") + (label_pos(a.ocols, c) >= 0 ? "column" : "batch") + " label `" +
                         c + "` of the matrix");
                if (ext(a.w, c) != ext(A, c)) fail(std::string("dimension of label `") + c + "` does not match");
            }
            for (char c : a.w.o)
                if (label_pos(A.o, c) < 0 || label_pos(a.orows, c) >= 0)
                    fail(std::string("w has the label `") + c + "`, which is neither a batch nor a column label of the matrix");
        }

        bool left = true;
        if (solve) {
            int nr = 0, nc = 0;
            for (char c : a.x.o) nr += label_pos(a.orows, c) >= 0, nc += label_pos(a.ocols, c) >= 0;
            left = nr == (int)a.orows.size() && nc == 0;
            const bool right = nc == (int)a.ocols.size() && nr == 0;
            if (!left && !right)
                fail("x must carry either every row label or every column label of the matrix, and no label of the "
                     "other set");
            const std::string &yvec = left ? a.ocols : a.orows;
            for (char c : A.o)
                if (label_pos(a.orows, c) < 0 && label_pos(a.ocols, c) < 0 && label_pos(a.x.o, c) < 0)
                    fail(std::string("x lacks the batch label `") + c + "` of the matrix");
            // y: the labels of x with the vector labels swapped, nothing else
            int expected = 0;
            for (char c : a.x.o) {
                const bool vec = label_pos(left ? a.orows : a.ocols, c) >= 0;
                if (!vec) {
                    ++expected;
                    if (label_pos(a.y.o, c) < 0) fail(std::string("y lacks the label `") + c + "` of x");
                    if (ext(a.y, c) != ext(a.x, c)) fail(std::string("dimension of label `") + c + "` does not match");
                }
                if (label_pos(A.o, c) >= 0 && ext(A, c) != ext(a.x, c))
                    fail(std::string("dimension of label `") + c + "` does not match");
            }
            for (char c : yvec) {
                if (label_pos(a.y.o, c) < 0) fail(std::string("y lacks the label `") + c + "` of the matrix");
                if (ext(a.y, c) != ext(A, c)) fail(std::string("dimension of label `") + c + "` does not match");
            }
            if ((int)a.y.o.size() != expected + (int)yvec.size())
                fail("y has a label that is neither in x nor a vector label of the matrix");
        }

        DensePlan plan;
        plan.op = a.op, plan.dtype = a.dtype;
        const TensorArg &D = solve ? a.y : a.a; // the output drives the items
        if (volume(D.dim) == 0) {
            plan.nothing = true;
            return plan;
        }

        // ---- items of every rank: one per non-empty output part -------------------------------------
        auto is_matrix = [&](char c) { return label_pos(a.orows, c) >= 0 || label_pos(a.ocols, c) >= 0; };
        // box of `t` an item driven by `part` of `drv` needs: matrix (vector) labels whole, the others as in
        // the part
        auto need_of = [&](const TensorArg &t, const TensorArg &drv, const Box &part) {
            Box b{Coor(t.nd, 0), t.dim};
            for (int k = 0; k < t.nd; ++k) {
                const int kd = label_pos(drv.o, t.o[k]);
                if (!is_matrix(t.o[k]) && kd >= 0) b.from[k] = part.from[kd], b.size[k] = part.size[kd];
            }
            return b;
        };
        struct Item {
            const TensorArg *drv; ///< the tensor of the part driving the item
            int part, slot = 0;
            Box na, nx, ny;       ///< eigh: ny is the box of W
            int ha = -1, hx = -1; ///< parts of A / X holding na / nx on the item's rank
            int hy = -1;          ///< eigh: the part of W that is exactly ny, written directly
            int writes = 0;
        };
        std::vector<Item> items;
        for (size_t i = 0; i < D.p.size(); ++i) {
            if (D.p[i].empty()) continue;
            Item it;
            it.drv = &D, it.part = (int)i;
            const int r = it.part / D.ncomp;
            it.na = need_of(A, D, D.p[i]);
            if (solve) {
                it.nx = need_of(a.x, D, D.p[i]);
                it.ny = need_of(a.y, D, D.p[i]);
                it.ha = holder(A, r, it.na);
                it.hx = holder(a.x, r, it.nx);
                plan.gather_x |= it.hx < 0;
            } else {
                it.ha = same(it.na, D.p[i]) ? (int)i : -1;
            }
            items.push_back(it);
        }
        if (eigh) {
            // W: the A item of a part's rank with exactly its batch box writes it; W-only items the rest
            const TensorArg &W = a.w;
            std::vector<char> served(W.p.size(), 0);
            for (Item &it : items) {
                it.writes = WRITES_A;
                it.ny = need_of(W, A, A.p[it.part]);
                const int r = it.part / A.ncomp;
                for (int c = 0; c < W.ncomp && it.hy < 0; ++c) {
                    const int k = r * W.ncomp + c;
                    if (!served[k] && !W.p[k].empty() && same(W.p[k], it.ny)) served[k] = 1, it.hy = k, it.writes |= WRITES_W;
                }
            }
            std::vector<Item> wonly;
            for (size_t i = 0; i < W.p.size(); ++i) {
                if (W.p[i].empty() || served[i]) continue;
                Item it;
                it.drv = &W, it.part = (int)i, it.writes = WRITES_W;
                it.na = need_of(A, W, W.p[i]);
                it.ny = need_of(W, W, W.p[i]);
                it.ha = holder(A, (int)i / W.ncomp, it.na);
                it.hy = same(it.ny, W.p[i]) ? (int)i : -1;
                wonly.push_back(it);
            }
            items.insert(items.begin(), wonly.begin(), wonly.end());
        }
        std::vector<int> per_rank(a.nranks, 0);
        for (Item &it : items) {
            it.slot = per_rank[it.part / it.drv->ncomp]++;
            plan.gather_a |= it.ha < 0;
        }
        plan.slots = *std::max_element(per_rank.begin(), per_rank.end());
        if (plan.gather_a) plan.a_args = gather_to_slots_args(A, plan.slots, a.nranks, a.rank, a.co, es);
        if (plan.gather_x) plan.x_args = gather_to_slots_args(a.x, plan.slots, a.nranks, a.rank, a.co, es);
        for (const Item &it : items) {
            const size_t at = (size_t)(it.part / it.drv->ncomp) * plan.slots + it.slot;
            if (plan.gather_a) plan.a_args.p1[at] = it.na;
            if (plan.gather_x) plan.x_args.p1[at] = it.nx;
        }

        // ---- the kernel of every item; every rank checks every item, so all ranks throw alike --------
        for (const Item &it : items) {
            const TensorArg &drv = *it.drv;
            DenseItem di;
            std::memset(&di.back, 0, sizeof di.back);
            di.comp = it.part % drv.ncomp, di.slot = it.slot, di.writes = it.writes;
            // storage of A, X and Y (eigh: W) for this item: (strides, offset)
            auto place = [&](const TensorArg &t, int held, const Box &need, bool gathered, int &comp, int64_t &off,
                             int64_t &elems) {
                comp = -1, off = 0, elems = volume(need.size);
                if (gathered || held < 0) return get_strides(need.size, a.co);
                comp = held % t.ncomp, elems = 0;
                const auto str = get_strides(t.p[held].size, a.co);
                off = offset_in(t.p[held], need, str);
                return str;
            };
            const auto sa = place(A, it.ha, it.na, plan.gather_a, di.a_comp, di.a_off, di.a_elems);
            std::vector<int64_t> sx, sy;
            di.x_comp = di.y_comp = -1, di.x_off = di.y_off = di.x_elems = di.y_elems = 0;
            if (solve) {
                sx = place(a.x, it.hx, it.nx, plan.gather_x, di.x_comp, di.x_off, di.x_elems);
                const bool direct = same(it.ny, D.p[it.part]);
                sy = place(a.y, direct ? it.part : -1, it.ny, false, di.y_comp, di.y_off, di.y_elems);
            }
            if (eigh && it.writes != WRITES_A) sy = place(a.w, it.hy, it.ny, false, di.y_comp, di.y_off, di.y_elems);
            // the output on a temporary: its own box goes back into the part
            const Box &nd = solve || it.writes == WRITES_W ? it.ny : it.na;
            di.write_back = solve ? di.y_comp < 0 : it.writes == WRITES_W ? di.y_comp < 0 : plan.gather_a;
            if (di.write_back) {
                const auto tstr = get_strides(nd.size, a.co);
                const auto pstr = get_strides(drv.p[it.part].size, a.co);
                sbk_box_desc &b = di.back;
                b.nd = drv.nd;
                for (int k = 0; k < drv.nd; ++k)
                    b.size[k] = drv.p[it.part].size[k], b.sstride[k] = tstr[k], b.dstride[k] = pstr[k];
                b.soff = offset_in(nd, drv.p[it.part], tstr), b.doff = 0;
            }

            sbk_dense_desc &d = di.desc;
            std::memset(&d, 0, sizeof d);
            d.op = a.op, d.n = (int)n, d.left = left, d.vectors = (it.writes & WRITES_A) != 0;
            auto dim_of = [&](char c, int size) {
                sbk_dense_dim x;
                x.size = size;
                const int ka = label_pos(A.o, c), kx = solve ? label_pos(a.x.o, c) : -1;
                const int ky = solve ? label_pos(a.y.o, c) : eigh && !sy.empty() ? label_pos(a.w.o, c) : -1;
                x.sa = ka >= 0 ? sa[ka] : 0;
                x.sx = kx >= 0 ? sx[kx] : 0;
                x.sy = ky >= 0 ? sy[ky] : 0;
                return x;
            };
            auto add = [&](sbk_dense_dim *g, int &ng, const sbk_dense_dim &x) {
                if (x.size == 1) return;
                if (ng >= SBK_MAX_GROUP_DIMS) fail("too many labels in a group");
                g[ng++] = x;
            };
            for (const std::string *s : {&a.orows, &a.ocols}) {
                std::string o = *s;
                if (a.co == SlowToFast) std::reverse(o.begin(), o.end()); // first listed label fastest
                for (char c : o)
                    s == &a.orows ? add(d.rows, d.nrows, dim_of(c, ext(A, c))) : add(d.cols, d.ncols, dim_of(c, ext(A, c)));
            }
            for (int k = 0; k < A.nd; ++k)
                if (!is_matrix(A.o[k])) add(d.batch, d.nbatch, dim_of(A.o[k], it.na.size[k]));
            if (solve)
                for (int k = 0; k < a.x.nd; ++k)
                    if (label_pos(A.o, a.x.o[k]) < 0) add(d.rhs, d.nrhs, dim_of(a.x.o[k], it.nx.size[k]));
            // batch entries and right-hand sides in any order: the smallest stride first, for coalescing
            std::stable_sort(d.batch, d.batch + d.nbatch, [](const sbk_dense_dim &u, const sbk_dense_dim &v) { return u.sa < v.sa; });
            std::stable_sort(d.rhs, d.rhs + d.nrhs, [](const sbk_dense_dim &u, const sbk_dense_dim &v) { return u.sx < v.sx; });
            // the blocked tier moves the matrices, X and Y with one box each (a dimension per label)
            const int wdims = d.nrows + d.ncols + d.nbatch, vdims = std::max(d.nrows, d.ncols) + d.nrhs + d.nbatch;
            if (blocked && std::max(wdims, solve ? vdims : 0) > SBK_MAX_DIMS)
                fail("a matrix over the shared-memory limit is gathered with one dimension per row, column, batch "
                     "(and right-hand-side) label: " + std::to_string(std::max(wdims, solve ? vdims : 0)) +
                     " labels of extent > 1 are more than " + std::to_string(SBK_MAX_DIMS));
            if (it.part / drv.ncomp == a.rank) plan.items.push_back(di), plan.w_only += it.writes == WRITES_W;
        }
        return plan;
    }

    std::string DensePlan::describe() const {
        std::stringstream ss;
        ss << "dense " << op_name(op) << " nothing " << nothing << " gather_a " << gather_a << " gather_x "
           << gather_x << " slots " << slots << "\n";
        const double one[2] = {1, 0};
        for (const auto &it : items) {
            const sbk_dense_desc &d = it.desc;
            ss << "item comp " << it.comp << " a " << it.a_comp << " " << it.a_off << " " << it.a_elems << " x "
               << it.x_comp << " " << it.x_off << " " << it.x_elems << " y " << it.y_comp << " " << it.y_off << " "
               << it.y_elems << " slot " << it.slot << " left " << d.left << " n " << d.n;
            const struct {
                const char *name;
                int n;
                const sbk_dense_dim *dims;
            } groups[] = {{"R", d.nrows, d.rows}, {"C", d.ncols, d.cols}, {"B", d.nbatch, d.batch}, {"H", d.nrhs, d.rhs}};
            for (const auto &g : groups) {
                ss << " " << g.name;
                for (int i = 0; i < g.n; ++i)
                    ss << " " << g.dims[i].size << " " << g.dims[i].sa << " " << g.dims[i].sx << " " << g.dims[i].sy;
            }
            if (op == SBB_EIGH) ss << " writes " << (it.writes & WRITES_A ? "a" : "") << (it.writes & WRITES_W ? "w" : "");
            std::string k;
            dense(d, dtype, one, nullptr, nullptr, nullptr, nullptr, &k);
            ss << "\nkernel " << k << "\n";
            if (it.write_back) {
                const sbk_box_desc &b = it.back;
                ss << "back comp " << it.comp << " soff " << b.soff << " size";
                for (int i = 0; i < b.nd; ++i) ss << " " << b.size[i];
                ss << " sstride";
                for (int i = 0; i < b.nd; ++i) ss << " " << b.sstride[i];
                ss << " dstride";
                for (int i = 0; i < b.nd; ++i) ss << " " << b.dstride[i];
                ss << "\n";
            }
        }
        if (gather_a) ss << "gather_a\n" << make_copy_plan(a_args)->describe();
        if (gather_x) ss << "gather_x\n" << make_copy_plan(x_args)->describe();
        return ss.str();
    }

    DenseSteps dense_steps(const DensePlan &plan) {
        DenseSteps s;
        // gather k fills slot `slot` from this rank's own parts alone: no unpack writes into it
        auto local_slots = [&](const CopyArgs &ca) {
            std::vector<char> local(plan.slots, 1);
            for (const BoxOp &op : get_copy_plan(ca)->ops)
                if (op.kind == BoxOp::Unpack) local[op.dst_comp] = 0;
            return local;
        };
        std::vector<char> la, lx;
        int ka = -1, kx = -1;
        if (plan.gather_a) ka = s.exchanges++, la = local_slots(plan.a_args);
        if (plan.gather_x) kx = s.exchanges++, lx = local_slots(plan.x_args);
        for (const DenseItem &it : plan.items) {
            int k = 0;
            if (ka >= 0) k = std::max(k, la[it.slot] ? ka : ka + 1);
            if (kx >= 0) k = std::max(k, lx[it.slot] ? kx : kx + 1);
            s.step.push_back(k);
        }
        return s;
    }

    std::string DenseSteps::describe() const {
        std::stringstream ss;
        ss << "steps " << exchanges + 1 << " exchanges " << exchanges << "\n";
        for (size_t i = 0; i < step.size(); ++i) ss << "item " << i << " step " << step[i] << "\n";
        return ss.str();
    }

    namespace {
        /// A dense call in steps, one exchange each (driver.hpp, StepRequest; the steps of dense_steps).
        /// The kernels of an item, their arithmetic and the work counted are those of the call without a
        /// request; only the step that queues them differs, so the results are bit-identical.
        class DenseExec : public StepRequest {
        public:
            DenseExec(const DenseArgs &a, const std::vector<Buffer> &va, const std::vector<Buffer> &vx,
                      const std::vector<Buffer> &vy, const std::vector<Buffer> &vw, Comm *comm)
                : StepRequest(op_name(a.op)), a(a), va(va), vx(vx), vy(vy), vw(vw), comm(comm) {}

            void begin() {
                plan = make_dense_plan(a);
                if (plan.nothing) return; // complete at the first progress()
                steps = dense_steps(plan);
                solve = solves(a.op), eigh = a.op == SBB_EIGH;
                es = dtype_bytes(a.dtype);
                // ---- home device of this rank, host components staged on it -------------------------------
                home = home_device(comm, {&vy, &va, &vx, &vw}, default_device(comm));
                sa = stage_in(va, a.a, a.rank, es, home, pool);
                if (solve) sx = stage_in(vx, a.x, a.rank, es, home, pool), sy = stage_in(vy, a.y, a.rank, es, home, pool);
                if (eigh) sw = stage_in(vw, a.w, a.rank, dtype_bytes(real_dtype()), home, pool);
                devs = call_devices(home, {&sa, &sx, &sy, &sw});
                // ---- gather slots: whole matrices (and vectors), one per item, on the item's device ----------
                auto slots = [&](bool on, int64_t DenseItem::*elems) {
                    if (!on) return std::vector<Buffer>(plan.slots);
                    std::vector<SlotNeed> need;
                    for (const auto &it : plan.items) need.push_back({it.slot, out(it).dev[it.comp].device, it.*elems});
                    return alloc_slots(plan.slots, need, es, home, pool);
                };
                aslot = slots(plan.gather_a, &DenseItem::a_elems);
                xslot = slots(plan.gather_x, &DenseItem::x_elems);
                progress();
            }

        private:
            const DenseArgs a;
            const std::vector<Buffer> va, vx, vy, vw;
            Comm *comm;
            DensePlan plan;
            DenseSteps steps;
            bool solve = false, eigh = false;
            int es = 0, home = 0, k = 0; ///< k: the step to take next
            PoolGuard pool;
            Staged sa, sx, sy, sw;
            std::set<int> devs;
            std::vector<Buffer> aslot, xslot;

            /// The staged tensor of the item's output part
            const Staged &out(const DenseItem &it) const { return solve ? sy : it.writes == WRITES_W ? sw : sa; }
            /// eigh: the element type of W
            int real_dtype() const { return a.dtype == SBB_C64 ? SBB_F32 : a.dtype == SBB_C128 ? SBB_F64 : a.dtype; }

            /// Begin the next gather and queue the items of this step
            bool step() override {
                if (plan.nothing) return true;
                if (k < steps.exchanges) {
                    const bool ga = k == 0 && plan.gather_a;
                    begin_exchange(ga ? plan.a_args : plan.x_args, a.dtype, ga ? sa.dev : sx.dev, ga ? aslot : xslot,
                                   comm);
                }
                launch(k);
                if (k++ < steps.exchanges) return false;
                // ---- host results back ------------------------------------------------------------------
                stage_out(solve ? vy : va, solve ? sy : sa, home);
                if (eigh) stage_out(vw, sw, home);
                pool.release();
                return true;
            }

            /// The items of step `s`, behind the local part of the gather in flight; several devices in this
            /// process: their streams ordered around them
            void launch(int s) {
                if (std::find(steps.step.begin(), steps.step.end(), s) == steps.step.end()) return;
                wait_local();
                order_streams(devs);
                const double one[2] = {1, 0};
                for (size_t i = 0; i < plan.items.size(); ++i) {
                    if (steps.step[i] != s) continue;
                    // W-only items read A in place before the other items of the rank overwrite it
                    if (i > 0 && (int)i == plan.w_only) order_streams(devs);
                    const DenseItem &it = plan.items[i];
                    const Buffer &o = out(it).dev[it.comp];
                    const int dev = o.device;
                    auto at = [&](int comp, int64_t off, const Staged &st, const std::vector<Buffer> &slot) -> char * {
                        const Buffer &b = comp >= 0 ? st.dev[comp] : slot[it.slot];
                        enable_peer(dev, b.device);
                        return (char *)b.ptr + (comp >= 0 ? off * es : 0);
                    };
                    char *pa = at(it.a_comp, it.a_off, sa, aslot);
                    char *px = solve ? at(it.x_comp, it.x_off, sx, xslot) : nullptr;
                    char *py = nullptr;
                    const int yt = eigh ? real_dtype() : a.dtype, yes = dtype_bytes(yt);
                    if (solve || (it.writes & WRITES_W)) {
                        const Buffer &yb = solve ? o : sw.dev[it.y_comp >= 0 ? it.y_comp : it.comp];
                        if (it.y_comp >= 0) enable_peer(dev, yb.device);
                        py = it.y_comp >= 0 ? (char *)yb.ptr + it.y_off * yes
                                            : (char *)pool.alloc(dev, (size_t)it.y_elems * yes);
                    }
                    use_device(dev);
                    const cudaStream_t stream = device_state(dev).stream;
                    dense(it.desc, a.dtype, a.alpha, pa, px, py, stream);
                    if (it.write_back) {
                        const bool y_out = solve || it.writes == WRITES_W;
                        permute_copy(it.back, y_out ? py : pa, y_out ? yt : a.dtype, o.ptr, y_out ? yt : a.dtype, one,
                                     false, dev, stream);
                    }
                    if (eigh) {
                        const sbk_dense_desc &d = it.desc;
                        double nb = 1;
                        for (int j = 0; j < d.nbatch; ++j) nb *= d.batch[j].size;
                        const double n = d.n;
                        work_counters().bytes += ((d.vectors ? 2 : 1) * n * n * es + (py ? n * yes : 0)) * nb;
                    } else {
                        const sbk_dense_desc &d = it.desc;
                        double nb = 1, nr = 1;
                        for (int j = 0; j < d.nbatch; ++j) nb *= d.batch[j].size;
                        for (int j = 0; j < d.nrhs; ++j) nr *= d.rhs[j].size;
                        const double n = d.n, cplx = (a.dtype == SBB_C64 || a.dtype == SBB_C128) ? 4 : 1;
                        const double flops = a.op == SBB_CHOLESKY    ? n * n * n / 3
                                             : a.op == SBB_INVERSION ? 2 * n * n * n
                                             : a.op == SBB_TRSM      ? n * n * nr
                                                                     : 2 * n * n * n / 3 + 2 * n * n * nr;
                        work_counters().flops += cplx * flops * nb;
                        work_counters().bytes += (solve ? n * n + 2 * n * nr : 2 * n * n) * nb * es;
                    }
                }
                order_streams(devs);
            }
        };
    }

    std::unique_ptr<Request> begin_dense(const DenseArgs &a, const std::vector<Buffer> &va,
                                         const std::vector<Buffer> &vx, const std::vector<Buffer> &vy,
                                         const std::vector<Buffer> &vw, Comm *comm) {
        std::unique_ptr<DenseExec> e(new DenseExec(a, va, vx, vy, vw, comm));
        e->begin();
        return e;
    }

} // namespace sbb
