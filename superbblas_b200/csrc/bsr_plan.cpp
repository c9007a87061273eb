// Distributed block-sparse operators. See bsr_plan.hpp.
#include "bsr_plan.hpp"
#include <algorithm>
#include <cstring>
#include <numeric>
#include <set>
#include <sstream>

namespace sbb {

    namespace {

        bool overlap(const Box &a, const Box &b) {
            if (a.empty() || b.empty()) return false;
            for (size_t k = 0; k < a.from.size(); ++k)
                if (a.from[k] + a.size[k] <= b.from[k] || b.from[k] + b.size[k] <= a.from[k]) return false;
            return true;
        }

        /// The dimension indices of an order, fastest first
        std::vector<int> fastest_first(int n, int co) {
            std::vector<int> r(n);
            for (int k = 0; k < n; ++k) r[k] = co == FastToSlow ? k : n - 1 - k;
            return r;
        }

        /// Shortest periodic arc of a ring of `d` sites covering every marked site: {from, size}
        std::pair<int, int> shortest_arc(const std::vector<char> &covered) {
            const int d = (int)covered.size();
            int c0 = -1;
            for (int i = 0; i < d && c0 < 0; ++i)
                if (covered[i]) c0 = i;
            if (c0 < 0) return {0, 0};
            int best = 0, best_start = 0, run = 0, start = 0;
            for (int s = 1; s <= d; ++s) { // from just after c0 round to c0 itself
                const int i = (c0 + s) % d;
                if (!covered[i]) {
                    if (run == 0) start = i;
                    if (++run > best) best = run, best_start = start;
                } else {
                    run = 0;
                }
            }
            if (best == 0) return {0, d};
            return {(best_start + best) % d, d - best};
        }
    }

    Coor BsrShape::effim() const {
        Coor r = blockim;
        for (int k = 0; k < ni; ++k) r[k] *= kronim[k];
        return r;
    }

    Coor BsrShape::effdom() const {
        Coor r = blockdom;
        for (int k = 0; k < nd; ++k) r[k] *= krondom[k];
        return r;
    }

    void check_bsr_shape(const BsrShape &s) {
        const std::string name = s.name();
        auto fail = [&](const std::string &m) { throw std::runtime_error(name + ": " + m); };
        check_float_dtype(s.dtype, name.c_str());
        if (s.ni > SBK_MAX_DIMS || s.nd > SBK_MAX_DIMS) fail("too many dimensions");
        if ((int)s.pim.size() != s.nranks * s.ncomp || (int)s.pdom.size() != s.nranks * s.ncomp)
            throw std::runtime_error("wtf");
        for (int k = 0; k < s.ni; ++k)
            if (s.blockim[k] < 1 || s.dimi[k] < 0) fail("blockim must be positive");
        for (int k = 0; k < s.nd; ++k)
            if (s.blockdom[k] < 1 || s.dimd[k] < 0) fail("blockdom must be positive");
        for (int k = 0; k < s.ni; ++k) {
            if (s.kronim[k] < 1) fail("kronim must be positive");
            if (s.kronim[k] > 1 && s.blockim[k] > 1) fail("kronim and blockim exceed 1 along the same image label");
        }
        for (int k = 0; k < s.nd; ++k) {
            if (s.krondom[k] < 1) fail("krondom must be positive");
            if (s.krondom[k] > 1 && s.blockdom[k] > 1) fail("krondom and blockdom exceed 1 along the same domain label");
        }
        const Coor bim = s.effim();
        for (const Box &b : s.pim) {
            if (b.empty()) continue;
            for (int k = 0; k < s.ni; ++k) {
                if (b.from[k] < 0 || b.from[k] + b.size[k] > s.dimi[k])
                    fail("an image part does not fit in the image lattice");
                if (b.from[k] % bim[k] != 0 || b.size[k] % bim[k] != 0)
                    fail(std::string("the from and size of every image part must be multiples of ") +
                         (s.kron ? "blockim * kronim" : "blockim"));
            }
        }
        int64_t covered = 0;
        for (size_t i = 0; i < s.pim.size(); ++i) {
            for (size_t j = 0; j < i; ++j)
                if (overlap(s.pim[i], s.pim[j])) fail("image parts overlap");
            covered += s.pim[i].empty() ? 0 : volume(s.pim[i].size);
        }
        if (covered != volume(s.dimi)) fail("the image parts must cover the image lattice");
    }

    int64_t bsr_rows(const BsrShape &s, const Box &part) {
        if (part.empty()) return 0;
        const Coor bim = s.effim();
        int64_t n = 1;
        for (int k = 0; k < s.ni; ++k) n *= part.size[k] / bim[k];
        return n;
    }

    namespace {
        /// Throws the message of an error code of BsrPart
        [[noreturn]] void bsr_error(const BsrShape &s, int code) {
            const std::string name = s.name(), block = s.kron ? "blockdom * krondom" : "blockdom";
            switch (code) {
            case 1: throw std::runtime_error(name + ": a block's domain coordinate (jj) is not a multiple of " + block);
            case 2:
                throw std::runtime_error(name + ": a block wraps around the domain lattice: (jj mod dimd) + " + block +
                                         " > dimd");
            case 3: throw std::runtime_error(name + ": negative number of blocks in a row (ii)");
            case 4:
                throw std::runtime_error(name + ": every block row of every component, on every rank, must have the "
                                                "same number of blocks (ii)");
            default: throw std::runtime_error(name + ": another rank failed");
            }
        }

        /// Ints per part in the create-time exchange: error code, halo from, halo size and, for a
        /// Kronecker operator, the blocks of every row (-1 without rows)
        int bsr_row_width(const BsrShape &s) { return 1 + 2 * s.nd + (s.kron ? 1 : 0); }

        /// Appends the exchange row of a part to `rows`
        void append_bsr_row(const BsrShape &s, const BsrPart &p, std::vector<int> &rows) {
            rows.push_back(p.error);
            rows.insert(rows.end(), p.halo.from.begin(), p.halo.from.end());
            rows.insert(rows.end(), p.halo.size.begin(), p.halo.size.end());
            if (s.kron) rows.push_back(p.u);
        }

        /// Every part's halo box from the exchange rows of all parts ([rank][component]), or the error:
        /// the first part's error code, then (Kronecker) parts with rows whose block counts differ
        std::vector<Box> bsr_halo(const BsrShape &s, const std::vector<int> &rows) {
            const size_t K = bsr_row_width(s), n = rows.size() / K;
            for (size_t q = 0; q < n; ++q)
                if (rows[q * K]) bsr_error(s, rows[q * K]);
            int u = -1;
            for (size_t q = 0; q < n && s.kron; ++q) {
                const int uq = rows[q * K + K - 1];
                if (uq < 0) continue;
                if (u >= 0 && uq != u) bsr_error(s, 4);
                u = uq;
            }
            std::vector<Box> halo;
            for (size_t q = 0; q < n; ++q) {
                const int *m = &rows[q * K];
                halo.push_back(Box{Coor(m + 1, m + 1 + s.nd), Coor(m + 1 + s.nd, m + 1 + 2 * s.nd)});
            }
            return halo;
        }
    }

    BsrPart make_bsr_part(const BsrShape &s, const Box &part, const int *ii, const int *jj) {
        BsrPart p;
        p.halo = Box{Coor(s.nd, 0), Coor(s.nd, 0)};
        const int64_t rows = bsr_rows(s, part);
        p.rowptr.assign(rows + 1, 0);
        for (int64_t r = 0; r < rows; ++r) {
            if (ii[r] < 0) {
                p.error = 3;
                return p;
            }
            p.rowptr[r + 1] = p.rowptr[r] + ii[r];
        }
        if (s.kron && rows > 0) {
            for (int64_t r = 0; r < rows; ++r)
                if (ii[r] != ii[0]) {
                    p.error = 4;
                    return p;
                }
            p.u = ii[0];
        }
        const int64_t nnz = p.rowptr[rows];
        const Coor bdom = s.effdom();
        std::vector<std::vector<char>> cov(s.nd);
        for (int k = 0; k < s.nd; ++k) cov[k].assign(s.dimd[k], 0);
        std::vector<int> jm((size_t)nnz * s.nd);
        for (int64_t b = 0; b < nnz; ++b)
            for (int k = 0; k < s.nd; ++k) {
                const int d = s.dimd[k], j = ((jj[b * s.nd + k] % d) + d) % d;
                if (j % bdom[k] != 0) p.error = std::max(p.error, 1);
                else if (j + bdom[k] > d) p.error = std::max(p.error, 2);
                else std::fill(cov[k].begin() + j, cov[k].begin() + j + bdom[k], 1);
                jm[b * s.nd + k] = j;
            }
        if (p.error) return p;
        if (nnz > 0)
            for (int k = 0; k < s.nd; ++k) {
                const auto arc = shortest_arc(cov[k]);
                p.halo.from[k] = arc.first, p.halo.size[k] = arc.second;
            }
        const auto hs = get_strides(p.halo.size, s.co);
        p.goff.assign(nnz, 0);
        for (int64_t b = 0; b < nnz; ++b)
            for (int k = 0; k < s.nd; ++k) {
                const int d = s.dimd[k];
                p.goff[b] += (int64_t)(((jm[b * s.nd + k] - p.halo.from[k]) % d + d) % d) * hs[k];
            }
        return p;
    }

    BsrGeometry bsr_geometry_from_all(const BsrShape &s, const int *ii_all, const int *jj_all) {
        check_bsr_shape(s);
        BsrGeometry g;
        g.s = s;
        std::vector<int> rows;
        for (size_t q = 0; q < s.pim.size(); ++q) {
            BsrPart p = make_bsr_part(s, s.pim[q], ii_all, jj_all);
            const int64_t nrows = bsr_rows(s, s.pim[q]);
            int64_t nnz = 0;
            for (int64_t r = 0; r < nrows; ++r) nnz += std::max(ii_all[r], 0);
            ii_all += nrows;
            jj_all += nnz * s.nd;
            append_bsr_row(s, p, rows);
            if ((int)q / s.ncomp == s.rank) g.mine.push_back(std::move(p));
        }
        g.halo = bsr_halo(s, rows);
        return g;
    }

    BsrPlan make_bsr_plan(const BsrGeometry &g, const BsrCall &c) {
        auto fail = [](const std::string &m) { throw std::runtime_error("bsr_krylov: " + m); };
        const BsrShape &s = g.s;
        check_float_dtype(c.dtype, "bsr_krylov");
        if (c.dtype != s.dtype) fail("the element type differs from the operator's");
        if ((int)c.oim.size() != s.ni || (int)c.odom.size() != s.nd)
            fail("oim and odom must have as many labels as the image and domain lattices have dimensions");
        if (c.nranks != s.nranks) fail("the communicator differs from the operator's");
        const TensorArg &x = c.x, &y = c.y;
        for (const TensorArg *t : {&x, &y})
            if ((int)t->p.size() != c.nranks * t->ncomp) throw std::runtime_error("wtf");
        if (!labels_unique(c.oim) || !labels_unique(c.odom) || !labels_unique(x.o) || !labels_unique(y.o))
            fail("repeated label in an order");
        for (const TensorArg *t : {&x, &y})
            for (int k = 0; k < t->nd; ++k)
                if (t->size[k] < 0 || t->size[k] > t->dim[k]) fail("range larger than the tensor");
        auto whole = [&](const TensorArg &t, const std::string &o, const Coor &dim, const char *what) {
            for (size_t k = 0; k < o.size(); ++k) {
                const int p = label_pos(t.o, o[k]);
                if (p < 0) fail(std::string(what) + " lacks the label `" + o[k] + "` of the operator");
                if (t.dim[p] != dim[k]) fail(std::string("dimension of label `") + o[k] + "` does not match");
                if (t.from[p] != 0 || t.size[p] != dim[k])
                    fail(std::string("the operator acts on whole lattices: from must be 0 and size the dimension "
                                     "along label `") + o[k] + "`");
            }
        };
        whole(x, c.odom, s.dimd, "x");
        whole(y, c.oim, s.dimi, "y");
        int P = 1;
        const int ypp = c.power ? label_pos(y.o, c.power) : -1;
        if (c.power) {
            if (label_pos(x.o, c.power) >= 0) fail("x must not carry the power label");
            if (ypp < 0) fail(std::string("y lacks the power label `") + c.power + "`");
            if (label_pos(c.oim, c.power) >= 0 || label_pos(c.odom, c.power) >= 0) fail("the power label is an operator label");
            P = y.size[ypp];
        }
        std::string cols;
        for (int k = 0; k < x.nd; ++k) {
            const char l = x.o[k];
            if (label_pos(c.odom, l) >= 0) continue;
            if (label_pos(c.oim, l) >= 0) fail(std::string("column label `") + l + "` of x is an image label");
            const int py = label_pos(y.o, l);
            if (py < 0) fail(std::string("y lacks the column label `") + l + "` of x");
            if (y.size[py] != x.size[k]) fail(std::string("dimension of label `") + l + "` does not match");
            cols += l;
        }
        for (char l : y.o)
            if (label_pos(c.oim, l) < 0 && label_pos(cols, l) < 0 && l != c.power)
                fail(std::string("y has the label `") + l + "`, which is neither an image label, a column label of x "
                                                             "nor the power label");
        if (P > 1 && (s.ni != s.nd || s.dimi != s.dimd))
            fail("powers above 1 need the same image and domain lattices");

        BsrPlan plan;
        plan.odom = c.odom;
        plan.powers = P;
        plan.kron = s.kron;
        int64_t ncols = 1;
        Coor csize;
        for (char l : cols) csize.push_back(x.size[label_pos(x.o, l)]), ncols *= csize.back();
        if (ncols == 0 || P == 0 || volume(s.dimi) == 0) {
            plan.nothing = true;
            return plan;
        }
        const int es = dtype_bytes(c.dtype), ncomp = s.ncomp;
        plan.slots = ncomp;

        // ---- direct: y's parts are the image parts, with every column and power -------------------
        bool direct = y.ncomp == ncomp;
        for (size_t q = 0; q < y.p.size() && direct; ++q) {
            const Box &yp = y.p[q], &ip = s.pim[q];
            if (ip.empty() || yp.empty()) {
                direct = ip.empty() && yp.empty();
                continue;
            }
            for (int k = 0; k < y.nd && direct; ++k) {
                const int ki = label_pos(c.oim, y.o[k]);
                if (ki >= 0) direct = yp.from[k] == ip.from[ki] && yp.size[k] == ip.size[ki];
                else direct = yp.from[k] <= y.from[k] && y.from[k] + y.size[k] <= yp.from[k] + yp.size[k];
            }
        }
        plan.direct = direct;

        // ---- the gathered input: columns fastest, then the domain labels of the halo box -----------
        const std::string og = s.co == FastToSlow ? cols + c.odom : c.odom + cols;
        Coor gdim;
        for (char l : og) gdim.push_back(label_pos(cols, l) >= 0 ? csize[label_pos(cols, l)] : s.dimd[label_pos(c.odom, l)]);
        auto gather_box = [&](const Box &halo) {
            Box b{Coor(og.size(), 0), Coor(og.size(), 0)};
            if (halo.empty()) return b;
            for (size_t k = 0; k < og.size(); ++k) {
                const int kc = label_pos(cols, og[k]), kd = label_pos(c.odom, og[k]);
                if (kc >= 0) b.size[k] = csize[kc];
                else b.from[k] = halo.from[kd], b.size[k] = halo.size[kd];
            }
            return b;
        };
        auto gather_to = [&](CopyArgs &ca) {
            ca.nd1 = (int)og.size(), ca.o1 = og, ca.ncomp1 = ncomp;
            ca.from1.assign(og.size(), 0), ca.dim1 = gdim;
            for (const Box &h : g.halo) ca.p1.push_back(gather_box(h));
        };
        plan.gather_x = copy_args(c.nranks, c.rank, s.co, es);
        {
            CopyArgs &ca = plan.gather_x;
            ca.nd0 = x.nd, ca.o0 = x.o, ca.p0 = x.p, ca.ncomp0 = x.ncomp;
            ca.from0 = x.from, ca.size0 = x.size, ca.dim0 = x.dim;
            gather_to(ca);
        }
        if (P > 1) {
            CopyArgs &ca = plan.gather_y;
            ca = copy_args(c.nranks, c.rank, s.co, es);
            ca.nd0 = y.nd, ca.o0 = y.o, ca.p0 = y.p, ca.ncomp0 = y.ncomp;
            for (char &l : ca.o0)
                if (label_pos(c.oim, l) >= 0) l = c.odom[label_pos(c.oim, l)]; // y_{p-1} read as an input
            ca.from0 = y.from, ca.size0 = y.size, ca.dim0 = y.dim;
            ca.size0[ypp] = 1;
            gather_to(ca);
        }
        plan.y_power_pos = ypp;

        // ---- temporaries and their way back into y ----------------------------------------------------
        const std::string ot = s.co == FastToSlow ? cols + c.oim : c.oim + cols;
        auto temp_box = [&](const Box &ip) {
            Box b{Coor(ot.size(), 0), Coor(ot.size(), 0)};
            if (ip.empty()) return b;
            for (size_t k = 0; k < ot.size(); ++k) {
                const int kc = label_pos(cols, ot[k]), ki = label_pos(c.oim, ot[k]);
                if (kc >= 0) b.size[k] = csize[kc];
                else b.from[k] = ip.from[ki], b.size[k] = ip.size[ki];
            }
            return b;
        };
        if (!direct) { // temporaries: columns fastest, then oim over the image box of the part
            CopyArgs &ca = plan.back;
            ca = copy_args(c.nranks, c.rank, s.co, es);
            ca.nd0 = (int)ot.size(), ca.o0 = ot, ca.ncomp0 = ncomp;
            for (const Box &ip : s.pim) ca.p0.push_back(temp_box(ip));
            ca.from0.assign(ot.size(), 0);
            for (char l : ot) ca.dim0.push_back(label_pos(cols, l) >= 0 ? csize[label_pos(cols, l)] : s.dimi[label_pos(c.oim, l)]);
            ca.size0 = ca.dim0;
            ca.nd1 = y.nd, ca.o1 = y.o, ca.p1 = y.p, ca.ncomp1 = y.ncomp;
            ca.from1 = y.from, ca.dim1 = y.dim;
            // y_p into the temporaries first, so that the kernel's epilogue applies beta as it does in y
            plan.fill_temps = !scalar_is(c.dtype, c.beta, 0);
            if (plan.fill_temps) {
                CopyArgs &fa = plan.fill;
                fa = copy_args(c.nranks, c.rank, s.co, es);
                fa.nd0 = y.nd, fa.o0 = y.o, fa.p0 = y.p, fa.ncomp0 = y.ncomp;
                fa.from0 = y.from, fa.size0 = y.size, fa.dim0 = y.dim;
                if (ypp >= 0) fa.size0[ypp] = 1;
                fa.nd1 = ca.nd0, fa.o1 = ca.o0, fa.p1 = ca.p0, fa.ncomp1 = ncomp;
                fa.from1.assign(ot.size(), 0), fa.dim1 = ca.dim0;
            }
        }

        // ---- one launch per operator component of this rank -------------------------------------------
        const auto ffi = fastest_first(s.ni, s.co), ffd = fastest_first(s.nd, s.co);
        const Coor bim = s.effim(), bdom = s.effdom();
        for (int k = 0; k < ncomp; ++k) {
            const int q = c.rank * ncomp + k;
            const Box &ip = s.pim[q];
            if (ip.empty()) continue;
            const BsrPart &part = g.mine[k];
            BsrItem it;
            it.comp = k;
            it.nnz = part.rowptr.back();
            it.x_elems = g.halo[q].empty() ? 0 : ncols * volume(g.halo[q].size);
            sbk_bsr_desc &d = it.desc;
            sbk_kron_desc &kr = it.kdesc;
            std::memset(&d, 0, sizeof d);
            std::memset(&kr, 0, sizeof kr);
            d.nrows = bsr_rows(s, ip);
            d.bi = (int)volume(s.blockim), d.bd = (int)volume(s.blockdom);
            d.im_fast = s.im_fast, d.ncols = (int)ncols;
            kr.ki = (int)volume(s.kronim), kr.kd = (int)volume(s.krondom), kr.u = std::max(part.u, 0);
            const auto hs = get_strides(g.halo[q].size, s.co);
            for (int kd : ffd)
                if (bdom[kd] > 1) {
                    kr.dksize[d.nd] = s.krondom[kd];
                    d.dsize[d.nd] = s.blockdom[kd], d.dstride[d.nd++] = hs[kd];
                }
            // strides of the output (a y part or the temporary) along oim, the columns and the power
            std::vector<int64_t> ostr;
            std::string oo;
            it.y_off = it.y_pstride = it.y_elems = 0;
            if (direct) {
                it.y_comp = k;
                const Box &yp = y.p[q];
                oo = y.o;
                ostr = get_strides(yp.size, s.co);
                for (int i = 0; i < y.nd; ++i)
                    if (label_pos(c.oim, y.o[i]) < 0) it.y_off += (int64_t)(y.from[i] - yp.from[i]) * ostr[i];
                if (ypp >= 0) it.y_pstride = ostr[ypp];
            } else {
                it.y_comp = -1;
                oo = ot;
                const Box tb = temp_box(ip);
                ostr = get_strides(tb.size, s.co);
                it.y_elems = volume(tb.size);
            }
            for (int ki : ffi) {
                kr.iksize[d.ni] = s.kronim[ki];
                d.iblocks[d.ni] = ip.size[ki] / bim[ki], d.isize[d.ni] = s.blockim[ki];
                d.istride[d.ni++] = ostr[label_pos(oo, c.oim[ki])];
            }
            std::string cf = cols;
            if (s.co != FastToSlow) std::reverse(cf.begin(), cf.end());
            for (char l : cf) {
                if (d.nc >= SBK_MAX_DIMS) fail("too many column labels");
                d.csize[d.nc] = csize[label_pos(cols, l)], d.cstride[d.nc++] = ostr[label_pos(oo, l)];
            }
            plan.items.push_back(it);
        }
        return plan;
    }

    std::string BsrPlan::describe(const BsrGeometry &g) const {
        std::stringstream ss;
        ss << "bsr nothing " << nothing << " direct " << direct << " powers " << powers << " slots " << slots
           << "\n";
        const double one[2] = {1, 0};
        for (const auto &it : items) {
            const sbk_bsr_desc &d = it.desc;
            ss << "item comp " << it.comp << " y " << it.y_comp << " " << it.y_off << " " << it.y_pstride << " "
               << it.y_elems << " x " << it.x_elems << " nnz " << it.nnz << " rows " << d.nrows << " bi " << d.bi
               << " bd " << d.bd << " imfast " << d.im_fast << " ncols " << d.ncols << " D";
            for (int i = 0; i < d.nd; ++i) ss << " " << d.dsize[i] << " " << d.dstride[i];
            ss << " I";
            for (int i = 0; i < d.ni; ++i) ss << " " << d.iblocks[i] << " " << d.isize[i] << " " << d.istride[i];
            ss << " C";
            for (int i = 0; i < d.nc; ++i) ss << " " << d.csize[i] << " " << d.cstride[i];
            ss << "\nrowptr";
            for (int64_t r : g.mine[it.comp].rowptr) ss << " " << r;
            ss << "\ngoff";
            for (int64_t o : g.mine[it.comp].goff) ss << " " << o;
            std::string k;
            if (kron) {
                const sbk_kron_desc &kr = it.kdesc;
                ss << "\nkron ki " << kr.ki << " kd " << kr.kd << " u " << kr.u << " IK";
                for (int i = 0; i < d.ni; ++i) ss << " " << kr.iksize[i];
                ss << " DK";
                for (int i = 0; i < d.nd; ++i) ss << " " << kr.dksize[i];
                kron_bsr(d, kr, g.s.dtype, one, one, nullptr, nullptr, nullptr, nullptr, nullptr, &k);
            } else {
                bsr(d, g.s.dtype, one, one, nullptr, nullptr, nullptr, nullptr, &k);
            }
            ss << "\nkernel " << k << "\n";
        }
        if (nothing) return ss.str();
        ss << "gather 0\n" << make_copy_plan(gather_x)->describe();
        for (int p = 1; p < powers; ++p) {
            CopyArgs ca = gather_y;
            ca.from0[y_power_pos] = (gather_y.from0[y_power_pos] + p - 1) % ca.dim0[y_power_pos];
            ss << "gather " << p << "\n" << make_copy_plan(ca)->describe();
        }
        if (!direct)
            for (int p = 0; p < powers; ++p) {
                if (fill_temps) ss << "fill " << p << "\n" << make_copy_plan(fill_args(p))->describe();
                ss << "back " << p << "\n" << make_copy_plan(back_args(p))->describe();
            }
        return ss.str();
    }

    CopyArgs BsrPlan::fill_args(int p) const {
        CopyArgs ca = fill;
        if (y_power_pos >= 0) ca.from0[y_power_pos] = (fill.from0[y_power_pos] + p) % ca.dim0[y_power_pos];
        return ca;
    }

    CopyArgs BsrPlan::back_args(int p) const {
        CopyArgs ca = back;
        if (y_power_pos >= 0) ca.from1[y_power_pos] = (back.from1[y_power_pos] + p) % ca.dim1[y_power_pos];
        return ca;
    }

    std::vector<BsrRowSplit> make_bsr_split(const BsrGeometry &g, const BsrPlan &plan, const CopyPlan &gather) {
        const BsrShape &s = g.s;
        const CopyArgs &ca = plan.gather_x;
        const int n1 = ca.nd1;
        const Coor bdom = s.effdom();
        std::vector<BsrRowSplit> out;
        for (const BsrItem &it : plan.items) {
            const int q = ca.rank * s.ncomp + it.comp;
            // the boxes of the slot (halo-relative domain coordinates) that come from another rank;
            // an unpack op lists the destination dims fastest first, without those of extent 1 but the
            // fastest one (plan.cpp), over the packed strides of the slot
            const Box &slot = ca.p1[q];
            const auto str = get_strides(slot.size, ca.co);
            const auto order = fastest_first(n1, ca.co);
            std::vector<Box> remote;
            for (const BoxOp &op : gather.ops) {
                if (op.kind != BoxOp::Unpack || op.dst_comp != it.comp) continue;
                Coor from(n1, 0), len(n1, 1);
                size_t j = 0;
                for (int i = 0; i < n1; ++i) {
                    const int m = order[i];
                    from[m] = (int)((op.doff / str[m]) % slot.size[m]);
                    if (j < op.size.size() && (i == 0 || (slot.size[m] > 1 && op.dstride[j] == str[m])))
                        len[m] = op.size[j++];
                }
                Box b{Coor(s.nd, 0), Coor(s.nd, 0)};
                for (int k = 0; k < s.nd; ++k) {
                    const int m = label_pos(ca.o1, plan.odom[k]);
                    b.from[k] = from[m], b.size[k] = len[m];
                }
                if (!b.empty()) remote.push_back(b);
            }
            const BsrPart &part = g.mine[it.comp];
            const Box &halo = g.halo[q];
            const auto hs = get_strides(halo.size, s.co);
            BsrRowSplit sp;
            Box blk{Coor(s.nd, 0), bdom};
            for (int64_t r = 0; r + 1 < (int64_t)part.rowptr.size(); ++r) {
                bool boundary = false;
                for (int64_t b = part.rowptr[r]; b < part.rowptr[r + 1] && !boundary && !remote.empty(); ++b) {
                    for (int k = 0; k < s.nd; ++k) blk.from[k] = (int)((part.goff[b] / hs[k]) % halo.size[k]);
                    for (const Box &rb : remote) boundary = boundary || overlap(blk, rb);
                }
                (boundary ? sp.boundary : sp.interior).push_back(r);
            }
            out.push_back(std::move(sp));
        }
        return out;
    }

    std::string describe_bsr_split(const BsrPlan &plan, const std::vector<BsrRowSplit> &split) {
        std::stringstream ss;
        for (size_t i = 0; i < split.size(); ++i) {
            ss << "split comp " << plan.items[i].comp << "\ninterior";
            for (int64_t r : split[i].interior) ss << " " << r;
            ss << "\nboundary";
            for (int64_t r : split[i].boundary) ss << " " << r;
            ss << "\n";
        }
        return ss.str();
    }

    BsrOperator::~BsrOperator() {
        for (auto *bv : {&rowptr, &goff})
            for (const Buffer &b : *bv)
                if (b.ptr) pool_free(b.device, b.ptr);
    }

    BsrOperator::Split::~Split() {
        for (const Buffer &b : rows)
            if (b.ptr) pool_free(b.device, b.ptr);
    }

    namespace {
        /// The second half of create_bsr: the exchange rows of every rank's parts arrive with one copy of
        /// an int32 tensor (begun by create_bsr_begin), then the errors that need every rank's data are
        /// thrown alike everywhere and the row pointers and block offsets go to the device of each
        /// component
        class BsrCreateExec : public StepRequest {
        public:
            BsrOperator *const op;
            std::vector<int> mine, full;

            explicit BsrCreateExec(BsrOperator *op) : StepRequest(op->g.s.name()), op(op) { ++op->requests; }
            ~BsrCreateExec() { --op->requests; }

        private:
            void on_failure() override { op->state = BsrOperator::Failed; }

            /// The completion; the operator is then ready
            bool step() override {
                const BsrShape &s = op->g.s;
                op->g.halo = bsr_halo(s, s.nranks > 1 ? full : mine);
                // ---- row pointers and block offsets on the device of each component ----------------------
                for (int k = 0; k < s.ncomp; ++k) {
                    const BsrPart &p = op->g.mine[k];
                    const int dev = op->v[k].host ? op->home : op->v[k].device;
                    auto up = [&](const std::vector<int64_t> &h) {
                        Buffer b{nullptr, false, dev};
                        b.ptr = pool_alloc(dev, std::max<size_t>(h.size(), 1) * sizeof(int64_t));
                        use_device(dev);
                        if (!h.empty())
                            cuda_check(cudaMemcpy(b.ptr, h.data(), h.size() * sizeof(int64_t), cudaMemcpyHostToDevice),
                                       "cudaMemcpy H2D");
                        return b;
                    };
                    op->rowptr.push_back(up(p.rowptr));
                    op->goff.push_back(up(p.goff));
                }
                op->state = BsrOperator::Ready;
                return true;
            }
        };
    }

    BsrOperator *create_bsr_begin(const BsrShape &s, const int *const *ii, const int *const *jj,
                                  const std::vector<Buffer> &v, const std::vector<Buffer> &kronv, Comm *comm,
                                  std::unique_ptr<Request> *request) {
        check_bsr_shape(s);
        std::unique_ptr<BsrOperator> op(new BsrOperator);
        op->g.s = s;
        op->v = v;
        op->kronv = kronv;
        const int home = op->home = home_device(comm, {&v}, default_device(comm), false);
        std::unique_ptr<BsrCreateExec> e(new BsrCreateExec(op.get()));

        // ---- this rank's parts, from host copies of ii and jj, and their exchange rows ------------------
        std::vector<int> &mine = e->mine;
        for (int k = 0; k < s.ncomp; ++k) {
            const Box &ip = s.pim[(size_t)s.rank * s.ncomp + k];
            const int64_t rows = bsr_rows(s, ip);
            std::vector<int> hi(rows), hj;
            auto fetch = [&](const int *src, int *dst, int64_t n) {
                if (n == 0) return;
                if (!src) throw std::runtime_error(std::string(s.name()) + ": null ii or jj for a non-empty component");
                if (v[k].host) {
                    std::memcpy(dst, src, n * sizeof(int));
                } else {
                    use_device(v[k].device);
                    cuda_check(cudaMemcpy(dst, src, n * sizeof(int), cudaMemcpyDeviceToHost), "cudaMemcpy D2H");
                }
            };
            fetch(ii[k], hi.data(), rows);
            int64_t nnz = 0;
            for (int x : hi) nnz += std::max(x, 0);
            hj.resize(nnz * s.nd);
            fetch(jj ? jj[k] : nullptr, hj.data(), nnz * s.nd);
            op->g.mine.push_back(make_bsr_part(s, ip, hi.data(), hj.data()));
            const BsrPart &p = op->g.mine.back();
            if (s.kron && p.u > 0 && !kronv[k].ptr) throw std::runtime_error("create_kron_bsr: null kronv for a component with blocks");
            append_bsr_row(s, p, mine);
        }

        // ---- begin the exchange of every rank's rows: rank-major, so that they arrive in part order -------
        if (s.nranks > 1) {
            if (!comm) throw std::runtime_error("wtf");
            const int W = (int)mine.size();
            CopyArgs ca = copy_args(s.nranks, s.rank, FastToSlow, 4);
            ca.nd0 = ca.nd1 = 2, ca.o0 = ca.o1 = "kr", ca.ncomp0 = ca.ncomp1 = 1;
            ca.dim0 = ca.dim1 = ca.size0 = Coor{W, s.nranks};
            ca.from0 = ca.from1 = Coor{0, 0};
            for (int r = 0; r < s.nranks; ++r) {
                ca.p0.push_back(Box{Coor{0, r}, Coor{W, 1}});
                ca.p1.push_back(Box{Coor{0, 0}, Coor{W, s.nranks}});
            }
            e->full.assign((size_t)s.nranks * W, 0);
            e->begin_exchange(ca, SBB_I32, {Buffer{mine.data(), true, home}}, {Buffer{e->full.data(), true, home}}, comm);
        }
        *request = std::move(e);
        return op.release();
    }

    namespace {
        /// bsr_krylov in steps, one exchange each (driver.hpp, StepRequest):
        ///   gather of x, [fill of the temporaries,] kernels, [write-back,] then the same per power >= 1.
        /// Power 0 runs the interior rows of every item right after the gather of x has begun (behind its
        /// local part) and the boundary rows once it is complete.  With temporaries to fill there is no
        /// split: every row runs after the fill.  An item whose split is trivial (no interior or no
        /// boundary row) runs in one launch after the gather, as before the split existed.
        class BsrExec : public StepRequest {
        public:
            BsrExec(const BsrOperator &op, const BsrCall &c, const std::vector<Buffer> &vx,
                    const std::vector<Buffer> &vy, Comm *comm)
                : StepRequest("bsr_krylov"), op(op), c(c), vx(vx), vy(vy), comm(comm) { ++op.requests; }
            ~BsrExec() { --op.requests; }

            void begin() {
                plan = make_bsr_plan(op.g, c);
                if (plan.nothing) return; // complete at the first progress()
                es = dtype_bytes(c.dtype);
                // ---- home device, host components staged on it -------------------------------------------
                home = home_device(comm, {&vy, &vx, &op.v}, op.home);
                sx = stage_in(vx, c.x, c.rank, es, home, pool);
                sy = stage_in(vy, c.y, c.rank, es, home, pool);
                // a host v (and kronv) is staged on every call, so that changes made to it between calls are seen
                std::vector<size_t> vbytes(op.v.size(), 0), kbytes(op.kronv.size(), 0);
                for (const BsrItem &it : plan.items) {
                    vbytes[it.comp] = (size_t)it.nnz * it.desc.bi * it.desc.bd * es;
                    if (plan.kron) kbytes[it.comp] = (size_t)it.kdesc.u * it.kdesc.ki * it.kdesc.kd * es;
                }
                sv = stage_in(op.v, vbytes, home, pool);
                sk = stage_in(op.kronv, kbytes, home, pool);
                devs = call_devices(home, {&sx, &sy, &sv, &sk});
                // ---- gathered inputs and temporaries, one slot per operator component ----------------------
                std::vector<SlotNeed> xneed, yneed;
                for (const BsrItem &it : plan.items) {
                    xneed.push_back({it.comp, item_device(it), it.x_elems});
                    if (!plan.direct) yneed.push_back({it.comp, item_device(it), it.y_elems});
                }
                slot = alloc_slots(plan.slots, xneed, es, home, pool);
                temp = alloc_slots(plan.slots, yneed, es, home, pool);
                progress();
            }

        private:
            const BsrOperator &op;
            const BsrCall c;
            const std::vector<Buffer> vx, vy;
            Comm *comm;
            BsrPlan plan;
            int es = 0, home = 0, p = 0;
            PoolGuard pool;
            Staged sx, sy, sv, sk;
            std::set<int> devs;
            std::vector<Buffer> slot, temp;
            std::shared_ptr<const BsrOperator::Split> split; ///< power 0 only; null: no item is split
            enum Next { Gather, Fill, Kernels, Back, End } next = Gather;
            enum Rows { All, Interior, Boundary };

            int item_device(const BsrItem &it) const { return sv.dev[it.comp].host ? home : sv.dev[it.comp].device; }

            /// Queue up to the next exchange and begin it
            bool step() override {
                if (plan.nothing) return true;
                for (;;) switch (next) {
                    case Gather: {
                        CopyArgs ca = plan.gather_x;
                        if (p > 0) {
                            ca = plan.gather_y;
                            const int k = plan.y_power_pos;
                            ca.from0[k] = (plan.gather_y.from0[k] + p - 1) % ca.dim0[k];
                        }
                        begin_exchange(ca, c.dtype, p == 0 ? sx.dev : sy.dev, slot, comm);
                        next = plan.fill_temps ? Fill : Kernels;
                        if (p == 0 && !plan.fill_temps) interior_rows();
                        return false;
                    }
                    case Fill:
                        begin_exchange(plan.fill_args(p), c.dtype, sy.dev, temp, comm);
                        next = Kernels;
                        return false;
                    case Kernels:
                        order_streams(devs);
                        launch(split ? Boundary : All);
                        order_streams(devs);
                        split = nullptr;
                        if (plan.direct) {
                            next = ++p < plan.powers ? Gather : End;
                        } else {
                            next = Back;
                        }
                        break;
                    case Back:
                        begin_exchange(plan.back_args(p), c.dtype, temp, sy.dev, comm);
                        next = ++p < plan.powers ? Gather : End;
                        return false;
                    case End:
                        // ---- host results back ----------------------------------------------------------------
                        stage_out(vy, sy, home);
                        pool.release();
                        return true;
                    }
            }

            /// The split of the gather just begun (cached with the operator), and the interior rows queued
            /// behind the gather's local part
            void interior_rows() {
                const std::shared_ptr<const CopyPlan> gp = get_copy_plan(plan.gather_x);
                split = nullptr;
                for (const auto &e : op.splits)
                    if (e->gather == gp) split = e;
                if (!split) {
                    const std::vector<BsrRowSplit> rs = make_bsr_split(op.g, plan, *gp);
                    std::shared_ptr<BsrOperator::Split> e(new BsrOperator::Split);
                    e->gather = gp;
                    for (size_t i = 0; i < rs.size(); ++i) {
                        const BsrRowSplit &r = rs[i];
                        e->ninterior.push_back((int64_t)r.interior.size());
                        Buffer b;
                        if (!r.interior.empty() && !r.boundary.empty()) {
                            std::vector<int64_t> h = r.interior;
                            h.insert(h.end(), r.boundary.begin(), r.boundary.end());
                            b.device = op.rowptr[plan.items[i].comp].device;
                            b.ptr = pool_alloc(b.device, h.size() * sizeof(int64_t));
                            use_device(b.device);
                            cuda_check(cudaMemcpy(b.ptr, h.data(), h.size() * sizeof(int64_t), cudaMemcpyHostToDevice),
                                       "cudaMemcpy H2D");
                        }
                        e->rows.push_back(b);
                    }
                    // the splits of a few gathers (x partitions) per operator
                    if (op.splits.size() >= 8) op.splits.erase(op.splits.begin());
                    op.splits.push_back(e);
                    split = e;
                }
                bool any = false;
                for (const Buffer &b : split->rows) any = any || b.ptr;
                if (!any) {
                    split = nullptr;
                    return;
                }
                wait_local();
                order_streams(devs);
                launch(Interior);
            }

            void launch(Rows which) {
                const int P = p;
                const bool cplx = c.dtype == SBB_C64 || c.dtype == SBB_C128;
                for (size_t i = 0; i < plan.items.size(); ++i) {
                    const BsrItem &it = plan.items[i];
                    const Buffer *list = split && split->rows[i].ptr ? &split->rows[i] : nullptr;
                    if (which == Interior && !list) continue;
                    const int dev = item_device(it);
                    char *out;
                    if (plan.direct) {
                        const Buffer &yb = sy.dev[it.y_comp];
                        enable_peer(dev, yb.device);
                        out = (char *)yb.ptr + (it.y_off + P * it.y_pstride) * es;
                    } else {
                        out = (char *)temp[it.comp].ptr;
                    }
                    enable_peer(dev, sv.dev[it.comp].device);
                    sbk_bsr_desc d = it.desc;
                    d.rowptr = (const int64_t *)op.rowptr[it.comp].ptr;
                    d.goff = (const int64_t *)op.goff[it.comp].ptr;
                    enable_peer(dev, op.rowptr[it.comp].device);
                    if (list && which != All) {
                        const int64_t ni = split->ninterior[i];
                        d.rows = (const int64_t *)list->ptr + (which == Interior ? 0 : ni);
                        d.nlist = which == Interior ? ni : d.nrows - ni;
                    }
                    if (plan.kron) enable_peer(dev, sk.dev[it.comp].device);
                    use_device(dev);
                    const sbk_kron_desc &kr = it.kdesc;
                    if (plan.kron)
                        kron_bsr(d, kr, c.dtype, c.alpha, c.beta, sv.dev[it.comp].ptr, sk.dev[it.comp].ptr,
                                 slot[it.comp].ptr, out, device_state(dev).stream);
                    else
                        bsr(d, c.dtype, c.alpha, c.beta, sv.dev[it.comp].ptr, slot[it.comp].ptr, out,
                            device_state(dev).stream);
                    if (which == Interior) continue; // the item's work is counted once
                    const double blk = (double)d.bi * d.bd;
                    if (plan.kron) {
                        // per block B x (bd -> bi for kd x columns), then the Kronecker sum (kd -> ki for bi x columns)
                        work_counters().flops +=
                            (cplx ? 8.0 : 2.0) * it.nnz * (blk * kr.kd + (double)kr.ki * kr.kd * d.bi) * d.ncols;
                        work_counters().bytes += ((double)it.nnz * blk + (double)kr.u * kr.ki * kr.kd + it.x_elems +
                                                  (double)d.nrows * d.bi * kr.ki * d.ncols) * es;
                    } else {
                        work_counters().flops += (cplx ? 8.0 : 2.0) * it.nnz * blk * d.ncols;
                        work_counters().bytes += ((double)it.nnz * blk + it.x_elems + (double)d.nrows * d.bi * d.ncols) * es;
                    }
                }
            }
        };
    }

    std::unique_ptr<Request> begin_bsr(const BsrOperator &op, const BsrCall &c, const std::vector<Buffer> &vx,
                                       const std::vector<Buffer> &vy, Comm *comm) {
        if (op.state == BsrOperator::Pending)
            throw std::runtime_error("bsr_krylov: the operator's create has not completed (wait for its request first)");
        if (op.state == BsrOperator::Failed) throw std::runtime_error("bsr_krylov: the operator's create failed");
        std::unique_ptr<BsrExec> e(new BsrExec(op, c, vx, vy, comm));
        e->begin();
        return e;
    }

} // namespace sbb
