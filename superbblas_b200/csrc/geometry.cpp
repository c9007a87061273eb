// Host-side label and box algebra on a periodic lattice. See geometry.hpp.
#include "geometry.hpp"
#include <algorithm>
#include <cstring>
#include <numeric>

namespace sbb {

    std::vector<int64_t> get_strides(const Coor &dim, int co) {
        const int n = (int)dim.size();
        std::vector<int64_t> s(n, 1);
        if (co == SlowToFast) {
            for (int i = n - 2; i >= 0; --i) s[i] = s[i + 1] * dim[i + 1];
        } else {
            for (int i = 1; i < n; ++i) s[i] = s[i - 1] * dim[i - 1];
        }
        return s;
    }

    std::vector<Box> read_partition(const int *p, int nparts, int nd) {
        std::vector<Box> r(nparts);
        for (int i = 0; i < nparts; ++i) {
            r[i].from.assign(p + (size_t)(2 * i) * nd, p + (size_t)(2 * i + 1) * nd);
            r[i].size.assign(p + (size_t)(2 * i + 1) * nd, p + (size_t)(2 * i + 2) * nd);
            for (int k = 0; k < nd; ++k)
                if (r[i].size[k] < 0) throw std::runtime_error("partition with negative size");
        }
        return r;
    }

    static inline int modp(int a, int d) {
        int r = a % d;
        return r < 0 ? r + d : r;
    }

    std::vector<Piece> ring_pieces(int pfrom, int psize, int rfrom, int rsize, int dim) {
        std::vector<Piece> out;
        if (psize <= 0 || rsize <= 0 || dim <= 0) return out;
        if (psize > dim || rsize > dim)
            throw std::runtime_error("range larger than the lattice dimension");
        // Start of the component measured from the start of the range
        const int r = modp(pfrom - rfrom, dim);
        // The component covers range-relative [r, r+psize) modulo dim: one or two plain segments
        // segment 1: [r, min(r+psize, dim)), local coordinate of u is u - r
        // segment 2: [0, r+psize-dim) when it wraps, local coordinate of u is u - r + dim
        const int e1 = std::min(r + psize, dim);
        const int e2 = r + psize - dim; // > 0 iff wraps
        if (e2 > 0) {
            const int len = std::min(e2, rsize);
            if (len > 0) out.push_back(Piece{0, len, dim - r});
        }
        {
            const int b = r, e = std::min(e1, rsize);
            if (e > b) out.push_back(Piece{b, e - b, 0});
        }
        return out;
    }

    bool intersect(const RBox &a, const RBox &b, Coor &u, Coor &len) {
        const int n = (int)a.u.size();
        u.resize(n);
        len.resize(n);
        for (int k = 0; k < n; ++k) {
            const int lo = std::max(a.u[k], b.u[k]);
            const int hi = std::min(a.u[k] + a.len[k], b.u[k] + b.len[k]);
            if (hi <= lo) return false;
            u[k] = lo;
            len[k] = hi - lo;
        }
        return true;
    }

    std::vector<RBox> subtract(const RBox &a, const RBox &b, const std::vector<int> &map) {
        std::vector<RBox> out;
        Coor iu, il;
        if (a.empty()) return out;
        if (!intersect(a, b, iu, il)) {
            out.push_back(a);
            return out;
        }
        const int n = (int)a.u.size();
        // Peel slabs dimension by dimension: dims < k are clipped to the intersection, dim k takes
        // what is left of / right of it, dims > k keep a's full extent.
        RBox cur = a;
        auto shifted = [&](const RBox &base, int k, int newu, int newlen) {
            RBox r = base;
            const int d = newu - base.u[k];
            r.u[k] = newu;
            r.len[k] = newlen;
            if (map[k] >= 0) r.lfrom[map[k]] += d;
            return r;
        };
        for (int k = 0; k < n; ++k) {
            const int a0 = cur.u[k], a1 = cur.u[k] + cur.len[k];
            const int i0 = iu[k], i1 = iu[k] + il[k];
            if (i0 > a0) out.push_back(shifted(cur, k, a0, i0 - a0));
            if (a1 > i1) out.push_back(shifted(cur, k, i1, a1 - i1));
            cur = shifted(cur, k, i0, il[k]);
        }
        return out;
    }

    std::vector<RBox> part_boxes(const Box &part, const Coor &rfrom, const Coor &rsize,
                                 const Coor &dim, const std::vector<int> &to_range, int nrange) {
        std::vector<RBox> out;
        const int n = (int)part.from.size();
        if (part.empty()) return out;
        std::vector<std::vector<Piece>> pieces(n);
        for (int k = 0; k < n; ++k) {
            pieces[k] = ring_pieces(part.from[k], part.size[k], rfrom[k], rsize[k], dim[k]);
            if (pieces[k].empty()) return out;
        }
        std::vector<int> idx(n, 0);
        for (;;) {
            RBox b;
            b.u.assign(nrange, 0);
            b.len.assign(nrange, 1);
            b.lfrom.resize(n);
            for (int k = 0; k < n; ++k) {
                const Piece &pc = pieces[k][idx[k]];
                b.lfrom[k] = pc.local;
                if (to_range[k] >= 0) b.u[to_range[k]] = pc.u, b.len[to_range[k]] = pc.len;
            }
            out.push_back(std::move(b));
            int k = 0;
            for (; k < n; ++k) {
                if (++idx[k] < (int)pieces[k].size()) break;
                idx[k] = 0;
            }
            if (k == n) break;
        }
        return out;
    }

    bool labels_unique(const std::string &o) {
        for (size_t i = 0; i < o.size(); ++i)
            if (o.find(o[i], i + 1) != std::string::npos) return false;
        return true;
    }

    // ---------------------------------------------------------------------------------------------
    // Partition generators
    // ---------------------------------------------------------------------------------------------

    namespace {
        /// Closest value of the form 2^a 3^b not above `number` by more than a quarter
        /// (reference: factors_2_3, dist.h:3268-3310; the partitions it induces are pinned by
        /// tests/dist.cpp:103-125, so the rounding rule has to be this one).
        unsigned smooth_23(unsigned number) {
            if (number == 0) throw std::runtime_error("unsupported value");
            unsigned twos = 0, threes = 0, value = 1, rest = number;
            while (rest % 2 == 0) ++twos, rest /= 2, value *= 2;
            while (rest % 3 == 0) ++threes, rest /= 3, value *= 3;
            while (rest >= 3) ++threes, rest /= 3, value *= 3;
            if (rest >= 2) ++twos, rest /= 2, value *= 2;
            while (threes > 0 && value * 4 / 3 <= number) --threes, twos += 2, value = value * 4 / 3;
            (void)twos;
            return value;
        }
    }

    Coor partitioning_distributed_procs(const std::string &order, const Coor &dim,
                                        const std::string &dist_labels, unsigned nprocs) {
        const int n = (int)dim.size();
        if ((int)order.size() != n)
            throw std::runtime_error("The length of the order should match the template argument; "
                                     "argument `order` should have length " +
                                     std::to_string(n));
        Coor procs(n, 1);
        // dimensions that may be split, in the order the caller listed them
        std::vector<int> cand;
        for (char l : dist_labels) {
            const auto pos = order.find(l);
            if (pos != std::string::npos && dim[pos] > 1) cand.push_back((int)pos);
        }
        if (cand.empty() || volume(dim) == 0 || nprocs <= 1) return procs;

        const unsigned target = smooth_23(nprocs);
        std::vector<unsigned> f(cand.size(), 1);
        unsigned placed = 1;
        for (;;) {
            // candidates by decreasing local extent; ties keep the first one found from the front
            std::vector<int> by_size(cand.size());
            std::iota(by_size.begin(), by_size.end(), 0);
            for (size_t j = 0; j < by_size.size(); ++j) {
                size_t best = j;
                size_t best_val = (size_t)dim[cand[by_size[j]]] / f[by_size[j]];
                for (size_t i = j + 1; i < by_size.size(); ++i) {
                    const size_t val = (size_t)dim[cand[by_size[i]]] / f[by_size[i]];
                    if (best_val < val) best = i, best_val = val;
                }
                std::swap(by_size[j], by_size[best]);
            }
            // give the first candidate that can take it a factor 3, else a factor 2
            bool done = true;
            for (size_t j = 0; j < by_size.size() && done; ++j) {
                for (unsigned factor : {3u, 2u}) {
                    if (target % (placed * factor) == 0) {
                        f[by_size[j]] *= factor;
                        placed *= factor;
                        done = false;
                        break;
                    }
                }
            }
            if (done) break;
        }
        for (size_t i = 0; i < cand.size(); ++i) procs[cand[i]] = (int)f[i];
        return procs;
    }

    namespace {
        /// Block distribution of `dim` sites among `np` owners: owner `c` gets [from, from+size)
        inline void block_1d(int dim, int np, int c, int &from, int &size) {
            size = dim / np + (dim % np > c ? 1 : 0);
            from = size == dim ? 0 : dim / np * c + std::min(c, dim % np);
        }
    }

    std::vector<Box> basic_partitioning(const char *order, const Coor &dim, const Coor &procs,
                                        const char *dist_labels, int nprocs, int ncomponents) {
        const int n = (int)dim.size();
        if ((int)procs.size() != n) throw std::runtime_error("basic_partitioning: bad `procs`");
        const int vol_procs = (int)volume(procs);
        // Process-grid axis order: the labels of dist_labels first (slowest), then the rest
        std::vector<int> axes;
        if (order != nullptr && dist_labels != nullptr) {
            if ((int)std::strlen(order) != n)
                throw std::runtime_error("basic_partitioning: invalid `order`, its length doesn't "
                                         "match the template parameter");
            const std::string o(order), dl(dist_labels);
            for (char l : dl) {
                const auto pos = o.find(l);
                if (pos != std::string::npos) axes.push_back((int)pos);
            }
            for (int i = 0; i < n; ++i)
                if (dl.find(o[i]) == std::string::npos) axes.push_back(i);
            if ((int)axes.size() != n) throw std::runtime_error("wtf");
        } else {
            axes.resize(n);
            std::iota(axes.begin(), axes.end(), 0);
        }

        const int nparts = (nprocs < 0 ? vol_procs : nprocs) * ncomponents;
        std::vector<Box> out(nparts, Box{Coor(n, 0), Coor(n, 0)});
        Coor grid(n);
        for (int i = 0; i < n; ++i) grid[i] = procs[axes[i]];
        const auto gstride = get_strides(grid, SlowToFast);
        for (int rank = 0; rank < vol_procs && rank * ncomponents < nparts; ++rank) {
            Box b{Coor(n, 0), Coor(n, 0)};
            for (int i = 0; i < n; ++i) {
                const int c = (int)((rank / gstride[i]) % grid[i]);
                block_1d(dim[axes[i]], grid[i], c, b.from[axes[i]], b.size[axes[i]]);
            }
            if (volume(b.size) == 0) b.from.assign(n, 0), b.size.assign(n, 0);
            if (ncomponents == 1) {
                out[rank] = b;
                continue;
            }
            // Components split the rank's box again along the same labels
            const std::string o(order ? order : ""), dl(dist_labels ? dist_labels : "");
            const Coor cprocs = partitioning_distributed_procs(o, b.size, dl, ncomponents);
            const auto sub = basic_partitioning(order, b.size, cprocs, dist_labels, ncomponents, 1);
            for (int c = 0; c < ncomponents; ++c) {
                Box &dst = out[rank * ncomponents + c];
                if (volume(sub[c].size) == 0) continue; // stays all zero
                dst.size = sub[c].size;
                for (int k = 0; k < n; ++k) dst.from[k] = sub[c].from[k] + b.from[k];
            }
        }
        return out;
    }

    std::vector<Box> basic_partitioning_ext(const Coor &dim, const Coor &procs, int nprocs,
                                            bool replicate, const Coor &ext_power) {
        const int n = (int)dim.size();
        const int vol_procs = (int)volume(procs);
        for (int e : ext_power)
            if (e < 0) throw std::runtime_error("Unsupported value for `power`");
        std::vector<Box> out(nprocs < 0 ? vol_procs : nprocs, Box{Coor(n, 0), Coor(n, 0)});
        const auto gstride = get_strides(procs, SlowToFast);
        for (int rank = 0; rank < vol_procs && rank < (int)out.size(); ++rank) {
            for (int i = 0; i < n; ++i) {
                const int c = (int)((rank / gstride[i]) % procs[i]);
                int from, size;
                block_1d(dim[i], procs[i], c, from, size);
                const int ext = (int)ext_power.size() > i ? ext_power[i] : 0;
                // widen by the halo on both sides, saturating at the whole dimension
                const int wsize = std::min(size + 2 * ext, dim[i]);
                const int core_from = dim[i] / procs[i] * c + std::min(c, dim[i] % procs[i]);
                out[rank].size[i] = wsize;
                out[rank].from[i] = wsize == dim[i] ? 0 : modp(core_from - ext, dim[i]);
            }
        }
        if (replicate && vol_procs == 1)
            for (auto &b : out) b = out[0];
        return out;
    }

    std::vector<Box> make_hole(const Coor &from, const Coor &size, const Coor &hole_from,
                               const Coor &hole_size, const Coor &dim) {
        const int n = (int)dim.size();
        std::vector<Box> out;
        if (n == 0) return out;
        if (volume(size) == 0) return out;
        if (volume(hole_size) == 0) {
            out.push_back(Box{from, size});
            return out;
        }
        // Work in the coordinates of the range: the hole meets it in up to 2^n plain boxes
        std::vector<int> map(n, -1);
        std::vector<RBox> rest(1);
        rest[0].u.assign(n, 0);
        rest[0].len = size;
        std::vector<std::vector<Piece>> pieces(n);
        bool touches = true;
        for (int k = 0; k < n; ++k) {
            pieces[k] = ring_pieces(hole_from[k], hole_size[k], from[k], size[k], dim[k]);
            if (pieces[k].empty()) touches = false;
        }
        if (touches) {
            std::vector<int> idx(n, 0);
            for (;;) {
                RBox h;
                h.u.resize(n), h.len.resize(n);
                for (int k = 0; k < n; ++k) h.u[k] = pieces[k][idx[k]].u, h.len[k] = pieces[k][idx[k]].len;
                std::vector<RBox> next;
                for (const auto &r : rest) {
                    auto parts = subtract(r, h, map);
                    next.insert(next.end(), parts.begin(), parts.end());
                }
                rest.swap(next);
                int k = 0;
                for (; k < n; ++k) {
                    if (++idx[k] < (int)pieces[k].size()) break;
                    idx[k] = 0;
                }
                if (k == n) break;
            }
        }
        for (const auto &r : rest) {
            if (r.empty()) continue;
            Box b{Coor(n), r.len};
            for (int k = 0; k < n; ++k)
                b.from[k] = r.len[k] == dim[k] ? from[k] : modp(from[k] + r.u[k], dim[k]);
            out.push_back(b);
        }
        return out;
    }

} // namespace sbb
