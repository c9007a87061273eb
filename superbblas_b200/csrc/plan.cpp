// Copy planner. See plan.hpp.
#include "plan.hpp"
#include <algorithm>
#include <map>
#include <mutex>
#include <sstream>

namespace sbb {

    void check_copy_args(const CopyArgs &a) {
        auto bad_len = [](const char *name, int n) {
            std::stringstream ss;
            ss << "The length of the order should match the template argument; argument `" << name
               << "` should have length " << n;
            throw std::runtime_error(ss.str());
        };
        if ((int)a.o0.size() != a.nd0) bad_len("o0", a.nd0);
        if ((int)a.o1.size() != a.nd1) bad_len("o1", a.nd1);
        auto invalid = [] { throw std::runtime_error("Invalid copy operation"); };
        if (!labels_unique(a.o0) || !labels_unique(a.o1)) invalid();
        for (int k = 0; k < a.nd0; ++k) {
            if (a.size0[k] < 0 || a.size0[k] > a.dim0[k]) invalid();
            if (a.size0[k] > 1 && a.o1.find(a.o0[k]) == std::string::npos) invalid();
        }
        if (volume(a.size0) != 0)
            for (int m = 0; m < a.nd1; ++m) {
                const auto k = a.o0.find(a.o1[m]);
                const int s = k == std::string::npos ? 1 : a.size0[k];
                if (s > a.dim1[m]) invalid();
            }
        if ((int)a.p0.size() != a.nranks * a.ncomp0 || (int)a.p1.size() != a.nranks * a.ncomp1)
            throw std::runtime_error("wtf");
    }

    namespace {
        int64_t align_up(int64_t x, int a) { return a <= 1 ? x : (x + a - 1) / a * a; }
    }

    std::shared_ptr<const CopyPlan> make_copy_plan(const CopyArgs &a) {
        check_copy_args(a);
        auto plan = std::make_shared<CopyPlan>();
        plan->nranks = a.nranks;
        plan->rank = a.rank;
        plan->send_elems.assign(a.nranks, 0);
        plan->recv_elems.assign(a.nranks, 0);
        const int n0 = a.nd0, n1 = a.nd1, me = a.rank;

        // Range space = destination label order
        std::vector<int> src_to_range(n0, -1), range_to_src(n1, -1), dst_to_range(n1);
        Coor size1(n1, 1);
        for (int m = 0; m < n1; ++m) {
            dst_to_range[m] = m;
            const auto k = a.o0.find(a.o1[m]);
            if (k != std::string::npos) {
                src_to_range[k] = m;
                range_to_src[m] = (int)k;
                size1[m] = a.size0[k];
            }
        }
        if (volume(a.size0) == 0) return plan;
        if (a.add && a.alpha_is_zero) return plan;

        const int P0 = (int)a.p0.size(), P1 = (int)a.p1.size();

        // Source boxes of every part (needed by every rank to agree on who sends what)
        std::vector<std::vector<RBox>> S(P0);
        std::vector<std::vector<int64_t>> sstr(P0);
        if (!a.alpha_is_zero)
            for (int i = 0; i < P0; ++i) {
                S[i] = part_boxes(a.p0[i], a.from0, a.size0, a.dim0, src_to_range, n1);
                sstr[i] = get_strides(a.p0[i].size, a.co);
            }

        // Order in which the dimensions of an op are listed: destination order, fastest first
        std::vector<int> dim_order(n1);
        for (int m = 0; m < n1; ++m) dim_order[m] = a.co == FastToSlow ? m : n1 - 1 - m;

        // running length (elements on the wire) of the message of every (sender, receiver) pair; all
        // pairs are tracked, not only mine, because the peer-memory transport needs to know where my
        // segment starts inside each receiver's arena
        std::vector<int64_t> pair((size_t)a.nranks * a.nranks, 0);
        auto wire = [&](int from, int to) -> int64_t & { return pair[(size_t)from * a.nranks + to]; };

        auto emit = [&](int i, int j, const RBox &sb, const RBox &db, const Coor &u,
                        const Coor &len, const std::vector<int64_t> &dstr) {
            const int ri = i / a.ncomp0, rj = j / a.ncomp1;
            const bool mine = ri == me || rj == me;
            if (ri == rj && !mine) return;
            BoxOp op;
            op.src_part = i, op.dst_part = j;
            int64_t soff = 0, doff = 0;
            for (int k = 0; k < n0; ++k) {
                int l = sb.lfrom[k];
                if (src_to_range[k] >= 0) l += u[src_to_range[k]] - sb.u[src_to_range[k]];
                soff += (int64_t)l * sstr[i][k];
            }
            for (int m = 0; m < n1; ++m) doff += (int64_t)(db.lfrom[m] + u[m] - db.u[m]) * dstr[m];
            for (int m : dim_order) {
                // extent-1 dims are dropped, except the fastest one (kept so that the two halves of
                // a wrapped row can be recognised and fused below)
                if (len[m] == 1 && m != dim_order[0]) continue;
                op.size.push_back(len[m]);
                op.sstride.push_back(range_to_src[m] >= 0 ? sstr[i][range_to_src[m]] : 0);
                op.dstride.push_back(dstr[m]);
            }
            if (ri == me && rj == me) {
                op.kind = BoxOp::Local;
                op.src_comp = i % a.ncomp0, op.dst_comp = j % a.ncomp1;
                op.soff = soff, op.doff = doff;
                plan->ops.push_back(std::move(op));
                return;
            }
            // Remote: big boxes are cut along their slowest dimension so that the exchange can be
            // pipelined (pack of piece k+1 and unpack of piece k-1 overlap the transfer of piece k).
            // Sender and receiver cut identically (the rule only depends on the box).
            const int64_t vol = volume(len);
            const int64_t wire_es = 16 / std::max(1, a.wire_align);
            int pieces = 1;
            const int last = (int)op.size.size() - 1;
            if (a.chunk_bytes > 0 && last >= 0 && vol * wire_es > a.chunk_bytes)
                pieces = (int)std::min<int64_t>(op.size[last],
                                                (vol * wire_es + a.chunk_bytes - 1) / a.chunk_bytes);
            for (int pc = 0; pc < pieces; ++pc) {
                BoxOp q = op;
                int64_t lo = 0;
                if (pieces > 1) {
                    lo = (int64_t)op.size[last] * pc / pieces;
                    const int64_t hi = (int64_t)op.size[last] * (pc + 1) / pieces;
                    q.size[last] = (int)(hi - lo);
                }
                const int64_t pvol = volume(q.size);
                // compact, destination-ordered layout on the wire
                std::vector<int64_t> wstr(q.size.size(), 1);
                for (size_t d = 1; d < q.size.size(); ++d) wstr[d] = wstr[d - 1] * q.size[d - 1];
                int64_t &w = wire(ri, rj);
                const int64_t at = w;
                w = align_up(w + pvol, a.wire_align);
                if (!mine) continue;
                if (ri == me) {
                    q.kind = BoxOp::Pack;
                    q.peer = rj;
                    q.src_comp = i % a.ncomp0;
                    q.soff = soff + (last >= 0 ? lo * op.sstride[last] : 0);
                    q.doff = at;
                    q.dstride = wstr;
                } else {
                    q.kind = BoxOp::Unpack;
                    q.peer = ri;
                    q.dst_comp = j % a.ncomp1;
                    q.doff = doff + (last >= 0 ? lo * op.dstride[last] : 0);
                    q.soff = at;
                    q.sstride = wstr;
                }
                plan->ops.push_back(std::move(q));
            }
        };

        auto emit_zero = [&](int j, const RBox &db, const std::vector<int64_t> &dstr) {
            if (j / a.ncomp1 != me) return;
            BoxOp op;
            op.kind = BoxOp::Zero;
            op.dst_part = j, op.dst_comp = j % a.ncomp1;
            int64_t doff = 0;
            for (int m = 0; m < n1; ++m) doff += (int64_t)db.lfrom[m] * dstr[m];
            op.doff = doff;
            for (int m : dim_order) {
                if (db.len[m] == 1) continue;
                op.size.push_back(db.len[m]);
                op.sstride.push_back(0);
                op.dstride.push_back(dstr[m]);
            }
            plan->ops.push_back(std::move(op));
        };

        for (int j = 0; j < P1; ++j) {
            const int rj = j / a.ncomp1;
            std::vector<RBox> D = part_boxes(a.p1[j], a.from1, size1, a.dim1, dst_to_range, n1);
            if (D.empty()) continue;
            const auto dstr = get_strides(a.p1[j].size, a.co);

            if (a.alpha_is_zero) { // Copy with alpha==0: zero the range, never read v0
                for (const auto &db : D) emit_zero(j, db, dstr);
                continue;
            }

            if (a.add) {
                // every holder contributes, in ascending part order
                for (int i = 0; i < P0; ++i)
                    for (const auto &sb : S[i])
                        for (const auto &db : D) {
                            Coor u, len;
                            if (intersect(sb, db, u, len)) emit(i, j, sb, db, u, len, dstr);
                        }
                continue;
            }

            // Copy: every destination element is written exactly once; holders on the destination's
            // own rank are preferred (no traffic), then ascending part order. What nobody holds is
            // zero-filled (the reference zeroes the whole range first, dist.h:2356-2382).
            std::vector<int> pref;
            for (int i = 0; i < P0; ++i)
                if (i / a.ncomp0 == rj) pref.push_back(i);
            for (int i = 0; i < P0; ++i)
                if (i / a.ncomp0 != rj) pref.push_back(i);
            std::vector<RBox> rest = D;
            for (int i : pref) {
                if (rest.empty()) break;
                for (const auto &sb : S[i]) {
                    std::vector<RBox> next;
                    for (const auto &db : rest) {
                        Coor u, len;
                        if (!intersect(sb, db, u, len)) {
                            next.push_back(db);
                            continue;
                        }
                        emit(i, j, sb, db, u, len, dstr);
                        auto left = subtract(db, sb, dst_to_range);
                        next.insert(next.end(), left.begin(), left.end());
                    }
                    rest.swap(next);
                }
            }
            for (const auto &db : rest) emit_zero(j, db, dstr);
        }

        // A periodic shift along the fastest label splits every row in two boxes (the part that
        // stays and the part that wraps around); when both halves of the same rows are local they
        // are fused back into one operation over whole rows with a rotation, so the rows are read
        // and written contiguously once (instead of a second, badly coalesced pass for the slab
        // that wrapped).
        for (size_t i = 0; i < plan->ops.size(); ++i) {
            BoxOp &A = plan->ops[i];
            if (A.kind != BoxOp::Local || A.rot != 0 || A.size.empty()) continue;
            if (A.sstride[0] != 1 || A.dstride[0] != 1) continue;
            for (size_t j = 0; j < plan->ops.size(); ++j) {
                BoxOp &B = plan->ops[j];
                if (i == j || B.kind != BoxOp::Local || B.rot != 0) continue;
                if (B.src_part != A.src_part || B.dst_part != A.dst_part) continue;
                if (B.size.size() != A.size.size() || B.sstride != A.sstride ||
                    B.dstride != A.dstride)
                    continue;
                bool same = true;
                for (size_t d = 1; d < A.size.size(); ++d) same = same && A.size[d] == B.size[d];
                if (!same) continue;
                // A: src [0,n-r) -> dst [r,n);  B: src [n-r,n) -> dst [0,r)
                if (B.soff != A.soff + A.size[0] || A.doff != B.doff + B.size[0]) continue;
                if (A.size[0] + B.size[0] > 2048) continue; // a whole row must fit in one tile
                A.rot = B.size[0];
                A.size[0] += B.size[0];
                A.doff = B.doff;
                plan->ops.erase(plan->ops.begin() + j);
                if (j < i) --i;
                break;
            }
        }

        plan->send_seg_off.assign(a.nranks, 0);
        plan->recv_seg_off.assign(a.nranks, 0);
        const int seg_align = 16 * std::max(1, a.wire_align); // 256 bytes
        for (int r = 0; r < a.nranks; ++r) {
            plan->send_elems[r] = wire(me, r);
            plan->recv_elems[r] = wire(r, me);
            if (wire(me, r) > 0 || wire(r, me) > 0) plan->needs_comm = true;
        }
        // layout of every rank's arena: one 256-byte aligned segment per sender, in rank order
        for (int q = 0; q < a.nranks; ++q) {
            int64_t off = 0;
            for (int r = 0; r < a.nranks; ++r) {
                if (q == me) plan->recv_seg_off[r] = off;
                if (r == me) plan->send_seg_off[q] = off;
                off += align_up(wire(r, q), seg_align);
                if (wire(r, q) > 0) plan->any_comm = true;
                plan->max_pair_elems = std::max(plan->max_pair_elems, wire(r, q));
            }
            plan->arena_elems = std::max(plan->arena_elems, off);
        }
        // Phases of the exchange: greedy edge colouring -- every edge (sender -> receiver) takes the
        // smallest phase not yet used at its sender or at its receiver.  Edges of the senders with the
        // fewest messages are coloured first: nothing synchronises the phases in time, every sender
        // simply starts with its phase 0, so a sender with a single message must own phase 0 at its
        // receiver (a redistribution t-slabs -> (z,t) blocks on 8 ranks: ranks 0 and 7 keep half of
        // their data and send one message; coloured in rank order rank 7 got phase 1, sent at once
        // and collided with rank 6 for half of the exchange).
        plan->send_phase.assign(a.nranks, 0);
        {
            std::vector<int> outdeg(a.nranks, 0);
            std::vector<std::pair<int, int>> edges;
            for (int r = 0; r < a.nranks; ++r)
                for (int q = 0; q < a.nranks; ++q)
                    if (r != q && wire(r, q) > 0) ++outdeg[r], edges.emplace_back(r, q);
            std::stable_sort(edges.begin(), edges.end(), [&](const std::pair<int, int> &x, const std::pair<int, int> &y) {
                return outdeg[x.first] < outdeg[y.first];
            });
            std::vector<std::vector<char>> used_s(a.nranks), used_r(a.nranks);
            for (const auto &e : edges) {
                const int r = e.first, q = e.second;
                size_t c = 0;
                for (;; ++c) {
                    const bool bs = c < used_s[r].size() && used_s[r][c];
                    const bool br = c < used_r[q].size() && used_r[q][c];
                    if (!bs && !br) break;
                }
                if (used_s[r].size() <= c) used_s[r].resize(c + 1, 0);
                if (used_r[q].size() <= c) used_r[q].resize(c + 1, 0);
                used_s[r][c] = used_r[q][c] = 1;
                plan->nphases = std::max(plan->nphases, (int)c + 1);
                if (r == me) plan->send_phase[q] = (int)c;
            }
        }
        return plan;
    }

    std::string CopyPlan::describe() const {
        std::stringstream ss;
        ss << "plan rank " << rank << " of " << nranks << "\n";
        for (int r = 0; r < nranks; ++r)
            if (send_elems[r] || recv_elems[r])
                ss << "wire peer " << r << " send " << send_elems[r] << " recv " << recv_elems[r]
                   << " phase " << (send_elems[r] ? send_phase[r] : -1) << "\n";
        static const char *names[] = {"local", "pack", "unpack", "zero"};
        for (const auto &op : ops) {
            ss << "op " << names[op.kind] << " src " << op.src_part << " dst " << op.dst_part
               << " peer " << op.peer << " soff " << op.soff << " doff " << op.doff << " size";
            for (int s : op.size) ss << " " << s;
            ss << " sstride";
            for (auto s : op.sstride) ss << " " << s;
            ss << " dstride";
            for (auto s : op.dstride) ss << " " << s;
            ss << " rot " << op.rot << "\n";
        }
        return ss.str();
    }

    // ---------------------------------------------------------------------------------------------
    // Plan cache (reference: cache keyed by the call geometry, dist.h:2305-2349)
    // ---------------------------------------------------------------------------------------------

    namespace {
        std::string key_of(const CopyArgs &a) {
            std::string k;
            auto put = [&](const void *p, size_t n) { k.append((const char *)p, n); };
            auto puti = [&](int v) { put(&v, sizeof v); };
            auto putc = [&](const Coor &c) {
                puti((int)c.size());
                if (!c.empty()) put(c.data(), c.size() * sizeof(int));
            };
            puti(a.nd0), puti(a.nd1), puti(a.ncomp0), puti(a.ncomp1), puti(a.nranks), puti(a.rank);
            puti(a.co), puti(a.add), puti(a.alpha_is_zero), puti(a.wire_align);
            put(&a.chunk_bytes, sizeof a.chunk_bytes);
            k += a.o0, k += '|', k += a.o1, k += '|';
            putc(a.from0), putc(a.size0), putc(a.dim0), putc(a.from1), putc(a.dim1);
            for (const auto &b : a.p0) putc(b.from), putc(b.size);
            for (const auto &b : a.p1) putc(b.from), putc(b.size);
            return k;
        }
        std::mutex cache_mutex;
        std::map<std::string, std::shared_ptr<const CopyPlan>> &cache() {
            static std::map<std::string, std::shared_ptr<const CopyPlan>> c;
            return c;
        }
    }

    std::shared_ptr<const CopyPlan> get_copy_plan(const CopyArgs &a) {
        const std::string k = key_of(a);
        {
            std::lock_guard<std::mutex> g(cache_mutex);
            auto it = cache().find(k);
            if (it != cache().end()) return it->second;
        }
        auto p = make_copy_plan(a);
        std::lock_guard<std::mutex> g(cache_mutex);
        if (cache().size() > 4096) cache().clear();
        cache()[k] = p;
        return p;
    }

    void clear_plan_cache() {
        std::lock_guard<std::mutex> g(cache_mutex);
        cache().clear();
    }

    size_t plan_cache_size() {
        std::lock_guard<std::mutex> g(cache_mutex);
        return cache().size();
    }

} // namespace sbb
