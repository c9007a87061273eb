// Host-side label and box algebra on a periodic lattice.
//
// Everything the planner needs is expressed in the "range space" of an operation: the coordinates
// u in [0, size) of the copied (or contracted) range, counted from its first element.  A component
// of a partitioned tensor intersects that range in at most two pieces per dimension (its box may
// wrap around the lattice, and so may the range), and inside each piece both the component's
// local storage and the range space are plain, non-periodic boxes.  Kernels therefore never see
// wrap-around: they get strided boxes.
//
// Reference semantics followed (not code): PartitionItem ownership `from <= c < from+size (mod
// dim)` (tensor.h:251-259, dist.h:36-51), intersection of periodic intervals (dist.h:353-423),
// basic_partitioning (dist.h:3393-3509), partitioning_distributed_procs (dist.h:3318-3383),
// make_hole (dist.h:3750-3825).
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

namespace sbb {

    using Coor = std::vector<int>;

    enum CoorOrder { SlowToFast = 0, FastToSlow = 1 };

    inline int64_t volume(const Coor &c) {
        int64_t v = 1;
        for (int x : c) v *= x;
        return c.empty() ? 1 : v; // a rank-0 tensor is a scalar
    }

    /// Jumps between consecutive coordinates in each dimension (tensor.h:282)
    std::vector<int64_t> get_strides(const Coor &dim, int co);

    /// One ownership box {from, size} of a partition (dist.h:39)
    struct Box {
        Coor from, size;
        bool empty() const {
            for (int s : size)
                if (s <= 0) return true;
            return false;
        }
    };

    /// A partition as the reference passes it: int[nparts][2][nd]
    std::vector<Box> read_partition(const int *p, int nparts, int nd);

    /// A piece of (component ∩ range) along one dimension
    struct Piece {
        int u;     ///< first range-relative coordinate
        int len;   ///< extent
        int local; ///< local coordinate inside the component of that first element
    };

    /// Pieces of [pfrom, pfrom+psize) ∩ [rfrom, rfrom+rsize) on a ring of `dim` sites, in
    /// range-relative coordinates, sorted by u. At most two.
    std::vector<Piece> ring_pieces(int pfrom, int psize, int rfrom, int rsize, int dim);

    /// A box in range space (extents follow some agreed dimension order) together with the local
    /// coordinates, in the owner's own dimension order, of its first element.
    struct RBox {
        Coor u, len; ///< range-space origin and extents
        Coor lfrom;  ///< owner-local coordinates of the origin (owner's dimension order)
        bool empty() const {
            for (int s : len)
                if (s <= 0) return true;
            return false;
        }
    };

    /// Set difference a \ b for two boxes in range space (plain, non periodic). `a`'s lfrom is
    /// carried along consistently. `map[k]` gives for range dimension k the index in lfrom that
    /// moves with it (or -1).
    std::vector<RBox> subtract(const RBox &a, const RBox &b, const std::vector<int> &map);

    /// Intersection of two range-space boxes; returns false when empty. `oa`/`ob` receive the
    /// offsets of the intersection's origin inside a and b (per range dimension).
    bool intersect(const RBox &a, const RBox &b, Coor &u, Coor &len);

    /// All range-space boxes of (part ∩ range). `to_range[k]` = range dimension of the part's
    /// k-th dimension or -1 (then the range has extent 1 there and only lfrom is recorded).
    std::vector<RBox> part_boxes(const Box &part, const Coor &rfrom, const Coor &rsize,
                                 const Coor &dim, const std::vector<int> &to_range, int nrange);

    /// No label appears twice in the order `o`
    bool labels_unique(const std::string &o);

    /// Position of label `c` in the order `o`, or -1
    inline int label_pos(const std::string &o, char c) {
        const auto p = o.find(c);
        return p == std::string::npos ? -1 : (int)p;
    }

    // --- partition generators (host only) ---------------------------------------------------------

    Coor partitioning_distributed_procs(const std::string &order, const Coor &dim,
                                        const std::string &dist_labels, unsigned nprocs);

    std::vector<Box> basic_partitioning(const char *order, const Coor &dim, const Coor &procs,
                                        const char *dist_labels, int nprocs, int ncomponents);

    std::vector<Box> basic_partitioning_ext(const Coor &dim, const Coor &procs, int nprocs,
                                            bool replicate, const Coor &ext_power);

    std::vector<Box> make_hole(const Coor &from, const Coor &size, const Coor &hole_from,
                               const Coor &hole_size, const Coor &dim);

} // namespace sbb
