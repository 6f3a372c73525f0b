// Coset-sharded commitment trees (multi-GPU, DESIGN.md section 7).
//
// A committed matrix has its level-0 items (row hashes for the trace tree, first-level nodes for the constraint tree, row hashes of a
// FRI layer) indexed i = (k * G + g) * blk + j : rank g owns, for every k < n, the aligned block of blk = 2^log_blk consecutive items.
//   local   each rank builds the n complete subtrees over its blocks (levels with more than n*G nodes);
//   mid     the n*G subtree roots are re-sharded by k-range with one all-to-all (rank g receives the G roots of every k in
//           [g n/G, (g+1) n/G): a contiguous run of n nodes of the global level n*G) and rank g builds the subtree over them -- the
//           levels with G < m <= n*G nodes, each rank holding m/G consecutive nodes of every such level;
//   top     the G mid-roots (32 bytes each) are all-gathered and the last log2(G) levels are hashed redundantly, so every rank
//           holds the same root at the Fiat-Shamir point.
// Per tree a rank moves (G-1)/G * 32 n bytes and hashes n blk + n nodes instead of all-gathering 32 n G bytes and hashing n G nodes
// redundantly (r02, 8 GPUs, 2^25 rows: trace tree 1.08 ms with the replicated upper tree).  With G == 1 the same code runs without
// communication and the three heaps are one.
#pragma once
#include <array>
#include "common.cuh"

namespace dg {

typedef std::array<uint8_t, 32> Digest;

enum { SHARD_LOCAL = 0, SHARD_TOP = 1, SHARD_MID = 2 };
struct ShardLocation { int owner; int kind; uint64_t index; };   // kind: which heap `index` points into (SHARD_TOP: replicated, owner = -1)

struct ShardGeom {
    uint64_t n;          // number of blocks per rank
    int log_blk;         // items per block
    int log_g;           // log2(world)
    uint64_t items() const { return (n << log_blk) << log_g; }
    // level-0 item i -> owner and index into the owner's local item array ([k][j])
    ShardLocation item(uint64_t i) const;
    // internal node with global heap index h (1 <= h < items())
    ShardLocation node(uint64_t h) const;
};

// one 16-byte unit (or 32-byte item = two consecutive units) to fetch: `index` counts items of `bytes` bytes from `base` on the
// rank `owner` (owner < 0: replicated, every rank reads its own copy)
struct FetchRef { const void *base; uint64_t index; int owner; };

// All device->host fetches of the openings stage in ONE pass: every rank registers the same requests in the same order, one kernel
// gathers the units this rank owns (zeros elsewhere), one all-gather + one copy bring every rank's units to every host, and the host
// picks each unit from its owner.  Replaces ~40 blocking index-upload / gather / download round trips per proof (r01: 1.3-1.6 ms).
class FetchBatch {
public:
    explicit FetchBatch(Context &c) : c_(c) {}
    size_t add16(const FetchRef &r) { return push(r.base, r.index, r.owner); }                       // returns the unit offset of the value
    size_t add32(const FetchRef &r) { size_t o = push(r.base, 2 * r.index, r.owner); push(r.base, 2 * r.index + 1, r.owner); return o; }
    void run();
    fe value(size_t off) const { fe v; memcpy(&v, out_.data() + off * 16, 16); return v; }
    Digest digest(size_t off) const { Digest d; memcpy(d.data(), out_.data() + off * 16, 32); return d; }
    size_t units() const { return owner_.size(); }
private:
    size_t push(const void *base, uint64_t unit, int owner) {
        const bool mine = owner < 0 || owner == c_.rank;
        req_.push_back(mine ? (unsigned long long)(uintptr_t)base : 0ULL);
        req_.push_back(mine ? unit : 0ULL);
        owner_.push_back(owner);
        return owner_.size() - 1;
    }
    Context &c_;
    std::vector<unsigned long long> req_;      // (base, unit) pairs
    std::vector<int> owner_;
    std::vector<uint8_t> out_;
};

struct ShardedTree {
    ShardGeom geom;
    const void *items_local = nullptr;   // n * blk digests, [k][j]
    DevBuf local_nodes;                  // heap over the local items (valid for levels with >= n nodes)
    DevBuf mid, top;                     // mid: heap over this rank's n nodes of the level n*G (2n digests); top: replicated heap of 2G digests
    const void *mid_p = nullptr, *top_p = nullptr;     // one rank: both alias the local heap (global heap indices)
    Digest root;

    // fetch_root = false leaves the root on the device (upper_p + 32): no host synchronisation; H = the proof's hash (digest.cuh)
    template <class H> void build(Context &c, const void *items_local_dev, uint64_t n, int log_blk, bool fetch_root = true);
    const void *root_dev() const { return (const uint8_t *)top_p + 32; }
    // locations as references for a FetchBatch
    FetchRef item_ref(uint64_t item_index) const { ShardLocation l = geom.item(item_index); return FetchRef{items_local, l.index, l.owner}; }
    FetchRef node_ref(uint64_t heap_index) const {
        ShardLocation l = geom.node(heap_index);
        if (l.kind == SHARD_TOP) return FetchRef{top_p, l.index, -1};
        if (l.kind == SHARD_MID) return FetchRef{mid_p, l.index, l.owner};
        return FetchRef{local_nodes.p, l.index, l.owner};
    }
};

template <class H> void merkle_build_partial(Context &c, const void *leaves, void *nodes, unsigned long long L, unsigned long long stop);
template <class H> void merkle_build(Context &c, const void *leaves, void *nodes, unsigned long long L);
template <class H> void merkle_finish(Context &c, void *nodes, unsigned long long m);
void interleave_roots(Context &c, const void *gathered, void *upper, unsigned long long n, int log_g);
template <class H> void constraint_items_local(Context &c, const fe *evals_local, int log_n, int log_nc, void *items);   // [k][c4_local] digests

}  // namespace dg
