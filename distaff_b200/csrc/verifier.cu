// GPU verifier for StarkProof bytes: the step after the prove path (SURVEY.md section 8f rank 3).
//
//   stark::verify                      /root/reference/src/stark/verifier.rs:11-75
//   evaluate_constraints / compose_*   /root/reference/src/stark/verifier.rs:79-162
//   fri::verify                        /root/reference/src/stark/fri/verifier.rs:11-131
//   MerkleTree::verify_batch           /root/reference/src/crypto/merkle.rs:154-263
//
// The reference walks the proof sequentially on one core.  Here the host parses the proof, redoes the Fiat-Shamir draws (PoW check,
// query positions, coefficients, FRI folding points) and turns every batch-Merkle verification into a plan of (left, right, out)
// hashing steps per tree level -- pure index logic, following verify_batch statement by statement, including its use of the current
// level's position as the slot of `proof.nodes` -- while the device does all of the arithmetic and hashing in five launches:
//   1. the hash (BLAKE3 or SHA3-256, from the proof's options) of the opened trace rows and of the opened FRI rows (the Merkle leaves),
//   2. all Merkle plans at once (one block per tree, one barrier per level),
//   3. the transition constraints at the out-of-domain point z: the prover's own constraint kernel (air.cu) in verify mode, with the
//      deep values as its two rows, the cycle polynomials evaluated at z^(n/16) and the powers z^inc from the host,
//   4. the DEEP composition at every query position (one thread per query, two Fermat inversions each),
//   5. every FRI row folded at its layer's point (closed-form 4-point fold of fri.cu; all layers in parallel, because each layer's
//      opened rows are in the proof and only the equality "fold of layer d == opened value of layer d + 1" chains them).
// The host then applies the reference's checks in the reference's order and returns its error strings.
#include <algorithm>
#include <array>
#include <map>
#include <set>
#include "air.h"
#include "digest.cuh"
#include "host_fs.h"
#include "poly.h"
#include "prover.h"
#include "shard.h"

namespace dg {

namespace {

// ---- bincode reader (proof.rs:10-37, fri/mod.rs:17-30, merkle.rs:14-18) -------------------------------------------------------
struct Reader {
    const uint8_t *p, *end;
    bool ok = true;
    Reader(const uint8_t *b, size_t n) : p(b), end(b + n) {}
    bool need(size_t n) { if (!ok || (size_t)(end - p) < n) { ok = false; return false; } return true; }
    uint8_t u8() { if (!need(1)) return 0; return *p++; }
    uint32_t u32() { if (!need(4)) return 0; uint32_t v; memcpy(&v, p, 4); p += 4; return v; }
    uint64_t u64() { if (!need(8)) return 0; uint64_t v; memcpy(&v, p, 8); p += 8; return v; }
    fe felt() { fe v = fe_make(0, 0); if (!need(16)) return v; memcpy(&v, p, 16); p += 16; return v; }
    Digest digest() { Digest d; d.fill(0); if (!need(32)) return d; memcpy(d.data(), p, 32); p += 32; return d; }
    size_t len(size_t elem_bytes) {                              // a Vec length that the remaining bytes can actually hold
        uint64_t n = u64();
        if (!ok || n > (uint64_t)(end - p) / (elem_bytes ? elem_bytes : 1)) { ok = false; return 0; }
        return (size_t)n;
    }
    std::vector<Digest> dvec() { size_t n = len(32); std::vector<Digest> v(n); for (auto &x : v) x = digest(); return v; }
    std::vector<std::vector<Digest>> dvv() { size_t n = len(8); std::vector<std::vector<Digest>> v(n); for (auto &x : v) x = dvec(); return v; }
    std::vector<fe> fvec() { size_t n = len(16); std::vector<fe> v(n); for (auto &x : v) x = felt(); return v; }
};

struct FriLayerProof { Digest root; std::vector<std::array<fe, 4>> values; std::vector<std::vector<Digest>> nodes; uint8_t depth; };
struct ParsedProof {
    Digest trace_root, constraint_root, rem_root;
    uint8_t domain_depth, ctx_depth, loop_depth, stack_depth, c_depth;
    uint32_t op_count;
    std::vector<std::vector<Digest>> trace_nodes, c_nodes;
    std::vector<std::vector<fe>> trace_evaluations;
    std::vector<Digest> c_values;
    std::vector<fe> z1, z2, rem_values;
    std::vector<FriLayerProof> layers;
    uint64_t pow_nonce;
    uint8_t log_ext, num_queries, grinding, hash_id;
};

bool parse_proof(const uint8_t *bytes, size_t n, ParsedProof &P) {
    Reader r(bytes, n);
    P.trace_root = r.digest();
    P.domain_depth = r.u8(); P.ctx_depth = r.u8(); P.loop_depth = r.u8(); P.stack_depth = r.u8();
    P.op_count = r.u32();
    P.trace_nodes = r.dvv();
    { size_t k = r.len(8); P.trace_evaluations.resize(k); for (auto &row : P.trace_evaluations) row = r.fvec(); }
    P.constraint_root = r.digest();
    P.c_values = r.dvec(); P.c_nodes = r.dvv(); P.c_depth = r.u8();
    P.z1 = r.fvec(); P.z2 = r.fvec();
    { size_t k = r.len(41); P.layers.resize(k); }
    for (auto &l : P.layers) {
        l.root = r.digest();
        size_t k = r.len(64);
        l.values.resize(k);
        for (auto &q : l.values) for (int j = 0; j < 4; j++) q[j] = r.felt();
        l.nodes = r.dvv();
        l.depth = r.u8();
    }
    P.rem_root = r.digest();
    P.rem_values = r.fvec();
    P.pow_nonce = r.u64();
    P.log_ext = r.u8(); P.num_queries = r.u8(); P.grinding = r.u8(); P.hash_id = r.u8();
    return r.ok && r.p == r.end;
}

// ---- batch Merkle verification as a hashing plan (merkle.rs:154-263) -------------------------------------------------------------
// pool slots: the caller lays out the proof's values and nodes in a pool of 32-byte digests; computed parents get fresh slots
struct MerklePlan {
    std::vector<uint32_t> ops;            // (left, right, out) pool indices
    std::vector<uint32_t> level_start;    // op index where each level starts (+ final end)
    uint32_t root_slot = 0;
    bool ok = false;
};
MerklePlan plan_verify_batch(const std::vector<uint64_t> &indexes_in, int depth, size_t n_values, uint32_t values_base,
                             const std::vector<std::vector<Digest>> &nodes, const std::vector<uint32_t> &nodes_base, uint32_t &next_slot) {
    MerklePlan plan;
    if (depth < 1 || depth > 40) return plan;
    const uint64_t offset = 1ULL << depth;
    std::map<uint64_t, uint64_t> index_map;
    for (size_t i = 0; i < indexes_in.size(); i++) {
        if (indexes_in[i] > offset - 1) return plan;             // the reference asserts here (map_indexes)
        index_map[indexes_in[i]] = i;
    }
    if (index_map.size() != indexes_in.size()) return plan;
    std::set<uint64_t> norm;
    for (uint64_t idx : indexes_in) norm.insert(idx - (idx & 1));
    std::vector<uint64_t> indexes(norm.begin(), norm.end());
    if (indexes.size() != nodes.size()) return plan;

    std::map<uint64_t, uint32_t> v;                              // node index -> pool slot of its computed hash
    std::vector<uint64_t> next;
    std::vector<size_t> ptrs;
    plan.level_start.push_back(0);
    for (size_t i = 0; i < indexes.size(); i++) {
        const uint64_t index = indexes[i];
        auto i1 = index_map.find(index), i2 = index_map.find(index + 1);
        uint32_t left, right;
        if (i1 != index_map.end()) {
            if (n_values <= i1->second) return plan;
            left = values_base + (uint32_t)i1->second;
            if (i2 != index_map.end()) {
                if (n_values <= i2->second) return plan;
                right = values_base + (uint32_t)i2->second;
                ptrs.push_back(0);
            } else {
                if (nodes[i].size() < 1) return plan;
                right = nodes_base[i];
                ptrs.push_back(1);
            }
        } else {
            if (nodes[i].size() < 1) return plan;
            left = nodes_base[i];
            if (i2 == index_map.end()) return plan;
            if (n_values <= i2->second) return plan;
            right = values_base + (uint32_t)i2->second;
            ptrs.push_back(1);
        }
        const uint32_t out = next_slot++;
        plan.ops.insert(plan.ops.end(), {left, right, out});
        const uint64_t parent = (offset + index) >> 1;
        v[parent] = out;
        next.push_back(parent);
    }
    for (int d = 1; d < depth; d++) {
        plan.level_start.push_back((uint32_t)(plan.ops.size() / 3));
        std::vector<uint64_t> cur = next;
        next.clear();
        std::map<uint64_t, uint32_t> vnext;
        size_t i = 0;
        while (i < cur.size()) {
            const uint64_t node_index = cur[i], sibling_index = node_index ^ 1;
            uint32_t sibling;
            if (i + 1 < cur.size() && cur[i + 1] == sibling_index) {
                auto s = v.find(sibling_index);
                if (s == v.end()) return plan;
                sibling = s->second;
                i += 1;
            } else {
                // the reference indexes proof.nodes and the pointers with the position inside the CURRENT level's list
                if (i >= ptrs.size() || i >= nodes.size()) return plan;
                const size_t pointer = ptrs[i];
                if (nodes[i].size() <= pointer) return plan;
                sibling = nodes_base[i] + (uint32_t)pointer;
                ptrs[i] += 1;
            }
            auto nd = v.find(node_index);
            if (nd == v.end()) return plan;
            const uint32_t out = next_slot++;
            if (node_index & 1) plan.ops.insert(plan.ops.end(), {sibling, nd->second, out});
            else plan.ops.insert(plan.ops.end(), {nd->second, sibling, out});
            const uint64_t parent = node_index >> 1;
            vnext[parent] = out;
            next.push_back(parent);
            i += 1;
        }
        for (auto &kv : vnext) v[kv.first] = kv.second;         // parents join the map (HashMap::insert in the reference)
    }
    plan.level_start.push_back((uint32_t)(plan.ops.size() / 3));
    auto rt = v.find(1);
    if (rt == v.end()) return plan;
    plan.root_slot = rt->second;
    plan.ok = true;
    return plan;
}

struct TreeDesc { uint32_t ops_base, n_levels, levels_base, pad; };

// one block per tree: ops of a level in parallel, levels separated by barriers
template <class H>
__global__ void __launch_bounds__(128) merkle_verify_kernel(uint4 *pool, const uint32_t *__restrict__ ops, const uint32_t *__restrict__ level_start,
                                                            const TreeDesc *__restrict__ trees) {
    const TreeDesc t = trees[blockIdx.x];
    for (uint32_t l = 0; l < t.n_levels; l++) {
        const uint32_t a = level_start[t.levels_base + l], b = level_start[t.levels_base + l + 1];
        for (uint32_t o = a + threadIdx.x; o < b; o += blockDim.x) {
            const uint32_t *op = ops + 3 * (size_t)(t.ops_base + o);
            uint32_t m[16], cv[8];
            const uint4 l0 = pool[2 * (size_t)op[0]], l1 = pool[2 * (size_t)op[0] + 1], r0 = pool[2 * (size_t)op[1]], r1 = pool[2 * (size_t)op[1] + 1];
            m[0] = l0.x; m[1] = l0.y; m[2] = l0.z; m[3] = l0.w; m[4] = l1.x; m[5] = l1.y; m[6] = l1.z; m[7] = l1.w;
            m[8] = r0.x; m[9] = r0.y; m[10] = r0.z; m[11] = r0.w; m[12] = r1.x; m[13] = r1.y; m[14] = r1.z; m[15] = r1.w;
            H::hash64(m, cv);
            pool[2 * (size_t)op[2]] = make_uint4(cv[0], cv[1], cv[2], cv[3]);
            pool[2 * (size_t)op[2] + 1] = make_uint4(cv[4], cv[5], cv[6], cv[7]);
        }
        __syncthreads();
    }
}

// DEEP composition at the query positions (verifier.rs:101-162): one thread per query
struct ComposeArgs {
    int nq, w;
    const fe *rows;                 // [w][nq]
    const unsigned long long *positions;
    const fe *z1, *z2, *cc1, *cc2;  // w each
    const fe *c_evals;              // constraint evaluation at each position
    fe z, zg, c_at_z, t1_degree, t2_degree, k_constraints;
    TwiddleRef twN;
    unsigned long long inc;
    fe *out;
};
__global__ void compose_at_queries_kernel(const ComposeArgs A) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= A.nq) return;
    const unsigned long long pos = A.positions[q];
    auto pw = [&](unsigned long long e) {
        const unsigned ee = (unsigned)(e & (unsigned long long)A.twN.mask);
        return fe_mul(A.twN.lo[ee & ((1u << A.twN.lo_bits) - 1u)], A.twN.hi[ee >> A.twN.lo_bits]);
    };
    const fe x = pw(pos);
    const fe inv1 = fe_inv(fe_sub(x, A.z)), inv2 = fe_inv(fe_sub(x, A.zg));
    fe comp = fe_make(0, 0);
    for (int i = 0; i < A.w; i++) {
        const fe r = A.rows[(size_t)i * A.nq + q];
        comp = fe_add(comp, fe_mul(fe_mul(fe_sub(r, A.z1[i]), inv1), A.cc1[i]));
        comp = fe_add(comp, fe_mul(fe_mul(fe_sub(r, A.z2[i]), inv2), A.cc2[i]));
    }
    const fe xp = pw(pos * A.inc);
    const fe adj = fe_mul(fe_mul(comp, xp), A.t2_degree);
    comp = fe_add(fe_mul(comp, A.t1_degree), adj);
    const fe cv = fe_mul(fe_sub(A.c_evals[q], A.c_at_z), inv1);
    A.out[q] = fe_add(comp, fe_mul(cv, A.k_constraints));
}

// every opened FRI row folded at its layer's point: rows[t] = 4 values, pos[t] = row index, shift[t] = 2 * depth, alpha index = layer[t]
__global__ void fri_fold_rows_kernel(const fe *__restrict__ rows, const unsigned long long *__restrict__ pos, const unsigned *__restrict__ layer, int count,
                                     const fe *__restrict__ alphas, TwiddleRef inv_root, fe tau_inv, fe inv4, fe *__restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const unsigned d = layer[t];
    const fe y0 = rows[4 * t], y1 = rows[4 * t + 1], y2 = rows[4 * t + 2], y3 = rows[4 * t + 3];
    const unsigned ee = (unsigned)((pos[t] << (2 * d)) & (unsigned long long)inv_root.mask);
    const fe xinv = fe_mul(inv_root.lo[ee & ((1u << inv_root.lo_bits) - 1u)], inv_root.hi[ee >> inv_root.lo_bits]);
    const fe u = fe_mul(alphas[d], xinv);
    const fe s02 = fe_add(y0, y2), d02 = fe_sub(y0, y2), s13 = fe_add(y1, y3), d13 = fe_mul(fe_sub(y1, y3), tau_inv);
    const fe a0 = fe_add(s02, s13), a1 = fe_add(d02, d13), a2 = fe_sub(s02, s13), a3 = fe_sub(d02, d13);
    fe acc = fe_add(a2, fe_mul(u, a3));
    acc = fe_add(a1, fe_mul(u, acc));
    acc = fe_add(a0, fe_mul(u, acc));
    out[t] = fe_mul(acc, inv4);
}

template <typename T> T *upload(Context &c, DevBuf &buf, const std::vector<T> &v) {
    buf.alloc(std::max<size_t>(16, v.size() * sizeof(T)));
    if (!v.empty()) DG_CUDA(cudaMemcpyAsync(buf.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, c.stream));
    return buf.as<T>();
}

// polynom::interpolate (Lagrange, polynom.rs:106-145) followed by polynom::eval, only for the remainder check (<= 256 points)
bool remainder_is_low_degree(const std::vector<fe> &xs_all, const std::vector<fe> &ys_all, size_t degree_plus_1) {
    const size_t m = degree_plus_1;
    std::vector<fe> xs(xs_all.begin(), xs_all.begin() + m), ys(ys_all.begin(), ys_all.begin() + m);
    // barycentric weights w_i = 1 / prod_{j != i} (x_i - x_j); p(x) = sum_i y_i w_i prod_{j != i} (x - x_j)
    std::vector<fe> wgt(m);
    for (size_t i = 0; i < m; i++) {
        fe d = fe_make(1, 0);
        for (size_t j = 0; j < m; j++) if (j != i) d = fe_mul(d, fe_sub(xs[i], xs[j]));
        wgt[i] = fe_mul(ys[i], fe_inv(d));
    }
    for (size_t t = m; t < xs_all.size(); t++) {
        const fe x = xs_all[t];
        // prefix / suffix products of (x - x_j)
        std::vector<fe> pre(m + 1), suf(m + 1);
        pre[0] = fe_make(1, 0);
        for (size_t j = 0; j < m; j++) pre[j + 1] = fe_mul(pre[j], fe_sub(x, xs[j]));
        suf[m] = fe_make(1, 0);
        for (size_t j = m; j-- > 0;) suf[j] = fe_mul(suf[j + 1], fe_sub(x, xs[j]));
        fe val = fe_make(0, 0);
        for (size_t i = 0; i < m; i++) val = fe_add(val, fe_mul(wgt[i], fe_mul(pre[i], suf[i + 1])));
        if (!fe_eq(val, ys_all[t])) return false;
    }
    return true;
}

}  // namespace

// host-only view of the batch-Merkle hashing plan (CPU tests): values occupy pool slots [0, n_values), the nodes of slot i start at
// n_values + sum of the earlier slots' sizes, computed parents follow.  Returns false where verify_batch returns false before hashing.
bool host_plan_verify_batch(const std::vector<uint64_t> &indexes, int depth, size_t n_values, const std::vector<uint32_t> &node_counts,
                            std::vector<uint32_t> &ops, std::vector<uint32_t> &level_start, uint32_t &root_slot) {
    std::vector<std::vector<Digest>> nodes(node_counts.size());
    std::vector<uint32_t> bases;
    uint32_t next = (uint32_t)n_values;
    for (size_t i = 0; i < node_counts.size(); i++) { nodes[i].resize(node_counts[i]); bases.push_back(next); next += node_counts[i]; }
    MerklePlan p = plan_verify_batch(indexes, depth, n_values, 0, nodes, bases, next);
    if (!p.ok) return false;
    ops = p.ops; level_start = p.level_start; root_slot = p.root_slot;
    return true;
}

namespace {
template <class H>
std::string verify_parsed(Context &c, const ParsedProof &P, const uint8_t program_hash[32], const std::vector<fe> &inputs,
                          const std::vector<fe> &outputs) {
    DG_REQUIRE(P.log_ext >= 4 && P.log_ext <= 8, "invalid extension factor in proof options");
    DG_REQUIRE(P.domain_depth >= P.log_ext + 4 && P.domain_depth <= 30, "invalid domain depth");
    DG_REQUIRE(inputs.size() <= 8 && outputs.size() <= 8, "cannot have more than 8 public inputs / outputs");
    const uint64_t b = 1ULL << P.log_ext, N = 1ULL << P.domain_depth, n = N >> P.log_ext;
    const int log_N = P.domain_depth, log_n = log_N - P.log_ext;
    const int w = 15 + P.ctx_depth + P.loop_depth + P.stack_depth;
    DG_REQUIRE(P.ctx_depth <= 16 && P.loop_depth <= 8 && P.stack_depth >= 1 && P.stack_depth <= 32 && w < 128, "invalid register counts in the proof");

    // ---- 1: PoW, query positions (verifier.rs:19-31)
    std::vector<uint8_t> fri_roots;
    for (auto &l : P.layers) fri_roots.insert(fri_roots.end(), l.root.begin(), l.root.end());
    fri_roots.insert(fri_roots.end(), P.rem_root.begin(), P.rem_root.end());
    DG_REQUIRE(fri_roots.size() <= 1024, "too many FRI layers");
    uint8_t seed[32], pseed[32];
    H::message(fri_roots.data(), fri_roots.size(), seed);
    pow_hash<H>(seed, P.pow_nonce, pseed);
    {
        uint64_t o0;
        memcpy(&o0, pseed, 8);
        const unsigned tz = o0 == 0 ? 64u : (unsigned)__builtin_ctzll(o0);
        if (tz < P.grinding) return "seed proof-of-work verification failed";
    }
    std::vector<uint64_t> t_positions;
    try { t_positions = fs::query_positions(pseed, N, b, P.num_queries); }
    catch (const std::exception &e) { return e.what(); }
    const std::vector<uint64_t> c_positions = fs::constraint_positions(t_positions);
    const int nq = (int)t_positions.size();
    // ---- 2: minimum op count (verifier.rs:34-37; MIN_TRACE_LENGTH = 16)
    if (P.op_count < 16) return "Verification of minimum operation count failed";
    if ((int)P.trace_evaluations.size() != nq) return "verification of trace Merkle proof failed";
    for (auto &row : P.trace_evaluations) DG_REQUIRE((int)row.size() == w, "trace evaluation row has wrong width");
    DG_REQUIRE((int)P.z1.size() == w && (int)P.z2.size() == w, "deep value vector has wrong width");

    // ---- pool of digests: [trace row hashes | constraint values | FRI row hashes per layer | all proof nodes | computed parents]
    std::vector<Digest> pool;
    auto reserve = [&](size_t k) { uint32_t base = (uint32_t)pool.size(); pool.resize(pool.size() + k); return base; };
    auto put_nodes = [&](const std::vector<std::vector<Digest>> &nodes) {
        std::vector<uint32_t> bases;
        for (auto &slot : nodes) { bases.push_back((uint32_t)pool.size()); pool.insert(pool.end(), slot.begin(), slot.end()); }
        return bases;
    };
    const uint32_t tv_base = reserve(nq);
    const uint32_t cv_base = (uint32_t)pool.size();
    pool.insert(pool.end(), P.c_values.begin(), P.c_values.end());
    std::vector<uint32_t> fv_base;
    for (auto &l : P.layers) fv_base.push_back(reserve(l.values.size()));
    const std::vector<uint32_t> tn_bases = put_nodes(P.trace_nodes), cn_bases = put_nodes(P.c_nodes);
    std::vector<std::vector<uint32_t>> fn_bases;
    for (auto &l : P.layers) fn_bases.push_back(put_nodes(l.nodes));
    uint32_t next_slot = (uint32_t)pool.size();

    // FRI positions per layer (fri/verifier.rs:24-31)
    std::vector<std::vector<uint64_t>> layer_pos(P.layers.size()), layer_aug(P.layers.size());
    {
        std::vector<uint64_t> pos = t_positions;
        uint64_t domain = N;
        for (size_t d = 0; d < P.layers.size(); d++) {
            layer_pos[d] = pos;
            layer_aug[d] = fs::augmented_positions(pos, domain);
            pos = layer_aug[d];
            domain /= 4;
        }
    }
    std::vector<MerklePlan> plans;
    plans.push_back(plan_verify_batch(t_positions, P.domain_depth, nq, tv_base, P.trace_nodes, tn_bases, next_slot));
    plans.push_back(plan_verify_batch(c_positions, P.c_depth, P.c_values.size(), cv_base, P.c_nodes, cn_bases, next_slot));
    for (size_t d = 0; d < P.layers.size(); d++)
        plans.push_back(plan_verify_batch(layer_aug[d], P.layers[d].depth, P.layers[d].values.size(), fv_base[d], P.layers[d].nodes, fn_bases[d], next_slot));
    pool.resize(next_slot);

    ArenaScope arena_scope;
    // ---- device: leaves
    DevBuf d_pool, d_rows, d_fri_rows;
    uint4 *pool_dev = (uint4 *)upload(c, d_pool, pool);
    std::vector<fe> rows_cm((size_t)w * nq);                       // column-major [w][nq]
    for (int q = 0; q < nq; q++) for (int j = 0; j < w; j++) rows_cm[(size_t)j * nq + q] = P.trace_evaluations[q][j];
    const fe *rows_dev = upload(c, d_rows, rows_cm);
    hash_rows_plain<H>(c, rows_dev, pool_dev + 2 * (size_t)tv_base, w, nq);
    std::vector<fe> fri_rows;
    std::vector<unsigned long long> fri_pos;
    std::vector<unsigned> fri_layer;
    std::vector<size_t> fri_off;
    for (size_t d = 0; d < P.layers.size(); d++) {
        fri_off.push_back(fri_pos.size());
        for (size_t j = 0; j < P.layers[d].values.size(); j++) {
            for (int k = 0; k < 4; k++) fri_rows.push_back(P.layers[d].values[j][k]);
            fri_pos.push_back(j < layer_aug[d].size() ? layer_aug[d][j] : 0);
            fri_layer.push_back((unsigned)d);
        }
    }
    const fe *fri_rows_dev = upload(c, d_fri_rows, fri_rows);
    for (size_t d = 0; d < P.layers.size(); d++)
        if (!P.layers[d].values.empty())
            hash64_contiguous<H>(c, fri_rows_dev + 4 * fri_off[d], pool_dev + 2 * (size_t)fv_base[d], P.layers[d].values.size());

    // ---- device: all Merkle plans
    std::vector<uint32_t> ops, level_start;
    std::vector<TreeDesc> trees;
    for (auto &pl : plans) {
        TreeDesc t{(uint32_t)(ops.size() / 3), 0, (uint32_t)level_start.size(), 0};
        if (pl.ok) {
            t.n_levels = (uint32_t)pl.level_start.size() - 1;
            ops.insert(ops.end(), pl.ops.begin(), pl.ops.end());
            level_start.insert(level_start.end(), pl.level_start.begin(), pl.level_start.end());
        } else {
            level_start.push_back(0);
        }
        trees.push_back(t);
    }
    DevBuf d_ops, d_ls, d_trees;
    const uint32_t *ops_dev = upload(c, d_ops, ops);
    const uint32_t *ls_dev = upload(c, d_ls, level_start);
    const TreeDesc *trees_dev = upload(c, d_trees, trees);
    merkle_verify_kernel<H><<<(unsigned)trees.size(), 128, 0, c.stream>>>(pool_dev, ops_dev, ls_dev, trees_dev); c.launches++;
    DG_CUDA(cudaGetLastError());

    // ---- 4: constraints at z (verifier.rs:47-52, 79-97)
    const fe z = fs::prng_vector(P.constraint_root.data(), 1)[0];
    const fe root_n = host_root_of_unity(log_n), x_last = host_inv(root_n);
    fe program_hash_fe[2];
    memcpy(program_hash_fe, program_hash, 32);
    fs::ConstraintCoefficients cc = fs::draw_constraint_coefficients(P.trace_root.data(), P.ctx_depth, P.loop_depth, P.stack_depth, inputs, outputs,
                                                                      fe_make(P.op_count, 0), program_hash_fe);
    const size_t T = cc.coefA.size();
    static const int GROUP_DEG[6] = {2, 3, 4, 6, 7, 8};
    std::vector<fe> hostvals;                                    // [coefA T | coefB T | periodic 23 | xpow 6]
    hostvals.insert(hostvals.end(), cc.coefA.begin(), cc.coefA.end());
    hostvals.insert(hostvals.end(), cc.coefB.begin(), cc.coefB.end());
    const std::vector<fe> per = fs::periodic_at(fe_pow_u64(z, n / 16));
    hostvals.insert(hostvals.end(), per.begin(), per.end());
    for (int gi = 0; gi < 6; gi++) hostvals.push_back(fe_pow_u64(z, (8 * n - 1) - (n - 1) * GROUP_DEG[gi]));
    DevBuf d_hostvals, d_fake, d_tev;
    const fe *hv = upload(c, d_hostvals, hostvals);
    // the two rows as a 128-step "trace" of one coset: step 0 = trace(z), step 1 = trace(z g) (its "next" row)
    std::vector<fe> fake((size_t)w * 128, fe_make(0, 0));
    for (int j = 0; j < w; j++) { fake[(size_t)j * 128] = P.z1[j]; fake[(size_t)j * 128 + 1] = P.z2[j]; }
    const fe *fake_dev = upload(c, d_fake, fake);
    d_tev.alloc(128 * 16);
    {
        AirParams A;
        memset(&A, 0, sizeof A);
        A.w = w; A.ctx_depth = P.ctx_depth; A.loop_depth = P.loop_depth; A.stack_depth = P.stack_depth;
        A.cl = std::max<int>(P.ctx_depth, 1); A.ll = std::max<int>(P.loop_depth, 1); A.sl = std::max<int>(P.stack_depth, 8);
        A.log_n = 7; A.log_blowup = 3;
        A.ext = fake_dev; A.col_stride = 128;
        A.c8_base = 0; A.num_c8 = 1;
        A.t_ev = d_tev.as<fe>();
        A.periodic = hv + 2 * T;                                   // unused in verify mode (per_override is set)
        A.coefA = hv; A.coefB = hv + T;
        A.twN = c.twiddle(10, false);
        A.violation = nullptr;
        A.verify_mode = 1;
        A.per_override = hv + 2 * T;
        A.xpow_override = hv + 2 * T + 23;
        launch_constraint_eval(c, A);
    }

    // ---- 5: DEEP composition at the query positions (verifier.rs:54-69, 101-162)
    fs::CompositionCoefficients dc = fs::draw_composition_coefficients(P.constraint_root.data(), w);
    // the constraint evaluation opened at each trace position: half of constraint leaf position / 2
    std::vector<fe> c_evals(nq);
    for (int q = 0; q < nq; q++) {
        const uint64_t position = t_positions[q];
        const size_t leaf_idx = std::find(c_positions.begin(), c_positions.end(), position / 2) - c_positions.begin();
        if (leaf_idx >= P.c_values.size()) return "verification of constraint Merkle proof failed";
        memcpy(&c_evals[q], P.c_values[leaf_idx].data() + (position % 2) * 16, 16);
    }
    DevBuf d_pos, d_zs, d_cev, d_comp;
    std::vector<unsigned long long> pos64(t_positions.begin(), t_positions.end());
    std::vector<fe> zs;                                            // [z1 w | z2 w | cc1 w | cc2 w]
    zs.insert(zs.end(), P.z1.begin(), P.z1.end()); zs.insert(zs.end(), P.z2.begin(), P.z2.end());
    zs.insert(zs.end(), dc.trace1.begin(), dc.trace1.end()); zs.insert(zs.end(), dc.trace2.begin(), dc.trace2.end());
    const fe *zs_dev = upload(c, d_zs, zs);
    d_comp.alloc(std::max(16, nq * 16));

    // t(z) is needed by the composition: read it back first (one small copy), then finish on the host what is scalar work
    fe t_at_z;
    DG_CUDA(cudaMemcpyAsync(&t_at_z, d_tev.p, 16, cudaMemcpyDeviceToHost, c.stream));
    DG_CUDA(cudaStreamSynchronize(c.stream));
    fe c_at_z;
    {
        // boundary numerators at z (evaluator.rs:181-326): I(z) = sum_j a_j s1_j - Ka + z^adj (sum_j b_j s1_j - Kb), same for the last step
        const fe zadj = fe_pow_u64(z, 6 * n + 2);
        fe ia = fe_make(0, 0), ib = ia, fa = ia, fb = ia;
        for (int j = 0; j < cc.n_boundary_regs; j++) {
            ia = fe_add(ia, fe_mul(P.z1[j], cc.bAi[j])); ib = fe_add(ib, fe_mul(P.z1[j], cc.bBi[j]));
            fa = fe_add(fa, fe_mul(P.z1[j], cc.bAf[j])); fb = fe_add(fb, fe_mul(P.z1[j], cc.bBf[j]));
        }
        const fe i_value = fe_add(fe_sub(ia, cc.KiA), fe_mul(zadj, fe_sub(ib, cc.KiB)));
        const fe f_value = fe_add(fe_sub(fa, cc.KfA), fe_mul(zadj, fe_sub(fb, cc.KfB)));
        // field::div(a, b) = a * inv(b) with inv(0) = 0 (field.rs:75-84)
        fe zz = fe_sub(z, fe_make(1, 0));
        fe result = fe_mul(i_value, fe_inv(zz));
        zz = fe_sub(z, x_last);
        result = fe_add(result, fe_mul(f_value, fe_inv(zz)));
        zz = fe_mul(fe_sub(fe_pow_u64(z, n), fe_make(1, 0)), fe_inv(zz));
        result = fe_add(result, fe_mul(t_at_z, fe_inv(zz)));
        c_at_z = result;
    }
    {
        ComposeArgs A;
        A.nq = nq; A.w = w; A.rows = rows_dev;
        A.positions = upload(c, d_pos, pos64);
        A.z1 = zs_dev; A.z2 = zs_dev + w; A.cc1 = zs_dev + 2 * w; A.cc2 = zs_dev + 3 * w;
        A.c_evals = upload(c, d_cev, c_evals);
        A.z = z; A.zg = fe_mul(z, root_n); A.c_at_z = c_at_z;
        A.t1_degree = dc.t1_degree; A.t2_degree = dc.t2_degree; A.k_constraints = dc.constraints;
        A.twN = c.twiddle(log_N, false);
        A.inc = (8 * n - 1 - n) - (n - 2);                        // get_incremental_trace_degree: composition degree - (n - 2), composition degree = 7n - 1
        A.out = d_comp.as<fe>();
        compose_at_queries_kernel<<<(nq + 63) / 64, 64, 0, c.stream>>>(A); c.launches++;
        DG_CUDA(cudaGetLastError());
    }

    // ---- 6: FRI rows folded at their layers' points (fri/verifier.rs:33-75)
    std::vector<fe> alphas;
    for (auto &l : P.layers) alphas.push_back(fs::prng_vector(l.root.data(), 1)[0]);
    DevBuf d_alphas, d_fpos, d_flayer, d_folded;
    const int n_fri = (int)fri_pos.size();
    d_folded.alloc(std::max(16, n_fri * 16));
    if (n_fri > 0) {
        const fe *al = upload(c, d_alphas, alphas);
        const unsigned long long *fp = upload(c, d_fpos, fri_pos);
        const unsigned *fl = upload(c, d_flayer, fri_layer);
        fri_fold_rows_kernel<<<(n_fri + 127) / 128, 128, 0, c.stream>>>(fri_rows_dev, fp, fl, n_fri, al, c.twiddle(log_N, true), host_inv(host_root_of_unity(2)),
                                                                          host_inv(fe_make(4, 0)), d_folded.as<fe>()); c.launches++;
        DG_CUDA(cudaGetLastError());
    }

    // ---- results back
    std::vector<Digest> pool_out(pool.size());
    std::vector<fe> comp(nq), folded(n_fri);
    DG_CUDA(cudaMemcpyAsync(pool_out.data(), pool_dev, pool.size() * 32, cudaMemcpyDeviceToHost, c.stream));
    DG_CUDA(cudaMemcpyAsync(comp.data(), d_comp.p, (size_t)nq * 16, cudaMemcpyDeviceToHost, c.stream));
    if (n_fri) DG_CUDA(cudaMemcpyAsync(folded.data(), d_folded.p, (size_t)n_fri * 16, cudaMemcpyDeviceToHost, c.stream));
    DG_CUDA(cudaStreamSynchronize(c.stream));

    // ---- the reference's checks, in its order
    auto root_ok = [&](const MerklePlan &pl, const Digest &root) { return pl.ok && pool_out[pl.root_slot] == root; };
    if (!root_ok(plans[0], P.trace_root)) return "verification of trace Merkle proof failed";
    if (!root_ok(plans[1], P.constraint_root)) return "verification of constraint Merkle proof failed";

    std::string fri_err;
    {
        if (P.layers.empty()) return "verification of low-degree proof failed: no FRI layers";
        std::vector<fe> evaluations = comp;
        std::vector<uint64_t> positions = t_positions;
        uint64_t domain_size = (1ULL << P.layers[0].depth) * 4;
        uint64_t max_degree_plus_1 = (7 * n - 1) + 1;           // get_composition_degree(n) + 1
        fe domain_root = host_root_of_unity(P.layers[0].depth + 2);
        for (size_t d = 0; d < P.layers.size() && fri_err.empty(); d++) {
            const FriLayerProof &layer = P.layers[d];
            const std::vector<uint64_t> aug = fs::augmented_positions(positions, domain_size);
            const uint64_t row_length = domain_size / 4;
            std::vector<fe> column_values;
            for (uint64_t p : positions) {
                const size_t idx = std::find(aug.begin(), aug.end(), p % row_length) - aug.begin();
                if (idx >= layer.values.size()) { fri_err = "layer values too short"; break; }
                column_values.push_back(layer.values[idx][p / row_length]);
            }
            if (!fri_err.empty()) break;
            bool same = evaluations.size() == column_values.size();
            for (size_t i = 0; same && i < evaluations.size(); i++) same = fe_eq(evaluations[i], column_values[i]);
            if (!same) { fri_err = "evaluations did not match column value at depth " + std::to_string(d); break; }
            if (!root_ok(plans[2 + d], layer.root)) { fri_err = "verification of Merkle proof failed at layer " + std::to_string(d); break; }
            if (layer.values.size() < aug.size()) { fri_err = "layer values too short"; break; }
            evaluations.assign(folded.begin() + fri_off[d], folded.begin() + fri_off[d] + aug.size());
            for (int s = 0; s < 2; s++) domain_root = fe_sqr(domain_root);
            max_degree_plus_1 /= 4;
            domain_size /= 4;
            positions = aug;
        }
        if (fri_err.empty()) {
            for (size_t i = 0; i < positions.size(); i++)
                if (positions[i] >= P.rem_values.size() || !fe_eq(P.rem_values[positions[i]], evaluations[i])) {
                    fri_err = "remainder values are inconsistent with values of the last column";
                    break;
                }
        }
        if (fri_err.empty()) {                                      // verify_remainder (fri/verifier.rs:97-131)
            const std::vector<fe> &rem = P.rem_values;
            if (max_degree_plus_1 > rem.size()) fri_err = "remainder degree is greater than number of remainder values";
            else {
                std::vector<fe> xs, ys;
                fe xpow = fe_make(1, 0);
                for (size_t i = 0; i < rem.size(); i++) {
                    if (i % b != 0) { xs.push_back(xpow); ys.push_back(rem[i]); }
                    xpow = fe_mul(xpow, domain_root);
                }
                if (max_degree_plus_1 > xs.size()) fri_err = "remainder degree is greater than number of remainder values";
                else if (!remainder_is_low_degree(xs, ys, (size_t)max_degree_plus_1))
                    fri_err = "remainder is not a valid degree " + std::to_string(max_degree_plus_1 - 1) + " polynomial";
            }
        }
    }
    if (!fri_err.empty()) return "verification of low-degree proof failed: " + fri_err;
    return "";
}
}  // namespace

// returns "" when the proof is accepted, the reference's error string otherwise; throws Error for malformed input / CUDA failures
std::string verify_proof(Context &c, const uint8_t program_hash[32], const std::vector<fe> &inputs, const std::vector<fe> &outputs,
                         const uint8_t *proof_bytes, size_t proof_len) {
    ParsedProof P;
    if (!parse_proof(proof_bytes, proof_len, P)) throw Error(DG_ERR_INVALID, "malformed proof bytes (bincode layout of StarkProof, proof.rs:10-37)");
    if (P.hash_id != Blake3Hash::id && P.hash_id != Sha3Hash::id) return "unsupported hash function";
    return with_proof_hash(P.hash_id, [&](auto h) { return verify_parsed<decltype(h)>(c, P, program_hash, inputs, outputs); });
}

}  // namespace dg
