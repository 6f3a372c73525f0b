// Host-side Fiat-Shamir glue (see host_fs.h for the reference lines each piece follows).
#include "host_fs.h"
#include <algorithm>
#include <cstring>
#include <mutex>
#include <stdexcept>
#include "air_constants.h"
#include "blake3.cuh"
#include "keccak.cuh"

namespace dg {
namespace fs {

typedef unsigned __int128 u128;

// ---- ChaCha20 (rand_chacha 0.2: 64-bit block counter in words 12-13, stream id 0, 20 rounds) -----------------------------
static inline uint32_t rol(uint32_t x, int n) { return (x << n) | (x >> (32 - n)); }
#define DG_QR(a, b, c, d) \
    a += b; d = rol(d ^ a, 16); c += d; b = rol(b ^ c, 12); a += b; d = rol(d ^ a, 8); c += d; b = rol(b ^ c, 7);

Rng::Rng(const uint8_t seed[32]) : counter_(0), pos_(16) { memcpy(key_, seed, 32); }

void Rng::refill() {
    uint32_t in[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u};
    for (int i = 0; i < 8; i++) in[4 + i] = key_[i];
    in[12] = (uint32_t)counter_; in[13] = (uint32_t)(counter_ >> 32); in[14] = 0; in[15] = 0;
    uint32_t x[16];
    memcpy(x, in, sizeof x);
    for (int r = 0; r < 10; r++) {
        DG_QR(x[0], x[4], x[8], x[12]) DG_QR(x[1], x[5], x[9], x[13]) DG_QR(x[2], x[6], x[10], x[14]) DG_QR(x[3], x[7], x[11], x[15])
        DG_QR(x[0], x[5], x[10], x[15]) DG_QR(x[1], x[6], x[11], x[12]) DG_QR(x[2], x[7], x[8], x[13]) DG_QR(x[3], x[4], x[9], x[14])
    }
    for (int i = 0; i < 16; i++) buf_[i] = x[i] + in[i];
    counter_++;
    pos_ = 0;
}
uint32_t Rng::next_u32() { if (pos_ >= 16) refill(); return buf_[pos_++]; }
uint64_t Rng::next_u64() { uint64_t lo = next_u32(); uint64_t hi = next_u32(); return lo | (hi << 32); }

// UniformInt<u128>::sample for the range [0, M): v*M as a 256-bit product, accept when the low half <= M - 1
fe Rng::field() {
    const u128 Mv = ((u128)DG_M_HI << 64) | DG_M_LO;
    for (;;) {
        uint64_t v0 = next_u64(), v1 = next_u64();           // Standard u128: low word first
        u128 p00 = (u128)v0 * DG_M_LO, p01 = (u128)v0 * DG_M_HI, p10 = (u128)v1 * DG_M_LO, p11 = (u128)v1 * DG_M_HI;
        u128 mid = (p00 >> 64) + (uint64_t)p01 + (uint64_t)p10;
        u128 lo = ((u128)(uint64_t)mid << 64) | (uint64_t)p00;
        u128 hi = p11 + (p01 >> 64) + (p10 >> 64) + (mid >> 64);
        if (lo <= Mv - 1) return fe_make((uint64_t)hi, (uint64_t)(hi >> 64));
    }
}
uint64_t Rng::below(uint64_t range) {
    const uint64_t reject = (0 - range) % range;
    const uint64_t zone = ~(uint64_t)0 - reject;
    for (;;) {
        u128 p = (u128)next_u64() * range;
        if ((uint64_t)p <= zone) return (uint64_t)(p >> 64);
    }
}
static RngHooks g_hooks = {nullptr, nullptr, nullptr};
static std::mutex g_hooks_mu;              // single-process multi-GPU: the ranks are host threads; callbacks run one at a time
void set_rng_hooks(const RngHooks *hooks) { if (hooks) g_hooks = *hooks; else g_hooks = RngHooks{nullptr, nullptr, nullptr}; }
bool rng_hooks_active() { return g_hooks.draw_field != nullptr || g_hooks.draw_positions != nullptr; }

std::vector<fe> prng_vector(const uint8_t seed[32], size_t count) {
    std::vector<fe> v(count);
    if (g_hooks.draw_field) {
        {
            std::lock_guard<std::mutex> lk(g_hooks_mu);
            if (g_hooks.draw_field(g_hooks.user, seed, count, reinterpret_cast<uint8_t *>(v.data())) != 0)
                throw std::runtime_error("draw_field callback failed");
        }
        for (auto &x : v)                                     // field::prng_vector yields canonical elements (Uniform over 0..M)
            if (x.hi == DG_M_HI && x.lo >= DG_M_LO) throw std::runtime_error("draw_field callback returned a non-canonical field element");
        return v;
    }
    Rng g(seed);
    for (size_t i = 0; i < count; i++) v[i] = g.field();
    return v;
}

// ---- BLAKE3, single chunk ------------------------------------------------------------------------------------------------
void blake3_short(const uint8_t *data, size_t len, uint8_t out[32]) {
    if (len > 1024) throw std::runtime_error("blake3_short: message longer than one chunk");
    uint32_t cv[8];
    b3::iv(cv);
    const size_t nblocks = len == 0 ? 1 : (len + 63) / 64;
    for (size_t b = 0; b < nblocks; b++) {
        uint8_t buf[64];
        memset(buf, 0, 64);
        const size_t take = len == 0 ? 0 : std::min<size_t>(64, len - b * 64);
        memcpy(buf, data + b * 64, take);
        uint32_t m[16];
        memcpy(m, buf, 64);
        uint32_t flags = 0;
        if (b == 0) flags |= b3::CHUNK_START;
        if (b == nblocks - 1) flags |= b3::CHUNK_END | b3::ROOT;
        b3::compress(cv, m, 0, (uint32_t)take, flags);
    }
    memcpy(out, cv, 32);
}

// ---- SHA3-256 ---------------------------------------------------------------------------------------------------------------
void sha3_256(const uint8_t *data, size_t len, uint8_t out[32]) {
    uint64_t a[25] = {0};
    for (size_t off = 0;; off += 136) {                          // 136-byte blocks; the last one (possibly empty) carries the padding
        uint8_t block[136] = {0};
        const size_t take = off < len ? std::min<size_t>(136, len - off) : 0;
        if (take) memcpy(block, data + off, take);
        const bool last = take < 136;
        if (last) { block[take] ^= 0x06; block[135] ^= 0x80; }
        for (int i = 0; i < 17; i++) { uint64_t v; memcpy(&v, block + 8 * i, 8); a[i] ^= v; }
        sha3::keccak_f(a);
        if (last) break;
    }
    uint32_t o[8];
    sha3::squeeze(a, o);
    memcpy(out, o, 32);
}

// ---- coefficients ----------------------------------------------------------------------------------------------------------
static const int DEG_STATIC[20] = {2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 8, 8, 6, 4, 6, 7, 6, 6, 4};

ConstraintCoefficients draw_constraint_coefficients(const uint8_t trace_root[32], int ctx_depth, int loop_depth, int stack_depth,
                                                    const std::vector<fe> &inputs, const std::vector<fe> &outputs, fe op_count,
                                                    const fe program_hash[2]) {
    const int NUM_BOUNDARY = 47, NUM_TRANSITION = 78;
    std::vector<fe> c = prng_vector(trace_root, 2 * (NUM_TRANSITION + 2 * NUM_BOUNDARY));
    const fe *bi = c.data(), *bf = c.data() + 2 * NUM_BOUNDARY, *tr = c.data() + 4 * NUM_BOUNDARY;
    const int cl = std::max(ctx_depth, 1), ll = std::max(loop_depth, 1), sl = std::max(stack_depth, 8);

    ConstraintCoefficients r;
    // ---- transition: compact the MAX-depth layout, then hand each constraint the pair of its flattened slot
    std::vector<fe> compact;
    auto take = [&](int src, int count) { for (int k = 0; k < count; k++) compact.push_back(tr[src + k]); };
    take(0, 40); take(40, 2 * cl); take(40 + 32, 2 * ll); take(40 + 32 + 16, 4); take(40 + 32 + 16 + 4, 2 * sl);
    const int T = 20 + cl + ll + 2 + stack_depth;
    std::vector<int> degree(T);
    for (int j = 0; j < 20; j++) degree[j] = DEG_STATIC[j];
    for (int j = 20; j < 20 + cl + ll; j++) degree[j] = 4;
    for (int j = 20 + cl + ll; j < T; j++) degree[j] = 7;
    r.coefA.assign(T, fe_make(0, 0));
    r.coefB.assign(T, fe_make(0, 0));
    int slot = 0;
    for (int d = 0; d <= 8; d++)
        for (int j = 0; j < T; j++)
            if (degree[j] == d) { r.coefA[j] = compact[2 * slot]; r.coefB[j] = compact[2 * slot + 1]; slot++; }

    // ---- boundary: per-register coefficient vectors + constants
    const int io = (int)std::max(inputs.size(), outputs.size());
    const int stack_regs = std::min(stack_depth, io);
    r.n_boundary_regs = 15 + ctx_depth + loop_depth + stack_regs;
    const fe Z = fe_make(0, 0), ONEv = fe_make(1, 0);
    r.bAi.assign(r.n_boundary_regs, Z); r.bBi.assign(r.n_boundary_regs, Z);
    r.bAf.assign(r.n_boundary_regs, Z); r.bBf.assign(r.n_boundary_regs, Z);
    r.KiA = r.KiB = r.KfA = r.KfB = Z;
    auto set = [&](int reg, int off, bool first, bool last, fe exp_i, fe exp_f) {
        // off = index of the coefficient pair inside a boundary block; reg < 0: register does not exist (constants only)
        if (first) {
            if (reg >= 0) { r.bAi[reg] = bi[off]; r.bBi[reg] = bi[off + 1]; }
            r.KiA = fe_add(r.KiA, fe_mul(exp_i, bi[off])); r.KiB = fe_add(r.KiB, fe_mul(exp_i, bi[off + 1]));
        }
        if (last) {
            if (reg >= 0) { r.bAf[reg] = bf[off]; r.bBf[reg] = bf[off + 1]; }
            r.KfA = fe_add(r.KfA, fe_mul(exp_f, bf[off])); r.KfB = fe_add(r.KfB, fe_mul(exp_f, bf[off + 1]));
        }
    };
    set(0, 0, true, true, Z, op_count);                                                        // op_counter
    for (int i = 0; i < 4; i++) set(1 + i, 2 + 2 * i, true, i < 2, Z, i < 2 ? program_hash[i] : Z);   // sponge / program hash
    for (int q = 0; q < 10; q++) set(5 + q, 10 + 2 * q, true, true, Z, ONEv);                  // op bits: 0 at the start, 1 at the end
    for (int i = 0; i < ctx_depth; i++) set(15 + i, 30 + 2 * i, true, true, Z, Z);
    for (int i = 0; i < loop_depth; i++) set(15 + ctx_depth + i, 62 + 2 * i, true, true, Z, Z);
    for (int i = 0; i < io; i++) {
        const int reg = i < stack_depth ? 15 + ctx_depth + loop_depth + i : -1;
        set(reg, 78 + 2 * i, i < (int)inputs.size(), i < (int)outputs.size(), i < (int)inputs.size() ? inputs[i] : Z,
            i < (int)outputs.size() ? outputs[i] : Z);
    }
    return r;
}

CompositionCoefficients draw_composition_coefficients(const uint8_t constraint_root[32], int width) {
    const int MAXR = 128;
    std::vector<fe> c = prng_vector(constraint_root, 1 + 4 * MAXR + 3);
    CompositionCoefficients r;
    r.z = c[0];
    r.trace1.assign(c.begin() + 1, c.begin() + 1 + width);
    r.trace2.assign(c.begin() + 1 + 2 * MAXR, c.begin() + 1 + 2 * MAXR + width);
    r.t1_degree = c[1 + 4 * MAXR];
    r.t2_degree = c[2 + 4 * MAXR];
    r.constraints = c[3 + 4 * MAXR];
    return r;
}

std::vector<uint64_t> query_positions(const uint8_t seed[32], uint64_t domain_size, uint64_t extension_factor, uint32_t num_queries) {
    if (g_hooks.draw_positions) {
        std::vector<uint64_t> got(num_queries);
        {
            std::lock_guard<std::mutex> lk(g_hooks_mu);
            if (g_hooks.draw_positions(g_hooks.user, seed, domain_size, (uint32_t)extension_factor, num_queries, got.data()) != 0)
                throw std::runtime_error("needed more query positions than could be generated");
        }
        for (size_t i = 0; i < got.size(); i++) {             // the invariants compute_query_positions guarantees (stark/utils/mod.rs:31-41)
            if (got[i] >= domain_size || got[i] % extension_factor == 0 || std::find(got.begin(), got.begin() + i, got[i]) != got.begin() + i)
                throw std::runtime_error("draw_positions callback returned an invalid position set");
        }
        return got;
    }
    Rng g(seed);
    std::vector<uint64_t> out;
    for (int attempt = 0; attempt < 1000 && out.size() < num_queries; attempt++) {
        const uint64_t v = g.below(domain_size);
        if (v % extension_factor == 0) continue;
        if (std::find(out.begin(), out.end(), v) != out.end()) continue;
        out.push_back(v);
    }
    if (out.size() < num_queries) throw std::runtime_error("needed more query positions than could be generated");
    return out;
}
std::vector<uint64_t> constraint_positions(const std::vector<uint64_t> &positions) {
    std::vector<uint64_t> out;
    for (uint64_t p : positions)
        if (std::find(out.begin(), out.end(), p / 2) == out.end()) out.push_back(p / 2);
    return out;
}
std::vector<uint64_t> augmented_positions(const std::vector<uint64_t> &positions, uint64_t column_length) {
    const uint64_t rows = column_length / 4;
    std::vector<uint64_t> out;
    for (uint64_t p : positions)
        if (std::find(out.begin(), out.end(), p % rows) == out.end()) out.push_back(p % rows);
    return out;
}

// ---- periodic tables --------------------------------------------------------------------------------------------------------
static fe g40() { return fe_make(0x86b8723e1920f4aaULL, 0x120532e7b364080aULL); }
static fe root_of_unity(int log_order) { fe r = g40(); for (int i = 0; i < 40 - log_order; i++) r = fe_sqr(r); return r; }

// the 23 periodic columns (sponge ARK 8 | masks 3 | hasher ARK 12) as polynomials of degree < 16 in y = x^(n/16): coefficient vectors
static std::vector<std::vector<fe>> periodic_polys() {
    std::vector<std::vector<fe>> cols;
    auto add_table = [&](const unsigned long long (*t)[2], int ncols) {
        for (int c = 0; c < ncols; c++) {
            std::vector<fe> v(16);
            for (int k = 0; k < 16; k++) v[k] = fe_make(t[c * 16 + k][0], t[c * 16 + k][1]);
            cols.push_back(v);
        }
    };
    add_table(DG_SPONGE_ARK, 8);
    static const int MASKS[3][16] = {{0, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1},      // decoder/mod.rs:219-223
                                     {1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0},
                                     {0, 1, 1, 1, 1, 1, 1, 1, 0, 1, 1, 1, 1, 1, 1, 1}};
    for (int m = 0; m < 3; m++) {
        std::vector<fe> v(16);
        for (int k = 0; k < 16; k++) v[k] = fe_make(MASKS[m][k], 0);
        cols.push_back(v);
    }
    add_table(DG_HASHER_ARK, 12);
    const fe w16_inv = fe_inv(root_of_unity(4)), inv16 = fe_inv(fe_make(16, 0));
    std::vector<fe> p16(16);
    p16[0] = fe_make(1, 0);
    for (int i = 1; i < 16; i++) p16[i] = fe_mul(p16[i - 1], w16_inv);
    std::vector<std::vector<fe>> polys(cols.size(), std::vector<fe>(16));
    for (size_t c = 0; c < cols.size(); c++)
        for (int k = 0; k < 16; k++) {                       // inverse DFT: cycle values -> coefficients
            fe acc = fe_make(0, 0);
            for (int r = 0; r < 16; r++) acc = fe_add(acc, fe_mul(cols[c][r], p16[(r * k) & 15]));
            polys[c][k] = fe_mul(acc, inv16);
        }
    return polys;
}

std::vector<fe> periodic_tables() {
    const std::vector<std::vector<fe>> polys = periodic_polys();
    const fe w128 = root_of_unity(7);
    std::vector<fe> p128(128);
    p128[0] = fe_make(1, 0);
    for (int i = 1; i < 128; i++) p128[i] = fe_mul(p128[i - 1], w128);
    std::vector<fe> out(128 * 23);
    for (size_t c = 0; c < polys.size(); c++)
        for (int s = 0; s < 128; s++) {                      // evaluate on the 8x extended cycle
            fe acc = fe_make(0, 0);
            for (int k = 0; k < 16; k++) acc = fe_add(acc, fe_mul(polys[c][k], p128[(s * k) & 127]));
            out[(size_t)s * 23 + c] = acc;
        }
    return out;
}

// the same 23 columns at an arbitrary point: y = x^(trace_length / 16)  (decoder/mod.rs evaluate_at, stack/mod.rs evaluate_at)
std::vector<fe> periodic_at(fe y) {
    const std::vector<std::vector<fe>> polys = periodic_polys();
    std::vector<fe> out(23);
    for (size_t c = 0; c < polys.size(); c++) {
        fe acc = fe_make(0, 0);
        for (int k = 15; k >= 0; k--) acc = fe_add(fe_mul(acc, y), polys[c][k]);
        out[c] = acc;
    }
    return out;
}

// ---- batch proofs --------------------------------------------------------------------------------------------------------------
BatchPlan plan_batch_proof(const std::vector<uint64_t> &indexes, uint64_t n_leaves) {
    BatchPlan plan;
    plan.value_leaves = indexes;
    std::vector<uint64_t> sorted(indexes);
    std::sort(sorted.begin(), sorted.end());
    if (std::adjacent_find(sorted.begin(), sorted.end()) != sorted.end()) throw std::runtime_error("repeating indexes detected");
    auto requested = [&](uint64_t i) { return std::binary_search(sorted.begin(), sorted.end(), i); };
    std::vector<uint64_t> pairs;                              // even-aligned, ascending, unique
    for (uint64_t i : sorted) {
        const uint64_t e = i & ~(uint64_t)1;
        if (pairs.empty() || pairs.back() != e) pairs.push_back(e);
    }
    std::vector<uint64_t> level;
    for (uint64_t e : pairs) {
        std::vector<NodeRef> first;
        const bool has0 = requested(e), has1 = requested(e + 1);
        if (has0 && !has1) first.push_back(NodeRef{true, e + 1});
        else if (!has0) first.push_back(NodeRef{true, e});
        plan.nodes.push_back(first);
        level.push_back((e + n_leaves) >> 1);
    }
    uint8_t depth = 0;
    while (((uint64_t)1 << depth) < n_leaves) depth++;
    plan.depth = depth;
    for (int d = 1; d < depth; d++) {
        std::vector<uint64_t> up;
        for (size_t i = 0; i < level.size(); i++) {
            const uint64_t sibling = level[i] ^ 1;
            if (i + 1 < level.size() && level[i + 1] == sibling) i++;
            else plan.nodes[i].push_back(NodeRef{false, sibling});     // slot = position in this level's list (merkle.rs:112)
            up.push_back(sibling >> 1);
        }
        level.swap(up);
    }
    return plan;
}

}  // namespace fs
}  // namespace dg
