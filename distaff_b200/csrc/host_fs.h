// Host-side Fiat-Shamir glue of the prover: everything in the reference's prove path that is a few hundred bytes of
// sequential work and therefore stays on the CPU:
//   field::prng / prng_vector (StdRng = ChaCha20, Uniform)      /root/reference/src/math/field.rs:264-275
//   ConstraintCoefficients / CompositionCoefficients             /root/reference/src/stark/utils/coefficients.rs:63-185
//   utils::compute_query_positions / map_trace_to_constraint...  /root/reference/src/stark/utils/mod.rs:25-53
//   MerkleTree::prove_batch index planning                       /root/reference/src/crypto/merkle.rs:64-124
//   fri::utils::get_augmented_positions                          /root/reference/src/stark/fri/utils.rs:4-14
//   periodic constant tables (extend_constants)                  /root/reference/src/stark/constraints/utils.rs:87-113
//   bincode encoding of StarkProof                               /root/reference/src/stark/proof.rs:10-37
// The rand 0.7.3 / bincode 1.3.1 crates are not vendored with the reference; their semantics are restated from the
// crates' documented algorithms (see DESIGN.md, "unpinned third-party semantics").
#pragma once
#include <cstdint>
#include <vector>
#include "fp128.cuh"

namespace dg {
namespace fs {

// ---- StdRng ---------------------------------------------------------------------------------------------------------
class Rng {
public:
    explicit Rng(const uint8_t seed[32]);
    uint64_t next_u64();
    fe field();                           // Uniform::from(0..M).sample
    uint64_t below(uint64_t range);       // Uniform::from(0..range).sample for usize
private:
    uint32_t key_[8], buf_[16];
    uint64_t counter_;
    int pos_;
    void refill();
    uint32_t next_u32();
};
std::vector<fe> prng_vector(const uint8_t seed[32], size_t count);

// Optional host-supplied randomness (dg_set_rng_callbacks): when set, prng_vector / query_positions ask the host instead of the
// built-in restatement of rand 0.7.3 -- a Rust host passes closures over the real StdRng / Uniform, which removes the one
// third-party semantic this library would otherwise have to reproduce from the crate's documentation (SURVEY.md section 8b).
struct RngHooks {
    void *user;
    int (*draw_field)(void *user, const uint8_t seed[32], uint64_t count, uint8_t *out16);
    int (*draw_positions)(void *user, const uint8_t seed[32], uint64_t domain_size, uint32_t extension_factor, uint32_t num_queries, uint64_t *out);
};
void set_rng_hooks(const RngHooks *hooks);     // nullptr: built-in generator
bool rng_hooks_active();

// ---- BLAKE3 of a short message (<= 1024 bytes) on the host -------------------------------------------------------------
void blake3_short(const uint8_t *data, size_t len, uint8_t out[32]);
// ---- SHA3-256 of a message of any length on the host (keccak.cuh) ---------------------------------------------------------
void sha3_256(const uint8_t *data, size_t len, uint8_t out[32]);

// ---- constraint coefficients, arranged for the evaluation kernel --------------------------------------------------------
struct ConstraintCoefficients {
    std::vector<fe> coefA, coefB;                 // per transition constraint in evaluation order
    std::vector<fe> bAi, bBi, bAf, bBf;           // per register (length n_boundary_regs)
    fe KiA, KiB, KfA, KfB;
    int n_boundary_regs;
};
ConstraintCoefficients draw_constraint_coefficients(const uint8_t trace_root[32], int ctx_depth, int loop_depth, int stack_depth,
                                                    const std::vector<fe> &inputs, const std::vector<fe> &outputs, fe op_count,
                                                    const fe program_hash[2]);
struct CompositionCoefficients {
    fe z;
    std::vector<fe> trace1, trace2;               // first `width` coefficients
    fe t1_degree, t2_degree, constraints;
};
CompositionCoefficients draw_composition_coefficients(const uint8_t constraint_root[32], int width);

std::vector<uint64_t> query_positions(const uint8_t seed[32], uint64_t domain_size, uint64_t extension_factor, uint32_t num_queries);
std::vector<uint64_t> constraint_positions(const std::vector<uint64_t> &positions);
std::vector<uint64_t> augmented_positions(const std::vector<uint64_t> &positions, uint64_t column_length);

// periodic tables of the evaluation domain: 128 rows x 23 columns (sponge ARK 8 | masks 3 | hasher ARK 12)
std::vector<fe> periodic_tables();
std::vector<fe> periodic_at(fe y);          // the 23 columns at y = x^(n/16) for an arbitrary x (verifier)

// ---- batch Merkle proof planning ----------------------------------------------------------------------------------------
struct NodeRef { bool leaf; uint64_t index; };
struct BatchPlan {
    std::vector<uint64_t> value_leaves;           // leaf index per requested index (request order)
    std::vector<std::vector<NodeRef>> nodes;      // per normalised index slot
    uint8_t depth;
};
BatchPlan plan_batch_proof(const std::vector<uint64_t> &indexes, uint64_t n_leaves);

// ---- bincode ------------------------------------------------------------------------------------------------------------
struct ByteWriter {
    std::vector<uint8_t> b;
    void u8(uint8_t v) { b.push_back(v); }
    void u32(uint32_t v) { for (int i = 0; i < 4; i++) b.push_back((uint8_t)(v >> (8 * i))); }
    void u64(uint64_t v) { for (int i = 0; i < 8; i++) b.push_back((uint8_t)(v >> (8 * i))); }
    void felt(fe v) { u64(v.lo); u64(v.hi); }
    void raw(const uint8_t *p, size_t n) { b.insert(b.end(), p, p + n); }
};

}  // namespace fs
}  // namespace dg
