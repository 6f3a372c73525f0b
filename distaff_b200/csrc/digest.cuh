// The commitment hash of a proof as a type: every digest site of the prover and verifier (row leaves, Merkle levels, FRI rows,
// constraint leaf pairs, proof of work, FRI-roots seed) is a template over it, and with_proof_hash() is the one place where the hash
// id of the proof options picks the instantiation.
//   blake3   hash id 0 (the default; the only hash the reference can serialise, options.rs:97-120)   blake3.cuh
//   sha3     hash id 4 (SHA3-256, hash.rs:212-218)                                                   keccak.cuh
#pragma once
#include "../../include/distaff_gpu.h"
#include "blake3.cuh"
#include "host_fs.h"
#include "keccak.cuh"

namespace dg {

struct Blake3Hash {
    static constexpr uint32_t id = DG_HASH_BLAKE3;
    __host__ __device__ static void hash64(const uint32_t m[16], uint32_t out[8]) { b3::hash64(m, out); }
    static void message(const uint8_t *data, size_t len, uint8_t out[32]) { fs::blake3_short(data, len, out); }
};
struct Sha3Hash {
    static constexpr uint32_t id = DG_HASH_SHA3;
    __host__ __device__ static void hash64(const uint32_t m[16], uint32_t out[8]) { sha3::hash64(m, out); }
    static void message(const uint8_t *data, size_t len, uint8_t out[32]) { fs::sha3_256(data, len, out); }
};

// nullptr when a proof can commit with `hash_id`, otherwise why not
inline const char *proof_hash_error(uint32_t hash_id) {
    if (hash_id == Blake3Hash::id || hash_id == Sha3Hash::id) return nullptr;
    if (hash_id >= 1 && hash_id <= 3)
        return "rescue, poseidon and gmimc (hash ids 1-3) absorb at most 64 bytes and a trace row is longer: the reference panics in "
               "build_merkle_tree with them; use blake3 (0) or sha3 (4)";
    return "unsupported hash function id (0 = blake3, 4 = sha3)";
}

// f(Blake3Hash{}) or f(Sha3Hash{}) for a hash id that proof_hash_error() accepts
template <class F>
auto with_proof_hash(uint32_t hash_id, F &&f) {
    return hash_id == Sha3Hash::id ? f(Sha3Hash{}) : f(Blake3Hash{});
}

}  // namespace dg
