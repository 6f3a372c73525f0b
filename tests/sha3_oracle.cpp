// TEST INFRASTRUCTURE ONLY.  The CPU oracle of oracle/ (a restatement of the reference's prover and verifier) with SHA3-256 as the
// commitment hash, for the tests of sha3 proofs.  Compiled on demand by tests/sha3_oracle.py; nothing in distaff_b200/ uses it.
//
//   hash::sha3  /root/reference/src/crypto/hash.rs:212-218 -> crate sha3 (Sha3_256; NOT in the reference tree): restated here from
//               FIPS 202 (August 2015) and pinned in tests against Python's hashlib.sha3_256.
//
// The oracle's prover already hashes every commitment with ProofOptions::hash_fn (stark.h), whose default is `blake3`, and its verifier
// accepts hash id 0 only.  This file keeps oracle/ as it is: the default `blake3` of stark.h is routed to commit_hash(), which calls the
// hash selected for the current call (one call at a time).  A sha3 proof is the oracle's proof with the options' hash byte set to 4 (what
// the reference stores for hash::sha3, options.rs:106-108); it is verified by the oracle's verifier with the byte read as 0 and sha3
// selected, so a proof relabelled from one hash to the other is checked with the wrong hash and rejected.
#include "../oracle/crypto.h"
#include <mutex>
#include <vector>

namespace oracle {
namespace keccak {
// section 3.2.5 (iota) via Algorithm 5: rc(t) = bit 0 of the LFSR x^8 + x^6 + x^5 + x^4 + 1 after t steps
static inline int rc_bit(int t) {
    if (t % 255 == 0) return 1;
    uint32_t r = 1;                                      // R[0] is bit 0, R[7] bit 7
    for (int i = 1; i <= t % 255; i++) {
        r <<= 1;                                         // R = 0 || R
        const uint32_t r8 = (r >> 8) & 1;
        r ^= r8 | (r8 << 4) | (r8 << 5) | (r8 << 6);     // R[0] ^= R[8], R[4] ^= R[8], R[5] ^= R[8], R[6] ^= R[8]
        r &= 0xff;                                       // Trunc_8
    }
    return r & 1;
}
struct Tables {
    int rho[25] = {0};
    uint64_t rc[24] = {0};
    Tables() {
        for (int t = 0, x = 1, y = 0; t < 24; t++) {     // section 3.2.2: offsets along the walk (x, y) <- (y, 2x + 3y) from (1, 0)
            rho[x + 5 * y] = ((t + 1) * (t + 2) / 2) % 64;
            const int nx = y, ny = (2 * x + 3 * y) % 5;
            x = nx; y = ny;
        }
        for (int ir = 0; ir < 24; ir++)                  // Algorithm 6: RC[2^j - 1] = rc(j + 7 ir)
            for (int j = 0; j <= 6; j++) rc[ir] |= (uint64_t)rc_bit(j + 7 * ir) << ((1 << j) - 1);
    }
};
static inline uint64_t rotl(uint64_t v, int n) { n %= 64; return n ? (v << n) | (v >> (64 - n)) : v; }
// Algorithm 7 with the step mappings of section 3.2 on A[x + 5y]
static inline void permute(uint64_t A[25]) {
    static const Tables T;
    for (int ir = 0; ir < 24; ir++) {
        uint64_t C[5], D[5], B[25];
        for (int x = 0; x < 5; x++) C[x] = A[x] ^ A[x + 5] ^ A[x + 10] ^ A[x + 15] ^ A[x + 20];          // theta
        for (int x = 0; x < 5; x++) D[x] = C[(x + 4) % 5] ^ rotl(C[(x + 1) % 5], 1);
        for (int i = 0; i < 25; i++) A[i] ^= D[i % 5];
        for (int x = 0; x < 5; x++)                                                                      // rho, then pi: A'[x, y] = A[x + 3y, x]
            for (int y = 0; y < 5; y++) B[x + 5 * y] = rotl(A[(x + 3 * y) % 5 + 5 * x], T.rho[(x + 3 * y) % 5 + 5 * x]);
        for (int x = 0; x < 5; x++)                                                                      // chi
            for (int y = 0; y < 5; y++) A[x + 5 * y] = B[x + 5 * y] ^ (~B[(x + 1) % 5 + 5 * y] & B[(x + 2) % 5 + 5 * y]);
        A[0] ^= T.rc[ir];                                                                                // iota
    }
}
} // namespace keccak

// section 6.1: SHA3-256(M) = Keccak[512](M || 01, 256); section 5.1 / B.2: the padded message ends 0x06 00 .. 00 0x80 (or 0x86)
static inline void sha3_256(const uint8_t *in, size_t len, uint8_t *out32) {
    const size_t rate = 136;
    std::vector<uint8_t> m(in, in + len);
    m.push_back(0x06);
    while (m.size() % rate) m.push_back(0);
    m.back() |= 0x80;
    uint64_t A[25] = {0};
    for (size_t off = 0; off < m.size(); off += rate) {
        for (size_t i = 0; i < rate / 8; i++)
            for (int b = 0; b < 8; b++) A[i] ^= (uint64_t)m[off + 8 * i + b] << (8 * b);
        keccak::permute(A);
    }
    for (int i = 0; i < 32; i++) out32[i] = (uint8_t)(A[i / 8] >> (8 * (i % 8)));
}

static HashFn g_commit = blake3;                        // the hash of the current call (read by the oracle's worker threads too)
static std::mutex g_call;                               // one call at a time
static inline void commit_hash(const uint8_t *in, size_t len, uint8_t *out32) { g_commit(in, len, out32); }
} // namespace oracle

#define blake3 commit_hash
#include "../oracle/stark.h"
#undef blake3

using namespace oracle;

namespace {
const uint8_t SHA3_ID = 4;
struct Select {                                         // selects the commitment hash for one call
    std::lock_guard<std::mutex> lk;
    explicit Select(HashFn h) : lk(g_call) { g_commit = h; }
    ~Select() { g_commit = blake3; }
};
} // namespace

extern "C" {

int so_set_threads(int t) { if (t >= 1) fft::host_threads() = t; return fft::host_threads(); }

void so_sha3(const uint8_t *in, uint64_t len, uint8_t *out32) { sha3_256(in, len, out32); }

// build_merkle_nodes (merkle.rs:269-294) with sha3; nodes_out: n * 32 bytes, heap layout
void so_merkle_nodes(const uint8_t *leaves, uint64_t n, uint8_t *nodes_out) {
    std::vector<Digest> l(n);
    memcpy(l.data(), leaves, n * 32);
    std::vector<Digest> nodes = build_merkle_nodes(l, sha3_256);
    memcpy(nodes_out, nodes.data(), n * 32);
}

// prove with ProofOptions(ext, num_queries, grinding, hash_fn = sha3); cols: column-major w x n field elements.  Returns the proof
// length (bytes copied to out when it fits in cap), or -1 with the error message in err.
int64_t so_prove(const uint8_t *cols, uint32_t w, uint64_t n, uint32_t ctx_depth, uint32_t loop_depth, const uint8_t *inputs, uint32_t n_in,
                 const uint8_t *outputs, uint32_t n_out, uint32_t ext, uint32_t num_queries, uint32_t grinding, uint8_t *out, uint64_t cap,
                 char *err, uint32_t err_cap) {
    try {
        std::vector<std::vector<u128>> regs(w, std::vector<u128>(n));
        for (uint32_t j = 0; j < w; j++) memcpy(regs[j].data(), cols + (size_t)j * n * 16, n * 16);
        std::vector<u128> in(n_in), o(n_out);
        if (n_in) memcpy(in.data(), inputs, n_in * 16);
        if (n_out) memcpy(o.data(), outputs, n_out * 16);
        ProofOptions opt;
        opt.extension_factor = ext; opt.num_queries = num_queries; opt.grinding_factor = grinding;
        StarkProof p;
        {
            Select s(sha3_256);
            p = prove(regs, ctx_depth, loop_depth, in, o, opt);
        }
        p.opt_hash_id = SHA3_ID;
        const std::vector<uint8_t> bytes = serialize(p);
        if (bytes.size() <= cap) memcpy(out, bytes.data(), bytes.size());
        return (int64_t)bytes.size();
    } catch (std::exception &e) {
        snprintf(err, err_cap, "%s", e.what());
        return -1;
    }
}

// stark::verify of blake3 (hash byte 0) and sha3 (hash byte 4) proofs: 0 when accepted, else 1 and the error message in err
int so_verify(const uint8_t *program_hash32, const uint8_t *inputs, uint32_t n_in, const uint8_t *outputs, uint32_t n_out, const uint8_t *proof,
              uint64_t proof_len, char *err, uint32_t err_cap) {
    std::string msg;
    try {
        std::vector<u128> in(n_in), o(n_out);
        if (n_in) memcpy(in.data(), inputs, n_in * 16);
        if (n_out) memcpy(o.data(), outputs, n_out * 16);
        StarkProof p = deserialize(proof, proof_len);
        const bool sha3 = p.opt_hash_id == SHA3_ID;
        if (sha3) p.opt_hash_id = 0;
        Select s(sha3 ? sha3_256 : blake3);
        msg = verify(program_hash32, in, o, p);
    } catch (std::exception &e) { msg = std::string("exception: ") + e.what(); }
    if (msg.empty()) return 0;
    snprintf(err, err_cap, "%s", msg.c_str());
    return 1;
}

}  // extern "C"
