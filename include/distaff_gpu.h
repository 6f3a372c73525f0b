/* distaff_gpu.h -- C-ABI of the B200 (sm_100a) STARK prover backend for Distaff.
 *
 * The reference has no FFI seam; the seam this library replaces is the single call
 *     stark::prove(&mut trace, inputs, outputs, options) -> StarkProof
 * at /root/reference/src/lib.rs:62  (definition: /root/reference/src/stark/prover.rs:17-169).
 * INTEGRATION.md shows the Rust binding (extern "C" block + replacement body of prover.rs::prove).
 *
 * Conventions
 *   - field elements are 16 little-endian bytes (a Rust u128, /root/reference/src/utils/mod.rs:35-41), canonical < M;
 *   - digests are 32 bytes; all sizes are in elements unless a name says bytes;
 *   - every function returns 0 on success and a negative code on failure; dg_last_error() describes the failure;
 *     nothing unwinds across the boundary;  there is NO CPU fallback: without a CUDA device every call fails with -3;
 *   - the caller owns input buffers (read-only for the duration of the call) and output buffers it passes in;
 *     objects returned through dg_proof_t** are owned by the library until dg_proof_free();
 *   - calls are serialised internally (one context per process, one device: $DG_DEVICE or dg_init()).
 */
#ifndef DISTAFF_GPU_H
#define DISTAFF_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DG_OK 0
#define DG_ERR_INVALID (-1)      /* bad argument (mirrors the reference's assert!s, e.g. trace_table.rs:23-58, options.rs:29-50) */
#define DG_ERR_CUDA (-2)         /* CUDA runtime failure */
#define DG_ERR_NO_DEVICE (-3)    /* no CUDA device: this backend has no CPU path */
#define DG_ERR_EXHAUSTED (-4)    /* PoW / query-position search exhausted (utils/mod.rs:39-41 panics in the reference) */
#define DG_ERR_UNSATISFIED (-5)  /* transition constraints do not vanish on the trace (evaluator.rs:152-157 panics) */
#define DG_ERR_REJECTED (-6)     /* dg_verify: the proof was rejected; the message is the reference's Err(String) (verifier.rs:28-73) */

/* ---- lifecycle ------------------------------------------------------------------------------------------------- */
int dg_init(int device);                     /* optional; device < 0 = $DG_DEVICE or 0; an error if the library already runs on another device */
/* Single-process multi-GPU: after dg_init_devices(n) (n = 1, 2, 4 or 8; devices 0 .. n-1) ONE call of dg_prove / dg_prove_device from one
 * host thread shards the proof over the n GPUs -- the library runs one internal host thread and one NCCL communicator per device -- and
 * returns the same bytes as the single-GPU call.  This is the mode the seam at lib.rs:62 (one synchronous call in one process) needs;
 * the one-process-per-GPU mode (dg_comm_init below) remains for hosts that already run one rank per GPU. */
int dg_init_devices(int n_devices);
const char *dg_last_error(void);             /* thread-local message of the last failing call */
int dg_device_info(char *name, size_t cap, int *sm_count, size_t *total_mem);

/* ---- the hot path: replaces stark::prove (prover.rs:17) ----------------------------------------------------------- */
typedef struct {
    const uint8_t *const *columns; /* width pointers, each to length*16 bytes: register traces, column-major (trace_table.rs:10) */
    uint32_t width;                /* 15 + ctx_depth + loop_depth + stack_depth (trace_state.rs:115-118)                    */
    uint64_t length;               /* trace length n, power of two >= 16                                                    */
    uint32_t ctx_depth, loop_depth;/* as returned by processor::execute (processor/mod.rs:23-46)                            */
} dg_trace_t;

typedef struct {                   /* ProofOptions (options.rs:16-23) */
    uint32_t extension_factor;     /* 16..256, power of two (default 32) */
    uint32_t num_queries;          /* 1..128 (default 50)                */
    uint32_t grinding_factor;      /* 0..32 (default 20)                 */
    uint32_t hash_id;              /* DG_HASH_BLAKE3 (0, default) or DG_HASH_SHA3 (4): the hash of every commitment of the proof */
} dg_options_t;

typedef struct dg_proof dg_proof_t;

typedef struct {                   /* per-stage device time in ms, the nine steps of prover.rs:19-167 */
    float stage_ms[9];
    float h2d_ms, total_ms;
    uint64_t kernel_launches;
} dg_prove_stats_t;

int dg_prove(const dg_trace_t *trace, const uint8_t *inputs16, uint32_t n_inputs, const uint8_t *outputs16, uint32_t n_outputs,
             const dg_options_t *options, dg_proof_t **proof_out, dg_prove_stats_t *stats /* may be NULL */);
/* same, with the register traces already resident in device memory: one allocation of width*length*16 bytes, column-major */
int dg_prove_device(const void *d_registers, uint32_t width, uint64_t length, uint32_t ctx_depth, uint32_t loop_depth,
                    const uint8_t *inputs16, uint32_t n_inputs, const uint8_t *outputs16, uint32_t n_outputs,
                    const dg_options_t *options, dg_proof_t **proof_out, dg_prove_stats_t *stats);

/* Optional: randomness supplied by the host.  The prover derives all of its Fiat-Shamir challenges from two reference functions,
 *   field::prng_vector(seed, n)                            (math/field.rs:264-275: StdRng::from_seed + Uniform(0..M))
 *   utils::compute_query_positions(seed, domain, options)  (stark/utils/mod.rs:25-44: StdRng + Uniform(0..domain), rejections)
 * both built on rand 0.7.3, which is not part of the reference tree.  By default the library uses its own restatement of that
 * generator (ChaCha20, rand's widening-multiply rejection sampling); a Rust host can instead register callbacks that call the real
 * functions, so that no third-party semantics are reproduced on this side of the boundary.  Callbacks return 0 on success; they are
 * called 20-30 times per proof (once per commitment), one at a time: on the thread that calls dg_prove, and after dg_init_devices(n) also
 * from the library's per-device host threads (every rank derives the same challenges; the calls are serialised by a mutex).  draw_field writes `count` canonical field
 * elements (16 LE bytes each); draw_positions writes exactly num_queries distinct positions < domain_size, none a multiple of
 * extension_factor (anything else is rejected with DG_ERR_INVALID; a non-zero return maps to DG_ERR_EXHAUSTED like the reference's panic).
 * Passing NULL restores the built-in generator.  Process-wide; not to be changed while a proof is running. */
typedef struct {
    void *user;
    int (*draw_field)(void *user, const uint8_t seed[32], uint64_t count, uint8_t *out16);
    int (*draw_positions)(void *user, const uint8_t seed[32], uint64_t domain_size, uint32_t extension_factor, uint32_t num_queries,
                          uint64_t *out_positions);
} dg_rng_callbacks_t;
int dg_set_rng_callbacks(const dg_rng_callbacks_t *callbacks);

/* bincode 1.3.1 encoding of StarkProof (proof.rs:10-37), what main.rs:45 serialises.  Its last byte is the hash id of the options
 * (the last field of StarkProof): 0 for blake3.  A sha3 proof is written in the same layout with that byte set to 4 -- an extension of
 * this interface: the reference's serializer refuses sha3 (options.rs:97-120), so a Rust caller deserialises such bytes with the byte
 * set to 0 and restores the options it proved with (INTEGRATION.md section 2).  dg_verify reads the byte back the same way. */
int dg_proof_serialized_len(const dg_proof_t *proof, size_t *len);
int dg_proof_serialize(const dg_proof_t *proof, uint8_t *buf, size_t cap);
/* intermediate commitments, for differential tests: which = 0 trace root, 1 constraint root, 2 PoW seed */
int dg_proof_digest(const dg_proof_t *proof, int which, uint8_t out32[32]);
int dg_proof_pow_nonce(const dg_proof_t *proof, uint64_t *nonce);
void dg_proof_free(dg_proof_t *proof);

/* ---- the step after the path: stark::verify (verifier.rs:11-75) on the GPU -------------------------------------------------------
 * Checks StarkProof bytes (the bincode encoding dg_proof_serialize emits / main.rs:45 writes) against a program hash and public
 * inputs / outputs.  Returns DG_OK when the reference would return Ok(true); DG_ERR_REJECTED when it would return Err(msg), with msg
 * copied to `message` (NUL-terminated, truncated to message_cap) and available from dg_last_error(); DG_ERR_INVALID for bytes that do
 * not deserialize.  Hashing, Merkle batch verification, the constraint evaluation at z, the DEEP composition at the query positions
 * and the FRI row folds run on the device (verifier.cu); the Fiat-Shamir draws use the same generator / callbacks as dg_prove. */
int dg_verify(const uint8_t program_hash[32], const uint8_t *inputs16, uint32_t n_inputs, const uint8_t *outputs16, uint32_t n_outputs,
              const uint8_t *proof_bytes, size_t proof_len, char *message, size_t message_cap);

/* ---- building blocks (micro-benchmarks of BASELINE.json config 5; same kernels the prover uses) ---------------------- */
/* math::fft / polynom::{eval_fft, interpolate_fft} (polynom.rs:23-28,82-86): natural-order DFT of `batch` vectors of 2^log_n
 * elements, in place in host memory */
int dg_ntt(uint8_t *values, uint32_t log_n, uint32_t batch, int inverse);
/* TraceTable::extend (trace_table.rs:143-169) for `batch` columns: n values in, n*blowup evaluations out in LOGICAL order
 * (out[i] = P(w_N^i)), host memory */
int dg_lde(const uint8_t *values, uint8_t *extended, uint32_t log_n, uint32_t log_blowup, uint32_t batch);
/* crypto::build_merkle_nodes (merkle.rs:269-294) with blake3: n_leaves*32 bytes in, n_leaves*32 bytes of nodes out */
int dg_merkle_build(const uint8_t *leaves, uint64_t n_leaves, uint8_t *nodes);
/* TraceTable::build_merkle_tree leaf step (trace_table.rs:176-183): hashes the rows of a column-major width x rows matrix */
int dg_hash_rows(const uint8_t *columns, uint32_t width, uint64_t rows, uint8_t *digests);
/* utils::find_pow_nonce (proof_of_work.rs:4-32) */
int dg_find_pow_nonce(const uint8_t seed[32], uint32_t grinding_factor, uint64_t *nonce, uint8_t new_seed[32]);
/* crypto::hash::{blake3, rescue, poseidon, sha3} (hash.rs:119-177,205-218) over n independent 64-byte messages -> n 32-byte digests
 * (benches/hash.rs), and build_merkle_nodes (merkle.rs:269-294) with any of them.  hash: 0 blake3, 1 rescue, 2 poseidon, 4 sha3 (SHA3-256)
 * -- ids of THIS interface (3 is GMiMC, which has no GPU kernel).  A proof can carry blake3 or sha3 (dg_options_t.hash_id): rescue,
 * poseidon and GMiMC absorb at most 64 bytes and a trace row is longer, so the reference panics when it commits with them.
 * Messages must hold valid field elements for 1 and 2 (field.rs:25). */
#define DG_HASH_BLAKE3 0
#define DG_HASH_RESCUE 1
#define DG_HASH_POSEIDON 2
#define DG_HASH_SHA3 4
int dg_hash64(int hash, const uint8_t *messages64, uint64_t n, uint8_t *digests32);
int dg_merkle_build_with(int hash, const uint8_t *leaves, uint64_t n_leaves, uint8_t *nodes);
/* element-wise field ops on vectors (op: 0 add, 1 sub, 2 mul, 3 inv, 4 exp(a, b)), for differential tests of the arithmetic;
 * impl: 0 = PTX path used by the kernels, 1 = portable C++ path, 2 / 3 = earlier PTX multiplies (op 2 only) */
int dg_field_op(int op, int impl, const uint8_t *a, const uint8_t *b, uint8_t *out, uint64_t n);

/* ---- device-resident variants (timed with CUDA events on the library's stream; *ms may be NULL) ----------------------- */
int dg_dev_alloc(void **ptr, size_t bytes);
int dg_dev_free(void *ptr);
int dg_dev_upload(void *dst, const void *src, size_t bytes);
int dg_dev_download(void *dst, const void *src, size_t bytes);
int dg_dev_sync(void);
int dg_dev_ntt(void *d_values, uint32_t log_n, uint32_t batch, int inverse, float *ms);
/* d_polys: batch x n coefficients; d_ext: batch x (n << log_blowup) evaluations, coset-major ([c][k] = LDE index k*blowup + c) */
int dg_dev_lde(const void *d_polys, void *d_ext, uint32_t log_n, uint32_t log_blowup, uint32_t batch, float *ms);
int dg_dev_merkle_build(const void *d_leaves, uint64_t n_leaves, void *d_nodes, float *ms);
int dg_dev_merkle_build_with(int hash, const void *d_leaves, uint64_t n_leaves, void *d_nodes, float *ms);
/* d_ext coset-major as produced by dg_dev_lde; d_leaves: (n << log_blowup) digests in logical row order */
int dg_dev_hash_rows(const void *d_ext, uint32_t width, uint32_t log_n, uint32_t log_blowup, void *d_leaves, float *ms);
/* writes > L2-size scratch to evict the L2 between timed iterations */
int dg_dev_flush_l2(void);

/* ---- multi-GPU: one process per GPU, the proof of ONE trace is sharded by LDE coset ranges over `world` ranks ----------------
 * Every rank calls dg_prove / dg_prove_device with the SAME trace and options; every rank returns the same proof bytes.
 * Rank 0 obtains the 128-byte NCCL id, the host distributes it (e.g. torch.distributed broadcast), all ranks call dg_comm_init. */
int dg_comm_unique_id(uint8_t id128[128]);
int dg_comm_init(int rank, int world /* 1, 2, 4 or 8 */, const uint8_t id128[128]);
int dg_comm_finalize(void);
/* index algebra of the sharded Merkle trees, exported for CPU tests: locates level-0 item `index` (is_node = 0) or the internal
 * node with global heap index `index` (is_node = 1) of a tree with n blocks of 2^log_blk items per rank over 2^log_g ranks;
 * out = {owner rank or -1 if replicated, 1 if in the replicated upper heap else 0, local index} */
int dg_host_shard_locate(uint64_t n, int log_blk, int log_g, int is_node, uint64_t index, int64_t out[3]);

/* ---- host-side Fiat-Shamir glue, exported so that it can be unit-tested without a GPU (none of these touch the device) ---- */
/* field::prng_vector (field.rs:271-275): count draws of StdRng::from_seed(seed) through Uniform(0..M) */
int dg_host_prng_vector(const uint8_t seed[32], uint64_t count, uint8_t *out16);
/* utils::compute_query_positions (stark/utils/mod.rs:25-44) */
int dg_host_query_positions(const uint8_t seed[32], uint64_t domain_size, uint32_t extension_factor, uint32_t num_queries, uint64_t *out);
/* blake3 of a message of at most 1024 bytes (the FRI-roots seed of prover.rs:119-127) */
int dg_host_blake3(const uint8_t *data, size_t len, uint8_t out32[32]);
/* SHA3-256 (FIPS 202) of a message of any length: the FRI-roots seed of a sha3 proof */
int dg_host_sha3(const uint8_t *data, size_t len, uint8_t out32[32]);
/* MerkleTree::prove_batch planning (merkle.rs:64-124): writes, per normalised slot, the count and then (is_leaf, index) pairs;
 * out layout: [n_slots][depth] then for each slot [count] (is_leaf, index)*count, all uint64 */
int dg_host_plan_batch(const uint64_t *indexes, uint32_t n_indexes, uint64_t n_leaves, uint64_t *out, size_t cap, size_t *written);
/* MerkleTree::verify_batch (merkle.rs:154-263) as the hashing plan dg_verify executes on the device: digests live in a pool -- the proof's
 * values in slots [0, n_values), the nodes of slot i from n_values + node_counts[0..i) on, computed parents after them; ops = (left, right,
 * out) slot triples, level_start[l] .. level_start[l+1] the ops of level l; the tree is accepted iff pool[root_slot] equals the root.
 * Returns DG_ERR_REJECTED where verify_batch returns false for structural reasons. */
int dg_host_merkle_verify_plan(const uint64_t *indexes, uint32_t n_indexes, uint32_t depth, uint32_t n_values, const uint32_t *node_counts,
                               uint32_t n_slots, uint32_t *ops, size_t ops_cap, uint32_t *n_ops, uint32_t *level_start, size_t levels_cap,
                               uint32_t *n_levels, uint32_t *root_slot);
/* extend_constants tables (constraints/utils.rs:87-113): 128 rows x 23 columns = sponge ARK 8 | masks 3 | hasher ARK 12 */
int dg_host_periodic_tables(uint8_t *out16 /* 128*23 elements */);

#ifdef __cplusplus
}
#endif
#endif /* DISTAFF_GPU_H */
