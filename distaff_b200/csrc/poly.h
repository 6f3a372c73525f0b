// Polynomial / scan / gather kernels (poly.cu) and FRI kernels (fri.cu).
#pragma once
#include "common.cuh"

namespace dg {

// two-level table of powers of an arbitrary base: base^e = lo[e & (2^lo_bits - 1)] * hi[e >> lo_bits],  e < len
struct PowRef { const fe *lo, *hi; int lo_bits; };
struct PowTable {
    DevBuf lo, hi;
    int lo_bits = 0;
    PowTable(Context &c, fe base, unsigned long long len);
    PowRef ref() const { PowRef r; r.lo = lo.as<fe>(); r.hi = hi.as<fe>(); r.lo_bits = lo_bits; return r; }
};

void suffix_scan_exclusive(Context &c, fe *data, unsigned long long len);
void syn_div(Context &c, const fe *in, fe *out, fe *scratch, unsigned long long len, const PowRef &b_pows, const PowRef &binv_pows, fe sub0);
void syn_div_expanded_sum(Context &c, const fe *a, fe *scratch, const fe *add0, const fe *add1, fe *out, unsigned long long n, unsigned long long len, fe e);
void eval_polys_at(Context &c, const fe *polys, unsigned long long n, int cols, const PowRef &zt, const TwiddleRef &gt, bool two_points, fe *out);
void boundary_coeffs(Context &c, const fe *polys, unsigned long long n, int nb, const fe *coef, fe KiA, fe KiB, fe KfA, fe KfB, fe *ic, fe *fc);
// finishes the coset-by-coset interpolation of 8n evaluations: b = [8][n] size-n inverse transforms of the cosets -> 8n coefficients
void coset_interp_finish(Context &c, const fe *b, fe *out, int log_n);
void lincomb2(Context &c, const fe *polys, unsigned long long n, int w, const fe *cc1, const fe *cc2, fe *t1, fe *t2);
void compose(Context &c, const fe *t1q, const fe *t2q, const fe *cq, fe *comp, unsigned long long n, unsigned long long len, unsigned long long inc,
             fe k1, fe k2, fe kc);

// ---- hashing (hash.cu); H = Blake3Hash or Sha3Hash (digest.cuh) ----
template <class H> void hash_trace_rows(Context &c, const fe *ext, void *leaves, int w, int log_n, int log_blowup);
template <class H> void hash_rows_plain(Context &c, const fe *cols, void *digests, int w, unsigned long long rows);
template <class H> void hash64_contiguous(Context &c, const void *in, void *out, unsigned long long count);
template <class H> void merkle_build(Context &c, const void *leaves, void *nodes, unsigned long long L);
template <class H> void merkle_finish(Context &c, void *nodes, unsigned long long m);     // level with m nodes already at nodes[m..2m)
template <class H> void merkle_levels_down_to(Context &c, const void *leaves, void *nodes, unsigned long long L, unsigned long long stop);
template <class H> unsigned long long pow_search(Context &c, const uint8_t seed[32], unsigned grinding);
template <class H> void pow_hash(const uint8_t seed[32], unsigned long long nonce, uint8_t out[32]);
// alghash.cu: blake3 / rescue / poseidon / sha3 over 64-byte messages, and Merkle trees with them
void alg_hash64(Context &c, int hash_id, const void *in, void *out, unsigned long long n);
void alg_merkle_build(Context &c, int hash_id, const void *leaves, void *nodes, unsigned long long L);

// ---- FRI (fri.cu) ----
// storage layout of a vector of D = 2^log_d evaluations: natural (log_b < 0) or coset-major with 2^log_b cosets:
// logical index i = (k << log_b) + c  lives at  (c << (log_d - log_b)) + k
struct Layout {
    int log_d, log_b;
    __host__ __device__ unsigned long long phys(unsigned long long i) const {
        if (log_b < 0) return i;
        return ((i & ((1ULL << log_b) - 1ULL)) << (log_d - log_b)) + (i >> log_b);
    }
    __host__ __device__ unsigned long long logical(unsigned long long p) const {
        if (log_b < 0) return p;
        const int log_k = log_d - log_b;
        return ((p & ((1ULL << log_k) - 1ULL)) << log_b) + (p >> log_k);
    }
};
// leaves[r] = H(v[r], v[r+R], v[r+2R], v[r+3R]),  R = D/4   (fri/prover.rs:16-17, fri/utils.rs:16-21)
template <class H> void fri_hash_rows(Context &c, const fe *values, Layout in, Layout rows, void *leaves);
// next[r] = f_r(alpha), f_r = cubic through (x_r t^j, v[r + jR])   (fri/prover.rs:26-32, quartic.rs:20-135)
// alpha: device pointer (derived on the device by fri_alpha, or uploaded by the host when RNG callbacks are registered)
void fri_fold(Context &c, const fe *values, Layout in, fe *next, Layout out, const fe *alpha, const TwiddleRef &inv_root_table, int log_n_total,
              fe tau_inv, fe inv4);
// alpha_dev[0] = field::prng(root) (fri/prover.rs:29); root_copy_dev receives the 32 root bytes (collected for one host copy at the end)
void fri_alpha(Context &c, const void *root_dev, fe *alpha_dev, void *root_copy_dev);
// coset-sharded variants (a rank holds cosets [c0, c0 + 2^log_nc) of the layer as [c - c0][k]); items in ShardedTree order [k'][c - c0]
template <class H> void fri_hash_rows_local(Context &c, const fe *values_local, int log_d, int log_b, int log_nc, void *items_local);
void fri_fold_local(Context &c, const fe *values_local, int log_d, int log_b, int log_nc, unsigned c0, fe *next_local, const fe *alpha,
                    const TwiddleRef &inv_root_table, int log_n_total, fe tau_inv, fe inv4);

}  // namespace dg
