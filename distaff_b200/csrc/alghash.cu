// Algebraic hash functions over F_M on the GPU: Rescue and Poseidon, one thread per 64-byte message, and Merkle trees built with them
// (and with BLAKE3 or SHA3-256, the hashes a proof commits with, under the same interface).
//
// Replaces (SURVEY.md section 8 row a10, micro-benchmark config C5)
//   hash::rescue     /root/reference/src/crypto/hash.rs:151-177
//   hash::poseidon   /root/reference/src/crypto/hash.rs:119-147
//   helpers          /root/reference/src/crypto/hash.rs:222-254  (add_constants, apply_sbox, apply_inv_sbox, apply_mds)
//   constants        /root/reference/src/crypto/hash.rs:9-115    (ALPHA = 3, INV_ALPHA, MDS[36], ARK[546])
//   build_merkle_nodes with these hash functions: /root/reference/src/crypto/merkle.rs:269-294
// Neither function is on the default prove path (ProofOptions can only serialise blake3, options.rs:97-125); the reference
// benchmarks them in benches/hash.rs and tests Merkle trees with them (merkle.rs:321-518).
//
// State = 6 field elements; a message of at most 64 bytes fills elements 0..3 as little-endian u128 (the rest is zero), the digest is
// elements 0..1.  Messages are expected to hold valid field elements (< M), as the reference's arithmetic assumes (field.rs:25).
// The inverse S-box x^INV_ALPHA (a 128-bit exponent) dominates Rescue: it is evaluated with a fixed 4-bit window
// (INV_ALPHA = 0xaaaaaaaaaaaaaaaaaaaa8caaaaaaaaab: digits a, 8, c, b only) = 124 squarings + 38 multiplications.
#define DG_MUL_CALL 1
#include "common.cuh"
#include "air_constants.h"
#include "digest.cuh"

namespace dg {

__constant__ fe c_alg_mds[36];
__constant__ fe c_alg_ark[546];

static void alg_upload_constants(Context &c) {
    if (c.alghash_consts) return;
    std::vector<fe> v(546);
    for (int i = 0; i < 36; i++) v[i] = fe_make(DG_HASH_MDS[i][0], DG_HASH_MDS[i][1]);
    DG_CUDA(cudaMemcpyToSymbol(c_alg_mds, v.data(), 36 * sizeof(fe)));
    for (int i = 0; i < 546; i++) v[i] = fe_make(DG_HASH_ARK[i][0], DG_HASH_ARK[i][1]);
    DG_CUDA(cudaMemcpyToSymbol(c_alg_ark, v.data(), 546 * sizeof(fe)));
    c.alghash_consts = true;
}

__device__ __forceinline__ void alg_add_constants(fe st[6], int off) {
#pragma unroll
    for (int i = 0; i < 6; i++) st[i] = fe_add(st[i], c_alg_ark[off + i]);
}
__device__ __forceinline__ void alg_mds(fe st[6]) {
    fe r[6];
#pragma unroll
    for (int i = 0; i < 6; i++) {
        fe acc = fe_mul(c_alg_mds[i * 6], st[0]);
#pragma unroll
        for (int j = 1; j < 6; j++) acc = fe_add(acc, fe_mul(c_alg_mds[i * 6 + j], st[j]));
        r[i] = acc;
    }
#pragma unroll
    for (int i = 0; i < 6; i++) st[i] = r[i];
}
// x^INV_ALPHA, hex digits of the exponent from the most significant: 20 x 'a', '8', 'c', 9 x 'a', 'b'
__device__ __noinline__ fe alg_inv_sbox(fe x) {
    const fe x2 = fe_sqr(x), x4 = fe_sqr(x2), x8 = fe_sqr(x4);
    const fe xa = fe_mul(x8, x2), xb = fe_mul(xa, x), xc = fe_mul(x8, x4);
    fe acc = xa;
#pragma unroll 1
    for (int d = 1; d < 32; d++) {
        acc = fe_sqr(acc); acc = fe_sqr(acc); acc = fe_sqr(acc); acc = fe_sqr(acc);
        const fe m = d == 20 ? x8 : (d == 21 ? xc : (d == 31 ? xb : xa));
        acc = fe_mul(acc, m);
    }
    return acc;
}

__device__ __forceinline__ void rescue_permute(fe st[6]) {          // hash.rs:160-173
    alg_add_constants(st, 0);
#pragma unroll 1
    for (int i = 0; i < 10; i++) {
#pragma unroll
        for (int j = 0; j < 6; j++) st[j] = alg_inv_sbox(st[j]);
        alg_mds(st);
        alg_add_constants(st, (i * 2 + 1) * 6);
#pragma unroll
        for (int j = 0; j < 6; j++) st[j] = fe_cube(st[j]);
        alg_mds(st);
        alg_add_constants(st, (i * 2 + 2) * 6);
    }
}
__device__ __forceinline__ void poseidon_permute(fe st[6]) {        // hash.rs:129-143: 4 full + 83 partial + 4 full rounds
#pragma unroll 1
    for (int i = 0; i < 91; i++) {
        alg_add_constants(st, i * 6);
        if (i < 4 || i >= 87) {
#pragma unroll
            for (int j = 0; j < 6; j++) st[j] = fe_cube(st[j]);
        } else {
            st[5] = fe_cube(st[5]);
        }
        alg_mds(st);
    }
}

// out[i] = H(in[64 i .. 64 i + 64))
template <int HASH>
__global__ void __launch_bounds__(128) alg_hash64_kernel(const uint4 *__restrict__ in, uint4 *__restrict__ out, unsigned long long n) {
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (HASH == DG_HASH_BLAKE3 || HASH == DG_HASH_SHA3) {
        uint32_t m[16], cv[8];
#pragma unroll
        for (int q = 0; q < 4; q++) { const uint4 v = in[4 * i + q]; m[4 * q] = v.x; m[4 * q + 1] = v.y; m[4 * q + 2] = v.z; m[4 * q + 3] = v.w; }
        if (HASH == DG_HASH_SHA3) Sha3Hash::hash64(m, cv);
        else Blake3Hash::hash64(m, cv);
        out[2 * i] = make_uint4(cv[0], cv[1], cv[2], cv[3]);
        out[2 * i + 1] = make_uint4(cv[4], cv[5], cv[6], cv[7]);
        return;
    }
    fe st[6];
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const uint4 v = in[4 * i + q];
        st[q] = fe_make(((unsigned long long)v.y << 32) | v.x, ((unsigned long long)v.w << 32) | v.z);
    }
    st[4] = fe_make(0, 0); st[5] = fe_make(0, 0);
    if (HASH == 1) rescue_permute(st); else poseidon_permute(st);
#pragma unroll
    for (int q = 0; q < 2; q++)
        out[2 * i + q] = make_uint4((unsigned)st[q].lo, (unsigned)(st[q].lo >> 32), (unsigned)st[q].hi, (unsigned)(st[q].hi >> 32));
}

void alg_hash64(Context &c, int hash_id, const void *in, void *out, unsigned long long n) {
    DG_REQUIRE((hash_id >= 0 && hash_id <= 2) || hash_id == DG_HASH_SHA3, "hash id must be 0 (blake3), 1 (rescue), 2 (poseidon) or 4 (sha3)");
    if (n == 0) return;
    alg_upload_constants(c);
    const unsigned grid = (unsigned)((n + 127) / 128);
    switch (hash_id) {
        case 0: alg_hash64_kernel<0><<<grid, 128, 0, c.stream>>>((const uint4 *)in, (uint4 *)out, n); break;
        case 1: alg_hash64_kernel<1><<<grid, 128, 0, c.stream>>>((const uint4 *)in, (uint4 *)out, n); break;
        case DG_HASH_SHA3: alg_hash64_kernel<DG_HASH_SHA3><<<grid, 128, 0, c.stream>>>((const uint4 *)in, (uint4 *)out, n); break;
        default: alg_hash64_kernel<2><<<grid, 128, 0, c.stream>>>((const uint4 *)in, (uint4 *)out, n); break;
    }
    c.launches++;
    DG_CUDA(cudaGetLastError());
}

// heap-layout Merkle nodes (merkle.rs:269-294): nodes[L/2 + i] = H(leaf[2i] | leaf[2i+1]), nodes[i] = H(nodes[2i] | nodes[2i+1]), nodes[0] = 0
void alg_merkle_build(Context &c, int hash_id, const void *leaves, void *nodes, unsigned long long L) {
    DG_REQUIRE(L >= 2 && (L & (L - 1)) == 0, "number of leaves must be a power of 2 and >= 2");
    uint8_t *nd = (uint8_t *)nodes;
    alg_hash64(c, hash_id, leaves, nd + (L / 2) * 32, L / 2);
    for (unsigned long long m = L / 2; m >= 2; m >>= 1)          // level with m nodes at [m, 2m) -> m/2 parents at [m/2, m)
        alg_hash64(c, hash_id, nd + m * 32, nd + (m / 2) * 32, m / 2);
    DG_CUDA(cudaMemsetAsync(nd, 0, 32, c.stream));
}

}  // namespace dg
