// Keccak-f[1600] and SHA3-256 for host and device code (32-byte digests).
// The reference's `hash::sha3` is crate sha3's Sha3_256 (/root/reference/src/crypto/hash.rs:212-218); the crate is not vendored, so
// this follows FIPS 202 (August 2015):
//   * state: 25 lanes of 64 bits, lane (x, y) at index x + 5y, bytes little-endian within a lane (section 3.1.2);
//   * one round = theta, rho, pi, chi, iota (section 3.2); 24 rounds (Keccak-p[1600, 24], section 3.3);
//   * rho offsets from the walk (x, y) <- (y, 2x + 3y) starting at (1, 0), offset (t + 1)(t + 2)/2 mod 64 (Algorithm 2);
//   * round constants from the degree-8 LFSR rc(t) (Algorithms 5 and 6);
//   * SHA3-256 = Keccak[c = 512]: rate 136 bytes (17 lanes), domain suffix 01 + pad10*1 -> bytes 0x06 ... 0x80 (section 6.1, B.2).
// Call sites on the prove path hash
//   * 64-byte inputs (Merkle nodes, FRI rows, constraint leaf pairs, proof-of-work): one permutation;
//   * trace rows of 16 w bytes (w < 128 field elements = 2 w lanes): floor(2 w / 17) + 1 permutations, streamed from the columns.
// On the device the lanes are 64-bit values that ptxas keeps as 32-bit register pairs: rotations are two funnel shifts, chi is one
// LOP3 per half, and the theta parities fold into 3-input LOP3s.
#pragma once
#include <cstdint>

namespace dg {
namespace sha3 {

#define DG_KECCAK_RC                                                                                                     \
    0x0000000000000001ULL, 0x0000000000008082ULL, 0x800000000000808aULL, 0x8000000080008000ULL, 0x000000000000808bULL,   \
    0x0000000080000001ULL, 0x8000000080008081ULL, 0x8000000000008009ULL, 0x000000000000008aULL, 0x0000000000000088ULL,   \
    0x0000000080008009ULL, 0x000000008000000aULL, 0x000000008000808bULL, 0x800000000000008bULL, 0x8000000000008089ULL,   \
    0x8000000000008003ULL, 0x8000000000008002ULL, 0x8000000000000080ULL, 0x000000000000800aULL, 0x800000008000000aULL,   \
    0x8000000080008081ULL, 0x8000000000008080ULL, 0x0000000080000001ULL, 0x8000000080008008ULL
static __constant__ uint64_t c_keccak_rc[24] = {DG_KECCAK_RC};
static const uint64_t h_keccak_rc[24] = {DG_KECCAK_RC};
#undef DG_KECCAK_RC

__host__ __device__ __forceinline__ uint64_t rotl64(uint64_t x, int n) {
#ifdef __CUDA_ARCH__
    uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    if (n >= 32) { const uint32_t t = lo; lo = hi; hi = t; n -= 32; }
    return ((uint64_t)__funnelshift_l(lo, hi, n) << 32) | __funnelshift_l(hi, lo, n);
#else
    return n == 0 ? x : (x << n) | (x >> (64 - n));
#endif
}
__host__ __device__ __forceinline__ uint64_t chi(uint64_t a, uint64_t b, uint64_t c) { return a ^ (~b & c); }

// Keccak-f[1600] in place
__host__ __device__ __forceinline__ void keccak_f(uint64_t a[25]) {
#pragma unroll 1
    for (int r = 0; r < 24; r++) {
        // theta
        const uint64_t c0 = a[0] ^ a[5] ^ a[10] ^ a[15] ^ a[20];
        const uint64_t c1 = a[1] ^ a[6] ^ a[11] ^ a[16] ^ a[21];
        const uint64_t c2 = a[2] ^ a[7] ^ a[12] ^ a[17] ^ a[22];
        const uint64_t c3 = a[3] ^ a[8] ^ a[13] ^ a[18] ^ a[23];
        const uint64_t c4 = a[4] ^ a[9] ^ a[14] ^ a[19] ^ a[24];
        const uint64_t d0 = c4 ^ rotl64(c1, 1);
        const uint64_t d1 = c0 ^ rotl64(c2, 1);
        const uint64_t d2 = c1 ^ rotl64(c3, 1);
        const uint64_t d3 = c2 ^ rotl64(c4, 1);
        const uint64_t d4 = c3 ^ rotl64(c0, 1);
        // rho and pi: lane (x, y) rotated by its offset lands at (y, 2x + 3y)
        const uint64_t b0 = a[0] ^ d0;
        const uint64_t b10 = rotl64(a[1] ^ d1, 1);
        const uint64_t b20 = rotl64(a[2] ^ d2, 62);
        const uint64_t b5 = rotl64(a[3] ^ d3, 28);
        const uint64_t b15 = rotl64(a[4] ^ d4, 27);
        const uint64_t b16 = rotl64(a[5] ^ d0, 36);
        const uint64_t b1 = rotl64(a[6] ^ d1, 44);
        const uint64_t b11 = rotl64(a[7] ^ d2, 6);
        const uint64_t b21 = rotl64(a[8] ^ d3, 55);
        const uint64_t b6 = rotl64(a[9] ^ d4, 20);
        const uint64_t b7 = rotl64(a[10] ^ d0, 3);
        const uint64_t b17 = rotl64(a[11] ^ d1, 10);
        const uint64_t b2 = rotl64(a[12] ^ d2, 43);
        const uint64_t b12 = rotl64(a[13] ^ d3, 25);
        const uint64_t b22 = rotl64(a[14] ^ d4, 39);
        const uint64_t b23 = rotl64(a[15] ^ d0, 41);
        const uint64_t b8 = rotl64(a[16] ^ d1, 45);
        const uint64_t b18 = rotl64(a[17] ^ d2, 15);
        const uint64_t b3 = rotl64(a[18] ^ d3, 21);
        const uint64_t b13 = rotl64(a[19] ^ d4, 8);
        const uint64_t b14 = rotl64(a[20] ^ d0, 18);
        const uint64_t b24 = rotl64(a[21] ^ d1, 2);
        const uint64_t b9 = rotl64(a[22] ^ d2, 61);
        const uint64_t b19 = rotl64(a[23] ^ d3, 56);
        const uint64_t b4 = rotl64(a[24] ^ d4, 14);
        // chi along each row, iota on lane (0, 0)
#ifdef __CUDA_ARCH__
        a[0] = chi(b0, b1, b2) ^ c_keccak_rc[r];
#else
        a[0] = chi(b0, b1, b2) ^ h_keccak_rc[r];
#endif
        a[1] = chi(b1, b2, b3);    a[2] = chi(b2, b3, b4);    a[3] = chi(b3, b4, b0);    a[4] = chi(b4, b0, b1);
        a[5] = chi(b5, b6, b7);    a[6] = chi(b6, b7, b8);    a[7] = chi(b7, b8, b9);    a[8] = chi(b8, b9, b5);    a[9] = chi(b9, b5, b6);
        a[10] = chi(b10, b11, b12); a[11] = chi(b11, b12, b13); a[12] = chi(b12, b13, b14); a[13] = chi(b13, b14, b10); a[14] = chi(b14, b10, b11);
        a[15] = chi(b15, b16, b17); a[16] = chi(b16, b17, b18); a[17] = chi(b17, b18, b19); a[18] = chi(b18, b19, b15); a[19] = chi(b19, b15, b16);
        a[20] = chi(b20, b21, b22); a[21] = chi(b21, b22, b23); a[22] = chi(b22, b23, b24); a[23] = chi(b23, b24, b20); a[24] = chi(b24, b20, b21);
    }
}

enum : uint64_t { PAD_FIRST = 0x06ULL, PAD_LAST = 0x8000000000000000ULL };     // first padding byte; last byte of the rate (lane 16)

// digest = lanes 0..3 as 8 little-endian words
__host__ __device__ __forceinline__ void squeeze(const uint64_t a[25], uint32_t out[8]) {
#pragma unroll
    for (int i = 0; i < 4; i++) { out[2 * i] = (uint32_t)a[i]; out[2 * i + 1] = (uint32_t)(a[i] >> 32); }
}

// SHA3-256 of exactly 64 bytes given as 16 little-endian words: 8 message lanes, padding in lanes 8 and 16, one permutation
__host__ __device__ __forceinline__ void hash64(const uint32_t m[16], uint32_t out[8]) {
    uint64_t a[25];
#pragma unroll
    for (int i = 0; i < 8; i++) a[i] = ((uint64_t)m[2 * i + 1] << 32) | m[2 * i];
    a[8] = PAD_FIRST;
#pragma unroll
    for (int i = 9; i < 25; i++) a[i] = 0;
    a[16] = PAD_LAST;
    keccak_f(a);
    squeeze(a, out);
}

// SHA3-256 of a message of `nlanes` whole lanes (8 nlanes bytes), lane g read by lane_at(g) as it is absorbed: the padded message has
// nlanes / 17 + 1 blocks, so the lane positions inside a block stay compile-time constants and the state stays in registers
template <typename LaneAt>
__host__ __device__ __forceinline__ void hash_lanes(int nlanes, LaneAt lane_at, uint32_t out[8]) {
    uint64_t a[25];
#pragma unroll
    for (int i = 0; i < 25; i++) a[i] = 0;
    const int nblocks = nlanes / 17 + 1;
#pragma unroll 1
    for (int b = 0; b < nblocks; b++) {
#pragma unroll
        for (int l = 0; l < 17; l++) {
            const int g = 17 * b + l;
            uint64_t v = g < nlanes ? lane_at(g) : 0;
            if (g == nlanes) v ^= PAD_FIRST;
            if (l == 16 && b == nblocks - 1) v ^= PAD_LAST;
            a[l] ^= v;
        }
        keccak_f(a);
    }
    squeeze(a, out);
}

}  // namespace sha3
}  // namespace dg
