// FRI layer kernels: row hashing and radix-4 folding.
//
//   fri::reduce                 /root/reference/src/stark/fri/prover.rs:11-53
//   quartic::transpose          /root/reference/src/math/quartic.rs:137-152   (rows r: v[r], v[r+R], v[r+2R], v[r+3R])
//   quartic::interpolate_batch  /root/reference/src/math/quartic.rs:37-135    (cubic through 4 points, batch inversion)
//   quartic::evaluate_batch     /root/reference/src/math/quartic.rs:20-31
//
// The reference interpolates every row with Lagrange formulas and one global batch inversion.  Because the four x
// coordinates of a row are x, x*t, x*t^2, x*t^3 with t a primitive 4th root of unity, the row polynomial evaluated at
// alpha is a 4-point inverse DFT followed by Horner in u = alpha / x:
//      f(alpha) = 1/4 * sum_j u^j * sum_k y_k t^(-jk)
// and 1/x is a power of the inverse LDE root (table lookup): no field inversion is needed.  The interpolating cubic is
// unique and the arithmetic exact, hence the values equal the reference's.
#include "poly.h"
#include "digest.cuh"

namespace dg {

template <class H>
__global__ void __launch_bounds__(256) fri_hash_rows_kernel(const fe *__restrict__ v, Layout in, Layout rows, uint4 *__restrict__ leaves) {
    const unsigned long long R = 1ULL << rows.log_d;
    const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= R) return;
    const unsigned long long r = rows.logical(t);
    uint32_t m[16], cv[8];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint4 x = reinterpret_cast<const uint4 *>(v)[in.phys(r + (unsigned long long)j * R)];
        m[4 * j] = x.x; m[4 * j + 1] = x.y; m[4 * j + 2] = x.z; m[4 * j + 3] = x.w;
    }
    H::hash64(m, cv);
    leaves[2 * r] = make_uint4(cv[0], cv[1], cv[2], cv[3]);
    leaves[2 * r + 1] = make_uint4(cv[4], cv[5], cv[6], cv[7]);
}
template <class H>
void fri_hash_rows(Context &c, const fe *values, Layout in, Layout rows, void *leaves) {
    const unsigned long long R = 1ULL << rows.log_d;
    fri_hash_rows_kernel<H><<<(unsigned)((R + 255) / 256), 256, 0, c.stream>>>(values, in, rows, (uint4 *)leaves); c.launches++;
    DG_CUDA(cudaGetLastError());
}
template void fri_hash_rows<Blake3Hash>(Context &, const fe *, Layout, Layout, void *);
template void fri_hash_rows<Sha3Hash>(Context &, const fe *, Layout, Layout, void *);

// special_x = field::prng(layer root) (fri/prover.rs:29) derived on the device, so that a layer's fold does not wait for a round trip
// to the host: StdRng::from_seed(root) = ChaCha20 (64-bit block counter, stream 0), Uniform(0..M) = widening multiply of a 128-bit
// draw by M with rejection of low halves > M - 1 -- the same steps as fs::Rng::field (host_fs.cu), which the CPU tests pin.
__device__ __forceinline__ uint32_t rol32(uint32_t x, int n) { return (x << n) | (x >> (32 - n)); }
#define DG_QRD(a, b, c, d) a += b; d = rol32(d ^ a, 16); c += d; b = rol32(b ^ c, 12); a += b; d = rol32(d ^ a, 8); c += d; b = rol32(b ^ c, 7);
__global__ void fri_alpha_kernel(const uint32_t *__restrict__ root, fe *__restrict__ alpha, uint32_t *__restrict__ root_copy) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    typedef unsigned __int128 u128;
    uint32_t key[8];
    for (int i = 0; i < 8; i++) { key[i] = root[i]; root_copy[i] = root[i]; }
    uint32_t buf[16];
    unsigned long long counter = 0;
    int pos = 16;
    auto next_u32 = [&]() {
        if (pos >= 16) {
            uint32_t in[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u, key[0], key[1], key[2], key[3], key[4], key[5], key[6], key[7],
                               (uint32_t)counter, (uint32_t)(counter >> 32), 0u, 0u};
            uint32_t x[16];
            for (int i = 0; i < 16; i++) x[i] = in[i];
            for (int r = 0; r < 10; r++) {
                DG_QRD(x[0], x[4], x[8], x[12]) DG_QRD(x[1], x[5], x[9], x[13]) DG_QRD(x[2], x[6], x[10], x[14]) DG_QRD(x[3], x[7], x[11], x[15])
                DG_QRD(x[0], x[5], x[10], x[15]) DG_QRD(x[1], x[6], x[11], x[12]) DG_QRD(x[2], x[7], x[8], x[13]) DG_QRD(x[3], x[4], x[9], x[14])
            }
            for (int i = 0; i < 16; i++) buf[i] = x[i] + in[i];
            counter++;
            pos = 0;
        }
        return buf[pos++];
    };
    auto next_u64 = [&]() { unsigned long long lo = next_u32(); unsigned long long hi = next_u32(); return lo | (hi << 32); };
    const u128 Mv = ((u128)DG_M_HI << 64) | DG_M_LO;
    for (;;) {
        const unsigned long long v0 = next_u64(), v1 = next_u64();
        const u128 p00 = (u128)v0 * DG_M_LO, p01 = (u128)v0 * DG_M_HI, p10 = (u128)v1 * DG_M_LO, p11 = (u128)v1 * DG_M_HI;
        const u128 mid = (p00 >> 64) + (unsigned long long)p01 + (unsigned long long)p10;
        const u128 lo = ((u128)(unsigned long long)mid << 64) | (unsigned long long)p00;
        const u128 hi = p11 + (p01 >> 64) + (p10 >> 64) + (mid >> 64);
        if (lo <= Mv - 1) { *alpha = fe_make((unsigned long long)hi, (unsigned long long)(hi >> 64)); return; }
    }
}
void fri_alpha(Context &c, const void *root_dev, fe *alpha_dev, void *root_copy_dev) {
    fri_alpha_kernel<<<1, 32, 0, c.stream>>>((const uint32_t *)root_dev, alpha_dev, (uint32_t *)root_copy_dev); c.launches++;
    DG_CUDA(cudaGetLastError());
}

__global__ void __launch_bounds__(256) fri_fold_kernel(const fe *__restrict__ v, Layout in, fe *__restrict__ next, Layout out, const fe *__restrict__ alpha_p,
                                                       TwiddleRef inv_root, int shift, fe tau_inv, fe inv4) {
    const fe alpha = *alpha_p;
    const unsigned long long R = 1ULL << out.log_d;
    const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= R) return;
    const unsigned long long r = out.logical(t);
    fe y0 = v[in.phys(r)], y1 = v[in.phys(r + R)], y2 = v[in.phys(r + 2 * R)], y3 = v[in.phys(r + 3 * R)];
    // x_r^-1 = (w_N^-1)^(r << shift)
    const unsigned ee = (unsigned)((r << shift) & (unsigned long long)inv_root.mask);
    fe xinv = fe_mul(inv_root.lo[ee & ((1u << inv_root.lo_bits) - 1u)], inv_root.hi[ee >> inv_root.lo_bits]);
    fe u = fe_mul(alpha, xinv);
    fe s02 = fe_add(y0, y2), d02 = fe_sub(y0, y2), s13 = fe_add(y1, y3), d13 = fe_mul(fe_sub(y1, y3), tau_inv);
    fe a0 = fe_add(s02, s13), a1 = fe_add(d02, d13), a2 = fe_sub(s02, s13), a3 = fe_sub(d02, d13);
    fe acc = fe_add(a2, fe_mul(u, a3));
    acc = fe_add(a1, fe_mul(u, acc));
    acc = fe_add(a0, fe_mul(u, acc));
    next[t] = fe_mul(acc, inv4);
}
void fri_fold(Context &c, const fe *values, Layout in, fe *next, Layout out, const fe *alpha, const TwiddleRef &inv_root_table, int log_n_total,
              fe tau_inv, fe inv4) {
    const unsigned long long R = 1ULL << out.log_d;
    const int shift = log_n_total - in.log_d;            // layer domain is the 4^depth-th powers of the LDE domain
    fri_fold_kernel<<<(unsigned)((R + 255) / 256), 256, 0, c.stream>>>(values, in, next, out, alpha, inv_root_table, shift, tau_inv, inv4); c.launches++;
    DG_CUDA(cudaGetLastError());
}

// ---- coset-sharded layers (multi-GPU): a rank holds the cosets [c0, c0 + 2^log_nc) of a layer of 2^log_d values as the slab
//      [c - c0][k], k < 2^(log_d - log_b).  Row r = b k' + c and its three companions r + jR (R = D/4) have k = k' + j R/b inside the
//      same coset, so hashing and folding need no other rank's data; the folded value of row r is element k' of coset c of the next layer.
template <class H>
__global__ void __launch_bounds__(256) fri_hash_rows_local_kernel(const fe *__restrict__ v, int log_d, int log_b, int log_nc, uint4 *__restrict__ items) {
    const int log_kr = log_d - 2 - log_b;                       // rows per coset
    const unsigned long long total = 1ULL << (log_kr + log_nc);
    const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const unsigned long long cl = t >> log_kr, kp = t & ((1ULL << log_kr) - 1ULL);
    const uint4 *col = reinterpret_cast<const uint4 *>(v) + (cl << (log_d - log_b)) + kp;
    uint32_t m[16], cv[8];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint4 x = col[(unsigned long long)j << log_kr];
        m[4 * j] = x.x; m[4 * j + 1] = x.y; m[4 * j + 2] = x.z; m[4 * j + 3] = x.w;
    }
    H::hash64(m, cv);
    const unsigned long long it = (kp << log_nc) + cl;        // ShardedTree item layout [k'][c - c0]
    items[2 * it] = make_uint4(cv[0], cv[1], cv[2], cv[3]);
    items[2 * it + 1] = make_uint4(cv[4], cv[5], cv[6], cv[7]);
}
template <class H>
void fri_hash_rows_local(Context &c, const fe *values_local, int log_d, int log_b, int log_nc, void *items_local) {
    const unsigned long long total = 1ULL << (log_d - 2 - log_b + log_nc);
    fri_hash_rows_local_kernel<H><<<(unsigned)((total + 255) / 256), 256, 0, c.stream>>>(values_local, log_d, log_b, log_nc, (uint4 *)items_local); c.launches++;
    DG_CUDA(cudaGetLastError());
}
template void fri_hash_rows_local<Blake3Hash>(Context &, const fe *, int, int, int, void *);
template void fri_hash_rows_local<Sha3Hash>(Context &, const fe *, int, int, int, void *);

__global__ void __launch_bounds__(256) fri_fold_local_kernel(const fe *__restrict__ v, int log_d, int log_b, int log_nc, unsigned c0, fe *__restrict__ next,
                                                             const fe *__restrict__ alpha_p, TwiddleRef inv_root, int shift, fe tau_inv, fe inv4) {
    const fe alpha = *alpha_p;
    const int log_kr = log_d - 2 - log_b;
    const unsigned long long total = 1ULL << (log_kr + log_nc);
    const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const unsigned long long cl = t >> log_kr, kp = t & ((1ULL << log_kr) - 1ULL);
    const fe *col = v + (cl << (log_d - log_b)) + kp;
    const fe y0 = col[0], y1 = col[1ULL << log_kr], y2 = col[2ULL << log_kr], y3 = col[3ULL << log_kr];
    const unsigned long long r = (kp << log_b) + c0 + cl;
    const unsigned ee = (unsigned)((r << shift) & (unsigned long long)inv_root.mask);
    fe xinv = fe_mul(inv_root.lo[ee & ((1u << inv_root.lo_bits) - 1u)], inv_root.hi[ee >> inv_root.lo_bits]);
    fe u = fe_mul(alpha, xinv);
    fe s02 = fe_add(y0, y2), d02 = fe_sub(y0, y2), s13 = fe_add(y1, y3), d13 = fe_mul(fe_sub(y1, y3), tau_inv);
    fe a0 = fe_add(s02, s13), a1 = fe_add(d02, d13), a2 = fe_sub(s02, s13), a3 = fe_sub(d02, d13);
    fe acc = fe_add(a2, fe_mul(u, a3));
    acc = fe_add(a1, fe_mul(u, acc));
    acc = fe_add(a0, fe_mul(u, acc));
    next[t] = fe_mul(acc, inv4);                               // [c - c0][k'] of the next layer
}
void fri_fold_local(Context &c, const fe *values_local, int log_d, int log_b, int log_nc, unsigned c0, fe *next_local, const fe *alpha,
                    const TwiddleRef &inv_root_table, int log_n_total, fe tau_inv, fe inv4) {
    const unsigned long long total = 1ULL << (log_d - 2 - log_b + log_nc);
    fri_fold_local_kernel<<<(unsigned)((total + 255) / 256), 256, 0, c.stream>>>(values_local, log_d, log_b, log_nc, c0, next_local, alpha, inv_root_table,
                                                                                  log_n_total - log_d, tau_inv, inv4); c.launches++;
    DG_CUDA(cudaGetLastError());
}

}  // namespace dg
