// Commitment kernels: trace-row leaf hashing, Merkle level sweeps, proof-of-work grinding.  Every kernel is a template over the
// proof's hash (digest.cuh): BLAKE3 (the default) or SHA3-256.
//
//   leaf hashing   /root/reference/src/stark/trace/trace_table.rs:174-185  (hash(as_bytes(row)) for every LDE row)
//   tree building  /root/reference/src/crypto/merkle.rs:269-294            (heap layout, nodes[0] = 0, root = nodes[1])
//   PoW grinding   /root/reference/src/stark/utils/proof_of_work.rs:4-32   (smallest nonce >= 1)
//
// Leaf hashing reads the extended trace in its coset-major layout ([column][coset][k]): a warp's 32 threads hash 32
// neighbouring k of one coset, so each column read is one 512-byte contiguous request; the 32-byte digest is written to
// its logical row position (one full 32-byte sector per thread).  The column->row "gather" that the reference performs
// on the CPU therefore costs no extra memory pass.
#include "common.cuh"
#include "digest.cuh"

namespace dg {

// ---- trace rows -----------------------------------------------------------------------------------------------------
// ext: [w][N] coset-major (N = n << log_blowup), leaves: N digests in logical row order
template <class H, bool FMA_ADDS>
__global__ void __launch_bounds__(256) hash_rows_kernel(const fe *__restrict__ ext, uint4 *__restrict__ leaves, int w, unsigned long long N,
                                                        int log_n, int log_blowup, uint32_t one) {
    const unsigned long long p = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= N) return;
    const unsigned long long n_mask = (1ULL << log_n) - 1ULL;
    const unsigned long long k = p & n_mask, c = p >> log_n;
    const unsigned long long row = (k << log_blowup) + c;
    const uint4 *col = reinterpret_cast<const uint4 *>(ext) + p;
    if constexpr (H::id == Sha3Hash::id) {
        // element j of the row = lanes 2j, 2j+1, read as two 8-byte halves of the 16-byte column entry as the sponge absorbs them
        uint32_t d[8];
        sha3::hash_lanes(2 * w, [&](int g) {
            const uint2 v = reinterpret_cast<const uint2 *>(col + (unsigned long long)(g >> 1) * N)[g & 1];
            return ((uint64_t)v.y << 32) | v.x;
        }, d);
        leaves[2 * row] = make_uint4(d[0], d[1], d[2], d[3]);
        leaves[2 * row + 1] = make_uint4(d[4], d[5], d[6], d[7]);
        return;
    }

    const int total_bytes = w * 16;
    uint32_t cv[8], cv0[8];
    int chunk_start_col = 0;
    const bool two_chunks = total_bytes > 1024;
    for (int chunk = 0; chunk < (two_chunks ? 2 : 1); chunk++) {
        const int chunk_cols = two_chunks ? (chunk == 0 ? 64 : w - 64) : w;
        const int nblocks = (chunk_cols + 3) >> 2;
        b3::iv(cv);
        for (int b = 0; b < nblocks; b++) {
            uint32_t m[16];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int j = b * 4 + q;
                uint4 v = make_uint4(0, 0, 0, 0);
                if (j < chunk_cols) v = col[(unsigned long long)(chunk_start_col + j) * N];
                m[4 * q] = v.x; m[4 * q + 1] = v.y; m[4 * q + 2] = v.z; m[4 * q + 3] = v.w;
            }
            const int rem = chunk_cols * 16 - b * 64;
            uint32_t flags = 0;
            if (b == 0) flags |= b3::CHUNK_START;
            if (b == nblocks - 1) { flags |= b3::CHUNK_END; if (!two_chunks) flags |= b3::ROOT; }
            if (FMA_ADDS) b3::compress_fma(cv, m, (uint64_t)chunk, rem < 64 ? rem : 64, flags, one);
            else b3::compress(cv, m, (uint64_t)chunk, rem < 64 ? rem : 64, flags);
        }
        if (two_chunks && chunk == 0) {
#pragma unroll
            for (int i = 0; i < 8; i++) cv0[i] = cv[i];
            chunk_start_col = 64;
        }
    }
    if (two_chunks) {
        uint32_t m[16];
#pragma unroll
        for (int i = 0; i < 8; i++) { m[i] = cv0[i]; m[8 + i] = cv[i]; }
        b3::iv(cv);
        b3::compress(cv, m, 0, 64, b3::PARENT | b3::ROOT);
    }
    leaves[2 * row] = make_uint4(cv[0], cv[1], cv[2], cv[3]);
    leaves[2 * row + 1] = make_uint4(cv[4], cv[5], cv[6], cv[7]);
}

template <class H>
void hash_trace_rows(Context &c, const fe *ext, void *leaves, int w, int log_n, int log_blowup) {
    const unsigned long long N = 1ULL << (log_n + log_blowup);
    static int fma = -1;
    if (fma < 0) { const char *e = getenv("DG_B3_FMA"); fma = e ? atoi(e) : 1; }      // FMA-pipe additions: trace tree 9.1 -> 8.1 ms at 2^25 rows x 26 columns
    if (H::id == Blake3Hash::id && fma) hash_rows_kernel<Blake3Hash, true><<<(unsigned)((N + 255) / 256), 256, 0, c.stream>>>(ext, (uint4 *)leaves, w, N, log_n, log_blowup, 1u);
    else hash_rows_kernel<H, false><<<(unsigned)((N + 255) / 256), 256, 0, c.stream>>>(ext, (uint4 *)leaves, w, N, log_n, log_blowup, 1u);
    c.launches++;
    DG_CUDA(cudaGetLastError());
}

// ---- Merkle levels ----------------------------------------------------------------------------------------------------
// out[i] = H(in[2i] || in[2i+1]),  i < count
template <class H>
__global__ void __launch_bounds__(256) merkle_level_kernel(const uint4 *__restrict__ in, uint4 *__restrict__ out, unsigned long long count) {
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    uint32_t m[16], cv[8];
#pragma unroll
    for (int q = 0; q < 4; q++) {
        uint4 v = in[4 * i + q];
        m[4 * q] = v.x; m[4 * q + 1] = v.y; m[4 * q + 2] = v.z; m[4 * q + 3] = v.w;
    }
    H::hash64(m, cv);
    out[2 * i] = make_uint4(cv[0], cv[1], cv[2], cv[3]);
    out[2 * i + 1] = make_uint4(cv[4], cv[5], cv[6], cv[7]);
}

// finishes a tree whose level with `count` (<= 1024, power of two) nodes sits at nodes[count .. 2*count): computes
// nodes[count/2 .. count), ..., nodes[1] in one block, and zeroes nodes[0]
template <class H>
__global__ void __launch_bounds__(512) merkle_top_kernel(uint4 *__restrict__ nodes, unsigned count) {
    __shared__ uint32_t s[2048 * 8 / 2];     // up to 1024 digests
    const unsigned tid = threadIdx.x;
    for (unsigned i = tid; i < count * 2; i += blockDim.x) {
        uint4 v = nodes[2 * count + i];
        s[4 * i] = v.x; s[4 * i + 1] = v.y; s[4 * i + 2] = v.z; s[4 * i + 3] = v.w;
    }
    __syncthreads();
    for (unsigned m = count / 2; m >= 1; m >>= 1) {
        // level with m nodes from 2m children held in s[0 .. 2m*8)
        uint32_t cv[8];
        uint32_t msg[16];
        const bool active = tid < m;
        if (active) {
#pragma unroll
            for (int q = 0; q < 16; q++) msg[q] = s[16 * tid + q];
            H::hash64(msg, cv);
        }
        __syncthreads();
        if (active) {
#pragma unroll
            for (int q = 0; q < 8; q++) s[8 * tid + q] = cv[q];
            nodes[2 * (m + tid)] = make_uint4(cv[0], cv[1], cv[2], cv[3]);
            nodes[2 * (m + tid) + 1] = make_uint4(cv[4], cv[5], cv[6], cv[7]);
        }
        __syncthreads();
    }
    if (tid == 0) { nodes[0] = make_uint4(0, 0, 0, 0); nodes[1] = make_uint4(0, 0, 0, 0); }
}

// computes the levels count/2, count/4, ... down to and including the level with `stop` nodes (stop >= 1, a power of two) from the
// input level `in` (count nodes) into the heap `nodes` (a level with m nodes sits at nodes[m .. 2m)).  One launch per level while a
// level has more than 1024 nodes -- BLAKE3 is ALU-bound with long dependency chains, so the per-level kernel at full occupancy is the
// fastest form (r02 measured a fused variant, 8 -> 4 -> 2 -> 1 nodes per thread in registers and 11 levels per launch: 104 registers,
// 16 resident warps per SM, 2^25-leaf tree 2.4 ms instead of 1.2 ms) -- then the last <= 1024 nodes level by level inside one block.
template <class H>
static void tree_levels(Context &c, const uint4 *in, uint4 *nodes, unsigned long long count, unsigned long long stop) {
    while (count > stop) {
        const unsigned long long m = count / 2;
        if (stop == 1 && count <= 1024 && count >= 2 && in == nodes + 2 * count) {     // the rest of a complete tree: one block
            merkle_top_kernel<H><<<1, 512, 0, c.stream>>>(nodes, (unsigned)count); c.launches++;
            DG_CUDA(cudaGetLastError());
            return;
        }
        merkle_level_kernel<H><<<(unsigned)((m + 255) / 256), 256, 0, c.stream>>>(in, nodes + 2 * m, m); c.launches++;
        DG_CUDA(cudaGetLastError());
        count = m;
        in = nodes + 2 * m;
    }
}

// leaves: L digests (L power of two >= 2); nodes: L digests (heap layout)
template <class H>
void merkle_build(Context &c, const void *leaves, void *nodes, unsigned long long L) {
    DG_REQUIRE(L >= 2 && (L & (L - 1)) == 0, "number of leaves must be a power of 2 and >= 2");
    uint4 *nd = (uint4 *)nodes;
    tree_levels<H>(c, (const uint4 *)leaves, nd, L, 1);
    DG_CUDA(cudaMemsetAsync(nd, 0, 32, c.stream));             // nodes[0] = 0 (merkle.rs:273)
}

// completes a tree whose level with m nodes (m a power of two) already sits at nodes[m .. 2m)
template <class H>
void merkle_finish(Context &c, void *nodes, unsigned long long m) {
    uint4 *nd = (uint4 *)nodes;
    tree_levels<H>(c, nd + 2 * m, nd, m, 1);
    DG_CUDA(cudaMemsetAsync(nd, 0, 32, c.stream));
}

// levels of a heap-layout tree from L/2 nodes down to (and including) the level with `stop` nodes
template <class H>
void merkle_levels_down_to(Context &c, const void *leaves, void *nodes, unsigned long long L, unsigned long long stop) {
    tree_levels<H>(c, (const uint4 *)leaves, (uint4 *)nodes, L, stop);
}

// ---- generic 64-byte hashing (tests / FRI rows given contiguously) ------------------------------------------------------
template <class H>
void hash64_contiguous(Context &c, const void *in, void *out, unsigned long long count) {
    merkle_level_kernel<H><<<(unsigned)((count + 255) / 256), 256, 0, c.stream>>>((const uint4 *)in, (uint4 *)out, count); c.launches++;
    DG_CUDA(cudaGetLastError());
}

// ---- proof of work ------------------------------------------------------------------------------------------------------
template <class H>
__global__ void __launch_bounds__(256) pow_kernel(const uint32_t *__restrict__ seed, unsigned long long start, unsigned long long count,
                                                  unsigned grinding, unsigned long long *best) {
    const unsigned long long g = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= count) return;
    const unsigned long long nonce = start + g;
    uint32_t m[16], cv[8];
#pragma unroll
    for (int i = 0; i < 8; i++) m[i] = seed[i];
    m[8] = (uint32_t)nonce; m[9] = (uint32_t)(nonce >> 32);
#pragma unroll
    for (int i = 10; i < 16; i++) m[i] = 0;
    H::hash64(m, cv);
    const unsigned long long o0 = ((unsigned long long)cv[1] << 32) | cv[0];
    const unsigned tz = o0 == 0 ? 64u : (unsigned)(__ffsll((long long)o0) - 1);
    if (tz >= grinding) atomicMin(best, nonce);
}

// returns the smallest nonce >= 1 whose hash has >= grinding trailing zero bits in its first 8 bytes
template <class H>
unsigned long long pow_search(Context &c, const uint8_t seed[32], unsigned grinding) {
    DevBuf d_seed(32), d_best(8);
    DG_CUDA(cudaMemcpyAsync(d_seed.p, seed, 32, cudaMemcpyHostToDevice, c.stream));
    const unsigned long long none = ~0ULL;
    DG_CUDA(cudaMemcpyAsync(d_best.p, &none, 8, cudaMemcpyHostToDevice, c.stream));
    unsigned long long start = 1;
    const unsigned long long batch = 1ULL << 22;
    for (int iter = 0; iter < (1 << 20); iter++) {
        pow_kernel<H><<<(unsigned)(batch / 256), 256, 0, c.stream>>>(d_seed.as<uint32_t>(), start, batch, grinding, d_best.as<unsigned long long>()); c.launches++;
        DG_CUDA(cudaGetLastError());
        unsigned long long best;
        DG_CUDA(cudaMemcpyAsync(&best, d_best.p, 8, cudaMemcpyDeviceToHost, c.stream));
        DG_CUDA(cudaStreamSynchronize(c.stream));
        if (best != none) return best;
        start += batch;
    }
    throw Error(-4, "proof-of-work search exhausted");
}

}  // namespace dg

namespace dg {
// rows of a plain column-major matrix (no coset permutation): physical position == logical row
template <class H>
void hash_rows_plain(Context &c, const fe *cols, void *digests, int w, unsigned long long rows) {
    hash_rows_kernel<H, false><<<(unsigned)((rows + 255) / 256), 256, 0, c.stream>>>(cols, (uint4 *)digests, w, rows, 63, 0, 1u); c.launches++;
    DG_CUDA(cudaGetLastError());
}
// host-side hash of the 64-byte proof-of-work input seed || nonce_le || 0^24 (proof_of_work.rs:12-24)
template <class H>
void pow_hash(const uint8_t seed[32], unsigned long long nonce, uint8_t out[32]) {
    uint32_t m[16], cv[8];
    memcpy(m, seed, 32);
    m[8] = (uint32_t)nonce; m[9] = (uint32_t)(nonce >> 32);
    for (int i = 10; i < 16; i++) m[i] = 0;
    H::hash64(m, cv);
    memcpy(out, cv, 32);
}

#define DG_HASH_SITES(H)                                                                                                    \
    template void hash_trace_rows<H>(Context &, const fe *, void *, int, int, int);                                         \
    template void merkle_build<H>(Context &, const void *, void *, unsigned long long);                                     \
    template void merkle_finish<H>(Context &, void *, unsigned long long);                                                  \
    template void merkle_levels_down_to<H>(Context &, const void *, void *, unsigned long long, unsigned long long);         \
    template void hash64_contiguous<H>(Context &, const void *, void *, unsigned long long);                                 \
    template unsigned long long pow_search<H>(Context &, const uint8_t[32], unsigned);                                      \
    template void hash_rows_plain<H>(Context &, const fe *, void *, int, unsigned long long);                               \
    template void pow_hash<H>(const uint8_t[32], unsigned long long, uint8_t[32]);
DG_HASH_SITES(Blake3Hash)
DG_HASH_SITES(Sha3Hash)
#undef DG_HASH_SITES
}  // namespace dg
