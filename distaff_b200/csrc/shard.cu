#include "shard.h"
#include "digest.cuh"
#include "poly.h"

namespace dg {

// ---- index algebra (host) ---------------------------------------------------------------------------------------------------
ShardLocation ShardGeom::item(uint64_t i) const {
    const uint64_t blk = 1ULL << log_blk, per_k = blk << log_g;
    const uint64_t k = i / per_k, within = i % per_k;
    ShardLocation r;
    r.owner = (int)(within >> log_blk);
    r.kind = SHARD_LOCAL;
    r.index = (k << log_blk) + (within & (blk - 1));
    return r;
}
ShardLocation ShardGeom::node(uint64_t h) const {
    const uint64_t G = 1ULL << log_g;
    const int lvl = 63 - __builtin_clzll(h);
    const uint64_t S = 1ULL << lvl, o = h - S;              // level size, position inside the level
    ShardLocation r;
    if (S <= G) { r.owner = -1; r.kind = SHARD_TOP; r.index = h; return r; }                   // replicated top heap (levels 1 .. G)
    if (S <= n * G) {                                       // mid: every rank holds S / G consecutive nodes of this level
        const uint64_t per = S / G;
        r.owner = (int)(o / per); r.kind = SHARD_MID; r.index = per + (o % per);
        return r;
    }
    const uint64_t span = items() / S;                    // level-0 items below this node (< blk)
    const uint64_t i0 = o * span;
    ShardLocation it = item(i0);
    const uint64_t local_level = (n << log_blk) / span;   // size of the local level with the same span
    r.owner = it.owner;
    r.kind = SHARD_LOCAL;
    r.index = local_level + it.index / span;
    return r;
}

// ---- kernels ------------------------------------------------------------------------------------------------------------------
// levels of a heap-layout tree from L/2 nodes down to (and including) the level with `stop` nodes (hash.cu)
template <class H>
void merkle_build_partial(Context &c, const void *leaves, void *nodes, unsigned long long L, unsigned long long stop) {
    merkle_levels_down_to<H>(c, leaves, nodes, L, stop);
}

// upper[(n << log_g) + (k << log_g) + g] = gathered[g][k]
__global__ void interleave_roots_kernel(const uint4 *__restrict__ gathered, uint4 *__restrict__ upper, unsigned long long n, int log_g) {
    const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (n << log_g)) return;
    const unsigned long long g = t / n, k = t % n;
    const unsigned long long dst = (n << log_g) + (k << log_g) + g;
    upper[2 * dst] = gathered[2 * t];
    upper[2 * dst + 1] = gathered[2 * t + 1];
}
void interleave_roots(Context &c, const void *gathered, void *upper, unsigned long long n, int log_g) {
    const unsigned long long total = n << log_g;
    interleave_roots_kernel<<<(unsigned)((total + 255) / 256), 256, 0, c.stream>>>((const uint4 *)gathered, (uint4 *)upper, n, log_g); c.launches++;
    DG_CUDA(cudaGetLastError());
}

// items[k * (nc/4) + c4] = H(ev[4c4][k], ev[4c4+1][k], ev[4c4+2][k], ev[4c4+3][k]) over the local cosets (prover.rs:84-86,180-187)
template <class H>
__global__ void __launch_bounds__(256) constraint_items_kernel(const fe *__restrict__ ev, int log_n, int log_nc, uint4 *__restrict__ items) {
    const unsigned long long n = 1ULL << log_n;
    const unsigned long long total = n << (log_nc - 2);
    const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const unsigned long long c4 = t >> log_n, k = t & (n - 1);
    const unsigned long long j = (k << (log_nc - 2)) + c4;
    uint32_t m[16], cv[8];
#pragma unroll
    for (int u = 0; u < 4; u++) {
        const uint4 x = reinterpret_cast<const uint4 *>(ev)[(4 * c4 + u) * n + k];
        m[4 * u] = x.x; m[4 * u + 1] = x.y; m[4 * u + 2] = x.z; m[4 * u + 3] = x.w;
    }
    H::hash64(m, cv);
    items[2 * j] = make_uint4(cv[0], cv[1], cv[2], cv[3]);
    items[2 * j + 1] = make_uint4(cv[4], cv[5], cv[6], cv[7]);
}
template <class H>
void constraint_items_local(Context &c, const fe *evals_local, int log_n, int log_nc, void *items) {
    const unsigned long long total = (1ULL << log_n) << (log_nc - 2);
    constraint_items_kernel<H><<<(unsigned)((total + 255) / 256), 256, 0, c.stream>>>(evals_local, log_n, log_nc, (uint4 *)items); c.launches++;
    DG_CUDA(cudaGetLastError());
}

// ---- sharded tree -------------------------------------------------------------------------------------------------------------------
template <class H>
void ShardedTree::build(Context &c, const void *items_local_dev, uint64_t n, int log_blk, bool fetch_root) {
    int log_g = 0;
    while ((1 << log_g) < c.world) log_g++;
    geom.n = n; geom.log_blk = log_blk; geom.log_g = log_g;
    items_local = items_local_dev;
    const uint64_t local_items = n << log_blk, G = 1ULL << log_g;
    if (c.world == 1) {
        // one rank: the local heap is the whole tree; the mid and top heaps alias it (their indices are global heap indices then)
        DG_REQUIRE(local_items >= 2, "tree needs at least 2 items");
        local_nodes.alloc(local_items * 32);
        merkle_build<H>(c, items_local_dev, local_nodes.p, local_items);
        mid_p = top_p = local_nodes.p;
    } else {
        DG_REQUIRE(n >= G && n % G == 0, "sharded tree needs at least one block per rank and k-range");
        const void *roots = items_local_dev;
        if (log_blk > 0) {
            local_nodes.alloc(local_items * 32);
            merkle_build_partial<H>(c, items_local_dev, local_nodes.p, local_items, n);
            roots = (const uint8_t *)local_nodes.p + n * 32;           // heap level with n nodes: the subtree roots, by k
        }
        // re-shard the roots by k-range: recv[g'][k'] = root (k = g n/G + k') of rank g'
        const uint64_t chunk = n / G;
        DevBuf recv(n * 32);
        if (c.mark) c.mark("tree.local");
        comm_all_to_all(c, roots, recv.p, chunk * 32);
        if (c.mark) c.mark("tree.a2a");
        mid.alloc(2 * n * 32);
        interleave_roots(c, recv.p, mid.p, chunk, log_g);           // mid[n + k' G + g'] : nodes [g n, (g + 1) n) of the global level n G
        merkle_finish<H>(c, mid.p, n);                                 // mid[1] = global node G + g
        top.alloc(2 * G * 32);
        comm_all_gather(c, (const uint8_t *)mid.p + 32, (uint8_t *)top.p + G * 32, 32);
        merkle_finish<H>(c, top.p, G);
        if (c.mark) c.mark("tree.mid+top");
        mid_p = mid.p; top_p = top.p;
    }
    if (fetch_root) {
        DG_CUDA(cudaMemcpyAsync(root.data(), (const uint8_t *)top_p + 32, 32, cudaMemcpyDeviceToHost, c.stream));
        DG_CUDA(cudaStreamSynchronize(c.stream));
    }
}
template void ShardedTree::build<Blake3Hash>(Context &, const void *, uint64_t, int, bool);
template void ShardedTree::build<Sha3Hash>(Context &, const void *, uint64_t, int, bool);
template void constraint_items_local<Blake3Hash>(Context &, const fe *, int, int, void *);
template void constraint_items_local<Sha3Hash>(Context &, const fe *, int, int, void *);

// out[t] = base_t ? ((const uint4 *)base_t)[unit_t] : 0
__global__ void fetch_units_kernel(const unsigned long long *__restrict__ req, unsigned count, uint4 *__restrict__ out) {
    const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const uint4 *base = reinterpret_cast<const uint4 *>(req[2 * t]);
    out[t] = base ? base[req[2 * t + 1]] : make_uint4(0, 0, 0, 0);
}

// replicated units are identical on every rank: all ranks but rank 0 zero theirs so that the sum over the ranks returns the value once
__global__ void zero_replicated_kernel(uint4 *__restrict__ out, const unsigned char *__restrict__ replicated, unsigned count, int zero_them) {
    const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < count && replicated[t] && zero_them) out[t] = make_uint4(0, 0, 0, 0);
}

void FetchBatch::run() {
    const size_t n = owner_.size();
    out_.assign(n * 16, 0);
    if (n == 0) return;
    DevBuf d_req(n * 16), d_out(n * 16);
    DG_CUDA(cudaMemcpyAsync(d_req.p, req_.data(), n * 16, cudaMemcpyHostToDevice, c_.stream));
    fetch_units_kernel<<<(unsigned)((n + 127) / 128), 128, 0, c_.stream>>>(d_req.as<unsigned long long>(), (unsigned)n, d_out.as<uint4>()); c_.launches++;
    DG_CUDA(cudaGetLastError());
    if (c_.world == 1) {
        DG_CUDA(cudaMemcpyAsync(out_.data(), d_out.p, n * 16, cudaMemcpyDeviceToHost, c_.stream));
        DG_CUDA(cudaStreamSynchronize(c_.stream));
        return;
    }
    // exactly one rank contributes each owned unit (the others wrote zeros), so a 32-bit integer sum over the ranks assembles the
    // result bit for bit; replicated units (owner < 0) were read by every rank: keep the local copy of those
    DevBuf summed(n * 16);
    std::vector<unsigned char> keep(n);
    bool any_replicated = false;
    for (size_t t = 0; t < n; t++) { keep[t] = owner_[t] < 0; any_replicated |= owner_[t] < 0; }
    if (any_replicated) {
        DevBuf d_keep(n);
        DG_CUDA(cudaMemcpyAsync(d_keep.p, keep.data(), n, cudaMemcpyHostToDevice, c_.stream));
        zero_replicated_kernel<<<(unsigned)((n + 127) / 128), 128, 0, c_.stream>>>(d_out.as<uint4>(), d_keep.as<unsigned char>(), (unsigned)n, c_.rank != 0); c_.launches++;
        DG_CUDA(cudaGetLastError());
        comm_all_reduce_sum_u32(c_, d_out.as<unsigned>(), summed.as<unsigned>(), n * 4);
    } else {
        comm_all_reduce_sum_u32(c_, d_out.as<unsigned>(), summed.as<unsigned>(), n * 4);
    }
    DG_CUDA(cudaMemcpyAsync(out_.data(), summed.p, n * 16, cudaMemcpyDeviceToHost, c_.stream));
    DG_CUDA(cudaStreamSynchronize(c_.stream));
}

}  // namespace dg
