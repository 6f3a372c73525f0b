// extern "C" surface declared in include/distaff_gpu.h.  Every entry point catches dg::Error and returns a code.
#include "../../include/distaff_gpu.h"
#include "common.cuh"
#include "prover.h"
#include "host_fs.h"
#include "shard.h"
#include "poly.h"
#include "digest.cuh"
#include <thread>

namespace dg {
std::string verify_proof(Context &c, const uint8_t program_hash[32], const std::vector<fe> &inputs, const std::vector<fe> &outputs,
                         const uint8_t *proof_bytes, size_t proof_len);
}

namespace dg {
bool host_plan_verify_batch(const std::vector<uint64_t> &indexes, int depth, size_t n_values, const std::vector<uint32_t> &node_counts,
                            std::vector<uint32_t> &ops, std::vector<uint32_t> &level_start, uint32_t &root_slot);
}

using namespace dg;

static thread_local std::string t_last_error;

template <typename F>
static int guarded(F &&f) {
    try {
        f();
        return DG_OK;
    } catch (const dg::Error &e) {
        t_last_error = e.what();
        return e.code;
    } catch (const std::exception &e) {
        t_last_error = e.what();
        return DG_ERR_INVALID;
    }
}

struct EventTimer {
    cudaEvent_t a = nullptr, b = nullptr;
    cudaStream_t s;
    float *out;
    EventTimer(cudaStream_t stream, float *ms) : s(stream), out(ms) {
        if (!out) return;
        DG_CUDA(cudaEventCreate(&a));
        DG_CUDA(cudaEventCreate(&b));
        DG_CUDA(cudaEventRecord(a, s));
    }
    void stop() {
        if (!out) return;
        DG_CUDA(cudaEventRecord(b, s));
        DG_CUDA(cudaEventSynchronize(b));
        DG_CUDA(cudaEventElapsedTime(out, a, b));
    }
    ~EventTimer() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
};

// ---- helper kernels ------------------------------------------------------------------------------------------------------
__global__ void coset_to_logical_kernel(const fe *__restrict__ in, fe *__restrict__ out, int log_n, int log_blowup) {
    const unsigned long long p = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long N = 1ULL << (log_n + log_blowup);
    if (p >= N) return;
    const unsigned long long k = p & ((1ULL << log_n) - 1ULL), c = p >> log_n;
    out[(unsigned long long)blockIdx.y * N + (k << log_blowup) + c] = in[(unsigned long long)blockIdx.y * N + p];
}

__global__ void field_op_kernel(int op, int impl, const fe *a, const fe *b, fe *out, unsigned long long n) {
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (op == 5) {                    // unreduced dot product of groups of 6: out[i] = sum_j a[6i+j] * b[6i+j]; impl 0 = 288-bit accumulation, 1 = reduced
        if (6 * i + 6 > n) return;
        fe xs[6], ys[6];
#pragma unroll
        for (int j = 0; j < 6; j++) { xs[j] = a[6 * i + j]; ys[j] = b[6 * i + j]; }
        if (impl == 0) out[i] = fe_dot<6>(xs, ys);
        else { fe acc = portable::fe_mul(xs[0], ys[0]); for (int j = 1; j < 6; j++) acc = portable::fe_add(acc, portable::fe_mul(xs[j], ys[j])); out[i] = acc; }
        return;
    }
    fe x = a[i], y = b ? b[i] : fe_make(0, 0), r;
    if ((impl == 2 || impl == 3) && op == 2) {
#ifdef __CUDA_ARCH__
        r = impl == 2 ? ptx::fe_mul_v1(x, y) : ptx::fe_mul_v3(x, y);      // earlier multiplies, kept for differential tests
#endif
    } else if (impl == 0) {
        switch (op) {
            case 0: r = fe_add(x, y); break;
            case 1: r = fe_sub(x, y); break;
            case 2: r = fe_mul(x, y); break;
            case 3: r = fe_inv(x); break;
            default: r = fe_is_zero(x) ? fe_make(0, 0) : fe_pow_u128(x, y.lo, y.hi); break;
        }
    } else {
        switch (op) {
            case 0: r = portable::fe_add(x, y); break;
            case 1: r = portable::fe_sub(x, y); break;
            case 2: r = portable::fe_mul(x, y); break;
            case 3: r = portable::fe_inv(x); break;
            default: r = fe_is_zero(x) ? fe_make(0, 0) : portable::fe_pow_u128(x, y.lo, y.hi); break;
        }
    }
    out[i] = r;
}

__global__ void fill_kernel(uint4 *p, size_t n, unsigned v) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = make_uint4(v, v + 1, v + 2, v + 3);
}

// Single-process multi-GPU (dg_init_devices): the proof is sharded exactly as in the one-process-per-GPU mode, but the ranks are host
// threads of this process, each bound to its own device context and NCCL communicator.  Rank 0 runs on the calling thread.
template <typename F>
static Proof *prove_on_all_devices(F &&prove_rank, dg_prove_stats_t *stats) {
    const int n = ctx_device_count();
    std::vector<Proof *> res(n, nullptr);
    std::vector<int> codes(n, 0);
    std::vector<std::string> msgs(n);
    auto run = [&](int g) {
        try {
            Context &cg = ctx_of(g);
            ctx_bind(&cg);
            res[g] = prove_rank(cg, g == 0 ? stats : nullptr);
        } catch (const dg::Error &e) { codes[g] = e.code; msgs[g] = e.what(); }
        catch (const std::exception &e) { codes[g] = DG_ERR_INVALID; msgs[g] = e.what(); }
    };
    std::vector<std::thread> th;
    for (int g = 1; g < n; g++) th.emplace_back(run, g);
    run(0);
    for (auto &t : th) t.join();
    ctx_bind(&ctx_of(0));
    for (int g = 0; g < n; g++)
        if (codes[g] != 0) {
            for (auto *p : res) delete p;
            throw Error(codes[g], "rank " + std::to_string(g) + ": " + msgs[g]);
        }
    for (int g = 1; g < n; g++) {
        const bool same = res[g] && res[g]->bytes == res[0]->bytes;
        delete res[g];
        if (!same) { delete res[0]; throw Error(DG_ERR_CUDA, "ranks produced different proofs"); }
    }
    return res[0];
}

extern "C" {

int dg_init(int device) { return guarded([&] { ctx_init(device); }); }
int dg_init_devices(int n_devices) { return guarded([&] { ctx_init_devices(n_devices); }); }
const char *dg_last_error(void) { return t_last_error.c_str(); }

int dg_device_info(char *name, size_t cap, int *sm_count, size_t *total_mem) {
    return guarded([&] {
        Context &c = ctx();
        cudaDeviceProp prop;
        DG_CUDA(cudaGetDeviceProperties(&prop, c.device));
        if (name && cap) { strncpy(name, prop.name, cap - 1); name[cap - 1] = 0; }
        if (sm_count) *sm_count = prop.multiProcessorCount;
        if (total_mem) *total_mem = prop.totalGlobalMem;
    });
}

// ---- device memory -------------------------------------------------------------------------------------------------------
int dg_dev_alloc(void **ptr, size_t bytes) { return guarded([&] { ctx(); DG_CUDA(cudaMalloc(ptr, bytes)); }); }
int dg_dev_free(void *ptr) { return guarded([&] { ctx(); DG_CUDA(cudaFree(ptr)); }); }
int dg_dev_upload(void *dst, const void *src, size_t bytes) {
    return guarded([&] { Context &c = ctx(); DG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c.stream)); DG_CUDA(cudaStreamSynchronize(c.stream)); });
}
int dg_dev_download(void *dst, const void *src, size_t bytes) {
    return guarded([&] { Context &c = ctx(); DG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c.stream)); DG_CUDA(cudaStreamSynchronize(c.stream)); });
}
int dg_dev_sync(void) { return guarded([&] { DG_CUDA(cudaStreamSynchronize(ctx().stream)); }); }
int dg_dev_flush_l2(void) {
    return guarded([&] {
        Context &c = ctx();
        const size_t bytes = (size_t)256 << 20;
        c.l2_scratch.ensure(bytes, true);
        fill_kernel<<<(unsigned)(bytes / 16 / 256), 256, 0, c.stream>>>(c.l2_scratch.as<uint4>(), bytes / 16, 7u); c.launches++;
        DG_CUDA(cudaGetLastError());
        DG_CUDA(cudaStreamSynchronize(c.stream));
    });
}

// ---- device-resident building blocks ----------------------------------------------------------------------------------------
int dg_dev_ntt(void *d_values, uint32_t log_n, uint32_t batch, int inverse, float *ms) {
    return guarded([&] {
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        c.twiddle(log_n, inverse != 0);       // table setup outside the timed region
        if (log_n > 20) c.twiddle(log_n - (log_n + 2) / 3, inverse != 0);
        c.ntt_tmp.ensure(((size_t)16 << log_n) * std::min<size_t>(batch, std::max<size_t>(1, ((size_t)1 << 30) / ((size_t)16 << log_n))), true);
        EventTimer t(c.stream, ms);
        ntt_batch(c, (const fe *)d_values, (fe *)d_values, log_n, batch, (size_t)1 << log_n, (size_t)1 << log_n, inverse != 0);
        t.stop();
        DG_CUDA(cudaStreamSynchronize(c.stream));
    });
}
int dg_dev_lde(const void *d_polys, void *d_ext, uint32_t log_n, uint32_t log_blowup, uint32_t batch, float *ms) {
    return guarded([&] {
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        c.twiddle(log_n + log_blowup, false);
        c.twiddle(log_n, false);
        if (log_n > 20) c.twiddle(log_n - (log_n + 2) / 3, false);
        EventTimer t(c.stream, ms);
        lde_batch(c, (const fe *)d_polys, (fe *)d_ext, log_n, log_blowup, 1, batch, (size_t)1 << log_n, (size_t)1 << (log_n + log_blowup));
        t.stop();
        DG_CUDA(cudaStreamSynchronize(c.stream));
    });
}
int dg_dev_merkle_build(const void *d_leaves, uint64_t n_leaves, void *d_nodes, float *ms) {
    return guarded([&] {
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        EventTimer t(c.stream, ms);
        merkle_build<Blake3Hash>(c, d_leaves, d_nodes, n_leaves);
        t.stop();
        DG_CUDA(cudaStreamSynchronize(c.stream));
    });
}
int dg_dev_merkle_build_with(int hash, const void *d_leaves, uint64_t n_leaves, void *d_nodes, float *ms) {
    return guarded([&] {
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        EventTimer t(c.stream, ms);
        alg_merkle_build(c, hash, d_leaves, d_nodes, n_leaves);
        t.stop();
        DG_CUDA(cudaStreamSynchronize(c.stream));
    });
}
int dg_dev_hash_rows(const void *d_ext, uint32_t width, uint32_t log_n, uint32_t log_blowup, void *d_leaves, float *ms) {
    return guarded([&] {
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        DG_REQUIRE(width >= 1 && width < 128, "width must be in 1..127");
        EventTimer t(c.stream, ms);
        hash_trace_rows<Blake3Hash>(c, (const fe *)d_ext, d_leaves, (int)width, (int)log_n, (int)log_blowup);
        t.stop();
        DG_CUDA(cudaStreamSynchronize(c.stream));
    });
}

// ---- host-memory building blocks -----------------------------------------------------------------------------------------------
int dg_ntt(uint8_t *values, uint32_t log_n, uint32_t batch, int inverse) {
    return guarded([&] {
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        DG_REQUIRE(values, "null buffer");
        DG_REQUIRE(log_n >= 1 && log_n <= 30 && batch >= 1, "invalid transform size");
        const size_t bytes = ((size_t)16 << log_n) * batch;
        DevBuf d(bytes);
        DG_CUDA(cudaMemcpyAsync(d.p, values, bytes, cudaMemcpyHostToDevice, c.stream));
        ntt_batch(c, d.as<fe>(), d.as<fe>(), log_n, batch, (size_t)1 << log_n, (size_t)1 << log_n, inverse != 0);
        DG_CUDA(cudaMemcpyAsync(values, d.p, bytes, cudaMemcpyDeviceToHost, c.stream));
        DG_CUDA(cudaStreamSynchronize(c.stream));
    });
}
int dg_lde(const uint8_t *values, uint8_t *extended, uint32_t log_n, uint32_t log_blowup, uint32_t batch) {
    return guarded([&] {
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        DG_REQUIRE(values && extended, "null buffer");
        DG_REQUIRE(log_n >= 1 && log_blowup >= 1 && log_n + log_blowup <= 30 && batch >= 1 && batch <= 65535, "invalid extension size");
        const size_t n = (size_t)1 << log_n, N = n << log_blowup;
        DevBuf d_in(n * batch * 16), d_ext(N * batch * 16), d_out(N * batch * 16);
        DG_CUDA(cudaMemcpyAsync(d_in.p, values, n * batch * 16, cudaMemcpyHostToDevice, c.stream));
        ntt_batch(c, d_in.as<fe>(), d_in.as<fe>(), log_n, batch, n, n, true);                 // interpolate (trace_table.rs:158)
        lde_batch(c, d_in.as<fe>(), d_ext.as<fe>(), log_n, log_blowup, 1, batch, n, N);       // evaluate over the LDE domain (:165)
        coset_to_logical_kernel<<<dim3((unsigned)((N + 255) / 256), batch), 256, 0, c.stream>>>(d_ext.as<fe>(), d_out.as<fe>(), log_n, log_blowup); c.launches++;
        DG_CUDA(cudaGetLastError());
        DG_CUDA(cudaMemcpyAsync(extended, d_out.p, N * batch * 16, cudaMemcpyDeviceToHost, c.stream));
        DG_CUDA(cudaStreamSynchronize(c.stream));
    });
}
int dg_merkle_build(const uint8_t *leaves, uint64_t n_leaves, uint8_t *nodes) {
    return guarded([&] {
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        DG_REQUIRE(leaves && nodes, "null buffer");
        DG_REQUIRE(n_leaves >= 2 && (n_leaves & (n_leaves - 1)) == 0, "number of leaves must be a power of 2 and >= 2");
        DevBuf d_l(n_leaves * 32), d_n(n_leaves * 32);
        DG_CUDA(cudaMemcpyAsync(d_l.p, leaves, n_leaves * 32, cudaMemcpyHostToDevice, c.stream));
        merkle_build<Blake3Hash>(c, d_l.p, d_n.p, n_leaves);
        DG_CUDA(cudaMemcpyAsync(nodes, d_n.p, n_leaves * 32, cudaMemcpyDeviceToHost, c.stream));
        DG_CUDA(cudaStreamSynchronize(c.stream));
    });
}
int dg_hash64(int hash, const uint8_t *messages64, uint64_t n, uint8_t *digests32) {
    return guarded([&] {
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        DG_REQUIRE((hash >= 0 && hash <= 2) || hash == DG_HASH_SHA3, "hash id must be 0 (blake3), 1 (rescue), 2 (poseidon) or 4 (sha3)");
        if (n == 0) return;
        DG_REQUIRE(messages64 && digests32, "null buffer");
        DevBuf d_in(n * 64), d_out(n * 32);
        DG_CUDA(cudaMemcpyAsync(d_in.p, messages64, n * 64, cudaMemcpyHostToDevice, c.stream));
        alg_hash64(c, hash, d_in.p, d_out.p, n);
        DG_CUDA(cudaMemcpyAsync(digests32, d_out.p, n * 32, cudaMemcpyDeviceToHost, c.stream));
        DG_CUDA(cudaStreamSynchronize(c.stream));
    });
}
int dg_merkle_build_with(int hash, const uint8_t *leaves, uint64_t n_leaves, uint8_t *nodes) {
    return guarded([&] {
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        DG_REQUIRE(n_leaves >= 2 && (n_leaves & (n_leaves - 1)) == 0, "number of leaves must be a power of 2 and >= 2");
        DevBuf d_l(n_leaves * 32), d_n(n_leaves * 32);
        DG_CUDA(cudaMemcpyAsync(d_l.p, leaves, n_leaves * 32, cudaMemcpyHostToDevice, c.stream));
        alg_merkle_build(c, hash, d_l.p, d_n.p, n_leaves);
        DG_CUDA(cudaMemcpyAsync(nodes, d_n.p, n_leaves * 32, cudaMemcpyDeviceToHost, c.stream));
        DG_CUDA(cudaStreamSynchronize(c.stream));
    });
}
int dg_hash_rows(const uint8_t *columns, uint32_t width, uint64_t rows, uint8_t *digests) {
    return guarded([&] {
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        DG_REQUIRE(columns && digests, "null buffer");
        DG_REQUIRE(width >= 1 && width < 128 && rows >= 1, "invalid matrix shape");
        DevBuf d_c((size_t)width * rows * 16), d_d(rows * 32);
        DG_CUDA(cudaMemcpyAsync(d_c.p, columns, (size_t)width * rows * 16, cudaMemcpyHostToDevice, c.stream));
        // reuse the trace-row kernel with a single "coset": physical position == logical row
        hash_rows_plain<Blake3Hash>(c, d_c.as<fe>(), d_d.p, (int)width, rows);
        DG_CUDA(cudaMemcpyAsync(digests, d_d.p, rows * 32, cudaMemcpyDeviceToHost, c.stream));
        DG_CUDA(cudaStreamSynchronize(c.stream));
    });
}
int dg_find_pow_nonce(const uint8_t seed[32], uint32_t grinding_factor, uint64_t *nonce, uint8_t new_seed[32]) {
    return guarded([&] {
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        DG_REQUIRE(seed && nonce, "null argument");
        DG_REQUIRE(grinding_factor <= 32, "grinding factor cannot be greater than 32");
        unsigned long long n = pow_search<Blake3Hash>(c, seed, grinding_factor);
        *nonce = n;
        if (new_seed) pow_hash<Blake3Hash>(seed, n, new_seed);
    });
}
int dg_field_op(int op, int impl, const uint8_t *a, const uint8_t *b, uint8_t *out, uint64_t n) {
    return guarded([&] {
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        DG_REQUIRE(a && out && n >= 1 && op >= 0 && op <= 5, "invalid argument");
        DG_REQUIRE(b || op == 3, "second operand missing");
        DevBuf da(n * 16), db(n * 16), dout(n * 16);
        DG_CUDA(cudaMemcpyAsync(da.p, a, n * 16, cudaMemcpyHostToDevice, c.stream));
        if (b) DG_CUDA(cudaMemcpyAsync(db.p, b, n * 16, cudaMemcpyHostToDevice, c.stream));
        field_op_kernel<<<(unsigned)((n + 127) / 128), 128, 0, c.stream>>>(op, impl, da.as<fe>(), b ? db.as<fe>() : nullptr, dout.as<fe>(), n); c.launches++;
        DG_CUDA(cudaGetLastError());
        DG_CUDA(cudaMemcpyAsync(out, dout.p, n * 16, cudaMemcpyDeviceToHost, c.stream));
        DG_CUDA(cudaStreamSynchronize(c.stream));
    });
}

// ---- prover ------------------------------------------------------------------------------------------------------------------------
int dg_prove(const dg_trace_t *trace, const uint8_t *inputs16, uint32_t n_inputs, const uint8_t *outputs16, uint32_t n_outputs,
             const dg_options_t *options, dg_proof_t **proof_out, dg_prove_stats_t *stats) {
    return guarded([&] {
        DG_REQUIRE(trace && options && proof_out, "null argument");
        DG_REQUIRE((n_inputs == 0 || inputs16) && (n_outputs == 0 || outputs16), "null public inputs / outputs");
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        if (ctx_device_count() > 1) {
            *proof_out = (dg_proof_t *)prove_on_all_devices([&](Context &cg, dg_prove_stats_t *st) {
                return prove_host(cg, *trace, inputs16, n_inputs, outputs16, n_outputs, *options, st); }, stats);
            return;
        }
        *proof_out = (dg_proof_t *)prove_host(c, *trace, inputs16, n_inputs, outputs16, n_outputs, *options, stats);
    });
}
int dg_prove_device(const void *d_registers, uint32_t width, uint64_t length, uint32_t ctx_depth, uint32_t loop_depth,
                    const uint8_t *inputs16, uint32_t n_inputs, const uint8_t *outputs16, uint32_t n_outputs,
                    const dg_options_t *options, dg_proof_t **proof_out, dg_prove_stats_t *stats) {
    return guarded([&] {
        DG_REQUIRE(d_registers && options && proof_out, "null argument");
        DG_REQUIRE((n_inputs == 0 || inputs16) && (n_outputs == 0 || outputs16), "null public inputs / outputs");
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        if (ctx_device_count() > 1) {          // the trace lives on device 0; the other devices read their columns over NVLink (peer access)
            *proof_out = (dg_proof_t *)prove_on_all_devices([&](Context &cg, dg_prove_stats_t *st) {
                return prove_device(cg, (const fe *)d_registers, width, length, ctx_depth, loop_depth, inputs16, n_inputs, outputs16, n_outputs, *options,
                                    st, 0.0f); }, stats);
            return;
        }
        *proof_out = (dg_proof_t *)prove_device(c, (const fe *)d_registers, width, length, ctx_depth, loop_depth, inputs16, n_inputs, outputs16,
                                                n_outputs, *options, stats, 0.0f);
    });
}
int dg_set_rng_callbacks(const dg_rng_callbacks_t *callbacks) {
    return guarded([&] {
        if (!callbacks) { fs::set_rng_hooks(nullptr); return; }
        fs::RngHooks h{callbacks->user, callbacks->draw_field, callbacks->draw_positions};
        fs::set_rng_hooks(&h);
    });
}
int dg_verify(const uint8_t program_hash[32], const uint8_t *inputs16, uint32_t n_inputs, const uint8_t *outputs16, uint32_t n_outputs,
              const uint8_t *proof_bytes, size_t proof_len, char *message, size_t message_cap) {
    if (message && message_cap) message[0] = 0;
    return guarded([&] {
        DG_REQUIRE(program_hash && proof_bytes, "null argument");
        DG_REQUIRE((n_inputs == 0 || inputs16) && (n_outputs == 0 || outputs16), "null public inputs / outputs");
        Context &c = ctx();
        std::lock_guard<std::mutex> lk(c.mu);
        std::vector<fe> in(n_inputs), out(n_outputs);
        if (n_inputs) memcpy(in.data(), inputs16, n_inputs * 16);
        if (n_outputs) memcpy(out.data(), outputs16, n_outputs * 16);
        const std::string verdict = dg::verify_proof(c, program_hash, in, out, proof_bytes, proof_len);
        if (!verdict.empty()) {
            if (message && message_cap) { strncpy(message, verdict.c_str(), message_cap - 1); message[message_cap - 1] = 0; }
            throw Error(DG_ERR_REJECTED, verdict);
        }
    });
}
int dg_proof_serialized_len(const dg_proof_t *proof, size_t *len) {
    return guarded([&] { DG_REQUIRE(proof && len, "null argument"); *len = ((const Proof *)proof)->bytes.size(); });
}
int dg_proof_serialize(const dg_proof_t *proof, uint8_t *buf, size_t cap) {
    return guarded([&] {
        DG_REQUIRE(proof && buf, "null argument");
        const Proof *p = (const Proof *)proof;
        DG_REQUIRE(cap >= p->bytes.size(), "buffer too small");
        memcpy(buf, p->bytes.data(), p->bytes.size());
    });
}
int dg_proof_digest(const dg_proof_t *proof, int which, uint8_t out32[32]) {
    return guarded([&] {
        DG_REQUIRE(proof && out32 && which >= 0 && which <= 2, "invalid argument");
        const Proof *p = (const Proof *)proof;
        memcpy(out32, which == 0 ? p->trace_root : which == 1 ? p->constraint_root : p->pow_seed, 32);
    });
}
int dg_proof_pow_nonce(const dg_proof_t *proof, uint64_t *nonce) {
    return guarded([&] { DG_REQUIRE(proof && nonce, "null argument"); *nonce = ((const Proof *)proof)->pow_nonce; });
}
void dg_proof_free(dg_proof_t *proof) { delete (Proof *)proof; }

// ---- multi-GPU ---------------------------------------------------------------------------------------------------------------------
int dg_comm_unique_id(uint8_t id128[128]) { return guarded([&] { comm_unique_id(id128); }); }
int dg_comm_init(int rank, int world, const uint8_t id128[128]) {
    return guarded([&] { Context &c = ctx(); std::lock_guard<std::mutex> lk(c.mu); comm_init(c, rank, world, id128); });
}
int dg_comm_finalize(void) { return guarded([&] { Context &c = ctx(); std::lock_guard<std::mutex> lk(c.mu); comm_finalize(c); }); }
int dg_host_shard_locate(uint64_t n, int log_blk, int log_g, int is_node, uint64_t index, int64_t out[3]) {
    return guarded([&] {
        ShardGeom geo; geo.n = n; geo.log_blk = log_blk; geo.log_g = log_g;
        ShardLocation l = is_node ? geo.node(index) : geo.item(index);
        out[0] = l.owner; out[1] = l.kind; out[2] = (int64_t)l.index;
    });
}

// ---- host-only helpers (no device access) ---------------------------------------------------------------------------------------------
int dg_host_prng_vector(const uint8_t seed[32], uint64_t count, uint8_t *out16) {
    return guarded([&] { DG_REQUIRE(seed && (out16 || count == 0), "null argument"); std::vector<fe> v = fs::prng_vector(seed, count); memcpy(out16, v.data(), count * 16); });
}
int dg_host_query_positions(const uint8_t seed[32], uint64_t domain_size, uint32_t extension_factor, uint32_t num_queries, uint64_t *out) {
    return guarded([&] {
        try {
            std::vector<uint64_t> p = fs::query_positions(seed, domain_size, extension_factor, num_queries);
            memcpy(out, p.data(), p.size() * 8);
        } catch (const std::exception &e) { throw Error(DG_ERR_EXHAUSTED, e.what()); }
    });
}
int dg_host_blake3(const uint8_t *data, size_t len, uint8_t out32[32]) { return guarded([&] { fs::blake3_short(data, len, out32); }); }
int dg_host_sha3(const uint8_t *data, size_t len, uint8_t out32[32]) {
    return guarded([&] { DG_REQUIRE(out32 && (data || len == 0), "null argument"); fs::sha3_256(data, len, out32); });
}
int dg_host_plan_batch(const uint64_t *indexes, uint32_t n_indexes, uint64_t n_leaves, uint64_t *out, size_t cap, size_t *written) {
    return guarded([&] {
        DG_REQUIRE(indexes && out && written, "null argument");
        DG_REQUIRE(n_leaves >= 2 && (n_leaves & (n_leaves - 1)) == 0, "number of leaves must be a power of 2 and >= 2");
        for (uint32_t i = 0; i < n_indexes; i++) DG_REQUIRE(indexes[i] < n_leaves, "invalid index (merkle.rs:296-303 asserts index <= max_valid)");
        fs::BatchPlan plan = fs::plan_batch_proof(std::vector<uint64_t>(indexes, indexes + n_indexes), n_leaves);
        std::vector<uint64_t> flat = {(uint64_t)plan.nodes.size(), (uint64_t)plan.depth};
        for (auto &slot : plan.nodes) {
            flat.push_back(slot.size());
            for (auto &r : slot) { flat.push_back(r.leaf ? 1 : 0); flat.push_back(r.index); }
        }
        DG_REQUIRE(flat.size() <= cap, "buffer too small");
        memcpy(out, flat.data(), flat.size() * 8);
        *written = flat.size();
    });
}
int dg_host_merkle_verify_plan(const uint64_t *indexes, uint32_t n_indexes, uint32_t depth, uint32_t n_values, const uint32_t *node_counts,
                               uint32_t n_slots, uint32_t *ops, size_t ops_cap, uint32_t *n_ops, uint32_t *level_start, size_t levels_cap,
                               uint32_t *n_levels, uint32_t *root_slot) {
    return guarded([&] {
        DG_REQUIRE(indexes && node_counts && ops && n_ops && level_start && n_levels && root_slot, "null argument");
        std::vector<uint32_t> o, ls;
        uint32_t root = 0;
        if (!host_plan_verify_batch(std::vector<uint64_t>(indexes, indexes + n_indexes), (int)depth, n_values,
                                    std::vector<uint32_t>(node_counts, node_counts + n_slots), o, ls, root))
            throw Error(DG_ERR_REJECTED, "batch proof structure rejected (merkle.rs:154-263 returns false)");
        DG_REQUIRE(o.size() <= ops_cap && ls.size() <= levels_cap, "buffer too small");
        memcpy(ops, o.data(), o.size() * 4);
        memcpy(level_start, ls.data(), ls.size() * 4);
        *n_ops = (uint32_t)(o.size() / 3);
        *n_levels = (uint32_t)ls.size() - 1;
        *root_slot = root;
    });
}
int dg_host_periodic_tables(uint8_t *out16) {
    return guarded([&] { std::vector<fe> t = fs::periodic_tables(); memcpy(out16, t.data(), t.size() * 16); });
}

}  // extern "C"
