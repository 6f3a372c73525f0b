// Host orchestration of the CUDA prove pipeline: the body that replaces /root/reference/src/stark/prover.rs:17-169.
// Stage numbering and names follow the reference's nine debug!() sections (prover.rs:19-167) so that per-stage timings of
// the CPU prover and of this backend line up.  Only 32-byte roots, a handful of challenges and the final openings cross
// the PCIe bus after the register traces have been uploaded.
#include "prover.h"
#include "air.h"
#include "digest.cuh"
#include "host_fs.h"
#include "poly.h"
#include "shard.h"
#include <array>
#include <atomic>
#include <memory>
#include <thread>

namespace dg {

namespace {

struct StageClock {
    cudaStream_t s;
    cudaEvent_t ev[10];
    explicit StageClock(cudaStream_t stream) : s(stream) { for (auto &e : ev) DG_CUDA(cudaEventCreate(&e)); }
    ~StageClock() { for (auto &e : ev) cudaEventDestroy(e); }
    void mark(int i) { DG_CUDA(cudaEventRecord(ev[i], s)); }
    float between(int a, int b) { float ms = 0; cudaEventElapsedTime(&ms, ev[a], ev[b]); return ms; }
};

// optional fine-grained device timeline (DG_SUBSTAGE=1): named event marks inside the nine stages, printed by rank 0 after the proof
struct SubClock {
    bool on;
    cudaStream_t s;
    std::vector<std::pair<std::string, cudaEvent_t>> marks;
    explicit SubClock(cudaStream_t stream) : on(getenv("DG_SUBSTAGE") != nullptr), s(stream) {}
    void mark(const char *name) {
        if (!on) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, s);
        marks.emplace_back(name, e);
    }
    void report(int rank) {
        if (!on) return;
        cudaStreamSynchronize(s);
        std::string line = "SUBSTAGE rank " + std::to_string(rank) + ":";
        for (size_t i = 1; i < marks.size(); i++) {
            float ms = 0;
            cudaEventElapsedTime(&ms, marks[i - 1].second, marks[i].second);
            char buf[96];
            snprintf(buf, sizeof buf, " %s=%.3f", marks[i].first.c_str(), ms);
            line += buf;
        }
        if (rank == 0 || atoi(getenv("DG_SUBSTAGE")) >= 2) fprintf(stderr, "%s\n", line.c_str());
        for (auto &m : marks) cudaEventDestroy(m.second);
        marks.clear();
    }
};

void d2h(Context &c, void *dst, const void *src, size_t bytes) {
    DG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c.stream));
    DG_CUDA(cudaStreamSynchronize(c.stream));
}
void h2d(Context &c, void *dst, const void *src, size_t bytes) {
    DG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c.stream));
}

// optional dump of intermediate device buffers (differential debugging against the oracle): DG_DEBUG_DUMP=<dir>
void debug_dump(Context &c, const char *name, const void *dev, size_t bytes) {
    const char *dir = getenv("DG_DEBUG_DUMP");
    if (!dir) return;
    std::vector<uint8_t> host(bytes);
    d2h(c, host.data(), dev, bytes);
    std::string path = std::string(dir) + "/" + name + ".bin";
    FILE *f = fopen(path.c_str(), "wb");
    if (!f) return;
    fwrite(host.data(), 1, bytes, f);
    fclose(f);
}

void debug_dump_host(const char *name, const void *host, size_t bytes) {
    const char *dir = getenv("DG_DEBUG_DUMP");
    if (!dir) return;
    std::string path = std::string(dir) + "/" + name + ".bin";
    FILE *f = fopen(path.c_str(), "wb");
    if (!f) return;
    fwrite(host, 1, bytes, f);
    fclose(f);
}


void write_digest_vec(fs::ByteWriter &w, const std::vector<Digest> &v) {
    w.u64(v.size());
    for (auto &d : v) w.raw(d.data(), 32);
}
void write_digest_vv(fs::ByteWriter &w, const std::vector<std::vector<Digest>> &v) {
    w.u64(v.size());
    for (auto &x : v) write_digest_vec(w, x);
}
void write_felt_vec(fs::ByteWriter &w, const std::vector<fe> &v) {
    w.u64(v.size());
    for (auto &x : v) w.felt(x);
}

int ilog2(uint64_t v) { int l = 0; while ((1ULL << l) < v) l++; return l; }

struct FriLayerDev {
    DevBuf leaves, nodes, folded;     // row hashes, tree, and the folded values (= values of the next layer)
    const fe *vals;                   // replicated layer: the whole vector; sharded layer: this rank's cosets [c - c0][k]
    Layout layout;                    // layout of the (whole) layer (domain size 2^layout.log_d)
    bool sharded = false;             // multi-GPU: rows hashed / folded per coset range, tree = ShardedTree over [k'][c - c0] items
    ShardedTree tree;
    Digest root;
};

}  // namespace

// Upload of a host trace, overlapped with stage 1: column chunk i is extended as soon as its copy has landed.
//   * pinned (page-locked / registered) columns: cudaMemcpyAsync straight from the caller's memory on the copy stream;
//   * pageable columns (what a Rust Vec<u128> is): cudaMemcpyAsync would stage them through the driver's bounce buffer at ~8 GB/s and
//     block the calling thread (r02: 155 ms end to end instead of 104).  Instead a few worker threads memcpy columns into the
//     library's own pinned slots and enqueue the DMA from there, so staging, DMA and the LDE of earlier columns run concurrently.
// The destructor joins the workers and drains the copy streams: on an error path no DMA from the caller's buffers is left in flight
// (the caller may free them as soon as dg_prove returns).
class TraceUploader {
public:
    static const int WORKERS = 4, SLOTS = 2;
    // chunk i = columns [bounds[i], bounds[i + 1])
    TraceUploader(Context &c, fe *d_regs, const uint8_t *const *host_cols, int w, uint64_t n, const std::vector<int> &bounds)
        : c_(c), w_(w), bounds_(bounds), nchunks_((int)bounds.size() - 1), col_bytes_(n * 16), done_(nchunks_, nullptr), recorded_(nchunks_) {
        for (auto &r : recorded_) r.store(0);
        for (auto &e : done_) DG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        // the destination comes from the stream-ordered pool / arena of the compute stream: order the copies after it
        cudaEvent_t ready;
        DG_CUDA(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
        DG_CUDA(cudaEventRecord(ready, c.stream));
        cudaPointerAttributes attr;
        bool pinned = cudaPointerGetAttributes(&attr, host_cols[0]) == cudaSuccess && attr.type != cudaMemoryTypeUnregistered;
        cudaGetLastError();
        if (getenv("DG_NO_STAGING")) pinned = true;
        if (pinned) {
            DG_CUDA(cudaStreamWaitEvent(c.copy_stream, ready, 0));
            for (int i = 0; i < nchunks_; i++) {           // enqueue every upload first: the copy engine runs ahead of the compute stream
                for (int j = bounds_[i]; j < bounds_[i + 1]; j++)
                    DG_CUDA(cudaMemcpyAsync(d_regs + (size_t)j * n, host_cols[j], col_bytes_, cudaMemcpyHostToDevice, c.copy_stream));
                DG_CUDA(cudaEventRecord(done_[i], c.copy_stream));
                recorded_[i].store(1);
            }
        } else {
            c.staging.ensure((size_t)WORKERS * SLOTS * col_bytes_);
            for (int t = 0; t < WORKERS; t++) {
                if (!c.staging_streams[t]) DG_CUDA(cudaStreamCreateWithFlags(&c.staging_streams[t], cudaStreamNonBlocking));
                DG_CUDA(cudaStreamWaitEvent(c.staging_streams[t], ready, 0));
            }
            const int dev = c.device;
            for (int t = 0; t < WORKERS; t++)
                workers_.emplace_back([this, t, dev, d_regs, host_cols, n]() {
                    cudaSetDevice(dev);
                    cudaStream_t st = c_.staging_streams[t];
                    cudaEvent_t slot_free[SLOTS] = {nullptr, nullptr};
                    int use = 0;
                    // worker t owns the chunks i = t, t + WORKERS, ... ; chunks complete in order per worker, the consumer waits per chunk
                    for (int i = t; i < nchunks_ && !failed_.load(); i += WORKERS) {
                        for (int j = bounds_[i]; j < bounds_[i + 1]; j++, use++) {
                            const int s = use % SLOTS;
                            uint8_t *slot = (uint8_t *)c_.staging.p + ((size_t)t * SLOTS + s) * col_bytes_;
                            if (slot_free[s]) cudaEventSynchronize(slot_free[s]);
                            else cudaEventCreateWithFlags(&slot_free[s], cudaEventDisableTiming);
                            memcpy(slot, host_cols[j], col_bytes_);
                            if (cudaMemcpyAsync(d_regs + (size_t)j * n, slot, col_bytes_, cudaMemcpyHostToDevice, st) != cudaSuccess) failed_.store(true);
                            cudaEventRecord(slot_free[s], st);
                        }
                        if (cudaEventRecord(done_[i], st) != cudaSuccess) failed_.store(true);
                        recorded_[i].store(1);
                    }
                    for (int i = t; i < nchunks_; i += WORKERS) recorded_[i].store(1);      // after a failure: release the consumer
                    cudaStreamSynchronize(st);
                    for (auto &e : slot_free) if (e) cudaEventDestroy(e);
                });
        }
        cudaEventDestroy(ready);
    }
    // makes the compute stream wait for chunk i (blocks the host only until the copy of that chunk has been enqueued)
    void wait_chunk(int i) {
        while (!recorded_[i].load()) std::this_thread::yield();
        if (failed_.load()) throw Error(DG_ERR_CUDA, "host trace upload failed");
        DG_CUDA(cudaStreamWaitEvent(c_.stream, done_[i], 0));
    }
    int chunks() const { return nchunks_; }
    ~TraceUploader() {
        failed_.store(true);                               // stops workers that have not started their next chunk (normal exit: all done)
        for (auto &t : workers_) t.join();
        cudaStreamSynchronize(c_.copy_stream);
        for (auto &e : done_) if (e) cudaEventDestroy(e);
    }
private:
    Context &c_;
    int w_;
    std::vector<int> bounds_;
    int nchunks_;
    size_t col_bytes_;
    std::vector<cudaEvent_t> done_;
    std::vector<std::atomic<int>> recorded_;
    std::atomic<bool> failed_{false};
    std::vector<std::thread> workers_;
};

// d_regs: register traces in device memory; when `host_cols` is given they are not there yet: column chunks are uploaded on the
// copy stream while the previous chunk is being interpolated and extended (the upload hides behind the LDE); H: the commitment hash
template <class H>
static Proof *prove_pipeline(Context &c, fe *d_regs, const uint8_t *const *host_cols, uint32_t width, uint64_t length, uint32_t ctx_depth,
                             uint32_t loop_depth, const uint8_t *inputs16, uint32_t n_inputs, const uint8_t *outputs16, uint32_t n_outputs,
                             const dg_options_t &opt, dg_prove_stats_t *stats) {
    // ---- argument checks (trace_table.rs:23-58, options.rs:29-50, lib.rs:33-34) -----------------------------------------------
    const uint64_t n = length, b = opt.extension_factor;
    DG_REQUIRE(b >= 16 && b <= 256 && (b & (b - 1)) == 0, "extension_factor must be a power of 2 between 16 and 256");
    DG_REQUIRE(opt.num_queries > 0 && opt.num_queries <= 128, "num_queries must be in 1..128");
    DG_REQUIRE(opt.grinding_factor <= 32, "grinding factor cannot be greater than 32");
    DG_REQUIRE(n >= 16 && (n & (n - 1)) == 0, "execution trace length must be a power of 2 and at least 16");
    DG_REQUIRE(ctx_depth <= 16, "context depth cannot be greater than 16");
    DG_REQUIRE(loop_depth <= 8, "loop depth cannot be greater than 8");
    DG_REQUIRE(width < 128, "execution trace cannot have more than 128 registers");
    DG_REQUIRE(width > 15 + ctx_depth + loop_depth, "user stack must consist of at least one register");
    DG_REQUIRE(n_inputs <= 8 && n_outputs <= 8, "cannot have more than 8 public inputs / outputs");
    const int w = (int)width, log_n = ilog2(n), log_b = ilog2(b), log_N = log_n + log_b;
    DG_REQUIRE(log_N <= 30, "LDE domain too large");
    const uint64_t N = n * b, E = n * 8;
    const int stack_depth = w - 15 - (int)ctx_depth - (int)loop_depth;
    DG_REQUIRE(stack_depth <= 32, "stack depth cannot be greater than 32");
    std::vector<fe> inputs(n_inputs), outputs(n_outputs);
    if (n_inputs) memcpy(inputs.data(), inputs16, n_inputs * 16);
    if (n_outputs) memcpy(outputs.data(), outputs16, n_outputs * 16);

    ArenaScope arena_scope;                   // all DevBufs below come from the per-proof arena (no driver allocation inside a proof)
    StageClock clk(c.stream);
    SubClock sub(c.stream);
    if (sub.on) c.mark = [&sub](const char *name) { sub.mark(name); }; else c.mark = nullptr;
    struct MarkReset { Context &c; ~MarkReset() { c.mark = nullptr; } } mark_reset{c};
    const unsigned long long launches0 = c.launches;
    Proof *proof = new Proof();
    std::unique_ptr<Proof> guard(proof);

    // ---- sharding: rank g owns the LDE cosets [c0, c0 + nc) of every column (world == 1: all of them) ------------------------------
    const int G = c.world, g = c.rank;
    int log_g = 0;
    while ((1 << log_g) < G) log_g++;
    DG_REQUIRE((b >> log_g) >= 4 && G <= 8, "extension factor too small for this many GPUs (need >= 4 cosets per rank)");
    const int log_nc = log_b - log_g;
    const uint64_t nc = 1ULL << log_nc, N_loc = n * nc;
    const unsigned c0 = (unsigned)(g * nc);

    // ---- 1: extend execution trace ---------------------------------------------------------------------------------------------------
    clk.mark(0);
    sub.mark("start");
    // G > 1: the interpolation is sharded by columns -- rank r interpolates the columns [col_start(r), col_start(r) + col_count(r)), an
    // even split (the first w mod G ranks own one more), and only needs (from a host trace: only uploads) those registers -- the
    // polynomials are all-gathered (equal slots of cpr columns per rank, then compacted into natural column order) and every rank
    // extends all columns on its cosets
    const int cpr = (w + G - 1) / G;                           // slot size of the gather = largest share
    auto col_count = [&](int r) { return w / G + (r < w % G ? 1 : 0); };
    auto col_start = [&](int r) { return r * (w / G) + std::min(r, w % G); };
    DevBuf polys((size_t)w * n * 16), ext((size_t)w * N_loc * 16);
    if (G == 1) {
        if (!host_cols) {
            ntt_batch(c, d_regs, polys.as<fe>(), log_n, w, n, n, true);
            lde_batch(c, polys.as<fe>(), ext.as<fe>(), log_n, log_b, 1, w, n, N_loc, c0, (unsigned)nc);
        } else {
            // chunks of ~64 MB, but a short ramp first (1, 2 columns): the first transform starts after one column's worth of copying
            const int chunk = (int)std::max<uint64_t>(1, std::min<uint64_t>(w, ((uint64_t)1 << 26) / (n * 16)));
            std::vector<int> bounds = {0};
            for (int step = 1; bounds.back() < w; step = std::min(chunk, step * 2)) bounds.push_back(std::min(w, bounds.back() + step));
            TraceUploader up(c, d_regs, host_cols, w, n, bounds);
            for (int i = 0; i < up.chunks(); i++) {
                const int j0 = bounds[i], cols = bounds[i + 1] - j0;
                up.wait_chunk(i);
                ntt_batch(c, d_regs + (size_t)j0 * n, polys.as<fe>() + (size_t)j0 * n, log_n, cols, n, n, true);
                lde_batch(c, polys.as<fe>() + (size_t)j0 * n, ext.as<fe>() + (size_t)j0 * N_loc, log_n, log_b, 1, cols, n, N_loc, c0, (unsigned)nc);
            }
        }
    } else {
        const int j0 = col_start(g), mine = col_count(g);
        DevBuf own((size_t)cpr * n * 16), slots((size_t)cpr * G * n * 16);
        if (mine > 0) {
            if (host_cols) {
                std::vector<int> bounds(mine + 1);
                for (int i = 0; i <= mine; i++) bounds[i] = i;
                TraceUploader up(c, d_regs + (size_t)j0 * n, host_cols + j0, mine, n, bounds);      // one column per chunk: all staging workers busy
                for (int i = 0; i < up.chunks(); i++) {              // interpolate every column as soon as it has landed
                    up.wait_chunk(i);
                    ntt_batch(c, d_regs + (size_t)(j0 + i) * n, own.as<fe>() + (size_t)i * n, log_n, 1, n, n, true);
                }
            } else {
                ntt_batch(c, d_regs + (size_t)j0 * n, own.as<fe>(), log_n, mine, n, n, true);
            }
        }
    sub.mark("1.intt");
        // the all-gather of the polynomials (and their compaction into column order) runs on the communication stream while this rank
        // already extends its own columns
        cudaEvent_t ev_own, ev_all;
        DG_CUDA(cudaEventCreateWithFlags(&ev_own, cudaEventDisableTiming));
        DG_CUDA(cudaEventCreateWithFlags(&ev_all, cudaEventDisableTiming));
        DG_CUDA(cudaEventRecord(ev_own, c.stream));
        DG_CUDA(cudaStreamWaitEvent(c.comm_stream, ev_own, 0));
        comm_all_gather(c, own.p, slots.p, (size_t)cpr * n * 16, c.comm_stream);
        for (int r = 0; r < G; r++)
            if (col_count(r) > 0)
                DG_CUDA(cudaMemcpyAsync(polys.as<fe>() + (size_t)col_start(r) * n, slots.as<fe>() + (size_t)r * cpr * n, (size_t)col_count(r) * n * 16,
                                        cudaMemcpyDeviceToDevice, c.comm_stream));
        DG_CUDA(cudaEventRecord(ev_all, c.comm_stream));
        if (mine > 0) lde_batch(c, own.as<fe>(), ext.as<fe>() + (size_t)j0 * N_loc, log_n, log_b, 1, mine, n, N_loc, c0, (unsigned)nc);
    sub.mark("1.lde_own");
        DG_CUDA(cudaStreamWaitEvent(c.stream, ev_all, 0));
        if (j0 > 0) lde_batch(c, polys.as<fe>(), ext.as<fe>(), log_n, log_b, 1, j0, n, N_loc, c0, (unsigned)nc);
        if (j0 + mine < w)
            lde_batch(c, polys.as<fe>() + (size_t)(j0 + mine) * n, ext.as<fe>() + (size_t)(j0 + mine) * N_loc, log_n, log_b, 1, w - j0 - mine, n, N_loc, c0,
                      (unsigned)nc);
        cudaEventDestroy(ev_own);
        cudaEventDestroy(ev_all);
    }

    // ---- 2: trace Merkle tree ----------------------------------------------------------------------------------------------------------
    clk.mark(1);
    sub.mark("1.lde");
    DevBuf t_leaves(N_loc * 32);
    hash_trace_rows<H>(c, ext.as<fe>(), t_leaves.p, w, log_n, log_nc);          // local rows, [k][c - c0]
    sub.mark("2.hash_rows");
    ShardedTree t_tree;
    t_tree.build<H>(c, t_leaves.p, n, log_nc);
    memcpy(proof->trace_root, t_tree.root.data(), 32);

    // ---- 3: evaluate constraints --------------------------------------------------------------------------------------------------------
    clk.mark(2);
    sub.mark("2.tree");
    fe last_row[3];     // op_counter and program hash of the last trace step (evaluator.rs:73-74)
    if (host_cols) {
        for (int j = 0; j < 3; j++) memcpy(&last_row[j], host_cols[j] + (n - 1) * 16, 16);
    } else {
        DevBuf d_last(48);
        for (int j = 0; j < 3; j++) DG_CUDA(cudaMemcpyAsync((uint8_t *)d_last.p + 16 * j, d_regs + (size_t)j * n + (n - 1), 16, cudaMemcpyDeviceToDevice, c.stream));
        d2h(c, last_row, d_last.p, 48);
    }
    const fe op_count = last_row[0];
    const fe program_hash[2] = {last_row[1], last_row[2]};
    fs::ConstraintCoefficients cc = fs::draw_constraint_coefficients(proof->trace_root, ctx_depth, loop_depth, stack_depth, inputs, outputs,
                                                                      op_count, program_hash);
    DevBuf &d_periodic = c.d_periodic;
    if (!d_periodic.p) {
        std::vector<fe> per = fs::periodic_tables();
        d_periodic.alloc(per.size() * 16, true);
        h2d(c, d_periodic.p, per.data(), per.size() * 16);
        DG_CUDA(cudaStreamSynchronize(c.stream));
    }
    const size_t T = cc.coefA.size(), nb = cc.bAi.size();
    DevBuf d_coef((2 * T + 4 * nb) * 16), d_violation(4);
    {
        std::vector<fe> pack;
        pack.insert(pack.end(), cc.coefA.begin(), cc.coefA.end());
        pack.insert(pack.end(), cc.coefB.begin(), cc.coefB.end());
        pack.insert(pack.end(), cc.bAi.begin(), cc.bAi.end());
        pack.insert(pack.end(), cc.bBi.begin(), cc.bBi.end());
        pack.insert(pack.end(), cc.bAf.begin(), cc.bAf.end());
        pack.insert(pack.end(), cc.bBf.begin(), cc.bBf.end());
        h2d(c, d_coef.p, pack.data(), pack.size() * 16);
        DG_CUDA(cudaStreamSynchronize(c.stream));
    }
    DG_CUDA(cudaMemsetAsync(d_violation.p, 0, 4, c.stream));
    DevBuf evals(3 * E * 16);                 // [boundary numerator, first step | boundary numerator, last step | transition combination]
    {
        const int num_c8 = 8 >> log_g;
        const uint64_t E_loc = n * num_c8;
        DevBuf evals_loc(E_loc * 16), gathered(E * 16);
        AirParams P;
        memset(&P, 0, sizeof P);
        P.w = w; P.ctx_depth = ctx_depth; P.loop_depth = loop_depth; P.stack_depth = stack_depth;
        P.cl = std::max<int>(ctx_depth, 1); P.ll = std::max<int>(loop_depth, 1); P.sl = std::max(stack_depth, 8);
        P.log_n = log_n; P.log_blowup = log_b;
        P.ext = ext.as<fe>(); P.col_stride = N_loc;
        P.c8_base = g * num_c8; P.num_c8 = num_c8;
        P.t_ev = evals_loc.as<fe>();
        P.periodic = d_periodic.as<fe>();
        const fe *base = d_coef.as<fe>();
        P.coefA = base; P.coefB = base + T;
        P.twN = c.twiddle(log_N, false);
        static const int GROUP_DEG[6] = {2, 3, 4, 6, 7, 8};
        for (int gi = 0; gi < 6; gi++) P.inc[gi] = (8 * n - 1) - (n - 1) * GROUP_DEG[gi];
        P.violation = d_violation.as<unsigned>();
    sub.mark("3.setup");
        launch_constraint_eval(c, P);
    sub.mark("3.eval");
        comm_all_reduce_max_u32(c, d_violation.as<unsigned>(), 1);
        unsigned violation = 0;
        d2h(c, &violation, d_violation.p, 4);
        if (violation) throw Error(DG_ERR_UNSATISFIED, "transition constraints at step " + std::to_string(violation - 1) + " were not satisfied");
        // interpolation of the transition combination (constraint_table.rs:54-63), coset by coset: size-n inverse transforms of the own
        // cosets (sharded), all-gather, then the 8-point inverse DFT across cosets (poly.cu: coset_interp_finish) -> the 8n coefficients
        // in natural order; no transposition and no replicated 8n-point transform
    sub.mark("3.violation_sync");
        ntt_batch(c, evals_loc.as<fe>(), evals_loc.as<fe>(), log_n, num_c8, n, n, true);
        comm_all_gather(c, evals_loc.as<fe>(), gathered.as<fe>(), E_loc * 16);
    sub.mark("3.intt+gather");
        coset_interp_finish(c, gathered.as<fe>(), evals.as<fe>() + 2 * E, log_n);
        // boundary constraints (evaluator.rs:181-326), directly as the 8n coefficients the reference obtains by interpolation
        boundary_coeffs(c, polys.as<fe>(), n, (int)nb, base + 2 * T, cc.KiA, cc.KiB, cc.KfA, cc.KfB, evals.as<fe>(), evals.as<fe>() + E);
    }
    debug_dump(c, "t_coeffs", evals.as<fe>() + 2 * E, E * 16);

    // ---- 4: convert constraint evaluations into a polynomial -----------------------------------------------------------------------------
    clk.mark(3);
    sub.mark("3.finish+boundary");
    DevBuf combined(E * 16), scratch(E * 16), scratch2(E * 16);
    const fe root_n = host_root_of_unity(log_n);
    const fe x_last = host_inv(root_n);                        // w_n^(n-1)   (evaluator.rs:128-131)
    {
        debug_dump(c, "i_coeffs", evals.as<fe>(), E * 16);
        debug_dump(c, "f_coeffs", evals.as<fe>() + E, E * 16);
        fe *ic = evals.as<fe>(), *fc = evals.as<fe>() + E, *tc = evals.as<fe>() + 2 * E;
        PowTable one_t(c, fe_make(1, 0), E + 1), xl_t(c, x_last, E + 1), xli_t(c, root_n, E + 1);
        syn_div(c, ic, ic, scratch.as<fe>(), E, one_t.ref(), one_t.ref(), fe_make(0, 0));            // / (x - 1)
        syn_div(c, fc, fc, scratch.as<fe>(), E, xl_t.ref(), xli_t.ref(), fe_make(0, 0));             // / (x - x_last)
        syn_div_expanded_sum(c, tc, scratch.as<fe>(), ic, fc, combined.as<fe>(), n, E, x_last);      // / ((x^n - 1)/(x - x_last)), summed
    }
    debug_dump(c, "constraint_poly", combined.p, E * 16);

    // ---- 5: constraint evaluations over the LDE domain + their Merkle tree -----------------------------------------------------------------
    clk.mark(4);
    sub.mark("4.combine");
    DevBuf c_ext(N_loc * 16), c_items((N_loc / 4) * 32);
    lde_batch(c, combined.as<fe>(), c_ext.as<fe>(), log_n, log_b, 8, 1, E, N_loc, c0, (unsigned)nc);
    sub.mark("5.lde");
    constraint_items_local<H>(c, c_ext.as<fe>(), log_n, log_nc, c_items.p);      // first tree level: H(4 evaluations), [k][c4 local]
    sub.mark("5.items");
    ShardedTree c_tree;
    c_tree.build<H>(c, c_items.p, n, log_nc - 2);
    memcpy(proof->constraint_root, c_tree.root.data(), 32);

    // ---- 6: DEEP composition polynomial ---------------------------------------------------------------------------------------------------------
    clk.mark(5);
    sub.mark("5.tree");
    fs::CompositionCoefficients dc = fs::draw_composition_coefficients(proof->constraint_root, w);
    const fe z = dc.z, zg = fe_mul(z, root_n);
    std::vector<fe> state1(w), state2(w);
    DevBuf comp(E * 16), comp_ext(N_loc * 16);
    {
        PowTable z_t(c, z, E + 1), zi_t(c, host_inv(z), E + 1), zg_t(c, zg, n + 1), zgi_t(c, host_inv(zg), n + 1);
        TwiddleRef g_t = c.twiddle(log_n, false);
        // trace polynomials at z and z*g: every rank evaluates its own columns (the split of stage 1); slots of 2 cpr values are gathered
        const int wp = cpr * G;
        DevBuf d_deep((size_t)(2 * wp + 2) * 16);
        DG_CUDA(cudaMemsetAsync(d_deep.p, 0, d_deep.bytes, c.stream));
        {
            const int j0 = col_start(g), mine = col_count(g);
            if (mine > 0) eval_polys_at(c, polys.as<fe>() + (size_t)j0 * n, n, mine, z_t.ref(), g_t, true, d_deep.as<fe>() + (size_t)2 * g * cpr);
            if (G > 1) comm_all_gather(c, d_deep.as<fe>() + (size_t)2 * g * cpr, d_deep.p, (size_t)2 * cpr * 16);
        }
        eval_polys_at(c, combined.as<fe>(), E, 1, z_t.ref(), g_t, false, d_deep.as<fe>() + 2 * wp);
        std::vector<fe> deep_slots(2 * wp + 2), deep(2 * w + 2);
        d2h(c, deep_slots.data(), d_deep.p, deep_slots.size() * 16);
        for (int r = 0; r < G; r++)
            for (int o = 0; o < col_count(r); o++) {
                deep[2 * (col_start(r) + o)] = deep_slots[2 * (r * cpr + o)];
                deep[2 * (col_start(r) + o) + 1] = deep_slots[2 * (r * cpr + o) + 1];
            }
        deep[2 * w] = deep_slots[2 * wp];
    sub.mark("6.deep_values");
        fe sub1 = fe_make(0, 0), sub2 = fe_make(0, 0);
        for (int i = 0; i < w; i++) {
            state1[i] = deep[2 * i]; state2[i] = deep[2 * i + 1];
            sub1 = fe_add(sub1, fe_mul(state1[i], dc.trace1[i]));
            sub2 = fe_add(sub2, fe_mul(state2[i], dc.trace2[i]));
        }
        const fe c_at_z = deep[2 * w];
        DevBuf d_cc((size_t)2 * w * 16), t12(2 * n * 16);
        h2d(c, d_cc.p, dc.trace1.data(), (size_t)w * 16);
        h2d(c, d_cc.as<fe>() + w, dc.trace2.data(), (size_t)w * 16);
        fe *t1 = t12.as<fe>(), *t2 = t12.as<fe>() + n;
        lincomb2(c, polys.as<fe>(), n, w, d_cc.as<fe>(), d_cc.as<fe>() + w, t1, t2);
        syn_div(c, t1, t1, scratch.as<fe>(), n, z_t.ref(), zi_t.ref(), sub1);                          // (T1(x) - T1(z)) / (x - z)
        syn_div(c, t2, t2, scratch.as<fe>(), n, zg_t.ref(), zgi_t.ref(), sub2);                        // (T2(x) - T2(zg)) / (x - zg)
        syn_div(c, combined.as<fe>(), scratch2.as<fe>(), scratch.as<fe>(), E, z_t.ref(), zi_t.ref(), c_at_z);   // (C(x) - C(z)) / (x - z)
    sub.mark("6.lincomb+syndiv");
        compose(c, t1, t2, scratch2.as<fe>(), comp.as<fe>(), n, E, 6 * n + 1, dc.t1_degree, dc.t2_degree, dc.constraints);
        debug_dump(c, "composition_poly", comp.p, E * 16);
        // every rank extends its own cosets; the first FRI layers work on these slabs directly (no all-gather of the N evaluations)
        lde_batch(c, comp.as<fe>(), comp_ext.as<fe>(), log_n, log_b, 8, 1, E, N_loc, c0, (unsigned)nc);
    }

    // ---- 7: FRI layers ---------------------------------------------------------------------------------------------------------------------------
    clk.mark(6);
    sub.mark("6.compose+lde");
    std::vector<FriLayerDev> layers;
    DevBuf fri_gathered;                                       // multi-GPU: the first replicated layer, gathered from the ranks' slabs
    {
        TwiddleRef inv_root = c.twiddle(log_N, true);
        const fe tau_inv = host_inv(host_root_of_unity(2));
        const fe inv4 = host_inv(fe_make(4, 0));
        const fe *cur = comp_ext.as<fe>();
        Layout lay{log_N, log_b};
        bool local = G > 1;                                    // `cur` is this rank's coset slab of the layer
        // layer roots and folding points stay on the device (special_x = prng(root) is derived by fri_alpha): the host sees the roots
        // in one copy after the last layer.  With host RNG callbacks registered each layer asks the host instead.
        const int MAX_LAYERS = 20;
        DevBuf d_alpha(MAX_LAYERS * 16), d_roots(MAX_LAYERS * 32);
        const bool host_rng = fs::rng_hooks_active();
        auto folding_point = [&](const void *root_dev, size_t layer) -> const fe * {
            DG_REQUIRE(layer < (size_t)MAX_LAYERS, "too many FRI layers");
            fe *a_dev = d_alpha.as<fe>() + layer;
            uint8_t *r_dev = (uint8_t *)d_roots.p + 32 * layer;
            if (!host_rng) { fri_alpha(c, root_dev, a_dev, r_dev); return a_dev; }
            Digest r;
            d2h(c, r.data(), root_dev, 32);
            const fe alpha = fs::prng_vector(r.data(), 1)[0];          // field::prng(seed) = first draw of the generator (field.rs:264-269)
            DG_CUDA(cudaMemcpyAsync(r_dev, root_dev, 32, cudaMemcpyDeviceToDevice, c.stream));
            DG_CUDA(cudaMemcpyAsync(a_dev, &alpha, 16, cudaMemcpyHostToDevice, c.stream));
            DG_CUDA(cudaStreamSynchronize(c.stream));
            return a_dev;
        };
        for (;;) {
            const int log_r = lay.log_d - 2;
            const uint64_t R = 1ULL << log_r;
            // layers below 2^22 values are latency-bound (two collectives per sharded tree cost more than hashing them whole): gather the
            // first such layer once (<= 32 MB) and finish redundantly on every rank
            if (local && (lay.log_d < 22 || log_r - log_b < 6)) {
                fri_gathered.alloc((size_t)16 << lay.log_d);
                comm_all_gather(c, cur, fri_gathered.p, ((size_t)16 << lay.log_d) >> log_g);     // rank-major == coset-major
                cur = fri_gathered.as<fe>();
                local = false;
            }
            layers.emplace_back();
            const size_t li = layers.size() - 1;
            FriLayerDev &L = layers.back();
            L.vals = cur; L.layout = lay; L.sharded = local;
            if (local) {
                // rows r = b k' + c of the own cosets: hashes in ShardedTree order, n' = R / b subtrees of nc leaves per rank
                L.leaves.alloc((R >> log_g) * 32);
                fri_hash_rows_local<H>(c, cur, lay.log_d, log_b, log_nc, L.leaves.p);
                L.tree.build<H>(c, L.leaves.p, R >> log_b, log_nc, false);
                const fe *alpha = folding_point(L.tree.root_dev(), li);
                L.folded.alloc((R >> log_g) * 16);
                fri_fold_local(c, cur, lay.log_d, log_b, log_nc, c0, L.folded.as<fe>(), alpha, inv_root, log_N, tau_inv, inv4);
                cur = L.folded.as<fe>();
                lay = Layout{log_r, log_b};
                continue;
            }
            const Layout rows{log_r, (lay.log_b >= 0 && log_r >= lay.log_b) ? lay.log_b : -1};
            L.leaves.alloc(R * 32); L.nodes.alloc(R * 32);
            fri_hash_rows<H>(c, cur, lay, rows, L.leaves.p);
            merkle_build<H>(c, L.leaves.p, L.nodes.p, R);
            if (R * 4 <= 256) {                                    // MAX_REMAINDER_LENGTH (fri/mod.rs:13): the remainder's root only
                DG_REQUIRE(li < (size_t)MAX_LAYERS, "too many FRI layers");
                DG_CUDA(cudaMemcpyAsync((uint8_t *)d_roots.p + 32 * li, (const uint8_t *)L.nodes.p + 32, 32, cudaMemcpyDeviceToDevice, c.stream));
                break;
            }
            const fe *alpha = folding_point((const uint8_t *)L.nodes.p + 32, li);     // special_x = prng(root)  (fri/prover.rs:29)
            L.folded.alloc(R * 16);                                // values of the next layer, owned by this one
            fri_fold(c, cur, lay, L.folded.as<fe>(), rows, alpha, inv_root, log_N, tau_inv, inv4);
            cur = L.folded.as<fe>();
            lay = rows;
        }
        std::vector<uint8_t> roots(32 * layers.size());
        d2h(c, roots.data(), d_roots.p, roots.size());
        for (size_t i = 0; i < layers.size(); i++) memcpy(layers[i].root.data(), roots.data() + 32 * i, 32);
    }

    // ---- 8: query positions ------------------------------------------------------------------------------------------------------------------------
    clk.mark(7);
    sub.mark("7.fri");
    std::vector<uint64_t> positions;
    {
        std::vector<uint8_t> roots;
        for (auto &L : layers) roots.insert(roots.end(), L.root.begin(), L.root.end());
        uint8_t seed[32];
        debug_dump_host("fri_roots", roots.data(), roots.size());
        H::message(roots.data(), roots.size(), seed);
        proof->pow_nonce = pow_search<H>(c, seed, opt.grinding_factor);
        pow_hash<H>(seed, proof->pow_nonce, proof->pow_seed);
        try {
            positions = fs::query_positions(proof->pow_seed, N, b, opt.num_queries);
        } catch (const std::exception &e) { throw Error(DG_ERR_EXHAUSTED, e.what()); }
        debug_dump_host("positions", positions.data(), positions.size() * 8);
    }

    // ---- 9: build proof object -------------------------------------------------------------------------------------------------------------------------
    clk.mark(8);
    sub.mark("8.pow");
    fs::ByteWriter out;
    {
        // Plan every opening on the host, fetch all opened values / digests in one batched pass (FetchBatch), then serialise.
        const int nq = (int)positions.size();
        FetchBatch fb(c);
        typedef std::vector<std::vector<size_t>> Offsets;
        // registers the nodes of a batch-proof plan; leaf_ref / node_ref map leaf indices / heap indices to fetch references
        auto plan_offsets = [&](const fs::BatchPlan &plan, auto leaf_ref, auto node_ref) {
            Offsets o(plan.nodes.size());
            for (size_t sidx = 0; sidx < plan.nodes.size(); sidx++)
                for (auto &r : plan.nodes[sidx]) o[sidx].push_back(fb.add32(r.leaf ? leaf_ref(r.index) : node_ref(r.index)));
            return o;
        };
        auto digests_at = [&](const Offsets &o) {
            std::vector<std::vector<Digest>> v(o.size());
            for (size_t i = 0; i < o.size(); i++)
                for (size_t off : o[i]) v[i].push_back(fb.digest(off));
            return v;
        };

        // trace rows at the queried positions (trace_table.rs:127-134): the rank owning the position's coset reads the row
        std::vector<size_t> row_off(nq);
        for (int q = 0; q < nq; q++) {
            const uint64_t cpos = positions[q] & (b - 1), k = positions[q] >> log_b;
            const int owner = (int)(cpos >> log_nc);
            const uint64_t phys = ((cpos - (uint64_t)owner * nc) << log_n) + k;
            for (int j = 0; j < w; j++) {
                const size_t off = fb.add16(FetchRef{ext.as<fe>() + (size_t)j * N_loc, phys, owner});
                if (j == 0) row_off[q] = off;
            }
        }
        // trace tree openings: leaves are the row hashes
        fs::BatchPlan tplan = fs::plan_batch_proof(positions, N);
        Offsets t_off = plan_offsets(tplan, [&](uint64_t i) { return t_tree.item_ref(i); }, [&](uint64_t h) { return t_tree.node_ref(h); });

        // constraint tree openings: leaf j = evaluations (2j, 2j+1), unhashed (prover.rs:180-187); evaluation 2j+1 lives in the next
        // coset at the same k, i.e. n elements further in the owner's slab: two 16-byte units registered back to back = one 32-byte item
        auto constraint_leaf = [&](uint64_t j) {
            const uint64_t i = 2 * j, cpos = i & (b - 1), k = i >> log_b;
            const int owner = (int)(cpos >> log_nc);
            const uint64_t p0 = ((cpos - (uint64_t)owner * nc) << log_n) + k;
            const size_t off = fb.add16(FetchRef{c_ext.as<fe>(), p0, owner});
            fb.add16(FetchRef{c_ext.as<fe>(), p0 + n, owner});
            return off;
        };
        std::vector<uint64_t> c_positions = fs::constraint_positions(positions);
        fs::BatchPlan cplan = fs::plan_batch_proof(c_positions, N / 2);
        std::vector<size_t> cval_off;
        for (uint64_t j : cplan.value_leaves) cval_off.push_back(constraint_leaf(j));
        Offsets c_off(cplan.nodes.size());
        for (size_t sidx = 0; sidx < cplan.nodes.size(); sidx++)
            for (auto &r : cplan.nodes[sidx]) {
                // heap indices of the tree over N/2 leaves: [N/4, N/2) is the first hashed level (= level-0 items of c_tree)
                if (r.leaf) c_off[sidx].push_back(constraint_leaf(r.index));
                else if (r.index >= N / 4) c_off[sidx].push_back(fb.add32(c_tree.item_ref(r.index - N / 4)));
                else c_off[sidx].push_back(fb.add32(c_tree.node_ref(r.index)));
            }

        // FRI layers (fri/prover.rs:55-95)
        struct LayerOpen { std::vector<uint64_t> pos; std::vector<size_t> val_off; Offsets node_off; uint8_t depth; };
        std::vector<LayerOpen> fri_open(layers.size() - 1);
        std::vector<uint64_t> fpos = positions;
        for (size_t d = 0; d + 1 < layers.size(); d++) {
            FriLayerDev &L = layers[d];
            LayerOpen &O = fri_open[d];
            const uint64_t D = 1ULL << L.layout.log_d, R = D / 4;
            fpos = fs::augmented_positions(fpos, D);
            O.pos = fpos;
            fs::BatchPlan plan = fs::plan_batch_proof(fpos, R);
            O.depth = plan.depth;
            for (uint64_t p : fpos)
                for (int j = 0; j < 4; j++) {
                    size_t off;
                    if (L.sharded) {
                        const uint64_t cpos = p & (b - 1), k = (p >> log_b) + (uint64_t)j * (R >> log_b);
                        const int owner = (int)(cpos >> log_nc);
                        off = fb.add16(FetchRef{L.vals, ((cpos - (uint64_t)owner * nc) << (L.layout.log_d - log_b)) + k, owner});
                    } else {
                        off = fb.add16(FetchRef{L.vals, L.layout.phys(p + j * R), -1});
                    }
                    if (j == 0) O.val_off.push_back(off);
                }
            if (L.sharded) O.node_off = plan_offsets(plan, [&](uint64_t i) { return L.tree.item_ref(i); }, [&](uint64_t h) { return L.tree.node_ref(h); });
            else O.node_off = plan_offsets(plan, [&](uint64_t i) { return FetchRef{L.leaves.p, i, -1}; }, [&](uint64_t h) { return FetchRef{L.nodes.p, h, -1}; });
        }
        std::vector<size_t> rem_off;
        {
            FriLayerDev &L = layers.back();
            const uint64_t D = 1ULL << L.layout.log_d;
            for (uint64_t i = 0; i < D; i++) rem_off.push_back(fb.add16(FetchRef{L.vals, L.layout.phys(i), -1}));   // remainder, natural order
        }
        fb.run();

        // ---- serialise (proof.rs:10-37; bincode: u64 length prefixes, arrays raw, little endian)
        out.raw(proof->trace_root, 32);
        out.u8(tplan.depth); out.u8((uint8_t)ctx_depth); out.u8((uint8_t)loop_depth); out.u8((uint8_t)stack_depth);
        out.u32((uint32_t)op_count.lo);                                               // op_count as u32 (proof.rs:62)
        write_digest_vv(out, digests_at(t_off));
        out.u64(nq);
        for (int q = 0; q < nq; q++) {
            out.u64(w);
            for (int j = 0; j < w; j++) out.felt(fb.value(row_off[q] + j));
        }
        out.raw(proof->constraint_root, 32);
        out.u64(cval_off.size());
        for (size_t off : cval_off) { Digest dgt = fb.digest(off); out.raw(dgt.data(), 32); }
        write_digest_vv(out, digests_at(c_off));
        out.u8(cplan.depth);
        write_felt_vec(out, state1);
        write_felt_vec(out, state2);

        out.u64(layers.size() - 1);
        for (size_t d = 0; d + 1 < layers.size(); d++) {
            LayerOpen &O = fri_open[d];
            out.raw(layers[d].root.data(), 32);
            out.u64(O.pos.size());
            for (size_t off : O.val_off)
                for (int j = 0; j < 4; j++) out.felt(fb.value(off + j));
            write_digest_vv(out, digests_at(O.node_off));
            out.u8(O.depth);
        }
        out.raw(layers.back().root.data(), 32);
        out.u64(rem_off.size());
        for (size_t off : rem_off) out.felt(fb.value(off));
        out.u64(proof->pow_nonce);
        out.u8((uint8_t)log_b); out.u8((uint8_t)opt.num_queries); out.u8((uint8_t)opt.grinding_factor); out.u8((uint8_t)H::id);
    }
    clk.mark(9);
    sub.mark("9.openings");
    sub.report(c.rank);
    DG_CUDA(cudaStreamSynchronize(c.stream));
    proof->bytes = std::move(out.b);
    if (stats) {
        for (int i = 0; i < 9; i++) stats->stage_ms[i] = clk.between(i, i + 1);
        stats->h2d_ms = 0.0f;                        // host variant: uploads overlap stage 1 and are part of stage_ms[0]
        stats->total_ms = clk.between(0, 9);
        stats->kernel_launches = c.launches - launches0;
    }
    return guard.release();
}

static Proof *prove_core(Context &c, fe *d_regs, const uint8_t *const *host_cols, uint32_t width, uint64_t length, uint32_t ctx_depth,
                         uint32_t loop_depth, const uint8_t *inputs16, uint32_t n_inputs, const uint8_t *outputs16, uint32_t n_outputs,
                         const dg_options_t &opt, dg_prove_stats_t *stats) {
    if (const char *why = proof_hash_error(opt.hash_id)) throw Error(DG_ERR_INVALID, why);
    return with_proof_hash(opt.hash_id, [&](auto h) {
        return prove_pipeline<decltype(h)>(c, d_regs, host_cols, width, length, ctx_depth, loop_depth, inputs16, n_inputs, outputs16, n_outputs,
                                           opt, stats);
    });
}

Proof *prove_device(Context &c, const fe *d_regs, uint32_t width, uint64_t length, uint32_t ctx_depth, uint32_t loop_depth,
                    const uint8_t *inputs16, uint32_t n_inputs, const uint8_t *outputs16, uint32_t n_outputs, const dg_options_t &opt,
                    dg_prove_stats_t *stats, float) {
    return prove_core(c, const_cast<fe *>(d_regs), nullptr, width, length, ctx_depth, loop_depth, inputs16, n_inputs, outputs16, n_outputs, opt, stats);
}

Proof *prove_host(Context &c, const dg_trace_t &trace, const uint8_t *inputs16, uint32_t n_inputs, const uint8_t *outputs16,
                  uint32_t n_outputs, const dg_options_t &opt, dg_prove_stats_t *stats) {
    DG_REQUIRE(trace.columns && trace.width >= 16 && trace.width < 128, "invalid trace");
    DG_REQUIRE(trace.length >= 16 && (trace.length & (trace.length - 1)) == 0, "execution trace length must be a power of 2 and at least 16");
    for (uint32_t j = 0; j < trace.width; j++) DG_REQUIRE(trace.columns[j] != nullptr, "null register column");
    c.upload_buf.ensure((size_t)trace.length * 16 * trace.width, true);
    return prove_core(c, c.upload_buf.as<fe>(), trace.columns, trace.width, trace.length, trace.ctx_depth, trace.loop_depth, inputs16, n_inputs,
                      outputs16, n_outputs, opt, stats);
}

}  // namespace dg
