#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200 STARK prover backend (contract: see the task brief / DESIGN.md section 6).

Metric (BASELINE.json): prove ms for a 2^20-step trace at default 120-bit ProofOptions (LDE blowup 32, 50 queries,
20-bit grinding, blake3).  One "step" = one complete proof of the same execution trace.

  python bench.py [--gpus N] [--steps K] [--warmup W]             our arm (CUDA prover)
  python bench.py --impl reference [--steps K] [--warmup W]       reference arm: the CPU restatement of the reference
                                                                  prover (oracle/, single thread) on a bounded sample
  --dump-outputs DIR (our arm): also write the proof of the last timed step to DIR/<name>.npy (see dump_outputs)
Workload: the reference's collatz example (src/examples/collatz.rs) with a start value whose trajectory has 2600 steps,
which the VM turns into 548k operations => a trace of 2^20 steps x 26 registers.
N > 1: one process per GPU (torchrun); ONE proof is sharded over the N ranks by LDE coset ranges (DESIGN.md section 7): every
rank holds the trace, extends / hashes / evaluates constraints on its own cosets and the ranks meet in NCCL all-gathers at the
commitment points.  Total work is fixed => "scaling": "strong"; `value` = time of that one proof (max over ranks).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

COLLATZ_START_2_20 = 6012607780440691934780549639      # 2600 Collatz steps, all iterates < 2^99
METRIC = "prove ms for 2^20-step trace (default 120-bit ProofOptions)"


def metric_name(log_n):
    return METRIC if log_n == 20 else "prove ms for 2^%d-step trace (default 120-bit ProofOptions)" % log_n


def collatz_start_for(log_n):
    """smallest-effort start values whose traces pad to 2^log_n steps (211 VM operations per Collatz iteration)"""
    table = {20: COLLATZ_START_2_20, 19: 93571393692802302, 18: 63728127, 17: 837799, 16: 6171, 15: 27, 14: 123, 13: 25, 12: 7}
    return table.get(log_n)


def build_workload(args, log_n=None):
    """--workload collatz (default, BASELINE configs[3]) | fibonacci (configs[1]: 2^16 steps) | merkle (configs[2]: 2^14 steps)"""
    from distaff_b200 import hostvm
    log_n = log_n or args.log_n
    kind = getattr(args, "workload", "collatz")
    if kind == "fibonacci":
        n_terms = (1 << log_n) // 16 - 6
        tr = hostvm.fibonacci(n_terms)
        assert tr.length == 1 << log_n, tr.length
        return tr, f"fibonacci({n_terms})"
    if kind == "merkle":
        count = {12: 1, 13: 2, 14: 4, 15: 8, 16: 16}.get(log_n)
        assert count, "--workload merkle supports --log-n 12..16 (depth-64 paths, 2^12 steps each)"
        tr = hostvm.merkle_paths(64, count)
        assert tr.length == 1 << log_n, tr.length
        return tr, f"merkle_paths(depth=64, count={count})"
    return build_trace(log_n)


def build_trace(log_n):
    from distaff_b200 import hostvm
    start = collatz_start_for(log_n)
    if start is not None:
        tr = hostvm.collatz(start)
        if tr.length == 1 << log_n:
            return tr, f"collatz(start={start})"
    # fallback: fibonacci with enough terms (16 operations per term)
    n_terms = (1 << log_n) // 16 - 6
    tr = hostvm.fibonacci(n_terms)
    assert tr.length == 1 << log_n, tr.length
    return tr, f"fibonacci({n_terms})"


class ClockSampler:
    """one background `nvidia-smi -lms` process (the recipe of B200_PROFILING.md) sampling clocks / throttle reasons during the
    timed region; a single long-lived process, because spawning nvidia-smi repeatedly perturbs the driver"""

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.samples = []

    def start(self):
        if os.environ.get("BENCH_NO_SMI"):
            return
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "250"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        for line in out.splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 7:
                self.samples.append(parts)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(self.samples)}


def peak_gbs():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "measured"
    except Exception:
        return 6650.0, "fallback"


# -------------------------------------------------------------------------------------------------------------------------
def oracle_threads():
    """threads for the CPU arm: all host threads unless BENCH_REF_THREADS says otherwise (1 = what the reference prover itself uses)"""
    # default: at most 32 -- on the 128-thread hosts of this pool the restatement is fastest there (2^16 steps: 25.7 s on 1 thread, 4.6 s on 8,
    # 2.2 s on 32, 4.6 s on 64, 9.6 s on 128: profiles/r02_oracle_threads.txt)
    return max(1, int(os.environ.get("BENCH_REF_THREADS", min(32, os.cpu_count() or 1))))


STAGE_NAMES = ["extend trace", "trace merkle tree", "evaluate constraints", "combine constraint polys", "constraint lde + tree",
               "deep composition", "fri layers", "pow + positions", "openings + proof"]


def workload_name(name, log_n, w):
    return f"{name}: trace 2^{log_n} steps x {w} registers, LDE blowup 32 (2^{log_n + 5} rows), 50 queries, 20-bit grinding, blake3"


def log_n_of(n):
    return int(n).bit_length() - 1


def dump_outputs(out_dir, proof):
    """--dump-outputs: what a caller of prove_device receives from the last timed proof, one DIR/<name>.npy per field, so that two
    builds can be compared output for output.  Every field is a byte string (the nonce as its 8 little-endian bytes), stored as one
    float32 element per byte, which is exact."""
    os.makedirs(out_dir, exist_ok=True)
    fields = {"proof": proof.bytes, "trace_root": proof.trace_root, "constraint_root": proof.constraint_root, "pow_seed": proof.pow_seed,
              "pow_nonce": proof.pow_nonce.to_bytes(8, "little")}
    for name, data in fields.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.frombuffer(data, dtype=np.uint8).astype(np.float32))


def golden_for(log_n):
    try:
        g = json.load(open(os.path.join(ROOT, "tests", "golden", "collatz_2_%d.json" % log_n)))
        return g
    except Exception:
        return None


def run_reference(args):
    """CPU arm, SAME workload as the GPU arm: the oracle prover (C++ restatement of the reference; no Rust toolchain in this image) proves
    the full 2^log_n-step collatz trace.  The reference prover is single-threaded by construction (every FFT / batch call passes
    num_threads = 1); the restatement can additionally split columns / rows / steps / sub-transforms over host threads (identical proof
    bytes), and this arm uses all of them so that the GPU is compared with the strongest CPU run available.  One step = one whole proof;
    a 2^20 proof takes minutes, so the number of timed proofs is bounded by BENCH_REF_BUDGET_S (default 240 s): at least one full
    proof is always measured, never a scaled sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import hashlib
    from oracle import pyoracle as po
    log_s = args.ref_log_n or args.log_n
    threads = po.set_threads(oracle_threads())
    tr, name = build_workload(args, log_s)
    budget_s = float(os.environ.get("BENCH_REF_BUDGET_S", "240"))
    times, stage_ms, proof = [], np.zeros(9), None
    t_start = time.perf_counter()
    planned = args.warmup + args.steps
    done_warm = 0
    for i in range(planned):
        t0 = time.perf_counter()
        r = po.prove(tr.registers, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs)
        dt = (time.perf_counter() - t0) * 1e3
        assert r.error is None, r.error
        proof = r.proof
        elapsed = time.perf_counter() - t_start
        # a proof that does not fit the budget twice is timed as it is (no warm-up pass: the CPU run has no lazy initialisation to hide)
        if i < args.warmup and elapsed + 2 * dt / 1e3 < budget_s:
            done_warm += 1
            continue
        times.append(dt)
        stage_ms += np.array(r.stage_ms)
        if elapsed + dt / 1e3 > budget_s or len(times) >= args.steps:
            break
    value = float(np.mean(times))
    sha = hashlib.sha256(proof).hexdigest()
    gold = golden_for(log_s) if args.workload == "collatz" else None
    sample = (f"{name}: the full 2^{log_s}-step trace x {tr.width} registers proven {len(times)}x in {value:.0f} ms per proof on {threads} host threads "
              f"(same workload as the GPU arm, no scaling)")
    line = {
        "impl": "reference", "metric": metric_name(log_s), "value": value, "unit": "ms", "n_gpus": args.gpus, "steps": len(times), "warmup": done_warm,
        "ms_per_step": value, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "u128 (128-bit prime field) + u32 (blake3)",
        "data": "synthetic",
        "config": {"workload": workload_name(name, log_s, tr.width),
                   "parallelism": "cpu: %d host threads" % threads, "l2": "n/a (CPU arm)", "proof_bytes": len(proof), "device": "host CPU",
                   "reference_impl": "oracle/ C++ restatement of the reference prover (Rust toolchain unavailable)"},
        "stage_ms": [float(x) / len(times) for x in stage_ms], "stage_names": STAGE_NAMES, "ms_steps": [round(float(x), 1) for x in times],
        "proof_sha256": sha, "matches_oracle_golden": (gold["proof_sha256"] == sha) if gold else None,
        "cpu_baseline": {"value": value, "unit": "ms", "cores": threads, "kind": "port", "sample": sample, "host_cores_available": os.cpu_count(),
                         "single_thread_note": "the reference itself runs on 1 thread; BENCH_REF_THREADS=1 reproduces that (756 s for this proof on the build box)"},
        "e2e": {"value": value, "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    os.environ["DG_DEVICE"] = str(local_rank)
    import torch
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import distaff_b200 as dg
    from distaff_b200 import backend
    info = backend.device_info()
    single_process = args.single_process and world == 1 and args.gpus > 1
    if world > 1:
        backend.comm_init_from_torch(dist, local_rank)
    elif single_process:
        # ONE process, one dg_prove call per proof, args.gpus GPUs: the library runs a host thread + NCCL communicator per device (dg_init_devices)
        backend.check(backend.lib().dg_init_devices(args.gpus))

    tr, name = build_workload(args)
    n, w = tr.length, tr.width
    regs = np.ascontiguousarray(tr.registers)
    opts = dg.ProofOptions()

    # device-resident arm (`value`): trace already in HBM
    dbuf = backend.DeviceBuffer(regs.nbytes).upload(regs)
    # end-to-end arm: pinned host copy of the trace, proof bytes back on the host
    pinned = torch.empty(regs.nbytes, dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = regs.reshape(-1).view(np.uint8)
    from distaff_b200 import hostvm
    pinned_regs = pinned.numpy().view(np.uint64).reshape(regs.shape)
    tr_pinned = hostvm.ExecutionTrace(pinned_regs, tr.ctx_depth, tr.loop_depth, tr.stack_depth, tr.program_hash, tr.public_inputs, tr.outputs)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                       # started before the warm-up so that its start-up cost is not inside the timed region
    proof = None
    for _ in range(args.warmup):
        proof = dg.prove_device(dbuf, w, n, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs, opts)
    barrier()
    dev_ms, stage_ms, launches = [], np.zeros(9), 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        proof = dg.prove_device(dbuf, w, n, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs, opts)
        dev_ms.append(proof.stats["total_ms"])           # CUDA events on the library's stream around the whole pipeline
        stage_ms += np.array(proof.stats["stage_ms"])
        launches += proof.stats["kernel_launches"]
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    total_dev_ms = float(np.sum(dev_ms))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, proof)

    # end-to-end: host trace (pinned) -> proof bytes on the host, through the public API call a user makes
    e2e_ms = []
    e2e_warm = min(args.warmup, 2)          # the host-buffer entry has its own first-use work (upload buffer, page pinning checks)
    for i in range(e2e_warm + args.steps):
        barrier()
        t1 = time.perf_counter()
        p2 = dg.prove(tr_pinned, opts)
        dt = (time.perf_counter() - t1) * 1e3
        if i >= e2e_warm:
            e2e_ms.append(dt)
    barrier()
    sampler.stop()
    assert p2.bytes == proof.bytes
    # the same call from ordinary pageable memory (what a Rust Vec<u128> is): not part of the headline, reported beside it
    e2e_pageable_ms = []
    for i in range(2):
        barrier()
        t1 = time.perf_counter()
        p3 = dg.prove(tr, opts)
        e2e_pageable_ms.append((time.perf_counter() - t1) * 1e3)
    barrier()
    assert p3.bytes == proof.bytes
    import hashlib
    proof_sha = hashlib.sha256(proof.bytes).hexdigest()

    if dist is not None:
        t = torch.tensor([total_dev_ms, float(np.sum(e2e_ms)), wall_ms, float(min(e2e_pageable_ms))], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_dev_ms, e2e_total, wall_ms, e2e_pageable = [float(x) for x in t.tolist()]
        # every rank must hold the same proof bytes: compare the digests
        mine = torch.frombuffer(bytearray(bytes.fromhex(proof_sha)), dtype=torch.uint8).to("cuda")
        alld = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(alld, mine)
        ranks_agree = all(bool(torch.equal(x, mine)) for x in alld)
    else:
        e2e_total = float(np.sum(e2e_ms))
        e2e_pageable = float(min(e2e_pageable_ms))
        ranks_agree = True
    if rank != 0:
        if dist is not None:
            backend.lib().dg_comm_finalize()
            dist.barrier()
            dist.destroy_process_group()
        return

    if dist is not None:
        backend.check(backend.lib().dg_comm_finalize())     # the remaining legs (roofline, CPU sample) are single-GPU work on rank 0
    ms_per_step = total_dev_ms / args.steps
    value = ms_per_step                         # one proof, sharded over `world` GPUs
    e2e_value = e2e_total / args.steps

    # ---- correctness of the timed proof (checker use of the oracle): the restated reference verifier (stark/verifier.rs) must accept it,
    #      and its SHA-256 must equal the digest of the CPU oracle's proof of the same trace committed under tests/golden/
    from oracle import pyoracle as po
    t_v = time.perf_counter()
    verdict = po.verify(tr.program_hash, tr.public_inputs, tr.outputs, proof.bytes)
    verify_ms = (time.perf_counter() - t_v) * 1e3
    gold = golden_for(log_n_of(n)) if args.workload == "collatz" else None
    trace_sha = hashlib.sha256(regs.tobytes()).hexdigest() if gold else None
    check = {"proof_sha256": proof_sha, "oracle_verifier": "accepted" if verdict is None else "REJECTED: %s" % verdict, "oracle_verify_ms": verify_ms,
             "all_ranks_same_proof": ranks_agree,
             "matches_oracle_golden": (gold["proof_sha256"] == proof_sha and gold["trace_sha256"] == trace_sha) if gold else None,
             "golden": "tests/golden/collatz_2_%d.json (CPU oracle proof of the same trace, %.0f s on the build box)" % (log_n_of(n), gold["oracle_prove_s"]) if gold else None}
    assert verdict is None, verdict
    assert ranks_agree, "ranks returned different proofs"
    if gold:
        assert check["matches_oracle_golden"], "GPU proof differs from the committed CPU-oracle digest"

    # ---- roofline of the dominant kernel (the NTT pass kernel of the trace LDE), measured live with CUDA events
    peak, peak_kind = peak_gbs()
    L = backend.lib()
    log_n = n.bit_length() - 1
    cols = min(w, 8)                            # the prover extends the trace eight columns per launch pair (4 GiB of NTT scratch): same shape here
    polys = backend.DeviceBuffer(cols * n * 16).upload(regs[:cols])
    ext = backend.DeviceBuffer(cols * n * 32 * 16)
    ms = ctypes.c_float(0)
    lde_ms = []
    for i in range(6):
        backend.check(L.dg_dev_flush_l2())
        backend.check(L.dg_dev_lde(polys.ptr, ext.ptr, log_n, 5, cols, ctypes.byref(ms)))   # CUDA events on the library's stream
        if i >= 1:
            lde_ms.append(ms.value)
    n_pass = 1 if log_n <= 10 else 2 if log_n <= 20 else 3      # ntt_pass_kernel launches per LDE call
    alg_bytes = cols * (16.0 * n + 16.0 * n * 32)          # SURVEY.md 8d: LDE of one column = 16 n + 16 N bytes
    lde = float(np.median(lde_ms))
    achieved = alg_bytes / (lde * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:                                        # DRAM bytes per launch from the committed ncu --set full capture of the same launch shape
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_roofline_traffic.json")))
        if log_n == 20 and cols == tj.get("columns_per_launch"):
            traffic, traffic_src = tj["per_launch_bytes"], "profiles/r02_roofline_traffic.json (ncu dram__bytes_read+write, mean of the two pass launches)"
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "ntt_pass_kernel (coset LDE x32 of %d trace columns = %d launches)" % (cols, n_pass), "achieved": achieved,
                "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_kind": peak_kind,
                "algorithmic_bytes_per_launch": alg_bytes / n_pass, "launch_ms": lde / n_pass,
                "note": "the kernel is integer-ALU bound, not HBM bound: ncu shows the ALU pipe 59-63% busy with math_pipe_throttle the top stall at 13-16% DRAM "
                        "throughput (profiles/r02_ncu_ntt_pass_kernel.txt); a 2-pass NTT writes and re-reads the 2^25-point intermediate (floor 3x the algorithmic bytes)"}
    # the bound that actually applies: 128-bit modular arithmetic.  One LDE column = 32 coset NTTs of n points = 32 * (n/2) * log2(n)
    # butterflies (1 modmul + 1 add + 1 sub) + 2 extra modmuls per point (coset factor, inter-pass twiddle), counted as 0.6 butterflies
    bfly = cols * 32.0 * ((n / 2) * log_n + 0.6 * 2 * n)
    peak_bfly = 224.6e9                         # tools/bench_modmul.cu, fe_mul v4 butterfly mix on B200 (profiles/r01_modmul_microbench.txt)
    roofline["compute"] = {"bound": "integer ALU pipe (128-bit modular butterflies)", "unit": "G butterflies/s", "achieved": bfly / (lde * 1e-3) / 1e9,
                           "peak": peak_bfly / 1e9, "frac": bfly / (lde * 1e-3) / peak_bfly,
                           "peak_source": "profiles/r01_modmul_microbench.txt (arithmetic in isolation, same GPU model)"}

    # ---- CPU baseline: the oracle (restated reference prover) on a bounded sample of the same workload (a shorter collatz trace), all host
    #      threads; the sample size is calibrated so that it costs ~10-30 s.  The same-size CPU number is the --impl reference arm.
    cpu = {"value": None, "unit": "ms", "cores": 1, "kind": "port", "sample": "skipped (--no-cpu-baseline)"}
    if not args.no_cpu_baseline and world == 1:
        threads = po.set_threads(oracle_threads())
        tr14, _ = build_workload(args, 14)
        t2 = time.perf_counter()
        r14 = po.prove(tr14.registers, tr14.ctx_depth, tr14.loop_depth, tr14.public_inputs, tr14.outputs)
        t14 = time.perf_counter() - t2
        assert r14.error is None
        log_s = args.ref_log_n or int(np.clip(14 + np.floor(np.log2(max(1.0, 20.0 / max(t14, 1e-3)))), 14, min(18, log_n)))
        trs, sname = build_workload(args, log_s)
        t2 = time.perf_counter()
        r = po.prove(trs.registers, trs.ctx_depth, trs.loop_depth, trs.public_inputs, trs.outputs)
        cpu_ms = (time.perf_counter() - t2) * 1e3
        assert r.error is None
        small = dg.prove(trs, opts)
        assert small.bytes == r.proof, "GPU proof differs from the CPU oracle's on the baseline sample"
        gpu_small_ms = small.stats["total_ms"]
        cpu = {"value": cpu_ms, "unit": "ms", "cores": threads, "kind": "port", "host_cores_available": os.cpu_count(),
               "sample_log_n": log_s, "gpu_ms_same_sample": gpu_small_ms, "stage_ms": [float(x) for x in r.stage_ms],
               "sample": f"{sname}: 2^{log_s}-step trace x {trs.width} registers proven by the C++ restatement on {threads} host threads in {cpu_ms:.0f} ms "
                         f"(not scaled; the GPU proof of the same trace is byte-identical and took {gpu_small_ms:.2f} ms on the device); "
                         f"the full 2^{log_n}-step CPU run is `bench.py --impl reference`"}
        po.set_threads(1)

    line = {
        "metric": metric_name(log_n), "value": value, "unit": "ms", "n_gpus": args.gpus if single_process else world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
        "dtype": "u128 (128-bit prime field) + u32 (blake3)", "data": "synthetic",
        "config": {"workload": workload_name(name, log_n, w),
                   "parallelism": ("coset-sharded x%d, one process per GPU (NCCL all-gather / all-to-all at commitment points)" % world) if world > 1 else
                                  ("coset-sharded x%d inside ONE process (dg_init_devices: host thread + NCCL communicator per device)" % args.gpus) if single_process else "single", "l2": "inputs exceed L2 (trace %d MB, extended trace %d MB)" % (regs.nbytes >> 20, (regs.nbytes * 32) >> 20),
                   "proof_bytes": len(proof.bytes), "device": info["name"]},
        "stage_ms": [float(x) / args.steps for x in stage_ms],
        "stage_names": STAGE_NAMES,
        "wall_ms_per_step": wall_ms / args.steps, "ms_steps": [round(float(x), 2) for x in dev_ms], "e2e_ms_steps": [round(float(x), 2) for x in e2e_ms],
        "e2e": {"value": e2e_value, "unit": "ms", "h2d_bytes_per_step": int(regs.nbytes), "d2h_bytes_per_step": len(proof.bytes),
                "api": "distaff_b200.prove(trace, options) -> dg_prove (pinned host trace in, proof bytes out)",
                "pageable_ms": e2e_pageable, "pageable_note": "same call from ordinary pageable memory (a Rust Vec<u128>), best of 2"},
        "proof_sha256": proof_sha, "proof_check": check,
        "gpu_launches": int(launches),
        "roofline": roofline, "cpu_baseline": cpu, "clocks": sampler.summary(),
    }
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()



# -------------------------------------------------------------------------------------------------------------------------
def run_microbench(args):
    """BASELINE.json config 5: NTT / LDE / leaf-hash / Merkle sweeps on device-resident data (benches/fft.rs:6, benches/hash.rs:16-27 shapes).
    Every rank runs the same sweep on its own GPU (independent vectors: the building blocks shard without any collective, "weak"
    scaling); times are CUDA events on the library's stream, L2 flushed between iterations, max over ranks; aggregate GB/s = N x bytes /
    max time.  Algorithmic bytes are SURVEY.md 8d's: NTT 32 n; LDE column 16 n + 16 N; leaf hash 16 w N + 32 N; tree 64 L.
    Rank 0 also times the CPU oracle (all host threads) on the same shapes up to 2^20 elements."""
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    os.environ["DG_DEVICE"] = str(local_rank)
    import torch
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from distaff_b200 import backend, felt
    L = backend.lib()
    info = backend.device_info()
    peak, peak_kind = peak_gbs()
    quick = args.quick
    iters = 3 if quick else 5

    def timed(fn):
        ms = ctypes.c_float(0)
        got = []
        for i in range(iters + 2):
            backend.check(L.dg_dev_flush_l2())
            if dist is not None:
                dist.barrier()
            fn(ctypes.byref(ms))
            if i >= 2:
                got.append(ms.value)
        med = float(np.median(got))
        if dist is not None:
            t = torch.tensor([med], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            med = float(t.item())
        return med

    po = None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import pyoracle as po
        threads = po.set_threads(oracle_threads())

    def cpu_time(fn):
        t0 = time.perf_counter()
        fn()
        return (time.perf_counter() - t0) * 1e3

    rows = []

    def emit(kind, shape, ms, alg_bytes, cpu_ms=None, extra=None):
        gbs = world * alg_bytes / (ms * 1e-3) / 1e9
        r = {"kernel": kind, "shape": shape, "ms": ms, "alg_gbs_aggregate": gbs, "alg_gbs_per_gpu": gbs / world, "frac_of_hbm_peak_per_gpu": gbs / world / peak,
             "cpu_ms": cpu_ms, "speedup_vs_cpu": (world * cpu_ms / ms) if cpu_ms else None}
        if extra:
            r.update(extra)
        rows.append(r)
        if rank == 0 and args.verbose:
            print("  %-10s %-28s %9.3f ms  %8.1f GB/s/GPU (%.1f%%)  cpu %s" % (kind, shape, ms, gbs / world, 100 * gbs / world / peak,
                                                                              "%.0f ms" % cpu_ms if cpu_ms else "-"), file=sys.stderr, flush=True)

    ntt_logs = (14, 18, 22) if quick else range(14, 25, 2)
    for log_n in ntt_logs:
        n = 1 << log_n
        vals = felt.random_elements(n, log_n)
        buf = backend.DeviceBuffer(n * 16).upload(vals)
        ms = timed(lambda m: backend.check(L.dg_dev_ntt(buf.ptr, log_n, 1, 0, m)))
        cpu = cpu_time(lambda: po.fft(vals)) if (po is not None and log_n <= 20) else None
        emit("ntt", "2^%d elements" % log_n, ms, 32.0 * n, cpu)
        buf.free()
    lde_logs = (14, 18) if quick else (12, 14, 16, 18, 20)
    for log_n in lde_logs:
        w, n = 16, 1 << log_n
        cols = felt.random_elements(w * n, 7)
        polys = backend.DeviceBuffer(w * n * 16).upload(cols)
        ext = backend.DeviceBuffer(w * n * 32 * 16)
        ms = timed(lambda m: backend.check(L.dg_dev_lde(polys.ptr, ext.ptr, log_n, 5, w, m)))
        cpu = None
        if po is not None and log_n <= 16:
            one = np.zeros((n * 32, 2), dtype=np.uint64)
            one[:n] = cols[:n]
            cpu = w * cpu_time(lambda: po.fft(one))           # one zero-padded column transform (trace_table.rs:165) x w columns
        emit("lde x32", "%d columns x 2^%d" % (w, log_n), ms, w * (16.0 * n + 16.0 * n * 32), cpu)
        leaves = backend.DeviceBuffer(n * 32 * 32)
        ms = timed(lambda m: backend.check(L.dg_dev_hash_rows(ext.ptr, w, log_n, 5, leaves.ptr, m)))
        emit("leaf hash", "2^%d rows x %d columns" % (log_n + 5, w), ms, 16.0 * w * n * 32 + 32.0 * n * 32)
        nodes = backend.DeviceBuffer(n * 32 * 32)
        ms = timed(lambda m: backend.check(L.dg_dev_merkle_build(leaves.ptr, n * 32, nodes.ptr, m)))
        cpu = None
        if po is not None and log_n + 5 <= 21:
            lv = np.frombuffer(np.random.Generator(np.random.PCG64(log_n)).bytes(n * 32 * 32), dtype=np.uint8)
            cpu = cpu_time(lambda: po.merkle_nodes("blake3", lv.tobytes()))
        emit("merkle", "2^%d leaves (blake3)" % (log_n + 5), ms, 64.0 * n * 32, cpu)
        for x in (polys, ext, leaves, nodes):
            x.free()
    if not quick:
        for name, hid in (("rescue", 1), ("poseidon", 2)):
            for log_l in (14, 18):
                L_ = 1 << log_l
                leaves = backend.DeviceBuffer(L_ * 32).upload(felt.random_elements(2 * L_, 7 + log_l))
                nodes = backend.DeviceBuffer(L_ * 32)
                ms = timed(lambda m: backend.check(L.dg_dev_merkle_build_with(hid, leaves.ptr, L_, nodes.ptr, m)))
                emit("merkle", "2^%d leaves (%s)" % (log_l, name), ms, 64.0 * L_, None, {"hashes_per_s_aggregate": world * (L_ - 1) / (ms * 1e-3)})
                leaves.free()
                nodes.free()
    out = {"microbench": rows, "n_gpus": world, "scaling": "weak", "device": info["name"], "hbm_peak_gbs": peak, "peak_kind": peak_kind,
           "cpu": {"kind": "port", "cores": oracle_threads() if po is not None else None}, "timing": "CUDA events, L2 flushed, median of %d, max over ranks" % iters}
    if po is not None:
        po.set_threads(1)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return out if rank == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log-n", type=int, default=20, help="log2 of the trace length (default: the 2^20-step headline workload)")
    ap.add_argument("--workload", default="collatz", choices=["collatz", "fibonacci", "merkle"],
                    help="collatz = the headline 2^20-step workload (default); fibonacci --log-n 16 and merkle --log-n 14 are BASELINE configs 2 and 3")
    ap.add_argument("--ref-log-n", type=int, default=0, help="log2 trace length of the CPU sample (default: chosen to fit the time budget)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--single-process", action="store_true", help="with --gpus N (no torchrun): shard the proof over N GPUs from this one process")
    ap.add_argument("--microbench", action="store_true", help="BASELINE config 5: NTT / LDE / leaf hash / Merkle sweep instead of the proof benchmark")
    ap.add_argument("--quick", action="store_true", help="--microbench: three sizes only")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the proof of the last timed step to DIR/<name>.npy (float32, one element per byte)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.microbench or args.impl != "ours"):
        ap.error("--dump-outputs applies to the CUDA prover benchmark only")
    if args.microbench:
        out = run_microbench(args)
        if out is not None:
            print(json.dumps(out), flush=True)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
