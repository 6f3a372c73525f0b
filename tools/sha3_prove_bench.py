#!/usr/bin/env python3
"""Cost of SHA3-256 commitments: proves the bench.py workload (2^20 steps by default) with hash_fn = blake3 and = sha3, alternating the
two over several repetitions in one process, and records the per-stage device times of every proof (proof.stats, CUDA events), plus
the SHA3-256 / BLAKE3 rate of 64-byte hashing as Merkle trees over 2^23 leaves (256 MB of leaves, twice the L2; the L2 is overwritten
before every timed tree).  The card's name and power limit are read in the same run.
    python tools/sha3_prove_bench.py [--log-n 20] [--reps 3] [--out profiles/r03_sha3_prove.json]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
STAGES = ["1 extend trace", "2 trace tree", "3 constraints", "4 constraint poly", "5 constraint tree", "6 composition", "7 FRI layers",
          "8 query positions + PoW", "9 proof object"]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                       text=True, check=True).stdout.strip().split(", ")
    return {"name": q[0], "power_limit": q[1], "max_sm_clock": q[2]}


def merkle_rate(backend, hash_id, log_leaves, reps):
    """64-byte hashes per second of dg_dev_merkle_build_with (L - 1 hashes per tree), device-event time, L2 overwritten before each tree"""
    L = backend.lib()
    n = 1 << log_leaves
    leaves = backend.DeviceBuffer(n * 32).upload(np.random.default_rng(1).integers(0, 2**63, size=n * 4, dtype=np.int64))
    nodes = backend.DeviceBuffer(n * 32)
    ms = ctypes.c_float(0)
    backend.check(L.dg_dev_merkle_build_with(hash_id, leaves.ptr, n, nodes.ptr, ctypes.byref(ms)))      # warm-up
    times = []
    for _ in range(reps):
        backend.check(L.dg_dev_flush_l2())
        backend.check(L.dg_dev_merkle_build_with(hash_id, leaves.ptr, n, nodes.ptr, ctypes.byref(ms)))
        times.append(ms.value)
    leaves.free()
    nodes.free()
    best = min(times)
    return {"leaves": n, "hashes": n - 1, "tree_ms": times, "ghash_per_s_best": (n - 1) / best / 1e6}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log-n", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_sha3_prove.json"))
    a = ap.parse_args()
    import bench
    import distaff_b200 as dg
    from distaff_b200 import backend
    res = {"card": card(), "device": backend.device_info(), "log_n": a.log_n, "reps": a.reps}
    tr, name = bench.build_trace(a.log_n)
    res["workload"] = f"{name}: 2^{a.log_n} steps x {tr.width} registers, blowup 32, 50 queries, 20-bit grinding"
    runs = {"blake3": [], "sha3": []}
    first = {}
    for h in ("blake3", "sha3"):                                       # warm-up: tables, arena sizing
        first[h] = dg.prove(tr, dg.ProofOptions(hash_fn=h)).bytes
    for _ in range(a.reps):
        for h in ("blake3", "sha3"):
            p = dg.prove(tr, dg.ProofOptions(hash_fn=h))
            assert p.bytes == first[h], "proof changed between repetitions"
            runs[h].append({"total_ms": p.stats["total_ms"], "stage_ms": p.stats["stage_ms"], "kernel_launches": p.stats["kernel_launches"]})
    for h, rs in runs.items():
        res[h] = {"runs": rs, "proof_len": len(first[h]), "hash_byte": first[h][-1],
                  "total_ms_median": float(np.median([r["total_ms"] for r in rs])),
                  "stage_ms_median": dict(zip(STAGES, [float(x) for x in np.median([r["stage_ms"] for r in rs], axis=0)]))}
    res["sha3_over_blake3_total"] = res["sha3"]["total_ms_median"] / res["blake3"]["total_ms_median"]
    res["hash64_merkle"] = {"sha3": merkle_rate(backend, 4, 23, 5), "blake3": merkle_rate(backend, 0, 23, 5)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)
    print(json.dumps({k: res[k] for k in ("card", "sha3_over_blake3_total")}))
    for h in ("blake3", "sha3"):
        print(h, "total %.2f ms" % res[h]["total_ms_median"], {k: round(v, 3) for k, v in res[h]["stage_ms_median"].items()})
    for h, r in res["hash64_merkle"].items():
        print(h, "64-byte hashes: %.2f G/s (tree of 2^23 leaves, best %.3f ms)" % (r["ghash_per_s_best"], min(r["tree_ms"])))


if __name__ == "__main__":
    main()
