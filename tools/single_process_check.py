#!/usr/bin/env python3
"""Single-process multi-GPU check: ONE process, dg_init_devices(n), one dg_prove call per proof (the seam of lib.rs:62) -- the proofs must be
byte-identical to the CPU oracle's.   python tools/single_process_check.py [n_devices] [log_n of the large trace] [--hash sha3]
--hash picks the commitment hash of every proof (default blake3)."""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np                                # noqa: E402
import bench                                      # noqa: E402
import distaff_b200 as dg                         # noqa: E402
from distaff_b200 import backend, hostvm          # noqa: E402
from oracle import pyoracle as po                 # noqa: E402
from tests import programs, sha3_oracle as so     # noqa: E402

args = sys.argv[1:]
HASH = "blake3"
if "--hash" in args:
    i = args.index("--hash")
    HASH = args[i + 1]
    del args[i:i + 2]
n_dev = int(args[0]) if len(args) > 0 else 2
log_n = int(args[1]) if len(args) > 1 else 16
opts = dg.ProofOptions(hash_fn=HASH)


def oracle_proof(tr):
    if HASH == "sha3":
        return so.prove(tr.registers, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs)
    return po.prove(tr.registers, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs).proof



backend.check(backend.lib().dg_init_devices(n_dev))
po.set_threads(min(32, os.cpu_count() or 1))
so.set_threads(min(32, os.cpu_count() or 1))
ok = True
cases = list(programs.small_programs().items()) + [("fib250", hostvm.fibonacci(250)), ("collatz7", hostvm.collatz(7))]
for name, tr in cases:
    p = dg.prove(tr, opts)
    same = p.bytes == oracle_proof(tr) and dg.verify(tr.program_hash, tr.public_inputs, tr.outputs, p.bytes) is None
    ok &= same
    print(f"[{n_dev} devices, 1 process] {name}: identical={same} ms={p.stats['total_ms']:.2f}", flush=True)
tr, name = bench.build_trace(log_n)
ref = oracle_proof(tr)
buf = backend.DeviceBuffer(tr.registers.nbytes).upload(tr.registers)
for i in range(3):
    t0 = time.perf_counter()
    p = dg.prove(tr, opts)
    wall = (time.perf_counter() - t0) * 1e3
    pd = dg.prove_device(buf, tr.width, tr.length, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs, opts)
same = p.bytes == ref and pd.bytes == ref
ok &= same
print(f"[{n_dev} devices, 1 process] {name} 2^{log_n}: identical={same} device_ms={pd.stats['total_ms']:.2f} host_call_ms={wall:.2f}", flush=True)
bad = hostvm.ExecutionTrace(tr.registers.copy(), tr.ctx_depth, tr.loop_depth, tr.stack_depth, tr.program_hash, tr.public_inputs, tr.outputs)
bad.registers[tr.width - 1, 100, 0] += 1
try:
    dg.prove(bad, opts)
    ok = False
except backend.DgError as e:
    ok &= e.code == -5
print("SINGLE_PROCESS_CHECK", "PASS" if ok else "FAIL", "devices", n_dev, flush=True)
sys.exit(0 if ok else 1)
