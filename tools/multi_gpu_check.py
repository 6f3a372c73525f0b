#!/usr/bin/env python3
"""Multi-GPU parity check (run under torchrun): one proof sharded over WORLD_SIZE GPUs must be byte-identical to the CPU oracle's.
    torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/multi_gpu_check.py [--hash sha3]
--hash picks the commitment hash of every proof (default blake3)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HASH = sys.argv[sys.argv.index("--hash") + 1] if "--hash" in sys.argv else "blake3"
rank, local_rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
os.environ["DG_DEVICE"] = str(local_rank)
import torch                       # noqa: E402
import torch.distributed as dist   # noqa: E402
import distaff_b200 as dg          # noqa: E402
from distaff_b200 import backend, hostvm   # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from tests import programs, sha3_oracle as so   # noqa: E402

torch.cuda.set_device(local_rank)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    backend.comm_init_from_torch(dist, local_rank)
ok = True
cases = list(programs.small_programs().items()) + [("fib250", hostvm.fibonacci(250)), ("collatz7", hostvm.collatz(7)), ("merkle20", programs.merkle_example(20, po))]
for name, tr in cases:
    for opts in ((32, 50, 20),) + (((64, 20, 8), (128, 10, 4)) if name in ("collatz3", "fib13") else ()):
        if opts[0] // world < 4:
            continue
        p = dg.prove(tr, dg.ProofOptions(*opts, hash_fn=HASH))
        if HASH == "sha3":
            ref = so.prove(tr.registers, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs, ext=opts[0], num_queries=opts[1], grinding=opts[2])
        else:
            ref = po.prove(tr.registers, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs, ext=opts[0], num_queries=opts[1],
                           grinding=opts[2]).proof
        same = p.bytes == ref
        ok &= same
        if rank == 0:
            print(f"[world {world}] {name} {opts}: identical={same} len={len(p.bytes)} ms={p.stats['total_ms']:.2f}", flush=True)
# an invalid trace must be rejected on every rank (the violation flag is max-reduced)
tr = programs.small_programs()["fib13"]
regs = tr.registers.copy()
regs[tr.width - 1, 100, 0] += 1
bad = hostvm.ExecutionTrace(regs, tr.ctx_depth, tr.loop_depth, tr.stack_depth, tr.program_hash, tr.public_inputs, tr.outputs)
try:
    dg.prove(bad, dg.ProofOptions(hash_fn=HASH))
    ok = False
    print(rank, "invalid trace was proven!?")
except backend.DgError as e:
    ok &= e.code == -5
t = torch.tensor([1 if ok else 0], device="cuda")
if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    backend.check(backend.lib().dg_comm_finalize())
    dist.destroy_process_group()
if rank == 0:
    print("MULTI_GPU_CHECK", "PASS" if int(t.item()) == 1 else "FAIL", "world", world, flush=True)
sys.exit(0 if int(t.item()) == 1 else 1)
