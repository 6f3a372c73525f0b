"""bench.py --dump-outputs and --steps: the arrays written after the timed steps are the proof of the last one (equal to the CPU
oracle's proof of the same trace), and --steps is the number of timed proofs."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    return subprocess.run([sys.executable, "bench.py", *args], cwd=ROOT, capture_output=True, text=True, timeout=600,
                          env=dict(os.environ, BENCH_NO_SMI="1"))


def test_bench_rejects_zero_steps_and_dumps_outside_the_prover_arm(tmp_path):
    r = _bench("--steps", "0")
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr
    r = _bench("--impl", "reference", "--dump-outputs", str(tmp_path))
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
    assert not os.listdir(tmp_path)


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_proof(tmp_path, po):
    import bench
    out = tmp_path / "dump"
    r = _bench("--log-n", "12", "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(out))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 3 and len(d["ms_steps"]) == 3 and len(d["e2e_ms_steps"]) == 3
    got = {p.stem: np.load(p) for p in out.glob("*.npy")}
    assert set(got) == {"proof", "trace_root", "constraint_root", "pow_seed", "pow_nonce"}
    assert all(a.dtype == np.float32 and a.ndim == 1 for a in got.values())
    raw = {k: a.astype(np.uint8).tobytes() for k, a in got.items()}
    assert hashlib.sha256(raw["proof"]).hexdigest() == d["proof_sha256"]
    tr, _ = bench.build_trace(12)
    ref = po.prove(tr.registers, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs)
    assert ref.error is None
    assert raw["proof"] == ref.proof
    assert raw["trace_root"] == ref.digest("trace_root") and raw["constraint_root"] == ref.digest("constraint_root")
    assert int.from_bytes(raw["pow_nonce"], "little") == ref.u64s("pow_nonce")[0]
    assert len(raw["pow_seed"]) == 32
