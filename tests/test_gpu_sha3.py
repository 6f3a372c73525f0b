"""-m gpu tests of SHA3-256 as the proof hash (ProofOptions(hash_fn="sha3")): the 64-byte hash and Merkle kernels against hashlib and the
oracle, proofs byte-identical to the CPU oracle's over programs, options, a multi-block row width and a 2^16-step trace, the GPU
verifier's verdicts against the oracle's, the refusal of hash ids that cannot hash a trace row, and both multi-GPU modes."""
import hashlib
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from tests import programs, sha3_oracle as so

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LDP = "verification of low-degree proof failed: evaluations did not match column value at depth 0"


@pytest.fixture(scope="module")
def dg():
    import distaff_b200
    from distaff_b200 import backend
    backend.device_info()
    return distaff_b200


def _oracle(po, tr, ext=32, num_queries=50, grinding=20):
    return so.prove(tr.registers, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs, ext=ext, num_queries=num_queries, grinding=grinding)


@pytest.fixture(scope="module")
def proofs(dg):
    return {name: (tr, dg.prove(tr, dg.ProofOptions(hash_fn="sha3")).bytes) for name, tr in programs.small_programs().items()}


def test_hash64_matches_hashlib(dg):
    rng = np.random.default_rng(3)
    msgs = rng.integers(0, 256, size=(1 << 16) * 64, dtype=np.uint8).tobytes()
    got = dg.hash64(msgs, "sha3")
    for i in list(range(0, 1 << 16, 97)) + [(1 << 16) - 1]:
        assert got[32 * i:32 * i + 32] == hashlib.sha3_256(msgs[64 * i:64 * i + 64]).digest(), i


def test_merkle_build_matches_oracle(dg, po):
    leaves = np.random.default_rng(4).integers(0, 256, size=(1 << 12) * 32, dtype=np.uint8).tobytes()
    assert dg.merkle_build(leaves, "sha3") == so.merkle_nodes(leaves)


def test_small_programs_match_the_oracle(po, proofs):
    for name, (tr, proof) in proofs.items():
        assert proof == _oracle(po, tr), name
        assert proof[-1] == 4


@pytest.mark.parametrize("prog,ext,queries,grinding", [("collatz3", 16, 30, 8), ("fib13", 64, 20, 12), ("collatz3", 256, 5, 4),
                                                      ("hash", 128, 128, 1), ("deep_stack", 32, 50, 0)])
def test_other_options_match_the_oracle(dg, po, prog, ext, queries, grinding):
    tr = programs.small_programs()[prog]
    assert dg.prove(tr, dg.ProofOptions(ext, queries, grinding, "sha3")).bytes == _oracle(po, tr, ext, queries, grinding)


def test_multi_block_rows_match_the_oracle(dg, po):
    tr = programs.wide_program()                    # 65 registers: 1040-byte rows = 130 lanes = 8 permutations per row
    assert tr.width == 65
    assert dg.prove(tr, dg.ProofOptions(hash_fn="sha3")).bytes == _oracle(po, tr)


def test_2_16_trace_matches_the_oracle(dg, po):
    import bench
    tr, _ = bench.build_trace(16)
    so.set_threads(min(32, os.cpu_count() or 1))
    proof = dg.prove(tr, dg.ProofOptions(hash_fn="sha3")).bytes
    assert proof == _oracle(po, tr)
    assert dg.verify(tr.program_hash, tr.public_inputs, tr.outputs, proof) is None


def test_verifier_agrees_with_the_oracle(dg, po, proofs):
    for name, (tr, proof) in proofs.items():
        assert so.verify(tr.program_hash, tr.public_inputs, tr.outputs, proof) is None, name
        assert dg.verify(tr.program_hash, tr.public_inputs, tr.outputs, proof) is None, name
    tr, proof = proofs["fib_span"]                  # src/tests/mod.rs:32-63: wrong inputs, wrong outputs, wrong program hash
    bad_hash = bytes([1]) + tr.program_hash[1:]
    for args in ((tr.program_hash, [1, 1], tr.outputs), (tr.program_hash, tr.public_inputs, [5]), (bad_hash, tr.public_inputs, tr.outputs)):
        assert so.verify(*args, proof) == LDP
        assert dg.verify(*args, proof) == LDP
    for name in ("fib13", "deep_stack"):            # the hash byte relabelled: blake3 <-> sha3, and ids without a proof hash
        tr, proof = proofs[name]
        for byte in (0, 1, 3, 5):
            bad = proof[:-1] + bytes([byte])
            assert dg.verify(tr.program_hash, tr.public_inputs, tr.outputs, bad) == so.verify(tr.program_hash, tr.public_inputs, tr.outputs, bad)
            assert dg.verify(tr.program_hash, tr.public_inputs, tr.outputs, bad) is not None
        b3 = dg.prove(tr).bytes
        assert dg.verify(tr.program_hash, tr.public_inputs, tr.outputs, b3[:-1] + b"\x04") == \
            so.verify(tr.program_hash, tr.public_inputs, tr.outputs, b3[:-1] + b"\x04") != None  # noqa: E711


def test_corrupted_bytes_get_the_same_verdict(dg, po, proofs):
    from distaff_b200 import backend
    rng = random.Random(11)
    checked = rejected = 0
    for name in ("fib13", "collatz3", "hash", "deep_stack"):
        tr, proof = proofs[name]
        offsets = [0, 31, 36, 40] + [rng.randrange(44, len(proof) - 16) for _ in range(30)] + [len(proof) - 12, len(proof) - 5]
        for off in offsets:
            bad = bytearray(proof)
            bad[off] ^= 1 << rng.randrange(8)
            bad = bytes(bad)
            want = so.verify(tr.program_hash, tr.public_inputs, tr.outputs, bad)
            try:
                got = dg.verify(tr.program_hash, tr.public_inputs, tr.outputs, bad)
            except backend.DgError:
                got = "malformed"
            if want is not None and (want.startswith("exception") or "too short" in want):
                assert got is not None, (name, off)
            else:
                assert got == want, (name, off, got, want)
            checked += 1
            rejected += want is not None
    assert checked > 120 and rejected > 80


def test_hashes_that_cannot_hash_a_row_are_refused(dg):
    from distaff_b200 import backend
    tr = programs.small_programs()["fib13"]
    for hid in (1, 2, 3, 5, 255):
        opt = dg.ProofOptions()
        c = opt._c
        opt._c = lambda c=c, hid=hid: backend.DgOptions(c().extension_factor, c().num_queries, c().grinding_factor, hid)
        with pytest.raises(backend.DgError) as e:
            dg.prove(tr, opt)
        assert e.value.code == -1
        if hid <= 3:
            assert "at most 64 bytes" in str(e.value)


def test_device_entry_point(dg, po):
    from distaff_b200 import backend
    tr = programs.small_programs()["collatz3"]
    buf = backend.DeviceBuffer(tr.registers.nbytes).upload(tr.registers)
    p = dg.prove_device(buf, tr.width, tr.length, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs, dg.ProofOptions(hash_fn="sha3"))
    assert p.bytes == _oracle(po, tr)


def _two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")


def test_two_ranks_sha3():
    _two_gpus()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29519", os.path.join(ROOT, "tools", "multi_gpu_check.py"), "--hash", "sha3"]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "MULTI_GPU_CHECK PASS world 2" in out.stdout


def test_single_process_two_devices_sha3():
    _two_gpus()
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "single_process_check.py"), "2", "14", "--hash", "sha3"], cwd=ROOT,
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "SINGLE_PROCESS_CHECK PASS devices 2" in out.stdout
