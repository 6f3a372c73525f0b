"""CPU tests of SHA3-256 as a proof hash: the sha3 oracle's SHA3-256 (tests/sha3_oracle.py) and the library's host SHA3-256 (dg_host_sha3, the FRI-roots seed of a
sha3 proof) against hashlib, oracle prove -> verify round trips with ProofOptions(hash_fn = sha3), the hash byte of the encoding, the
argument checks of distaff_b200.ProofOptions, and the committed sha3 proof fixture."""
import ctypes
import hashlib
import json
import os
import random

import pytest

from tests import programs, sha3_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LENGTHS = list(range(0, 301)) + [400, 416, 2048]          # 0..300 covers the rate boundaries 135/136/137 and 271/272/273


def _messages():
    rng = random.Random(2026)
    return [bytes(rng.randrange(256) for _ in range(n)) for n in LENGTHS]


def test_oracle_sha3_matches_hashlib():
    for m in _messages():
        assert so.hash(m) == hashlib.sha3_256(m).digest(), len(m)


def test_host_sha3_matches_hashlib():
    from distaff_b200 import backend
    if not os.path.exists(backend.LIB_PATH):
        pytest.skip("libdistaff_gpu.so not built (run __graft_entry__.build())")
    L = ctypes.CDLL(backend.LIB_PATH)
    out = ctypes.create_string_buffer(32)
    for m in _messages():
        assert L.dg_host_sha3(m, len(m), out) == 0
        assert out.raw == hashlib.sha3_256(m).digest(), len(m)


@pytest.fixture(scope="module")
def sha3_proofs():
    return {name: (tr, so.prove(tr.registers, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs))
            for name, tr in programs.small_programs().items()}


def test_oracle_sha3_round_trip(sha3_proofs):
    for name, (tr, proof) in sha3_proofs.items():
        assert proof[-1] == 4, name                                  # options.hash_fn is the last byte of the encoding
        assert so.verify(tr.program_hash, tr.public_inputs, tr.outputs, proof) is None, name


def test_relabelled_hash_byte_is_rejected(po, sha3_proofs):
    tr, proof = sha3_proofs["fib13"]
    assert so.verify(tr.program_hash, tr.public_inputs, tr.outputs, proof[:-1] + b"\x00") is not None
    b3 = po.prove(tr.registers, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs).proof
    assert b3[-1] == 0 and b3 != proof
    assert so.verify(tr.program_hash, tr.public_inputs, tr.outputs, b3) is None          # the blake3 proof itself verifies
    assert so.verify(tr.program_hash, tr.public_inputs, tr.outputs, b3[:-1] + b"\x04") is not None
    for other in (1, 2, 3, 5, 255):
        assert so.verify(tr.program_hash, tr.public_inputs, tr.outputs, proof[:-1] + bytes([other])) == "unsupported hash function"


def test_sha3_golden_fixture(sha3_proofs):
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "oracle_sha3_proofs.json")))
    assert set(golden) == set(sha3_proofs)
    for name, (tr, proof) in sha3_proofs.items():
        assert hashlib.sha256(tr.registers.tobytes()).hexdigest() == golden[name]["trace_sha256"], name
        assert hashlib.sha256(proof).hexdigest() == golden[name]["proof_sha256"], name


def test_proof_options_hash_argument():
    from distaff_b200 import ProofOptions
    assert ProofOptions().hash_fn == "blake3" and ProofOptions()._c().hash_id == 0
    assert ProofOptions(hash_fn="sha3")._c().hash_id == 4
    o = ProofOptions(64, 20, 8, "sha3")                              # positional, in the reference's field order
    assert (o.extension_factor, o.num_queries, o.grinding_factor, o.hash_fn) == (64, 20, 8, "sha3")
    assert ProofOptions(16, 30, 8)._c().hash_id == 0
    for name in ("rescue", "poseidon", "gmimc"):
        with pytest.raises(ValueError, match="at most 64 bytes"):
            ProofOptions(hash_fn=name)
    for name in ("sha256", "", None, 4):
        with pytest.raises(ValueError):
            ProofOptions(hash_fn=name)
