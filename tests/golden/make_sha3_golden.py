#!/usr/bin/env python3
"""Regenerates tests/golden/oracle_sha3_proofs.json: for every program of tests.programs.small_programs(), the SHA-256 of the
execution trace and of the CPU oracle's proof with ProofOptions(hash_fn = sha3) (tests/sha3_oracle.py) (default options otherwise).  The fixture freezes
the oracle's sha3 proofs so that oracle regressions are caught and the -m gpu tests compare against committed values as well as
against the live oracle.   Run:  python tests/golden/make_sha3_golden.py
"""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import programs, sha3_oracle as so   # noqa: E402

out = {}
for name, tr in programs.small_programs().items():
    proof = so.prove(tr.registers, tr.ctx_depth, tr.loop_depth, tr.public_inputs, tr.outputs)
    assert proof[-1] == 4
    assert so.verify(tr.program_hash, tr.public_inputs, tr.outputs, proof) is None
    out[name] = {"trace_sha256": hashlib.sha256(tr.registers.tobytes()).hexdigest(), "proof_sha256": hashlib.sha256(proof).hexdigest()}
path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_sha3_proofs.json")
json.dump(out, open(path, "w"), indent=1, sort_keys=True)
print("wrote", path, len(out), "programs")
