"""Host-side mirror of the reference's public interface for the prove path (names and argument meaning follow
/root/reference/src/lib.rs:30-75, /root/reference/src/stark/options.rs:16-91, /root/reference/src/stark/proof.rs:10-77)."""
import ctypes

import numpy as np

from . import backend, felt, hostvm


# hashes a proof can commit with (dg_options_t.hash_id); the others cannot hash a trace row (include/distaff_gpu.h)
PROOF_HASHES = {"blake3": 0, "sha3": 4}


class ProofOptions:
    """stark::ProofOptions (options.rs:29-50): same argument checks, same defaults (options.rs:82-91).  hash_fn is "blake3" (the
    default) or "sha3" (SHA3-256, hash.rs:212-218)."""

    def __init__(self, extension_factor=32, num_queries=50, grinding_factor=20, hash_fn="blake3"):
        if hash_fn not in PROOF_HASHES:
            if hash_fn in ("rescue", "poseidon", "gmimc"):
                raise ValueError(f"hash_fn {hash_fn!r} cannot commit to a proof: it absorbs at most 64 bytes and a trace row is longer "
                                 "(the reference panics in build_merkle_tree); use 'blake3' or 'sha3'")
            raise ValueError(f"unknown hash_fn {hash_fn!r}: use 'blake3' or 'sha3'")
        assert extension_factor & (extension_factor - 1) == 0, "extension_factor must be a power of 2"
        assert extension_factor >= 16, "extension_factor cannot be smaller than 16"
        assert extension_factor <= 256, "extension_factor cannot be greater than 256"
        assert num_queries > 0, "num_queries must be greater than 0"
        assert num_queries <= 128, "num_queries cannot be greater than 128"
        assert grinding_factor <= 32, "grinding factor cannot be greater than 32"
        self.extension_factor = extension_factor
        self.num_queries = num_queries
        self.grinding_factor = grinding_factor
        self.hash_fn = hash_fn

    def _c(self):
        return backend.DgOptions(self.extension_factor, self.num_queries, self.grinding_factor, PROOF_HASHES[self.hash_fn])


class StarkProof:
    """Result of prove(): the bincode bytes of the reference's StarkProof plus a few commitments for differential tests."""

    def __init__(self, data, trace_root, constraint_root, pow_seed, pow_nonce, stats):
        self.bytes = data
        self.trace_root = trace_root
        self.constraint_root = constraint_root
        self.pow_seed = pow_seed
        self.pow_nonce = pow_nonce
        self.stats = stats

    def __len__(self):
        return len(self.bytes)


def _collect(handle, stats):
    L = backend.lib()
    try:
        n = ctypes.c_size_t(0)
        backend.check(L.dg_proof_serialized_len(handle, ctypes.byref(n)))
        buf = ctypes.create_string_buffer(n.value)
        backend.check(L.dg_proof_serialize(handle, buf, n.value))
        digs = []
        for which in range(3):
            d = ctypes.create_string_buffer(32)
            backend.check(L.dg_proof_digest(handle, which, d))
            digs.append(d.raw)
        nonce = backend.u64(0)
        backend.check(L.dg_proof_pow_nonce(handle, ctypes.byref(nonce)))
    finally:
        L.dg_proof_free(handle)
    st = {"stage_ms": [float(x) for x in stats.stage_ms], "h2d_ms": float(stats.h2d_ms), "total_ms": float(stats.total_ms),
          "kernel_launches": int(stats.kernel_launches)}
    return StarkProof(buf.raw, digs[0], digs[1], digs[2], nonce.value, st)


def prove(trace, options=None):
    """stark::prove(&mut trace, inputs, outputs, options) for a hostvm.ExecutionTrace (host memory in, proof bytes out)."""
    options = options or ProofOptions()
    regs = np.ascontiguousarray(trace.registers, dtype=np.uint64)
    w, n = regs.shape[0], regs.shape[1]
    cols = (backend.vp * w)(*[regs[j].ctypes.data for j in range(w)])
    t = backend.DgTrace(cols, w, n, trace.ctx_depth, trace.loop_depth)
    fi, fo = felt.from_ints(trace.public_inputs), felt.from_ints(trace.outputs)
    opt = options._c()
    handle = backend.vp()
    stats = backend.DgStats()
    backend.check(backend.lib().dg_prove(ctypes.byref(t), fi.ctypes.data, len(fi), fo.ctypes.data, len(fo), ctypes.byref(opt),
                                        ctypes.byref(handle), ctypes.byref(stats)))
    return _collect(handle, stats)


def prove_device(d_registers, width, length, ctx_depth, loop_depth, public_inputs, outputs, options=None):
    """Same, for register traces already resident in device memory (backend.DeviceBuffer or raw pointer)."""
    options = options or ProofOptions()
    ptr = d_registers.ptr if isinstance(d_registers, backend.DeviceBuffer) else int(d_registers)
    fi, fo = felt.from_ints(public_inputs), felt.from_ints(outputs)
    opt = options._c()
    handle = backend.vp()
    stats = backend.DgStats()
    backend.check(backend.lib().dg_prove_device(ptr, width, length, ctx_depth, loop_depth, fi.ctypes.data, len(fi), fo.ctypes.data, len(fo),
                                               ctypes.byref(opt), ctypes.byref(handle), ctypes.byref(stats)))
    return _collect(handle, stats)


def verify(program_hash, public_inputs, outputs, proof):
    """distaff::verify (lib.rs:68-75 -> stark/verifier.rs:11-75) on the GPU.  Returns None when the proof is accepted, otherwise the
    reference's error string (what `Err(msg)` carries); raises DgError for bytes that are not a serialized StarkProof.  The hash
    (blake3 or sha3) is the one the proof's options name: the last byte of the bytes."""
    data = proof.bytes if isinstance(proof, StarkProof) else bytes(proof)
    fi, fo = felt.from_ints(public_inputs), felt.from_ints(outputs)
    msg = ctypes.create_string_buffer(256)
    rc = backend.lib().dg_verify(bytes(program_hash), fi.ctypes.data, len(fi), fo.ctypes.data, len(fo), data, len(data), msg, 256)
    if rc == 0:
        return None
    if rc == -6:
        return msg.value.decode()
    backend.check(rc)


def execute(source, public_inputs=(), secret_a=(), secret_b=(), num_outputs=1, options=None):
    """distaff::execute (lib.rs:30-65): run the program on the host VM, then prove on the GPU. Returns (outputs, proof)."""
    trace = hostvm.execute(source, public_inputs, secret_a, secret_b, num_outputs)
    return trace.outputs, prove(trace, options)


# ---- building blocks ------------------------------------------------------------------------------------------------------
def ntt(values, inverse=False):
    """polynom::eval_fft / interpolate_fft on (batch, n, 2) or (n, 2) uint64 arrays; returns a new array"""
    a = np.ascontiguousarray(values, dtype=np.uint64).copy()
    shape = a.shape
    n = shape[-2]
    batch = int(np.prod(shape[:-2])) if len(shape) > 2 else 1
    assert n & (n - 1) == 0 and n >= 2
    backend.check(backend.lib().dg_ntt(a.ctypes.data, n.bit_length() - 1, batch, 1 if inverse else 0))
    return a


def intt(values):
    return ntt(values, inverse=True)


def lde(values, blowup=32):
    """TraceTable::extend for a (batch, n, 2) array of register traces: returns (batch, n*blowup, 2) evaluations in LDE order"""
    a = np.ascontiguousarray(values, dtype=np.uint64)
    if a.ndim == 2:
        a = a[None]
    batch, n = a.shape[0], a.shape[1]
    out = np.empty((batch, n * blowup, 2), dtype=np.uint64)
    backend.check(backend.lib().dg_lde(a.ctypes.data, out.ctypes.data, n.bit_length() - 1, blowup.bit_length() - 1, batch))
    return out


HASH_IDS = {"blake3": 0, "rescue": 1, "poseidon": 2, "sha3": 4}


def merkle_build(leaves, hash="blake3"):
    """crypto::build_merkle_nodes (merkle.rs:269-294): bytes (n*32) -> bytes (n*32), heap layout; hash in blake3 | rescue | poseidon | sha3"""
    leaves = bytes(leaves)
    n = len(leaves) // 32
    out = ctypes.create_string_buffer(n * 32)
    if hash == "blake3":
        backend.check(backend.lib().dg_merkle_build(leaves, n, out))
    else:
        backend.check(backend.lib().dg_merkle_build_with(HASH_IDS[hash], leaves, n, out))
    return out.raw


def hash64(messages, hash="rescue"):
    """crypto::hash::{blake3, rescue, poseidon, sha3} of n independent 64-byte messages: bytes (n*64) -> bytes (n*32)"""
    messages = bytes(messages)
    assert len(messages) % 64 == 0
    n = len(messages) // 64
    out = ctypes.create_string_buffer(max(1, n * 32))
    backend.check(backend.lib().dg_hash64(HASH_IDS[hash], messages, n, out))
    return out.raw[:n * 32]


def hash_rows(columns):
    """blake3 of every row of a column-major (w, rows, 2) uint64 matrix -> bytes rows*32"""
    a = np.ascontiguousarray(columns, dtype=np.uint64)
    w, rows = a.shape[0], a.shape[1]
    out = ctypes.create_string_buffer(rows * 32)
    backend.check(backend.lib().dg_hash_rows(a.ctypes.data, w, rows, out))
    return out.raw


def find_pow_nonce(seed, grinding_factor=20):
    nonce = backend.u64(0)
    out = ctypes.create_string_buffer(32)
    backend.check(backend.lib().dg_find_pow_nonce(bytes(seed), grinding_factor, ctypes.byref(nonce), out))
    return out.raw, nonce.value


def field_op(op, a, b=None, impl=0):
    code = {"add": 0, "sub": 1, "mul": 2, "inv": 3, "exp": 4, "dot6": 5}[op]
    fa = np.ascontiguousarray(a, dtype=np.uint64)
    fb = np.ascontiguousarray(b, dtype=np.uint64) if b is not None else None
    out = np.empty_like(fa)
    backend.check(backend.lib().dg_field_op(code, impl, fa.ctypes.data, fb.ctypes.data if fb is not None else None, out.ctypes.data, fa.shape[0]))
    return out[:fa.shape[0] // 6] if op == "dot6" else out
