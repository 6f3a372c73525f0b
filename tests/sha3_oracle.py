"""TEST INFRASTRUCTURE ONLY.  ctypes face of tests/sha3_oracle.cpp: the CPU oracle (oracle/) proving and verifying with SHA3-256
commitments.  The library is compiled on first use, with the oracle's compiler flags, into the temporary directory (keyed by the
sources, so the tree stays untouched and concurrent processes reuse one build)."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_SOURCES = [os.path.join(_HERE, "sha3_oracle.cpp")] + [os.path.join(_ROOT, "oracle", f) for f in
                                                       ("math.h", "crypto.h", "air.h", "stark.h", "ref_constants.h")]
_FLAGS = ["-O3", "-march=x86-64-v3", "-fPIC", "-fopenmp", "-B/usr/lib/gcc/x86_64-linux-gnu/13", "-std=c++17", "-Wall",
          "-Wno-unused-function", "-shared"]             # oracle/Makefile
_LIB = None
vp = ctypes.c_void_p


def lib():
    global _LIB
    if _LIB is None:
        key = hashlib.sha256(b"".join(open(p, "rb").read() for p in _SOURCES)).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"distaff_sha3_oracle_{os.getuid()}_{key}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}"
            subprocess.check_call([os.environ.get("CXX", "g++"), *_FLAGS, "-o", tmp, _SOURCES[0]])
            os.replace(tmp, path)
        L = ctypes.CDLL(path)
        L.so_set_threads.restype = ctypes.c_int
        L.so_set_threads.argtypes = [ctypes.c_int]
        L.so_sha3.argtypes = [vp, ctypes.c_uint64, vp]
        L.so_merkle_nodes.argtypes = [vp, ctypes.c_uint64, vp]
        L.so_prove.restype = ctypes.c_int64
        L.so_prove.argtypes = [vp, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32, vp, ctypes.c_uint32, vp, ctypes.c_uint32,
                               ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32, vp, ctypes.c_uint64, ctypes.c_char_p, ctypes.c_uint32]
        L.so_verify.restype = ctypes.c_int
        L.so_verify.argtypes = [vp, vp, ctypes.c_uint32, vp, ctypes.c_uint32, vp, ctypes.c_uint64, ctypes.c_char_p, ctypes.c_uint32]
        _LIB = L
    return _LIB


def _fvec(values):
    a = np.empty((len(values), 2), dtype=np.uint64)
    for i, v in enumerate(values):
        a[i, 0] = v & (2**64 - 1)
        a[i, 1] = v >> 64
    return a


def set_threads(t):
    return lib().so_set_threads(int(t))


def hash(data):
    data = bytes(data)
    out = ctypes.create_string_buffer(32)
    lib().so_sha3(data, len(data), out)
    return out.raw


def merkle_nodes(leaves):
    """leaves: bytes of n*32 -> bytes of n*32 (heap layout), hashed with sha3"""
    leaves = bytes(leaves)
    n = len(leaves) // 32
    out = ctypes.create_string_buffer(n * 32)
    lib().so_merkle_nodes(leaves, n, out)
    return out.raw


def prove(registers, ctx_depth, loop_depth, inputs, outputs, ext=32, num_queries=50, grinding=20):
    """registers: (w, n, 2) uint64 column-major.  Returns the bytes of the sha3 proof; raises RuntimeError with the prover's message."""
    regs = np.ascontiguousarray(registers, dtype=np.uint64)
    fi, fo = _fvec(list(inputs)), _fvec(list(outputs))
    err = ctypes.create_string_buffer(512)
    cap = 1 << 20
    while True:
        out = ctypes.create_string_buffer(cap)
        n = lib().so_prove(regs.ctypes.data, regs.shape[0], regs.shape[1], ctx_depth, loop_depth, fi.ctypes.data, len(fi), fo.ctypes.data,
                           len(fo), ext, num_queries, grinding, out, cap, err, 512)
        if n < 0:
            raise RuntimeError(err.value.decode())
        if n <= cap:
            return out.raw[:n]
        cap = n


def verify(program_hash, inputs, outputs, proof):
    """None when the proof (hash byte 0 = blake3 or 4 = sha3) verifies, else the verifier's error string"""
    fi, fo = _fvec(list(inputs)), _fvec(list(outputs))
    err = ctypes.create_string_buffer(512)
    proof = bytes(proof)
    rc = lib().so_verify(bytes(program_hash), fi.ctypes.data, len(fi), fo.ctypes.data, len(fo), proof, len(proof), err, 512)
    return None if rc == 0 else err.value.decode()
