"""ctypes binding of distaff_b200/libdistaff_gpu.so (C-ABI in include/distaff_gpu.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device is visible, every call raises.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DG_LIB_PATH") or os.path.join(_HERE, "libdistaff_gpu.so")   # DG_LIB_PATH: A/B builds of the same C-ABI
_LIB = None

vp = ctypes.c_void_p
u32 = ctypes.c_uint32
u64 = ctypes.c_uint64
fp = ctypes.POINTER(ctypes.c_float)


class DgError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"distaff_gpu error {code}: {message}")
        self.code = code


class DgTrace(ctypes.Structure):
    _fields_ = [("columns", ctypes.POINTER(vp)), ("width", u32), ("length", u64), ("ctx_depth", u32), ("loop_depth", u32)]


class DgOptions(ctypes.Structure):
    _fields_ = [("extension_factor", u32), ("num_queries", u32), ("grinding_factor", u32), ("hash_id", u32)]


class DgStats(ctypes.Structure):
    _fields_ = [("stage_ms", ctypes.c_float * 9), ("h2d_ms", ctypes.c_float), ("total_ms", ctypes.c_float), ("kernel_launches", u64)]


DRAW_FIELD_FN = ctypes.CFUNCTYPE(ctypes.c_int, vp, vp, u64, vp)
DRAW_POSITIONS_FN = ctypes.CFUNCTYPE(ctypes.c_int, vp, vp, u64, u32, u32, vp)


class DgRngCallbacks(ctypes.Structure):
    _fields_ = [("user", vp), ("draw_field", DRAW_FIELD_FN), ("draw_positions", DRAW_POSITIONS_FN)]


EXPORTS = {
    "dg_init": [ctypes.c_int],
    "dg_init_devices": [ctypes.c_int],
    "dg_set_rng_callbacks": [ctypes.POINTER(DgRngCallbacks)],
    "dg_device_info": [ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_size_t)],
    "dg_prove": [ctypes.POINTER(DgTrace), vp, u32, vp, u32, ctypes.POINTER(DgOptions), ctypes.POINTER(vp), ctypes.POINTER(DgStats)],
    "dg_prove_device": [vp, u32, u64, u32, u32, vp, u32, vp, u32, ctypes.POINTER(DgOptions), ctypes.POINTER(vp), ctypes.POINTER(DgStats)],
    "dg_verify": [vp, vp, u32, vp, u32, vp, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t],
    "dg_proof_serialized_len": [vp, ctypes.POINTER(ctypes.c_size_t)],
    "dg_proof_serialize": [vp, vp, ctypes.c_size_t],
    "dg_proof_digest": [vp, ctypes.c_int, vp],
    "dg_proof_pow_nonce": [vp, ctypes.POINTER(u64)],
    "dg_ntt": [vp, u32, u32, ctypes.c_int],
    "dg_lde": [vp, vp, u32, u32, u32],
    "dg_merkle_build": [vp, u64, vp],
    "dg_hash_rows": [vp, u32, u64, vp],
    "dg_hash64": [ctypes.c_int, vp, u64, vp],
    "dg_merkle_build_with": [ctypes.c_int, vp, u64, vp],
    "dg_find_pow_nonce": [vp, u32, ctypes.POINTER(u64), vp],
    "dg_field_op": [ctypes.c_int, ctypes.c_int, vp, vp, vp, u64],
    "dg_dev_alloc": [ctypes.POINTER(vp), ctypes.c_size_t],
    "dg_dev_free": [vp],
    "dg_dev_upload": [vp, vp, ctypes.c_size_t],
    "dg_dev_download": [vp, vp, ctypes.c_size_t],
    "dg_dev_sync": [],
    "dg_dev_ntt": [vp, u32, u32, ctypes.c_int, fp],
    "dg_dev_lde": [vp, vp, u32, u32, u32, fp],
    "dg_dev_merkle_build": [vp, u64, vp, fp],
    "dg_dev_merkle_build_with": [ctypes.c_int, vp, u64, vp, fp],
    "dg_dev_hash_rows": [vp, u32, u32, u32, vp, fp],
    "dg_dev_flush_l2": [],
    "dg_comm_unique_id": [vp],
    "dg_comm_init": [ctypes.c_int, ctypes.c_int, vp],
    "dg_comm_finalize": [],
    "dg_host_shard_locate": [u64, ctypes.c_int, ctypes.c_int, ctypes.c_int, u64, ctypes.POINTER(ctypes.c_int64)],
    "dg_host_prng_vector": [vp, u64, vp],
    "dg_host_query_positions": [vp, u64, u32, u32, vp],
    "dg_host_blake3": [vp, ctypes.c_size_t, vp],
    "dg_host_sha3": [vp, ctypes.c_size_t, vp],
    "dg_host_plan_batch": [vp, u32, u64, vp, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)],
    "dg_host_merkle_verify_plan": [vp, u32, u32, u32, vp, u32, vp, ctypes.c_size_t, vp, vp, ctypes.c_size_t, vp, vp],
    "dg_host_periodic_tables": [vp],
}
VOID_EXPORTS = {"dg_proof_free": [vp]}


def lib():
    """Loads the CUDA backend; raises if it has not been built (`python -c 'import __graft_entry__ as g; g.build()'`)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with make -C distaff_b200/csrc (there is no CPU fallback)")
        L = ctypes.CDLL(LIB_PATH)
        for name, args in EXPORTS.items():
            fn = getattr(L, name)
            fn.restype = ctypes.c_int
            fn.argtypes = args
        for name, args in VOID_EXPORTS.items():
            fn = getattr(L, name)
            fn.restype = None
            fn.argtypes = args
        L.dg_last_error.restype = ctypes.c_char_p
        L.dg_last_error.argtypes = []
        _LIB = L
    return _LIB


def check(rc):
    if rc != 0:
        raise DgError(rc, lib().dg_last_error().decode(errors="replace"))


_RNG_KEEPALIVE = None


def set_rng_callbacks(draw_field=None, draw_positions=None):
    """dg_set_rng_callbacks: draw_field(seed: bytes, count) -> bytes (count*16), draw_positions(seed, domain, ext, nq) -> list[int];
    called with no arguments it restores the built-in generator.  (The binding a Rust host would use is in INTEGRATION.md.)"""
    global _RNG_KEEPALIVE
    if draw_field is None and draw_positions is None:
        check(lib().dg_set_rng_callbacks(None))
        _RNG_KEEPALIVE = None
        return

    def _field(user, seed, count, out):
        try:
            data = draw_field(ctypes.string_at(seed, 32), int(count))
            ctypes.memmove(out, data, int(count) * 16)
            return 0
        except Exception:
            return 1

    def _positions(user, seed, domain, ext, nq, out):
        try:
            pos = draw_positions(ctypes.string_at(seed, 32), int(domain), int(ext), int(nq))
            if len(pos) != nq:
                return 1
            arr = (ctypes.c_uint64 * nq)(*pos)
            ctypes.memmove(out, arr, 8 * nq)
            return 0
        except Exception:
            return 1

    cb = DgRngCallbacks(None, DRAW_FIELD_FN(_field) if draw_field else DRAW_FIELD_FN(0),
                        DRAW_POSITIONS_FN(_positions) if draw_positions else DRAW_POSITIONS_FN(0))
    _RNG_KEEPALIVE = cb
    check(lib().dg_set_rng_callbacks(ctypes.byref(cb)))


def device_info():
    name = ctypes.create_string_buffer(128)
    sms = ctypes.c_int(0)
    mem = ctypes.c_size_t(0)
    check(lib().dg_device_info(name, 128, ctypes.byref(sms), ctypes.byref(mem)))
    return {"name": name.value.decode(), "sm_count": sms.value, "total_mem": mem.value}


def comm_init_from_torch(dist, device_index):
    """Joins the NCCL communicator used to shard one proof over the ranks of an initialised torch.distributed group."""
    import torch
    rank, world = dist.get_rank(), dist.get_world_size()
    ident = torch.zeros(128, dtype=torch.uint8, device=f"cuda:{device_index}")
    if rank == 0:
        buf = ctypes.create_string_buffer(128)
        check(lib().dg_comm_unique_id(buf))
        ident.copy_(torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8))
    dist.broadcast(ident, src=0)
    raw = bytes(ident.cpu().numpy().tobytes())
    check(lib().dg_comm_init(rank, world, raw))
    return rank, world


class DeviceBuffer:
    """Raw device allocation owned by the backend's context."""

    def __init__(self, nbytes):
        self.nbytes = int(nbytes)
        p = vp()
        check(lib().dg_dev_alloc(ctypes.byref(p), self.nbytes))
        self.ptr = p.value

    def upload(self, array):
        a = np.ascontiguousarray(array)
        assert a.nbytes <= self.nbytes
        check(lib().dg_dev_upload(self.ptr, a.ctypes.data, a.nbytes))
        return self

    def download(self, shape, dtype=np.uint64):
        out = np.empty(shape, dtype=dtype)
        assert out.nbytes <= self.nbytes
        check(lib().dg_dev_download(out.ctypes.data, self.ptr, out.nbytes))
        return out

    def free(self):
        if self.ptr:
            lib().dg_dev_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
