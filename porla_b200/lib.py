"""ctypes binding of libmultiexp.so -- the same binding a Porla maintainer gets from
``#include "libmultiexp.h"`` + ``-lmultiexp`` (/root/reference/porla/Makefile:13), written in Python
because the tests and the benchmark are Python.  Function names and argument meaning follow
/root/reference/porla/Utils/utils.h:235-305.
"""
from __future__ import annotations

import ctypes as C
import os
import struct
from typing import Optional, Sequence

LIB_PATH = os.environ.get("PORLA_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libmultiexp.so")

CURVE_BN254, CURVE_SECP256K1 = 0, 1
SCALAR_BE32, SCALAR_LE32 = 0, 1
POINT_BE64, POINT_LE64 = 0, 1
PLAN_GLV_ON, PLAN_GLV_OFF, PLAN_FIXED = 0x100, 0x200, 0x400     # plan-code flags of porla_msm_plan (include/porla_multiexp.h)

# every symbol include/porla_multiexp.h declares (checked by tests/test_abi_symbols.py)
LEGACY_SYMBOLS = [
    "init_key", "init_SRS", "init_SRS_from_data", "compute_digest", "compute_digest_complement",
    "compute_digest_from_srs", "compute_multi_exp", "compare_commitment", "create_proof",
    "verify_proof", "add_point", "mult_point", "neg_point", "set_inf_point",
]
NEW_SYMBOLS = [
    "porla_device_init", "porla_launch_count", "compute_multi_exp_batch",
    "compute_digest_from_srs_batch", "porla_table_create", "porla_table_create_multiples",
    "porla_table_precompute", "porla_table_len", "porla_table_num_infinity", "porla_table_export", "porla_table_destroy",
    "porla_msm_device", "porla_msm_resident", "porla_msm_plan", "porla_msm_window_sums_device",
    "porla_msm_finalize_host", "porla_msm_combine_device", "porla_msm_host", "porla_choose_window",
    "porla_scalar_mul_batch_device", "porla_secp256k1_ecmult_multi_var",
    "porla_secp256k1_gej_serialize", "porla_debug_field_mul", "porla_debug_field_op", "porla_debug_point_add_host", "porla_measure_pint",
    "porla_stage_timing_enable", "porla_stage_timing_read",
    "porla_butterfly_stage_device", "bn254_butterfly_stage", "bn254_align_mac_batch", "bn254_audit_aggregate", "porla_data_butterfly_stage", "porla_data_butterfly_stage_device",
    "porla_msm_table_host_scalars", "porla_msm_table_host_scalars_batch", "porla_secp256k1_table_create", "porla_secp256k1_ecmult_multi_table",
    "porla_debug_pairing_selfcheck", "porla_debug_latency", "porla_secp256k1_inner_product_prove", "porla_secp256k1_inner_product_verify",
    "porla_secp256k1_butterfly_stage", "porla_secp256k1_align_mac_batch", "porla_secp256k1_audit_aggregate",
    "porla_secp256k1_ecmult_multi_gej", "porla_secp256k1_ecmult_multi_table_batch", "porla_secp256k1_ecmult_const_batch",
    "porla_device_count", "porla_mtable_create", "porla_mtable_devices", "porla_mtable_len", "porla_mtable_range",
    "porla_mtable_msm_host_scalars", "porla_mtable_msm_resident", "porla_mtable_scalars_upload", "porla_mtable_scalars_free",
    "porla_mtable_destroy", "porla_debug_copy_ring_bytes", "porla_msm_host_devices", "porla_debug_h2d_rate",
    "porla_debug_quad_op", "compute_digest_batch", "compute_digest_complement_batch",
]


class GoSlice(C.Structure):
    """libmultiexp.h:61."""
    _fields_ = [("data", C.c_void_p), ("len", C.c_longlong), ("cap", C.c_longlong)]


class SecpFe(C.Structure):
    _fields_ = [("n", C.c_uint64 * 5)]


class SecpGe(C.Structure):
    _fields_ = [("x", SecpFe), ("y", SecpFe), ("infinity", C.c_int)]


class SecpGej(C.Structure):
    _fields_ = [("x", SecpFe), ("y", SecpFe), ("z", SecpFe), ("infinity", C.c_int)]


class SecpScalar(C.Structure):
    _fields_ = [("d", C.c_uint64 * 4)]


SECP_CB = C.CFUNCTYPE(C.c_int, C.POINTER(SecpScalar), C.POINTER(SecpGe), C.c_size_t, C.c_void_p)

_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """dlopen the CUDA library.  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `make` (nvcc, sm_100a). porla_b200 has no "
            "Python/CPU implementation of the MSM path.")
    lib = C.CDLL(LIB_PATH)
    P, LL, I = C.c_void_p, C.c_longlong, C.c_int
    GS = C.POINTER(GoSlice)
    sig = {
        "init_key": (None, [GS, GS]),
        "init_SRS": (None, [LL, GS, C.POINTER(LL)]),
        "init_SRS_from_data": (None, [LL, GS]),
        "compute_digest": (None, [GS, GS]),
        "compute_digest_complement": (None, [GS, GS]),
        "compute_digest_from_srs": (None, [GS, GS]),
        "compute_multi_exp": (None, [GS, GS, LL, GS]),
        "compare_commitment": (C.c_ubyte, [GS, GS]),
        "create_proof": (None, [C.c_ulonglong, GS, GS, GS, GS, GS]),
        "verify_proof": (C.c_ubyte, [GS, GS, GS, GS]),
        "add_point": (None, [GS, GS]),
        "mult_point": (None, [GS, GS]),
        "neg_point": (None, [GS]),
        "set_inf_point": (None, [GS]),
        "porla_device_init": (I, []),
        "porla_launch_count": (C.c_uint64, []),
        "compute_multi_exp_batch": (None, [GS, GS, LL, LL, GS]),
        "compute_digest_from_srs_batch": (None, [GS, LL, GS]),
        "compute_digest_batch": (None, [GS, LL, GS]),
        "compute_digest_complement_batch": (None, [GS, LL, GS]),
        "porla_table_create": (P, [I, P, C.c_int64, I, I, P]),
        "porla_table_create_multiples": (P, [I, P, C.c_int64, I, I, P]),
        "porla_table_precompute": (I, [P, I, C.c_int64, C.c_int64, P]),
        "porla_table_len": (C.c_int64, [P]),
        "porla_table_num_infinity": (C.c_int64, [P]),
        "porla_table_export": (None, [P, I, P, I, P]),
        "porla_table_destroy": (None, [P]),
        "porla_msm_device": (None, [P, P, C.c_int64, C.c_int64, I, I, I, I, P, P, P]),
        "porla_msm_resident": (None, [P, P, C.c_int64, I, I, I, P, P]),
        "porla_msm_plan": (None, [I, C.c_int64, C.c_int64, I, C.POINTER(I), C.POINTER(I)]),
        "porla_msm_window_sums_device": (None, [P, P, C.c_int64, I, I, P, P]),
        "porla_msm_finalize_host": (None, [I, P, C.c_int64, I, I, I, P]),
        "porla_msm_combine_device": (None, [I, P, C.c_int64, C.c_int64, I, P, P]),
        "porla_msm_host": (None, [I, P, P, C.c_int64, C.c_int64, I, I, P]),
        "porla_choose_window": (I, [I, C.c_int64, C.c_int64]),
        "porla_scalar_mul_batch_device": (None, [P, P, C.c_int64, I, I, P, P]),
        "porla_secp256k1_ecmult_multi_var": (I, [P, P, C.POINTER(SecpGej), C.POINTER(SecpScalar), SECP_CB, P, C.c_size_t]),
        "porla_secp256k1_gej_serialize": (I, [C.POINTER(SecpGej), C.c_char_p]),
        "porla_measure_pint": (C.c_double, [I, C.c_double]),
        "porla_stage_timing_enable": (None, [I]),
        "porla_stage_timing_read": (I, [C.POINTER(C.c_float)]),
        "porla_butterfly_stage_device": (None, [P, C.c_int64, P, I, I, P]),
        "bn254_butterfly_stage": (None, [GS, LL, LL, GS]),
        "bn254_align_mac_batch": (None, [GS, LL, GS]),
        "bn254_audit_aggregate": (None, [GS, GS, LL, GS, GS]),
        "porla_data_butterfly_stage": (None, [P, C.c_int64, C.c_int64, C.c_int64, C.c_char_p, C.c_char_p]),
        "porla_data_butterfly_stage_device": (None, [P, C.c_int64, C.c_int64, C.c_int64, P, C.c_char_p, P]),
        "porla_msm_table_host_scalars": (None, [P, C.c_int64, P, C.c_int64, I, I, P]),
        "porla_msm_table_host_scalars_batch": (None, [P, C.c_int64, P, C.c_int64, C.c_int64, I, I, P]),
        "porla_secp256k1_table_create": (P, [C.POINTER(SecpGe), C.c_size_t]),
        "porla_secp256k1_ecmult_multi_table": (I, [P, C.c_size_t, C.POINTER(SecpScalar), C.c_size_t, C.POINTER(SecpGej)]),
        "porla_secp256k1_ecmult_multi_table_batch": (I, [P, C.c_size_t, C.POINTER(SecpScalar), C.c_size_t, C.c_size_t,
                                                         C.POINTER(SecpGej)]),
        "porla_secp256k1_ecmult_const_batch": (I, [P, C.POINTER(SecpScalar), C.c_size_t, C.POINTER(SecpGej)]),
        "porla_debug_pairing_selfcheck": (I, [I]),
        "porla_secp256k1_inner_product_prove": (C.c_size_t, [P, C.c_size_t, C.c_char_p, C.c_char_p, C.c_char_p]),
        "porla_secp256k1_inner_product_verify": (I, [P, C.c_size_t, C.POINTER(SecpGej), C.c_char_p]),
        "porla_secp256k1_butterfly_stage": (I, [C.POINTER(SecpGej), C.c_size_t, C.c_size_t, C.POINTER(SecpScalar)]),
        "porla_secp256k1_align_mac_batch": (I, [P, C.c_size_t, P, C.c_size_t, C.POINTER(SecpGej)]),
        "porla_secp256k1_audit_aggregate": (I, [P, C.c_size_t, P, P, C.c_size_t, P, C.POINTER(SecpGej)]),
        "porla_secp256k1_ecmult_multi_gej": (I, [C.POINTER(SecpGej), C.POINTER(SecpScalar), C.c_size_t, C.c_size_t,
                                                 C.POINTER(SecpGej)]),
        "porla_debug_latency": (I, [I, I, I, I, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
        "porla_debug_quad_op": (None, [I, I, P, P, C.c_int64, I, P]),
        "porla_debug_field_mul": (None, [I, P, P, C.c_int64, P]),
        "porla_debug_field_op": (None, [I, I, P, P, C.c_int64, P]),
        "porla_debug_point_add_host": (None, [I, P, P, C.c_int64, I, P]),
        "porla_device_count": (I, []),
        "porla_mtable_create": (P, [I, P, C.c_int64, I, I]),
        "porla_mtable_devices": (I, [P]),
        "porla_mtable_len": (C.c_int64, [P]),
        "porla_mtable_range": (None, [P, I, C.POINTER(I), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
        "porla_mtable_msm_host_scalars": (None, [P, P, I, I, P]),
        "porla_mtable_msm_resident": (None, [P, C.POINTER(P), I, I, P]),
        "porla_mtable_scalars_upload": (P, [P, I, P]),
        "porla_mtable_scalars_free": (None, [P, I, P]),
        "porla_mtable_destroy": (None, [P]),
        "porla_debug_copy_ring_bytes": (C.c_uint64, []),
        "porla_debug_h2d_rate": (C.c_double, [P, C.c_uint64, I]),
        "porla_msm_host_devices": (None, [I, P, P, C.c_int64, I, I, I, P]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


# ------------------------------------------------------------------------------- helpers
def _slice(buf) -> GoSlice:
    """GoSlice over a ctypes buffer / bytearray (caller keeps `buf` alive)."""
    if isinstance(buf, (bytes, bytearray)):
        arr = (C.c_ubyte * len(buf)).from_buffer(buf) if isinstance(buf, bytearray) else (C.c_ubyte * len(buf)).from_buffer_copy(buf)
    else:
        arr = buf
    s = GoSlice(C.cast(arr, C.c_void_p), C.sizeof(arr), C.sizeof(arr))
    s._keep = arr
    return s


def _ptr_slice(ptr: int, nbytes: int) -> GoSlice:
    return GoSlice(C.c_void_p(ptr), nbytes, nbytes)


# ------------------------------------------------------------------------------- utils.h mirrors
def bn254_add(a: bytearray, b: bytes) -> None:
    """utils.h:235 -- a += b, in place on the 64-byte MAC_Block."""
    load().add_point(C.byref(_slice(a)), C.byref(_slice(bytearray(b))))


def bn254_mult(a: bytearray, scalar: bytes) -> None:
    """utils.h:245 -- a = scalar * a, scalar a 32-byte big-endian bn254_scalar."""
    load().mult_point(C.byref(_slice(a)), C.byref(_slice(bytearray(scalar))))


def bn254_neg(a: bytearray) -> None:
    """utils.h:255."""
    load().neg_point(C.byref(_slice(a)))


def bn254_set_infinity(a: bytearray) -> None:
    """utils.h:263."""
    load().set_inf_point(C.byref(_slice(a)))


def bn254_scalar_set_int(value: int) -> bytes:
    """utils.h:271 -- words 0..6 zero, word 7 = htonl(value)."""
    return bytes(28) + struct.pack(">I", value & 0xFFFFFFFF)


def bn254_multi_exp(points: bytes, scalars: bytes, length: int) -> bytes:
    """utils.h:277 -- result = sum scalars[i] * points[i]; 64-byte MAC_Block out."""
    out = bytearray(64)
    sc, pt = bytearray(scalars), bytearray(points)
    load().compute_multi_exp(C.byref(_slice(sc)), C.byref(_slice(pt)), length, C.byref(_slice(out)))
    return bytes(out)


def bn254_multi_exp_batch(points: bytes, scalars: bytes, length: int, batch: int) -> bytes:
    out = bytearray(64 * batch)
    sc, pt = bytearray(scalars), bytearray(points)
    load().compute_multi_exp_batch(C.byref(_slice(sc)), C.byref(_slice(pt)), length, batch, C.byref(_slice(out)))
    return bytes(out)


def bn254_butterfly_stage(points: bytearray, n: int, m: int, twiddles: bytes) -> None:
    """One stage of the FFT in the exponent, in place on n 64-byte MAC_Blocks (the loop body of
    Server.hpp:1577-1608 for every butterfly of the stage): twiddles = m/2 bn254_scalars (32 B BE)."""
    load().bn254_butterfly_stage(C.byref(_slice(points)), n, m, C.byref(_slice(bytearray(twiddles))))


def bn254_compare(a: bytes, b: bytes) -> bool:
    """utils.h:294."""
    return bool(load().compare_commitment(C.byref(_slice(bytearray(a))), C.byref(_slice(bytearray(b)))))


class Kzg:
    """The KZG half of the C-ABI as Porla's Client/Server drive it
    (Client.hpp:159-167,348-354,408-419,439-453; Server.hpp:179-188,363-398,550-558)."""

    def __init__(self, tau_key: bytes, alpha_key: bytes):
        self.lib = load()
        self.lib.init_key(C.byref(_slice(bytearray(tau_key))), C.byref(_slice(bytearray(alpha_key))))
        self.n = 0

    def init_srs(self, n: int) -> bytes:
        out = bytearray(n * 32 + 132)
        ln = C.c_longlong(0)
        self.lib.init_SRS(n, C.byref(_slice(out)), C.byref(ln))
        self.n = n
        return bytes(out[: ln.value])

    def init_srs_from_data(self, n: int, blob: bytes) -> None:
        self.lib.init_SRS_from_data(n, C.byref(_slice(bytearray(blob))))
        self.n = n

    def compute_digest(self, data: bytes) -> bytes:
        out = bytearray(64)
        self.lib.compute_digest(C.byref(_slice(bytearray(data))), C.byref(_slice(out)))
        return bytes(out)

    def compute_digest_complement(self, s: bytes) -> bytes:
        out = bytearray(64)
        self.lib.compute_digest_complement(C.byref(_slice(bytearray(s))), C.byref(_slice(out)))
        return bytes(out)

    def compute_digest_batch(self, data: bytes, batch: int) -> bytes:
        """`batch` records of n_samples x 32-byte BE coefficients; returns batch x 64 bytes, record j equal to
        compute_digest of record j."""
        out = bytearray(64 * batch)
        self.lib.compute_digest_batch(C.byref(_slice(bytearray(data))), batch, C.byref(_slice(out)))
        return bytes(out)

    def compute_digest_complement_batch(self, scalars: bytes, batch: int) -> bytes:
        """`batch` 32-byte BE scalars; returns batch x 64 bytes, record j equal to compute_digest_complement of scalar j."""
        out = bytearray(64 * batch)
        self.lib.compute_digest_complement_batch(C.byref(_slice(bytearray(scalars))), batch, C.byref(_slice(out)))
        return bytes(out)

    def compute_digest_from_srs(self, data: bytes) -> bytes:
        out = bytearray(64)
        self.lib.compute_digest_from_srs(C.byref(_slice(bytearray(data))), C.byref(_slice(out)))
        return bytes(out)

    def compute_digest_from_srs_batch(self, data: bytes, batch: int) -> bytes:
        out = bytearray(64 * batch)
        self.lib.compute_digest_from_srs_batch(C.byref(_slice(bytearray(data))), batch, C.byref(_slice(out)))
        return bytes(out)

    def align_mac_batch(self, data: bytearray, batch: int) -> bytes:
        """Server::align_MAC for `batch` blocks at once (Server.hpp:478-562): data = batch*n*64 bytes of LE
        chunk values below PRIME_MODULUS*r, reduced mod PRIME_MODULUS in place; returns batch*64 bytes."""
        out = bytearray(64 * batch)
        self.lib.bn254_align_mac_batch(C.byref(_slice(data)), batch, C.byref(_slice(out)))
        return bytes(out)

    def audit_aggregate(self, coefs: bytes, blocks: bytes, n: int):
        """Server::audit's B = sum coef_i * block_i followed by align_MAC on B (Server.hpp:790-828, 903): coefs n x 4 B
        LE, blocks n x n_samples x 64 B LE; returns (B % PRIME_MODULUS as n_samples x 32 B BE, 64-byte alignment value)."""
        b_out, al = bytearray(32 * self.n), bytearray(64)
        self.lib.bn254_audit_aggregate(C.byref(_slice(bytearray(coefs))), C.byref(_slice(bytearray(blocks))), n,
                                       C.byref(_slice(b_out)), C.byref(_slice(al)))
        return bytes(b_out), bytes(al)

    def create_proof(self, random_point: int, data: bytes):
        c, h, z, y = bytearray(64), bytearray(64), bytearray(32), bytearray(32)
        self.lib.create_proof(random_point, C.byref(_slice(bytearray(data))), C.byref(_slice(c)), C.byref(_slice(h)),
                              C.byref(_slice(z)), C.byref(_slice(y)))
        return bytes(c), bytes(h), bytes(z), bytes(y)

    def verify_proof(self, c: bytes, h: bytes, z: bytes, y: bytes) -> bool:
        return bool(self.lib.verify_proof(C.byref(_slice(bytearray(c))), C.byref(_slice(bytearray(h))),
                                          C.byref(_slice(bytearray(z))), C.byref(_slice(bytearray(y)))))


# ------------------------------------------------------------------------------- new entry points
class Table:
    """A point table resident in HBM (SRS / generator table), internal Montgomery form."""

    def __init__(self, handle: int, curve: int):
        self.handle, self.curve = handle, curve

    @classmethod
    def from_host(cls, curve: int, points: bytes, point_fmt: int = POINT_BE64) -> "Table":
        n = len(points) // 64
        buf = bytearray(points)
        h = load().porla_table_create(curve, C.cast((C.c_ubyte * len(buf)).from_buffer(buf), C.c_void_p), n, point_fmt, 0, None)
        return cls(h, curve)

    @classmethod
    def from_device(cls, curve: int, dev_ptr: int, n: int, point_fmt: int = POINT_BE64, stream: int = 0) -> "Table":
        return cls(load().porla_table_create(curve, C.c_void_p(dev_ptr), n, point_fmt, 1, C.c_void_p(stream)), curve)

    @classmethod
    def multiples_of_generator(cls, curve: int, scalars, n: int, scalar_fmt: int = SCALAR_LE32,
                               on_device: bool = False, stream: int = 0) -> "Table":
        """table[i] = k_i * G.  `scalars`: bytes (host) or a device pointer."""
        if on_device:
            ptr = C.c_void_p(scalars)
        else:
            buf = bytearray(scalars)
            ptr = C.cast((C.c_ubyte * len(buf)).from_buffer(buf), C.c_void_p)
        return cls(load().porla_table_create_multiples(curve, ptr, n, scalar_fmt, int(on_device), C.c_void_p(stream)), curve)

    def precompute(self, window_bits: int = 0, n_hint: int = 0, batch_hint: int = 1, stream: int = 0) -> int:
        """Fixed-base expansion (2^(c*w) * P_i for every window); returns the window size used."""
        return int(load().porla_table_precompute(C.c_void_p(self.handle), window_bits, n_hint, batch_hint, C.c_void_p(stream)))

    def __len__(self) -> int:
        return int(load().porla_table_len(C.c_void_p(self.handle)))

    @property
    def num_infinity(self) -> int:
        return int(load().porla_table_num_infinity(C.c_void_p(self.handle)))

    def export(self, point_fmt: int = POINT_BE64) -> bytes:
        out = bytearray(64 * len(self))
        if len(self):
            load().porla_table_export(C.c_void_p(self.handle), point_fmt, C.cast((C.c_ubyte * len(out)).from_buffer(out), C.c_void_p), 0, None)
        return bytes(out)

    def msm_device(self, d_scalars: int, n: int, d_out: int = 0, nbatch: int = 1, scalar_fmt: int = SCALAR_BE32,
                   shared_points: bool = True, window_bits: int = 0, out_fmt: int = POINT_BE64, d_out_xyzz: int = 0,
                   stream: int = 0) -> None:
        """Asynchronous MSM on device buffers (raw pointers, e.g. torch.Tensor.data_ptr())."""
        load().porla_msm_device(C.c_void_p(self.handle), C.c_void_p(d_scalars), n, nbatch, scalar_fmt, int(shared_points),
                                window_bits, out_fmt, C.c_void_p(d_out) if d_out else None,
                                C.c_void_p(d_out_xyzz) if d_out_xyzz else None, C.c_void_p(stream))

    def msm_resident(self, d_scalars: int, n: int, scalar_fmt: int = SCALAR_BE32, window_bits: int = 0,
                     out_fmt: int = POINT_BE64, stream: int = 0) -> bytes:
        """Synchronous MSM with device-resident scalars; the 64-byte result comes back to the host."""
        out = (C.c_ubyte * 64)()
        load().porla_msm_resident(C.c_void_p(self.handle), C.c_void_p(d_scalars), n, scalar_fmt, window_bits, out_fmt,
                                  C.cast(out, C.c_void_p), C.c_void_p(stream))
        return bytes(out)

    def butterfly_stage(self, m: int, twiddles: bytes, scalar_fmt: int = SCALAR_BE32, stream: int = 0) -> None:
        """In-place radix-2 butterfly stage over the resident table (host twiddles, m/2 x 32 bytes)."""
        tw = bytearray(twiddles)
        load().porla_butterfly_stage_device(C.c_void_p(self.handle), m, C.cast((C.c_ubyte * len(tw)).from_buffer(tw), C.c_void_p),
                                            scalar_fmt, 0, C.c_void_p(stream))

    def destroy(self) -> None:
        if self.handle:
            load().porla_table_destroy(C.c_void_p(self.handle))
            self.handle = 0


def _as_void_p(buf):
    """void* of a bytes-like object / ctypes buffer / integer address (caller keeps it alive)."""
    if isinstance(buf, int):
        return C.c_void_p(buf)
    if isinstance(buf, bytes):
        return C.cast(C.c_char_p(buf), C.c_void_p)
    if isinstance(buf, bytearray):
        return C.cast((C.c_ubyte * len(buf)).from_buffer(buf), C.c_void_p)
    return C.cast(buf, C.c_void_p)


class MultiTable:
    """A point table resident in HBM and range-sharded over the GPUs of the box inside ONE process (the in-call
    partition of Client.hpp:747-787 with devices in place of host threads)."""

    def __init__(self, curve: int, points, n: int, point_fmt: int = POINT_BE64, ndev: int = 0):
        self.curve, self.n = curve, n
        self._keep = points
        self.handle = load().porla_mtable_create(curve, _as_void_p(points), n, point_fmt, ndev)
        self.ndev = int(load().porla_mtable_devices(C.c_void_p(self.handle)))

    def part_range(self, part: int):
        d, f, c = C.c_int(0), C.c_int64(0), C.c_int64(0)
        load().porla_mtable_range(C.c_void_p(self.handle), part, C.byref(d), C.byref(f), C.byref(c))
        return d.value, f.value, c.value

    def msm_host_scalars(self, scalars, scalar_fmt: int = SCALAR_BE32, out_fmt: int = POINT_BE64) -> bytes:
        out = (C.c_ubyte * 64)()
        load().porla_mtable_msm_host_scalars(C.c_void_p(self.handle), _as_void_p(scalars), scalar_fmt, out_fmt, C.cast(out, C.c_void_p))
        return bytes(out)

    def upload_scalars(self, scalars: bytes):
        """Per-part resident copies of an n x 32-byte scalar array; returns the handle list msm_resident takes."""
        ptrs = []
        for p in range(self.ndev):
            _, first, count = self.part_range(p)
            chunk = bytes(scalars[32 * first:32 * (first + count)])
            ptrs.append(load().porla_mtable_scalars_upload(C.c_void_p(self.handle), p, _as_void_p(chunk)))
        return ptrs

    def free_scalars(self, ptrs) -> None:
        for p, d in enumerate(ptrs):
            load().porla_mtable_scalars_free(C.c_void_p(self.handle), p, C.c_void_p(d))

    def msm_resident(self, ptrs, scalar_fmt: int = SCALAR_BE32, out_fmt: int = POINT_BE64) -> bytes:
        out = (C.c_ubyte * 64)()
        arr = (C.c_void_p * self.ndev)(*ptrs)
        load().porla_mtable_msm_resident(C.c_void_p(self.handle), arr, scalar_fmt, out_fmt, C.cast(out, C.c_void_p))
        return bytes(out)

    def destroy(self) -> None:
        if self.handle:
            load().porla_mtable_destroy(C.c_void_p(self.handle))
            self.handle = 0


def msm_host_devices(curve: int, scalars, points, n: int, ndev: int = 0, scalar_fmt: int = SCALAR_BE32,
                     point_fmt: int = POINT_BE64) -> bytes:
    """One MSM from host buffers, its point range split over `ndev` GPUs inside the call (0 = all visible)."""
    out = (C.c_ubyte * 64)()
    load().porla_msm_host_devices(curve, _as_void_p(scalars), _as_void_p(points), n, scalar_fmt, point_fmt, ndev, C.cast(out, C.c_void_p))
    return bytes(out)


def msm_host(curve: int, scalars: bytes, points: bytes, n: int, nbatch: int = 1, scalar_fmt: int = SCALAR_BE32,
             point_fmt: int = POINT_BE64) -> bytes:
    out = bytearray(64 * nbatch)
    sc, pt = bytearray(scalars), bytearray(points)
    load().porla_msm_host(curve, C.cast((C.c_ubyte * len(sc)).from_buffer(sc), C.c_void_p) if sc else None,
                          C.cast((C.c_ubyte * len(pt)).from_buffer(pt), C.c_void_p) if pt else None,
                          n, nbatch, scalar_fmt, point_fmt,
                          C.cast((C.c_ubyte * len(out)).from_buffer(out), C.c_void_p))
    return bytes(out)


def _int_to_fe(v: int) -> SecpFe:
    fe = SecpFe()
    for i in range(5):
        fe.n[i] = (v >> (52 * i)) & ((1 << 52) - 1) if i < 4 else (v >> 208)
    return fe


def _fe_to_int(fe: SecpFe) -> int:
    return sum(int(fe.n[i]) << (52 * i) for i in range(5))


def _scalar_array(values: Sequence[int]):
    """ctypes array of SecpScalar (at least one element) holding integers below 2^256 as stored, not reduced."""
    return (SecpScalar * max(1, len(values))).from_buffer_copy(
        b"".join((s % (1 << 256)).to_bytes(32, "little") for s in values).ljust(32 * max(1, len(values)), b"\0"))


def _affine_or_none(g: SecpGej):
    return None if g.infinity else (_fe_to_int(g.x), _fe_to_int(g.y))


class SecpGenerators:
    """secp256k1 generator array resident in HBM (the `generators[]` of Server.hpp:347 / Client.hpp:393)."""

    def __init__(self, points: Sequence):
        arr = (SecpGe * max(1, len(points)))()
        for i, Pt in enumerate(points):
            if Pt is None:
                arr[i].infinity = 1
            else:
                arr[i].x, arr[i].y, arr[i].infinity = _int_to_fe(Pt[0]), _int_to_fe(Pt[1]), 0
        self.n = len(points)
        self.handle = load().porla_secp256k1_table_create(arr, self.n)

    def multi(self, first: int, scalars: Sequence[int]):
        """(ok, affine result or None) of sum scalars[i] * generators[first + i]."""
        n = len(scalars)
        sc = (SecpScalar * max(1, n))()
        for k, s in enumerate(scalars):
            for i in range(4):
                sc[k].d[i] = (s >> (64 * i)) & 0xFFFFFFFFFFFFFFFF
        r = SecpGej()
        ok = load().porla_secp256k1_ecmult_multi_table(C.c_void_p(self.handle), first, sc, n, C.byref(r))
        if r.infinity:
            return ok, None
        return ok, (_fe_to_int(r.x), _fe_to_int(r.y))

    def multi_batch(self, first: int, scalars: Sequence[int], n: int, batch: int):
        """(ok, list of `batch` affine results or None) of sum_i scalars[b*n + i] * generators[first + i] for b < batch:
        the per-block commitments of Client::initialize / Server::compute_commitment in one call.  (0, None) when the
        shape is refused."""
        r = (SecpGej * max(1, batch))()
        ok = load().porla_secp256k1_ecmult_multi_table_batch(C.c_void_p(self.handle), first, _scalar_array(scalars[:n * batch]),
                                                             n, batch, r)
        return (ok, [_affine_or_none(g) for g in r[:batch]]) if ok else (0, None)

    def align_mac_batch(self, data: bytearray, batch: int, n_chunks: int):
        """Server::align_MAC, IPA branch, for `batch` blocks of n_chunks chunks over generators [0, n_chunks): data =
        batch*n_chunks*64 bytes of LE values below PRIME_MODULUS*n, reduced mod PRIME_MODULUS in place.  Returns (the C
        entry's result, a ctypes array of `batch` SecpGej alignments)."""
        out = (SecpGej * max(1, batch))()
        ok = load().porla_secp256k1_align_mac_batch(C.c_void_p(self.handle), n_chunks, _as_void_p(data) if data else None,
                                                    batch, out)
        return ok, out

    def audit_aggregate(self, coefs: bytes, blocks: bytes, n: int, n_chunks: int):
        """Server::audit's B = sum coef_j * block_j, then align_MAC on B: coefs n x 4 B LE, blocks n x n_chunks x 64 B LE.
        Returns (the C entry's result, B % PRIME_MODULUS as n_chunks x 32 B LE, the alignment as a SecpGej)."""
        b_out, al = bytearray(32 * n_chunks), SecpGej()
        cf, bl = bytearray(coefs), bytearray(blocks)
        ok = load().porla_secp256k1_audit_aggregate(C.c_void_p(self.handle), n_chunks, _as_void_p(cf) if cf else None,
                                                    _as_void_p(bl) if bl else None, n, _as_void_p(b_out) if b_out else None,
                                                    C.byref(al))
        return ok, bytes(b_out), al

    def inner_product_prove(self, a: Sequence[int], b: Sequence[int]) -> bytes:
        """Server::inner_product_prove (Server.hpp:2279-2443); the table must hold the generators followed by u."""
        n = self.n - 1
        buf = C.create_string_buffer(32 + 66 * max(0, n.bit_length() - 2) + 128)
        ln = load().porla_secp256k1_inner_product_prove(C.c_void_p(self.handle), n,
                                                        b"".join((x % (1 << 256)).to_bytes(32, "little") for x in a),
                                                        b"".join((x % (1 << 256)).to_bytes(32, "little") for x in b), buf)
        return buf.raw[:ln]

    def inner_product_verify(self, commitment, proof: bytes) -> bool:
        """Client::inner_product_verify (Client.hpp:1465-1630); commitment: affine point or None."""
        g = SecpGej()
        if commitment is None:
            g.infinity = 1
        else:
            g.x, g.y, g.infinity = _int_to_fe(commitment[0]), _int_to_fe(commitment[1]), 0
            g.z = _int_to_fe(1)
        return bool(load().porla_secp256k1_inner_product_verify(C.c_void_p(self.handle), self.n - 1, C.byref(g), proof))

    def destroy(self) -> None:
        if self.handle:
            load().porla_table_destroy(C.c_void_p(self.handle))
            self.handle = 0


def secp256k1_butterfly_stage(gejs, m: int, twiddles: Sequence[int]) -> int:
    """One stage of the FFT in the exponent on IPA-mode MACs, in place on `gejs` (a ctypes array of SecpGej: any z, any
    field magnitude).  twiddles: m/2 integers below 2^256, taken mod n.  Returns the C entry's result (0: m is not a power
    of two >= 2 dividing len(gejs), buffer untouched)."""
    tw = (SecpScalar * max(1, len(twiddles)))()
    for k, w in enumerate(twiddles):
        for i in range(4):
            tw[k].d[i] = (w >> (64 * i)) & 0xFFFFFFFFFFFFFFFF
    return load().porla_secp256k1_butterfly_stage(gejs, len(gejs), m, tw)


def secp256k1_ecmult_multi_gej(gejs, scalars: Sequence[int], n: int, nbatch: int = 1):
    """r[b] = sum_i scalars[b*n + i] * gejs[b*n + i] on MACs as stored (a ctypes array of SecpGej: any z, any field
    magnitude); scalars: n*nbatch integers below 2^256, taken mod the group order.  Returns (the C entry's result, a
    ctypes array of nbatch SecpGej with z = 1)."""
    r = (SecpGej * max(1, nbatch))()
    return load().porla_secp256k1_ecmult_multi_gej(gejs, _scalar_array(scalars[:n * nbatch]), n, nbatch, r), r


def secp256k1_ecmult_const_batch(base: SecpGenerators, scalars: Sequence[int]):
    """The client's MAC complements in one call: scalars[i] * h for the one point h of `base` (a SecpGenerators of length
    1).  scalars: integers below 2^256, taken mod the group order.  Returns (ok, list of affine results or None), or
    (0, None) when the base is refused."""
    r = (SecpGej * max(1, len(scalars)))()
    ok = load().porla_secp256k1_ecmult_const_batch(C.c_void_p(base.handle), _scalar_array(scalars), len(scalars), r)
    return (ok, [_affine_or_none(g) for g in r[:len(scalars)]]) if ok else (0, None)


def secp256k1_ecmult_multi_var(scalars: Sequence[int], points: Sequence, g_scalar: Optional[int] = None):
    """Drive the IPA adapter exactly as utils.h:166-178 does: scalars/points are delivered one
    index at a time through the callback.  points: affine (x, y) tuples or None for infinity.
    Returns (ok, affine result or None)."""
    lib = load()
    n = len(scalars)

    def cb(sc_p, pt_p, idx, _data):
        s = scalars[idx]
        for i in range(4):
            sc_p.contents.d[i] = (s >> (64 * i)) & 0xFFFFFFFFFFFFFFFF
        P = points[idx]
        if P is None:
            C.memset(pt_p, 0, C.sizeof(SecpGe))
            pt_p.contents.infinity = 1
        else:
            pt_p.contents.x = _int_to_fe(P[0])
            pt_p.contents.y = _int_to_fe(P[1])
            pt_p.contents.infinity = 0
        return 1

    r = SecpGej()
    gs = None
    if g_scalar is not None:
        gs = SecpScalar()
        for i in range(4):
            gs.d[i] = (g_scalar >> (64 * i)) & 0xFFFFFFFFFFFFFFFF
    ok = lib.porla_secp256k1_ecmult_multi_var(None, None, C.byref(r), C.byref(gs) if gs is not None else None, SECP_CB(cb), None, n)
    if r.infinity:
        return ok, None
    assert _fe_to_int(r.z) == 1
    return ok, (_fe_to_int(r.x), _fe_to_int(r.y))
