"""ctypes bindings for the CPU oracle (oracle/liboracle.so) and, when it has been
built, the unmodified reference (oracle/_ref/libsnappy_ref.so).

Test infrastructure only: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  The product never imports it.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "liboracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libsnappy_ref.so")
REF_BIN = os.path.join(ORACLE_DIR, "_ref", "snappy_ref")

MODE_HASH, MODE_BST = 0, 1
BLOCK = 65536

_u8p = C.POINTER(C.c_uint8)


def build(ref: bool = True) -> None:
    """Compile oracle/ (and oracle/_ref when the reference sources are present: oracle/Makefile)."""
    targets = ["all"] + (["ref"] if ref else [])
    import sys
    # (make's chatter goes to stderr: bench.py's stdout is one JSON line)
    subprocess.run(["make", "-s", "-C", ORACLE_DIR] + targets, check=True, stdout=sys.stderr)


def _as_u8(buf) -> np.ndarray:
    if isinstance(buf, np.ndarray):
        return np.ascontiguousarray(buf, dtype=np.uint8)
    return np.frombuffer(bytes(buf), dtype=np.uint8)


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(_u8p)


class Oracle:
    """Our C restatement (oracle/snappy_oracle.c)."""

    def __init__(self):
        if not os.path.exists(ORACLE_SO):
            build(ref=False)
        L = C.CDLL(ORACLE_SO)
        L.oracle_varint_encode.restype = C.c_uint
        L.oracle_varint_encode.argtypes = [C.c_uint64, _u8p]
        L.oracle_varint_decode.restype = C.c_uint
        L.oracle_varint_decode.argtypes = [_u8p, C.c_size_t, C.POINTER(C.c_uint64)]
        L.oracle_max_compressed_size.restype = C.c_uint64
        L.oracle_max_compressed_size.argtypes = [C.c_uint64]
        L.oracle_compress.restype = C.c_uint64
        L.oracle_compress.argtypes = [_u8p, C.c_uint64, _u8p, C.c_int, C.POINTER(C.c_uint32)]
        L.oracle_decompress.restype = C.c_int
        L.oracle_decompress.argtypes = [_u8p, C.c_uint64, _u8p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.oracle_block_index.restype = C.c_int64
        L.oracle_block_index.argtypes = [_u8p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        self.L = L

    def varint_encode(self, v: int) -> bytes:
        buf = np.zeros(16, dtype=np.uint8)
        k = self.L.oracle_varint_encode(v, _ptr(buf))
        return buf[:k].tobytes()

    def varint_decode(self, data) -> tuple[int, int]:
        a = _as_u8(data)
        out = C.c_uint64(0)
        k = self.L.oracle_varint_decode(_ptr(a), a.size, C.byref(out))
        return out.value, k

    def compress(self, data, mode: int = MODE_HASH, with_sizes: bool = False):
        a = _as_u8(data)
        cap = self.L.oracle_max_compressed_size(a.size)
        out = np.empty(cap, dtype=np.uint8)
        nb = (a.size + BLOCK - 1) // BLOCK
        sizes = np.zeros(max(nb, 1), dtype=np.uint32)
        n = self.L.oracle_compress(_ptr(a), a.size, _ptr(out), mode, sizes.ctypes.data_as(C.POINTER(C.c_uint32)))
        res = out[:n].copy()
        return (res, sizes[:nb]) if with_sizes else res

    def decompress(self, stream, cap: int | None = None) -> np.ndarray:
        a = _as_u8(stream)
        if cap is None:
            cap, _ = self.varint_decode(a[:10])
        out = np.empty(max(cap, 1), dtype=np.uint8)
        n = C.c_uint64(0)
        rc = self.L.oracle_decompress(_ptr(a), a.size, _ptr(out), cap, C.byref(n))
        if rc != 0:
            raise ValueError(f"oracle_decompress error {rc}")
        return out[: n.value].copy()

    def block_index(self, stream) -> tuple[np.ndarray, int]:
        a = _as_u8(stream)
        total, _ = self.varint_decode(a[:10])
        offs = np.zeros((total + BLOCK - 1) // BLOCK + 1, dtype=np.uint64)
        tot = C.c_uint64(0)
        nb = self.L.oracle_block_index(_ptr(a), a.size, offs.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(tot))
        if nb < 0:
            raise ValueError(f"oracle_block_index error {-nb}")
        return offs[: nb + 1].copy(), tot.value


class Reference:
    """The unmodified reference, compiled from its own sources by oracle/Makefile (`make ref`)."""

    def __init__(self):
        if not os.path.exists(REF_SO):
            raise FileNotFoundError(REF_SO)
        L = C.CDLL(REF_SO)
        L.ref_compress.restype = C.c_uint64
        L.ref_compress.argtypes = [_u8p, C.c_uint64, _u8p, C.c_uint64, C.c_int]
        L.ref_decompress.restype = C.c_uint64
        L.ref_decompress.argtypes = [_u8p, C.c_uint64, _u8p, C.c_uint64]
        L.parse_to_varint.restype = C.c_uint
        L.parse_to_varint.argtypes = [C.c_ulonglong, _u8p]
        L.str_varint_to_dim_.restype = C.c_int
        L.str_varint_to_dim_.argtypes = [_u8p]
        self.L = L

    @staticmethod
    def available() -> bool:
        return os.path.exists(REF_SO)

    def compress(self, data, mode: int = MODE_HASH) -> np.ndarray:
        a = _as_u8(data)
        cap = a.size + (a.size // BLOCK + 1) * 1024 + 64
        out = np.empty(cap, dtype=np.uint8)
        n = self.L.ref_compress(_ptr(a), a.size, _ptr(out), cap, mode)
        if n == 2**64 - 1:
            raise RuntimeError("ref_compress failed")
        return out[:n].copy()

    def decompress(self, stream, cap: int) -> np.ndarray:
        a = _as_u8(stream)
        out = np.empty(max(cap, 1), dtype=np.uint8)
        n = self.L.ref_decompress(_ptr(a), a.size, _ptr(out), cap)
        if n == 2**64 - 1:
            raise RuntimeError("ref_decompress failed")
        return out[:n].copy()

    def varint_encode(self, v: int) -> bytes:
        buf = np.zeros(16, dtype=np.uint8)
        k = self.L.parse_to_varint(v, _ptr(buf))
        return buf[:k].tobytes()

    def varint_decode(self, data) -> int:
        a = np.concatenate([_as_u8(data), np.zeros(4, dtype=np.uint8)])
        return self.L.str_varint_to_dim_(_ptr(a))
