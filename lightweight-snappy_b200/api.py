"""ctypes host mirror of libsnappy_b200.so (include/snappy_b200.h).

This module adds nothing to the codec: it loads the C-ABI library, checks that every
declared symbol is exported, and wraps the calls for numpy arrays (host-buffer API) and
torch CUDA tensors (device-level API; torch is only the owner of device memory and
streams).  There is no fallback of any kind: if the library is missing or a call fails,
an exception is raised.

Naming follows the reference's operator interface (src/snappy_compression.h:8,
src/snappy_compression_tree.h:10, src/snappy_decompression.h:15):
    snappy_compress(data)      -> stream   (hash-table path)
    snappy_compress_bst(data)  -> stream   (BST / exact-key path)
    snappy_decompress(stream)  -> data

MODE_PARALLEL selects the block-parallel parse: a valid Snappy stream in the same format that
every decoder reads, deterministic, but not byte-identical to the reference's.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsnappy_b200.so")
CLI_PATH = os.path.join(HERE, "snappy_b200")

BLOCK = 65536
SLOT_STRIDE = 66560
MODE_HASH, MODE_BST, MODE_PARALLEL = 0, 1, 2
OK = 0
ERR_CUDA, ERR_ARG, ERR_CAPACITY, ERR_CORRUPT, ERR_FRAMING, ERR_IO, ERR_CHECKSUM = -1, -2, -3, -4, -5, -6, -7
ST_CAPACITY, ST_CORRUPT, ST_FRAMING, ST_CHECKSUM = 1, 2, 4, 16

_u8p = C.c_void_p

# name -> (restype, argtypes); this is also the export list tests/test_abi.py checks
SIGNATURES = {
    "snappy_b200_last_error": (C.c_char_p, []),
    "snappy_b200_device_count": (C.c_int, []),
    "snappy_b200_launch_count": (C.c_uint64, []),
    "snappy_b200_index_rounds": (C.c_uint64, []),
    "snappy_b200_max_compressed_bytes": (C.c_uint64, [C.c_uint64]),
    "snappy_b200_block_count": (C.c_uint64, [C.c_uint64]),
    "snappy_b200_compress_workspace_bytes": (C.c_size_t, [C.c_uint64, C.c_int]),
    "snappy_b200_compress_device": (C.c_int, [_u8p, C.c_uint64, C.c_int, _u8p, C.c_uint64, _u8p, _u8p, _u8p, _u8p,
                                              C.c_size_t, C.c_void_p]),
    "snappy_b200_decompress_device_indexed": (C.c_int, [_u8p, _u8p, C.c_uint64, C.c_uint64, _u8p, _u8p, C.c_void_p]),
    "snappy_b200_index_workspace_bytes": (C.c_size_t, [C.c_uint64]),
    "snappy_b200_index_device": (C.c_int, [_u8p, C.c_uint64, C.c_uint64, C.c_uint64, _u8p, _u8p, _u8p, C.c_size_t,
                                           C.c_void_p]),
    "snappy_b200_decode_segments_device": (C.c_int, [_u8p, C.c_uint64, C.c_uint64, C.c_uint64, _u8p, _u8p, _u8p, _u8p,
                                                     C.c_size_t, C.c_void_p]),
    "snappy_b200_decompress_workspace_bytes": (C.c_size_t, [C.c_uint64, C.c_uint64]),
    "snappy_b200_decompress_device": (C.c_int, [_u8p, C.c_uint64, C.c_uint64, C.c_uint64, _u8p, _u8p, _u8p, _u8p,
                                                C.c_size_t, C.c_void_p]),
    "snappy_b200_decompress_async_workspace_bytes": (C.c_size_t, [C.c_uint64, C.c_uint64]),
    "snappy_b200_decompress_device_async": (C.c_int, [_u8p, C.c_uint64, C.c_uint64, C.c_uint64, _u8p, _u8p, _u8p, _u8p,
                                                      C.c_size_t, C.c_uint, C.c_void_p]),
    "snappy_b200_compress_host": (C.c_int, [_u8p, C.c_uint64, C.c_int, _u8p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "snappy_b200_uncompressed_length": (C.c_int, [_u8p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "snappy_b200_decompress_host": (C.c_int, [_u8p, C.c_uint64, _u8p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "snappy_b200_compress_host_indexed": (C.c_int, [_u8p, C.c_uint64, C.c_int, _u8p, C.c_uint64, C.POINTER(C.c_uint64),
                                                    _u8p]),
    "snappy_b200_decompress_host_indexed": (C.c_int, [_u8p, C.c_uint64, _u8p, C.c_uint64, _u8p, C.c_uint64,
                                                      C.POINTER(C.c_uint64)]),
    "snappy_b200_compress_host_multi": (C.c_int, [_u8p, C.c_uint64, C.c_int, _u8p, C.c_uint64, C.POINTER(C.c_uint64), _u8p,
                                                  C.c_int]),
    "snappy_b200_compress_host_range": (C.c_int, [_u8p, C.c_uint64, C.c_int, _u8p, C.c_uint64, C.POINTER(C.c_uint64), _u8p,
                                                  C.c_uint64]),
    "snappy_b200_compress_host_multi_range": (C.c_int, [_u8p, C.c_uint64, C.c_int, _u8p, C.c_uint64,
                                                        C.POINTER(C.c_uint64), _u8p, C.c_int, C.c_uint64]),
    "snappy_b200_decompress_host_multi": (C.c_int, [_u8p, C.c_uint64, _u8p, C.c_uint64, C.POINTER(C.c_uint64), C.c_int]),
    "snappy_b200_decompress_host_indexed_multi": (C.c_int, [_u8p, C.c_uint64, _u8p, C.c_uint64, _u8p, C.c_uint64,
                                                            C.POINTER(C.c_uint64), C.c_int]),
    "snappy_b200_decompress_file": (C.c_int, [C.c_void_p, C.c_void_p]),
    "snappy_b200_compress_file_indexed": (C.c_int, [C.c_void_p, C.c_ulonglong, C.c_int, C.c_void_p, C.c_void_p]),
    "snappy_b200_decompress_file_indexed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "snappy_b200_frame_max_compressed_bytes": (C.c_uint64, [C.c_uint64]),
    "snappy_b200_frame_compress_workspace_bytes": (C.c_size_t, [C.c_uint64, C.c_int]),
    "snappy_b200_frame_compress_device": (C.c_int, [_u8p, C.c_uint64, C.c_int, _u8p, C.c_uint64, _u8p, _u8p, _u8p,
                                                    C.c_size_t, C.c_void_p]),
    "snappy_b200_frame_compress_host": (C.c_int, [_u8p, C.c_uint64, C.c_int, _u8p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "snappy_b200_frame_uncompressed_length": (C.c_int, [_u8p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "snappy_b200_frame_decompress_host": (C.c_int, [_u8p, C.c_uint64, _u8p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "snappy_b200_frame_compress_file": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "snappy_b200_frame_decompress_file": (C.c_int, [C.c_void_p, C.c_void_p]),
    "snappy_b200_release": (None, []),
    "snappy_b200_host_alloc": (C.c_void_p, [C.c_size_t]),
    "snappy_b200_host_free": (None, [C.c_void_p]),
    # the reference's own symbols (drop-in layer)
    "snappy_compress": (None, [C.c_void_p, C.c_ulonglong, C.c_void_p]),
    "snappy_compress_bst": (C.c_int, [C.c_void_p, C.c_ulonglong, C.c_void_p]),
    "snappy_decompress": (C.c_int, [C.c_void_p, C.c_void_p]),
    "parse_to_varint": (C.c_uint, [C.c_ulonglong, _u8p]),
    "varint_to_dim": (C.c_int, [C.c_void_p]),
    "str_varint_to_dim_": (C.c_int, [_u8p]),
    "init_Buffer": (None, [C.c_void_p, C.c_uint]),
    "move_current": (None, [C.c_void_p, C.c_uint]),
    "reset": (None, [C.c_void_p]),
}


class SnappyError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libsnappy_b200 error {code}: {msg}")
        self.code = code


def build() -> None:
    """Compile libsnappy_b200.so + the CLI in-tree for sm_100a (make; nvcc cross-compiles)."""
    subprocess.run(["make", "-s", "-C", HERE], check=True)


_lib = None


def lib() -> C.CDLL:
    """The loaded C-ABI library.  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(f"{LIB_PATH} is missing: run `make -C {HERE}` (or __graft_entry__.build())")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the export is missing
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _check(rc: int) -> None:
    if rc != OK:
        raise SnappyError(rc, lib().snappy_b200_last_error().decode(errors="replace"))


def max_compressed_bytes(n: int) -> int:
    return lib().snappy_b200_max_compressed_bytes(n)


def block_count(n: int) -> int:
    return (n + BLOCK - 1) // BLOCK


# ------------------------------------------------------------------ host-buffer API (numpy)
def _host_u8(buf) -> np.ndarray:
    if isinstance(buf, np.ndarray):
        return np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
    if hasattr(buf, "numpy") and hasattr(buf, "is_cuda"):  # torch CPU tensor (possibly pinned)
        return buf.contiguous().view(-1).numpy().view(np.uint8)
    return np.frombuffer(bytes(buf), dtype=np.uint8)


def compress_host(data, mode: int = MODE_HASH, out: np.ndarray | None = None) -> np.ndarray:
    a = _host_u8(data)
    cap = max_compressed_bytes(a.size)
    if out is None:
        out = np.empty(max(cap, 1), dtype=np.uint8)
    n = C.c_uint64(0)
    _check(lib().snappy_b200_compress_host(a.ctypes.data, a.size, mode, out.ctypes.data, out.size, C.byref(n)))
    return out[: n.value]


def compress_host_indexed(data, mode: int = MODE_HASH) -> tuple[np.ndarray, np.ndarray]:
    """Stream + side index (u64 block offsets, block_count + 1 entries)."""
    a = _host_u8(data)
    out = np.empty(max(max_compressed_bytes(a.size), 1), dtype=np.uint8)
    offs = np.zeros(block_count(a.size) + 1, dtype=np.uint64)
    n = C.c_uint64(0)
    _check(lib().snappy_b200_compress_host_indexed(a.ctypes.data, a.size, mode, out.ctypes.data, out.size, C.byref(n),
                                                   offs.ctypes.data))
    return out[: n.value], offs


def decompress_host_indexed(stream, block_offsets, out: np.ndarray | None = None) -> np.ndarray:
    a = _host_u8(stream)
    offs = np.ascontiguousarray(block_offsets, dtype=np.uint64)
    total = uncompressed_length(a)
    if out is None:
        out = np.empty(max(total, 1), dtype=np.uint8)
    n = C.c_uint64(0)
    _check(lib().snappy_b200_decompress_host_indexed(a.ctypes.data, a.size, offs.ctypes.data, offs.size - 1,
                                                     out.ctypes.data, out.size, C.byref(n)))
    return out[: n.value]


def compress_host_multi(data, mode: int = MODE_HASH, n_devices: int = 8, with_index: bool = False):
    """The host-buffer compressor over the first n_devices GPUs (block ranges per device, no collective)."""
    a = _host_u8(data)
    out = np.empty(max(max_compressed_bytes(a.size), 1), dtype=np.uint8)
    offs = np.zeros(block_count(a.size) + 1, dtype=np.uint64)
    n = C.c_uint64(0)
    _check(lib().snappy_b200_compress_host_multi(a.ctypes.data, a.size, mode, out.ctypes.data, out.size, C.byref(n),
                                                 offs.ctypes.data if with_index else None, n_devices))
    return (out[: n.value], offs) if with_index else out[: n.value]


def decompress_host_multi(stream, n_devices: int = 8, block_offsets=None, out: np.ndarray | None = None) -> np.ndarray:
    a = _host_u8(stream)
    total = uncompressed_length(a)
    if out is None:
        out = np.empty(max(total, 1), dtype=np.uint8)
    n = C.c_uint64(0)
    if block_offsets is None:
        _check(lib().snappy_b200_decompress_host_multi(a.ctypes.data, a.size, out.ctypes.data, out.size, C.byref(n),
                                                       n_devices))
    else:
        offs = np.ascontiguousarray(block_offsets, dtype=np.uint64)
        _check(lib().snappy_b200_decompress_host_indexed_multi(a.ctypes.data, a.size, offs.ctypes.data, offs.size - 1,
                                                               out.ctypes.data, out.size, C.byref(n), n_devices))
    return out[: n.value]


def uncompressed_length(stream) -> int:
    a = _host_u8(stream)
    n = C.c_uint64(0)
    _check(lib().snappy_b200_uncompressed_length(a.ctypes.data, min(a.size, 16), C.byref(n)))
    return n.value


def decompress_host(stream, out: np.ndarray | None = None) -> np.ndarray:
    a = _host_u8(stream)
    total = uncompressed_length(a)
    if out is None:
        out = np.empty(max(total, 1), dtype=np.uint8)
    n = C.c_uint64(0)
    _check(lib().snappy_b200_decompress_host(a.ctypes.data, a.size, out.ctypes.data, out.size, C.byref(n)))
    return out[: n.value]


def snappy_compress(data) -> np.ndarray:
    """Hash-table path; stream byte-identical to the reference's snappy_compress."""
    return compress_host(data, MODE_HASH)


def snappy_compress_bst(data) -> np.ndarray:
    """BST (exact-key) path; stream byte-identical to the reference's snappy_compress_bst."""
    return compress_host(data, MODE_BST)


def snappy_decompress(stream) -> np.ndarray:
    return decompress_host(stream)


# ------------------------------------------------------------------ framing format (.sz, framing_format.txt)
def compress_framed(data, mode: int = MODE_HASH) -> np.ndarray:
    """A framed stream: the stream identifier, then one CRC-checked chunk per 64 KiB block."""
    a = _host_u8(data)
    out = np.empty(int(lib().snappy_b200_frame_max_compressed_bytes(a.size)), dtype=np.uint8)
    n = C.c_uint64(0)
    _check(lib().snappy_b200_frame_compress_host(a.ctypes.data, a.size, mode, out.ctypes.data, out.size, C.byref(n)))
    return out[: n.value]


def framed_uncompressed_length(stream) -> int:
    """Total uncompressed length of a framed stream; walks the chunk headers on the host (no device needed)."""
    a = _host_u8(stream)
    n = C.c_uint64(0)
    _check(lib().snappy_b200_frame_uncompressed_length(a.ctypes.data, a.size, C.byref(n)))
    return n.value


def decompress_framed(stream, out: np.ndarray | None = None) -> np.ndarray:
    """Decodes a framed stream; SnappyError with code ERR_CHECKSUM when a chunk's CRC-32C does not match."""
    a = _host_u8(stream)
    total = framed_uncompressed_length(a)
    if out is None:
        out = np.empty(max(total, 1), dtype=np.uint8)
    n = C.c_uint64(0)
    _check(lib().snappy_b200_frame_decompress_host(a.ctypes.data, a.size, out.ctypes.data, out.size, C.byref(n)))
    return out[: n.value]


# ------------------------------------------------------------------ device-level API (torch)
class DeviceCodec:
    """Pre-allocated device buffers for repeated device-resident calls on one size class.

    All tensors live on the current CUDA device; calls are enqueued on torch's current
    stream and are asynchronous.  The workspace fits every mode, MODE_PARALLEL included, whose
    candidate offsets take 2 bytes per byte of max_bytes on top of what the other modes need.  `status` / `out_bytes` are device scalars: read them
    (which synchronises) when the result is needed.
    """

    def __init__(self, max_bytes: int, device="cuda"):
        import torch

        self.torch = torch
        self.device = torch.device(device)
        self.max_bytes = max_bytes
        nb = block_count(max_bytes)
        L = lib()
        self.comp_capacity = max(int(L.snappy_b200_max_compressed_bytes(max_bytes)), 16)
        ws = max(*(int(L.snappy_b200_compress_workspace_bytes(max_bytes, m)) for m in (MODE_BST, MODE_PARALLEL)),
                 int(L.snappy_b200_index_workspace_bytes(self.comp_capacity)),
                 int(L.snappy_b200_decompress_workspace_bytes(self.comp_capacity, max_bytes)),
                 int(L.snappy_b200_decompress_async_workspace_bytes(self.comp_capacity, max_bytes)),
                 *(int(L.snappy_b200_frame_compress_workspace_bytes(max_bytes, m)) for m in (MODE_BST, MODE_PARALLEL)))
        self.workspace = torch.empty(ws + 256, dtype=torch.uint8, device=self.device)
        self.stream_buf = torch.empty(self.comp_capacity + 256, dtype=torch.uint8, device=self.device)
        self.block_offsets = torch.zeros(nb + 1, dtype=torch.int64, device=self.device)
        self.out_bytes = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.status = torch.zeros(1, dtype=torch.int32, device=self.device)

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def compress(self, data, mode: int = MODE_HASH):
        """data: uint8 CUDA tensor.  Fills stream_buf / out_bytes / block_offsets / status."""
        n = data.numel()
        assert data.is_cuda and data.dtype == self.torch.uint8 and data.is_contiguous() and n <= self.max_bytes
        _check(lib().snappy_b200_compress_device(
            data.data_ptr(), n, mode, self.stream_buf.data_ptr(), self.comp_capacity, self.out_bytes.data_ptr(),
            self.block_offsets.data_ptr(), self.status.data_ptr(), self.workspace.data_ptr(),
            self.workspace.numel(), self._stream()))

    def compress_framed(self, data, mode: int = MODE_HASH):
        """data: uint8 CUDA tensor.  A framed stream into stream_buf / out_bytes / status (enqueue only)."""
        n = data.numel()
        assert data.is_cuda and data.dtype == self.torch.uint8 and data.is_contiguous() and n <= self.max_bytes
        _check(lib().snappy_b200_frame_compress_device(
            data.data_ptr(), n, mode, self.stream_buf.data_ptr(), self.stream_buf.numel(), self.out_bytes.data_ptr(),
            self.status.data_ptr(), self.workspace.data_ptr(), self.workspace.numel(), self._stream()))

    def decompress_indexed(self, stream_t, block_offsets, total_out: int, out):
        """Decodes with a known block index (e.g. the one compress() produced)."""
        self.status.zero_()
        _check(lib().snappy_b200_decompress_device_indexed(
            stream_t.data_ptr(), block_offsets.data_ptr(), block_count(total_out), total_out, out.data_ptr(),
            self.status.data_ptr(), self._stream()))

    def decompress(self, stream_t, stream_bytes: int, body_offset: int, total_out: int, out, block_offsets=None):
        """Index-less decode: K0 + segment-driven decoder (synchronises between K0 rounds)."""
        if block_offsets is None:
            block_offsets = self.block_offsets
        self.status.zero_()
        _check(lib().snappy_b200_decompress_device(
            stream_t.data_ptr(), stream_bytes, body_offset, total_out, out.data_ptr(), block_offsets.data_ptr(),
            self.status.data_ptr(), self.workspace.data_ptr(), self.workspace.numel(), self._stream()))
        return block_offsets

    def decompress_async(self, stream_t, stream_bytes: int, body_offset: int, total_out: int, out, block_offsets=None,
                         max_rounds: int = 64, zero_status: bool = True):
        """Index-less decode, enqueue-only (no host synchronisation: may be captured into a CUDA graph).
        K0 runs a fixed batch of `max_rounds` self-terminating relaxation rounds; status gets
        ST_UNRESOLVED if the stream needed more."""
        if zero_status:
            self.status.zero_()
        _check(lib().snappy_b200_decompress_device_async(
            stream_t.data_ptr(), stream_bytes, body_offset, total_out, out.data_ptr(),
            block_offsets.data_ptr() if block_offsets is not None else None,
            self.status.data_ptr(), self.workspace.data_ptr(), self.workspace.numel(), max_rounds, self._stream()))

    def decode_segments(self, stream_t, stream_bytes: int, body_offset: int, total_out: int, out, block_offsets):
        """Second half of decompress(): needs the workspace as index() left it (status is kept)."""
        _check(lib().snappy_b200_decode_segments_device(
            stream_t.data_ptr(), stream_bytes, body_offset, total_out, out.data_ptr(), block_offsets.data_ptr(),
            self.status.data_ptr(), self.workspace.data_ptr(), self.workspace.numel(), self._stream()))

    def index(self, stream_t, stream_bytes: int, body_offset: int, total_out: int, block_offsets=None):
        """K0: block boundaries of an index-less stream (synchronises between rounds)."""
        if block_offsets is None:
            block_offsets = self.block_offsets
        self.status.zero_()
        _check(lib().snappy_b200_index_device(
            stream_t.data_ptr(), stream_bytes, body_offset, total_out, block_offsets.data_ptr(),
            self.status.data_ptr(), self.workspace.data_ptr(), self.workspace.numel(), self._stream()))
        return block_offsets

    def result_stream(self):
        """The compressed stream of the last compress() as a tensor view (synchronises)."""
        st = int(self.status.item())
        if st:
            raise SnappyError(-st, f"device status 0x{st:x}")
        return self.stream_buf[: int(self.out_bytes.item())]

    def check_status(self):
        st = int(self.status.item())
        if st:
            raise SnappyError(-st, f"device status 0x{st:x}")


def device_count() -> int:
    return int(lib().snappy_b200_device_count())


def index_rounds() -> int:
    return int(lib().snappy_b200_index_rounds())


def launch_count() -> int:
    return int(lib().snappy_b200_launch_count())
